// Test-only driver of lld::Optimizer::OptimizeSim3 (lld_slam_b200/host/lld_shim.h): builds two POD keyframes, their map points
// and vpMatches1 from the arrays written by tests/test_optimize_sim3.py (rows of kind 0 are valid correspondences; kind 1 has no
// match, 2 no map point in KF1, 3 a bad KF1 point, 4 a bad matched point, 5 a matched point not observed in KF2), runs the shim
// as LoopClosing::ComputeSim3 does, then once more with all but 8 correspondences moved far away (the early return), and dumps
// vpMatches1 (1 = set), g2oS12 and the return values.
//   shim_sim3 <in.bin> <out.bin>
// Built against liblldba.so (GPU) and, with -DLLD_SHIM_ORACLE, against tests/hostcheck/libsim3_oracle.so.
#ifdef LLD_SHIM_ORACLE
#define lld_sim3_opt lldo_sim3_opt
#endif
#include <cstdio>
#include <map>
#include <memory>
#include <string>

#include "../../lld_slam_b200/host/lld_shim.h"

#ifdef LLD_SHIM_ORACLE
extern "C" {
int lldo_sim3_opt(void*, const lld_sim3_problem*, lld_sim3_result*);
}
#endif

static std::map<std::string, std::vector<uint8_t>> g_in, g_out;
static std::map<std::string, char> g_type;

static bool read_all(const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) return false;
  for (;;) {
    uint32_t nl;
    if (fread(&nl, 4, 1, f) != 1) break;
    std::string name(nl, ' ');
    char t;
    uint64_t nb;
    if (fread(&name[0], 1, nl, f) != nl || fread(&t, 1, 1, f) != 1 || fread(&nb, 8, 1, f) != 1) return false;
    std::vector<uint8_t> b(nb);
    if (nb && fread(b.data(), 1, nb, f) != nb) return false;
    g_in[name] = b;
  }
  fclose(f);
  return true;
}
template <typename T> static const T* in(const char* k) { return reinterpret_cast<const T*>(g_in.at(k).data()); }
template <typename T> static void out(const char* k, char type, const T* p, size_t n) {
  g_out[k].assign(reinterpret_cast<const uint8_t*>(p), reinterpret_cast<const uint8_t*>(p) + n * sizeof(T));
  g_type[k] = type;
}

int main(int argc, char** argv) {
  if (argc != 3 || !read_all(argv[1])) { fprintf(stderr, "usage: shim_sim3 <in.bin> <out.bin>\n"); return 2; }
  void* ctx = nullptr;
#ifndef LLD_SHIM_ORACLE
  if (lld_ctx_create(0, &ctx)) { fprintf(stderr, "lld_ctx_create failed\n"); return 3; }
#endif
  const int N = (int)(g_in.at("kind").size() / 4);
  const int* kind = in<int>("kind");
  const float* cam = in<float>("cam");
  lld::KeyFrame KF1, KF2;
  for (int s = 0; s < 2; s++) {
    lld::KeyFrame& K = s ? KF2 : KF1;
    for (int c = 0; c < 12; c++) K.Tcw[c] = in<float>(s ? "T2" : "T1")[c];
    K.fx = cam[4 * s]; K.fy = cam[4 * s + 1]; K.cx = cam[4 * s + 2]; K.cy = cam[4 * s + 3];
    K.mvInvLevelSigma2.assign(in<float>("inv_level_sigma2"), in<float>("inv_level_sigma2") + g_in.at("inv_level_sigma2").size() / 4);
    for (int i = 0; i < N; i++) {
      const float* kp = in<float>(s ? "kp2" : "kp1") + 2 * i;
      K.mvKeysUn.push_back({kp[0], kp[1], in<int>(s ? "oct2" : "oct1")[i], 0.f});
    }
    K.mvpMapPoints.assign(N, nullptr);
  }
  std::vector<std::unique_ptr<lld::MapPoint>> pts;
  auto point = [&](const char* key, int i) {
    pts.emplace_back(new lld::MapPoint());
    for (int c = 0; c < 3; c++) pts.back()->pos[c] = in<float>(key)[3 * i + c];
    return pts.back().get();
  };
  std::vector<lld::MapPoint*> vpMatches1(N, nullptr);
  for (int i = 0; i < N; i++) {
    lld::MapPoint* p1 = point("X1w", i);
    lld::MapPoint* p2 = point("X2w", i);
    p1->observations[&KF1] = (size_t)i;
    if (kind[i] != 5) p2->observations[&KF2] = (size_t)i;
    if (kind[i] != 2) KF1.mvpMapPoints[i] = p1;
    p1->bad = kind[i] == 3;
    p2->bad = kind[i] == 4;
    if (kind[i] != 1) vpMatches1[i] = p2;
  }
  const double* S0 = in<double>("S12");
  auto sim3 = [&]() {
    lld::Sim3 S;
    for (int k = 0; k < 4; k++) S.q[k] = S0[k];
    for (int k = 0; k < 3; k++) S.t[k] = S0[4 + k];
    S.s = S0[7];
    return S;
  };
  auto dump = [](const lld::Sim3& S, double* o) {
    for (int k = 0; k < 4; k++) o[k] = S.q[k];
    for (int k = 0; k < 3; k++) o[4 + k] = S.t[k];
    o[7] = S.s;
  };
  const float th2 = in<float>("th2")[0];
  const bool fix = in<int>("fix")[0] != 0;
  std::vector<lld::MapPoint*> vpEarly = vpMatches1;
  lld::Sim3 S = sim3();
  const int n_in = lld::Optimizer::OptimizeSim3(ctx, &KF1, &KF2, vpMatches1, S, th2, fix);
  std::vector<int> matched;
  for (auto* p : vpMatches1) matched.push_back(p != nullptr);
  double so[8];
  dump(S, so);
  out("n_in", 'i', &n_in, 1);
  out("S12", 'd', so, 8);
  out("matched", 'i', matched.data(), matched.size());
  // all but 8 valid correspondences observed 300 px away in KF1: fewer than 10 survive round 1
  int kept = 0;
  for (int i = 0; i < N; i++)
    if (kind[i] == 0 && kept++ >= 8) KF1.mvKeysUn[i].x += 300.f;
  lld::Sim3 Se = sim3();
  const int n_early = lld::Optimizer::OptimizeSim3(ctx, &KF1, &KF2, vpEarly, Se, th2, fix);
  dump(Se, so);
  out("n_in_early", 'i', &n_early, 1);
  out("S12_early", 'd', so, 8);
  FILE* f = fopen(argv[2], "wb");
  if (!f) return 4;
  for (auto& kv : g_out) {
    const uint32_t nl = (uint32_t)kv.first.size();
    const uint64_t nb = kv.second.size();
    fwrite(&nl, 4, 1, f); fwrite(kv.first.data(), 1, nl, f); fwrite(&g_type[kv.first], 1, 1, f); fwrite(&nb, 8, 1, f);
    if (nb) fwrite(kv.second.data(), 1, nb, f);
  }
  fclose(f);
  return 0;
}
