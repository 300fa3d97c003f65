// Test-only driver of lld::PnPsolver (lld_slam_b200/host/lld_shim.h) in Tracking::Relocalization's loop: one POD current
// frame (keypoints with octaves, mvLevelSigma2) and per relocalisation candidate c a vpMapPointMatches over the frame's
// keypoints, from the arrays written by tests/test_pnp_ransac.py: candidate c owns the keypoints [coff[c], coff[c+1]) (kind 0
// a good map point, 1 no map point, 2 a bad map point); every other entry of its vector is null.  Rounds of
// PnPsolver::IterateBatch(5) over the candidates neither found nor discarded (SetRansacParameters(0.99, 10, 300, 4, 0.5,
// 5.991)); a candidate with bNoMore is discarded, a candidate that returns a pose is done.  Draws come from the injected rand()
// values `rands`.  Dumps per candidate the round of its pose (-1: none), nInliers, the pose, vbInliers over the frame's
// keypoints and mnIterations; one candidate is also run alone through iterate() to check it against IterateBatch.
//   shim_pnp_ransac <in.bin> <out.bin>
// Built against liblldba.so (GPU) and, with -DLLD_SHIM_ORACLE, against tests/hostcheck/libpnp_ransac_oracle.so.
#ifdef LLD_SHIM_ORACLE
#define lld_pnp_ransac lldo_pnp_ransac
#define lld_pnp_ransac_params lldo_pnp_ransac_params
#endif
#include <cstdio>
#include <map>
#include <memory>
#include <string>

#include "../../lld_slam_b200/host/lld_shim.h"

#ifdef LLD_SHIM_ORACLE
extern "C" {
int lldo_pnp_ransac(void*, const lld_pnp_ransac_problem*, lld_pnp_ransac_result*);
int lldo_pnp_ransac_params(int32_t, double, int32_t, int32_t, int32_t, float, int32_t*);
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
  if (argc != 3 || !read_all(argv[1])) { fprintf(stderr, "usage: shim_pnp_ransac <in.bin> <out.bin>\n"); return 2; }
  void* ctx = nullptr;
#ifndef LLD_SHIM_ORACLE
  if (lld_ctx_create(0, &ctx)) { fprintf(stderr, "lld_ctx_create failed\n"); return 3; }
#endif
  const int nc = (int)(g_in.at("coff").size() / 4) - 1;
  const int* coff = in<int>("coff");
  const int* kind = in<int>("kind");
  const float* cam = in<float>("cam");
  const int* rands = in<int>("rands");
  const size_t n_rands = g_in.at("rands").size() / 4;
  size_t next_rand = 0;
  auto random_int = [&](int mn, int mx) {   // DUtils::Random::RandomInt on the injected rand() values
    const int d = mx - mn + 1;
    const int r = next_rand < n_rands ? rands[next_rand++] : 0;
    return int(((double)r / ((double)RAND_MAX + 1.0)) * d) + mn;
  };
  lld::Frame F;
  F.fx = cam[0]; F.fy = cam[1]; F.cx = cam[2]; F.cy = cam[3];
  F.N = coff[nc];
  const size_t nl = g_in.at("level_sigma2").size() / 4;
  F.mvLevelSigma2.assign(in<float>("level_sigma2"), in<float>("level_sigma2") + nl);
  for (int i = 0; i < F.N; i++) F.mvKeysUn.push_back({in<float>("kp")[2 * i], in<float>("kp")[2 * i + 1], in<int>("oct")[i], 0.f});
  std::vector<std::unique_ptr<lld::MapPoint>> pts;
  std::vector<std::unique_ptr<lld::PnPsolver>> solvers;
  for (int c = 0; c < nc; c++) {
    std::vector<lld::MapPoint*> vpMapPointMatches((size_t)F.N, nullptr);
    for (int i = coff[c]; i < coff[c + 1]; i++) {
      if (kind[i] == 1) continue;
      pts.emplace_back(new lld::MapPoint());
      for (int k = 0; k < 3; k++) pts.back()->pos[k] = in<float>("Xw")[3 * i + k];
      pts.back()->bad = kind[i] == 2;
      vpMapPointMatches[(size_t)i] = pts.back().get();
    }
    solvers.emplace_back(new lld::PnPsolver(F, vpMapPointMatches));
    solvers.back()->SetRansacParameters(0.99, 10, 300, 4, 0.5, 5.991);
    solvers.back()->RandomInt = random_int;
  }
  std::vector<int> found_round((size_t)nc, -1), n_in((size_t)nc, 0), its((size_t)nc, 0);
  std::vector<float> T(12 * (size_t)nc, 0.f);
  std::vector<uint8_t> inl((size_t)nc * (size_t)F.N, 0);
  std::vector<bool> done((size_t)nc, false);
  int rounds = 0;
  for (int live = nc; live > 0; rounds++) {
    std::vector<lld::PnPsolver*> batch;
    std::vector<int> ids;
    for (int c = 0; c < nc; c++)
      if (!done[(size_t)c]) { batch.push_back(solvers[(size_t)c].get()); ids.push_back(c); }
    const int rc = lld::PnPsolver::IterateBatch(ctx, batch, 5);
    if (rc) { fprintf(stderr, "IterateBatch: %d\n", rc); return 5; }
    for (size_t j = 0; j < ids.size(); j++) {
      const int c = ids[j];
      lld::PnPsolver* S = batch[j];
      its[(size_t)c] = S->Iterations();
      if (S->Found()) {
        found_round[(size_t)c] = rounds;
        n_in[(size_t)c] = S->NumInliers();
        S->GetTcw(&T[12 * (size_t)c]);
        for (int i = 0; i < F.N; i++) inl[(size_t)c * F.N + i] = S->Inliers()[(size_t)i];
      }
      if (S->Found() || S->NoMore()) { done[(size_t)c] = true; live--; }
    }
  }
  // iterate() on a fresh solver of candidate 0 with the draws IterateBatch consumed for it in the first round
  {
    std::vector<lld::MapPoint*> vp((size_t)F.N, nullptr);
    int k = 0;   // candidate 0's map points are the first ones created
    for (int i = coff[0]; i < coff[1]; i++)
      if (kind[i] != 1) vp[(size_t)i] = pts[(size_t)k++].get();
    lld::PnPsolver S(F, vp);
    S.SetRansacParameters(0.99, 10, 300, 4, 0.5, 5.991);
    size_t r1 = 0;
    S.RandomInt = [&](int mn, int mx) {
      const int d = mx - mn + 1;
      return int(((double)rands[r1++] / ((double)RAND_MAX + 1.0)) * d) + mn;
    };
    bool bNoMore = false;
    std::vector<bool> vbInliers;
    int nInliers = -1;
    float Tcw[12] = {0};
    const bool got = S.iterate(ctx, 5, bNoMore, vbInliers, nInliers, Tcw);
    const int one[3] = {got ? 1 : 0, bNoMore ? 1 : 0, nInliers};
    out("one_flags", 'i', one, 3);
    out("one_Tcw", 'f', Tcw, 12);
    std::vector<uint8_t> m((size_t)F.N, 0);
    for (size_t i = 0; i < vbInliers.size(); i++) m[i] = vbInliers[i];
    out("one_inlier", 'b', m.data(), m.size());
    const int nv = (int)vbInliers.size();
    out("one_n_vb", 'i', &nv, 1);
  }
  out("found_round", 'i', found_round.data(), found_round.size());
  out("n_in", 'i', n_in.data(), n_in.size());
  out("its", 'i', its.data(), its.size());
  out("Tcw", 'f', T.data(), T.size());
  out("inlier", 'b', inl.data(), inl.size());
  out("rounds", 'i', &rounds, 1);
  const int used = (int)next_rand;
  out("rands_used", 'i', &used, 1);
  FILE* f = fopen(argv[2], "wb");
  if (!f) return 4;
  for (auto& kv : g_out) {
    const uint32_t nl2 = (uint32_t)kv.first.size();
    const uint64_t nb = kv.second.size();
    fwrite(&nl2, 4, 1, f); fwrite(kv.first.data(), 1, nl2, f); fwrite(&g_type[kv.first], 1, 1, f); fwrite(&nb, 8, 1, f);
    if (nb) fwrite(kv.second.data(), 1, nb, f);
  }
  fclose(f);
#ifndef LLD_SHIM_ORACLE
  lld_ctx_destroy(ctx);
#endif
  return 0;
}
