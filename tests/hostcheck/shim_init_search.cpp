// Test-only driver of lld::ORBmatcher::SearchForInitialization (lld_slam_b200/host/lld_shim.h): builds two POD Frames from a
// single-pair lld_init_search problem (written by tests/shim_io.py), runs the shim twice -- the second call takes vbPrevMatched
// from the first, as Tracking::MonocularInitialization does -- and dumps vnMatches12, vbPrevMatched and the counts.
//   shim_init_search <in.bin> <out.bin>
// Built against liblldba.so (GPU) and, with -DLLD_SHIM_ORACLE, against tests/hostcheck/libinit_search_oracle.so.
#ifdef LLD_SHIM_ORACLE
#define lld_init_search lldo_init_search
#endif
#include <cstdio>
#include <map>
#include <string>

#include "../../lld_slam_b200/host/lld_shim.h"

#ifdef LLD_SHIM_ORACLE
extern "C" {
int lldo_init_search(void*, const lld_init_search_problem*, lld_init_search_result*);
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
  if (argc != 3 || !read_all(argv[1])) { fprintf(stderr, "usage: shim_init_search <in.bin> <out.bin>\n"); return 2; }
  void* ctx = nullptr;
#ifndef LLD_SHIM_ORACLE
  if (lld_ctx_create(0, &ctx)) { fprintf(stderr, "lld_ctx_create failed\n"); return 3; }
#endif
  const int N1 = (int)(g_in.at("kp1_octave").size()), N2 = (int)(g_in.at("kp2_octave").size());
  const float* bounds = in<float>("bounds");
  lld::Frame F1, F2;
  for (lld::Frame* F : {&F1, &F2}) {
    F->mnMinX = bounds[0]; F->mnMaxX = bounds[1]; F->mnMinY = bounds[2]; F->mnMaxY = bounds[3];
    F->mvScaleFactors.assign(in<float>("scale_factors"), in<float>("scale_factors") + g_in.at("scale_factors").size() / 4);
  }
  for (int i = 0; i < N1; i++)
    F1.mvKeysUn.push_back({0.f, 0.f, (int)in<uint8_t>("kp1_octave")[i], in<float>("kp1_angle")[i]});
  F1.mDescriptors.assign(in<uint8_t>("kp1_desc"), in<uint8_t>("kp1_desc") + 32 * (size_t)N1);
  auto set_f2 = [&](const char* xy_key) {
    F2.mvKeysUn.clear();
    for (int i = 0; i < N2; i++)
      F2.mvKeysUn.push_back({in<float>(xy_key)[2 * i], in<float>(xy_key)[2 * i + 1], (int)in<uint8_t>("kp2_octave")[i], in<float>("kp2_angle")[i]});
  };
  F2.mDescriptors.assign(in<uint8_t>("kp2_desc"), in<uint8_t>("kp2_desc") + 32 * (size_t)N2);
  std::vector<lld::Point2f> prev;
  for (int i = 0; i < N1; i++) prev.push_back({in<float>("prev_matched")[2 * i], in<float>("prev_matched")[2 * i + 1]});
  const float* cfg = in<float>("config");   // window, nn_ratio, check_orientation
  lld::ORBmatcher matcher(cfg[1], cfg[2] != 0.f);
  std::vector<int> m12(7, 123);             // assigned by the call
  int n[2];
  for (int call = 0; call < 2; call++) {
    set_f2(call ? "kp2_xy_next" : "kp2_xy");
    n[call] = matcher.SearchForInitialization(ctx, F1, F2, prev, m12, (int)cfg[0]);
    std::vector<float> pm;
    for (auto& q : prev) { pm.push_back(q.x); pm.push_back(q.y); }
    out(call ? "match12_1" : "match12_0", 'i', m12.data(), m12.size());
    out(call ? "prev_1" : "prev_0", 'f', pm.data(), pm.size());
  }
  out("n_matches", 'i', n, 2);
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
