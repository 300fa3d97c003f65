// Test-only driver of lld::Sim3Solver (lld_slam_b200/host/lld_shim.h) in LoopClosing::ComputeSim3's loop: per loop candidate c
// two POD keyframes, their map points and vpMatched12 from the arrays written by tests/test_sim3_ransac.py (rows [coff[c],
// coff[c+1]); kind 0 is a valid correspondence, 1 no match, 2 no map point in KF1, 3 a bad KF1 point, 4 a bad matched point,
// 5 a matched point not observed in KF2).  Rounds of Sim3Solver::IterateBatch(5) over the candidates not yet discarded; in
// candidate order a candidate with bNoMore is discarded, a success goes through ToSim3 into Optimizer::OptimizeSim3(th2 = 10)
// with the RANSAC inliers, and the first candidate with nInliers >= 20 ends the loop.  Draws come from the injected rand()
// values `rands`.  Dumps the matched candidate, its g2oS12 and n_in, and every candidate's mnIterations / successes.
//   shim_sim3_ransac <in.bin> <out.bin>
// Built against liblldba.so (GPU) and, with -DLLD_SHIM_ORACLE, against the two oracle libraries of tests/hostcheck.
#ifdef LLD_SHIM_ORACLE
#define lld_sim3_opt lldo_sim3_opt
#define lld_sim3_ransac lldo_sim3_ransac
#endif
#include <cstdio>
#include <map>
#include <memory>
#include <string>

#include "../../lld_slam_b200/host/lld_shim.h"

#ifdef LLD_SHIM_ORACLE
extern "C" {
int lldo_sim3_opt(void*, const lld_sim3_problem*, lld_sim3_result*);
int lldo_sim3_ransac(void*, const lld_sim3_ransac_problem*, lld_sim3_ransac_result*);
int32_t lld_sim3_ransac_max_its(int32_t n_corr, double probability, int32_t min_inliers, int32_t max_iterations) {
  // the oracle build has no product library: the same host arithmetic
  if (n_corr < min_inliers) return 1;
  const float epsilon = (float)min_inliers / n_corr;
  int nIterations = 1;
  if (min_inliers != n_corr) {
    const double it = std::ceil(std::log(1 - probability) / std::log(1 - std::pow((double)epsilon, 3.0)));
    nIterations = it >= 2147483647.0 ? 2147483647 : (int)it;
  }
  return std::max(1, std::min(nIterations, max_iterations));
}
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
  if (argc != 3 || !read_all(argv[1])) { fprintf(stderr, "usage: shim_sim3_ransac <in.bin> <out.bin>\n"); return 2; }
  void* ctx = nullptr;
#ifndef LLD_SHIM_ORACLE
  if (lld_ctx_create(0, &ctx)) { fprintf(stderr, "lld_ctx_create failed\n"); return 3; }
#endif
  const int nc = (int)(g_in.at("coff").size() / 4) - 1;
  const int* coff = in<int>("coff");
  const int* kind = in<int>("kind");
  const float* cam = in<float>("cam");
  const bool fix = in<int>("fix")[0] != 0;
  const int* rands = in<int>("rands");
  const size_t n_rands = g_in.at("rands").size() / 4;
  size_t next_rand = 0;
  auto random_int = [&](int mn, int mx) {   // DUtils::Random::RandomInt on the injected rand() values
    const int d = mx - mn + 1;
    const int r = next_rand < n_rands ? rands[next_rand++] : 0;
    return int(((double)r / ((double)RAND_MAX + 1.0)) * d) + mn;
  };
  std::vector<std::unique_ptr<lld::KeyFrame>> kfs;
  std::vector<std::unique_ptr<lld::MapPoint>> pts;
  std::vector<std::vector<lld::MapPoint*>> matches((size_t)nc);
  std::vector<std::unique_ptr<lld::Sim3Solver>> solvers;
  std::vector<lld::KeyFrame*> kf1s, kf2s;
  for (int c = 0; c < nc; c++) {
    const int a = coff[c], n = coff[c + 1] - a;
    lld::KeyFrame* K[2];
    for (int s = 0; s < 2; s++) {
      kfs.emplace_back(new lld::KeyFrame());
      K[s] = kfs.back().get();
      for (int k = 0; k < 12; k++) K[s]->Tcw[k] = in<float>(s ? "T2" : "T1")[12 * c + k];
      K[s]->fx = cam[0]; K[s]->fy = cam[1]; K[s]->cx = cam[2]; K[s]->cy = cam[3];   // one camera for both keyframes
      const size_t nl = g_in.at("level_sigma2").size() / 4;
      K[s]->mvLevelSigma2.assign(in<float>("level_sigma2"), in<float>("level_sigma2") + nl);
      K[s]->mvInvLevelSigma2.assign(in<float>("inv_level_sigma2"), in<float>("inv_level_sigma2") + nl);
      for (int i = 0; i < n; i++) {
        const float* kp = in<float>(s ? "kp2" : "kp1") + 2 * (a + i);
        K[s]->mvKeysUn.push_back({kp[0], kp[1], in<int>(s ? "oct2" : "oct1")[a + i], 0.f});
      }
      K[s]->mvpMapPoints.assign((size_t)n, nullptr);
    }
    matches[(size_t)c].assign((size_t)n, nullptr);
    for (int i = 0; i < n; i++) {
      const int row = a + i;
      pts.emplace_back(new lld::MapPoint());
      lld::MapPoint* p1 = pts.back().get();
      pts.emplace_back(new lld::MapPoint());
      lld::MapPoint* p2 = pts.back().get();
      for (int k = 0; k < 3; k++) { p1->pos[k] = in<float>("X1w")[3 * row + k]; p2->pos[k] = in<float>("X2w")[3 * row + k]; }
      p1->observations[K[0]] = (size_t)i;
      if (kind[row] != 5) p2->observations[K[1]] = (size_t)i;
      if (kind[row] != 2) K[0]->mvpMapPoints[(size_t)i] = p1;
      p1->bad = kind[row] == 3;
      p2->bad = kind[row] == 4;
      if (kind[row] != 1) matches[(size_t)c][(size_t)i] = p2;
    }
    kf1s.push_back(K[0]); kf2s.push_back(K[1]);
    solvers.emplace_back(new lld::Sim3Solver(K[0], K[1], matches[(size_t)c], fix));
    solvers.back()->SetRansacParameters(0.99, 20, 300);
    solvers.back()->RandomInt = random_int;
  }
  std::vector<bool> discarded((size_t)nc, false);
  std::vector<int> successes((size_t)nc, 0);
  int matched = -1, n_in_matched = 0, rounds = 0;
  double S_out[8] = {0};
  for (int live = nc; live > 0 && matched < 0; rounds++) {
    std::vector<lld::Sim3Solver*> batch;
    std::vector<int> ids;
    for (int c = 0; c < nc; c++)
      if (!discarded[(size_t)c]) { batch.push_back(solvers[(size_t)c].get()); ids.push_back(c); }
    const int rc = lld::Sim3Solver::IterateBatch(ctx, batch, 5);
    if (rc) { fprintf(stderr, "IterateBatch: %d\n", rc); return 5; }
    for (size_t j = 0; j < ids.size(); j++) {
      const int c = ids[j];
      lld::Sim3Solver* S = batch[j];
      if (S->NoMore()) { discarded[(size_t)c] = true; live--; }
      if (!S->Found()) continue;
      successes[(size_t)c]++;
      std::vector<lld::MapPoint*> vpMapPointMatches(matches[(size_t)c].size(), nullptr);
      for (size_t k = 0; k < S->Inliers().size(); k++)
        if (S->Inliers()[k]) vpMapPointMatches[k] = matches[(size_t)c][k];
      float R[9], t[3];
      S->GetEstimatedRotation(R);
      S->GetEstimatedTranslation(t);
      lld::Sim3 gScm = lld::ToSim3(R, t, S->GetEstimatedScale());
      const int nInliers = lld::Optimizer::OptimizeSim3(ctx, kf1s[(size_t)c], kf2s[(size_t)c], vpMapPointMatches, gScm, 10, fix);
      if (nInliers < 0) return 6;
      if (nInliers >= 20) {
        matched = c;
        n_in_matched = nInliers;
        for (int k = 0; k < 4; k++) S_out[k] = gScm.q[k];
        for (int k = 0; k < 3; k++) S_out[4 + k] = gScm.t[k];
        S_out[7] = gScm.s;
        break;
      }
    }
  }
  out("matched", 'i', &matched, 1);
  out("n_in", 'i', &n_in_matched, 1);
  out("rounds", 'i', &rounds, 1);
  out("S12", 'd', S_out, 8);
  out("successes", 'i', successes.data(), successes.size());
  const int used = (int)next_rand;
  out("rands_used", 'i', &used, 1);
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
