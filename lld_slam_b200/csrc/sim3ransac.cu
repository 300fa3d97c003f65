// sim3ransac.cu — batched loop-candidate Sim3 RANSAC (Sim3Solver::iterate / ComputeSim3 / CheckInliers, ORB-SLAM2
// src/Sim3Solver.cc).
//
// One CTA per loop candidate, one warp per minimal set.  The CTA evaluates the candidate's sets in waves of NW: each warp
// forms the Horn estimate of its set (every lane the same, so nothing is broadcast) and counts the inliers over the
// candidate's correspondences, lanes striding over them, with __ballot_sync / __popc.  After a wave one thread applies
// iterate()'s sequential rule to the wave's counts in set order (mnIterations, the carried best, the strict success test) and
// stops the CTA at the first success.  The winner's inlier mask is then recomputed with the same arithmetic; per-set masks
// are never stored.  Correspondence data is read from global memory (a candidate's 300 correspondences are 9.6 KB and stay
// in L1 across the waves).
// Compiled with --fmad=false: the estimate and the projections mirror the reference's CV_32F operation order.
#include <algorithm>
#include <climits>
#include <cmath>

#include "lld_ctx.h"
#include "lld_math.cuh"

using namespace lld;

namespace {

constexpr int RTPB = 256;
constexpr int NW = RTPB / 32;

struct RansacView {
  const float* cam;
  const int* fix_scale;
  const int* off;
  const float* x1c;
  const float* x2c;
  const float* sig1;
  const float* sig2;
  int min_inliers;
  const int* max_its;
  const int* its_in;
  const int* best_in;
  int n_iterations;
  const int* hyp_off;
  const int* hyp_idx;
  uint8_t* found;
  uint8_t* no_more;
  int* n_inliers;
  float* T12;
  uint8_t* inlier;
  int* its_out;
  int* best_out;
  int* hyp_inliers;
};

__global__ void __launch_bounds__(RTPB) k_sim3_ransac(RansacView v) {
  __shared__ float s_est[NW][13];
  __shared__ int s_cnt[NW];
  __shared__ int s_win;   // -1: keep going, >= 0: the warp of the last wave whose set succeeded
  const int pb = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int e0 = v.off[pb], n = v.off[pb + 1] - e0;
  const int h0 = v.hyp_off[pb], B = v.hyp_off[pb + 1] - h0;
  const bool fix = v.fix_scale[pb] != 0;
  float K[8];
#pragma unroll
  for (int k = 0; k < 8; k++) K[k] = v.cam[8 * (size_t)pb + k];
  const float* X1 = v.x1c + 3 * (size_t)e0;
  const float* X2 = v.x2c + 3 * (size_t)e0;
  const float* S1 = v.sig1 + e0;
  const float* S2 = v.sig2 + e0;
  if (v.hyp_inliers)
    for (int k = tid; k < B; k += RTPB) v.hyp_inliers[h0 + k] = -1;
  int its = v.its_in[pb], best = v.best_in[pb];   // thread 0's copies are the ones written back
  if (tid == 0) s_win = -1;
  __syncthreads();
  for (int base = 0; base < B; base += NW) {
    const int k = base + w;
    if (k < B) {
      const int* id = v.hyp_idx + 3 * (size_t)(h0 + k);
      float P1[9], P2[9];
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const int i = id[j];
#pragma unroll
        for (int r = 0; r < 3; r++) {
          P1[3 * j + r] = X1[3 * (size_t)i + r];
          P2[3 * j + r] = X2[3 * (size_t)i + r];
        }
      }
      float R[9], t[3], s;
      sim3r_horn(P1, P2, fix, R, t, &s);
      Sim3Pair T;
      sim3r_pair(R, t, s, &T);
      int cnt = 0;
      for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        bool in = false;
        if (i < n) {
          float e[2];
          in = sim3r_inlier(T, X1 + 3 * (size_t)i, X2 + 3 * (size_t)i, S1[i], S2[i], K, e);
        }
        cnt += __popc(__ballot_sync(0xffffffffu, in));
      }
      if (lane == 0) {
        s_cnt[w] = cnt;
#pragma unroll
        for (int j = 0; j < 9; j++) s_est[w][j] = R[j];
        s_est[w][9] = t[0]; s_est[w][10] = t[1]; s_est[w][11] = t[2];
        s_est[w][12] = s;
      }
    }
    __syncthreads();
    if (tid == 0) {
      for (int j = 0; j < NW && base + j < B; j++) {   // iterate()'s loop body, in set order
        its++;
        const int c = s_cnt[j];
        if (v.hyp_inliers) v.hyp_inliers[h0 + base + j] = c;
        if (c >= best) {
          best = c;
          if (c > v.min_inliers) { s_win = j; break; }
        }
      }
    }
    __syncthreads();
    if (s_win >= 0) break;
  }
  const int win = s_win;
  const bool found = win >= 0;
  if (tid == 0) {
    v.found[pb] = found;
    v.no_more[pb] = n < v.min_inliers ? 1 : (!found && its >= v.max_its[pb]);
    v.its_out[pb] = its;
    v.best_out[pb] = best;
  }
  if (tid < 13) v.T12[13 * (size_t)pb + tid] = found ? s_est[win][tid] : 0.f;
  Sim3Pair T;
  if (found) sim3r_pair(s_est[win], s_est[win] + 9, s_est[win][12], &T);
  int cnt = 0;
  for (int i = tid; i < n; i += RTPB) {
    bool in = false;
    if (found) {
      float e[2];
      in = sim3r_inlier(T, X1 + 3 * (size_t)i, X2 + 3 * (size_t)i, S1[i], S2[i], K, e);
    }
    v.inlier[e0 + i] = in;
    cnt += in;
  }
  __syncthreads();
  if (tid == 0) s_cnt[0] = 0;
  __syncthreads();
  if (cnt) atomicAdd(&s_cnt[0], cnt);
  __syncthreads();
  if (tid == 0) v.n_inliers[pb] = found ? s_cnt[0] : 0;
}

}  // namespace

extern "C" int32_t lld_sim3_ransac_max_its(int32_t n_corr, double probability, int32_t min_inliers, int32_t max_iterations) {
  if (n_corr < min_inliers) return 1;
  const float epsilon = (float)min_inliers / n_corr;
  int nIterations;
  if (min_inliers == n_corr) {
    nIterations = 1;
  } else {
    const double it = std::ceil(std::log(1 - probability) / std::log(1 - std::pow((double)epsilon, 3.0)));
    nIterations = it >= (double)INT_MAX ? INT_MAX : (int)it;
  }
  return std::max(1, std::min(nIterations, max_iterations));
}

extern "C" int lld_sim3_ransac(void* ctx, const lld_sim3_ransac_problem* p, lld_sim3_ransac_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  const int n = p->n_problems;
  LLD_ARG(c, n >= 0);
  LLD_ARG(c, p->min_inliers >= 0);
  LLD_ARG(c, p->n_iterations >= 0);
  if (n == 0) return LLD_OK;
  LLD_ARG(c, p->off && p->off[0] == 0);
  LLD_ARG(c, p->hyp_off && p->hyp_off[0] == 0);
  for (int i = 0; i < n; i++) {
    LLD_ARG(c, p->off[i + 1] >= p->off[i]);
    LLD_ARG(c, p->hyp_off[i + 1] >= p->hyp_off[i]);
    LLD_ARG(c, p->fix_scale[i] == 0 || p->fix_scale[i] == 1);
    LLD_ARG(c, p->max_its[i] >= 1);
    LLD_ARG(c, p->its_done[i] >= 0 && p->best_inliers[i] >= 0);
    const int N = p->off[i + 1] - p->off[i];
    const int budget = N < p->min_inliers ? 0 : std::min(p->n_iterations, std::max(0, p->max_its[i] - p->its_done[i]));
    if (p->hyp_off[i + 1] - p->hyp_off[i] != budget) {
      snprintf(c->err, sizeof(c->err), "lld_sim3_ransac: problem %d has %d minimal sets, its budget is %d", i,
               p->hyp_off[i + 1] - p->hyp_off[i], budget);
      return LLD_ERR_ARG;
    }
    for (int h = p->hyp_off[i]; h < p->hyp_off[i + 1]; h++) {
      const int32_t* id = p->hyp_idx + 3 * (size_t)h;
      if (id[0] < 0 || id[0] >= N || id[1] < 0 || id[1] >= N || id[2] < 0 || id[2] >= N || id[0] == id[1] || id[0] == id[2] ||
          id[1] == id[2]) {
        snprintf(c->err, sizeof(c->err), "lld_sim3_ransac: minimal set %d of problem %d is (%d, %d, %d): indices must be distinct and in [0, %d)",
                 h - p->hyp_off[i], i, id[0], id[1], id[2], N);
        return LLD_ERR_ARG;
      }
    }
  }
  const int m = p->off[n], h = p->hyp_off[n];
  if (int r = lld_call_begin(c, true)) return r;
  RansacView v{};
  LLD_UP(c, v.cam, p->cam, 8 * (size_t)n);
  LLD_UP(c, v.fix_scale, p->fix_scale, n);
  LLD_UP(c, v.off, p->off, n + 1);
  LLD_UP(c, v.x1c, p->x1c, 3 * (size_t)m);
  LLD_UP(c, v.x2c, p->x2c, 3 * (size_t)m);
  LLD_UP(c, v.sig1, p->sigma2_1, m);
  LLD_UP(c, v.sig2, p->sigma2_2, m);
  v.min_inliers = p->min_inliers;
  LLD_UP(c, v.max_its, p->max_its, n);
  LLD_UP(c, v.its_in, p->its_done, n);
  LLD_UP(c, v.best_in, p->best_inliers, n);
  v.n_iterations = p->n_iterations;
  LLD_UP(c, v.hyp_off, p->hyp_off, n + 1);
  LLD_UP(c, v.hyp_idx, p->hyp_idx, 3 * (size_t)h);
  LLD_DEV(c, v.found, n);
  LLD_DEV(c, v.no_more, n);
  LLD_DEV(c, v.n_inliers, n);
  LLD_DEV(c, v.T12, 13 * (size_t)n);
  LLD_DEV(c, v.inlier, m);
  LLD_DEV(c, v.its_out, n);
  LLD_DEV(c, v.best_out, n);
  if (out->hyp_inliers) LLD_DEV(c, v.hyp_inliers, h);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_LAUNCH(c, k_sim3_ransac, n, RTPB, 0, v);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, out->found, v.found, (size_t)n);
  LLD_DOWN(c, out->no_more, v.no_more, (size_t)n);
  LLD_DOWN(c, out->n_inliers, v.n_inliers, (size_t)n);
  LLD_DOWN(c, out->T12, v.T12, 13 * (size_t)n);
  LLD_DOWN(c, out->inlier, v.inlier, (size_t)m);
  LLD_DOWN(c, out->its_done, v.its_out, (size_t)n);
  LLD_DOWN(c, out->best_inliers, v.best_out, (size_t)n);
  LLD_DOWN(c, out->hyp_inliers, v.hyp_inliers, (size_t)h);
  return lld_call_end(c);
}
