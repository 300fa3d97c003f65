// pnpransac.cu — batched relocalisation EPnP RANSAC (PnPsolver::iterate / Refine / CheckInliers / compute_pose, ORB-SLAM2
// src/PnPsolver.cc).
//
// One CTA per relocalisation candidate, one warp per minimal set.  The CTA evaluates the candidate's sets in waves of NW: each
// warp runs EPnP on its four correspondences (lanes split the M^T M entries and the Jacobi rotation rows, lane 0 the small
// serial pieces; lld_math.cuh pnp_epnp) and counts the inliers over the candidate's correspondences with __ballot_sync /
// __popc.  After a wave the CTA applies iterate()'s sequential rule to the wave's sets in order: the count test (>=
// min_inliers), the new best (> best_inliers: its mask and pose are written to the carried state) and Refine, which runs EPnP
// over the best mask's correspondences with the whole CTA (one thread per M^T M entry, each summing serially in
// correspondence order) and stops the CTA when the refined count exceeds min_inliers.  Correspondence data is read from global
// memory; the per-warp EPnP state lives in shared memory (PnpWork).
// Compiled with --fmad=false: the EPnP arithmetic and CheckInliers' float / double mix mirror the reference's operation order.
#include <algorithm>
#include <climits>
#include <cmath>

#include "lld_ctx.h"
#include "lld_math.cuh"

using namespace lld;

namespace {

constexpr int RTPB = 256;
constexpr int NW = RTPB / 32;

struct PnpView {
  const float* cam;
  const int* min_in;
  const int* max_its;
  const int* its_in;
  const int* best_in;
  const int* off;
  const float* p2d;
  const float* p3dw;
  const float* max_err;
  uint8_t* bmask;   // carried mvbBestInliers, updated in place
  float* bTcw;      // carried mBestTcw, updated in place
  int n_iterations;
  const int* hyp_off;
  const int* hyp_idx;
  uint8_t* found;
  uint8_t* no_more;
  int* n_inliers;
  float* Tcw;
  uint8_t* inlier;
  int* its_out;
  int* best_out;
  int* hyp_inliers;
  int* ridx;        // [m] scratch: the best inliers' indices, the correspondences Refine runs EPnP on
};

// CheckInliers over the candidate's n correspondences, the CTA striding over them; the count is returned on every thread
__device__ int cta_count(const double* R, const double* t, const float* X3, const float* UV, const float* ME, int n,
                         const PnpCam& cam, int* s_red) {
  int cnt = 0;
  for (int i = threadIdx.x; i < n; i += RTPB) cnt += pnp_inlier(R, t, X3 + 3 * (size_t)i, UV + 2 * (size_t)i, ME[i], cam);
  if (threadIdx.x == 0) *s_red = 0;
  __syncthreads();
  if (cnt) atomicAdd(s_red, cnt);
  __syncthreads();
  const int r = *s_red;
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(RTPB) k_pnp_ransac(PnpView v) {
  __shared__ PnpWork s_w[NW];
  __shared__ double s_pose[NW][12];
  __shared__ int s_cnt[NW];
  __shared__ int s_red, s_nidx;
  const int pb = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int e0 = v.off[pb], n = v.off[pb + 1] - e0;
  const int h0 = v.hyp_off[pb], B = v.hyp_off[pb + 1] - h0;
  const int min_in = v.min_in[pb];
  const PnpCam cam{v.cam[4 * (size_t)pb], v.cam[4 * (size_t)pb + 1], v.cam[4 * (size_t)pb + 2], v.cam[4 * (size_t)pb + 3]};
  const float* X3 = v.p3dw + 3 * (size_t)e0;
  const float* UV = v.p2d + 2 * (size_t)e0;
  const float* ME = v.max_err + e0;
  uint8_t* BM = v.bmask + e0;
  float* BT = v.bTcw + 12 * (size_t)pb;
  if (v.hyp_inliers)
    for (int k = tid; k < B; k += RTPB) v.hyp_inliers[h0 + k] = -1;
  int its = v.its_in[pb], best = v.best_in[pb];   // uniform over the CTA
  bool found = false;
  int n_found = 0;
  for (int base = 0; base < B && !found; base += NW) {
    const int k = base + w;
    if (k < B) {
      const PnpWarp par{lane};
      pnp_epnp(par, s_w[w], X3, UV, v.hyp_idx + 4 * (size_t)(h0 + k), 4, cam);
      const int b = pnp_pick(s_w[w]);
      const double* R = s_w[w].R[b];
      const double* t = s_w[w].t[b];
      int cnt = 0;
      for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        const bool in = i < n && pnp_inlier(R, t, X3 + 3 * (size_t)i, UV + 2 * (size_t)i, ME[i], cam);
        cnt += __popc(__ballot_sync(0xffffffffu, in));
      }
      if (lane < 9) s_pose[w][lane] = R[lane];
      else if (lane < 12) s_pose[w][lane] = t[lane - 9];
      if (lane == 0) s_cnt[w] = cnt;
    }
    __syncthreads();
    const int nw = min(NW, B - base);
    for (int j = 0; j < nw; j++) {   // iterate()'s loop body, in set order
      const int c = s_cnt[j];
      its++;
      if (tid == 0 && v.hyp_inliers) v.hyp_inliers[h0 + base + j] = c;
      if (c < min_in) continue;
      if (c > best) {
        best = c;
        for (int i = tid; i < n; i += RTPB)
          BM[i] = pnp_inlier(s_pose[j], s_pose[j] + 9, X3 + 3 * (size_t)i, UV + 2 * (size_t)i, ME[i], cam);
        if (tid < 12) BT[tid] = (float)s_pose[j][tid];
      }
      __syncthreads();
      // Refine() on the best mask, the whole CTA (s_w[0]: warp 0's set of this wave is already in s_pose)
      if (tid == 0) {
        int r = 0;
        for (int i = 0; i < n; i++)
          if (BM[i]) v.ridx[e0 + r++] = i;
        s_nidx = r;
      }
      __syncthreads();
      const PnpCta cta;
      pnp_epnp(cta, s_w[0], X3, UV, v.ridx + e0, s_nidx, cam);
      const int rb = pnp_pick(s_w[0]);
      const double* R = s_w[0].R[rb];
      const double* t = s_w[0].t[rb];
      const int rc = cta_count(R, t, X3, UV, ME, n, cam, &s_red);
      if (rc > min_in) {
        found = true;
        n_found = rc;
        for (int i = tid; i < n; i += RTPB)
          v.inlier[e0 + i] = pnp_inlier(R, t, X3 + 3 * (size_t)i, UV + 2 * (size_t)i, ME[i], cam);
        if (tid < 9) v.Tcw[12 * (size_t)pb + tid] = (float)R[tid];
        else if (tid < 12) v.Tcw[12 * (size_t)pb + tid] = (float)t[tid - 9];
        break;
      }
    }
    __syncthreads();   // s_w[0] and s_pose are rewritten by the next wave
  }
  bool no_more = false;
  if (n < min_in) {
    no_more = true;
  } else if (!found && its >= v.max_its[pb]) {
    no_more = true;
    if (best >= min_in) {   // the budget is spent: the best pose so far
      found = true;
      n_found = best;
      for (int i = tid; i < n; i += RTPB) v.inlier[e0 + i] = BM[i];
      if (tid < 12) v.Tcw[12 * (size_t)pb + tid] = BT[tid];
    }
  }
  if (!found) {
    for (int i = tid; i < n; i += RTPB) v.inlier[e0 + i] = 0;
    if (tid < 12) v.Tcw[12 * (size_t)pb + tid] = 0.f;
  }
  if (tid == 0) {
    v.found[pb] = found;
    v.no_more[pb] = no_more;
    v.n_inliers[pb] = found ? n_found : 0;
    v.its_out[pb] = its;
    v.best_out[pb] = best;
  }
}

}  // namespace

extern "C" int lld_pnp_ransac_params(int32_t n_corr, double probability, int32_t min_inliers, int32_t max_iterations,
                                     int32_t min_set, float epsilon, int32_t out[2]) {
  if (n_corr < 0 || !out) return LLD_ERR_ARG;
  int nMinInliers = (int)((float)n_corr * epsilon);
  if (nMinInliers < min_inliers) nMinInliers = min_inliers;
  if (nMinInliers < min_set) nMinInliers = min_set;
  if (epsilon < (float)nMinInliers / (float)n_corr) epsilon = (float)nMinInliers / (float)n_corr;
  int nIterations;
  if (nMinInliers == n_corr) {
    nIterations = 1;
  } else {
    const double it = std::ceil(std::log(1 - probability) / std::log(1 - std::pow((double)epsilon, 3.0)));
    nIterations = it >= (double)INT_MAX ? INT_MAX : (it > (double)INT_MIN ? (int)it : INT_MIN);   // NaN: INT_MIN, as x86 converts
  }
  out[0] = nMinInliers;
  out[1] = std::max(1, std::min(nIterations, max_iterations));
  return LLD_OK;
}

extern "C" int lld_pnp_ransac(void* ctx, const lld_pnp_ransac_problem* p, lld_pnp_ransac_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  const int n = p->n_problems;
  LLD_ARG(c, n >= 0);
  LLD_ARG(c, p->n_iterations >= 0);
  if (n == 0) return LLD_OK;
  LLD_ARG(c, p->off && p->off[0] == 0);
  LLD_ARG(c, p->hyp_off && p->hyp_off[0] == 0);
  LLD_ARG(c, p->best_Tcw && out->best_Tcw && out->best_mask);
  for (int i = 0; i < n; i++) {
    LLD_ARG(c, p->off[i + 1] >= p->off[i]);
    LLD_ARG(c, p->hyp_off[i + 1] >= p->hyp_off[i]);
    LLD_ARG(c, p->min_inliers[i] >= 4);
    LLD_ARG(c, p->max_its[i] >= 1);
    LLD_ARG(c, p->its_done[i] >= 0 && p->best_inliers[i] >= 0);
    const int N = p->off[i + 1] - p->off[i];
    const int budget = N < p->min_inliers[i] ? 0 : std::max(p->n_iterations, p->max_its[i] - p->its_done[i]);
    if (p->hyp_off[i + 1] - p->hyp_off[i] != budget) {
      snprintf(c->err, sizeof(c->err), "lld_pnp_ransac: problem %d has %d minimal sets, its budget is %d", i,
               p->hyp_off[i + 1] - p->hyp_off[i], budget);
      return LLD_ERR_ARG;
    }
    for (int h = p->hyp_off[i]; h < p->hyp_off[i + 1]; h++) {
      const int32_t* id = p->hyp_idx + 4 * (size_t)h;
      bool ok = true;
      for (int a = 0; a < 4; a++) {
        ok = ok && id[a] >= 0 && id[a] < N;
        for (int b = 0; b < a; b++) ok = ok && id[a] != id[b];
      }
      if (!ok) {
        snprintf(c->err, sizeof(c->err),
                 "lld_pnp_ransac: minimal set %d of problem %d is (%d, %d, %d, %d): indices must be distinct and in [0, %d)",
                 h - p->hyp_off[i], i, id[0], id[1], id[2], id[3], N);
        return LLD_ERR_ARG;
      }
    }
  }
  const int m = p->off[n], h = p->hyp_off[n];
  LLD_ARG(c, m == 0 || p->best_mask);
  if (int r = lld_call_begin(c, true)) return r;
  PnpView v{};
  LLD_UP(c, v.cam, p->cam, 4 * (size_t)n);
  LLD_UP(c, v.min_in, p->min_inliers, n);
  LLD_UP(c, v.max_its, p->max_its, n);
  LLD_UP(c, v.its_in, p->its_done, n);
  LLD_UP(c, v.best_in, p->best_inliers, n);
  LLD_UP(c, v.off, p->off, n + 1);
  LLD_UP(c, v.p2d, p->p2d, 2 * (size_t)m);
  LLD_UP(c, v.p3dw, p->p3dw, 3 * (size_t)m);
  LLD_UP(c, v.max_err, p->max_err, m);
  LLD_UP(c, v.bmask, p->best_mask, m);
  LLD_UP(c, v.bTcw, p->best_Tcw, 12 * (size_t)n);
  v.n_iterations = p->n_iterations;
  LLD_UP(c, v.hyp_off, p->hyp_off, n + 1);
  LLD_UP(c, v.hyp_idx, p->hyp_idx, 4 * (size_t)h);
  LLD_DEV(c, v.found, n);
  LLD_DEV(c, v.no_more, n);
  LLD_DEV(c, v.n_inliers, n);
  LLD_DEV(c, v.Tcw, 12 * (size_t)n);
  LLD_DEV(c, v.inlier, m);
  LLD_DEV(c, v.its_out, n);
  LLD_DEV(c, v.best_out, n);
  LLD_DEV(c, v.ridx, m);
  if (out->hyp_inliers) LLD_DEV(c, v.hyp_inliers, h);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_LAUNCH(c, k_pnp_ransac, n, RTPB, 0, v);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, out->found, v.found, (size_t)n);
  LLD_DOWN(c, out->no_more, v.no_more, (size_t)n);
  LLD_DOWN(c, out->n_inliers, v.n_inliers, (size_t)n);
  LLD_DOWN(c, out->Tcw, v.Tcw, 12 * (size_t)n);
  LLD_DOWN(c, out->inlier, v.inlier, (size_t)m);
  LLD_DOWN(c, out->its_done, v.its_out, (size_t)n);
  LLD_DOWN(c, out->best_inliers, v.best_out, (size_t)n);
  LLD_DOWN(c, out->best_mask, v.bmask, (size_t)m);
  LLD_DOWN(c, out->best_Tcw, v.bTcw, 12 * (size_t)n);
  LLD_DOWN(c, out->hyp_inliers, v.hyp_inliers, (size_t)h);
  return lld_call_end(c);
}
