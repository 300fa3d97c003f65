// lineassoc.cu — temporal line association, Tracking::AddLinesFrom (src/Tracking.cc:996-1124), batched over frames.
//
// One warp per frame replays the reference's sequential loop over the offered map lines; the candidates of a map line
// (sub_inds) sit one per lane: claimed / no-stereo-match / behind-the-camera rejections, the reprojection gate
// vgl::LineReprojErrorL1 (src/vgl.cc:548-559) in the left and the right image against the octave-scaled threshold, the
// float-descriptor L2 distance in double.  The smallest distance wins, the first candidate on ties (strict < in list
// order: warp argmin on the key (distance, position in the list)); an accepted match claims the current line for the
// rest of the loop (mCurrentFrame.mvpMapLines[mi] = pML).  FP64 arithmetic in the reference's operation order (this file
// is compiled with --fmad=false), so the gates and the argmin agree with the CPU path bit for bit.
#include <algorithm>

#include "lld_ctx.h"

namespace {

struct AssocView {
  lld_line_assoc_problem p;   // device pointers
  int* cur_assoc;
  int* n_added;
  int max_cur;
};

__device__ __forceinline__ void map_point_c2w(const double* T, const double* X, double* o) {
  const double d[3] = {X[0] - T[3], X[1] - T[7], X[2] - T[11]};
#pragma unroll
  for (int i = 0; i < 3; i++) o[i] = T[0 * 4 + i] * d[0] + T[1 * 4 + i] * d[1] + T[2 * 4 + i] * d[2];
}
__device__ __forceinline__ double line_reproj_err_l1(const float* seg, const double* T, const double* X0, const double* dir, const double* K) {
  double Xa[3], Xb[3];
  const double P2[3] = {X0[0] + dir[0], X0[1] + dir[1], X0[2] + dir[2]};
  map_point_c2w(T, X0, Xa);
  map_point_c2w(T, P2, Xb);
  double c1[3], c2[3];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    c1[i] = K[3 * i] * Xa[0] + K[3 * i + 1] * Xa[1] + K[3 * i + 2] * Xa[2];
    c2[i] = K[3 * i] * Xb[0] + K[3 * i + 1] * Xb[1] + K[3 * i + 2] * Xb[2];
  }
  double l[3] = {c1[1] * c2[2] - c1[2] * c2[1], c1[2] * c2[0] - c1[0] * c2[2], c1[0] * c2[1] - c1[1] * c2[0]};
  const double n = sqrt(l[0] * l[0] + l[1] * l[1]);
  l[0] /= n; l[1] /= n; l[2] /= n;
  const double e1 = fabs((double)seg[0] * l[0] + (double)seg[1] * l[1] + l[2]);
  const double e2 = fabs((double)seg[2] * l[0] + (double)seg[3] * l[1] + l[2]);
  return e1 + e2;
}

__global__ void __launch_bounds__(32) k_line_associate(AssocView v) {
  extern __shared__ unsigned s_taken[];   // bit per current line of the frame
  const lld_line_assoc_problem& p = v.p;
  const int f = blockIdx.x, lane = threadIdx.x;
  const int m0 = p.ml_off[f], m1 = p.ml_off[f + 1];
  const int c0 = p.cur_off[f], nc = p.cur_off[f + 1] - c0;
  const int r0 = p.right_off[f];
  const int D = p.desc_dim;
  const double* Tc = p.T_curr + 16 * (size_t)f;
  const double* Tr = p.T_right + 16 * (size_t)f;
  for (int w = lane; w < (nc + 31) / 32; w += 32) {
    unsigned bits = 0;
    for (int b = 0; b < 32; b++) {
      const int i = 32 * w + b;
      if (i < nc && p.cur_taken[c0 + i]) bits |= 1u << b;
    }
    s_taken[w] = bits;
  }
  for (int i = lane; i < nc; i += 32) v.cur_assoc[c0 + i] = -1;
  __syncwarp();
  int added = 0;
  for (int i = m0; i < m1; i++) {
    if (!p.ml_valid[i]) continue;    // warp-uniform
    const double* X0 = p.ml_x0_dir + 6 * (size_t)i;
    const double* dir = X0 + 3;
    double X1c[3], X2c[3];
    map_point_c2w(Tc, p.ml_x1x2 + 6 * (size_t)i, X1c);
    map_point_c2w(Tc, p.ml_x1x2 + 6 * (size_t)i + 3, X2c);
    const bool front = !(X1c[2] < 0 || X2c[2] < 0);
    const int q0 = p.cand_off[i], q1 = p.cand_off[i + 1];
    double md = 1e10;
    int best_pos = 0x7fffffff, match_id = -1;
    for (int qb = q0; qb < q1; qb += 32) {
      const int q = qb + lane;
      double cd = 1e300;
      int si = -1;
      if (q < q1 && front) {
        si = p.cand_idx[q];
        bool ok = !((s_taken[si >> 5] >> (si & 31)) & 1u);
        const int ri = p.cur_line_match[c0 + si];
        if (ri < 0 && !p.monocular) ok = false;
        if (ok) {
          double thr = p.thr_reproj_base;
          for (int l = 0; l < p.cur_octave[c0 + si]; l++) thr *= 1.44;
          const double se = line_reproj_err_l1(p.cur_left + 4 * (size_t)(c0 + si), Tc, X0, dir, p.K);
          double se2 = 0;
          if (!p.monocular) se2 = line_reproj_err_l1(p.cur_right + 4 * (size_t)(r0 + ri), Tr, X0, dir, p.K);
          if (se > thr || se2 > thr) ok = false;
        }
        if (ok) {
          const float* da = p.ml_desc + (size_t)D * i;
          const float* db = p.cur_desc + (size_t)D * (c0 + si);
          double ss = 0;
          for (int k = 0; k < D; k++) {
            const double df = (double)da[k] - (double)db[k];
            ss += df * df;
          }
          cd = sqrt(ss);
          // the reference accepts only cd < md, md starting at 1e10; dropping the rest here also keeps a NaN distance (from a
          // NaN in a descriptor) out of the argmin, whose comparisons would otherwise leave the lanes with different winners
          if (!(cd < 1e10)) { cd = 1e300; si = -1; }
        } else {
          si = -1;
        }
      }
      // warp argmin on (distance, list position): the reference's strict < keeps the first of equal distances
      int pos = si >= 0 ? q : 0x7fffffff;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, cd, o);
        const int op = __shfl_xor_sync(0xffffffffu, pos, o);
        const int os = __shfl_xor_sync(0xffffffffu, si, o);
        if (os >= 0 && (si < 0 || od < cd || (od == cd && op < pos))) { cd = od; pos = op; si = os; }
      }
      if (si >= 0 && cd < md) { md = cd; match_id = si; best_pos = pos; }
    }
    (void)best_pos;
    if (md > p.md_thr) continue;
    if (match_id >= 0) {   // not taken: taken candidates were skipped above
      if (lane == 0) {
        s_taken[match_id >> 5] |= 1u << (match_id & 31);
        v.cur_assoc[c0 + match_id] = i - m0;
      }
      added++;
      __syncwarp();
    }
  }
  if (lane == 0 && v.n_added) v.n_added[f] = added;
}

}  // namespace

extern "C" int lld_line_associate(void* ctx, const lld_line_assoc_problem* p, lld_line_assoc_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  c->launches = 0;   // a rejected call reports no launches
  LLD_ARG(c, p->n_frames >= 1 && p->desc_dim >= 1);
  const int F = p->n_frames, n_ml = p->ml_off[F], n_cur = p->cur_off[F], n_r = p->right_off[F], n_cand = p->cand_off[n_ml], D = p->desc_dim;
  // candidates index the frame's current lines (taken bitset, cur_line_match); a stereo match indexes its right lines
  for (int f = 0; f < F; f++) {
    const int nc = p->cur_off[f + 1] - p->cur_off[f], nr = p->right_off[f + 1] - p->right_off[f];
    for (int q = p->cand_off[p->ml_off[f]]; q < p->cand_off[p->ml_off[f + 1]]; q++) LLD_ARG(c, p->cand_idx[q] >= 0 && p->cand_idx[q] < nc);
    if (!p->monocular)
      for (int i = p->cur_off[f]; i < p->cur_off[f + 1]; i++) LLD_ARG(c, p->cur_line_match[i] < nr);
  }
  int max_cur = 1;
  for (int f = 0; f < F; f++) max_cur = std::max(max_cur, p->cur_off[f + 1] - p->cur_off[f]);
  const size_t smem = 4 * (size_t)((max_cur + 31) / 32);
  LLD_ARG(c, smem <= 48 * 1024);
  if (int r = lld_call_begin(c, true)) return r;
  AssocView v{};
  v.p = *p;
  LLD_UP(c, v.p.ml_off, p->ml_off, F + 1);
  LLD_UP(c, v.p.ml_valid, p->ml_valid, n_ml);
  LLD_UP(c, v.p.ml_x0_dir, p->ml_x0_dir, 6 * (size_t)n_ml);
  LLD_UP(c, v.p.ml_x1x2, p->ml_x1x2, 6 * (size_t)n_ml);
  LLD_UP(c, v.p.ml_desc, p->ml_desc, (size_t)D * n_ml);
  LLD_UP(c, v.p.cand_off, p->cand_off, n_ml + 1);
  LLD_UP(c, v.p.cand_idx, p->cand_idx, n_cand);
  LLD_UP(c, v.p.cur_off, p->cur_off, F + 1);
  LLD_UP(c, v.p.cur_left, p->cur_left, 4 * (size_t)n_cur);
  LLD_UP(c, v.p.cur_octave, p->cur_octave, n_cur);
  LLD_UP(c, v.p.cur_line_match, p->cur_line_match, n_cur);
  LLD_UP(c, v.p.cur_taken, p->cur_taken, n_cur);
  LLD_UP(c, v.p.cur_desc, p->cur_desc, (size_t)D * n_cur);
  LLD_UP(c, v.p.right_off, p->right_off, F + 1);
  LLD_UP(c, v.p.cur_right, p->cur_right, 4 * (size_t)n_r);
  LLD_UP(c, v.p.T_curr, p->T_curr, 16 * (size_t)F);
  LLD_UP(c, v.p.T_right, p->T_right, 16 * (size_t)F);
  LLD_DEV(c, v.cur_assoc, n_cur);
  LLD_DEV(c, v.n_added, F);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_LAUNCH(c, k_line_associate, F, 32, smem, v);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, out->cur_assoc, v.cur_assoc, n_cur);
  LLD_DOWN(c, out->n_added, v.n_added, F);
  return lld_call_end(c);
}
