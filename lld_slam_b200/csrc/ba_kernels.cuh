// ba_kernels.cuh — sm_100a kernels of the batched point+line bundle adjustment.
//
// One LM "step" of every window in the batch is the fixed kernel sequence
//   [k_lin_points, k_lin_lines, k_lin_poses, k_reduce_pose, k_reduce_lin, k_begin]   (windows in PH_LIN only)
//   k_schur_points, k_schur_lines, k_schur_rows, k_reduce_rows, k_solve,
//   k_backsub_points, k_backsub_lines, k_reduce_trial, k_decide
// Each kernel looks at the per-window phase and returns early for windows that do not need it, so the
// whole batch advances in lock step while every window follows its own Levenberg-Marquardt trajectory
// (Thirdparty/g2o/g2o/core/optimization_algorithm_levenberg.cpp:61-164).
// Reductions are fixed-order (no floating-point atomics): results are run-to-run reproducible.
#pragma once
#include <cfloat>
#include <cstdio>

#include "ba.cuh"
#include "lld_math.cuh"

namespace lld {

#define LM_TPB 128

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
  return v;
}
// fixed-order block sum (blockDim.x multiple of 32, <= 1024); result valid in thread 0
__device__ __forceinline__ double block_sum(double v, double* sm /*>=32*/) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  double r = 0;
  if (wid == 0) {
    r = (lane < (int)(blockDim.x >> 5)) ? sm[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;
}
__device__ __forceinline__ double block_max(double v, double* sm) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  double r = 0;
  if (wid == 0) {
    r = (lane < (int)(blockDim.x >> 5)) ? sm[lane] : 0.0;
    r = warp_max(r);
  }
  return r;
}

// ------------------------------------------------------------------------------------------------
// state initialisation
// ------------------------------------------------------------------------------------------------
__global__ void k_init_state(BaView v, const double* __restrict__ kf_Tcw, const double* __restrict__ pt_xyz,
                             const double* __restrict__ ln_x0_dir, const float* __restrict__ lc_right) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < v.n_kf) {
    double qt[7], Rt[12];
    pose_from_Rt(kf_Tcw + 12 * (size_t)i, qt);
    pose_to_Rt(qt, Rt);
    for (int b = 0; b < 2; b++) {
      for (int k = 0; k < 7; k++) v.pose_qt[b][7 * (size_t)i + k] = qt[k];
      for (int k = 0; k < 12; k++) v.pose_Rt[b][12 * (size_t)i + k] = Rt[k];
    }
  }
  if (i < v.n_pt)
    for (int k = 0; k < 3; k++) {
      const double x = pt_xyz[3 * (size_t)i + k];
      v.pt_xyz[0][3 * (size_t)i + k] = x;
      v.pt_xyz[1][3 * (size_t)i + k] = x;
    }
  if (i < v.n_ln) {
    double st[5];
    line_from_x0_dir(ln_x0_dir + 6 * (size_t)i, ln_x0_dir + 6 * (size_t)i + 3, st);
    for (int k = 0; k < 5; k++) {
      v.ln_st[0][5 * (size_t)i + k] = st[k];
      v.ln_st[1][5 * (size_t)i + k] = st[k];
    }
    v.ln_removed[i] = 0;
  }
  if (i < v.n_pe) {
    v.pe_level[i] = 0;
    v.pe_chi2[i] = 0.0;
  }
  if (i < v.n_lc) {
    v.lc_level[2 * i] = 0;
    v.lc_level[2 * i + 1] = (lc_right[4 * (size_t)i] < 0.f) ? 2 : 0;  // src/LineOptimizer.cc:65-68
    v.lc_chi2[2 * i] = 0.0;
    v.lc_chi2[2 * i + 1] = 0.0;
  }
  if (i < v.n_free_total)
    for (int k = 0; k < 6; k++) v.g_x[6 * (size_t)i + k] = 0.0;
  if (i < v.n_pt)
    for (int k = 0; k < 3; k++) v.pt_xl[3 * (size_t)i + k] = 0.0;
  if (i < v.n_ln)
    for (int k = 0; k < 4; k++) v.ln_xl[4 * (size_t)i + k] = 0.0;
}

// ------------------------------------------------------------------------------------------------
// index arrays derived on the device at upload time (nothing to index on the host, nothing to move over PCIe)
// ------------------------------------------------------------------------------------------------
// out[e] = the segment i of the CSR offsets off[0..n] that contains e (largest i with off[i] <= e: skips empty segments)
__global__ void k_expand_owner(int n_out, int n, const int* __restrict__ off, int* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_out) return;
  int lo = 0, hi = n;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= e) lo = mid;
    else hi = mid;
  }
  out[e] = lo;
}

// Sparse-mode position tables: per list entry i of free block g (a point edge / line cell observed by g) and per neighbour block
// nb_g[nb_off[g] + j] >= g, the list position of the same landmark's edge on that neighbour, or -1 (the table is pre-set to -1).
// One thread per list entry: its block row by bisection in the list offsets, then the landmark's other edges.
__global__ void k_build_tab(int n_list, int nG, const int* __restrict__ l_off, const int* __restrict__ l_ref, const int* __restrict__ off,
                            const int* __restrict__ e_lm, const int* __restrict__ ekf, const int* __restrict__ kf_g,
                            const int* __restrict__ e_pos, const int* __restrict__ nb_off, const int* __restrict__ nb_g,
                            const long long* __restrict__ t_off, int* __restrict__ tab) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_list) return;
  int lo = 0, hi = nG;   // largest g with l_off[g] <= i
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (l_off[mid] <= i) lo = mid;
    else hi = mid;
  }
  const int g = lo, nnb = nb_off[g + 1] - nb_off[g];
  const int* nbl = nb_g + nb_off[g];
  int* row = tab + t_off[g] + (long long)(i - l_off[g]) * nnb;
  const int lm = e_lm[l_ref[i]];
  for (int e2 = off[lm]; e2 < off[lm + 1]; e2++) {
    const int b = kf_g[ekf[e2]];
    if (b < g) continue;
    int a = 0, z = nnb;   // lower_bound of b in the neighbour list
    while (a < z) {
      const int mid = (a + z) >> 1;
      if (nbl[mid] < b) a = mid + 1;
      else z = mid;
    }
    row[a] = e_pos[e2];
  }
}

// sparse mode, a landmark seen more than once by one free keyframe: the position tables name ONE co-edge per (landmark,
// keyframe) (the last one, above), so k_schur_rows would pair W_e with only that edge.  H holds one landmark-pose block per
// (landmark, keyframe) that all those edges add into (block_solver.hpp), so the records of the other edges are added into
// the named one and zeroed: the Schur rows and the back-substitution then see the summed block.  Runs after the
// linearisation has rewritten every record; a group is summed by one thread in list order.
__global__ void k_fold_dup(BaView v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n_fold) return;
  const bool pt = i < v.n_fold_pt;
  const int rec = pt ? 27 : 38, nw = pt ? 18 : 24;
  double* base = pt ? v.P_rec : v.L_rec;
  double* d = base + (size_t)rec * v.fold_dst[i];
  for (int k = v.fold_off[i]; k < v.fold_off[i + 1]; k++) {
    double* s = base + (size_t)rec * v.fold_src[k];
    for (int q = 0; q < nw; q++) {
      d[q] += s[q];
      s[q] = 0.0;
    }
  }
}

// dense mode: the W blocks of a landmark are contiguous (first slot w0[sorted position]) and sorted by keyframe, so the
// slot of an edge is w0 + the rank of its keyframe's block among the set bits of the landmark's mask; -1 = fixed keyframe
__global__ void k_dense_wpos(int n_e, const int* __restrict__ e_lm, const int* __restrict__ e_kf, const int* __restrict__ kf_g,
                             const int* __restrict__ lm_win, const int* __restrict__ w_g0, const int* __restrict__ spos,
                             const uint32_t* __restrict__ mask, const int* __restrict__ w0, int* __restrict__ wpos) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_e) return;
  const int g = kf_g[e_kf[e]];
  if (g < 0) {
    wpos[e] = -1;
    return;
  }
  const int lm = e_lm[e], oi = spos[lm];
  const int bit = g - w_g0[lm_win[lm]];
  wpos[e] = w0[oi] + __popc(mask[oi] & ((1u << bit) - 1u));
}

__global__ void k_round_init(BaView v, int maxit, int round) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= v.n_win) return;
  v.w_phase[w] = (maxit > 0) ? PH_LIN : PH_DONE;
  v.w_iter[w] = 0;
  v.w_trials[w] = 0;
  v.w_maxit[w] = maxit;
  v.w_nbad[w] = 0;
  v.w_ok[w] = 1;
  v.w_lambda[w] = -1.0;
  v.w_ni[w] = 2.0;
  if (round == 0) {
    v.w_sel[w] = 0;
    v.w_nlog[w] = 0;
    v.iter_done[2 * w] = 0;
    v.iter_done[2 * w + 1] = 0;
  }
  if (w == 0) *v.n_active_win = (maxit > 0) ? v.n_win : 0;
}

// ------------------------------------------------------------------------------------------------
// linearisation: one thread per landmark
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void make_line_obs(const BaView& v, int kf, const float* seg, LineObs& o) {
  if (v.prm.ln_norm) {  // K^-1 (x,y,1)  src/Optimizer.cc:234-235
    const double* in = v.kf_intr + 5 * (size_t)kf;
    o.x1[0] = ((double)seg[0] - in[2]) / in[0]; o.x1[1] = ((double)seg[1] - in[3]) / in[1];
    o.x2[0] = ((double)seg[2] - in[2]) / in[0]; o.x2[1] = ((double)seg[3] - in[3]) / in[1];
  } else {
    o.x1[0] = seg[0]; o.x1[1] = seg[1];
    o.x2[0] = seg[2]; o.x2[1] = seg[3];
  }
  o.x1[2] = 1.0;
  o.x2[2] = 1.0;
}

// PT_G lanes per map point (4 for single windows, where one lane per point fills a third of the SMs; 1 for batches):
// lane g takes edges e0 + g, e0 + g + PT_G, ...; the sums are combined by a fixed xor butterfly inside the lane group.
// WITH_D (dense mode, every LM step but the first of a round, where lambda is known when the step starts): the kernel also
// forms (H_ll + lambda I)^-1 and D^-1 b_l (k_schur_points' work, block_solver.hpp:389) — for windows that retry a rejected
// step with a new lambda from the stored H_ll, without linearising again.
template <int PT_G, bool WITH_D = false>
__global__ void __launch_bounds__(LM_TPB) k_lin_points(BaView v) {
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int pl = gt / PT_G, gl = gt - pl * PT_G;
  const bool live = pl < v.n_pt;
  const int p = live ? pl : v.n_pt - 1;  // dead lanes shadow the last point (shuffles stay full-warp), no stores
  const int w = v.pt_win[p];
  const int phase = v.w_phase[w];
  const bool run = live && phase == PH_LIN;
  if (PT_G == 1 && !run && !(WITH_D && live && phase == PH_RETRY)) return;
  const int sel = v.w_sel[w];
  const double* Xp = v.pt_xyz[sel] + 3 * (size_t)p;
  const double X[3] = {Xp[0], Xp[1], Xp[2]};
  double H[6] = {0, 0, 0, 0, 0, 0}, bl[3] = {0, 0, 0};
  double chi = 0;
  int nact = 0;
  const int e0 = v.pt_obs_off[p], e1 = v.pt_obs_off[p + 1];
  const bool dense = v.dense_mode != 0;
  const int* epos = dense ? v.pe_wpos : v.pe_pos;
  // edge header (keyframe, W slot, level, observation, information) one edge ahead of the arithmetic
  int e = e0 + gl;
  int kf = 0, pos = -1, lvl = 1;
  float ou = 0.f, ov = 0.f, orr = 0.f, oinfo = 0.f;
  if (e < e1 && run) {
    kf = v.pe_kf[e]; pos = epos[e]; lvl = v.pe_level[e];
    ou = v.pe_uvr[3 * (size_t)e]; ov = v.pe_uvr[3 * (size_t)e + 1]; orr = v.pe_uvr[3 * (size_t)e + 2];
    oinfo = v.pe_info[e];
  }
  while (e < e1 && run) {
    const int en = e + PT_G;
    int kf_n = 0, pos_n = -1, lvl_n = 1;
    float ou_n = 0.f, ov_n = 0.f, or_n = 0.f, oinfo_n = 0.f;
    if (en < e1) {
      kf_n = v.pe_kf[en]; pos_n = epos[en]; lvl_n = v.pe_level[en];
      ou_n = v.pe_uvr[3 * (size_t)en]; ov_n = v.pe_uvr[3 * (size_t)en + 1]; or_n = v.pe_uvr[3 * (size_t)en + 2];
      oinfo_n = v.pe_info[en];
    }
    double* W = dense ? v.pe_Wl + 18 * (size_t)(pos < 0 ? 0 : pos) : v.P_rec + 27 * (size_t)(pos < 0 ? 0 : pos);
    double Wv[18];
#pragma unroll
    for (int k = 0; k < 18; k++) Wv[k] = 0.0;
    if (lvl == 0) {
      nact++;
      double Rt[12];
      {
        const double2* rp = reinterpret_cast<const double2*>(v.pose_Rt[sel] + 12 * (size_t)kf);
#pragma unroll
        for (int k = 0; k < 6; k++) {
          const double2 t2 = rp[k];
          Rt[2 * k] = t2.x; Rt[2 * k + 1] = t2.y;
        }
      }
      const double* intr = v.kf_intr + 5 * (size_t)kf;
      const float obs[3] = {ou, ov, orr};
      const bool stereo = !(orr < 0.f);
      double xc[3], err[3], Jl[9];
      map_Rt(Rt, X, xc);
      pt_residual<true>(xc, intr, obs, stereo, err);
      const double info = (double)oinfo;
      const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
      double wgt = 1.0, rho = c2;
      if (v.prm.robust_pt) rho = huber(c2, stereo ? v.prm.delta_pt_stereo : v.prm.delta_pt_mono, &wgt);
      chi += rho;
      const double wo = wgt * info;
      pt_jac_point(xc, Rt, intr, stereo, Jl);
      // Hll += Jl^T wo Jl ; bl -= Jl^T wo err
      double JW[9];
#pragma unroll
      for (int k = 0; k < 9; k++) JW[k] = wo * Jl[k];
      H[0] += JW[0] * Jl[0] + JW[3] * Jl[3] + JW[6] * Jl[6];
      H[1] += JW[0] * Jl[1] + JW[3] * Jl[4] + JW[6] * Jl[7];
      H[2] += JW[0] * Jl[2] + JW[3] * Jl[5] + JW[6] * Jl[8];
      H[3] += JW[1] * Jl[1] + JW[4] * Jl[4] + JW[7] * Jl[7];
      H[4] += JW[1] * Jl[2] + JW[4] * Jl[5] + JW[7] * Jl[8];
      H[5] += JW[2] * Jl[2] + JW[5] * Jl[5] + JW[8] * Jl[8];
#pragma unroll
      for (int c = 0; c < 3; c++) bl[c] -= JW[c] * err[0] + JW[3 + c] * err[1] + JW[6 + c] * err[2];
      if (pos >= 0) {
        double Jp[18];
        pt_jac_pose(xc, intr, stereo, Jp);
#pragma unroll
        for (int r = 0; r < 6; r++)
#pragma unroll
          for (int c = 0; c < 3; c++) Wv[r * 3 + c] = Jp[r] * JW[c] + Jp[6 + r] * JW[3 + c] + Jp[12 + r] * JW[6 + c];
      }
    }
    if (pos >= 0) {  // W of a gated-out edge is zero
      if (dense) {   // 144-byte blocks: 16-byte stores
        double2* wp = reinterpret_cast<double2*>(W);
#pragma unroll
        for (int k = 0; k < 9; k++) wp[k] = make_double2(Wv[2 * k], Wv[2 * k + 1]);
      } else {
#pragma unroll
        for (int k = 0; k < 18; k++) W[k] = Wv[k];
      }
    }
    e = en; kf = kf_n; pos = pos_n; lvl = lvl_n;
    ou = ou_n; ov = ov_n; orr = or_n; oinfo = oinfo_n;
  }
#pragma unroll
  for (int o = PT_G / 2; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < 6; k++) H[k] += __shfl_xor_sync(0xffffffffu, H[k], o);
#pragma unroll
    for (int k = 0; k < 3; k++) bl[k] += __shfl_xor_sync(0xffffffffu, bl[k], o);
    chi += __shfl_xor_sync(0xffffffffu, chi, o);
    nact += __shfl_xor_sync(0xffffffffu, nact, o);
  }
  if (gl != 0 || !live) return;
  double* Ho = v.pt_H + 9 * (size_t)p;
  if (run) {
#pragma unroll
    for (int k = 0; k < 6; k++) Ho[k] = H[k];
    Ho[6] = bl[0]; Ho[7] = bl[1]; Ho[8] = bl[2];
    v.lm_chi2lin[p] = chi;
    v.lm_maxdiag[p] = nact ? fmax(fabs(H[0]), fmax(fabs(H[3]), fabs(H[5]))) : 0.0;
    v.lm_active[p] = nact > 0;
  } else if (WITH_D && phase == PH_RETRY) {
#pragma unroll
    for (int k = 0; k < 6; k++) H[k] = Ho[k];
    bl[0] = Ho[6]; bl[1] = Ho[7]; bl[2] = Ho[8];
  } else {
    return;
  }
  if (WITH_D) {
    const double lam = v.w_lambda[w];
    double Di[9];
    {
      const double A[9] = {H[0] + lam, H[1], H[2], H[1], H[3] + lam, H[4], H[2], H[4], H[5] + lam};
      inv3_sym(A, Di);
    }
    double* Do = v.pts_D + 10 * (size_t)v.pt_spos[p];
    Do[0] = Di[0]; Do[1] = Di[1]; Do[2] = Di[2]; Do[3] = Di[4]; Do[4] = Di[5]; Do[5] = Di[8];
#pragma unroll
    for (int i = 0; i < 3; i++) Do[6 + i] = Di[3 * i] * bl[0] + Di[3 * i + 1] * bl[1] + Di[3 * i + 2] * bl[2];
  }
}

// index of (r,c), r<=c, in the packed upper triangle of a 4x4
__device__ __forceinline__ constexpr int u4(int r, int c) { return r * 4 - (r * (r - 1)) / 2 + (c - r); }

// Lines: LN_G lanes per map line, lane g linearises cells c0 + g, c0 + g + LN_G, ... (a cell = one keyframe's left + right
// edge, ~1100 FP64 flops each with divisions and a square root: one thread per line is a 10-evaluation latency chain);
// H_ll, b_l, chi2 and the active count are then summed over the group by a fixed xor-butterfly (deterministic).
// (LN_G = 8 below ~8k lines, where one lane per line leaves the SMs idle; 1 for large batches, where the extra lanes only cost)
template <int LN_G, bool WITH_D = false>
__global__ void __launch_bounds__(LM_TPB) k_lin_lines(BaView v) {
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int l = gt / LN_G, gl = gt - l * LN_G;
  const bool live = l < v.n_ln;
  const int lc = live ? l : v.n_ln - 1;      // dead lanes shadow the last line (no stores) so that shuffles stay full-warp
  const int w = v.ln_win[lc];
  const int phase = v.w_phase[w];
  const bool run = live && phase == PH_LIN;
  const int sel = v.w_sel[w];
  const double* stp = v.ln_st[sel] + 5 * (size_t)lc;
  const double st[5] = {stp[0], stp[1], stp[2], stp[3], stp[4]};
  double r1[3], r2[3], X1[3], X2[3];
  line_axes(st, r1, r2);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    X1[i] = st[4] * r2[i];
    X2[i] = X1[i] + r1[i];
  }
  double H[10], bl[4] = {0, 0, 0, 0};
#pragma unroll
  for (int k = 0; k < 10; k++) H[k] = 0;
  double chi = 0;
  int nact = 0;
  const bool removed = v.ln_removed[lc] != 0;
  const int c0 = v.ln_obs_off[lc], c1 = v.ln_obs_off[lc + 1];
  const int* cpos = v.dense_mode ? v.lc_wpos : v.lc_pos;
  // cell header (keyframe, W slot, levels) one cell ahead of the arithmetic
  int c = c0 + gl, kf = 0, pos = -1;
  unsigned lv = 0x0101u;
  if (c < c1 && run) {
    kf = v.lc_kf[c]; pos = cpos[c];
    lv = *reinterpret_cast<const unsigned short*>(v.lc_level + 2 * (size_t)c);
  }
  while (c < c1 && run) {
    const int cn = c + LN_G;
    int kf_n = 0, pos_n = -1;
    unsigned lv_n = 0x0101u;
    if (cn < c1) {
      kf_n = v.lc_kf[cn]; pos_n = cpos[cn];
      lv_n = *reinterpret_cast<const unsigned short*>(v.lc_level + 2 * (size_t)cn);
    }
    double W[24];
#pragma unroll
    for (int k = 0; k < 24; k++) W[k] = 0.0;
    const unsigned lv0 = lv & 0xffu, lv1 = lv >> 8;
    if (!removed && (lv0 == 0 || lv1 == 0)) {
      double Rt[12];
      {
        const double2* rp = reinterpret_cast<const double2*>(v.pose_Rt[sel] + 12 * (size_t)kf);
#pragma unroll
        for (int k = 0; k < 6; k++) {
          const double2 t2 = rp[k];
          Rt[2 * k] = t2.x; Rt[2 * k + 1] = t2.y;
        }
      }
      const double* cam = v.kf_lcam + 4 * (size_t)kf;
      double P1[3], P2[3];
      map_Rt(Rt, X1, P1);
      map_Rt(Rt, X2, P2);
      const double delta = v.lc_stereo[c] ? v.prm.delta_ln_stereo : v.prm.delta_ln_mono;
#pragma unroll 1
      for (int side = 0; side < 2; side++) {
        if ((side == 0 ? lv0 : lv1) != 0) continue;
        nact++;
        LineObs o;
        make_line_obs(v, kf, (side == 0 ? v.lc_left : v.lc_right) + 4 * (size_t)c, o);
        double err[2], Jp[12], Jl[8];
        line_linearize<true>(P1, P2, cam[0], cam[1], cam[2], side ? -cam[3] : 0.0, o, Rt, X1, X2, r2, err, Jp, Jl);
        const double info = v.lc_info[2 * (size_t)c + side];
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
        double wgt = 1.0, rho = c2;
        if (v.prm.robust_ln) rho = huber(c2, delta, &wgt);
        chi += rho;
        const double wo = wgt * info;
        double JW[8];
#pragma unroll
        for (int k = 0; k < 8; k++) JW[k] = wo * Jl[k];
#pragma unroll
        for (int r = 0; r < 4; r++) {
#pragma unroll
          for (int cc = r; cc < 4; cc++) H[u4(r, cc)] += JW[r] * Jl[cc] + JW[4 + r] * Jl[4 + cc];
          bl[r] -= JW[r] * err[0] + JW[4 + r] * err[1];
        }
        if (pos >= 0) {
#pragma unroll
          for (int r = 0; r < 6; r++)
#pragma unroll
            for (int cc = 0; cc < 4; cc++) W[r * 4 + cc] += Jp[r] * JW[cc] + Jp[6 + r] * JW[4 + cc];
        }
      }
    }
    if (pos >= 0) {   // 192- / 304-byte records: 16-byte stores
      double2* Wo = reinterpret_cast<double2*>(v.dense_mode ? v.lc_Wl + 24 * (size_t)pos : v.L_rec + 38 * (size_t)pos);
#pragma unroll
      for (int k = 0; k < 12; k++) Wo[k] = make_double2(W[2 * k], W[2 * k + 1]);
    }
    c = cn; kf = kf_n; pos = pos_n; lv = lv_n;
  }
  // group sum (xor 4, 2, 1 inside the aligned group of LN_G lanes): every lane ends with the line's totals
#pragma unroll
  for (int o = LN_G / 2; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < 10; k++) H[k] += __shfl_xor_sync(0xffffffffu, H[k], o);
#pragma unroll
    for (int k = 0; k < 4; k++) bl[k] += __shfl_xor_sync(0xffffffffu, bl[k], o);
    chi += __shfl_xor_sync(0xffffffffu, chi, o);
    nact += __shfl_xor_sync(0xffffffffu, nact, o);
  }
  if (gl != 0 || !live) return;
  double* Ho = v.ln_H + 14 * (size_t)l;
  if (run) {
#pragma unroll
    for (int k = 0; k < 10; k++) Ho[k] = H[k];
#pragma unroll
    for (int k = 0; k < 4; k++) Ho[10 + k] = bl[k];
    const int li = v.n_pt + l;
    v.lm_chi2lin[li] = chi;
    v.lm_maxdiag[li] = nact ? fmax(fmax(fabs(H[u4(0, 0)]), fabs(H[u4(1, 1)])), fmax(fabs(H[u4(2, 2)]), fabs(H[u4(3, 3)]))) : 0.0;
    v.lm_active[li] = nact > 0;
  } else if (WITH_D && phase == PH_RETRY) {
#pragma unroll
    for (int k = 0; k < 10; k++) H[k] = Ho[k];
#pragma unroll
    for (int k = 0; k < 4; k++) bl[k] = Ho[10 + k];
  } else {
    return;
  }
  if (WITH_D) {   // k_schur_lines' work
    const double lam = v.w_lambda[w];
    double A[16], Di[16];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
      for (int c2 = 0; c2 < 4; c2++) A[4 * r + c2] = H[r <= c2 ? u4(r, c2) : u4(c2, r)] + (r == c2 ? lam : 0.0);
    inv4(A, Di);
    double* Do = v.lns_D + 14 * (size_t)v.ln_spos[l];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
      for (int c2 = r; c2 < 4; c2++) Do[u4(r, c2)] = Di[4 * r + c2];
#pragma unroll
    for (int i = 0; i < 4; i++) Do[10 + i] = Di[4 * i] * bl[0] + Di[4 * i + 1] * bl[1] + Di[4 * i + 2] * bl[2] + Di[4 * i + 3] * bl[3];
  }
}

// fixed-order reduction of NV per-thread values over the CTA (LM_TPB threads); result in out[0..NV) for all threads
template <int NV>
__device__ __forceinline__ void block_reduce_nv(const double* acc, double (*part)[NV], double* out) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    double x = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) part[wid][k] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s2 = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s2 += part[w][threadIdx.x];
    out[threadIdx.x] = s2;
  }
  __syncthreads();
}

// pose pass: one CTA per chunk of a free keyframe's edge list; recomputes residual, weight and the pose Jacobian
// and reduces Jp^T (w Omega) Jp and -Jp^T (w Omega) r in fixed order.
// measured on B200 (64 windows of 20/5k/1k, ms per bench step / ms in this kernel): plain 16.09 / 2.86, four resident CTAs per
// SM (128 registers) 15.77 / 2.55, data prefetch 15.88 / 2.67, both 15.67 / 2.45, five CTAs (96 registers, spills) 16.14 / 2.96
#ifndef LLD_POSES_MINB
#define LLD_POSES_MINB 4
#endif
#ifndef LLD_POSES_PREFETCH
#define LLD_POSES_PREFETCH 1
#endif
__global__ void __launch_bounds__(LM_TPB, LLD_POSES_MINB) k_lin_poses(BaView v) {
  const int ch = blockIdx.x;
  const int g = v.ch_g[ch];
  const int kf = v.g_kf[g];
  const int w = v.kf_win[kf];
  if (v.w_phase[w] != PH_LIN) return;
  const int sel = v.w_sel[w];
  __shared__ double tr[28][LM_TPB + 1];        // per-thread partials, transposed (row stride 129: conflict-free)
  __shared__ double part[LM_TPB / 32][28];
  const double* Rt = v.pose_Rt[sel] + 12 * (size_t)kf;
  const double* intr = v.kf_intr + 5 * (size_t)kf;
  const double* cam = v.kf_lcam + 4 * (size_t)kf;
  const bool is_pt = ch < v.n_chunks_pt;
  double acc[28];
#pragma unroll
  for (int k = 0; k < 28; k++) acc[k] = 0.0;
  // entry header (edge / cell, its landmark) one entry ahead: the list -> edge -> landmark -> state chain is four loads deep
  const int i_end = v.ch_end[ch];
  int i = v.ch_begin[ch] + threadIdx.x, id = 0, lm = 0;
  if (i < i_end) {
    id = is_pt ? v.pl_edge[i] : v.ll_cell[i];
    lm = is_pt ? v.pe_pt[id] : v.lc_ln[id];
  }
#if LLD_POSES_PREFETCH
  if (is_pt) {
    // point chunks: the DATA of the next entry (level, landmark position, observation, information) is loaded before the
    // arithmetic of the current one as well -- the kernel is bound by the latency of these gathers (ncu: 8.5 warps stalled
    // on the long scoreboard per issue at 12 warps per SM)
    struct PtData { uint8_t lvl; double X[3]; float obs[3]; float info; };
    auto load = [&](int e, int l, PtData& d) {
      d.lvl = v.pe_level[e];
      const double* X = v.pt_xyz[sel] + 3 * (size_t)l;
      d.X[0] = X[0]; d.X[1] = X[1]; d.X[2] = X[2];
      const float* o = v.pe_uvr + 3 * (size_t)e;
      d.obs[0] = o[0]; d.obs[1] = o[1]; d.obs[2] = o[2];
      d.info = v.pe_info[e];
    };
    PtData nxt;
    nxt.lvl = 1;
    if (i < i_end) load(id, lm, nxt);
    for (; i < i_end; i += blockDim.x) {
      const PtData cur = nxt;
      const int i2 = i + (int)blockDim.x;
      if (i2 < i_end) {
        const int e2 = v.pl_edge[i2];
        load(e2, v.pe_pt[e2], nxt);
      }
      if (cur.lvl != 0) continue;
      const bool stereo = !(cur.obs[2] < 0.f);
      double xc[3], err[3], Jp[18];
      map_Rt(Rt, cur.X, xc);
      pt_residual<true>(xc, intr, cur.obs, stereo, err);
      const double info = (double)cur.info;
      const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
      double wgt = 1.0;
      if (v.prm.robust_pt) huber(c2, stereo ? v.prm.delta_pt_stereo : v.prm.delta_pt_mono, &wgt);
      const double wo = wgt * info;
      pt_jac_pose(xc, intr, stereo, Jp);
      int k = 0;
#pragma unroll
      for (int r = 0; r < 6; r++) {
#pragma unroll
        for (int c = r; c < 6; c++, k++) acc[k] += wo * (Jp[r] * Jp[c] + Jp[6 + r] * Jp[6 + c] + Jp[12 + r] * Jp[12 + c]);
        acc[21 + r] -= wo * (Jp[r] * err[0] + Jp[6 + r] * err[1] + Jp[12 + r] * err[2]);
      }
      acc[27] += 1.0;
    }
    i = i_end;
  }
#endif
  for (; i < i_end; i += blockDim.x) {
    const int id_c = id, lm_c = lm;
    if (i + (int)blockDim.x < i_end) {
      id = is_pt ? v.pl_edge[i + blockDim.x] : v.ll_cell[i + blockDim.x];
      lm = is_pt ? v.pe_pt[id] : v.lc_ln[id];
    }
    if (is_pt) {
      const int e = id_c;
      if (v.pe_level[e] != 0) continue;
      const double* X = v.pt_xyz[sel] + 3 * (size_t)lm_c;
      const float* obs = v.pe_uvr + 3 * (size_t)e;
      const bool stereo = !(obs[2] < 0.f);
      double xc[3], err[3], Jp[18];
      map_Rt(Rt, X, xc);
      pt_residual<true>(xc, intr, obs, stereo, err);
      const double info = (double)v.pe_info[e];
      const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
      double wgt = 1.0;
      if (v.prm.robust_pt) huber(c2, stereo ? v.prm.delta_pt_stereo : v.prm.delta_pt_mono, &wgt);
      const double wo = wgt * info;
      pt_jac_pose(xc, intr, stereo, Jp);
      int k = 0;
#pragma unroll
      for (int r = 0; r < 6; r++) {
#pragma unroll
        for (int c = r; c < 6; c++, k++) acc[k] += wo * (Jp[r] * Jp[c] + Jp[6 + r] * Jp[6 + c] + Jp[12 + r] * Jp[12 + c]);
        acc[21 + r] -= wo * (Jp[r] * err[0] + Jp[6 + r] * err[1] + Jp[12 + r] * err[2]);
      }
      acc[27] += 1.0;
    } else {
      const int c = id_c;
      const int l = lm_c;
      if (v.ln_removed[l]) continue;
      const uint8_t lv0 = v.lc_level[2 * c], lv1 = v.lc_level[2 * c + 1];
      if (lv0 != 0 && lv1 != 0) continue;
      const double* stp = v.ln_st[sel] + 5 * (size_t)l;
      const double st[5] = {stp[0], stp[1], stp[2], stp[3], stp[4]};
      double r1[3], r2[3], X1[3], X2[3], P1[3], P2[3];
      line_axes(st, r1, r2);
#pragma unroll
      for (int q = 0; q < 3; q++) {
        X1[q] = st[4] * r2[q];
        X2[q] = X1[q] + r1[q];
      }
      map_Rt(Rt, X1, P1);
      map_Rt(Rt, X2, P2);
      const double delta = v.lc_stereo[c] ? v.prm.delta_ln_stereo : v.prm.delta_ln_mono;
#pragma unroll 1
      for (int side = 0; side < 2; side++) {
        if ((side == 0 ? lv0 : lv1) != 0) continue;
        LineObs o;
        make_line_obs(v, kf, (side == 0 ? v.lc_left : v.lc_right) + 4 * (size_t)c, o);
        double err[2], Jp[12];
        line_linearize<false>(P1, P2, cam[0], cam[1], cam[2], side ? -cam[3] : 0.0, o, Rt, X1, X2, r2, err, Jp, nullptr);
        const double info = v.lc_info[2 * (size_t)c + side];
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
        double wgt = 1.0;
        if (v.prm.robust_ln) huber(c2, delta, &wgt);
        const double wo = wgt * info;
        int k = 0;
#pragma unroll
        for (int r = 0; r < 6; r++) {
#pragma unroll
          for (int cc = r; cc < 6; cc++, k++) acc[k] += wo * (Jp[r] * Jp[cc] + Jp[6 + r] * Jp[6 + cc]);
          acc[21 + r] -= wo * (Jp[r] * err[0] + Jp[6 + r] * err[1]);
        }
        acc[27] += 1.0;
      }
    }
  }
  // fixed-order sum over the CTA through shared memory: 28 stores + 32 loads per thread instead of 28 five-step shuffle trees
#pragma unroll
  for (int k = 0; k < 28; k++) tr[k][threadIdx.x] = acc[k];
  __syncthreads();
  if (threadIdx.x < 28 * (LM_TPB / 32)) {
    const int k = threadIdx.x % 28, q = threadIdx.x / 28;
    double s2 = 0;
#pragma unroll 8
    for (int t = 0; t < 32; t++) s2 += tr[k][32 * q + t];
    part[q][k] = s2;
  }
  __syncthreads();
  if (threadIdx.x < 28) {
    double s2 = 0;
#pragma unroll
    for (int q = 0; q < LM_TPB / 32; q++) s2 += part[q][threadIdx.x];
    v.ch_pose[28 * (size_t)ch + threadIdx.x] = s2;
  }
}

// sum the chunk partials of each free keyframe (fixed order)
__global__ void k_reduce_pose(BaView v) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int g = t / 28, k = t % 28;
  if (g >= v.n_free_total) return;
  const int w = v.kf_win[v.g_kf[g]];
  if (v.w_phase[w] != PH_LIN) return;
  double s = 0;
  for (int ch = v.g_chp0[g]; ch < v.g_chp0[g + 1]; ch++) s += v.ch_pose[28 * (size_t)ch + k];
  for (int ch = v.g_chl0[g]; ch < v.g_chl0[g + 1]; ch++) s += v.ch_pose[28 * (size_t)ch + k];
  if (k < 21) v.g_Hpp[21 * (size_t)g + k] = s;
  else if (k < 27) v.g_bp[6 * (size_t)g + (k - 21)] = s;
  else v.g_nact[g] = (int)(s + 0.5);
}

// two-level per-window reduction of the landmark scalars written by the linearisation (chi2, max diag, #active):
// n_slices CTAs per window write partials, k_sum_lin adds them in fixed order
__global__ void __launch_bounds__(256) k_reduce_lin(BaView v) {
  const int w = blockIdx.x / v.n_slices, sl = blockIdx.x % v.n_slices;
  if (v.w_phase[w] != PH_LIN) return;
  __shared__ double sm[32];
  double chi = 0, mx = 0, na = 0;
  const int np = v.pt_off[w + 1] - v.pt_off[w], nl = v.ln_off[w + 1] - v.ln_off[w];
  const int p0 = v.pt_off[w] + (int)((long long)np * sl / v.n_slices), p1 = v.pt_off[w] + (int)((long long)np * (sl + 1) / v.n_slices);
  const int l0 = v.ln_off[w] + (int)((long long)nl * sl / v.n_slices), l1 = v.ln_off[w] + (int)((long long)nl * (sl + 1) / v.n_slices);
  for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    chi += v.lm_chi2lin[p];
    mx = fmax(mx, v.lm_maxdiag[p]);
    na += v.lm_active[p] ? 1.0 : 0.0;
  }
  for (int l = l0 + threadIdx.x; l < l1; l += blockDim.x) {
    chi += v.lm_chi2lin[v.n_pt + l];
    mx = fmax(mx, v.lm_maxdiag[v.n_pt + l]);
    na += v.lm_active[v.n_pt + l] ? 1.0 : 0.0;
  }
  chi = block_sum(chi, sm);
  na = block_sum(na, sm);
  mx = block_max(mx, sm);
  if (threadIdx.x == 0) {
    double* o = v.w_part + 4 * (size_t)blockIdx.x;
    o[0] = chi; o[1] = mx; o[2] = na;
  }
}
__global__ void k_sum_lin(BaView v) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= v.n_win || v.w_phase[w] != PH_LIN) return;
  double chi = 0, mx = 0, na = 0;
  for (int s2 = 0; s2 < v.n_slices; s2++) {
    const double* o = v.w_part + 4 * ((size_t)w * v.n_slices + s2);
    chi += o[0]; mx = fmax(mx, o[1]); na += o[2];
  }
  v.w_red_sum[4 * w + 0] = chi;
  v.w_red_sum[4 * w + 1] = 0.0;
  v.w_red_sum[4 * w + 2] = na;
  v.w_red_max[w] = mx;
}

// iteration start: currentChi, iniChi, lambda init at iteration 0 (optimization_algorithm_levenberg.cpp:75-97,166-180)
__device__ __forceinline__ void begin_window(const BaView& v, int w, bool pose_diag_in_max = false) {
  const double chi = v.w_red_sum[4 * w + 0];
  const int nact = (int)(v.w_red_sum[4 * w + 2] + 0.5);
  if (nact == 0 && v.w_iter[w] == 0) {  // empty index mapping: optimize() returns without iterating
    v.w_phase[w] = PH_DONE;
    atomicSub(v.n_active_win, 1);
    return;
  }
  v.w_curchi[w] = chi;
  v.w_inichi[w] = chi;
  v.w_trials[w] = 0;
  if (v.w_iter[w] == 0) {
    double mx = v.w_red_max[w];
    for (int g = v.w_g0[w]; g < v.w_g0[w + 1] && !pose_diag_in_max; g++) {
      if (v.g_nact[g] == 0) continue;
      const double* H = v.g_Hpp + 21 * (size_t)g;
      int k = 0;
      for (int r = 0; r < 6; r++) {
        mx = fmax(mx, fabs(H[k]));
        k += 6 - r;
      }
    }
    v.w_lambda[w] = 1e-5 * mx;
    v.w_ni[w] = 2.0;
    v.w_nbad[w] = 0;
    const int n = v.w_nlog[w];
    if (n < v.log_stride) v.chi2_log[(size_t)w * v.log_stride + n] = chi;
    v.w_nlog[w] = n + 1;
  }
}

__global__ void k_begin(BaView v) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= v.n_win) return;
  if (v.w_phase[w] != PH_LIN) return;
  begin_window(v, w);
}

// single-rank fast path: chunk partial sums of the window's keyframes, landmark scalars and the iteration-start
// bookkeeping in one CTA per window (saves two launches and their dependent-load latency per LM step).
// 1024 threads and 4-way unrolled independent loads: for a single window this kernel is pure memory latency.
constexpr int FUSED_RED_TPB = 1024;
__global__ void __launch_bounds__(FUSED_RED_TPB) k_begin_fused(BaView v) {
  const int w = blockIdx.x;
  if (v.w_phase[w] != PH_LIN) return;
  __shared__ double sm[32];
  __shared__ double spart[4][32 * 28];  // up to 32 free keyframes (dense mode) x 28 values x 4 chunk quarters
  const int g0 = v.w_g0[w], nf = v.w_g0[w + 1] - g0;
  const int tid = threadIdx.x;
  const bool small = nf >= 1 && nf <= 32;
  const int parts = small ? min(4, FUSED_RED_TPB / (nf * 28)) : 1;   // 1..4 slices of every keyframe's chunk range
  if (small) {  // thread = (slice of the chunk range, keyframe, value); the slices are added in fixed order
    const int qtr = tid / (nf * 28), x = tid - qtr * (nf * 28);
    if (qtr < parts) {
      const int g = g0 + x / 28, k = x % 28;
      double s2 = 0;
      for (int rng = 0; rng < 2; rng++) {  // the quarter's share of the point chunks, then of the line chunks
        const int c0 = rng == 0 ? v.g_chp0[g] : v.g_chl0[g], c1 = rng == 0 ? v.g_chp0[g + 1] : v.g_chl0[g + 1];
        const int n = c1 - c0, b = c0 + (n * qtr) / parts, e = c0 + (n * (qtr + 1)) / parts;
        int ch = b;
        for (; ch + 4 <= e; ch += 4) {
          const double a0 = v.ch_pose[28 * (size_t)ch + k], a1 = v.ch_pose[28 * (size_t)(ch + 1) + k],
                       a2 = v.ch_pose[28 * (size_t)(ch + 2) + k], a3 = v.ch_pose[28 * (size_t)(ch + 3) + k];
          s2 += a0; s2 += a1; s2 += a2; s2 += a3;
        }
        for (; ch < e; ch++) s2 += v.ch_pose[28 * (size_t)ch + k];
      }
      spart[qtr][x] = s2;
    }
  }
  __syncthreads();
  if (small) {
    for (int x = tid; x < nf * 28; x += blockDim.x) {
      const int g = g0 + x / 28, k = x % 28;
      double s2 = spart[0][x];
      for (int q = 1; q < parts; q++) s2 += spart[q][x];
      if (k < 21) v.g_Hpp[21 * (size_t)g + k] = s2;
      else if (k < 27) v.g_bp[6 * (size_t)g + (k - 21)] = s2;
      else v.g_nact[g] = (int)(s2 + 0.5);
    }
  } else {
    for (int x = tid; x < nf * 28; x += blockDim.x) {
      const int g = g0 + x / 28, k = x % 28;
      double s2 = 0;
      for (int ch = v.g_chp0[g]; ch < v.g_chp0[g + 1]; ch++) s2 += v.ch_pose[28 * (size_t)ch + k];
      for (int ch = v.g_chl0[g]; ch < v.g_chl0[g + 1]; ch++) s2 += v.ch_pose[28 * (size_t)ch + k];
      if (k < 21) v.g_Hpp[21 * (size_t)g + k] = s2;
      else if (k < 27) v.g_bp[6 * (size_t)g + (k - 21)] = s2;
      else v.g_nact[g] = (int)(s2 + 0.5);
    }
  }
  __syncthreads();
  double chi = 0, mx = 0, na = 0;
  for (int x = tid; x < nf * 6; x += blockDim.x) {  // lambda init also looks at the pose diagonal (levenberg.cpp:166-180)
    const int g = g0 + x / 6, r = x % 6;
    if (v.g_nact[g] != 0) mx = fmax(mx, fabs(v.g_Hpp[21 * (size_t)g + (r * 6 - (r * (r - 1)) / 2)]));
  }
  {
    const int p0 = v.pt_off[w], p1 = v.pt_off[w + 1];
    int p = p0 + tid;
    for (; p + 3 * FUSED_RED_TPB < p1; p += 4 * FUSED_RED_TPB) {
      const double c0 = v.lm_chi2lin[p], c1 = v.lm_chi2lin[p + FUSED_RED_TPB], c2 = v.lm_chi2lin[p + 2 * FUSED_RED_TPB],
                   c3 = v.lm_chi2lin[p + 3 * FUSED_RED_TPB];
      const double m0 = v.lm_maxdiag[p], m1 = v.lm_maxdiag[p + FUSED_RED_TPB], m2 = v.lm_maxdiag[p + 2 * FUSED_RED_TPB],
                   m3 = v.lm_maxdiag[p + 3 * FUSED_RED_TPB];
      const int a0 = v.lm_active[p], a1 = v.lm_active[p + FUSED_RED_TPB], a2 = v.lm_active[p + 2 * FUSED_RED_TPB],
                a3 = v.lm_active[p + 3 * FUSED_RED_TPB];
      chi += c0; chi += c1; chi += c2; chi += c3;
      mx = fmax(fmax(fmax(mx, m0), fmax(m1, m2)), m3);
      na += (a0 ? 1.0 : 0.0) + (a1 ? 1.0 : 0.0) + (a2 ? 1.0 : 0.0) + (a3 ? 1.0 : 0.0);
    }
    for (; p < p1; p += FUSED_RED_TPB) {
      chi += v.lm_chi2lin[p];
      mx = fmax(mx, v.lm_maxdiag[p]);
      na += v.lm_active[p] ? 1.0 : 0.0;
    }
  }
  for (int l = v.ln_off[w] + tid; l < v.ln_off[w + 1]; l += blockDim.x) {
    chi += v.lm_chi2lin[v.n_pt + l];
    mx = fmax(mx, v.lm_maxdiag[v.n_pt + l]);
    na += v.lm_active[v.n_pt + l] ? 1.0 : 0.0;
  }
  chi = block_sum(chi, sm);
  na = block_sum(na, sm);
  mx = block_max(mx, sm);
  if (tid == 0) {
    v.w_red_sum[4 * w + 0] = chi;
    v.w_red_sum[4 * w + 1] = 0.0;
    v.w_red_sum[4 * w + 2] = na;
    v.w_red_max[w] = mx;
  }
  if (tid == 0) begin_window(v, w, true);
}

// per free keyframe: fixed-order sum of its chunk partials (k_lin_poses) into H_pp, b_p and the active-edge count; the
// part of k_begin_fused that every LM step needs (the rest of it is the lambda_0 / chi2 bookkeeping of a first step)
__global__ void __launch_bounds__(128) k_pose_sum(BaView v) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int g = t / 28, k = t - 28 * g;
  if (g >= v.n_free_total) return;
  const int w = v.kf_win[v.g_kf[g]];
  if (v.w_phase[w] != PH_LIN) return;
  double s2 = 0;
  for (int rng = 0; rng < 2; rng++) {
    const int c0 = rng == 0 ? v.g_chp0[g] : v.g_chl0[g], c1 = rng == 0 ? v.g_chp0[g + 1] : v.g_chl0[g + 1];
    int ch = c0;
    for (; ch + 4 <= c1; ch += 4) {
      const double a0 = v.ch_pose[28 * (size_t)ch + k], a1 = v.ch_pose[28 * (size_t)(ch + 1) + k],
                   a2 = v.ch_pose[28 * (size_t)(ch + 2) + k], a3 = v.ch_pose[28 * (size_t)(ch + 3) + k];
      s2 += a0; s2 += a1; s2 += a2; s2 += a3;
    }
    for (; ch < c1; ch++) s2 += v.ch_pose[28 * (size_t)ch + k];
  }
  if (k < 21) v.g_Hpp[21 * (size_t)g + k] = s2;
  else if (k < 27) v.g_bp[6 * (size_t)g + (k - 21)] = s2;
  else v.g_nact[g] = (int)(s2 + 0.5);
}

// ------------------------------------------------------------------------------------------------
// trial: Schur complement pieces per landmark (lambda dependent)
// ------------------------------------------------------------------------------------------------
// per landmark: Dinv = (Hll + lambda I)^-1 (general inverse, block_solver.hpp:389), c = Dinv b_l; both are also
// scattered into the list-order records so that k_schur_rows reads one contiguous record per entry.
__global__ void __launch_bounds__(LM_TPB) k_schur_points(BaView v) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= v.n_pt) return;
  const int w = v.pt_win[p];
  if (v.w_phase[w] == PH_DONE) return;
  const double lam = v.w_lambda[w];
  const double* Hi = v.pt_H + 9 * (size_t)p;
  double Di[9];
  {
    const double A[9] = {Hi[0] + lam, Hi[1], Hi[2], Hi[1], Hi[3] + lam, Hi[4], Hi[2], Hi[4], Hi[5] + lam};
    inv3_sym(A, Di);
  }
  double rec[9] = {Di[0], Di[1], Di[2], Di[4], Di[5], Di[8], 0, 0, 0};
#pragma unroll
  for (int i = 0; i < 3; i++) rec[6 + i] = Di[3 * i] * Hi[6] + Di[3 * i + 1] * Hi[7] + Di[3 * i + 2] * Hi[8];
  double* Do = v.dense_mode ? v.pts_D + 10 * (size_t)v.pt_spos[p] : v.pt_D + 9 * (size_t)p;
#pragma unroll
  for (int k = 0; k < 9; k++) Do[k] = rec[k];
  if (v.dense_mode) return;
  for (int e = v.pt_obs_off[p]; e < v.pt_obs_off[p + 1]; e++) {
    const int pos = v.pe_pos[e];
    if (pos < 0) continue;
    double* R = v.P_rec + 27 * (size_t)pos + 18;
#pragma unroll
    for (int k = 0; k < 9; k++) R[k] = rec[k];
  }
}

__global__ void __launch_bounds__(LM_TPB) k_schur_lines(BaView v) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= v.n_ln) return;
  const int w = v.ln_win[l];
  if (v.w_phase[w] == PH_DONE) return;
  const double lam = v.w_lambda[w];
  const double* Hi = v.ln_H + 14 * (size_t)l;
  double Di[16];
  {
    double A[16];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
      for (int c = 0; c < 4; c++) A[4 * r + c] = Hi[r <= c ? u4(r, c) : u4(c, r)] + (r == c ? lam : 0.0);
    inv4(A, Di);
  }
  double rec[14];
#pragma unroll
  for (int r = 0; r < 4; r++)
#pragma unroll
    for (int c = r; c < 4; c++) rec[u4(r, c)] = Di[4 * r + c];
#pragma unroll
  for (int i = 0; i < 4; i++)
    rec[10 + i] = Di[4 * i] * Hi[10] + Di[4 * i + 1] * Hi[11] + Di[4 * i + 2] * Hi[12] + Di[4 * i + 3] * Hi[13];
  double* Do = v.dense_mode ? v.lns_D + 14 * (size_t)v.ln_spos[l] : v.ln_D + 14 * (size_t)l;
#pragma unroll
  for (int k = 0; k < 14; k++) Do[k] = rec[k];
  if (v.dense_mode) return;
  for (int cc = v.ln_obs_off[l]; cc < v.ln_obs_off[l + 1]; cc++) {
    const int pos = v.lc_pos[cc];
    if (pos < 0) continue;
    double* R = v.L_rec + 38 * (size_t)pos + 24;
#pragma unroll
    for (int k = 0; k < 14; k++) R[k] = rec[k];
  }
}

// Schur rows: CTA = one chunk of free keyframe a's list; thread t = (neighbour j, column c) owns the 6 accumulators
// S[a, nb_j][0..5][c] in registers.  Per list entry (landmark l seen by a) and every free b >= a that also sees l:
//   S[a,b] -= W_(l,a) Dinv_l W_(l,b)^T ;   bschur[a] -= W_(l,a) (Dinv_l b_l)          (block_solver.hpp:381-440)
// Entries are grouped into segments that share one set of co-observing keyframes, so a thread tests "does my
// neighbour see these landmarks" once per segment; own records (W_a, Dinv, c) are staged through shared memory in
// coalesced blocks; the co-edge row W_b[c][:] is a gather through the int position table.
constexpr int ROW_SB = 32;  // entries staged per block
template <int D, int MAXT>
__global__ void __launch_bounds__(MAXT) k_schur_rows(BaView v, int chunk_base) {
  constexpr int REC = 6 * D + D * (D + 1) / 2 + D;
  constexpr int OFF_D = 6 * D, OFF_C = 6 * D + D * (D + 1) / 2;
  const int ch = chunk_base + blockIdx.x;
  const int g = v.ch_g[ch];
  const int kf = v.g_kf[g];
  const int w = v.kf_win[kf];
  if (v.w_phase[w] == PH_DONE) return;
  __shared__ double srec[ROW_SB * REC];
  const int nnb = v.nb_off[g + 1] - v.nb_off[g];
  const int t = threadIdx.x;
  const bool live = t < 6 * nnb;
  const int j = live ? t / 6 : 0, c = t - 6 * (t / 6);
  double acc[6] = {0, 0, 0, 0, 0, 0};
  double bacc = 0;
  const int i0 = v.ch_begin[ch], i1 = v.ch_end[ch];
  const double* rec_g = D == 3 ? v.P_rec : v.L_rec;
  const int l_off = (D == 3 ? v.pl_off : v.ll_off)[g];
  const int* tab = (D == 3 ? v.pl_tab : v.ll_tab) + (D == 3 ? v.pl_tab_off : v.ll_tab_off)[g] + (long long)(i0 - l_off) * nnb + j;
  int seg = v.ch_seg0[ch];
  const int seg_end_idx = v.ch_seg0[ch + 1];
  for (int blk = i0; blk < i1; blk += ROW_SB) {
    const int nb = min(ROW_SB, i1 - blk);
    __syncthreads();
    for (int q = t; q < nb * REC; q += blockDim.x) srec[q] = rec_g[(size_t)blk * REC + q];
    __syncthreads();
    // segments intersecting [blk, blk+nb)
    while (seg < seg_end_idx && v.seg_end[seg] <= blk) seg++;
    for (int s2 = seg; s2 < seg_end_idx && v.seg_begin[s2] < blk + nb; s2++) {
      const int a = max(v.seg_begin[s2], blk), b = min(v.seg_end[s2], blk + nb);
      if (!live) continue;
      if (j == 0) {  // b_schur part (every entry)
        for (int i = a; i < b; i++) {
          const double* R = srec + (i - blk) * REC;
          double sb = 0;
#pragma unroll
          for (int k = 0; k < D; k++) sb += R[D * c + k] * R[OFF_C + k];
          bacc += sb;
        }
      }
      if (tab[(long long)(a - i0) * nnb] < 0) continue;  // the whole segment misses this neighbour
#pragma unroll 4
      for (int i = a; i < b; i++) {
        const int pos2 = tab[(long long)(i - i0) * nnb];
        const double* Wb = rec_g + (size_t)pos2 * REC + D * c;
        const double* R = srec + (i - blk) * REC;
        double wb[D], z[D];
#pragma unroll
        for (int k = 0; k < D; k++) wb[k] = Wb[k];
        if (D == 3) {
          z[0] = R[OFF_D + 0] * wb[0] + R[OFF_D + 1] * wb[1] + R[OFF_D + 2] * wb[2];
          z[1] = R[OFF_D + 1] * wb[0] + R[OFF_D + 3] * wb[1] + R[OFF_D + 4] * wb[2];
          z[2] = R[OFF_D + 2] * wb[0] + R[OFF_D + 4] * wb[1] + R[OFF_D + 5] * wb[2];
        } else {
#pragma unroll
          for (int r = 0; r < D; r++) {
            double zz = 0;
#pragma unroll
            for (int k = 0; k < D; k++) zz += R[OFF_D + (r <= k ? u4(r, k) : u4(k, r))] * wb[k];
            z[r] = zz;
          }
        }
#pragma unroll
        for (int r = 0; r < 6; r++) {
          double a2 = 0;
#pragma unroll
          for (int k = 0; k < D; k++) a2 += R[D * r + k] * z[k];
          acc[r] += a2;
        }
      }
    }
  }
  if (live) {
    double* out = v.ch_S + v.ch_S_off[ch];
    const int ld = 6 * nnb;
#pragma unroll
    for (int r = 0; r < 6; r++) out[(size_t)r * ld + t] = acc[r];
    if (j == 0) out[(size_t)6 * ld + c] = bacc;
  }
}

// S(a, nb_j) = [j==0] (Hpp_a + lambda I) - sum_chunks partial ; bschur_a = bp_a - sum_chunks partial_b
__global__ void k_reduce_rows(BaView v, int with_diag) {
  const int g = blockIdx.x;
  const int w = v.kf_win[v.g_kf[g]];
  if (v.w_phase[w] == PH_DONE) return;
  const int nnb = v.nb_off[g + 1] - v.nb_off[g];
  const int ld = 6 * nnb;
  const double lam = v.w_lambda[w];
  for (int t = threadIdx.x; t < ld; t += blockDim.x) {
    const int j = t / 6, c = t - 6 * j;
    double s[6] = {0, 0, 0, 0, 0, 0};
    double sb = 0;
    for (int rng = 0; rng < 2; rng++) {
      const int c0 = rng == 0 ? v.g_chp0[g] : v.g_chl0[g], c1 = rng == 0 ? v.g_chp0[g + 1] : v.g_chl0[g + 1];
      for (int ch = c0; ch < c1; ch++) {
        const double* part = v.ch_S + v.ch_S_off[ch];
#pragma unroll
        for (int r = 0; r < 6; r++) s[r] += part[(size_t)r * ld + t];
        if (j == 0) sb += part[(size_t)6 * ld + c];
      }
    }
    double* S = v.S_blk + 36 * (size_t)(v.nb_off[g] + j);
#pragma unroll
    for (int r = 0; r < 6; r++) {
      double d = 0.0;
      if (j == 0 && with_diag) {
        const int rr = r < c ? r : c, cc = r < c ? c : r;
        d = v.g_Hpp[21 * (size_t)g + (rr * 6 - (rr * (rr - 1)) / 2 + (cc - rr))];
        if (r == c) d += lam;
      }
      S[6 * r + c] = d - s[r];
    }
    if (j == 0) v.g_bs[6 * (size_t)g + c] = (with_diag ? v.g_bp[6 * (size_t)g + c] : 0.0) - sb;
  }
}

// ------------------------------------------------------------------------------------------------
// k_schur_tile: dense mode Schur complement by co-visibility classes, staged through shared memory by persistent CTAs.
// Landmarks are stored in signature order; a "piece" is a run of landmarks seen by exactly the same n free keyframes,
// with their W blocks contiguous and sorted by keyframe.  Per piece: S_(a,b) += sum_l W_(l,a) Dinv_l W_(l,b)^T for every
// pair a <= b of its keyframes and b_schur_a += sum_l W_(l,a) (Dinv_l b_l); outputs go to a scratch slot per task and
// k_reduce_piece sums them per S block in fixed order (block_solver.hpp:381-440 without atomics).
// An item = (piece, block of <= SP_TPB tasks); a task is half of a pair's 6x6 block (6 rows x 3 columns) or one b_schur
// vector.  Every CTA walks its items (blockIdx.x, + gridDim.x, ...; windows that are done are skipped 32 items at a
// time) as one stream of landmark chunks: while chunk i is computed, chunk i + 1 (of the same or of the next item) is
// already in flight (cp.async, two buffers), so the DRAM latency is paid once per CTA, not once per piece.  Per chunk:
// the piece's contiguous W blocks and inverse records land in shared memory (every byte read once, coalesced),
// Z_(l,b) = W_(l,b) Dinv_l is formed once per (landmark, keyframe) (plus a pseudo block [Dinv_l b_l, 0..], so that the
// b_schur tasks run the same code), and thread (task, slice s) accumulates W_(l,ia) Z_(l,ib)^T over the landmarks
// l = s, s + S, ... : 18 + 3 D shared loads per 18 D FMAs, no global loads in the loop.  Slices are summed in fixed
// order through shared memory; outputs land in the scratch slots k_reduce_piece gathers.
// ------------------------------------------------------------------------------------------------
constexpr int SP_TPB = 128;
constexpr int SP_CAP_WD = 2304;  // doubles per W + inverse-record buffer (two of them)
constexpr int SP_CAP_Z = 2560;   // doubles of the Z buffer (>= SP_TPB * 18: it also carries the slice sums)
constexpr int SP_SMEM_BYTES = (2 * SP_CAP_WD + SP_CAP_Z) * 8;
constexpr int SP_MAX_S = 16;

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(dst_smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(src));
}

// host side: chunk length / slices of an item (D = 3 points, 4 lines)
inline void schur_item_shape(int D, int n, int nl, int t0, int* lc, int* S, int* nchunk) {
  const int WS = 6 * D, DS = D == 3 ? 10 : 14;
  const int ntask = n * (n + 1) + n;
  int ntb = ntask - t0 < SP_TPB ? ntask - t0 : SP_TPB;
  if (ntb < 1) ntb = 1;
  int L = SP_CAP_WD / (n * WS + DS);
  const int Lz = SP_CAP_Z / ((n + 1) * WS);
  if (Lz < L) L = Lz;
  if (nl < L) L = nl;
  int s = SP_TPB / ntb;
  if (s > SP_MAX_S) s = SP_MAX_S;
  if (s > L / 2) s = L / 2;
  if (s < 1) s = 1;
  *lc = L; *S = s; *nchunk = (nl + L - 1) / L;
}

template <int D>
__global__ void __launch_bounds__(SP_TPB, 4) k_schur_tile(BaView v, int item_base, int n_items) {
  constexpr int WS = 6 * D;
  constexpr int DS = D == 3 ? 10 : 14;
  constexpr int OFF_C = D * (D + 1) / 2;
  extern __shared__ __align__(16) double sp_smem[];
  double* const sZ = sp_smem + 2 * SP_CAP_WD;
  const int tid = threadIdx.x, lane = tid & 31;
  const int G = gridDim.x;
  const int cnt = (n_items - (int)blockIdx.x + G - 1) / G;
  const SchurItem* items = v.it_rec + item_base + blockIdx.x;
  const double* Wbase = D == 3 ? v.pe_Wl : v.lc_Wl;
  const double* Dbase = D == 3 ? v.pts_D : v.lns_D;

  // the CTA's items whose window is still running, 32 at a time (every warp evaluates the same ballot)
  int scan_base = -32;
  unsigned scan_mask = 0;
  auto next_item = [&]() -> int {
    while (true) {
      if (scan_mask) {
        const int j = __ffs(scan_mask) - 1;
        scan_mask &= scan_mask - 1;
        return scan_base + j;
      }
      scan_base += 32;
      if (scan_base >= cnt) return -1;
      const int j = scan_base + lane;
      bool a = false;
      if (j < cnt) a = v.w_phase[items[(size_t)j * G].w] != PH_DONE;
      scan_mask = __ballot_sync(0xffffffffu, a);
    }
  };
  auto load_item = [&](int k, SchurItem& R) {
    const int4* p = reinterpret_cast<const int4*>(items + (size_t)k * G);
    const int4 a = p[0], b = p[1];
    R.l0 = a.x; R.nl = a.y; R.n = a.z; R.t0 = a.w;
    R.w = b.x;
    R.w0 = ((long long)(unsigned)b.w << 32) | (unsigned)b.z;
    const int4 c2 = p[2];
    R.out = ((long long)(unsigned)c2.y << 32) | (unsigned)c2.x;
    R.lc = b.y; R.S = c2.z; R.nchunk = c2.w;
  };
  auto issue = [&](const SchurItem& R, int c, int b) {
    const int rowW = R.n * WS;
    const int Lc = R.lc;
    const int lc0 = c * Lc, m = min(Lc, R.nl - lc0);
    double* sW = sp_smem + b * SP_CAP_WD;
    double* sD = sW + Lc * rowW;
    const double* gW = Wbase + (size_t)R.w0 * WS + (size_t)lc0 * rowW;
    const int nW = m * rowW / 2;
    for (int i = tid; i < nW; i += SP_TPB) cp_async16(sW + 2 * i, gW + 2 * i);
    const double* gD = Dbase + (size_t)(R.l0 + lc0) * DS;
    const int nD = m * DS / 2;
    for (int i = tid; i < nD; i += SP_TPB) cp_async16(sD + 2 * i, gD + 2 * i);
  };

  int cur = next_item();
  if (cur < 0) return;
  SchurItem R, Rn;
  load_item(cur, R);
  issue(R, 0, 0);
  asm volatile("cp.async.commit_group;\n" ::);
  int nxt = next_item();
  Rn = R;
  if (nxt >= 0) load_item(nxt, Rn);
  int buf = 0, c = 0;
  while (true) {
    // ---- per item: task of this thread ----
    const int n = R.n, nl = R.nl;
    const int npair = n * (n + 1) / 2, ntask = 2 * npair + n;
    const int ntb = min(SP_TPB, ntask - R.t0);
    const int rowW = n * WS, rowZ = (n + 1) * WS;
    const int Lc = R.lc, nchunk = R.nchunk, S = R.S;
    const int s = tid / ntb, tl = tid - s * ntb;
    const bool act = s < S;
    int ia = 0, zb = n, h = 0;
    {
      const int task = R.t0 + tl;
      if (task < 2 * npair) {
        int pr = task >> 1;
        h = task & 1;
        while (pr >= n - ia) { pr -= n - ia; ia++; }
        zb = ia + pr;
      } else {
        ia = min(task - 2 * npair, n - 1);
      }
    }
    // (landmark, block) of this thread's Z blocks: start and stride of tid + k SP_TPB in base n + 1
    const int zl0 = tid / (n + 1), zb0 = tid - zl0 * (n + 1);
    const int zdl = SP_TPB / (n + 1), zdb = SP_TPB - zdl * (n + 1);
    double acc[18];
#pragma unroll
    for (int q = 0; q < 18; q++) acc[q] = 0.0;
    for (c = 0; c < nchunk; c++, buf ^= 1) {
      // next chunk of the stream into the other buffer
      if (c + 1 < nchunk) issue(R, c + 1, buf ^ 1);
      else if (nxt >= 0) issue(Rn, 0, buf ^ 1);
      asm volatile("cp.async.commit_group;\n" ::);
      asm volatile("cp.async.wait_group 1;\n" ::: "memory");
      __syncthreads();
      const int m = min(Lc, nl - c * Lc);
      const double* sW = sp_smem + buf * SP_CAP_WD;
      const double* sD = sW + Lc * rowW;
      for (int i = tid, l = zl0, b = zb0; i < m * (n + 1); i += SP_TPB) {
        const double* Dv = sD + l * DS;
        double* z = sZ + l * rowZ + b * WS;
        if (b < n) {
          const double* wv = sW + l * rowW + b * WS;
          double dm[D][D];
#pragma unroll
          for (int k = 0; k < D; k++)
#pragma unroll
            for (int j = 0; j < D; j++) {
              const int r = k < j ? k : j, c2 = k < j ? j : k;
              dm[k][j] = Dv[r * D - (r * (r - 1)) / 2 + (c2 - r)];
            }
#pragma unroll
          for (int cc = 0; cc < 6; cc++) {
            double wb[D];
#pragma unroll
            for (int j = 0; j < D; j++) wb[j] = wv[cc * D + j];
#pragma unroll
            for (int k = 0; k < D; k++) {
              double zz = 0;
#pragma unroll
              for (int j = 0; j < D; j++) zz += dm[k][j] * wb[j];
              z[cc * D + k] = zz;
            }
          }
        } else {
#pragma unroll
          for (int k = 0; k < WS; k++) z[k] = k < D ? Dv[OFF_C + k] : 0.0;
        }
        l += zdl; b += zdb;
        if (b > n) { b -= n + 1; l++; }
      }
      __syncthreads();
      if (act) {
        const double* wa_p = sW + ia * WS;
        const double* z_p = sZ + zb * WS + h * 3 * D;
#pragma unroll 2
        for (int l = s; l < m; l += S) {
          double wa[WS];
          const double* wp = wa_p + l * rowW;
#pragma unroll
          for (int k = 0; k < WS; k += 2) {
            const double2 t2 = *reinterpret_cast<const double2*>(wp + k);
            wa[k] = t2.x; wa[k + 1] = t2.y;
          }
          const double* zp = z_p + l * rowZ;
#pragma unroll
          for (int cc = 0; cc < 3; cc++) {
            double z[D];
#pragma unroll
            for (int k = 0; k < D; k++) z[k] = zp[cc * D + k];
#pragma unroll
            for (int r = 0; r < 6; r++) {
              double a2 = acc[cc * 6 + r];
#pragma unroll
              for (int k = 0; k < D; k++) a2 += wa[D * r + k] * z[k];
              acc[cc * 6 + r] = a2;
            }
          }
        }
      }
      __syncthreads();
    }
    // ---- outputs: slices summed in fixed order (the Z buffer is free until the next chunk's barrier) ----
    double* out = v.dpart + R.out;
    if (S == 1) {
      if (tid < ntb) {
        const int task = R.t0 + tl;
        if (task < 2 * npair) {
          double* o = out + (size_t)(task >> 1) * 36 + (task & 1) * 18;
#pragma unroll
          for (int q = 0; q < 18; q++) o[q] = acc[q];
        } else {
          double* o = out + (size_t)36 * npair + (size_t)(task - 2 * npair) * SCHUR_KS;
#pragma unroll
          for (int q = 0; q < 6; q++) o[q] = acc[q];
        }
      }
    } else {
      double* red = sZ;
      if (act)
#pragma unroll
        for (int q = 0; q < 18; q++) red[(s * ntb + tl) * 18 + q] = acc[q];
      __syncthreads();
      for (int e = tid; e < ntb * 18; e += SP_TPB) {
        const int tl2 = e / 18, q = e - 18 * tl2;
        const int task = R.t0 + tl2;
        size_t o;
        if (task < 2 * npair) o = (size_t)(task >> 1) * 36 + (task & 1) * 18 + q;
        else if (q < 6) o = (size_t)36 * npair + (size_t)(task - 2 * npair) * SCHUR_KS + q;
        else continue;
        double sum = 0;
        for (int s2 = 0; s2 < S; s2++) sum += red[(s2 * ntb + tl2) * 18 + q];
        out[o] = sum;
      }
    }
    if (nxt < 0) break;
    cur = nxt;
    R = Rn;
    nxt = next_item();
    if (nxt >= 0) load_item(nxt, Rn);
  }
}

// S(a,b) = [a==b] (Hpp_a + lambda I) - sum over contributing (piece, pair) ; bschur_a = bp_a - sum b tasks
// one thread per element of an S block (36 consecutive threads read 288 contiguous bytes of every contribution) and per
// element of b_schur; the gather list is walked in its fixed order
__global__ void __launch_bounds__(256) k_reduce_piece(BaView v, int n_blocks) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_blocks * 36) {
    const int blk = t / 36, e = t - 36 * blk, c = e / 6, r = e - 6 * c;
    int lo = 0, hi = v.n_free_total;   // owning free block row g: largest g with nb_off[g] <= blk
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (v.nb_off[mid] <= blk) lo = mid;
      else hi = mid;
    }
    const int g = lo, j = blk - v.nb_off[g];
    const int w = v.kf_win[v.g_kf[g]];
    if (v.w_phase[w] == PH_DONE) return;
    double s = 0;
    const int q1 = v.gb_off[blk + 1];
    int q = v.gb_off[blk];
    for (; q + 8 <= q1; q += 8) {   // eight gathers in flight (the kernel is bound by their latency); the sum stays in list order
      long long o[8];
      double a[8];
#pragma unroll
      for (int k = 0; k < 8; k++) o[k] = v.gb_src[q + k];
#pragma unroll
      for (int k = 0; k < 8; k++) a[k] = v.dpart[o[k] + e];
#pragma unroll
      for (int k = 0; k < 8; k++) s += a[k];
    }
    for (; q + 4 <= q1; q += 4) {
      const long long o0 = v.gb_src[q], o1 = v.gb_src[q + 1], o2 = v.gb_src[q + 2], o3 = v.gb_src[q + 3];
      const double a0 = v.dpart[o0 + e], a1 = v.dpart[o1 + e], a2 = v.dpart[o2 + e], a3 = v.dpart[o3 + e];
      s += a0; s += a1; s += a2; s += a3;
    }
    for (; q < q1; q++) s += v.dpart[v.gb_src[q] + e];
    double d = 0.0;
    if (j == 0) {
      const int rr = r < c ? r : c, cc = r < c ? c : r;
      d = v.g_Hpp[21 * (size_t)g + (rr * 6 - (rr * (rr - 1)) / 2 + (cc - rr))];
      if (r == c) d += v.w_lambda[w];
    }
    v.S_blk[36 * (size_t)blk + 6 * r + c] = d - s;
  } else {
    const int u = t - n_blocks * 36;
    const int g = u / 6, r = u - 6 * g;
    if (g >= v.n_free_total) return;
    const int w = v.kf_win[v.g_kf[g]];
    if (v.w_phase[w] == PH_DONE) return;
    double s = 0;
    for (int q = v.gv_off[g]; q < v.gv_off[g + 1]; q++) s += v.dpart[v.gv_src[q] + r];
    v.g_bs[6 * (size_t)g + r] = v.g_bp[6 * (size_t)g + r] - s;
  }
}

// the same sums for long gather lists (few windows cut into many short pieces): one warp per (block, column c) and per
// free keyframe, lanes stride over the gather list, fixed-order shuffle tree
__global__ void __launch_bounds__(256) k_reduce_piece_warp(BaView v, int n_blocks) {
  const int wi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (wi < n_blocks * 6) {
    const int blk = wi / 6, c = wi - 6 * blk;
    int lo = 0, hi = v.n_free_total;   // owning free block row g: largest g with nb_off[g] <= blk
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (v.nb_off[mid] <= blk) lo = mid;
      else hi = mid;
    }
    const int g = lo, j = blk - v.nb_off[g];
    const int w = v.kf_win[v.g_kf[g]];
    if (v.w_phase[w] == PH_DONE) return;
    double s[6] = {0, 0, 0, 0, 0, 0};
    for (int q = v.gb_off[blk] + lane; q < v.gb_off[blk + 1]; q += 32) {
      const double* src = v.dpart + v.gb_src[q] + 6 * c;
#pragma unroll
      for (int r = 0; r < 6; r++) s[r] += src[r];
    }
#pragma unroll
    for (int r = 0; r < 6; r++) s[r] = warp_sum(s[r]);
    if (lane == 0) {
      const double lam = v.w_lambda[w];
#pragma unroll
      for (int r = 0; r < 6; r++) {
        double d = 0.0;
        if (j == 0) {
          const int rr = r < c ? r : c, cc = r < c ? c : r;
          d = v.g_Hpp[21 * (size_t)g + (rr * 6 - (rr * (rr - 1)) / 2 + (cc - rr))];
          if (r == c) d += lam;
        }
        v.S_blk[36 * (size_t)blk + 6 * r + c] = d - s[r];
      }
    }
  } else {
    const int g = wi - n_blocks * 6;
    if (g >= v.n_free_total) return;
    const int w = v.kf_win[v.g_kf[g]];
    if (v.w_phase[w] == PH_DONE) return;
    double s[6] = {0, 0, 0, 0, 0, 0};
    for (int q = v.gv_off[g] + lane; q < v.gv_off[g + 1]; q += 32) {
      const double* src = v.dpart + v.gv_src[q];
#pragma unroll
      for (int r = 0; r < 6; r++) s[r] += src[r];
    }
#pragma unroll
    for (int r = 0; r < 6; r++) s[r] = warp_sum(s[r]);
    if (lane == 0)
#pragma unroll
      for (int r = 0; r < 6; r++) v.g_bs[6 * (size_t)g + r] = v.g_bp[6 * (size_t)g + r] - s[r];
  }
}

// ------------------------------------------------------------------------------------------------
// reduced camera system: dense LDL^T of one window by one CTA (lower triangle, row-major, leading dim ld)
// stands in for LinearSolverEigen / LinearSolverDense (Thirdparty/g2o/g2o/solvers/*.h); failure = zero or
// non-finite pivot.
// ------------------------------------------------------------------------------------------------
// reciprocal for the pivot chain of the small LDL^T factorisations: MUFU seed (~20 bits) + two Newton steps (<= 1 ulp),
// a third of the latency of the IEEE division sequence; zero / non-finite pivots are rejected by the caller beforehand
__device__ __forceinline__ double rcp_newton(double d) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  double e = fma(-d, r, 1.0);
  r = fma(r, e, r);
  e = fma(-d, r, 1.0);
  r = fma(r, e, r);
  return r;
}

// Blocked (6-column supernode) LDL^T of the reduced camera system by one CTA, diagonal blocks factored one pivot ahead:
//   (0) warp 0 factors diagonal block 0: lanes 0..20 hold the lower-triangle entries, lanes 21..26 the rhs block as a
//       seventh row (its elimination is the forward substitution), pivots are broadcast by shuffles;
//   per block column k:
//   (1) one thread per row below solves its 1x6 panel row  T = A_ik L_kk^-T  and  L = T D^-1  (L_kk and D^-1 in registers),
//   (2) rank-6 trailing update  A_ij -= sum_c L_ic T_jc,  b_i -= sum_c L_ic z_c : warp 0 takes the six rows of
//       diagonal block k + 1 and factors it at once (the dependent chain of the 6x6 LDL^T runs under the other warps'
//       update instead of between two barriers), the other warps take one row each;
//   backward substitution by 6-column blocks in one warp (6x6 triangle by shuffles, one shared-memory round trip per block).
// n is a multiple of 6.  tmp: >= 6 n + 32 doubles (T transposed [6][n] + {z[6], 1/D[6]} x 2).
__device__ bool ldlt_solve_cta(double* __restrict__ A, int n, int ld, double* __restrict__ b /*in: rhs, out: x*/, double* __restrict__ tmp, int* flag) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  double* Tt = tmp;          // [6][n]
  double* zb = tmp + 6 * n;  // [2][16]: z block at 0..5, 1/D at 8..13
  int li = 0, lj = lane;     // lanes 0..20: entry (li, lj), lj <= li, of a diagonal block (look-ahead update below)
  while (li < 5 && lj > li) { lj -= li + 1; li++; }
  // unblocked right-looking LDL^T of the 6x6 diagonal block at k0 with the rhs block as a seventh row (its elimination
  // is the forward substitution), in the registers of one thread: the pivot chain is reciprocal -> multiply -> fma per
  // pivot with no shuffle or shared-memory round trip in between (a lane-parallel variant measured 300 cycles / pivot)
  auto factor = [&](int k0, double* zq) -> bool {
    bool okk = true;
    if (lane == 0) {
      double M[7][6];
#pragma unroll
      for (int i = 0; i < 6; i++)
#pragma unroll
        for (int j = 0; j < 6; j++)
          if (j <= i) M[i][j] = A[(size_t)(k0 + i) * ld + k0 + j];
#pragma unroll
      for (int j = 0; j < 6; j++) M[6][j] = b[k0 + j];
      double inv[6];
#pragma unroll
      for (int pv = 0; pv < 6; pv++) {
        const double d = M[pv][pv];
        if (!(d != 0.0) || !isfinite(d)) okk = false;
        const double id = rcp_newton(d);
        inv[pv] = id;
#pragma unroll
        for (int i = 0; i < 7; i++)
          if (i > pv) {
            const double l = M[i][pv] * id;
#pragma unroll
            for (int k = 0; k < 6; k++)
              if (k > pv && k <= i) M[i][k] -= l * M[k][pv];   // T(k, pv) is still unscaled: rows are scaled after use
          }
#pragma unroll
        for (int i = 0; i < 6; i++)
          if (i > pv) M[i][pv] *= id;
      }
#pragma unroll
      for (int i = 0; i < 6; i++) {
#pragma unroll
        for (int j = 0; j < 6; j++)
          if (j <= i) A[(size_t)(k0 + i) * ld + k0 + j] = M[i][j];
        zq[8 + i] = inv[i];
        zq[i] = M[6][i];
        b[k0 + i] = M[6][i];
      }
    }
    return __shfl_sync(0xffffffffu, okk ? 1 : 0, 0) != 0;
  };
  if (tid == 0) *flag = 1;
  __syncthreads();
  if (wid == 0 && n > 0) {
    const bool okk = factor(0, zb);
    if (!okk && lane == 0) *flag = 0;
  }
  __syncthreads();
  if (!*flag) return false;
  for (int k0 = 0, kb = 0; k0 < n; k0 += 6, kb ^= 1) {
    const double* zk = zb + 16 * kb;
    // panel rows: T_i = A_i,k L_kk^-T  (forward substitution along the row), L_i = T_i D^-1
    for (int i = k0 + 6 + tid; i < n; i += nt) {
      double Lk[15], invd[6], t6[6];
#pragma unroll
      for (int c = 1; c < 6; c++)
#pragma unroll
        for (int q = 0; q < 6; q++)
          if (q < c) Lk[c * (c - 1) / 2 + q] = A[(size_t)(k0 + c) * ld + k0 + q];
#pragma unroll
      for (int c = 0; c < 6; c++) invd[c] = zk[8 + c];
      double* row = A + (size_t)i * ld + k0;
#pragma unroll
      for (int c = 0; c < 6; c++) t6[c] = row[c];
#pragma unroll
      for (int c = 1; c < 6; c++)
#pragma unroll
        for (int q = 0; q < 6; q++)
          if (q < c) t6[c] -= t6[q] * Lk[c * (c - 1) / 2 + q];
#pragma unroll
      for (int c = 0; c < 6; c++) {
        Tt[(size_t)c * n + i] = t6[c];
        row[c] = t6[c] * invd[c];
      }
    }
    __syncthreads();
    if (wid == 0) {
      // rows of diagonal block k + 1 (they end inside that block), then its factorisation
      if (k0 + 6 < n) {
        if (lane < 21) {
          const int i = k0 + 6 + li, j = k0 + 6 + lj;
          const double* row = A + (size_t)i * ld;
          double a2 = 0;
#pragma unroll
          for (int c = 0; c < 6; c++) a2 += row[k0 + c] * Tt[(size_t)c * n + j];
          A[(size_t)i * ld + j] -= a2;
        } else if (lane < 27) {
          const int i = k0 + 6 + (lane - 21);
          const double* row = A + (size_t)i * ld;
          double a2 = 0;
#pragma unroll
          for (int c = 0; c < 6; c++) a2 += row[k0 + c] * zk[c];
          b[i] -= a2;
        }
        __syncwarp();
        const bool okk = factor(k0 + 6, zb + 16 * (kb ^ 1));
        if (!okk && lane == 0) *flag = 0;
      }
    } else {
      // rank-6 trailing update of the rows below block k + 1, one warp per row
      for (int i = k0 + 12 + (wid - 1); i < n; i += nw - 1) {
        double* row = A + (size_t)i * ld;
        const double l0 = row[k0], l1 = row[k0 + 1], l2 = row[k0 + 2], l3 = row[k0 + 3], l4 = row[k0 + 4], l5 = row[k0 + 5];
        for (int j = k0 + 6 + lane; j <= i; j += 32)
          row[j] -= l0 * Tt[j] + l1 * Tt[n + j] + l2 * Tt[2 * n + j] + l3 * Tt[3 * n + j] + l4 * Tt[4 * n + j] + l5 * Tt[5 * n + j];
        if (lane == 0) b[i] -= l0 * zk[0] + l1 * zk[1] + l2 * zk[2] + l3 * zk[3] + l4 * zk[4] + l5 * zk[5];
      }
    }
    __syncthreads();
    if (!*flag) return false;
  }
  for (int i = tid; i < n; i += nt) b[i] /= A[(size_t)i * ld + i];
  __syncthreads();
  // backward: L^T x = D^-1 z by 6-column blocks, one warp
  if (wid == 0) {
    for (int k0 = n - 6; k0 >= 0; k0 -= 6) {
      // lane c < 6: x_c = z_c - sum_{q > c} L(k0 + q, k0 + c) x_q
      double z = lane < 6 ? b[k0 + lane] : 0.0;
      double Lc[5];
#pragma unroll
      for (int q = 1; q < 6; q++) Lc[q - 1] = (lane < q) ? A[(size_t)(k0 + q) * ld + k0 + lane] : 0.0;
#pragma unroll
      for (int q = 5; q >= 1; q--) {
        const double xq = __shfl_sync(0xffffffffu, z, q);
        z -= Lc[q - 1] * xq;   // lanes >= q hold Lc = 0
      }
      double x6[6];
#pragma unroll
      for (int c = 0; c < 6; c++) x6[c] = __shfl_sync(0xffffffffu, z, c);
      if (lane < 6) b[k0 + lane] = z;
      for (int i = lane; i < k0; i += 32) {
        double a2 = 0;
#pragma unroll
        for (int c = 0; c < 6; c++) a2 += A[(size_t)(k0 + c) * ld + i] * x6[c];
        b[i] -= a2;
      }
      __syncwarp();
    }
  }
  __syncthreads();
  return true;
}

// ------------------------------------------------------------------------------------------------
// envelope (skyline) LDL^T for the global-BA reduced camera system: same 6-column supernode algorithm as
// ldlt_solve_cta, restricted to the profile  first[i] <= j <= i  (no fill outside the envelope).  One CTA, matrix in
// global memory (L2 resident), panel / rhs scratch in shared memory.  Stands in for Eigen::SimplicialLDLT
// (Thirdparty/g2o/g2o/solvers/linear_solver_eigen.h:94-124).
// ------------------------------------------------------------------------------------------------
#define ENV_A(i, j) A[rowptr[i] + ((j) - first[i])]
constexpr int ENV_BS_ROWS = 32;  // rows staged per chunk in the backward substitution
__global__ void __launch_bounds__(1024) k_solve_env(BaView v) {
  extern __shared__ double esm[];
  const int w = 0;
  if (v.w_phase[w] == PH_DONE) return;
  const int g0 = v.w_g0[w], nf = v.w_g0[w + 1] - g0;
  const int n = 6 * nf;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const int ph = v.env_panel_h;
  double* Tt = esm;                    // [6][ph]
  double* zb = esm + 6 * (size_t)ph;   // [6]
  double* stage = zb + 8;              // [ENV_BS_ROWS][maxlen]
  double* b = stage + (size_t)ENV_BS_ROWS * v.env_maxlen;  // rhs / solution in shared memory, n doubles
  __shared__ int flag;
  __shared__ double red[32];
  double* A = v.env_A;
  const long long* rowptr = v.env_rowptr;
  const int* first = v.env_first;
  const int sel = v.w_sel[w];
  // assemble: zero the envelope, scatter the block rows (upper blocks (a,b) -> lower entries), rhs
  const long long nnz = rowptr[n];
  for (long long i = tid; i < nnz; i += nt) A[i] = 0.0;
  if (tid == 0) flag = 1;
  __syncthreads();
  for (int a = 0; a < nf; a++) {
    const int g = g0 + a;
    const int nb0 = v.nb_off[g], nnb = v.nb_off[g + 1] - nb0;
    for (int idx = tid; idx < nnb * 36; idx += nt) {
      const int j = idx / 36, rc = idx - 36 * j, r = rc / 6, c = rc - 6 * r;
      const int bb = v.nb_g[nb0 + j] - g0;
      if (j == 0 && c < r) continue;
      ENV_A(6 * bb + c, 6 * a + r) = v.S_blk[36 * (size_t)(nb0 + j) + rc];
    }
  }
  for (int i = tid; i < n; i += nt) b[i] = v.g_bs[6 * (size_t)g0 + i];
  __syncthreads();
  bool ok = true;
  for (int k0 = 0; k0 < n && ok; k0 += 6) {
    const int kb = k0 / 6;
    const int i_end = 6 * (v.env_blk_last[kb] + 1);
    if (tid == 0) {
      double M[6][6], zz[6];
#pragma unroll
      for (int i = 0; i < 6; i++) {
        zz[i] = b[k0 + i];
#pragma unroll
        for (int j = 0; j < 6; j++) M[i][j] = (j <= i) ? ENV_A(k0 + i, k0 + j) : 0.0;
      }
      bool okk = true;
#pragma unroll
      for (int j = 0; j < 6; j++) {
        double d = M[j][j];
#pragma unroll
        for (int q = 0; q < 6; q++)
          if (q < j) d -= M[j][q] * M[j][q] * M[q][q];
        if (!(d != 0.0) || !isfinite(d)) okk = false;
        M[j][j] = d;
        const double id = 1.0 / d;
#pragma unroll
        for (int i = 0; i < 6; i++)
          if (i > j) {
            double s2 = M[i][j];
#pragma unroll
            for (int q = 0; q < 6; q++)
              if (q < j) s2 -= M[i][q] * M[j][q] * M[q][q];
            M[i][j] = s2 * id;
          }
      }
      if (!okk) flag = 0;
      else {
#pragma unroll
        for (int i = 0; i < 6; i++)
#pragma unroll
          for (int q = 0; q < 6; q++)
            if (q < i) zz[i] -= M[i][q] * zz[q];
#pragma unroll
        for (int i = 0; i < 6; i++) {
          zb[i] = zz[i];
          b[k0 + i] = zz[i];
#pragma unroll
          for (int j = 0; j < 6; j++)
            if (j <= i) ENV_A(k0 + i, k0 + j) = M[i][j];
        }
      }
    }
    __syncthreads();
    if (!flag) { ok = false; break; }
    // panel rows
    for (int i = k0 + 6 + tid; i < i_end; i += nt) {
      double t6[6] = {0, 0, 0, 0, 0, 0};
      if (first[i] <= k0) {
        double* row = &ENV_A(i, k0);
#pragma unroll
        for (int c = 0; c < 6; c++) {
          double s2 = row[c];
#pragma unroll
          for (int q = 0; q < 6; q++)
            if (q < c) s2 -= t6[q] * ENV_A(k0 + c, k0 + q);
          t6[c] = s2;
        }
#pragma unroll
        for (int c = 0; c < 6; c++) row[c] = t6[c] / ENV_A(k0 + c, k0 + c);
      }
#pragma unroll
      for (int c = 0; c < 6; c++) Tt[(size_t)c * ph + (i - k0 - 6)] = t6[c];
    }
    __syncthreads();
    for (int i = k0 + 6 + wid; i < i_end; i += nw) {
      if (first[i] > k0) continue;
      double* row = A + rowptr[i] - first[i];
      const double l0 = row[k0], l1 = row[k0 + 1], l2 = row[k0 + 2], l3 = row[k0 + 3], l4 = row[k0 + 4], l5 = row[k0 + 5];
      const int jb = max(k0 + 6, first[i]);
      for (int j = jb + lane; j <= i; j += 32) {
        const int q = j - k0 - 6;
        row[j] -= l0 * Tt[q] + l1 * Tt[ph + q] + l2 * Tt[2 * (size_t)ph + q] + l3 * Tt[3 * (size_t)ph + q] + l4 * Tt[4 * (size_t)ph + q] +
                  l5 * Tt[5 * (size_t)ph + q];
      }
      if (lane == 0) b[i] -= l0 * zb[0] + l1 * zb[1] + l2 * zb[2] + l3 * zb[3] + l4 * zb[4] + l5 * zb[5];
    }
    __syncthreads();
  }
  if (ok) {
    for (int i = tid; i < n; i += nt) b[i] /= ENV_A(i, i);
    __syncthreads();
    // backward substitution, rows staged through shared memory in chunks (one warp does the dependent chain)
    const int ml = v.env_maxlen;
    for (int j1 = n; j1 > 0; j1 -= ENV_BS_ROWS) {
      const int j0 = max(0, j1 - ENV_BS_ROWS);
      for (int r = j0 + wid; r < j1; r += nw) {
        const int len = r - first[r];
        for (int q = lane; q < len; q += 32) stage[(size_t)(r - j0) * ml + q] = A[rowptr[r] + q];
      }
      __syncthreads();
      if (wid == 0) {
        for (int j = j1 - 1; j >= j0; j--) {
          const double xj = b[j];
          const int f = first[j], len = j - f;
          for (int q = lane; q < len; q += 32) b[f + q] -= stage[(size_t)(j - j0) * ml + q] * xj;
          __syncwarp();
        }
      }
      __syncthreads();
    }
    for (int i = tid; i < n; i += nt) v.g_x[6 * (size_t)g0 + i] = b[i];
  }
  __syncthreads();
  for (int k = v.kf_off[w] + tid; k < v.kf_off[w + 1]; k += nt) {
    const int g = v.kf_g[k];
    double qt[7];
    const double* src = v.pose_qt[sel] + 7 * (size_t)k;
    if (g >= 0 && v.g_nact[g] > 0) {
      pose_oplus(src, v.g_x + 6 * (size_t)g, qt);
    } else {
#pragma unroll
      for (int q = 0; q < 7; q++) qt[q] = src[q];
    }
    double Rt[12];
    pose_to_Rt(qt, Rt);
    double* dq = v.pose_qt[sel ^ 1] + 7 * (size_t)k;
    double* dr = v.pose_Rt[sel ^ 1] + 12 * (size_t)k;
#pragma unroll
    for (int q = 0; q < 7; q++) dq[q] = qt[q];
#pragma unroll
    for (int q = 0; q < 12; q++) dr[q] = Rt[q];
  }
  const double lam = v.w_lambda[w];
  double sc = 0;
  for (int i = tid; i < n; i += nt) {
    const int g = g0 + i / 6;
    if (v.g_nact[g] == 0) continue;
    const double x = v.g_x[6 * (size_t)g0 + i];
    sc += x * (lam * x + v.g_bp[6 * (size_t)g0 + i]);
  }
  sc = block_sum(sc, red);
  if (tid == 0) {
    v.w_scale_p[w] = sc;
    v.w_ok[w] = ok ? 1 : 0;
  }
}
#undef ENV_A

// one CTA per window: assemble the dense reduced camera system from the block rows, factor, solve, apply the
// pose update T <- exp(x) T into the trial buffer and accumulate the pose part of computeScale().
template <bool SMEM>
__global__ void __launch_bounds__(512) k_solve(BaView v) {
  extern __shared__ double smem[];
  const int w = blockIdx.x;
  if (v.w_phase[w] == PH_DONE) return;
  const int g0 = v.w_g0[w], nf = v.w_g0[w + 1] - g0;
  const int n = 6 * nf;
  const int tid = threadIdx.x, nt = blockDim.x;
  __shared__ int flag;
  __shared__ double red[32];
  double* A = SMEM ? smem : (v.solve_scratch + v.w_scratch_off[w]);
  double* rhs = SMEM ? (smem + (size_t)n * n) : (A + (size_t)n * n);
  double* tmp = rhs + n;  // 6n + 16 doubles
  const int sel = v.w_sel[w];
  bool ok = true;
  if (n > 0) {
    if (v.dense_mode) {
      // local BA: every block (a, b >= a) exists, block row a starts at nb_off[g0] + a nf - a (a - 1) / 2; nothing to
      // zero (the factorisation reads the lower triangle only)
      const int base = v.nb_off[g0], tot = 36 * (nf * (nf + 1) / 2);
      const double* Sg = v.S_blk + 36 * (size_t)base;
      // coalesced sweep, eight loads in flight per thread before the first store (A may alias S_blk for the compiler);
      // the (a, j) of a thread's elements is found incrementally (their block index only grows)
      int a = 0, off = 0;
      for (int i0 = tid; i0 < tot; i0 += 8 * nt) {
        double val[8];
        int dst[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          const int idx = i0 + u * nt;
          dst[u] = -1;
          val[u] = 0.0;
          if (idx < tot) {
            const int blk = idx / 36, rc = idx - 36 * blk, r = rc / 6, c = rc - 6 * r;
            while (off + (nf - a) <= blk) { off += nf - a; a++; }
            const int j = blk - off;
            if (!(j == 0 && c < r)) dst[u] = (6 * (a + j) + c) * n + (6 * a + r);   // diagonal block: keep one triangle
            val[u] = Sg[idx];
          }
        }
#pragma unroll
        for (int u = 0; u < 8; u++)
          if (dst[u] >= 0) A[dst[u]] = val[u];
      }
    } else {
      for (int idx = tid; idx < n * n; idx += nt) A[idx] = 0.0;
      __syncthreads();
      for (int a = 0; a < nf; a++) {
        const int g = g0 + a;
        const int nb0 = v.nb_off[g], nnb = v.nb_off[g + 1] - nb0;
        for (int idx = tid; idx < nnb * 36; idx += nt) {
          const int j = idx / 36, rc = idx - 36 * j, r = rc / 6, c = rc - 6 * r;
          const int b = v.nb_g[nb0 + j] - g0;
          if (j == 0 && c < r) continue;  // diagonal block: keep one triangle
          A[(size_t)(6 * b + c) * n + (6 * a + r)] = v.S_blk[36 * (size_t)(nb0 + j) + rc];
        }
      }
    }
    for (int i = tid; i < n; i += nt) rhs[i] = v.g_bs[6 * (size_t)g0 + i];
    __syncthreads();
    ok = ldlt_solve_cta(A, n, n, rhs, tmp, &flag);
    __syncthreads();
    if (ok)
      for (int i = tid; i < n; i += nt) v.g_x[6 * (size_t)g0 + i] = rhs[i];
    __syncthreads();
  }
  // pose update into the trial buffer; fixed / inactive keyframes are carried over unchanged
  for (int k = v.kf_off[w] + tid; k < v.kf_off[w + 1]; k += nt) {
    const int g = v.kf_g[k];
    double qt[7];
    const double* src = v.pose_qt[sel] + 7 * (size_t)k;
    if (g >= 0 && v.g_nact[g] > 0) {
      pose_oplus(src, v.g_x + 6 * (size_t)g, qt);
    } else {
#pragma unroll
      for (int q = 0; q < 7; q++) qt[q] = src[q];
    }
    double Rt[12];
    pose_to_Rt(qt, Rt);
    double* dq = v.pose_qt[sel ^ 1] + 7 * (size_t)k;
    double* dr = v.pose_Rt[sel ^ 1] + 12 * (size_t)k;
#pragma unroll
    for (int q = 0; q < 7; q++) dq[q] = qt[q];
#pragma unroll
    for (int q = 0; q < 12; q++) dr[q] = Rt[q];
  }
  // scale contribution of the poses: sum x (lambda x + b)   (computeScale, levenberg.cpp:182-189)
  const double lam = v.w_lambda[w];
  double sc = 0;
  for (int i = tid; i < n; i += nt) {
    const int g = g0 + i / 6;
    if (v.g_nact[g] == 0) continue;
    const double x = v.g_x[6 * (size_t)g0 + i];
    sc += x * (lam * x + v.g_bp[6 * (size_t)g0 + i]);
  }
  sc = block_sum(sc, red);
  if (tid == 0) {
    v.w_scale_p[w] = sc;
    v.w_ok[w] = ok ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// back-substitution + update + error at the trial state (one thread per landmark)
// ------------------------------------------------------------------------------------------------
template <int PT_G>
__global__ void __launch_bounds__(LM_TPB) k_backsub_points(BaView v) {
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int pl = gt / PT_G, gl = gt - pl * PT_G;
  const bool live = pl < v.n_pt;
  const int p = live ? pl : v.n_pt - 1;
  const int w = v.pt_win[p];
  const bool run = live && v.w_phase[w] != PH_DONE;
  if (PT_G == 1 && !run) return;
  const int sel = v.w_sel[w];
  const double* Xo = v.pt_xyz[sel] + 3 * (size_t)p;
  double* Xn = v.pt_xyz[sel ^ 1] + 3 * (size_t)p;
  const bool active = v.lm_active[p] != 0;
  const bool go = run && active;
  const double* Dp = v.dense_mode ? v.pts_D + 10 * (size_t)v.pt_spos[p] : v.pt_D + 9 * (size_t)p;
  double s3[3] = {0, 0, 0};
  const int e0 = v.pt_obs_off[p], e1 = v.pt_obs_off[p + 1];
  {
    const bool dense = v.dense_mode != 0;
    const int* epos = dense ? v.pe_wpos : v.pe_pos;
    // a gated-out edge has W = 0 and is skipped, unless W records were folded (k_fold_dup): then it may hold the sum
    const bool skip_gated = v.n_fold == 0;
    // (W slot, update block) of the edge one ahead of the arithmetic: the keyframe -> block -> x chain is three loads deep
    int e = e0 + gl, pos = -1, g = 0;
    if (e < e1 && go) {
      pos = (skip_gated && v.pe_level[e] != 0) ? -1 : epos[e];
      g = v.kf_g[v.pe_kf[e]];
    }
    while (e < e1 && go) {
      const int en = e + PT_G;
      int pos_n = -1, g_n = 0;
      if (en < e1) {
        pos_n = (skip_gated && v.pe_level[en] != 0) ? -1 : epos[en];
        g_n = v.kf_g[v.pe_kf[en]];
      }
      if (pos >= 0) {
        double Wv[18];
        if (dense) {
          const double2* wp = reinterpret_cast<const double2*>(v.pe_Wl + 18 * (size_t)pos);
#pragma unroll
          for (int k = 0; k < 9; k++) {
            const double2 t2 = wp[k];
            Wv[2 * k] = t2.x; Wv[2 * k + 1] = t2.y;
          }
        } else {
          const double* wp = v.P_rec + 27 * (size_t)pos;
#pragma unroll
          for (int k = 0; k < 18; k++) Wv[k] = wp[k];
        }
        const double2* xp2 = reinterpret_cast<const double2*>(v.g_x + 6 * (size_t)g);
        const double2 x01 = xp2[0], x23 = xp2[1], x45 = xp2[2];
        const double xp[6] = {x01.x, x01.y, x23.x, x23.y, x45.x, x45.y};
#pragma unroll
        for (int r = 0; r < 6; r++) {
          const double x = xp[r];
          s3[0] += Wv[3 * r] * x; s3[1] += Wv[3 * r + 1] * x; s3[2] += Wv[3 * r + 2] * x;
        }
      }
      e = en; pos = pos_n; g = g_n;
    }
  }
#pragma unroll
  for (int o = PT_G / 2; o > 0; o >>= 1)
#pragma unroll
    for (int k = 0; k < 3; k++) s3[k] += __shfl_xor_sync(0xffffffffu, s3[k], o);
  // xl = Dinv (bl - W^T xp) = c - Dinv (W^T xp)
  // A failed linear solve leaves the solver's x untouched and the reference still applies it (update(_solver->x()) and
  // computeScale() run before the failure is looked at, optimization_algorithm_levenberg.cpp:112-131): the landmark
  // keeps the update of its last successful solve (zero before the first one).
  double xl[3] = {0, 0, 0};
  double* xs = v.pt_xl + 3 * (size_t)p;
  if (active) {
    if (v.w_ok[w]) {
      xl[0] = Dp[6] - (Dp[0] * s3[0] + Dp[1] * s3[1] + Dp[2] * s3[2]);
      xl[1] = Dp[7] - (Dp[1] * s3[0] + Dp[3] * s3[1] + Dp[4] * s3[2]);
      xl[2] = Dp[8] - (Dp[2] * s3[0] + Dp[4] * s3[1] + Dp[5] * s3[2]);
      if (run && gl == 0) { xs[0] = xl[0]; xs[1] = xl[1]; xs[2] = xl[2]; }
    } else {
      xl[0] = xs[0]; xl[1] = xs[1]; xl[2] = xs[2];
    }
  }
  const double X[3] = {Xo[0] + xl[0], Xo[1] + xl[1], Xo[2] + xl[2]};
  double chi = 0;
  {
    int e = e0 + gl, kf = 0, lvl = 1;
    float ou = 0.f, ov = 0.f, orr = 0.f, oinfo = 0.f;
    if (e < e1 && go) {
      kf = v.pe_kf[e]; lvl = v.pe_level[e];
      ou = v.pe_uvr[3 * (size_t)e]; ov = v.pe_uvr[3 * (size_t)e + 1]; orr = v.pe_uvr[3 * (size_t)e + 2];
      oinfo = v.pe_info[e];
    }
    while (e < e1 && go) {
      const int en = e + PT_G;
      int kf_n = 0, lvl_n = 1;
      float ou_n = 0.f, ov_n = 0.f, or_n = 0.f, oinfo_n = 0.f;
      if (en < e1) {
        kf_n = v.pe_kf[en]; lvl_n = v.pe_level[en];
        ou_n = v.pe_uvr[3 * (size_t)en]; ov_n = v.pe_uvr[3 * (size_t)en + 1]; or_n = v.pe_uvr[3 * (size_t)en + 2];
        oinfo_n = v.pe_info[en];
      }
      if (lvl == 0) {
        double Rt[12];
        const double2* rp = reinterpret_cast<const double2*>(v.pose_Rt[sel ^ 1] + 12 * (size_t)kf);
#pragma unroll
        for (int k = 0; k < 6; k++) {
          const double2 t2 = rp[k];
          Rt[2 * k] = t2.x; Rt[2 * k + 1] = t2.y;
        }
        const float obs[3] = {ou, ov, orr};
        const bool stereo = !(orr < 0.f);
        double xc[3], err[3];
        map_Rt(Rt, X, xc);
        pt_residual<true>(xc, v.kf_intr + 5 * (size_t)kf, obs, stereo, err);
        const double info = (double)oinfo;
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
        v.pe_chi2[e] = c2;
        double wgt;
        chi += v.prm.robust_pt ? huber(c2, stereo ? v.prm.delta_pt_stereo : v.prm.delta_pt_mono, &wgt) : c2;
      }
      e = en; kf = kf_n; lvl = lvl_n;
      ou = ou_n; ov = ov_n; orr = or_n; oinfo = oinfo_n;
    }
  }
#pragma unroll
  for (int o = PT_G / 2; o > 0; o >>= 1) chi += __shfl_xor_sync(0xffffffffu, chi, o);
  if (!run || gl != 0) return;
  if (!active) {
    Xn[0] = Xo[0]; Xn[1] = Xo[1]; Xn[2] = Xo[2];
    v.lm_chi2[p] = 0.0;
    v.lm_scale[p] = 0.0;
    return;
  }
  Xn[0] = X[0]; Xn[1] = X[1]; Xn[2] = X[2];
  const double lam = v.w_lambda[w];
  const double* bl = v.pt_H + 9 * (size_t)p + 6;
  v.lm_scale[p] = xl[0] * (lam * xl[0] + bl[0]) + xl[1] * (lam * xl[1] + bl[1]) + xl[2] * (lam * xl[2] + bl[2]);
  v.lm_chi2[p] = chi;
}

template <int LN_G>
__global__ void __launch_bounds__(LM_TPB) k_backsub_lines(BaView v) {
  // LN_G lanes per line (as k_lin_lines): W^T x_p and the trial residuals are summed over the group in fixed order
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int l = gt / LN_G, gl = gt - l * LN_G;
  const bool live = l < v.n_ln;
  const int lc = live ? l : v.n_ln - 1;
  const int w = v.ln_win[lc];
  const bool run = live && v.w_phase[w] != PH_DONE;
  const int sel = v.w_sel[w];
  const int li = v.n_pt + lc;
  const double* so = v.ln_st[sel] + 5 * (size_t)lc;
  double* sn = v.ln_st[sel ^ 1] + 5 * (size_t)lc;
  const bool active = v.lm_active[li] != 0;
  const double* Dp = v.dense_mode ? v.lns_D + 14 * (size_t)v.ln_spos[lc] : v.ln_D + 14 * (size_t)lc;
  double s4[4] = {0, 0, 0, 0};
  const int c0 = v.ln_obs_off[lc], c1 = v.ln_obs_off[lc + 1];
  {
    const int* cpos = v.dense_mode ? v.lc_wpos : v.lc_pos;
    const bool go = run && active;
    // (W slot, update block) of the cell one ahead of the arithmetic
    int c = c0 + gl, pos = -1, g = 0;
    if (c < c1 && go) {
      pos = cpos[c];
      g = v.kf_g[v.lc_kf[c]];
    }
    while (c < c1 && go) {
      const int cn = c + LN_G;
      int pos_n = -1, g_n = 0;
      if (cn < c1) {
        pos_n = cpos[cn];
        g_n = v.kf_g[v.lc_kf[cn]];
      }
      if (pos >= 0) {
        const double2* wp = reinterpret_cast<const double2*>(v.dense_mode ? v.lc_Wl + 24 * (size_t)pos : v.L_rec + 38 * (size_t)pos);
        double W[24];
#pragma unroll
        for (int k = 0; k < 12; k++) {
          const double2 t2 = wp[k];
          W[2 * k] = t2.x; W[2 * k + 1] = t2.y;
        }
        const double2* xp2 = reinterpret_cast<const double2*>(v.g_x + 6 * (size_t)g);
        const double2 x01 = xp2[0], x23 = xp2[1], x45 = xp2[2];
        const double xp[6] = {x01.x, x01.y, x23.x, x23.y, x45.x, x45.y};
#pragma unroll
        for (int r = 0; r < 6; r++) {
          const double x = xp[r];
          s4[0] += W[4 * r] * x; s4[1] += W[4 * r + 1] * x; s4[2] += W[4 * r + 2] * x; s4[3] += W[4 * r + 3] * x;
        }
      }
      c = cn; pos = pos_n; g = g_n;
    }
  }
#pragma unroll
  for (int o = LN_G / 2; o > 0; o >>= 1)
#pragma unroll
    for (int k = 0; k < 4; k++) s4[k] += __shfl_xor_sync(0xffffffffu, s4[k], o);
  double xl[4] = {0, 0, 0, 0};
  double st[5] = {so[0], so[1], so[2], so[3], so[4]};
  if (active) {
    double* xs = v.ln_xl + 4 * (size_t)lc;
    if (v.w_ok[w]) {
#pragma unroll
      for (int r = 0; r < 4; r++) {
        double zz = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) zz += Dp[r <= k ? u4(r, k) : u4(k, r)] * s4[k];
        xl[r] = Dp[10 + r] - zz;
      }
      if (run && gl == 0) { xs[0] = xl[0]; xs[1] = xl[1]; xs[2] = xl[2]; xs[3] = xl[3]; }
    } else {   // failed linear solve: the stale update is applied, as in the reference (see k_backsub_points)
      xl[0] = xs[0]; xl[1] = xs[1]; xl[2] = xs[2]; xl[3] = xs[3];
    }
    const double st0[5] = {so[0], so[1], so[2], so[3], so[4]};
    line_oplus(st0, xl, st);
  }
  double r1[3], r2[3], X1[3], X2[3];
  line_axes(st, r1, r2);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    X1[i] = st[4] * r2[i];
    X2[i] = X1[i] + r1[i];
  }
  double chi = 0;
  for (int c = c0 + gl; c < c1 && run && active; c += LN_G) {
    const uint8_t lv0 = v.lc_level[2 * c], lv1 = v.lc_level[2 * c + 1];
    if (lv0 != 0 && lv1 != 0) continue;
    const int kf = v.lc_kf[c];
    const double* Rt = v.pose_Rt[sel ^ 1] + 12 * (size_t)kf;
    const double* cam = v.kf_lcam + 4 * (size_t)kf;
    double P1[3], P2[3];
    map_Rt(Rt, X1, P1);
    map_Rt(Rt, X2, P2);
    const double delta = v.lc_stereo[c] ? v.prm.delta_ln_stereo : v.prm.delta_ln_mono;
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
      if ((side == 0 ? lv0 : lv1) != 0) continue;
      LineObs o;
      make_line_obs(v, kf, (side == 0 ? v.lc_left : v.lc_right) + 4 * (size_t)c, o);
      double err[2];
      line_residual(P1, P2, cam[0], cam[1], cam[2], side ? -cam[3] : 0.0, o, err);
      const double info = v.lc_info[2 * (size_t)c + side];
      const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
      v.lc_chi2[2 * (size_t)c + side] = c2;
      double wgt;
      chi += v.prm.robust_ln ? huber(c2, delta, &wgt) : c2;
    }
  }
#pragma unroll
  for (int o = LN_G / 2; o > 0; o >>= 1) chi += __shfl_xor_sync(0xffffffffu, chi, o);
  if (!run || gl != 0) return;
  if (!active) {
#pragma unroll
    for (int k = 0; k < 5; k++) sn[k] = so[k];
    v.lm_chi2[li] = 0.0;
    v.lm_scale[li] = 0.0;
    return;
  }
#pragma unroll
  for (int k = 0; k < 5; k++) sn[k] = st[k];
  const double lam = v.w_lambda[w];
  const double* bl = v.ln_H + 14 * (size_t)l + 10;
  v.lm_scale[li] = xl[0] * (lam * xl[0] + bl[0]) + xl[1] * (lam * xl[1] + bl[1]) + xl[2] * (lam * xl[2] + bl[2]) +
                   xl[3] * (lam * xl[3] + bl[3]);
  v.lm_chi2[li] = chi;
}

__global__ void __launch_bounds__(256) k_reduce_trial(BaView v) {
  const int w = blockIdx.x / v.n_slices, sl = blockIdx.x % v.n_slices;
  if (v.w_phase[w] == PH_DONE) return;
  __shared__ double sm[32];
  double chi = 0, sc = 0;
  const int np = v.pt_off[w + 1] - v.pt_off[w], nl = v.ln_off[w + 1] - v.ln_off[w];
  const int p0 = v.pt_off[w] + (int)((long long)np * sl / v.n_slices), p1 = v.pt_off[w] + (int)((long long)np * (sl + 1) / v.n_slices);
  const int l0 = v.ln_off[w] + (int)((long long)nl * sl / v.n_slices), l1 = v.ln_off[w] + (int)((long long)nl * (sl + 1) / v.n_slices);
  for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    chi += v.lm_chi2[p];
    sc += v.lm_scale[p];
  }
  for (int l = l0 + threadIdx.x; l < l1; l += blockDim.x) {
    chi += v.lm_chi2[v.n_pt + l];
    sc += v.lm_scale[v.n_pt + l];
  }
  chi = block_sum(chi, sm);
  sc = block_sum(sc, sm);
  if (threadIdx.x == 0) {
    double* o = v.w_part + 4 * (size_t)blockIdx.x;
    o[0] = chi; o[1] = sc;
  }
}
__global__ void k_sum_trial(BaView v) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= v.n_win || v.w_phase[w] == PH_DONE) return;
  double chi = 0, sc = 0;
  for (int s2 = 0; s2 < v.n_slices; s2++) {
    const double* o = v.w_part + 4 * ((size_t)w * v.n_slices + s2);
    chi += o[0]; sc += o[1];
  }
  v.w_red_sum[4 * w + 0] = chi;
  v.w_red_sum[4 * w + 1] = sc;
}

// accept / reject and the outer-iteration bookkeeping (optimization_algorithm_levenberg.cpp:99-164,
// sparse_optimizer.cpp:376-418)
__device__ __forceinline__ void decide_window(const BaView& v, int w, int round, int stop_now) {
  double tempChi = v.w_red_sum[4 * w + 0];
  if (!v.w_ok[w]) tempChi = DBL_MAX;
  const double cur = v.w_curchi[w];
  double rho = cur - tempChi;
  double scale = v.w_scale_p[w] + v.w_red_sum[4 * w + 1];
  scale += 1e-3;
  rho /= scale;
  double lam = v.w_lambda[w], ni = v.w_ni[w];
  double newcur = cur;
  if (rho > 0 && isfinite(tempChi)) {
    double alpha = 1. - pow((2 * rho - 1), 3);
    alpha = fmin(alpha, 2. / 3.);
    const double sf = fmax(1. / 3., alpha);
    lam *= sf;
    ni = 2;
    newcur = tempChi;
    v.w_sel[w] ^= 1;  // the trial buffer becomes the estimate (discardTop)
  } else {
    lam *= ni;
    ni *= 2;  // pop(): the estimate buffer is untouched
  }
  v.w_lambda[w] = lam;
  v.w_ni[w] = ni;
  v.w_curchi[w] = newcur;
  const int q = v.w_trials[w] + 1;
  v.w_trials[w] = q;
  if (rho < 0 && q < 10 && !stop_now) {
    v.w_phase[w] = PH_RETRY;
    return;
  }
  // end of this outer iteration
  const int n = v.w_nlog[w];
  if (n < v.log_stride) {
    v.chi2_log[(size_t)w * v.log_stride + n] = newcur;
    v.lambda_log[(size_t)w * v.log_stride + n - 1 - round] = lam;
    v.trials_log[(size_t)w * v.log_stride + n - 1 - round] = q;
  }
  v.w_nlog[w] = n + 1;
  const int it = v.w_iter[w] + 1;
  v.w_iter[w] = it;
  v.iter_done[2 * w + round] = it;
  bool term = (q == 10 || rho == 0);
  if (!term) {
    const double ini = v.w_inichi[w];
    int nb = v.w_nbad[w];
    if ((ini - newcur) * 1e3 < ini) nb++;
    else nb = 0;
    v.w_nbad[w] = nb;
    if (nb >= 3) term = true;
  }
  if (term || it >= v.w_maxit[w] || stop_now) {
    v.w_phase[w] = PH_DONE;
    atomicSub(v.n_active_win, 1);
  } else {
    v.w_phase[w] = PH_LIN;
  }
}

__global__ void k_decide(BaView v, int round, int stop_now) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= v.n_win) return;
  if (v.w_phase[w] == PH_DONE) return;
  decide_window(v, w, round, stop_now);
}

// single-rank fast path: trial reduction + decision in one CTA per window
__global__ void __launch_bounds__(FUSED_RED_TPB) k_decide_fused(BaView v, int round, int stop_now) {
  const int w = blockIdx.x;
  if (v.w_phase[w] == PH_DONE) return;
  __shared__ double sm[32];
  const int tid = threadIdx.x;
  double chi = 0, sc = 0;
  {
    const int p1 = v.pt_off[w + 1];
    int p = v.pt_off[w] + tid;
    for (; p + 3 * FUSED_RED_TPB < p1; p += 4 * FUSED_RED_TPB) {
      const double c0 = v.lm_chi2[p], c1 = v.lm_chi2[p + FUSED_RED_TPB], c2 = v.lm_chi2[p + 2 * FUSED_RED_TPB],
                   c3 = v.lm_chi2[p + 3 * FUSED_RED_TPB];
      const double s0 = v.lm_scale[p], s1 = v.lm_scale[p + FUSED_RED_TPB], s2 = v.lm_scale[p + 2 * FUSED_RED_TPB],
                   s3 = v.lm_scale[p + 3 * FUSED_RED_TPB];
      chi += c0; chi += c1; chi += c2; chi += c3;
      sc += s0; sc += s1; sc += s2; sc += s3;
    }
    for (; p < p1; p += FUSED_RED_TPB) {
      chi += v.lm_chi2[p];
      sc += v.lm_scale[p];
    }
  }
  for (int l = v.ln_off[w] + tid; l < v.ln_off[w + 1]; l += blockDim.x) {
    chi += v.lm_chi2[v.n_pt + l];
    sc += v.lm_scale[v.n_pt + l];
  }
  chi = block_sum(chi, sm);
  sc = block_sum(sc, sm);
  if (tid == 0) {
    v.w_red_sum[4 * w + 0] = chi;
    v.w_red_sum[4 * w + 1] = sc;
    decide_window(v, w, round, stop_now);
  }
}

// trial reduction + decision of the lean step: a window that starts a new outer iteration (PH_LIN) carries its chi2 over
// from the accepted trial of the previous step — the same state, so activeRobustChi2() of
// optimization_algorithm_levenberg.cpp:75 would return the same sum — instead of reducing it again.
__global__ void __launch_bounds__(FUSED_RED_TPB) k_decide_carry(BaView v, int round, int stop_now) {
  const int w = blockIdx.x;
  if (v.w_phase[w] == PH_DONE) return;
  __shared__ double sm[32];
  const int tid = threadIdx.x;
  double chi = 0, sc = 0;
  for (int p = v.pt_off[w] + tid; p < v.pt_off[w + 1]; p += FUSED_RED_TPB) {
    chi += v.lm_chi2[p];
    sc += v.lm_scale[p];
  }
  for (int l = v.ln_off[w] + tid; l < v.ln_off[w + 1]; l += FUSED_RED_TPB) {
    chi += v.lm_chi2[v.n_pt + l];
    sc += v.lm_scale[v.n_pt + l];
  }
  chi = block_sum(chi, sm);
  sc = block_sum(sc, sm);
  if (tid == 0) {
    if (v.w_phase[w] == PH_LIN) {   // solve() entry of a new outer iteration
      v.w_inichi[w] = v.w_curchi[w];
      v.w_trials[w] = 0;
    }
    v.w_red_sum[4 * w + 0] = chi;
    v.w_red_sum[4 * w + 1] = sc;
    decide_window(v, w, round, stop_now);
  }
}

// ------------------------------------------------------------------------------------------------
// outlier gating between the two rounds of LocalBundleAdjustment and final classification
// ------------------------------------------------------------------------------------------------
// src/Optimizer.cc:1239-1267 : chi2 of the LAST computed error (stale semantics) and depth at the current estimate
__global__ void k_flag_points(BaView v, uint8_t* bad_out /*nullptr: gate (set level); else: final flags*/) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= v.n_pe) return;
  const int p = v.pe_pt[e];
  const int w = v.pt_win[p];
  const int sel = v.w_sel[w];
  const float* obs = v.pe_uvr + 3 * (size_t)e;
  const bool stereo = !(obs[2] < 0.f);
  const double th = stereo ? v.prm.chi2_pt_stereo : v.prm.chi2_pt_mono;
  double xc[3];
  map_Rt(v.pose_Rt[sel] + 12 * (size_t)v.pe_kf[e], v.pt_xyz[sel] + 3 * (size_t)p, xc);
  const bool bad = (v.pe_chi2[e] > th) || !(xc[2] > 0.0);
  if (bad_out) bad_out[e] = bad ? 1 : 0;
  else if (bad) v.pe_level[e] = 1;
}

__device__ __forceinline__ bool line_edge_depth_ok(const BaView& v, int sel, int kf, const double* X1, const double* X2,
                                                   int side, const LineObs& o) {
  const double* Rt = v.pose_Rt[sel] + 12 * (size_t)kf;
  const double* cam = v.kf_lcam + 4 * (size_t)kf;
  double P1[3], P2[3];
  map_Rt(Rt, X1, P1);
  map_Rt(Rt, X2, P2);
  const double bx = side ? -cam[3] : 0.0;
  const double X0c[3] = {P1[0] + bx, P1[1], P1[2]};
  const double ldc[3] = {P2[0] - P1[0], P2[1] - P1[1], P2[2] - P1[2]};
  return line_depth_positive(X0c, ldc, cam[0], cam[1], cam[2], o.x1, o.x2);
}

// LineOptimizer::DisableOutliers  src/LineOptimizer.cc:129-170 (one thread per line)
__global__ void k_flag_lines(BaView v) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= v.n_ln) return;
  const int w = v.ln_win[l];
  const int sel = v.w_sel[w];
  const double* stp = v.ln_st[sel] + 5 * (size_t)l;
  const double st[5] = {stp[0], stp[1], stp[2], stp[3], stp[4]};
  double r1[3], r2[3], X1[3], X2[3];
  line_axes(st, r1, r2);
  for (int i = 0; i < 3; i++) {
    X1[i] = st[4] * r2[i];
    X2[i] = X1[i] + r1[i];
  }
  int cnt = 0, nedge = 0;
  for (int c = v.ln_obs_off[l]; c < v.ln_obs_off[l + 1]; c++) {
    const int kf = v.lc_kf[c];
    const double d = v.lc_stereo[c] ? v.prm.delta_ln_stereo : v.prm.delta_ln_mono;
    const double thr = d * d;
    for (int side = 0; side < 2; side++) {
      if (v.lc_level[2 * c + side] == 2) continue;
      nedge++;
      LineObs o;
      make_line_obs(v, kf, (side == 0 ? v.lc_left : v.lc_right) + 4 * (size_t)c, o);
      const bool dp = line_edge_depth_ok(v, sel, kf, X1, X2, side, o);
      if (v.lc_chi2[2 * (size_t)c + side] > thr || !dp) v.lc_level[2 * c + side] = 1;
      else cnt += 2;
    }
  }
  if (nedge > 0 && cnt <= v.prm.ln_filter) v.ln_removed[l] = 1;
}

// LineOptimizer::GetLineData  src/LineOptimizer.cc:172-201 : depth first, then the error recomputed at the final state
__global__ void k_final_lines(BaView v, uint8_t* bad_out /*[n_lc][2]*/) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= v.n_ln) return;
  const int w = v.ln_win[l];
  const int sel = v.w_sel[w];
  const bool removed = v.ln_removed[l] != 0;
  const double* stp = v.ln_st[sel] + 5 * (size_t)l;
  const double st[5] = {stp[0], stp[1], stp[2], stp[3], stp[4]};
  double r1[3], r2[3], X1[3], X2[3];
  line_axes(st, r1, r2);
  for (int i = 0; i < 3; i++) {
    X1[i] = st[4] * r2[i];
    X2[i] = X1[i] + r1[i];
  }
  for (int c = v.ln_obs_off[l]; c < v.ln_obs_off[l + 1]; c++) {
    const int kf = v.lc_kf[c];
    const double d = v.lc_stereo[c] ? v.prm.delta_ln_stereo : v.prm.delta_ln_mono;
    const double thr = d * d;
    for (int side = 0; side < 2; side++) {
      uint8_t bad = 0;
      if (!removed && v.lc_level[2 * c + side] != 2) {
        LineObs o;
        make_line_obs(v, kf, (side == 0 ? v.lc_left : v.lc_right) + 4 * (size_t)c, o);
        const bool dp = line_edge_depth_ok(v, sel, kf, X1, X2, side, o);
        const double* Rt = v.pose_Rt[sel] + 12 * (size_t)kf;
        const double* cam = v.kf_lcam + 4 * (size_t)kf;
        double P1[3], P2[3], err[2];
        map_Rt(Rt, X1, P1);
        map_Rt(Rt, X2, P2);
        line_residual(P1, P2, cam[0], cam[1], cam[2], side ? -cam[3] : 0.0, o, err);
        const double info = v.lc_info[2 * (size_t)c + side];
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
        bad = (c2 > thr || !dp) ? 1 : 0;
      }
      bad_out[2 * (size_t)c + side] = bad;
    }
  }
}

// gather the selected state buffers into the output layout
__global__ void k_export(BaView v, double* kf_Tcw, double* pt_xyz, double* ln_x0_dir, const double* ln_x0_dir_in) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < v.n_kf) {
    const int sel = v.w_sel[v.kf_win[i]];
    for (int k = 0; k < 12; k++) kf_Tcw[12 * (size_t)i + k] = v.pose_Rt[sel][12 * (size_t)i + k];
  }
  if (i < v.n_pt) {
    const int sel = v.w_sel[v.pt_win[i]];
    for (int k = 0; k < 3; k++) pt_xyz[3 * (size_t)i + k] = v.pt_xyz[sel][3 * (size_t)i + k];
  }
  if (i < v.n_ln) {
    const int sel = v.w_sel[v.ln_win[i]];
    if (v.ln_removed[i]) {
      for (int k = 0; k < 6; k++) ln_x0_dir[6 * (size_t)i + k] = ln_x0_dir_in[6 * (size_t)i + k];
    } else {
      const double* stp = v.ln_st[sel] + 5 * (size_t)i;
      const double st[5] = {stp[0], stp[1], stp[2], stp[3], stp[4]};
      double r1[3], r2[3];
      line_axes(st, r1, r2);
      for (int k = 0; k < 3; k++) {
        ln_x0_dir[6 * (size_t)i + k] = st[4] * r2[k];
        ln_x0_dir[6 * (size_t)i + 3 + k] = r1[k];
      }
    }
  }
}

}  // namespace lld
