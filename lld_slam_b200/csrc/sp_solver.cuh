// sp_solver.cuh — block elimination of the global-BA reduced camera system over a general super-block graph.
//
// Cyclic reduction (cr_solver.cuh) needs a block-tridiagonal system: every landmark spans at most mb free keyframes.  After
// a loop closure some landmarks are seen by keyframes at both ends of the map, and those blocks become extra edges of the
// super-block graph (a ring instead of a chain, plus chords).  The host builds a symbolic plan from the block pattern alone
// (ba.cu, sp_plan_build): elimination levels of independent super-blocks, chosen by ascending degree; one m x m slot per
// block (I, J), I <= J, fill included; the offsets of Z_i = D_i^-1 [U_ij ...] and, per output block, the ordered list of
// Schur contributions.  Each level then runs
//   k_sp_factor : CTA per eliminated node : LDL^T of D_i (ldlt_solve_cta), zc_i = D_i^-1 b_i
//   k_sp_solve  : CTA per (node, 64 of its m deg right-hand-side columns) : Z_i (cr_subst_cols)
//   k_sp_update : CTA per 64x64 tile of an output block, or per right-hand side : W_jk -= sum_i U_ij^T Z_ik, b_j -= U_ij^T zc_i
// in the plan's fixed order (no atomics: bit-reproducible).  Updating in place is safe: the nodes of one level are
// independent, so a level never writes a block that it reads.  The back-substitution x_i = zc_i - sum_j Z_ij x_j runs the
// levels in reverse.  A zero / non-finite pivot clears *ok and the LM trial is rejected, as in cyclic reduction.
#pragma once
#include "cr_solver.cuh"

namespace lld {

struct SpView {
  int N;                 // super-blocks
  int m;                 // scalars per super-block (6 * mb)
  int mb;                // keyframe blocks per super-block
  double* W;             // [n_slot][m][m]: slot I < N = diagonal block of node I, then the off-diagonal blocks (I < J)
  double* b;             // [N][m]
  double* L;             // [N][m][m] factor of each node: strict lower = L, diagonal = D
  double* Z;             // eliminated node at position p: [m][m deg_p] at z_off[p]
  double* zc;            // [N][m] D^-1 b
  double* x;             // [N][m] solution
  int* ok;               // [1]
  const int* q_slot;     // [n_blocks]: slot of the keyframe block nb_g[q] (assembly)
  const int* el_node;    // [N] node eliminated at position p (level by level)
  const int* el_nb_off;  // [N + 1] neighbour list of position p in nb_node / nb_slot2
  const long long* z_off;// [N]
  const int* nb_node;    // neighbour j (ascending within a list)
  const int* nb_slot2;   // 2 slot(i, j) + (1 when the block is stored as (j, i), i.e. j < i)
  const int* up_out;     // update item: output slot (block items) or node j (right-hand-side items)
  const int* up_c_off;   // [n_items + 1] its contributions
  const int* c_slot2;    // contribution: 2 slot(i, j) + transposed, as nb_slot2
  const int* c_pos;      // position p of the eliminated node i
  const int* c_col;      // index of k in the neighbour list of i (block items)
};

// y <- L^-T D^-1 L^-1 y for the CR_TC columns of one CTA, the substitution of k_cr_solve (kept as a copy there, so that
// the cyclic-reduction kernels compile to the same code): thread (column pair c, row group rg) holds rows
// [rg RPT, (rg+1) RPT) of columns c and c + CR_TC / 2 in y; block forward / backward substitution with the L block row /
// column read from shared memory (broadcast reads; one load feeds two FMAs), two barriers per block step.  Every thread
// of the CTA calls it.
template <int RPT>
__device__ __forceinline__ void cr_subst_cols(const double* Ls, double* yp, int m, int c, int rg, double (&y)[2][RPT]) {
  constexpr int HC = CR_TC / 2;
  const int r0 = rg * RPT;
  const int ngrp = (m + RPT - 1) / RPT;
  // forward: L y = r
  for (int g = 0; g < ngrp; g++) {
    if (rg == g) {
#pragma unroll
      for (int k = 0; k < RPT; k++) {
        if (r0 + k < m) {
          double a0 = y[0][k], a1 = y[1][k];
#pragma unroll
          for (int q = 0; q < RPT; q++)
            if (q < k) {
              const double l = Ls[(size_t)(r0 + k) * m + r0 + q];
              a0 -= l * y[0][q]; a1 -= l * y[1][q];
            }
          y[0][k] = a0; y[1][k] = a1;
          yp[k * CR_TC + c] = a0; yp[k * CR_TC + c + HC] = a1;
        }
      }
    }
    __syncthreads();
    if (rg > g && rg < ngrp) {
      const int q0 = g * RPT;
#pragma unroll
      for (int q = 0; q < RPT; q++) {
        if (q0 + q < m) {
          const double y0 = yp[q * CR_TC + c], y1 = yp[q * CR_TC + c + HC];
#pragma unroll
          for (int k = 0; k < RPT; k++)
            if (r0 + k < m) {
              const double l = Ls[(size_t)(r0 + k) * m + q0 + q];
              y[0][k] -= l * y0; y[1][k] -= l * y1;
            }
        }
      }
    }
    __syncthreads();
  }
  // diagonal
#pragma unroll
  for (int k = 0; k < RPT; k++)
    if (r0 + k < m) {
      const double id = 1.0 / Ls[(size_t)(r0 + k) * m + r0 + k];
      y[0][k] *= id; y[1][k] *= id;
    }
  // backward: L^T x = y
  for (int g = ngrp - 1; g >= 0; g--) {
    if (rg == g) {
#pragma unroll
      for (int k = RPT - 1; k >= 0; k--) {
        if (r0 + k < m) {
          double a0 = y[0][k], a1 = y[1][k];
#pragma unroll
          for (int q = 0; q < RPT; q++)
            if (q > k && r0 + q < m) {
              const double l = Ls[(size_t)(r0 + q) * m + r0 + k];
              a0 -= l * y[0][q]; a1 -= l * y[1][q];
            }
          y[0][k] = a0; y[1][k] = a1;
          yp[k * CR_TC + c] = a0; yp[k * CR_TC + c + HC] = a1;
        }
      }
    }
    __syncthreads();
    if (rg < g) {
      const int q0 = g * RPT;
#pragma unroll
      for (int q = 0; q < RPT; q++) {
        if (q0 + q < m) {
          const double x0 = yp[q * CR_TC + c], x1 = yp[q * CR_TC + c + HC];
#pragma unroll
          for (int k = 0; k < RPT; k++)
            if (r0 + k < m) {
              const double l = Ls[(size_t)(q0 + q) * m + r0 + k];
              y[0][k] -= l * x0; y[1][k] -= l * x1;
            }
        }
      }
    }
    __syncthreads();
  }
}

// scatter the upper keyframe blocks of S and b_schur into the slots (zeroed beforehand); padding rows of the last
// super-block get a unit diagonal
__global__ void __launch_bounds__(256) k_sp_assemble(BaView v, SpView sp, int n_blocks) {
  if (v.w_phase[0] == PH_DONE) return;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int g0 = v.w_g0[0], nf = v.w_g0[1] - g0;
  const int m = sp.m, mb = sp.mb;
  const size_t mm = (size_t)m * m;
  if (t == 0) *sp.ok = 1;
  if (t < n_blocks * 36) {
    const int q = t / 36, e = t - 36 * q, r = e / 6, c = e - 6 * r;
    int lo = 0, hi = v.n_free_total;   // owning block row: largest g with nb_off[g] <= q
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (v.nb_off[mid] <= q) lo = mid;
      else hi = mid;
    }
    const int a = lo - g0, h = v.nb_g[q] - g0;   // block (a, h), h >= a
    const double val = v.S_blk[36 * (size_t)q + e];
    const int I = a / mb, J = h / mb;
    const int ra = (a - I * mb) * 6 + r, ch = (h - J * mb) * 6 + c;
    double* Wb = sp.W + (size_t)sp.q_slot[q] * mm;
    if (I == J) {
      if (a == h) {
        if (c >= r) { Wb[(size_t)ra * m + ch] = val; Wb[(size_t)ch * m + ra] = val; }
      } else {
        Wb[(size_t)ra * m + ch] = val;
        Wb[(size_t)ch * m + ra] = val;
      }
    } else {
      Wb[(size_t)ra * m + ch] = val;
    }
  } else {
    const int i = t - n_blocks * 36;
    if (i < sp.N * m) {
      double bv = 0.0;
      if (i < 6 * nf) bv = v.g_bs[6 * (size_t)g0 + i];
      else sp.W[(size_t)(i / m) * mm + (size_t)(i % m) * m + (i % m)] = 1.0;
      sp.b[i] = bv;
    }
  }
}

// eliminated node at position p0 + blockIdx.x: LDL^T of D_i, zc_i = D_i^-1 b_i
__global__ void __launch_bounds__(512) k_sp_factor(BaView v, SpView sp, int p0) {
  if (v.w_phase[0] == PH_DONE) return;
  extern __shared__ double crsm[];
  __shared__ int flag;
  const int m = sp.m, tid = threadIdx.x, nt = blockDim.x;
  const int i = sp.el_node[p0 + blockIdx.x];
  if (!*sp.ok) return;
  double* A = crsm;
  double* rhs = A + (size_t)m * m;
  double* tmp = rhs + m;
  const double* Dg = sp.W + (size_t)i * m * m;
  for (int k = tid; k < m * m; k += nt) A[k] = Dg[k];
  for (int k = tid; k < m; k += nt) rhs[k] = sp.b[(size_t)i * m + k];
  __syncthreads();
  const bool ok = ldlt_solve_cta(A, m, m, rhs, tmp, &flag);
  __syncthreads();
  if (!ok) {
    if (tid == 0) *sp.ok = 0;
    return;
  }
  double* Lg = sp.L + (size_t)i * m * m;
  for (int k = tid; k < m * m; k += nt) Lg[k] = A[k];
  for (int k = tid; k < m; k += nt) sp.zc[(size_t)i * m + k] = rhs[k];
}

// Z_i = D_i^-1 [U_ij ...] for the nodes at positions [p0, p0 + gridDim.x / ntile); CTA = (node, tile of CR_TC columns),
// ntile = tiles of the level's widest node (CTAs past a node's own m deg columns return at once).  Column block a holds
// U_ij for j = the a-th neighbour, read transposed when the block is stored as (j, i).
template <int RPT>
__global__ void __launch_bounds__(CR_TC / 2 * CR_RG) k_sp_solve(BaView v, SpView sp, int p0, int ntile) {
  if (v.w_phase[0] == PH_DONE) return;
  extern __shared__ double crsm[];
  const int m = sp.m, tid = threadIdx.x;
  const int pos = p0 + blockIdx.x / ntile, tile = blockIdx.x % ntile;
  const int nb0 = sp.el_nb_off[pos], ncol = m * (sp.el_nb_off[pos + 1] - nb0);
  if (tile * CR_TC >= ncol || !*sp.ok) return;
  const int i = sp.el_node[pos];
  const size_t mm = (size_t)m * m;
  constexpr int HC = CR_TC / 2;
  double* Ls = crsm;                     // [m][m]
  double* yp = Ls + mm;                  // [RPT][CR_TC] published block
  {
    const double2* Lg = reinterpret_cast<const double2*>(sp.L + (size_t)i * mm);
    double2* L2 = reinterpret_cast<double2*>(Ls);
    for (int k = tid; k < m * m / 2; k += blockDim.x) L2[k] = Lg[k];   // m is even
  }
  const int c = tid % HC, rg = tid / HC;
  const int r0 = rg * RPT;
  double y[2][RPT];
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int col = tile * CR_TC + c + h * HC;
    const int a = col / m, cc = col - a * m;
    const int s2 = col < ncol ? sp.nb_slot2[nb0 + a] : 0;
    const double* U = sp.W + (size_t)(s2 >> 1) * mm;
#pragma unroll
    for (int k = 0; k < RPT; k++) {
      const int r = r0 + k;
      double val = 0.0;
      if (col < ncol && r < m) val = (s2 & 1) ? U[(size_t)cc * m + r] : U[(size_t)r * m + cc];
      y[h][k] = val;
    }
  }
  __syncthreads();
  cr_subst_cols<RPT>(Ls, yp, m, c, rg, y);
  double* Zg = sp.Z + sp.z_off[pos];
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int col = tile * CR_TC + c + h * HC;
    if (col < ncol)
#pragma unroll
      for (int k = 0; k < RPT; k++)
        if (r0 + k < m) Zg[(size_t)(r0 + k) * ncol + col] = y[h][k];
  }
}

// update items [u0, u0 + n_blk) are output blocks (T x T tiles each), [u0 + n_blk, u0 + n_blk + n_rhs) right-hand sides;
// each sums its contribution list in plan order, then subtracts the sum
__global__ void __launch_bounds__(256) k_sp_update(BaView v, SpView sp, int u0, int n_blk) {
  if (v.w_phase[0] == PH_DONE) return;
  if (!*sp.ok) return;
  __shared__ double As[CR_KC][CR_TILE + 4];
  __shared__ double Bs[CR_KC][CR_TILE + 4];
  const int m = sp.m;
  const size_t mm = (size_t)m * m;
  const int T = (m + CR_TILE - 1) / CR_TILE;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  if ((int)blockIdx.x >= n_blk * T * T) {   // b_j -= sum_i U_ij^T zc_i
    const int it = u0 + n_blk + (int)blockIdx.x - n_blk * T * T;
    const int j = sp.up_out[it];
    for (int r = tid; r < m; r += 256) {
      double acc = 0.0;
      for (int q = sp.up_c_off[it]; q < sp.up_c_off[it + 1]; q++) {
        const int s2 = sp.c_slot2[q];
        const double* U = sp.W + (size_t)(s2 >> 1) * mm;
        const double* z = sp.zc + (size_t)sp.el_node[sp.c_pos[q]] * m;
        double a = 0.0;
        if (s2 & 1) for (int k = 0; k < m; k++) a += U[(size_t)r * m + k] * z[k];
        else for (int k = 0; k < m; k++) a += U[(size_t)k * m + r] * z[k];
        acc += a;
      }
      sp.b[(size_t)j * m + r] -= acc;
    }
    return;
  }
  const int it = u0 + (int)blockIdx.x / (T * T), tl = (int)blockIdx.x % (T * T);
  const int r0 = (tl / T) * CR_TILE, c0 = (tl % T) * CR_TILE;
  double acc[4][4];
#pragma unroll
  for (int u = 0; u < 4; u++)
#pragma unroll
    for (int w2 = 0; w2 < 4; w2++) acc[u][w2] = 0.0;
  for (int q = sp.up_c_off[it]; q < sp.up_c_off[it + 1]; q++) {   // U_ij^T Z_ik : A(k, r) = U_ij[k][r], B(k, c) = Z_ik[k][c]
    const int s2 = sp.c_slot2[q], pos = sp.c_pos[q];
    const int zs = m * (sp.el_nb_off[pos + 1] - sp.el_nb_off[pos]);
    const double* U = sp.W + (size_t)(s2 >> 1) * mm;
    const double* Zk = sp.Z + sp.z_off[pos] + (size_t)sp.c_col[q] * m;
    if (s2 & 1) cr_tile_product<true>(U, m, Zk, zs, m, r0, c0, As, Bs, acc);
    else cr_tile_product<false>(U, m, Zk, zs, m, r0, c0, As, Bs, acc);
  }
  double* Wo = sp.W + (size_t)sp.up_out[it] * mm;
#pragma unroll
  for (int u = 0; u < 4; u++)
#pragma unroll
    for (int w2 = 0; w2 < 4; w2++) {
      const int r = r0 + ty + 16 * u, c = c0 + tx + 16 * w2;
      if (r < m && c < m) Wo[(size_t)r * m + c] -= acc[u][w2];
    }
}

// back-substitution of the nodes at positions [p0, p0 + gridDim.x / per): x_i = zc_i - sum_a Z_i,a x_(nb a); one warp
// per row
__global__ void __launch_bounds__(256) k_sp_backsub(BaView v, SpView sp, int p0) {
  if (v.w_phase[0] == PH_DONE) return;
  if (!*sp.ok) return;
  const int m = sp.m;
  const int rows_per_cta = 8;
  const int per = (m + rows_per_cta - 1) / rows_per_cta;
  const int pos = p0 + (int)blockIdx.x / per, chunk = (int)blockIdx.x % per;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int r = chunk * rows_per_cta + wid;
  if (r >= m) return;
  const int i = sp.el_node[pos], nb0 = sp.el_nb_off[pos], deg = sp.el_nb_off[pos + 1] - nb0;
  const double* Zr = sp.Z + sp.z_off[pos] + (size_t)r * m * deg;
  double acc = 0.0;
  for (int a = 0; a < deg; a++) {
    const double* xj = sp.x + (size_t)sp.nb_node[nb0 + a] * m;
    for (int k = lane; k < m; k += 32) acc += Zr[(size_t)a * m + k] * xj[k];
  }
  acc = warp_sum(acc);
  if (lane == 0) sp.x[(size_t)i * m + r] = sp.zc[(size_t)i * m + r] - acc;
}

}  // namespace lld
