// sim3.cu — batched loop-candidate Sim3 optimisation (Optimizer::OptimizeSim3, src/Optimizer.cc:1656-1858).
//
// One CTA per loop candidate runs the whole schedule of the reference on the device: optimize(5), the chi2 test that drops
// correspondences, the early return below 10 survivors, optimize(10 | 5) and the final test.  The graph is one
// VertexSim3Expmap and two edges per correspondence (EdgeSim3ProjectXYZ e12, EdgeInverseSim3ProjectXYZ e21) whose point
// vertices are fixed, so the normal equations are a dense 7x7.  The edges have no analytic Jacobian in the reference: g2o
// differentiates them numerically (BaseBinaryEdge::linearizeOplus, central differences at delta = 1e-9).  The 14 perturbed
// states do not depend on the edge, so they are formed once per LM iteration in shared memory (with their inverses for
// e21); every thread then evaluates its correspondences at the current state and at the 14 perturbed ones.  H (28 unique
// entries), b (7) and the robust chi2 are reduced in fixed order, thread 0 solves the 7x7 LDL^T with the isPositive gate
// and forms the trial state, and every thread runs the same LM bookkeeping (optimization_algorithm_levenberg.cpp) on the
// reduced values.  Edge records are staged in shared memory when the batch's largest problem fits.
// Compiled with --fmad=false: the numeric Jacobian divides differences of nearly equal errors by 2e-9, so the errors are
// evaluated in the source's operation order without contraction.
#include <algorithm>
#include <cfloat>

#include "lld_ctx.h"
#include "lld_math.cuh"

using namespace lld;

namespace {

constexpr int STPB = 128;
constexpr int NW = STPB / 32;
constexpr int NACC = 28 + 7 + 1;     // upper H, b, robust chi2
constexpr int EDGE_BYTES = 48;       // p1c, p2c (3 f32), obs1, obs2 (2 f32), info1, info2 (f32)
constexpr size_t SMEM_LIMIT = 200 * 1024;

struct Sim3View {
  int n;
  const double* S12;
  const double* cam;
  const int* fix_scale;
  const float* th2;
  const int* off;
  const float* p1c;
  const float* p2c;
  const float* obs1;
  const float* obs2;
  const float* info1;
  const float* info2;
  int its1, its_bad, its_clean;
  double* chi2;        // scratch [m][2]: stale chi2 of e12 / e21 (the error of the last evaluation, as g2o keeps it)
  double* out_S12;
  uint8_t* inlier;     // doubles as the edge level: 1 = in the graph
  int* n_in;
  int log_stride;
  double* chi2_log;
  double* lambda_log;
  int* trials_log;
  int* n_iter_done;
};

struct Edges {
  const float *p1c, *p2c, *obs1, *obs2, *info1, *info2;
};

template <int NV>
__device__ __forceinline__ void block_reduce(double* acc, double (*part)[NV], double* out) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) part[wid][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = 0;
#pragma unroll
    for (int w = 0; w < NW; w++) s += part[w][threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// error of one edge of correspondence i at state S (inverse Si): e12 (side 0) from P2c with K1, e21 (side 1) from P1c with K2
__device__ __forceinline__ void edge_error(const Edges& E, int i, int side, const double* cam, const double* S, const double* Si,
                                           double* e) {
  const float* P = (side ? E.p1c : E.p2c) + 3 * i;
  const float* o = (side ? E.obs2 : E.obs1) + 2 * i;
  const double Pd[3] = {P[0], P[1], P[2]};
  const double od[2] = {o[0], o[1]};
  sim3_edge_error(side ? Si : S, Pd, cam + 4 * side, od, e);
}

__device__ __forceinline__ double chi2_2(const double* e, double info) { return e[0] * (info * e[0]) + e[1] * (info * e[1]); }

// BaseBinaryEdge::constructQuadraticForm for the Sim3 vertex with a Huber kernel
__device__ __forceinline__ void accumulate(const double* e, const double* J, double info, double delta, double* acc) {
  const double c2 = chi2_2(e, info);
  double w;
  const double rho = huber(c2, delta, &w);
  acc[35] += rho;
  const double wo = w * info;
  int k = 0;
#pragma unroll
  for (int r = 0; r < 7; r++) {
#pragma unroll
    for (int c = r; c < 7; c++, k++) acc[k] += wo * (J[r] * J[c] + J[7 + r] * J[7 + c]);
    acc[28 + r] -= wo * (J[r] * e[0] + J[7 + r] * e[1]);
  }
}

// dense 7x7 LDL^T with the isPositive() gate of Eigen::LDLT (linear_solver_dense.h)
__device__ bool solve7(const double* Hu /*upper packed*/, double lambda, const double* b, double* x) {
  double A[7][7];
  int k = 0;
#pragma unroll
  for (int r = 0; r < 7; r++)
#pragma unroll
    for (int c = r; c < 7; c++, k++) {
      A[r][c] = Hu[k];
      A[c][r] = Hu[k];
    }
#pragma unroll
  for (int r = 0; r < 7; r++) A[r][r] += lambda;
  double D[7];
#pragma unroll
  for (int j = 0; j < 7; j++) {
    double d = A[j][j];
#pragma unroll
    for (int q = 0; q < j; q++) d -= A[j][q] * A[j][q] * D[q];
    if (!(d > 0.0) || !isfinite(d)) return false;
    D[j] = d;
#pragma unroll
    for (int i = j + 1; i < 7; i++) {
      double s = A[i][j];
#pragma unroll
      for (int q = 0; q < j; q++) s -= A[i][q] * A[j][q] * D[q];
      A[i][j] = s / d;
    }
  }
  double z[7];
#pragma unroll
  for (int i = 0; i < 7; i++) {
    double s = b[i];
#pragma unroll
    for (int q = 0; q < i; q++) s -= A[i][q] * z[q];
    z[i] = s;
  }
#pragma unroll
  for (int i = 0; i < 7; i++) z[i] /= D[i];
#pragma unroll
  for (int i = 6; i >= 0; i--) {
    double s = z[i];
#pragma unroll
    for (int q = i + 1; q < 7; q++) s -= A[q][i] * x[q];
    x[i] = s;
  }
  return true;
}

struct Shared {
  double st[15][2][8];   // [0] current state, [1 + k] perturbed state k; [.][0] state, [.][1] inverse
  double trial[2][8];    // trial state and its inverse
  double x[7];           // the solver's x: zero at each optimize(), kept across its iterations (a failed solve leaves it)
  double Hb[35];
  double part[NW][NACC];
  double red[NACC];
  int ok;
};

template <bool STAGE>
__device__ void sim3_body(const Sim3View& v) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ Shared sh;
  const int pb = blockIdx.x, tid = threadIdx.x;
  const int e0 = v.off[pb], m = v.off[pb + 1] - e0;
  const bool fix = v.fix_scale[pb] != 0;
  const float th2 = v.th2[pb];
  const double delta = (double)sqrtf(th2);
  double cam[8];
#pragma unroll
  for (int k = 0; k < 8; k++) cam[k] = v.cam[8 * (size_t)pb + k];
  Edges E{v.p1c + 3 * (size_t)e0, v.p2c + 3 * (size_t)e0, v.obs1 + 2 * (size_t)e0, v.obs2 + 2 * (size_t)e0,
          v.info1 + e0, v.info2 + e0};
  if (STAGE) {
    float* sf = reinterpret_cast<float*>(dyn);
    float* s_p1 = sf; sf += 3 * m;
    float* s_p2 = sf; sf += 3 * m;
    float* s_o1 = sf; sf += 2 * m;
    float* s_o2 = sf; sf += 2 * m;
    float* s_i1 = sf; sf += m;
    float* s_i2 = sf;
    for (int i = tid; i < 3 * m; i += STPB) { s_p1[i] = E.p1c[i]; s_p2[i] = E.p2c[i]; }
    for (int i = tid; i < 2 * m; i += STPB) { s_o1[i] = E.obs1[i]; s_o2[i] = E.obs2[i]; }
    for (int i = tid; i < m; i += STPB) { s_i1[i] = E.info1[i]; s_i2[i] = E.info2[i]; }
    E = Edges{s_p1, s_p2, s_o1, s_o2, s_i1, s_i2};
  }
  double* chi = v.chi2 + 2 * (size_t)e0;
  uint8_t* lev = v.inlier + e0;
  for (int i = tid; i < m; i += STPB) { lev[i] = 1; chi[2 * i] = 0.0; chi[2 * i + 1] = 0.0; }
  if (tid < 8) sh.st[0][0][tid] = v.S12[8 * (size_t)pb + tid];
  double* logc = v.chi2_log ? v.chi2_log + (size_t)pb * v.log_stride : nullptr;
  double* logl = v.lambda_log ? v.lambda_log + (size_t)pb * v.log_stride : nullptr;
  int* logt = v.trials_log ? v.trials_log + (size_t)pb * v.log_stride : nullptr;
  if (tid == 0 && v.chi2_log)
    for (int k = 0; k < v.log_stride; k++) logc[k] = 0.0;
  if (tid == 0 && v.lambda_log)
    for (int k = 0; k < v.log_stride; k++) logl[k] = 0.0;
  if (tid == 0 && v.trials_log)
    for (int k = 0; k < v.log_stride; k++) logt[k] = 0;
  __syncthreads();

  int n_bad = 0, n_in = 0;
  bool early = false;
  for (int round = 0; round < 2; round++) {
    const int its = round == 0 ? v.its1 : (n_bad > 0 ? v.its_bad : v.its_clean);
    const int base = round == 0 ? 0 : v.its1 + 1;
    // ---- optimize(its) over the edges still in the graph ----
    if (tid < 7) sh.x[tid] = 0.0;
    double nact = 0;
    for (int i = tid; i < m; i += STPB) nact += lev[i];
    block_reduce<1>(&nact, reinterpret_cast<double(*)[1]>(&sh.part[0][0]), sh.red);
    bool go = sh.red[0] > 0.5;   // no edge: optimize() returns without an iteration
    __syncthreads();
    double lambda = 0.0, ni = 2.0;
    int n_bad_it = 0, done = 0;
    for (int it = 0; it < its && go; it++) {
      if (tid == 0) sim3_inverse(sh.st[0][0], sh.st[0][1]);
      else if (tid <= 14) sim3_perturbed(sh.st[0][0], tid - 1, fix, sh.st[tid][0], sh.st[tid][1]);
      __syncthreads();
      double acc[NACC];
#pragma unroll
      for (int k = 0; k < NACC; k++) acc[k] = 0.0;
      for (int i = tid; i < m; i += STPB) {
        if (!lev[i]) continue;
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
          double e[2], J[14];
          edge_error(E, i, side, cam, sh.st[0][0], sh.st[0][1], e);
#pragma unroll 1
          for (int d = 0; d < 7; d++) {
            double ep[2], em[2];
            edge_error(E, i, side, cam, sh.st[1 + 2 * d][0], sh.st[1 + 2 * d][1], ep);
            edge_error(E, i, side, cam, sh.st[2 + 2 * d][0], sh.st[2 + 2 * d][1], em);
            sim3_jac_col(ep, em, J, d);
          }
          accumulate(e, J, (double)(side ? E.info2[i] : E.info1[i]), delta, acc);
        }
      }
      block_reduce<NACC>(acc, sh.part, sh.red);
      if (tid < 35) sh.Hb[tid] = sh.red[tid];   // H (upper packed), b: kept for the trials of this iteration
      double currentChi = sh.red[35];
      const double iniChi = currentChi;
      __syncthreads();
      if (it == 0) {
        double mx = 0;
        int k = 0;
        for (int r = 0; r < 7; r++) {
          mx = fmax(mx, fabs(sh.Hb[k]));
          k += 7 - r;
        }
        lambda = 1e-5 * mx;
        ni = 2.0;
        n_bad_it = 0;
        if (logc && tid == 0) logc[base] = currentChi;
      }
      double rho = 0;
      int qmax = 0;
      bool again;
      do {
        if (tid == 0) {
          double xn[7];
          const bool ok2 = solve7(sh.Hb, lambda, sh.Hb + 28, xn);
          if (ok2)
#pragma unroll
            for (int k = 0; k < 7; k++) sh.x[k] = xn[k];
          sim3_oplus(sh.st[0][0], sh.x, fix, sh.trial[0]);   // oplusImpl may zero x[6] in place
          sim3_inverse(sh.trial[0], sh.trial[1]);
          sh.ok = ok2;
        }
        __syncthreads();
        double a1 = 0.0;
        for (int i = tid; i < m; i += STPB) {
          if (!lev[i]) continue;
          double e12[2], e21[2], w;
          edge_error(E, i, 0, cam, sh.trial[0], sh.trial[1], e12);
          edge_error(E, i, 1, cam, sh.trial[0], sh.trial[1], e21);
          const double c12 = chi2_2(e12, (double)E.info1[i]), c21 = chi2_2(e21, (double)E.info2[i]);
          chi[2 * i] = c12;
          chi[2 * i + 1] = c21;
          a1 += huber(c12, delta, &w);
          a1 += huber(c21, delta, &w);
        }
        block_reduce<1>(&a1, reinterpret_cast<double(*)[1]>(&sh.part[0][0]), sh.red);
        double tempChi = sh.red[0];
        if (!sh.ok) tempChi = DBL_MAX;
        rho = currentChi - tempChi;
        double scale = 0;
#pragma unroll
        for (int k = 0; k < 7; k++) scale += sh.x[k] * (lambda * sh.x[k] + sh.Hb[28 + k]);
        scale += 1e-3;
        rho /= scale;
        const bool accept = rho > 0 && isfinite(tempChi);
        if (accept) {
          double alpha = 1. - pow((2 * rho - 1), 3);
          alpha = fmin(alpha, 2. / 3.);
          lambda *= fmax(1. / 3., alpha);
          ni = 2;
          currentChi = tempChi;
        } else {
          lambda *= ni;
          ni *= 2;
        }
        __syncthreads();
        if (accept && tid < 8) sh.st[0][0][tid] = sh.trial[0][tid];
        qmax++;
        again = (rho < 0 && qmax < 10);
        __syncthreads();
      } while (again);
      done++;
      if (tid == 0) {
        if (logc) logc[base + done] = currentChi;
        if (logl) logl[base + done] = lambda;
        if (logt) logt[base + done] = qmax;
      }
      if (qmax == 10 || rho == 0) go = false;
      else {
        if ((iniChi - currentChi) * 1e3 < iniChi) n_bad_it++;
        else n_bad_it = 0;
        if (n_bad_it >= 3) go = false;
      }
    }
    if (tid == 0 && v.n_iter_done) v.n_iter_done[2 * (size_t)pb + round] = done;
    // ---- chi2 test on the stale errors: e12->chi2() > th2 || e21->chi2() > th2 ----
    double cnt[2] = {0.0, 0.0};   // dropped, kept
    for (int i = tid; i < m; i += STPB) {
      if (!lev[i]) continue;
      if (chi[2 * i] > (double)th2 || chi[2 * i + 1] > (double)th2) { lev[i] = 0; cnt[0] += 1.0; }
      else cnt[1] += 1.0;
    }
    block_reduce<2>(cnt, reinterpret_cast<double(*)[2]>(&sh.part[0][0]), sh.red);
    const int dropped = (int)(sh.red[0] + 0.5), kept = (int)(sh.red[1] + 0.5);
    __syncthreads();
    if (round == 0) {
      n_bad = dropped;
      if (m - n_bad < 10) { early = true; break; }   // return 0, g2oS12 unchanged
    } else {
      n_in = kept;
    }
  }
  if (tid < 8) v.out_S12[8 * (size_t)pb + tid] = early ? v.S12[8 * (size_t)pb + tid] : sh.st[0][0][tid];
  if (tid == 0) {
    v.n_in[pb] = early ? 0 : n_in;
    if (early && v.n_iter_done) v.n_iter_done[2 * (size_t)pb + 1] = 0;
  }
}

__global__ void __launch_bounds__(STPB) k_sim3_opt_smem(Sim3View v) { sim3_body<true>(v); }
__global__ void __launch_bounds__(STPB) k_sim3_opt_global(Sim3View v) { sim3_body<false>(v); }

}  // namespace

extern "C" int lld_sim3_opt(void* ctx, const lld_sim3_problem* p, lld_sim3_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  const int n = p->n_problems;
  LLD_ARG(c, n >= 0);
  LLD_ARG(c, p->its_first >= 0 && p->its_more_outliers >= 0 && p->its_more_clean >= 0);
  if (n == 0) return LLD_OK;
  LLD_ARG(c, p->off && p->off[0] == 0);
  size_t max_m = 0;
  for (int i = 0; i < n; i++) {
    LLD_ARG(c, p->off[i + 1] >= p->off[i]);
    LLD_ARG(c, p->fix_scale[i] == 0 || p->fix_scale[i] == 1);
    LLD_ARG(c, p->th2[i] > 0.f);
    max_m = std::max(max_m, (size_t)(p->off[i + 1] - p->off[i]));
  }
  const bool logs = out->chi2_log || out->lambda_log || out->trials_log;
  const int its2 = std::max(p->its_more_outliers, p->its_more_clean);
  LLD_ARG(c, !logs || out->log_stride >= p->its_first + its2 + 2);
  const int m = p->off[n];
  if (int r = lld_call_begin(c, true)) return r;
  Sim3View v{};
  v.n = n;
  LLD_UP(c, v.S12, p->S12, 8 * (size_t)n);
  LLD_UP(c, v.cam, p->cam, 8 * (size_t)n);
  LLD_UP(c, v.fix_scale, p->fix_scale, n);
  LLD_UP(c, v.th2, p->th2, n);
  LLD_UP(c, v.off, p->off, n + 1);
  LLD_UP(c, v.p1c, p->p1c, 3 * (size_t)m);
  LLD_UP(c, v.p2c, p->p2c, 3 * (size_t)m);
  LLD_UP(c, v.obs1, p->obs1, 2 * (size_t)m);
  LLD_UP(c, v.obs2, p->obs2, 2 * (size_t)m);
  LLD_UP(c, v.info1, p->info1, m);
  LLD_UP(c, v.info2, p->info2, m);
  v.its1 = p->its_first; v.its_bad = p->its_more_outliers; v.its_clean = p->its_more_clean;
  LLD_DEV(c, v.chi2, 2 * (size_t)m);
  LLD_DEV(c, v.out_S12, 8 * (size_t)n);
  LLD_DEV(c, v.inlier, m);
  LLD_DEV(c, v.n_in, n);
  v.log_stride = out->log_stride;
  if (out->chi2_log) LLD_DEV(c, v.chi2_log, (size_t)n * out->log_stride);
  if (out->lambda_log) LLD_DEV(c, v.lambda_log, (size_t)n * out->log_stride);
  if (out->trials_log) LLD_DEV(c, v.trials_log, (size_t)n * out->log_stride);
  if (out->n_iter_done) LLD_DEV(c, v.n_iter_done, 2 * (size_t)n);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  const size_t smem = EDGE_BYTES * max_m;
  if (smem <= SMEM_LIMIT) {
    LLD_CUDA(c, lld_raise_dyn_smem(k_sim3_opt_smem, smem));
    LLD_LAUNCH(c, k_sim3_opt_smem, n, STPB, smem, v);
  } else {
    LLD_LAUNCH(c, k_sim3_opt_global, n, STPB, 0, v);
  }
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, out->S12, v.out_S12, 8 * (size_t)n);
  LLD_DOWN(c, out->inlier, v.inlier, (size_t)m);
  LLD_DOWN(c, out->n_in, v.n_in, (size_t)n);
  LLD_DOWN(c, out->chi2_log, v.chi2_log, (size_t)n * out->log_stride);
  LLD_DOWN(c, out->lambda_log, v.lambda_log, (size_t)n * out->log_stride);
  LLD_DOWN(c, out->trials_log, v.trials_log, (size_t)n * out->log_stride);
  LLD_DOWN(c, out->n_iter_done, v.n_iter_done, 2 * (size_t)n);
  return lld_call_end(c);
}
