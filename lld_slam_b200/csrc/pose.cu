// pose.cu — batched motion-only pose optimisation (Optimizer::PoseOptimization, src/Optimizer.cc:562-932).
//
// One CTA per frame runs the whole 4 x 10 Levenberg-Marquardt schedule on the device: every thread owns a
// strided slice of the frame's unary edges (EdgeSE3ProjectXYZOnlyPose, EdgeStereoSE3ProjectXYZOnlyPose,
// EdgeSE3ProjectLineOnlyPose), the 6x6 normal equations are reduced in fixed order through shuffles + shared
// memory, thread 0 does the dense LDL^T (LinearSolverDense) and the LM bookkeeping
// (optimization_algorithm_levenberg.cpp:61-164), and the edge records are staged in shared memory once so the
// ~80 passes over them never touch HBM again.
#include <cfloat>

#include "lld_ctx.h"
#include "lld_math.cuh"

using namespace lld;

namespace {

constexpr int PTPB = 128;
constexpr int NW = PTPB / 32;

struct PoseView {
  int n_frames;
  const double* Tcw;
  const double* intr;
  const double* line_cam;
  const int* pt_off;
  const float* pt_xw;
  const float* pt_uvr;
  const float* pt_info;
  const int* ln_off;
  const double* ln_x0_dir;
  const float* ln_left;
  const float* ln_right;
  const double* ln_info;
  const uint8_t* ln_stereo;
  const uint8_t* ln_gate_stereo;
  double delta_mono, delta_stereo, delta_ln_mono, delta_ln_stereo;
  float chi2_mono, chi2_stereo;
  double gate_ln_mono, gate_ln_stereo;
  int n_rounds, its;
  // scratch (global): per-edge stale chi2 and level
  double* pt_chi2;
  double* ln_chi2;   // [n_ln][2]
  uint8_t* pt_level;
  uint8_t* ln_level; // [n_ln][2]  0 active, 1 outlier, 2 absent
  // outputs
  double* out_Tcw;
  uint8_t* pt_outlier;
  uint8_t* ln_outlier;
  int* n_inliers;
  double* chi2_final;
};

// fixed-order block reduction of NV values held per thread; result in out[] (shared), visible to all after return
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

struct FrameCtx {
  const float* xw;
  const float* uvr;
  const float* info;
  const double* x0d;
  const float* left;
  const float* right;
  const double* linfo;
  const uint8_t* lstereo;
  int np, nl;
  double intr[5];
  double cam[4];
};

// residual (+ optional pose Jacobian) of point edge i at pose Rt; returns dim
__device__ __forceinline__ int pt_edge(const FrameCtx& F, int i, const double* Rt, double* err, double* Jp) {
  const float* X = F.xw + 3 * i;
  const double Xd[3] = {X[0], X[1], X[2]};
  double xc[3];
  map_Rt(Rt, Xd, xc);
  const float* obs = F.uvr + 3 * i;
  const bool stereo = !(obs[2] < 0.f);
  pt_residual<false>(xc, F.intr, obs, stereo, err);
  if (Jp) pt_jac_pose(xc, F.intr, stereo, Jp);
  return stereo ? 3 : 2;
}
__device__ __forceinline__ void ln_edge(const FrameCtx& F, int i, int side, const double* Rt, double* err, double* Jp) {
  const double* xd = F.x0d + 6 * i;
  const double X1[3] = {xd[0], xd[1], xd[2]};
  const double X2[3] = {xd[0] + xd[3], xd[1] + xd[4], xd[2] + xd[5]};  // X2 = X0 + dir  (src/Optimizer.cc:629-630)
  double P1[3], P2[3];
  map_Rt(Rt, X1, P1);
  map_Rt(Rt, X2, P2);
  const float* seg = (side ? F.right : F.left) + 4 * i;
  LineObs o;
  o.x1[0] = seg[0]; o.x1[1] = seg[1]; o.x1[2] = 1.0;
  o.x2[0] = seg[2]; o.x2[1] = seg[3]; o.x2[2] = 1.0;
  const double bx = side ? -F.cam[3] : 0.0;
  if (Jp) line_linearize<false>(P1, P2, F.cam[0], F.cam[1], F.cam[2], bx, o, Rt, X1, X2, X1, err, Jp, nullptr);
  else line_residual(P1, P2, F.cam[0], F.cam[1], F.cam[2], bx, o, err);
}

// dense 6x6 LDL^T with the isPositive() gate of Eigen::LDLT (linear_solver_dense.h:107-112)
__device__ bool solve6(const double* H21 /*upper packed*/, double lambda, const double* b, double* x) {
  double A[6][6];
  int k = 0;
  for (int r = 0; r < 6; r++)
    for (int c = r; c < 6; c++, k++) {
      A[r][c] = H21[k];
      A[c][r] = H21[k];
    }
  for (int r = 0; r < 6; r++) A[r][r] += lambda;
  double D[6];
  for (int j = 0; j < 6; j++) {
    double d = A[j][j];
    for (int q = 0; q < j; q++) d -= A[j][q] * A[j][q] * D[q];
    if (!(d > 0.0) || !isfinite(d)) return false;
    D[j] = d;
    for (int i = j + 1; i < 6; i++) {
      double s = A[i][j];
      for (int q = 0; q < j; q++) s -= A[i][q] * A[j][q] * D[q];
      A[i][j] = s / d;
    }
  }
  double z[6];
  for (int i = 0; i < 6; i++) {
    double s = b[i];
    for (int q = 0; q < i; q++) s -= A[i][q] * z[q];
    z[i] = s;
  }
  for (int i = 0; i < 6; i++) z[i] /= D[i];
  for (int i = 5; i >= 0; i--) {
    double s = z[i];
    for (int q = i + 1; q < 6; q++) s -= A[q][i] * x[q];
    x[i] = s;
  }
  return true;
}

__global__ void __launch_bounds__(PTPB) k_pose_opt(PoseView v, int stage_smem) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ double part[NW][28];
  __shared__ double red[28];
  const int f = blockIdx.x;
  const int tid = threadIdx.x;
  const int p0 = v.pt_off[f], np = v.pt_off[f + 1] - p0;
  const int l0 = v.ln_off[f], nl = v.ln_off[f + 1] - l0;
  FrameCtx F;
  F.np = np; F.nl = nl;
#pragma unroll
  for (int k = 0; k < 5; k++) F.intr[k] = v.intr[5 * (size_t)f + k];
#pragma unroll
  for (int k = 0; k < 4; k++) F.cam[k] = v.line_cam[4 * (size_t)f + k];
  F.xw = v.pt_xw + 3 * (size_t)p0; F.uvr = v.pt_uvr + 3 * (size_t)p0; F.info = v.pt_info + p0;
  F.x0d = v.ln_x0_dir + 6 * (size_t)l0; F.left = v.ln_left + 4 * (size_t)l0; F.right = v.ln_right + 4 * (size_t)l0;
  F.linfo = v.ln_info + 2 * (size_t)l0; F.lstereo = v.ln_stereo + l0;
  if (stage_smem) {
    // layout: x0d (6 f64 / line), linfo (2 f64 / line), xw, uvr, info (f32 / point), left, right (4 f32 / line), lstereo
    double* sd = reinterpret_cast<double*>(dyn);
    double* s_x0d = sd; sd += 6 * nl;
    double* s_linfo = sd; sd += 2 * nl;
    float* sf = reinterpret_cast<float*>(sd);
    float* s_xw = sf; sf += 3 * np;
    float* s_uvr = sf; sf += 3 * np;
    float* s_info = sf; sf += np;
    float* s_left = sf; sf += 4 * nl;
    float* s_right = sf; sf += 4 * nl;
    uint8_t* s_st = reinterpret_cast<uint8_t*>(sf);
    for (int i = tid; i < 6 * nl; i += PTPB) s_x0d[i] = F.x0d[i];
    for (int i = tid; i < 2 * nl; i += PTPB) s_linfo[i] = F.linfo[i];
    for (int i = tid; i < 3 * np; i += PTPB) { s_xw[i] = F.xw[i]; s_uvr[i] = F.uvr[i]; }
    for (int i = tid; i < np; i += PTPB) s_info[i] = F.info[i];
    for (int i = tid; i < 4 * nl; i += PTPB) { s_left[i] = F.left[i]; s_right[i] = F.right[i]; }
    for (int i = tid; i < nl; i += PTPB) s_st[i] = F.lstereo[i];
    F.x0d = s_x0d; F.linfo = s_linfo; F.xw = s_xw; F.uvr = s_uvr; F.info = s_info;
    F.left = s_left; F.right = s_right; F.lstereo = s_st;
    __syncthreads();
  }
  double* pchi = v.pt_chi2 + p0;
  double* lchi = v.ln_chi2 + 2 * (size_t)l0;
  uint8_t* plev = v.pt_level + p0;
  uint8_t* llev = v.ln_level + 2 * (size_t)l0;
  uint8_t* pout = v.pt_outlier + p0;
  uint8_t* lout = v.ln_outlier + l0;
  // edge set-up
  int n_line_edges_local = 0;
  for (int i = tid; i < np; i += PTPB) { plev[i] = 0; pout[i] = 0; pchi[i] = 0.0; }
  for (int i = tid; i < nl; i += PTPB) {
    llev[2 * i] = 0;
    const bool has_r = !(F.right[4 * i] < 0.f);
    llev[2 * i + 1] = has_r ? 0 : 2;
    lout[i] = 0;
    n_line_edges_local += has_r ? 2 : 1;
  }
  double qt0[7];
  pose_from_Rt(v.Tcw + 12 * (size_t)f, qt0);
  {
    double a1[1] = {(double)n_line_edges_local};
    block_reduce<1>(a1, reinterpret_cast<double(*)[1]>(&part[0][0]), red);
  }
  const int n_edges_total = np + (int)(red[0] + 0.5);
  __syncthreads();
  if (np < 3) {  // src/Optimizer.cc:809-810
    if (tid == 0) {
      for (int k = 0; k < 12; k++) v.out_Tcw[12 * (size_t)f + k] = v.Tcw[12 * (size_t)f + k];
      v.n_inliers[f] = 0;
      if (v.chi2_final) v.chi2_final[f] = 0.0;
    }
    return;
  }
  int nBad = 0;
  double last_chi = 0.0;
  bool robust = true;
  double qt[7];
  for (int round = 0; round < v.n_rounds; round++) {
#pragma unroll
    for (int k = 0; k < 7; k++) qt[k] = qt0[k];  // vSE3->setEstimate(initial)  :823
    // ---- optimize(its) ----
    double lambda = -1.0, ni = 2.0;
    int n_bad_it = 0;
    double x[6] = {0, 0, 0, 0, 0, 0};
    // any active edge?  (empty index mapping -> optimize() does nothing)
    double nact_l = 0;
    for (int i = tid; i < np; i += PTPB) nact_l += (plev[i] == 0);
    for (int i = tid; i < 2 * nl; i += PTPB) nact_l += (llev[i] == 0);
    {
      double a1[1] = {nact_l};
      block_reduce<1>(a1, reinterpret_cast<double(*)[1]>(&part[0][0]), red);
    }
    const bool any_active = red[0] > 0.5;
    __syncthreads();
    bool go = any_active;
    for (int it = 0; it < v.its && go; it++) {
      // linearise at qt
      double Rt[12];
      pose_to_Rt(qt, Rt);
      double acc[28];
#pragma unroll
      for (int k = 0; k < 28; k++) acc[k] = 0.0;
      for (int i = tid; i < np; i += PTPB) {
        if (plev[i] != 0) continue;
        double err[3], Jp[18];
        const int D = pt_edge(F, i, Rt, err, Jp);
        const double info = (double)F.info[i];
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
        double wgt = 1.0, rho = c2;
        if (robust) rho = huber(c2, D == 3 ? v.delta_stereo : v.delta_mono, &wgt);
        acc[27] += rho;
        const double wo = wgt * info;
        int k = 0;
#pragma unroll
        for (int r = 0; r < 6; r++) {
#pragma unroll
          for (int c = r; c < 6; c++, k++) acc[k] += wo * (Jp[r] * Jp[c] + Jp[6 + r] * Jp[6 + c] + Jp[12 + r] * Jp[12 + c]);
          acc[21 + r] -= wo * (Jp[r] * err[0] + Jp[6 + r] * err[1] + Jp[12 + r] * err[2]);
        }
      }
      for (int e = tid; e < 2 * nl; e += PTPB) {
        if (llev[e] != 0) continue;
        const int i = e >> 1, side = e & 1;
        double err[2], Jp[12];
        ln_edge(F, i, side, Rt, err, Jp);
        const double info = F.linfo[e];
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
        double wgt = 1.0, rho = c2;
        if (robust) rho = huber(c2, F.lstereo[i] ? v.delta_ln_stereo : v.delta_ln_mono, &wgt);
        acc[27] += rho;
        const double wo = wgt * info;
        int k = 0;
#pragma unroll
        for (int r = 0; r < 6; r++) {
#pragma unroll
          for (int c = r; c < 6; c++, k++) acc[k] += wo * (Jp[r] * Jp[c] + Jp[6 + r] * Jp[6 + c]);
          acc[21 + r] -= wo * (Jp[r] * err[0] + Jp[6 + r] * err[1]);
        }
      }
      block_reduce<28>(acc, part, red);
      double H[21], b[6];
#pragma unroll
      for (int k = 0; k < 21; k++) H[k] = red[k];
#pragma unroll
      for (int k = 0; k < 6; k++) b[k] = red[21 + k];
      double currentChi = red[27];
      const double iniChi = currentChi;
      __syncthreads();
      if (it == 0) {
        double mx = 0;
        int k = 0;
        for (int r = 0; r < 6; r++) {
          mx = fmax(mx, fabs(H[k]));
          k += 6 - r;
        }
        lambda = 1e-5 * mx;
        ni = 2.0;
        n_bad_it = 0;
      }
      double rho = 0;
      int qmax = 0;
      bool again;
      do {
        // every thread solves the same 6x6 (cheaper than a broadcast round trip)
        double xn[6];
        const bool ok2 = solve6(H, lambda, b, xn);
        if (ok2)
#pragma unroll
          for (int k = 0; k < 6; k++) x[k] = xn[k];
        double qn[7];
        pose_oplus(qt, x, qn);
        double Rn[12];
        pose_to_Rt(qn, Rn);
        double a1[1] = {0.0};
        for (int i = tid; i < np; i += PTPB) {
          if (plev[i] != 0) continue;
          double err[3];
          const int D = pt_edge(F, i, Rn, err, nullptr);
          const double info = (double)F.info[i];
          const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
          pchi[i] = c2;
          double wgt;
          a1[0] += robust ? huber(c2, D == 3 ? v.delta_stereo : v.delta_mono, &wgt) : c2;
        }
        for (int e = tid; e < 2 * nl; e += PTPB) {
          if (llev[e] != 0) continue;
          const int i = e >> 1, side = e & 1;
          double err[2];
          ln_edge(F, i, side, Rn, err, nullptr);
          const double info = F.linfo[e];
          const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
          lchi[e] = c2;
          double wgt;
          a1[0] += robust ? huber(c2, F.lstereo[i] ? v.delta_ln_stereo : v.delta_ln_mono, &wgt) : c2;
        }
        block_reduce<1>(a1, reinterpret_cast<double(*)[1]>(&part[0][0]), red);
        double tempChi = red[0];
        __syncthreads();
        if (!ok2) tempChi = DBL_MAX;
        rho = currentChi - tempChi;
        double scale = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) scale += x[k] * (lambda * x[k] + b[k]);
        scale += 1e-3;
        rho /= scale;
        if (rho > 0 && isfinite(tempChi)) {
          double alpha = 1. - pow((2 * rho - 1), 3);
          alpha = fmin(alpha, 2. / 3.);
          lambda *= fmax(1. / 3., alpha);
          ni = 2;
          currentChi = tempChi;
#pragma unroll
          for (int k = 0; k < 7; k++) qt[k] = qn[k];
        } else {
          lambda *= ni;
          ni *= 2;
        }
        qmax++;
        again = (rho < 0 && qmax < 10);
      } while (again);
      last_chi = currentChi;
      if (qmax == 10 || rho == 0) go = false;
      else {
        if ((iniChi - currentChi) * 1e3 < iniChi) n_bad_it++;
        else n_bad_it = 0;
        if (n_bad_it >= 3) go = false;
      }
    }
    // ---- classification at the optimised pose (src/Optimizer.cc:828-912) ----
    double Rt[12];
    pose_to_Rt(qt, Rt);
    double nb[1] = {0.0};
    for (int i = tid; i < np; i += PTPB) {
      double c2 = pchi[i];
      const bool stereo = !(F.uvr[3 * i + 2] < 0.f);
      if (pout[i]) {  // only edges currently flagged are re-evaluated  :834-837
        double err[3];
        pt_edge(F, i, Rt, err, nullptr);
        const double info = (double)F.info[i];
        c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]) + err[2] * (info * err[2]);
        pchi[i] = c2;
      }
      const float chi2f = (float)c2;
      if (chi2f > (stereo ? v.chi2_stereo : v.chi2_mono)) { pout[i] = 1; plev[i] = 1; nb[0] += 1.0; }
      else { pout[i] = 0; plev[i] = 0; }
    }
    block_reduce<1>(nb, reinterpret_cast<double(*)[1]>(&part[0][0]), red);
    nBad = (int)(red[0] + 0.5);
    __syncthreads();
    if (n_edges_total < 10) break;  // optimizer.edges().size()<10  :886
    // lines: always re-evaluated (:895); the right edge, when present, has the last word on mvbOutlierLines[idx]
    for (int i = tid; i < nl; i += PTPB) {
      for (int side = 0; side < 2; side++) {
        const int e = 2 * i + side;
        if (llev[e] == 2) continue;
        double err[2];
        ln_edge(F, i, side, Rt, err, nullptr);
        const double info = F.linfo[e];
        const double c2 = err[0] * (info * err[0]) + err[1] * (info * err[1]);
        lchi[e] = c2;
        const float chi2f = (float)c2;
        const double thr = v.ln_gate_stereo[2 * (size_t)(l0 + i) + side] ? v.gate_ln_stereo : v.gate_ln_mono;
        if ((double)chi2f > thr) { lout[i] = 1; llev[e] = 1; }
        else { lout[i] = 0; llev[e] = 0; }
      }
    }
    if (round == 2) robust = false;  // it==2: setRobustKernel(0)
    __syncthreads();
  }
  if (tid == 0) {
    double Rt[12];
    pose_to_Rt(qt, Rt);
    for (int k = 0; k < 12; k++) v.out_Tcw[12 * (size_t)f + k] = Rt[k];
    v.n_inliers[f] = np - nBad;
    if (v.chi2_final) v.chi2_final[f] = last_chi;
  }
}

// resident-mode view (bench), owned by the context; invalid once another entry point of the context recycles the device pool
struct PoseResident { PoseView v; size_t smem = 0; };
PoseResident* pose_resident(LldCtx* c, bool create) {
  if (!c->resident[1] && create) {
    c->resident[1] = new PoseResident();
    c->resident_free[1] = [](void* p) { delete static_cast<PoseResident*>(p); };
  }
  return static_cast<PoseResident*>(c->resident[1]);
}
bool pose_resident_valid(LldCtx* c) {
  if (c->resident[1] && c->resident_gen[1] == c->pool_gen) return true;
  snprintf(c->err, sizeof(c->err), "no resident pose problem (not uploaded, or another call on this context recycled the device pool)");
  return false;
}

int pose_upload(LldCtx* c, const lld_pose_problem* p, PoseView& v, size_t* smem_out) {
  v = PoseView();
  const int F = p->n_frames;
  LLD_ARG(c, F >= 1);
  const int np = p->pt_off[F], nl = p->ln_off[F];
  v.n_frames = F;
  LLD_UP(c, v.Tcw, p->Tcw, 12 * (size_t)F);
  LLD_UP(c, v.intr, p->intr, 5 * (size_t)F);
  LLD_UP(c, v.line_cam, p->line_cam, 4 * (size_t)F);
  LLD_UP(c, v.pt_off, p->pt_off, F + 1);
  LLD_UP(c, v.pt_xw, p->pt_xw, 3 * (size_t)np);
  LLD_UP(c, v.pt_uvr, p->pt_uvr, 3 * (size_t)np);
  LLD_UP(c, v.pt_info, p->pt_info, np);
  LLD_UP(c, v.ln_off, p->ln_off, F + 1);
  LLD_UP(c, v.ln_x0_dir, p->ln_x0_dir, 6 * (size_t)nl);
  LLD_UP(c, v.ln_left, p->ln_left, 4 * (size_t)nl);
  LLD_UP(c, v.ln_right, p->ln_right, 4 * (size_t)nl);
  LLD_UP(c, v.ln_info, p->ln_info, 2 * (size_t)nl);
  LLD_UP(c, v.ln_stereo, p->ln_stereo, nl);
  LLD_UP(c, v.ln_gate_stereo, p->ln_gate_stereo, 2 * (size_t)nl);
  v.delta_mono = p->delta_mono; v.delta_stereo = p->delta_stereo;
  v.delta_ln_mono = p->delta_ln_mono; v.delta_ln_stereo = p->delta_ln_stereo;
  v.chi2_mono = p->chi2_mono; v.chi2_stereo = p->chi2_stereo;
  v.gate_ln_mono = p->gate_ln_mono; v.gate_ln_stereo = p->gate_ln_stereo;
  v.n_rounds = p->n_rounds; v.its = p->its;
  LLD_DEV(c, v.pt_chi2, np);
  LLD_DEV(c, v.ln_chi2, 2 * (size_t)nl);
  LLD_DEV(c, v.pt_level, np);
  LLD_DEV(c, v.ln_level, 2 * (size_t)nl);
  LLD_DEV(c, v.out_Tcw, 12 * (size_t)F);
  LLD_DEV(c, v.pt_outlier, np);
  LLD_DEV(c, v.ln_outlier, nl);
  LLD_DEV(c, v.n_inliers, F);
  LLD_DEV(c, v.chi2_final, F);
  // shared-memory staging size = largest frame
  size_t mx = 0;
  for (int f = 0; f < F; f++) {
    const size_t a = p->pt_off[f + 1] - p->pt_off[f], b = p->ln_off[f + 1] - p->ln_off[f];
    const size_t s = 8 * (6 * b + 2 * b) + 4 * (3 * a + 3 * a + a + 4 * b + 4 * b) + b + 16;
    mx = s > mx ? s : mx;
  }
  *smem_out = mx;
  return LLD_OK;
}

int pose_run(LldCtx* c, PoseView& v, size_t smem_need) {
  const size_t limit = 200 * 1024;
  const int stage = smem_need <= limit ? 1 : 0;
  const size_t smem = stage ? smem_need : 0;
  if (stage) LLD_CUDA(c, lld_raise_dyn_smem(k_pose_opt, (size_t)(int)smem));
  LLD_LAUNCH(c, k_pose_opt, v.n_frames, PTPB, smem, v, stage);
  LLD_CUDA(c, cudaGetLastError());
  return LLD_OK;
}

int pose_download(LldCtx* c, PoseView& v, const lld_pose_problem* p, lld_pose_result* out) {
  const int F = v.n_frames;
  const int np = p->pt_off[F], nl = p->ln_off[F];
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, out->Tcw, v.out_Tcw, 12 * (size_t)F);
  LLD_DOWN(c, out->pt_outlier, v.pt_outlier, (size_t)np);
  LLD_DOWN(c, out->ln_outlier, v.ln_outlier, (size_t)nl);
  LLD_DOWN(c, out->n_inliers, v.n_inliers, (size_t)F);
  LLD_DOWN(c, out->chi2_final, v.chi2_final, (size_t)F);
  return lld_call_end(c);
}

}  // namespace

extern "C" int lld_pose_opt(void* ctx, const lld_pose_problem* p, lld_pose_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, true)) return r;
  PoseView v;
  size_t smem = 0;
  int r = pose_upload(c, p, v, &smem);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  r = pose_run(c, v, smem);
  if (r) return r;
  return pose_download(c, v, p, out);
}

// resident mode (bench)
extern "C" int lld_pose_upload(void* ctx, const lld_pose_problem* p) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, false)) return r;
  PoseResident* R = pose_resident(c, true);
  int r = pose_upload(c, p, R->v, &R->smem);
  c->resident_gen[1] = r ? 0 : c->pool_gen;
  if (r) return r;
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  return LLD_OK;
}
extern "C" int lld_pose_run(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !pose_resident_valid(c)) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaSetDevice(c->device));
  PoseResident* R = pose_resident(c, false);
  return pose_run(c, R->v, R->smem);
}
extern "C" int lld_pose_download(void* ctx, const lld_pose_problem* p, lld_pose_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !out || !pose_resident_valid(c)) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  return pose_download(c, pose_resident(c, false)->v, p, out);
}
