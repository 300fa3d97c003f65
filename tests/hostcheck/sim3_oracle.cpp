// ORACLE — TEST INFRASTRUCTURE ONLY.  CPU restatement of Optimizer::OptimizeSim3 (src/Optimizer.cc:1656-1858; the ORB-SLAM2
// function LLD-SLAM inherits unchanged) under the C-ABI of include/lldba.h with the lldo_ prefix, like the oracle library in
// oracle/.  A plain sequential transcription of the g2o pieces it runs: g2o::Sim3 (types/sim3.h), VertexSim3Expmap,
// EdgeSim3ProjectXYZ / EdgeInverseSim3ProjectXYZ (ORB-SLAM2's types_seven_dof_expmap.h, numeric Jacobian of
// BaseBinaryEdge::linearizeOplus with push / oplus / computeError / pop), BlockSolverX + LinearSolverDense (LDL^T with the
// isPositive gate) and OptimizationAlgorithmLevenberg.  Built by __graft_entry__.build() into
// tests/hostcheck/libsim3_oracle.so with -ffp-contract=off.  The product never loads it.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <limits>
#include <vector>

#include "../../include/lldba.h"

namespace {

struct Sim3 {
  double q[4] = {0, 0, 0, 1};  // x y z w
  double t[3] = {0, 0, 0};
  double s = 1;
};

// Eigen's Quaternion::_transformVector: uv = 2 (q.vec x v); v + w uv + q.vec x uv
void rotate(const double* q, const double* v, double* o) {
  double uv[3] = {q[1] * v[2] - q[2] * v[1], q[2] * v[0] - q[0] * v[2], q[0] * v[1] - q[1] * v[0]};
  for (int k = 0; k < 3; k++) uv[k] += uv[k];
  const double c[3] = {q[1] * uv[2] - q[2] * uv[1], q[2] * uv[0] - q[0] * uv[2], q[0] * uv[1] - q[1] * uv[0]};
  for (int k = 0; k < 3; k++) o[k] = v[k] + q[3] * uv[k] + c[k];
}

// Eigen's quaternion product
void qmul(const double* a, const double* b, double* o) {
  const double w = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
  const double x = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
  const double y = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
  const double z = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z; o[3] = w;
}

// Quaterniond(const Matrix3d&): Eigen's quaternion_assign_impl
void quat_of(const double m[3][3], double* q) {
  double t = m[0][0] + m[1][1] + m[2][2];
  if (t > 0) {
    t = std::sqrt(t + 1.0);
    q[3] = 0.5 * t;
    t = 0.5 / t;
    q[0] = (m[2][1] - m[1][2]) * t;
    q[1] = (m[0][2] - m[2][0]) * t;
    q[2] = (m[1][0] - m[0][1]) * t;
  } else {
    int i = 0;
    if (m[1][1] > m[0][0]) i = 1;
    if (m[2][2] > m[i][i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = std::sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0);
    q[i] = 0.5 * t;
    t = 0.5 / t;
    q[3] = (m[k][j] - m[j][k]) * t;
    q[j] = (m[j][i] + m[i][j]) * t;
    q[k] = (m[k][i] + m[i][k]) * t;
  }
}

// Sim3(const Vector7d& update)
Sim3 sim3_from_update(const double* u) {
  const double omega[3] = {u[0], u[1], u[2]};
  const double upsilon[3] = {u[3], u[4], u[5]};
  const double sigma = u[6];
  const double theta = std::sqrt(omega[0] * omega[0] + omega[1] * omega[1] + omega[2] * omega[2]);
  const double Om[3][3] = {{0, -omega[2], omega[1]}, {omega[2], 0, -omega[0]}, {-omega[1], omega[0], 0}};
  Sim3 S;
  S.s = std::exp(sigma);
  double Om2[3][3];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) Om2[i][j] = Om[i][0] * Om[0][j] + Om[i][1] * Om[1][j] + Om[i][2] * Om[2][j];
  const double I[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  double R[3][3];
  const double eps = 0.00001;
  double A, B, C;
  auto rodrigues = [&]() {
    const double a = std::sin(theta) / theta, b = (1 - std::cos(theta)) / (theta * theta);
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) R[i][j] = I[i][j] + a * Om[i][j] + b * Om2[i][j];
  };
  auto small = [&]() {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) R[i][j] = I[i][j] + Om[i][j] + Om2[i][j];
  };
  if (std::fabs(sigma) < eps) {
    C = 1;
    if (theta < eps) {
      A = 1. / 2.;
      B = 1. / 6.;
      small();
    } else {
      const double theta2 = theta * theta;
      A = (1 - std::cos(theta)) / (theta2);
      B = (theta - std::sin(theta)) / (theta2 * theta);
      rodrigues();
    }
  } else {
    C = (S.s - 1) / sigma;
    if (theta < eps) {
      const double sigma2 = sigma * sigma;
      A = ((sigma - 1) * S.s + 1) / sigma2;
      B = ((0.5 * sigma2 - sigma + 1) * S.s) / (sigma2 * sigma);
      small();
    } else {
      rodrigues();
      const double a = S.s * std::sin(theta);
      const double b = S.s * std::cos(theta);
      const double theta2 = theta * theta;
      const double sigma2 = sigma * sigma;
      const double c = theta2 + sigma2;
      A = (a * sigma + (1 - b) * theta) / (theta * c);
      B = (C - ((b - 1) * sigma + a * theta) / (c)) * 1. / (theta2);
    }
  }
  quat_of(R, S.q);
  double W[3][3];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) W[i][j] = A * Om[i][j] + B * Om2[i][j] + C * I[i][j];
  for (int i = 0; i < 3; i++) S.t[i] = W[i][0] * upsilon[0] + W[i][1] * upsilon[1] + W[i][2] * upsilon[2];
  return S;
}

Sim3 operator*(const Sim3& A, const Sim3& B) {
  Sim3 r;
  qmul(A.q, B.q, r.q);
  double rt[3];
  rotate(A.q, B.t, rt);
  for (int k = 0; k < 3; k++) r.t[k] = A.s * rt[k] + A.t[k];
  r.s = A.s * B.s;
  return r;
}

Sim3 inverse(const Sim3& S) {
  Sim3 r;
  r.q[0] = -S.q[0]; r.q[1] = -S.q[1]; r.q[2] = -S.q[2]; r.q[3] = S.q[3];
  const double c = -1. / S.s;
  const double v[3] = {c * S.t[0], c * S.t[1], c * S.t[2]};
  rotate(r.q, v, r.t);
  r.s = 1. / S.s;
  return r;
}

void map(const Sim3& S, const double* x, double* o) {
  double rx[3];
  rotate(S.q, x, rx);
  for (int k = 0; k < 3; k++) o[k] = S.s * rx[k] + S.t[k];
}

struct Vertex {  // VertexSim3Expmap
  Sim3 est;
  std::vector<Sim3> stack;
  bool fix_scale = false;
  double f1[2], pp1[2], f2[2], pp2[2];
  void push() { stack.push_back(est); }
  void pop() { est = stack.back(); stack.pop_back(); }
  void oplus(double* update) {
    if (fix_scale) update[6] = 0;
    est = sim3_from_update(update) * est;
  }
};

struct Edge {  // EdgeSim3ProjectXYZ (inverse = false) / EdgeInverseSim3ProjectXYZ (inverse = true)
  bool inverse_edge;
  double P[3];       // the fixed point vertex
  double obs[2];
  double info;
  double err[2] = {0, 0};
  double J[2][7];
  int pair;
  void computeError(const Vertex& v) {
    double x[3];
    if (inverse_edge) map(inverse(v.est), P, x);
    else map(v.est, P, x);
    const double p0 = x[0] / x[2], p1 = x[1] / x[2];
    const double* f = inverse_edge ? v.f2 : v.f1;
    const double* pp = inverse_edge ? v.pp2 : v.pp1;
    err[0] = obs[0] - (p0 * f[0] + pp[0]);
    err[1] = obs[1] - (p1 * f[1] + pp[1]);
  }
  double chi2() const { return err[0] * (info * err[0]) + err[1] * (info * err[1]); }
  // BaseBinaryEdge::linearizeOplus, numeric; the point vertex is fixed and skipped
  void linearizeOplus(Vertex& v) {
    const double delta = 1e-9;
    const double scalar = 1.0 / (2 * delta);
    const double before[2] = {err[0], err[1]};
    double add[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int d = 0; d < 7; d++) {
      v.push();
      add[d] = delta;
      v.oplus(add);
      computeError(v);
      double bak[2] = {err[0], err[1]};
      v.pop();
      v.push();
      add[d] = -delta;
      v.oplus(add);
      computeError(v);
      bak[0] -= err[0];
      bak[1] -= err[1];
      v.pop();
      add[d] = 0.0;
      J[0][d] = scalar * bak[0];
      J[1][d] = scalar * bak[1];
    }
    err[0] = before[0];
    err[1] = before[1];
  }
};

// RobustKernelHuber::robustify
void huber(double e, double delta, double* rho0, double* rho1) {
  const double dsqr = delta * delta;
  if (e <= dsqr) { *rho0 = e; *rho1 = 1.; return; }
  const double sqrte = std::sqrt(e);
  *rho0 = 2 * sqrte * delta - dsqr;
  *rho1 = delta / sqrte;
}

struct Optimizer {
  Vertex v;
  std::vector<Edge> edges;      // insertion order: e12, e21 of each correspondence
  std::vector<char> active;     // edge still in the graph
  double delta = 0;
  double lambda = 0, ni = 2;
  int n_bad = 0;
  double x[7];
  // logs of the current round
  std::vector<double> chi2_log, lambda_log;
  std::vector<int> trials_log;

  void computeActiveErrors() {
    for (size_t k = 0; k < edges.size(); k++)
      if (active[k]) edges[k].computeError(v);
  }
  double activeRobustChi2() const {
    double chi = 0;
    for (size_t k = 0; k < edges.size(); k++) {
      if (!active[k]) continue;
      double r0, r1;
      huber(edges[k].chi2(), delta, &r0, &r1);
      chi += r0;
    }
    return chi;
  }
  // BlockSolverX::buildSystem for the single Sim3 vertex: H = sum J^T (rho' Omega) J, b = -sum J^T (rho' Omega) e
  void buildSystem(double H[7][7], double b[7]) {
    for (int r = 0; r < 7; r++) {
      b[r] = 0;
      for (int c = 0; c < 7; c++) H[r][c] = 0;
    }
    for (size_t k = 0; k < edges.size(); k++) {
      if (!active[k]) continue;
      Edge& e = edges[k];
      e.linearizeOplus(v);
      double r0, r1;
      huber(e.chi2(), delta, &r0, &r1);
      const double wo = r1 * e.info;
      for (int r = 0; r < 7; r++) {
        for (int c = 0; c < 7; c++) H[r][c] += wo * (e.J[0][r] * e.J[0][c] + e.J[1][r] * e.J[1][c]);
        b[r] -= wo * (e.J[0][r] * e.err[0] + e.J[1][r] * e.err[1]);
      }
    }
  }
  // LinearSolverDense: LDL^T, fails unless every pivot is positive (Eigen::LDLT::isPositive)
  static bool solve(const double H[7][7], double lam, const double b[7], double xo[7]) {
    double A[7][7], D[7];
    for (int r = 0; r < 7; r++)
      for (int c = 0; c < 7; c++) A[r][c] = H[r][c] + (r == c ? lam : 0.0);
    for (int j = 0; j < 7; j++) {
      double d = A[j][j];
      for (int q = 0; q < j; q++) d -= A[j][q] * A[j][q] * D[q];
      if (!(d > 0.0) || !std::isfinite(d)) return false;
      D[j] = d;
      for (int i = j + 1; i < 7; i++) {
        double s = A[i][j];
        for (int q = 0; q < j; q++) s -= A[i][q] * A[j][q] * D[q];
        A[i][j] = s / d;
      }
    }
    double y[7], z[7];   // L y = b, z = D^-1 y, L^T x = z
    for (int i = 0; i < 7; i++) {
      double s = b[i];
      for (int q = 0; q < i; q++) s -= A[i][q] * y[q];
      y[i] = s;
    }
    for (int i = 0; i < 7; i++) z[i] = y[i] / D[i];
    for (int i = 6; i >= 0; i--) {
      double s = z[i];
      for (int q = i + 1; q < 7; q++) s -= A[q][i] * xo[q];
      xo[i] = s;
    }
    return true;
  }
  // OptimizationAlgorithmLevenberg::solve; 1 = stop
  int lmSolve(int iteration) {
    computeActiveErrors();
    double currentChi = activeRobustChi2();
    const double iniChi = currentChi;
    double H[7][7], b[7];
    buildSystem(H, b);
    if (iteration == 0) {
      double mx = 0;
      for (int j = 0; j < 7; j++) mx = std::max(std::fabs(H[j][j]), mx);
      lambda = 1e-5 * mx;
      ni = 2;
      n_bad = 0;
      chi2_log.push_back(currentChi);
    }
    double rho = 0;
    int qmax = 0;
    do {
      v.push();
      double xn[7];
      const bool ok2 = solve(H, lambda, b, xn);
      if (ok2) std::copy(xn, xn + 7, x);
      v.oplus(x);
      computeActiveErrors();
      double tempChi = activeRobustChi2();
      if (!ok2) tempChi = std::numeric_limits<double>::max();
      rho = currentChi - tempChi;
      double scale = 0;
      for (int j = 0; j < 7; j++) scale += x[j] * (lambda * x[j] + b[j]);
      scale += 1e-3;
      rho /= scale;
      if (rho > 0 && std::isfinite(tempChi)) {
        double alpha = 1. - std::pow((2 * rho - 1), 3);
        alpha = std::min(alpha, 2. / 3.);
        lambda *= std::max(1. / 3., alpha);
        ni = 2;
        currentChi = tempChi;
        v.stack.pop_back();   // discardTop
      } else {
        lambda *= ni;
        ni *= 2;
        v.pop();
      }
      qmax++;
    } while (rho < 0 && qmax < 10);
    chi2_log.push_back(currentChi);
    lambda_log.push_back(lambda);
    trials_log.push_back(qmax);
    if (qmax == 10 || rho == 0) return 1;
    if ((iniChi - currentChi) * 1e3 < iniChi) n_bad++;
    else n_bad = 0;
    if (n_bad >= 3) return 1;
    return 0;
  }
  // initializeOptimization(); optimize(its): returns the iterations run
  int optimize(int its) {
    chi2_log.clear(); lambda_log.clear(); trials_log.clear();
    std::fill(x, x + 7, 0.0);
    bool any = false;
    for (char a : active) any |= a != 0;
    if (!any) return 0;
    int done = 0;
    for (int i = 0; i < its; i++) {
      done++;
      if (lmSolve(i)) break;
    }
    return done;
  }
};

void put(const Sim3& S, double* o) {
  for (int k = 0; k < 4; k++) o[k] = S.q[k];
  for (int k = 0; k < 3; k++) o[4 + k] = S.t[k];
  o[7] = S.s;
}
Sim3 get(const double* o) {
  Sim3 S;
  for (int k = 0; k < 4; k++) S.q[k] = o[k];
  for (int k = 0; k < 3; k++) S.t[k] = o[4 + k];
  S.s = o[7];
  return S;
}

}  // namespace

extern "C" int lldo_sim3_opt(void*, const lld_sim3_problem* p, lld_sim3_result* out) {
  for (int pb = 0; pb < p->n_problems; pb++) {
    const int e0 = p->off[pb], m = p->off[pb + 1] - e0;
    Optimizer O;
    const double* K = p->cam + 8 * (size_t)pb;
    O.v.est = get(p->S12 + 8 * (size_t)pb);
    O.v.fix_scale = p->fix_scale[pb] != 0;
    O.v.f1[0] = K[0]; O.v.f1[1] = K[1]; O.v.pp1[0] = K[2]; O.v.pp1[1] = K[3];
    O.v.f2[0] = K[4]; O.v.f2[1] = K[5]; O.v.pp2[0] = K[6]; O.v.pp2[1] = K[7];
    const float th2 = p->th2[pb];
    O.delta = (double)std::sqrt(th2);   // const float deltaHuber = sqrt(th2)
    for (int i = 0; i < m; i++) {
      const size_t g = (size_t)(e0 + i);
      Edge e12, e21;
      e12.inverse_edge = false; e21.inverse_edge = true;
      for (int k = 0; k < 3; k++) { e12.P[k] = p->p2c[3 * g + k]; e21.P[k] = p->p1c[3 * g + k]; }
      for (int k = 0; k < 2; k++) { e12.obs[k] = p->obs1[2 * g + k]; e21.obs[k] = p->obs2[2 * g + k]; }
      e12.info = p->info1[g]; e21.info = p->info2[g];
      e12.pair = e21.pair = i;
      O.edges.push_back(e12);
      O.edges.push_back(e21);
      out->inlier[g] = 1;
    }
    O.active.assign(O.edges.size(), 1);
    const Sim3 initial = O.v.est;
    double* lc = out->chi2_log ? out->chi2_log + (size_t)pb * out->log_stride : nullptr;
    double* ll = out->lambda_log ? out->lambda_log + (size_t)pb * out->log_stride : nullptr;
    int* lt = out->trials_log ? out->trials_log + (size_t)pb * out->log_stride : nullptr;
    for (int k = 0; lc && k < out->log_stride; k++) lc[k] = 0;
    for (int k = 0; ll && k < out->log_stride; k++) ll[k] = 0;
    for (int k = 0; lt && k < out->log_stride; k++) lt[k] = 0;
    auto log_round = [&](int base) {
      for (size_t k = 0; lc && k < O.chi2_log.size(); k++) lc[base + k] = O.chi2_log[k];
      for (size_t k = 0; ll && k < O.lambda_log.size(); k++) ll[base + 1 + k] = O.lambda_log[k];
      for (size_t k = 0; lt && k < O.trials_log.size(); k++) lt[base + 1 + k] = O.trials_log[k];
    };
    // optimize(5) and the first test
    const int done1 = O.optimize(p->its_first);
    log_round(0);
    int nBad = 0;
    for (int i = 0; i < m; i++) {
      Edge &e12 = O.edges[2 * i], &e21 = O.edges[2 * i + 1];
      if (e12.chi2() > th2 || e21.chi2() > th2) {
        out->inlier[e0 + i] = 0;
        O.active[2 * i] = O.active[2 * i + 1] = 0;
        nBad++;
      }
    }
    const int nMore = nBad > 0 ? p->its_more_outliers : p->its_more_clean;
    if (out->n_iter_done) { out->n_iter_done[2 * pb] = done1; out->n_iter_done[2 * pb + 1] = 0; }
    if (m - nBad < 10) {
      put(initial, out->S12 + 8 * (size_t)pb);
      out->n_in[pb] = 0;
      continue;
    }
    const int done2 = O.optimize(nMore);
    log_round(p->its_first + 1);
    if (out->n_iter_done) out->n_iter_done[2 * pb + 1] = done2;
    int nIn = 0;
    for (int i = 0; i < m; i++) {
      if (!O.active[2 * i]) continue;
      if (O.edges[2 * i].chi2() > th2 || O.edges[2 * i + 1].chi2() > th2) out->inlier[e0 + i] = 0;
      else nIn++;
    }
    put(O.v.est, out->S12 + 8 * (size_t)pb);
    out->n_in[pb] = nIn;
  }
  return 0;
}

// pieces of the listing, for the host check of the device math (tests/test_optimize_sim3.py)
extern "C" void lldo_sim3_exp(const double* u, double* S) { put(sim3_from_update(u), S); }
extern "C" void lldo_sim3_mul(const double* A, const double* B, double* O) { put(get(A) * get(B), O); }
extern "C" void lldo_sim3_inverse(const double* S, double* O) { put(inverse(get(S)), O); }
extern "C" void lldo_sim3_map(const double* S, const double* x, double* o) { map(get(S), x, o); }
// e12 / e21 of one correspondence at S and their numeric Jacobians ([2][7] each); cam = K1, K2
extern "C" void lldo_sim3_edges(const double* S, int fix_scale, const double* cam, const float* p1c, const float* p2c,
                                const float* obs1, const float* obs2, double* e12, double* e21, double* J12, double* J21) {
  Vertex v;
  v.est = get(S);
  v.fix_scale = fix_scale != 0;
  v.f1[0] = cam[0]; v.f1[1] = cam[1]; v.pp1[0] = cam[2]; v.pp1[1] = cam[3];
  v.f2[0] = cam[4]; v.f2[1] = cam[5]; v.pp2[0] = cam[6]; v.pp2[1] = cam[7];
  Edge a, b;
  a.inverse_edge = false; b.inverse_edge = true;
  for (int k = 0; k < 3; k++) { a.P[k] = p2c[k]; b.P[k] = p1c[k]; }
  for (int k = 0; k < 2; k++) { a.obs[k] = obs1[k]; b.obs[k] = obs2[k]; }
  a.info = b.info = 1;
  a.computeError(v); b.computeError(v);
  a.linearizeOplus(v); b.linearizeOplus(v);
  for (int k = 0; k < 2; k++) { e12[k] = a.err[k]; e21[k] = b.err[k]; }
  for (int r = 0; r < 2; r++)
    for (int d = 0; d < 7; d++) { J12[7 * r + d] = a.J[r][d]; J21[7 * r + d] = b.J[r][d]; }
}
