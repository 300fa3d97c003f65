// CPU oracle of lld_pnp_ransac (include/lldba.h): a plain sequential restatement of ORB-SLAM2's PnPsolver (iterate, Refine,
// CheckInliers) and of Lepetit's epnp.cpp (compute_pose and its stages) in that file's structure: the correspondences are
// copied into pws / us, the barycentric coordinates and camera points are stored per correspondence, M is filled row by
// row.  The SVDs and the eigen decomposition are the cyclic Jacobi solvers the header describes (the contract does not ask
// for OpenCV's bits there); every sum over correspondences runs in correspondence order.  Test infrastructure: built by
// __graft_entry__.build() into libpnp_ransac_oracle.so and bound by capi.load_oracle(); tests/test_pnp_ransac.py pins it
// with an independent Python transcription that calls cv2 (SVDecomp, solve, invert).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/lldba.h"

namespace {

double dot(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// two-sided cyclic Jacobi on the symmetric n x n A; eigenvectors in V's columns; ord by decreasing eigenvalue (stable)
void sym_jacobi(double* A, double* V, int n, int* ord) {
  for (int k = 0; k < n * n; k++) V[k] = (k / n == k % n) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 32; sweep++) {
    double off = 0, dia = 0;
    for (int i = 0; i < n; i++) {
      dia += std::fabs(A[i * n + i]);
      for (int j = i + 1; j < n; j++) off += std::fabs(A[i * n + j]);
    }
    if (!(off > 1e-15 * dia)) break;
    for (int p = 0; p < n - 1; p++)
      for (int q = p + 1; q < n; q++) {
        const double apq = A[p * n + q];
        if (apq == 0.0) continue;
        const double theta = (A[q * n + q] - A[p * n + p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < n; k++) {
          const double x = A[k * n + p], y = A[k * n + q];
          A[k * n + p] = c * x - s * y;
          A[k * n + q] = s * x + c * y;
          const double vx = V[k * n + p], vy = V[k * n + q];
          V[k * n + p] = c * vx - s * vy;
          V[k * n + q] = s * vx + c * vy;
        }
        for (int k = 0; k < n; k++) {
          const double x = A[p * n + k], y = A[q * n + k];
          A[p * n + k] = c * x - s * y;
          A[q * n + k] = s * x + c * y;
        }
      }
  }
  for (int i = 0; i < n; i++) ord[i] = i;
  for (int i = 1; i < n; i++) {
    const int x = ord[i];
    int j = i;
    for (; j > 0 && A[x * n + x] > A[ord[j - 1] * n + ord[j - 1]]; j--) ord[j] = ord[j - 1];
    ord[j] = x;
  }
}

// one-sided Jacobi SVD of the m x k A (overwritten by U diag(sig)), V right singular vectors, ord by decreasing sig
void svd_jacobi(double* A, int m, int k, double* V, double* sig, int* ord) {
  for (int i = 0; i < k * k; i++) V[i] = (i / k == i % k) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 32; sweep++) {
    bool rotated = false;
    for (int p = 0; p < k - 1; p++)
      for (int q = p + 1; q < k; q++) {
        double al = 0, be = 0, ga = 0;
        for (int r = 0; r < m; r++) {
          al += A[r * k + p] * A[r * k + p];
          be += A[r * k + q] * A[r * k + q];
          ga += A[r * k + p] * A[r * k + q];
        }
        if (!(std::fabs(ga) > 1e-15 * std::sqrt(al * be))) continue;
        const double zeta = (be - al) / (2.0 * ga);
        const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / std::sqrt(1.0 + t * t), s = c * t;
        for (int r = 0; r < m; r++) {
          const double x = A[r * k + p], y = A[r * k + q];
          A[r * k + p] = c * x - s * y;
          A[r * k + q] = s * x + c * y;
        }
        for (int r = 0; r < k; r++) {
          const double x = V[r * k + p], y = V[r * k + q];
          V[r * k + p] = c * x - s * y;
          V[r * k + q] = s * x + c * y;
        }
        rotated = true;
      }
    if (!rotated) break;
  }
  for (int j = 0; j < k; j++) {
    double s2 = 0;
    for (int r = 0; r < m; r++) s2 += A[r * k + j] * A[r * k + j];
    sig[j] = std::sqrt(s2);
  }
  for (int i = 0; i < k; i++) ord[i] = i;
  for (int i = 1; i < k; i++) {
    const int x = ord[i];
    int j = i;
    for (; j > 0 && sig[x] > sig[ord[j - 1]]; j--) ord[j] = ord[j - 1];
    ord[j] = x;
  }
}

// cvSolve(A, b, x, CV_SVD)
void svd_solve(double* A, int m, int k, const double* b, double* x) {
  double V[25], sig[5];
  int ord[5];
  svd_jacobi(A, m, k, V, sig, ord);
  for (int i = 0; i < k; i++) x[i] = 0.0;
  double thr = 0;   // OpenCV's back-substitution skips singular values <= 2 DBL_EPSILON sum(sig)
  for (int jj = 0; jj < k; jj++) thr += sig[ord[jj]];
  thr *= 2 * 2.220446049250313e-16;
  for (int jj = 0; jj < k; jj++) {
    const int j = ord[jj];
    if (std::fabs(sig[j]) <= thr) continue;
    double ub = 0;
    for (int r = 0; r < m; r++) ub += (A[r * k + j] / sig[j]) * b[r];
    const double w = ub / sig[j];
    for (int i = 0; i < k; i++) x[i] += V[i * k + j] * w;
  }
}

struct Epnp {
  double fu, fv, uc, vc;
  int n = 0;
  std::vector<double> pws, us, alphas, pcs;
  double cws[4][3], ccs[4][3];

  void reset() { n = 0; pws.clear(); us.clear(); }
  void add(double X, double Y, double Z, double u, double v) {
    pws.push_back(X); pws.push_back(Y); pws.push_back(Z);
    us.push_back(u); us.push_back(v);
    n++;
  }

  void choose_control_points() {
    for (int j = 0; j < 3; j++) cws[0][j] = 0;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) cws[0][j] += pws[3 * i + j];
    for (int j = 0; j < 3; j++) cws[0][j] /= n;
    std::vector<double> PW0(3 * (size_t)n);
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) PW0[3 * i + j] = pws[3 * i + j] - cws[0][j];
    double A[9], V[9];
    int ord[3];
    for (int a = 0; a < 3; a++)
      for (int b = a; b < 3; b++) {
        double s = 0;
        for (int i = 0; i < n; i++) s += PW0[3 * i + a] * PW0[3 * i + b];
        A[3 * a + b] = A[3 * b + a] = s;
      }
    sym_jacobi(A, V, 3, ord);
    for (int i = 1; i < 4; i++) {
      const int e = ord[i - 1];
      const double d = A[4 * e];
      const double k = std::sqrt((d > 0.0 ? d : 0.0) / n);
      for (int j = 0; j < 3; j++) cws[i][j] = cws[0][j] + k * V[3 * j + e];
    }
  }

  void compute_barycentric_coordinates(double* cci) {
    double CC[9], V[9], sig[3];
    int ord[3];
    for (int i = 0; i < 3; i++)
      for (int j = 1; j < 4; j++) CC[3 * i + j - 1] = cws[j][i] - cws[0][i];
    svd_jacobi(CC, 3, 3, V, sig, ord);
    double thr = 0;   // cvInvert(CV_SVD): singular values <= 2 DBL_EPSILON sum(sig) are skipped (a pseudo-inverse)
    for (int kk = 0; kk < 3; kk++) thr += sig[ord[kk]];
    thr *= 2 * 2.220446049250313e-16;
    for (int i = 0; i < 3; i++)
      for (int r = 0; r < 3; r++) {
        double s = 0;
        for (int kk = 0; kk < 3; kk++) {
          const int c = ord[kk];
          if (std::fabs(sig[c]) <= thr) continue;
          s += V[3 * i + c] * ((CC[3 * r + c] / sig[c]) / sig[c]);
        }
        cci[3 * i + r] = s;
      }
    alphas.assign(4 * (size_t)n, 0.0);
    for (int i = 0; i < n; i++) {
      const double* pi = &pws[3 * i];
      double* a = &alphas[4 * i];
      for (int j = 0; j < 3; j++)
        a[1 + j] = cci[3 * j] * (pi[0] - cws[0][0]) + cci[3 * j + 1] * (pi[1] - cws[0][1]) + cci[3 * j + 2] * (pi[2] - cws[0][2]);
      a[0] = 1.0 - a[1] - a[2] - a[3];
    }
  }

  void fill_M(double* M, int row, const double* as, double u, double v) {
    double* M1 = M + row * 12;
    double* M2 = M1 + 12;
    for (int i = 0; i < 4; i++) {
      M1[3 * i] = as[i] * fu;
      M1[3 * i + 1] = 0.0;
      M1[3 * i + 2] = as[i] * (uc - u);
      M2[3 * i] = 0.0;
      M2[3 * i + 1] = as[i] * fv;
      M2[3 * i + 2] = as[i] * (vc - v);
    }
  }

  void compute_L_6x10(const double* ut, double* l) {
    const double* v[4] = {ut + 12 * 11, ut + 12 * 10, ut + 12 * 9, ut + 12 * 8};
    double dv[4][6][3];
    for (int i = 0; i < 4; i++) {
      int a = 0, b = 1;
      for (int j = 0; j < 6; j++) {
        for (int k = 0; k < 3; k++) dv[i][j][k] = v[i][3 * a + k] - v[i][3 * b + k];
        b++;
        if (b > 3) {
          a++;
          b = a + 1;
        }
      }
    }
    for (int i = 0; i < 6; i++) {
      double* row = l + 10 * i;
      row[0] = dot(dv[0][i], dv[0][i]);
      row[1] = 2 * dot(dv[0][i], dv[1][i]);
      row[2] = dot(dv[1][i], dv[1][i]);
      row[3] = 2 * dot(dv[0][i], dv[2][i]);
      row[4] = 2 * dot(dv[1][i], dv[2][i]);
      row[5] = dot(dv[2][i], dv[2][i]);
      row[6] = 2 * dot(dv[0][i], dv[3][i]);
      row[7] = 2 * dot(dv[1][i], dv[3][i]);
      row[8] = 2 * dot(dv[2][i], dv[3][i]);
      row[9] = dot(dv[3][i], dv[3][i]);
    }
  }

  static double dist2(const double* p1, const double* p2) {
    return (p1[0] - p2[0]) * (p1[0] - p2[0]) + (p1[1] - p2[1]) * (p1[1] - p2[1]) + (p1[2] - p2[2]) * (p1[2] - p2[2]);
  }

  void compute_rho(double* rho) {
    rho[0] = dist2(cws[0], cws[1]);
    rho[1] = dist2(cws[0], cws[2]);
    rho[2] = dist2(cws[0], cws[3]);
    rho[3] = dist2(cws[1], cws[2]);
    rho[4] = dist2(cws[1], cws[3]);
    rho[5] = dist2(cws[2], cws[3]);
  }

  static void find_betas_approx_1(const double* L, const double* rho, double* betas) {
    double A[24], b4[4];
    const int c[4] = {0, 1, 3, 6};
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 4; j++) A[4 * i + j] = L[10 * i + c[j]];
    svd_solve(A, 6, 4, rho, b4);
    if (b4[0] < 0) {
      betas[0] = std::sqrt(-b4[0]);
      betas[1] = -b4[1] / betas[0];
      betas[2] = -b4[2] / betas[0];
      betas[3] = -b4[3] / betas[0];
    } else {
      betas[0] = std::sqrt(b4[0]);
      betas[1] = b4[1] / betas[0];
      betas[2] = b4[2] / betas[0];
      betas[3] = b4[3] / betas[0];
    }
  }

  static void find_betas_approx_2(const double* L, const double* rho, double* betas) {
    double A[18], b3[3];
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 3; j++) A[3 * i + j] = L[10 * i + j];
    svd_solve(A, 6, 3, rho, b3);
    if (b3[0] < 0) {
      betas[0] = std::sqrt(-b3[0]);
      betas[1] = (b3[2] < 0) ? std::sqrt(-b3[2]) : 0.0;
    } else {
      betas[0] = std::sqrt(b3[0]);
      betas[1] = (b3[2] > 0) ? std::sqrt(b3[2]) : 0.0;
    }
    if (b3[1] < 0) betas[0] = -betas[0];
    betas[2] = 0.0;
    betas[3] = 0.0;
  }

  static void find_betas_approx_3(const double* L, const double* rho, double* betas) {
    double A[30], b5[5];
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 5; j++) A[5 * i + j] = L[10 * i + j];
    svd_solve(A, 6, 5, rho, b5);
    if (b5[0] < 0) {
      betas[0] = std::sqrt(-b5[0]);
      betas[1] = (b5[2] < 0) ? std::sqrt(-b5[2]) : 0.0;
    } else {
      betas[0] = std::sqrt(b5[0]);
      betas[1] = (b5[2] > 0) ? std::sqrt(b5[2]) : 0.0;
    }
    if (b5[1] < 0) betas[0] = -betas[0];
    betas[2] = b5[3] / betas[0];
    betas[3] = 0.0;
  }

  static void qr_solve(double* A, double* b, double* X) {
    const int nr = 6, nc = 4;
    double A1[4], A2[4];
    for (int k = 0; k < nc; k++) X[k] = 0.0;
    for (int k = 0; k < nc; k++) {
      double eta = std::fabs(A[k * nc + k]);
      for (int i = k + 1; i < nr; i++) {
        const double elt = std::fabs(A[i * nc + k]);
        if (eta < elt) eta = elt;
      }
      if (eta == 0) return;   // the reference reports a singular A and leaves X as it was
      double sum = 0.0;
      for (int i = k; i < nr; i++) {
        A[i * nc + k] /= eta;
        sum += A[i * nc + k] * A[i * nc + k];
      }
      double sigma = std::sqrt(sum);
      if (A[k * nc + k] < 0) sigma = -sigma;
      A[k * nc + k] += sigma;
      A1[k] = sigma * A[k * nc + k];
      A2[k] = -eta * sigma;
      for (int j = k + 1; j < nc; j++) {
        double s = 0;
        for (int i = k; i < nr; i++) s += A[i * nc + k] * A[i * nc + j];
        const double tau = s / A1[k];
        for (int i = k; i < nr; i++) A[i * nc + j] -= tau * A[i * nc + k];
      }
    }
    for (int j = 0; j < nc; j++) {
      double tau = 0;
      for (int i = j; i < nr; i++) tau += A[i * nc + j] * b[i];
      tau /= A1[j];
      for (int i = j; i < nr; i++) b[i] -= tau * A[i * nc + j];
    }
    X[nc - 1] = b[nc - 1] / A2[nc - 1];
    for (int i = nc - 2; i >= 0; i--) {
      double s = 0;
      for (int j = i + 1; j < nc; j++) s += A[i * nc + j] * X[j];
      X[i] = (b[i] - s) / A2[i];
    }
  }

  static void gauss_newton(const double* L, const double* rho, double* betas) {
    for (int k = 0; k < 5; k++) {
      double A[24], b[6], x[4];
      for (int i = 0; i < 6; i++) {
        const double* rowL = L + 10 * i;
        double* rowA = A + 4 * i;
        rowA[0] = 2 * rowL[0] * betas[0] + rowL[1] * betas[1] + rowL[3] * betas[2] + rowL[6] * betas[3];
        rowA[1] = rowL[1] * betas[0] + 2 * rowL[2] * betas[1] + rowL[4] * betas[2] + rowL[7] * betas[3];
        rowA[2] = rowL[3] * betas[0] + rowL[4] * betas[1] + 2 * rowL[5] * betas[2] + rowL[8] * betas[3];
        rowA[3] = rowL[6] * betas[0] + rowL[7] * betas[1] + rowL[8] * betas[2] + 2 * rowL[9] * betas[3];
        b[i] = rho[i] - (rowL[0] * betas[0] * betas[0] + rowL[1] * betas[0] * betas[1] + rowL[2] * betas[1] * betas[1] +
                         rowL[3] * betas[0] * betas[2] + rowL[4] * betas[1] * betas[2] + rowL[5] * betas[2] * betas[2] +
                         rowL[6] * betas[0] * betas[3] + rowL[7] * betas[1] * betas[3] + rowL[8] * betas[2] * betas[3] +
                         rowL[9] * betas[3] * betas[3]);
      }
      qr_solve(A, b, x);
      for (int i = 0; i < 4; i++) betas[i] += x[i];
    }
  }

  void compute_ccs(const double* betas, const double* ut) {
    for (int i = 0; i < 4; i++) ccs[i][0] = ccs[i][1] = ccs[i][2] = 0.0;
    for (int i = 0; i < 4; i++) {
      const double* v = ut + 12 * (11 - i);
      for (int j = 0; j < 4; j++)
        for (int k = 0; k < 3; k++) ccs[j][k] += betas[i] * v[3 * j + k];
    }
  }

  void compute_pcs() {
    pcs.assign(3 * (size_t)n, 0.0);
    for (int i = 0; i < n; i++) {
      const double* a = &alphas[4 * i];
      double* pc = &pcs[3 * i];
      for (int j = 0; j < 3; j++) pc[j] = a[0] * ccs[0][j] + a[1] * ccs[1][j] + a[2] * ccs[2][j] + a[3] * ccs[3][j];
    }
  }

  void solve_for_sign() {
    if (pcs[2] < 0.0) {
      for (int i = 0; i < 4; i++)
        for (int j = 0; j < 3; j++) ccs[i][j] = -ccs[i][j];
      for (int i = 0; i < n; i++) {
        pcs[3 * i] = -pcs[3 * i];
        pcs[3 * i + 1] = -pcs[3 * i + 1];
        pcs[3 * i + 2] = -pcs[3 * i + 2];
      }
    }
  }

  void estimate_R_and_t(double R[3][3], double t[3]) {
    double pc0[3] = {0, 0, 0}, pw0[3] = {0, 0, 0};
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) {
        pc0[j] += pcs[3 * i + j];
        pw0[j] += pws[3 * i + j];
      }
    for (int j = 0; j < 3; j++) {
      pc0[j] /= n;
      pw0[j] /= n;
    }
    double abt[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n; i++) {
      const double* pc = &pcs[3 * i];
      const double* pw = &pws[3 * i];
      for (int j = 0; j < 3; j++) {
        abt[3 * j] += (pc[j] - pc0[j]) * (pw[0] - pw0[0]);
        abt[3 * j + 1] += (pc[j] - pc0[j]) * (pw[1] - pw0[1]);
        abt[3 * j + 2] += (pc[j] - pc0[j]) * (pw[2] - pw0[2]);
      }
    }
    double V[9], sig[3];
    int ord[3];
    svd_jacobi(abt, 3, 3, V, sig, ord);
    double u[3][3];   // abt_u: u[i][k] = row i of the k-th left singular vector
    for (int i = 0; i < 3; i++)
      for (int k = 0; k < 3; k++) u[i][k] = abt[3 * i + ord[k]] / sig[ord[k]];
    if (sig[ord[2]] <= (sig[ord[0]] + sig[ord[1]] + sig[ord[2]]) * (2 * 2.220446049250313e-16)) {
      // rank 2 (coplanar world points): the third left vector is the cross product of the first two
      u[0][2] = u[1][0] * u[2][1] - u[2][0] * u[1][1];
      u[1][2] = u[2][0] * u[0][1] - u[0][0] * u[2][1];
      u[2][2] = u[0][0] * u[1][1] - u[1][0] * u[0][1];
    }
    for (int i = 0; i < 3; i++) {
      double vr[3];
      for (int j = 0; j < 3; j++) {
        for (int k = 0; k < 3; k++) vr[k] = V[3 * j + ord[k]];
        R[i][j] = dot(u[i], vr);
      }
    }
    const double det = R[0][0] * R[1][1] * R[2][2] + R[0][1] * R[1][2] * R[2][0] + R[0][2] * R[1][0] * R[2][1] -
                       R[0][2] * R[1][1] * R[2][0] - R[0][1] * R[1][0] * R[2][2] - R[0][0] * R[1][2] * R[2][1];
    if (det < 0) {
      R[2][0] = -R[2][0];
      R[2][1] = -R[2][1];
      R[2][2] = -R[2][2];
    }
    t[0] = pc0[0] - dot(R[0], pw0);
    t[1] = pc0[1] - dot(R[1], pw0);
    t[2] = pc0[2] - dot(R[2], pw0);
  }

  double reprojection_error(const double R[3][3], const double t[3]) {
    double sum2 = 0.0;
    for (int i = 0; i < n; i++) {
      const double* pw = &pws[3 * i];
      const double Xc = dot(R[0], pw) + t[0];
      const double Yc = dot(R[1], pw) + t[1];
      const double inv_Zc = 1.0 / (dot(R[2], pw) + t[2]);
      const double ue = uc + fu * Xc * inv_Zc;
      const double ve = vc + fv * Yc * inv_Zc;
      const double u = us[2 * i], v = us[2 * i + 1];
      sum2 += std::sqrt((u - ue) * (u - ue) + (v - ve) * (v - ve));
    }
    return sum2 / n;
  }

  double compute_R_and_t(const double* ut, const double* betas, double R[3][3], double t[3]) {
    compute_ccs(betas, ut);
    compute_pcs();
    solve_for_sign();
    estimate_R_and_t(R, t);
    return reprojection_error(R, t);
  }

  void compute_pose(double R[3][3], double t[3]) {
    choose_control_points();
    double cci[9];
    compute_barycentric_coordinates(cci);
    std::vector<double> M(24 * (size_t)n);
    for (int i = 0; i < n; i++) fill_M(M.data(), 2 * i, &alphas[4 * i], us[2 * i], us[2 * i + 1]);
    double MtM[144], V[144], ut[144];
    int ord[12];
    for (int a = 0; a < 12; a++)
      for (int b = a; b < 12; b++) {
        double s = 0;
        for (int r = 0; r < 2 * n; r++) s += M[12 * r + a] * M[12 * r + b];
        MtM[12 * a + b] = MtM[12 * b + a] = s;
      }
    sym_jacobi(MtM, V, 12, ord);
    for (int r = 0; r < 12; r++)
      for (int k = 0; k < 12; k++) ut[12 * r + k] = V[12 * k + ord[r]];
    double L[60], rho[6];
    compute_L_6x10(ut, L);
    compute_rho(rho);
    double Betas[4][4], rep_errors[4], Rs[4][3][3], ts[4][3];
    find_betas_approx_1(L, rho, Betas[1]);
    gauss_newton(L, rho, Betas[1]);
    rep_errors[1] = compute_R_and_t(ut, Betas[1], Rs[1], ts[1]);
    find_betas_approx_2(L, rho, Betas[2]);
    gauss_newton(L, rho, Betas[2]);
    rep_errors[2] = compute_R_and_t(ut, Betas[2], Rs[2], ts[2]);
    find_betas_approx_3(L, rho, Betas[3]);
    gauss_newton(L, rho, Betas[3]);
    rep_errors[3] = compute_R_and_t(ut, Betas[3], Rs[3], ts[3]);
    int N = 1;
    if (rep_errors[2] < rep_errors[1]) N = 2;
    if (rep_errors[3] < rep_errors[N]) N = 3;
    std::memcpy(R, Rs[N], sizeof(Rs[N]));
    std::memcpy(t, ts[N], sizeof(ts[N]));
  }
};

// PnPsolver::CheckInliers for one correspondence
bool check_one(const double R[3][3], const double t[3], const float* P3Dw, const float* P2D, float maxErr, double fu, double fv,
               double uc, double vc) {
  const float Xc = R[0][0] * P3Dw[0] + R[0][1] * P3Dw[1] + R[0][2] * P3Dw[2] + t[0];
  const float Yc = R[1][0] * P3Dw[0] + R[1][1] * P3Dw[1] + R[1][2] * P3Dw[2] + t[1];
  const float invZc = 1 / (R[2][0] * P3Dw[0] + R[2][1] * P3Dw[1] + R[2][2] * P3Dw[2] + t[2]);
  const double ue = uc + fu * Xc * invZc;
  const double ve = vc + fv * Yc * invZc;
  const float distX = P2D[0] - ue;
  const float distY = P2D[1] - ve;
  const float error2 = distX * distX + distY * distY;
  return error2 < maxErr;
}

struct Solver {
  int N;
  const float *p2d, *p3dw, *maxErr;
  Epnp pnp;
  double mRi[3][3], mti[3];
  std::vector<uint8_t> inl;

  int check_inliers() {
    int c = 0;
    inl.assign((size_t)N, 0);
    for (int i = 0; i < N; i++) {
      inl[i] = check_one(mRi, mti, p3dw + 3 * i, p2d + 2 * i, maxErr[i], pnp.fu, pnp.fv, pnp.uc, pnp.vc);
      c += inl[i];
    }
    return c;
  }
  void add(int idx) { pnp.add(p3dw[3 * idx], p3dw[3 * idx + 1], p3dw[3 * idx + 2], p2d[2 * idx], p2d[2 * idx + 1]); }
};

void to_float_pose(const double R[3][3], const double t[3], float* T) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) T[3 * i + j] = (float)R[i][j];
  for (int i = 0; i < 3; i++) T[9 + i] = (float)t[i];
}

}  // namespace

extern "C" {

int lldo_pnp_ransac(void*, const lld_pnp_ransac_problem* p, lld_pnp_ransac_result* out) {
  if (!p || !out || p->n_problems < 0 || p->n_iterations < 0) return LLD_ERR_ARG;
  for (int pb = 0; pb < p->n_problems; pb++) {
    const int e0 = p->off[pb], N = p->off[pb + 1] - e0;
    const int h0 = p->hyp_off[pb], nh = p->hyp_off[pb + 1] - h0;
    const int minIn = p->min_inliers[pb], maxIts = p->max_its[pb];
    const int budget = N < minIn ? 0 : std::max(p->n_iterations, maxIts - p->its_done[pb]);
    if (nh != budget || minIn < 4 || maxIts < 1) return LLD_ERR_ARG;
    Solver S;
    S.N = N; S.p2d = p->p2d + 2 * e0; S.p3dw = p->p3dw + 3 * e0; S.maxErr = p->max_err + e0;
    S.pnp.fu = p->cam[4 * pb]; S.pnp.fv = p->cam[4 * pb + 1]; S.pnp.uc = p->cam[4 * pb + 2]; S.pnp.vc = p->cam[4 * pb + 3];
    int mnIterations = p->its_done[pb], mnBestInliers = p->best_inliers[pb];
    std::vector<uint8_t> bestMask(p->best_mask + e0, p->best_mask + e0 + N);
    float bestTcw[12];
    std::memcpy(bestTcw, p->best_Tcw + 12 * pb, sizeof(bestTcw));
    if (out->hyp_inliers)
      for (int k = 0; k < nh; k++) out->hyp_inliers[h0 + k] = -1;
    bool found = false, bNoMore = false;
    int nInliers = 0;
    std::vector<uint8_t> retMask((size_t)N, 0);
    float retTcw[12] = {0};
    if (N < minIn) {
      bNoMore = true;
    } else {
      int nCurrent = 0;
      while (mnIterations < maxIts || nCurrent < p->n_iterations) {
        nCurrent++;
        mnIterations++;
        const int32_t* id = p->hyp_idx + 4 * (h0 + nCurrent - 1);
        S.pnp.reset();
        for (int k = 0; k < 4; k++) S.add(id[k]);
        S.pnp.compute_pose(S.mRi, S.mti);
        const int mnInliersi = S.check_inliers();
        if (out->hyp_inliers) out->hyp_inliers[h0 + nCurrent - 1] = mnInliersi;
        if (mnInliersi >= minIn) {
          if (mnInliersi > mnBestInliers) {
            bestMask = S.inl;
            mnBestInliers = mnInliersi;
            to_float_pose(S.mRi, S.mti, bestTcw);
          }
          // Refine()
          S.pnp.reset();
          for (int i = 0; i < N; i++)
            if (bestMask[i]) S.add(i);
          S.pnp.compute_pose(S.mRi, S.mti);
          const int refined = S.check_inliers();
          if (refined > minIn) {
            found = true;
            nInliers = refined;
            retMask = S.inl;
            to_float_pose(S.mRi, S.mti, retTcw);
            break;
          }
        }
      }
      if (!found && mnIterations >= maxIts) {
        bNoMore = true;
        if (mnBestInliers >= minIn) {
          found = true;
          nInliers = mnBestInliers;
          retMask = bestMask;
          std::memcpy(retTcw, bestTcw, sizeof(retTcw));
        }
      }
    }
    out->found[pb] = found;
    out->no_more[pb] = bNoMore;
    out->n_inliers[pb] = nInliers;
    std::memcpy(out->Tcw + 12 * pb, retTcw, sizeof(retTcw));
    for (int i = 0; i < N; i++) out->inlier[e0 + i] = retMask[i];
    out->its_done[pb] = mnIterations;
    out->best_inliers[pb] = mnBestInliers;
    for (int i = 0; i < N; i++) out->best_mask[e0 + i] = bestMask[i];
    std::memcpy(out->best_Tcw + 12 * pb, bestTcw, sizeof(bestTcw));
  }
  return LLD_OK;
}

// PnPsolver::SetRansacParameters' host arithmetic (lld_pnp_ransac_params), for the shim's oracle build
int lldo_pnp_ransac_params(int32_t n_corr, double probability, int32_t min_inliers, int32_t max_iterations, int32_t min_set,
                           float epsilon, int32_t out[2]) {
  if (n_corr < 0 || !out) return LLD_ERR_ARG;
  int nMinInliers = n_corr * epsilon;
  if (nMinInliers < min_inliers) nMinInliers = min_inliers;
  if (nMinInliers < min_set) nMinInliers = min_set;
  if (epsilon < (float)nMinInliers / n_corr) epsilon = (float)nMinInliers / n_corr;
  int nIterations = 1;
  if (nMinInliers != n_corr) {
    const double it = std::ceil(std::log(1 - probability) / std::log(1 - std::pow(epsilon, 3)));
    nIterations = it >= 2147483647.0 ? 2147483647 : (it > -2147483648.0 ? (int)it : -2147483647 - 1);
  }
  out[0] = nMinInliers;
  out[1] = std::max(1, std::min(nIterations, max_iterations));
  return LLD_OK;
}

// pieces for the host build of the device math (tests/hostcheck/devmath_pnp_ransac_host.cpp): EPnP over n correspondences
// (X3 [n][3], uv [n][2], cam fu fv uc vc) -> R (9), t (3) in double; CheckInliers of one correspondence
void lldo_pnp_epnp(const float* X3, const float* uv, int n, const double* cam, double* Rt) {
  Epnp e;
  e.fu = cam[0]; e.fv = cam[1]; e.uc = cam[2]; e.vc = cam[3];
  for (int i = 0; i < n; i++) e.add(X3[3 * i], X3[3 * i + 1], X3[3 * i + 2], uv[2 * i], uv[2 * i + 1]);
  double R[3][3], t[3];
  e.compute_pose(R, t);
  std::memcpy(Rt, R, 9 * sizeof(double));
  std::memcpy(Rt + 9, t, 3 * sizeof(double));
}
int lldo_pnp_inlier(const double* Rt, const float* X, const float* uv, float max_err, const double* cam) {
  double R[3][3];
  std::memcpy(R, Rt, sizeof(R));
  return check_one(R, Rt + 9, X, uv, max_err, cam[0], cam[1], cam[2], cam[3]);
}
void lldo_pnp_sym_jacobi(double* A, double* V, int n, int* ord) { sym_jacobi(A, V, n, ord); }
void lldo_pnp_svd_solve(double* A, int m, int k, const double* b, double* x) { svd_solve(A, m, k, b, x); }

}  // extern "C"
