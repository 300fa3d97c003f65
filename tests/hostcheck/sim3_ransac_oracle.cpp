// CPU oracle of lld_sim3_ransac (include/lldba.h): a plain sequential restatement of ORB-SLAM2's Sim3Solver::iterate,
// ComputeSim3, CheckInliers, Project and FromCameraToImage, in float with the double intermediates of the source (ang, nom,
// den, the dot products) and cv::gemm's rounding for the small CV_32F products (see the header).  The eigen solver is the
// library's cyclic Jacobi (the contract does not ask for OpenCV's bits there).  Test infrastructure: built by
// __graft_entry__.build() into libsim3_ransac_oracle.so and bound by capi.load_oracle(); tests/test_sim3_ransac.py pins it
// with an independent Python transcription that calls cv2.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/lldba.h"

namespace {

typedef float Mat3[3][3];

// cv::gemm, 3-long, no transposition: float products summed in float, then s0 * alpha + c * beta in double, rounded once
float gemm_row(const float* a, const float* b, int bstride) {
  float s0 = a[0] * b[0];
  s0 = s0 + a[1] * b[bstride];
  s0 = s0 + a[2] * b[2 * bstride];
  return s0;
}

void eigen_top(const float N[4][4], float q[4]) {
  double A[4][4], V[4][4];
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) {
      A[i][j] = N[i][j];
      V[i][j] = i == j;
    }
  for (int sweep = 0; sweep < 32; sweep++) {
    double off = 0, dia = 0;
    for (int i = 0; i < 4; i++) {
      dia += std::fabs(A[i][i]);
      for (int j = i + 1; j < 4; j++) off += std::fabs(A[i][j]);
    }
    if (!(off > 1e-15 * dia)) break;
    for (int p = 0; p < 3; p++)
      for (int r = p + 1; r < 4; r++) {
        if (A[p][r] == 0.0) continue;
        const double theta = (A[r][r] - A[p][p]) / (2.0 * A[p][r]);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 4; k++) {
          const double x = A[k][p], y = A[k][r];
          A[k][p] = c * x - s * y;
          A[k][r] = s * x + c * y;
        }
        for (int k = 0; k < 4; k++) {
          const double x = A[p][k], y = A[r][k];
          A[p][k] = c * x - s * y;
          A[r][k] = s * x + c * y;
        }
        for (int k = 0; k < 4; k++) {
          const double x = V[k][p], y = V[k][r];
          V[k][p] = c * x - s * y;
          V[k][r] = s * x + c * y;
        }
      }
  }
  int im = 0;
  for (int i = 1; i < 4; i++)
    if (A[i][i] > A[im][im]) im = i;
  for (int i = 0; i < 4; i++) q[i] = (float)V[i][im];
}

void rodrigues(const float v[3], Mat3 R) {
  double r[3] = {v[0], v[1], v[2]};
  const double theta = std::sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  if (theta < 2.220446049250313e-16) {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) R[i][j] = i == j ? 1.f : 0.f;
    return;
  }
  const double c = std::cos(theta), s = std::sin(theta), c1 = 1. - c;
  const double itheta = 1. / theta;
  for (double& x : r) x *= itheta;
  const double rx[3][3] = {{0, -r[2], r[1]}, {r[2], 0, -r[0]}, {-r[1], r[0], 0}};
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) R[i][j] = (float)((c * (i == j) + c1 * (r[i] * r[j])) + s * rx[i][j]);
}

struct Estimate {
  Mat3 R;
  float t[3], s;
  Mat3 sR, sRinv;
  float tinv[3];
};

// Sim3Solver::ComputeSim3(P1, P2): P[coordinate][point]
void compute_sim3(const Mat3 P1, const Mat3 P2, bool fix_scale, Estimate& E) {
  float O1[3], O2[3];
  Mat3 Pr1, Pr2;
  for (int r = 0; r < 3; r++) {
    O1[r] = (P1[r][0] + P1[r][1] + P1[r][2]) * (float)(1.0 / 3);
    O2[r] = (P2[r][0] + P2[r][1] + P2[r][2]) * (float)(1.0 / 3);
    for (int k = 0; k < 3; k++) {
      Pr1[r][k] = P1[r][k] - O1[r];
      Pr2[r][k] = P2[r][k] - O2[r];
    }
  }
  Mat3 M;   // Pr2 * Pr1.t()
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double acc = 0;
      for (int k = 0; k < 3; k++) acc += (double)Pr2[i][k] * Pr1[j][k];
      M[i][j] = (float)acc;
    }
  float N11 = M[0][0] + M[1][1] + M[2][2];
  float N12 = M[1][2] - M[2][1];
  float N13 = M[2][0] - M[0][2];
  float N14 = M[0][1] - M[1][0];
  float N22 = M[0][0] - M[1][1] - M[2][2];
  float N23 = M[0][1] + M[1][0];
  float N24 = M[2][0] + M[0][2];
  float N33 = -M[0][0] + M[1][1] - M[2][2];
  float N34 = M[1][2] + M[2][1];
  float N44 = -M[0][0] - M[1][1] + M[2][2];
  const float N[4][4] = {{N11, N12, N13, N14}, {N12, N22, N23, N24}, {N13, N23, N33, N34}, {N14, N24, N34, N44}};
  float evec[4];
  eigen_top(N, evec);
  float vec[3] = {evec[1], evec[2], evec[3]};
  const double nv = std::sqrt(((double)vec[0] * vec[0] + (double)vec[2] * vec[2]) + (double)vec[1] * vec[1]);   // cv::norm
  const double ang = std::atan2(nv, (double)evec[0]);
  const double alpha = 2 * ang * (1. / nv);
  for (float& x : vec) x = (float)(alpha * x);
  rodrigues(vec, E.R);
  if (!fix_scale) {
    Mat3 P3;   // mR12i * Pr2
    for (int i = 0; i < 3; i++)
      for (int k = 0; k < 3; k++) P3[i][k] = gemm_row(E.R[i], &Pr2[0][k], 3);
    double nom = 0, den = 0;
    for (int i = 0; i < 3; i++)
      for (int k = 0; k < 3; k++) nom += (double)Pr1[i][k] * P3[i][k];
    for (int i = 0; i < 3; i++)
      for (int k = 0; k < 3; k++) {
        const float sq = P3[i][k] * P3[i][k];   // cv::pow(P3, 2)
        den += sq;
      }
    E.s = (float)(nom / den);
  } else {
    E.s = 1.0f;
  }
  for (int r = 0; r < 3; r++) E.t[r] = (float)((double)gemm_row(E.R[r], O2, 1) * (-(double)E.s) + (double)O1[r]);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      E.sR[i][j] = E.s * E.R[i][j];
      E.sRinv[i][j] = (float)((1.0 / E.s) * E.R[j][i]);
    }
  for (int r = 0; r < 3; r++) E.tinv[r] = (float)((double)gemm_row(E.sRinv[r], E.t, 1) * -1.0);
}

void project(const float X[3], const Mat3 Rcw, const float tcw[3], const float* K, float uv[2]) {
  float P[3];
  for (int r = 0; r < 3; r++) P[r] = (float)((double)gemm_row(Rcw[r], X, 1) + (double)tcw[r]);
  const float invz = 1 / P[2];
  const float x = P[0] * invz;
  const float y = P[1] * invz;
  uv[0] = K[0] * x + K[2];
  uv[1] = K[1] * y + K[3];
}

void to_image(const float X[3], const float* K, float uv[2]) {
  const float invz = 1 / X[2];
  const float x = X[0] * invz;
  const float y = X[1] * invz;
  uv[0] = K[0] * x + K[2];
  uv[1] = K[1] * y + K[3];
}

float dot2(const float a[2], const float b[2]) {
  const float d[2] = {a[0] - b[0], a[1] - b[1]};
  double r = 0;
  r += (double)d[0] * d[0];
  r += (double)d[1] * d[1];
  return (float)r;
}

struct Solver {
  int N;
  const float *K, *x1, *x2;
  std::vector<size_t> maxErr1, maxErr2;
  std::vector<float> P1im1, P2im2;
  bool fix;
  void init(const float* cam, int fixs, const float* x1c, const float* x2c, const float* s1, const float* s2, int n) {
    N = n; K = cam; x1 = x1c; x2 = x2c; fix = fixs != 0;
    for (int i = 0; i < n; i++) {
      maxErr1.push_back((size_t)(9.210 * s1[i]));
      maxErr2.push_back((size_t)(9.210 * s2[i]));
      float a[2], b[2];
      to_image(x1 + 3 * i, K, a);
      to_image(x2 + 3 * i, K + 4, b);
      P1im1.push_back(a[0]); P1im1.push_back(a[1]);
      P2im2.push_back(b[0]); P2im2.push_back(b[1]);
    }
  }
  int check_inliers(const Estimate& E, uint8_t* inl) const {
    int n_in = 0;
    for (int i = 0; i < N; i++) {
      float p21[2], p12[2];
      project(x2 + 3 * i, E.sR, E.t, K, p21);
      project(x1 + 3 * i, E.sRinv, E.tinv, K + 4, p12);
      const float err1 = dot2(&P1im1[2 * i], p21);
      const float err2 = dot2(p12, &P2im2[2 * i]);
      const bool in = err1 < maxErr1[i] && err2 < maxErr2[i];
      if (inl) inl[i] = in;
      n_in += in;
    }
    return n_in;
  }
};

}  // namespace

extern "C" {

int lldo_sim3_ransac(void*, const lld_sim3_ransac_problem* p, lld_sim3_ransac_result* out) {
  if (!p || !out || p->n_problems < 0 || p->min_inliers < 0 || p->n_iterations < 0) return LLD_ERR_ARG;
  for (int pb = 0; pb < p->n_problems; pb++) {
    const int e0 = p->off[pb], N = p->off[pb + 1] - e0;
    const int h0 = p->hyp_off[pb], nh = p->hyp_off[pb + 1] - h0;
    const int budget = N < p->min_inliers ? 0 : std::min(p->n_iterations, std::max(0, p->max_its[pb] - p->its_done[pb]));
    if (nh != budget) return LLD_ERR_ARG;
    Solver S;
    S.init(p->cam + 8 * pb, p->fix_scale[pb], p->x1c + 3 * e0, p->x2c + 3 * e0, p->sigma2_1 + e0, p->sigma2_2 + e0, N);
    int mnIterations = p->its_done[pb], mnBestInliers = p->best_inliers[pb];
    if (out->hyp_inliers)
      for (int k = 0; k < nh; k++) out->hyp_inliers[h0 + k] = -1;
    for (int i = 0; i < N; i++) out->inlier[e0 + i] = 0;
    for (int k = 0; k < 13; k++) out->T12[13 * pb + k] = 0.f;
    bool bNoMore = false, found = false;
    int nInliers = 0;
    if (N < p->min_inliers) {
      bNoMore = true;
    } else {
      int nCurrentIterations = 0;
      while (mnIterations < p->max_its[pb] && nCurrentIterations < p->n_iterations) {
        nCurrentIterations++;
        mnIterations++;
        const int32_t* id = p->hyp_idx + 3 * (h0 + nCurrentIterations - 1);
        Mat3 P1, P2;
        for (int c = 0; c < 3; c++)
          for (int r = 0; r < 3; r++) {
            P1[r][c] = S.x1[3 * id[c] + r];
            P2[r][c] = S.x2[3 * id[c] + r];
          }
        Estimate E;
        compute_sim3(P1, P2, S.fix, E);
        const int mnInliersi = S.check_inliers(E, nullptr);
        if (out->hyp_inliers) out->hyp_inliers[h0 + nCurrentIterations - 1] = mnInliersi;
        if (mnInliersi >= mnBestInliers) {
          mnBestInliers = mnInliersi;
          if (mnInliersi > p->min_inliers) {
            found = true;
            nInliers = mnInliersi;
            S.check_inliers(E, out->inlier + e0);
            float* T = out->T12 + 13 * pb;
            for (int i = 0; i < 3; i++)
              for (int j = 0; j < 3; j++) T[3 * i + j] = E.R[i][j];
            for (int r = 0; r < 3; r++) T[9 + r] = E.t[r];
            T[12] = E.s;
            break;
          }
        }
      }
      if (!found && mnIterations >= p->max_its[pb]) bNoMore = true;
    }
    out->found[pb] = found;
    out->no_more[pb] = bNoMore;
    out->n_inliers[pb] = nInliers;
    out->its_done[pb] = mnIterations;
    out->best_inliers[pb] = mnBestInliers;
  }
  return LLD_OK;
}

// pieces for the host build of the device math (tests/hostcheck/devmath_sim3_ransac_host.cpp): P1, P2 point-major
// ([k][3]); out = R (9), t (3), s
void lldo_sim3r_horn(const float* P1, const float* P2, int fix_scale, float* out) {
  Mat3 A, B;
  for (int k = 0; k < 3; k++)
    for (int r = 0; r < 3; r++) {
      A[r][k] = P1[3 * k + r];
      B[r][k] = P2[3 * k + r];
    }
  Estimate E;
  compute_sim3(A, B, fix_scale != 0, E);
  std::memcpy(out, E.R, 9 * sizeof(float));
  std::memcpy(out + 9, E.t, 3 * sizeof(float));
  out[12] = E.s;
}
void lldo_sym4_top_eigvec(const float* N, float* q) {
  float A[4][4];
  std::memcpy(A, N, sizeof(A));
  eigen_top(A, q);
}
void lldo_rodrigues(const float* v, float* R) { rodrigues(v, reinterpret_cast<float(*)[3]>(R)); }
// err1, err2 of one correspondence under the estimate est (R, t, s); returns the inlier flag
int lldo_sim3r_errors(const float* est, const float* cam, const float* x1, const float* x2, float s1, float s2, float* err) {
  Estimate E;
  std::memcpy(E.R, est, 9 * sizeof(float));
  std::memcpy(E.t, est + 9, 3 * sizeof(float));
  E.s = est[12];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      E.sR[i][j] = E.s * E.R[i][j];
      E.sRinv[i][j] = (float)((1.0 / E.s) * E.R[j][i]);
    }
  for (int r = 0; r < 3; r++) E.tinv[r] = (float)((double)gemm_row(E.sRinv[r], E.t, 1) * -1.0);
  float a[2], b[2], p21[2], p12[2];
  to_image(x1, cam, a);
  to_image(x2, cam + 4, b);
  project(x2, E.sR, E.t, cam, p21);
  project(x1, E.sRinv, E.tinv, cam + 4, p12);
  err[0] = dot2(a, p21);
  err[1] = dot2(p12, b);
  return err[0] < (size_t)(9.210 * s1) && err[1] < (size_t)(9.210 * s2);
}

}  // extern "C"
