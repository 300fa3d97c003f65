// lld_math.cuh — device math of the point+line BA kernels (sm_100a).
//
// Every function is __host__ __device__ so that tests/ can compile this header with g++ and check the
// arithmetic against the CPU oracle before any GPU time is spent (tests/test_device_math_host.py).
// The formulas are closed-form re-derivations, not transcriptions, of the g2o edge types
// (reference: Thirdparty/g2o/g2o/types/types_six_dof_expmap.{h,cpp}, types_sba.{h,cpp}, se3quat.h):
//
//  * point edges use the camera-frame point once and build both Jacobians from shared sub-terms;
//  * line edges use (K a) x (K b) = cof(K) (a x b): with m = P1 x P2 (camera-frame points incl. baseline shift)
//        l~ = cof(K) m ,  n = f * hypot(m0, m1) ,  r_i = (u~_i m0 + v~_i m1 + f w_i m2) / hypot(m0, m1)
//    (u~ = u - cx w, v~ = v - cy w), and the chain rule through the triple products
//        g_i = (x_i - r_i (l0, l1, 0)) / n ,   h1 = K^T (g_i x A1) ,  h2 = K^T (g_i x A2)
//        d r_i / d omega   = X2m x h1 - X1m x h2        d r_i / d upsilon = h1 - h2
//        d r_i / d delta_r = 2 (X2 x k1 - X1 x k2)      d r_i / d alpha   = r2 . (k1 - k2) ,  k = R_cam^T h
//    which equals FormJacobianLineWRTCam / EdgeSE3ProjectLine::linearize (.cpp:472-553) term by term.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define LLD_HD __host__ __device__ __forceinline__
#else
#define LLD_HD inline
#endif

namespace lld {

LLD_HD void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
LLD_HD double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// ---- quaternion (x y z w) / rotation ---------------------------------------------------------
LLD_HD void quat_to_R(const double* q, double* R) {
  const double tx = 2 * q[0], ty = 2 * q[1], tz = 2 * q[2];
  const double twx = tx * q[3], twy = ty * q[3], twz = tz * q[3];
  const double txx = tx * q[0], txy = ty * q[0], txz = tz * q[0];
  const double tyy = ty * q[1], tyz = tz * q[1], tzz = tz * q[2];
  R[0] = 1 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
  R[3] = txy + twz; R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1 - (txx + tyy);
}
LLD_HD void quat_from_R(const double* m, double* q) {  // Eigen Quaterniond(Matrix3d) branch structure
  double t = m[0] + m[4] + m[8];
  if (t > 0.0) {
    t = sqrt(t + 1.0);
    q[3] = 0.5 * t;
    t = 0.5 / t;
    q[0] = (m[7] - m[5]) * t; q[1] = (m[2] - m[6]) * t; q[2] = (m[3] - m[1]) * t;
  } else {
    int i = 0;
    if (m[4] > m[0]) i = 1;
    if (m[8] > m[4 * i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrt(m[4 * i] - m[4 * j] - m[4 * k] + 1.0);
    double qq[4];
    qq[i] = 0.5 * t;
    t = 0.5 / t;
    qq[3] = (m[3 * k + j] - m[3 * j + k]) * t;
    qq[j] = (m[3 * j + i] + m[3 * i + j]) * t;
    qq[k] = (m[3 * k + i] + m[3 * i + k]) * t;
    q[0] = qq[0]; q[1] = qq[1]; q[2] = qq[2]; q[3] = qq[3];
  }
}
LLD_HD void quat_mul(const double* a, const double* b, double* o) {
  const double w = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
  const double x = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
  const double y = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
  const double z = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z; o[3] = w;
}
LLD_HD void quat_normalize_pos(double* q) {  // SE3Quat::normalizeRotation  se3quat.h:280-285
  double s = 1.0 / sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (q[3] < 0) s = -s;
  q[0] *= s; q[1] *= s; q[2] *= s; q[3] *= s;
}
LLD_HD void quat_rot(const double* q, const double* v, double* o) {
  double uv[3], c2[3];
  cross3(q, v, uv);
  uv[0] += uv[0]; uv[1] += uv[1]; uv[2] += uv[2];
  cross3(q, uv, c2);
  o[0] = v[0] + q[3] * uv[0] + c2[0];
  o[1] = v[1] + q[3] * uv[1] + c2[1];
  o[2] = v[2] + q[3] * uv[2] + c2[2];
}

// Pose stored as q[4] (x y z w), t[3].  qt = 7 doubles.
// VertexSE3Expmap::oplusImpl: T <- exp(u) * T   (types_six_dof_expmap.h:76-79, se3quat.h:104-110,223-257)
LLD_HD void pose_oplus(const double* qt, const double* u, double* out) {
  const double wx = u[0], wy = u[1], wz = u[2];
  const double theta = sqrt(wx * wx + wy * wy + wz * wz);
  // Omega = skew(w), Omega^2 = w w^T - theta^2 I
  double a, b, c;
  if (theta < 0.00001) {  // R = I + Omega + Omega^2 ; V = R   (the reference's small-angle branch, sic)
    a = 1.0; b = 1.0; c = 1.0;
  } else {
    const double s = sin(theta), co = cos(theta);
    a = s / theta;
    b = (1 - co) / (theta * theta);
    c = (theta - s) / (theta * theta * theta);
  }
  const double O2[9] = {-(wy * wy + wz * wz), wx * wy, wx * wz, wx * wy, -(wx * wx + wz * wz), wy * wz,
                        wx * wz, wy * wz, -(wx * wx + wy * wy)};
  const double O[9] = {0, -wz, wy, wz, 0, -wx, -wy, wx, 0};
  double R[9], V[9];
  const double vb = (theta < 0.00001) ? 1.0 : b;  // V's Omega coefficient
#pragma unroll
  for (int i = 0; i < 9; i++) {
    const double id = (i == 0 || i == 4 || i == 8) ? 1.0 : 0.0;
    R[i] = id + a * O[i] + b * O2[i];
    V[i] = id + vb * O[i] + c * O2[i];
  }
  double qd[4], td[3];
  quat_from_R(R, qd);
  quat_normalize_pos(qd);
  td[0] = V[0] * u[3] + V[1] * u[4] + V[2] * u[5];
  td[1] = V[3] * u[3] + V[4] * u[4] + V[5] * u[5];
  td[2] = V[6] * u[3] + V[7] * u[4] + V[8] * u[5];
  double rt[3];
  quat_rot(qd, qt + 4, rt);
  double qo[4];
  quat_mul(qd, qt, qo);
  quat_normalize_pos(qo);
  out[0] = qo[0]; out[1] = qo[1]; out[2] = qo[2]; out[3] = qo[3];
  out[4] = td[0] + rt[0]; out[5] = td[1] + rt[1]; out[6] = td[2] + rt[2];
}
// SE3Quat(R,t): Converter::toSE3Quat  src/Converter.cc:37-47
LLD_HD void pose_from_Rt(const double* Rt, double* qt) {
  quat_from_R(Rt, qt);
  quat_normalize_pos(qt);
  qt[4] = Rt[9]; qt[5] = Rt[10]; qt[6] = Rt[11];
}
LLD_HD void pose_to_Rt(const double* qt, double* Rt) {
  quat_to_R(qt, Rt);
  Rt[9] = qt[4]; Rt[10] = qt[5]; Rt[11] = qt[6];
}
LLD_HD void map_Rt(const double* Rt, const double* X, double* o) {
  o[0] = Rt[0] * X[0] + Rt[1] * X[1] + Rt[2] * X[2] + Rt[9];
  o[1] = Rt[3] * X[0] + Rt[4] * X[1] + Rt[5] * X[2] + Rt[10];
  o[2] = Rt[6] * X[0] + Rt[7] * X[1] + Rt[8] * X[2] + Rt[11];
}

// ---- line vertex: state = q[4] (un-normalised) + alpha ---------------------------------------
// LineOptimizer::AddLineMinimal  src/LineOptimizer.cc:44-50
LLD_HD void line_from_x0_dir(const double* x0, const double* dir, double* st) {
  const double n = sqrt(dot3(x0, x0));
  double c[3];
  cross3(dir, x0, c);
  const double in = 1.0 / n;
  const double R[9] = {dir[0], x0[0] * in, c[0] * in, dir[1], x0[1] * in, c[1] * in, dir[2], x0[2] * in, c[2] * in};
  quat_from_R(R, st);
  st[4] = n;
}
// r1 = R[:,0] (direction), r2 = R[:,1] of normalized(q)
LLD_HD void line_axes(const double* st, double* r1, double* r2) {
  const double s = 1.0 / sqrt(st[0] * st[0] + st[1] * st[1] + st[2] * st[2] + st[3] * st[3]);
  const double q[4] = {st[0] * s, st[1] * s, st[2] * s, st[3] * s};
  double R[9];
  quat_to_R(q, R);
  r1[0] = R[0]; r1[1] = R[3]; r1[2] = R[6];
  r2[0] = R[1]; r2[1] = R[4]; r2[2] = R[7];
}
// VertexSBALine::oplusImpl  types_sba.h:95-108 (NaN when |u[0:3]| > 1, exactly like the reference)
LLD_HD void line_oplus(const double* st, const double* u, double* out) {
  const double s = 1.0 / sqrt(st[0] * st[0] + st[1] * st[1] + st[2] * st[2] + st[3] * st[3]);
  const double qn[4] = {st[0] * s, st[1] * s, st[2] * s, st[3] * s};
  const double qr[4] = {u[0], u[1], u[2], sqrt(1.0 - (u[0] * u[0] + u[1] * u[1] + u[2] * u[2]))};
  quat_mul(qr, qn, out);
  out[4] = st[4] + u[3];
}

// ---- robust kernel -----------------------------------------------------------------------------
// RobustKernelHuber::robustify  robust_kernel_impl.cpp:78-91 : returns rho(e), sets w = rho'(e)
LLD_HD double huber(double e, double delta, double* w) {
  const double dsqr = delta * delta;
  if (e <= dsqr) {
    *w = 1.0;
    return e;
  }
  const double sqrte = sqrt(e);
  *w = delta / sqrte;
  return 2 * sqrte * delta - dsqr;
}

// ---- point edges -------------------------------------------------------------------------------
// residual only.  stereo residual mirrors the float `invz` (and, for the binary edge, the float `bf`) of
// EdgeStereoSE3ProjectXYZ::cam_project (.cpp:158-165) / ...OnlyPose::cam_project (.cpp:307-314).
template <bool BF_FLOAT>
LLD_HD void pt_residual(const double* xc, const double* intr, const float* obs, bool stereo, double* err) {
  if (stereo) {
    const float invz = (float)(1.0 / xc[2]);
    const double r0 = xc[0] * (double)invz * intr[0] + intr[2];
    const double r1 = xc[1] * (double)invz * intr[1] + intr[3];
    double bfz;
    if (BF_FLOAT) {
#if defined(__CUDA_ARCH__)
      bfz = (double)__fmul_rn((float)intr[4], invz);
#else
      volatile float prod = (float)intr[4] * invz;
      bfz = (double)prod;
#endif
    } else {
      bfz = intr[4] * (double)invz;
    }
    err[0] = (double)obs[0] - r0;
    err[1] = (double)obs[1] - r1;
    err[2] = (double)obs[2] - (r0 - bfz);
  } else {
    const double p0 = xc[0] / xc[2], p1 = xc[1] / xc[2];
    err[0] = (double)obs[0] - (p0 * intr[0] + intr[2]);
    err[1] = (double)obs[1] - (p1 * intr[1] + intr[3]);
    err[2] = 0.0;
  }
}
// d err / d pose (rows 0..2 x 6), shared by the binary (.cpp:134-146,222-241) and unary (.cpp:283-295,352-371) edges
LLD_HD void pt_jac_pose(const double* xc, const double* intr, bool stereo, double* Jp) {
  const double x = xc[0], y = xc[1];
  const double iz = 1.0 / xc[2], iz2 = iz * iz;
  const double fx = intr[0], fy = intr[1], bf = intr[4];
  Jp[0] = x * y * iz2 * fx;
  Jp[1] = -(1 + x * x * iz2) * fx;
  Jp[2] = y * iz * fx;
  Jp[3] = -iz * fx;
  Jp[4] = 0;
  Jp[5] = x * iz2 * fx;
  Jp[6] = (1 + y * y * iz2) * fy;
  Jp[7] = -x * y * iz2 * fy;
  Jp[8] = -x * iz * fy;
  Jp[9] = 0;
  Jp[10] = -iz * fy;
  Jp[11] = y * iz2 * fy;
  if (stereo) {
    Jp[12] = Jp[0] - bf * y * iz2;
    Jp[13] = Jp[1] + bf * x * iz2;
    Jp[14] = Jp[2];
    Jp[15] = Jp[3];
    Jp[16] = 0;
    Jp[17] = Jp[5] - bf * iz2;
  } else {
    Jp[12] = Jp[13] = Jp[14] = Jp[15] = Jp[16] = Jp[17] = 0;
  }
}
// d err / d point (rows 0..2 x 3)  (.cpp:123-132 mono, :210-220 stereo)
LLD_HD void pt_jac_point(const double* xc, const double* R, const double* intr, bool stereo, double* Jl) {
  const double iz = 1.0 / xc[2], iz2 = iz * iz;
  const double fx = intr[0], fy = intr[1], bf = intr[4];
  const double ax = fx * xc[0] * iz2, ay = fy * xc[1] * iz2;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    Jl[c] = -fx * R[c] * iz + ax * R[6 + c];
    Jl[3 + c] = -fy * R[3 + c] * iz + ay * R[6 + c];
    Jl[6 + c] = stereo ? (Jl[c] - bf * R[6 + c] * iz2) : 0.0;
  }
}

// ---- line edges --------------------------------------------------------------------------------
struct LineObs {   // one endpoint pair already in the space the edge uses (pixel-homogeneous or K^-1-normalised)
  double x1[3], x2[3];
};
// residual of one image (left: bx = 0, right: bx = -baseline).  P1,P2: camera-frame points WITHOUT the shift.
LLD_HD void line_residual(const double* P1, const double* P2, double f, double cx, double cy, double bx,
                          const LineObs& o, double* err) {
  const double a[3] = {P1[0] + bx, P1[1], P1[2]}, b[3] = {P2[0] + bx, P2[1], P2[2]};
  double m[3];
  cross3(a, b, m);
  const double hn = sqrt(m[0] * m[0] + m[1] * m[1]);
  const double ih = 1.0 / hn;
  err[0] = ((o.x1[0] - cx * o.x1[2]) * m[0] + (o.x1[1] - cy * o.x1[2]) * m[1] + f * o.x1[2] * m[2]) * ih;
  err[1] = ((o.x2[0] - cx * o.x2[2]) * m[0] + (o.x2[1] - cy * o.x2[2]) * m[1] + f * o.x2[2] * m[2]) * ih;
}
// residual + pose Jacobian (2x6) and, when WITH_LINE, line Jacobian (2x4).
// Rcam: camera rotation (row-major); X1,X2: world-frame line points, r2: world-frame R_l[:,1].
template <bool WITH_LINE>
LLD_HD void line_linearize(const double* P1, const double* P2, double f, double cx, double cy, double bx,
                           const LineObs& o, const double* Rcam, const double* X1, const double* X2,
                           const double* r2, double* err, double* Jp, double* Jl) {
  const double a[3] = {P1[0] + bx, P1[1], P1[2]}, b[3] = {P2[0] + bx, P2[1], P2[2]};
  double m[3];
  cross3(a, b, m);
  const double hn = sqrt(m[0] * m[0] + m[1] * m[1]);
  const double ih = 1.0 / hn;
  // l = l~/n with l~ = cof(K) m, n = f*hn
  const double l0 = m[0] * ih, l1 = m[1] * ih;
  const double n_inv = ih / f;
  // A_k = K (P_k + b)
  const double A1[3] = {f * a[0] + cx * a[2], f * a[1] + cy * a[2], a[2]};
  const double A2[3] = {f * b[0] + cx * b[2], f * b[1] + cy * b[2], b[2]};
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const double* x = i == 0 ? o.x1 : o.x2;
    const double r = ((x[0] - cx * x[2]) * m[0] + (x[1] - cy * x[2]) * m[1] + f * x[2] * m[2]) * ih;
    err[i] = r;
    const double g[3] = {(x[0] - r * l0) * n_inv, (x[1] - r * l1) * n_inv, x[2] * n_inv};
    double c1[3], c2[3];
    cross3(g, A1, c1);
    cross3(g, A2, c2);
    // h = K^T c
    const double h1[3] = {f * c1[0], f * c1[1], cx * c1[0] + cy * c1[1] + c1[2]};
    const double h2[3] = {f * c2[0], f * c2[1], cx * c2[0] + cy * c2[1] + c2[2]};
    double w1[3], w2[3];
    cross3(P2, h1, w1);
    cross3(P1, h2, w2);
    double* J = Jp + 6 * i;
    J[0] = w1[0] - w2[0]; J[1] = w1[1] - w2[1]; J[2] = w1[2] - w2[2];
    J[3] = h1[0] - h2[0]; J[4] = h1[1] - h2[1]; J[5] = h1[2] - h2[2];
    if (WITH_LINE) {
      // k = Rcam^T h
      const double k1[3] = {Rcam[0] * h1[0] + Rcam[3] * h1[1] + Rcam[6] * h1[2],
                            Rcam[1] * h1[0] + Rcam[4] * h1[1] + Rcam[7] * h1[2],
                            Rcam[2] * h1[0] + Rcam[5] * h1[1] + Rcam[8] * h1[2]};
      const double k2[3] = {Rcam[0] * h2[0] + Rcam[3] * h2[1] + Rcam[6] * h2[2],
                            Rcam[1] * h2[0] + Rcam[4] * h2[1] + Rcam[7] * h2[2],
                            Rcam[2] * h2[0] + Rcam[5] * h2[1] + Rcam[8] * h2[2]};
      double v1[3], v2[3];
      cross3(X2, k1, v1);
      cross3(X1, k2, v2);
      double* L = Jl + 4 * i;
      L[0] = 2 * (v1[0] - v2[0]); L[1] = 2 * (v1[1] - v2[1]); L[2] = 2 * (v1[2] - v2[2]);
      L[3] = r2[0] * (k1[0] - k2[0]) + r2[1] * (k1[1] - k2[1]) + r2[2] * (k1[2] - k2[2]);
    }
  }
}
// EdgeSE3ProjectLine::IsDepthPositive (.h:312-342) + vgl::ReprojectLinePointTo3D (src/vgl.cc:336-346):
// least squares [ (px,py,1) | -K ld ] (depth, s) = K X0 ; closed form through the 2x2 normal equations.
// X0c: camera-frame X0 (incl. shift), ldc: camera-frame direction.
LLD_HD bool line_depth_positive(const double* X0c, const double* ldc, double f, double cx, double cy,
                                const double* x1, const double* x2) {
  const double y[3] = {f * X0c[0] + cx * X0c[2], f * X0c[1] + cy * X0c[2], X0c[2]};
  const double c[3] = {-(f * ldc[0] + cx * ldc[2]), -(f * ldc[1] + cy * ldc[2]), -ldc[2]};
  const double cc = dot3(c, c), cy_ = dot3(c, y);
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const double* x = i == 0 ? x1 : x2;
    const double a[3] = {x[0], x[1], 1.0};
    const double aa = dot3(a, a), ac = dot3(a, c), ay = dot3(a, y);
    const double det = aa * cc - ac * ac;
    const double depth = (cc * ay - ac * cy_) / det;
    if (depth < 0) ok = false;
  }
  return ok;
}

// ---- Sim3 (g2o::Sim3 of ORB-SLAM2's vendored g2o, types/sim3.h) -----------------------------------
// State S[8] = q (x y z w), t[3], s.  Every expression follows the source's evaluation order (Eigen evaluates the
// 3x3 products coefficient-wise, k = 0..2 left to right), so that the host build of this header, the CPU oracle and
// the kernel agree to the bit wherever no transcendental function is involved.
LLD_HD void sim3_map(const double* S, const double* x, double* o) {  // s * (r * x) + t
  double rx[3];
  quat_rot(S, x, rx);
  o[0] = S[7] * rx[0] + S[4];
  o[1] = S[7] * rx[1] + S[5];
  o[2] = S[7] * rx[2] + S[6];
}
LLD_HD void sim3_mul(const double* A, const double* B, double* O) {  // (r_A r_B, s_A (r_A t_B) + t_A, s_A s_B)
  double q[4], rt[3];
  quat_mul(A, B, q);
  quat_rot(A, B + 4, rt);
  O[0] = q[0]; O[1] = q[1]; O[2] = q[2]; O[3] = q[3];
  O[4] = A[7] * rt[0] + A[4];
  O[5] = A[7] * rt[1] + A[5];
  O[6] = A[7] * rt[2] + A[6];
  O[7] = A[7] * B[7];
}
LLD_HD void sim3_inverse(const double* S, double* O) {  // (r^-1, r^-1 ((-1/s) t), 1/s), r^-1 = conjugate
  const double qc[4] = {-S[0], -S[1], -S[2], S[3]};
  const double c = -1. / S[7];
  const double v[3] = {c * S[4], c * S[5], c * S[6]};
  double rt[3];
  quat_rot(qc, v, rt);
  O[0] = qc[0]; O[1] = qc[1]; O[2] = qc[2]; O[3] = qc[3];
  O[4] = rt[0]; O[5] = rt[1]; O[6] = rt[2];
  O[7] = 1. / S[7];
}
// Sim3(const Vector7d& update): omega = u[0:3], upsilon = u[3:6], sigma = u[6]
LLD_HD void sim3_exp(const double* u, double* S) {
  const double w0 = u[0], w1 = u[1], w2 = u[2], sigma = u[6];
  const double theta = sqrt(w0 * w0 + w1 * w1 + w2 * w2);
  const double O[9] = {0, -w2, w1, w2, 0, -w0, -w1, w0, 0};
  double O2[9];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) O2[3 * i + j] = O[3 * i] * O[j] + O[3 * i + 1] * O[3 + j] + O[3 * i + 2] * O[6 + j];
  const double s = exp(sigma);
  const double eps = 0.00001;
  double A, B, C, ra = 1.0, rb = 1.0;  // R = I + ra * Omega + rb * Omega^2
  bool small = false;                     // theta < eps: R = I + Omega + Omega^2 (sic)
  if (fabs(sigma) < eps) {
    C = 1;
    if (theta < eps) {
      A = 1. / 2.;
      B = 1. / 6.;
      small = true;
    } else {
      const double theta2 = theta * theta;
      A = (1 - cos(theta)) / (theta2);
      B = (theta - sin(theta)) / (theta2 * theta);
      ra = sin(theta) / theta; rb = (1 - cos(theta)) / (theta * theta);
    }
  } else {
    C = (s - 1) / sigma;
    if (theta < eps) {
      const double sigma2 = sigma * sigma;
      A = ((sigma - 1) * s + 1) / sigma2;
      B = ((0.5 * sigma2 - sigma + 1) * s) / (sigma2 * sigma);
      small = true;
    } else {
      ra = sin(theta) / theta; rb = (1 - cos(theta)) / (theta * theta);
      const double a = s * sin(theta);
      const double b = s * cos(theta);
      const double theta2 = theta * theta;
      const double sigma2 = sigma * sigma;
      const double c = theta2 + sigma2;
      A = (a * sigma + (1 - b) * theta) / (theta * c);
      B = (C - ((b - 1) * sigma + a * theta) / (c)) * 1. / (theta2);
    }
  }
  double R[9], W[9];
#pragma unroll
  for (int i = 0; i < 9; i++) {
    const double id = (i == 0 || i == 4 || i == 8) ? 1.0 : 0.0;
    R[i] = small ? id + O[i] + O2[i] : id + ra * O[i] + rb * O2[i];
    W[i] = A * O[i] + B * O2[i] + C * id;
  }
  quat_from_R(R, S);
  S[4] = W[0] * u[3] + W[1] * u[4] + W[2] * u[5];
  S[5] = W[3] * u[3] + W[4] * u[4] + W[5] * u[5];
  S[6] = W[6] * u[3] + W[7] * u[4] + W[8] * u[5];
  S[7] = s;
}
// VertexSim3Expmap::oplusImpl: with _fix_scale the caller's update[6] is set to 0, then estimate = Sim3(update) * estimate
LLD_HD void sim3_oplus(const double* S, double* u, bool fix_scale, double* out) {
  if (fix_scale) u[6] = 0;
  double E[8];
  sim3_exp(u, E);
  sim3_mul(E, S, out);
}
// EdgeSim3ProjectXYZ / EdgeInverseSim3ProjectXYZ::computeError: obs - cam_map(project(S.map(P))), where S is the
// estimate (e12, P = P2c, K1) or its inverse (e21, P = P1c, K2); K = fx fy cx cy
LLD_HD void sim3_edge_error(const double* S, const double* P, const double* K, const double* obs, double* err) {
  double x[3];
  sim3_map(S, P, x);
  const double p0 = x[0] / x[2], p1 = x[1] / x[2];
  err[0] = obs[0] - (p0 * K[0] + K[2]);
  err[1] = obs[1] - (p1 * K[1] + K[3]);
}
// The 14 states of g2o's numeric Jacobian (BaseBinaryEdge::linearizeOplus, delta = 1e-9): Sk[2d] = oplus(S, +delta e_d),
// Sk[2d+1] = oplus(S, -delta e_d); each with its inverse for the e21 edge.  Writes 8 doubles per state.
LLD_HD void sim3_perturbed(const double* S, int k, bool fix_scale, double* Sk, double* Skinv) {
  const double delta = 1e-9;
  double add[7] = {0, 0, 0, 0, 0, 0, 0};
  add[k >> 1] = (k & 1) ? -delta : delta;
  sim3_oplus(S, add, fix_scale, Sk);
  sim3_inverse(Sk, Skinv);
}
// One column of the 2x7 numeric Jacobian from the errors at the +delta / -delta states: scalar * (e+ - e-)
LLD_HD void sim3_jac_col(const double* ep, const double* em, double* J, int d) {
  const double scalar = 1.0 / (2 * 1e-9);
  J[d] = scalar * (ep[0] - em[0]);
  J[7 + d] = scalar * (ep[1] - em[1]);
}

// ---- Sim3Solver (ORB-SLAM2 src/Sim3Solver.cc): Horn's closed form and the inlier test in CV_32F -----------------------
// Small CV_32F products follow cv::gemm: a 3-long product without transposition sums float products in float (k = 0..2)
// and then rounds s0 * alpha + c * beta, formed in double, once to float.
LLD_HD float cv_gemm3(float a0, float a1, float a2, float b0, float b1, float b2) {
  const float p0 = a0 * b0, p1 = a1 * b1, p2 = a2 * b2;
  return (p0 + p1) + p2;
}
// Largest eigenpair of a symmetric 4x4 (cv::eigen's row 0): cyclic Jacobi in double on the float matrix, eigenvector rounded
// to float.  Ties go to the lowest index; a zero matrix gives e0.
LLD_HD void sym4_top_eigvec(const float* Nf, float* q) {
  double A[4][4], V[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      A[i][j] = (double)Nf[4 * i + j];
      V[i][j] = i == j ? 1.0 : 0.0;
    }
  for (int sweep = 0; sweep < 32; sweep++) {
    double off = 0.0, dia = 0.0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      dia += fabs(A[i][i]);
#pragma unroll
      for (int j = i + 1; j < 4; j++) off += fabs(A[i][j]);
    }
    if (!(off > 1e-15 * dia)) break;
#pragma unroll
    for (int p = 0; p < 3; p++)
#pragma unroll
      for (int r = p + 1; r < 4; r++) {
        const double apr = A[p][r];
        if (apr == 0.0) continue;
        const double th = (A[r][r] - A[p][p]) / (2.0 * apr);
        const double t = (th >= 0.0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const double akp = A[k][p], akr = A[k][r];
          A[k][p] = c * akp - s * akr;
          A[k][r] = s * akp + c * akr;
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const double apk = A[p][k], ark = A[r][k];
          A[p][k] = c * apk - s * ark;
          A[r][k] = s * apk + c * ark;
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const double vkp = V[k][p], vkr = V[k][r];
          V[k][p] = c * vkp - s * vkr;
          V[k][r] = s * vkp + c * vkr;
        }
      }
  }
  int im = 0;
  double best = A[0][0];
#pragma unroll
  for (int i = 1; i < 4; i++)
    if (A[i][i] > best) { best = A[i][i]; im = i; }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    double v = V[i][0];
#pragma unroll
    for (int j = 1; j < 4; j++) v = im == j ? V[i][j] : v;
    q[i] = (float)v;
  }
}
// cv::Rodrigues of a float rotation vector into a float 3x3 (computed in double)
LLD_HD void cv_rodrigues(const float* rv, float* R) {
  double r[3] = {(double)rv[0], (double)rv[1], (double)rv[2]};
  const double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  if (theta < 2.220446049250313e-16) {
#pragma unroll
    for (int i = 0; i < 9; i++) R[i] = (i == 0 || i == 4 || i == 8) ? 1.f : 0.f;
    return;
  }
  const double c = cos(theta), s = sin(theta), c1 = 1. - c;
  const double it = 1. / theta;
  r[0] *= it; r[1] *= it; r[2] *= it;
  const double rx[9] = {0, -r[2], r[1], r[2], 0, -r[0], -r[1], r[0], 0};
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) R[3 * i + j] = (float)((c * (i == j ? 1.0 : 0.0) + c1 * (r[i] * r[j])) + s * rx[3 * i + j]);
}
// Sim3Solver::ComputeSim3 on one minimal set.  P1, P2: the three points, point-major ([k][3] = column k of P3Dc1i / P3Dc2i).
// Writes the unscaled rotation R (row-major), t and s as GetEstimatedRotation / Translation / Scale return them.
LLD_HD void sim3r_horn(const float* P1, const float* P2, bool fix_scale, float* R, float* t, float* s_out) {
  float O1[3], O2[3], Pr1[3][3], Pr2[3][3];   // Pr[coordinate][point]
#pragma unroll
  for (int r = 0; r < 3; r++) {
    O1[r] = ((P1[r] + P1[3 + r]) + P1[6 + r]) * (1.0f / 3.0f);   // cv::reduce(SUM), C / P.cols
    O2[r] = ((P2[r] + P2[3 + r]) + P2[6 + r]) * (1.0f / 3.0f);
#pragma unroll
    for (int k = 0; k < 3; k++) {
      Pr1[r][k] = P1[3 * k + r] - O1[r];
      Pr2[r][k] = P2[3 * k + r] - O2[r];
    }
  }
  float M[3][3];   // Pr2 * Pr1^T
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++)
      M[i][j] = (float)(((double)Pr2[i][0] * (double)Pr1[j][0] + (double)Pr2[i][1] * (double)Pr1[j][1]) +
                        (double)Pr2[i][2] * (double)Pr1[j][2]);
  const float N11 = (M[0][0] + M[1][1]) + M[2][2], N12 = M[1][2] - M[2][1], N13 = M[2][0] - M[0][2], N14 = M[0][1] - M[1][0];
  const float N22 = (M[0][0] - M[1][1]) - M[2][2], N23 = M[0][1] + M[1][0], N24 = M[2][0] + M[0][2];
  const float N33 = (-M[0][0] + M[1][1]) - M[2][2], N34 = M[1][2] + M[2][1], N44 = (-M[0][0] - M[1][1]) + M[2][2];
  const float N[16] = {N11, N12, N13, N14, N12, N22, N23, N24, N13, N23, N33, N34, N14, N24, N34, N44};
  float q[4];
  sym4_top_eigvec(N, q);
  // cv::norm of the float 1x3 (double, in OpenCV's lane order), ang = atan2(|v|, w), v = 2 ang v / |v|
  const double nrm = sqrt(((double)q[1] * (double)q[1] + (double)q[3] * (double)q[3]) + (double)q[2] * (double)q[2]);
  const double ang = atan2(nrm, (double)q[0]);
  const double al = (2 * ang) * (1. / nrm);
  const float rv[3] = {(float)(al * (double)q[1]), (float)(al * (double)q[2]), (float)(al * (double)q[3])};
  cv_rodrigues(rv, R);
  float s = 1.0f;
  if (!fix_scale) {
    float P3[3][3];   // R * Pr2
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int k = 0; k < 3; k++) P3[r][k] = cv_gemm3(R[3 * r], R[3 * r + 1], R[3 * r + 2], Pr2[0][k], Pr2[1][k], Pr2[2][k]);
    double nom = 0, den = 0;
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int k = 0; k < 3; k++) {
        nom += (double)Pr1[r][k] * (double)P3[r][k];
        den += (double)(P3[r][k] * P3[r][k]);
      }
    s = (float)(nom / den);
  }
#pragma unroll
  for (int r = 0; r < 3; r++)   // t = O1 - s R O2: gemm(R, O2, -s, O1, 1)
    t[r] = (float)((double)cv_gemm3(R[3 * r], R[3 * r + 1], R[3 * r + 2], O2[0], O2[1], O2[2]) * -(double)s + (double)O1[r]);
  *s_out = s;
}
// T12 = [sR | t], T21 = [(1/s) R^T | -(1/s) R^T t] of one estimate (R, t, s)
struct Sim3Pair {
  float A12[9], b12[3], A21[9], b21[3];
};
LLD_HD void sim3r_pair(const float* R, const float* t, float s, Sim3Pair* T) {
  const double is = 1.0 / (double)s;
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) {
      T->A12[3 * i + j] = s * R[3 * i + j];
      T->A21[3 * i + j] = (float)(is * (double)R[3 * j + i]);
    }
#pragma unroll
  for (int r = 0; r < 3; r++) {
    T->b12[r] = t[r];
    T->b21[r] = -cv_gemm3(T->A21[3 * r], T->A21[3 * r + 1], T->A21[3 * r + 2], t[0], t[1], t[2]);
  }
}
// Sim3Solver::Project of one point (Rcw * X + tcw, float invz, no depth test); K = fx fy cx cy
LLD_HD void sim3r_project(const float* A, const float* b, const float* X, const float* K, float* uv) {
  float Y[3];
#pragma unroll
  for (int r = 0; r < 3; r++) Y[r] = (float)((double)cv_gemm3(A[3 * r], A[3 * r + 1], A[3 * r + 2], X[0], X[1], X[2]) + (double)b[r]);
  const float invz = 1 / Y[2];
  const float x = Y[0] * invz, y = Y[1] * invz;
  uv[0] = K[0] * x + K[2];
  uv[1] = K[1] * y + K[3];
}
// Sim3Solver::FromCameraToImage of one point
LLD_HD void sim3r_own(const float* X, const float* K, float* uv) {
  const float invz = 1 / X[2];
  const float x = X[0] * invz, y = X[1] * invz;
  uv[0] = K[0] * x + K[2];
  uv[1] = K[1] * y + K[3];
}
// dist.dot(dist) of a float 2-vector (double accumulation, stored in a float)
LLD_HD float sim3r_err(const float* a, const float* b) {
  const float d0 = a[0] - b[0], d1 = a[1] - b[1];
  return (float)((double)d0 * (double)d0 + (double)d1 * (double)d1);
}
// mvnMaxError = 9.210 * sigma2 stored in a size_t
LLD_HD float sim3r_max_err(float sigma2) { return (float)(unsigned long long)(9.210 * (double)sigma2); }
// CheckInliers for one correspondence; K = K1 (4), K2 (4).  err1 / err2 out for the tests.
LLD_HD bool sim3r_inlier(const Sim3Pair& T, const float* x1, const float* x2, float sig1, float sig2, const float* K, float* e) {
  float own1[2], own2[2], p21[2], p12[2];
  sim3r_own(x1, K, own1);
  sim3r_own(x2, K + 4, own2);
  sim3r_project(T.A12, T.b12, x2, K, p21);
  sim3r_project(T.A21, T.b21, x1, K + 4, p12);
  e[0] = sim3r_err(own1, p21);
  e[1] = sim3r_err(p12, own2);
  return e[0] < sim3r_max_err(sig1) && e[1] < sim3r_max_err(sig2);
}

// ---- PnPsolver (ORB-SLAM2 src/PnPsolver.cc: EPnP of Lepetit et al., epnp.cpp) -------------------------------------
// One EPnP runs on a group of threads described by a Par: the serial host build (PnpSerial), one warp (a minimal set) or
// one CTA (Refine over the best inliers).  Every sum over correspondences is formed by one thread, serially in
// correspondence order, so all three give the same bits; the group splits only over independent outputs (matrix entries,
// Jacobi rotation rows) and joins with Par::sync().  Shared state lives in a PnpWork the group can all read.
struct PnpSerial {
  LLD_HD int rank() const { return 0; }
  LLD_HD int size() const { return 1; }
  LLD_HD void sync() const {}
};
#if defined(__CUDACC__)
struct PnpWarp {
  int lane;
  __device__ int rank() const { return lane; }
  __device__ int size() const { return 32; }
  __device__ void sync() const { __syncwarp(); }
};
struct PnpCta {
  __device__ int rank() const { return (int)threadIdx.x; }
  __device__ int size() const { return (int)blockDim.x; }
  __device__ void sync() const { __syncthreads(); }
};
#endif

struct PnpCam {
  double fu, fv, uc, vc;
};

struct PnpWork {
  double c0[3];         // cws[0]: centroid of the world points
  double cws[4][3];     // control points
  double cci[9];        // CC^-1 (cvInvert(CC, CV_SVD))
  double a[144];        // the symmetric matrix under Jacobi (PW0^T PW0 in a[0..8], M^T M)
  double v[144];        // its eigenvectors (columns)
  int ord[12];          // eigen indices by decreasing eigenvalue
  double ccs[3][12];    // camera control points of the three beta solutions (sign resolved)
  double pw0[3], pc0[3][3];
  double abt[3][9];
  double R[3][9], t[3][3], err[3];
};

// cyclic Jacobi on the symmetric n x n A (row-major, overwritten; the diagonal ends as the eigenvalues), eigenvectors in the
// columns of V, ord = eigen indices by decreasing eigenvalue (first index on ties).  The group splits each rotation over rows.
template <class P>
LLD_HD void pnp_sym_jacobi(const P& par, double* A, double* V, int n, int* ord) {
  for (int k = par.rank(); k < n * n; k += par.size()) V[k] = (k / n == k % n) ? 1.0 : 0.0;
  par.sync();
  for (int sweep = 0; sweep < 32; sweep++) {
    double off = 0, dia = 0;
    for (int i = 0; i < n; i++) {
      dia += fabs(A[i * n + i]);
      for (int j = i + 1; j < n; j++) off += fabs(A[i * n + j]);
    }
    if (!(off > 1e-15 * dia)) break;
    for (int p = 0; p < n - 1; p++)
      for (int q = p + 1; q < n; q++) {
        const double apq = A[p * n + q];
        if (apq == 0.0) continue;
        const double theta = (A[q * n + q] - A[p * n + p]) / (2.0 * apq);
        const double tt = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(tt * tt + 1.0), s = tt * c;
        par.sync();
        for (int k = par.rank(); k < n; k += par.size()) {
          const double x = A[k * n + p], y = A[k * n + q];
          A[k * n + p] = c * x - s * y;
          A[k * n + q] = s * x + c * y;
          const double vx = V[k * n + p], vy = V[k * n + q];
          V[k * n + p] = c * vx - s * vy;
          V[k * n + q] = s * vx + c * vy;
        }
        par.sync();
        for (int k = par.rank(); k < n; k += par.size()) {
          const double x = A[p * n + k], y = A[q * n + k];
          A[p * n + k] = c * x - s * y;
          A[q * n + k] = s * x + c * y;
        }
        par.sync();
      }
  }
  if (par.rank() == 0) {
    for (int i = 0; i < n; i++) ord[i] = i;
    for (int i = 1; i < n; i++) {   // insertion sort by decreasing eigenvalue, stable
      const int x = ord[i];
      int j = i;
      for (; j > 0 && A[x * n + x] > A[ord[j - 1] * n + ord[j - 1]]; j--) ord[j] = ord[j - 1];
      ord[j] = x;
    }
  }
  par.sync();
}

// one-sided (Hestenes) Jacobi SVD of the m x k A (row-major, m <= 6, k <= 5): A is overwritten by U diag(sig), V (k x k)
// holds the right singular vectors in its columns, ord the column indices by decreasing singular value.
LLD_HD void pnp_svd_jacobi(double* A, int m, int k, double* V, double* sig, int* ord) {
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
        if (!(fabs(ga) > 1e-15 * sqrt(al * be))) continue;
        const double zeta = (be - al) / (2.0 * ga);
        const double tt = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + tt * tt), s = c * tt;
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
    sig[j] = sqrt(s2);
  }
  for (int i = 0; i < k; i++) ord[i] = i;
  for (int i = 1; i < k; i++) {   // insertion sort by decreasing sig, stable
    const int x = ord[i];
    int j = i;
    for (; j > 0 && sig[x] > sig[ord[j - 1]]; j--) ord[j] = ord[j - 1];
    ord[j] = x;
  }
}

// least-squares solve of the m x k system A x = b through the SVD (cvSolve(..., CV_SVD)); A is destroyed
LLD_HD void pnp_svd_solve(double* A, int m, int k, const double* b, double* x) {
  double V[25], sig[5];
  int ord[5];
  pnp_svd_jacobi(A, m, k, V, sig, ord);
  for (int i = 0; i < k; i++) x[i] = 0.0;
  double thr = 0;   // OpenCV's back-substitution skips singular values <= 2 DBL_EPSILON sum(sig)
  for (int jj = 0; jj < k; jj++) thr += sig[ord[jj]];
  thr *= 2 * 2.220446049250313e-16;
  for (int jj = 0; jj < k; jj++) {
    const int j = ord[jj];
    if (fabs(sig[j]) <= thr) continue;
    double ub = 0;
    for (int r = 0; r < m; r++) ub += (A[r * k + j] / sig[j]) * b[r];
    const double w = ub / sig[j];
    for (int i = 0; i < k; i++) x[i] += V[i * k + j] * w;
  }
}

// Lepetit's qr_solve on the 6 x 4 Gauss-Newton system (unpivoted Householder); a singular A leaves x at 0
LLD_HD void pnp_qr_solve_6x4(double* A, double* b, double* x) {
  const int nr = 6, nc = 4;
  double A1[4], A2[4];
  for (int k = 0; k < nc; k++) x[k] = 0.0;
  for (int k = 0; k < nc; k++) {
    double eta = fabs(A[k * nc + k]);
    for (int i = k + 1; i < nr; i++) {
      const double elt = fabs(A[i * nc + k]);
      if (eta < elt) eta = elt;
    }
    if (eta == 0) return;
    double sum = 0.0;
    for (int i = k; i < nr; i++) {
      A[i * nc + k] /= eta;
      sum += A[i * nc + k] * A[i * nc + k];
    }
    double sigma = sqrt(sum);
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
  x[nc - 1] = b[nc - 1] / A2[nc - 1];
  for (int i = nc - 2; i >= 0; i--) {
    double s = 0;
    for (int j = i + 1; j < nc; j++) s += A[i * nc + j] * x[j];
    x[i] = (b[i] - s) / A2[i];
  }
}

LLD_HD double pnp_dot(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// compute_barycentric_coordinates for one world point
LLD_HD void pnp_alphas(const PnpWork& w, const float* X, double* al) {
  const double p0 = X[0], p1 = X[1], p2 = X[2];
  for (int j = 0; j < 3; j++)
    al[1 + j] = w.cci[3 * j] * (p0 - w.cws[0][0]) + w.cci[3 * j + 1] * (p1 - w.cws[0][1]) + w.cci[3 * j + 2] * (p2 - w.cws[0][2]);
  al[0] = 1.0 - al[1] - al[2] - al[3];
}

// compute_pcs for one point: camera coordinate j under the control points ccs
LLD_HD double pnp_pc(const double* al, const double* ccs, int j) {
  return al[0] * ccs[j] + al[1] * ccs[3 + j] + al[2] * ccs[6 + j] + al[3] * ccs[9 + j];
}

// compute_L_6x10 on the eigenvectors of the four smallest eigenvalues, compute_rho
LLD_HD void pnp_L_rho(const PnpWork& w, double* L, double* rho) {
  double v[4][12];
  for (int i = 0; i < 4; i++)
    for (int k = 0; k < 12; k++) v[i][k] = w.v[k * 12 + w.ord[11 - i]];   // ut row 11 - i
  double dv[4][6][3];
  for (int i = 0; i < 4; i++) {
    int a = 0, b = 1;
    for (int j = 0; j < 6; j++) {
      dv[i][j][0] = v[i][3 * a] - v[i][3 * b];
      dv[i][j][1] = v[i][3 * a + 1] - v[i][3 * b + 1];
      dv[i][j][2] = v[i][3 * a + 2] - v[i][3 * b + 2];
      b++;
      if (b > 3) {
        a++;
        b = a + 1;
      }
    }
  }
  for (int i = 0; i < 6; i++) {
    double* row = L + 10 * i;
    row[0] = pnp_dot(dv[0][i], dv[0][i]);
    row[1] = 2.0 * pnp_dot(dv[0][i], dv[1][i]);
    row[2] = pnp_dot(dv[1][i], dv[1][i]);
    row[3] = 2.0 * pnp_dot(dv[0][i], dv[2][i]);
    row[4] = 2.0 * pnp_dot(dv[1][i], dv[2][i]);
    row[5] = pnp_dot(dv[2][i], dv[2][i]);
    row[6] = 2.0 * pnp_dot(dv[0][i], dv[3][i]);
    row[7] = 2.0 * pnp_dot(dv[1][i], dv[3][i]);
    row[8] = 2.0 * pnp_dot(dv[2][i], dv[3][i]);
    row[9] = pnp_dot(dv[3][i], dv[3][i]);
  }
  auto d2 = [](const double* p, const double* q) {
    return (p[0] - q[0]) * (p[0] - q[0]) + (p[1] - q[1]) * (p[1] - q[1]) + (p[2] - q[2]) * (p[2] - q[2]);
  };
  rho[0] = d2(w.cws[0], w.cws[1]);
  rho[1] = d2(w.cws[0], w.cws[2]);
  rho[2] = d2(w.cws[0], w.cws[3]);
  rho[3] = d2(w.cws[1], w.cws[2]);
  rho[4] = d2(w.cws[1], w.cws[3]);
  rho[5] = d2(w.cws[2], w.cws[3]);
}

// find_betas_approx_1 / 2 / 3 (s = 0, 1, 2): the columns of L each approximation keeps, its SVD solve and its sign rules
LLD_HD void pnp_betas_approx(int s, const double* L, const double* rho, double* betas) {
  const int cols[3][5] = {{0, 1, 3, 6, -1}, {0, 1, 2, -1, -1}, {0, 1, 2, 3, 4}};
  const int k = s == 0 ? 4 : (s == 1 ? 3 : 5);
  double A[30], b[5];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < k; c++) A[r * k + c] = L[10 * r + cols[s][c]];
  pnp_svd_solve(A, 6, k, rho, b);
  if (s == 0) {
    if (b[0] < 0) {
      betas[0] = sqrt(-b[0]);
      betas[1] = -b[1] / betas[0];
      betas[2] = -b[2] / betas[0];
      betas[3] = -b[3] / betas[0];
    } else {
      betas[0] = sqrt(b[0]);
      betas[1] = b[1] / betas[0];
      betas[2] = b[2] / betas[0];
      betas[3] = b[3] / betas[0];
    }
    return;
  }
  if (b[0] < 0) {
    betas[0] = sqrt(-b[0]);
    betas[1] = (b[2] < 0) ? sqrt(-b[2]) : 0.0;
  } else {
    betas[0] = sqrt(b[0]);
    betas[1] = (b[2] > 0) ? sqrt(b[2]) : 0.0;
  }
  if (b[1] < 0) betas[0] = -betas[0];
  betas[2] = s == 2 ? b[3] / betas[0] : 0.0;
  betas[3] = 0.0;
}

// gauss_newton: 5 iterations of compute_A_and_b_gauss_newton + qr_solve
LLD_HD void pnp_gauss_newton(const double* L, const double* rho, double* betas) {
  for (int it = 0; it < 5; it++) {
    double A[24], b[6], x[4];
    for (int i = 0; i < 6; i++) {
      const double* l = L + 10 * i;
      double* a = A + 4 * i;
      a[0] = 2 * l[0] * betas[0] + l[1] * betas[1] + l[3] * betas[2] + l[6] * betas[3];
      a[1] = l[1] * betas[0] + 2 * l[2] * betas[1] + l[4] * betas[2] + l[7] * betas[3];
      a[2] = l[3] * betas[0] + l[4] * betas[1] + 2 * l[5] * betas[2] + l[8] * betas[3];
      a[3] = l[6] * betas[0] + l[7] * betas[1] + l[8] * betas[2] + 2 * l[9] * betas[3];
      b[i] = rho[i] - (l[0] * betas[0] * betas[0] + l[1] * betas[0] * betas[1] + l[2] * betas[1] * betas[1] +
                       l[3] * betas[0] * betas[2] + l[4] * betas[1] * betas[2] + l[5] * betas[2] * betas[2] +
                       l[6] * betas[0] * betas[3] + l[7] * betas[1] * betas[3] + l[8] * betas[2] * betas[3] +
                       l[9] * betas[3] * betas[3]);
    }
    pnp_qr_solve_6x4(A, b, x);
    for (int i = 0; i < 4; i++) betas[i] += x[i];
  }
}

// estimate_R_and_t's SVD part: ABt = U S V^T, R = U V^T (columns by decreasing singular value), row 2 negated if det < 0,
// t = pc0 - R pw0
LLD_HD void pnp_R_t(const double* abt_in, const double* pc0, const double* pw0, double* R, double* t) {
  double U[9], V[9], sig[3];
  int ord[3];
  for (int i = 0; i < 9; i++) U[i] = abt_in[i];
  pnp_svd_jacobi(U, 3, 3, V, sig, ord);
  double Un[9];   // left singular vectors, columns by decreasing singular value
  for (int i = 0; i < 3; i++)
    for (int k = 0; k < 3; k++) Un[3 * i + k] = U[i * 3 + ord[k]] / sig[ord[k]];
  const double thr = (sig[ord[0]] + sig[ord[1]] + sig[ord[2]]) * (2 * 2.220446049250313e-16);
  if (sig[ord[2]] <= thr) {   // coplanar world points: complete U to a proper basis (V is a product of rotations)
    Un[2] = Un[3] * Un[7] - Un[6] * Un[4];
    Un[5] = Un[6] * Un[1] - Un[0] * Un[7];
    Un[8] = Un[0] * Un[4] - Un[3] * Un[1];
  }
  for (int i = 0; i < 3; i++) {
    double vr[3];
    for (int j = 0; j < 3; j++) {
      for (int k = 0; k < 3; k++) vr[k] = V[j * 3 + ord[k]];
      R[3 * i + j] = pnp_dot(Un + 3 * i, vr);
    }
  }
  const double det = R[0] * R[4] * R[8] + R[1] * R[5] * R[6] + R[2] * R[3] * R[7] - R[2] * R[4] * R[6] - R[1] * R[3] * R[8] -
                     R[0] * R[5] * R[7];
  if (det < 0) {
    R[6] = -R[6];
    R[7] = -R[7];
    R[8] = -R[8];
  }
  t[0] = pc0[0] - pnp_dot(R, pw0);
  t[1] = pc0[1] - pnp_dot(R + 3, pw0);
  t[2] = pc0[2] - pnp_dot(R + 6, pw0);
}

// reprojection_error term of one correspondence
LLD_HD double pnp_reproj(const double* R, const double* t, const float* X, const float* uv, const PnpCam& cam) {
  const double pw[3] = {X[0], X[1], X[2]};
  const double Xc = pnp_dot(R, pw) + t[0];
  const double Yc = pnp_dot(R + 3, pw) + t[1];
  const double inv_Zc = 1.0 / (pnp_dot(R + 6, pw) + t[2]);
  const double ue = cam.uc + cam.fu * Xc * inv_Zc;
  const double ve = cam.vc + cam.fv * Yc * inv_Zc;
  const double u = uv[0], v = uv[1];
  return sqrt((u - ue) * (u - ue) + (v - ve) * (v - ve));
}

// compute_pose over the n correspondences id(0..n-1) (idx == nullptr: 0..n-1) of X3 ([.][3]) / uv ([.][2]).  R (9), t
// (3) in double, as mRi / mti; valid on every rank after the call.
template <class P>
LLD_HD void pnp_epnp(const P& par, PnpWork& w, const float* X3, const float* uv, const int* idx, int n, const PnpCam& cam) {
  const int rk = par.rank(), sz = par.size();
  const double dn = (double)n;
#define LLD_PNP_ID(i) (idx ? idx[i] : (i))
  // choose_control_points: centroid, then PW0^T PW0
  for (int j = rk; j < 3; j += sz) {
    double s = 0;
    for (int i = 0; i < n; i++) s += (double)X3[3 * (size_t)LLD_PNP_ID(i) + j];
    w.c0[j] = s / dn;
  }
  par.sync();
  for (int e = rk; e < 6; e += sz) {
    const int a = e < 3 ? 0 : (e < 5 ? 1 : 2), b = e < 3 ? e : (e < 5 ? e - 2 : 2);
    double s = 0;
    for (int i = 0; i < n; i++) {
      const float* X = X3 + 3 * (size_t)LLD_PNP_ID(i);
      s += ((double)X[a] - w.c0[a]) * ((double)X[b] - w.c0[b]);
    }
    w.a[3 * a + b] = s;
    w.a[3 * b + a] = s;
  }
  par.sync();
  pnp_sym_jacobi(par, w.a, w.v, 3, w.ord);
  if (rk == 0) {
    for (int j = 0; j < 3; j++) w.cws[0][j] = w.c0[j];
    for (int i = 1; i < 4; i++) {
      const int e = w.ord[i - 1];
      const double d = w.a[4 * e];
      const double k = sqrt((d > 0.0 ? d : 0.0) / dn);
      for (int j = 0; j < 3; j++) w.cws[i][j] = w.cws[0][j] + k * w.v[3 * j + e];
    }
    // compute_barycentric_coordinates: CC^-1 through the SVD, V diag(1 / s) U^T
    double CC[9], V[9], sig[3];
    int ord[3];
    for (int i = 0; i < 3; i++)
      for (int j = 1; j < 4; j++) CC[3 * i + j - 1] = w.cws[j][i] - w.cws[0][i];
    pnp_svd_jacobi(CC, 3, 3, V, sig, ord);
    double thr = 0;   // cvInvert(CV_SVD): singular values <= 2 DBL_EPSILON sum(sig) are skipped (a pseudo-inverse)
    for (int kk = 0; kk < 3; kk++) thr += sig[ord[kk]];
    thr *= 2 * 2.220446049250313e-16;
    for (int i = 0; i < 3; i++)
      for (int r = 0; r < 3; r++) {
        double s = 0;
        for (int kk = 0; kk < 3; kk++) {
          const int c = ord[kk];
          if (fabs(sig[c]) <= thr) continue;
          s += V[3 * i + c] * ((CC[3 * r + c] / sig[c]) / sig[c]);
        }
        w.cci[3 * i + r] = s;
      }
  }
  par.sync();
  // fill_M, M^T M: entry (a, b), rows in correspondence order (u row, then v row)
  for (int e = rk; e < 78; e += sz) {
    int a = 0, rem = e;
    while (rem >= 12 - a) {
      rem -= 12 - a;
      a++;
    }
    const int b = a + rem;
    double s = 0;
    for (int i = 0; i < n; i++) {
      const int id = LLD_PNP_ID(i);
      double al[4];
      pnp_alphas(w, X3 + 3 * (size_t)id, al);
      const double u = uv[2 * (size_t)id], v = uv[2 * (size_t)id + 1];
      const double m1a = (a % 3 == 0) ? al[a / 3] * cam.fu : (a % 3 == 1 ? 0.0 : al[a / 3] * (cam.uc - u));
      const double m1b = (b % 3 == 0) ? al[b / 3] * cam.fu : (b % 3 == 1 ? 0.0 : al[b / 3] * (cam.uc - u));
      const double m2a = (a % 3 == 0) ? 0.0 : (a % 3 == 1 ? al[a / 3] * cam.fv : al[a / 3] * (cam.vc - v));
      const double m2b = (b % 3 == 0) ? 0.0 : (b % 3 == 1 ? al[b / 3] * cam.fv : al[b / 3] * (cam.vc - v));
      s += m1a * m1b;
      s += m2a * m2b;
    }
    w.a[12 * a + b] = s;
    w.a[12 * b + a] = s;
  }
  par.sync();
  pnp_sym_jacobi(par, w.a, w.v, 12, w.ord);
  // L, rho, the three beta approximations with Gauss-Newton, ccs and solve_for_sign (the first point's depth)
  if (rk == 0) {
    double L[60], rho[6];
    pnp_L_rho(w, L, rho);
    for (int s = 0; s < 3; s++) {
      double betas[4];
      pnp_betas_approx(s, L, rho, betas);
      pnp_gauss_newton(L, rho, betas);
      double* ccs = w.ccs[s];
      for (int k = 0; k < 12; k++) ccs[k] = 0.0;
      for (int i = 0; i < 4; i++)
        for (int k = 0; k < 12; k++) ccs[k] += betas[i] * w.v[k * 12 + w.ord[11 - i]];
      double al[4];
      pnp_alphas(w, X3 + 3 * (size_t)LLD_PNP_ID(0), al);
      if (pnp_pc(al, ccs, 2) < 0)
        for (int k = 0; k < 12; k++) ccs[k] = -ccs[k];
    }
  }
  par.sync();
  // estimate_R_and_t: centroids of the camera points of each solution and of the world points
  for (int e = rk; e < 12; e += sz) {
    const int s = e / 3, j = e % 3;
    double acc = 0;
    for (int i = 0; i < n; i++) {
      const int id = LLD_PNP_ID(i);
      if (s == 3) {
        acc += (double)X3[3 * (size_t)id + j];
      } else {
        double al[4];
        pnp_alphas(w, X3 + 3 * (size_t)id, al);
        acc += pnp_pc(al, w.ccs[s], j);
      }
    }
    if (s == 3)
      w.pw0[j] = acc / dn;
    else
      w.pc0[s][j] = acc / dn;
  }
  par.sync();
  for (int e = rk; e < 27; e += sz) {
    const int s = e / 9, j = (e % 9) / 3, c = e % 3;
    double acc = 0;
    for (int i = 0; i < n; i++) {
      const int id = LLD_PNP_ID(i);
      double al[4];
      pnp_alphas(w, X3 + 3 * (size_t)id, al);
      acc += (pnp_pc(al, w.ccs[s], j) - w.pc0[s][j]) * ((double)X3[3 * (size_t)id + c] - w.pw0[c]);
    }
    w.abt[s][3 * j + c] = acc;
  }
  par.sync();
  for (int s = rk; s < 3; s += sz) pnp_R_t(w.abt[s], w.pc0[s], w.pw0, w.R[s], w.t[s]);
  par.sync();
  for (int s = rk; s < 3; s += sz) {
    double acc = 0;
    for (int i = 0; i < n; i++) {
      const int id = LLD_PNP_ID(i);
      acc += pnp_reproj(w.R[s], w.t[s], X3 + 3 * (size_t)id, uv + 2 * (size_t)id, cam);
    }
    w.err[s] = acc / dn;
  }
  par.sync();
#undef LLD_PNP_ID
}

// the solution compute_pose keeps: 1, replaced by 2 if its error is smaller, then by 3 if smaller than the kept one
LLD_HD int pnp_pick(const PnpWork& w) {
  int b = 0;
  if (w.err[1] < w.err[0]) b = 1;
  if (w.err[2] < w.err[b]) b = 2;
  return b;
}

// PnPsolver::CheckInliers for one correspondence: Xc, Yc, invZc stored to float, ue / ve in double, distX / distY and
// error2 in float; inlier iff error2 < mvMaxError (a NaN is an outlier, no depth test)
LLD_HD bool pnp_inlier(const double* R, const double* t, const float* X, const float* uv, float max_err, const PnpCam& cam) {
  const float Xc = (float)(R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + t[0]);
  const float Yc = (float)(R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + t[1]);
  const float invZc = (float)(1 / (R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + t[2]));
  const double ue = cam.uc + cam.fu * Xc * invZc;
  const double ve = cam.vc + cam.fv * Yc * invZc;
  const float distX = (float)(uv[0] - ue);
  const float distY = (float)(uv[1] - ve);
  const float error2 = distX * distX + distY * distY;
  return error2 < max_err;
}

// ---- tiny dense helpers --------------------------------------------------------------------------
// symmetric 3x3 / 4x4 inverse via cofactors / blockwise (general inverse, like MatrixXd::inverse()).
LLD_HD void inv3_sym(const double* A /*full 9*/, double* I) {
  const double c00 = A[4] * A[8] - A[5] * A[7];
  const double c01 = A[5] * A[6] - A[3] * A[8];
  const double c02 = A[3] * A[7] - A[4] * A[6];
  const double det = A[0] * c00 + A[1] * c01 + A[2] * c02;
  const double id = 1.0 / det;
  I[0] = c00 * id;
  I[1] = (A[2] * A[7] - A[1] * A[8]) * id;
  I[2] = (A[1] * A[5] - A[2] * A[4]) * id;
  I[3] = c01 * id;
  I[4] = (A[0] * A[8] - A[2] * A[6]) * id;
  I[5] = (A[2] * A[3] - A[0] * A[5]) * id;
  I[6] = c02 * id;
  I[7] = (A[1] * A[6] - A[0] * A[7]) * id;
  I[8] = (A[0] * A[4] - A[1] * A[3]) * id;
}
// general 4x4 inverse through 2x2 sub-determinants (adjugate); no pivoting, no dynamic indexing
LLD_HD void inv4(const double* a, double* b) {
  const double s0 = a[0] * a[5] - a[4] * a[1], s1 = a[0] * a[6] - a[4] * a[2], s2 = a[0] * a[7] - a[4] * a[3];
  const double s3 = a[1] * a[6] - a[5] * a[2], s4 = a[1] * a[7] - a[5] * a[3], s5 = a[2] * a[7] - a[6] * a[3];
  const double c5 = a[10] * a[15] - a[14] * a[11], c4 = a[9] * a[15] - a[13] * a[11], c3 = a[9] * a[14] - a[13] * a[10];
  const double c2 = a[8] * a[15] - a[12] * a[11], c1 = a[8] * a[14] - a[12] * a[10], c0 = a[8] * a[13] - a[12] * a[9];
  const double det = s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0;
  const double id = 1.0 / det;
  b[0] = (a[5] * c5 - a[6] * c4 + a[7] * c3) * id;
  b[1] = (-a[1] * c5 + a[2] * c4 - a[3] * c3) * id;
  b[2] = (a[13] * s5 - a[14] * s4 + a[15] * s3) * id;
  b[3] = (-a[9] * s5 + a[10] * s4 - a[11] * s3) * id;
  b[4] = (-a[4] * c5 + a[6] * c2 - a[7] * c1) * id;
  b[5] = (a[0] * c5 - a[2] * c2 + a[3] * c1) * id;
  b[6] = (-a[12] * s5 + a[14] * s2 - a[15] * s1) * id;
  b[7] = (a[8] * s5 - a[10] * s2 + a[11] * s1) * id;
  b[8] = (a[4] * c4 - a[5] * c2 + a[7] * c0) * id;
  b[9] = (-a[0] * c4 + a[1] * c2 - a[3] * c0) * id;
  b[10] = (a[12] * s4 - a[13] * s2 + a[15] * s0) * id;
  b[11] = (-a[8] * s4 + a[9] * s2 - a[11] * s0) * id;
  b[12] = (-a[4] * c3 + a[5] * c1 - a[6] * c0) * id;
  b[13] = (a[0] * c3 - a[1] * c1 + a[2] * c0) * id;
  b[14] = (-a[12] * s3 + a[13] * s1 - a[14] * s0) * id;
  b[15] = (a[8] * s3 - a[9] * s1 + a[10] * s0) * id;
}

}  // namespace lld
