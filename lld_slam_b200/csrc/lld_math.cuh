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
