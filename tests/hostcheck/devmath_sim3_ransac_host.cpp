// Test-only: compiles the Sim3Solver part of the product's device math header (lld_slam_b200/csrc/lld_math.cuh) for the host
// so that tests/test_sim3_ransac.py can compare it with the CPU oracle (libsim3_ransac_oracle.so) without a GPU.
#include "../../lld_slam_b200/csrc/lld_math.cuh"
using namespace lld;
extern "C" {
// P1, P2 point-major ([k][3]); out = R (9), t (3), s
void dm_sim3r_horn(const float* P1, const float* P2, int fix_scale, float* out) { sim3r_horn(P1, P2, fix_scale != 0, out, out + 9, out + 12); }
void dm_sym4_top_eigvec(const float* N, float* q) { sym4_top_eigvec(N, q); }
void dm_rodrigues(const float* v, float* R) { cv_rodrigues(v, R); }
int dm_sim3r_errors(const float* est, const float* cam, const float* x1, const float* x2, float s1, float s2, float* err) {
  Sim3Pair T;
  sim3r_pair(est, est + 9, est[12], &T);
  return sim3r_inlier(T, x1, x2, s1, s2, cam, err);
}
}
