// Test-only: compiles the PnPsolver part of the product's device math header (lld_slam_b200/csrc/lld_math.cuh) for the host
// so that tests/test_pnp_ransac.py can compare it with the CPU oracle (libpnp_ransac_oracle.so) without a GPU.
#include "../../lld_slam_b200/csrc/lld_math.cuh"
using namespace lld;
extern "C" {
// EPnP over n correspondences (X3 [n][3], uv [n][2], cam fu fv uc vc) -> R (9), t (3) of the kept solution
void dm_pnp_epnp(const float* X3, const float* uv, int n, const double* cam, double* Rt) {
  static PnpWork w;
  const PnpCam c{cam[0], cam[1], cam[2], cam[3]};
  pnp_epnp(PnpSerial{}, w, X3, uv, nullptr, n, c);
  const int b = pnp_pick(w);
  for (int k = 0; k < 9; k++) Rt[k] = w.R[b][k];
  for (int k = 0; k < 3; k++) Rt[9 + k] = w.t[b][k];
}
int dm_pnp_inlier(const double* Rt, const float* X, const float* uv, float max_err, const double* cam) {
  const PnpCam c{cam[0], cam[1], cam[2], cam[3]};
  return pnp_inlier(Rt, Rt + 9, X, uv, max_err, c);
}
void dm_pnp_sym_jacobi(double* A, double* V, int n, int* ord) { pnp_sym_jacobi(PnpSerial{}, A, V, n, ord); }
void dm_pnp_svd_solve(double* A, int m, int k, const double* b, double* x) { pnp_svd_solve(A, m, k, b, x); }
}
