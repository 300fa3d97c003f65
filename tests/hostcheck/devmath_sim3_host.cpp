// Test-only: compiles the Sim3 part of the product's device math header (lld_slam_b200/csrc/lld_math.cuh) for the host so that
// tests/test_optimize_sim3.py can compare it with the CPU oracle (libsim3_oracle.so) without a GPU.
#include "../../lld_slam_b200/csrc/lld_math.cuh"
using namespace lld;
extern "C" {
// Sim3 (state q[4], t[3], s)
void dm_sim3_exp(const double* u, double* S) { sim3_exp(u, S); }
void dm_sim3_mul(const double* A, const double* B, double* O) { sim3_mul(A, B, O); }
void dm_sim3_inverse(const double* S, double* O) { sim3_inverse(S, O); }
void dm_sim3_map(const double* S, const double* x, double* o) { sim3_map(S, x, o); }
// e12 / e21 of one correspondence at S and their numeric Jacobians ([2][7] each), as the kernel forms them; cam = K1, K2
void dm_sim3_edges(const double* S, int fix_scale, const double* cam, const float* p1c, const float* p2c, const float* obs1,
                   const float* obs2, double* e12, double* e21, double* J12, double* J21) {
  double Si[8], Sk[14][2][8];
  sim3_inverse(S, Si);
  for (int k = 0; k < 14; k++) sim3_perturbed(S, k, fix_scale != 0, Sk[k][0], Sk[k][1]);
  const double P1[3] = {p1c[0], p1c[1], p1c[2]}, P2[3] = {p2c[0], p2c[1], p2c[2]};
  const double o1[2] = {obs1[0], obs1[1]}, o2[2] = {obs2[0], obs2[1]};
  sim3_edge_error(S, P2, cam, o1, e12);
  sim3_edge_error(Si, P1, cam + 4, o2, e21);
  for (int d = 0; d < 7; d++) {
    double ep[2], em[2];
    sim3_edge_error(Sk[2 * d][0], P2, cam, o1, ep);
    sim3_edge_error(Sk[2 * d + 1][0], P2, cam, o1, em);
    sim3_jac_col(ep, em, J12, d);
    sim3_edge_error(Sk[2 * d][1], P1, cam + 4, o2, ep);
    sim3_edge_error(Sk[2 * d + 1][1], P1, cam + 4, o2, em);
    sim3_jac_col(ep, em, J21, d);
  }
}
}
