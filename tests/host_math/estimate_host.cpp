// TEST HARNESS (not product code): runs the per-branch math of csrc/estimate_math.cuh on the host so that a CPU test can compare
// the estimator's flows and hand-derived partials with torch autograd.  Built by tests/test_wls_estimate.py with g++ -ffp-contract=off.
#include <stdint.h>

#include "../../deep-statistical-solver-for-distribution-system-state-estimation_b200/csrc/estimate_math.cuh"

// in [E,8] = (V_i, V_j, th_i, th_j, G, B, Gs, Bs); out [E,20] = (P_f, Q_f, P_t, Q_t, d[4][4] row-major)
extern "C" int est_host_branch(const double* in, int64_t E, double c, double* out) {
  for (int64_t e = 0; e < E; ++e) {
    const double* r = in + 8 * e;
    EstBranch b;
    est_branch(r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], c, b);
    double* o = out + 20 * e;
    o[0] = b.pf;
    o[1] = b.qf;
    o[2] = b.pt;
    o[3] = b.qt;
    for (int f = 0; f < 4; ++f)
      for (int k = 0; k < 4; ++k) o[4 + 4 * f + k] = b.d[f][k];
  }
  return 0;
}
