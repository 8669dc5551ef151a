// Per-branch arithmetic of the WLS state estimator (estimate.cu), fp64: the pi-model flows of data.py:370-376 (phase shift ignored,
// data.py:362-363) and their partials with respect to (theta_i, V_i, theta_j, V_j), the rows of the measurement Jacobian H that a
// branch contributes (SURVEY.md Appendix B.1 / B.2).  Plain inline functions, compiled for the device by estimate.cu and for the host
// by tests/host_math/estimate_host.cpp, which lets a CPU test check them against torch autograd without a GPU.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define EST_HD __host__ __device__ __forceinline__
#else
#define EST_HD inline
#endif

struct EstBranch {
  double pf, qf, pt, qt;   // MW / MVAr
  double d[4][4];          // d[flow][var]: flow in (pf, qf, pt, qt), var in (theta_i, V_i, theta_j, V_j)
};

// g, b, gs, bs: edge_attr columns 6-9; c = V_lv^2 (V_lv = min vn_kv of the grid)
EST_HD void est_branch(double vi, double vj, double thi, double thj, double g, double b, double gs, double bs, double c,
                       EstBranch& o) {
  double sn, cs;
#if defined(__CUDA_ARCH__)
  sincos(thi - thj, &sn, &cs);
#else
  sn = sin(thi - thj);
  cs = cos(thi - thj);
#endif
  const double A = g * cs + b * sn, Bm = -g * sn + b * cs;    // from side: P_f, Q_f bracket; dA/ddelta = Bm, dBm/ddelta = -A
  const double A2 = g * cs - b * sn, B2 = g * sn + b * cs;    // to side: dA2/ddelta = -B2, dB2/ddelta = A2
  const double gsh = g + gs / 2, bsh = b + bs / 2;
  const double vv = vi * vj, cvv = c * vv;
  o.pf = (-vv * A + gsh * vi * vi) * c;
  o.qf = (vv * Bm - bsh * vi * vi) * c;
  o.pt = (-vv * A2 + gsh * vj * vj) * c;
  o.qt = (vv * B2 - bsh * vj * vj) * c;
  // d/dtheta_j = -d/dtheta_i for every flow
  o.d[0][0] = -cvv * Bm;
  o.d[0][1] = c * (-vj * A + 2 * gsh * vi);
  o.d[0][3] = -c * vi * A;
  o.d[1][0] = -cvv * A;
  o.d[1][1] = c * (vj * Bm - 2 * bsh * vi);
  o.d[1][3] = c * vi * Bm;
  o.d[2][0] = cvv * B2;
  o.d[2][1] = -c * vj * A2;
  o.d[2][3] = c * (-vi * A2 + 2 * gsh * vj);
  o.d[3][0] = cvv * A2;
  o.d[3][1] = c * vj * B2;
  o.d[3][3] = c * (vi * B2 - 2 * bsh * vj);
  for (int f = 0; f < 4; ++f) o.d[f][2] = -o.d[f][0];
}

// a measurement of the loss (data.py:397-409): the de-normalised value, 0 where the normalised value is exactly 0 (absent)
EST_HD double est_unnorm(float z, float sd, float mu) { return z != 0.0f ? (double)z * (double)sd + (double)mu : 0.0; }
