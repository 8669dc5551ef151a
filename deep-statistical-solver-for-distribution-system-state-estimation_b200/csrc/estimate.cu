// Classical WLS state estimation, batched (include/dss2_b200.h, dss2_wls_estimate): Gauss-Newton on the measurements of the
// physics-informed loss (data.py:393-459), the estimator the reference runs beside DSS2 (case_study.py:1226-1357).  fp64, the factorisation double-double.
//   k_wls_estimate  one thread per scenario of a chunk.  Per iteration:
//     1. branch flows and their 16 partials w.r.t. (th_i, V_i, th_j, V_j), once per edge (estimate_math.cuh), into the workspace;
//        the partials w.r.t. the slack's th are dropped (th_slack = 0 is not an unknown);
//     2. per bus, the V and th rows, and the p and q rows over its support {i} u nbr(i) with their residuals;
//     3. per measured edge, the P_f and Q_f rows over {i, j};
//     4. both accumulated into H^T W H (2x2 blocks on the host's pattern) and H^T W r in one pass; the slack's th row and column
//        are identity;
//     5. block LU and substitutions (block_lu.cuh, shared with k_pf_newton) in double-double: the gain matrix is assembled in fp64,
//        but its Schur complements cancel by up to 16 digits where a pseudo-measurement of a small load carries a weight near 1e12,
//        and an fp64 factorisation then returns a step with no correct digit (2 % of the noisy Oberrhein scenarios);
//     6. (th, V) += alpha dx, alpha = 1, 1/2, 1/4, ... the first that does not increase J_s beyond rounding;
//     7. stop when the full step max |dx| <= tol (converged) or after max_iter updates.
//   J_s is returned at the final state.
// Workspace per chunk of C scenarios: 16 N + 28 E + 8 blocks + 4 max_support doubles per scenario, stored index-major ([index][C]) so
// that the threads of a warp touch consecutive addresses.  No atomics: every sum is one thread's loop in a fixed order, so a scenario's
// result does not depend on the other scenarios of the call or on the chunk size.
#include <math.h>

#include "block_lu.cuh"
#include "common.cuh"
#include "estimate_math.cuh"

namespace {

// one warp per block: a batch of a few thousand scenarios still spreads over most of the 148 SMs
constexpr int SE_THREADS = 32;

struct SeArgs {
  dss2_se_topology_t t;
  int64_t B, s0, C;              // scenarios, first scenario of this chunk, chunk stride of the workspace
  const float *x, *ea, *st;      // x [B N, xs], edge_attr [B E, es], stats28
  int64_t xs, es;
  double w_v, w_p, w_pf, tol;
  int max_iter;
  double *vm, *va, *obj, *step;
  float* out;
  int32_t* iters;
  uint8_t* conv;
  double* ws;
};

// the gain matrix and right-hand side are accumulated in fp64 into the high parts of their double-double workspace (block_lu.cuh DD)
__device__ __forceinline__ void add_blk(double* A, int64_t C, int p, double a, double b, double c, double d) {
  double* r = A + (int64_t)8 * p * C;
  r[0] += a;
  r[2 * C] += b;
  r[4 * C] += c;
  r[6 * C] += d;
}

// flows (and, with partials, the 16 partials) of every edge at the current state into fl [20][E]
__device__ __forceinline__ void edge_pass(const dss2_se_topology_t& t, const double* V, const double* th, const double* prm, double c2,
                                          double* fl, int64_t C, bool partials) {
  const int E = t.num_edges;
  for (int e = 0; e < E; ++e) {
    const int i = __ldg(t.edge_ft + 2 * e), j = __ldg(t.edge_ft + 2 * e + 1);
    EstBranch b;
    est_branch(V[i * C], V[j * C], th[i * C], th[j * C], prm[e * C], prm[(E + e) * C], prm[(2 * E + e) * C], prm[(3 * E + e) * C], c2, b);
    fl[e * C] = b.pf;
    fl[(E + e) * C] = b.qf;
    fl[(2 * E + e) * C] = b.pt;
    fl[(3 * E + e) * C] = b.qt;
    if (!partials) continue;
    const double mi = i == t.slack ? 0.0 : 1.0, mj = j == t.slack ? 0.0 : 1.0;
#pragma unroll
    for (int f = 0; f < 4; ++f) {
      fl[((4 + 4 * f) * E + e) * C] = b.d[f][0] * mi;
      fl[((5 + 4 * f) * E + e) * C] = b.d[f][1];
      fl[((6 + 4 * f) * E + e) * C] = b.d[f][2] * mj;
      fl[((7 + 4 * f) * E + e) * C] = b.d[f][3];
    }
  }
}

// rows of p_n and q_n over the support of bus n (m slots) into H [4][m] = (dp/dth, dp/dV, dq/dth, dq/dV), and p_n, q_n themselves
__device__ __forceinline__ void bus_rows(const dss2_se_topology_t& t, int n, int m, const double* fl, double* H, int64_t C, double& P,
                                         double& Q) {
  const int E = t.num_edges;
  for (int k = 0; k < 4 * m; ++k) H[k * C] = 0.0;
  P = 0.0;
  Q = 0.0;
  for (int z = __ldg(t.inc_ptr + n); z < __ldg(t.inc_ptr + n + 1); ++z) {
    const int e = __ldg(t.inc + 3 * z), end = __ldg(t.inc + 3 * z + 1), o = __ldg(t.inc + 3 * z + 2);
    const int fp = 2 * end, fq = 2 * end + 1;          // (P_f, Q_f) at the from-end, (P_t, Q_t) at the to-end
    const int vs = 2 * end, vo = 2 - 2 * end;          // this bus's (th, V) partials, the other end's
    P -= fl[(fp * E + e) * C];
    Q -= fl[(fq * E + e) * C];
    H[0] -= fl[((4 + 4 * fp + vs) * E + e) * C];
    H[(int64_t)m * C] -= fl[((5 + 4 * fp + vs) * E + e) * C];
    H[(int64_t)2 * m * C] -= fl[((4 + 4 * fq + vs) * E + e) * C];
    H[(int64_t)3 * m * C] -= fl[((5 + 4 * fq + vs) * E + e) * C];
    H[o * C] -= fl[((4 + 4 * fp + vo) * E + e) * C];
    H[(m + o) * C] -= fl[((5 + 4 * fp + vo) * E + e) * C];
    H[(2 * m + o) * C] -= fl[((4 + 4 * fq + vo) * E + e) * C];
    H[(3 * m + o) * C] -= fl[((5 + 4 * fq + vo) * E + e) * C];
  }
}

// J_s at the current state: the flows (values only) into fl, then bus terms and edge terms in a fixed order
__device__ __forceinline__ double objective(const dss2_se_topology_t& t, const double* V, const double* th, const double* Zb, const double* Wb,
                                            const double* Ze, const double* We, const double* prm, double c2, double* fl, int64_t C) {
  const int N = t.num_buses, E = t.num_edges;
  edge_pass(t, V, th, prm, c2, fl, C, false);
  double J = 0.0;
  for (int n = 0; n < N; ++n) {
    double P = 0.0, Q = 0.0;
    for (int z = __ldg(t.inc_ptr + n); z < __ldg(t.inc_ptr + n + 1); ++z) {
      const int e = __ldg(t.inc + 3 * z), end = __ldg(t.inc + 3 * z + 1);
      P -= fl[(2 * end * E + e) * C];
      Q -= fl[((2 * end + 1) * E + e) * C];
    }
    const double d0 = Zb[n * C] - V[n * C], d1 = Zb[(N + n) * C] - th[n * C];
    const double d2 = Zb[(2 * N + n) * C] - P, d3 = Zb[(3 * N + n) * C] - Q;
    J += Wb[n * C] * d0 * d0 + Wb[(N + n) * C] * d1 * d1 + Wb[(2 * N + n) * C] * d2 * d2 + Wb[(3 * N + n) * C] * d3 * d3;
  }
  for (int e = 0; e < E; ++e) {
    const double d0 = Ze[e * C] - fl[e * C], d1 = Ze[(E + e) * C] - fl[(E + e) * C];
    J += We[e * C] * d0 * d0 + We[(E + e) * C] * d1 * d1;
  }
  return J;
}

__global__ void __launch_bounds__(SE_THREADS, 12) k_wls_estimate(SeArgs a) {
  const int64_t c = blockIdx.x * (int64_t)SE_THREADS + threadIdx.x;
  const int64_t s = a.s0 + c;
  if (s >= a.B || c >= a.C) return;
  const dss2_se_topology_t& t = a.t;
  const int N = t.num_buses, E = t.num_edges;
  const int64_t C = a.C;
  // this thread's columns of the workspace
  double* V = a.ws + c;
  double* th = V + (int64_t)N * C;
  double* Zb = th + (int64_t)N * C;          // [4][N] bus measurements (V, th, p, q)
  double* Wb = Zb + (int64_t)4 * N * C;      // [4][N] their weights times w_v / w_p
  double* Ze = Wb + (int64_t)4 * N * C;      // [2][E] P_f, Q_f measurements
  double* We = Ze + (int64_t)2 * E * C;      // [2][E] their weights times w_pf
  double* prm = We + (int64_t)2 * E * C;     // [4][E] G, B, Gs, Bs
  double* fl = prm + (int64_t)4 * E * C;     // [20][E] P_f, Q_f, P_t, Q_t, then d(flow f)/d(var k) at row 4 + 4 f + k
  double* F = fl + (int64_t)20 * E * C;      // [2N] dd: right-hand side by position (th rows, then V rows), then the step
  double* A = F + (int64_t)4 * N * C;        // [blocks][4] dd
  double* H = A + (int64_t)8 * t.num_blocks * C;   // [4][max_support] rows of p (th, V) and q (th, V) over one bus's support
  double* Vo = H + (int64_t)4 * t.max_support * C; // [N] the state before the step, for the line search
  double* tho = Vo + (int64_t)N * C;

  // measurements of the loss (data.py:397-409), promoted to fp64
  const float* xs = a.x + s * N * a.xs;
  const float* es = a.ea + s * E * a.es;
  float vlv = __ldg(xs + 8);
  for (int n = 0; n < N; ++n) {
    const float* r = xs + n * a.xs;
    vlv = fminf(vlv, __ldg(r + 8));
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      Zb[(k * N + n) * C] = est_unnorm(__ldg(r + 2 * k), __ldg(a.st + 8 + 2 * k), __ldg(a.st + 2 * k));
      Wb[(k * N + n) * C] = (k < 2 ? a.w_v : a.w_p) * est_unnorm(__ldg(r + 2 * k + 1), __ldg(a.st + 8 + 2 * k + 1), __ldg(a.st + 2 * k + 1));
    }
    V[n * C] = 1.0;
    th[n * C] = 0.0;
  }
  for (int e = 0; e < E; ++e) {
    const float* r = es + e * a.es;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      Ze[(k * E + e) * C] = est_unnorm(__ldg(r + 2 * k), __ldg(a.st + 22 + 2 * k), __ldg(a.st + 16 + 2 * k));
      We[(k * E + e) * C] = a.w_pf * est_unnorm(__ldg(r + 2 * k + 1), __ldg(a.st + 22 + 2 * k + 1), __ldg(a.st + 16 + 2 * k + 1));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) prm[(k * E + e) * C] = (double)__ldg(r + 6 + k);
  }
  const double c2 = (double)vlv * (double)vlv;
  const BlockLu lu = {N, t.blk_ptr, t.blk_col, t.diag, t.upd_ptr, t.upd};
  const int slack_diag = __ldg(t.pair_blk + __ldg(t.pair_ptr + t.slack));
  const int slack_pos = __ldg(t.sup_pos + __ldg(t.sup_ptr + t.slack));

  int it = 0;
  bool ok = false;
  double mx = 0.0;
  double J = objective(t, V, th, Zb, Wb, Ze, We, prm, c2, fl, C);
  while (it < a.max_iter) {
    edge_pass(t, V, th, prm, c2, fl, C, true);
    for (int p = 0; p < 8 * t.num_blocks; ++p) A[p * C] = 0.0;
    for (int k = 0; k < 4 * N; ++k) F[k * C] = 0.0;
    // buses: V, th, then p and q over the support
    for (int n = 0; n < N; ++n) {
      const int s0 = __ldg(t.sup_ptr + n), m = __ldg(t.sup_ptr + n + 1) - s0;
      const int p0 = __ldg(t.pair_ptr + n);
      const int kn = __ldg(t.sup_pos + s0), dn = __ldg(t.pair_blk + p0);
      const double wv = Wb[n * C], wt = Wb[(N + n) * C], wp = Wb[(2 * N + n) * C], wq = Wb[(3 * N + n) * C];
      if (wv != 0.0) {
        add_blk(A, C, dn, 0.0, 0.0, 0.0, wv);
        F[2 * (N + kn) * C] += wv * (Zb[n * C] - V[n * C]);
      }
      if (wt != 0.0 && n != t.slack) {
        add_blk(A, C, dn, wt, 0.0, 0.0, 0.0);
        F[2 * kn * C] += wt * (Zb[(N + n) * C] - th[n * C]);
      }
      if (wp == 0.0 && wq == 0.0) continue;
      double P, Q;
      bus_rows(t, n, m, fl, H, C, P, Q);
      const double rp = wp * (Zb[(2 * N + n) * C] - P), rq = wq * (Zb[(3 * N + n) * C] - Q);
      for (int u = 0; u < m; ++u) {
        const double pta = H[u * C], pva = H[(m + u) * C], qta = H[(2 * m + u) * C], qva = H[(3 * m + u) * C];
        const int ka = __ldg(t.sup_pos + s0 + u);
        F[2 * ka * C] += rp * pta + rq * qta;
        F[2 * (N + ka) * C] += rp * pva + rq * qva;
        const double wpa = wp * pta, wpv = wp * pva, wqa = wq * qta, wqv = wq * qva;
        for (int v = 0; v < m; ++v) {
          const double ptb = H[v * C], pvb = H[(m + v) * C], qtb = H[(2 * m + v) * C], qvb = H[(3 * m + v) * C];
          add_blk(A, C, __ldg(t.pair_blk + p0 + u * m + v), wpa * ptb + wqa * qtb, wpa * pvb + wqa * qvb, wpv * ptb + wqv * qtb,
                  wpv * pvb + wqv * qvb);
        }
      }
    }
    // measured edges: P_f and Q_f over (th_i, V_i, th_j, V_j)
    for (int e = 0; e < E; ++e) {
      const double w0 = We[e * C], w1 = We[(E + e) * C];
      if (w0 == 0.0 && w1 == 0.0) continue;
      const int i = __ldg(t.edge_ft + 2 * e), j = __ldg(t.edge_ft + 2 * e + 1);
      const int ki = __ldg(t.sup_pos + __ldg(t.sup_ptr + i)), kj = __ldg(t.sup_pos + __ldg(t.sup_ptr + j));
      double hp[4], hq[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        hp[k] = fl[((4 + k) * E + e) * C];
        hq[k] = fl[((8 + k) * E + e) * C];
      }
      const double r0 = w0 * (Ze[e * C] - fl[e * C]), r1 = w1 * (Ze[(E + e) * C] - fl[(E + e) * C]);
      F[2 * ki * C] += r0 * hp[0] + r1 * hq[0];
      F[2 * (N + ki) * C] += r0 * hp[1] + r1 * hq[1];
      F[2 * kj * C] += r0 * hp[2] + r1 * hq[2];
      F[2 * (N + kj) * C] += r0 * hp[3] + r1 * hq[3];
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int ra = 2 * u, cb = 2 * v;
          add_blk(A, C, __ldg(t.edge_blk + 4 * e + 2 * u + v),
                  w0 * hp[ra] * hp[cb] + w1 * hq[ra] * hq[cb], w0 * hp[ra] * hp[cb + 1] + w1 * hq[ra] * hq[cb + 1],
                  w0 * hp[ra + 1] * hp[cb] + w1 * hq[ra + 1] * hq[cb], w0 * hp[ra + 1] * hp[cb + 1] + w1 * hq[ra + 1] * hq[cb + 1]);
        }
    }
    // th_slack is not an unknown: identity in its row and column (every other entry there is zero), zero right-hand side
    A[(int64_t)8 * slack_diag * C] = 1.0;
    F[(int64_t)2 * slack_pos * C] = 0.0;
    if (!block_lu_factor<DD>(lu, A, C)) break;
    block_lu_solve<DD>(lu, A, F, C);
    for (int k = 0; k < 2 * N; ++k) F[k * C] = F[2 * k * C] + F[(2 * k + 1) * C];   // the step, rounded to fp64, packed
    mx = 0.0;
    bool finite = true;
    for (int k = 0; k < N; ++k) {
      const double dt = F[k * C], dv = F[(N + k) * C];
      finite = finite && isfinite(dt) && isfinite(dv);
      mx = fmax(mx, fmax(fabs(dt), fabs(dv)));
    }
    if (!finite) {
      mx = NAN;
      break;
    }
    // step halving until J_s does not grow beyond rounding: plain Gauss-Newton diverges from the flat start on scenarios with large
    // residuals; near the solution the full step is taken
    for (int i = 0; i < N; ++i) {
      Vo[i * C] = V[i * C];
      tho[i * C] = th[i * C];
    }
    double alpha = 1.0, Jn = 0.0;
    bool descent = false;
    for (int h = 0; h < 40 && !descent; ++h, alpha *= 0.5) {
      for (int k = 0; k < N; ++k) {
        const int i = __ldg(t.bus + k);
        th[i * C] = tho[i * C] + alpha * F[k * C];
        V[i * C] = Vo[i * C] + alpha * F[(N + k) * C];
      }
      Jn = objective(t, V, th, Zb, Wb, Ze, We, prm, c2, fl, C);
      descent = Jn <= J + 1e-12 * J;
    }
    if (!descent) {
      for (int i = 0; i < N; ++i) {
        V[i * C] = Vo[i * C];
        th[i * C] = tho[i * C];
      }
      break;
    }
    J = Jn;
    ++it;
    if (mx <= a.tol) {
      ok = true;
      break;
    }
  }

  if (!isfinite(J)) ok = false;
  const float xm0 = __ldg(a.st), xs0 = __ldg(a.st + 8);
  for (int n = 0; n < N; ++n) {
    const double v = V[n * C], h = th[n * C];
    a.vm[s * N + n] = v;
    a.va[s * N + n] = h;
    a.out[2 * (s * N + n)] = (float)((v - (double)xm0) / (double)xs0);
    a.out[2 * (s * N + n) + 1] = (float)h;
  }
  a.obj[s] = J;
  a.iters[s] = it;
  a.conv[s] = ok ? 1 : 0;
  a.step[s] = mx;
}

}  // namespace

extern "C" size_t dss2_wls_estimate_workspace_bytes(const dss2_se_topology_t* t, int64_t chunk) {
  if (!t || chunk < 1) return 0;
  return (size_t)chunk * sizeof(double) *
         (16 * (size_t)t->num_buses + 28 * (size_t)t->num_edges + 8 * (size_t)t->num_blocks + 4 * (size_t)t->max_support);
}

extern "C" int dss2_wls_estimate(const dss2_se_topology_t* topo, int64_t B, const float* x, int64_t x_stride, const float* edge_attr,
                                 int64_t ea_stride, const float* stats28, double w_v, double w_p, double w_pf, double tol, int max_iter,
                                 double* vm_pu, double* va_rad, float* output, double* objective, int32_t* iterations,
                                 uint8_t* converged, double* max_step, void* workspace, size_t workspace_bytes, int64_t chunk,
                                 void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(topo && x && edge_attr && stats28 && vm_pu && va_rad && output && objective && iterations && converged && max_step &&
                     workspace,
                 "dss2_wls_estimate: null argument");
  const dss2_se_topology_t& t = *topo;
  DSS2_CHECK_ARG(t.num_buses >= 2 && t.num_edges >= 1 && t.slack >= 0 && t.slack < t.num_buses && t.num_blocks >= t.num_buses &&
                     t.num_updates >= 0 && t.num_pairs >= t.num_buses && t.max_support >= 1,
                 "dss2_wls_estimate: bad topology sizes");
  DSS2_CHECK_ARG(t.edge_ft && t.inc_ptr && t.inc && t.sup_ptr && t.sup_pos && t.pair_ptr && t.pair_blk && t.edge_blk && t.bus && t.blk_ptr &&
                     t.blk_col && t.diag && t.upd_ptr && (t.upd || t.num_updates == 0),
                 "dss2_wls_estimate: null topology array");
  DSS2_CHECK_ARG(B >= 1 && chunk >= 1 && max_iter >= 0 && tol > 0.0 && x_stride >= 11 && ea_stride >= 13,
                 "dss2_wls_estimate: bad sizes, strides or tolerance");
  const int64_t C = chunk < B ? chunk : B;
  DSS2_CHECK_ARG(workspace_bytes >= dss2_wls_estimate_workspace_bytes(topo, C), "dss2_wls_estimate: workspace too small for %lld scenarios",
                 (long long)C);
  SeArgs a = {};
  a.t = t;
  a.B = B;
  a.C = C;
  a.x = x;
  a.ea = edge_attr;
  a.st = stats28;
  a.xs = x_stride;
  a.es = ea_stride;
  a.w_v = w_v;
  a.w_p = w_p;
  a.w_pf = w_pf;
  a.tol = tol;
  a.max_iter = max_iter;
  a.vm = vm_pu;
  a.va = va_rad;
  a.out = output;
  a.obj = objective;
  a.iters = iterations;
  a.conv = converged;
  a.step = max_step;
  a.ws = (double*)workspace;
  for (int64_t s0 = 0; s0 < B; s0 += C) {
    a.s0 = s0;
    const int64_t m = (B - s0) < C ? (B - s0) : C;
    k_wls_estimate<<<(unsigned)((m + SE_THREADS - 1) / SE_THREADS), SE_THREADS, 0, stream>>>(a);
    DSS2_LAUNCH_CHECK();
  }
  return 0;
}
