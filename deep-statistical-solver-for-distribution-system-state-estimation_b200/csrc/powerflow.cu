// (f-2) Batched AC power flow: Newton-Raphson in polar form, fp64, on the reference's pi-model (data.py:370-376, phase shift ignored), the
// offline solve the reference does with pandapower runpp (toy_network.py:160-250).  One slack bus, PQ buses, one topology per call.
//   k_pf_newton  one thread per scenario of a chunk.  Per iteration: mismatch S_calc - S_spec over the PQ buses from Y (CSR, MVA at 1 pu);
//                if max |.| <= tol stop; else assemble the reduced Jacobian as 2x2 blocks (dP/dth, dP/dV; dQ/dth, dQ/dV) on the host's
//                block pattern, factorise it row by row (IKJ block LU in the host's elimination order, diagonal pivots inverted in place),
//                forward / back substitution, update (th, V).  At the end: the state and the slack injection.
//   k_pf_flows   one thread per (scenario, closed edge): the pi-model branch flows of the solved state, rounded as synth.branch_flows.
// Workspace: per chunk of C scenarios, 4 N + 2 n + 4 * blocks doubles per scenario, stored index-major ([index][C]) so that the threads of
// a warp touch consecutive addresses.  No atomics: every sum is one thread's loop in a fixed order, so a scenario's result does not
// depend on the other scenarios of the call or on the chunk size.  A singular pivot or max_iter updates without convergence give
// converged = 0 for that scenario only.
#include <math.h>

#include "block_lu.cuh"
#include "common.cuh"

namespace {

constexpr int PF_THREADS = 128;

struct PfArgs {
  dss2_pf_topology_t t;
  int64_t S, s0, C;              // scenarios, first scenario of this chunk, chunk stride of the workspace
  const double *p, *q, *vs;      // [S,N] load-positive injections, [S] slack voltage
  double tol;
  int max_iter;
  double *vm, *va, *p_out, *q_out;
  int32_t* iters;
  uint8_t* conv;
  double* mism;
  double* ws;
};

// S_calc of bus i (MVA): U_i conj(sum_j Y_ij U_j) with U = e + j f
__device__ __forceinline__ void bus_power(const dss2_pf_topology_t& t, const double* e, const double* f, int64_t C, int i, double& P,
                                          double& Q) {
  double ir = 0.0, ii = 0.0;
  for (int z = __ldg(t.y_ptr + i); z < __ldg(t.y_ptr + i + 1); ++z) {
    const int j = __ldg(t.y_col + z);
    const double g = __ldg(t.y_gb + 2 * z), b = __ldg(t.y_gb + 2 * z + 1);
    const double ej = e[j * C], fj = f[j * C];
    ir += g * ej - b * fj;
    ii += g * fj + b * ej;
  }
  const double ei = e[i * C], fi = f[i * C];
  P = ei * ir + fi * ii;
  Q = fi * ir - ei * ii;
}

__global__ void __launch_bounds__(PF_THREADS) k_pf_newton(PfArgs a) {
  const int64_t c = blockIdx.x * (int64_t)PF_THREADS + threadIdx.x;
  const int64_t s = a.s0 + c;
  if (s >= a.S || c >= a.C) return;
  const dss2_pf_topology_t& t = a.t;
  const int N = t.num_buses, n = t.num_pq;
  const int64_t C = a.C;
  // this thread's columns of the workspace
  double* V = a.ws + c;
  double* th = V + (int64_t)N * C;
  double* e = th + (int64_t)N * C;
  double* f = e + (int64_t)N * C;
  double* F = f + (int64_t)N * C;           // [2n]: mismatch (P rows then Q rows), then the Newton step in place
  double* A = F + (int64_t)2 * n * C;       // [blocks][4]
  const double* ps = a.p + s * N;
  const double* qs = a.q + s * N;

  for (int i = 0; i < N; ++i) {
    V[i * C] = i == t.slack ? a.vs[s] : 1.0;
    th[i * C] = 0.0;
  }
  int it = 0;
  bool ok = false;
  double mx = 0.0;
  for (;; ++it) {
    for (int i = 0; i < N; ++i) {
      double sn, cs;
      sincos(th[i * C], &sn, &cs);
      e[i * C] = V[i * C] * cs;
      f[i * C] = V[i * C] * sn;
    }
    // mismatch over the PQ buses, in elimination order
    mx = 0.0;
    for (int k = 0; k < n; ++k) {
      const int i = __ldg(t.bus + k);
      double P, Q;
      bus_power(t, e, f, C, i, P, Q);
      const double dp = P + ps[i], dq = Q + qs[i];   // S_spec = -(p + j q)
      F[k * C] = dp;
      F[(n + k) * C] = dq;
      mx = fmax(mx, fmax(fabs(dp), fabs(dq)));
    }
    if (mx <= a.tol) {
      ok = true;
      break;
    }
    if (it == a.max_iter) break;
    // Jacobian blocks, row k = bus i, column m = bus j
    for (int k = 0; k < n; ++k) {
      const int i = __ldg(t.bus + k);
      const double ei = e[i * C], fi = f[i * C], Vi = V[i * C];
      for (int p = __ldg(t.blk_ptr + k); p < __ldg(t.blk_ptr + k + 1); ++p) {
        const int yz = __ldg(t.blk_y + p);
        Blk J = {0.0, 0.0, 0.0, 0.0};
        if (yz >= 0) {
          const double g = __ldg(t.y_gb + 2 * yz), b = __ldg(t.y_gb + 2 * yz + 1);
          const int m = __ldg(t.blk_col + p);
          if (m == k) {
            const double P = F[k * C] - ps[i], Q = F[(n + k) * C] - qs[i];
            J = {-Q - b * Vi * Vi, P / Vi + g * Vi, P - g * Vi * Vi, Q / Vi - b * Vi};
          } else {
            const int j = __ldg(t.bus + m);
            const double ej = e[j * C], fj = f[j * C], Vj = V[j * C];
            const double cr = ei * ej + fi * fj, sr = fi * ej - ei * fj;   // Vi Vj cos(th_ij), Vi Vj sin(th_ij)
            const double u = g * sr - b * cr, w = g * cr + b * sr;
            J = {u, w / Vj, -w, u / Vj};
          }
        }
        st_blk(A, C, p, J);
      }
    }
    // block LU (block_lu.cuh), forward / back substitution, then the update (th, V) -= x
    const BlockLu lu = {n, t.blk_ptr, t.blk_col, t.diag, t.upd_ptr, t.upd};
    if (!block_lu_factor(lu, A, C)) break;
    block_lu_solve(lu, A, F, C);
    for (int k = n - 1; k >= 0; --k) {
      const int i = __ldg(t.bus + k);
      th[i * C] -= F[k * C];
      V[i * C] -= F[(n + k) * C];
    }
  }
  // the state, and the slack injection in the load-positive convention
  for (int i = 0; i < N; ++i) {
    a.vm[s * N + i] = V[i * C];
    a.va[s * N + i] = th[i * C];
  }
  double P, Q;
  bus_power(t, e, f, C, t.slack, P, Q);
  a.p_out[s * N + t.slack] = -P;
  a.q_out[s * N + t.slack] = -Q;
  a.iters[s] = it;
  a.conv[s] = ok ? 1 : 0;
  a.mism[s] = mx;
}

// synth.branch_flows (data.py:370-376) with its operation order, every product and sum rounded on its own
__global__ void __launch_bounds__(256) k_pf_flows(const int32_t* __restrict__ ft, const double* __restrict__ gb, int E, int N, int64_t S,
                                                  double base, const double* __restrict__ vm, const double* __restrict__ va,
                                                  double* __restrict__ pf, double* __restrict__ qf, double* __restrict__ pt,
                                                  double* __restrict__ qt) {
  const int64_t total = S * E;
  for (int64_t r = blockIdx.x * 256ll + threadIdx.x; r < total; r += (int64_t)gridDim.x * 256) {
    const int64_t s = r / E;
    const int e = (int)(r % E);
    const int fb = ft[2 * e], tb = ft[2 * e + 1];
    const double g = gb[4 * e], b = gb[4 * e + 1], gs = gb[4 * e + 2], bs = gb[4 * e + 3];
    const double vi = vm[s * N + fb], vj = vm[s * N + tb];
    const double d = __dsub_rn(va[s * N + fb], va[s * N + tb]);
    const double c = cos(d), sn = sin(d);
    const double vv = __dmul_rn(-vi, vj);
    const double gsh = __dadd_rn(g, __dmul_rn(gs, 0.5)), bsh = __dadd_rn(b, __dmul_rn(bs, 0.5));
    const double vi2 = __dmul_rn(vi, vi), vj2 = __dmul_rn(vj, vj), vivj = __dmul_rn(vi, vj);
    pf[r] = __dmul_rn(__dadd_rn(__dmul_rn(vv, __dadd_rn(__dmul_rn(g, c), __dmul_rn(b, sn))), __dmul_rn(gsh, vi2)), base);
    qf[r] = __dmul_rn(__dsub_rn(__dmul_rn(vivj, __dadd_rn(__dmul_rn(-g, sn), __dmul_rn(b, c))), __dmul_rn(bsh, vi2)), base);
    pt[r] = __dmul_rn(__dadd_rn(__dmul_rn(vv, __dsub_rn(__dmul_rn(g, c), __dmul_rn(b, sn))), __dmul_rn(gsh, vj2)), base);
    qt[r] = __dmul_rn(__dsub_rn(__dmul_rn(vivj, __dadd_rn(__dmul_rn(g, sn), __dmul_rn(b, c))), __dmul_rn(bsh, vj2)), base);
  }
}

}  // namespace

extern "C" size_t dss2_powerflow_workspace_bytes(const dss2_pf_topology_t* t, int64_t chunk) {
  if (!t || chunk < 1) return 0;
  return (size_t)chunk * sizeof(double) * (4 * (size_t)t->num_buses + 2 * (size_t)t->num_pq + 4 * (size_t)t->num_blocks);
}

extern "C" int dss2_powerflow(const dss2_pf_topology_t* topo, int64_t S, const double* p_mw, const double* q_mvar, const double* v_slack,
                              double tol_mva, int max_iter, double* vm_pu, double* va_rad, double* p_out, double* q_out, double* p_from,
                              double* q_from, double* p_to, double* q_to, int32_t* iterations, uint8_t* converged, double* max_mismatch,
                              void* workspace, size_t workspace_bytes, int64_t chunk, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(topo && p_mw && q_mvar && v_slack && vm_pu && va_rad && p_out && q_out && p_from && q_from && p_to && q_to && iterations &&
                     converged && max_mismatch && workspace,
                 "dss2_powerflow: null argument");
  const dss2_pf_topology_t& t = *topo;
  DSS2_CHECK_ARG(t.num_buses >= 2 && t.num_pq == t.num_buses - 1 && t.slack >= 0 && t.slack < t.num_buses && t.num_blocks >= t.num_pq &&
                     t.num_edges >= 1 && t.num_updates >= 0 && t.v_lv > 0.0,
                 "dss2_powerflow: bad topology sizes");
  DSS2_CHECK_ARG(t.y_ptr && t.y_col && t.y_gb && t.bus && t.blk_ptr && t.blk_col && t.blk_y && t.diag && t.upd_ptr && t.edge_ft && t.edge_gb &&
                     (t.upd || t.num_updates == 0),
                 "dss2_powerflow: null topology array");
  DSS2_CHECK_ARG(S >= 1 && chunk >= 1 && max_iter >= 0 && tol_mva > 0.0, "dss2_powerflow: bad sizes or tolerance");
  const int64_t C = chunk < S ? chunk : S;
  DSS2_CHECK_ARG(workspace_bytes >= dss2_powerflow_workspace_bytes(topo, C), "dss2_powerflow: workspace too small for %lld scenarios",
                 (long long)C);
  PfArgs a = {};
  a.t = t;
  a.S = S;
  a.C = C;
  a.p = p_mw;
  a.q = q_mvar;
  a.vs = v_slack;
  a.tol = tol_mva;
  a.max_iter = max_iter;
  a.vm = vm_pu;
  a.va = va_rad;
  a.p_out = p_out;
  a.q_out = q_out;
  a.iters = iterations;
  a.conv = converged;
  a.mism = max_mismatch;
  a.ws = (double*)workspace;
  for (int64_t s0 = 0; s0 < S; s0 += C) {
    a.s0 = s0;
    const int64_t m = (S - s0) < C ? (S - s0) : C;
    k_pf_newton<<<(unsigned)((m + PF_THREADS - 1) / PF_THREADS), PF_THREADS, 0, stream>>>(a);
    DSS2_LAUNCH_CHECK();
  }
  const int64_t total = S * t.num_edges;
  const int grid = (int)(((total + 255) / 256) < (int64_t)dss2_sm_count() * 16 ? (total + 255) / 256 : (int64_t)dss2_sm_count() * 16);
  k_pf_flows<<<grid, 256, 0, stream>>>(t.edge_ft, t.edge_gb, t.num_edges, t.num_buses, S, t.v_lv * t.v_lv, vm_pu, va_rad, p_from, q_from,
                                        p_to, q_to);
  DSS2_LAUNCH_CHECK();
  return 0;
}
