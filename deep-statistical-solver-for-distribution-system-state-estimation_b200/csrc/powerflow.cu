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

struct Blk {
  double a, b, c, d;             // [[a, b], [c, d]]
};

__device__ __forceinline__ Blk ld_blk(const double* A, int64_t C, int p) {
  const double* r = A + (int64_t)4 * p * C;
  return {r[0], r[C], r[2 * C], r[3 * C]};
}
__device__ __forceinline__ void st_blk(double* A, int64_t C, int p, const Blk& x) {
  double* r = A + (int64_t)4 * p * C;
  r[0] = x.a;
  r[C] = x.b;
  r[2 * C] = x.c;
  r[3 * C] = x.d;
}
__device__ __forceinline__ Blk mul(const Blk& x, const Blk& y) {
  return {x.a * y.a + x.b * y.c, x.a * y.b + x.b * y.d, x.c * y.a + x.d * y.c, x.c * y.b + x.d * y.d};
}

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
    // block LU, row by row: L[k,m] = A[k,m] inv(A[m,m]) for m < k ascending, A[k,j] -= L[k,m] A[m,j] (j > m); then invert A[k,k]
    bool singular = false;
    for (int k = 0; k < n && !singular; ++k) {
      const int dk = __ldg(t.diag + k);
      for (int p = __ldg(t.blk_ptr + k); p < dk; ++p) {
        const Blk L = mul(ld_blk(A, C, p), ld_blk(A, C, __ldg(t.diag + __ldg(t.blk_col + p))));
        st_blk(A, C, p, L);
        for (int u = __ldg(t.upd_ptr + p); u < __ldg(t.upd_ptr + p + 1); ++u) {
          const int dst = __ldg(t.upd + 2 * u), src = __ldg(t.upd + 2 * u + 1);
          const Blk x = ld_blk(A, C, dst), y = mul(L, ld_blk(A, C, src));
          st_blk(A, C, dst, {x.a - y.a, x.b - y.b, x.c - y.c, x.d - y.d});
        }
      }
      const Blk D = ld_blk(A, C, dk);
      const double det = D.a * D.d - D.b * D.c;
      if (!(fabs(det) > 1e-12 * (fabs(D.a * D.d) + fabs(D.b * D.c)))) {
        singular = true;
        break;
      }
      const double r = 1.0 / det;
      st_blk(A, C, dk, {D.d * r, -D.b * r, -D.c * r, D.a * r});
    }
    if (singular) break;
    // forward: y_k = F_k - sum_{m<k} L[k,m] y_m
    for (int k = 0; k < n; ++k) {
      double yp = F[k * C], yq = F[(n + k) * C];
      for (int p = __ldg(t.blk_ptr + k); p < __ldg(t.diag + k); ++p) {
        const Blk L = ld_blk(A, C, p);
        const int m = __ldg(t.blk_col + p);
        const double xp = F[m * C], xq = F[(n + m) * C];
        yp -= L.a * xp + L.b * xq;
        yq -= L.c * xp + L.d * xq;
      }
      F[k * C] = yp;
      F[(n + k) * C] = yq;
    }
    // back: x_k = inv(A[k,k]) (y_k - sum_{j>k} A[k,j] x_j), then the update (th, V) -= x
    for (int k = n - 1; k >= 0; --k) {
      const int dk = __ldg(t.diag + k);
      double yp = F[k * C], yq = F[(n + k) * C];
      for (int p = dk + 1; p < __ldg(t.blk_ptr + k + 1); ++p) {
        const Blk U = ld_blk(A, C, p);
        const int j = __ldg(t.blk_col + p);
        const double xp = F[j * C], xq = F[(n + j) * C];
        yp -= U.a * xp + U.b * xq;
        yq -= U.c * xp + U.d * xq;
      }
      const Blk D = ld_blk(A, C, dk);
      const double xp = D.a * yp + D.b * yq, xq = D.c * yp + D.d * yq;
      F[k * C] = xp;
      F[(n + k) * C] = xq;
      const int i = __ldg(t.bus + k);
      th[i * C] -= xp;
      V[i * C] -= xq;
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
