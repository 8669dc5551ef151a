// (c) Fused branch-flow + WLS loss, forward and backward.  Replaces data.py:328-390, 393-459 + autograd.
//
// One shared-memory tile = a few whole scenarios (graphs never share a branch), so bus voltages,
// branch flows, bus injections and every adjoint live in shared memory; HBM sees x, edge_attr,
// edge_index and the model output once per pass, and writes grad_out once.  No per-branch tensor ever
// reaches HBM and no floating-point atomics are used: bus sums walk the CSR by destination in the
// order of PyG's scatter.  The three soft-constraint penalties are squares of batch means
// (data.py:453-455), so the gradient needs batch-global sums first: pass 1 (k_wls<false>) produces
// them (last-CTA-done reduction in fixed order, fp64), pass 2 (k_wls<true>) recomputes the cheap flow
// arithmetic and applies the adjoints.
//
// Compiled with -fmad=false: see wls_math.cuh.
#include "common.cuh"
#include "wls_math.cuh"

namespace {

constexpr int WLS_THREADS = 256;
// tile kernel: 128 threads so that 16 CTAs fit an SM; a tile's passes are a chain of short dependent phases, and with 8 resident CTAs
// the 9.2 tiles per SM of the bench workload needed two nearly serial rounds
constexpr int WLS_TILE_THREADS = 128;
constexpr int WLS_TILE_CTAS_PER_SM = 16;
enum { S_JN = 0, S_JE, S_V, S_TH, S_LOAD, S_N = 5 };

struct WlsArgs {
  dss2_graph_t g;
  const float* x;
  int64_t xs;
  const float* ea;
  int64_t eas;
  float* out;
  const float* stats;
  WlsCoefs k;
  const float* vminmax;
  int mask_inplace;
  float* loss;
  const float* grad_loss;
  float* grad_out;
  double* partial;     // [grid][S_N]
  unsigned* counter;
  double* sums;        // [S_N] batch sums, then [5] = bus count, [6] = branch count they were taken over
  int global_batch;    // pass 2 only: sums[0..6] describe the GLOBAL batch (all-reduced over the data-parallel ranks between the passes)
};

__device__ __forceinline__ WlsBranchIn load_branch(const float* row, const float* s_v, const float* s_th, int i, int j) {
  WlsBranchIn in;
  in.vi = s_v[i];
  in.vj = s_v[j];
  in.thi = s_th[i];
  in.thj = s_th[j];
  in.G = row[6];
  in.B = row[7];
  in.Gs = row[8];
  in.Bs = row[9];
  in.shift = row[11];
  in.rating = row[12];
  return in;
}

template <bool BWD>
__global__ void __launch_bounds__(WLS_TILE_THREADS) k_wls(WlsArgs a) {
  extern __shared__ float smem[];
  const dss2_graph_t& g = a.g;
  const int T = g.max_tile_nodes, E = g.max_tile_edges;
  float* s_v = smem;
  float* s_th = s_v + T;
  float* s_ap = s_th + T;
  float* s_aq = s_ap + T;
  float* s_gv = s_aq + T;
  float* s_gth = s_gv + T;
  float* s_pf = s_gth + T;   // bwd: reused as cvi
  float* s_qf = s_pf + E;    // bwd: reused as cvj
  float* s_pt = s_qf + E;    // bwd: reused as cdel
  float* s_qt = s_pt + E;
  __shared__ WlsStats st;
  __shared__ double s_red[S_N][WLS_TILE_THREADS / 32];
  __shared__ bool s_last;

  const int tid = threadIdx.x;
  if (tid < 28) ((float*)&st)[tid] = a.stats[tid];
  const WlsGrid grid = wls_grid(a.vminmax[0], a.vminmax[1]);
  const WlsCoefs k = a.k;
  const int64_t Nt = g.num_nodes, Et = g.num_edges;
  const int64_t* ei = g.edge_index;
  __syncthreads();

  double acc[S_N] = {0, 0, 0, 0, 0};
  float cN = 0.f, cE = 0.f, mv = 0.f, mth = 0.f, ml = 0.f;
  if (BWD) {
    float gl = a.grad_loss ? a.grad_loss[0] : 1.0f;
    // exact-global-batch data parallelism (data.py:450-455 on the union of all ranks' batches): the means and the 1/N, 1/E factors of the
    // gradient come from the all-reduced sums and counts; every rank then holds its buses' share of the global gradient
    const double Ng = a.global_batch ? a.sums[5] : (double)Nt, Eg = a.global_batch ? a.sums[6] : (double)Et;
    cN = gl / (float)Ng;
    cE = gl / (float)Eg;
    mv = (float)(a.sums[S_V] / Ng);
    mth = (float)(a.sums[S_TH] / Eg);
    ml = (float)(a.sums[S_LOAD] / Eg);
    if (a.global_batch && blockIdx.x == 0 && tid == 0) {   // the loss of the global batch, identical on every rank
      const double jv = a.sums[S_V] / Ng, jt = a.sums[S_TH] / Eg, jl = a.sums[S_LOAD] / Eg, lam = (double)k.lam_reg;
      a.loss[0] = (float)(a.sums[S_JN] / Ng + a.sums[S_JE] / Eg + lam * jv * jv + lam * jt * jt + lam * jl * jl);
    }
  }

  for (int t = blockIdx.x; t < g.num_tiles; t += gridDim.x) {
    const TileRange r = tile_range(g, t);
    const int nT = r.n1 - r.n0, nE = (int)(r.e1 - r.e0);
    // pass A: bus state
    for (int ln = tid; ln < nT; ln += WLS_TILE_THREADS) {
      int64_t n = r.n0 + ln;
      float o0 = a.out[2 * n], o1 = a.out[2 * n + 1];
      float slack = a.x[n * a.xs + 9];
      float th = o1 * (1.0f - slack);
      s_v[ln] = o0 * st.xs[0] + st.xm[0];
      s_th[ln] = th;
      if (!BWD && a.mask_inplace) a.out[2 * n + 1] = th;
    }
    __syncthreads();
    // pass B: branch flows
    for (int le = tid; le < nE; le += WLS_TILE_THREADS) {
      int64_t e = r.e0 + le;
      int i = (int)(ei[e] - r.n0), j = (int)(ei[Et + e] - r.n0);
      const float* row = a.ea + e * a.eas;
      WlsBranchIn in = load_branch(row, s_v, s_th, i, j);
      WlsBranch b;
      wls_branch_forward(in, grid, b);
      s_pf[le] = b.pf;
      s_qf[le] = b.qf;
      s_pt[le] = b.pt;
      s_qt[le] = b.qt;
      if (!BWD) {
        float eZ0 = wls_unnorm(row[0], st.es[0], st.em[0]), eR0 = wls_unnorm(row[1], st.es[1], st.em[1]);
        float eZ1 = wls_unnorm(row[2], st.es[2], st.em[2]), eR1 = wls_unnorm(row[3], st.es[3], st.em[3]);
        acc[S_JE] += (double)wls_branch_residual(eZ0, eR0, eZ1, eR1, b.pf, b.qf, k);
        acc[S_TH] += (double)fmaxf(fabsf(b.delta) - 0.5f, 0.0f);
        acc[S_LOAD] += (double)fmaxf(b.loading - 1.5f, 0.0f);
      }
    }
    __syncthreads();
    // pass C: bus injections (data.py:428-429) in PyG scatter order, residuals / adjoints
    for (int ln = tid; ln < nT; ln += WLS_TILE_THREADS) {
      int64_t n = r.n0 + ln;
      float sp_to = 0.f, sq_to = 0.f, sp_fr = 0.f, sq_fr = 0.f;
      for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
        uint32_t id = g.eid[z];
        int le = (int)((int64_t)(id & 0x7fffffffu) - r.e0);
        if (id >> 31) {
          sp_fr += s_pf[le];
          sq_fr += s_qf[le];
        } else {
          sp_to += s_pt[le];
          sq_to += s_qt[le];
        }
      }
      float p_bus = -sp_to - sp_fr, q_bus = -sq_to - sq_fr;
      WlsBus b;
      wls_bus_load(a.x + n * a.xs, a.out[2 * n], a.out[2 * n + 1], st, b);
      b.v = s_v[ln];
      b.th = s_th[ln];
      if (!BWD) {
        acc[S_JN] += (double)wls_bus_residual(b, p_bus, q_bus, k);
        acc[S_V] += (double)wls_bus_vband(b);
      } else {
        s_ap[ln] = -2.0f * k.lam_p * b.R[2] * (b.Z[2] - p_bus) * cN;
        s_aq[ln] = -2.0f * k.lam_p * b.R[3] * (b.Z[3] - q_bus) * cN;
        float band = (b.v - 1.1f > 0.0f ? 1.0f : 0.0f) - (0.9f - b.v > 0.0f ? 1.0f : 0.0f);
        s_gv[ln] = -2.0f * k.lam_v * b.R[0] * (b.Z[0] - b.v) * cN + 2.0f * k.lam_reg * mv * cN * band;
        s_gth[ln] = -2.0f * k.lam_v * b.R[1] * (b.Z[1] - b.th) * cN;
      }
    }
    if (BWD) {
      __syncthreads();
      // pass D: branch adjoints -> (dV_i, dV_j, d delta) per branch, kept in shared memory
      for (int le = tid; le < nE; le += WLS_TILE_THREADS) {
        int64_t e = r.e0 + le;
        int i = (int)(ei[e] - r.n0), j = (int)(ei[Et + e] - r.n0);
        const float* row = a.ea + e * a.eas;
        WlsBranchIn in = load_branch(row, s_v, s_th, i, j);
        WlsBranch b;
        wls_branch_forward(in, grid, b);
        float eZ0 = wls_unnorm(row[0], st.es[0], st.em[0]), eR0 = wls_unnorm(row[1], st.es[1], st.em[1]);
        float eZ1 = wls_unnorm(row[2], st.es[2], st.em[2]), eR1 = wls_unnorm(row[3], st.es[3], st.em[3]);
        float dpf = -s_ap[i] - 2.0f * k.lam_pf * eR0 * (eZ0 - b.pf) * cE;
        float dqf = -s_aq[i] - 2.0f * k.lam_pf * eR1 * (eZ1 - b.qf) * cE;
        float dpt = -s_ap[j], dqt = -s_aq[j];
        float ad = fabsf(b.delta);
        float ddelta = (ad - 0.5f > 0.0f) ? 2.0f * k.lam_reg * mth * cE * (b.delta > 0.0f ? 1.0f : -1.0f) : 0.0f;
        float dload = (b.loading - 1.5f > 0.0f) ? 2.0f * k.lam_reg * ml * cE : 0.0f;
        float dvi, dvj, ddel;
        wls_branch_backward(in, grid, b, dpf, dqf, dpt, dqt, ddelta, dload, dvi, dvj, ddel);
        s_pf[le] = dvi;
        s_qf[le] = dvj;
        s_pt[le] = ddel;
      }
      __syncthreads();
      // pass E: gather branch adjoints into the bus, chain through un-normalisation and slack mask
      for (int ln = tid; ln < nT; ln += WLS_TILE_THREADS) {
        int64_t n = r.n0 + ln;
        float gv = s_gv[ln], gth = s_gth[ln];
        for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
          uint32_t id = g.eid[z];
          int le = (int)((int64_t)(id & 0x7fffffffu) - r.e0);
          if (id >> 31) {  // this bus is the branch's "from" end
            gv += s_pf[le];
            gth += s_pt[le];
          } else {
            gv += s_qf[le];
            gth -= s_pt[le];
          }
        }
        float slack = a.x[n * a.xs + 9];
        a.grad_out[2 * n] = gv * st.xs[0];
        a.grad_out[2 * n + 1] = gth * (1.0f - slack);
      }
    }
    __syncthreads();
  }

  if (!BWD) {
    // block reduction (fp64) -> per-CTA partial -> the last CTA to finish adds the partials in CTA order
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int q = 0; q < S_N; ++q) {
      double v = warp_sum(acc[q]);
      if (lane == 0) s_red[q][warp] = v;
    }
    __syncthreads();
    if (tid < S_N) {
      double v = 0;
      for (int w = 0; w < WLS_TILE_THREADS / 32; ++w) v += s_red[tid][w];
      a.partial[(size_t)blockIdx.x * S_N + tid] = v;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
      __threadfence();
      // all threads of the last CTA add the per-CTA partials: thread t takes rows t, t + 128, ... in order, then a fixed butterfly /
      // warp order combines them - deterministic, and ~100x shorter than 5 threads walking >1000 rows (measured 68 us for 1184 rows)
      double v[S_N] = {0, 0, 0, 0, 0};
      for (unsigned c = tid; c < gridDim.x; c += WLS_TILE_THREADS)
#pragma unroll
        for (int q = 0; q < S_N; ++q) v[q] += ((volatile double*)a.partial)[(size_t)c * S_N + q];
      __syncthreads();   // s_red is reused below
#pragma unroll
      for (int q = 0; q < S_N; ++q) {
        const double r = warp_sum(v[q]);
        if (lane == 0) s_red[q][warp] = r;
      }
      __syncthreads();
      if (tid < S_N) {
        double r = 0;
        for (int w = 0; w < WLS_TILE_THREADS / 32; ++w) r += s_red[tid][w];
        a.sums[tid] = r;
        s_red[tid][0] = r;
      }
      __syncthreads();
      if (tid == 0) {
        double n = (double)Nt, e = (double)Et;
        double jv = s_red[S_V][0] / n, jt = s_red[S_TH][0] / e, jl = s_red[S_LOAD][0] / e;
        double lam = (double)k.lam_reg;
        a.loss[0] = (float)(s_red[S_JN][0] / n + s_red[S_JE][0] / e + lam * jv * jv + lam * jt * jt + lam * jl * jl);
        a.sums[5] = n;   // the counts travel with the sums (exact-global-batch mode all-reduces all seven)
        a.sums[6] = e;
        *a.counter = 0;  // ready for the next launch / graph replay
      }
    }
  }
}

// -------------------------------------------------------------------------------------------------
// large-graph path (a scenario with more buses than a tile holds): the same passes A-E as k_wls, one
// launch per pass, the per-bus / per-branch intermediates in the graph's global scratch
// (6 Nt + 4 Et floats).  Same arithmetic (wls_math.cuh), same fixed-order fp64 reductions.
// -------------------------------------------------------------------------------------------------
struct WlsScratch {
  float *v, *th, *ap, *aq, *gv, *gth;   // [Nt]
  float *pf, *qf, *pt, *qt;             // [Et]; backward reuses pf/qf/pt as dV_i / dV_j / d delta
};

__device__ __forceinline__ void wls_block_partial(double (&acc)[S_N], double* partial_row) {
  __shared__ double s_red[S_N][WLS_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int q = 0; q < S_N; ++q) {
    double v = warp_sum(acc[q]);
    if (lane == 0) s_red[q][warp] = v;
  }
  __syncthreads();
  if (tid < S_N) {
    double v = 0;
    for (int w = 0; w < WLS_THREADS / 32; ++w) v += s_red[tid][w];
    partial_row[tid] = v;
  }
}

__global__ void __launch_bounds__(WLS_THREADS) k_wls_g_state(WlsArgs a, WlsScratch s) {
  const float xs0 = a.stats[8], xm0 = a.stats[0];
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < a.g.num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    float o0 = a.out[2 * n], o1 = a.out[2 * n + 1];
    float slack = a.x[n * a.xs + 9];
    float th = o1 * (1.0f - slack);
    s.v[n] = o0 * xs0 + xm0;
    s.th[n] = th;
    if (a.mask_inplace) a.out[2 * n + 1] = th;
  }
}

template <bool BWD>
__global__ void __launch_bounds__(WLS_THREADS) k_wls_g_branch(WlsArgs a, WlsScratch s) {
  __shared__ WlsStats st;
  const dss2_graph_t& g = a.g;
  const int tid = threadIdx.x;
  if (tid < 28) ((float*)&st)[tid] = a.stats[tid];
  __syncthreads();
  const WlsGrid grid = wls_grid(a.vminmax[0], a.vminmax[1]);
  const WlsCoefs k = a.k;
  const int64_t Nt = g.num_nodes, Et = g.num_edges;
  const int64_t* ei = g.edge_index;
  double acc[S_N] = {0, 0, 0, 0, 0};
  float cE = 0.f, mth = 0.f, ml = 0.f;
  if (BWD) {
    float gl = a.grad_loss ? a.grad_loss[0] : 1.0f;
    cE = gl / (float)Et;
    mth = (float)(a.sums[S_TH] / (double)Et);
    ml = (float)(a.sums[S_LOAD] / (double)Et);
  }
  (void)Nt;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + tid; e < Et; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = ei[e], j = ei[Et + e];
    const float* row = a.ea + e * a.eas;
    WlsBranchIn in;
    in.vi = s.v[i];
    in.vj = s.v[j];
    in.thi = s.th[i];
    in.thj = s.th[j];
    in.G = row[6];
    in.B = row[7];
    in.Gs = row[8];
    in.Bs = row[9];
    in.shift = row[11];
    in.rating = row[12];
    WlsBranch b;
    wls_branch_forward(in, grid, b);
    float eZ0 = wls_unnorm(row[0], st.es[0], st.em[0]), eR0 = wls_unnorm(row[1], st.es[1], st.em[1]);
    float eZ1 = wls_unnorm(row[2], st.es[2], st.em[2]), eR1 = wls_unnorm(row[3], st.es[3], st.em[3]);
    if (!BWD) {
      s.pf[e] = b.pf;
      s.qf[e] = b.qf;
      s.pt[e] = b.pt;
      s.qt[e] = b.qt;
      acc[S_JE] += (double)wls_branch_residual(eZ0, eR0, eZ1, eR1, b.pf, b.qf, k);
      acc[S_TH] += (double)fmaxf(fabsf(b.delta) - 0.5f, 0.0f);
      acc[S_LOAD] += (double)fmaxf(b.loading - 1.5f, 0.0f);
    } else {
      float dpf = -s.ap[i] - 2.0f * k.lam_pf * eR0 * (eZ0 - b.pf) * cE;
      float dqf = -s.aq[i] - 2.0f * k.lam_pf * eR1 * (eZ1 - b.qf) * cE;
      float dpt = -s.ap[j], dqt = -s.aq[j];
      float ad = fabsf(b.delta);
      float ddelta = (ad - 0.5f > 0.0f) ? 2.0f * k.lam_reg * mth * cE * (b.delta > 0.0f ? 1.0f : -1.0f) : 0.0f;
      float dload = (b.loading - 1.5f > 0.0f) ? 2.0f * k.lam_reg * ml * cE : 0.0f;
      float dvi, dvj, ddel;
      wls_branch_backward(in, grid, b, dpf, dqf, dpt, dqt, ddelta, dload, dvi, dvj, ddel);
      s.pf[e] = dvi;
      s.qf[e] = dvj;
      s.pt[e] = ddel;
    }
  }
  if (!BWD) wls_block_partial(acc, a.partial + (size_t)blockIdx.x * S_N);
}

template <bool BWD>
__global__ void __launch_bounds__(WLS_THREADS) k_wls_g_bus(WlsArgs a, WlsScratch s, int partial_base) {
  __shared__ WlsStats st;
  const dss2_graph_t& g = a.g;
  const int tid = threadIdx.x;
  if (tid < 28) ((float*)&st)[tid] = a.stats[tid];
  __syncthreads();
  const WlsCoefs k = a.k;
  const int64_t Nt = g.num_nodes;
  double acc[S_N] = {0, 0, 0, 0, 0};
  float cN = 0.f, mv = 0.f;
  if (BWD) {
    float gl = a.grad_loss ? a.grad_loss[0] : 1.0f;
    cN = gl / (float)Nt;
    mv = (float)(a.sums[S_V] / (double)Nt);
  }
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + tid; n < Nt; n += (int64_t)gridDim.x * blockDim.x) {
    float sp_to = 0.f, sq_to = 0.f, sp_fr = 0.f, sq_fr = 0.f;
    for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
      const uint32_t id = g.eid[z];
      const int64_t e = id & 0x7fffffffu;
      if (id >> 31) {
        sp_fr += s.pf[e];
        sq_fr += s.qf[e];
      } else {
        sp_to += s.pt[e];
        sq_to += s.qt[e];
      }
    }
    float p_bus = -sp_to - sp_fr, q_bus = -sq_to - sq_fr;
    WlsBus b;
    wls_bus_load(a.x + n * a.xs, a.out[2 * n], a.out[2 * n + 1], st, b);
    b.v = s.v[n];
    b.th = s.th[n];
    if (!BWD) {
      acc[S_JN] += (double)wls_bus_residual(b, p_bus, q_bus, k);
      acc[S_V] += (double)wls_bus_vband(b);
    } else {
      s.ap[n] = -2.0f * k.lam_p * b.R[2] * (b.Z[2] - p_bus) * cN;
      s.aq[n] = -2.0f * k.lam_p * b.R[3] * (b.Z[3] - q_bus) * cN;
      float band = (b.v - 1.1f > 0.0f ? 1.0f : 0.0f) - (0.9f - b.v > 0.0f ? 1.0f : 0.0f);
      s.gv[n] = -2.0f * k.lam_v * b.R[0] * (b.Z[0] - b.v) * cN + 2.0f * k.lam_reg * mv * cN * band;
      s.gth[n] = -2.0f * k.lam_v * b.R[1] * (b.Z[1] - b.th) * cN;
    }
  }
  if (!BWD) wls_block_partial(acc, a.partial + (size_t)(partial_base + blockIdx.x) * S_N);
}

// one CTA: add the per-CTA partials (fp64, fixed order: thread t takes rows t, t + 256, ..., then butterfly / warp order), publish the
// sums and the loss
__global__ void __launch_bounds__(WLS_THREADS) k_wls_g_finish(WlsArgs a, int rows) {
  __shared__ double s_red[S_N][WLS_THREADS / 32];
  __shared__ double s_sum[S_N];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double v[S_N] = {0, 0, 0, 0, 0};
  for (int c = tid; c < rows; c += WLS_THREADS)
#pragma unroll
    for (int q = 0; q < S_N; ++q) v[q] += a.partial[(size_t)c * S_N + q];
#pragma unroll
  for (int q = 0; q < S_N; ++q) {
    const double r = warp_sum(v[q]);
    if (lane == 0) s_red[q][warp] = r;
  }
  __syncthreads();
  if (tid < S_N) {
    double r = 0;
    for (int w = 0; w < WLS_THREADS / 32; ++w) r += s_red[tid][w];
    a.sums[tid] = r;
    s_sum[tid] = r;
  }
  __syncthreads();
  if (tid == 0) {
    double n = (double)a.g.num_nodes, e = (double)a.g.num_edges;
    double jv = s_sum[S_V] / n, jt = s_sum[S_TH] / e, jl = s_sum[S_LOAD] / e;
    double lam = (double)a.k.lam_reg;
    a.loss[0] = (float)(s_sum[S_JN] / n + s_sum[S_JE] / e + lam * jv * jv + lam * jt * jt + lam * jl * jl);
  }
}

__global__ void __launch_bounds__(WLS_THREADS) k_wls_g_gather(WlsArgs a, WlsScratch s) {
  const dss2_graph_t& g = a.g;
  const float xs0 = a.stats[8];
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < g.num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    float gv = s.gv[n], gth = s.gth[n];
    for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
      const uint32_t id = g.eid[z];
      const int64_t e = id & 0x7fffffffu;
      if (id >> 31) {
        gv += s.pf[e];
        gth += s.pt[e];
      } else {
        gv += s.qf[e];
        gth -= s.pt[e];
      }
    }
    float slack = a.x[n * a.xs + 9];
    a.grad_out[2 * n] = gv * xs0;
    a.grad_out[2 * n + 1] = gth * (1.0f - slack);
  }
}

int wls_generic(const WlsArgs& a, bool want_grad, cudaStream_t stream) {
  const dss2_graph_t* g = &a.g;
  const int64_t Nt = g->num_nodes, Et = g->num_edges;
  DSS2_NEED_SCRATCH(g, "dss2_wls_fwd_bwd");
  DSS2_CHECK_ARG((size_t)(6 * Nt + 4 * Et) * sizeof(float) <= g->scratch_bytes, "dss2_wls_fwd_bwd: graph scratch too small for %lld branches",
                 (long long)Et);
  WlsScratch s;
  s.v = g->scratch;
  s.th = s.v + Nt;
  s.ap = s.th + Nt;
  s.aq = s.ap + Nt;
  s.gv = s.aq + Nt;
  s.gth = s.gv + Nt;
  s.pf = s.gth + Nt;
  s.qf = s.pf + Et;
  s.pt = s.qf + Et;
  s.qt = s.pt + Et;
  const int half = dss2_sm_count() * 4;   // the partial buffer holds sm*8 rows: branches first, buses after
  const int gn = (int)max((int64_t)1, min((int64_t)half, (Nt + WLS_THREADS - 1) / WLS_THREADS));
  const int ge = (int)max((int64_t)1, min((int64_t)half, (Et + WLS_THREADS - 1) / WLS_THREADS));
  k_wls_g_state<<<gn, WLS_THREADS, 0, stream>>>(a, s);
  DSS2_LAUNCH_CHECK();
  k_wls_g_branch<false><<<ge, WLS_THREADS, 0, stream>>>(a, s);
  DSS2_LAUNCH_CHECK();
  k_wls_g_bus<false><<<gn, WLS_THREADS, 0, stream>>>(a, s, ge);
  DSS2_LAUNCH_CHECK();
  k_wls_g_finish<<<1, WLS_THREADS, 0, stream>>>(a, ge + gn);
  DSS2_LAUNCH_CHECK();
  if (want_grad) {
    k_wls_g_bus<true><<<gn, WLS_THREADS, 0, stream>>>(a, s, 0);
    DSS2_LAUNCH_CHECK();
    k_wls_g_branch<true><<<ge, WLS_THREADS, 0, stream>>>(a, s);
    DSS2_LAUNCH_CHECK();
    k_wls_g_gather<<<gn, WLS_THREADS, 0, stream>>>(a, s);
    DSS2_LAUNCH_CHECK();
  }
  return 0;
}

// get_pflow as a plain per-branch kernel (evaluation path, dss2_run.py:193-194): outputs are API tensors.
// EST: y is the model output (normalised V, raw theta) and the bus state is the de-normalised estimate of dss2_run.py:183-184,
// V = y0 * x_std0 + x_mean0 and theta = y1 * (1 - x[:, 9]) - the arithmetic of k_eval_metrics' estimate branch.
struct PflowEst {
  const float* x;   // [Nt, >= 10]: column 9 = slack flag
  int64_t xs;
  float xm0, xs0;
};
template <bool EST>
__device__ __forceinline__ void pflow_bus(const float* y, int64_t ys, const PflowEst& est, int64_t n, float& v, float& th) {
  if (EST) {
    v = y[n * ys] * est.xs0 + est.xm0;
    th = y[n * ys + 1] * (1.0f - est.x[n * est.xs + 9]);
  } else {
    v = y[n * ys];
    th = y[n * ys + 1];
  }
}
template <bool EST>
__global__ void k_pflow(const int64_t* __restrict__ ei, int64_t Et, const float* __restrict__ y, int64_t ys, PflowEst est,
                        const float* __restrict__ ep, int64_t eps_, const float* __restrict__ vminmax, float* out8, int use_shift) {
  const WlsGrid grid = wls_grid(vminmax[0], vminmax[1]);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < Et; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = ei[e], j = ei[Et + e];
    const float* row = ep + e * eps_;
    WlsBranchIn in;
    pflow_bus<EST>(y, ys, est, i, in.vi, in.thi);
    pflow_bus<EST>(y, ys, est, j, in.vj, in.thj);
    in.G = row[0];
    in.B = row[1];
    in.Gs = row[2];
    in.Bs = row[3];
    in.shift = row[5];
    in.rating = row[6];
    WlsBranch b;
    wls_branch_forward_delta(in, grid, b, use_shift ? (in.thi - in.thj) - in.shift : in.thi - in.thj);   // data.py:362-365
    out8[e] = b.ll;
    out8[Et + e] = b.lt;
    out8[2 * Et + e] = b.pf;
    out8[3 * Et + e] = b.qf;
    out8[4 * Et + e] = b.pt;
    out8[5 * Et + e] = b.qt;
    out8[6 * Et + e] = b.i_f;
    out8[7 * Et + e] = b.i_t;
  }
}

// Adjoint of get_pflow w.r.t. y = (V, theta): thread = bus n, which walks its incident branches through the CSR row of the doubled
// graph (a non-reversed entry: n is the `to` end; a reversed one: n is the `from` end), re-evaluates the branch and keeps its own
// end's share - every branch is evaluated once per end, no atomics, fixed order.
__global__ void k_pflow_bwd(dss2_graph_t g, const float* __restrict__ y, int64_t ys, const float* __restrict__ ep, int64_t eps_,
                            const float* __restrict__ vminmax, const float* __restrict__ gout8, int use_shift, float* __restrict__ gy) {
  const WlsGrid grid = wls_grid(vminmax[0], vminmax[1]);
  const int64_t Et = g.num_edges;
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < g.num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    float gv = 0.0f, gth = 0.0f;
    for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
      const uint32_t id = g.eid[z];
      const int64_t e = id & 0x7fffffffu;
      const bool from_end = id >> 31;
      const int64_t i = from_end ? n : g.col[z], j = from_end ? g.col[z] : n;
      const float* row = ep + e * eps_;
      WlsBranchIn in;
      in.vi = y[i * ys];
      in.thi = y[i * ys + 1];
      in.vj = y[j * ys];
      in.thj = y[j * ys + 1];
      in.G = row[0];
      in.B = row[1];
      in.Gs = row[2];
      in.Bs = row[3];
      in.shift = row[5];
      in.rating = row[6];
      WlsBranch b;
      wls_branch_forward_delta(in, grid, b, use_shift ? (in.thi - in.thj) - in.shift : in.thi - in.thj);
      float go[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) go[q] = gout8[q * Et + e];
      float dvi, dvj, ddel;
      wls_pflow_backward(in, grid, b, go, dvi, dvj, ddel);
      gv += from_end ? dvi : dvj;
      gth += from_end ? ddel : -ddel;
    }
    gy[2 * n] = gv;
    gy[2 * n + 1] = gth;
  }
}

// -------------------------------------------------------------------------------------------------
// (f-4) Validation metrics of one batch, dss2_run.py:183-209: de-normalise V, mask the slack angle, squared / absolute errors of V and
// theta, column sums for the std ratio, and line / transformer loading errors over the branches whose TRUE loading is non-zero -
// both branch-flow evaluations (truth and estimate) in registers, 19 fp64 sums out, fixed-order last-CTA reduction.
// -------------------------------------------------------------------------------------------------
enum { M_SE_V = 0, M_AE_V, M_SE_TH, M_AE_TH, M_SV, M_SVV, M_STH, M_STHTH, M_YV, M_YVV, M_YTH, M_YTHTH,
       M_CNT_L, M_SE_L, M_AE_L, M_CNT_T, M_SE_T, M_AE_T, M_PAD, M_N = 19 };
struct EvalArgs {
  int64_t Nt, Et;
  const int64_t* ei;
  const float* x;      // [Nt, >= 11]: column 9 = slack flag
  int64_t xs;
  const float* ea;     // [Et, >= 13]: columns 6.. = edge_param
  int64_t eas;
  const float* out;    // [Nt, 2] model output (normalised V, raw theta)
  int64_t os;
  const float* y;      // [Nt, 2] labels (V pu, theta rad)
  int64_t ys;
  float xm0, xs0;
  const float* vminmax;
  double* partial;     // [grid][M_N]
  unsigned* counter;
  double* sums;        // [M_N] or NULL
  double* acc;         // [EVAL_ACC_N] or NULL: the batch's finalised metrics are added here (eval_finalise)
};

// The ten metrics of one batch from its 19 sums, in the order of dss2.metrics.evaluate_batch's dict, exactly as the script's formulas
// compute them in fp64 (wls.o is built with -fmad=false; double sqrt and division are IEEE): the epoch accumulator gets each value
// added, and one more batch counted in [10].  Python semantics kept where CUDA's differ: ratio(a, 0) = NaN, the std of n <= 1 values is
// NaN, and max(v, 0.0) keeps a NaN v (fmax would return 0).
enum { EVAL_ACC_N = 11 };
__device__ __forceinline__ double eval_nan() { return __longlong_as_double(0x7ff8000000000000LL); }   // Python's float("nan")
__device__ __forceinline__ double eval_ratio(double a, double b) { return b != 0.0 ? a / b : eval_nan(); }
__device__ __forceinline__ double eval_std(double sx, double sxx, double n) {   // torch.std: unbiased
  if (!(n > 1.0)) return eval_nan();
  const double v = (sxx - sx * sx / n) / (n - 1.0);
  return sqrt(0.0 > v ? 0.0 : v);
}
__device__ void eval_finalise(const double* s, double n, double* acc) {
  const double m[10] = {
      sqrt(s[M_SE_V] / n), s[M_AE_V] / n, sqrt(s[M_SE_TH] / n), s[M_AE_TH] / n,
      sqrt(eval_ratio(s[M_SE_L], s[M_CNT_L])), eval_ratio(s[M_AE_L], s[M_CNT_L]),
      sqrt(eval_ratio(s[M_SE_T], s[M_CNT_T])), eval_ratio(s[M_AE_T], s[M_CNT_T]),
      100.0 * eval_ratio(eval_std(s[M_SV], s[M_SVV], n), eval_std(s[M_YV], s[M_YVV], n)),
      100.0 * eval_ratio(eval_std(s[M_STH], s[M_STHTH], n), eval_std(s[M_YTH], s[M_YTHTH], n))};
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] += m[k];
  acc[10] += 1.0;
}

__global__ void __launch_bounds__(WLS_THREADS) k_eval_metrics(EvalArgs a) {
  __shared__ double s_red[M_N][WLS_THREADS / 32];
  __shared__ double s_tot[M_N];
  __shared__ bool s_last;
  const WlsGrid grid = wls_grid(a.vminmax[0], a.vminmax[1]);
  double acc[M_N];
#pragma unroll
  for (int q = 0; q < M_N; ++q) acc[q] = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (int64_t n = t0; n < a.Nt; n += stride) {
    const float v = a.out[n * a.os] * a.xs0 + a.xm0;                               // dss2_run.py:183
    const float th = a.out[n * a.os + 1] * (1.0f - a.x[n * a.xs + 9]);             // :184
    const float yv = a.y[n * a.ys], yth = a.y[n * a.ys + 1];
    const float dv = v - yv, dth = th - yth;
    acc[M_SE_V] += (double)(dv * dv);
    acc[M_AE_V] += (double)fabsf(dv);
    acc[M_SE_TH] += (double)(dth * dth);
    acc[M_AE_TH] += (double)fabsf(dth);
    acc[M_SV] += v;
    acc[M_SVV] += (double)v * v;
    acc[M_STH] += th;
    acc[M_STHTH] += (double)th * th;
    acc[M_YV] += yv;
    acc[M_YVV] += (double)yv * yv;
    acc[M_YTH] += yth;
    acc[M_YTHTH] += (double)yth * yth;
  }
  for (int64_t e = t0; e < a.Et; e += stride) {
    const int64_t i = a.ei[e], j = a.ei[a.Et + e];
    const float* row = a.ea + e * a.eas;
    WlsBranchIn in;
    in.G = row[6];
    in.B = row[7];
    in.Gs = row[8];
    in.Bs = row[9];
    in.shift = row[11];
    in.rating = row[12];
    WlsBranch bt, bo;
    in.vi = a.y[i * a.ys];
    in.thi = a.y[i * a.ys + 1];
    in.vj = a.y[j * a.ys];
    in.thj = a.y[j * a.ys + 1];
    wls_branch_forward(in, grid, bt);                                               // truth, :193
    in.vi = a.out[i * a.os] * a.xs0 + a.xm0;
    in.thi = a.out[i * a.os + 1] * (1.0f - a.x[i * a.xs + 9]);
    in.vj = a.out[j * a.os] * a.xs0 + a.xm0;
    in.thj = a.out[j * a.os + 1] * (1.0f - a.x[j * a.xs + 9]);
    wls_branch_forward(in, grid, bo);                                               // estimate, :194
    if (bt.ll != 0.0f) {                                                            // :196-197
      const float d = bo.ll - bt.ll;
      acc[M_CNT_L] += 1.0;
      acc[M_SE_L] += (double)(d * d);
      acc[M_AE_L] += (double)fabsf(d);
    }
    if (bt.lt != 0.0f) {                                                            // :199-200
      const float d = bo.lt - bt.lt;
      acc[M_CNT_T] += 1.0;
      acc[M_SE_T] += (double)(d * d);
      acc[M_AE_T] += (double)fabsf(d);
    }
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int q = 0; q < M_N; ++q) {
    const double v = warp_sum(acc[q]);
    if (lane == 0) s_red[q][warp] = v;
  }
  __syncthreads();
  if (tid < M_N) {
    double v = 0;
    for (int w = 0; w < WLS_THREADS / 32; ++w) v += s_red[tid][w];
    a.partial[(size_t)blockIdx.x * M_N + tid] = v;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (s_last) {
    __threadfence();
    for (int q = warp; q < M_N; q += WLS_THREADS / 32) {   // warp w adds quantity q over all CTAs: lanes stride the rows, butterfly combine
      double v = 0;
      for (unsigned c = lane; c < gridDim.x; c += 32) v += ((volatile double*)a.partial)[(size_t)c * M_N + q];
      v = warp_sum(v);
      if (lane == 0) {
        if (a.sums) a.sums[q] = v;
        s_tot[q] = v;
      }
    }
    if (tid == 0) *a.counter = 0;
    if (a.acc) {          // s_last is uniform over the CTA
      __syncthreads();
      if (tid == 0) eval_finalise(s_tot, (double)a.Nt, a.acc);
    }
  }
}

int wls_grid_size(const dss2_graph_t* g) { return max(1, min(g->num_tiles, dss2_sm_count() * WLS_TILE_CTAS_PER_SM)); }
size_t wls_smem(const dss2_graph_t* g) { return (size_t)(6 * g->max_tile_nodes + 4 * g->max_tile_edges) * sizeof(float); }

}  // namespace

extern "C" size_t dss2_wls_workspace_bytes(const dss2_graph_t* g) {
  (void)g;
  return (size_t)(dss2_sm_count() * WLS_TILE_CTAS_PER_SM) * S_N * sizeof(double) + 256 + 16 * sizeof(double);
}

static int wls_launch(int phase, const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, float* output,
                      const float* stats, float lam_v, float lam_p, float lam_pf, float lam_reg, const float* vminmax, int mask_inplace, float* loss,
                      const float* grad_loss, float* grad_out, void* ws, size_t ws_bytes, void* stream_);

extern "C" int dss2_wls_fwd_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr,
                                int64_t ea_stride, float* output, const float* stats, float lam_v, float lam_p, float lam_pf,
                                float lam_reg, const float* vminmax, int mask_inplace, float* loss, const float* grad_loss,
                                float* grad_out, void* ws, size_t ws_bytes, void* stream_) {
  return wls_launch(0, g, x, x_stride, edge_attr, ea_stride, output, stats, lam_v, lam_p, lam_pf, lam_reg, vminmax, mask_inplace, loss, grad_loss,
                    grad_out, ws, ws_bytes, stream_);
}

// Exact-global-batch data parallelism (SURVEY.md 8e, data.py:450-455): phase 1 = the reduction pass only; it leaves seven doubles at
// dss2_wls_sums(ws): the five batch sums (bus residual, branch residual, voltage-band, angle and loading penalties) and the bus / branch
// counts.  The caller sum-all-reduces those seven over the ranks IN PLACE, then phase 2 = the gradient pass with the global means and
// 1/N, 1/E factors (it also overwrites *loss with the loss of the global batch).  Summing the ranks' parameter gradients afterwards
// gives the gradient of ONE batch that is the union of the ranks' batches.  Tiled batches only.
extern "C" double* dss2_wls_sums(void* ws) { return (double*)((char*)ws + 256); }
extern "C" int dss2_wls_pass(int phase, const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride,
                             float* output, const float* stats, float lam_v, float lam_p, float lam_pf, float lam_reg, const float* vminmax,
                             int mask_inplace, float* loss, const float* grad_loss, float* grad_out, void* ws, size_t ws_bytes, void* stream_) {
  DSS2_CHECK_ARG(phase == 1 || phase == 2, "dss2_wls_pass: phase must be 1 (reduction pass) or 2 (gradient pass on all-reduced sums)");
  DSS2_CHECK_ARG(g && g->num_tiles > 0, "dss2_wls_pass: the split passes serve tiled batches only");
  DSS2_CHECK_ARG(phase == 1 || grad_out, "dss2_wls_pass: phase 2 needs grad_out");
  return wls_launch(phase, g, x, x_stride, edge_attr, ea_stride, output, stats, lam_v, lam_p, lam_pf, lam_reg, vminmax, mask_inplace, loss, grad_loss,
                    grad_out, ws, ws_bytes, stream_);
}

static int wls_launch(int phase, const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, float* output,
                      const float* stats, float lam_v, float lam_p, float lam_pf, float lam_reg, const float* vminmax, int mask_inplace, float* loss,
                      const float* grad_loss, float* grad_out, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(g && x && edge_attr && output && stats && vminmax && loss && ws, "dss2_wls_fwd_bwd: null argument");
  DSS2_CHECK_ARG(g->undirected == 1, "dss2_wls_fwd_bwd: needs a graph built from the one-way edge list with undirect=1");
  DSS2_CHECK_ARG(ws_bytes >= dss2_wls_workspace_bytes(g), "dss2_wls_fwd_bwd: workspace too small");
  DSS2_CHECK_ARG(x_stride >= 11 && ea_stride >= 13, "dss2_wls_fwd_bwd: x needs 11 columns and edge_attr 13");
  WlsArgs a;
  a.g = *g;
  a.x = x;
  a.xs = x_stride;
  a.ea = edge_attr;
  a.eas = ea_stride;
  a.out = output;
  a.stats = stats;
  a.k = WlsCoefs{lam_v, lam_p, lam_pf, lam_reg};
  a.vminmax = vminmax;
  a.mask_inplace = mask_inplace;
  a.loss = loss;
  a.grad_loss = grad_loss;
  a.grad_out = grad_out;
  a.global_batch = phase == 2;
  int grid = wls_grid_size(g);
  char* base = (char*)ws;
  a.counter = (unsigned*)base;                       // zero-initialised by the caller once; self-resetting
  a.sums = (double*)(base + 256);
  a.partial = a.sums + 16;
  if (g->num_nodes == 0 || g->num_edges == 0) {
    DSS2_CHECK_ARG(false, "dss2_wls_fwd_bwd: empty batch (the reference's means over buses / branches would be NaN)");
  }
  if (g->num_tiles == 0) return wls_generic(a, grad_out != nullptr, stream);
  size_t smem = wls_smem(g);
  DSS2_CHECK_ARG(smem <= 200 * 1024, "dss2_wls_fwd_bwd: tile needs %zu bytes of shared memory", smem);
  if (smem > 48 * 1024) {
    DSS2_CUDA(cudaFuncSetAttribute(k_wls<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DSS2_CUDA(cudaFuncSetAttribute(k_wls<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  if (phase != 2) {
    k_wls<false><<<grid, WLS_TILE_THREADS, smem, stream>>>(a);
    DSS2_LAUNCH_CHECK();
  }
  if (grad_out && phase != 1) {
    k_wls<true><<<grid, WLS_TILE_THREADS, smem, stream>>>(a);
    DSS2_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" size_t dss2_eval_workspace_bytes(void) { return 256 + (size_t)(dss2_sm_count() * 4 + 1) * M_N * sizeof(double); }

// sums19 and acc11: exactly one of them is set (dss2_eval_metrics / dss2_eval_metrics_acc)
static int eval_launch(const int64_t* edge_index, int64_t num_nodes, int64_t num_edges, const float* x, int64_t x_stride,
                       const float* edge_attr, int64_t ea_stride, const float* output, int64_t out_stride, const float* y, int64_t y_stride,
                       float x_mean0, float x_std0, const float* vminmax, double* sums19, double* acc11, void* ws, size_t ws_bytes,
                       void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const char* who = acc11 ? "dss2_eval_metrics_acc" : "dss2_eval_metrics";
  DSS2_CHECK_ARG(edge_index && x && edge_attr && output && y && vminmax && (sums19 || acc11) && ws, "%s: null argument", who);
  DSS2_CHECK_ARG(x_stride >= 11 && ea_stride >= 13 && out_stride >= 2 && y_stride >= 2, "%s: x needs 11 columns, edge_attr 13", who);
  DSS2_CHECK_ARG(ws_bytes >= dss2_eval_workspace_bytes(), "%s: workspace too small", who);
  EvalArgs a;
  a.Nt = num_nodes;
  a.Et = num_edges;
  a.ei = edge_index;
  a.x = x;
  a.xs = x_stride;
  a.ea = edge_attr;
  a.eas = ea_stride;
  a.out = output;
  a.os = out_stride;
  a.y = y;
  a.ys = y_stride;
  a.xm0 = x_mean0;
  a.xs0 = x_std0;
  a.vminmax = vminmax;
  a.counter = (unsigned*)ws;                      // zero-initialised by the caller once; self-resetting
  a.partial = (double*)((char*)ws + 256);
  a.sums = sums19;
  a.acc = acc11;
  const int grid = (int)max((int64_t)1, min((int64_t)dss2_sm_count() * 4, (max(num_nodes, num_edges) + WLS_THREADS - 1) / WLS_THREADS));
  k_eval_metrics<<<grid, WLS_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_eval_metrics(const int64_t* edge_index, int64_t num_nodes, int64_t num_edges, const float* x, int64_t x_stride,
                                 const float* edge_attr, int64_t ea_stride, const float* output, int64_t out_stride, const float* y,
                                 int64_t y_stride, float x_mean0, float x_std0, const float* vminmax, double* sums19, void* ws,
                                 size_t ws_bytes, void* stream_) {
  DSS2_CHECK_ARG(sums19, "dss2_eval_metrics: null argument");
  return eval_launch(edge_index, num_nodes, num_edges, x, x_stride, edge_attr, ea_stride, output, out_stride, y, y_stride, x_mean0, x_std0,
                     vminmax, sums19, nullptr, ws, ws_bytes, stream_);
}

extern "C" int dss2_eval_metrics_acc(const int64_t* edge_index, int64_t num_nodes, int64_t num_edges, const float* x, int64_t x_stride,
                                     const float* edge_attr, int64_t ea_stride, const float* output, int64_t out_stride, const float* y,
                                     int64_t y_stride, float x_mean0, float x_std0, const float* vminmax, double* acc11, void* ws,
                                     size_t ws_bytes, void* stream_) {
  DSS2_CHECK_ARG(acc11, "dss2_eval_metrics_acc: null argument");
  return eval_launch(edge_index, num_nodes, num_edges, x, x_stride, edge_attr, ea_stride, output, out_stride, y, y_stride, x_mean0, x_std0,
                     vminmax, nullptr, acc11, ws, ws_bytes, stream_);
}

extern "C" int dss2_pflow(const int64_t* edge_index, int64_t Et, const float* y, int64_t y_stride, const float* edge_param,
                          int64_t ep_stride, const float* vminmax, float* out8, void* stream_) {
  return dss2_pflow_ex(edge_index, Et, y, y_stride, edge_param, ep_stride, vminmax, 0, out8, stream_);
}

static int pflow_grid(int64_t Et) { return (int)max((int64_t)1, min((int64_t)148 * 8, (Et + 255) / 256)); }

extern "C" int dss2_pflow_ex(const int64_t* edge_index, int64_t Et, const float* y, int64_t y_stride, const float* edge_param,
                             int64_t ep_stride, const float* vminmax, int use_shift, float* out8, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(edge_index && y && edge_param && vminmax && out8, "dss2_pflow: null argument");
  if (Et == 0) return 0;
  k_pflow<false><<<pflow_grid(Et), 256, 0, stream>>>(edge_index, Et, y, y_stride, PflowEst{}, edge_param, ep_stride, vminmax, out8, use_shift);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_pflow_est(const int64_t* edge_index, int64_t Et, const float* output, int64_t out_stride, const float* x, int64_t x_stride,
                              float x_mean0, float x_std0, const float* edge_param, int64_t ep_stride, const float* vminmax, float* out8,
                              void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(edge_index && output && x && edge_param && vminmax && out8, "dss2_pflow_est: null argument");
  DSS2_CHECK_ARG(out_stride >= 2 && x_stride >= 10, "dss2_pflow_est: output needs 2 columns, x 10");
  if (Et == 0) return 0;
  k_pflow<true><<<pflow_grid(Et), 256, 0, stream>>>(edge_index, Et, output, out_stride, PflowEst{x, x_stride, x_mean0, x_std0}, edge_param,
                                                    ep_stride, vminmax, out8, 0);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_pflow_bwd(const dss2_graph_t* g, const float* y, int64_t y_stride, const float* edge_param, int64_t ep_stride,
                              const float* vminmax, int use_shift, const float* grad_out8, float* grad_y, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(g && y && edge_param && vminmax && grad_out8 && grad_y, "dss2_pflow_bwd: null argument");
  DSS2_CHECK_ARG(g->undirected == 1, "dss2_pflow_bwd: needs a graph built from the one-way edge list with undirect=1");
  if (g->num_nodes == 0) return 0;
  int grid = (int)max((int64_t)1, min((int64_t)148 * 8, (g->num_nodes + 255) / 256));
  k_pflow_bwd<<<grid, 256, 0, stream>>>(*g, y, y_stride, edge_param, ep_stride, vminmax, grad_out8, use_shift, grad_y);
  DSS2_LAUNCH_CHECK();
  return 0;
}
