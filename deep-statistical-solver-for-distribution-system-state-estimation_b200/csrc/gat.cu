// (f-1) GAT_DSSE: fused GATv2 layer (+ LeakyReLU) forward / backward and the two-Linear head.
// Replaces networks.py:113-156 (PyG GATv2Conv(8, 8, heads=1, edge_dim=6, add_self_loops=True, fill_value='mean') x 7, each followed by
// LeakyReLU(0.01), then Linear(8,32), Linear(32,2)) and its autograd.
//
// The script hands the ONE-WAY edge list to the model (networks.py:155-156 does not undirect).  The kernels walk the doubled-graph CSR
// the other layers use: in row i the entries WITHOUT the reversed bit are the edges pointing at i (in edge order = PyG's scatter
// order), the entries WITH it are the edges leaving i.  One thread owns one bus: channels are 8 wide, everything lives in registers,
// the 208 layer parameters sit in shared memory.  PyG's attention per edge (j -> i), restated:
//     x_l = W_l x + b_l, x_r = W_r x + b_r;  s = x_r[i] + x_l[j] + W_e a_e;  score = att . leaky_relu(s, 0.2)
//     alpha = exp(score - max_i) / (sum_i exp(.) + 1e-16);  out[i] = sum_j alpha_ij x_l[j] + bias
// with input self loops dropped and one loop per bus appended LAST whose attribute is the mean of the attributes of the edges pointing
// at the bus (0 without any).  No per-edge tensor reaches HBM; the backward recomputes the edge terms (pass A: per-destination softmax
// statistics, pass B: adjoints gathered per bus from its in- and out-edges: no atomics), weight gradients of the two node-level
// Linears come from one outer-product reduction over the stored node adjoints.
#include "common.cuh"

namespace {

constexpr int GC = 8;       // channels = dim_feat (heads = 1)
constexpr int GFE = 8;      // edge_dim <= 8
constexpr int GAT_THREADS = 128;
constexpr int GAT_BWD_THREADS = 256;   // k_gat_bwd runs one CTA per partial row (= per SM): 8 warps instead of 4 hide its gather latency
constexpr int GAT_NODE_WS = 36;   // floats per bus of backward scratch: m, den, t, pad, g[8], x_r[8], d x_l[8], d x_r[8]

struct GatW {
  float wl[GC * GC], bl[GC], wr[GC * GC], br[GC], we[GC * GFE], att[GC], bias[GC];
};
// Prepared weights in constant memory, one slot per layer (dss2_gat_upload): with SLOT a template parameter every weight is an
// immediate constant-bank operand of its FMA - no shared-memory load and no register holds a weight (the shared-memory variant made ptxas
// park ~200 weights in registers: 255 registers, 8 warps per SM).  SLOT = -1: weights from the launch's pointers through shared memory.
constexpr int GAT_SLOTS = 8;
__constant__ GatW c_gat[GAT_SLOTS];
__device__ GatW g_gat_stage[GAT_SLOTS];

// Attention dropout (GATv2Conv / FAConv `dropout`, applied to the normalised coefficients in training mode).  The keep bit of an
// attention coefficient is a pure function of (seed, step, layer_uid, head, edge key): edge key = one-way edge id for a real edge (the
// destination's entry and the source's reversed entry see the same bit), Et + i for the loop appended at bus i.  Every site that
// visits the coefficient (forward, statistics pass, both backward branches) re-draws the same bit; nothing is stored.
struct AttnDropArgs {
  int mode;             // 1 philox (seed / step from rng[0..1] on the device), 2 caller mask (uint8 [Et + Nt], 1 = keep)
  float scale;          // 1 / (1 - p)
  uint32_t keep_thr;    // philox: keep iff draw < keep_thr
  uint32_t layer_uid, head;
  const uint64_t* rng;
  const uint8_t* mask;
  int64_t num_edges;    // Et: first edge key of the appended loops
};
// third counter word: every TAG dropout draw puts a value below 32 there, so this domain tag keeps the two streams disjoint
constexpr uint32_t ATTN_DROP_DOMAIN = 0xA7700000u;
struct AttnKey {
  uint2 key;
  uint32_t step_lo;
};
__device__ __forceinline__ AttnKey attn_key(const AttnDropArgs& d) {
  AttnKey k = {make_uint2(0u, 0u), 0u};
  if (d.mode == 1) {
    const uint64_t seed = d.rng[0], step = d.rng[1];
    k.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (d.layer_uid * 0x9E3779B9u) ^ (uint32_t)(step >> 32));
    k.step_lo = (uint32_t)step;
  }
  return k;
}
__device__ __forceinline__ bool attn_keep(const AttnDropArgs& d, const AttnKey& k, uint64_t e) {
  if (d.mode == 2) return d.mask[e] != 0;
  const uint4 q = philox4x32_10(make_uint4((uint32_t)e, (uint32_t)(e >> 32), ATTN_DROP_DOMAIN | d.head, k.step_lo), k.key);
  return q.x < d.keep_thr;
}
// d_k = mask_k / (1 - p): the factor the coefficient of edge key e is multiplied with
__device__ __forceinline__ float attn_factor(const AttnDropArgs& d, const AttnKey& k, uint64_t e) { return attn_keep(d, k, e) ? d.scale : 0.0f; }

__global__ void k_attn_drop_mask(AttnDropArgs d, int64_t n, uint8_t* out) {
  const AttnKey k = attn_key(d);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) out[e] = attn_keep(d, k, e) ? 1 : 0;
}

struct GatArgs {
  dss2_graph_t g;
  const float* x;
  int64_t xs;
  const float* ea;
  int64_t eas;
  int fe;
  const float *wl, *bl, *wr, *br, *we, *att, *bias;
  float slope_att, slope_act;
  int act;     // 0 none, 1 leaky_relu(slope_act) (relu = slope 0), 2 tanh
  int loops;   // 1: PyG add_self_loops=True (drop input loops, append one per bus with the mean in-attribute); 0: edges as given
  float* y;           // fwd
  const float* yout;  // bwd: the layer's output (activation gate)
  const float* gy;
  float* ws;          // [Nt][GAT_NODE_WS]
  float* gx;
  float* partials;     // k_gat_bwd: the lin_edge.w block of the partial row
  int64_t partial_stride;
  int64_t off_att, off_bias;   // k_gat_bwd: att and bias blocks relative to `partials`
  AttnDropArgs drop;           // read by the DROP = true kernels only
};

__device__ __forceinline__ void load_weights(GatW& w, const GatArgs& a) {
  for (int i = threadIdx.x; i < GC * GC; i += blockDim.x) {
    w.wl[i] = a.wl[i];
    w.wr[i] = a.wr[i];
  }
  for (int i = threadIdx.x; i < GC * GFE; i += blockDim.x) {
    const int c = i / GFE, f = i % GFE;
    w.we[i] = f < a.fe ? a.we[c * a.fe + f] : 0.0f;
  }
  if (threadIdx.x < GC) {
    w.bl[threadIdx.x] = a.bl[threadIdx.x];
    w.br[threadIdx.x] = a.br[threadIdx.x];
    w.att[threadIdx.x] = a.att[threadIdx.x];
    w.bias[threadIdx.x] = a.bias[threadIdx.x];
  }
}

template <int SLOT>
__device__ __forceinline__ const GatW& gat_weights(GatW& sh, const GatArgs& a) {
  if constexpr (SLOT >= 0) {
    return c_gat[SLOT];
  } else {
    load_weights(sh, a);
    __syncthreads();
    return sh;
  }
}

__device__ __forceinline__ void load_x(const GatArgs& a, int64_t n, float (&v)[GC]) {
  const float* p = a.x + n * a.xs;
#pragma unroll
  for (int i = 0; i < GC; ++i) v[i] = p[i];
}
__device__ __forceinline__ void load_attr(const GatArgs& a, int64_t e, float (&v)[GFE]) {
  const float* p = a.ea + e * a.eas;
#pragma unroll
  for (int i = 0; i < GFE; ++i) v[i] = i < a.fe ? p[i] : 0.0f;
}
// out = W v + b, W row-major [8][8] in shared memory
__device__ __forceinline__ void lin8(const float* W, const float* b, const float (&v)[GC], float (&out)[GC]) {
#pragma unroll
  for (int c = 0; c < GC; ++c) {
    float s = b[c];
#pragma unroll
    for (int i = 0; i < GC; ++i) s = fmaf(W[c * GC + i], v[i], s);
    out[c] = s;
  }
}
// s = x_r + x_l + W_e a
__device__ __forceinline__ void edge_pre(const GatW& w, const float (&xr)[GC], const float (&xl)[GC], const float (&at)[GFE], float (&s)[GC]) {
#pragma unroll
  for (int c = 0; c < GC; ++c) {
    float e = 0.0f;
#pragma unroll
    for (int f = 0; f < GFE; ++f) e = fmaf(w.we[c * GFE + f], at[f], e);
    s[c] = (xr[c] + xl[c]) + e;
  }
}
__device__ __forceinline__ float edge_score(const GatW& w, const float (&s)[GC], float slope) {
  float sc = 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) sc = fmaf(s[c] > 0.0f ? s[c] : s[c] * slope, w.att[c], sc);
  return sc;
}

// Per-destination softmax statistics of bus i: max score m, denominator den (incl. PyG's 1e-16), un-normalised weighted sum acc of
// x_l over the in-edges and the loop, mean in-attribute abar.  `G` (optional) additionally gives t = sum_k alpha_k (G . x_l[k]).
// DROP: acc and t weight edge k with alpha_k d_k (the denominator is the softmax's, before the dropout).
struct DstStats {
  float m, den, t;
};
template <bool WITH_T, bool DROP = false>
__device__ __forceinline__ DstStats dst_pass(const GatArgs& a, const GatW& w, int64_t i, const float (&xr)[GC], const float (&xl_i)[GC],
                                             float (&abar)[GFE], float (&acc)[GC], const float (&G)[GC], const AttnKey& dk = AttnKey{}) {
  const dss2_graph_t& g = a.g;
  const int beg = g.rowptr[i], end = g.rowptr[i + 1];
  float m = -INFINITY;
  int cnt = 0;
#pragma unroll
  for (int f = 0; f < GFE; ++f) abar[f] = 0.0f;
  for (int z = beg; z < end; ++z) {
    const uint32_t id = g.eid[z];
    const int j = g.col[z];
    if ((id >> 31) || (a.loops && j == i)) continue;
    float xj[GC], xl[GC], at[GFE], s[GC];
    load_x(a, j, xj);
    lin8(w.wl, w.bl, xj, xl);
    load_attr(a, id, at);
#pragma unroll
    for (int f = 0; f < GFE; ++f) abar[f] += at[f];
    ++cnt;
    edge_pre(w, xr, xl, at, s);
    m = fmaxf(m, edge_score(w, s, a.slope_att));
  }
  if (cnt > 0) {
    const float c = (float)cnt;
#pragma unroll
    for (int f = 0; f < GFE; ++f) abar[f] = abar[f] / c;
  }
  float s_loop[GC];
  float sc_loop = -INFINITY;
  if (a.loops) {
    edge_pre(w, xr, xl_i, abar, s_loop);
    sc_loop = edge_score(w, s_loop, a.slope_att);
    m = fmaxf(m, sc_loop);
  }
  float den = 0.0f, t = 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) acc[c] = 0.0f;
  for (int z = beg; z < end; ++z) {
    const uint32_t id = g.eid[z];
    const int j = g.col[z];
    if ((id >> 31) || (a.loops && j == i)) continue;
    float xj[GC], xl[GC], at[GFE], s[GC];
    load_x(a, j, xj);
    lin8(w.wl, w.bl, xj, xl);
    load_attr(a, id, at);
    edge_pre(w, xr, xl, at, s);
    const float ex = expf(edge_score(w, s, a.slope_att) - m);
    den += ex;
    float exd = ex;
    if constexpr (DROP) exd = ex * attn_factor(a.drop, dk, id);
    float dot = 0.0f;
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      acc[c] = fmaf(exd, xl[c], acc[c]);
      if (WITH_T) dot = fmaf(G[c], xl[c], dot);
    }
    if (WITH_T) t = fmaf(exd, dot, t);
  }
  if (a.loops) {
    const float ex = expf(sc_loop - m);
    den += ex;
    float exd = ex;
    if constexpr (DROP) exd = ex * attn_factor(a.drop, dk, (uint64_t)a.drop.num_edges + (uint64_t)i);
    float dot = 0.0f;
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      acc[c] = fmaf(exd, xl_i[c], acc[c]);
      if (WITH_T) dot = fmaf(G[c], xl_i[c], dot);
    }
    if (WITH_T) t = fmaf(exd, dot, t);
  }
  den += 1e-16f;   // a bus without in-edges and without loop: acc = 0, den = 1e-16 -> out = bias, like PyG's empty softmax segment
  DstStats r;
  r.m = m;
  r.den = den;
  r.t = t / den;
  return r;
}

template <int SLOT, bool DROP>
__global__ void __launch_bounds__(GAT_THREADS) k_gat_fwd(GatArgs a) {
  __shared__ GatW w_sh;
  const GatW& w = gat_weights<SLOT>(w_sh, a);
  const float zero[GC] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  AttnKey dk = {};
  if constexpr (DROP) dk = attn_key(a.drop);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    float xi[GC], xr[GC], xl[GC], abar[GFE], acc[GC];
    load_x(a, i, xi);
    lin8(w.wr, w.br, xi, xr);
    lin8(w.wl, w.bl, xi, xl);
    const DstStats st = dst_pass<false, DROP>(a, w, i, xr, xl, abar, acc, zero, dk);
    float out[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      const float v = acc[c] / st.den + w.bias[c];
      out[c] = a.act == 2 ? tanhf(v) : ((a.act == 1 && !(v > 0.0f)) ? v * a.slope_act : v);
    }
    float4* dst = reinterpret_cast<float4*>(a.y + i * GC);
    dst[0] = make_float4(out[0], out[1], out[2], out[3]);
    dst[1] = make_float4(out[4], out[5], out[6], out[7]);
  }
}

// backward pass A: per bus g = grad_y * gate, x_r, softmax statistics (m, den, t)
template <int SLOT, bool DROP>
__global__ void __launch_bounds__(GAT_THREADS) k_gat_bwd_stats(GatArgs a) {
  __shared__ GatW w_sh;
  const GatW& w = gat_weights<SLOT>(w_sh, a);
  AttnKey dk = {};
  if constexpr (DROP) dk = attn_key(a.drop);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    float xi[GC], xr[GC], xl[GC], abar[GFE], acc[GC], G[GC];
    load_x(a, i, xi);
    lin8(w.wr, w.br, xi, xr);
    lin8(w.wl, w.bl, xi, xl);
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      const float yv = a.yout[i * GC + c];
      const float gate = a.act == 2 ? 1.0f - yv * yv : ((a.act == 1 && !(yv > 0.0f)) ? a.slope_act : 1.0f);
      G[c] = a.gy[i * GC + c] * gate;
    }
    const DstStats st = dst_pass<true, DROP>(a, w, i, xr, xl, abar, acc, G, dk);
    float* o = a.ws + i * GAT_NODE_WS;
    o[0] = st.m;
    o[1] = st.den;
    o[2] = st.t;
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      o[4 + c] = G[c];
      o[12 + c] = xr[c];
    }
  }
}

// adjoint of one edge (j -> i) given the destination's statistics: returns alpha, fills ds = d loss / d s, adds to d att.
// DROP (d = the edge's dropout factor): returns alpha d, the weight of x_l[j] in out[i]; d score = alpha (d (G_i . x_l[j]) - t_i).
template <bool DROP = false>
__device__ __forceinline__ float edge_adjoint(const GatArgs& a, const GatW& w, const float (&s)[GC], float m, float den, float t,
                                              const float (&Gi)[GC], const float (&xl_j)[GC], float (&ds)[GC], float* datt, float d = 1.0f) {
  const float alpha = expf(edge_score(w, s, a.slope_att) - m) / den;
  float dal = 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) dal = fmaf(Gi[c], xl_j[c], dal);
  float dsc;
  // d * dal rounded on its own (no fused multiply-add), as t's terms were: a segment of one kept coefficient (a bus with one in-edge
  // and no loop) then gets exactly t = d dal and d score = 0, like the softmax adjoint it stands for
  if constexpr (DROP) dsc = alpha * (__fmul_rn(d, dal) - t);
  else dsc = alpha * (dal - t);
#pragma unroll
  for (int c = 0; c < GC; ++c) {
    const bool pos = s[c] > 0.0f;
    ds[c] = dsc * w.att[c] * (pos ? 1.0f : a.slope_att);
    if (datt) datt[c] = fmaf(dsc, pos ? s[c] : s[c] * a.slope_att, datt[c]);
  }
  if constexpr (DROP) return alpha * d;
  return alpha;
}

// backward pass B: thread = bus n.  As destination it owns d x_r[n], d W_e, d att of its in-edges and loop; as source it gathers d x_l[n]
// from its out-edges.  partial layout per CTA: [W_e 8 x fe | att 8 | bias 8] at the offsets the host passes via partials pointer.
template <int SLOT, bool DROP>
__global__ void __launch_bounds__(GAT_BWD_THREADS) k_gat_bwd(GatArgs a) {
  __shared__ GatW w_sh;
  __shared__ float red[GAT_BWD_THREADS / 32][GC * GFE + 2 * GC];
  const GatW& w = gat_weights<SLOT>(w_sh, a);
  const dss2_graph_t& g = a.g;
  AttnKey dk = {};
  if constexpr (DROP) dk = attn_key(a.drop);
  float dWe[GC * GFE], datt[GC], dbias[GC];
#pragma unroll
  for (int i = 0; i < GC * GFE; ++i) dWe[i] = 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) datt[c] = dbias[c] = 0.0f;
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < g.num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    float xn[GC], xl_n[GC], dxl[GC], dxr[GC];
    load_x(a, n, xn);
    lin8(w.wl, w.bl, xn, xl_n);
#pragma unroll
    for (int c = 0; c < GC; ++c) dxl[c] = dxr[c] = 0.0f;
    const float* sn = a.ws + n * GAT_NODE_WS;
    const float m_n = sn[0], den_n = sn[1], t_n = sn[2];
    float Gn[GC], xr_n[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      Gn[c] = sn[4 + c];
      xr_n[c] = sn[12 + c];
      dbias[c] += Gn[c];
    }
    const int beg = g.rowptr[n], end = g.rowptr[n + 1];
    float abar[GFE];
    int cnt = 0;
#pragma unroll
    for (int f = 0; f < GFE; ++f) abar[f] = 0.0f;
    for (int z = beg; z < end; ++z) {
      const uint32_t id = g.eid[z];
      const int o = g.col[z];
      if (a.loops && o == n) continue;   // self loops of the input are dropped (remove_self_loops, part of add_self_loops=True)
      float at[GFE], s[GC], ds[GC];
      load_attr(a, id & 0x7fffffffu, at);
      if (!(id >> 31)) {      // in-edge (o -> n): this bus is the destination
        float xo[GC], xl_o[GC];
        load_x(a, o, xo);
        lin8(w.wl, w.bl, xo, xl_o);
#pragma unroll
        for (int f = 0; f < GFE; ++f) abar[f] += at[f];
        ++cnt;
        edge_pre(w, xr_n, xl_o, at, s);
        float d = 1.0f;
        if constexpr (DROP) d = attn_factor(a.drop, dk, id);
        edge_adjoint<DROP>(a, w, s, m_n, den_n, t_n, Gn, xl_o, ds, datt, d);
#pragma unroll
        for (int c = 0; c < GC; ++c) {
          dxr[c] += ds[c];
#pragma unroll
          for (int f = 0; f < GFE; ++f) dWe[c * GFE + f] = fmaf(ds[c], at[f], dWe[c * GFE + f]);
        }
      } else {                // out-edge (n -> o): this bus is the source
        const float* so = a.ws + (int64_t)o * GAT_NODE_WS;
        float Go[GC], xr_o[GC];
#pragma unroll
        for (int c = 0; c < GC; ++c) {
          Go[c] = so[4 + c];
          xr_o[c] = so[12 + c];
        }
        edge_pre(w, xr_o, xl_n, at, s);
        float d = 1.0f;
        if constexpr (DROP) d = attn_factor(a.drop, dk, id & 0x7fffffffu);
        const float alpha = edge_adjoint<DROP>(a, w, s, so[0], so[1], so[2], Go, xl_n, ds, nullptr, d);
#pragma unroll
        for (int c = 0; c < GC; ++c) dxl[c] += fmaf(alpha, Go[c], ds[c]);
      }
    }
    if (a.loops) {   // the appended self loop (n -> n) with the mean in-attribute
      if (cnt > 0) {
        const float c = (float)cnt;
#pragma unroll
        for (int f = 0; f < GFE; ++f) abar[f] = abar[f] / c;
      }
      float s[GC], ds[GC];
      edge_pre(w, xr_n, xl_n, abar, s);
      float d = 1.0f;
      if constexpr (DROP) d = attn_factor(a.drop, dk, (uint64_t)a.drop.num_edges + (uint64_t)n);
      const float alpha = edge_adjoint<DROP>(a, w, s, m_n, den_n, t_n, Gn, xl_n, ds, datt, d);
#pragma unroll
      for (int c = 0; c < GC; ++c) {
        dxr[c] += ds[c];
        dxl[c] += fmaf(alpha, Gn[c], ds[c]);
#pragma unroll
        for (int f = 0; f < GFE; ++f) dWe[c * GFE + f] = fmaf(ds[c], abar[f], dWe[c * GFE + f]);
      }
    }
    float* o = a.ws + n * GAT_NODE_WS;
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      o[20 + c] = dxl[c];
      o[28 + c] = dxr[c];
    }
    if (a.gx) {   // grad_x = W_l^T d x_l + W_r^T d x_r
      float gx[GC];
#pragma unroll
      for (int i = 0; i < GC; ++i) {
        float s = 0.0f;
#pragma unroll
        for (int c = 0; c < GC; ++c) s = fmaf(w.wl[c * GC + i], dxl[c], fmaf(w.wr[c * GC + i], dxr[c], s));
        gx[i] = s;
      }
      float4* dst = reinterpret_cast<float4*>(a.gx + n * GC);
      dst[0] = make_float4(gx[0], gx[1], gx[2], gx[3]);
      dst[1] = make_float4(gx[4], gx[5], gx[6], gx[7]);
    }
  }
  // per-CTA partial: warp sums -> shared memory -> fixed-order sum over the warps
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < GC * GFE; ++i) {
    const float v = warp_sum(dWe[i]);
    if (lane == 0) red[warp][i] = v;
  }
#pragma unroll
  for (int c = 0; c < GC; ++c) {
    const float v1 = warp_sum(datt[c]), v2 = warp_sum(dbias[c]);
    if (lane == 0) {
      red[warp][GC * GFE + c] = v1;
      red[warp][GC * GFE + GC + c] = v2;
    }
  }
  __syncthreads();
  float* part = a.partials + (size_t)blockIdx.x * a.partial_stride;
  for (int i = threadIdx.x; i < GC * a.fe + 2 * GC; i += blockDim.x) {
    int src;
    if (i < GC * a.fe) src = (i / a.fe) * GFE + (i % a.fe);
    else src = GC * GFE + (i - GC * a.fe);
    float s = 0.0f;
#pragma unroll
    for (int wv = 0; wv < GAT_BWD_THREADS / 32; ++wv) s += red[wv][src];
    const int j = i - GC * a.fe;
    part[j < 0 ? (int64_t)i : j < GC ? a.off_att + j : a.off_bias + (j - GC)] = s;
  }
}

// out_w[c][i] = sum_n A[n][c] * B[n][i], out_b[c] = sum_n A[n][c]: per-CTA partial sums of the weight / bias gradient of a node-level
// Linear (A = adjoint of its output, B = its input), rows split contiguously over the CTAs, 64-row chunks staged in shared memory.
constexpr int OR_THREADS = 256, OR_ROWS = 64;
__global__ void __launch_bounds__(OR_THREADS) k_outer_reduce(int64_t num_rows, const float* __restrict__ A, int64_t as, int ca,
                                                             const float* __restrict__ B, int64_t bs, int cb, float* partials,
                                                             int64_t partial_stride, int64_t w_off, int64_t b_off) {
  __shared__ float sA[OR_ROWS][33], sB[OR_ROWS][33];
  __shared__ float s_part[OR_THREADS];
  const int tid = threadIdx.x;
  const int nout = ca * (cb + 1);
  // few outputs (a GATv2 layer has 72): several threads share one output and take the rows of a chunk round robin (`slices`), combined
  // in a fixed order at the end; many outputs (the head: up to 1056): every thread owns up to 5 outputs and walks all rows
  const int slices = nout <= OR_THREADS ? OR_THREADS / nout : 1;
  const bool sliced = nout <= OR_THREADS;
  const int my_o = tid % nout, my_sl = tid / nout;
  float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // ca, cb <= 32 -> at most 1056 outputs over 256 threads
  const int64_t per = (num_rows + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = blockIdx.x * per, r1 = min(num_rows, r0 + per);
  for (int64_t base = r0; base < r1; base += OR_ROWS) {
    const int rows = (int)min((int64_t)OR_ROWS, r1 - base);
    for (int idx = tid; idx < rows * ca; idx += OR_THREADS) sA[idx / ca][idx % ca] = A[(base + idx / ca) * as + idx % ca];
    for (int idx = tid; idx < rows * cb; idx += OR_THREADS) sB[idx / cb][idx % cb] = B[(base + idx / cb) * bs + idx % cb];
    __syncthreads();
    if (sliced) {
      if (my_sl < slices) {
        const int c = my_o / (cb + 1), i = my_o % (cb + 1);
        float s = acc[0];
        if (i < cb) {
          for (int r = my_sl; r < rows; r += slices) s = fmaf(sA[r][c], sB[r][i], s);
        } else {
          for (int r = my_sl; r < rows; r += slices) s += sA[r][c];
        }
        acc[0] = s;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 5; ++q) {
        const int o = tid + q * OR_THREADS;
        if (o < nout) {
          const int c = o / (cb + 1), i = o % (cb + 1);
          float s = acc[q];
          if (i < cb) {
            for (int r = 0; r < rows; ++r) s = fmaf(sA[r][c], sB[r][i], s);
          } else {
            for (int r = 0; r < rows; ++r) s += sA[r][c];
          }
          acc[q] = s;
        }
      }
    }
    __syncthreads();
  }
  float* part = partials + (size_t)blockIdx.x * partial_stride;
  if (sliced) {
    s_part[tid] = acc[0];
    __syncthreads();
    if (tid < nout) {
      float s = 0.0f;
      for (int sl = 0; sl < slices; ++sl) s += s_part[sl * nout + tid];
      const int c = tid / (cb + 1), i = tid % (cb + 1);
      if (i < cb) part[w_off + (int64_t)c * cb + i] = s;
      else part[b_off + c] = s;
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    const int o = tid + q * OR_THREADS;
    if (o < nout) {
      const int c = o / (cb + 1), i = o % (cb + 1);
      if (i < cb) part[w_off + (int64_t)c * cb + i] = acc[q];
      else part[b_off + c] = acc[q];
    }
  }
}

// The same reduction with register accumulators: a warp owns one 8 x 8 block (ba, bb) of the [ca, cb] product (ca, cb <= 32, the number
// of blocks a power of two <= 8: every GATv2 / GINE / gnn_dsse layer is one block, the head's two Linears are 4 blocks each) and a slice
// of the rows; thread = bus row, the row's 8 x 9 outer product (column 8 = the bias sum, block column 0 only) accumulates in registers
// over the rows the thread owns, then ONE fixed-order reduction per CTA: butterfly inside the warps, the warp totals of a block summed in
// warp order.  No shared-memory staging, two barriers per launch instead of two per 64 rows.
__global__ void __launch_bounds__(OR_THREADS) k_outer_reduce8(int64_t num_rows, const float* __restrict__ A, int64_t as, int ca,
                                                              const float* __restrict__ B, int64_t bs, int cb, float* partials,
                                                              int64_t partial_stride, int64_t w_off, int64_t b_off) {
  constexpr int NW = OR_THREADS / 32;
  __shared__ float red[NW][8 * 9];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nba = (ca + 7) >> 3, nbb = (cb + 7) >> 3, nblk = nba * nbb, nsl = NW / nblk;   // nblk in {1, 2, 4, 8}
  const int blk = warp % nblk, sl = warp / nblk, ba = blk / nbb, bb = blk % nbb;
  const int ca0 = 8 * ba, cb0 = 8 * bb, nca = min(8, ca - ca0), ncb = min(8, cb - cb0);
  float acc[8][9];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int i = 0; i < 9; ++i) acc[c][i] = 0.0f;
  const bool a_vec = nca == 8 && (as & 3) == 0 && (((uintptr_t)A) & 15) == 0, b_vec = ncb == 8 && (bs & 3) == 0 && (((uintptr_t)B) & 15) == 0;
  const int64_t rows_per_pass = (int64_t)gridDim.x * nsl * 32;
  for (int64_t n = ((int64_t)blockIdx.x * nsl + sl) * 32 + lane; n < num_rows; n += rows_per_pass) {
    float a[8], b[8];
    const float *pa = A + n * as + ca0, *pb = B + n * bs + cb0;
    if (a_vec) {
      const float4 u = *reinterpret_cast<const float4*>(pa), v = *reinterpret_cast<const float4*>(pa + 4);
      a[0] = u.x, a[1] = u.y, a[2] = u.z, a[3] = u.w, a[4] = v.x, a[5] = v.y, a[6] = v.z, a[7] = v.w;
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) a[c] = c < nca ? pa[c] : 0.0f;
    }
    if (b_vec) {
      const float4 u = *reinterpret_cast<const float4*>(pb), v = *reinterpret_cast<const float4*>(pb + 4);
      b[0] = u.x, b[1] = u.y, b[2] = u.z, b[3] = u.w, b[4] = v.x, b[5] = v.y, b[6] = v.z, b[7] = v.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) b[i] = i < ncb ? pb[i] : 0.0f;
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[c][i] = fmaf(a[c], b[i], acc[c][i]);
      acc[c][8] += a[c];
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const float v = warp_sum(acc[c][i]);
      if (lane == 0) red[warp][c * 9 + i] = v;
    }
  __syncthreads();
  float* part = partials + (size_t)blockIdx.x * partial_stride;
  for (int o = threadIdx.x; o < ca * (cb + 1); o += OR_THREADS) {
    const int c = o / (cb + 1), i = o % (cb + 1);
    const int ib = i < cb ? i : 0;                       // the bias column lives in block column 0
    const int b_ = (c >> 3) * nbb + (ib >> 3);
    float s = 0.0f;
    for (int w = 0; w < nsl; ++w) s += red[w * nblk + b_][(c & 7) * 9 + (i < cb ? (i & 7) : 8)];
    if (i < cb) part[w_off + (int64_t)c * cb + i] = s;
    else part[b_off + c] = s;
  }
}

// launches the outer-product reduction that fits the operand widths
static void launch_outer_reduce(int np, cudaStream_t stream, int64_t num_rows, const float* A, int64_t as, int ca, const float* B, int64_t bs, int cb,
                                float* partials, int64_t partial_stride, int64_t w_off, int64_t b_off) {
  const int nblk = ((ca + 7) / 8) * ((cb + 7) / 8);
  if (ca <= 32 && cb <= 32 && (nblk == 1 || nblk == 2 || nblk == 4 || nblk == 8))
    k_outer_reduce8<<<np, OR_THREADS, 0, stream>>>(num_rows, A, as, ca, B, bs, cb, partials, partial_stride, w_off, b_off);
  else
    k_outer_reduce<<<np, OR_THREADS, 0, stream>>>(num_rows, A, as, ca, B, bs, cb, partials, partial_stride, w_off, b_off);
}

// ---- head: z = W2 (W1 x + b1) + b2 (no non-linearity in between, networks.py:150-151) ----
constexpr int MLP_MAX = 32;
struct MlpArgs {
  int64_t n;
  const float* x;
  int din;
  const float *w1, *b1;
  int dmid;
  const float *w2, *b2;
  int dout;
  float* h;          // [n, dmid]
  float* z;          // [n, dout]
  const float* gz;   // bwd
  float* gh;         // [n, dmid]
  float* gx;         // [n, din]
};
__global__ void __launch_bounds__(128) k_mlp2_fwd(MlpArgs a) {
  __shared__ float w1[MLP_MAX * MLP_MAX], w2[MLP_MAX * MLP_MAX], b1[MLP_MAX], b2[MLP_MAX];
  for (int i = threadIdx.x; i < a.dmid * a.din; i += blockDim.x) w1[i] = a.w1[i];
  for (int i = threadIdx.x; i < a.dout * a.dmid; i += blockDim.x) w2[i] = a.w2[i];
  if (threadIdx.x < a.dmid) b1[threadIdx.x] = a.b1[threadIdx.x];
  if (threadIdx.x < a.dout) b2[threadIdx.x] = a.b2[threadIdx.x];
  __syncthreads();
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < a.n; n += (int64_t)gridDim.x * blockDim.x) {
    float x[MLP_MAX], z[8];
    for (int i = 0; i < a.din; ++i) x[i] = a.x[n * a.din + i];
    for (int o = 0; o < a.dout; ++o) z[o] = b2[o];
    for (int c = 0; c < a.dmid; ++c) {
      float h = b1[c];
      for (int i = 0; i < a.din; ++i) h = fmaf(w1[c * a.din + i], x[i], h);
      a.h[n * a.dmid + c] = h;
      for (int o = 0; o < a.dout; ++o) z[o] = fmaf(w2[o * a.dmid + c], h, z[o]);
    }
    for (int o = 0; o < a.dout; ++o) a.z[n * a.dout + o] = z[o];
  }
}
__global__ void __launch_bounds__(128) k_mlp2_bwd(MlpArgs a) {
  __shared__ float w1[MLP_MAX * MLP_MAX], w2[MLP_MAX * MLP_MAX];
  for (int i = threadIdx.x; i < a.dmid * a.din; i += blockDim.x) w1[i] = a.w1[i];
  for (int i = threadIdx.x; i < a.dout * a.dmid; i += blockDim.x) w2[i] = a.w2[i];
  __syncthreads();
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < a.n; n += (int64_t)gridDim.x * blockDim.x) {
    float gz[8], gx[MLP_MAX];
    for (int o = 0; o < a.dout; ++o) gz[o] = a.gz[n * a.dout + o];
    for (int i = 0; i < a.din; ++i) gx[i] = 0.0f;
    for (int c = 0; c < a.dmid; ++c) {
      float gh = 0.0f;
      for (int o = 0; o < a.dout; ++o) gh = fmaf(w2[o * a.dmid + c], gz[o], gh);
      a.gh[n * a.dmid + c] = gh;
      for (int i = 0; i < a.din; ++i) gx[i] = fmaf(w1[c * a.din + i], gh, gx[i]);
    }
    for (int i = 0; i < a.din; ++i) a.gx[n * a.din + i] = gx[i];
  }
}

// the sizes of the script (dss2_run.py:73-76: 8 -> 32 -> 2) fully unrolled: rows in registers instead of runtime-indexed local arrays
template <int DIN, int DMID, int DOUT>
__global__ void __launch_bounds__(128) k_mlp2_fwd_fixed(MlpArgs a) {
  __shared__ float w1[DMID * DIN], w2[DOUT * DMID], b1[DMID], b2[DOUT];
  for (int i = threadIdx.x; i < DMID * DIN; i += blockDim.x) w1[i] = a.w1[i];
  for (int i = threadIdx.x; i < DOUT * DMID; i += blockDim.x) w2[i] = a.w2[i];
  if (threadIdx.x < DMID) b1[threadIdx.x] = a.b1[threadIdx.x];
  if (threadIdx.x < DOUT) b2[threadIdx.x] = a.b2[threadIdx.x];
  __syncthreads();
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < a.n; n += (int64_t)gridDim.x * blockDim.x) {
    float x[DIN], z[DOUT];
#pragma unroll
    for (int i = 0; i < DIN; ++i) x[i] = a.x[n * DIN + i];
#pragma unroll
    for (int o = 0; o < DOUT; ++o) z[o] = b2[o];
#pragma unroll
    for (int c = 0; c < DMID; ++c) {
      float h = b1[c];
#pragma unroll
      for (int i = 0; i < DIN; ++i) h = fmaf(w1[c * DIN + i], x[i], h);
      if (a.h) a.h[n * DMID + c] = h;      // NULL: the backward is dss2_mlp2_bwd_nh, which never reads it
#pragma unroll
      for (int o = 0; o < DOUT; ++o) z[o] = fmaf(w2[o * DMID + c], h, z[o]);
    }
#pragma unroll
    for (int o = 0; o < DOUT; ++o) a.z[n * DOUT + o] = z[o];
  }
}
// The head has no non-linearity between its two Linears (networks.py:150-151), so every weight gradient is linear in the two small
// sums S = sum_n grad_z[n] (x) x[n] (DOUT x DIN) and s = sum_n grad_z[n]:
//   d W1 = W2^T S,  d b1 = W2^T s,  d W2 = S W1^T + s b1^T,  d b2 = s.
// One pass: grad_x per bus, S and s in registers, one fixed-order reduction per CTA, then the CTA expands ITS S, s into its partial row
// (the expansion is linear, so the sum over the CTA rows is the gradient).  Neither h nor grad_h ever touch memory (the stored-h
// version moved 2 x 128 B per bus for them and ran two more outer-product reductions).
constexpr int MLP_NH_THREADS = 256;
template <int DIN, int DMID, int DOUT>
__global__ void __launch_bounds__(MLP_NH_THREADS) k_mlp2_bwd_nh(MlpArgs a, float* partials, int64_t partial_stride) {
  constexpr int NS = DOUT * (DIN + 1), NW = MLP_NH_THREADS / 32;
  __shared__ float w1[DMID * DIN], w2[DOUT * DMID], b1[DMID], red[NW][NS], tot[NS];
  for (int i = threadIdx.x; i < DMID * DIN; i += blockDim.x) w1[i] = a.w1[i];
  for (int i = threadIdx.x; i < DOUT * DMID; i += blockDim.x) w2[i] = a.w2[i];
  if (threadIdx.x < DMID) b1[threadIdx.x] = a.b1[threadIdx.x];
  __syncthreads();
  float S[DOUT][DIN + 1];
#pragma unroll
  for (int o = 0; o < DOUT; ++o)
#pragma unroll
    for (int i = 0; i <= DIN; ++i) S[o][i] = 0.0f;
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < a.n; n += (int64_t)gridDim.x * blockDim.x) {
    float gz[DOUT], x[DIN], gx[DIN];
#pragma unroll
    for (int o = 0; o < DOUT; ++o) gz[o] = a.gz[n * DOUT + o];
#pragma unroll
    for (int i = 0; i < DIN; ++i) {
      x[i] = a.x[n * DIN + i];
      gx[i] = 0.0f;
    }
#pragma unroll
    for (int c = 0; c < DMID; ++c) {
      float gh = 0.0f;
#pragma unroll
      for (int o = 0; o < DOUT; ++o) gh = fmaf(w2[o * DMID + c], gz[o], gh);
#pragma unroll
      for (int i = 0; i < DIN; ++i) gx[i] = fmaf(w1[c * DIN + i], gh, gx[i]);
    }
#pragma unroll
    for (int i = 0; i < DIN; ++i) a.gx[n * DIN + i] = gx[i];
#pragma unroll
    for (int o = 0; o < DOUT; ++o) {
#pragma unroll
      for (int i = 0; i < DIN; ++i) S[o][i] = fmaf(gz[o], x[i], S[o][i]);
      S[o][DIN] += gz[o];
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 0; o < DOUT; ++o)
#pragma unroll
    for (int i = 0; i <= DIN; ++i) {
      const float v = warp_sum(S[o][i]);
      if (lane == 0) red[warp][o * (DIN + 1) + i] = v;
    }
  __syncthreads();
  if (threadIdx.x < NS) {
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += red[w][threadIdx.x];
    tot[threadIdx.x] = s;
  }
  __syncthreads();
  // partial row layout: [w1 dmid x din | b1 dmid | w2 dout x dmid | b2 dout]
  float* part = partials + (size_t)blockIdx.x * partial_stride;
  constexpr int O_B1 = DMID * DIN, O_W2 = O_B1 + DMID, O_B2 = O_W2 + DOUT * DMID, TOTAL = O_B2 + DOUT;
  for (int idx = threadIdx.x; idx < TOTAL; idx += blockDim.x) {
    float v = 0.0f;
    if (idx < O_B1) {
      const int c = idx / DIN, i = idx % DIN;
#pragma unroll
      for (int o = 0; o < DOUT; ++o) v = fmaf(w2[o * DMID + c], tot[o * (DIN + 1) + i], v);
    } else if (idx < O_W2) {
      const int c = idx - O_B1;
#pragma unroll
      for (int o = 0; o < DOUT; ++o) v = fmaf(w2[o * DMID + c], tot[o * (DIN + 1) + DIN], v);
    } else if (idx < O_B2) {
      const int o = (idx - O_W2) / DMID, c = (idx - O_W2) % DMID;
      v = tot[o * (DIN + 1) + DIN] * b1[c];
#pragma unroll
      for (int i = 0; i < DIN; ++i) v = fmaf(tot[o * (DIN + 1) + i], w1[c * DIN + i], v);
    } else {
      v = tot[(idx - O_B2) * (DIN + 1) + DIN];
    }
    part[idx] = v;
  }
}

template <int DIN, int DMID, int DOUT>
__global__ void __launch_bounds__(128) k_mlp2_bwd_fixed(MlpArgs a) {
  __shared__ float w1[DMID * DIN], w2[DOUT * DMID];
  for (int i = threadIdx.x; i < DMID * DIN; i += blockDim.x) w1[i] = a.w1[i];
  for (int i = threadIdx.x; i < DOUT * DMID; i += blockDim.x) w2[i] = a.w2[i];
  __syncthreads();
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < a.n; n += (int64_t)gridDim.x * blockDim.x) {
    float gz[DOUT], gx[DIN];
#pragma unroll
    for (int o = 0; o < DOUT; ++o) gz[o] = a.gz[n * DOUT + o];
#pragma unroll
    for (int i = 0; i < DIN; ++i) gx[i] = 0.0f;
#pragma unroll
    for (int c = 0; c < DMID; ++c) {
      float gh = 0.0f;
#pragma unroll
      for (int o = 0; o < DOUT; ++o) gh = fmaf(w2[o * DMID + c], gz[o], gh);
      a.gh[n * DMID + c] = gh;
#pragma unroll
      for (int i = 0; i < DIN; ++i) gx[i] = fmaf(w1[c * DIN + i], gh, gx[i]);
    }
#pragma unroll
    for (int i = 0; i < DIN; ++i) a.gx[n * DIN + i] = gx[i];
  }
}

// -------------------------------------------------------------------------------------------------
// GINE_DSSE layer (networks.py:71-111, PyG GINEConv): out_i = nn((1 + eps) x_i + sum_{j -> i} relu(x_j + lin(a_ji))), LeakyReLU.
// `nn` is ONE Linear(8, 8) shared by all layers of the model, `lin` = Linear(edge_dim, 8) per layer.  Same thread-per-bus structure
// as the GATv2 kernels: one-way edge list, in-edges = CSR entries without the reversed bit, out-edges = entries with it.
// -------------------------------------------------------------------------------------------------
constexpr int GINE_NODE_WS = 24;   // per bus: g[8] (gated output gradient), gh[8] (= W_nn^T g), h[8] (input of nn)
struct GineW {
  float wn[GC * GC], bn[GC], we[GC * GFE], be[GC];
};
struct GineArgs {
  dss2_graph_t g;
  const float* x;
  int64_t xs;
  const float* ea;
  int64_t eas;
  int fe;
  const float *wn, *bn, *we, *be;
  float eps, slope_act;
  const float* eps_dev;   // train_eps=True: this layer's eps parameter (device); its gradient lands behind lin.bias in the partial row
  int act;
  float* y;
  const float* yout;
  const float* gy;
  float* ws;
  float* gx;
  float* partials;
  int64_t partial_stride;
};
__device__ __forceinline__ void gine_load_weights(GineW& w, const GineArgs& a) {
  for (int i = threadIdx.x; i < GC * GC; i += blockDim.x) w.wn[i] = a.wn[i];
  for (int i = threadIdx.x; i < GC * GFE; i += blockDim.x) {
    const int c = i / GFE, f = i % GFE;
    w.we[i] = f < a.fe ? a.we[c * a.fe + f] : 0.0f;
  }
  if (threadIdx.x < GC) {
    w.bn[threadIdx.x] = a.bn[threadIdx.x];
    w.be[threadIdx.x] = a.be[threadIdx.x];
  }
}
__device__ __forceinline__ void gine_load_x(const GineArgs& a, int64_t n, float (&v)[GC]) {
  const float* p = a.x + n * a.xs;
#pragma unroll
  for (int i = 0; i < GC; ++i) v[i] = p[i];
}
// pre = x_src + (W_e a + b_e)
__device__ __forceinline__ void gine_pre(const GineArgs& a, const GineW& w, const float (&xs_)[GC], uint32_t id, float (&at)[GFE], float (&pre)[GC]) {
  const float* p = a.ea + (int64_t)(id & 0x7fffffffu) * a.eas;
#pragma unroll
  for (int f = 0; f < GFE; ++f) at[f] = f < a.fe ? p[f] : 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) {
    float e = 0.0f;
#pragma unroll
    for (int f = 0; f < GFE; ++f) e = fmaf(w.we[c * GFE + f], at[f], e);
    pre[c] = xs_[c] + (e + w.be[c]);
  }
}
// h = (1 + eps) x_i + sum over the in-edges of relu(pre)
__device__ __forceinline__ void gine_h(const GineArgs& a, const GineW& w, int64_t i, const float (&xi)[GC], float (&h)[GC]) {
  const dss2_graph_t& g = a.g;
  float agg[GC];
#pragma unroll
  for (int c = 0; c < GC; ++c) agg[c] = 0.0f;
  for (int z = g.rowptr[i]; z < g.rowptr[i + 1]; ++z) {
    const uint32_t id = g.eid[z];
    if (id >> 31) continue;
    float xj[GC], at[GFE], pre[GC];
    gine_load_x(a, g.col[z], xj);
    gine_pre(a, w, xj, id, at, pre);
#pragma unroll
    for (int c = 0; c < GC; ++c) agg[c] += fmaxf(pre[c], 0.0f);
  }
  const float eps = a.eps_dev ? *a.eps_dev : a.eps;
#pragma unroll
  for (int c = 0; c < GC; ++c) h[c] = agg[c] + (1.0f + eps) * xi[c];
}
__global__ void __launch_bounds__(GAT_THREADS) k_gine_fwd(GineArgs a) {
  __shared__ GineW w;
  gine_load_weights(w, a);
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    float xi[GC], h[GC], out[GC];
    gine_load_x(a, i, xi);
    gine_h(a, w, i, xi, h);
    lin8(w.wn, w.bn, h, out);
#pragma unroll
    for (int c = 0; c < GC; ++c) out[c] = a.act == 2 ? tanhf(out[c]) : ((a.act == 1 && !(out[c] > 0.0f)) ? out[c] * a.slope_act : out[c]);
    float4* dst = reinterpret_cast<float4*>(a.y + i * GC);
    dst[0] = make_float4(out[0], out[1], out[2], out[3]);
    dst[1] = make_float4(out[4], out[5], out[6], out[7]);
  }
}
// backward pass A: per bus g = grad_y * gate, gh = W_nn^T g, h (recomputed)
__global__ void __launch_bounds__(GAT_THREADS) k_gine_bwd_a(GineArgs a) {
  __shared__ GineW w;
  gine_load_weights(w, a);
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    float xi[GC], h[GC], G[GC];
    gine_load_x(a, i, xi);
    gine_h(a, w, i, xi, h);
    float* o = a.ws + i * GINE_NODE_WS;
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      const float yv = a.yout[i * GC + c];
      const float gate = a.act == 2 ? 1.0f - yv * yv : ((a.act == 1 && !(yv > 0.0f)) ? a.slope_act : 1.0f);
      G[c] = a.gy[i * GC + c] * gate;
      o[c] = G[c];
      o[16 + c] = h[c];
    }
#pragma unroll
    for (int k = 0; k < GC; ++k) {
      float s = 0.0f;
#pragma unroll
      for (int c = 0; c < GC; ++c) s = fmaf(w.wn[c * GC + k], G[c], s);
      o[8 + k] = s;
    }
  }
}
// backward pass B: thread = bus n: d W_e / d b_e of its in-edges, d x[n] from its own term and its out-edges.
// partial layout per CTA at a.partials: [lin.weight 8 x fe | lin.bias 8]
__global__ void __launch_bounds__(GAT_BWD_THREADS) k_gine_bwd_b(GineArgs a) {
  __shared__ GineW w;
  __shared__ float red[GAT_BWD_THREADS / 32][GC * GFE + GC];
  gine_load_weights(w, a);
  __syncthreads();
  const dss2_graph_t& g = a.g;
  float dWe[GC * GFE], dbe[GC], deps = 0.0f;
  const float eps = a.eps_dev ? *a.eps_dev : a.eps;
#pragma unroll
  for (int i = 0; i < GC * GFE; ++i) dWe[i] = 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) dbe[c] = 0.0f;
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < g.num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    float xn[GC], ghn[GC], dx[GC];
    gine_load_x(a, n, xn);
    const float* sn = a.ws + n * GINE_NODE_WS;
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      ghn[c] = sn[8 + c];
      dx[c] = (1.0f + eps) * ghn[c];
      deps = fmaf(ghn[c], xn[c], deps);   // d/d eps of (1 + eps) x_n . gh_n
    }
    for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
      const uint32_t id = g.eid[z];
      const int o = g.col[z];
      float at[GFE], pre[GC];
      if (!(id >> 31)) {   // in-edge (o -> n)
        float xo[GC];
        gine_load_x(a, o, xo);
        gine_pre(a, w, xo, id, at, pre);
#pragma unroll
        for (int c = 0; c < GC; ++c) {
          const float t = pre[c] > 0.0f ? ghn[c] : 0.0f;
          dbe[c] += t;
#pragma unroll
          for (int f = 0; f < GFE; ++f) dWe[c * GFE + f] = fmaf(t, at[f], dWe[c * GFE + f]);
        }
      } else {             // out-edge (n -> o)
        gine_pre(a, w, xn, id, at, pre);
        const float* so = a.ws + (int64_t)o * GINE_NODE_WS;
#pragma unroll
        for (int c = 0; c < GC; ++c) dx[c] += pre[c] > 0.0f ? so[8 + c] : 0.0f;
      }
    }
    if (a.gx) {
      float4* dst = reinterpret_cast<float4*>(a.gx + n * GC);
      dst[0] = make_float4(dx[0], dx[1], dx[2], dx[3]);
      dst[1] = make_float4(dx[4], dx[5], dx[6], dx[7]);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < GC * GFE; ++i) {
    const float v = warp_sum(dWe[i]);
    if (lane == 0) red[warp][i] = v;
  }
#pragma unroll
  for (int c = 0; c < GC; ++c) {
    const float v = warp_sum(dbe[c]);
    if (lane == 0) red[warp][GC * GFE + c] = v;
  }
  __shared__ float red_eps[GAT_BWD_THREADS / 32];
  {
    const float v = warp_sum(deps);
    if (lane == 0) red_eps[warp] = v;
  }
  __syncthreads();
  float* part = a.partials + (size_t)blockIdx.x * a.partial_stride;
  for (int i = threadIdx.x; i < GC * a.fe + GC; i += blockDim.x) {
    const int src = i < GC * a.fe ? (i / a.fe) * GFE + (i % a.fe) : GC * GFE + (i - GC * a.fe);
    float s = 0.0f;
#pragma unroll
    for (int wv = 0; wv < GAT_BWD_THREADS / 32; ++wv) s += red[wv][src];
    part[i] = s;
  }
  if (a.eps_dev && threadIdx.x == 0) {
    float s = 0.0f;
#pragma unroll
    for (int wv = 0; wv < GAT_BWD_THREADS / 32; ++wv) s += red_eps[wv];
    part[GC * a.fe + GC] = s;
  }
}

// -------------------------------------------------------------------------------------------------
// gnn_dsse (networks.py:11-69): GCN2Conv / TAGConv stacks at width dim_feat <= 8 on the ONE-WAY edge list as given (the model does not
// un-direct it), built from four small thread-per-bus kernels.  The CSR rows of dss2_graph_t hold the in-edges of a bus (entries
// without the reversed flag, in edge order = PyG's scatter order) and, flagged, its out-edges: the transposed propagation of the
// backward walks the same row.
// self_loops = 1 is gcn_norm(add_self_loops=True), i.e. PyG's add_remaining_self_loops: the self loops of the input are dropped (an
// entry with col == i) and exactly one loop of weight 1 per bus is appended last.  self_loops = 0 takes the edge list as given: an
// input loop is an ordinary edge (TAGConv's gcn_norm(add_self_loops=False)).
// -------------------------------------------------------------------------------------------------
struct GnnArgs {
  dss2_graph_t g;
  const float* dinv;     // [Nt] deg^-1/2 of gcn_norm (in-degree; with self loops: input loops not counted, + 1), inf -> 0
  int self_loops;
  int transposed;
  const float* x;        // [Nt, >= 8], row stride xs
  int64_t xs;
  float scale;           // out = scale * (A x) + add_scale * add
  const float* add;
  int64_t adds;
  float add_scale;
  float* out;            // [Nt, 8]
};

__global__ void __launch_bounds__(GAT_THREADS) k_gcn_dinv(dss2_graph_t g, int self_loops, float* dinv) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    int deg = self_loops ? 1 : 0;
    for (int z = g.rowptr[i]; z < g.rowptr[i + 1]; ++z) deg += ((g.eid[z] >> 31) || (self_loops && g.col[z] == i)) ? 0 : 1;
    dinv[i] = deg > 0 ? 1.0f / sqrtf((float)deg) : 0.0f;   // deg.pow(-0.5), inf -> 0 (gcn_norm)
  }
}

// out[i] = scale * sum_{j -> i} dinv[j] dinv[i] x[j] (+ self loop last, as add_remaining_self_loops appends it) + add_scale * add[i];
// with self loops the input loops (j == i) are skipped, in both directions.
// transposed: the sum runs over the out-edges i -> j instead (adjoint of the propagation).  Every product / sum is rounded on its own
// like the eager ops of the reference (no fused multiply-add).
__global__ void __launch_bounds__(GAT_THREADS) k_prop8(GnnArgs a) {
  const dss2_graph_t& g = a.g;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    const float di = a.dinv[i];
    float acc[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) acc[c] = 0.0f;
    for (int z = g.rowptr[i]; z < g.rowptr[i + 1]; ++z) {
      const bool rev = g.eid[z] >> 31;
      if (rev != (a.transposed != 0)) continue;
      const int64_t j = g.col[z];
      if (a.self_loops && j == i) continue;   // an input loop: replaced by the appended one
      const float w = __fmul_rn(a.dinv[j], di);
      const float* xj = a.x + j * a.xs;
#pragma unroll
      for (int c = 0; c < GC; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(w, xj[c]));
    }
    if (a.self_loops) {
      const float w = __fmul_rn(di, di);
      const float* xi = a.x + i * a.xs;
#pragma unroll
      for (int c = 0; c < GC; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(w, xi[c]));
    }
    float o[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      o[c] = __fmul_rn(acc[c], a.scale);
      if (a.add) o[c] = __fadd_rn(o[c], __fmul_rn(a.add_scale, a.add[i * a.adds + c]));
    }
    float4* dst = reinterpret_cast<float4*>(a.out + i * GC);
    dst[0] = make_float4(o[0], o[1], o[2], o[3]);
    dst[1] = make_float4(o[4], o[5], o[6], o[7]);
  }
}

struct Lin8Args {
  int64_t num_nodes;
  int M;                  // matrices (1 for GCN2Conv, K + 1 for TAGConv)
  int wt;                 // 0: z = in W (GCN2Conv weight1 [in, out]); 1: z = in W^T (Linear weight [out, in])
  const float* in[4];     // [Nt, >= 8] each
  int64_t ins[4];
  const float* w;         // [M][8][8]
  const float* bias;      // [8] or NULL
  int act;                // 0 none, 1 leaky_relu(slope), 2 relu, 3 tanh
  float slope;
  float* y;               // fwd: [Nt, 8]
  const float* yout;      // bwd: the forward's y
  const float* gy;        // bwd: [Nt, 8]
  float* gz;              // bwd: [Nt, 8] adjoint of the pre-activation (input of the weight-gradient reduction)
  float* gin[4];          // bwd: [Nt, 8] adjoint of in[m]
  float* acc;             // bwd, optional: acc[n] += acc_scale * gin[0][n]   (GCN2Conv: the x_0 path)
  float acc_scale;
};
struct Lin8W {
  float w[4][GC * GC], b[GC];
};
__device__ __forceinline__ void lin8_load(Lin8W& s, const Lin8Args& a) {
  for (int i = threadIdx.x; i < a.M * GC * GC; i += blockDim.x) s.w[i / (GC * GC)][i % (GC * GC)] = a.w[i];
  if (threadIdx.x < GC) s.b[threadIdx.x] = a.bias ? a.bias[threadIdx.x] : 0.0f;
}
__global__ void __launch_bounds__(GAT_THREADS) k_lin8_fwd(Lin8Args a) {
  __shared__ Lin8W s;
  lin8_load(s, a);
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    float z[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) z[c] = 0.0f;
    for (int m = 0; m < a.M; ++m) {
      float v[GC], t[GC];
      const float* p = a.in[m] + i * a.ins[m];
#pragma unroll
      for (int j = 0; j < GC; ++j) v[j] = p[j];
#pragma unroll
      for (int c = 0; c < GC; ++c) {
        float d = 0.0f;
#pragma unroll
        for (int j = 0; j < GC; ++j) d = fmaf(v[j], a.wt ? s.w[m][c * GC + j] : s.w[m][j * GC + c], d);
        t[c] = d;
      }
#pragma unroll
      for (int c = 0; c < GC; ++c) z[c] = m == 0 ? t[c] : z[c] + t[c];   // out = lins[0](x); out = out + lins[k](x_k)
    }
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      float v = a.bias ? z[c] + s.b[c] : z[c];
      if (a.act == 1) v = v > 0.0f ? v : v * a.slope;
      else if (a.act == 2) v = fmaxf(v, 0.0f);
      else if (a.act == 3) v = tanhf(v);
      z[c] = v;
    }
    float4* dst = reinterpret_cast<float4*>(a.y + i * GC);
    dst[0] = make_float4(z[0], z[1], z[2], z[3]);
    dst[1] = make_float4(z[4], z[5], z[6], z[7]);
  }
}
__global__ void __launch_bounds__(GAT_THREADS) k_lin8_bwd(Lin8Args a) {
  __shared__ Lin8W s;
  lin8_load(s, a);
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    float g[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      const float y = a.yout ? a.yout[i * GC + c] : 0.0f;
      float d = 1.0f;
      if (a.act == 1) d = y > 0.0f ? 1.0f : a.slope;
      else if (a.act == 2) d = y > 0.0f ? 1.0f : 0.0f;
      else if (a.act == 3) d = 1.0f - y * y;
      g[c] = a.gy[i * GC + c] * d;
    }
    float4* gz = reinterpret_cast<float4*>(a.gz + i * GC);
    gz[0] = make_float4(g[0], g[1], g[2], g[3]);
    gz[1] = make_float4(g[4], g[5], g[6], g[7]);
    for (int m = 0; m < a.M; ++m) {
      float o[GC];
#pragma unroll
      for (int j = 0; j < GC; ++j) {
        float d = 0.0f;
#pragma unroll
        for (int c = 0; c < GC; ++c) d = fmaf(g[c], a.wt ? s.w[m][c * GC + j] : s.w[m][j * GC + c], d);
        o[j] = d;
      }
      float4* dst = reinterpret_cast<float4*>(a.gin[m] + i * GC);
      dst[0] = make_float4(o[0], o[1], o[2], o[3]);
      dst[1] = make_float4(o[4], o[5], o[6], o[7]);
      if (m == 0 && a.acc) {
#pragma unroll
        for (int j = 0; j < GC; ++j) a.acc[i * GC + j] += a.acc_scale * o[j];
      }
    }
  }
}

struct GatPrepArgs {
  const float *wl[GAT_SLOTS], *bl[GAT_SLOTS], *wr[GAT_SLOTS], *br[GAT_SLOTS], *we[GAT_SLOTS], *att[GAT_SLOTS], *bias[GAT_SLOTS];
  int fe, first;
};
__global__ void k_gat_prep(GatPrepArgs p) {
  const int s = p.first + blockIdx.x, q = blockIdx.x;
  GatW& w = g_gat_stage[s];
  for (int i = threadIdx.x; i < GC * GC; i += blockDim.x) {
    w.wl[i] = p.wl[q][i];
    w.wr[i] = p.wr[q][i];
  }
  for (int i = threadIdx.x; i < GC * GFE; i += blockDim.x) {
    const int c = i / GFE, f = i % GFE;
    w.we[i] = f < p.fe ? p.we[q][c * p.fe + f] : 0.0f;
  }
  if (threadIdx.x < GC) {
    w.bl[threadIdx.x] = p.bl[q][threadIdx.x];
    w.br[threadIdx.x] = p.br[q][threadIdx.x];
    w.att[threadIdx.x] = p.att[q][threadIdx.x];
    w.bias[threadIdx.x] = p.bias[q][threadIdx.x];
  }
}

#define GAT_SLOT_CASE(S, KERN, GRID, THREADS)                  \
  case S:                                                      \
    if (a.drop.mode) KERN<S, true><<<GRID, THREADS, 0, stream>>>(a); \
    else KERN<S, false><<<GRID, THREADS, 0, stream>>>(a);            \
    break;
#define GAT_SLOT_LAUNCH(slot, KERN, GRID, THREADS) \
  switch (slot) {                                  \
    GAT_SLOT_CASE(-1, KERN, GRID, THREADS)         \
    GAT_SLOT_CASE(0, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(1, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(2, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(3, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(4, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(5, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(6, KERN, GRID, THREADS)          \
    GAT_SLOT_CASE(7, KERN, GRID, THREADS)          \
    default:                                \
      dss2_set_error("GAT weight slot %d outside -1..%d", slot, GAT_SLOTS - 1); \
      return -1;                            \
  }

// dss2_attn_drop_t -> kernel arguments; mode stays 0 (the DROP = false kernels) for a NULL descriptor, p = 0 or mode 0
int fill_drop(const char* who, AttnDropArgs& d, const dss2_attn_drop_t* drop, int64_t num_edges) {
  d = AttnDropArgs{};
  if (!drop) return 0;
  DSS2_CHECK_ARG(drop->p >= 0.0f && drop->p < 1.0f, "%s: attention dropout p %f outside [0, 1)", who, drop->p);
  DSS2_CHECK_ARG(drop->mode >= 0 && drop->mode <= 2, "%s: attention dropout mode %d outside 0..2", who, drop->mode);
  DSS2_CHECK_ARG(drop->mode != 1 || drop->rng_state, "%s: philox attention dropout needs rng_state", who);
  DSS2_CHECK_ARG(drop->mode != 2 || drop->mask, "%s: mask attention dropout needs a mask", who);
  DSS2_CHECK_ARG(drop->head < 0x10000u, "%s: head %u outside 0..65535", who, drop->head);
  if (drop->p == 0.0f || drop->mode == 0) return 0;
  d.mode = drop->mode;
  d.scale = 1.0f / (float)(1.0 - (double)drop->p);
  const double thr = (1.0 - (double)drop->p) * 4294967296.0;
  d.keep_thr = thr >= 4294967295.0 ? 0xffffffffu : (uint32_t)thr;
  d.layer_uid = drop->layer_uid;
  d.head = drop->head;
  d.rng = drop->rng_state;
  d.mask = drop->mask;
  d.num_edges = num_edges;
  return 0;
}

int grid_for(int64_t n, int threads) { return (int)max((int64_t)1, min((int64_t)dss2_sm_count() * 8, (n + threads - 1) / threads)); }

int fill_args(const char* who, GatArgs& a, const dss2_graph_t* g, const float* x, int64_t xs, const float* ea, int64_t eas, int fe,
              const float* wl, const float* bl, const float* wr, const float* br, const float* we, const float* att, const float* bias,
              float slope_att, int act, float slope_act, int slot = -1) {
  DSS2_CHECK_ARG(g && x && ea, "%s: null argument", who);
  DSS2_CHECK_ARG(slot >= 0 || (wl && bl && wr && br && we && att && bias), "%s: null weight pointer", who);
  DSS2_CHECK_ARG(fe >= 1 && fe <= GFE, "%s: edge_dim %d outside 1..%d", who, fe, GFE);
  DSS2_CHECK_ARG(xs >= GC && eas >= fe, "%s: row strides too small", who);
  a.g = *g;
  a.x = x;
  a.xs = xs;
  a.ea = ea;
  a.eas = eas;
  a.fe = fe;
  a.wl = wl;
  a.bl = bl;
  a.wr = wr;
  a.br = br;
  a.we = we;
  a.att = att;
  a.bias = bias;
  a.slope_att = slope_att;
  a.act = act & 0xff;
  a.loops = (act & DSS2_GAT_NO_SELF_LOOPS) ? 0 : 1;
  a.slope_act = slope_act;
  return 0;
}

}  // namespace

extern "C" size_t dss2_gat_ws_bytes(int64_t num_nodes) { return (size_t)num_nodes * GAT_NODE_WS * sizeof(float); }

static int gat_fwd_impl(int slot, const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                        const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                        const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                        const dss2_attn_drop_t* drop, float* y, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  GatArgs a = {};
  if (fill_args("dss2_gat_fwd", a, g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias,
                att_slope, act, act_slope, slot))
    return -1;
  if (fill_drop("dss2_gat_fwd", a.drop, drop, g->num_edges)) return -1;
  DSS2_CHECK_ARG(y && ((uintptr_t)y & 15) == 0, "dss2_gat_fwd: y must be a 16-byte aligned [Nt, 8] buffer");
  if (g->num_nodes == 0) return 0;
  a.y = y;
  GAT_SLOT_LAUNCH(slot, k_gat_fwd, grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_gat_fwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                            const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                            const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                            float* y, void* stream_) {
  return gat_fwd_impl(-1, g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias, att_slope, act,
                      act_slope, nullptr, y, stream_);
}

extern "C" int dss2_gat_fwd_drop(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                 int slot, const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                                 const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                                 const dss2_attn_drop_t* drop, float* y, void* stream_) {
  return gat_fwd_impl(slot, g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias, att_slope, act,
                      act_slope, drop, y, stream_);
}

extern "C" int dss2_attn_drop_mask(const dss2_attn_drop_t* drop, int64_t num_edges, int64_t num_nodes, uint8_t* out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(drop && out && num_edges >= 0 && num_nodes >= 0, "dss2_attn_drop_mask: null or negative argument");
  AttnDropArgs d;
  if (fill_drop("dss2_attn_drop_mask", d, drop, num_edges)) return -1;
  const int64_t n = num_edges + num_nodes;
  if (n == 0) return 0;
  if (!d.mode) {   // no dropout: every coefficient kept
    DSS2_CUDA(cudaMemsetAsync(out, 1, (size_t)n, stream));
    return 0;
  }
  k_attn_drop_mask<<<grid_for(n, 256), 256, 0, stream>>>(d, n, out);
  DSS2_LAUNCH_CHECK();
  return 0;
}

// Weights of `count` layers -> constant-memory slots first .. first + count - 1: one layout kernel + one device-to-device copy (both
// capturable).  The slot variants of the layer kernels then read every weight as an immediate constant operand.
extern "C" int dss2_gat_upload(int first, int count, const float* const* lin_l_w, const float* const* lin_l_b, const float* const* lin_r_w,
                               const float* const* lin_r_b, const float* const* lin_edge_w, const float* const* att, const float* const* bias,
                               int fe, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(first >= 0 && count >= 1 && first + count <= GAT_SLOTS, "dss2_gat_upload: slots %d..%d outside 0..%d", first, first + count - 1,
                 GAT_SLOTS - 1);
  DSS2_CHECK_ARG(fe >= 1 && fe <= GFE, "dss2_gat_upload: edge_dim %d outside 1..%d", fe, GFE);
  GatPrepArgs p = {};
  for (int q = 0; q < count; ++q) {
    DSS2_CHECK_ARG(lin_l_w[q] && lin_l_b[q] && lin_r_w[q] && lin_r_b[q] && lin_edge_w[q] && att[q] && bias[q], "dss2_gat_upload: null pointer");
    p.wl[q] = lin_l_w[q], p.bl[q] = lin_l_b[q], p.wr[q] = lin_r_w[q], p.br[q] = lin_r_b[q], p.we[q] = lin_edge_w[q], p.att[q] = att[q];
    p.bias[q] = bias[q];
  }
  p.fe = fe;
  p.first = first;
  k_gat_prep<<<count, 64, 0, stream>>>(p);
  DSS2_LAUNCH_CHECK();
  void* stage = nullptr;
  DSS2_CUDA(cudaGetSymbolAddress(&stage, g_gat_stage));
  DSS2_CUDA(cudaMemcpyToSymbolAsync(c_gat, (const char*)stage + (size_t)first * sizeof(GatW), (size_t)count * sizeof(GatW),
                                    (size_t)first * sizeof(GatW), cudaMemcpyDeviceToDevice, stream));
  return 0;
}

extern "C" int dss2_gat_fwd_slot(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                 int slot, float att_slope, int act, float act_slope, float* y, void* stream_) {
  DSS2_CHECK_ARG(slot >= 0 && slot < GAT_SLOTS, "dss2_gat_fwd_slot: slot %d outside 0..%d", slot, GAT_SLOTS - 1);
  return gat_fwd_impl(slot, g, x, x_stride, edge_attr, ea_stride, fe, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, att_slope,
                      act, act_slope, nullptr, y, stream_);
}

// part_off[7]: offsets (floats, relative to `partials`) of the blocks [lin_l.w 64, lin_l.b 8, lin_r.w 64, lin_r.b 8, lin_edge.w 8 fe, att 8,
// bias 8] inside a partial row: one head of a multi-head layer writes into that head's slice of every parameter.
static int gat_bwd_impl(int slot, const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                        const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                        const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                        const dss2_attn_drop_t* drop, const float* y, const float* grad_y, float* grad_x, float* node_ws,
                        size_t node_ws_bytes, float* partials, int64_t partial_stride, const int64_t* part_off, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  GatArgs a = {};
  if (fill_args("dss2_gat_bwd", a, g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias,
                att_slope, act, act_slope, slot))
    return -1;
  if (fill_drop("dss2_gat_bwd", a.drop, drop, g->num_edges)) return -1;
  DSS2_CHECK_ARG(grad_y && node_ws && partials && part_off && (!(act & 0xff) || y), "dss2_gat_bwd: null argument");
  DSS2_CHECK_ARG(g->undirected == 1, "dss2_gat_bwd: needs a graph built from the one-way edge list with undirect=1 (out-edges of a bus are "
                 "found through the reversed entries)");
  DSS2_CHECK_ARG(node_ws_bytes >= dss2_gat_ws_bytes(g->num_nodes), "dss2_gat_bwd: node workspace too small");
  for (int i = 0; i < 7; ++i) {
    const int64_t n = i == 0 || i == 2 ? GC * GC : i == 4 ? GC * fe : GC;
    DSS2_CHECK_ARG(part_off[i] >= 0 && part_off[i] + n <= partial_stride, "dss2_gat_bwd: partial block %d outside the partial row", i);
  }
  DSS2_CHECK_ARG(!grad_x || ((uintptr_t)grad_x & 15) == 0, "dss2_gat_bwd: grad_x must be 16-byte aligned");
  if (g->num_nodes == 0) return 0;
  a.yout = y;
  a.gy = grad_y;
  a.ws = node_ws;
  a.gx = grad_x;
  GAT_SLOT_LAUNCH(slot, k_gat_bwd_stats, grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS);
  DSS2_LAUNCH_CHECK();
  const int np = dss2_num_partials();
  a.partials = partials + part_off[4];
  a.off_att = part_off[5] - part_off[4];
  a.off_bias = part_off[6] - part_off[4];
  a.partial_stride = partial_stride;
  GAT_SLOT_LAUNCH(slot, k_gat_bwd, np, GAT_BWD_THREADS);
  DSS2_LAUNCH_CHECK();
  // d W_l | d b_l and d W_r | d b_r from the stored node adjoints (columns 20..27 and 28..35 of the workspace)
  if (part_off[2] == part_off[0] + GC * GC && part_off[3] == part_off[1] + GC) {
    // [lin_l.w | lin_r.w] and [lin_l.b | lin_r.b] adjacent in the partial row: ONE reduction over the 16 adjoint columns
    launch_outer_reduce(np, stream, g->num_nodes, node_ws + 20, GAT_NODE_WS, 2 * GC, x, x_stride, GC, partials, partial_stride, part_off[0],
                        part_off[1]);
    DSS2_LAUNCH_CHECK();
    return 0;
  }
  launch_outer_reduce(np, stream, g->num_nodes, node_ws + 20, GAT_NODE_WS, GC, x, x_stride, GC, partials, partial_stride, part_off[0], part_off[1]);
  DSS2_LAUNCH_CHECK();
  launch_outer_reduce(np, stream, g->num_nodes, node_ws + 28, GAT_NODE_WS, GC, x, x_stride, GC, partials, partial_stride, part_off[2], part_off[3]);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_gat_bwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                               const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                               const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                               const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes, float* partials,
                               int64_t partial_stride, const int64_t* part_off, void* stream_) {
  return gat_bwd_impl(-1, g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias, att_slope, act,
                      act_slope, nullptr, y, grad_y, grad_x, node_ws, node_ws_bytes, partials, partial_stride, part_off, stream_);
}

extern "C" int dss2_gat_bwd_drop(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                 int slot, const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                                 const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                                 const dss2_attn_drop_t* drop, const float* y, const float* grad_y, float* grad_x, float* node_ws,
                                 size_t node_ws_bytes, float* partials, int64_t partial_stride, const int64_t* part_off, void* stream_) {
  const int64_t w = GC * GC, e0 = 2 * (w + GC);
  const int64_t off[7] = {0, w, w + GC, 2 * w + GC, e0, e0 + (int64_t)GC * fe, e0 + (int64_t)GC * fe + GC};
  return gat_bwd_impl(slot, g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias, att_slope, act,
                      act_slope, drop, y, grad_y, grad_x, node_ws, node_ws_bytes, partials, partial_stride, part_off ? part_off : off, stream_);
}

// the backward of a layer whose weights sit in constant-memory slot `slot` (part_off as in dss2_gat_bwd_ex; NULL: the standard partial row)
extern "C" int dss2_gat_bwd_slot(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                 int slot, float att_slope, int act, float act_slope, const float* y, const float* grad_y, float* grad_x,
                                 float* node_ws, size_t node_ws_bytes, float* partials, int64_t partial_stride, const int64_t* part_off,
                                 void* stream_) {
  DSS2_CHECK_ARG(slot >= 0 && slot < GAT_SLOTS, "dss2_gat_bwd_slot: slot %d outside 0..%d", slot, GAT_SLOTS - 1);
  const int64_t w = GC * GC, e0 = 2 * (w + GC);
  const int64_t off[7] = {0, w, w + GC, 2 * w + GC, e0, e0 + (int64_t)GC * fe, e0 + (int64_t)GC * fe + GC};
  return gat_bwd_impl(slot, g, x, x_stride, edge_attr, ea_stride, fe, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, att_slope,
                      act, act_slope, nullptr, y, grad_y, grad_x, node_ws, node_ws_bytes, partials, partial_stride, part_off ? part_off : off,
                      stream_);
}

// partial row: [lin_l.w 64 | lin_l.b 8 | lin_r.w 64 | lin_r.b 8 | lin_edge.w 8 fe | att 8 | bias 8]
extern "C" int dss2_gat_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                            const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                            const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                            const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes, float* partials,
                            int64_t partial_stride, void* stream_) {
  const int64_t w = GC * GC, e0 = 2 * (w + GC);
  const int64_t off[7] = {0, w, w + GC, 2 * w + GC, e0, e0 + (int64_t)GC * fe, e0 + (int64_t)GC * fe + GC};
  return dss2_gat_bwd_ex(g, x, x_stride, edge_attr, ea_stride, fe, lin_l_w, lin_l_b, lin_r_w, lin_r_b, lin_edge_w, att, bias, att_slope, act,
                         act_slope, y, grad_y, grad_x, node_ws, node_ws_bytes, partials, partial_stride, off, stream_);
}

extern "C" size_t dss2_gine_ws_bytes(int64_t num_nodes) { return (size_t)num_nodes * GINE_NODE_WS * sizeof(float); }

static int gine_fill(const char* who, GineArgs& a, const dss2_graph_t* g, const float* x, int64_t xs, const float* ea, int64_t eas, int fe,
                     const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, int act, float act_slope) {
  DSS2_CHECK_ARG(g && x && ea && nn_w && nn_b && lin_w && lin_b, "%s: null argument", who);
  DSS2_CHECK_ARG(fe >= 1 && fe <= GFE && xs >= GC && eas >= fe, "%s: edge_dim %d outside 1..%d or row strides too small", who, fe, GFE);
  a.g = *g;
  a.x = x;
  a.xs = xs;
  a.ea = ea;
  a.eas = eas;
  a.fe = fe;
  a.wn = nn_w;
  a.bn = nn_b;
  a.we = lin_w;
  a.be = lin_b;
  a.eps = eps;
  a.act = act;
  a.slope_act = act_slope;
  return 0;
}

extern "C" int dss2_gine_fwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, const float* eps_param,
                                int act, float act_slope, float* y, void* stream_);
extern "C" int dss2_gine_fwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                             const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, int act,
                             float act_slope, float* y, void* stream_) {
  return dss2_gine_fwd_ex(g, x, x_stride, edge_attr, ea_stride, fe, nn_w, nn_b, lin_w, lin_b, eps, nullptr, act, act_slope, y, stream_);
}
extern "C" int dss2_gine_fwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, const float* eps_param,
                                int act, float act_slope, float* y, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  GineArgs a = {};
  if (gine_fill("dss2_gine_fwd", a, g, x, x_stride, edge_attr, ea_stride, fe, nn_w, nn_b, lin_w, lin_b, eps, act, act_slope)) return -1;
  a.eps_dev = eps_param;
  DSS2_CHECK_ARG(y && ((uintptr_t)y & 15) == 0, "dss2_gine_fwd: y must be a 16-byte aligned [Nt, 8] buffer");
  if (g->num_nodes == 0) return 0;
  a.y = y;
  k_gine_fwd<<<grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

// partials_lin: per-CTA rows [lin.weight 8 fe | lin.bias 8]; partials_nn: per-CTA rows [nn.weight 64 | nn.bias 8] of THIS layer's share of
// the shared Linear's gradient (the host adds the layers' shares); both with row stride partial_stride, dss2_num_partials() rows.
extern "C" int dss2_gine_bwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, const float* eps_param,
                                int act, float act_slope, const float* y, const float* grad_y, float* grad_x, float* node_ws,
                                size_t node_ws_bytes, float* partials_lin, float* partials_nn, int64_t partial_stride, void* stream_);
extern "C" int dss2_gine_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                             const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, int act,
                             float act_slope, const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes,
                             float* partials_lin, float* partials_nn, int64_t partial_stride, void* stream_) {
  return dss2_gine_bwd_ex(g, x, x_stride, edge_attr, ea_stride, fe, nn_w, nn_b, lin_w, lin_b, eps, nullptr, act, act_slope, y, grad_y, grad_x, node_ws,
                          node_ws_bytes, partials_lin, partials_nn, partial_stride, stream_);
}
// eps_param != NULL (train_eps=True): eps is read from the device and its gradient is written as one more element of the partials_lin
// row: [lin.weight 8 fe | lin.bias 8 | eps 1]
extern "C" int dss2_gine_bwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                                const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, const float* eps_param,
                                int act, float act_slope, const float* y, const float* grad_y, float* grad_x, float* node_ws,
                                size_t node_ws_bytes, float* partials_lin, float* partials_nn, int64_t partial_stride, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  GineArgs a = {};
  if (gine_fill("dss2_gine_bwd", a, g, x, x_stride, edge_attr, ea_stride, fe, nn_w, nn_b, lin_w, lin_b, eps, act, act_slope)) return -1;
  a.eps_dev = eps_param;
  DSS2_CHECK_ARG(grad_y && node_ws && partials_lin && partials_nn && (!act || y), "dss2_gine_bwd: null argument");
  DSS2_CHECK_ARG(g->undirected == 1, "dss2_gine_bwd: needs a graph built from the one-way edge list with undirect=1");
  DSS2_CHECK_ARG(node_ws_bytes >= dss2_gine_ws_bytes(g->num_nodes), "dss2_gine_bwd: node workspace too small");
  DSS2_CHECK_ARG(!grad_x || ((uintptr_t)grad_x & 15) == 0, "dss2_gine_bwd: grad_x must be 16-byte aligned");
  if (g->num_nodes == 0) return 0;
  a.yout = y;
  a.gy = grad_y;
  a.ws = node_ws;
  a.gx = grad_x;
  k_gine_bwd_a<<<grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  const int np = dss2_num_partials();
  a.partials = partials_lin;
  a.partial_stride = partial_stride;
  k_gine_bwd_b<<<np, GAT_BWD_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  // d W_nn | d b_nn = sum_n g[n] (x) [h[n], 1]
  launch_outer_reduce(np, stream, g->num_nodes, node_ws, GINE_NODE_WS, GC, node_ws + 16, GINE_NODE_WS, GC, partials_nn,
                                                partial_stride, 0, GC * GC);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_mlp2_fwd(int64_t num_nodes, const float* x, int din, const float* w1, const float* b1, int dmid, const float* w2,
                             const float* b2, int dout, float* h, float* z, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x && w1 && b1 && w2 && b2 && z, "dss2_mlp2_fwd: null argument");
  DSS2_CHECK_ARG(din >= 1 && din <= MLP_MAX && dmid >= 1 && dmid <= MLP_MAX && dout >= 1 && dout <= 8, "dss2_mlp2_fwd: sizes %d -> %d -> %d unsupported",
                 din, dmid, dout);
  if (num_nodes == 0) return 0;
  MlpArgs a = {};
  a.n = num_nodes;
  a.x = x;
  a.din = din;
  a.w1 = w1;
  a.b1 = b1;
  a.dmid = dmid;
  a.w2 = w2;
  a.b2 = b2;
  a.dout = dout;
  a.h = h;
  a.z = z;
  DSS2_CHECK_ARG(h || (din == 8 && dmid == 32 && dout == 2), "dss2_mlp2_fwd: h may be NULL only where dss2_mlp2_nh_supported()");
  if (din == 8 && dmid == 32 && dout == 2) k_mlp2_fwd_fixed<8, 32, 2><<<grid_for(num_nodes, 128), 128, 0, stream>>>(a);
  else k_mlp2_fwd<<<grid_for(num_nodes, 128), 128, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

// partial row layout: [w1 dmid x din | b1 dmid | w2 dout x dmid | b2 dout]
extern "C" int dss2_mlp2_bwd(int64_t num_nodes, const float* x, int din, const float* w1, int dmid, const float* w2, int dout,
                             const float* h, const float* grad_z, float* grad_h_ws, float* grad_x, float* partials, int64_t partial_stride,
                             void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x && w1 && w2 && h && grad_z && grad_h_ws && grad_x && partials, "dss2_mlp2_bwd: null argument");
  DSS2_CHECK_ARG(din >= 1 && din <= MLP_MAX && dmid >= 1 && dmid <= MLP_MAX && dout >= 1 && dout <= 8, "dss2_mlp2_bwd: sizes %d -> %d -> %d unsupported",
                 din, dmid, dout);
  DSS2_CHECK_ARG(partial_stride >= (int64_t)dmid * din + dmid + dout * dmid + dout, "dss2_mlp2_bwd: partial_stride too small");
  if (num_nodes == 0) return 0;
  MlpArgs a = {};
  a.n = num_nodes;
  a.x = x;
  a.din = din;
  a.w1 = w1;
  a.dmid = dmid;
  a.w2 = w2;
  a.dout = dout;
  a.gz = grad_z;
  a.gh = grad_h_ws;
  a.gx = grad_x;
  if (din == 8 && dmid == 32 && dout == 2) k_mlp2_bwd_fixed<8, 32, 2><<<grid_for(num_nodes, 128), 128, 0, stream>>>(a);
  else k_mlp2_bwd<<<grid_for(num_nodes, 128), 128, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  const int np = dss2_num_partials();
  const int64_t o_w1 = 0, o_b1 = (int64_t)dmid * din, o_w2 = o_b1 + dmid, o_b2 = o_w2 + (int64_t)dout * dmid;
  launch_outer_reduce(np, stream, num_nodes, grad_h_ws, dmid, dmid, x, din, din, partials, partial_stride, o_w1, o_b1);
  DSS2_LAUNCH_CHECK();
  launch_outer_reduce(np, stream, num_nodes, grad_z, dout, dout, h, dmid, dmid, partials, partial_stride, o_w2, o_b2);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_mlp2_nh_supported(int din, int dmid, int dout) { return din == 8 && dmid == 32 && dout == 2; }

// the same gradients without h / grad_h in memory (k_mlp2_bwd_nh); sizes: dss2_mlp2_nh_supported
extern "C" int dss2_mlp2_bwd_nh(int64_t num_nodes, const float* x, int din, const float* w1, const float* b1, int dmid, const float* w2, int dout,
                                const float* grad_z, float* grad_x, float* partials, int64_t partial_stride, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x && w1 && b1 && w2 && grad_z && grad_x && partials, "dss2_mlp2_bwd_nh: null argument");
  DSS2_CHECK_ARG(dss2_mlp2_nh_supported(din, dmid, dout), "dss2_mlp2_bwd_nh: sizes %d -> %d -> %d unsupported", din, dmid, dout);
  DSS2_CHECK_ARG(partial_stride >= (int64_t)dmid * din + dmid + dout * dmid + dout, "dss2_mlp2_bwd_nh: partial_stride too small");
  MlpArgs a = {};
  a.n = num_nodes;
  a.x = x;
  a.din = din;
  a.w1 = w1;
  a.b1 = b1;
  a.dmid = dmid;
  a.w2 = w2;
  a.dout = dout;
  a.gz = grad_z;
  a.gx = grad_x;
  k_mlp2_bwd_nh<8, 32, 2><<<dss2_num_partials(), MLP_NH_THREADS, 0, stream>>>(a, partials, partial_stride);   // idle CTAs write zeros
  DSS2_LAUNCH_CHECK();
  return 0;
}

// -------------------------------------------------------------------------------------------------
// gnn_dsse building blocks (networks.py:11-69), see the kernels above
// -------------------------------------------------------------------------------------------------
extern "C" int dss2_gcn_dinv(const dss2_graph_t* g, int self_loops, float* dinv, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(g && dinv, "dss2_gcn_dinv: null argument");
  DSS2_CHECK_ARG(g->undirected == 1, "dss2_gcn_dinv: needs a graph built from the one-way edge list with undirect=1");
  if (g->num_nodes == 0) return 0;
  k_gcn_dinv<<<grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(*g, self_loops, dinv);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_gcn_prop8(const dss2_graph_t* g, const float* dinv, int self_loops, int transposed, const float* x, int64_t x_stride,
                              float scale, const float* add, int64_t add_stride, float add_scale, float* out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(g && dinv && x && out, "dss2_gcn_prop8: null argument");
  DSS2_CHECK_ARG(x_stride >= GC && (!add || add_stride >= GC) && ((uintptr_t)out & 15) == 0, "dss2_gcn_prop8: rows must hold 8 floats, out 16-byte aligned");
  DSS2_CHECK_ARG(x != out, "dss2_gcn_prop8: in-place propagation is not possible");
  if (g->num_nodes == 0) return 0;
  GnnArgs a = {};
  a.g = *g;
  a.dinv = dinv;
  a.self_loops = self_loops;
  a.transposed = transposed;
  a.x = x;
  a.xs = x_stride;
  a.scale = scale;
  a.add = add;
  a.adds = add_stride;
  a.add_scale = add_scale;
  a.out = out;
  k_prop8<<<grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

static int lin8_fill(const char* who, Lin8Args& a, int64_t num_nodes, int M, int wt, const float* const* in, const int64_t* in_strides, const float* w,
                     const float* bias, int act, float slope) {
  DSS2_CHECK_ARG(M >= 1 && M <= 4 && in && in_strides && w, "%s: 1..4 input matrices", who);
  DSS2_CHECK_ARG(act >= 0 && act <= 3, "%s: act %d outside 0..3", who, act);
  a.num_nodes = num_nodes;
  a.M = M;
  a.wt = wt;
  for (int m = 0; m < M; ++m) {
    DSS2_CHECK_ARG(in[m] && in_strides[m] >= GC, "%s: input %d missing or narrower than 8", who, m);
    a.in[m] = in[m];
    a.ins[m] = in_strides[m];
  }
  a.w = w;
  a.bias = bias;
  a.act = act;
  a.slope = slope;
  return 0;
}

extern "C" int dss2_lin8_fwd(int64_t num_nodes, int M, int weight_is_out_by_in, const float* const* in, const int64_t* in_strides, const float* w,
                             const float* bias, int act, float slope, float* y, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  Lin8Args a = {};
  if (lin8_fill("dss2_lin8_fwd", a, num_nodes, M, weight_is_out_by_in, in, in_strides, w, bias, act, slope)) return -1;
  DSS2_CHECK_ARG(y && ((uintptr_t)y & 15) == 0, "dss2_lin8_fwd: y must be a 16-byte aligned [Nt, 8] buffer");
  if (num_nodes == 0) return 0;
  a.y = y;
  k_lin8_fwd<<<grid_for(num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

// grad_in[m] [Nt, 8] for every input, grad_z [Nt, 8]; weight gradients: per-CTA partial sums at partials + m * 64 (layout of `w`),
// bias gradient (sum of grad_z) at partials + bias_offset (pass scratch space when the layer has no bias).  acc (optional):
// acc += acc_scale * grad_in[0] (GCN2Conv's x_0 path).
extern "C" int dss2_lin8_bwd(int64_t num_nodes, int M, int weight_is_out_by_in, const float* const* in, const int64_t* in_strides, const float* w,
                             int act, float slope, const float* y, const float* grad_y, float* grad_z, float* const* grad_in, float* acc,
                             float acc_scale, float* partials, int64_t partial_stride, int64_t bias_offset, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  Lin8Args a = {};
  if (lin8_fill("dss2_lin8_bwd", a, num_nodes, M, weight_is_out_by_in, in, in_strides, w, nullptr, act, slope)) return -1;
  DSS2_CHECK_ARG(grad_y && grad_z && grad_in && partials && (!act || y), "dss2_lin8_bwd: null argument");
  if (num_nodes == 0) return 0;
  a.yout = y;
  a.gy = grad_y;
  a.gz = grad_z;
  for (int m = 0; m < M; ++m) {
    DSS2_CHECK_ARG(grad_in[m] && ((uintptr_t)grad_in[m] & 15) == 0, "dss2_lin8_bwd: grad_in[%d] missing or unaligned", m);
    a.gin[m] = grad_in[m];
  }
  a.acc = acc;
  a.acc_scale = acc_scale;
  k_lin8_bwd<<<grid_for(num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  const int np = dss2_num_partials();
  for (int m = 0; m < M; ++m) {
    // Linear weight [out c][in j]: sum_n gz[n][c] in[n][j];  GCN2Conv weight1 [in j][out c]: sum_n in[n][j] gz[n][c]
    if (weight_is_out_by_in)
      launch_outer_reduce(np, stream, num_nodes, grad_z, GC, GC, in[m], in_strides[m], GC, partials, partial_stride, (int64_t)m * GC * GC,
                                                    bias_offset);
    else
      launch_outer_reduce(np, stream, num_nodes, in[m], in_strides[m], GC, grad_z, GC, GC, partials, partial_stride, (int64_t)m * GC * GC,
                                                    bias_offset);
    DSS2_LAUNCH_CHECK();
  }
  return 0;
}

// -------------------------------------------------------------------------------------------------
// gnn_dsse(model='fagcn'): FAConv (networks.py:44-50; torch_geometric.nn.conv.FAConv) at width 8 on the one-way edge list:
//   out[i] = sum_{j -> i} tanh(att_l . x[j] + att_r . x[i]) * dinv[j] dinv[i] * x[j]  (+ the self loop, appended last)  + eps * x_0[i]
// followed by the model's non-linearity (fused here).  Thread per bus; the attention logits of the neighbours are recomputed from their
// rows (8 FMAs) instead of stored.  FAConv's own dropout acts on the attention coefficient tanh(.) (DROP kernels, edge keys as for GATv2).
// With self loops the input loops are skipped (add_remaining_self_loops), so their dropout keys are never read, as for GATv2.
// -------------------------------------------------------------------------------------------------
namespace {
struct FaArgs {
  dss2_graph_t g;
  const float* dinv;
  int self_loops;
  const float* x;        // [Nt, >= 8], row stride xs
  int64_t xs;
  const float* x0;       // [Nt, >= 8], row stride x0s
  int64_t x0s;
  const float *att_l, *att_r;   // [8] each
  float eps;
  int act;
  float slope;
  float* y;              // fwd: [Nt, 8]
  const float* yout;     // bwd: the forward's y
  const float* gy;       // bwd
  float* gx;             // bwd: [Nt, 8] adjoint of x
  float* acc;            // bwd, optional: acc[n] += eps * gz[n]  (the x_0 path)
  float* partials;       // bwd: per-CTA partial sums: [0, 8) att_l, [8, 16) att_r
  int64_t partial_stride;
  AttnDropArgs drop;     // read by the DROP = true kernels only
};
__device__ __forceinline__ void fa_row(const float* p, float (&v)[GC]) {
#pragma unroll
  for (int c = 0; c < GC; ++c) v[c] = p[c];
}
__device__ __forceinline__ float fa_dot(const float (&a)[GC], const float (&b)[GC]) {
  float d = 0.0f;
#pragma unroll
  for (int c = 0; c < GC; ++c) d = fmaf(a[c], b[c], d);
  return d;
}
__device__ __forceinline__ float fa_act_grad(int act, float slope, float y) {
  if (act == 1) return y > 0.0f ? 1.0f : slope;
  if (act == 2) return y > 0.0f ? 1.0f : 0.0f;
  if (act == 3) return 1.0f - y * y;
  return 1.0f;
}

template <bool DROP>
__global__ void __launch_bounds__(GAT_THREADS) k_fa_fwd(FaArgs a) {
  const dss2_graph_t& g = a.g;
  float wl[GC], wr[GC];
  fa_row(a.att_l, wl);
  fa_row(a.att_r, wr);
  AttnKey dk = {};
  if constexpr (DROP) dk = attn_key(a.drop);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < g.num_nodes; i += (int64_t)gridDim.x * blockDim.x) {
    const float di = a.dinv[i];
    float xi[GC], acc[GC];
    fa_row(a.x + i * a.xs, xi);
    const float ar = fa_dot(xi, wr);
#pragma unroll
    for (int c = 0; c < GC; ++c) acc[c] = 0.0f;
    for (int z = g.rowptr[i]; z < g.rowptr[i + 1]; ++z) {
      if (g.eid[z] >> 31) continue;           // out-edge of i
      const int64_t j = g.col[z];
      if (a.self_loops && j == i) continue;   // an input loop: replaced by the appended one
      float xj[GC];
      fa_row(a.x + j * a.xs, xj);
      float t = tanhf(fa_dot(xj, wl) + ar);
      if constexpr (DROP) t *= attn_factor(a.drop, dk, g.eid[z]);
      const float coef = t * (a.dinv[j] * di);
#pragma unroll
      for (int c = 0; c < GC; ++c) acc[c] = fmaf(coef, xj[c], acc[c]);
    }
    if (a.self_loops) {
      float t = tanhf(fa_dot(xi, wl) + ar);
      if constexpr (DROP) t *= attn_factor(a.drop, dk, (uint64_t)a.drop.num_edges + (uint64_t)i);
      const float coef = t * (di * di);
#pragma unroll
      for (int c = 0; c < GC; ++c) acc[c] = fmaf(coef, xi[c], acc[c]);
    }
    float o[GC];
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      float v = a.eps != 0.0f ? fmaf(a.eps, a.x0[i * a.x0s + c], acc[c]) : acc[c];
      if (a.act == 1) v = v > 0.0f ? v : v * a.slope;
      else if (a.act == 2) v = fmaxf(v, 0.0f);
      else if (a.act == 3) v = tanhf(v);
      o[c] = v;
    }
    float4* dst = reinterpret_cast<float4*>(a.y + i * GC);
    dst[0] = make_float4(o[0], o[1], o[2], o[3]);
    dst[1] = make_float4(o[4], o[5], o[6], o[7]);
  }
}

// adjoint: with gz = grad_y * act'(y) and, per edge j -> i, t = tanh(al[j] + ar[i]), c = dinv[j] dinv[i], q = (1 - t^2) c (gz[i] . x[j]):
//   grad_x[j] += t c gz[i] + q att_l,   grad_x[i] += q att_r,   grad_att_l += q x[j],   grad_att_r += q x[i].
// A thread owns bus n: its in-edges give the att_r terms, its out-edges (same CSR row, flagged) the att_l terms and the message adjoint.
// DROP: c includes the edge's dropout factor d (tc = t d c, q = (1 - t^2) c d (gz[i] . x[j])); the formulas above hold unchanged.
template <bool DROP>
__global__ void __launch_bounds__(GAT_THREADS) k_fa_bwd(FaArgs a) {
  const dss2_graph_t& g = a.g;
  __shared__ float red[GAT_THREADS / 32][2 * GC];
  float wl[GC], wr[GC], dwl[GC], dwr[GC];
  fa_row(a.att_l, wl);
  fa_row(a.att_r, wr);
  AttnKey dk = {};
  if constexpr (DROP) dk = attn_key(a.drop);
#pragma unroll
  for (int c = 0; c < GC; ++c) dwl[c] = dwr[c] = 0.0f;
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < g.num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    const float dn = a.dinv[n];
    float xn[GC], gzn[GC], gx[GC];
    fa_row(a.x + n * a.xs, xn);
#pragma unroll
    for (int c = 0; c < GC; ++c) {
      gzn[c] = a.gy[n * GC + c] * fa_act_grad(a.act, a.slope, a.yout ? a.yout[n * GC + c] : 0.0f);
      gx[c] = 0.0f;
    }
    if (a.acc) {
#pragma unroll
      for (int c = 0; c < GC; ++c) a.acc[n * GC + c] += a.eps * gzn[c];
    }
    const float al_n = fa_dot(xn, wl), ar_n = fa_dot(xn, wr);
    float q_l = 0.0f, q_r = 0.0f;   // sums of q over the out-edges (n is the source) and the in-edges (n is the target)
    for (int z = g.rowptr[n]; z < g.rowptr[n + 1]; ++z) {
      const int64_t m = g.col[z];
      if (a.self_loops && m == n) continue;   // an input loop (its in- and its out-entry): replaced by the appended one
      float xm[GC];
      fa_row(a.x + m * a.xs, xm);
      float c = a.dinv[m] * dn;
      if constexpr (DROP) c *= attn_factor(a.drop, dk, g.eid[z] & 0x7fffffffu);
      if (g.eid[z] >> 31) {   // n -> m
        float gzm[GC];
#pragma unroll
        for (int k = 0; k < GC; ++k) gzm[k] = a.gy[m * GC + k] * fa_act_grad(a.act, a.slope, a.yout ? a.yout[m * GC + k] : 0.0f);
        const float t = tanhf(al_n + fa_dot(xm, wr));
        const float tc = t * c;
#pragma unroll
        for (int k = 0; k < GC; ++k) gx[k] = fmaf(tc, gzm[k], gx[k]);
        q_l += (1.0f - t * t) * c * fa_dot(gzm, xn);
      } else {                // m -> n
        const float t = tanhf(fa_dot(xm, wl) + ar_n);
        q_r += (1.0f - t * t) * c * fa_dot(gzn, xm);
      }
    }
    if (a.self_loops) {
      const float t = tanhf(al_n + ar_n);
      float c = dn * dn;
      if constexpr (DROP) c *= attn_factor(a.drop, dk, (uint64_t)a.drop.num_edges + (uint64_t)n);
      const float tc = t * c, q = (1.0f - t * t) * c * fa_dot(gzn, xn);
#pragma unroll
      for (int k = 0; k < GC; ++k) gx[k] = fmaf(tc, gzn[k], gx[k]);
      q_l += q;
      q_r += q;
    }
#pragma unroll
    for (int k = 0; k < GC; ++k) {
      gx[k] = fmaf(q_l, wl[k], fmaf(q_r, wr[k], gx[k]));
      dwl[k] = fmaf(q_l, xn[k], dwl[k]);
      dwr[k] = fmaf(q_r, xn[k], dwr[k]);
    }
    float4* dst = reinterpret_cast<float4*>(a.gx + n * GC);
    dst[0] = make_float4(gx[0], gx[1], gx[2], gx[3]);
    dst[1] = make_float4(gx[4], gx[5], gx[6], gx[7]);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < GC; ++k) {
    const float v1 = warp_sum(dwl[k]), v2 = warp_sum(dwr[k]);
    if (lane == 0) {
      red[warp][k] = v1;
      red[warp][GC + k] = v2;
    }
  }
  __syncthreads();
  if (threadIdx.x < 2 * GC) {
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < GAT_THREADS / 32; ++w) s += red[w][threadIdx.x];
    a.partials[(size_t)blockIdx.x * a.partial_stride + threadIdx.x] = s;
  }
}

int fa_fill(const char* who, FaArgs& a, const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t xs, const float* x0,
            int64_t x0s, const float* att_l, const float* att_r, float eps, int act, float slope) {
  DSS2_CHECK_ARG(g && dinv && x && att_l && att_r && (eps == 0.0f || x0), "%s: null argument", who);
  DSS2_CHECK_ARG(xs >= GC && (eps == 0.0f || x0s >= GC), "%s: row strides below %d", who, GC);
  DSS2_CHECK_ARG(act >= 0 && act <= 3, "%s: act %d outside 0..3", who, act);
  a.g = *g;
  a.dinv = dinv;
  a.self_loops = self_loops;
  a.x = x;
  a.xs = xs;
  a.x0 = x0;
  a.x0s = x0s;
  a.att_l = att_l;
  a.att_r = att_r;
  a.eps = eps;
  a.act = act;
  a.slope = slope;
  return 0;
}
}  // namespace

extern "C" int dss2_fa_fwd_drop(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* x0,
                                int64_t x0_stride, const float* att_l, const float* att_r, float eps, int act, float slope,
                                const dss2_attn_drop_t* drop, float* y, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FaArgs a = {};
  if (fa_fill("dss2_fa_fwd", a, g, dinv, self_loops, x, x_stride, x0, x0_stride, att_l, att_r, eps, act, slope)) return -1;
  if (fill_drop("dss2_fa_fwd", a.drop, drop, g->num_edges)) return -1;
  DSS2_CHECK_ARG(y && ((uintptr_t)y & 15) == 0, "dss2_fa_fwd: y missing or unaligned");
  if (g->num_nodes == 0) return 0;
  a.y = y;
  if (a.drop.mode) k_fa_fwd<true><<<grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  else k_fa_fwd<false><<<grid_for(g->num_nodes, GAT_THREADS), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_fa_fwd(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* x0,
                           int64_t x0_stride, const float* att_l, const float* att_r, float eps, int act, float slope, float* y,
                           void* stream_) {
  return dss2_fa_fwd_drop(g, dinv, self_loops, x, x_stride, x0, x0_stride, att_l, att_r, eps, act, slope, nullptr, y, stream_);
}

extern "C" int dss2_fa_bwd_drop(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* att_l,
                                const float* att_r, float eps, int act, float slope, const dss2_attn_drop_t* drop, const float* y,
                                const float* grad_y, float* grad_x, float* acc_x0, float* partials, int64_t partial_stride, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  FaArgs a = {};
  if (fa_fill("dss2_fa_bwd", a, g, dinv, self_loops, x, x_stride, x, x_stride, att_l, att_r, eps, act, slope)) return -1;
  if (fill_drop("dss2_fa_bwd", a.drop, drop, g->num_edges)) return -1;
  DSS2_CHECK_ARG(grad_y && grad_x && partials && (!act || y) && ((uintptr_t)grad_x & 15) == 0, "dss2_fa_bwd: null or unaligned argument");
  a.yout = y;
  a.gy = grad_y;
  a.gx = grad_x;
  a.acc = acc_x0;
  a.partials = partials;
  a.partial_stride = partial_stride;
  // every partial row is written (idle CTAs write zeros)
  if (a.drop.mode) k_fa_bwd<true><<<dss2_num_partials(), GAT_THREADS, 0, stream>>>(a);
  else k_fa_bwd<false><<<dss2_num_partials(), GAT_THREADS, 0, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_fa_bwd(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* att_l,
                           const float* att_r, float eps, int act, float slope, const float* y, const float* grad_y, float* grad_x,
                           float* acc_x0, float* partials, int64_t partial_stride, void* stream_) {
  return dss2_fa_bwd_drop(g, dinv, self_loops, x, x_stride, att_l, att_r, eps, act, slope, nullptr, y, grad_y, grad_x, acc_x0, partials,
                          partial_stride, stream_);
}
