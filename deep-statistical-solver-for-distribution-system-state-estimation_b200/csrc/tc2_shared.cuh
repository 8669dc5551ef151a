// Pieces shared by the tcgen05 TAG-layer kernels (tag_tc2.cu: k_tag_tc2, k_tag_gw; tag_tc3.cu: k_tag_tc3).
#pragma once
#include "common.cuh"
#include "tc.cuh"

// kernel arguments of the layer kernels (global type: it crosses translation units)
struct Tc2Args {
  dss2_graph_t g;
  const float* in;          // FWD: x [Nt,32].  BGX: grad_y [Nt,cout]
  const uint32_t* in_bits;  // BGX: sign words of the forward output (NULL when the layer had no activation)
  const float* w;           // [K+1][cout][32]
  const float* bias;        // FWD
  int cout;
  int act;                  // FWD: apply dropout + ReLU
  float scale;              // 1/(1-p)
  uint32_t keep_thr16;
  int drop_mode;
  const uint64_t* rng;
  uint32_t layer_uid;
  const uint8_t* mask;
  const float* res;
  int64_t res_stride;
  float* out;               // FWD: y [Nt,cout].  BGX: grad_x [Nt,32]
  uint32_t* out_bits;       // FWD
  float* lvl_out;           // BGX: [K][Nt,32] hop levels 1..K of g (for k_tag_gw)
  const float* dense_lvl;   // large-graph path: hop levels 1..K precomputed in global memory ([K][Nt,32]); tiles are plain row chunks
  int flags;                // measurement switches (DSS2_TC2_FLAGS): 1 = BGX prefetches the next tile behind the last publish like FWD
  // Layer chaining (k_tag_tc3 only): a tile of layer l+1 needs nothing but the SAME tile of layer l (message passing never leaves a tile),
  // so consecutive layer launches are linked per tile instead of per grid.  done_flags[t] is set to the chain sequence number (device
  // step counter + 1) once tile t's outputs are in global memory; a launch given wait_flags reads tile t's input only after the
  // producer's flag carries this step's number, and is launched with programmatic stream serialization WITHOUT a grid-wide wait: its
  // CTAs start on the SMs the producer's CTAs leave and run ahead (no empty last round, prologue hidden behind the producer's tail).
  uint32_t* done_flags;
  const uint32_t* wait_flags;
  const uint64_t* chain_seq;   // device {seed, step}: sequence number = (uint32)step + 1
};

namespace {

constexpr int T2_MAX = 256;                      // rows per tile (2 MMA blocks of 128)
constexpr uint32_t W_TILE = 32 * tc::ROW_BYTES;  // 4 KB
enum { MODE_FWD = 0, MODE_BGX = 1 };


__device__ __forceinline__ char* align1024(char* p) {
  const uint32_t a = smem_u32(p);
  return p + (((a + 1023u) & ~1023u) - a);
}

// Thread mapping of the layer kernel: 256 threads per tile, thread = (row, half): row = tid & 127 (= its TMEM lane), half = tid >> 7
// owns features [16*half, 16*half + 16).  Two threads per row double the number of busy warps on grids whose tile holds a single
// graph (Oberrhein: 70 of 128 rows) and halve every per-thread dependency chain.
// NB = MMA blocks (128 rows each) per tile: NB = 2 packs e.g. 3 Oberrhein graphs (210 rows) or 17 CIGRE graphs (255 rows) into one
// tile, so that more live rows share one pass through the per-tile dependency chain; workers = 256 per block + 1 issuer warp.
constexpr int HF = 16;

__device__ __forceinline__ void store_half_sw128(const float (&v)[HF], char* pt, char* lt, uint32_t row, uint32_t half) {
  const uint32_t code = tc::row_code(row);
#pragma unroll
  for (uint32_t q = 0; q < 4; ++q)
    tc::plain_store4(make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]), pt, lt, code ^ ((half * 4 + q) << 4));
}

// h += w * plain[src row][16*half ...]: one neighbour, exact fp32 values from the plain tile, whose 16-byte chunk c of row `src` sits at
// chunk c ^ key (key = src & 7 in the hardware-swizzled tiles of k_tag_tc2, the row's swizzle key in the plain tiles of k_tag_tc3)
__device__ __forceinline__ uint32_t row_code_key(uint32_t row, uint32_t key) { return (row << 7) | (key << 4); }
__device__ __forceinline__ void gather_half(float (&h)[HF], const char* pt, uint32_t src, uint32_t key, float w, uint32_t half) {
  const uint32_t code = row_code_key(src, key);
#pragma unroll
  for (uint32_t q = 0; q < 4; ++q) {
    const float4 a = *reinterpret_cast<const float4*>(pt + (code ^ ((half * 4 + q) << 4)));
    h[4 * q + 0] = fmaf(w, a.x, h[4 * q + 0]);
    h[4 * q + 1] = fmaf(w, a.y, h[4 * q + 1]);
    h[4 * q + 2] = fmaf(w, a.z, h[4 * q + 2]);
    h[4 * q + 3] = fmaf(w, a.w, h[4 * q + 3]);
  }
}

struct RowTopo {
  float4 w;        // weights of the first 4 entries
  uint32_t cols;   // 4 x 8-bit tile-local sources
  uint32_t deg;    // degree (saturated at DSS2_ELL_DEG_MASK: hub rows take their extent from rowptr)
  uint32_t keys;   // swizzle keys: bits 0..2 the row's own, 3 + 3d..5 + 3d those of ELL source d
};
__device__ __forceinline__ RowTopo row_topo(float4 w, uint2 ci) {
  RowTopo t;
  t.w = w;
  t.cols = ci.x;
  t.deg = ci.y & DSS2_ELL_DEG_MASK;
  t.keys = ci.y >> DSS2_ELL_KEY_SHIFT;
  return t;
}
__device__ __forceinline__ RowTopo load_row_topo(const dss2_graph_t& g, size_t n) {
  return row_topo(reinterpret_cast<const float4*>(g.ell_w)[n], reinterpret_cast<const uint2*>(g.ell_ci)[n]);
}

// one hop for this thread's half row: entries in CSR order = PyG scatter order.  BUS_KEYS: the plain tile is swizzled by the graph's
// per-row keys (k_tag_tc3), else by the tile row (k_tag_tc2's hardware swizzle)
template <bool BUS_KEYS>
__device__ __forceinline__ void hop_thread(float (&h)[HF], const dss2_graph_t& g, const RowTopo& tp, const char* pt, size_t n, int n0,
                                           uint32_t half) {
#pragma unroll
  for (int i = 0; i < HF; ++i) h[i] = 0.0f;
  const float wv[4] = {tp.w.x, tp.w.y, tp.w.z, tp.w.w};
#pragma unroll
  for (uint32_t d = 0; d < 4; ++d) {
    const uint32_t src = (tp.cols >> (8 * d)) & 0xffu;
    if (d < tp.deg) gather_half(h, pt, src, BUS_KEYS ? (tp.keys >> (3 + 3 * d)) & 7u : src & 7u, wv[d], half);
  }
  if (tp.deg > 4) {   // rare: hub nodes
    const int beg = g.rowptr[n], end = g.rowptr[n + 1];
    for (int z = beg + 4; z < end; ++z) {
      const int c = g.col[z];
      gather_half(h, pt, (uint32_t)(c - n0), BUS_KEYS ? (uint32_t)g.hop_key[c] : (uint32_t)(c - n0) & 7u, g.w[z], half);
    }
  }
}

// 16 Bernoulli(keep) decisions: features [16*half, 16*half+16) of one node row
__device__ __forceinline__ uint32_t keep_half(uint2 key, uint32_t tile, uint32_t row, uint32_t half, uint32_t step_lo, uint32_t thr16) {
  uint32_t word = 0;
#pragma unroll
  for (uint32_t q = 0; q < 2; ++q) {
    const uint4 r = philox4x32_10(make_uint4(tile, row, half * 2 + q, step_lo), key);
    const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (uint32_t i = 0; i < 4; ++i) {
      word |= ((u[i] & 0xffffu) < thr16 ? 1u : 0u) << (q * 8 + 2 * i);
      word |= ((u[i] >> 16) < thr16 ? 1u : 0u) << (q * 8 + 2 * i + 1);
    }
  }
  return word;
}

struct TileNodes {
  int n0, n1;
};
__device__ __forceinline__ TileNodes tile_nodes(const dss2_graph_t& g, int t, int dense_rows = 0) {
  TileNodes r;
  r.n0 = r.n1 = 0;
  if (dense_rows) {   // hop-free mode: tile t = rows [t * dense_rows, (t + 1) * dense_rows)
    const int64_t n0 = (int64_t)t * dense_rows;
    if (n0 < g.num_nodes) {
      r.n0 = (int)n0;
      r.n1 = (int)min(g.num_nodes, n0 + dense_rows);
    }
    return r;
  }
  if (t < g.num_tiles) {
    const int g0 = t * g.graphs_per_tile, g1 = min(g0 + g.graphs_per_tile, g.num_graphs);
    r.n0 = (int)g.ptr[g0];
    r.n1 = (int)g.ptr[g1];
  }
  return r;
}

// RW = warps per half tile (32 rows each): 8 -> 256-row tiles (two MMA blocks), one 17-warp CTA per SM; 4 -> 128-row tiles, two 9-warp
// CTAs per SM; 3 -> 96-row tiles, THREE 7-warp CTAs per SM.  The RW = 3 shape exists for grids whose graphs fill little more than
// half of a 128-row block (Oberrhein: 70 buses): a CTA is a per-tile dependency chain (store -> fence -> barrier -> gather -> ... ->
// MMA -> TMEM -> epilogue), so what fills the SM's issue slots is the number of INDEPENDENT chains in flight, not the rows per
// chain; three one-graph CTAs keep as many rows in flight as one three-graph CTA and never meet at a barrier.  Warp w may read TMEM
// lanes [32 (w % 4), +32) only, so the half-0 workers are warps 0..2, the half-1 workers warps 4..6 and warp 3 - which has no rows -
// is the MMA issuer.  The MMAs stay M = 128: rows 96..127 of the A operand alias the next shared-memory buffer (any bits will do,
// row m of D depends on row m of A only and those accumulator lanes are never read).
template <int RW>
struct Tc2Shape {
  static constexpr int NB = (RW + 3) / 4;
  static constexpr int ROWS = 32 * RW;
  static constexpr int WORKERS = 64 * RW;
  static constexpr int ISSUER_WARP = RW == 3 ? 3 : 2 * RW;
  static constexpr int THREADS = RW == 3 ? 224 : 64 * RW + 32;
  static constexpr int CTAS_PER_SM = RW == 3 ? 3 : (RW == 4 ? 2 : 1);
};

}  // namespace

// tag_tc3.cu: the TMA-fed variant of the layer kernel (returns < 0 on error, 1 when the shape is not served and the caller should use
// k_tag_tc2, 0 when launched)
int dss2_tc3_launch(int mode, const Tc2Args& a, int K, cudaStream_t stream);
