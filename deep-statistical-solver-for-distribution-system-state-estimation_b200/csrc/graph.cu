#include <cstdlib>
// Library runtime (errors, launch counter) + batch structure kernels:
//   dss2_graph_build  - doubled-graph CSR by destination, gcn degree norm, tiling   (networks.py:236-258, PyG gcn_norm)
//   dss2_pack_batch   - PyG Batch.from_data_list as a gather kernel                   (dss2_run.py:68-69,134)
//   dss2_col_minmax   - batch-global V_hv / V_lv                                      (data.py:334-336)
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <cub/cub.cuh>

#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// runtime
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void dss2_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void dss2_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int dss2_sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  }
  return sms;
}
int dss2_launch_priority(int level) {
  static const int max_level = [] {
    const char* e = getenv("DSS2_CHAIN_PRIO");
    return e ? atoi(e) : 1;
  }();
  static const int greatest = [] {
    int least = 0, g = 0;
    return cudaDeviceGetStreamPriorityRange(&least, &g) == cudaSuccess ? g : 0;
  }();
  return level <= max_level ? greatest : 0;
}
extern "C" const char* dss2_last_error(void) { return g_err; }
extern "C" int dss2_version(void) { return 100; }
extern "C" int64_t dss2_launch_count(void) { return g_launches.load(); }

// ---------------------------------------------------------------------------------------------
// graph build
// ---------------------------------------------------------------------------------------------
namespace {

enum { ST_REVERSE_FOUND = 0, ST_BAD_INDEX, ST_NOT_TILEABLE, ST_MAX_SEG_NODES, ST_MAX_TILE_NODES, ST_MAX_TILE_NNZ, ST_MAX_TILE_EDGES, ST_COUNT = 16 };

__global__ void k_detect_reverse(const int64_t* __restrict__ ei, int64_t Et, int* stats) {
  // networks.py:236-238: graph counts as undirected iff some edge (t0 -> s0) exists, (s0 -> t0) being edge 0
  int64_t s0 = ei[0], t0 = ei[Et];
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < Et; e += (int64_t)gridDim.x * blockDim.x)
    if (ei[e] == t0 && ei[Et + e] == s0) atomicOr(&stats[ST_REVERSE_FOUND], 1);
}

__device__ __forceinline__ void doubled_edge(const int64_t* ei, int64_t Et, int64_t q, int64_t& src, int64_t& dst) {
  if (q < Et) {
    src = ei[q];
    dst = ei[Et + q];
  } else {
    src = ei[Et + (q - Et)];
    dst = ei[q - Et];
  }
}

__global__ void k_count(const int64_t* __restrict__ ei, int64_t Et, int64_t nnz, int64_t Nt, int* cnt, int* stats) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
    int64_t s, d;
    doubled_edge(ei, Et, q, s, d);
    if (s < 0 || s >= Nt || d < 0 || d >= Nt) {
      atomicOr(&stats[ST_BAD_INDEX], 1);
      continue;
    }
    atomicAdd(&cnt[d], 1);
  }
}

__global__ void k_fill(const int64_t* __restrict__ ei, int64_t Et, int64_t nnz, int64_t Nt, const int* __restrict__ rowptr,
                       int* cursor, int* col, uint32_t* eid) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
    int64_t s, d;
    doubled_edge(ei, Et, q, s, d);
    if (s < 0 || s >= Nt || d < 0 || d >= Nt) continue;
    int pos = rowptr[d] + atomicAdd(&cursor[d], 1);
    col[pos] = (int)s;
    eid[pos] = q < Et ? (uint32_t)q : ((uint32_t)(q - Et) | 0x80000000u);
  }
}

// Order every row by doubled edge id (= PyG scatter order) and write the degree norm.
__global__ void k_sort_rows(int64_t Nt, const int* __restrict__ rowptr, int* col, uint32_t* eid, float* dis) {
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < Nt; n += (int64_t)gridDim.x * blockDim.x) {
    int b = rowptr[n], e = rowptr[n + 1];
    for (int i = b + 1; i < e; ++i) {
      uint32_t key = eid[i];
      int c = col[i];
      int j = i - 1;
      while (j >= b && eid[j] > key) {
        eid[j + 1] = eid[j];
        col[j + 1] = col[j];
        --j;
      }
      eid[j + 1] = key;
      col[j + 1] = c;
    }
    int deg = e - b;
    dis[n] = deg > 0 ? 1.0f / sqrtf((float)deg) : 0.0f;   // deg.pow(-0.5), inf -> 0
  }
}

// gcn_norm edge weight per CSR entry: dis[src] * 1 * dis[dst]
__global__ void k_entry_weights(int64_t Nt, const int* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ dis, float* w) {
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < Nt; n += (int64_t)gridDim.x * blockDim.x) {
    const float dn = dis[n];
    for (int z = rowptr[n]; z < rowptr[n + 1]; ++z) w[z] = dis[col[z]] * dn;
  }
}

__device__ __forceinline__ int graph_of(const int64_t* ptr, int B, int64_t node) {
  int lo = 0, hi = B;  // largest g with ptr[g] <= node
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (ptr[mid] <= node) lo = mid; else hi = mid;
  }
  return lo;
}

// eptr[g] = first one-way edge whose source lies in graph >= g (edges are graph-major in a PyG batch)
__global__ void k_eptr(const int64_t* __restrict__ ei, int64_t Et, const int64_t* __restrict__ ptr, int B, int64_t* eptr, int* stats) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g > B) return;
  if (g == B) { eptr[B] = Et; return; }
  int64_t lo = 0, hi = Et, key = ptr[g];
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (ei[mid] < key) lo = mid + 1; else hi = mid;
  }
  eptr[g] = lo;
  atomicMax(&stats[ST_MAX_SEG_NODES], (int)min((int64_t)INT_MAX, ptr[g + 1] - ptr[g]));
}

// every edge must stay inside one graph and graphs must appear in order
__global__ void k_check_edges(const int64_t* __restrict__ ei, int64_t Et, const int64_t* __restrict__ ptr, int B, int* stats) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < Et; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t s = ei[e], d = ei[Et + e];
    int gs = graph_of(ptr, B, s);
    bool ok = d >= ptr[gs] && d < ptr[gs + 1];
    if (e + 1 < Et) ok = ok && (ei[e + 1] >= ptr[gs]);
    if (!ok) atomicOr(&stats[ST_NOT_TILEABLE], 1);
  }
}

// ELL view of the first 4 entries of every row, with sources numbered relative to the row's tile (thread-per-row kernels)
__global__ void k_build_ell(dss2_graph_t g) {
  int t = blockIdx.x;
  if (t >= g.num_tiles) return;
  TileRange r = tile_range(g, t);
  for (int n = r.n0 + threadIdx.x; n < r.n1; n += blockDim.x) {
    const int beg = g.rowptr[n], deg = g.rowptr[n + 1] - beg;
    uint32_t cols = 0;
    float w[4] = {0.f, 0.f, 0.f, 0.f};
    for (int d = 0; d < 4; ++d) {
      int local = n - r.n0;          // padding points at the row itself with weight 0
      if (d < deg) {
        local = g.col[beg + d] - r.n0;
        w[d] = g.w[beg + d];
      }
      cols |= (uint32_t)(local & 0xff) << (8 * d);
    }
    reinterpret_cast<float4*>(g.ell_w)[n] = make_float4(w[0], w[1], w[2], w[3]);
    reinterpret_cast<uint2*>(g.ell_ci)[n] = make_uint2(cols, (uint32_t)min(deg, (int)DSS2_ELL_DEG_MASK));
  }
}

// Swizzle keys of one tile's rows (see DSS2_HOP_KEYS_COLOR in dss2_b200.h).  ci = the tile's ELL words before key packing, key = out.
// The 8 lanes of one LDS.128 / STS.128 phase of the layer kernels are 8 consecutive tile rows (group G = rows 8j..8j+7), each
// reading or writing 16 bytes of one row of the plain level tile; two of them hit the same banks iff their rows differ and have the
// same key.  Costs, per pair of distinct rows with equal keys:
//   (a) 4 for the slot-d sources of two rows of one group (gathered together: up to 4 slots x 4 loads per thread and hop),
//   (b) 1 for two rows of one group (stored together: 4 stores per thread and level).
// Greedy colouring in row order, then two sweeps that move each row to its cheapest key (more sweeps change nothing on the grids
// in the repository); ties keep the identity key (n0 + r) & 7.  Deterministic: integer costs, fixed order.
__host__ __device__ void hop_keys_tile(const uint2* ci, int nT, int n0, int policy, uint8_t* key) {
  constexpr int WA = 4, WB = 1, NO_KEY = 0xff;
  if (policy != DSS2_HOP_KEYS_COLOR) {
    for (int r = 0; r < nT; ++r) key[r] = (uint8_t)((n0 + r) & 7);
    return;
  }
  uint16_t start[DSS2_TILE_CAP + 1], occ[4 * DSS2_TILE_CAP];   // (row, slot) pairs grouped by source row
  for (int v = 0; v <= nT; ++v) start[v] = 0;
  auto active = [&](int r) { return (int)min(ci[r].y & DSS2_ELL_DEG_MASK, 4u); };
  auto src = [&](int r, int d) { return (int)((ci[r].x >> (8 * d)) & 0xffu); };
  for (int r = 0; r < nT; ++r)
    for (int d = 0; d < active(r); ++d) ++start[src(r, d) + 1];
  for (int v = 0; v < nT; ++v) start[v + 1] += start[v];
  {
    uint16_t fill[DSS2_TILE_CAP];
    for (int v = 0; v < nT; ++v) fill[v] = start[v];
    for (int r = 0; r < nT; ++r)
      for (int d = 0; d < active(r); ++d) occ[fill[src(r, d)]++] = (uint16_t)(4 * r + d);
  }
  for (int r = 0; r < nT; ++r) key[r] = NO_KEY;
  for (int pass = 0; pass < 3; ++pass) {
    for (int v = 0; v < nT; ++v) {
      int cost[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      const int g0 = v & ~7, g1 = min(g0 + 8, nT);
      for (int u = g0; u < g1; ++u)
        if (u != v && key[u] != NO_KEY) cost[key[u]] += WB;
      for (int o = start[v]; o < start[v + 1]; ++o) {
        const int r = occ[o] >> 2, d = occ[o] & 3, h0 = r & ~7, h1 = min(h0 + 8, nT);
        for (int q = h0; q < h1; ++q) {
          if (q == r || d >= active(q)) continue;
          const int s = src(q, d);
          if (s != v && key[s] != NO_KEY) cost[key[s]] += WA;
        }
      }
      int best = key[v] != NO_KEY ? key[v] : (n0 + v) & 7;   // ties keep the current (first pass: identity) key
      for (int k = 0; k < 8; ++k)
        if (cost[k] < cost[best]) best = k;
      key[v] = (uint8_t)best;
    }
  }
}

// one thread per tile: keys -> hop_key[] and the upper bits of the tile's ELL degree words
__global__ void k_hop_keys(dss2_graph_t g, int policy) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.num_tiles) return;
  const TileRange r = tile_range(g, t);
  const int nT = r.n1 - r.n0;
  uint2* ci = reinterpret_cast<uint2*>(g.ell_ci) + r.n0;
  uint8_t* key = g.hop_key + r.n0;
  hop_keys_tile(ci, nT, r.n0, policy, key);
  for (int i = 0; i < nT; ++i) {
    const uint2 c = ci[i];
    uint32_t word = (c.y & DSS2_ELL_DEG_MASK) | ((uint32_t)key[i] << DSS2_ELL_KEY_SHIFT);
    const int act = (int)min(c.y & DSS2_ELL_DEG_MASK, 4u);
    for (int d = 0; d < act; ++d) word |= (uint32_t)key[(c.x >> (8 * d)) & 0xffu] << (DSS2_ELL_KEY_SHIFT + 3 + 3 * d);
    ci[i].y = word;
  }
}

__global__ void k_tile_stats(dss2_graph_t g, int* stats) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.num_tiles) return;
  TileRange r = tile_range(g, t);
  atomicMax(&stats[ST_MAX_TILE_NODES], r.n1 - r.n0);
  atomicMax(&stats[ST_MAX_TILE_NNZ], r.z1 - r.z0);
  atomicMax(&stats[ST_MAX_TILE_EDGES], (int)(r.e1 - r.e0));
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WsLayout {
  size_t rowptr, col, eid, dis, w, ell_w, ell_ci, hop_key, eptr, cursor, stats, cub, total, cub_bytes;
};
WsLayout ws_layout(int64_t Nt, int64_t Et, int32_t B) {
  WsLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  L.rowptr = take((size_t)(Nt + 1) * 4);
  L.col = take((size_t)(2 * Et + 1) * 4);
  L.eid = take((size_t)(2 * Et + 1) * 4);
  L.dis = take((size_t)(Nt + 1) * 4);
  L.w = take((size_t)(2 * Et + 1) * 4);
  L.ell_w = take((size_t)(Nt + 1) * 16);
  L.ell_ci = take((size_t)(Nt + 1) * 8);
  L.hop_key = take((size_t)(Nt + 1));
  L.eptr = take((size_t)(B + 1) * 8);
  L.cursor = take((size_t)(Nt + 1) * 4);
  L.stats = take(ST_COUNT * 4);
  size_t cub_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (int*)nullptr, (int*)nullptr, (int)(Nt + 1));
  L.cub_bytes = cub_bytes + 256;
  L.cub = take(L.cub_bytes);
  L.total = off;
  return L;
}
inline int grid_for(int64_t n, int threads) { return (int)max((int64_t)1, min((int64_t)148 * 16, (n + threads - 1) / threads)); }

}  // namespace

extern "C" size_t dss2_generic_scratch_bytes(int64_t Nt) { return ((size_t)4 * Nt * HID + 16384) * sizeof(float); }

extern "C" size_t dss2_graph_workspace_bytes(int64_t Nt, int64_t Et, int32_t B) { return ws_layout(Nt, Et, B).total; }

extern "C" int dss2_graph_build(dss2_graph_t* g, const int64_t* edge_index, int64_t Et, int64_t Nt, const int64_t* ptr,
                                int32_t B, int undirect, int tile_cap, int hop_keys, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(g && ws && ptr && (edge_index || Et == 0), "dss2_graph_build: null argument");
  DSS2_CHECK_ARG(Nt >= 0 && Et >= 0 && B >= 1, "dss2_graph_build: bad sizes Nt=%lld Et=%lld B=%d", (long long)Nt, (long long)Et, B);
  DSS2_CHECK_ARG(Nt < (1LL << 31) - 2 && 2 * Et < (1LL << 31) - 2, "dss2_graph_build: batch too large for the int32 CSR");
  DSS2_CHECK_ARG(tile_cap >= 1 && tile_cap <= DSS2_TILE_CAP, "dss2_graph_build: tile_cap %d outside 1..%d", tile_cap, DSS2_TILE_CAP);
  DSS2_CHECK_ARG(hop_keys == DSS2_HOP_KEYS_IDENTITY || hop_keys == DSS2_HOP_KEYS_COLOR, "dss2_graph_build: hop_keys %d is not a policy", hop_keys);
  WsLayout L = ws_layout(Nt, Et, B);
  DSS2_CHECK_ARG(ws_bytes >= L.total, "dss2_graph_build: workspace %zu < %zu bytes", ws_bytes, L.total);
  char* base = (char*)ws;
  memset(g, 0, sizeof(*g));
  g->num_nodes = Nt;
  g->num_edges = Et;
  g->num_graphs = B;
  g->edge_index = edge_index;
  g->ptr = ptr;
  g->rowptr = (int32_t*)(base + L.rowptr);
  g->col = (int32_t*)(base + L.col);
  g->eid = (uint32_t*)(base + L.eid);
  g->dis = (float*)(base + L.dis);
  g->w = (float*)(base + L.w);
  g->ell_w = (float*)(base + L.ell_w);
  g->ell_ci = (uint32_t*)(base + L.ell_ci);
  g->hop_key = (uint8_t*)(base + L.hop_key);
  g->hop_keys = hop_keys;
  g->eptr = (int64_t*)(base + L.eptr);
  int* cursor = (int*)(base + L.cursor);
  int* stats = (int*)(base + L.stats);
  int h_stats[ST_COUNT];
  const int T = 256;

  DSS2_CUDA(cudaMemsetAsync(stats, 0, ST_COUNT * 4, stream));
  if (undirect < 0) {
    if (Et > 0) {
      k_detect_reverse<<<grid_for(Et, T), T, 0, stream>>>(edge_index, Et, stats);
      DSS2_LAUNCH_CHECK();
      DSS2_CUDA(cudaMemcpyAsync(h_stats, stats, 4, cudaMemcpyDeviceToHost, stream));
      DSS2_CUDA(cudaStreamSynchronize(stream));
      undirect = h_stats[ST_REVERSE_FOUND] ? 0 : 1;
    } else {
      undirect = 1;
    }
  }
  g->undirected = undirect ? 1 : 0;
  int64_t nnz = undirect ? 2 * Et : Et;
  g->nnz = nnz;

  DSS2_CUDA(cudaMemsetAsync(cursor, 0, (size_t)(Nt + 1) * 4, stream));
  if (nnz > 0) {
    k_count<<<grid_for(nnz, T), T, 0, stream>>>(edge_index, Et, nnz, Nt, cursor, stats);
    DSS2_LAUNCH_CHECK();
  }
  size_t cub_bytes = L.cub_bytes;
  DSS2_CUDA(cub::DeviceScan::ExclusiveSum(base + L.cub, cub_bytes, cursor, g->rowptr, (int)(Nt + 1), stream));
  dss2_count_launch(2);
  DSS2_CUDA(cudaMemsetAsync(cursor, 0, (size_t)(Nt + 1) * 4, stream));
  if (nnz > 0) {
    k_fill<<<grid_for(nnz, T), T, 0, stream>>>(edge_index, Et, nnz, Nt, g->rowptr, cursor, g->col, g->eid);
    DSS2_LAUNCH_CHECK();
  }
  if (Nt > 0) {
    k_sort_rows<<<grid_for(Nt, T), T, 0, stream>>>(Nt, g->rowptr, g->col, g->eid, g->dis);
    DSS2_LAUNCH_CHECK();
    k_entry_weights<<<grid_for(Nt, T), T, 0, stream>>>(Nt, g->rowptr, g->col, g->dis, g->w);
    DSS2_LAUNCH_CHECK();
  }
  k_eptr<<<(B + 1 + T - 1) / T, T, 0, stream>>>(edge_index, Et, ptr, B, g->eptr, stats);
  DSS2_LAUNCH_CHECK();
  if (Et > 0) {
    k_check_edges<<<grid_for(Et, T), T, 0, stream>>>(edge_index, Et, ptr, B, stats);
    DSS2_LAUNCH_CHECK();
  }
  DSS2_CUDA(cudaMemcpyAsync(h_stats, stats, ST_COUNT * 4, cudaMemcpyDeviceToHost, stream));
  DSS2_CUDA(cudaStreamSynchronize(stream));
  DSS2_CHECK_ARG(!h_stats[ST_BAD_INDEX], "dss2_graph_build: edge_index entry outside [0, %lld)", (long long)Nt);

  int max_seg = h_stats[ST_MAX_SEG_NODES];
  if (h_stats[ST_NOT_TILEABLE] || max_seg > tile_cap || max_seg == 0) {
    g->graphs_per_tile = 0;  // generic (large-graph) kernels only
    g->num_tiles = 0;
    return 0;
  }
  g->graphs_per_tile = tile_cap / max_seg;
  g->num_tiles = (B + g->graphs_per_tile - 1) / g->graphs_per_tile;
  k_tile_stats<<<(g->num_tiles + T - 1) / T, T, 0, stream>>>(*g, stats);
  DSS2_LAUNCH_CHECK();
  DSS2_CUDA(cudaMemcpyAsync(h_stats, stats, ST_COUNT * 4, cudaMemcpyDeviceToHost, stream));
  DSS2_CUDA(cudaStreamSynchronize(stream));
  g->max_tile_nodes = h_stats[ST_MAX_TILE_NODES];
  g->max_tile_nnz = h_stats[ST_MAX_TILE_NNZ];
  g->max_tile_edges = h_stats[ST_MAX_TILE_EDGES];
  k_build_ell<<<g->num_tiles, 128, 0, stream>>>(*g);
  DSS2_LAUNCH_CHECK();
  k_hop_keys<<<(g->num_tiles + 63) / 64, 64, 0, stream>>>(*g, hop_keys);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_hop_keys_host(const uint32_t* ell_ci, const int64_t* tile_ptr, int32_t num_tiles, int hop_keys, uint8_t* keys) {
  DSS2_CHECK_ARG(ell_ci && tile_ptr && keys && num_tiles >= 0, "dss2_hop_keys_host: bad argument");
  DSS2_CHECK_ARG(hop_keys == DSS2_HOP_KEYS_IDENTITY || hop_keys == DSS2_HOP_KEYS_COLOR, "dss2_hop_keys_host: hop_keys %d is not a policy", hop_keys);
  for (int t = 0; t < num_tiles; ++t) {
    const int64_t n0 = tile_ptr[t], nT = tile_ptr[t + 1] - n0;
    DSS2_CHECK_ARG(nT >= 0 && nT <= DSS2_TILE_CAP, "dss2_hop_keys_host: tile %d has %lld rows", t, (long long)nT);
    hop_keys_tile(reinterpret_cast<const uint2*>(ell_ci) + n0, (int)nT, (int)n0, hop_keys, keys + n0);
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// batch packer
// ---------------------------------------------------------------------------------------------
namespace {

// single block: exclusive scan of the selected scenarios' node / edge counts -> ptr, eptr; resets vminmax
__global__ void __launch_bounds__(1024) k_pack_scan(const int64_t* __restrict__ node_off, const int64_t* __restrict__ edge_off,
                            const int64_t* __restrict__ ids, int B, int64_t* ptr, int64_t* eptr, float* vminmax) {
  typedef cub::BlockScan<long long, 1024> Scan;
  __shared__ typename Scan::TempStorage tmp_n, tmp_e;
  int per = (B + 1023) / 1024;
  int b0 = threadIdx.x * per, b1 = min(B, b0 + per);
  long long sn = 0, se = 0;
  for (int b = b0; b < b1; ++b) {
    int64_t s = ids[b];
    sn += node_off[s + 1] - node_off[s];
    se += edge_off[s + 1] - edge_off[s];
  }
  long long pn, pe, tn, te;
  Scan(tmp_n).ExclusiveSum(sn, pn, tn);
  Scan(tmp_e).ExclusiveSum(se, pe, te);
  for (int b = b0; b < b1; ++b) {
    int64_t s = ids[b];
    ptr[b] = pn;
    eptr[b] = pe;
    pn += node_off[s + 1] - node_off[s];
    pe += edge_off[s + 1] - edge_off[s];
  }
  if (threadIdx.x == 0) {
    ptr[B] = tn;
    eptr[B] = te;
    if (vminmax) {
      vminmax[0] = __int_as_float(0x7f800000);  // +inf
      vminmax[1] = 0.0f;
    }
  }
}

// grid (slices, B): slice `blockIdx.x` of graph `blockIdx.y`; pure gathers, coalesced in the innermost index
__global__ void k_pack_copy(const float* __restrict__ x_all, const float* __restrict__ ea_all, const float* __restrict__ y_all,
                            const int64_t* __restrict__ ei_all, int64_t ei_all_cols, const int64_t* __restrict__ node_off,
                            const int64_t* __restrict__ edge_off, const int64_t* __restrict__ ids,
                            const int64_t* __restrict__ ptr, const int64_t* __restrict__ eptr, float* x, int64_t* ei,
                            int64_t ei_cols, float* ea, float* y, int64_t* batch, float* vminmax) {
  int b = blockIdx.y;
  int64_t s = ids[b];
  int64_t n_src = node_off[s], nn = node_off[s + 1] - n_src, n_dst = ptr[b];
  int64_t e_src = edge_off[s], ne = edge_off[s + 1] - e_src, e_dst = eptr[b];
  // element indices inside one graph fit 32 bits (64-bit `i % 11` alone cost ~20 instructions per copied float: the kernel was issue bound)
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
  const int nx = (int)nn * 11, nea = (int)ne * 13, nn32 = (int)nn, ne32 = (int)ne;
  float vmin = __int_as_float(0x7f800000), vmax = 0.0f;
  const float* xs = x_all + n_src * 11;
  float* xd = x + n_dst * 11;
  for (int i = tid; i < nx; i += nth) {
    float v = xs[i];
    xd[i] = v;
    if (i % 11 == 8) {
      vmin = fminf(vmin, v);
      vmax = fmaxf(vmax, v);
    }
  }
  const float* es = ea_all + e_src * 13;
  float* ed = ea + e_dst * 13;
  for (int i = tid; i < nea; i += nth) ed[i] = es[i];
  if (y) {
    const float* ys = y_all + n_src * 2;
    float* yd = y + n_dst * 2;
    for (int i = tid; i < 2 * nn32; i += nth) yd[i] = ys[i];
  }
  const int64_t* ei_s0 = ei_all + e_src;
  const int64_t* ei_s1 = ei_all + ei_all_cols + e_src;
  int64_t* ei_d0 = ei + e_dst;
  int64_t* ei_d1 = ei + ei_cols + e_dst;
  for (int i = tid; i < ne32; i += nth) {
    ei_d0[i] = ei_s0[i] + n_dst;
    ei_d1[i] = ei_s1[i] + n_dst;
  }
  if (batch) {
    int64_t* bd = batch + n_dst;
    for (int i = tid; i < nn32; i += nth) bd[i] = b;
  }
  if (vminmax) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    // one atomic pair per CTA (all launches hit the same two words: per-warp atomics queued 32 k deep at B = 4096)
    __shared__ float s_mm[2][32];
    const int warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if ((threadIdx.x & 31) == 0) {
      s_mm[0][warp] = vmin;
      s_mm[1][warp] = vmax;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < nw; ++w) {
        vmin = fminf(vmin, s_mm[0][w]);
        vmax = fmaxf(vmax, s_mm[1][w]);
      }
      // vn_kv > 0: IEEE order == integer order; CTAs that saw no bus row (slices beyond the graph) hold the neutral elements
      if (vmin <= vmax) {
        atomicMin((int*)&vminmax[0], __float_as_int(vmin));
        atomicMax((int*)&vminmax[1], __float_as_int(vmax));
      }
    }
  }
}

__global__ void k_minmax_init(float* vminmax) {
  vminmax[0] = __int_as_float(0x7f800000);
  vminmax[1] = 0.0f;
}
__global__ void k_col_minmax(const float* __restrict__ x, int64_t stride, int col, int64_t n, float* vminmax) {
  float vmin = __int_as_float(0x7f800000), vmax = 0.0f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float v = x[i * stride + col];
    vmin = fminf(vmin, v);
    vmax = fmaxf(vmax, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
    vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin((int*)&vminmax[0], __float_as_int(vmin));
    atomicMax((int*)&vminmax[1], __float_as_int(vmax));
  }
}

}  // namespace

extern "C" int dss2_pack_batch(const float* x_all, const float* ea_all, const float* y_all, const int64_t* ei_all,
                               int64_t ei_all_cols, const int64_t* node_off, const int64_t* edge_off, const int64_t* scen_ids,
                               int32_t B, float* x, int64_t* edge_index, int64_t edge_index_cols, float* edge_attr, float* y,
                               int64_t* batch, int64_t* ptr, int64_t* eptr, float* vminmax, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x_all && ea_all && ei_all && node_off && edge_off && scen_ids && x && edge_index && edge_attr && ptr && eptr,
                 "dss2_pack_batch: null argument");
  DSS2_CHECK_ARG(B >= 1 && B <= 65535, "dss2_pack_batch: num_graphs %d outside 1..65535", B);
  DSS2_CHECK_ARG(!y || y_all, "dss2_pack_batch: y requested without y_all");
  k_pack_scan<<<1, 1024, 0, stream>>>(node_off, edge_off, scen_ids, B, ptr, eptr, vminmax);
  DSS2_LAUNCH_CHECK();
  // slices per graph: enough CTAs to fill the machine when B is small, one CTA per graph otherwise
  int slices = max(1, min(64, (148 * 8) / B));
  k_pack_copy<<<dim3(slices, B), 128, 0, stream>>>(x_all, ea_all, y_all, ei_all, ei_all_cols, node_off, edge_off, scen_ids, ptr,
                                                   eptr, x, edge_index, edge_index_cols, edge_attr, y, batch, vminmax);
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_col_minmax(const float* x, int64_t stride, int col, int64_t n, float* vminmax, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x && vminmax && n > 0, "dss2_col_minmax: bad argument");
  k_minmax_init<<<1, 1, 0, stream>>>(vminmax);
  DSS2_LAUNCH_CHECK();
  k_col_minmax<<<grid_for(n, 256), 256, 0, stream>>>(x, stride, col, n, vminmax);
  DSS2_LAUNCH_CHECK();
  return 0;
}
