// (b2) TAG layer on tcgen05, third generation: k_tag_tc3 = k_tag_tc2's arithmetic with every global-memory access of the worker
// threads moved onto the TMA engine.
//
// Why (clock64 stamps of one worker thread, Oberrhein B=4096, profiles/r2_stamps_tc2.txt): of the 12.3 k (forward) / 14.8 k
// (backward-to-input) cycles a 210-row tile spent in k_tag_tc2, ~2.2 k were the next tile's row prefetch (16 warps x 7 LDG: the
// LSU moves 64 B per cycle and the gathers of the hops queue behind it) and, in the backward, ~2.8 k the hop-level spill (8
// STG.128 per thread).  Here
//   * the MMA-issuer warp's elected lane lands the NEXT-BUT-ONE tile in a two-stage shared-memory ring: the 32-wide rows with one
//     cp.async.bulk.tensor (SWIZZLE_128B tensor map: a thread then reads its own row without bank conflicts), the ELL topology and
//     the sign words with 1-D bulk copies; the tile's node range travels through shared memory with them, so a worker issues no
//     global load at all;
//   * the backward's hop levels leave as ONE cp.async.bulk store per level straight from the plain level tile the next hop
//     gathers from.  That tile is software-swizzled by the graph's per-row keys (16-byte chunk c of row n sits at chunk
//     c ^ hop_key[n], see DSS2_HOP_KEYS_COLOR), so its byte image in global memory can be un-swizzled by the weight-gradient kernel
//     without knowing the tiling (format word 1 and the key array behind the levels, see GwArgs::lvl_fmt);
//   * the A operand lives in tensor memory as in k_tag_tc2<TA> (tcgen05.st by the thread that owns the row), so shared memory is
//     read by generic-proxy gathers only and the sole proxy fence left is the one in front of the spill (cheap now: a worker has
//     no global access in flight when it executes it).
// Everything else (thread = (row, half), hop order = PyG scatter order, 3xTF32 with all four terms, epilogue) is k_tag_tc2's.
// Served: tiled graphs, K in 1..2, forward with any cout, backward-to-input with cout == 32 (the 35 hidden layers); the caller
// falls back to k_tag_tc2 otherwise.
#include <cuda.h>

#include "tc2_shared.cuh"

#ifdef DSS2_STAMPS
// diagnostic build only (tools/stamps.sh): per-phase clock64 totals of worker thread 0 and of the issuer of CTA 0
__device__ unsigned long long g_tc3_stamps[32];
#define STAMP(i)                                                    \
  do {                                                              \
    if (blockIdx.x == 0 && (tid == 0)) {                            \
      const long long now_ = clock64();                             \
      g_tc3_stamps[i] += (unsigned long long)(now_ - stamp_prev_);  \
      stamp_prev_ = now_;                                           \
    }                                                               \
  } while (0)
#define STAMP_I(i)                                                  \
  do {                                                              \
    if (blockIdx.x == 0 && (tid & 31) == 0) {                       \
      const long long now_ = clock64();                             \
      g_tc3_stamps[i] += (unsigned long long)(now_ - stamp_prev_);  \
      stamp_prev_ = now_;                                           \
    }                                                               \
  } while (0)
extern "C" int dss2_tc3_stamps(unsigned long long* host_out) {
  unsigned long long zero[32] = {};
  if (cudaMemcpyFromSymbol(host_out, g_tc3_stamps, sizeof(zero)) != cudaSuccess) return -1;
  if (cudaMemcpyToSymbol(g_tc3_stamps, zero, sizeof(zero)) != cudaSuccess) return -1;
  return 0;
}
#else
#define STAMP(i)
#define STAMP_I(i)
#endif

namespace {

// ---- tensor map (driver entry point fetched at run time: the library must load on machines without libcuda) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// [rows, 32] fp32 row-major, box = [box_rows, 32], 128-byte swizzle, out-of-range rows read as zeros
int make_row_map(CUtensorMap* m, const float* base, int64_t rows, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return -1;
  const cuuint64_t dims[2] = {32, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {128};
  const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS
             ? 0
             : -1;
}

__device__ __forceinline__ void tma_load_rows(void* smem_dst, const CUtensorMap* map, int row0, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(map), "r"(0), "r"(row0), "r"(smem_u32(bar))
               : "memory");
}

template <int RW>
struct Tc3Smem {
  static constexpr int ROWS = 32 * RW;
  static constexpr uint32_t LV_TILE = ROWS * tc::ROW_BYTES;
  // one input stage: rows (hardware swizzle, 1024-byte aligned) | ELL weights (16 B / row) | ELL columns + degree (8 B / row, the
  // copy starts at an even row) | sign words (4 B / row, the copy starts at a multiple of 4 rows)
  static constexpr uint32_t ST_W = LV_TILE, ST_CI = ST_W + ROWS * 16, ST_BITS = ST_CI + ROWS * 8 + 16, ST_END = ST_BITS + ROWS * 4 + 16;
  static constexpr uint32_t STAGE = (ST_END + 1023u) & ~1023u;
  static size_t bytes(int K) { return 1024 + 2 * (size_t)LV_TILE + 2 * (size_t)STAGE + (size_t)(K + 1) * 2 * W_TILE + 512; }
};

template <int MODE, int K, int RW>
__global__ void __launch_bounds__(Tc2Shape<RW>::THREADS + 32, RW == 8 ? 1 : 2) k_tag_tc3(Tc2Args a, const __grid_constant__ CUtensorMap in_map) {
  using Shape = Tc2Shape<RW>;
  using Sm = Tc3Smem<RW>;
  constexpr int NB = Shape::NB;
  constexpr int WORKERS = Shape::WORKERS;
  constexpr int THREADS = Shape::THREADS + 32;   // workers + MMA-issuer warp + one publisher warp (layer chaining: tile marks)
  constexpr int ROWS = Shape::ROWS;
  constexpr uint32_t LV_TILE = Sm::LV_TILE;
  constexpr uint32_t TMEM_COLS = NB == 1 ? 256u : 512u;   // D: 64 per block; A: [2 buffers][NB blocks][plain 32 | residual 32]
  extern __shared__ char raw[];
  const dss2_graph_t& g = a.g;
  char* base = align1024(raw);
  char* Lv = base;                                  // [2] plain level tiles (gather sources, spill sources)
  char* St = Lv + 2 * LV_TILE;                      // [2] input stages
  char* Wt = St + 2 * Sm::STAGE;                    // [(K+1)] x 8 KB: rows 0-31 plain W_k, rows 32-63 residual -> one N = 64 operand
  char* tail = Wt + (K + 1) * 2 * W_TILE;
  float* bias_s = reinterpret_cast<float*>(tail);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail + 128);   // [2] "MMAs reading TMEM buffer b have completed"            (tcgen05.commit)
  uint64_t* full = bars + 2;                                  // [2] "all workers have written buffer b"
  uint64_t* in_full = full + 2;                               // [2] "input stage s has landed"
  uint64_t* sp_done = in_full + 2;                            // [2] "the spill has read plain tile b" (once per tile and buffer)
  int* tinfo = reinterpret_cast<int*>(sp_done + 2);           // [2][2] node range of the tile in stage s
  uint32_t* tslot = reinterpret_cast<uint32_t*>(tinfo + 4);
  const int tid = threadIdx.x, warp = tid >> 5;
  const bool issuer = warp == Shape::ISSUER_WARP, publisher = warp == Shape::ISSUER_WARP + 1;
  const uint32_t row = (uint32_t)tid % ROWS, half = ((uint32_t)tid / ROWS) & 1u;
  const int cout = a.cout;
  const bool spill = MODE == MODE_BGX && a.lvl_out != nullptr;
  const bool has_bits = MODE == MODE_BGX && a.in_bits != nullptr;
  // narrow grad_y rows (the last layer of a sub-net: cout 2, 4, 8 or 16 floats): the stage takes them as ONE dense 1-D bulk copy
  // (16-byte-aligned superset of the tile's rows, like the topology words) and the upper feature half of level 0 is zero
  const bool narrow = MODE == MODE_BGX && cout != HID;
  const int nalign = narrow && cout * 4 < 16 ? 16 / (cout * 4) : 1;   // rows per 16 bytes

  // ---- layer chaining: let the next layer launch now (it links to this one per tile through done_flags, see Tc2Args) ----
  if (a.done_flags) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t chain_seq = (a.done_flags || a.wait_flags) ? (uint32_t)a.chain_seq[1] + 1u : 0u;
  // ---- one-time setup ----
  // The first two input tiles are requested BEFORE the weight operand is staged (measured with %globaltimer stamps: staging took 3.2 us and
  // the first tile's loads another 2.2 us after it, every launch, on every SM): one lane of the issuer warp initialises the barriers and
  // issues the loads, which then land while all threads build the weight tiles.
  const int lane = tid & 31;
  if (issuer && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars[i], 1);
      mbar_init(&full[i], WORKERS);
      mbar_init(&in_full[i], 1);
      mbar_init(&sp_done[i], 1);
    }
    fence_mbar_init();
    if (spill && blockIdx.x == 0) {   // spill format: rows swizzled by the keys in g.hop_key
      uint32_t* fmt = reinterpret_cast<uint32_t*>(a.lvl_out + (size_t)K * g.num_nodes * 32);
      fmt[0] = 1u;
      *reinterpret_cast<const uint8_t**>(fmt + 2) = g.hop_key;
    }
  }
  if (warp == 0) tc::tmem_alloc(tslot, TMEM_COLS);
  // land tile `tn` in stage s; the node range goes with it (written before the arrive.expect_tx, which releases it)
  auto issue_in = [&](const TileNodes& tn, int s, int tile) {
    const int nT = tn.n1 - tn.n0;
    if (nT <= 0) return;
    if (a.wait_flags) {   // the producer layer has stored this tile (acquire), and the TMA engine may read it (proxy fence)
      const uint32_t* f = a.wait_flags + tile;
      uint32_t v;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      } while (v != chain_seq);
      asm volatile("fence.proxy.async.global;" ::: "memory");
    }
    char* st = St + (size_t)s * Sm::STAGE;
    const int r2 = tn.n0 & ~1, r4 = tn.n0 & ~3;
    const uint32_t ci_bytes = (uint32_t)(((tn.n0 - r2 + nT) * 8 + 15) & ~15);
    const uint32_t bit_bytes = has_bits ? (uint32_t)(((tn.n0 - r4 + nT) * 4 + 15) & ~15) : 0u;
    tinfo[2 * s] = tn.n0;
    tinfo[2 * s + 1] = tn.n1;
    const int rn = tn.n0 & ~(nalign - 1);
    const uint32_t in_bytes = narrow ? (uint32_t)(((tn.n0 - rn + nT) * cout * 4 + 15) & ~15) : LV_TILE;
    mbar_expect_tx(&in_full[s], in_bytes + (uint32_t)nT * 16u + ci_bytes + bit_bytes);
    if (narrow) bulk_g2s(st, reinterpret_cast<const char*>(a.in) + (size_t)rn * cout * 4, in_bytes, &in_full[s]);
    else tma_load_rows(st, &in_map, tn.n0, &in_full[s]);
    bulk_g2s(st + Sm::ST_W, reinterpret_cast<const char*>(g.ell_w) + (size_t)tn.n0 * 16, (uint32_t)nT * 16u, &in_full[s]);
    bulk_g2s(st + Sm::ST_CI, reinterpret_cast<const char*>(g.ell_ci) + (size_t)r2 * 8, ci_bytes, &in_full[s]);
    if (has_bits) bulk_g2s(st + Sm::ST_BITS, reinterpret_cast<const char*>(a.in_bits) + (size_t)r4 * 4, bit_bytes, &in_full[s]);
  };
  TileNodes t0 = {0, 0}, t1 = {0, 0}, t2 = {0, 0};
  if (issuer) {
    t0 = tile_nodes(g, blockIdx.x);
    t1 = tile_nodes(g, blockIdx.x + gridDim.x);
    t2 = tile_nodes(g, blockIdx.x + 2 * gridDim.x);
    if (lane == 0) {
      issue_in(t0, 0, blockIdx.x);
      issue_in(t1, 1, blockIdx.x + gridDim.x);
    }
  }
  {
    // weight operand, as in k_tag_tc2: all of a thread's loads first (one L2 round trip instead of one per element), then split and store
    constexpr int PER = ((K + 1) * 32 * 32 + THREADS - 1) / THREADS;
    float wv[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int idx = tid + q * THREADS;
      const int k = idx >> 10, nrow = (idx >> 5) & 31, kk = idx & 31;
      const int c = MODE == MODE_FWD ? nrow : kk, j = MODE == MODE_FWD ? kk : nrow;
      wv[q] = (idx < (K + 1) * 32 * 32 && c < cout) ? __ldg(a.w + ((size_t)k * cout + c) * HID + j) : 0.0f;
    }
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int idx = tid + q * THREADS;
      if (idx < (K + 1) * 32 * 32) {
        const int k = idx >> 10, nrow = (idx >> 5) & 31, kk = idx & 31;
        const uint32_t off = tc::swz_off((uint32_t)nrow, (uint32_t)kk);
        *reinterpret_cast<float*>(Wt + (size_t)(2 * k) * W_TILE + off) = wv[q];
        *reinterpret_cast<float*>(Wt + (size_t)(2 * k + 1) * W_TILE + off) = tc::tf32_residual(wv[q]);
      }
    }
  }
  if (tid < 32) bias_s[tid] = (MODE == MODE_FWD && tid < cout) ? a.bias[tid] : 0.0f;
  uint2 key = make_uint2(0u, 0u);
  uint32_t step_lo = 0;
  if (MODE == MODE_FWD && a.drop_mode == 1) {
    const uint64_t seed = a.rng[0], step = a.rng[1];
    key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (a.layer_uid * 0x9E3779B9u) ^ (uint32_t)(step >> 32));
    step_lo = (uint32_t)step;
  }
  fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tslot, 0);
  const int ntiles = g.num_tiles;

  if (issuer) {
    // ===== issuer warp: input ring, MMAs, hop-level spill (all by the elected lane) =====
    const uint32_t idesc = tc::idesc_tf32(128, 64);
    uint32_t fpar[2] = {0u, 0u};
    int it = 0;
#ifdef DSS2_STAMPS
    long long stamp_prev_ = clock64();
#endif
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
      const int s = it & 1;
      const int n0 = t0.n0, nT = t0.n1 - t0.n0;
      const int nmb = (NB == 2 && nT > 128) ? 2 : 1;
      const TileNodes t3 = tile_nodes(g, t + 3 * gridDim.x);   // node range three tiles ahead: its loads have a whole tile to land
#pragma unroll
      for (int k = 0; k <= K; ++k) {
        const int b = k & 1;
        mbar_wait(&full[b], fpar[b]);
        fpar[b] ^= 1u;
        STAMP_I(16 + 2 * k);
        tc::fence_after_sync();
        if (tc::elect_one()) {
          // every worker has read stage s (it arrives on full[0] after storing level 0): refill it with the tile after next
          if (k == 0) issue_in(t2, s, t + 2 * gridDim.x);
          if (spill && k >= 1) {
            bulk_s2g(a.lvl_out + ((size_t)(k - 1) * g.num_nodes + n0) * 32, Lv + (size_t)b * LV_TILE, (uint32_t)nT * 128u);
            bulk_commit();
          }
          const uint64_t dW = tc::smem_desc_sw128(smem_u32(Wt + (size_t)(2 * k) * W_TILE));
          for (int mb = 0; mb < nmb; ++mb) {
            const uint32_t aT = tmem + 64 * NB + (uint32_t)(b * NB + mb) * 64;   // plain word columns [0, 32), residual [32, 64)
#pragma unroll
            for (uint32_t kk = 0; kk < 4; ++kk) {
              const uint32_t o = kk * tc::KSTEP_BYTES;
              tc::mma_tf32_ts(tmem + mb * 64, aT + 32 + kk * 8, tc::desc_advance(dW, o), idesc, (k == 0 && kk == 0) ? 0u : 1u);
              tc::mma_tf32_ts(tmem + mb * 64, aT + kk * 8, tc::desc_advance(dW, o), idesc, 1u);
            }
          }
          tc::mma_commit(&bars[b]);
          if (spill && k >= 1) {   // the plain tile may be overwritten once the bulk engine has read it (separate from the MMAs' commit:
            bulk_wait_read0();     // the epilogue only waits for the accumulators)
            tc::mbar_arrive(&sp_done[b]);
          }
        }
        __syncwarp();
        STAMP_I(17 + 2 * k);
      }
      t0 = t1;
      t1 = t2;
      t2 = t3;
    }
    if (spill && tc::elect_one()) bulk_wait0();   // the spilled levels are complete in global memory before the kernel ends
    __syncwarp();
  } else if (publisher) {
    // ===== publisher warp (layer chaining): once every worker has issued a tile's output stores, make them visible device-wide and
    // publish the tile's mark - off the workers' path (a gpu-scope fence costs ~1 us; measured on a worker it cancelled the overlap) =====
    if (a.done_flags) {
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        named_bar_sync(2, WORKERS + 32);
        if (lane == 0) {
          __threadfence();
          asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(a.done_flags + t), "r"(chain_seq) : "memory");
        }
        __syncwarp();
      }
    }
  } else {
    // ===== worker warps: thread = (row, half) =====
    uint32_t par[2] = {0u, 0u}, ipar[2] = {0u, 0u}, spar[2] = {0u, 0u};
    const uint32_t tlane = (uint32_t)((warp & 3) * 32) << 16;
    auto publish = [&](int b, bool meet, bool spilled) {
      if (spilled) fence_proxy_async();   // the bulk store reads this thread's STS through the async proxy
      tc::tmem_wait_st();
      tc::fence_before_sync();
      tc::mbar_arrive(&full[b]);
      if (meet) named_bar_sync(1, WORKERS);
    };
    auto store_level = [&](const float (&v)[HF], uint32_t key, int b, bool to_smem) {
      if (to_smem) {
        const uint32_t code = row_code_key(row, key);
        char* pt = Lv + (size_t)b * LV_TILE;
#pragma unroll
        for (uint32_t q = 0; q < 4; ++q)
          *reinterpret_cast<float4*>(pt + (code ^ ((half * 4 + q) << 4))) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
      }
      const uint32_t ta = tmem + tlane + 64 * NB + (uint32_t)(b * NB + (row >> 7)) * 64 + half * HF;
      tc::tmem_st16(ta, v);
      float r[HF];
#pragma unroll
      for (int i = 0; i < HF; ++i) r[i] = tc::tf32_residual(v[i]);
      tc::tmem_st16(ta + 32, r);
    };

    int it = 0;
#ifdef DSS2_STAMPS
    long long stamp_prev_ = clock64();
#endif
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
      const int s = it & 1;
      const char* st = St + (size_t)s * Sm::STAGE;
      mbar_wait(&in_full[s], ipar[s]);
      ipar[s] ^= 1u;
      STAMP(0);   // wait for the input stage
      const int n0 = tinfo[2 * s], nT = tinfo[2 * s + 1] - n0;
      const bool live = (int)row < nT;
      const size_t n = (size_t)n0 + row;
      // ---- this thread's half row and topology out of the stage (the tensor map swizzles by the stage row) ----
      float xr[HF];
      RowTopo tp;
      {
        if (narrow) {
          const float* p = reinterpret_cast<const float*>(st) + ((uint32_t)(n0 & (nalign - 1)) + row) * (uint32_t)cout;
#pragma unroll
          for (int c = 0; c < HF; ++c) xr[c] = 0.0f;
          if (half == 0) {
            if (cout == 8) {
              const float4 v0 = *reinterpret_cast<const float4*>(p), v1 = *reinterpret_cast<const float4*>(p + 4);
              xr[0] = v0.x, xr[1] = v0.y, xr[2] = v0.z, xr[3] = v0.w, xr[4] = v1.x, xr[5] = v1.y, xr[6] = v1.z, xr[7] = v1.w;
            } else if (cout == 2) {
              const float2 v0 = *reinterpret_cast<const float2*>(p);
              xr[0] = v0.x, xr[1] = v0.y;
            } else {
#pragma unroll
              for (int c = 0; c < HF; ++c)
                if (c < cout) xr[c] = p[c];
            }
          }
        } else {
          const uint32_t code = tc::row_code(row);
#pragma unroll
          for (uint32_t q = 0; q < 4; ++q) {
            const float4 v = *reinterpret_cast<const float4*>(st + (code ^ ((half * 4 + q) << 4)));
            xr[4 * q] = v.x;
            xr[4 * q + 1] = v.y;
            xr[4 * q + 2] = v.z;
            xr[4 * q + 3] = v.w;
          }
        }
        tp = row_topo(*reinterpret_cast<const float4*>(st + Sm::ST_W + row * 16),
                      *reinterpret_cast<const uint2*>(st + Sm::ST_CI + ((uint32_t)(n0 & 1) + row) * 8));
        uint32_t word = 0xffffu;
        if (has_bits) word = *reinterpret_cast<const uint32_t*>(st + Sm::ST_BITS + ((uint32_t)(n0 & 3) + row) * 4) >> (half * HF);
        if (!live) word = 0u;   // rows past the tile hold the next tile's data: the MMA input of dead rows is zero
#pragma unroll
        for (int c = 0; c < HF; ++c) {
          const float sc = has_bits ? xr[c] * a.scale : xr[c];
          xr[c] = ((word >> c) & 1u) ? sc : 0.0f;
        }
      }
      // ---- level 0 (TMEM buffer 0 is free: the previous tile's epilogue waited for its last MMAs; the plain tile once the
      //      previous tile's spill of the level that shared it has been read) ----
      if (spill && K >= 2 && it > 0) {
        mbar_wait(&sp_done[0], spar[0]);
        spar[0] ^= 1u;
      }
      const uint32_t skey = tp.keys & 7u;   // this row's swizzle key in the plain level tiles
      store_level(xr, skey, 0, true);
      STAMP(1);   // stage read + store L0
      publish(0, true, false);
      STAMP(2);
      // ---- levels 1..K ----
#pragma unroll
      for (int k = 1; k <= K; ++k) {
        const int b = k & 1, pb = (k - 1) & 1;
        float h[HF];
        if (live) hop_thread<true>(h, g, tp, Lv + (size_t)pb * LV_TILE, n, n0, half);
        else {
#pragma unroll
          for (int i = 0; i < HF; ++i) h[i] = 0.0f;
        }
        STAMP(3 + 4 * (k - 1));
        if (k >= 2) {   // TMEM buffer b still feeds the MMAs of level k-2
          mbar_wait(&bars[b], par[b]);
          par[b] ^= 1u;
        }
        if (spill && k == 1 && it > 0) {   // plain tile 1: the previous tile's level-1 spill (level 2 shares tile 0 with the unspilled level 0)
          mbar_wait(&sp_done[1], spar[1]);
          spar[1] ^= 1u;
        }
        STAMP(4 + 4 * (k - 1));
        store_level(h, skey, b, k < K || spill);
        STAMP(5 + 4 * (k - 1));
        publish(b, k < K, spill);
        STAMP(6 + 4 * (k - 1));
      }
      // dropout keep bits do not depend on the MMAs: generate them while the tensor core finishes
      uint32_t keep_rng = 0xffffu;
      if (MODE == MODE_FWD && a.act && a.drop_mode == 1 && live) keep_rng = keep_half(key, (uint32_t)t, row, half, step_lo, a.keep_thr16);
      STAMP(11);
      // ---- all MMAs of the tile complete when the last two commits have arrived ----
      if (K >= 1) {
        const int b2 = (K - 1) & 1;
        mbar_wait(&bars[b2], par[b2]);
        par[b2] ^= 1u;
      }
      {
        const int b1 = K & 1;
        mbar_wait(&bars[b1], par[b1]);
        par[b1] ^= 1u;
      }
      tc::fence_after_sync();
      STAMP(12);
      float v[HF];
      {
        uint32_t r1[HF], r2[HF];
        const uint32_t taddr = tmem + (row >> 7) * 64 + half * HF + tlane;
        tc::tmem_ld16_nowait(taddr, r1);
        tc::tmem_ld16_nowait(taddr + 32, r2);
        tc::tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < HF; ++c) v[c] = __uint_as_float(r1[c]) + __uint_as_float(r2[c]);
      }
      tc::fence_before_sync();        // orders these TMEM reads before the next tile's "buffer written" arrival -> issuer -> overwrite of D
      STAMP(13);
      if (live) {
        if (MODE == MODE_FWD) {
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 bq = *reinterpret_cast<const float4*>(bias_s + half * HF + 4 * c4);
            v[4 * c4 + 0] += bq.x;
            v[4 * c4 + 1] += bq.y;
            v[4 * c4 + 2] += bq.z;
            v[4 * c4 + 3] += bq.w;
          }
          if (a.act) {
            uint32_t keep = 0xffffu;
            if (a.drop_mode == 1) {
              keep = keep_rng;
            } else if (a.drop_mode == 2) {
              const uint4 m0 = *reinterpret_cast<const uint4*>(a.mask + n * HID + half * HF);
              const uint32_t mw[4] = {m0.x, m0.y, m0.z, m0.w};
              keep = 0u;
#pragma unroll
              for (int c = 0; c < HF; ++c) keep |= (((mw[c >> 2] >> ((c & 3) * 8)) & 0xffu) != 0u ? 1u : 0u) << c;
            }
            uint32_t word = 0u;
#pragma unroll
            for (int c = 0; c < HF; ++c) {
              float xv = v[c];
              if (a.drop_mode != 0) xv = ((keep >> c) & 1u) ? xv * a.scale : 0.0f;
              xv = fmaxf(xv, 0.0f);
              word |= (xv > 0.0f ? 1u : 0u) << c;
              v[c] = xv;
            }
            if (a.out_bits) reinterpret_cast<uint16_t*>(a.out_bits)[2 * n + half] = (uint16_t)word;   // little endian halves
          }
          if (a.res) {
#pragma unroll
            for (int c = 0; c < HF; ++c)
              if ((int)(half * HF) + c < cout) v[c] += a.res[n * a.res_stride + half * HF + c];
          }
        }
        const int ow = MODE == MODE_FWD ? cout : 32;
        if (ow == 32) {
          // stored below, after a 4x4 lane transpose
        } else if (ow == 8) {
          if (half == 0) {
            float4* dst = reinterpret_cast<float4*>(a.out + n * 8);
            dst[0] = make_float4(v[0], v[1], v[2], v[3]);
            dst[1] = make_float4(v[4], v[5], v[6], v[7]);
          }
        } else if (ow == 2) {
          if (half == 0) *reinterpret_cast<float2*>(a.out + n * 2) = make_float2(v[0], v[1]);
        } else {
#pragma unroll
          for (int c = 0; c < HF; ++c)
            if ((int)(half * HF) + c < ow) a.out[n * ow + half * HF + c] = v[c];
        }
      }
      if ((MODE == MODE_FWD ? cout : 32) == 32) {
        // A thread holds 64 contiguous bytes of ITS row, so a plain STG.128 of the warp touches 32 different 128-byte lines (16 bytes
        // each): ~2000 cycles per tile in the stamps.  Transpose 4x4 chunks inside each group of 4 lanes (rows 4g..4g+3): lane i ends
        // up with chunk i of all four rows, and one warp store then writes 8 rows x 64 contiguous bytes.
        const uint32_t li = (uint32_t)tid & 3u;
        float4 c[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) c[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        auto sel = [](bool p, const float4& x, const float4& y) { return p ? x : y; };
        auto xchg = [](const float4& x, int m) {
          return make_float4(__shfl_xor_sync(0xffffffffu, x.x, m), __shfl_xor_sync(0xffffffffu, x.y, m), __shfl_xor_sync(0xffffffffu, x.z, m),
                             __shfl_xor_sync(0xffffffffu, x.w, m));
        };
        const bool hi2 = li & 2u, hi1 = li & 1u;
        // step A (lanes i, i^2): lane keeps the chunk pair {0,1} (i < 2) or {2,3} of its own row and of row i^2
        const float4 ra0 = xchg(sel(hi2, c[0], c[2]), 2), ra1 = xchg(sel(hi2, c[1], c[3]), 2);
        const float4 b0 = sel(hi2, ra0, c[0]), b1 = sel(hi2, ra1, c[1]), b2 = sel(hi2, c[2], ra0), b3 = sel(hi2, c[3], ra1);
        // step B (lanes i, i^1): lane keeps chunk i of its two rows and receives chunk i of the partner's two rows
        const float4 rb0 = xchg(sel(hi1, b0, b1), 1), rb1 = xchg(sel(hi1, b2, b3), 1);
        const float4 k0 = sel(hi1, b1, b0), k1 = sel(hi1, b3, b2);
        const float4 w0 = sel(hi1, rb0, k0), w1 = sel(hi1, k0, rb0), w2 = sel(hi1, rb1, k1), w3 = sel(hi1, k1, rb1);
        const uint32_t rbase = row & ~3u;
        float* dst = a.out + ((size_t)n0 + rbase) * 32 + (half * 4 + li) * 4;
        if ((int)rbase + 0 < nT) *reinterpret_cast<float4*>(dst) = w0;
        if ((int)rbase + 1 < nT) *reinterpret_cast<float4*>(dst + 32) = w1;
        if ((int)rbase + 2 < nT) *reinterpret_cast<float4*>(dst + 64) = w2;
        if ((int)rbase + 3 < nT) *reinterpret_cast<float4*>(dst + 96) = w3;
      }
      STAMP(14);
      if (a.done_flags) asm volatile("bar.arrive 2, %0;" ::"r"(WORKERS + 32) : "memory");   // this thread's stores of the tile are issued
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, TMEM_COLS);
}

template <int MODE, int K, int RW>
int launch_tc3(const Tc2Args& a, cudaStream_t stream) {
  using Shape = Tc2Shape<RW>;
  CUtensorMap map;
  if (make_row_map(&map, a.in, a.g.num_nodes, Shape::ROWS)) return 1;   // no driver entry point / rejected: the caller falls back
  const size_t smem = Tc3Smem<RW>::bytes(K);
  const int grid = max(1, min(a.g.num_tiles, (RW == 8 ? 1 : 2) * dss2_sm_count()));
  DSS2_CUDA(cudaFuncSetAttribute(k_tag_tc3<MODE, K, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  {
    // chained to the previous layer per tile (wait_flags): may start while that launch still runs (see Tc2Args)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)Shape::THREADS + 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (a.wait_flags) {
      attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[na].val.programmaticStreamSerializationAllowed = 1;
      ++na;
    }
    const int prio = dss2_launch_priority(a.wait_flags ? 1 : 2);
    if (prio != 0) {
      attr[na].id = cudaLaunchAttributePriority;
      attr[na].val.priority = prio;
      ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = (unsigned)na;
    DSS2_CUDA(cudaLaunchKernelEx(&cfg, k_tag_tc3<MODE, K, RW>, a, map));
  }
  DSS2_LAUNCH_CHECK();
  return 0;
}
template <int MODE, int K>
int launch_tc3_k(const Tc2Args& a, cudaStream_t stream) {
  return a.g.max_tile_nodes <= 128 ? launch_tc3<MODE, K, 4>(a, stream) : launch_tc3<MODE, K, 8>(a, stream);
}

}  // namespace

int dss2_tc3_launch(int mode, const Tc2Args& a, int K, cudaStream_t stream) {
  static const bool enabled = [] {
    const char* e = getenv("DSS2_TC3");
    return !(e && e[0] == '0');
  }();
  const dss2_graph_t& g = a.g;
  if (!enabled || g.num_tiles <= 0 || g.max_tile_nodes > T2_MAX || K < 1 || K > 2 || !g.ell_w || !g.ell_ci) return 1;
  static const bool narrow_ok = [] {
    const char* e = getenv("DSS2_TC3_NARROW");
    return !(e && e[0] == '0');
  }();
  // narrow grad_y rows: dense bulk copy of 2 / 4 / 8 / 16-float rows (other widths: k_tag_tc2 loads them directly)
  if (mode == MODE_BGX && a.cout != 32 && !(narrow_ok && (a.cout == 2 || a.cout == 4 || a.cout == 8 || a.cout == 16))) return 1;
  if ((((uintptr_t)a.in | (uintptr_t)a.in_bits | (uintptr_t)a.lvl_out) & 15) != 0) return 1;   // TMA / bulk-copy alignment
  if (mode == MODE_FWD) return K == 1 ? launch_tc3_k<MODE_FWD, 1>(a, stream) : launch_tc3_k<MODE_FWD, 2>(a, stream);
  return K == 1 ? launch_tc3_k<MODE_BGX, 1>(a, stream) : launch_tc3_k<MODE_BGX, 2>(a, stream);
}
