// (b2) TAG layer on tcgen05, second generation: forward, backward-to-input and weight gradients.
//
// ncu on the first tensor-core kernel (profiles/r1c) showed the remaining cost was CUDA-core instruction issue and latency: a
// warp-per-row / lane-per-feature layout spends one warp instruction per 32 floats of ONE row.  Here every CUDA-core stage is
// thread-per-row: a thread owns one node row (32 fp32 in registers), so one warp instruction advances 32 rows.  That cuts the
// non-GEMM work ~4x (gathers are LDS.128 of whole neighbour rows, the epilogue needs no ballots or broadcasts), and the three
// 32x32 transforms stay on the tensor core (3xTF32, accumulators in TMEM).
//
//   k_tag_tc2<FWD>  y = sum_k (A^k x) W_k^T + b, dropout, ReLU, sign word, residual                 (replaces k_tag_fwd; the first tcgen05 version, k_tag_fwd_tc, was removed in round 2)
//   k_tag_tc2<BGX>  grad_x = sum_k (A^k g) W_k with g = grad_y * [y>0]/(1-p): hops commute with the right-multiplication and A is
//                   symmetric on the doubled graph, so the backward-to-input is the SAME kernel with transposed weights; it also
//                   stores A g and A^2 g for the weight-gradient kernel
//   k_tag_gw        grad_W_k = (A^k g)^T x, grad_b = sum g: one streaming MN-major GEMM over 64-row chunks (contraction over node
//                   rows), accumulated in TMEM across the whole persistent CTA; no hop recomputation on x at all
//
// Tiles are <= 128 node rows of whole graphs (graph built with tile_cap = 128).  Operand tiles of hop level k live in one of two
// rotating shared-memory buffers (level k+2 reuses the buffer of level k once its MMAs have committed), so a CTA needs ~90 KB and
// two CTAs share an SM; the next tile's rows are prefetched into registers while the current tile is processed.
#include "common.cuh"
#include "tc.cuh"

#ifdef DSS2_STAMPS
// diagnostic build only (tools/stamps.sh): per-phase clock64 totals of worker thread 0 and of the issuer of CTA 0
__device__ unsigned long long g_tc2_stamps[32];
#define STAMP(i)                                                    \
  do {                                                              \
    if (blockIdx.x == 0 && (tid == 0)) {                            \
      const long long now_ = clock64();                             \
      g_tc2_stamps[i] += (unsigned long long)(now_ - stamp_prev_);  \
      stamp_prev_ = now_;                                           \
    }                                                               \
  } while (0)
#define STAMP_I(i)                                                  \
  do {                                                              \
    if (blockIdx.x == 0 && (tid & 31) == 0) {                       \
      const long long now_ = clock64();                             \
      g_tc2_stamps[i] += (unsigned long long)(now_ - stamp_prev_);  \
      stamp_prev_ = now_;                                           \
    }                                                               \
  } while (0)
#else
#define STAMP(i)
#define STAMP_I(i)
#endif

#include "tc2_shared.cuh"

namespace {

// TA = "A operand in tensor memory": thread (row, half) IS TMEM lane `row`, so a hop level goes straight from the thread's registers
// into the A operand with tcgen05.st (plain fp32 word + rounded residual, 64 columns per level and 128-row block); the MMAs read A
// from TMEM and only the 8 KB weight operand from shared memory.  What that removes from the per-tile chain (clock64 stamps,
// profiles/r2_stamps_*.txt): the residual tiles and their 12 STS.128 per thread, the shared-memory copy of the last level (nobody
// gathers from it), the 4 KB A read of every MMA (the K-major 32-byte slices made an M128 N64 K8 MMA take 100-180 cycles against a
// 32-cycle floor while the workers' gathers hammered the same banks) and all three fence.proxy.async per tile - shared memory is
// only read by generic-proxy gathers now, so a plain bar.sync orders it, and the TMEM hand-over is tcgen05.wait::st + fence.
template <int MODE, int K, int RW, bool DENSE, bool TA>
__global__ void __launch_bounds__(Tc2Shape<RW>::THREADS, Tc2Shape<RW>::CTAS_PER_SM) k_tag_tc2(Tc2Args a) {
  using Shape = Tc2Shape<RW>;
  constexpr int NB = Shape::NB;
  constexpr int TC2_WORKERS = Shape::WORKERS;
  constexpr int TC2_THREADS = Shape::THREADS;
  constexpr int ROWS = Shape::ROWS;
  constexpr uint32_t LV_TILE = ROWS * tc::ROW_BYTES;   // one operand tile (plain or residual) of one hop level
  constexpr int NLV = TA ? 2 : 4;                      // TA: two rotating plain tiles (gather sources); else [2 buffers][plain, residual]
  constexpr uint32_t TMEM_COLS = TA ? (NB == 1 ? 256u : 512u) : 64u * NB;   // D: 64 per block; TA: + [2 buffers][NB blocks][plain 32 | residual 32]
  extern __shared__ char raw[];
  const dss2_graph_t& g = a.g;
  char* base = align1024(raw);
  char* Lv = base;                                  // level tiles
  char* Wt = Lv + NLV * LV_TILE;                    // [(K+1)] x 8 KB: rows 0-31 plain W_k, rows 32-63 residual -> one N = 64 operand
  char* tail = Wt + (K + 1) * 2 * W_TILE;           // (behind the level tiles: a 96-row tile's M = 128 operand read runs 4 KB past its end)
  float* bias_s = reinterpret_cast<float*>(tail);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail + 128);   // [2]: "MMAs reading buffer b have completed"   (tcgen05.commit)
  uint64_t* full = bars + 2;                                  // [2]: "all workers have written buffer b"       (256 arrivals)
  uint32_t* tslot = reinterpret_cast<uint32_t*>(full + 2);
  const int tid = threadIdx.x, warp = tid >> 5;
  const bool issuer = warp == Shape::ISSUER_WARP;
  // worker tid = half * ROWS + row (RW = 3: half * 128 + row): warp % 4 == (row / 32) % 4 = the TMEM lane quarter this warp may read
  const uint32_t row = RW == 3 ? ((uint32_t)tid & 127u) : (uint32_t)tid % ROWS;
  const uint32_t half = RW == 3 ? ((uint32_t)tid >> 7) : (((uint32_t)tid / ROWS) & 1u);
  const int cout = a.cout;
  auto lv_p = [&](int b) { return Lv + (size_t)(TA ? b : 2 * b) * LV_TILE; };
  auto lv_l = [&](int b) { return Lv + (size_t)(2 * b + 1) * LV_TILE; };   // !TA only

  // ---- one-time setup ----
  if (warp == 0) tc::tmem_alloc(tslot, TMEM_COLS);
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&full[0], TC2_WORKERS);
    mbar_init(&full[1], TC2_WORKERS);
    fence_mbar_init();
  }
  // weight operand B[n][kk] (K-major rows n): FWD n = output feature c, kk = input feature j: W_k[c][j];
  //                                           BGX n = input feature j, kk = output feature c: W_k[c][j] transposed
  for (int idx = tid; idx < (K + 1) * 32 * 32; idx += TC2_THREADS) {
    const int k = idx >> 10, nrow = (idx >> 5) & 31, kk = idx & 31;
    const int c = MODE == MODE_FWD ? nrow : kk, j = MODE == MODE_FWD ? kk : nrow;
    const float v = c < cout ? a.w[((size_t)k * cout + c) * HID + j] : 0.0f;
    const uint32_t off = tc::swz_off((uint32_t)nrow, (uint32_t)kk);
    *reinterpret_cast<float*>(Wt + (size_t)(2 * k) * W_TILE + off) = v;
    *reinterpret_cast<float*>(Wt + (size_t)(2 * k + 1) * W_TILE + off) = tc::tf32_residual(v);
  }
  if (tid < 32) bias_s[tid] = (MODE == MODE_FWD && tid < cout) ? a.bias[tid] : 0.0f;
  if (MODE == MODE_BGX && a.lvl_out && blockIdx.x == 0 && tid == 0)   // format word of the hop-level spill: plain rows
    *reinterpret_cast<uint32_t*>(a.lvl_out + (size_t)K * g.num_nodes * 32) = 0u;
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
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tslot, 0);   // warp-uniform for the compiler (MMA operands live in uniform registers)
  constexpr int dense_rows = DENSE ? ROWS : 0;   // compile-time: the tiled instantiations carry none of the hop-free code
  const int ntiles = DENSE ? (int)((g.num_nodes + ROWS - 1) / ROWS) : g.num_tiles;

  if (issuer) {
    // ===== MMA issuer warp: D[:, 0:32] += A W_plain^T, D[:, 32:64] += A W_resid^T for A in {plain, residual} of every level =====
    const uint32_t idesc = tc::idesc_tf32(128, 64);
    uint32_t fpar[2] = {0u, 0u};
#ifdef DSS2_STAMPS
    long long stamp_prev_ = clock64();
#endif
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const TileNodes tn = tile_nodes(g, t, dense_rows);
      const int nmb = (NB == 2 && tn.n1 - tn.n0 > 128) ? 2 : 1;
#pragma unroll
      for (int k = 0; k <= K; ++k) {
        const int b = k & 1;
        mbar_wait(&full[b], fpar[b]);
        fpar[b] ^= 1u;
        STAMP_I(16 + 2 * k);
        tc::fence_after_sync();
        if (tc::elect_one()) {
          const uint64_t dW = tc::smem_desc_sw128(smem_u32(Wt + (size_t)(2 * k) * W_TILE));
          for (int mb = 0; mb < nmb; ++mb) {
            if (TA) {
              const uint32_t aT = tmem + 64 * NB + (uint32_t)(b * NB + mb) * 64;   // plain word columns [0, 32), residual [32, 64)
#pragma unroll
              for (uint32_t kk = 0; kk < 4; ++kk) {
                const uint32_t o = kk * tc::KSTEP_BYTES;
                tc::mma_tf32_ts(tmem + mb * 64, aT + 32 + kk * 8, tc::desc_advance(dW, o), idesc, (k == 0 && kk == 0) ? 0u : 1u);
                tc::mma_tf32_ts(tmem + mb * 64, aT + kk * 8, tc::desc_advance(dW, o), idesc, 1u);
              }
            } else {
              const uint64_t dP = tc::smem_desc_sw128(smem_u32(lv_p(b)) + mb * 128 * tc::ROW_BYTES);
              const uint64_t dL = tc::smem_desc_sw128(smem_u32(lv_l(b)) + mb * 128 * tc::ROW_BYTES);
#pragma unroll
              for (uint32_t kk = 0; kk < 4; ++kk) {
                const uint32_t o = kk * tc::KSTEP_BYTES;
                tc::mma_tf32(tmem + mb * 64, tc::desc_advance(dL, o), tc::desc_advance(dW, o), idesc, (k == 0 && kk == 0) ? 0u : 1u);
                tc::mma_tf32(tmem + mb * 64, tc::desc_advance(dP, o), tc::desc_advance(dW, o), idesc, 1u);
              }
            }
          }
          tc::mma_commit(&bars[b]);
        }
        __syncwarp();
        STAMP_I(17 + 2 * k);
      }
    }
  } else {
    // ===== worker warps: thread = (row, half) =====
    uint32_t par[2] = {0u, 0u};
    // software pipeline over this CTA's tiles: node range two tiles ahead, rows + topology one tile ahead (all in registers)
    float xr[HF];
    uint32_t xr_bits = 0;
    RowTopo tp_next = row_topo(make_float4(0.f, 0.f, 0.f, 0.f), make_uint2(0u, 0u));
    auto load_row = [&](const TileNodes& tn) {   // this thread's half row of the tile, zero padded; BGX: masked grad_y
#pragma unroll
      for (int i = 0; i < HF; ++i) xr[i] = 0.0f;
      if ((int)row >= tn.n1 - tn.n0) return;
      const size_t n = (size_t)tn.n0 + row;
      if (!dense_rows) tp_next = load_row_topo(g, n);
      if (MODE == MODE_FWD || cout == 32) {
        const float4* src = reinterpret_cast<const float4*>(a.in + n * 32 + half * HF);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 v = ldg_stream4(src + q);
          xr[4 * q] = v.x;
          xr[4 * q + 1] = v.y;
          xr[4 * q + 2] = v.z;
          xr[4 * q + 3] = v.w;
        }
      } else {
#pragma unroll
        for (int c = 0; c < HF; ++c)
          if ((int)(half * HF) + c < cout) xr[c] = a.in[n * cout + half * HF + c];
      }
      // BGX: the sign word is only LOADED here; the mask is applied when the tile starts (apply_mask), so that this prefetch never
      // waits for its own loads (clock64 stamps: masking in place exposed ~3000 cycles of DRAM latency per tile)
      if (MODE == MODE_BGX && a.in_bits) xr_bits = a.in_bits[n] >> (half * HF);
    };
    auto apply_mask = [&]() {
      if (MODE == MODE_BGX && a.in_bits) {
#pragma unroll
        for (int c = 0; c < HF; ++c) xr[c] = ((xr_bits >> c) & 1u) ? xr[c] * a.scale : 0.0f;
      }
    };
    // my part of buffer b is written: make it visible to the tensor core, tell the issuer and - when the next stage gathers other
    // threads' rows - meet the workers (after the last level nobody gathers: the MMAs are the only readers, no barrier needed)
    auto publish = [&](int b, bool meet = true) {
      if (TA) {
        tc::tmem_wait_st();
        tc::fence_before_sync();
      } else {
        fence_proxy_async();
      }
      tc::mbar_arrive(&full[b]);
      if (meet) named_bar_sync(1, TC2_WORKERS);
    };
    // this thread's half row of a hop level -> operand storage of buffer b (and, when a later hop gathers from it, the plain tile)
    const uint32_t tlane = (uint32_t)((warp & 3) * 32) << 16;
    auto store_level = [&](const float (&v)[HF], int b, bool gathered) {
      if (!TA) {
        store_half_sw128(v, lv_p(b), lv_l(b), row, half);
        return;
      }
      if (gathered) {
        const uint32_t code = tc::row_code(row);
        char* pt = lv_p(b);
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

    TileNodes cur = tile_nodes(g, blockIdx.x, dense_rows);
    TileNodes nxt = tile_nodes(g, blockIdx.x + gridDim.x, dense_rows);
    load_row(cur);
#ifdef DSS2_STAMPS
    long long stamp_prev_ = clock64();
#endif
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      STAMP(0);
      const int nT = cur.n1 - cur.n0, n0 = cur.n0;
      const bool live = (int)row < nT;
      const size_t n = (size_t)n0 + row;
      const RowTopo tp = tp_next;
      // ---- level 0 (buffer 0 is free: the previous tile's epilogue waited for its last MMAs) ----
      apply_mask();
      store_level(xr, 0, true);                                   // dead rows store zeros: keeps the MMA input finite
      STAMP(1);
      publish(0);
      STAMP(2);
      if (MODE == MODE_BGX && !(a.flags & 1)) {   // see the note on the prefetch below: with the spill stores in flight the backward measures best here
        cur = nxt;
        load_row(cur);
        nxt = tile_nodes(g, t + 2 * gridDim.x, dense_rows);
      }
      // ---- levels 1..K ----
#pragma unroll
      for (int k = 1; k <= K; ++k) {
        const int b = k & 1, pb = (k - 1) & 1;
        float h[HF];
        if (DENSE && live) {   // large-graph path: the level was computed by a hop kernel over the whole graph
          const float4* src = reinterpret_cast<const float4*>(a.dense_lvl + ((size_t)(k - 1) * g.num_nodes + n) * 32 + half * HF);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 v = ldg_stream4(src + q);
            h[4 * q] = v.x;
            h[4 * q + 1] = v.y;
            h[4 * q + 2] = v.z;
            h[4 * q + 3] = v.w;
          }
        } else if (!DENSE && live) hop_thread<false>(h, g, tp, lv_p(pb), n, n0, half);
        else {
#pragma unroll
          for (int i = 0; i < HF; ++i) h[i] = 0.0f;
        }
        STAMP(3 + 4 * (k - 1));   // hop
        if (k >= 2) {   // buffer b still feeds the MMAs of level k-2
          mbar_wait(&bars[b], par[b]);
          par[b] ^= 1u;
        }
        STAMP(4 + 4 * (k - 1));   // wait for the buffer
        store_level(h, b, k < K);
        STAMP(5 + 4 * (k - 1));   // store
        publish(b, k < K);
        STAMP(6 + 4 * (k - 1));   // publish
        // hop-level spill for the weight-gradient pass.  Its stores drain during the next hop; the fence of the next publish still
        // waits for their tail (measured: cheaper than deferring all spills to the tile end, where they pile up with the output
        // stores in front of the next tile's first fence: 88 vs 103 us)
        if (MODE == MODE_BGX && a.lvl_out && live && !(a.flags & 2)) {
          float4* dst = reinterpret_cast<float4*>(a.lvl_out + ((size_t)(k - 1) * g.num_nodes + n) * 32 + half * HF);
#pragma unroll
          for (int q = 0; q < 4; ++q) dst[q] = make_float4(h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]);
        }
      }
      // The prefetch of the next tile sits here, behind the tile's LAST proxy fence: fence.proxy.async waits for every earlier memory
      // operation of the thread, global ones included (clock64 stamps: a prefetch issued before a publish costs ~2000 cycles of
      // exposed DRAM latency at that publish).  From here the loads have the whole epilogue to land.
      if (MODE == MODE_FWD || (a.flags & 1)) {
        cur = nxt;
        load_row(cur);                                             // next tile: rows (same registers) + topology
        nxt = tile_nodes(g, t + 2 * gridDim.x, dense_rows);                    // and the node range of the tile after it
      }
      // dropout keep bits do not depend on the MMAs: generate them while the tensor core finishes
      uint32_t keep_rng = 0xffffu;
      if (MODE == MODE_FWD && a.act && a.drop_mode == 1 && live) keep_rng = keep_half(key, (uint32_t)t, row, half, step_lo, a.keep_thr16);
      STAMP(11);   // spill / prefetch / rng
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
      STAMP(12);   // wait for the MMAs
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
      STAMP(13);   // TMEM loads
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
          float4* dst = reinterpret_cast<float4*>(a.out + n * 32 + half * HF);
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) dst[c4] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
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
      STAMP(14);   // epilogue
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, TMEM_COLS);
}

// -------------------------------------------------------------------------------------------------
// weight gradients: D[32*k + c, j] = sum_r G_k[r][c] * x[r][j]  (k <= K), D[c, 32] = sum_r G_0[r][c]  (bias gradient, ones column)
// -------------------------------------------------------------------------------------------------
constexpr int GW_ROWS = 64;                       // node rows per chunk (contraction block)
constexpr uint32_t GW_TILE = GW_ROWS * tc::ROW_BYTES;   // 8 KB

struct GwArgs {
  int64_t num_nodes;
  const float* x;          // layer input [Nt,32]
  const float* gy;         // grad wrt layer output [Nt,cout]
  const uint32_t* bits;    // sign words or NULL
  const float* lvl;        // [K][Nt,32] = A g, A^2 g from the backward-to-input kernel
  const uint32_t* lvl_fmt; // device words behind the levels: [0] = 0: plain rows; 1: rows as k_tag_tc3 spills them (byte image of its
                           // shared-memory tiles: 16-byte chunk c of row n stored at chunk c ^ key[n]), with the key array (uint8 [Nt],
                           // the graph's hop_key) as a pointer in words [2, 4).  NULL = plain
  int cout;
  float scale;
  float* partials;         // row = blockIdx.x
  int64_t partial_stride;
  int64_t bias_offset;
};

// the key array of a spill in format 1, NULL for plain rows
__device__ __forceinline__ const uint8_t* lvl_keys(const GwArgs& a) {
  return a.lvl_fmt && a.lvl_fmt[0] == 1u ? *reinterpret_cast<const uint8_t* const*>(a.lvl_fmt + 2) : nullptr;
}

constexpr int GW_STAGES = 3;
constexpr uint32_t GW_STAGE_BYTES = 4 * GW_TILE + 320;   // x, grad_y, A g, A^2 g rows + sign words + level swizzle keys of one 64-row chunk
constexpr int GW_CONV = 512;                             // converter threads (16 warps): thread = (16-byte column chunk, row of the chunk)
constexpr int GW_THREADS = GW_CONV + 64;                 // + 1 MMA-issuer warp + 1 bulk-copy producer warp
// one operand buffer: A.hi[K+1 blocks] A.lo[K+1 blocks] B.hi B.lo.  The M = 128 descriptors span 4 blocks: the blocks past the K+1
// levels alias whatever follows in the buffer (finite or not: they only feed rows of D that are never read).
__host__ __device__ constexpr uint32_t gw_ops_bytes(int K) { return (uint32_t)(2 * (K + 1) + 2) * GW_TILE; }

// Roles (ncu on the one-role version: 4 warps, 12 % issue utilisation, the converting thread 0 also spent ~1.9 k cycles per chunk
// issuing 32 MMAs while the other warps waited at the barrier; on the single-buffer version: 45 % of the converter samples waiting
// for the previous chunk's MMAs):
//   warp 16, lane 0: per chunk - once all converters have arrived on `ready[b]` - issues 16 MMAs M128 x N64 x K8: A in {G.lo, G.hi}
//                    x B = [x.hi ; x.lo] stacked along N (the two halves of D are added in the epilogue), commits to `bar[b]`;
//   warp 17, lane 0: lands chunks with bulk copies (3-stage ring); a slot is refilled as soon as `ready[b]` says that every
//                    converter has read it (clock64 stamps: issuing 16 MMAs costs ~980 cycles and 5 bulk copies ~430, so the two
//                    jobs get a thread each);
//   warps 0-15:      thread = (16-byte column chunk cq, row rs): staged row -> registers -> mask -> hi/lo split; wait until the
//                    MMAs that last read operand buffer b (two chunks ago) are complete, store the operand tiles, arrive on
//                    `ready[b]`.
// The operand tiles are double buffered, so conversion and tile stores of chunk i+1 overlap the MMAs of chunk i.
template <int K>
__global__ void __launch_bounds__(GW_THREADS, 1) k_tag_gw(GwArgs a) {
  extern __shared__ char raw[];
  char* base = align1024(raw);
  constexpr uint32_t OPS = gw_ops_bytes(K);
  constexpr uint32_t A_LO = (K + 1) * GW_TILE, B_HI = 2 * (K + 1) * GW_TILE, B_LO = B_HI + GW_TILE;
  char* ops = base;
  char* stage0 = ops + 2 * OPS;                          // raw rows landed by the TMA engine, GW_STAGES deep
  char* tail = stage0 + GW_STAGES * GW_STAGE_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(tail);    // [GW_STAGES] "chunk has landed"
  uint64_t* empty = full + GW_STAGES;                    // [GW_STAGES] "every converter has read the slot" (GW_CONV arrivals)
  uint64_t* ready = empty + GW_STAGES;                   // [2] "operand buffer b is written" (GW_CONV arrivals)
  uint64_t* bar = ready + 2;                             // [2] "the MMAs reading operand buffer b have completed"
  uint64_t* grp_done = bar + 2;                          // [2] "the MMAs of the chunk group accumulating in TMEM accumulator a have completed"
  uint64_t* flushed = grp_done + 2;                      // [2] "every converter has added accumulator a to its registers" (GW_CONV arrivals)
  uint32_t* tslot = reinterpret_cast<uint32_t*>(flushed + 2);
  const int tid = threadIdx.x, warp = tid >> 5;
  const bool issuer = warp == GW_CONV / 32, producer = warp == GW_CONV / 32 + 1;
  const uint32_t cq = tid & 7, rs = (tid >> 3) & 63;
  const int cout = a.cout;

  if (warp == 0) tc::tmem_alloc(tslot, 128);   // two accumulators of 64 columns
  if (tid == 0) {
    for (int s = 0; s < GW_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], GW_CONV);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&ready[b], GW_CONV);
      mbar_init(&bar[b], 1);
      mbar_init(&grp_done[b], 1);
      mbar_init(&flushed[b], GW_CONV);
    }
    fence_mbar_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tslot, 0);   // warp-uniform for the compiler

  const int64_t num_chunks = (a.num_nodes + GW_ROWS - 1) / GW_ROWS;
  const int64_t full_chunks = a.num_nodes / GW_ROWS;       // only whole chunks go through the bulk-copy engine
  const uint8_t* lvl_key = lvl_keys(a);
  float gb[4] = {0.f, 0.f, 0.f, 0.f};
  int it = 0;                                              // chunks this CTA has processed (same count in every role)
  // The tensor core adds into its fp32 accumulator with truncation, and a CTA adds ~500 MMAs into the same words: measured on the
  // full-size batch (tests: ...full_parity_vs_fp64_oracle) that chain alone put one weight gradient at 1.16e-5 of its scale.  So the
  // chunks go in groups of GW_GROUP into two alternating TMEM accumulators, and every finished group is added - rounded to nearest -
  // into registers: converter thread (warp w, lane l) owns TMEM lane 32 (w % 4) + l, columns [16 (w / 4), +16).
  constexpr int GW_GROUP = 4;
  float facc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) facc[i] = 0.0f;
  const int my_chunks = blockIdx.x < num_chunks ? (int)((num_chunks - 1 - blockIdx.x) / gridDim.x) + 1 : 0;
  const int my_groups = (my_chunks + GW_GROUP - 1) / GW_GROUP;

  if (producer) {
    if (tc::elect_one()) {
      const uint32_t gy_bytes = (uint32_t)(GW_ROWS * cout * 4);
      const uint32_t tx = GW_TILE * (K >= 2 ? 3 : 2) + gy_bytes + (a.bits ? 256u : 0u) + (lvl_key ? 64u : 0u);
      auto issue = [&](int64_t ch, int s) {
        if (ch >= full_chunks) return;
        char* st = stage0 + (size_t)s * GW_STAGE_BYTES;
        const int64_t n = ch * GW_ROWS;
        mbar_expect_tx(&full[s], tx);
        bulk_g2s(st, a.x + n * 32, GW_TILE, &full[s]);
        bulk_g2s(st + GW_TILE, a.gy + n * cout, gy_bytes, &full[s]);
        bulk_g2s(st + 2 * GW_TILE, a.lvl + n * 32, GW_TILE, &full[s]);
        if (K >= 2) bulk_g2s(st + 3 * GW_TILE, a.lvl + (a.num_nodes + n) * 32, GW_TILE, &full[s]);
        if (a.bits) bulk_g2s(st + 4 * GW_TILE, a.bits + n, 256, &full[s]);
        if (lvl_key) bulk_g2s(st + 4 * GW_TILE + 256, lvl_key + n, 64, &full[s]);
      };
      for (int i = 0; i < GW_STAGES; ++i) issue(blockIdx.x + (int64_t)i * gridDim.x, i);
      for (int64_t ch = blockIdx.x; ch < num_chunks; ch += gridDim.x, ++it) {
        const int s = it % GW_STAGES;
        mbar_wait(&empty[s], (uint32_t)((it / GW_STAGES) & 1));      // every converter has read the slot into registers
        issue(ch + (int64_t)GW_STAGES * gridDim.x, s);
      }
    }
    __syncwarp();
  } else if (issuer) {
    if (tc::elect_one()) {
      const uint32_t idesc = tc::idesc_tf32(128, 64, 1, 1);
      for (int64_t ch = blockIdx.x; ch < num_chunks; ch += gridDim.x, ++it) {
        const int b = it & 1;
        const int grp = it / GW_GROUP, ga = grp & 1;
        const bool first = it % GW_GROUP == 0, last = it % GW_GROUP == GW_GROUP - 1 || it == my_chunks - 1;
        const uint32_t ob = smem_u32(ops + b * OPS);
        const uint64_t dAh = tc::smem_desc_mn32(ob, GW_TILE), dAl = tc::smem_desc_mn32(ob + A_LO, GW_TILE);
        const uint64_t dB = tc::smem_desc_mn32(ob + B_HI, GW_TILE);
        mbar_wait(&ready[b], (uint32_t)((it >> 1) & 1));
        if (first && grp >= 2) mbar_wait(&flushed[ga], (uint32_t)(((grp >> 1) - 1) & 1));   // accumulator ga has been read out
        tc::fence_after_sync();
        const uint32_t acc = tmem + (uint32_t)ga * 64u;
#pragma unroll
        for (uint32_t ks = 0; ks < GW_ROWS / 8; ++ks) {
          const uint32_t o = ks * 1024;
          tc::mma_tf32(acc, tc::desc_advance(dAl, o), tc::desc_advance(dB, o), idesc, (first && ks == 0) ? 0u : 1u);
          tc::mma_tf32(acc, tc::desc_advance(dAh, o), tc::desc_advance(dB, o), idesc, 1u);
        }
        tc::mma_commit(&bar[b]);
        if (last) tc::mma_commit(&grp_done[ga]);
      }
    }
    __syncwarp();
  } else {
    int next_flush = 0;   // first group not yet added to facc
    auto flush = [&](int grp) {
      const int ga = grp & 1;
      mbar_wait(&grp_done[ga], (uint32_t)((grp >> 1) & 1));
      tc::fence_after_sync();
      uint32_t r[16];
      tc::tmem_ld16_nowait(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)ga * 64u + (uint32_t)(warp >> 2) * 16u, r);
      tc::tmem_wait_ld();
      tc::fence_before_sync();
      tc::mbar_arrive(&flushed[ga]);
#pragma unroll
      for (int i = 0; i < 16; ++i) facc[i] += __uint_as_float(r[i]);
    };
    for (int64_t ch = blockIdx.x; ch < num_chunks; ch += gridDim.x, ++it) {
      const int s = it % GW_STAGES, b = it & 1;
      const bool staged = ch < full_chunks;
      // one chunk after a group's last: its MMAs have had a whole chunk's conversion time to finish
      if (next_flush < it / GW_GROUP && it % GW_GROUP >= 1) {
        flush(next_flush);
        ++next_flush;
      }
      const char* st = stage0 + (size_t)s * GW_STAGE_BYTES;
      if (staged) mbar_wait(&full[s], (uint32_t)((it / GW_STAGES) & 1));
      const uint32_t r = rs;
      const int64_t n = ch * GW_ROWS + r;
      float4 vx, vg, v1, v2;
      vx = vg = v1 = v2 = make_float4(0.f, 0.f, 0.f, 0.f);
      uint32_t word = 0xffffffffu;
      uint32_t cl = cq;   // chunk position of columns [4 cq, 4 cq + 4) in a spilled level row
      if (lvl_key) cl ^= staged ? (uint32_t)reinterpret_cast<const uint8_t*>(st + 4 * GW_TILE + 256)[r] : n < a.num_nodes ? (uint32_t)lvl_key[n] : 0u;
      if (staged) {
        vx = *reinterpret_cast<const float4*>(st + r * 128 + cq * 16);
        v1 = *reinterpret_cast<const float4*>(st + 2 * GW_TILE + r * 128 + cl * 16);
        if (K >= 2) v2 = *reinterpret_cast<const float4*>(st + 3 * GW_TILE + r * 128 + cl * 16);
        if (cout == 32) {
          vg = *reinterpret_cast<const float4*>(st + GW_TILE + r * 128 + cq * 16);
        } else {
          const float* gp = reinterpret_cast<const float*>(st + GW_TILE) + r * cout;
          float t4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if ((int)(cq * 4 + e) < cout) t4[e] = gp[cq * 4 + e];
          vg = make_float4(t4[0], t4[1], t4[2], t4[3]);
        }
        if (a.bits) word = reinterpret_cast<const uint32_t*>(st + 4 * GW_TILE)[r];
      } else if (n < a.num_nodes) {   // the one ragged chunk at the end of the batch: plain bounded loads
        vx = *reinterpret_cast<const float4*>(a.x + n * 32 + cq * 4);
        v1 = *reinterpret_cast<const float4*>(a.lvl + n * 32 + cl * 4);
        if (K >= 2) v2 = *reinterpret_cast<const float4*>(a.lvl + (a.num_nodes + n) * 32 + cl * 4);
        float t4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if ((int)(cq * 4 + e) < cout) t4[e] = a.gy[n * cout + cq * 4 + e];
        vg = make_float4(t4[0], t4[1], t4[2], t4[3]);
        if (a.bits) word = a.bits[n];
      }
      if (a.bits) {
        const uint32_t w4 = word >> (cq * 4);
        vg.x = (w4 & 1u) ? vg.x * a.scale : 0.0f;
        vg.y = (w4 & 2u) ? vg.y * a.scale : 0.0f;
        vg.z = (w4 & 4u) ? vg.z * a.scale : 0.0f;
        vg.w = (w4 & 8u) ? vg.w * a.scale : 0.0f;
      }
      tc::mbar_arrive(&empty[s]);   // slot s is in registers: the producer may refill it
      // grad_b = column sums of the masked output gradient, exact fp32 on the CUDA cores (a ones-column in the GEMM would inherit
      // the 2^-23 TF32-pair representation error, visible in this cancelling sum)
      gb[0] += vg.x;
      gb[1] += vg.y;
      gb[2] += vg.z;
      gb[3] += vg.w;
      if (it >= 2) mbar_wait(&bar[b], (uint32_t)(((it >> 1) - 1) & 1));   // the MMAs of chunk it-2 read this operand buffer
      char* Ah = ops + b * OPS;
      char* Al = Ah + A_LO;
      char* Bh = Ah + B_HI;
      char* Bl = Ah + B_LO;
      const uint32_t off = tc::swz32_off(r, cq * 4);
      tc::split_store4(vx, Bh, Bl, off);                                      // x
      tc::split_store4(vg, Ah, Al, off);                                      // G_0
      tc::split_store4(v1, Ah + GW_TILE, Al + GW_TILE, off);                  // G_1
      if (K >= 2) tc::split_store4(v2, Ah + 2 * GW_TILE, Al + 2 * GW_TILE, off);   // G_2
      fence_proxy_async();
      tc::mbar_arrive(&ready[b]);
    }
    while (next_flush < my_groups) {   // the remaining groups (the last group's commit covers every MMA issued before it)
      flush(next_flush);
      ++next_flush;
    }
  }
  // ---- write this CTA's partial sums: converter thread = TMEM lane m = 32*level + c, 16 of the 64 columns; columns 0-31 (x.hi part)
  //      and 32-63 (x.lo part) of the same weight are added through the partial row itself (hi part stored, barrier, lo part added) ----
  float* part = a.partials + (size_t)blockIdx.x * a.partial_stride;
  {
    const int m = (warp & 3) * 32 + (tid & 31), k = m >> 5, c = m & 31, cg = warp >> 2;   // cg: column group of 16 (converter warps only)
    const bool mine = tid < GW_CONV && k <= K && c < cout;
    float4* dst = reinterpret_cast<float4*>(part + ((size_t)k * cout + c) * 32 + (cg & 1) * 16);
    if (mine && cg < 2) {
#pragma unroll
      for (int q = 0; q < 4; ++q) dst[q] = make_float4(facc[4 * q], facc[4 * q + 1], facc[4 * q + 2], facc[4 * q + 3]);
    }
    __syncthreads();
    if (mine && cg >= 2) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float4 v = dst[q];
        v.x += facc[4 * q];
        v.y += facc[4 * q + 1];
        v.z += facc[4 * q + 2];
        v.w += facc[4 * q + 3];
        dst[q] = v;
      }
    }
  }
  // bias gradient: 64 row partials per column -> shared memory -> 32 column sums in fixed order
  float* red = reinterpret_cast<float*>(stage0);
  __syncthreads();
  if (tid < GW_CONV) {
#pragma unroll
    for (int e = 0; e < 4; ++e) red[rs * 33 + cq * 4 + e] = gb[e];
  }
  __syncthreads();
  if (tid < 32 && tid < cout) {
    float sum = 0.0f;
    for (int r = 0; r < 64; ++r) sum += red[r * 33 + tid];
    part[a.bias_offset + tid] = sum;
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, 128);
}

// -------------------------------------------------------------------------------------------------
// The same weight gradients on the fp32 FMA pipe, exact fp32 (no TF32 split, no TMEM accumulation order): a pure streaming
// kernel - no hops, no dependency chain - so the CUDA cores are not the handicap they are in the layer kernels.  The bulk-copy
// ring lands raw 64-row chunks; a short pre-pass applies the dropout/ReLU mask to grad_y (and sums the bias gradient); then
// thread (i = input feature, cg = group of 4 output columns) keeps 4(K+1) accumulators and walks the chunk's rows:
// per row 1 LDS (x[r][i], conflict free) + (K+1) broadcast LDS.128 + 4(K+1) FFMA.
// -------------------------------------------------------------------------------------------------
constexpr int GWF_STAGES = 4;
constexpr int GWF_THREADS = 256;
#define GWF_STAGE_BYTES(K) ((uint32_t)((K) + 2) * GW_TILE + 320u)   // x, grad_y, K hop levels, sign words, level swizzle keys
template <int K>
size_t gwf_smem() { return 1024 + GWF_STAGES * GWF_STAGE_BYTES(K) + 2 * GW_TILE + 32 * 33 * 4 + 64; }

template <int K>
__global__ void __launch_bounds__(GWF_THREADS, 1) k_tag_gw_ffma(GwArgs a) {
  extern __shared__ char raw[];
  char* base = align1024(raw);
  constexpr uint32_t STAGE = GWF_STAGE_BYTES(K);
  char* stage0 = base;
  float* G0 = reinterpret_cast<float*>(stage0 + GWF_STAGES * STAGE);   // [2][64][32] masked, scaled grad_y (double buffered)
  float* red = G0 + 2 * GW_ROWS * 32;                                   // [32][33] bias-gradient partials
  uint64_t* full = reinterpret_cast<uint64_t*>(red + 32 * 33);
  const int tid = threadIdx.x;
  const int cout = a.cout;
  if (tid == 0) {
    for (int s = 0; s < GWF_STAGES; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const int64_t num_chunks = (a.num_nodes + GW_ROWS - 1) / GW_ROWS;
  const int64_t full_chunks = a.num_nodes / GW_ROWS;
  const uint32_t gy_bytes = (uint32_t)(GW_ROWS * cout * 4);
  const uint8_t* lvl_key = lvl_keys(a);
  const uint32_t tx = GW_TILE * (K + 1) + gy_bytes + (a.bits ? 256u : 0u) + (lvl_key ? 64u : 0u);
  auto issue = [&](int64_t ch, int s) {
    if (ch >= full_chunks) return;
    char* st = stage0 + (size_t)s * STAGE;
    const int64_t n = ch * GW_ROWS;
    mbar_expect_tx(&full[s], tx);
    bulk_g2s(st, a.x + n * 32, GW_TILE, &full[s]);
    bulk_g2s(st + GW_TILE, a.gy + n * cout, gy_bytes, &full[s]);
#pragma unroll
    for (int k = 0; k < K; ++k) bulk_g2s(st + (2 + k) * GW_TILE, a.lvl + ((int64_t)k * a.num_nodes + n) * 32, GW_TILE, &full[s]);
    if (a.bits) bulk_g2s(st + (K + 2) * GW_TILE, a.bits + n, 256, &full[s]);
    if (lvl_key) bulk_g2s(st + (K + 2) * GW_TILE + 256, lvl_key + n, 64, &full[s]);
  };
  if (tid == 0)
    for (int i = 0; i < GWF_STAGES - 1; ++i) issue(blockIdx.x + (int64_t)i * gridDim.x, i);

  const uint32_t cq = tid & 7, rs = tid >> 3;          // pre-pass mapping: 16-byte column chunk, row (and row + 32)
  const int i_feat = tid & 31, c0 = (tid >> 5) * 4;    // main mapping
  float gb[4] = {0.f, 0.f, 0.f, 0.f};
  float acc[K + 1][4];
#pragma unroll
  for (int k = 0; k <= K; ++k)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[k][e] = 0.0f;

  int it = 0;
  for (int64_t ch = blockIdx.x; ch < num_chunks; ch += gridDim.x, ++it) {
    const int s = it % GWF_STAGES;
    char* st = stage0 + (size_t)s * STAGE;
    float* g0 = G0 + (it & 1) * GW_ROWS * 32;
    if (ch < full_chunks) {
      mbar_wait(&full[s], (uint32_t)((it / GWF_STAGES) & 1));
    } else {   // the one ragged chunk at the end of the batch: bounded loads by all threads into the (idle) slot, zero filled
      const int64_t n0 = ch * GW_ROWS;
      for (int idx = tid; idx < GW_ROWS * 32; idx += GWF_THREADS) {
        const int r = idx >> 5, j = idx & 31;
        const bool inb = n0 + r < a.num_nodes;
        reinterpret_cast<float*>(st)[idx] = inb ? a.x[(n0 + r) * 32 + j] : 0.0f;
#pragma unroll
        for (int k = 0; k < K; ++k)
          reinterpret_cast<float*>(st + (2 + k) * GW_TILE)[idx] = inb ? a.lvl[((int64_t)k * a.num_nodes + n0 + r) * 32 + j] : 0.0f;   // byte image: keeps the level format
        if (j < cout) reinterpret_cast<float*>(st + GW_TILE)[r * cout + j] = inb ? a.gy[(n0 + r) * cout + j] : 0.0f;
        if (a.bits && j == 0) reinterpret_cast<uint32_t*>(st + (K + 2) * GW_TILE)[r] = inb ? a.bits[n0 + r] : 0u;
        if (lvl_key && j == 0) reinterpret_cast<uint8_t*>(st + (K + 2) * GW_TILE + 256)[r] = inb ? lvl_key[n0 + r] : 0u;
      }
      __syncthreads();
    }
    // pre-pass: masked, scaled output gradient -> g0, bias gradient
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t r = rs + 32 * h;
      float4 vg;
      if (cout == 32) {
        vg = *reinterpret_cast<const float4*>(st + GW_TILE + r * 128 + cq * 16);
      } else {
        const float* gp = reinterpret_cast<const float*>(st + GW_TILE) + r * cout;
        float t4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if ((int)(cq * 4 + e) < cout) t4[e] = gp[cq * 4 + e];
        vg = make_float4(t4[0], t4[1], t4[2], t4[3]);
      }
      if (a.bits) {
        const uint32_t w4 = reinterpret_cast<const uint32_t*>(st + (K + 2) * GW_TILE)[r] >> (cq * 4);
        vg.x = (w4 & 1u) ? vg.x * a.scale : 0.0f;
        vg.y = (w4 & 2u) ? vg.y * a.scale : 0.0f;
        vg.z = (w4 & 4u) ? vg.z * a.scale : 0.0f;
        vg.w = (w4 & 8u) ? vg.w * a.scale : 0.0f;
      }
      gb[0] += vg.x;
      gb[1] += vg.y;
      gb[2] += vg.z;
      gb[3] += vg.w;
      *reinterpret_cast<float4*>(g0 + r * 32 + cq * 4) = vg;
    }
    __syncthreads();   // g0 complete; every thread has left the main loop of the previous chunk -> its slot may be refilled
    if (tid == 0) issue(ch + (int64_t)(GWF_STAGES - 1) * gridDim.x, (it + GWF_STAGES - 1) % GWF_STAGES);
    const float* xs = reinterpret_cast<const float*>(st) + i_feat;
    const uint8_t* ks = reinterpret_cast<const uint8_t*>(st + (K + 2) * GW_TILE + 256);
#pragma unroll 4
    for (int r = 0; r < GW_ROWS; ++r) {
      const float xv = xs[r * 32];
      const uint32_t cl = (uint32_t)(c0 >> 2) ^ (lvl_key ? (uint32_t)ks[r] : 0u);
      const float4 l0 = *reinterpret_cast<const float4*>(g0 + r * 32 + c0);
      acc[0][0] = fmaf(l0.x, xv, acc[0][0]);
      acc[0][1] = fmaf(l0.y, xv, acc[0][1]);
      acc[0][2] = fmaf(l0.z, xv, acc[0][2]);
      acc[0][3] = fmaf(l0.w, xv, acc[0][3]);
#pragma unroll
      for (int k = 1; k <= K; ++k) {
        const float4 lk = *reinterpret_cast<const float4*>(st + (1 + k) * GW_TILE + r * 128 + (cl << 4));
        acc[k][0] = fmaf(lk.x, xv, acc[k][0]);
        acc[k][1] = fmaf(lk.y, xv, acc[k][1]);
        acc[k][2] = fmaf(lk.z, xv, acc[k][2]);
        acc[k][3] = fmaf(lk.w, xv, acc[k][3]);
      }
    }
  }
  // ---- this CTA's partial sums ----
  float* part = a.partials + (size_t)blockIdx.x * a.partial_stride;
#pragma unroll
  for (int k = 0; k <= K; ++k)
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (c0 + e < cout) part[((size_t)k * cout + c0 + e) * 32 + i_feat] = acc[k][e];
#pragma unroll
  for (int e = 0; e < 4; ++e) red[rs * 33 + cq * 4 + e] = gb[e];
  __syncthreads();
  if (tid < cout) {
    float sum = 0.0f;
    for (int r = 0; r < 32; ++r) sum += red[r * 33 + tid];
    part[a.bias_offset + tid] = sum;
  }
}

size_t tc2_smem(int K, int rw, bool ta) { return 1024 + (size_t)(K + 1) * 2 * W_TILE + (ta ? 2 : 4) * (size_t)rw * 32 * tc::ROW_BYTES + 256; }   // K = 2: 73 KB (3 CTAs/SM), 89 KB (2) or 153 KB
size_t gw_smem(int K) { return 1024 + 2 * gw_ops_bytes(K) + GW_STAGES * GW_STAGE_BYTES + 128; }   // 128: 14 mbarriers + TMEM slot

int tc2_supported(const dss2_graph_t* g, int K) {
  return g && g->num_tiles > 0 && g->max_tile_nodes <= T2_MAX && K >= 1 && K <= 2 && g->ell_w && g->ell_ci;
}

// DSS2_TC2_TA=0 selects the shared-memory A operand (the round-1 kernels) for A/B measurements
bool tc2_use_ta() {
  static const bool v = [] {
    const char* e = getenv("DSS2_TC2_TA");
    return !(e && e[0] == '0');
  }();
  return v;
}

template <int MODE, int K, int RW, bool DENSE, bool TA>
int launch_tc2_inst2(const Tc2Args& a, cudaStream_t stream) {
  using Shape = Tc2Shape<RW>;
  const size_t smem = tc2_smem(K, RW, TA);
  const int tiles = DENSE ? (int)((a.g.num_nodes + Shape::ROWS - 1) / Shape::ROWS) : a.g.num_tiles;
  const int per_sm = TA ? (Shape::NB == 1 ? 2 : 1) : Shape::CTAS_PER_SM;   // TA: 256 / 512 of the SM's 512 TMEM columns per CTA
  const int grid = max(1, min(tiles, per_sm * dss2_sm_count()));
  DSS2_CUDA(cudaFuncSetAttribute(k_tag_tc2<MODE, K, RW, DENSE, TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_tag_tc2<MODE, K, RW, DENSE, TA><<<grid, Shape::THREADS, smem, stream>>>(a);
  DSS2_LAUNCH_CHECK();
  return 0;
}
template <int MODE, int K, int RW, bool DENSE = false>
int launch_tc2_inst(const Tc2Args& a, cudaStream_t stream) {
  return tc2_use_ta() ? launch_tc2_inst2<MODE, K, RW, DENSE, true>(a, stream) : launch_tc2_inst2<MODE, K, RW, DENSE, false>(a, stream);
}
template <int MODE, int K>
int launch_tc2_k(const Tc2Args& a, cudaStream_t stream) {
  const int rows = a.g.max_tile_nodes;
  if (rows <= 96 && getenv("DSS2_TC2_RW3")) return launch_tc2_inst<MODE, K, 3>(a, stream);
  if (rows <= 128) return launch_tc2_inst<MODE, K, 4>(a, stream);
  return launch_tc2_inst<MODE, K, 8>(a, stream);
}
template <int MODE>
int launch_tc2(const Tc2Args& a_in, int K, cudaStream_t stream) {
  Tc2Args a = a_in;
  static const int flags = [] { const char* e = getenv("DSS2_TC2_FLAGS"); return e ? atoi(e) : 0; }();
  a.flags = flags;
  return K == 1 ? launch_tc2_k<MODE, 1>(a, stream) : launch_tc2_k<MODE, 2>(a, stream);
}

}  // namespace

extern "C" int dss2_tag_tc2_supported(const dss2_graph_t* g, int K) { return tc2_supported(g, K); }

#ifdef DSS2_STAMPS
// diagnostic build: read (and clear) the phase counters
extern "C" int dss2_tc2_stamps(unsigned long long* host_out) {
  unsigned long long zero[32] = {};
  if (cudaMemcpyFromSymbol(host_out, g_tc2_stamps, sizeof(zero)) != cudaSuccess) return -1;
  if (cudaMemcpyToSymbol(g_tc2_stamps, zero, sizeof(zero)) != cudaSuccess) return -1;
  return 0;
}
#endif

// Large-graph path (tag.cu): the transform of a layer on hop levels that already sit in global memory (lvl = [K][Nt,32], levels 1..K),
// through the same tcgen05 kernel with plain 256-row tiles and the hop stage replaced by loads.  K in 1..2.
int dss2_tc2_dense_fwd(const dss2_graph_t* g, const float* x, const float* lvl, const float* w, const float* bias, int cout, int K, int act,
                       float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid, const uint8_t* mask, const float* res,
                       int64_t res_stride, float* y, uint32_t* act_bits, cudaStream_t stream) {
  Tc2Args a = {};
  a.g = *g;
  a.in = x;
  a.dense_lvl = lvl;
  a.w = w;
  a.bias = bias;
  a.cout = cout;
  a.act = act;
  if (p_drop == 0.0f) drop_mode = 0;
  a.drop_mode = act ? drop_mode : 0;
  a.scale = 1.0f / (float)(1.0 - (double)p_drop);
  double thr = (1.0 - (double)p_drop) * 65536.0 + 0.5;
  a.keep_thr16 = thr >= 65536.0 ? 65536u : (uint32_t)thr;
  a.rng = rng_state;
  a.layer_uid = layer_uid;
  a.mask = mask;
  a.res = res;
  a.res_stride = res_stride;
  a.out = y;
  a.out_bits = act_bits;
  return K == 1 ? launch_tc2_inst<MODE_FWD, 1, 8, true>(a, stream) : launch_tc2_inst<MODE_FWD, 2, 8, true>(a, stream);
}
int dss2_tc2_dense_bgx(const dss2_graph_t* g, const float* grad_y, const uint32_t* act_bits, float p_drop, const float* lvl, const float* w,
                       int cout, int K, float* grad_x, cudaStream_t stream) {
  Tc2Args a = {};
  a.g = *g;
  a.in = grad_y;        // [Nt,cout]; level 0 = grad_y * [y>0]/(1-p) is formed while loading, exactly as in the tiled backward
  a.in_bits = act_bits;
  a.dense_lvl = lvl;    // levels 1..K of that masked gradient (hop kernels)
  a.w = w;
  a.cout = cout;
  a.scale = 1.0f / (float)(1.0 - (double)p_drop);
  a.out = grad_x;
  return K == 1 ? launch_tc2_inst<MODE_BGX, 1, 8, true>(a, stream) : launch_tc2_inst<MODE_BGX, 2, 8, true>(a, stream);
}

// every tile of a launch that did not go through the chained kernel is complete at its end: mark them all
__global__ void k_fill_marks(uint32_t* marks, int n, const uint64_t* seq) {
  const uint32_t v = (uint32_t)seq[1] + 1u;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) marks[i] = v;
}

extern "C" int dss2_tag_fwd_tc2_chain(const dss2_graph_t* g, const float* x, const float* w, const float* bias, int cout, int K, int act,
                                      float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid, const uint8_t* mask,
                                      const float* res, int64_t res_stride, float* y, uint32_t* act_bits, uint32_t* done_flags,
                                      const uint32_t* wait_flags, void* stream_);
extern "C" int dss2_tag_fwd_tc2(const dss2_graph_t* g, const float* x, const float* w, const float* bias, int cout, int K, int act,
                                float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid, const uint8_t* mask,
                                const float* res, int64_t res_stride, float* y, uint32_t* act_bits, void* stream_) {
  return dss2_tag_fwd_tc2_chain(g, x, w, bias, cout, K, act, p_drop, drop_mode, rng_state, layer_uid, mask, res, res_stride, y, act_bits, nullptr,
                                nullptr, stream_);
}

// Chained variant for a stack of layers inside one captured step (see Tc2Args): done_flags [num_tiles] receives this launch's per-tile
// completion marks, wait_flags = the done_flags of the launch that produced x.  Either may be NULL.  Both need rng_state (the device
// {seed, step} pair: the marks carry step + 1, so a replayed graph needs no reset).  When the TMA-fed kernel cannot serve the shape the
// flags are ignored and the launch is an ordinary one (correct, just not overlapped) - then done_flags is filled by a plain kernel.
extern "C" int dss2_tag_fwd_tc2_chain(const dss2_graph_t* g, const float* x, const float* w, const float* bias, int cout, int K, int act,
                                      float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid, const uint8_t* mask,
                                      const float* res, int64_t res_stride, float* y, uint32_t* act_bits, uint32_t* done_flags,
                                      const uint32_t* wait_flags, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(!(done_flags || wait_flags) || rng_state, "dss2_tag_fwd_tc2_chain: the tile marks need rng_state (device {seed, step})");
  DSS2_CHECK_ARG(g && x && w && bias && y, "dss2_tag_fwd_tc2: null argument");
  DSS2_CHECK_ARG(cout >= 1 && cout <= HID, "dss2_tag_fwd_tc2: cout %d outside 1..%d", cout, HID);
  DSS2_CHECK_ARG(tc2_supported(g, K), "dss2_tag_fwd_tc2: needs a tiled graph (tile_cap <= 256) and K in 1..2");
  DSS2_CHECK_ARG(p_drop >= 0.0f && p_drop < 1.0f, "dss2_tag_fwd_tc2: dropout p %f outside [0,1)", p_drop);
  DSS2_CHECK_ARG(!(act && drop_mode == 1) || rng_state, "dss2_tag_fwd_tc2: philox dropout needs rng_state");
  DSS2_CHECK_ARG(!(act && drop_mode == 2) || mask, "dss2_tag_fwd_tc2: mask dropout needs a mask");
  if (g->num_nodes == 0) return 0;
  Tc2Args a = {};
  a.g = *g;
  a.in = x;
  a.w = w;
  a.bias = bias;
  a.cout = cout;
  a.act = act;
  if (p_drop == 0.0f) drop_mode = 0;
  a.drop_mode = act ? drop_mode : 0;
  a.scale = 1.0f / (float)(1.0 - (double)p_drop);
  double thr = (1.0 - (double)p_drop) * 65536.0 + 0.5;
  a.keep_thr16 = thr >= 65536.0 ? 65536u : (uint32_t)thr;
  a.rng = rng_state;
  a.layer_uid = layer_uid;
  a.mask = mask;
  a.res = res;
  a.res_stride = res_stride;
  a.out = y;
  a.out_bits = act_bits;
  a.done_flags = done_flags;
  a.wait_flags = wait_flags;
  a.chain_seq = rng_state;
  const int rc3 = dss2_tc3_launch(MODE_FWD, a, K, stream);   // the TMA-fed kernel when it serves the shape
  if (rc3 <= 0) return rc3;
  a.done_flags = nullptr;
  a.wait_flags = nullptr;
  const int rc2 = launch_tc2<MODE_FWD>(a, K, stream);        // ordinary launch: ordered after the producer, complete before any consumer
  if (rc2 == 0 && done_flags) {
    k_fill_marks<<<max(1, min(g->num_tiles, 1024) / 256 + 1), 256, 0, stream>>>(done_flags, g->num_tiles, rng_state);
    DSS2_LAUNCH_CHECK();
  }
  return rc2;
}

extern "C" size_t dss2_tag_bwd_tc2_workspace_bytes(int64_t num_nodes, int K) { return (size_t)K * num_nodes * HID * sizeof(float) + 256; }

// the two halves of the backward, individually launchable (bench.py times them separately; dss2_tag_bwd_tc2 = both)
extern "C" int dss2_tag_bwd_tc2_gx_chain(const dss2_graph_t* g, const float* w, int cout, int K, int act, float p_drop, const uint32_t* act_bits,
                                         const float* grad_y, float* grad_x, void* ws, size_t ws_bytes, const uint64_t* rng_state,
                                         uint32_t* done_flags, const uint32_t* wait_flags, void* stream_);
extern "C" int dss2_tag_bwd_tc2_gx(const dss2_graph_t* g, const float* w, int cout, int K, int act, float p_drop, const uint32_t* act_bits,
                                   const float* grad_y, float* grad_x, void* ws, size_t ws_bytes, void* stream_) {
  return dss2_tag_bwd_tc2_gx_chain(g, w, cout, K, act, p_drop, act_bits, grad_y, grad_x, ws, ws_bytes, nullptr, nullptr, nullptr, stream_);
}

// Chained variant (see dss2_tag_fwd_tc2_chain): the backward-to-input of layer l-1 needs only the same tile of layer l's grad_x, so a
// stack of these launches links per tile.  The weight-gradient pass of a layer (dss2_tag_bwd_tc2_gw) needs the WHOLE launch (it streams
// 64-row chunks across tiles and reads the spilled levels): run it behind an event on a second stream with its own workspace per layer.
extern "C" int dss2_tag_bwd_tc2_gx_chain(const dss2_graph_t* g, const float* w, int cout, int K, int act, float p_drop, const uint32_t* act_bits,
                                         const float* grad_y, float* grad_x, void* ws, size_t ws_bytes, const uint64_t* rng_state,
                                         uint32_t* done_flags, const uint32_t* wait_flags, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(!(done_flags || wait_flags) || rng_state, "dss2_tag_bwd_tc2_gx_chain: the tile marks need rng_state (device {seed, step})");
  DSS2_CHECK_ARG(g && w && grad_y && grad_x && ws, "dss2_tag_bwd_tc2_gx: null argument");
  DSS2_CHECK_ARG(cout >= 1 && cout <= HID, "dss2_tag_bwd_tc2_gx: cout %d outside 1..%d", cout, HID);
  DSS2_CHECK_ARG(tc2_supported(g, K), "dss2_tag_bwd_tc2_gx: needs a tiled graph (tile_cap <= 256) and K in 1..2");
  DSS2_CHECK_ARG(!act || act_bits, "dss2_tag_bwd_tc2_gx: activation layers need act_bits from the forward");
  DSS2_CHECK_ARG(ws_bytes >= dss2_tag_bwd_tc2_workspace_bytes(g->num_nodes, K), "dss2_tag_bwd_tc2_gx: workspace too small");
  DSS2_CHECK_ARG((((uintptr_t)grad_y | (uintptr_t)ws | (uintptr_t)grad_x) & 15) == 0, "dss2_tag_bwd_tc2_gx: pointers must be 16-byte aligned");
  if (g->num_nodes == 0) return 0;
  Tc2Args a = {};
  a.g = *g;
  a.in = grad_y;
  a.in_bits = act ? act_bits : nullptr;
  a.w = w;
  a.cout = cout;
  a.scale = 1.0f / (float)(1.0 - (double)p_drop);
  a.out = grad_x;
  a.lvl_out = (float*)ws;
  a.done_flags = done_flags;
  a.wait_flags = wait_flags;
  a.chain_seq = rng_state;
  const int rc3 = dss2_tc3_launch(MODE_BGX, a, K, stream);
  if (rc3 <= 0) return rc3;
  a.done_flags = nullptr;
  a.wait_flags = nullptr;
  const int rc2 = launch_tc2<MODE_BGX>(a, K, stream);
  if (rc2 == 0 && done_flags) {
    k_fill_marks<<<max(1, min(g->num_tiles, 1024) / 256 + 1), 256, 0, stream>>>(done_flags, g->num_tiles, rng_state);
    DSS2_LAUNCH_CHECK();
  }
  return rc2;
}

extern "C" int dss2_tag_bwd_tc2_gw(int64_t num_nodes, const float* x, int cout, int K, int act, float p_drop, const uint32_t* act_bits,
                                   const float* grad_y, float* partials, int64_t partial_stride, int64_t bias_offset, const void* ws,
                                   size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x && grad_y && partials && ws, "dss2_tag_bwd_tc2_gw: null argument");
  DSS2_CHECK_ARG(cout >= 1 && cout <= HID && K >= 1 && K <= 2, "dss2_tag_bwd_tc2_gw: cout %d / K %d unsupported", cout, K);
  DSS2_CHECK_ARG(!act || act_bits, "dss2_tag_bwd_tc2_gw: activation layers need act_bits from the forward");
  DSS2_CHECK_ARG(ws_bytes >= dss2_tag_bwd_tc2_workspace_bytes(num_nodes, K), "dss2_tag_bwd_tc2_gw: workspace too small");
  DSS2_CHECK_ARG(partial_stride >= (int64_t)(K + 1) * cout * HID + cout, "dss2_tag_bwd_tc2_gw: partial_stride too small");
  DSS2_CHECK_ARG((((uintptr_t)x | (uintptr_t)grad_y | (uintptr_t)ws | (uintptr_t)act_bits | (uintptr_t)partials) & 15) == 0,
                 "dss2_tag_bwd_tc2_gw: x, grad_y, act_bits, partials and ws must be 16-byte aligned (bulk-copy sources / 128-bit stores)");
  if (num_nodes == 0) return 0;
  GwArgs b;
  b.num_nodes = num_nodes;
  b.x = x;
  b.gy = grad_y;
  b.bits = act ? act_bits : nullptr;
  b.lvl = (const float*)ws;
  b.lvl_fmt = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(ws) + (size_t)K * num_nodes * HID * sizeof(float));
  b.cout = cout;
  b.scale = 1.0f / (float)(1.0 - (double)p_drop);
  b.partials = partials;
  b.partial_stride = partial_stride;
  b.bias_offset = bias_offset;
  const size_t smem = gw_smem(K);
  const int grid = dss2_sm_count();    // = dss2_num_partials(): every partial row is written
  if (K == 1) {
    DSS2_CUDA(cudaFuncSetAttribute(k_tag_gw<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_tag_gw<1><<<grid, GW_THREADS, smem, stream>>>(b);
  } else {
    DSS2_CUDA(cudaFuncSetAttribute(k_tag_gw<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_tag_gw<2><<<grid, GW_THREADS, smem, stream>>>(b);
  }
  DSS2_LAUNCH_CHECK();
  return 0;
}

// exact fp32 variant of the weight-gradient pass (CUDA cores); same contract, K up to 3
extern "C" int dss2_tag_gw_ffma(int64_t num_nodes, const float* x, int cout, int K, int act, float p_drop, const uint32_t* act_bits,
                                const float* grad_y, float* partials, int64_t partial_stride, int64_t bias_offset, const void* ws,
                                size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(x && grad_y && partials && ws, "dss2_tag_gw_ffma: null argument");
  DSS2_CHECK_ARG(cout >= 1 && cout <= HID && K >= 1 && K <= 3, "dss2_tag_gw_ffma: cout %d / K %d unsupported", cout, K);
  DSS2_CHECK_ARG(!act || act_bits, "dss2_tag_gw_ffma: activation layers need act_bits from the forward");
  DSS2_CHECK_ARG(ws_bytes >= dss2_tag_bwd_tc2_workspace_bytes(num_nodes, K), "dss2_tag_gw_ffma: workspace too small");
  DSS2_CHECK_ARG(partial_stride >= (int64_t)(K + 1) * cout * HID + cout, "dss2_tag_gw_ffma: partial_stride too small");
  DSS2_CHECK_ARG((((uintptr_t)x | (uintptr_t)grad_y | (uintptr_t)ws | (uintptr_t)act_bits) & 15) == 0 && (num_nodes * HID * 4) % 16 == 0,
                 "dss2_tag_gw_ffma: x, grad_y, act_bits and ws must be 16-byte aligned (bulk-copy sources)");
  if (num_nodes == 0) return 0;
  GwArgs b;
  b.num_nodes = num_nodes;
  b.x = x;
  b.gy = grad_y;
  b.bits = act ? act_bits : nullptr;
  b.lvl = (const float*)ws;
  b.lvl_fmt = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(ws) + (size_t)K * num_nodes * HID * sizeof(float));
  b.cout = cout;
  b.scale = 1.0f / (float)(1.0 - (double)p_drop);
  b.partials = partials;
  b.partial_stride = partial_stride;
  b.bias_offset = bias_offset;
  const int grid = dss2_sm_count();    // = dss2_num_partials(): every partial row is written
#define DSS2_GWF(KK)                                                                                                     \
  {                                                                                                                      \
    DSS2_CUDA(cudaFuncSetAttribute(k_tag_gw_ffma<KK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gwf_smem<KK>())); \
    k_tag_gw_ffma<KK><<<grid, GWF_THREADS, gwf_smem<KK>(), stream>>>(b);                                                 \
  }
  if (K == 1) DSS2_GWF(1) else if (K == 2) DSS2_GWF(2) else DSS2_GWF(3)
#undef DSS2_GWF
  DSS2_LAUNCH_CHECK();
  return 0;
}

extern "C" int dss2_tag_bwd_tc2(const dss2_graph_t* g, const float* x, const float* w, int cout, int K, int act, float p_drop,
                                const uint32_t* act_bits, const float* grad_y, float* grad_x, float* partials, int64_t partial_stride,
                                int64_t bias_offset, void* ws, size_t ws_bytes, void* stream_) {
  DSS2_CHECK_ARG(g, "dss2_tag_bwd_tc2: null graph");
  int rc = dss2_tag_bwd_tc2_gx(g, w, cout, K, act, p_drop, act_bits, grad_y, grad_x, ws, ws_bytes, stream_);
  if (rc) return rc;
  return dss2_tag_bwd_tc2_gw(g->num_nodes, x, cout, K, act, p_drop, act_bits, grad_y, partials, partial_stride, bias_offset, ws, ws_bytes, stream_);
}
