/*
 * dss2_b200.h - C ABI of the B200-native DSS2 hot path (libdss2_b200.so).
 *
 * The reference (TU-Delft-AI-Energy-Lab/Deep-Statistical-Solver-for-Distribution-System-State-Estimation)
 * is pure Python and has no FFI; its hot path is reached through the Python surface that
 * dss2_run.py touches (SURVEY.md 8b).  This header is the boundary the Python host mirror
 * (`networks.py`, `data.py` in the package directory) binds with ctypes; every entry point names the
 * reference code it replaces.  See INTEGRATION.md for the reference-side binding.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer owned by the caller unless it is marked
 *     "host"; kernels never allocate or free; all work is enqueued on `stream` (a cudaStream_t passed
 *     as void*) and is safe to capture in a CUDA graph unless stated otherwise;
 *   - return value 0 = success, negative = error (dss2_last_error() gives the thread-local message);
 *   - fp32 features, int64 indices at the API (as PyG), int32 kernel-private CSR;
 *   - hidden width is 32 (one warp lane per hidden feature); other widths are rejected loudly.
 */
#ifndef DSS2_B200_H
#define DSS2_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSS2_HID 32            /* hidden width the layer kernels are specialised for */
#define DSS2_TILE_CAP 256      /* max nodes of a shared-memory tile (whole graphs) */

const char* dss2_last_error(void);
int dss2_version(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches claim) */
int64_t dss2_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Graph structure of one batch (kernel-private; built once per batch topology).
 * Replaces: MPN.is_directed / undirect_graph (networks.py:236-258, redone in each of the 5 sub-nets),
 *           PyG gcn_norm inside every TAGConv.forward (recomputed 40x per forward),
 *           PyG degree (networks.py:197, dead).
 * The doubled graph (forward edges then reversed edges, networks.py:245-248) is stored as CSR by
 * destination; within a row entries are ordered by doubled edge id, i.e. the order in which PyG's
 * sequential scatter_add_ visits them.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dss2_graph {
  int64_t num_nodes;        /* Nt */
  int64_t num_edges;        /* Et one-way edges as given at the API */
  int64_t nnz;              /* CSR entries: 2*Et if reversed edges were appended, else Et */
  int32_t num_graphs;       /* B segments (graphs) */
  int32_t undirected;       /* 1: reversed edges appended (input was one-way) */
  int32_t graphs_per_tile;  /* G; 0 = no shared-memory tiling possible (graph larger than a tile) */
  int32_t num_tiles;
  int32_t max_tile_nodes;
  int32_t max_tile_nnz;
  int32_t max_tile_edges;   /* one-way edges */
  int32_t hop_keys;         /* swizzle-key policy the build used (DSS2_HOP_KEYS_*) */
  const int64_t* edge_index;/* [2,Et] caller's tensor */
  const int64_t* ptr;       /* [B+1] node offset of every graph (caller's or builder's) */
  int64_t* eptr;            /* [B+1] one-way edge offset of every graph */
  int32_t* rowptr;          /* [Nt+1] */
  int32_t* col;             /* [nnz] source node */
  uint32_t* eid;            /* [nnz] original edge id | reversed << 31 */
  float* dis;               /* [Nt] in-degree^-1/2 on the doubled graph, 0 where degree is 0 */
  float* w;                 /* [nnz] gcn_norm weight of the entry: dis[src] * dis[dst] */
  float* ell_w;             /* [Nt][4] weights of the first 4 entries of every row (0 = padding): thread-per-row kernels */
  uint32_t* ell_ci;         /* [Nt][2] .x = 4 x 8-bit tile-local source rows of those entries, .y = row degree (saturated at
                               DSS2_ELL_DEG_MASK) | swizzle keys of the row and of its 4 ELL sources (DSS2_ELL_KEY_SHIFT) */
  float* scratch;           /* caller-provided, only needed when num_tiles == 0 (a graph exceeds a tile): */
  size_t scratch_bytes;     /*   dss2_generic_scratch_bytes(Nt) bytes of device memory for the large-graph kernels */
  uint8_t* hop_key;         /* [Nt] swizzle key (0..7) of every row of a tiled graph */
} dss2_graph_t;

/* Swizzle keys.  The TAG layer kernels keep each hop level of a tile in shared memory as 128-byte rows, with 16-byte chunk c of
 * row n stored at chunk c ^ key[n].  Eight consecutive tile rows form one phase of a 128-bit shared-memory access, so rows whose
 * keys differ never share banks.  IDENTITY: key = n & 7 (consecutive rows differ).  COLOR: keys chosen per tile at graph build so
 * that the rows gathered together by one phase (the slot-d ELL sources of 8 consecutive rows) differ as well.  The keys move
 * bytes only: every sum, and so every result, is the same under both policies. */
#define DSS2_HOP_KEYS_IDENTITY 0
#define DSS2_HOP_KEYS_COLOR 1
#define DSS2_ELL_DEG_MASK 0x1ffffu   /* ell_ci[n].y bits 0..16: degree; 17..19: key of n; 20 + 3d..22 + 3d: key of ELL source d */
#define DSS2_ELL_KEY_SHIFT 17

/* Large graphs (a graph with more nodes than a tile, e.g. a 10k-bus feeder): num_tiles == 0 after the build and every layer /
 * loss entry point switches to its global-memory variant (hops as separate SpMM launches, row-streaming transforms, node-centric
 * loss passes).  Those need scratch: set g->scratch / g->scratch_bytes to a device buffer of this many bytes. */
size_t dss2_generic_scratch_bytes(int64_t num_nodes);

/* Bytes of device workspace dss2_graph_build needs for (Nt, Et, B). */
size_t dss2_graph_workspace_bytes(int64_t num_nodes, int64_t num_edges, int32_t num_graphs);

/* Builds the structure into `g` (host struct).  `ws` must stay alive as long as `g` is used: all
 * arrays of `g` except edge_index/ptr point into it.  undirect: 1 append reversed edges, 0 do not,
 * -1 decide like MPN.is_directed (networks.py:236-238).  tile_cap: max nodes per tile (<= DSS2_TILE_CAP).
 * hop_keys: DSS2_HOP_KEYS_IDENTITY or DSS2_HOP_KEYS_COLOR.
 * Synchronises `stream` (reads sizes back); not graph-capturable. */
int dss2_graph_build(dss2_graph_t* g, const int64_t* edge_index, int64_t num_edges, int64_t num_nodes,
                     const int64_t* ptr, int32_t num_graphs, int undirect, int tile_cap, int hop_keys,
                     void* ws, size_t ws_bytes, void* stream);

/* The keys dss2_graph_build assigns, computed on the host (tests, tools/hop_conflicts.py).  All pointers are HOST pointers:
 * ell_ci [Nt][2] = the ELL words with the plain degree in .y, tile_ptr [num_tiles+1] = first row of every tile; keys [Nt] out. */
int dss2_hop_keys_host(const uint32_t* ell_ci, const int64_t* tile_ptr, int32_t num_tiles, int hop_keys, uint8_t* keys);

/* ------------------------------------------------------------------------------------------------
 * (a) Batch packer.  Replaces PyG DataLoader -> Batch.from_data_list (dss2_run.py:18,68-69,134).
 * Scenario-major store: scenario s owns node rows node_off[s]..node_off[s+1] of x_all[.,11] / y_all[.,2]
 * and edge rows edge_off[s]..edge_off[s+1] of ea_all[.,13] / columns of ei_all[2,E_all] (local ids).
 * Output is PyG's disjoint-union batch, bit-exact: x, edge_index (+node offset), edge_attr, y,
 * batch, ptr, plus eptr (edge offsets) and vminmax = {min, max} of vn_kv = x[:,8] (data.py:334-336).
 * Any of y/batch may be NULL.  ptr/eptr ([B+1]) are produced by an on-device scan of the selected sizes.
 * ---------------------------------------------------------------------------------------------- */
int dss2_pack_batch(const float* x_all, const float* ea_all, const float* y_all, const int64_t* ei_all,
                    int64_t ei_all_cols, const int64_t* node_off, const int64_t* edge_off,
                    const int64_t* scen_ids, int32_t num_graphs,
                    float* x, int64_t* edge_index, int64_t edge_index_cols, float* edge_attr, float* y,
                    int64_t* batch, int64_t* ptr, int64_t* eptr, float* vminmax, void* stream);

/* vminmax[0] = min, [1] = max of column `col` of x (row stride `stride` floats). */
int dss2_col_minmax(const float* x, int64_t stride, int col, int64_t n, float* vminmax, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (b1) EdgeAggregation.  Replaces networks.py:159-209 (+ its autograd):
 *   out[n] = sum_{e: dst(e)=n} ( W2 relu(W1 [x_n | x_src(e) | a_e] + b1) + b2 )   on the doubled graph,
 * reversed edges using a_e with columns 0 and 2 negated (networks.py:252).
 * x: [Nt, fn] with row stride x_stride floats (fn <= 8); edge_attr: [Et, fe] row stride ea_stride (fe <= 8).
 * w1 [32, 2*fn+fe], b1 [32], w2 [32,32], b2 [32] row-major as torch Linear.  out [Nt,32].
 * ---------------------------------------------------------------------------------------------- */
int dss2_edgeagg_fwd(const dss2_graph_t* g, const float* x, int64_t x_stride, int fn,
                     const float* edge_attr, int64_t ea_stride, int fe,
                     const float* w1, const float* b1, const float* w2, const float* b2,
                     float* out, void* stream);

/* Backward.  grad_out [Nt,32].  grad_x [Nt,fn] (dense, stride fn) may be NULL; if `skip_grad`
 * (row stride skip_stride) is given it is added into grad_x (the SkipMPN residual path, networks.py:336).
 * Weight gradients are written as per-CTA partial sums: partials[cta][edgeagg_param_count] with
 * layout (w1, b1, w2, b2); *num_partials CTAs were used.  Reduce with dss2_reduce_partials. */
int dss2_edgeagg_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, int fn,
                     const float* edge_attr, int64_t ea_stride, int fe,
                     const float* w1, const float* b1, const float* w2, const float* b2,
                     const float* grad_out, const float* skip_grad, int64_t skip_stride,
                     float* grad_x, float* partials, int64_t partial_stride, void* stream);

/* Prepared-weights variant of (b1) for a captured step: the thread-per-row kernels (csrc/edgeagg_row.cu) read the two Linears from
 * constant memory.  dss2_edgeagg_upload writes the weights of n modules (host arrays of n device pointers each) into slots
 * slot0 .. slot0+n-1 (0..6) with one layout kernel and one device-to-device copy node; the _slot entry points then take a slot instead of
 * the four weight pointers (same contracts as dss2_edgeagg_fwd / dss2_edgeagg_bwd).  dss2_edgeagg_slots_ok != 0 when the batch structure,
 * strides (<= 16 floats) and fe (<= 6) fit those kernels; otherwise use the pointer API, which picks the kernel itself (and routes through
 * a scratch slot when it can).  A slot's contents stay valid until the next upload into it. */
int dss2_edgeagg_slots_ok(const dss2_graph_t* g, int64_t x_stride, int64_t ea_stride, int fe);
int dss2_edgeagg_upload(int slot0, int n, const float* const* w1, const float* const* b1, const float* const* w2,
                        const float* const* b2, int fn, int fe, void* stream);
int dss2_edgeagg_fwd_slot(const dss2_graph_t* g, const float* x, int64_t x_stride, int fn, const float* edge_attr,
                          int64_t ea_stride, int fe, int slot, float* out, void* stream);
int dss2_edgeagg_bwd_slot(const dss2_graph_t* g, const float* x, int64_t x_stride, int fn, const float* edge_attr,
                          int64_t ea_stride, int fe, int slot, const float* grad_out, const float* skip_grad,
                          int64_t skip_stride, float* grad_x, float* partials, int64_t partial_stride, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (b2) TAGConv(32 -> cout, K) [+ Dropout + ReLU] [+ residual].  Replaces PyG TAGConv.forward with
 * gcn_norm(add_self_loops=False) and the inline Dropout/ReLU of networks.py:268-269 (+ autograd):
 *   out = sum_{k=0..K} (A_hat^k x) W_k^T + b ;  y = relu(dropout_p(out)) if act else out ; y += res
 * w: K+1 matrices [cout,32] contiguous ([K+1,cout,32]); bias [cout]; y [Nt,cout].
 * Dropout: mode 0 none; 1 counter-based Philox keyed by (seed, layer_uid, node, feature) with the
 * seed/step pair read from DEVICE memory rng_state[2] (graph-replay safe); 2 caller-supplied mask
 * (uint8 [Nt,32], 1 = keep) for exact parity with a recorded torch mask.
 * act_bits [Nt] (out, may be NULL when !act): bit c = y[n][c] > 0, all the backward needs.
 * res: optional [Nt,cout] residual input with row stride res_stride (SkipMPN, networks.py:336).
 * ---------------------------------------------------------------------------------------------- */
int dss2_tag_fwd(const dss2_graph_t* g, const float* x, const float* w, const float* bias, int cout, int K,
                 int act, float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid,
                 const uint8_t* mask, const float* res, int64_t res_stride,
                 float* y, uint32_t* act_bits, void* stream);

/* Tensor-core layer kernels: the (K+1) 32x32 transforms on tcgen05 (kind::tf32, 3xTF32 split = fp32-equivalent accuracy, accumulators in
 * TMEM), thread = (row, half row), A operand in tensor memory; tiled graphs with
 * tile_cap <= 256 and K <= 2).  Forward: same contract as dss2_tag_fwd.  Backward: same contract as dss2_tag_bwd plus a workspace of
 * dss2_tag_bwd_tc2_workspace_bytes() for the hop levels of the masked output gradient; it runs the backward-to-input as the forward
 * kernel with transposed weights (grad_x = sum_k (A^k g) W_k) and the weight gradients as one streaming MN-major GEMM
 * (grad_W_k = (A^k g)^T x), with no hop recomputation on x.  When every pointer is 16-byte aligned the entry points launch the
 * TMA-fed kernel k_tag_tc3 (inputs by cp.async.bulk[.tensor], hop levels spilled by bulk store; the forward for any cout, the
 * backward-to-input for cout == 32), else k_tag_tc2 with direct loads (DSS2_TC3=0 forces that).  Contract details of the TMA path:
 * act_bits buffers hold (num_nodes + 3) & ~3 words (the sign words of a tile are copied from a 16-byte aligned start);
 * the last 256 bytes of the backward workspace carry a format word written by _gx and read by _gw / dss2_tag_gw_ffma (0 = plain
 * level rows, 1 = rows whose 16-byte chunk c is stored at chunk c ^ g->hop_key[row], followed by that key array's address):
 * pass the SAME workspace to both, while the graph is alive. */
int dss2_tag_tc2_supported(const dss2_graph_t* g, int K);
int dss2_tag_fwd_tc2(const dss2_graph_t* g, const float* x, const float* w, const float* bias, int cout, int K,
                     int act, float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid,
                     const uint8_t* mask, const float* res, int64_t res_stride,
                     float* y, uint32_t* act_bits, void* stream);
/* Chained variant for a stack of layers inside one step: a tile of layer l+1 needs only the SAME tile of layer l (message passing never
 * leaves a tile), so the launches are linked per tile instead of per grid.  done_flags [num_tiles] (u32) receives step+1 for every tile
 * whose outputs are in global memory; wait_flags = the done_flags of the launch that produced x: this launch then starts (programmatic
 * stream serialization, no grid-wide wait) on the SMs the producer's CTAs leave and reads a tile once its mark carries this step's number.
 * rng_state (device {seed, step}) supplies the step; marks need no reset between steps.  Either pointer may be NULL. */
int dss2_tag_fwd_tc2_chain(const dss2_graph_t* g, const float* x, const float* w, const float* bias, int cout, int K,
                           int act, float p_drop, int drop_mode, const uint64_t* rng_state, uint32_t layer_uid,
                           const uint8_t* mask, const float* res, int64_t res_stride, float* y, uint32_t* act_bits,
                           uint32_t* done_flags, const uint32_t* wait_flags, void* stream);
/* The same for a stack of backward-to-input launches (dss2_tag_bwd_tc2_gx): layer l-1 needs only the same tile of layer l's grad_x.  The
 * weight-gradient pass of a layer (dss2_tag_bwd_tc2_gw) needs the whole launch: run it behind an event on a second stream, with a
 * workspace per layer (it then fills the SMs the chained launches leave idle). */
int dss2_tag_bwd_tc2_gx_chain(const dss2_graph_t* g, const float* w, int cout, int K, int act, float p_drop,
                              const uint32_t* act_bits, const float* grad_y, float* grad_x, void* ws, size_t ws_bytes,
                              const uint64_t* rng_state, uint32_t* done_flags, const uint32_t* wait_flags, void* stream);
size_t dss2_tag_bwd_tc2_workspace_bytes(int64_t num_nodes, int K);
int dss2_tag_bwd_tc2(const dss2_graph_t* g, const float* x, const float* w, int cout, int K,
                     int act, float p_drop, const uint32_t* act_bits, const float* grad_y,
                     float* grad_x, float* partials, int64_t partial_stride, int64_t bias_offset,
                     void* ws, size_t ws_bytes, void* stream);
/* Its two launches on their own: _gx writes grad_x and the hop levels of the masked output gradient into ws; _gw consumes x,
 * grad_y (+act_bits) and ws and writes the per-CTA partial sums of grad_W / grad_b. */
int dss2_tag_bwd_tc2_gx(const dss2_graph_t* g, const float* w, int cout, int K, int act, float p_drop,
                        const uint32_t* act_bits, const float* grad_y, float* grad_x, void* ws, size_t ws_bytes, void* stream);
int dss2_tag_bwd_tc2_gw(int64_t num_nodes, const float* x, int cout, int K, int act, float p_drop,
                        const uint32_t* act_bits, const float* grad_y, float* partials, int64_t partial_stride,
                        int64_t bias_offset, const void* ws, size_t ws_bytes, void* stream);
/* The weight-gradient pass of dss2_tag_bwd_tc2_gw in exact fp32 on the CUDA cores (bulk-copy ring + FFMA, K <= 3): same arguments,
 * same partial layout.  It is a pure streaming pass, and ncu / CUDA events decide which of the two the host uses (DESIGN.md 4). */
int dss2_tag_gw_ffma(int64_t num_nodes, const float* x, int cout, int K, int act, float p_drop, const uint32_t* act_bits,
                     const float* grad_y, float* partials, int64_t partial_stride, int64_t bias_offset, const void* ws,
                     size_t ws_bytes, void* stream);
/* D[128,32] = A[128,32] * B[32,32]^T through the tensor-core operand / descriptor / TMEM path (bring-up and regression test). */
int dss2_tc_selftest(const float* A, const float* B, float* D, void* stream);
/* D[32*t + j, n] = sum_r A[t][r][j] * B[r][n], A = [4,64,32], B = [64,32]: MN-major TF32 operands (SWIZZLE_128B_BASE32B), the
 * weight-gradient GEMM shape (contraction over node rows). */
int dss2_tc_selftest_mn(const float* A, const float* B, float* D, void* stream);

/* Backward with recomputation of A_hat^k x from the saved layer input x.
 * grad_y [Nt,cout]; act_bits as written by the forward (NULL when !act); grad_x [Nt,32].
 * Per-CTA partial sums: row c of the partials buffer starts at partials + c*partial_stride; grad_W
 * ([K+1,cout,32]) is written at offset 0 of the row and grad_bias ([cout]) at offset `bias_offset`
 * (signed: in the flat parameter layout the bias precedes the weights). */
int dss2_tag_bwd(const dss2_graph_t* g, const float* x, const float* w, int cout, int K,
                 int act, float p_drop, const uint32_t* act_bits, const float* grad_y,
                 float* grad_x, float* partials, int64_t partial_stride, int64_t bias_offset,
                 void* stream);

/* Number of CTAs (= rows of a partials buffer) the layer backward kernels use on this device. */
int dss2_num_partials(void);

/* grad[i] = sum_{c < num_partials} partials[c*partial_stride + i], i < count; deterministic order.
 * accumulate != 0 adds into grad instead of overwriting. */
int dss2_reduce_partials(const float* partials, int64_t partial_stride, int num_partials, int64_t count,
                         float* grad, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (c) Branch flows + WLS loss, fused forward and backward.  Replaces data.py:328-390 (get_pflow) and
 * data.py:393-459 (gsp_wls_edge) + autograd.  x [Nt,11] (stride x_stride), edge_attr [Et,13]
 * (stride ea_stride), output [Nt,2] (dense).  stats = {x_mean[8], x_std[8], edge_mean[6], edge_std[6]}
 * (device, 28 floats).  coefs = {lam_v, lam_p, lam_pf, lam_reg} by value.  vminmax: device {V_lv, V_hv}.
 * mask_inplace != 0 reproduces the reference's in-place zeroing of slack theta in `output`
 * (data.py:412-413).  loss: device scalar.  grad_out [Nt,2] may be NULL (forward only);
 * grad_loss: device scalar upstream gradient or NULL (= 1).  ws: dss2_wls_workspace_bytes(g).
 * ---------------------------------------------------------------------------------------------- */
size_t dss2_wls_workspace_bytes(const dss2_graph_t* g);
int dss2_wls_fwd_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr,
                     int64_t ea_stride, float* output, const float* stats, float lam_v, float lam_p,
                     float lam_pf, float lam_reg, const float* vminmax, int mask_inplace,
                     float* loss, const float* grad_loss, float* grad_out, void* ws, size_t ws_bytes,
                     void* stream);
/* Exact-global-batch data parallelism (SURVEY.md 8e; the loss squares batch means, data.py:450-455, so per-rank losses do not add up):
 * dss2_wls_pass(1, ...) runs the reduction pass only and leaves seven doubles at dss2_wls_sums(ws) - the five batch sums and the bus /
 * branch counts; the caller sum-all-reduces them over the ranks in place; dss2_wls_pass(2, ...) runs the gradient pass with the global
 * means and 1/N, 1/E factors and overwrites *loss with the loss of the union batch.  Summing (not averaging) the ranks' parameter
 * gradients then gives the gradient of one batch made of all ranks' scenarios.  Same arguments as dss2_wls_fwd_bwd; tiled batches only. */
double* dss2_wls_sums(void* ws);
int dss2_wls_pass(int phase, const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride,
                  float* output, const float* stats, float lam_v, float lam_p, float lam_pf, float lam_reg, const float* vminmax,
                  int mask_inplace, float* loss, const float* grad_loss, float* grad_out, void* ws, size_t ws_bytes, void* stream);

/* get_pflow (data.py:328-390, phase_shift=True): y [Nt,2] (V pu, theta rad, row stride y_stride);
 * node vn_kv via vminmax; edge_param columns (G,B,Gs,Bs,closed,shift,imax) = edge_attr[:,6:13] given
 * as pointer to column 0 of the parameter block with row stride ep_stride.
 * out8 [8,Et]: loading_lines, loading_trafo, P_from, Q_from, P_to, Q_to, I_from, I_to. */
int dss2_pflow(const int64_t* edge_index, int64_t num_edges, const float* y, int64_t y_stride,
               const float* edge_param, int64_t ep_stride, const float* vminmax, float* out8, void* stream);
/* dss2_pflow_ex: use_shift != 0 evaluates delta = (theta_i - theta_j) - phase_shift (get_pflow(..., phase_shift=False), data.py:364-365).
 * dss2_pflow_bwd: adjoint of the eight outputs w.r.t. y (the reference's get_pflow is plain autograd code): grad_out8 [8, Et] dense
 * (zeros for unused outputs), grad_y [Nt, 2] dense; g = the batch structure of the one-way edge list (undirect = 1). */
int dss2_pflow_ex(const int64_t* edge_index, int64_t num_edges, const float* y, int64_t y_stride, const float* edge_param,
                  int64_t ep_stride, const float* vminmax, int use_shift, float* out8, void* stream);
int dss2_pflow_bwd(const dss2_graph_t* g, const float* y, int64_t y_stride, const float* edge_param, int64_t ep_stride,
                   const float* vminmax, int use_shift, const float* grad_out8, float* grad_y, void* stream);
/* dss2_pflow_est: get_pflow of the model's de-normalised estimate (inference, dss2_run.py:183-194) without materialising it: per bus
 * V = output[:,0] * x_std0 + x_mean0 and theta = output[:,1] * (1 - x[:,9]) (separately rounded fp32, as the torch ops compute it),
 * then the branch flows of dss2_pflow into the same out8 [8,Et] layout.  output [Nt,>=2] (row stride out_stride), x [Nt,>=10]
 * (x_stride); x_mean0 / x_std0 by value.  No host reads, no allocation: graph-capturable. */
int dss2_pflow_est(const int64_t* edge_index, int64_t num_edges, const float* output, int64_t out_stride, const float* x, int64_t x_stride,
                   float x_mean0, float x_std0, const float* edge_param, int64_t ep_stride, const float* vminmax, float* out8, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (f-3) Dataset builder.  Replaces the feature engineering of data_from_pickles (data.py:96-206) for S scenarios of one grid:
 * nodes [S,N,7] f64 (vn_kv, bool_slack, bool_zero_inj, vm_pu, va_rad, p_mw, q_mvar), closed_edges [S,E,11] f64 (the closed branches:
 * from_bus, to_bus, G, B, Gs, Bs, closed line, phase shift, imax or sn, p_from_mw, q_from_mvar), noise_nodes [S,N,4] / noise_edges [S,E,2]
 * f64 standard-normal draws (np.random.normal(0, s) = s * draw: a caller can replay the reference's stream), meas_v_mask [N] / meas_pflow_mask
 * [E] u8 (dss2_run.py:48-53), noise_param6 = HOST array (p_noise, v_noise, i_noise, pm_noise, sgen_noise, zero_inj_coef).
 * Out: x [S*N,11], edge_attr [S*E,13] with the first 8 / 6 columns z-scored over their non-zero entries (data.py:179-190), and
 * stats28 = x_mean[8], edge_mean[6], x_std[8], edge_std[6].  Five launches; deterministic (fixed-order float64 reductions). */
size_t dss2_build_scenarios_workspace_bytes(void);
int dss2_build_scenarios(const double* nodes, const double* closed_edges, const double* noise_nodes, const double* noise_edges,
                         const uint8_t* meas_v_mask, const uint8_t* meas_pflow_mask, const double* noise_param6, int64_t S, int N,
                         int E, float* x, float* edge_attr, float* stats28, void* workspace, size_t workspace_bytes, void* stream);

/* Synthetic scenario sampler of the offline generator (toy_network.py:83-126 with loadsampling.py:75-107), bit-exact with the
 * reference's numpy arithmetic for the same random draws.
 * dss2_load_profiles: base [L] loads (or static generators); mu[l*H+h] = weight_a[l] * (base[l] * profile_a[h]) + weight_b[l] * (base[l] *
 *   profile_b[h]) over the H hours of two daily profiles (toy_network.py:106-107), written as the sampler's two arguments [L*H]:
 *   dist 0 'uniform': arg_a = mu (1 - spread), arg_b = mu (1 + spread); dist 1 'normal': arg_a = mu, arg_b = mu * spread (:119-123).
 * dss2_mc_sample: out[u,i] = arg_a[u] + draws[u,i] * (arg_b[u] - arg_a[u]) (dist 0, samplermontecarlo, draws uniform in [0,1)) or
 *   arg_a[u] + arg_b[u] * draws[u,i] (dist 1, samplermontecarlo_normal, standard-normal draws); draws, out [U, iters] f64. */
int dss2_load_profiles(const double* base, const double* weight_a, const double* weight_b, const double* profile_a,
                       const double* profile_b, int L, int H, int dist, double spread, double* arg_a, double* arg_b, void* stream);
int dss2_mc_sample(const double* arg_a, const double* arg_b, int64_t U, int iters, int dist, const double* draws, double* out,
                   void* stream);

/* ------------------------------------------------------------------------------------------------
 * (f-2) AC power flow of the offline generator.  Replaces pandapower runpp (toy_network.py:180, in the loop of :160-250) on the
 * reference's own pi-model (data.py:370-376, phase shift ignored): Y_ff, Y_tt += y + ys/2 and Y_ft, Y_tf -= y per closed edge, parallel
 * edges summed; S_calc = V_lv^2 U conj(Y U), V_lv = min(vn_kv); S_spec = -(p_mw + j q_mvar) (load-positive, data.py:428-429).
 * Newton-Raphson in polar form, fp64, from a flat start (V = 1, theta = 0; the slack at (v_slack[s], 0)); one slack bus, PQ buses.
 * Topology (built once on the host, dss2.powerflow.symbolic; every array DEVICE, int32 unless stated):
 *   y_ptr [N+1], y_col, y_gb [nnz,2] f64: Y * V_lv^2 as CSR over all buses (MVA at 1 pu);
 *   bus [n]: bus of elimination position k (n = N - 1, the slack removed);
 *   blk_ptr [n+1], blk_col [blocks]: 2x2-block pattern of the reduced Jacobian in position order with fill, columns ascending;
 *   blk_y [blocks]: Y entry of each block (-1 = fill); diag [n]: position of block (k,k);
 *   upd_ptr [blocks+1], upd [updates,2]: for lower block p = (k,m), the pairs (block (k,j), block (m,j)), j > m, of the row-wise block LU;
 *   edge_ft [E,2], edge_gb [E,4] f64 (G, B, Gs, Bs): the closed edges, whose flows are returned.
 * dss2_powerflow: p_mw, q_mvar [S,N] (slack entries ignored), v_slack [S].  Per scenario, convergence (max |S_calc - S_spec| over the PQ
 *   buses <= tol_mva) is tested before each update; iterations [S] = updates applied.  Out: vm_pu, va_rad [S,N]; p_out, q_out [S,N] get
 *   the slack's computed injection at the slack column (other entries untouched: the caller copies the inputs in); p_from, q_from,
 *   p_to, q_to [S,E] (rounded like synth.branch_flows); converged [S] u8; max_mismatch [S] (MVA, at the last evaluation).  max_iter
 *   updates without convergence, or a pivot with |det| <= 1e-12 (|ad| + |bc|), give converged = 0 and undefined outputs for that
 *   scenario only.  Scenarios run `chunk` per launch in `workspace` (dss2_powerflow_workspace_bytes(topo, chunk) = 8 chunk (4 N + 2 n +
 *   4 blocks) bytes); no atomics, so a scenario's result does not depend on the chunk or the other scenarios.  No host synchronisation,
 *   no allocation.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dss2_pf_topology {
  int32_t num_buses;        /* N */
  int32_t slack;
  int32_t num_pq;           /* n = N - 1 */
  int32_t num_blocks;
  int32_t num_updates;
  int32_t num_edges;        /* E closed edges */
  double v_lv;              /* min(vn_kv), kV */
  const int32_t* y_ptr;
  const int32_t* y_col;
  const double* y_gb;
  const int32_t* bus;
  const int32_t* blk_ptr;
  const int32_t* blk_col;
  const int32_t* blk_y;
  const int32_t* diag;
  const int32_t* upd_ptr;
  const int32_t* upd;
  const int32_t* edge_ft;
  const double* edge_gb;
} dss2_pf_topology_t;
size_t dss2_powerflow_workspace_bytes(const dss2_pf_topology_t* topo, int64_t chunk);
int dss2_powerflow(const dss2_pf_topology_t* topo, int64_t S, const double* p_mw, const double* q_mvar, const double* v_slack,
                   double tol_mva, int max_iter, double* vm_pu, double* va_rad, double* p_out, double* q_out, double* p_from,
                   double* q_from, double* p_to, double* q_to, int32_t* iterations, uint8_t* converged, double* max_mismatch,
                   void* workspace, size_t workspace_bytes, int64_t chunk, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Classical weighted-least-squares state estimation, batched: the estimator the reference compares DSS2 against
 * (case_study.py:1226-1357, pandapower's WLS estimator) on the measurements of the physics-informed loss (data.py:393-459).
 * Per scenario of N buses and E closed edges, with Z, R, Z', R' the de-normalised, masked measurements and weights of the loss
 * (data.py:397-409; a normalised value of exactly 0 is absent), fp64 on the fp32 inputs promoted exactly:
 *   J_s(V, th) = w_v sum_n [R_n0 (Z_n0 - V_n)^2 + R_n1 (Z_n1 - th_n)^2] + w_p sum_n [R_n2 (Z_n2 - p_n)^2 + R_n3 (Z_n3 - q_n)^2]
 *              + w_pf sum_e [R'_e0 (Z'_e0 - P_f,e)^2 + R'_e1 (Z'_e1 - Q_f,e)^2]
 * th_slack = 0 (x column 9, data.py:412-413); p_n = -sum_{to=n} P_t - sum_{from=n} P_f and the same for q (data.py:428-429); the
 * flows of the pi-model (data.py:370-376, phase shift ignored) with c = V_lv^2, V_lv = min vn_kv (x column 8) of the scenario, and
 * G, B, Gs, Bs from edge_attr columns 6-9.  Classical WLS: w_v = w_p = w_pf = 1; the loss's data term: lam_v / N, lam_p / N, lam_pf / E.
 * Gauss-Newton over the 2N - 1 unknowns (th, V) from a flat start (V = 1, th = 0): the gain matrix H^T W H as 2x2 (th, V) blocks per
 * pair of buses that share a measurement, the slack's block with identity in its th row and column, factorised by the block LU of
 * the power flow in the host's elimination order, in double-double (a weight near 1e12 makes the fp64 Schur complements cancel).
 * The step is halved until J_s does not grow (beyond 1e-12 relative), which keeps Gauss-Newton from diverging on scenarios with
 * large residuals.  Stops when the full step max |dx| <= tol (converged), after max_iter updates, or when no halving (down to
 * 2^-39) decreases J_s.
 * Topology (built once on the host, dss2.estimation.symbolic; every array DEVICE, int32; "position" = elimination position):
 *   edge_ft [E,2]: local (from, to) of the closed edges, the batch's edge order;
 *   inc_ptr [N+1], inc [.,3]: per bus its incident edges as (edge, end 0 = from / 1 = to, support slot of the other end);
 *   sup_ptr [N+1], sup_pos: per bus the positions of its support {i} u nbr(i), slot 0 = the bus itself;
 *   pair_ptr [N+1], pair_blk: per bus the block of every (slot a, slot b) of its support, row-major over (a, b);
 *   edge_blk [E,4]: blocks (ii, ij, ji, jj) of every edge; bus [N]: bus at each position;
 *   blk_ptr, blk_col, diag, upd_ptr, upd: the block pattern with fill and the LU's update lists (as dss2_pf_topology_t).
 * dss2_wls_estimate: B scenarios of one topology in PyG order: x [B N, >= 11] (row stride x_stride), edge_attr [B E, >= 13],
 * stats28 = x_mean[8], x_std[8], edge_mean[6], edge_std[6] (fp32, device).  Out: vm_pu, va_rad [B N] f64, output [B N, 2] f32 =
 * ((V - x_mean0) / x_std0, th) (the model's output convention), objective [B] = J_s at the returned state, iterations [B] = updates
 * applied, converged [B] u8, max_step [B] = the last full step max |dx|.  A pivot with |det| <= 1e-12 (|ad| + |bc|), a
 * non-finite value, max_iter updates without convergence or a step without descent give converged = 0 for that scenario only.
 * Scenarios run `chunk` per launch, one thread each, in `workspace` (dss2_wls_estimate_workspace_bytes(topo, chunk) = 8 chunk
 * (16 N + 28 E + 8 blocks + 4 max_support) bytes, index-major, the blocks and the right-hand side in double-double); no atomics, so a scenario's result does not depend on the chunk or the other scenarios.  No host synchronisation, no allocation.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dss2_se_topology {
  int32_t num_buses;        /* N */
  int32_t num_edges;        /* E */
  int32_t slack;
  int32_t num_blocks;
  int32_t num_updates;
  int32_t num_pairs;        /* sum over buses of |support|^2 */
  int32_t max_support;
  const int32_t* edge_ft;
  const int32_t* inc_ptr;
  const int32_t* inc;
  const int32_t* sup_ptr;
  const int32_t* sup_pos;
  const int32_t* pair_ptr;
  const int32_t* pair_blk;
  const int32_t* edge_blk;
  const int32_t* bus;
  const int32_t* blk_ptr;
  const int32_t* blk_col;
  const int32_t* diag;
  const int32_t* upd_ptr;
  const int32_t* upd;
} dss2_se_topology_t;
size_t dss2_wls_estimate_workspace_bytes(const dss2_se_topology_t* topo, int64_t chunk);
int dss2_wls_estimate(const dss2_se_topology_t* topo, int64_t B, const float* x, int64_t x_stride, const float* edge_attr,
                      int64_t ea_stride, const float* stats28, double w_v, double w_p, double w_pf, double tol, int max_iter,
                      double* vm_pu, double* va_rad, float* output, double* objective, int32_t* iterations, uint8_t* converged,
                      double* max_step, void* workspace, size_t workspace_bytes, int64_t chunk, void* stream);

/* Validation metrics of one batch (SURVEY.md 8f-4, dss2_run.py:183-209) in one kernel: x [Nt,>=11] (column 9 = slack flag),
 * edge_attr [Et,>=13] (columns 6.. = branch parameters), output [Nt,2] = model output (normalised V, raw theta), y [Nt,2] = labels.
 * sums19 (device, fp64): [0..3] sum (dV)^2, |dV|, (dth)^2, |dth| with V = out0*x_std0 + x_mean0 and th = out1*(1-slack);
 * [4..7] sum V, V^2, th, th^2; [8..11] the same of the labels; [12..14] count, sum d^2, sum |d| of the line loading over branches whose
 * TRUE line loading is non-zero; [15..17] the same for the transformer loading; [18] unused.  ws: dss2_eval_workspace_bytes(),
 * zero-initialised once. */
size_t dss2_eval_workspace_bytes(void);
int dss2_eval_metrics(const int64_t* edge_index, int64_t num_nodes, int64_t num_edges, const float* x, int64_t x_stride,
                      const float* edge_attr, int64_t ea_stride, const float* output, int64_t out_stride, const float* y,
                      int64_t y_stride, float x_mean0, float x_std0, const float* vminmax, double* sums19, void* ws, size_t ws_bytes,
                      void* stream);
/* Same kernel and arguments, with the batch finalised on the device for an epoch average that needs no host synchronisation: the last
 * CTA turns the 19 sums into the ten metrics of dss2.metrics.evaluate_batch in fp64 (rmse_v, mae_v, rmse_th, mae_th, rmse_loading,
 * mae_loading, rmse_loading_trafos, mae_loading_trafos, prop_std_v, prop_std_th; the script's formulas in its operation order, NaN where
 * a count is zero or a std has n <= 1) and ADDS them to acc11[0..9], and 1 to acc11[10] (the batch count).  Epoch value k =
 * acc11[k] / acc11[10], the script's mean over batches (dss2_run.py:165-236).  acc11: device fp64, zeroed by the caller per epoch. */
int dss2_eval_metrics_acc(const int64_t* edge_index, int64_t num_nodes, int64_t num_edges, const float* x, int64_t x_stride,
                          const float* edge_attr, int64_t ea_stride, const float* output, int64_t out_stride, const float* y,
                          int64_t y_stride, float x_mean0, float x_std0, const float* vminmax, double* acc11, void* ws, size_t ws_bytes,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * Adjacent: flat-buffer Adamax (torch.optim.Adamax defaults, dss2_run.py:91-92,143).
 * step_state: device {uint64 seed, uint64 step}; the kernel uses step+1 for bias correction and, when
 * bump != 0, increments it (so a captured graph advances its own clock).  grad_scale multiplies the
 * gradient first (1/world_size after a sum all-reduce).
 * ---------------------------------------------------------------------------------------------- */
int dss2_adamax_step(float* param, const float* grad, float* exp_avg, float* exp_inf, int64_t count,
                     float lr, float beta1, float beta2, float eps, float grad_scale,
                     uint64_t* step_state, int bump, void* stream);
/* step_state[1] += 1 on the device: the clock of a forward-only stream (a captured evaluator advances it once per forward, so that its
 * dropout draws and the tile-mark sequence numbers of the chained layers differ on every replay). */
int dss2_step_advance(uint64_t* step_state, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Next row (SURVEY.md 8f-1): GAT_DSSE, the as-shipped default model of dss2_run.py:86 (networks.py:113-156):
 * 7 x [PyG GATv2Conv(8, 8, heads=1, negative_slope=0.2, add_self_loops=True, edge_dim=6, fill_value='mean') + LeakyReLU(0.01)],
 * Linear(8, dim_dense), Linear(dim_dense, 2).
 *
 * dss2_gat_fwd: one GATv2 layer + activation (act: 0 none, 1 leaky_relu with act_slope - ReLU = slope 0 -, 2 tanh; or-ed with
 * DSS2_GAT_NO_SELF_LOOPS for add_self_loops=False: edges as given, no appended loop) on the ONE-WAY edge list the script passes: x [Nt,8] (row stride
 * x_stride), edge_attr [Et,fe] (row stride ea_stride) -> y [Nt,8] dense.  Input self loops are dropped and one loop per bus is appended
 * last with the mean attribute of the edges pointing at the bus; segment softmax as PyG (max-shifted, + 1e-16).
 * Parameters with PyG's names and shapes: lin_l.weight/bias [8,8]/[8], lin_r.weight/bias, lin_edge.weight [8,fe], att [8], bias [8].
 * dss2_gat_bwd: recompute-based backward.  y = the forward output (activation gate), grad_y its gradient, grad_x [Nt,8] or NULL,
 * node_ws: dss2_gat_ws_bytes(Nt) of scratch; per-CTA partial gradients (dss2_num_partials() rows) in the order
 * [lin_l.w 64 | lin_l.b 8 | lin_r.w 64 | lin_r.b 8 | lin_edge.w 8 fe | att 8 | bias 8].  Needs a graph built with undirect=1.
 * dss2_mlp2_fwd/bwd: z = W2 (W1 x + b1) + b2 per bus (no non-linearity in between, networks.py:150-151); h [Nt,dmid] is kept for the
 * backward; partial layout [w1 dmid x din | b1 dmid | w2 dout x dmid | b2 dout].
 * ---------------------------------------------------------------------------------------------- */
#define DSS2_GAT_NO_SELF_LOOPS 0x100
size_t dss2_gat_ws_bytes(int64_t num_nodes);
int dss2_gat_fwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                 const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                 const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                 float* y, void* stream);
int dss2_gat_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                 const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                 const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                 const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes, float* partials,
                 int64_t partial_stride, void* stream);
/* Prepared weights: dss2_gat_upload puts the seven tensors of `count` layers into constant-memory slots first .. first + count - 1 (8
 * slots; one layout kernel + one device-to-device copy, both capturable); dss2_gat_fwd_slot / dss2_gat_bwd_slot are the layer kernels
 * reading slot `slot` - every weight an immediate constant operand, 92-96 registers per thread instead of 255 (the pointer variants
 * stage the weights in shared memory).  Slots are process-wide state: upload, then launch, on one stream.  part_off: as for
 * dss2_gat_bwd_ex below, or NULL for the standard partial row; with [lin_l.w | lin_r.w] and [lin_l.b | lin_r.b] adjacent the two Linear
 * gradients come from ONE outer-product reduction. */
int dss2_gat_upload(int first, int count, const float* const* lin_l_w, const float* const* lin_l_b, const float* const* lin_r_w,
                    const float* const* lin_r_b, const float* const* lin_edge_w, const float* const* att, const float* const* bias, int fe,
                    void* stream);
int dss2_gat_fwd_slot(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe, int slot,
                      float att_slope, int act, float act_slope, float* y, void* stream);
int dss2_gat_bwd_slot(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe, int slot,
                      float att_slope, int act, float act_slope, const float* y, const float* grad_y, float* grad_x, float* node_ws,
                      size_t node_ws_bytes, float* partials, int64_t partial_stride, const int64_t* part_off, void* stream);
/* One head of a multi-head layer (GATv2Conv(heads = H, concat = False), networks.py:145-146: the heads' outputs are averaged): the same
 * backward with the seven blocks of the partial row at explicit offsets part_off[7] (floats, relative to `partials`, order as above), so
 * that head h writes into its slice of every parameter.  The host side (dss2/gat.py) runs the heads with act = 0 and a zero bias and
 * combines them with dss2_lin8_fwd / dss2_lin8_bwd (M = H inputs, weight blocks I / H, the layer's bias and activation). */
int dss2_gat_bwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                    const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b,
                    const float* lin_edge_w, const float* att, const float* bias, float att_slope, int act, float act_slope,
                    const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes, float* partials,
                    int64_t partial_stride, const int64_t* part_off, void* stream);
/* GINE_DSSE layer (networks.py:71-111, PyG GINEConv + LeakyReLU): y_i = leaky(nn((1 + eps) x_i + sum_{j->i} relu(x_j + lin(a_ji)))) with
 * nn = the model's ONE shared Linear(8,8) and lin = this layer's Linear(edge_dim, 8); one-way edge list.  Backward: node_ws of
 * dss2_gine_ws_bytes(Nt); per-CTA partial rows [lin.weight 8 fe | lin.bias 8] at partials_lin and [nn.weight 64 | nn.bias 8] (this
 * layer's share of the shared Linear's gradient) at partials_nn, both with row stride partial_stride. */
size_t dss2_gine_ws_bytes(int64_t num_nodes);
int dss2_gine_fwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                  const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, int act, float act_slope,
                  float* y, void* stream);
int dss2_gine_bwd(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                  const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, int act, float act_slope,
                  const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes, float* partials_lin,
                  float* partials_nn, int64_t partial_stride, void* stream);
/* train_eps=True: eps_param = this layer's trainable eps on the device (NULL = the value `eps`); the backward appends its gradient to the
 * partials_lin row: [lin.weight 8 fe | lin.bias 8 | eps 1]. */
int dss2_gine_fwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                     const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, const float* eps_param,
                     int act, float act_slope, float* y, void* stream);
int dss2_gine_bwd_ex(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe,
                     const float* nn_w, const float* nn_b, const float* lin_w, const float* lin_b, float eps, const float* eps_param,
                     int act, float act_slope, const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes,
                     float* partials_lin, float* partials_nn, int64_t partial_stride, void* stream);
int dss2_mlp2_fwd(int64_t num_nodes, const float* x, int din, const float* w1, const float* b1, int dmid, const float* w2,
                  const float* b2, int dout, float* h, float* z, void* stream);
int dss2_mlp2_bwd(int64_t num_nodes, const float* x, int din, const float* w1, int dmid, const float* w2, int dout,
                  const float* h, const float* grad_z, float* grad_h_ws, float* grad_x, float* partials, int64_t partial_stride,
                  void* stream);
/* The head without h or grad_h in memory, for the sizes dss2_mlp2_nh_supported() accepts (8 -> 32 -> 2, dss2_run.py:73-76): there is no
 * non-linearity between the two Linears, so all four gradients are linear in S = sum_n grad_z[n] (x) x[n] and s = sum_n grad_z[n]; one
 * pass over the buses, same partial-row layout.  dss2_mlp2_fwd takes h = NULL for these sizes. */
int dss2_mlp2_nh_supported(int din, int dmid, int dout);
int dss2_mlp2_bwd_nh(int64_t num_nodes, const float* x, int din, const float* w1, const float* b1, int dmid, const float* w2, int dout,
                     const float* grad_z, float* grad_x, float* partials, int64_t partial_stride, void* stream);

/* ------------------------------------------------------------------------------------------------
 * gnn_dsse building blocks (networks.py:11-69: GCN2Conv / TAGConv / FAConv stacks at width dim_feat <= 8 on the one-way edge list as given).
 * self_loops != 0 is gcn_norm(add_self_loops=True), i.e. PyG's add_remaining_self_loops: the self loops of the input are dropped and
 * one loop of weight 1 per bus is appended; self_loops == 0 takes the edge list as given (an input loop is an ordinary edge).
 * dss2_gcn_dinv: gcn_norm's deg^-1/2 per bus (in-degree; with add_self_loops input loops not counted, + 1; inf -> 0).
 * dss2_gcn_prop8: out = scale * (A_hat x) + add_scale * add with A_hat = D^-1/2 (A [+ I]) D^-1/2 over the in-edges in PyG's scatter
 *   order (self loop last; with self_loops the input loops skipped), or - transposed != 0 - over the out-edges (adjoint).  Rows are
 *   8 floats (zero padded), x with row stride.
 * dss2_lin8_fwd/bwd: y = act(sum_m in_m W_m [+ b]) per bus for M <= 4 inputs of width 8; weight_is_out_by_in = 1 for torch Linear
 *   weights [out, in] (TAGConv.lins), 0 for GCN2Conv.weight1 [in, out]; act: 0 none, 1 leaky_relu(slope), 2 relu, 3 tanh.  The backward
 *   writes grad_z, grad_in[m], optionally acc += acc_scale * grad_in[0], and per-CTA partial sums of the weight gradients (layout of w)
 *   at partials, of the bias gradient at partials + bias_offset.
 * ---------------------------------------------------------------------------------------------- */
int dss2_gcn_dinv(const dss2_graph_t* g, int self_loops, float* dinv, void* stream);
int dss2_gcn_prop8(const dss2_graph_t* g, const float* dinv, int self_loops, int transposed, const float* x, int64_t x_stride,
                   float scale, const float* add, int64_t add_stride, float add_scale, float* out, void* stream);
int dss2_lin8_fwd(int64_t num_nodes, int M, int weight_is_out_by_in, const float* const* in, const int64_t* in_strides, const float* w,
                  const float* bias, int act, float slope, float* y, void* stream);
int dss2_lin8_bwd(int64_t num_nodes, int M, int weight_is_out_by_in, const float* const* in, const int64_t* in_strides, const float* w,
                  int act, float slope, const float* y, const float* grad_y, float* grad_z, float* const* grad_in, float* acc,
                  float acc_scale, float* partials, int64_t partial_stride, int64_t bias_offset, void* stream);

/* gnn_dsse(model='fagcn') (networks.py:44-50, torch_geometric FAConv; dropout: dss2_fa_fwd_drop below) at width 8 on the one-way edge list:
 *   y[i] = act( sum_{j -> i} tanh(att_l . x[j] + att_r . x[i]) dinv[j] dinv[i] x[j]  (+ self loop, last)  + eps x0[i] ).
 * With self_loops the input loops are skipped and one loop per bus is appended (as dss2_gcn_prop8; dinv from dss2_gcn_dinv alike).
 * dss2_fa_bwd: grad_x (adjoint of x, message and attention paths), optionally acc_x0 += eps * grad_z (the x_0 path), and per-CTA
 * partial sums of the attention gradients at partials[0..8) (att_l) and partials[8..16) (att_r), dss2_num_partials() rows. */
int dss2_fa_fwd(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* x0,
                int64_t x0_stride, const float* att_l, const float* att_r, float eps, int act, float slope, float* y, void* stream);
int dss2_fa_bwd(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* att_l,
                const float* att_r, float eps, int act, float slope, const float* y, const float* grad_y, float* grad_x,
                float* acc_x0, float* partials, int64_t partial_stride, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention dropout of GATv2Conv (networks.py:145-146, `dropout` of GAT_DSSE) and FAConv (networks.py:46, `dropout` of
 * gnn_dsse(model='fagcn')) in training mode: alpha = F.dropout(softmax_i(score), p) for GATv2, coef = F.dropout(tanh(.), p) * w for
 * FAConv, every coefficient of a softmax segment - the appended self loop too - kept with probability 1 - p and scaled by 1 / (1 - p).
 * Descriptor (host struct, one per layer and head):
 *   p in [0, 1); mode 0 none, 1 counter-based Philox keyed by (seed, step) read from DEVICE memory rng_state[2] (graph-replay safe, as
 *   dss2_tag_fwd) with layer_uid and head, 2 caller mask `mask` (uint8 [Et + Nt], 1 = keep).  p == 0 or mode 0 = no dropout.
 *   Edge key of a coefficient: the one-way edge id e for a real edge, Et + i for the loop appended at bus i.  With add_self_loops both
 *   GATv2 and FAConv drop the input self loops, so their keys are never read (mode 2: their mask entries are ignored); without it an
 *   input loop is an ordinary edge with its own key and the loop entries Et + i are unused.
 * The forward and both backward passes re-draw the same bit wherever they visit a coefficient; nothing is stored between them.
 * dss2_gat_fwd_drop / dss2_gat_bwd_drop: dss2_gat_fwd / dss2_gat_bwd_ex with a weight slot (slot >= 0: dss2_gat_upload's weights, the
 *   pointers are ignored; -1: weights from the pointers) and a descriptor (NULL = none).  bwd: part_off NULL = the standard partial row.
 * dss2_fa_fwd_drop / dss2_fa_bwd_drop: dss2_fa_fwd / dss2_fa_bwd with a descriptor.
 * dss2_attn_drop_mask: writes the mask [Et + Nt] (1 = keep) that the descriptor applies, from the same device function as the layer
 *   kernels (mode 1: what the Philox stream draws for this seed, step, layer_uid and head).
 * All of them are capturable: no host synchronisation, no allocation.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dss2_attn_drop {
  float p;
  int mode;
  const uint64_t* rng_state;
  uint32_t layer_uid;
  uint32_t head;
  const uint8_t* mask;
} dss2_attn_drop_t;
int dss2_gat_fwd_drop(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe, int slot,
                      const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b, const float* lin_edge_w,
                      const float* att, const float* bias, float att_slope, int act, float act_slope, const dss2_attn_drop_t* drop,
                      float* y, void* stream);
int dss2_gat_bwd_drop(const dss2_graph_t* g, const float* x, int64_t x_stride, const float* edge_attr, int64_t ea_stride, int fe, int slot,
                      const float* lin_l_w, const float* lin_l_b, const float* lin_r_w, const float* lin_r_b, const float* lin_edge_w,
                      const float* att, const float* bias, float att_slope, int act, float act_slope, const dss2_attn_drop_t* drop,
                      const float* y, const float* grad_y, float* grad_x, float* node_ws, size_t node_ws_bytes, float* partials,
                      int64_t partial_stride, const int64_t* part_off, void* stream);
int dss2_fa_fwd_drop(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* x0,
                     int64_t x0_stride, const float* att_l, const float* att_r, float eps, int act, float slope,
                     const dss2_attn_drop_t* drop, float* y, void* stream);
int dss2_fa_bwd_drop(const dss2_graph_t* g, const float* dinv, int self_loops, const float* x, int64_t x_stride, const float* att_l,
                     const float* att_r, float eps, int act, float slope, const dss2_attn_drop_t* drop, const float* y,
                     const float* grad_y, float* grad_x, float* acc_x0, float* partials, int64_t partial_stride, void* stream);
int dss2_attn_drop_mask(const dss2_attn_drop_t* drop, int64_t num_edges, int64_t num_nodes, uint8_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSS2_B200_H */
