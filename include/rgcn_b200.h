/*
 * rgcn_b200.h — C ABI of the B200-native RGCN message-passing hot path.
 *
 * Drop-in boundary for arnold117/PrimeKG-RGCN-LinkPrediction (reference paths are relative
 * to /root/reference).  The reference has no FFI: its hot path is the Python call chain
 *   DrugDiseaseModel.forward            src/models/rgcn.py:300-331
 *   -> DrugDiseaseRGCN.forward          src/models/rgcn.py:97-130
 *   -> torch_geometric RGCNConv.forward called at src/models/rgcn.py:123, :128 (third party)
 *   -> LinkPredictor.forward            src/models/rgcn.py:189-213
 *   -> LinkPredictor.score_all_tails    src/models/rgcn.py:215-243
 * Each entry point below names the reference computation it replaces.  The Python host side
 * (primekg-rgcn-linkprediction_b200/) binds these with ctypes; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - sizes are explicit, nothing is allocated inside: workspaces are passed in and sized by
 *     the *_workspace_bytes twin;
 *   - all work is enqueued on `stream` (a cudaStream_t), no implicit synchronisation unless
 *     the function's comment says so;
 *   - return value 0 = ok, otherwise an RGCN_E* code; rgcn_last_error() gives the message of
 *     the calling thread's last failure.
 *   - feature matrices are row-major fp32, rows 16-byte aligned (ld % 4 == 0), feature width d
 *     a multiple of 4 and at most 1024.
 */
#ifndef RGCN_B200_H_
#define RGCN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RGCN_B200_ABI_VERSION 8

enum {
  RGCN_OK = 0,
  RGCN_EINVAL = 1,      /* bad argument (shape / alignment / null)            */
  RGCN_ERANGE = 2,      /* an edge endpoint or relation id is out of range    */
  RGCN_ECUDA = 3,       /* a CUDA runtime call failed                         */
  RGCN_EWORKSPACE = 4,  /* workspace too small                                */
  RGCN_EUNSUPPORTED = 5 /* device is not sm_100 / feature not compiled        */
};

typedef void* rgcn_stream_t; /* cudaStream_t */

int rgcn_abi_version(void);
/* Copies the calling thread's last error message (NUL terminated) into buf; returns its length. */
int rgcn_last_error(char* buf, size_t buf_len);
/* 0 when the current device is compute capability 10.x, RGCN_EUNSUPPORTED otherwise. */
int rgcn_check_device(void);
/* Number of kernels of this library launched so far by this process (all threads). */
int64_t rgcn_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Measurement aid (no reference counterpart): the row-gather access pattern of the aggregation with everything else
 * removed, so that bench.py can MEASURE, on the box it runs on, what the L2 (table smaller than the L2) or the HBM
 * (larger table) delivers for that pattern — the denominators of the roofline block.  Sums table[idx[i], 0:d] over
 * i in [0, n_idx) (idx == NULL: rows i % n_rows in order, a streaming read) with sm_count * blocks_per_sm blocks;
 * sink: rgcn_probe_gather_sink_floats(blocks_per_sm) floats of scratch.  Bytes moved = n_idx * d * 4.
 * ------------------------------------------------------------------------------------------ */
int64_t rgcn_probe_gather_sink_floats(int32_t blocks_per_sm);
int rgcn_probe_gather(const float* table, int64_t ld, int64_t n_rows, int32_t d, const int32_t* idx, int64_t n_idx,
                      int32_t blocks_per_sm, float* sink, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Graph preprocessing.  Replaces, once per graph, the per-relation boolean masks
 * `edge_index[:, edge_type == r]` that RGCNConv evaluates on every call
 * (call sites src/models/rgcn.py:123, :128; input format src/preprocess.py:240-261).
 *
 * Builds the CSR keyed by (dst, relation)  [key = dst * R + rel, n_dst * R keys] and the
 * transposed CSR keyed by (src, relation) [key = src * R + rel, n_src * R keys].  Inside one
 * key the ORIGINAL edge order is kept (stable LSD radix sort), so the result is bit-identical
 * to a stable sort of the keys.
 *
 *   src, dst, rel   [E] int64 (edge_index row 0, row 1, edge_type)
 *   rowptr   [n_dst*R + 1] int32    col   [E] int32 (= src[perm])     perm   [E] int32
 *   rowptr_t [n_src*R + 1] int32    row_t [E] int32 (= dst[perm_t])   perm_t [E] int32
 *   inv_cnt  [n_dst*R] float   1 / max(in-degree of (dst, rel), 1)
 *   w_t      [E] float         inv_cnt[row_t[e] * R + rel(e)] in transposed order
 *   status   [4] int32         [0] bit0: src out of range, bit1: dst, bit2: rel;
 *                              [1] number of hub segments (> hub_threshold edges);
 *                              [2] longest (dst, rel) segment; [3] longest (src, rel) segment
 * The call is asynchronous; the caller synchronises and inspects status[0] (non-zero => the
 * arrays are unspecified and the Python layer raises IndexError, where PyG would hit a
 * device-side assert).
 * ------------------------------------------------------------------------------------------ */
size_t rgcn_csr_build_workspace_bytes(int64_t E, int64_t n_dst, int64_t n_src, int32_t R);
int rgcn_csr_build(const int64_t* src, const int64_t* dst, const int64_t* rel, int64_t E,
                   int64_t n_dst, int64_t n_src, int32_t R,
                   int32_t* rowptr, int32_t* col, int32_t* perm,
                   int32_t* rowptr_t, int32_t* row_t, int32_t* perm_t,
                   float* inv_cnt, float* w_t, int32_t* status,
                   void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Hub plan (one per CSR orientation, once per graph).  Power-law graphs have (row, relation)
 * segments with 10^4 edges; segments longer than hub_threshold edges are cut into 128-edge chunks that
 * whole thread blocks reduce in a fixed order (no atomics).  The threshold bounds the longest serial walk
 * of one lane group, i.e. the critical path of the row kernel (64 is the default of the Python layer).  hub_keys receives the sorted keys of
 * those segments, hub_chunk_ptr the exclusive prefix of their chunk counts (cap_hubs + 1 entries;
 * entries past n_hubs repeat the total).  cap_hubs >= E / hub_threshold + 1 is always enough.
 * SYNCHRONISES the stream: the two counts are returned to the host.
 * ------------------------------------------------------------------------------------------ */
size_t rgcn_hub_plan_workspace_bytes(int64_t n_keys, int64_t cap_hubs);
int rgcn_hub_plan(const int32_t* rowptr, int64_t n_keys, int32_t hub_threshold, int32_t* hub_keys,
                  int32_t* hub_chunk_ptr, int64_t cap_hubs, int32_t* n_hubs_host, int32_t* n_chunks_host,
                  void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* Chunk table of a hub plan, one int32[4] entry per chunk: {key of the chunk's segment, first chunk of that segment,
 * index of the first hub segment of the same row, number of chunks of that row}.  16-byte aligned. */
int rgcn_hub_chunk_table(const int32_t* hub_keys, const int32_t* hub_chunk_ptr, int32_t n_hubs, int32_t R,
                         int32_t* chunk_table, rgcn_stream_t stream);

/* One orientation of the relation-keyed CSR as the aggregation kernels consume it. */
typedef struct rgcn_csr {
  const int32_t* rowptr;        /* [n_rows * R + 1]                                   */
  const int32_t* idx;           /* [E] gathered row per edge (col, or row_t)          */
  const float* w;               /* [E] per-edge weight, or NULL => mean per segment   */
  int64_t n_rows;
  int64_t E;
  int32_t R;
  int32_t n_hubs;
  int32_t n_chunks;
  int32_t hub_threshold;        /* the threshold the hub plan was made with            */
  const int32_t* hub_keys;      /* [n_hubs]                                           */
  const int32_t* hub_chunk_ptr; /* [n_hubs + 1]                                       */
  const int32_t* chunk_table;   /* [n_chunks][4] from rgcn_hub_chunk_table            */
  const int32_t* row_order;     /* [n_rows] or NULL: a permutation of the rows, the order in which the lane
                                   groups take them (by decreasing edge count: balanced blocks, long walks first) */
  int64_t order_chunk_rows;     /* 0: row_order sorts all rows globally; c > 0: it sorts inside consecutive blocks of c
                                   rows (positions [k c, (k+1) c) hold exactly the rows [k c, (k+1) c)), so the walk can be
                                   launched block by block and pipelined with the transform of the finished rows */
} rgcn_csr_t;

/* ------------------------------------------------------------------------------------------
 * Neighbourhood aggregation, forward.  Replaces, for all relations at once,
 *   x_j = x.index_select(0, src_r);  s = scatter_add(x_j, dst_r);  h_r = s / clamp(cnt, 1)
 * of RGCNConv's loop path (src/models/rgcn.py:123, :128).
 *
 *   H[i, r*d : (r+1)*d] = (1 / max(cnt(i, r), 1)) * sum_{e in seg(i, r)} X[col[e], :]
 * One group of d/4 lanes per destination row, 128-bit loads, serial left-to-right fp32 sum inside
 * a segment (= the order of CPU index_add_), no atomics; segments longer than the hub threshold
 * are split over whole thread blocks and reduced in a fixed order.
 *   out_mode 0: H is fp32 [n_rows, ldh].  out_mode 1: H is one bf16 plane (values rounded to bf16, the
 *   "bf16-transform" mode).  out_mode 2: two bf16 planes H (hi) and H_lo with hi + lo = value to 2^-17 — the
 *   TMA-loadable operand format of rgcn_transform_* in the fp32 mode.  ldh counts elements of the output type.
 *   comp != NULL (basis decomposition, comp [R, B] fp32): instead of R blocks the kernel writes the
 *   B basis-mixed blocks  Z[i, b*d:(b+1)*d] = sum_r comp[r, b] * h_r[i]   (H is then [n_rows, B*d]).
 *   With a weighted CSR (g->w != NULL, i.e. the transposed orientation) h_r is the weighted SUM instead of
 *   the mean: called on the transposed CSR with X = the masked output gradient this is the mirrored
 *   backward of the basis form,  T_b[j] = sum_r comp[r, b] * sum_{e in seg_t(j, r)} w_t[e] * G[row_t[e]].
 *   x_root != NULL (unmixed form only): row i of x_root [n_rows, d] is appended as block R of output row i, so the
 *   transform operand [H | X] (self-loop term last) is complete after this one kernel (H must be R+1 blocks wide).
 *   dot_p != NULL (needs comp, B <= 8): additionally  gc[r, b] = sum_i <h_r[i], dot_p[i, b*d:(b+1)*d]>, the
 *   gradient of comp when dot_p = X @ [V_1 .. V_B]; written as rgcn_aggregate_blocks(g, d) partial rows of
 *   R*B floats into gc_partial, to be summed with rgcn_reduce_partials (fixed order).
 * ------------------------------------------------------------------------------------------ */
size_t rgcn_aggregate_workspace_bytes(const rgcn_csr_t* g, int32_t d);
int64_t rgcn_aggregate_blocks(const rgcn_csr_t* g, int32_t d);
int rgcn_aggregate_fwd(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d,
                       const float* comp, int32_t B,
                       void* H, void* H_lo, int64_t ldh, int32_t out_mode,
                       const float* dot_p, int64_t ld_dot_p, float* gc_partial,
                       const float* x_root, int64_t ld_x_root,
                       void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
/* out[c] = sum over the n_part rows of part[., n_cols] in a fixed order (deterministic). */
int rgcn_reduce_partials(const float* part, int64_t n_part, int32_t n_cols, float* out, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Neighbourhood aggregation, backward (grad-X).  Replaces autograd's backward of the gather /
 * scatter-mean (index_select backward = index_add_ with atomics on CUDA), reached from
 * loss.backward() at src/train.py:306.  Runs over the TRANSPOSED CSR, atomic-free and
 * deterministic:
 *   gX[j, :] = init[j, :] + sum_r sum_{e in seg_t(j, r)} w_t[e] * gH[row_t[e], r*d : (r+1)*d]
 * `init` (may be NULL) carries the root/self-loop term gO @ root^T.
 * ------------------------------------------------------------------------------------------ */
/* Optional second output of the backward walk: gX once more, masked for the layer UPSTREAM of this one —
 * v = mask > 0 ? gX * scale : 0, mask = that layer's ReLU / dropout output (src/models/rgcn.py:124-125), scale its
 * 1 / (1 - p) — written as the bf16 operand planes (hi [, lo]) its backward GEMMs read, with the per-block column sums of
 * v (its bias gradient, [rgcn_aggregate_row_blocks(gt, d), d]).  Replaces that layer's rgcn_split_planes pass. */
typedef struct rgcn_masked_planes_out {
  const float* mask; int64_t ld_mask; float scale;
  void* hi; void* lo; int64_t ldp;          /* lo == NULL: hi plane only (bf16 mode) */
  float* colsum_partial;                    /* nullable */
} rgcn_masked_planes_out;
int64_t rgcn_aggregate_row_blocks(const rgcn_csr_t* g, int32_t d);
/* Row-range form of the unmixed forward walk (comp == NULL form of rgcn_aggregate_fwd): only the positions
 * [row_begin, row_end) of the walk order; hub_pass = 0 when an earlier call of the same layer has already reduced the hub
 * chunks into `workspace` (an empty range with hub_pass = 1 runs the hub pass alone).  With a row order the range must
 * consist of whole order chunks (order_chunk_rows).  rgcn_layer_fwd pipelines these calls with the transform. */
int rgcn_aggregate_fwd_rows(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d, void* H, void* H_lo, int64_t ldh,
                            int32_t out_mode, const float* x_root, int64_t ld_x_root, int64_t row_begin, int64_t row_end,
                            int32_t hub_pass, void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
/* The same walk over a BF16 feature matrix X16 [n_src, d] (the bf16-transform mode: half the gathered bytes; sums, means and
 * hub partials stay fp32), written as the bf16 hi plane H_hi of the transform's operand; x_root16 (bf16 [n_rows, d]) is
 * appended as block R.  Leading dimensions in elements, multiples of 8; d % 8 == 0. */
int rgcn_aggregate_fwd_bf16(const rgcn_csr_t* g, const void* X16, int64_t ldx, int32_t d, void* H_hi, int64_t ldh,
                            const void* x_root16, int64_t ld_x_root, int64_t row_begin, int64_t row_end, int32_t hub_pass,
                            void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* Listed-rows forward walk (the last layer of a link-prediction step is only read at the 2 * batch head / tail rows of its
 * output, src/models/rgcn.py:325-326): position c of rows[0 .. n_list) walks row rows[c] and writes row c of a COMPACT
 * operand [rgcn_rows_compact_size(n_list), >= (R+1) d]; a row listed several times is walked ONCE, into its first position
 * (slot: node -> first list position or m_c, rgcn_rows_list_build); later duplicates and padding positions are zero rows.
 * Hub chunks of unlisted rows are skipped.  On graphs of moderate size the walk goes through the rows in the CSR's
 * degree order and unlisted rows leave at once (long walks start first), otherwise through the list positions.
 * rgcn_rows_list_build: rows [2 n] = heads then tails (out-of-range indices parked on row 0), slot [n_nodes]. */
int rgcn_rows_list_build(const int64_t* head, const int64_t* tail, int64_t n_pairs, int64_t n_nodes, int64_t* rows,
                         int32_t* slot, rgcn_stream_t stream);
int rgcn_aggregate_fwd_list(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d, void* H, void* H_lo, int64_t ldh,
                            int32_t out_mode, const float* x_root, int64_t ld_x_root, const int64_t* rows, int64_t n_list,
                            const int32_t* slot, void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
int rgcn_aggregate_fwd_bf16_list(const rgcn_csr_t* g, const void* X16, int64_t ldx, int32_t d, void* H_hi, int64_t ldh,
                                 const void* x_root16, int64_t ld_x_root, const int64_t* rows, int64_t n_list,
                                 const int32_t* slot, void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

int rgcn_aggregate_bwd(const rgcn_csr_t* gt, const float* gH, int64_t ldg, int32_t d,
                       const float* init, int64_t ld_init,
                       float* gX, int64_t ldgx, const rgcn_masked_planes_out* masked_planes,
                       void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
/* Same walk over a ROW-SPARSE gH: gH_rows holds only the listed rows (see rgcn_rows_compact), slot[i] is the compact
 * row of node i or zero_row (an all-zero row of gH_rows / init_rows) for every other node; init_rows is indexed through
 * slot as well.  Edges whose gathered row is absent are skipped — they would add exact zeros — so the result equals
 * rgcn_aggregate_bwd on the dense matrix bit for bit. */
int rgcn_aggregate_bwd_rows(const rgcn_csr_t* gt, const float* gH_rows, int64_t ldg, int32_t d,
                            const int32_t* slot, int32_t zero_row, const float* init_rows, int64_t ld_init,
                            float* gX, int64_t ldgx, const rgcn_masked_planes_out* masked_planes,
                            void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* rgcn_aggregate_bwd_rows on a graph much larger than the row list (a partitioned shard walks ALL sources of the graph for
 * the ~2 * batch listed rows): src_flag (scratch, gt->n_rows bytes) is cleared, the sources of the listed rows' in-edges are
 * marked from the FORWARD-orientation CSR g_fwd (rows / slot of rgcn_rows_list_build or rgcn_link_loss_bwd_rows), and
 * unmarked rows leave the walk at once.  Same results (the skipped rows only ever add exact zeros). */
int rgcn_aggregate_bwd_rows_marked(const rgcn_csr_t* gt, const rgcn_csr_t* g_fwd, const int64_t* rows, int64_t n_list,
                                   uint8_t* src_flag, const float* gH_rows, int64_t ldg, int32_t d, const int32_t* slot,
                                   int32_t zero_row, const float* init_rows, int64_t ld_init, float* gX, int64_t ldgx,
                                   void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Max aggregation (RGCNConv(aggr='max'), csrc/aggregate_max.cu).  Forward over the forward-orientation CSR g:
 *   Hmax[i, r*d + c] = max_{e in seg(i, r)} X[col[e], c]     (NaN propagates; 0 for an empty segment)
 *   Hcnt[i, r*d + c] = |{e in seg(i, r) : X[col[e], c] == Hmax}| + [Hmax == 0]
 * = torch's zeros(..).scatter_reduce_(0, idx, src, 'amax', include_self=False) and the divisor of its backward (the zero
 * initial value counts as a tie when the maximum is exactly 0).  Hmax is also written as the transform's operand planes
 * (out_mode 1: bf16 hi plane, 2: hi + lo) with x_root (optional) appended as block R, like rgcn_aggregate_fwd.
 * Backward over the TRANSPOSED CSR gt (no weights used), deterministic, no atomics:
 *   gX[j] = init[j] + sum_r sum_{e: j -> i in seg_t(j, r)} [X[j] == Hmax[i, r]] * gH[i, r] / Hcnt[i, r]
 * (and NaN where Hmax is NaN, as torch's backward gives).  init (optional): e.g. the root-term gradient.
 * Segments longer than the hub threshold go through the orientation's hub plan (chunk partials reduced by whole blocks
 * first: (max, ties) pairs forward, sums backward), into `workspace` of rgcn_aggregate_max_workspace_bytes(g, d,
 * backward) bytes.  Deterministic; neither call allocates; both check their arguments before any CUDA call.
 * ------------------------------------------------------------------------------------------ */
size_t rgcn_aggregate_max_workspace_bytes(const rgcn_csr_t* g, int32_t d, int32_t backward);
int rgcn_aggregate_max_fwd(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d, void* H, void* H_lo, int64_t ldh,
                           int32_t out_mode, const float* x_root, int64_t ld_x_root, float* Hmax, float* Hcnt, int64_t ldm,
                           void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
int rgcn_aggregate_max_bwd(const rgcn_csr_t* gt, const float* gH, int64_t ldg, const float* Hmax, const float* Hcnt,
                           int64_t ldm, const float* X, int64_t ldx, int32_t d, const float* init, int64_t ld_init,
                           float* gX, int64_t ldgx, void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Relational transform on the tensor cores (tcgen05.mma, fp32 accumulators in TMEM, every operand tile
 * streamed by TMA).  Replaces the R+1 matmuls `h_r @ W_r`, `x @ root` per layer of RGCNConv's loop path
 * (src/models/rgcn.py:123, :128) and their autograd transposes (src/train.py:306), concatenated
 * along K:  A = [H | X]  ([n_rows, K1 + K2]),  W = [W1 ; W2] = [weight.view(R*d_in, d_out) ; root].
 *
 * Activations are passed as "bf16 planes": row-major bf16 matrices `hi` (value rounded to bf16) and, in
 * mode 0, `lo` (value - hi rounded to bf16).  rgcn_aggregate_fwd(out_mode 1|2) writes H planes directly;
 * rgcn_split_planes converts any fp32 matrix, optionally zeroing elements where relu_mask <= 0 (ReLU
 * backward) and emitting per-block column sums (the bias gradient; rgcn_split_planes_blocks() rows of
 * `cols` floats) and / or the masked values themselves as fp32 (out_f32, nullable).  Planes: base 16-byte aligned, ld (elements) a multiple of 8.
 *   fwd   : out = A @ W + bias (, ReLU)                       [n_rows, d_out] fp32
 *   dgrad : gA  = G @ W^T                                     [n_rows, K1 + K2] fp32
 *   wgrad : [gW1 ; gW2] = A^T @ G ;  gbias = sum of the n_colsum column-sum partials
 * Fused dropout (F.relu + nn.Dropout of src/models/rgcn.py:124-125 in ONE epilogue): with dropout_p > 0 (needs
 * relu = 1) fwd zeroes each output element with probability p and scales the kept ones by 1 / (1 - p).  The mask is
 * a counter-based hash of (dropout_seed, *dropout_counter, element index); the device-side counter is advanced by the
 * call itself, so a captured CUDA graph draws a fresh mask on every replay.  Backward needs no stored mask: the
 * output is zero exactly where ReLU or dropout killed the element, so rgcn_split_planes(gO, relu_mask = out,
 * mask_scale = 1 / (1 - p)) yields G (mask_scale multiplies the masked values; pass 1 without dropout).
 * Fused all-gather (destination-range partition over the GPUs of one NVSwitch domain): peer_out_host is a HOST array
 * of n_peer (<= 8) device pointers to feature buffers [*, peer_ld] that live in other GPUs' memory and are mapped
 * into this process (CUDA IPC / symmetric memory).  fwd's epilogue stores every finished tile into `out` AND into
 * rows peer_row0 + i of each peer buffer, so the transfer of the layer's output overlaps its own GEMM tile by tile
 * and the next layer's all-gather disappears; the caller only has to put a cross-GPU barrier before the next read.
 * mode 0 = "fp32": hi*hi + hi*lo + lo*hi (error ~1e-5 relative); mode 1 = "bf16": hi*hi only.
 * Everything is deterministic (fixed split-K / partial reduction order).  K1, K2, d_out multiples of 4.
 * ------------------------------------------------------------------------------------------ */
int64_t rgcn_split_planes_blocks(int64_t rows, int32_t cols);
int rgcn_split_planes(const float* x, int64_t ldx, const float* relu_mask, int64_t ldm, int64_t rows,
                      int32_t cols, void* hi, void* lo, int64_t ldp, float* colsum_partial,
                      float mask_scale, float* out_f32, int64_t ld_f32, rgcn_stream_t stream);
size_t rgcn_transform_workspace_bytes(int64_t n_rows, int32_t K, int32_t d_out);
int rgcn_transform_fwd(const void* A_hi, const void* A_lo, int64_t lda, int32_t K1, int32_t K2,
                       const float* W1, const float* W2, const float* bias, int32_t relu,
                       int64_t n_rows, int32_t d_out, float* out, int64_t ldo, int32_t mode,
                       float dropout_p, uint32_t dropout_seed, unsigned long long* dropout_counter,
                       float* const* peer_out_host, int32_t n_peer, int64_t peer_row0, int64_t peer_ld,
                       void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
int rgcn_transform_dgrad(const void* G_hi, const void* G_lo, int64_t ldg, int32_t d_out,
                         const float* W1, int32_t K1, const float* W2, int32_t K2,
                         int64_t n_rows, float* gA, int64_t ldga, int32_t mode,
                         void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
int rgcn_transform_wgrad(const void* A_hi, const void* A_lo, int64_t lda, int32_t K1, int32_t K2,
                         const void* G_hi, const void* G_lo, int64_t ldg, int32_t d_out, int64_t n_rows,
                         const float* colsum_partial, int32_t n_colsum,
                         float* gW1, float* gW2, float* gbias, int32_t mode,
                         void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Basis decomposition of the relation weights, RGCNConv(num_bases = B) (plumbed at src/models/rgcn.py:58, :76, :84):
 *   rgcn_basis_combine     : W[r, :] = sum_b comp[r, b] * V[b, :]          (PyG: (comp @ weight.view(B, -1)).view(R, in, out))
 *   rgcn_basis_combine_bwd : g_V[b, :] = sum_r comp[r, b] * gW[r, :],  g_comp[r, b] = <gW[r, :], V[b, :]>   (either may be NULL)
 * comp [R, B], V / g_V [B, in_out], W / gW [R, in_out], all row-major fp32; R, B <= 64 (g_comp: B <= 16).
 * ------------------------------------------------------------------------------------------ */
int rgcn_basis_combine(const float* comp, const float* V, int32_t R, int32_t B, int64_t in_out, float* W,
                       rgcn_stream_t stream);
int rgcn_basis_combine_bwd(const float* comp, const float* V, const float* gW, int32_t R, int32_t B, int64_t in_out,
                           float* g_V, float* g_comp, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Block-diagonal relation weights, RGCNConv(num_blocks = nb) (PyG's `weight [R, nb, in/nb, out/nb]`):
 *   rgcn_block_diag_expand : W [R, nb*bi, nb*bo] = blockdiag(blocks[r, 0], .., blocks[r, nb-1]) per relation; every
 *                            element is written (explicit zeros off the blocks)
 *   rgcn_block_diag_gather : g_blocks[r, k, c, d] = gW[r, k*bi + c, k*bo + d]   (the compact gradient; copies only)
 * blocks / g_blocks [R, nb, bi, bo], W / gW [R, nb*bi, nb*bo], row-major fp32, 16-byte aligned; allocate nothing.
 * ------------------------------------------------------------------------------------------ */
int rgcn_block_diag_expand(const float* blocks, int32_t R, int32_t nb, int32_t bi, int32_t bo, float* W,
                           rgcn_stream_t stream);
int rgcn_block_diag_gather(const float* gW, int32_t R, int32_t nb, int32_t bi, int32_t bo, float* g_blocks,
                           rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * One layer per call.  rgcn_layer_fwd = rgcn_aggregate_fwd (H into the first R blocks of the operand planes, x_root
 * appended as the last block by the same kernel) + rgcn_transform_fwd: everything `RGCNConv.forward` does at
 * src/models/rgcn.py:123 / :128 (+ the ReLU / dropout of :124-125 when asked).  rgcn_layer_bwd = rgcn_split_planes
 * (G = g_out * mask) + rgcn_transform_dgrad + rgcn_aggregate_bwd + rgcn_transform_wgrad: its autograd backward
 * (src/train.py:306).  Same kernels, same results as the separate calls; one foreign call instead of 5-7, which is
 * what bounds the step when the reference's unmodified loop drives the modules eagerly from Python.
 * weight is [R * d_in, d_out] row-major (RGCNConv.weight viewed 2-D), modes / dropout / peers as in rgcn_transform_fwd.
 * ------------------------------------------------------------------------------------------ */
typedef struct rgcn_layer_fwd_args {
  const rgcn_csr_t* csr;                    /* (dst, relation) orientation                                   */
  const float* x_src; int64_t ld_x_src;     /* [n_src, d_in] rows the edges gather from                      */
  const float* x_root; int64_t ld_x_root;   /* [n_dst, d_in] rows being updated (== x_src on one GPU)        */
  int32_t d_in, d_out, relu, mode;
  const float* weight; const float* root; const float* bias;
  float dropout_p; uint32_t dropout_seed; unsigned long long* dropout_counter;
  void* A_hi; void* A_lo; int64_t lda;      /* out: operand planes [n_dst, >= (R+1) d_in], kept for backward */
  float* out; int64_t ldo;                  /* out: [n_dst, d_out]                                           */
  float* const* peer_out_host; int32_t n_peer; int64_t peer_row0, peer_ld;
  void* agg_workspace; size_t agg_workspace_bytes;     /* rgcn_aggregate_workspace_bytes(csr, d_in)           */
  void* gemm_workspace; size_t gemm_workspace_bytes;   /* rgcn_transform_workspace_bytes(n_dst, (R+1) d_in, d_out) */
  /* Optional (NULL: the weights are converted into gemm_workspace on every call, forward and dgrad each): persistent
   * buffer of rgcn_weight_planes_bytes((R+1) d_in, d_out) bytes, 256-byte aligned.  The call converts [weight; root] into
   * it ONCE (rgcn_prepare_weights), reads it as the MN-major operand of the transform, and rgcn_layer_bwd reads the same
   * buffer for its dgrad.  With it the call may also PIPELINE: the walk of row chunk c + 1 runs on `stream` while the
   * transform of chunk c (and, in the partitioned path, its peer stores = the all-gather) runs on an internal side
   * stream, joined before the call returns.  pipeline: 0 = the library decides (never: measured slower on one and
   * two GPUs, see csrc/layer.cu; RGCN_PIPELINE=1 opts in), 1 = never, 2 = always, 3 = the FUSED schedule: walk and
   * transform in one kernel, the operand [H | X] handed over through shared memory (csrc/fused_layer.cu; d_in a
   * multiple of 64, d_out a multiple of 16 up to 256, fp32 gathers; otherwise the call falls back to schedule 1;
   * RGCN_FUSED_FWD=1 selects it for schedule 0.  Measured slower than schedule 1 on the B200, so never the default). */
  void* w_planes; size_t w_planes_bytes; int32_t pipeline;
  /* bf16-transform mode (mode 1, needs w_planes), all optional: x_bf16 = a bf16 copy of x (x_src == x_root, d_in % 8 == 0):
   * the walk gathers IT (half the bytes of the dominant kernel; sums stay fp32);  out_bf16 = where to leave the bf16 copy
   * of this layer's output for the next layer (d_out % 4 == 0). */
  const void* x_bf16; int64_t ld_x_bf16; void* out_bf16; int64_t ld_out_bf16;
  /* Listed-rows form (rows != NULL; needs w_planes, no dropout; peers receive the listed rows only): only rows[0 .. n_list) of the layer's output
   * are wanted — the 2 * batch (head, tail) rows the link-prediction decoder reads from the LAST layer,
   * src/models/rgcn.py:325-326.  The walk visits those rows only, A_hi / A_lo are COMPACT planes
   * [rgcn_rows_compact_size(n_list), >= (R+1) d_in] in list order (padding rows zero; hand them to rgcn_layer_bwd with
   * a_compact = 1), the transform runs over them and stores row c at out[rows[c], :]; all other rows of `out` are left
   * untouched.  rows / slot as built by rgcn_rows_list_build; a row listed twice is computed once (later duplicate
   * positions of A are zero rows). */
  const int64_t* rows; int64_t n_list; const int32_t* slot;
  /* Row of the LAYER'S output that local row 0 is, for the fused dropout's element index only (0 on one GPU).  A
   * destination-range shard passes the global id of its first node, so node v draws the same keep mask on every shard
   * count; without it every shard would repeat the mask of the first shard's rows.  Needs w_planes when dropout_p > 0. */
  int64_t dropout_row0;
} rgcn_layer_fwd_args;

typedef struct rgcn_layer_bwd_args {
  const rgcn_csr_t* csr_t;                  /* (src, relation) orientation with edge weights                 */
  const float* g_out; int64_t ld_g_out;     /* [n_dst, d_out]                                                */
  const float* relu_mask; int64_t ld_mask; float mask_scale;   /* layer output (NULL: no ReLU), 1 / (1 - p)  */
  int64_t n_dst; int32_t d_in, d_out, mode, add_root_term;
  const float* weight; const float* root;
  const void* A_hi; const void* A_lo; int64_t lda;             /* planes saved by rgcn_layer_fwd             */
  void* G_hi; void* G_lo; int64_t ldg;      /* scratch planes [n_dst, d_out]                                 */
  float* colsum_partial;                    /* scratch [rgcn_split_planes_blocks(n_dst, d_out), d_out]       */
  float* gA; int64_t ld_gA;                 /* scratch [n_dst, (R+1) d_in]; NULL: no input gradient wanted   */
  float* g_x; int64_t ld_g_x;               /* out [n_src, d_in] (NULL: only gA is wanted); with add_root_term the
                                               root-term gradient gA[:, R d_in:] is added (one-GPU case)       */
  float* g_weight; float* g_root; float* g_bias;               /* out, NULL: not wanted                      */
  void* agg_workspace; size_t agg_workspace_bytes;
  void* gemm_workspace; size_t gemm_workspace_bytes;
  /* Row-sparse form (rows != NULL): the caller guarantees that g_out is zero outside the listed rows — the 2 * batch
   * (head, tail) rows the link-prediction loss reads from the encoder output, src/models/rgcn.py:325-326, so this is the
   * backward of the LAST layer in the reference's training step (src/train.py:291-306).  With m_c =
   * rgcn_rows_compact_size(n_list) the scratch shapes become: G planes [m_c, d_out], gA [m_c + 1, (R+1) d_in] (row m_c
   * is the zero row), colsum_partial [rgcn_rows_compact_blocks(n_list), d_out], gemm workspace for m_c rows; relu_mask
   * must be NULL and add_root_term set.  Results equal the dense form (absent rows only ever add exact zeros). */
  const int64_t* rows; int64_t n_list;      /* device list of node ids, duplicates allowed                    */
  int32_t* slot;                            /* scratch [n_dst]                                                */
  void* Ac_hi; void* Ac_lo; int64_t ldac;   /* scratch planes [m_c, (R+1) d_in] (weight gradient wanted)      */
  /* Cross-layer hand-over of the masked output gradient (both optional):
   * next_G   : the walk also writes g_x masked for the upstream layer as that layer's G planes (see above);
   * g_ready  : G_hi / G_lo / colsum_partial (n_colsum_ready rows) ALREADY hold this layer's masked output gradient —
   *            written by the downstream layer's next_G — so the rgcn_split_planes pass over g_out is skipped. */
  const rgcn_masked_planes_out* next_G;
  int32_t g_ready; int32_t n_colsum_ready;
  int32_t slot_ready;                       /* row-sparse form: `slot` already holds the map for `rows` (written by
                                               rgcn_link_loss_bwd_rows for this very list): skip building it        */
  const void* w_planes;                     /* optional: the weight planes rgcn_layer_fwd prepared (dgrad reads them) */
  int32_t a_compact;                        /* row-sparse form: A_hi / A_lo are the compact planes of the listed-rows
                                               forward over this very list (no copy; Ac_* unused)                   */
  const rgcn_csr_t* csr_fwd; uint8_t* src_flag;   /* row-sparse form, optional (both or none): the forward-orientation CSR
                                               and n_src bytes of scratch -> the walk skips the sources that have no edge
                                               into a listed row (rgcn_aggregate_bwd_rows_marked); for graphs much
                                               larger than the row list                                             */
} rgcn_layer_bwd_args;

/* Compaction step of the row-sparse backward (csrc/rowsparse.cu), also callable on its own:
 * slot[i] = first position of node i in rows[0 .. n_list) or m_c; G planes row c = g_out[rows[c]] when slot[rows[c]] == c
 * else zeros; Ac planes likewise from A (optional); colsum_partial = per-block column sums of the G rows (optional);
 * zero_row[0 .. zero_cols) is cleared (optional: the zero row of the dgrad output).  slot_ready != 0: `slot` was built
 * for this list already (rgcn_link_loss_bwd_rows) and is used as it is. */
int64_t rgcn_rows_compact_size(int64_t n_list);       /* m_c = n_list rounded up to a multiple of 128 */
int64_t rgcn_rows_compact_blocks(int64_t n_list);     /* rows of colsum_partial                       */
int rgcn_rows_compact(const int64_t* rows, int64_t n_list, int64_t n_nodes, int32_t* slot,
                      const float* g_out, int64_t ld_g_out, int32_t d_out, void* G_hi, void* G_lo, int64_t ldg,
                      const void* A_hi, const void* A_lo, int64_t lda, int32_t K, void* Ac_hi, void* Ac_lo,
                      int64_t ldac, float* colsum_partial, float* zero_row, int32_t zero_cols, int32_t slot_ready,
                      rgcn_stream_t stream);

/* Weights converted once per layer call: bf16 hi (, lo) planes of the row-major [K1 + K2, d_out] block [W1; W2] exactly
 * as PyTorch stores it (row stride padded to a multiple of 8).  rgcn_transform_fwd_w reads them as the MN-major B operand
 * of the tcgen05 kernel (no transposed copy), rgcn_transform_dgrad_w as the K-major one; otherwise they are
 * rgcn_transform_fwd / rgcn_transform_dgrad.  dropout_counter (nullable) is advanced by the conversion kernel, as the
 * conversion inside rgcn_transform_fwd does.  row_offset: row of the layer's output that row 0 of this call is (the
 * fused dropout hashes the GLOBAL element index, so row-chunked calls of one layer draw one consistent mask).
 * out_bf16 (nullable, [n_rows, ld_out_bf16] bf16): the same output rounded to bf16 — the gather source of the next layer
 * in the bf16-transform mode (rgcn_aggregate_fwd_bf16). */
size_t rgcn_weight_planes_bytes(int32_t K, int32_t d_out);
int rgcn_prepare_weights(const float* W1, int32_t K1, const float* W2, int32_t K2, int32_t d_out, int32_t mode,
                         void* w_planes, unsigned long long* dropout_counter, rgcn_stream_t stream);
int rgcn_transform_fwd_w(const void* A_hi, const void* A_lo, int64_t lda, int32_t K, const void* w_planes,
                         const float* bias, int32_t relu, int64_t n_rows, int32_t d_out, float* out, int64_t ldo,
                         int32_t mode, float dropout_p, uint32_t dropout_seed, const unsigned long long* dropout_counter,
                         int64_t row_offset, float* const* peer_out_host, int32_t n_peer, int64_t peer_row0, int64_t peer_ld,
                         void* out_bf16, int64_t ld_out_bf16, rgcn_stream_t stream);
int rgcn_transform_dgrad_w(const void* G_hi, const void* G_lo, int64_t ldg, int32_t d_out, const void* w_planes, int32_t K,
                           int64_t n_rows, float* gA, int64_t ldga, int32_t mode, rgcn_stream_t stream);
/* rgcn_transform_fwd_w over a COMPACT operand [n_rows, K] whose row c belongs to node out_rows[c] (c < n_list; the rows
 * beyond are padding): the epilogue stores row c at out[out_rows[c], :]; only the listed rows of `out` are written.
 * slot (nullable): node -> first list position; a later duplicate position is then not stored.  peer_out_host (n_peer
 * > 0): the listed rows are also stored at rows peer_row0 + out_rows[c] of the peers' buffers. */
int rgcn_transform_fwd_w_rows(const void* A_hi, const void* A_lo, int64_t lda, int32_t K, const void* w_planes,
                              const float* bias, int32_t relu, int64_t n_rows, int32_t d_out, float* out, int64_t ldo,
                              int32_t mode, const int64_t* out_rows, int64_t n_list, const int32_t* slot,
                              float* const* peer_out_host, int32_t n_peer, int64_t peer_row0, int64_t peer_ld,
                              rgcn_stream_t stream);

int rgcn_layer_fwd(const rgcn_layer_fwd_args* a, rgcn_stream_t stream);
int rgcn_layer_bwd(const rgcn_layer_bwd_args* a, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Peer-memory exchange kernels of the destination-range partitioned path (graphs too large for one GPU; the
 * reference is single-device, this is the scale-out of src/models/rgcn.py:123-128 and of its autograd backward).
 * All `*_host` arguments are HOST arrays of DEVICE pointers into buffers of the n GPUs of one NVSwitch domain,
 * peer-mapped into this process; entry q belongs to rank q.  No collective library call is involved: the caller
 * places a cross-GPU barrier between a producer and its consumers.
 *   rgcn_p2p_push_rows    : dst_q[row0 + i, :] = src[i, :] for every q  (all-gather by push of this rank's shard)
 *   rgcn_p2p_reduce_split : v[i, :] = extra[i, :] + sum_q part_q[row0 + i, :]  in rank order (deterministic reduce-
 *                           scatter by pull), then optionally zeroed where relu_mask <= 0 and scaled by mask_scale,
 *                           written as fp32 `out` and / or as bf16 planes hi (, lo) with the same column-sum partials
 *                           as rgcn_split_planes (rgcn_split_planes_blocks(rows, cols) rows of `cols` floats).
 * ------------------------------------------------------------------------------------------ */
/*   rgcn_p2p_pull_rows    : out[rows[c], :] = sum_q part_q[row0 + rows[c], :] (rank order) for the n_list listed LOCAL rows only
 *                           (int64 device list, duplicates allowed; out is [n_rows_out, ldo], other rows untouched): the
 *                           reduce-scatter of a gradient that is zero outside a short row list. */
int rgcn_p2p_pull_rows(const float* const* part_host, int32_t n_part, int64_t row0, int64_t ld_part, const int64_t* rows,
                       int64_t n_list, int64_t n_rows_out, int32_t cols, float* out, int64_t ldo, rgcn_stream_t stream);
int rgcn_p2p_push_rows(const float* src, int64_t ld_src, int64_t rows, int32_t cols,
                       float* const* dst_host, int32_t n_dst, int64_t row0, int64_t ld_dst, rgcn_stream_t stream);
int rgcn_p2p_reduce_split(const float* const* part_host, int32_t n_part, int64_t row0, int64_t ld_part,
                          const float* extra, int64_t ld_extra, const float* relu_mask, int64_t ldm, float mask_scale,
                          int64_t rows, int32_t cols, float* out, int64_t ldo, void* hi, void* lo, int64_t ldp,
                          float* colsum_partial, rgcn_stream_t stream);

/* All-reduce of one flat fp32 buffer over the n GPUs (data-parallel replicas of graphs that fit one GPU exchange their
 * parameter gradients with it; no reference counterpart — reference README.md:624-627 lists multi-GPU as future work).
 * Two-shot over peer-mapped memory, CUDA-graph capturable, deterministic: rank r sums slice r of every rank's `in` in rank
 * order, scales it and stores it into slice r of EVERY rank's `out` (in and out must be different buffers); arrival / done
 * flags are monotone epochs kept by a device-side counter that the call itself advances.
 *   in_host / out_host / flags_host : host arrays of n device pointers (peer-mapped; entry q = rank q); every flag block
 *                                     is rgcn_p2p_allreduce_flag_bytes() bytes, ZEROED once before first use
 *   epoch_counter : local device uint32, zeroed once; status (nullable): bit 1 set when a peer never arrived (the waits
 *                   give up after a few seconds instead of hanging the GPU). */
size_t rgcn_p2p_allreduce_flag_bytes(void);
int rgcn_p2p_allreduce(const float* const* in_host, float* const* out_host, unsigned int* const* flags_host,
                       int32_t n_ranks, int32_t rank, int64_t n_floats, float scale, unsigned int* epoch_counter,
                       int32_t* status, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * DistMult decoder.  Replaces node_embeddings[head], [tail] (src/models/rgcn.py:325-326) +
 * LinkPredictor.forward (src/models/rgcn.py:207-211) with one gather-and-score kernel:
 *   score[p] = sum_k emb_h[hp, k] * r_p[k] * emb_t[tp, k],   hp = head ? head[p] : p, tp likewise
 * (head == tail == NULL is the stand-alone LinkPredictor.forward on already gathered rows;
 *  emb_h == emb_t == encoder output with index arrays is the fused DrugDiseaseModel.forward).
 * r_p = rel_rows[p, :] when rel_rows != NULL (rows already gathered and dropped-out by the
 * caller), else rel_table[rel[p], :]; either is multiplied element-wise by rel_scale[p, :] when
 * rel_scale != NULL (the dropout mask / (1 - p) of src/models/rgcn.py:208, drawn by the caller).
 * Backward: g_h[hp] += g[p] * r_p * t_p ; g_t[tp] += g[p] * h_p * r_p ;
 *           g_rel_rows[p] = g[p] * h_p * t_p  and/or  g_rel_table[rel[p]] += the same.
 * With an index array the target rows may repeat: the buffer must be zero-filled by the caller
 * and duplicates are combined with fp32 atomics; without one the rows are plain stores.
 * ------------------------------------------------------------------------------------------ */
int rgcn_distmult_fwd(const float* emb_h, int64_t ld_h, const float* emb_t, int64_t ld_t,
                      const int64_t* head, const int64_t* tail, const int64_t* rel,
                      const float* rel_table, const float* rel_rows, const float* rel_scale,
                      int64_t n_pairs, int32_t d, float* score, rgcn_stream_t stream);
int rgcn_distmult_bwd(const float* emb_h, int64_t ld_h, const float* emb_t, int64_t ld_t,
                      const int64_t* head, const int64_t* tail, const int64_t* rel,
                      const float* rel_table, const float* rel_rows, const float* rel_scale,
                      const float* g_score, int64_t n_pairs, int32_t d, float* g_h, int64_t ld_gh, float* g_t, int64_t ld_gt,
                      float* g_rel_table, float* g_rel_rows, rgcn_stream_t stream);
/* ------------------------------------------------------------------------------------------
 * All-pairs scoring / ranking (fp32).  A is a prepared query matrix (rgcn_rows_prepare: gather rows of the
 * encoder output, optionally times the relation row (DistMult h * r, src/models/rgcn.py:235-238) and / or
 * L2-normalised (cosine, src/compare_methods.py:384-397)); B is the candidate matrix, optionally gathered
 * through b_idx.
 *   rgcn_allpairs_scores: out[i, j] = alpha * <A[i], B[b_idx[j]]> + beta      (score_all_tails, src/models/rgcn.py:241;
 *                          (cos + 1) / 2 with alpha = beta = 0.5; the 6,282 x 5,593 drug-disease sweep)
 *   rgcn_allpairs_rank  : thr[i] = <A[i], B[true_pos[i]]>;  greater[i] / equal[i] = number of candidates j != true_pos[i]
 *                          scoring above / exactly at thr[i].  rank = 1 + greater reproduces the argsort loop of
 *                          src/evaluate.py:260-276 without materialising the [queries, candidates] matrix.
 * true_pos indexes the candidate list (positions in b_idx when given).
 * ------------------------------------------------------------------------------------------ */
int rgcn_rows_prepare(const float* emb, int64_t ld, const int64_t* idx, int64_t n, int32_t d,
                      const float* rel_table, const int64_t* rel, int32_t normalize,
                      float* out, int64_t ldo, rgcn_stream_t stream);
int rgcn_allpairs_scores(const float* A, int64_t lda, int64_t na, const float* B, int64_t ldb,
                         const int64_t* b_idx, int64_t nb, int32_t d, float alpha, float beta,
                         float* out, int64_t ldo, rgcn_stream_t stream);
int rgcn_allpairs_rank(const float* A, int64_t lda, int64_t nq, const float* B, int64_t ldb,
                       const int64_t* b_idx, int64_t nb, int32_t d, const int64_t* true_pos,
                       float* thr, int32_t* greater, int32_t* equal, rgcn_stream_t stream);
/* The same two counts from a MATERIALISED score block scores[nq, ld] (first n_cand columns; e.g. produced on the tensor
 * cores by rgcn_transform_dgrad(A' planes, candidate rows)): the threshold is scores[i, true_pos[i]], the true tail is
 * excluded by index.  thr (optional) receives the thresholds. */
int rgcn_rank_count(const float* scores, int64_t ld, int64_t nq, int64_t n_cand, const int64_t* true_pos,
                    float* thr, int32_t* greater, int32_t* equal, rgcn_stream_t stream);
/* Exclusion lists (filtered ranking, top-k of novel links): row i of the queries excludes the candidate positions
 * excl_pos[excl_begin[i] .. excl_end[i]) (int32, sorted ascending and distinct within each range; positions >= n_cand are
 * ignored; ranges of different rows may overlap or share storage).  The excluding entry points take the three pointers
 * together: all null (no filter) or none.
 *   rgcn_rank_excl_correct : turns the counts of rgcn_rank_count / rgcn_allpairs_rank into filtered counts: for every
 *                            excluded j != true_pos[i] it subtracts [s_ij > thr[i]] from greater[i] and [s_ij == thr[i]]
 *                            from equal[i].  s_ij is read from the score block `scores` (ld) when it is given, else
 *                            recomputed as rgcn_allpairs_rank computes it (A, B, b_idx, d: fmaf in ascending k).  thr is the
 *                            counting pass's threshold (its thr output). */
int rgcn_rank_excl_correct(const float* scores, int64_t ld, const float* A, int64_t lda, const float* B, int64_t ldb,
                           const int64_t* b_idx, int32_t d, int64_t nq, int64_t n_cand, const int64_t* true_pos,
                           const float* thr, const int64_t* excl_begin, const int64_t* excl_end, const int32_t* excl_pos,
                           int32_t* greater, int32_t* equal, rgcn_stream_t stream);
/* The same sweeps on the tensor cores WITHOUT the [queries, candidates] matrix: the tcgen05 kernel's epilogue consumes the
 * accumulator (three bf16 products, fp32 accumulation, as the fp32 mode of the transforms).
 *   Q_hi / Q_lo     : the prepared query rows (rgcn_rows_prepare) as bf16 planes [n_q, d] (rgcn_split_planes)
 *   cand_planes     : rgcn_prepare_weights(candidate rows [n_cand, d], K1 = n_cand, d_out = d, mode 0)
 *   rgcn_scores_diag_w : thr[i] = <q_i, c_i> from the DIAGONAL tiles of Q x T^T, T = the true tails gathered per query and
 *                        prepared like cand_planes ([n_q, d]): same K order and products as the sweep, so thr[i] carries the
 *                        bits the sweep computes for (i, true_pos[i]) and exact ties with other candidates count as ties
 *   rgcn_scores_rank_w : greater[i] / equal[i] += #{j != true_pos[i] : s_ij > / == thr[i]}   (zero both first)
 *                        -> rank = 1 + greater: score_all_tails + the per-row argsort of src/evaluate.py:260-276
 *   rgcn_scores_topk_w : per query the k <= 16 best candidates, value alpha * s + beta (alpha > 0) and position in the
 *                        candidate list, sorted by value (ties: lower position first): the cosine sweeps + top-k /
 *                        threshold filters of src/compare_methods.py:384-397, src/medical_validation.py:222-239,
 *                        src/case_studies.py:260-274.  Scratch: cand_val / cand_idx [n_q, n_slots, 16] with n_slots >=
 *                        rgcn_scores_topk_slots(n_q, n_cand), slot_ctr [n_q] (cleared by the call).  The slot count is
 *                        the number of partial lists a row can receive (two per CTA run over its row tile, at most
 *                        2 (#SMs + 1)); fewer slots are rejected.
 *   rgcn_scores_rank_excl_w / rgcn_scores_topk_excl_w : the same with exclusion lists (format above rgcn_rank_excl_correct;
 *                        all three null = the unfiltered call).  rank: an excluded column counts in neither greater nor
 *                        equal (the true tail stays excluded by index; listing it changes nothing).  top-k: an excluded
 *                        column is never a candidate; a row with fewer than k admissible columns ends in -inf / -1. */
int rgcn_scores_diag_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* tail_planes, int64_t n_q,
                       float* thr, rgcn_stream_t stream);
int rgcn_scores_rank_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes, int64_t n_cand,
                       int64_t n_q, const float* thr, const int64_t* true_pos, int32_t* greater, int32_t* equal,
                       rgcn_stream_t stream);
int32_t rgcn_scores_topk_slots(int64_t n_q, int64_t n_cand);
int rgcn_scores_topk_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes, int64_t n_cand,
                       int64_t n_q, int32_t k, float alpha, float beta, float* cand_val, int32_t* cand_idx,
                       int32_t* slot_ctr, int32_t n_slots, float* out_val, int64_t* out_idx, rgcn_stream_t stream);
int rgcn_scores_rank_excl_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                            int64_t n_cand, int64_t n_q, const float* thr, const int64_t* true_pos, int32_t* greater,
                            int32_t* equal, const int64_t* excl_begin, const int64_t* excl_end, const int32_t* excl_pos,
                            rgcn_stream_t stream);
int rgcn_scores_topk_excl_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                            int64_t n_cand, int64_t n_q, int32_t k, float alpha, float beta, float* cand_val,
                            int32_t* cand_idx, int32_t* slot_ctr, int32_t n_slots, float* out_val, int64_t* out_idx,
                            const int64_t* excl_begin, const int64_t* excl_end, const int32_t* excl_pos,
                            rgcn_stream_t stream);
/* ------------------------------------------------------------------------------------------
 * Fused link-prediction loss.  Replaces nn.BCEWithLogitsLoss (mean) over the batch logits and the
 * sigmoid > 0.5 accuracy count (src/train.py:139, :300, :321-322):
 *   loss = mean_i [ max(x,0) - x*y + log1p(exp(-|x|)) ],  n_correct = #{(x_i > 0) == y_i}   (one block, fixed order)
 *   g_logits[i] = g_loss * (sigmoid(x_i) - y_i) / n
 * ------------------------------------------------------------------------------------------ */
int rgcn_bce_logits_fwd(const float* logits, const float* labels, int64_t n, float* loss,
                        int32_t* n_correct, rgcn_stream_t stream);
int rgcn_bce_logits_bwd(const float* logits, const float* labels, int64_t n, const float* g_loss,
                        float* g_logits, rgcn_stream_t stream);
/* ------------------------------------------------------------------------------------------
 * Fused tail of the training step (the caller-side code of src/train.py:276-300, :321-322 around the model call).
 *   rgcn_link_batch    : NegativeSampler.sample (src/train.py:59-97) + the pos/neg concatenation and labels of :281-288:
 *                        out[0 .. n_pos) = positives (label 1), out[n_pos + i*num_neg + k] = positive i with its head
 *                        (probability 1/2) or else its tail replaced by a uniform node (label 0).  Counter-based RNG
 *                        (seed, device counter advanced by the call): fresh negatives on every CUDA-graph replay.
 *   rgcn_link_loss_fwd : scores (src/models/rgcn.py:325-329, relation dropout of :207-208 by counter-based mask),
 *                        loss = mean BCE-with-logits (src/train.py:139, :300) and the count of correct sigmoid > 0.5
 *                        predictions (:321-322) in ONE kernel; `state` receives the dropout counter value used.
 *   rgcn_link_loss_bwd : d loss / d emb scattered into the dense, pre-zeroed g_emb [N, d]; d loss / d rel_table (optional,
 *                        pre-zeroed; n_rel = its row count, used to pre-reduce the block's pairs in shared memory).
 *                        Scores-only form (LinkPredictor.score_pairs with the same counter-based relation dropout):
 *                        labels = loss = NULL in the forward; g_score [n_pairs] = the incoming gradient of the scores
 *                        in the backward (labels, score, g_loss then unused).
 *                        workspace: rgcn_link_loss_workspace_bytes(n_pairs), ZEROED once before first use.
 *                        (fp32 atomics on repeated rows: the sum order differs from run to run.)
 *   rgcn_link_loss_bwd_rows : the DETERMINISTIC form of the same backward, and the one the modules use.  No floating-point
 *                        atomics: slot[i] (int32 [n_nodes], out) = first position of node i in rows (int64 [2 n_pairs],
 *                        out: the heads then the tails) or rgcn_rows_compact_size(2 n_pairs) when nobody lists it; every
 *                        position's contribution is computed in parallel, then the owner position's warp adds the
 *                        contributions to its node in ascending position order and every row of g_emb [n_nodes, d] is
 *                        written exactly once (no pre-zeroing); listed_only != 0: only the LISTED rows are written —
 *                        for a consumer that reads nothing else, the listed-rows form of the last encoder layer
 *                        (rgcn_layer_fwd with rows) — and the rest of g_emb stays undefined.
 *                        g_rel_table = fixed-order sum of per-32-pair partials.
 *                        workspace (always needed, 16-byte aligned): rgcn_link_bwd_rows_workspace_bytes.
 *                        slot / rows are exactly what rgcn_layer_bwd's row-sparse form wants (slot_ready = 1).
 *   Index range: with n_nodes > 0 a pair whose head / tail is outside [0, n_nodes) or whose relation is outside
 *                        [0, n_rel) is skipped — NaN score and loss, no gradient — and bit 0 of *status (nullable) is
 *                        set; the reference's nn.Embedding raises a device-side assert at the same place.
 * ------------------------------------------------------------------------------------------ */
int rgcn_link_batch(const int64_t* pos_head, const int64_t* pos_tail, const int64_t* pos_rel, int64_t n_pos,
                    int32_t num_neg, int64_t num_nodes, uint32_t seed, unsigned long long* counter,
                    int64_t* heads, int64_t* tails, int64_t* rels, float* labels, rgcn_stream_t stream);

/* Generalised negative sampler: rgcn_link_batch plus filtered (Bordes et al. 2013), type-constrained (Krompaß et al.
 * 2015) and Bernoulli head / tail (Wang et al. 2014) negatives.  Same layout as rgcn_link_batch; rgcn_link_batch is
 * this call with no tables and one block.
 *   side    : negative i of positive q replaces its head with probability head_prob[rel_q] (NULL: 1/2), else its tail;
 *             chosen once, from attempt 0's draw.
 *   entity  : attempt j draws uniformly from the side's admissible list of rel_q (the multiply-shift of a 32-bit
 *             draw into the list length; an empty list = all num_nodes nodes) and is rejected when the corrupted
 *             triple is in the filter.  After max_tries rejections the last draw is kept (label 0 all the same) and
 *             *exhausted (nullable) is incremented.
 *   draws   : a counter-based hash of (seed, *counter, i, j); attempt 0 is rgcn_link_batch's draw, so with no tables
 *             and head_prob = NULL the output is rgcn_link_batch's, bit for bit.  A positive whose relation is outside
 *             [0, num_rel) gets an unconstrained, unfiltered draw with head probability 1/2.
 *   filter  : the forward index of known triples: filter_keys [n_filter] = head * num_rel + rel ascending, filter_tails
 *             [n_filter] ascending within each key (KnownTriples.keys / .tails).  Both NULL: no filter.
 *   types   : head_offsets / tail_offsets [num_rel + 1] (CSR) into head_nodes / tail_nodes: the admissible heads /
 *             tails of each relation.  All four NULL: unconstrained.
 *   counter : advanced by exactly one per call; every block draws with the value before the call.  ticket NULL: one
 *             block of 1024 threads; otherwise one thread per output entry, and the last block to finish advances the
 *             counter and resets *ticket (an unsigned int, ZEROED once before first use).
 * The struct is read on the host and passed to the kernel by value.  Arguments are checked before any CUDA call. */
typedef struct rgcn_link_batch_args {
  const int64_t* pos_head;
  const int64_t* pos_tail;
  const int64_t* pos_rel;
  int64_t n_pos;
  int32_t num_neg;
  int32_t num_rel;            /* rows of head_prob and of the type tables; may be 0 when none is given */
  int64_t num_nodes;
  uint32_t seed;
  int32_t max_tries;          /* >= 1 */
  unsigned long long* counter;
  int64_t* heads;
  int64_t* tails;
  int64_t* rels;
  float* labels;
  const float* head_prob;     /* [num_rel] in [0, 1], nullable */
  const int64_t* filter_keys;
  const int32_t* filter_tails;
  int64_t n_filter;
  const int64_t* head_offsets;
  const int32_t* head_nodes;
  const int64_t* tail_offsets;
  const int32_t* tail_nodes;
  unsigned long long* exhausted;
  unsigned int* ticket;
} rgcn_link_batch_args;

int rgcn_link_batch_ex(const rgcn_link_batch_args* args_host, rgcn_stream_t stream);
size_t rgcn_link_loss_workspace_bytes(int64_t n_pairs);
int rgcn_link_loss_fwd(const float* emb, int64_t ld, const int64_t* head, const int64_t* tail, const int64_t* rel,
                       const float* rel_table, const float* labels, int64_t n_pairs, int32_t d, float dropout_p,
                       uint32_t seed, unsigned long long* counter, unsigned long long* state, float* score,
                       float* loss, int32_t* n_correct, int64_t n_nodes, int32_t n_rel, int32_t* status,
                       void* workspace, size_t workspace_bytes, rgcn_stream_t stream);
int rgcn_link_loss_bwd(const float* emb, int64_t ld, const int64_t* head, const int64_t* tail, const int64_t* rel,
                       const float* rel_table, const float* labels, const float* score, const float* g_loss,
                       const float* g_score,
                       int64_t n_pairs, int32_t d, float dropout_p, uint32_t seed, const unsigned long long* state,
                       float* g_emb, int64_t ld_g, float* g_rel_table, int32_t n_rel, int64_t n_nodes,
                       rgcn_stream_t stream);
size_t rgcn_link_bwd_rows_workspace_bytes(int64_t n_pairs, int32_t n_rel, int32_t d);
int rgcn_link_loss_bwd_rows(const float* emb, int64_t ld, const int64_t* head, const int64_t* tail, const int64_t* rel,
                            const float* rel_table, const float* labels, const float* score, const float* g_loss,
                            const float* g_score, int64_t n_pairs, int32_t d, float dropout_p, uint32_t seed,
                            const unsigned long long* state, int64_t n_nodes, int32_t n_rel, float* g_emb, int64_t ld_g,
                            float* g_rel_table, int32_t* slot, int64_t* rows, int32_t* status, int32_t listed_only,
                            void* workspace, size_t workspace_bytes, rgcn_stream_t stream);

/* flag[0] = 1 when any head/tail is outside [0, n_nodes) or any rel outside [0, n_rel). */
int rgcn_check_pairs(const int64_t* head, const int64_t* tail, const int64_t* rel, int64_t n_pairs,
                     int64_t n_nodes, int32_t n_rel, int32_t* flag, rgcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Optimiser step.  Replaces torch.nn.utils.clip_grad_norm_(params, max_norm) + torch.optim.Adam / AdamW .step()
 * (reference src/train.py:311-318) with two kernels (one without clipping) over a table of parameter segments.
 *
 *   clipping (max_grad_norm >= 0): total_norm = ||all grads||_2 (per-block partial sums, fp64, reduced in a fixed
 *     order: bitwise run-to-run deterministic), clip_coef = min(max_grad_norm / (total_norm + 1e-6), 1);
 *     *grad_norm = total_norm (nullable).  The clipped gradient is used on the fly; grad is NOT written.
 *   update, per element, in the order of torch.optim.Adam's single-tensor path (fp32; the per-step scalars in fp64
 *     from the segment's step + 1, rounded to fp32):
 *     g = grad * clip_coef;  decoupled ? p *= 1 - lr*wd : g += wd*p  (when wd != 0);  m = lerp(m, g, 1 - beta1);
 *     v = beta2*v + (1 - beta2)*g*g;  p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps);
 *     and every segment's *step += 1 once all blocks have read it.
 *
 *   segments_host : host array of n_segments (at most RGCN_ADAM_MAX_SEGMENTS) descriptors, passed to the kernels BY
 *                   VALUE (a captured CUDA graph keeps the pointers; no table copy).  param / exp_avg / exp_avg_sq /
 *                   grad are fp32 [numel]; step is one fp32 (torch's state['step']); group indexes hparams.
 *   hparams       : DEVICE array of n_groups rgcn_adam_hparams, read by every launch (an lr change between replays of
 *                   a captured step takes effect without re-capturing).
 *   workspace     : rgcn_adam_workspace_bytes(total numel of the segments, n_segments) bytes, ZEROED once before first
 *                   use (it holds two arrival counters that every call leaves at zero).
 * n_segments == 0 enqueues nothing; it loads the kernels, so that a later call under stream capture loads no module.
 * ------------------------------------------------------------------------------------------ */
#define RGCN_ADAM_MAX_SEGMENTS 64

typedef struct rgcn_adam_segment {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  float* step;
  int64_t numel;
  int32_t group;
} rgcn_adam_segment;

typedef struct rgcn_adam_hparams {
  double lr, beta1, beta2, eps, weight_decay;
  int32_t decoupled_weight_decay; /* 1: AdamW's p *= 1 - lr*wd; 0: Adam's L2 term g += wd*p */
} rgcn_adam_hparams;

size_t rgcn_adam_workspace_bytes(int64_t total_numel, int32_t n_segments);
int rgcn_adam_step(const rgcn_adam_segment* segments_host, int32_t n_segments, const rgcn_adam_hparams* hparams,
                   int32_t n_groups, float max_grad_norm, float* grad_norm, void* workspace, size_t workspace_bytes,
                   rgcn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RGCN_B200_H_ */
