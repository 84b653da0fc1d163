// One RGCN layer per call: the sequences of kernels behind `RGCNConv.forward` (reference call sites
// src/models/rgcn.py:123, :128) and behind its autograd backward (src/train.py:306), enqueued by ONE C call each.
// Nothing new is computed here — the calls below are the library's own entry points — but a Python host then pays
// one foreign call per layer and direction instead of five to seven, which is what bounds the step when the
// reference's unmodified training loop drives the modules eagerly (no CUDA graph).
#include "common.cuh"

#include <stdlib.h>

using namespace rgcn;

// csrc/fused_layer.cu: walk + transform of one layer in one kernel (the operand [H | X] goes through shared memory)
namespace rgcn {
int fused_layer_fwd_eligible(const rgcn_layer_fwd_args* a);
int fused_layer_fwd_launch(const rgcn_layer_fwd_args* a, cudaStream_t st);
}

// The weight-gradient contraction (tensor pipe) and the transposed walk (L2 / latency bound) of one layer's backward
// both depend only on G and on the dgrad output respectively, not on each other: the wgrad runs on a side stream while
// the main stream walks the graph, forked AFTER the dgrad launch (so the dgrad, which the walk waits for, gets the SMs
// first) and joined before the call returns.  Inside a stream capture the fork / join becomes two branches of the graph.
// Default: only while the stream is being captured into a CUDA graph — an eagerly driven step is bound by the host, and
// the four extra event calls per layer only add to that.  RGCN_OVERLAP_WGRAD=0 never forks, =1 always does.
namespace {
struct SideStream {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
// `create` = false while a capture is in progress: creating streams / events there could invalidate the capture, so the
// objects are made by the first eager call (GraphedTrainStep warms up eagerly before it captures)
SideStream* side_stream(bool create) {
  static SideStream ss[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStream& f = ss[dev];
  if (!f.join) {
    if (!create) return nullptr;
    if (cudaStreamCreateWithFlags(&f.side, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&f.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&f.join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
  }
  return &f;
}
SideStream* overlap_wgrad(cudaStream_t st) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RGCN_OVERLAP_WGRAD");
    v = !e ? 2 : (e[0] == '0' ? 0 : 1);
  }
  if (v == 0) return nullptr;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  const bool capturing = cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive;
  SideStream* ss = side_stream(!capturing);
  return (v == 1 || capturing) ? ss : nullptr;
}
}  // namespace

// dgrad -> [fork: wgrad on the side stream] -> transposed walk -> join.  `m` rows of G / A; `walk` launches the gather.
template <typename Walk>
static int dgrad_walk_wgrad(const rgcn_layer_bwd_args* a, int64_t m, const void* A_hi, const void* A_lo, int64_t lda,
                            int32_t n_colsum, Walk walk, rgcn_stream_t stream) {
  const int R = a->csr_t->R;
  const int K1 = R * a->d_in, K2 = a->d_in;
  const bool need_w = a->g_weight != nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (a->gA) {
    if (a->w_planes)
      rc = rgcn_transform_dgrad_w(a->G_hi, a->G_lo, a->ldg, a->d_out, a->w_planes, K1 + K2, m, a->gA, a->ld_gA, a->mode, stream);
    else
      rc = rgcn_transform_dgrad(a->G_hi, a->G_lo, a->ldg, a->d_out, a->weight, K1, a->root, K2, m, a->gA, a->ld_gA,
                                a->mode, a->gemm_workspace, a->gemm_workspace_bytes, stream);
    if (rc) return rc;
  }
  SideStream* ss = (need_w && a->gA && a->g_x) ? overlap_wgrad(st) : nullptr;
  cudaStream_t wst = st;
  if (ss) {
    RGCN_CUDA(cudaEventRecord(ss->fork, st));
    RGCN_CUDA(cudaStreamWaitEvent(ss->side, ss->fork, 0));
    wst = ss->side;
  }
  if (need_w) {
    rc = rgcn_transform_wgrad(A_hi, A_lo, lda, K1, K2, a->G_hi, a->G_lo, a->ldg, a->d_out, m,
                              a->g_bias ? a->colsum_partial : nullptr, a->g_bias ? n_colsum : 0, a->g_weight, a->g_root,
                              a->g_bias, a->mode, a->gemm_workspace, a->gemm_workspace_bytes, (rgcn_stream_t)wst);
    if (rc) return rc;
  }
  if (ss) RGCN_CUDA(cudaEventRecord(ss->join, ss->side));
  if (a->gA && a->g_x) {
    rc = walk();
    if (rc) return rc;
  }
  if (ss) RGCN_CUDA(cudaStreamWaitEvent(st, ss->join, 0));
  return RGCN_OK;
}

// ---- forward: the walk of row chunk c + 1 under the transform of chunk c --------------------------------------------
// The walk is bound by L2 / HBM gathers, the transform by the tensor pipe and (in the partitioned path) by the NVLink
// stores of its epilogue: run on two streams they overlap instead of adding up.  The hub chunks are reduced once, up
// front; the weights are converted once (rgcn_prepare_weights) and shared by all chunks; a chunk-wise row order
// (rgcn_csr_t::order_chunk_rows) keeps every chunk's rows a contiguous range, which is what the transform needs.
static int pipeline_mode(const rgcn_layer_fwd_args* a, cudaStream_t st, SideStream** ss_out) {
  static int env = -1;
  if (env < 0) {
    const char* e = getenv("RGCN_PIPELINE");
    env = !e ? 2 : (e[0] == '0' ? 0 : 1);
  }
  *ss_out = nullptr;
  int want = a->pipeline == 1 ? 0 : (a->pipeline == 2 ? 1 : env);        // 0 never, 1 always, 2 library decides
  if (want == 0) return 0;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  const bool capturing = cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive;
  SideStream* ss = side_stream(!capturing);
  if (!ss) return 0;
  // Measured, and it LOSES everywhere it was tried, so the library never pipelines on its own (RGCN_PIPELINE=1 or
  // pipeline = 2 opt in): cfg2 (30,926 rows, 4 chunks) 0.530 against 0.446 ms per step — one-wave chunk transforms pay
  // their prologue and pipeline fill per tile while walk blocks hold the SMs; one GPU, 1.25 M rows / 50 M edges / 30
  // relations 89.1 against 84.6 ms; two GPUs with the peer stores in the epilogue 98.5 against 92.8 ms — walk and
  // transform are both bound by the same memory system there (operand planes of 19.8 GB per layer), not by different units.
  if (want == 2) return 0;
  *ss_out = ss;
  return 1;
}

static int64_t pipeline_chunk_rows(const rgcn_csr_t* g) {
  if (g->row_order) return g->order_chunk_rows;                           // 0: global order, cannot be walked in ranges
  int64_t c = (g->n_rows + 7) / 8;                                         // ~8 chunks, whole 128-row tiles
  c = (c + 127) / 128 * 128;
  return c < 8192 ? 8192 : c;
}

extern "C" int rgcn_layer_fwd(const rgcn_layer_fwd_args* a, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(a && a->csr, "layer_fwd: null arguments");
  const int R = a->csr->R;
  const int K1 = R * a->d_in, K2 = a->d_in, K = K1 + K2;
  const int out_mode = a->mode == 0 ? 2 : 1;
  RGCN_CHECK_ARG(a->mode == 0 || a->mode == 1, "layer_fwd: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(a->A_hi && (a->mode == 1 || a->A_lo) && a->lda >= K1 + K2, "layer_fwd: operand planes missing or too narrow");
  RGCN_CHECK_ARG(a->dropout_row0 >= 0 && (a->dropout_row0 == 0 || a->dropout_p == 0.f || a->w_planes),
                 "layer_fwd: dropout_row0 must be >= 0 and needs w_planes with dropout");
  if (!a->w_planes) {
    // the row walk also appends x_root[i] as the last block of row i: the operand [H | X] in one kernel
    int rc = rgcn_aggregate_fwd(a->csr, a->x_src, a->ld_x_src, a->d_in, nullptr, 0, a->A_hi, a->mode == 0 ? a->A_lo : nullptr,
                                a->lda, out_mode, nullptr, 0, nullptr, a->x_root, a->ld_x_root, a->agg_workspace,
                                a->agg_workspace_bytes, stream);
    if (rc) return rc;
    return rgcn_transform_fwd(a->A_hi, a->A_lo, a->lda, K1, K2, a->weight, a->root, a->bias, a->relu, a->csr->n_rows, a->d_out,
                              a->out, a->ldo, a->mode, a->dropout_p, a->dropout_seed, a->dropout_counter, a->peer_out_host,
                              a->n_peer, a->peer_row0, a->peer_ld, a->gemm_workspace, a->gemm_workspace_bytes, stream);
  }
  RGCN_CHECK_ARG(a->w_planes_bytes >= rgcn_weight_planes_bytes(K, a->d_out), "layer_fwd: w_planes too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = a->csr->n_rows;
  int rc = rgcn_prepare_weights(a->weight, K1, a->root, K2, a->d_out, a->mode, a->w_planes,
                                a->dropout_p > 0.f ? a->dropout_counter : nullptr, stream);
  if (rc) return rc;
  void* A_lo = a->mode == 0 ? a->A_lo : nullptr;
  if (a->rows) {
    // listed-rows form: only the rows the caller will read (the 2 * batch head / tail rows of a link-prediction step,
    // src/models/rgcn.py:325-326) are walked and transformed; A comes back COMPACT [m_c, K] in list order, which is the
    // operand layout the row-sparse backward wants (rgcn_layer_bwd, a_compact)
    RGCN_CHECK_ARG(a->n_list > 0 && a->slot && a->dropout_p == 0.f, "layer_fwd: the listed-rows form needs the slot map and excludes dropout");
    const int64_t m_c = rgcn_rows_compact_size(a->n_list);
    const bool g16l = a->mode == 1 && a->x_bf16 && a->d_in % 8 == 0 && a->lda % 8 == 0 && a->x_src == a->x_root;
    if (g16l)
      rc = rgcn_aggregate_fwd_bf16_list(a->csr, a->x_bf16, a->ld_x_bf16, a->d_in, a->A_hi, a->lda, a->x_bf16, a->ld_x_bf16, a->rows,
                                        a->n_list, a->slot, a->agg_workspace, a->agg_workspace_bytes, stream);
    else
      rc = rgcn_aggregate_fwd_list(a->csr, a->x_src, a->ld_x_src, a->d_in, a->A_hi, A_lo, a->lda, out_mode, a->x_root, a->ld_x_root,
                                   a->rows, a->n_list, a->slot, a->agg_workspace, a->agg_workspace_bytes, stream);
    if (rc) return rc;
    return rgcn_transform_fwd_w_rows(a->A_hi, A_lo, a->lda, K, a->w_planes, a->bias, a->relu, m_c, a->d_out, a->out, a->ldo,
                                     a->mode, a->rows, a->n_list, a->slot, a->peer_out_host, a->n_peer, a->peer_row0, a->peer_ld,
                                     stream);
  }
  if (fused_layer_fwd_eligible(a)) {
    // hub chunks first (their partials are what the fused kernel's row walk adds for the long segments)
    if (a->csr->n_chunks > 0) {
      rc = rgcn_aggregate_fwd_rows(a->csr, a->x_src, a->ld_x_src, a->d_in, a->A_hi, A_lo, a->lda, out_mode, a->x_root,
                                   a->ld_x_root, 0, 0, 1, a->agg_workspace, a->agg_workspace_bytes, stream);
      if (rc) return rc;
    }
    return fused_layer_fwd_launch(a, st);
  }
  auto transform = [&](int64_t r0, int64_t r1, rgcn_stream_t s) {
    const char* hi = (const char*)a->A_hi + (size_t)r0 * a->lda * 2;
    const char* lo = A_lo ? (const char*)A_lo + (size_t)r0 * a->lda * 2 : nullptr;
    void* o16 = a->out_bf16 ? (void*)((char*)a->out_bf16 + (size_t)r0 * a->ld_out_bf16 * 2) : nullptr;
    return rgcn_transform_fwd_w(hi, lo, a->lda, K, a->w_planes, a->bias, a->relu, r1 - r0, a->d_out, a->out + r0 * a->ldo,
                                a->ldo, a->mode, a->dropout_p, a->dropout_seed, a->dropout_counter, a->dropout_row0 + r0, a->peer_out_host,
                                a->n_peer, a->peer_row0 + r0, a->peer_ld, o16, a->ld_out_bf16, s);
  };
  // bf16-transform mode with a bf16 copy of the input: the walk gathers the copy
  const bool g16 = a->mode == 1 && a->x_bf16 && a->d_in % 8 == 0 && a->lda % 8 == 0 && a->x_src == a->x_root;
  auto walk = [&](int64_t r0, int64_t r1, int hub_pass, bool whole) {
    if (g16)
      return rgcn_aggregate_fwd_bf16(a->csr, a->x_bf16, a->ld_x_bf16, a->d_in, a->A_hi, a->lda, a->x_bf16, a->ld_x_bf16, r0, r1,
                                     hub_pass, a->agg_workspace, a->agg_workspace_bytes, stream);
    if (whole)
      return rgcn_aggregate_fwd(a->csr, a->x_src, a->ld_x_src, a->d_in, nullptr, 0, a->A_hi, A_lo, a->lda, out_mode, nullptr, 0,
                                nullptr, a->x_root, a->ld_x_root, a->agg_workspace, a->agg_workspace_bytes, stream);
    return rgcn_aggregate_fwd_rows(a->csr, a->x_src, a->ld_x_src, a->d_in, a->A_hi, A_lo, a->lda, out_mode, a->x_root,
                                   a->ld_x_root, r0, r1, hub_pass, a->agg_workspace, a->agg_workspace_bytes, stream);
  };
  SideStream* ss = nullptr;
  const int64_t chunk = pipeline_chunk_rows(a->csr);
  if (chunk <= 0 || n < 2 * chunk || !pipeline_mode(a, st, &ss)) {
    rc = walk(0, n, 1, true);
    if (rc) return rc;
    return transform(0, n, stream);
  }
  // hub chunks first (all rows' hub segments), then chunk by chunk
  if (a->csr->n_chunks > 0) {
    rc = walk(0, 0, 1, false);
    if (rc) return rc;
  }
  RGCN_CUDA(cudaEventRecord(ss->fork, st));
  RGCN_CUDA(cudaStreamWaitEvent(ss->side, ss->fork, 0));
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    const int64_t r1 = r0 + chunk < n ? r0 + chunk : n;
    rc = walk(r0, r1, 0, false);
    if (rc) return rc;
    if (r1 < n) {
      RGCN_CUDA(cudaEventRecord(ss->fork, st));
      RGCN_CUDA(cudaStreamWaitEvent(ss->side, ss->fork, 0));
      rc = transform(r0, r1, (rgcn_stream_t)ss->side);
    } else {
      // the last chunk's transform has nothing left to hide behind: join first, then run it on the main stream
      RGCN_CUDA(cudaEventRecord(ss->join, ss->side));
      RGCN_CUDA(cudaStreamWaitEvent(st, ss->join, 0));
      rc = transform(r0, r1, stream);
    }
    if (rc) return rc;
  }
  return RGCN_OK;
}

// g_out is zero outside the listed rows (csrc/rowsparse.cu): compact, then the same four steps over m_c rows
static int layer_bwd_rows(const rgcn_layer_bwd_args* a, rgcn_stream_t stream) {
  const int R = a->csr_t->R;
  const int K1 = R * a->d_in, K2 = a->d_in, K = K1 + K2;
  const bool need_w = a->g_weight != nullptr;
  const int64_t m_c = rgcn_rows_compact_size(a->n_list);
  RGCN_CHECK_ARG(a->n_list > 0 && a->slot, "layer_bwd: the row-sparse form needs a row list and the slot scratch");
  RGCN_CHECK_ARG(!a->relu_mask && !a->g_ready, "layer_bwd: the row-sparse form serves a layer without ReLU (the last one)");
  // add_root_term = 0 (a destination-range shard: sources and destinations live in different id spaces): the root-term
  // gradient stays in the compact gA[:, R d_in:] rows for the caller
  // a_compact: the forward was the listed-rows form over this very list, so A already is the compact operand
  const bool copy_a = need_w && !a->a_compact;
  RGCN_CHECK_ARG(!copy_a || (a->Ac_hi && (a->mode == 1 || a->Ac_lo)), "layer_bwd: compact operand planes missing");
  int rc = rgcn_rows_compact(a->rows, a->n_list, a->n_dst, a->slot, a->g_out, a->ld_g_out, a->d_out, a->G_hi,
                             a->mode == 0 ? a->G_lo : nullptr, a->ldg, a->A_hi, a->mode == 0 ? a->A_lo : nullptr, a->lda, K,
                             copy_a ? a->Ac_hi : nullptr, (copy_a && a->mode == 0) ? a->Ac_lo : nullptr, a->ldac,
                             a->g_bias ? a->colsum_partial : nullptr, a->gA ? a->gA + m_c * a->ld_gA : nullptr, a->gA ? K : 0,
                             a->slot_ready, stream);
  if (rc) return rc;
  const void* Aw_hi = a->a_compact ? a->A_hi : a->Ac_hi;
  const void* Aw_lo = a->a_compact ? a->A_lo : a->Ac_lo;
  const int64_t ldw = a->a_compact ? a->lda : a->ldac;
  return dgrad_walk_wgrad(a, m_c, Aw_hi, Aw_lo, ldw, (int32_t)rgcn_rows_compact_blocks(a->n_list), [&]() {
    if (a->csr_fwd && a->src_flag && !a->next_G)
      return rgcn_aggregate_bwd_rows_marked(a->csr_t, a->csr_fwd, a->rows, a->n_list, a->src_flag, a->gA, a->ld_gA, a->d_in, a->slot,
                                            (int32_t)m_c, a->add_root_term ? a->gA + K1 : nullptr, a->ld_gA, a->g_x, a->ld_g_x,
                                            a->agg_workspace, a->agg_workspace_bytes, stream);
    return rgcn_aggregate_bwd_rows(a->csr_t, a->gA, a->ld_gA, a->d_in, a->slot, (int32_t)m_c,
                                   a->add_root_term ? a->gA + K1 : nullptr, a->ld_gA, a->g_x, a->ld_g_x, a->next_G,
                                   a->agg_workspace, a->agg_workspace_bytes, stream);
  }, stream);
}

extern "C" int rgcn_layer_bwd(const rgcn_layer_bwd_args* a, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(a && a->csr_t, "layer_bwd: null arguments");
  const int R = a->csr_t->R;
  const int K1 = R * a->d_in, K2 = a->d_in;
  RGCN_CHECK_ARG(a->mode == 0 || a->mode == 1, "layer_bwd: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(a->G_hi && (a->mode == 1 || a->G_lo), "layer_bwd: scratch planes for G missing");
  const bool need_w = a->g_weight != nullptr;
  RGCN_CHECK_ARG(!need_w || (a->g_root && a->A_hi && (a->mode == 1 || a->A_lo)), "layer_bwd: weight gradient needs g_root and the saved planes");
  RGCN_CHECK_ARG(!a->g_bias || (need_w && a->colsum_partial), "layer_bwd: g_bias needs the weight gradient and colsum_partial");
  if (a->rows) return layer_bwd_rows(a, stream);
  // G = g_out * [mask > 0] * mask_scale as planes, column sums = bias gradient — unless the downstream layer's walk
  // has written them already (g_ready)
  int32_t n_colsum = a->n_colsum_ready;
  if (!a->g_ready) {
    int rc = rgcn_split_planes(a->g_out, a->ld_g_out, a->relu_mask, a->ld_mask, a->n_dst, a->d_out, a->G_hi,
                               a->mode == 0 ? a->G_lo : nullptr, a->ldg, a->g_bias ? a->colsum_partial : nullptr,
                               a->mask_scale, nullptr, 0, stream);
    if (rc) return rc;
    n_colsum = (int32_t)rgcn_split_planes_blocks(a->n_dst, a->d_out);
  }
  return dgrad_walk_wgrad(a, a->n_dst, a->A_hi, a->A_lo, a->lda, n_colsum, [&]() {
    return rgcn_aggregate_bwd(a->csr_t, a->gA, a->ld_gA, a->d_in, a->add_root_term ? a->gA + K1 : nullptr, a->ld_gA, a->g_x,
                              a->ld_g_x, a->next_G, a->agg_workspace, a->agg_workspace_bytes, stream);
  }, stream);
}
