// Optimiser step: torch.nn.utils.clip_grad_norm_ + torch.optim.Adam / AdamW (reference src/train.py:311-318) as two
// memory-bound kernels over a table of parameter segments (include/rgcn_b200.h, rgcn_adam_step).
//
//   adam_grad_sqnorm_kernel  one block per 4096-float chunk of a segment: fp64 partial sum of g^2 -> partials[block];
//                            the last block to arrive (integer ticket) sums the partials in index order and writes
//                            total_norm and clip_coef.  No floating-point atomics: the same bits on every run.
//   adam_update_kernel       same chunking: one read of p, g, m, v and one write of p, m, v per element.  Every block
//                            forms the bias corrections from its segment's step; the last block to arrive (all others
//                            have read it by then) advances every segment's step.
// The table travels by value as a kernel parameter, so a captured CUDA graph bakes the pointers in.
#include <math.h>

#include "common.cuh"

namespace rgcn {

constexpr int kAdamThreads = 256;
constexpr int kAdamVec = 4;                                     // float4 per thread per chunk
constexpr int64_t kAdamChunk = (int64_t)kAdamThreads * kAdamVec * 4;   // floats per block
constexpr size_t kAdamHeader = 64;                              // counters + clip coefficient, then the partials

struct AdamTable {
  rgcn_adam_segment seg[RGCN_ADAM_MAX_SEGMENTS];
  int32_t chunk_begin[RGCN_ADAM_MAX_SEGMENTS + 1];              // first block of each segment; [n_seg] = grid size
  uint64_t vec_ok;                                               // bit s: segment s is 16-byte aligned throughout
  int32_t n_seg;
};

struct AdamWs {
  unsigned int* norm_ticket;
  unsigned int* update_ticket;
  float* clip_coef;
  double* partials;
};

static inline AdamWs adam_ws(void* workspace) {
  char* b = static_cast<char*>(workspace);
  return AdamWs{reinterpret_cast<unsigned int*>(b), reinterpret_cast<unsigned int*>(b + 4),
                reinterpret_cast<float*>(b + 8), reinterpret_cast<double*>(b + kAdamHeader)};
}

__device__ __forceinline__ int adam_find_segment(const AdamTable& t, int b) {
  int s = 0;
  while (s + 1 < t.n_seg && t.chunk_begin[s + 1] <= b) ++s;
  return s;
}

// fixed-order block sum of one double per thread (shuffle tree, then the 8 warp sums in warp order); valid in thread 0
__device__ __forceinline__ double adam_block_sum(double v, double* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kAdamThreads / 32; ++w) s += red[w];
  return s;
}

__global__ void __launch_bounds__(kAdamThreads) adam_grad_sqnorm_kernel(const AdamTable tab, float max_norm, AdamWs ws,
                                                                        float* __restrict__ grad_norm) {
  pdl_enter();
  __shared__ double red[kAdamThreads / 32];
  __shared__ bool s_last;
  const int s = adam_find_segment(tab, blockIdx.x);
  const rgcn_adam_segment& sg = tab.seg[s];
  const int64_t lo = (int64_t)(blockIdx.x - tab.chunk_begin[s]) * kAdamChunk;
  const int64_t hi = min(lo + kAdamChunk, sg.numel);
  double acc = 0.0;
  if ((tab.vec_ok >> s) & 1) {
    const int64_t hi4 = hi & ~(int64_t)3;
    const float4* g4 = reinterpret_cast<const float4*>(sg.grad);
    for (int64_t i = lo / 4 + threadIdx.x; i < hi4 / 4; i += kAdamThreads) {
      const float4 g = __ldg(g4 + i);
      acc = fma((double)g.x, (double)g.x, acc);
      acc = fma((double)g.y, (double)g.y, acc);
      acc = fma((double)g.z, (double)g.z, acc);
      acc = fma((double)g.w, (double)g.w, acc);
    }
    const int64_t i = hi4 + threadIdx.x;
    if (i < hi) {
      const double g = __ldg(sg.grad + i);
      acc = fma(g, g, acc);
    }
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kAdamThreads) {
      const double g = __ldg(sg.grad + i);
      acc = fma(g, g, acc);
    }
  }
  const double part = adam_block_sum(acc, red);
  if (threadIdx.x == 0) {
    ws.partials[blockIdx.x] = part;
    __threadfence();
    s_last = atomicAdd(ws.norm_ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double t = 0.0;
  for (int i = threadIdx.x; i < (int)gridDim.x; i += kAdamThreads) t += __ldcg(ws.partials + i);
  __syncthreads();                                              // red is reused
  const double total = adam_block_sum(t, red);
  if (threadIdx.x == 0) {
    const float norm = (float)sqrt(total);
    // torch: clip_coef = max_norm / (total_norm + 1e-6) is reciprocal(total_norm + 1e-6) * max_norm in fp32, then
    // clamp(max=1), which keeps a NaN
    float c = __fmul_rn(__frcp_rn(__fadd_rn(norm, 1e-6f)), max_norm);
    c = c > 1.f ? 1.f : c;
    *ws.clip_coef = c;
    if (grad_norm) *grad_norm = norm;
    *ws.norm_ticket = 0u;
  }
}

struct AdamScalars {
  float clip, decay, wd, w1, beta2, w2, inv_bc2, eps, neg_step;
  int mode;                                                     // 0: no decay, 1: L2 (Adam), 2: decoupled (AdamW)
};

__device__ __forceinline__ float adam_elem(float& p, float g, float& m, float& v, const AdamScalars& c, bool clip) {
  if (clip) g = __fmul_rn(g, c.clip);
  if (c.mode == 2) p = __fmul_rn(p, c.decay);
  else if (c.mode == 1) g = fmaf(c.wd, p, g);
  const float d = __fsub_rn(g, m);                              // torch's lerp: the form depends on |weight| < 0.5
  m = fabsf(c.w1) < 0.5f ? fmaf(c.w1, d, m) : fmaf(-d, __fsub_rn(1.f, c.w1), g);
  v = fmaf(__fmul_rn(c.w2, g), g, __fmul_rn(v, c.beta2));
  const float denom = __fadd_rn(__fmul_rn(__fsqrt_rn(v), c.inv_bc2), c.eps);
  p = fmaf(c.neg_step, __fdiv_rn(m, denom), p);
  return p;
}

__global__ void __launch_bounds__(kAdamThreads) adam_update_kernel(const AdamTable tab,
                                                                   const rgcn_adam_hparams* __restrict__ hp, int clip,
                                                                   AdamWs ws) {
  pdl_enter();
  __shared__ AdamScalars s_c;
  __shared__ bool s_last;
  const int s = adam_find_segment(tab, blockIdx.x);
  const rgcn_adam_segment& sg = tab.seg[s];
  if (threadIdx.x == 0) {
    // torch (capturable=False): step_t += 1 in fp32, then the bias corrections in Python floats (fp64), rounded to
    // fp32 where they meet the tensors
    const rgcn_adam_hparams h = hp[sg.group];
    const double t = (double)__fadd_rn(__ldcg(sg.step), 1.f);
    const double bc1 = 1.0 - pow(h.beta1, t), bc2 = 1.0 - pow(h.beta2, t);
    AdamScalars c;
    c.clip = clip ? __ldcg(ws.clip_coef) : 1.f;
    c.mode = h.weight_decay != 0.0 ? (h.decoupled_weight_decay ? 2 : 1) : 0;
    c.decay = (float)(1.0 - h.lr * h.weight_decay);
    c.wd = (float)h.weight_decay;
    c.w1 = (float)(1.0 - h.beta1);
    c.beta2 = (float)h.beta2;
    c.w2 = (float)(1.0 - h.beta2);
    c.inv_bc2 = __frcp_rn((float)sqrt(bc2));                    // tensor / CPU scalar: a * (1 / (float)b) in torch
    c.eps = (float)h.eps;
    c.neg_step = (float)(-(h.lr / bc1));
    s_c = c;
  }
  __syncthreads();
  const AdamScalars c = s_c;
  const bool do_clip = clip != 0;
  const int64_t lo = (int64_t)(blockIdx.x - tab.chunk_begin[s]) * kAdamChunk;
  const int64_t hi = min(lo + kAdamChunk, sg.numel);
  if ((tab.vec_ok >> s) & 1) {
    const int64_t hi4 = hi & ~(int64_t)3;
    float4* p4 = reinterpret_cast<float4*>(sg.param);
    const float4* g4 = reinterpret_cast<const float4*>(sg.grad);
    float4* m4 = reinterpret_cast<float4*>(sg.exp_avg);
    float4* v4 = reinterpret_cast<float4*>(sg.exp_avg_sq);
    for (int64_t k = lo / 4 + threadIdx.x; k < hi4 / 4; k += kAdamThreads) {
      float4 p = p4[k], m = m4[k], v = v4[k];
      const float4 g = __ldg(g4 + k);
      adam_elem(p.x, g.x, m.x, v.x, c, do_clip);
      adam_elem(p.y, g.y, m.y, v.y, c, do_clip);
      adam_elem(p.z, g.z, m.z, v.z, c, do_clip);
      adam_elem(p.w, g.w, m.w, v.w, c, do_clip);
      p4[k] = p; m4[k] = m; v4[k] = v;
    }
    const int64_t i = hi4 + threadIdx.x;                        // scalar tail (numel % 4 elements)
    if (i < hi) adam_elem(sg.param[i], __ldg(sg.grad + i), sg.exp_avg[i], sg.exp_avg_sq[i], c, do_clip);
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kAdamThreads)
      adam_elem(sg.param[i], __ldg(sg.grad + i), sg.exp_avg[i], sg.exp_avg_sq[i], c, do_clip);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(ws.update_ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int k = threadIdx.x; k < tab.n_seg; k += kAdamThreads) *tab.seg[k].step = __fadd_rn(__ldcg(tab.seg[k].step), 1.f);
  if (threadIdx.x == 0) *ws.update_ticket = 0u;
}

static int64_t adam_chunks(int64_t numel) { return (numel + kAdamChunk - 1) / kAdamChunk; }

// cudaFuncGetAttributes loads a lazily loaded module; done once per device outside any capture (see the header)
static int adam_load_kernels() {
  static bool loaded[64] = {false};
  int dev = 0;
  RGCN_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && loaded[dev]) return RGCN_OK;
  cudaFuncAttributes a;
  RGCN_CUDA(cudaFuncGetAttributes(&a, adam_grad_sqnorm_kernel));
  RGCN_CUDA(cudaFuncGetAttributes(&a, adam_update_kernel));
  if (dev >= 0 && dev < 64) loaded[dev] = true;
  return RGCN_OK;
}

}  // namespace rgcn

using namespace rgcn;

extern "C" size_t rgcn_adam_workspace_bytes(int64_t total_numel, int32_t n_segments) {
  if (total_numel < 0 || n_segments < 0) return 0;
  return kAdamHeader + (size_t)(total_numel / kAdamChunk + n_segments + 1) * sizeof(double);
}

extern "C" int rgcn_adam_step(const rgcn_adam_segment* segments_host, int32_t n_segments,
                              const rgcn_adam_hparams* hparams, int32_t n_groups, float max_grad_norm,
                              float* grad_norm, void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n_segments >= 0, "adam_step: negative n_segments %d", n_segments);
  RGCN_CHECK_ARG(n_segments <= RGCN_ADAM_MAX_SEGMENTS, "adam_step: %d segments, at most %d per call", n_segments,
                 RGCN_ADAM_MAX_SEGMENTS);
  RGCN_CHECK_ARG(n_segments == 0 || segments_host, "adam_step: null segment table");
  RGCN_CHECK_ARG(n_segments == 0 || (hparams && n_groups > 0), "adam_step: null hparams or no groups");
  RGCN_CHECK_ARG(!(max_grad_norm != max_grad_norm), "adam_step: max_grad_norm is NaN (negative disables clipping)");
  AdamTable tab;
  memset(&tab, 0, sizeof(tab));
  int64_t total = 0, blocks = 0;
  for (int s = 0; s < n_segments; ++s) {
    const rgcn_adam_segment& g = segments_host[s];
    RGCN_CHECK_ARG(g.numel >= 0, "adam_step: segment %d has negative numel", s);
    RGCN_CHECK_ARG(g.group >= 0 && g.group < n_groups, "adam_step: segment %d group %d outside [0, %d)", s, g.group,
                   n_groups);
    RGCN_CHECK_ARG(g.step, "adam_step: segment %d has a null step pointer", s);
    RGCN_CHECK_ARG(g.numel == 0 || (g.param && g.grad && g.exp_avg && g.exp_avg_sq),
                   "adam_step: segment %d has a null pointer", s);
    tab.seg[s] = g;
    tab.chunk_begin[s] = (int32_t)blocks;
    // an empty segment still gets one (idle) block: its step advances like torch's
    blocks += g.numel ? adam_chunks(g.numel) : 1;
    RGCN_CHECK_ARG(blocks < (int64_t)INT32_MAX, "adam_step: too many elements");
    total += g.numel;
    const bool aligned = ((reinterpret_cast<uintptr_t>(g.param) | reinterpret_cast<uintptr_t>(g.grad) |
                           reinterpret_cast<uintptr_t>(g.exp_avg) | reinterpret_cast<uintptr_t>(g.exp_avg_sq)) & 15) == 0;
    if (aligned) tab.vec_ok |= 1ull << s;
  }
  tab.chunk_begin[n_segments] = (int32_t)blocks;
  tab.n_seg = n_segments;
  RGCN_CHECK_ARG(n_segments == 0 || workspace, "adam_step: null workspace");
  RGCN_CHECK_ARG(n_segments == 0 || workspace_bytes >= kAdamHeader + (size_t)blocks * sizeof(double),
                 "adam_step: workspace of %zu bytes, need %zu", workspace_bytes,
                 kAdamHeader + (size_t)blocks * sizeof(double));
  if (int rc = adam_load_kernels()) return rc;
  if (n_segments == 0) return RGCN_OK;
  const AdamWs ws = adam_ws(workspace);
  const bool clip = max_grad_norm >= 0.f;
  cudaStream_t st = (cudaStream_t)stream;
  if (clip) {
    RGCN_CUDA(launch_pdl(adam_grad_sqnorm_kernel, dim3((unsigned)blocks), dim3(kAdamThreads), 0, st, tab, max_grad_norm,
                         ws, grad_norm));
    RGCN_LAUNCH_CHECK();
  }
  RGCN_CUDA(launch_pdl(adam_update_kernel, dim3((unsigned)blocks), dim3(kAdamThreads), 0, st, tab, hparams, (int)clip,
                       ws));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}
