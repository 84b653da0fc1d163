// Basis decomposition of the relation weights (RGCNConv(num_bases = B), plumbed at reference src/models/rgcn.py:58, :76,
// :84): W_r = sum_b comp[r, b] * V_b, i.e. PyG's `(comp @ weight.view(B, -1)).view(R, in, out)`, and its backward
//   g_V[b]       = sum_r comp[r, b] * g_W[r]
//   g_comp[r, b] = <g_W[r], V_b>
// B and R are tens, in * out is 10^4 .. 10^5: three bandwidth-bound streaming kernels over the [*, in * out] matrices
// (a library SGEMM sees a 30 x 8 product with K = 65,536 and spends 150 us on it; these take a few us).
// Fixed summation orders: deterministic.
#include "common.cuh"

namespace rgcn {

constexpr int kMaxCombine = 64;      // rows of comp held per thread loop (R and B up to this)

// out[i, :] = sum_j coef(i, j) * in[j, :]   over float4 columns; coef(i, j) = c[i * ldc + j] or c[j * ldc + i]
template <bool TRANSPOSED>
__global__ void __launch_bounds__(256) combine_rows_kernel(const float* __restrict__ c, int ldc, int n_out, int n_in,
                                                           const float* __restrict__ in, float* __restrict__ out,
                                                           int64_t cols4) {
  pdl_enter();
  extern __shared__ float s_c[];                       // [n_out][n_in]
  for (int t = threadIdx.x; t < n_out * n_in; t += 256) {
    const int i = t / n_in, j = t % n_in;
    s_c[t] = TRANSPOSED ? c[j * ldc + i] : c[i * ldc + j];
  }
  __syncthreads();
  const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (k >= cols4) return;
  const float4* __restrict__ in4 = reinterpret_cast<const float4*>(in);
  float4* __restrict__ out4 = reinterpret_cast<float4*>(out);
  // inputs in chunks of 8 rows held in registers, every output row accumulated in input order
  for (int i0 = 0; i0 < n_out; i0 += 8) {
    float4 acc[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < n_in; ++j) {
      const float4 v = __ldg(in4 + (int64_t)j * cols4 + k);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (i0 + u < n_out) fma4(acc[u], s_c[(i0 + u) * n_in + j], v);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (i0 + u < n_out) out4[(int64_t)(i0 + u) * cols4 + k] = acc[u];
  }
}

// g_comp[r, b] = <gW[r, :], V[b, :]>: one block per r, B accumulators per thread (B <= 16), fixed-order block reduce
__global__ void __launch_bounds__(256) comp_grad_kernel(const float* __restrict__ gW, const float* __restrict__ V, int B,
                                                        int64_t cols4, float* __restrict__ g_comp, int ldg) {
  pdl_enter();
  __shared__ float red[8][16];
  const int r = blockIdx.x;
  const float4* __restrict__ g4 = reinterpret_cast<const float4*>(gW) + (int64_t)r * cols4;
  const float4* __restrict__ v4 = reinterpret_cast<const float4*>(V);
  float acc[16];
#pragma unroll
  for (int b = 0; b < 16; ++b) acc[b] = 0.f;
  for (int64_t k = threadIdx.x; k < cols4; k += 256) {
    const float4 g = __ldg(g4 + k);
#pragma unroll
    for (int b = 0; b < 16; ++b) {
      if (b < B) {
        const float4 v = __ldg(v4 + (int64_t)b * cols4 + k);
        acc[b] = fmaf(g.x, v.x, acc[b]); acc[b] = fmaf(g.y, v.y, acc[b]);
        acc[b] = fmaf(g.z, v.z, acc[b]); acc[b] = fmaf(g.w, v.w, acc[b]);
      }
    }
  }
#pragma unroll
  for (int b = 0; b < 16; ++b) {
    float s = acc[b];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][b] = s;
  }
  __syncthreads();
  if (threadIdx.x < B) {
    float s = red[0][threadIdx.x];
    for (int w = 1; w < 8; ++w) s += red[w][threadIdx.x];
    g_comp[r * ldg + threadIdx.x] = s;
  }
}

// Block-diagonal relation weights (RGCNConv(num_blocks = nb), PyG's second regulariser, Schlichtkrull et al. 2018):
// W_r = blockdiag(blocks[r, 0], .., blocks[r, nb - 1]),  W[r, k*bi + c, k*bo + d] = blocks[r, k, c, d], zero off the blocks.
// The expanded W_r feeds the unchanged layer kernels; the backward copies the diagonal blocks of the dense gradient
// back.  Pure copies (no arithmetic): bit-exact and deterministic.  VEC: 4 consecutive columns per thread (bo % 4 == 0,
// so they never straddle a block).  One thread per output vector, 32-bit index arithmetic (the host caps the sizes).
template <bool VEC>
__global__ void __launch_bounds__(256) block_diag_expand_kernel(const float* __restrict__ blocks, int nb, int bi, int bo,
                                                                float* __restrict__ W, unsigned n_vec) {
  pdl_enter();
  constexpr unsigned V = VEC ? 4 : 1;
  const unsigned t = blockIdx.x * 256u + threadIdx.x;
  if (t >= n_vec) return;
  const unsigned d_in = (unsigned)nb * bi, cols = (unsigned)nb * bo / V;
  const unsigned ri = t / cols, j = (t - ri * cols) * V;       // row r * d_in + i of W, first column
  const unsigned r = ri / d_in, i = ri - r * d_in;
  const unsigned k = i / bi;
  const bool on = j >= k * bo && j < (k + 1) * bo;
  const size_t src = ((size_t)(r * nb + k) * bi + (i - k * bi)) * bo + (j - k * bo);
  if (VEC) {
    reinterpret_cast<float4*>(W)[t] = on ? __ldg(reinterpret_cast<const float4*>(blocks + src)) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    W[t] = on ? __ldg(blocks + src) : 0.f;
  }
}

template <bool VEC>
__global__ void __launch_bounds__(256) block_diag_gather_kernel(const float* __restrict__ gW, int nb, int bi, int bo,
                                                                float* __restrict__ g_blocks, unsigned n_vec) {
  pdl_enter();
  constexpr unsigned V = VEC ? 4 : 1;
  const unsigned t = blockIdx.x * 256u + threadIdx.x;
  if (t >= n_vec) return;
  const unsigned cols = (unsigned)bo / V;
  const unsigned rkc = t / cols, d = (t - rkc * cols) * V;    // (r * nb + k) * bi + c, column in the block
  const unsigned rk = rkc / bi, c = rkc - rk * bi;
  const unsigned r = rk / nb, k = rk - r * nb;
  const size_t src = ((size_t)r * nb * bi + k * bi + c) * ((size_t)nb * bo) + k * bo + d;
  if (VEC) {
    reinterpret_cast<float4*>(g_blocks)[t] = __ldg(reinterpret_cast<const float4*>(gW + src));
  } else {
    g_blocks[t] = __ldg(gW + src);
  }
}

}  // namespace rgcn

using namespace rgcn;

static int check_combine(const float* comp, const float* a, const float* b, int32_t R, int32_t B, int64_t io) {
  RGCN_CHECK_ARG(comp && a && b && R >= 1 && B >= 1 && R <= kMaxCombine && B <= kMaxCombine && io >= 4 && io % 4 == 0,
                 "basis_combine: need 1 <= R, B <= %d and in * out a positive multiple of 4", kMaxCombine);
  RGCN_CHECK_ARG((((uintptr_t)a | (uintptr_t)b) & 15) == 0, "basis_combine: matrices must be 16-byte aligned");
  return RGCN_OK;
}

extern "C" int rgcn_basis_combine(const float* comp, const float* V, int32_t R, int32_t B, int64_t in_out, float* W,
                                  rgcn_stream_t stream) {
  int rc = check_combine(comp, V, W, R, B, in_out);
  if (rc) return rc;
  const int64_t cols4 = in_out / 4;
  RGCN_CUDA(launch_pdl(combine_rows_kernel<false>, dim3((unsigned)((cols4 + 255) / 256)), dim3(256), (size_t)R * B * sizeof(float),
                       (cudaStream_t)stream, comp, (int)B, (int)R, (int)B, V, W, cols4));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_basis_combine_bwd(const float* comp, const float* V, const float* gW, int32_t R, int32_t B,
                                      int64_t in_out, float* g_V, float* g_comp, rgcn_stream_t stream) {
  int rc = check_combine(comp, V, gW, R, B, in_out);
  if (rc) return rc;
  RGCN_CHECK_ARG(!g_comp || B <= 16, "basis_combine_bwd: the coefficient gradient handles at most 16 bases");
  RGCN_CHECK_ARG(!g_V || ((uintptr_t)g_V & 15) == 0, "basis_combine_bwd: g_V must be 16-byte aligned");
  const int64_t cols4 = in_out / 4;
  if (g_V) {
    RGCN_CUDA(launch_pdl(combine_rows_kernel<true>, dim3((unsigned)((cols4 + 255) / 256)), dim3(256), (size_t)R * B * sizeof(float),
                         (cudaStream_t)stream, comp, (int)B, (int)B, (int)R, gW, g_V, cols4));
    RGCN_LAUNCH_CHECK();
  }
  if (g_comp) {
    RGCN_CUDA(launch_pdl(comp_grad_kernel, dim3((unsigned)R), dim3(256), 0, (cudaStream_t)stream, gW, V, (int)B, cols4, g_comp, (int)B));
    RGCN_LAUNCH_CHECK();
  }
  return RGCN_OK;
}

static int check_block_diag(const char* who, const float* a, const float* b, int32_t R, int32_t nb, int32_t bi, int32_t bo) {
  RGCN_CHECK_ARG(a && b && R >= 1 && nb >= 1 && bi >= 1 && bo >= 1, "%s: need non-null matrices and R, nb, bi, bo >= 1", who);
  RGCN_CHECK_ARG((int64_t)nb * bi <= (1 << 20) && (int64_t)nb * bo <= (1 << 20) && R <= (1 << 20),
                 "%s: in, out = nb * bi, nb * bo and R must be at most 2^20", who);
  RGCN_CHECK_ARG((int64_t)R * nb * bi * nb * bo < ((int64_t)1 << 31), "%s: the dense W must have fewer than 2^31 elements", who);
  RGCN_CHECK_ARG((((uintptr_t)a | (uintptr_t)b) & 15) == 0, "%s: matrices must be 16-byte aligned", who);
  return RGCN_OK;
}

extern "C" int rgcn_block_diag_expand(const float* blocks, int32_t R, int32_t nb, int32_t bi, int32_t bo, float* W,
                                      rgcn_stream_t stream) {
  int rc = check_block_diag("block_diag_expand", blocks, W, R, nb, bi, bo);
  if (rc) return rc;
  const int64_t n = (int64_t)R * nb * bi * nb * bo;
  if (bo % 4 == 0) {
    RGCN_CUDA(launch_pdl(block_diag_expand_kernel<true>, dim3((unsigned)((n / 4 + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                         blocks, (int)nb, (int)bi, (int)bo, W, (unsigned)(n / 4)));
  } else {
    RGCN_CUDA(launch_pdl(block_diag_expand_kernel<false>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                         blocks, (int)nb, (int)bi, (int)bo, W, (unsigned)n));
  }
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_block_diag_gather(const float* gW, int32_t R, int32_t nb, int32_t bi, int32_t bo, float* g_blocks,
                                      rgcn_stream_t stream) {
  int rc = check_block_diag("block_diag_gather", gW, g_blocks, R, nb, bi, bo);
  if (rc) return rc;
  const int64_t n = (int64_t)R * nb * bi * bo;
  if (bo % 4 == 0) {
    RGCN_CUDA(launch_pdl(block_diag_gather_kernel<true>, dim3((unsigned)((n / 4 + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                         gW, (int)nb, (int)bi, (int)bo, g_blocks, (unsigned)(n / 4)));
  } else {
    RGCN_CUDA(launch_pdl(block_diag_gather_kernel<false>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                         gW, (int)nb, (int)bi, (int)bo, g_blocks, (unsigned)n));
  }
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}
