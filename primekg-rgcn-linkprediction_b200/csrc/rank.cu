// All-pairs scoring and ranking without the [queries, candidates] score matrix round trip.
//
//   rows_prepare : A'[i] = emb[idx[i]] (* rel_table[rel[i]]) (/ ||.||)          gather + DistMult scale / L2 normalise
//   allpairs_scores : out[i, j] = alpha * <A'[i], B[b_idx[j]]> + beta
//        -> LinkPredictor.score_all_tails (reference src/models/rgcn.py:234-241), compare_methods.predict_all
//           ((cos + 1) / 2, src/compare_methods.py:384-397), the 6,282 x 5,593 drug-disease sweep (BASELINE cfg4)
//   allpairs_rank : greater[i] = #{j != t_i : s_ij > s_i,t_i},  equal[i] = #{j != t_i : s_ij == s_i,t_i}
//        -> the per-row `argsort` + position search of the ranking evaluation (src/evaluate.py:260-276):
//           rank = 1 + greater (ties: torch.argsort is unstable, the reference's rank lies in [1+greater, 1+greater+equal])
//
// fp32 FMA tiles (64 x 64 outputs per block, 4 x 4 per thread, K staged through shared memory in 16-wide slabs).
// Every output accumulates k = 0..d-1 in ascending order with fmaf, and so does the threshold kernel, which makes
// s_i,t_i bit-identical to the tile's own value for j = t_i (no self-comparison artefacts).
#include "common.cuh"

namespace rgcn {

constexpr int TM = 64, TN = 64, TK = 16;

__global__ void __launch_bounds__(256) rows_prepare_kernel(const float* __restrict__ emb, int64_t ld,
                                                           const int64_t* __restrict__ idx, int64_t n, int32_t d,
                                                           const float* __restrict__ rel_table,
                                                           const int64_t* __restrict__ rel, int normalize,
                                                           float* __restrict__ out, int64_t ldo) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= n) return;
  const float* src = emb + (idx ? idx[i] : i) * ld;
  const float* r = (rel_table && rel) ? rel_table + rel[i] * d : nullptr;
  float ss = 0.f;
  for (int k = lane; k < d; k += 32) {
    float v = src[k];
    if (r) v *= r[k];
    ss += v * v;
  }
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float nrm = sqrtf(ss);
  for (int k = lane; k < d; k += 32) {
    float v = src[k];
    if (r) v *= r[k];
    if (normalize) v = v / nrm;                       // x / ||x||, as numpy does (0/0 -> nan, like the reference)
    out[i * ldo + k] = v;
  }
}

// thr[i] = <A[i], B[t_i]> with the tile kernel's accumulation order
__global__ void threshold_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb,
                                 const int64_t* __restrict__ b_idx, const int64_t* __restrict__ true_pos, int64_t nq,
                                 int32_t d, float* __restrict__ thr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  const int64_t t = true_pos[i];
  const float* a = A + i * lda;
  const float* b = B + (b_idx ? b_idx[t] : t) * ldb;
  float acc = 0.f;
  for (int k = 0; k < d; ++k) acc = fmaf(a[k], b[k], acc);
  thr[i] = acc;
}

// MODE 0: store alpha * s + beta.   MODE 1: count against thr.
template <int MODE>
__global__ void __launch_bounds__(256) allpairs_kernel(const float* __restrict__ A, int64_t lda, int64_t na,
                                                       const float* __restrict__ B, int64_t ldb,
                                                       const int64_t* __restrict__ b_idx, int64_t nb, int32_t d,
                                                       float alpha, float beta, float* __restrict__ out, int64_t ldo,
                                                       const float* __restrict__ thr,
                                                       const int64_t* __restrict__ true_pos,
                                                       int32_t* __restrict__ greater, int32_t* __restrict__ equal) {
  __shared__ float sa[TK][TM + 4], sb[TK][TN + 4];
  const int64_t i0 = (int64_t)blockIdx.y * TM, j0 = (int64_t)blockIdx.x * TN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 x 16 threads, 4 x 4 outputs each
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  // loader mapping: thread loads one float4 (4 consecutive k) of one row per slab
  const int lr = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;  // row 0..63, k offset 0,4,8,12
  const int64_t ai = i0 + lr, bj = j0 + lr;
  const float* arow = (ai < na) ? A + ai * lda : nullptr;
  const float* brow = (bj < nb) ? B + (b_idx ? b_idx[bj] : bj) * ldb : nullptr;
  for (int k0 = 0; k0 < d; k0 += TK) {
    float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
    if (k0 + lk < d) {                                          // d % 4 == 0
      if (arow) va = ldg4(arow + k0 + lk);
      if (brow) vb = ldg4(brow + k0 + lk);
    }
    __syncthreads();
    sa[lk][lr] = va.x; sa[lk + 1][lr] = va.y; sa[lk + 2][lr] = va.z; sa[lk + 3][lr] = va.w;
    sb[lk][lr] = vb.x; sb[lk + 1][lr] = vb.y; sb[lk + 2][lr] = vb.z; sb[lk + 3][lr] = vb.w;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&sa[k][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&sb[k][tx * 4]);
      const float av[4] = {a4.x, a4.y, a4.z, a4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int64_t i = i0 + ty * 4 + a;
    const bool valid = i < na;
    if (MODE == 0) {
      if (!valid) continue;
      const int64_t j = j0 + tx * 4;
      float* o = out + i * ldo + j;
      if (j + 3 < nb && (ldo & 3) == 0 && (((uintptr_t)out) & 15) == 0) {
        *reinterpret_cast<float4*>(o) = make_float4(alpha * acc[a][0] + beta, alpha * acc[a][1] + beta,
                                                    alpha * acc[a][2] + beta, alpha * acc[a][3] + beta);
      } else {
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if (j + b < nb) o[b] = alpha * acc[a][b] + beta;
      }
    } else {
      const float t = valid ? thr[i] : 0.f;
      const int64_t tp = valid ? true_pos[i] : -1;
      int g = 0, e = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int64_t j = j0 + tx * 4 + b;
        if (valid && j < nb && j != tp) {
          g += acc[a][b] > t;
          e += acc[a][b] == t;
        }
      }
      // the 16 threads of one row group (same ty) sit in 16 consecutive lanes: every lane takes part in the
      // shuffles, then one integer atomic per row and tile (integer adds: order independent => deterministic)
      for (int o = 8; o; o >>= 1) {
        g += __shfl_xor_sync(0xffffffffu, g, o);
        e += __shfl_xor_sync(0xffffffffu, e, o);
      }
      if (valid && tx == 0) {
        if (g) atomicAdd(greater + i, g);
        if (e) atomicAdd(equal + i, e);
      }
    }
  }
}

}  // namespace rgcn

using namespace rgcn;

static int check_ap(const float* A, int64_t lda, const float* B, int64_t ldb, int32_t d) {
  RGCN_CHECK_ARG(d >= 4 && d % 4 == 0, "allpairs: d=%d must be a positive multiple of 4", d);
  RGCN_CHECK_ARG(A && B && lda % 4 == 0 && ldb % 4 == 0 && (((uintptr_t)A | (uintptr_t)B) & 15) == 0,
                 "allpairs: operands must be 16-byte aligned rows (ld %% 4 == 0)");
  return RGCN_OK;
}

extern "C" int rgcn_rows_prepare(const float* emb, int64_t ld, const int64_t* idx, int64_t n, int32_t d,
                                 const float* rel_table, const int64_t* rel, int32_t normalize, float* out, int64_t ldo,
                                 rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n >= 0 && d > 0 && (n == 0 || (emb && out)), "rows_prepare: bad arguments");
  RGCN_CHECK_ARG((rel_table == nullptr) == (rel == nullptr), "rows_prepare: rel_table and rel go together");
  if (n == 0) return RGCN_OK;
  rows_prepare_kernel<<<(unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream>>>(emb, ld, idx, n, d, rel_table, rel,
                                                                                normalize, out, ldo);
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_allpairs_scores(const float* A, int64_t lda, int64_t na, const float* B, int64_t ldb,
                                    const int64_t* b_idx, int64_t nb, int32_t d, float alpha, float beta, float* out,
                                    int64_t ldo, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(na >= 0 && nb >= 0, "allpairs_scores: negative size");
  if (na == 0 || nb == 0) return RGCN_OK;
  int rc = check_ap(A, lda, B, ldb, d);
  if (rc) return rc;
  RGCN_CHECK_ARG(out && ldo >= nb, "allpairs_scores: bad output");
  dim3 grid((unsigned)((nb + TN - 1) / TN), (unsigned)((na + TM - 1) / TM));
  allpairs_kernel<0><<<grid, 256, 0, (cudaStream_t)stream>>>(A, lda, na, B, ldb, b_idx, nb, d, alpha, beta, out, ldo,
                                                             nullptr, nullptr, nullptr, nullptr);
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_allpairs_rank(const float* A, int64_t lda, int64_t nq, const float* B, int64_t ldb,
                                  const int64_t* b_idx, int64_t nb, int32_t d, const int64_t* true_pos, float* thr,
                                  int32_t* greater, int32_t* equal, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(nq >= 0 && nb >= 0, "allpairs_rank: negative size");
  if (nq == 0) return RGCN_OK;
  int rc = check_ap(A, lda, B, ldb, d);
  if (rc) return rc;
  RGCN_CHECK_ARG(true_pos && thr && greater && equal, "allpairs_rank: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  RGCN_CUDA(cudaMemsetAsync(greater, 0, (size_t)nq * sizeof(int32_t), st));
  RGCN_CUDA(cudaMemsetAsync(equal, 0, (size_t)nq * sizeof(int32_t), st));
  threshold_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, st>>>(A, lda, B, ldb, b_idx, true_pos, nq, d, thr);
  RGCN_LAUNCH_CHECK();
  if (nb == 0) return RGCN_OK;
  dim3 grid((unsigned)((nb + TN - 1) / TN), (unsigned)((nq + TM - 1) / TM));
  allpairs_kernel<1><<<grid, 256, 0, st>>>(A, lda, nq, B, ldb, b_idx, nb, d, 1.f, 0.f, nullptr, 0, thr, true_pos, greater,
                                           equal);
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

// ---- rank from a materialised score block (the tensor-core path) ---------------------------------------------------
// greater[i] = #{j != t_i : s[i, j] > s[i, t_i]}, equal[i] = #{j != t_i : s[i, j] == s[i, t_i]} over the first n_cand
// columns of row i; the threshold is read from the same matrix, the true tail is excluded by INDEX, so there are no
// self-comparison artefacts whatever the accumulation order of the GEMM that produced the scores.
namespace rgcn {
__global__ void __launch_bounds__(256) rank_count_kernel(const float* __restrict__ s, int64_t ld, int64_t nq, int64_t n_cand,
                                                         const int64_t* __restrict__ true_pos, float* __restrict__ thr,
                                                         int32_t* __restrict__ greater, int32_t* __restrict__ equal) {
  pdl_enter();
  __shared__ int sg[8], se[8];
  const int64_t i = blockIdx.x;
  if (i >= nq) return;
  const float* __restrict__ row = s + i * ld;
  const int64_t t = true_pos[i];
  const float th = row[t];
  int g = 0, e = 0;
  for (int64_t j = threadIdx.x; j < n_cand; j += 256) {
    const float v = row[j];
    if (j != t) { g += v > th; e += v == th; }
  }
  for (int o = 16; o; o >>= 1) {
    g += __shfl_xor_sync(0xffffffffu, g, o);
    e += __shfl_xor_sync(0xffffffffu, e, o);
  }
  if ((threadIdx.x & 31) == 0) { sg[threadIdx.x >> 5] = g; se[threadIdx.x >> 5] = e; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { g += sg[w]; e += se[w]; }
    greater[i] = g; equal[i] = e;
    if (thr) thr[i] = th;
  }
}
}  // namespace rgcn

extern "C" int rgcn_rank_count(const float* scores, int64_t ld, int64_t nq, int64_t n_cand, const int64_t* true_pos,
                               float* thr, int32_t* greater, int32_t* equal, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(nq >= 0 && n_cand > 0 && ld >= n_cand, "rank_count: bad sizes");
  RGCN_CHECK_ARG(nq == 0 || (scores && true_pos && greater && equal), "rank_count: null argument");
  if (nq == 0) return RGCN_OK;
  RGCN_CUDA(launch_pdl(rgcn::rank_count_kernel, dim3((unsigned)nq), dim3(256), 0, (cudaStream_t)stream, scores, ld, nq, n_cand,
                       true_pos, thr, greater, equal));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

// ---- filtered ranks from an unfiltered count -------------------------------------------------------------------------
// After rgcn_rank_count (materialised block) or rgcn_allpairs_rank (fp32 FMA tiles): every excluded position j != t_i of
// row i whose score is > / == thr[i] is taken back out of greater[i] / equal[i].  The score carries the counting pass's
// own bits: read from the block, or recomputed with the tile kernel's accumulation (fmaf, k ascending).  One warp per
// row, integer updates: deterministic.
namespace rgcn {
__global__ void __launch_bounds__(256) rank_excl_correct_kernel(const float* __restrict__ s, int64_t lds,
                                                                const float* __restrict__ A, int64_t lda,
                                                                const float* __restrict__ B, int64_t ldb,
                                                                const int64_t* __restrict__ b_idx, int32_t d, int64_t nq,
                                                                int64_t n_cand, const int64_t* __restrict__ true_pos,
                                                                const float* __restrict__ thr,
                                                                const int64_t* __restrict__ excl_begin,
                                                                const int64_t* __restrict__ excl_end,
                                                                const int32_t* __restrict__ excl_pos,
                                                                int32_t* __restrict__ greater, int32_t* __restrict__ equal) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= nq) return;
  const int64_t t = true_pos[i];
  const float th = thr[i];
  int g = 0, e = 0;
  for (int64_t x = excl_begin[i] + lane; x < excl_end[i]; x += 32) {
    const int64_t j = excl_pos[x];
    if (j == t || j < 0 || j >= n_cand) continue;
    float v;
    if (s) {
      v = s[i * lds + j];
    } else {
      const float* a = A + i * lda;
      const float* b = B + (b_idx ? b_idx[j] : j) * ldb;
      float acc = 0.f;
      for (int k = 0; k < d; ++k) acc = fmaf(a[k], b[k], acc);
      v = acc;
    }
    g += v > th;
    e += v == th;
  }
  for (int o = 16; o; o >>= 1) {
    g += __shfl_xor_sync(0xffffffffu, g, o);
    e += __shfl_xor_sync(0xffffffffu, e, o);
  }
  if (lane == 0) { greater[i] -= g; equal[i] -= e; }
}
}  // namespace rgcn

extern "C" int rgcn_rank_excl_correct(const float* scores, int64_t ld, const float* A, int64_t lda, const float* B,
                                      int64_t ldb, const int64_t* b_idx, int32_t d, int64_t nq, int64_t n_cand,
                                      const int64_t* true_pos, const float* thr, const int64_t* excl_begin,
                                      const int64_t* excl_end, const int32_t* excl_pos, int32_t* greater, int32_t* equal,
                                      rgcn_stream_t stream) {
  RGCN_CHECK_ARG(nq >= 0 && n_cand >= 0, "rank_excl_correct: negative size");
  if (nq == 0) return RGCN_OK;
  RGCN_CHECK_ARG(true_pos && thr && excl_begin && excl_end && excl_pos && greater && equal,
                 "rank_excl_correct: null argument");
  if (scores) {
    RGCN_CHECK_ARG(ld >= n_cand, "rank_excl_correct: ld < n_cand");
  } else {
    RGCN_CHECK_ARG(A && B && d > 0, "rank_excl_correct: needs the score block or the operands A, B");
  }
  RGCN_CUDA(launch_pdl(rgcn::rank_excl_correct_kernel, dim3((unsigned)((nq + 7) / 8)), dim3(256), 0, (cudaStream_t)stream,
                       scores, ld, A, lda, B, ldb, b_idx, d, nq, n_cand, true_pos, thr, excl_begin, excl_end, excl_pos,
                       greater, equal));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

