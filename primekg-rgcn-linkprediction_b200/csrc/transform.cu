// Relational transform of one RGCN layer on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
//   forward  O  = [H | X] @ [Wf ; root] + bias (, ReLU)          M = nodes, N = d_out, K = (R+1) d_in
//   dgrad    gA = G @ [Wf ; root]^T                              M = nodes, N = (R+1) d_in, K = d_out
//   wgrad    [gWf ; g_root] = [H | X]^T @ G,  g_bias = column sums of G       M = (R+1) d_in, N = d_out, K = nodes
//   (G = gO * relu', formed once by rgcn_split_planes)
//
// These are the R+1 per-relation `h_r @ W_r` / `x @ root` products of RGCNConv (reference call sites
// src/models/rgcn.py:123, :128) and their autograd transposes (src/train.py:306), concatenated along K so
// that one tile pass serves all relations.
//
// Operand format: "bf16 planes".  Every fp32 activation matrix is kept as a bf16 `hi` plane (x rounded to bf16)
// and, in the fp32 mode, a bf16 `lo` plane (x - hi rounded to bf16; hi + lo = x to 2^-17).  The aggregation kernel
// writes H straight into planes, rgcn_split_planes converts X / gO (fusing the ReLU-backward mask and the bias-gradient
// column sums), and the weights are split by a tiny prep kernel.  Same bytes as fp32, but every GEMM operand is then
// TMA-loadable into the 128B-swizzled UMMA layout: no loader warps, no conversions in the GEMM.
//   mode 0 "fp32": D += hi*hi + hi*lo + lo*hi   (three tcgen05.mma per K step, ~1e-5 relative error)
//   mode 1 "bf16": D += hi*hi                   (the "bf16-transform" mode, tolerance 2e-2)
// fp32 accumulation in TMEM in both.
//
// Kernel anatomy (one CTA = one 128 x BN output tile, BN <= 256 TMEM columns):
//   TMA warp : one thread streams A and B tiles with cp.async.bulk.tensor (SWIZZLE_128B) into a ring of stages
//   MMA warp : one thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) and tcgen05.commit
//   epilogue : tcgen05.ld -> bias / ReLU -> staging tile in the idle operand smem -> coalesced 128-bit row stores
#include <cuda.h>
#include <limits.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm_common.cuh"
#include "tc05.cuh"

namespace rgcn {
using namespace tc05;

__device__ __forceinline__ float4 lds4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts4(uint32_t a, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

constexpr int BM = 128;         // UMMA M
constexpr int BK = 64;          // K per stage for K-major operands (= one 128-byte swizzle row of bf16)
constexpr int BNMAX = 256;      // UMMA N max = TMEM columns per accumulator
constexpr int WG_BK = 32;       // nodes per stage in the weight-gradient kernel
constexpr int kMaxPeers = 8;    // GPUs of one NVSwitch domain the fused all-gather epilogue can address

// ------------------------------------------------------------------------------------------------
// fp32 -> bf16 planes
// ------------------------------------------------------------------------------------------------

// x [rows, cols] fp32 -> hi (, lo) planes; optional ReLU-backward mask (x zeroed where mask <= 0); optional
// per-block column sums of the masked x (fixed order => deterministic bias gradient).
__global__ void __launch_bounds__(256) split_planes_kernel(const float* __restrict__ x, int64_t ldx,
                                                           const float* __restrict__ mask, int64_t ldm, int64_t rows,
                                                           int cols, __nv_bfloat16* __restrict__ hi,
                                                           __nv_bfloat16* __restrict__ lo, int64_t ldp,
                                                           float* __restrict__ colsum_partial, int64_t rows_per_block,
                                                           float scale, float* __restrict__ out_f32, int64_t ldf) {
  pdl_enter();
  __shared__ float4 red[256];
  const int tpr = cols >> 2;                       // threads per row (<= 256)
  const int rpp = 256 / tpr;                       // rows per pass
  const int c4 = threadIdx.x % tpr, rsub = threadIdx.x / tpr;
  const int64_t r_beg = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r_end = min(r_beg + rows_per_block, rows);
  float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
  if (rsub < rpp) {
    constexpr int U = 4;                           // independent rows in flight per thread
    for (int64_t r0 = r_beg + rsub; r0 < r_end; r0 += (int64_t)U * rpp) {
      float4 v[U], m[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t r = r0 + (int64_t)u * rpp;
        const bool ok = r < r_end;
        v[u] = ok ? ldg4(x + r * ldx + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (mask) m[u] = ok ? ldg4(mask + r * ldm + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t r = r0 + (int64_t)u * rpp;
        if (r < r_end) {
          if (mask) {
            if (!(m[u].x > 0.f)) v[u].x = 0.f;
            if (!(m[u].y > 0.f)) v[u].y = 0.f;
            if (!(m[u].z > 0.f)) v[u].z = 0.f;
            if (!(m[u].w > 0.f)) v[u].w = 0.f;
            v[u] = scale4(v[u], scale);                // 1 / (1 - p) of a fused dropout, else 1
          }
          add4(cs, v[u]);
          if (out_f32) *reinterpret_cast<float4*>(out_f32 + r * ldf + c4 * 4) = v[u];
          uint2 h, l;
          split4(v[u], h, l);
          *reinterpret_cast<uint2*>(hi + r * ldp + c4 * 4) = h;
          if (lo) *reinterpret_cast<uint2*>(lo + r * ldp + c4 * 4) = l;
        }
      }
    }
  }
  if (colsum_partial) {
    red[threadIdx.x] = cs;
    __syncthreads();
    if (rsub == 0) {
      float4 s = red[c4];
      for (int j = 1; j < rpp; ++j) add4(s, red[j * tpr + c4]);
      *reinterpret_cast<float4*>(colsum_partial + (size_t)blockIdx.x * cols + c4 * 4) = s;
    }
  }
}


// weights: fp32 [K1 + K2, N] (two row blocks) -> bf16 hi / lo, optionally transposed, zero padded.
// seed_state (nullable): the dropout step counter, advanced here once per layer call (stream-ordered before the GEMM
// that reads it, and replayed with the CUDA graph, so every step draws a fresh mask without host involvement).
__global__ void split_weights_kernel(const float* __restrict__ w1, int K1, const float* __restrict__ w2, int K2, int N,
                                     int transpose, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                     int rows_pad, int cols_pad, unsigned long long* seed_state) {
  pdl_enter();
  if (seed_state && blockIdx.x == 0 && threadIdx.x == 0) *seed_state += 1ull;
  // output [rows_pad, cols_pad]; transpose: out[n][k] = W[k][n], else out[k][n] = W[k][n]
  const int64_t total = (int64_t)rows_pad * cols_pad;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols_pad), c = (int)(i % cols_pad);
    const int k = transpose ? c : r, n = transpose ? r : c;
    float v = 0.f;
    if (k < K1 + K2 && n < N) v = (k < K1) ? w1[(int64_t)k * N + n] : w2[(int64_t)(k - K1) * N + n];
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    hi[i] = h;
    if (lo) lo[i] = l;
  }
}

// ------------------------------------------------------------------------------------------------
// K-major GEMM: out[M, N] = A[M, K] @ B[N, K]^T   (forward and dgrad); A and B are bf16 planes fed by TMA
// ------------------------------------------------------------------------------------------------
struct GemmKParams {
  int64_t M;
  int N;                                      // valid output columns
  int BN;                                     // tile width: multiple of 32, <= 128
  int n_tiles;                                // column tiles
  int num_kb;                                 // K blocks of 64 (TMA zero-fills past the true K)
  const float* bias; int relu;
  float* out; int64_t ldo;
  __nv_bfloat16* out16; int64_t ldo16;        // optional second output: the same values rounded to bf16 (the next layer's
                                              // gather source in the bf16-transform mode)
  // fused dropout after the ReLU (training): keep iff drop_bits(...) >= drop_thresh, kept values times drop_scale
  uint32_t drop_thresh; float drop_scale; uint32_t drop_seed; const unsigned long long* drop_ctr;
  int64_t row_offset;                         // row of the layer's output that local row 0 is (row-chunked calls): dropout index
  // ---- epilogues that consume the accumulator instead of storing it (all-pairs scoring, csrc/rank.cu comments) ----
  int tile_contig;                            // CTA c takes a CONTIGUOUS run of tiles (mostly one row tile): per-row state
                                              // stays in registers across column tiles
  int diag;                                   // only the diagonal tiles (row tile t with column tile t), BN == 128
  int64_t n_cols_valid;                       // candidates beyond this column are padding
  const float* thr_in; float* thr_out;        // EPI_RANK: per-row threshold;  EPI_THR: out[row] = acc[row, row]
  const int64_t* true_pos; int32_t* greater; int32_t* equal;
  float alpha, beta;                          // EPI_TOPK: reported value = alpha * acc + beta (alpha > 0)
  float* cand_val; int32_t* cand_idx; int32_t* slot_ctr; int32_t n_slots;    // [M, n_slots, kTopK] partial lists, [M] counters
  // fused all-gather: every output tile is also stored into the same-shaped slot (rows peer_row0 ...) of up to
  // kMaxPeers feature buffers that live in OTHER GPUs' memory (peer-mapped, NVLink stores issued by the epilogue)
  float* peer_out[kMaxPeers]; int n_peer; int64_t peer_row0; int64_t peer_ld;
  // scattered output rows (listed-rows forward of the last layer): row c of the product goes to out[out_rows[c]] for
  // c < n_out_rows, the padding rows beyond are dropped (duplicates in the list write identical values)
  const int64_t* out_rows; int64_t n_out_rows;
  const int32_t* out_slot;                    // nullable: node -> first list position; later duplicates are not stored
  // TMA-store epilogue (plain / dropout store loops): every warp's 32 x 16 patch leaves shared memory as ONE bulk tensor
  // store (cp.async.bulk.tensor: the patch's XOR swizzle is the tensor map's 64-byte swizzle); rows / columns beyond the
  // matrix are clipped by the copy engine
  int tma_store;
  alignas(64) CUtensorMap tm_out;
  // EPI_RANK / EPI_TOPK with exclusion (the EXCL instantiations): row i skips the candidate positions
  // excl_pos[excl_begin[i] .. excl_end[i]), sorted ascending and distinct.  (Last, so that the fields above keep their
  // offsets: the unfiltered rank / top-k instantiations compile to the same SASS.)
  const int64_t* excl_begin; const int64_t* excl_end; const int32_t* excl_pos;
};

enum { EPI_STORE = 0, EPI_RANK = 1, EPI_THR = 2, EPI_TOPK = 3 };
constexpr int kTopK = 16;                     // entries every epilogue lane keeps per row (top-K requests up to this)
constexpr int KBN = 128;                      // N tile of the persistent kernel: two accumulators fit 256 TMEM columns
// Epilogue warps: a warp may only address the TMEM lane quarter 32 (w % 4) .. +31, so the warps of a quarter share the
// tile's COLUMNS.  The storing epilogue is latency bound (TMEM load -> patch -> global stores, a few hundred dependent
// cycles per 16-column chunk) and takes four warps per quarter; the consuming epilogues (rank / threshold / top-k) keep
// per-row state over a contiguous half of the columns and stay at two.
constexpr int K_EPI_WARPS = 8;                // consuming epilogues: two warps per quarter, half of the columns each
constexpr int K_EPI_WARPS_STORE = 16;         // storing epilogue: four per quarter, 16-column chunks dealt round robin
constexpr int K_PATCH = 32 * 20 * 4;          // per-warp patch, consuming epilogues: 32 lanes x 10 staged (value, index) pairs
constexpr int K_PATCH_STORE = 32 * 16 * 4;    // per-warp transpose patch, storing epilogue: 32 rows x 16 floats, XOR swizzled
constexpr int K_THREADS = (K_EPI_WARPS + 2) * 32;
constexpr int K_THREADS_STORE = (K_EPI_WARPS_STORE + 2) * 32;
constexpr int epi_warps(int epi) { return epi == 0 ? K_EPI_WARPS_STORE : K_EPI_WARPS; }
constexpr int epi_patch(int epi) { return epi == 0 ? K_PATCH_STORE : K_PATCH; }

// BNT = widest column tile the instantiation can hold: 128 (two accumulators in 256 TMEM columns, 3 / 6 stages) or 256
// (two accumulators fill the 512 TMEM columns; A is then read once for 256 output columns — the K = 1,024 forward is
// bound by the L2 -> SM ingest of its operands, not by the tensor pipe — at the price of a 2 / 4 stage ring)
template <bool SPLIT, int BNT = 128>
struct KStage {
  static constexpr int A_BYTES = BM * 128;              // 128 rows x 64 bf16
  static constexpr int B_BYTES = BNT * 128;
  static constexpr int BYTES = (SPLIT ? 2 : 1) * (A_BYTES + B_BYTES);
  static constexpr int STAGES = BNT == 256 ? (SPLIT ? 2 : 4) : (SPLIT ? 3 : 6);
  static constexpr int A_HI = 0, A_LO = A_BYTES;
  static constexpr int B_HI = (SPLIT ? 2 : 1) * A_BYTES, B_LO = B_HI + B_BYTES;
  static constexpr int SMEM = STAGES * BYTES + K_EPI_WARPS * K_PATCH + 1024;                    // consuming epilogues
  static constexpr int SMEM_STORE = STAGES * BYTES + K_EPI_WARPS_STORE * K_PATCH_STORE + 1024;  // storing epilogue
};

// Persistent, warp-specialised: CTA c walks tiles c, c + grid, ... (column tile fastest, so neighbouring CTAs share
// the A rows in L2).  The smem ring and the two TMEM accumulators are continuous across tiles: the MMA warp starts
// tile i+1 while the epilogue warps drain tile i.
// B_MN = false: B is K-major ([N, K] rows of K, the dgrad / all-pairs operand);  B_MN = true: B is MN-major ([K, N] rows
// of N — the weight matrix exactly as PyTorch stores it, so the forward needs no transposed copy): the stage then holds
// ceil(BN / 64) chunks of 64 k-rows x 128 B, the layout of the weight-gradient kernel's operands.
// XF (EPI_STORE only) specialises the store loop, which is where an epilogue-bound launch spends its instructions:
// 0 = plain store, 1 = + fused dropout, 2 = everything decided at run time (bf16 copy, peer stores, scattered rows)
// EXCL (EPI_RANK / EPI_TOPK only): skip each row's excluded candidate positions (p.excl_*).  A lane visits its row's
// columns in ascending order (a CTA run walks its column tiles in order, the warp its half of each tile chunk by chunk),
// so one cursor per lane walks the sorted list: one comparison per element, a load only when the cursor advances.
template <bool SPLIT, bool B_MN, int EPI = EPI_STORE, int BNT = 128, int XF = 2, bool EXCL = false>
__global__ void __launch_bounds__((epi_warps(EPI) + 2) * 32, 1)
gemm_kmajor_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                   const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                   const __grid_constant__ GemmKParams p) {
  using S = KStage<SPLIT, BNT>;
  constexpr int EW = epi_warps(EPI);              // epilogue warps; warp EW = TMA producer, warp EW + 1 = MMA issuer
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[S::STAGES], empty_bar[S::STAGES], tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float s_bias[256];      // the whole bias when N <= 256 (wider layers read it from global memory)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t m_tiles = (p.M + BM - 1) / BM;
  const int64_t n_tiles_total = p.diag ? m_tiles : m_tiles * p.n_tiles;
  // tile schedule, the same in all three roles: strided (neighbouring CTAs share the A rows in L2) or contiguous runs
  int64_t t_begin = blockIdx.x, t_end = n_tiles_total, t_step = gridDim.x;
  if (p.tile_contig) {
    const int64_t per = (n_tiles_total + gridDim.x - 1) / gridDim.x;
    t_begin = (int64_t)blockIdx.x * per;
    t_end = t_begin + per < n_tiles_total ? t_begin + per : n_tiles_total;
    t_step = 1;
  }
  auto tile_mi = [&](int64_t t) { return p.diag ? t : t / p.n_tiles; };
  auto tile_ni = [&](int64_t t) { return p.diag ? t : t % p.n_tiles; };
  const uint32_t acc_cols = p.BN <= 32 ? 32 : p.BN <= 64 ? 64 : p.BN <= 128 ? 128 : 256;     // columns of one accumulator
  const uint32_t tmem_cols = 2 * acc_cols;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);               // the TMA thread's arrive.expect_tx
      mbar_init(&empty_bar[s], 1);              // one tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);              // tcgen05.commit after the tile's last MMA
      mbar_init(&tempty_bar[a], EW);            // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == EW && lane == 0) {
    tma_prefetch_desc(&tm_a_hi);
    tma_prefetch_desc(&tm_b_hi);
    if (SPLIT) { tma_prefetch_desc(&tm_a_lo); tma_prefetch_desc(&tm_b_lo); }
  }
  if (warp == 0) tmem_alloc(&tmem_base_smem, tmem_cols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_smem;
  // everything above is independent of the predecessor's data: barriers, TMEM, descriptor prefetch
  pdl_launch_dependents();
  pdl_wait();
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_bias[i] = (p.bias && i < p.N) ? p.bias[i] : 0.f;
  __syncthreads();

  if (warp < EW) {
    // ===================== epilogue: warp w drains TMEM lanes 32 (w % 4) .. +31 (the quarter a warp may address) in
    // sub-chunks of 16 columns: the storing epilogue deals the chunks round robin to the quarter's four warps (chunk
    // w / 4, w / 4 + 4, ...), the consuming ones give warp w the contiguous half w / 4 of the columns ===============
    const int quarter = warp & 3, half = warp >> 2;
    const int c_lo = EPI == EPI_STORE ? half * 16 : half * (p.BN >> 1);
    const int c_hi = EPI == EPI_STORE ? p.BN : c_lo + (p.BN >> 1);
    constexpr int c_step = EPI == EPI_STORE ? (EW / 4) * 16 : 16;
    float* patch = reinterpret_cast<float*>(smem + (size_t)S::STAGES * S::BYTES + (size_t)warp * epi_patch(EPI));
    const uint32_t patch_s = smem_u32(patch);              // (explicit shared-space accesses: the pointer arithmetic above
                                                           //  hides the address space from the compiler -> generic LD / ST)
    constexpr bool DROP = XF >= 1, EXTRA = XF == 2;
    uint32_t drop_key = 0, bk_small = 0;
    bool drop_small = false;
    if (DROP && p.drop_thresh) {
      const unsigned long long ctr = *p.drop_ctr;
      drop_key = pcg_hash(p.drop_seed ^ (uint32_t)ctr) + (uint32_t)(ctr >> 32);
      // fewer than 2^32 elements: every element lies in block 0, whose key is computed once
      drop_small = (unsigned long long)(p.M + p.row_offset) * (unsigned long long)p.N < (1ull << 32);
      bk_small = drop_block_key(drop_key, 0);
    }
    // per-row state of the consuming epilogues (one row per lane)
    int64_t cur_m0 = -1;
    int cnt_g = 0, cnt_e = 0;
    float thr = 0.f;
    int64_t tpos = -1;
    float topv[EPI == EPI_TOPK ? kTopK : 1];
    int topi[EPI == EPI_TOPK ? kTopK : 1];
    constexpr int kTopBuf = 10;                               // staged candidates per lane (K_PATCH = 32 lanes x 10 x 8 B)
    uint2* tbuf = reinterpret_cast<uint2*>(patch);
    int bcnt = 0;
    float kth = -INFINITY;                                    // the list's last entry as of the last drain
    // exclusion cursor (EXCL): x_next = excl_pos[x_cur], or INT_MAX past the end of the row's list
    int64_t x_cur = 0, x_end = 0;
    int x_next = INT_MAX;
    auto x_advance = [&]() { ++x_cur; x_next = x_cur < x_end ? p.excl_pos[x_cur] : INT_MAX; };
    auto drain = [&]() {
      const int mx = __reduce_max_sync(0xffffffffu, bcnt);
      for (int e = 0; e < mx; ++e) {
        const bool has = e < bcnt;
        const uint2 c = has ? tbuf[lane + 32 * e] : make_uint2(0u, 0u);
        float v = __uint_as_float(c.x);
        int ci = (int)c.y;
        if (has && v > topv[(EPI == EPI_TOPK ? kTopK : 1) - 1]) {
          // insertion into the descending list; candidates arrive in ascending column order, so an equal value keeps
          // the earlier (lower) column first
#pragma unroll
          for (int i = 0; i < (EPI == EPI_TOPK ? kTopK : 1); ++i) {
            if (v > topv[i]) {
              const float tv = topv[i]; const int ti = topi[i];
              topv[i] = v; topi[i] = ci; v = tv; ci = ti;
            }
          }
        }
      }
      bcnt = 0;
      kth = topv[(EPI == EPI_TOPK ? kTopK : 1) - 1];
      __syncwarp();
    };
    auto flush_row_state = [&]() {
      if (cur_m0 < 0) return;
      if (EPI == EPI_TOPK) drain();
      const int64_t row = cur_m0 + quarter * 32 + lane;
      if (row >= p.M) return;
      if (EPI == EPI_RANK) {
        if (cnt_g) atomicAdd(p.greater + row, cnt_g);        // integer adds: order independent, deterministic
        if (cnt_e) atomicAdd(p.equal + row, cnt_e);
      } else if (EPI == EPI_TOPK) {
        const int slot = atomicAdd(p.slot_ctr + row, 1);     // (slot order varies; the merge sorts by value, then index)
        if (slot < p.n_slots) {
          float* cv = p.cand_val + ((size_t)row * p.n_slots + slot) * kTopK;
          int32_t* ci = p.cand_idx + ((size_t)row * p.n_slots + slot) * kTopK;
#pragma unroll
          for (int i = 0; i < (EPI == EPI_TOPK ? kTopK : 1); ++i) { cv[i] = topv[i]; ci[i] = topi[i]; }
        }
      }
    };
    int iter = 0;
    for (int64_t t = t_begin; t < t_end; t += t_step, ++iter) {
      const int64_t m0 = tile_mi(t) * BM;
      const int n0 = (int)tile_ni(t) * p.BN;
      const int a = iter & 1;
      if (EPI != EPI_STORE && m0 != cur_m0) {
        flush_row_state();
        cur_m0 = m0;
        const int64_t row = m0 + quarter * 32 + lane;
        cnt_g = cnt_e = 0;
        if (EPI == EPI_RANK) {
          thr = row < p.M ? p.thr_in[row] : 0.f;
          tpos = row < p.M ? p.true_pos[row] : -1;
        }
        if (EPI == EPI_TOPK) {
#pragma unroll
          for (int i = 0; i < (EPI == EPI_TOPK ? kTopK : 1); ++i) { topv[i] = -INFINITY; topi[i] = -1; }
          kth = -INFINITY;
          bcnt = 0;
        }
        if (EXCL) {
          // the run may enter the row tile mid-row: start at the lower bound of the first column this warp visits
          int64_t lo = 0, hi = 0;
          if (row < p.M) { lo = p.excl_begin[row]; hi = x_end = p.excl_end[row]; }
          else x_end = 0;
          const int first = n0 + c_lo;
          while (lo < hi) {
            const int64_t mid = lo + ((hi - lo) >> 1);
            if (p.excl_pos[mid] < first) lo = mid + 1; else hi = mid;
          }
          x_cur = lo;
          x_next = x_cur < x_end ? p.excl_pos[x_cur] : INT_MAX;
        }
      }
      mbar_wait(&tfull_bar[a], (uint32_t)((iter >> 1) & 1));
      fence_after_sync();
      const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)a * acc_cols;
      for (int cc = c_lo; cc < c_hi; cc += c_step) {
        uint32_t r[16];
        tmem_ld_32x16(t_lane + cc, r);
        tmem_ld_wait();
        if (EPI != EPI_STORE) {
          const int64_t row = m0 + quarter * 32 + lane;
          if (EXCL) {
            // entries below this chunk: columns of the other half, or of tiles this run does not visit
            while (x_next < n0 + cc) x_advance();
          }
          if (EPI == EPI_RANK) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int64_t col = n0 + cc + j;
              const float v = __uint_as_float(r[j]);
              bool skip = false;
              if (EXCL && x_next == n0 + cc + j) { skip = true; x_advance(); }
              if (row < p.M && col < p.n_cols_valid && col != tpos && !skip) { cnt_g += v > thr; cnt_e += v == thr; }
            }
          } else if (EPI == EPI_THR) {
            // the diagonal element of this lane's row, if it lies in this warp's 16 columns
            const int want = quarter * 32 + lane - cc;
            float v = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j == want) v = __uint_as_float(r[j]);
            if (want >= 0 && want < 16 && row < p.M) p.thr_out[row] = v;
          } else {
            // Staged insertion.  A lane inserting into its sorted list costs the whole warp ~80 instructions, and with 32
            // rows per warp SOME lane wants to insert at almost every column.  So a passing element is only appended
            // to the lane's small buffer in shared memory (the idle transpose patch), and when any lane's buffer fills
            // the warp drains all 32 buffers together: the insertion cost is paid once per ~5 elements per lane.
#pragma unroll
            for (int j0 = 0; j0 < 16; j0 += 4) {
#pragma unroll
              for (int j = j0; j < j0 + 4; ++j) {
                const int col = n0 + cc + j;
                const float v = __uint_as_float(r[j]);
                bool skip = false;
                if (EXCL && x_next == col) { skip = true; x_advance(); }
                if (row < p.M && col < p.n_cols_valid && v > kth && !skip) {
                  tbuf[lane + 32 * bcnt] = make_uint2(r[j], (uint32_t)col);
                  ++bcnt;
                }
              }
              if (__any_sync(0xffffffffu, bcnt >= kTopBuf - 4)) drain();
            }
          }
          continue;
        }
        const bool tma_out = XF < 2 && p.tma_store;            // (kernel-uniform)
        if (tma_out) {
          // the previous chunk's bulk store must have read the patch before it is rewritten
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
        }
        // registers (one row per lane) -> patch, + bias / ReLU
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          float4 b;
          if (p.N <= 256) {
            b = *reinterpret_cast<const float4*>(s_bias + ((n0 + cc + j) & 255));
          } else {
            const int c0 = n0 + cc + j;
            const bool on = p.bias != nullptr && c0 < p.N;                   // (N % 4 == 0)
            b = on ? make_float4(__ldg(p.bias + c0), __ldg(p.bias + c0 + 1), __ldg(p.bias + c0 + 2), __ldg(p.bias + c0 + 3))
                   : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          float4 qv = make_float4(__uint_as_float(r[j]) + b.x, __uint_as_float(r[j + 1]) + b.y,
                                  __uint_as_float(r[j + 2]) + b.z, __uint_as_float(r[j + 3]) + b.w);
          if (p.relu) { qv.x = fmaxf(qv.x, 0.f); qv.y = fmaxf(qv.y, 0.f); qv.z = fmaxf(qv.z, 0.f); qv.w = fmaxf(qv.w, 0.f); }
          // row `lane`, 16-byte chunk j / 4, XOR swizzled by the row pair: conflict-free for the row-wise writes here and
          // for the 8-rows x 64-byte reads below, without padding (16 warps' patches must fit beside the operand ring)
          if (tma_out && DROP && (XF == 1 || p.drop_thresh)) {
            // lane = row: the same (row, column) -> bits map as the store loop below
            const int64_t row = m0 + quarter * 32 + lane;
            const uint32_t e32 = (uint32_t)(row + p.row_offset) * (uint32_t)p.N + (uint32_t)(n0 + cc + j);
            const uint32_t bk = drop_small ? bk_small
                                           : drop_block_key(drop_key, (uint64_t)(row + p.row_offset) * (uint64_t)p.N + (uint64_t)(n0 + cc + j));
            const uint32_t h0 = pcg_hash(e32 ^ bk), h1 = pcg_hash((e32 + 2) ^ bk);
            qv.x = (h0 & 0xffffu) >= p.drop_thresh ? qv.x * p.drop_scale : 0.f;
            qv.y = (h0 >> 16) >= p.drop_thresh ? qv.y * p.drop_scale : 0.f;
            qv.z = (h1 & 0xffffu) >= p.drop_thresh ? qv.z * p.drop_scale : 0.f;
            qv.w = (h1 >> 16) >= p.drop_thresh ? qv.w * p.drop_scale : 0.f;
          }
          sts4(patch_s + (uint32_t)(lane * 16 + (((j >> 2) ^ ((lane >> 1) & 3)) << 2)) * 4u, qv);
        }
        if (tma_out) {
          fence_proxy_async();                                   // generic-proxy patch writes -> visible to the copy engine
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&p.tm_out, patch_s, n0 + cc, (int)(m0 + quarter * 32));
            bulk_commit();
          }
          continue;
        }
        __syncwarp();
        // patch -> global: each instruction writes 8 rows x 64 contiguous bytes
        const int c4 = (lane & 3) * 4;
        const bool col_ok = n0 + cc + c4 < p.N;
#pragma unroll
        for (int rr = 0; rr < 32; rr += 8) {
          const int rl = rr + (lane >> 2);
          int64_t row = m0 + quarter * 32 + rl;
          if (row < p.M && col_ok) {
            if (EXTRA && p.out_rows) {
              if (row >= p.n_out_rows) continue;
              const int64_t pos = row;
              row = __ldg(p.out_rows + pos);
              if (p.out_slot && __ldg(p.out_slot + row) != (int32_t)pos) continue;
            }
            float4 v = lds4(patch_s + (uint32_t)(rl * 16 + (((c4 >> 2) ^ ((rl >> 1) & 3)) << 2)) * 4u);
            if (DROP && (XF == 1 || p.drop_thresh)) {
              // N % 4 == 0, so the four elements of one store never straddle a 2^32 block; the low 32 bits of the element
              // index are a 32-bit product, the block key needs the high part only beyond 2^32 elements
              const uint32_t e32 = (uint32_t)(row + p.row_offset) * (uint32_t)p.N + (uint32_t)(n0 + cc + c4);
              const uint32_t bk = drop_small ? bk_small
                                             : drop_block_key(drop_key, (uint64_t)(row + p.row_offset) * (uint64_t)p.N + (uint64_t)(n0 + cc + c4));
              // two hashes per store, 16 random bits per element (p is resolved to 2^-16)
              const uint32_t h0 = pcg_hash(e32 ^ bk), h1 = pcg_hash((e32 + 2) ^ bk);
              v.x = (h0 & 0xffffu) >= p.drop_thresh ? v.x * p.drop_scale : 0.f;
              v.y = (h0 >> 16) >= p.drop_thresh ? v.y * p.drop_scale : 0.f;
              v.z = (h1 & 0xffffu) >= p.drop_thresh ? v.z * p.drop_scale : 0.f;
              v.w = (h1 >> 16) >= p.drop_thresh ? v.w * p.drop_scale : 0.f;
            }
            *reinterpret_cast<float4*>(p.out + row * p.ldo + n0 + cc + c4) = v;
            if (EXTRA) {
              if (p.out16) {
                __nv_bfloat162 b01 = __floats2bfloat162_rn(v.x, v.y), b23 = __floats2bfloat162_rn(v.z, v.w);
                uint2 o;
                o.x = *reinterpret_cast<uint32_t*>(&b01);
                o.y = *reinterpret_cast<uint32_t*>(&b23);
                *reinterpret_cast<uint2*>(p.out16 + row * p.ldo16 + n0 + cc + c4) = o;
              }
              for (int q = 0; q < p.n_peer; ++q)
                *reinterpret_cast<float4*>(p.peer_out[q] + (p.peer_row0 + row) * p.peer_ld + n0 + cc + c4) = v;
            }
          }
        }
        __syncwarp();
      }
      fence_before_sync();
      if (lane == 0) mbar_arrive(&tempty_bar[a]);       // accumulator a may be overwritten
    }
    if (EPI != EPI_STORE) flush_row_state();
    if (EPI == EPI_STORE && XF < 2 && p.tma_store && lane == 0) bulk_wait0();     // the last bulk stores have landed
  } else if (warp == EW) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      // a TMA box always delivers its full byte count (out-of-range elements arrive as zeros)
      const int b_chunks = (p.BN + 63) / 64;                                // MN-major B: boxes of 64 n x BK k
      const uint32_t b_bytes = B_MN ? (uint32_t)b_chunks * (uint32_t)(BK * 128) : (uint32_t)p.BN * 128u;
      const uint32_t bytes = ((uint32_t)BM * 128u + b_bytes) * (SPLIT ? 2u : 1u);
      uint32_t it = 0;
      for (int64_t t = t_begin; t < t_end; t += t_step) {
        const int m0 = (int)(tile_mi(t) * BM);
        const int n0 = (int)tile_ni(t) * p.BN;
        for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
          const int s = it % S::STAGES;
          const uint32_t ph = (it / S::STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);      // slot free (passes immediately on the first round)
          uint8_t* st = smem + (size_t)s * S::BYTES;
          mbar_arrive_expect_tx(&full_bar[s], bytes);
          tma_load_2d(st + S::A_HI, &tm_a_hi, &full_bar[s], kb * BK, m0);
          if (SPLIT) tma_load_2d(st + S::A_LO, &tm_a_lo, &full_bar[s], kb * BK, m0);
          if (B_MN) {
            for (int ch = 0; ch < b_chunks; ++ch) {
              tma_load_2d(st + S::B_HI + ch * (BK * 128), &tm_b_hi, &full_bar[s], n0 + ch * 64, kb * BK);
              if (SPLIT) tma_load_2d(st + S::B_LO + ch * (BK * 128), &tm_b_lo, &full_bar[s], n0 + ch * 64, kb * BK);
            }
          } else {
            tma_load_2d(st + S::B_HI, &tm_b_hi, &full_bar[s], kb * BK, n0);
            if (SPLIT) tma_load_2d(st + S::B_LO, &tm_b_lo, &full_bar[s], kb * BK, n0);
          }
        }
      }
    }
  } else {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = idesc_bf16(BM, p.BN, 0, B_MN ? 1 : 0);
      uint32_t it = 0;
      int iter = 0;
      for (int64_t t = t_begin; t < t_end; t += t_step, ++iter) {
        const int a = iter & 1;
        mbar_wait(&tempty_bar[a], (uint32_t)(((iter >> 1) & 1) ^ 1));   // epilogue has drained this accumulator
        fence_after_sync();
        const uint32_t tacc = tmem_base + (uint32_t)a * acc_cols;
        for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
          const int s = it % S::STAGES;
          const uint32_t ph = (it / S::STAGES) & 1;
          mbar_wait(&full_bar[s], ph);
          fence_after_sync();
          const uint32_t base = smem_u32(smem + (size_t)s * S::BYTES);
          const uint64_t da_hi = smem_desc_sw128(base + S::A_HI, 16, 1024);
          const uint64_t da_lo = smem_desc_sw128(base + S::A_LO, 16, 1024);
          // MN-major B: LBO = stride between the 64-column chunks, SBO = stride between 8-k groups (as in the wgrad kernel)
          const uint64_t db_hi = B_MN ? smem_desc_sw128(base + S::B_HI, BK * 128, 1024) : smem_desc_sw128(base + S::B_HI, 16, 1024);
          const uint64_t db_lo = B_MN ? smem_desc_sw128(base + S::B_LO, BK * 128, 1024) : smem_desc_sw128(base + S::B_LO, 16, 1024);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t adv = (uint64_t)(k * 32 >> 4);      // 16 bf16 = 32 bytes along K inside the swizzle row
            const uint64_t adv_b = B_MN ? (uint64_t)(k * 2048 >> 4) : adv;   // MN-major: 16 k = two 8-k atoms of 1024 B
            mma_bf16_ss(tacc, da_hi + adv, db_hi + adv_b, idesc, (kb | k) ? 1u : 0u);
            if (SPLIT) {
              mma_bf16_ss(tacc, da_hi + adv, db_lo + adv_b, idesc, 1u);
              mma_bf16_ss(tacc, da_lo + adv, db_hi + adv_b, idesc, 1u);
            }
          }
          mma_commit(&empty_bar[s]);            // frees the stage once these MMAs have read it
        }
        mma_commit(&tfull_bar[a]);              // this tile's accumulator is complete
      }
    }
  }
  __syncthreads();
  if (warp == 0) {
    fence_after_sync();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------
// weight gradient: P[split][m, n] = sum_{node in split} A[node, m] * G[node, n]   (both operands MN-major, TMA fed)
// ------------------------------------------------------------------------------------------------
struct WgradParams {
  int64_t nodes;
  int BN;                                     // tile columns (multiple of 64, <= 256)
  int64_t nodes_per_split;                    // multiple of WG_BK
  float* partial;                             // [splits, m_tiles * 128, ldp]
  int ldp;                                    // = n_tiles * BN
};

template <bool SPLIT>
struct WStage {
  static constexpr int A_BYTES = 2 * WG_BK * 128;        // 2 chunks of 64 m  x 32 nodes x 128 B
  static constexpr int B_BYTES = 4 * WG_BK * 128;        // 4 chunks of 64 n
  static constexpr int BYTES = (SPLIT ? 2 : 1) * (A_BYTES + B_BYTES);
  static constexpr int STAGES = SPLIT ? 4 : 8;
  static constexpr int A_HI = 0, A_LO = A_BYTES;
  static constexpr int B_HI = (SPLIT ? 2 : 1) * A_BYTES, B_LO = B_HI + B_BYTES;
};

template <bool SPLIT>
__global__ void __launch_bounds__(192, 1)
gemm_wgrad_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                  const __grid_constant__ CUtensorMap tm_g_hi, const __grid_constant__ CUtensorMap tm_g_lo,
                  const WgradParams p) {
  using S = WStage<SPLIT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[S::STAGES], empty_bar[S::STAGES], accum_bar;
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x, n_tile = blockIdx.y, split = blockIdx.z;
  const int m0 = m_tile * BM, n0 = n_tile * p.BN;
  const uint32_t tmem_cols = p.BN <= 64 ? 64 : p.BN <= 128 ? 128 : 256;
  const int64_t node_beg = (int64_t)split * p.nodes_per_split;
  const int64_t node_end = min(node_beg + p.nodes_per_split, p.nodes);
  const int num_kb = node_end > node_beg ? (int)((node_end - node_beg + WG_BK - 1) / WG_BK) : 0;
  const int n_chunks = p.BN / 64;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tm_a_hi);
    tma_prefetch_desc(&tm_g_hi);
    if (SPLIT) { tma_prefetch_desc(&tm_a_lo); tma_prefetch_desc(&tm_g_lo); }
  }
  if (warp == 0) tmem_alloc(&tmem_base_smem, tmem_cols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_launch_dependents();
  pdl_wait();

  if (warp < 4) {
    // ===================== epilogue: TMEM -> partial buffer (warp w owns TMEM lanes 32w..32w+31) ==========
    float* prow = p.partial + ((size_t)split * gridDim.x * BM + (size_t)(m0 + warp * 32 + lane)) * p.ldp + n0;
    if (num_kb > 0) {
      mbar_wait(&accum_bar, 0);
      fence_after_sync();
      const uint32_t t_lane = tmem_base + ((uint32_t)(warp * 32) << 16);
      for (int cc = 0; cc < p.BN; cc += 32) {
        uint32_t r[32];
        tmem_ld_32x32(t_lane + cc, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(prow + cc + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                                  __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
      }
      fence_before_sync();
    } else {
      for (int cc = 0; cc < p.BN; cc += 4) *reinterpret_cast<float4*>(prow + cc) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else if (warp == 4) {
    // ===================== TMA producer: boxes of 64 columns x WG_BK node rows =====================
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)(2 + n_chunks) * WG_BK * 128u * (SPLIT ? 2u : 1u);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % S::STAGES;
        const uint32_t ph = (kb / S::STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        uint8_t* st = smem + (size_t)s * S::BYTES;
        const int nd0 = (int)(node_beg + (int64_t)kb * WG_BK);
        mbar_arrive_expect_tx(&full_bar[s], bytes);
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
          tma_load_2d(st + S::A_HI + ch * (WG_BK * 128), &tm_a_hi, &full_bar[s], m0 + ch * 64, nd0);
          if (SPLIT) tma_load_2d(st + S::A_LO + ch * (WG_BK * 128), &tm_a_lo, &full_bar[s], m0 + ch * 64, nd0);
        }
        for (int ch = 0; ch < n_chunks; ++ch) {
          tma_load_2d(st + S::B_HI + ch * (WG_BK * 128), &tm_g_hi, &full_bar[s], n0 + ch * 64, nd0);
          if (SPLIT) tma_load_2d(st + S::B_LO + ch * (WG_BK * 128), &tm_g_lo, &full_bar[s], n0 + ch * 64, nd0);
        }
      }
    }
  } else {
    // ===================== MMA issuer (warp 5) =====================
    if (lane == 0 && num_kb > 0) {
      const uint32_t idesc = idesc_bf16(BM, p.BN, 1, 1);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % S::STAGES;
        const uint32_t ph = (kb / S::STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        fence_after_sync();
        const uint32_t base = smem_u32(smem + (size_t)s * S::BYTES);
        // MN-major: LBO = stride between 64-element M/N chunks, SBO = stride between 8-node groups
        const uint64_t da_hi = smem_desc_sw128(base + S::A_HI, WG_BK * 128, 1024);
        const uint64_t db_hi = smem_desc_sw128(base + S::B_HI, WG_BK * 128, 1024);
        const uint64_t da_lo = smem_desc_sw128(base + S::A_LO, WG_BK * 128, 1024);
        const uint64_t db_lo = smem_desc_sw128(base + S::B_LO, WG_BK * 128, 1024);
#pragma unroll
        for (int k = 0; k < WG_BK / 16; ++k) {
          const uint64_t adv = (uint64_t)(k * 2048 >> 4);      // 16 nodes = two 8-node atoms of 1024 B
          mma_bf16_ss(tmem_base, da_hi + adv, db_hi + adv, idesc, (kb | k) ? 1u : 0u);
          if (SPLIT) {
            mma_bf16_ss(tmem_base, da_hi + adv, db_lo + adv, idesc, 1u);
            mma_bf16_ss(tmem_base, da_lo + adv, db_hi + adv, idesc, 1u);
          }
        }
        mma_commit(&empty_bar[s]);
      }
      mma_commit(&accum_bar);
    }
  }
  __syncthreads();
  if (warp == 0) {
    fence_after_sync();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// fixed-order reduction of the split partials into gW1 [K1, N], gW2 [K2, N]: 4 lanes per output float4, lane q adds
// splits q, q+4, ... in order, then a fixed two-step shuffle combine (deterministic)
__device__ __forceinline__ void colsum_reduce_block(const float* __restrict__ part, int n_part, int N, int c4,
                                                    float* __restrict__ out);

// The last N / 4 blocks of the launch reduce the bias-gradient column sums instead (one launch for both).
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int m_pad,
                                                           int ldp, int K1, int K2, int N, float* __restrict__ gw1,
                                                           float* __restrict__ gw2, int main_blocks,
                                                           const float* __restrict__ colsum_part, int n_colsum,
                                                           float* __restrict__ gbias) {
  pdl_enter();
  if ((int)blockIdx.x >= main_blocks) {
    colsum_reduce_block(colsum_part, n_colsum, N, blockIdx.x - main_blocks, gbias);
    return;
  }
  const int64_t total = (int64_t)(K1 + K2) * (N >> 2);
  const int q = threadIdx.x & 3;
  const int64_t stride_i = (int64_t)main_blocks * (blockDim.x >> 2);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 2) + (threadIdx.x >> 2); i < ((total + 7) & ~int64_t(7));
       i += stride_i) {
    const bool valid = i < total;
    const int m = valid ? (int)(i / (N >> 2)) : 0, n = valid ? (int)(i % (N >> 2)) * 4 : 0;
    const float* src = partial + (size_t)m * ldp + n;
    const size_t stride = (size_t)m_pad * ldp;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid)
      for (int sp = q; sp < splits; sp += 4) add4(s, *reinterpret_cast<const float4*>(src + (size_t)sp * stride));
    for (int o = 1; o <= 2; o <<= 1) {
      s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
      s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
      s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
      s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
    }
    if (valid && q == 0) {
      float* dst = (m < K1) ? gw1 + (size_t)m * N + n : gw2 + (size_t)(m - K1) * N + n;
      *reinterpret_cast<float4*>(dst) = s;
    }
  }
}

// g_bias[n] = sum over the column-sum partials [n_part, N]: one block per float4 column; thread t adds partials
// t, t+256, ...; fixed shuffle tree inside each warp, then the 8 warp sums in order => deterministic
__device__ __forceinline__ void colsum_reduce_block(const float* __restrict__ part, int n_part, int N, int c4,
                                                    float* __restrict__ out) {
  __shared__ float4 wsum[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int p = threadIdx.x; p < n_part; p += 256) add4(s, *reinterpret_cast<const float4*>(part + (size_t)p * N + c4 * 4));
  for (int o = 16; o; o >>= 1) {
    s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
    s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
    s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
    s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
  }
  if (lane == 0) wsum[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float4 t = wsum[0];
    for (int w = 1; w < 8; ++w) add4(t, wsum[w]);
    *reinterpret_cast<float4*>(out + c4 * 4) = t;
  }
}

__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ part, int n_part, int N,
                                                              float* __restrict__ out) {
  pdl_enter();
  colsum_reduce_block(part, n_part, N, blockIdx.x, out);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

struct Tiling { int n_tiles, BN, n_pad; };
static Tiling tile_n(int N, int gran, int bn_max = BNMAX) {
  Tiling t;
  const int np = round_up(N, gran);
  t.n_tiles = (np + bn_max - 1) / bn_max;
  t.BN = round_up((np + t.n_tiles - 1) / t.n_tiles, gran);
  t.n_pad = t.n_tiles * t.BN;
  return t;
}


static int check_plane(const void* p, int64_t ld, const char* what) {
  RGCN_CHECK_ARG(p && ((uintptr_t)p & 15) == 0 && ld % 8 == 0, "transform: plane %s must be non-null, 16-byte aligned, ld %% 8 == 0", what);
  return RGCN_OK;
}

// out[M, N] = A @ B^T with A planes [M, K] (ld lda) and weight planes [n_pad, k_pad]
// B operand: a bf16 matrix [b_rows, b_cols] with leading dimension b_ld.  K-major (b_mn = false): rows = N, cols = K;
// MN-major (b_mn = true): rows = K, cols = N (TMA boxes of 64 columns x BK rows).
template <bool SPLIT, bool B_MN, int BNT, int XF>
static int launch_kmajor_x(const GemmKParams& p, const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& mhi,
                           const CUtensorMap& mlo, unsigned grid, cudaStream_t st) {
  int rc = set_smem(gemm_kmajor_kernel<SPLIT, B_MN, EPI_STORE, BNT, XF>, KStage<SPLIT, BNT>::SMEM_STORE);
  if (rc) return rc;
  RGCN_CUDA(launch_pdl(gemm_kmajor_kernel<SPLIT, B_MN, EPI_STORE, BNT, XF>, dim3(grid), dim3(K_THREADS_STORE), KStage<SPLIT, BNT>::SMEM_STORE, st,
                       ahi, alo, mhi, mlo, p));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

template <bool SPLIT, bool B_MN>
static int launch_kmajor_q(const GemmKParams& p, int xf, const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& mhi,
                           const CUtensorMap& mlo, unsigned grid, cudaStream_t st);

template <bool SPLIT, bool B_MN>
static int launch_kmajor_t(const GemmKParams& p, const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& mhi,
                           const CUtensorMap& mlo, unsigned grid, cudaStream_t st) {
  // the store loop's variant: 2 = run-time everything (bf16 copy, peer stores, scattered rows), 1 = dropout, 0 = plain
  static int force_generic = -1;
  if (force_generic < 0) { const char* e = getenv("RGCN_GENERIC_EPILOGUE"); force_generic = (e && e[0] == '1') ? 1 : 0; }
  const int xf = (force_generic || p.out_rows || p.out16 || p.n_peer) ? 2 : (p.drop_thresh ? 1 : 0);
  static int tma_store = -1;                           // RGCN_TMA_STORE=0: the st.global store loop
  if (tma_store < 0) { const char* e = getenv("RGCN_TMA_STORE"); tma_store = (e && e[0] == '0') ? 0 : 1; }
  GemmKParams q = p;
  if (xf < 2 && tma_store && ((uintptr_t)p.out & 15) == 0 && p.ldo % 4 == 0 && p.N % 4 == 0) {
    int rc = make_out_map(&q.tm_out, p.out, p.M, p.N, p.ldo);
    if (rc) return rc;
    q.tma_store = 1;
  }
  return launch_kmajor_q<SPLIT, B_MN>(q, xf, ahi, alo, mhi, mlo, grid, st);
}

template <bool SPLIT, bool B_MN>
static int launch_kmajor_q(const GemmKParams& p, int xf, const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& mhi,
                           const CUtensorMap& mlo, unsigned grid, cudaStream_t st) {
  if (p.BN > 128) {
    if (xf == 0) return launch_kmajor_x<SPLIT, B_MN, 256, 0>(p, ahi, alo, mhi, mlo, grid, st);
    if (xf == 1) return launch_kmajor_x<SPLIT, B_MN, 256, 1>(p, ahi, alo, mhi, mlo, grid, st);
    return launch_kmajor_x<SPLIT, B_MN, 256, 2>(p, ahi, alo, mhi, mlo, grid, st);
  }
  if (xf == 0) return launch_kmajor_x<SPLIT, B_MN, 128, 0>(p, ahi, alo, mhi, mlo, grid, st);
  if (xf == 1) return launch_kmajor_x<SPLIT, B_MN, 128, 1>(p, ahi, alo, mhi, mlo, grid, st);
  return launch_kmajor_x<SPLIT, B_MN, 128, 2>(p, ahi, alo, mhi, mlo, grid, st);
}

// widest column tile of the prepared-weights transforms (RGCN_WIDE_TILES=0: always 128)
static int wide_bn() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RGCN_WIDE_TILES");
    v = (e && e[0] == '0') ? KBN : 256;
  }
  return v;
}

template <bool SPLIT, bool B_MN, int EPI, bool EXCL = false>
static int launch_kmajor_e(const GemmKParams& p, const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& mhi,
                           const CUtensorMap& mlo, unsigned grid, cudaStream_t st) {
  auto kern = gemm_kmajor_kernel<SPLIT, B_MN, EPI, 128, 2, EXCL>;
  int rc = set_smem(kern, KStage<SPLIT>::SMEM);
  if (rc) return rc;
  RGCN_CUDA(launch_pdl(kern, dim3(grid), dim3(K_THREADS), KStage<SPLIT>::SMEM, st, ahi, alo, mhi, mlo, p));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

static int launch_kmajor(GemmKParams p, const void* a_hi, const void* a_lo, int64_t lda, int K,
                         const __nv_bfloat16* bhi, const __nv_bfloat16* blo, int64_t b_rows, int64_t b_cols, int64_t b_ld,
                         bool b_mn, int n_tiles, bool split, cudaStream_t st, int epi = EPI_STORE) {
  CUtensorMap ahi, alo, mhi, mlo;
  int rc = make_map(&ahi, a_hi, p.M, K, lda, BM);
  if (rc) return rc;
  rc = make_map(&alo, split ? a_lo : a_hi, p.M, K, lda, BM);
  if (rc) return rc;
  rc = make_map(&mhi, bhi, b_rows, b_cols, b_ld, b_mn ? BK : p.BN);
  if (rc) return rc;
  rc = make_map(&mlo, split ? blo : bhi, b_rows, b_cols, b_ld, b_mn ? BK : p.BN);
  if (rc) return rc;
  p.n_tiles = n_tiles;
  const int64_t tiles = p.diag ? (p.M + BM - 1) / BM : ((p.M + BM - 1) / BM) * n_tiles;
  const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
  if (epi != EPI_STORE) {
    // the consuming epilogues serve the all-pairs scorers: K-major candidates, three-product (fp32) mode
    if (b_mn || !split) { set_error("transform: the scoring epilogues need K-major candidates in fp32 mode"); return RGCN_EINVAL; }
    const bool excl = p.excl_pos != nullptr;
    if (epi == EPI_RANK) return excl ? launch_kmajor_e<true, false, EPI_RANK, true>(p, ahi, alo, mhi, mlo, grid, st)
                                     : launch_kmajor_e<true, false, EPI_RANK>(p, ahi, alo, mhi, mlo, grid, st);
    if (epi == EPI_THR) return launch_kmajor_e<true, false, EPI_THR>(p, ahi, alo, mhi, mlo, grid, st);
    return excl ? launch_kmajor_e<true, false, EPI_TOPK, true>(p, ahi, alo, mhi, mlo, grid, st)
                : launch_kmajor_e<true, false, EPI_TOPK>(p, ahi, alo, mhi, mlo, grid, st);
  }
  if (split) return b_mn ? launch_kmajor_t<true, true>(p, ahi, alo, mhi, mlo, grid, st)
                         : launch_kmajor_t<true, false>(p, ahi, alo, mhi, mlo, grid, st);
  return b_mn ? launch_kmajor_t<false, true>(p, ahi, alo, mhi, mlo, grid, st)
              : launch_kmajor_t<false, false>(p, ahi, alo, mhi, mlo, grid, st);
}

static int wgrad_splits(int64_t nodes, int tiles) {
  int s = sm_count() / tiles;                                     // one wave: tiles * splits <= #SMs
  const int64_t max_s = (nodes + 4 * WG_BK - 1) / (4 * WG_BK);      // at least 4 stages of work per split
  if (s > max_s) s = (int)max_s;
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  return s;
}

}  // namespace rgcn

using namespace rgcn;

extern "C" int64_t rgcn_split_planes_blocks(int64_t rows, int32_t cols) {
  if (rows <= 0 || cols < 4) return 0;
  const int rpp = 256 / (cols / 4) > 0 ? 256 / (cols / 4) : 1;
  int64_t nb = (rows + 31) / 32;
  if (nb > 1184) nb = 1184;
  const int64_t rpb = ((rows + nb - 1) / nb + rpp - 1) / rpp * rpp;
  return (rows + rpb - 1) / rpb;
}

extern "C" int rgcn_reduce_partials(const float* part, int64_t n_part, int32_t n_cols, float* out, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(part && out && n_part >= 0 && n_part < (1ll << 31) && n_cols >= 4 && n_cols % 4 == 0,
                 "reduce_partials: n_cols must be a positive multiple of 4");
  RGCN_CHECK_ARG(((uintptr_t)part & 15) == 0 && ((uintptr_t)out & 15) == 0, "reduce_partials: buffers must be 16-byte aligned");
  RGCN_CUDA(launch_pdl(reduce_partials_kernel, dim3((unsigned)(n_cols / 4)), dim3(256), 0, (cudaStream_t)stream, part, (int)n_part, n_cols, out));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_split_planes(const float* x, int64_t ldx, const float* relu_mask, int64_t ldm, int64_t rows,
                                 int32_t cols, void* hi, void* lo, int64_t ldp, float* colsum_partial,
                                 float mask_scale, float* out_f32, int64_t ld_f32, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(rows >= 0 && cols >= 4 && cols % 4 == 0 && cols <= 1024, "split_planes: cols=%d must be a multiple of 4 in [4, 1024]", cols);
  if (rows == 0) return RGCN_OK;                 // nothing is read or written (an empty tensor may have a null pointer)
  RGCN_CHECK_ARG(!out_f32 || (((uintptr_t)out_f32 & 15) == 0 && ld_f32 % 4 == 0), "split_planes: fp32 output misaligned");
  RGCN_CHECK_ARG(x && ((uintptr_t)x & 15) == 0 && ldx % 4 == 0, "split_planes: x must be 16-byte aligned, ld %% 4 == 0");
  RGCN_CHECK_ARG(!relu_mask || (((uintptr_t)relu_mask & 15) == 0 && ldm % 4 == 0), "split_planes: mask misaligned");
  RGCN_CHECK_ARG(hi && ((uintptr_t)hi & 7) == 0 && (!lo || ((uintptr_t)lo & 7) == 0) && ldp % 4 == 0,
                 "split_planes: planes must be 8-byte aligned, ld %% 4 == 0");
  RGCN_CHECK_ARG(!colsum_partial || ((uintptr_t)colsum_partial & 15) == 0, "split_planes: colsum_partial misaligned");
  const int64_t nb = rgcn_split_planes_blocks(rows, cols);
  const int rpp = 256 / (cols / 4) > 0 ? 256 / (cols / 4) : 1;
  const int64_t rows_per_block = ((rows + nb - 1) / nb + rpp - 1) / rpp * rpp;
  RGCN_CUDA(launch_pdl(split_planes_kernel, dim3((unsigned)nb), dim3(256), 0, (cudaStream_t)stream, x, ldx, relu_mask, ldm, rows, cols,
                                                                     (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ldp,
                                                                     colsum_partial, rows_per_block, mask_scale,
                                                                     out_f32, ld_f32));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" size_t rgcn_transform_workspace_bytes(int64_t n_rows, int32_t K, int32_t d_out) {
  if (n_rows < 0 || K <= 0 || d_out <= 0) return 0;
  // forward: weights^T [n_pad(d_out), k_pad(K)];  dgrad: weights [n_pad(K), k_pad(d_out)];  2 bf16 planes each
  const size_t fwd = (size_t)tile_n(d_out, 32, KBN).n_pad * round_up(K, BK) * 2 * 2;
  const size_t dgr = (size_t)tile_n(K, 32, KBN).n_pad * round_up(d_out, BK) * 2 * 2;
  const Tiling t = tile_n(d_out, 64);
  const int m_tiles = (K + BM - 1) / BM;
  const int splits = wgrad_splits(n_rows, m_tiles * t.n_tiles);
  const size_t wg = (size_t)splits * m_tiles * BM * t.n_pad * 4;
  size_t need = fwd > dgr ? fwd : dgr;
  if (wg > need) need = wg;
  return align_up(need, 256) + 1024;
}

extern "C" int rgcn_transform_fwd(const void* A_hi, const void* A_lo, int64_t lda, int32_t K1, int32_t K2, const float* W1,
                                  const float* W2, const float* bias, int32_t relu, int64_t n_rows, int32_t d_out,
                                  float* out, int64_t ldo, int32_t mode, float dropout_p, uint32_t dropout_seed,
                                  unsigned long long* dropout_counter, float* const* peer_out_host, int32_t n_peer,
                                  int64_t peer_row0, int64_t peer_ld, void* workspace, size_t workspace_bytes,
                                  rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n_peer >= 0 && n_peer <= kMaxPeers && (n_peer == 0 || (peer_out_host && peer_ld % 4 == 0 && peer_row0 >= 0)),
                 "transform_fwd: bad peer outputs (at most %d, ld %% 4 == 0)", kMaxPeers);
  RGCN_CHECK_ARG(n_rows >= 0 && K1 > 0 && K2 >= 0 && d_out > 0, "transform_fwd: bad sizes");
  RGCN_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, "transform_fwd: dropout_p must be in [0, 1)");
  RGCN_CHECK_ARG(dropout_p == 0.f || (dropout_counter && relu), "transform_fwd: fused dropout needs relu = 1 and a counter");
  RGCN_CHECK_ARG(K1 % 4 == 0 && K2 % 4 == 0 && d_out % 4 == 0, "transform_fwd: K1, K2, d_out must be multiples of 4");
  RGCN_CHECK_ARG(mode == 0 || mode == 1, "transform_fwd: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(n_rows < (1ll << 31), "transform_fwd: too many rows for one call");
  int rc = check_plane(A_hi, lda, "A_hi"); if (rc) return rc;
  if (mode == 0) { rc = check_plane(A_lo, lda, "A_lo"); if (rc) return rc; }
  RGCN_CHECK_ARG(out && ((uintptr_t)out & 15) == 0 && ldo % 4 == 0, "transform_fwd: out must be 16-byte aligned, ld %% 4 == 0");
  RGCN_CHECK_ARG(W1 && (K2 == 0 || W2) && (!bias || ((uintptr_t)bias & 3) == 0), "transform_fwd: null weights");
  if (n_rows == 0) return RGCN_OK;
  const int K = K1 + K2, k_pad = round_up(K, BK);
  const Tiling t = tile_n(d_out, 32, KBN);
  RGCN_CHECK_ARG(!bias || d_out <= 1024, "transform_fwd: bias needs d_out <= 1024");
  const size_t plane = (size_t)t.n_pad * k_pad * 2;
  if (!workspace || workspace_bytes < align_up(2 * plane, 256) + 1024) {
    set_error("transform_fwd: workspace too small"); return RGCN_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)align_up((size_t)workspace, 1024);
  __nv_bfloat16* bhi = (__nv_bfloat16*)ws;
  __nv_bfloat16* blo = (__nv_bfloat16*)(ws + plane);
  const bool split = mode == 0;
  {
    const int64_t total = (int64_t)t.n_pad * k_pad;
    RGCN_CUDA(launch_pdl(split_weights_kernel, dim3(grid_cap((total + 255) / 256, 1184)), dim3(256), 0, st, W1, K1, W2, K2, d_out, 1, bhi,
                                                                              split ? blo : nullptr, t.n_pad, k_pad,
                                                                              dropout_p > 0.f ? dropout_counter : nullptr));
    RGCN_LAUNCH_CHECK();
  }
  GemmKParams p{};
  p.M = n_rows; p.N = d_out; p.BN = t.BN; p.num_kb = k_pad / BK;
  p.bias = bias; p.relu = relu; p.out = out; p.ldo = ldo;
  if (dropout_p > 0.f) {
    const double th = (double)dropout_p * 65536.0 + 0.5;
    p.drop_thresh = th >= 65535.0 ? 65535u : (th < 1.0 ? 1u : (uint32_t)th);
    p.drop_scale = 1.f / (1.f - dropout_p);
    p.drop_seed = dropout_seed; p.drop_ctr = dropout_counter;
  }
  p.n_peer = n_peer; p.peer_row0 = peer_row0; p.peer_ld = peer_ld;
  for (int q = 0; q < n_peer; ++q) {
    RGCN_CHECK_ARG(peer_out_host[q] && ((uintptr_t)peer_out_host[q] & 15) == 0, "transform_fwd: peer output %d is null or misaligned", q);
    p.peer_out[q] = peer_out_host[q];
  }
  return launch_kmajor(p, A_hi, A_lo, lda, K, bhi, blo, t.n_pad, k_pad, k_pad, false, t.n_tiles, split, st);
}

extern "C" int rgcn_transform_dgrad(const void* G_hi, const void* G_lo, int64_t ldg, int32_t d_out, const float* W1,
                                    int32_t K1, const float* W2, int32_t K2, int64_t n_rows, float* gA, int64_t ldga,
                                    int32_t mode, void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n_rows >= 0 && K1 > 0 && K2 >= 0 && d_out > 0, "transform_dgrad: bad sizes");
  RGCN_CHECK_ARG(K1 % 4 == 0 && K2 % 4 == 0 && d_out % 4 == 0, "transform_dgrad: K1, K2, d_out must be multiples of 4");
  RGCN_CHECK_ARG(mode == 0 || mode == 1, "transform_dgrad: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(n_rows < (1ll << 31), "transform_dgrad: too many rows for one call");
  int rc = check_plane(G_hi, ldg, "G_hi"); if (rc) return rc;
  if (mode == 0) { rc = check_plane(G_lo, ldg, "G_lo"); if (rc) return rc; }
  RGCN_CHECK_ARG(gA && ((uintptr_t)gA & 15) == 0 && ldga % 4 == 0, "transform_dgrad: gA must be 16-byte aligned, ld %% 4 == 0");
  RGCN_CHECK_ARG(W1 && (K2 == 0 || W2), "transform_dgrad: null weights");
  if (n_rows == 0) return RGCN_OK;
  const int K = K1 + K2;                      // = N of this GEMM
  const int k_pad = round_up(d_out, BK);      // = K of this GEMM
  const Tiling t = tile_n(K, 32, KBN);
  const size_t plane = (size_t)t.n_pad * k_pad * 2;
  if (!workspace || workspace_bytes < align_up(2 * plane, 256) + 1024) {
    set_error("transform_dgrad: workspace too small"); return RGCN_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)align_up((size_t)workspace, 1024);
  __nv_bfloat16* bhi = (__nv_bfloat16*)ws;
  __nv_bfloat16* blo = (__nv_bfloat16*)(ws + plane);
  const bool split = mode == 0;
  {
    const int64_t total = (int64_t)t.n_pad * k_pad;
    RGCN_CUDA(launch_pdl(split_weights_kernel, dim3(grid_cap((total + 255) / 256, 1184)), dim3(256), 0, st, W1, K1, W2, K2, d_out, 0, bhi,
                                                                              split ? blo : nullptr, t.n_pad, k_pad, nullptr));
    RGCN_LAUNCH_CHECK();
  }
  GemmKParams p{};
  p.M = n_rows; p.N = K; p.BN = t.BN; p.num_kb = k_pad / BK;
  p.bias = nullptr; p.relu = 0; p.out = gA; p.ldo = ldga;
  return launch_kmajor(p, G_hi, G_lo, ldg, d_out, bhi, blo, t.n_pad, k_pad, k_pad, false, t.n_tiles, split, st);
}

extern "C" int rgcn_transform_wgrad(const void* A_hi, const void* A_lo, int64_t lda, int32_t K1, int32_t K2,
                                    const void* G_hi, const void* G_lo, int64_t ldg, int32_t d_out, int64_t n_rows,
                                    const float* colsum_partial, int32_t n_colsum, float* gW1, float* gW2, float* gbias,
                                    int32_t mode, void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n_rows >= 0 && K1 > 0 && K2 >= 0 && d_out > 0, "transform_wgrad: bad sizes");
  RGCN_CHECK_ARG(K1 % 4 == 0 && K2 % 4 == 0 && d_out % 4 == 0, "transform_wgrad: K1, K2, d_out must be multiples of 4");
  RGCN_CHECK_ARG(mode == 0 || mode == 1, "transform_wgrad: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(n_rows < (1ll << 31), "transform_wgrad: too many rows for one call");
  int rc;
  if (n_rows > 0) {                           // no rows: the planes are not read (the outputs are zero)
    rc = check_plane(A_hi, lda, "A_hi"); if (rc) return rc;
    rc = check_plane(G_hi, ldg, "G_hi"); if (rc) return rc;
    if (mode == 0) {
      rc = check_plane(A_lo, lda, "A_lo"); if (rc) return rc;
      rc = check_plane(G_lo, ldg, "G_lo"); if (rc) return rc;
    }
  }
  RGCN_CHECK_ARG(gW1 && (K2 == 0 || gW2), "transform_wgrad: null outputs");
  RGCN_CHECK_ARG(!gbias || (colsum_partial && n_colsum >= 0), "transform_wgrad: g_bias needs the column-sum partials");
  const int K = K1 + K2;
  const Tiling t = tile_n(d_out, 64);
  const int m_tiles = (K + BM - 1) / BM;
  const int splits = wgrad_splits(n_rows, m_tiles * t.n_tiles);
  const size_t part = (size_t)splits * m_tiles * BM * t.n_pad * 4;
  if (!workspace || workspace_bytes < align_up(part, 256) + 1024) {
    set_error("transform_wgrad: workspace too small"); return RGCN_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)align_up((size_t)workspace, 1024);
  WgradParams p{};
  p.nodes = n_rows; p.BN = t.BN;
  p.nodes_per_split = ((n_rows + splits - 1) / splits + WG_BK - 1) / WG_BK * WG_BK;
  if (p.nodes_per_split == 0) p.nodes_per_split = WG_BK;
  p.partial = (float*)ws; p.ldp = t.n_pad;
  if (n_rows > 0) {
    const bool split = mode == 0;
    CUtensorMap ahi, alo, ghi, glo;
    rc = make_map(&ahi, A_hi, n_rows, K, lda, WG_BK); if (rc) return rc;
    rc = make_map(&alo, split ? A_lo : A_hi, n_rows, K, lda, WG_BK); if (rc) return rc;
    rc = make_map(&ghi, G_hi, n_rows, d_out, ldg, WG_BK); if (rc) return rc;
    rc = make_map(&glo, split ? G_lo : G_hi, n_rows, d_out, ldg, WG_BK); if (rc) return rc;
    dim3 grid((unsigned)m_tiles, (unsigned)t.n_tiles, (unsigned)splits);
    if (split) {
      const int smem = WStage<true>::STAGES * WStage<true>::BYTES + 1024;
      rc = set_smem(gemm_wgrad_kernel<true>, smem); if (rc) return rc;
      RGCN_CUDA(launch_pdl(gemm_wgrad_kernel<true>, dim3(grid), dim3(192), smem, st, ahi, alo, ghi, glo, p));
    } else {
      const int smem = WStage<false>::STAGES * WStage<false>::BYTES + 1024;
      rc = set_smem(gemm_wgrad_kernel<false>, smem); if (rc) return rc;
      RGCN_CUDA(launch_pdl(gemm_wgrad_kernel<false>, dim3(grid), dim3(192), smem, st, ahi, alo, ghi, glo, p));
    }
    RGCN_LAUNCH_CHECK();
  }
  const int64_t total = (int64_t)K * (d_out / 4);
  const unsigned main_blocks = grid_cap((total + 63) / 64, 4736);
  RGCN_CUDA(launch_pdl(wgrad_reduce_kernel, dim3(main_blocks + (gbias ? (unsigned)(d_out / 4) : 0u)), dim3(256), 0, st, 
      p.partial, n_rows > 0 ? splits : 0, m_tiles * BM, t.n_pad, K1, K2, d_out, gW1, gW2, (int)main_blocks,
      colsum_partial, n_colsum, gbias));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

// ------------------------------------------------------------------------------------------------
// Weights converted ONCE per layer call: bf16 hi (, lo) planes of the row-major [K1 + K2, d_out] weight block exactly as
// PyTorch stores it.  The forward reads them as the MN-major B operand (no transposed copy), the dgrad as the K-major one;
// row-chunked calls of one layer share them.
// ------------------------------------------------------------------------------------------------
namespace rgcn {
}  // namespace rgcn

extern "C" size_t rgcn_weight_planes_bytes(int32_t K, int32_t d_out) {
  if (K <= 0 || d_out <= 0) return 0;
  return 2 * wplane_bytes(K, d_out) + 1024;
}

extern "C" int rgcn_prepare_weights(const float* W1, int32_t K1, const float* W2, int32_t K2, int32_t d_out, int32_t mode,
                                    void* w_planes, unsigned long long* dropout_counter, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(W1 && K1 > 0 && K2 >= 0 && (K2 == 0 || W2) && d_out > 0 && d_out % 4 == 0, "prepare_weights: bad sizes");
  RGCN_CHECK_ARG(mode == 0 || mode == 1, "prepare_weights: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(w_planes && ((uintptr_t)w_planes & 255) == 0, "prepare_weights: w_planes must be 256-byte aligned");
  const int K = K1 + K2;
  const int ld = (int)wplane_ld(d_out);
  __nv_bfloat16* hi = (__nv_bfloat16*)w_planes;
  __nv_bfloat16* lo = (__nv_bfloat16*)((char*)w_planes + wplane_bytes(K, d_out));
  const int64_t total = (int64_t)K * ld;
  RGCN_CUDA(launch_pdl(split_weights_kernel, dim3(grid_cap((total + 255) / 256, 1184)), dim3(256), 0, (cudaStream_t)stream,
                       W1, K1, W2, K2, d_out, 0, hi, mode == 0 ? lo : (__nv_bfloat16*)nullptr, K, ld, dropout_counter));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

static int transform_fwd_w_impl(const void* A_hi, const void* A_lo, int64_t lda, int32_t K, const void* w_planes,
                                const float* bias, int32_t relu, int64_t n_rows, int32_t d_out, float* out, int64_t ldo,
                                int32_t mode, float dropout_p, uint32_t dropout_seed,
                                const unsigned long long* dropout_counter, int64_t row_offset,
                                float* const* peer_out_host, int32_t n_peer, int64_t peer_row0, int64_t peer_ld,
                                void* out_bf16, int64_t ld_out_bf16, const int64_t* out_rows, int64_t n_out_rows,
                                const int32_t* out_slot, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(!out_rows || (n_out_rows >= 0 && n_out_rows <= n_rows && dropout_p == 0.f),
                 "transform_fwd_w: scattered output rows exclude the fused dropout");
  RGCN_CHECK_ARG(n_peer >= 0 && n_peer <= kMaxPeers && (n_peer == 0 || (peer_out_host && peer_ld % 4 == 0 && peer_row0 >= 0)),
                 "transform_fwd_w: bad peer outputs (at most %d, ld %% 4 == 0)", kMaxPeers);
  RGCN_CHECK_ARG(!out_bf16 || (((uintptr_t)out_bf16 & 7) == 0 && ld_out_bf16 % 4 == 0), "transform_fwd_w: bf16 output misaligned");
  RGCN_CHECK_ARG(n_rows >= 0 && n_rows < (1ll << 31) && K > 0 && K % 4 == 0 && d_out > 0 && d_out % 4 == 0, "transform_fwd_w: bad sizes");
  RGCN_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f && (dropout_p == 0.f || (dropout_counter && relu)),
                 "transform_fwd_w: dropout_p in [0, 1), fused dropout needs relu = 1 and a counter");
  RGCN_CHECK_ARG(mode == 0 || mode == 1, "transform_fwd_w: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(w_planes && ((uintptr_t)w_planes & 255) == 0, "transform_fwd_w: w_planes must come from rgcn_prepare_weights");
  int rc = check_plane(A_hi, lda, "A_hi"); if (rc) return rc;
  if (mode == 0) { rc = check_plane(A_lo, lda, "A_lo"); if (rc) return rc; }
  RGCN_CHECK_ARG(out && ((uintptr_t)out & 15) == 0 && ldo % 4 == 0, "transform_fwd_w: out must be 16-byte aligned, ld %% 4 == 0");
  RGCN_CHECK_ARG(!bias || d_out <= 1024, "transform_fwd_w: bias needs d_out <= 1024");
  if (n_rows == 0) return RGCN_OK;
  // measured (scripts/ab_gemm.py, 30,926 x 1,024 x 256): 256-wide tiles win with one product per k-step (4-stage ring:
  // 34.3 against 36.9 us) and lose with three (2-stage ring: 63.5 against 57.4 us)
  static int wide_fp32 = -1;                       // A/B switch: 256-wide tiles in the three-product mode too
  if (wide_fp32 < 0) { const char* e = getenv("RGCN_WIDE_FP32"); wide_fp32 = e ? atoi(e) : 0; }
  const bool wide = d_out > KBN && (mode == 1 || (wide_fp32 == 1) || (wide_fp32 == 2 && K <= 256));
  Tiling t = tile_n(d_out, 32, wide ? wide_bn() : KBN);
  // few rows (the listed-rows transform: 4,096 x 1,024 -> 256 is 64 tiles of 128 x 128): 64-wide tiles fill the machine
  static int narrow_small = -1;
  if (narrow_small < 0) { const char* e = getenv("RGCN_NARROW_SMALL"); narrow_small = (e && e[0] == '0') ? 0 : 1; }
  if (narrow_small && d_out % 64 == 0 && d_out >= 128 && ((n_rows + BM - 1) / BM) * t.n_tiles * 2 <= sm_count()) t = tile_n(d_out, 32, 64);
  const __nv_bfloat16* bhi = (const __nv_bfloat16*)w_planes;
  const __nv_bfloat16* blo = (const __nv_bfloat16*)((const char*)w_planes + wplane_bytes(K, d_out));
  GemmKParams p{};
  p.M = n_rows; p.N = d_out; p.BN = t.BN; p.num_kb = round_up(K, BK) / BK;
  p.bias = bias; p.relu = relu; p.out = out; p.ldo = ldo; p.row_offset = row_offset;
  p.out16 = (__nv_bfloat16*)out_bf16; p.ldo16 = ld_out_bf16;
  p.out_rows = out_rows; p.n_out_rows = n_out_rows; p.out_slot = out_slot;
  if (dropout_p > 0.f) {
    const double th = (double)dropout_p * 65536.0 + 0.5;
    p.drop_thresh = th >= 65535.0 ? 65535u : (th < 1.0 ? 1u : (uint32_t)th);
    p.drop_scale = 1.f / (1.f - dropout_p);
    p.drop_seed = dropout_seed; p.drop_ctr = dropout_counter;
  }
  p.n_peer = n_peer; p.peer_row0 = peer_row0; p.peer_ld = peer_ld;
  for (int q = 0; q < n_peer; ++q) {
    RGCN_CHECK_ARG(peer_out_host[q] && ((uintptr_t)peer_out_host[q] & 15) == 0, "transform_fwd_w: peer output %d is null or misaligned", q);
    p.peer_out[q] = peer_out_host[q];
  }
  return launch_kmajor(p, A_hi, A_lo, lda, K, bhi, blo, K, d_out, wplane_ld(d_out), true, t.n_tiles, mode == 0, (cudaStream_t)stream);
}

extern "C" int rgcn_transform_fwd_w(const void* A_hi, const void* A_lo, int64_t lda, int32_t K, const void* w_planes,
                                    const float* bias, int32_t relu, int64_t n_rows, int32_t d_out, float* out, int64_t ldo,
                                    int32_t mode, float dropout_p, uint32_t dropout_seed,
                                    const unsigned long long* dropout_counter, int64_t row_offset,
                                    float* const* peer_out_host, int32_t n_peer, int64_t peer_row0, int64_t peer_ld,
                                    void* out_bf16, int64_t ld_out_bf16, rgcn_stream_t stream) {
  return transform_fwd_w_impl(A_hi, A_lo, lda, K, w_planes, bias, relu, n_rows, d_out, out, ldo, mode, dropout_p, dropout_seed,
                              dropout_counter, row_offset, peer_out_host, n_peer, peer_row0, peer_ld, out_bf16, ld_out_bf16,
                              nullptr, 0, nullptr, stream);
}

// The same product over a COMPACT operand [n_rows, K] whose row c belongs to node out_rows[c] (c < n_list; the rows
// beyond are padding): the epilogue stores row c at out[out_rows[c], :] — only the listed rows of `out` are written.
// slot (nullable): node -> first list position; a later duplicate position is not stored (its operand row may be zero).
// peer_out_host (n_peer > 0): the listed rows also go to rows peer_row0 + out_rows[c] of the peers' buffers (the
// partitioned path's all-gather of the rows the decoders read).
extern "C" int rgcn_transform_fwd_w_rows(const void* A_hi, const void* A_lo, int64_t lda, int32_t K, const void* w_planes,
                                         const float* bias, int32_t relu, int64_t n_rows, int32_t d_out, float* out, int64_t ldo,
                                         int32_t mode, const int64_t* out_rows, int64_t n_list, const int32_t* slot,
                                         float* const* peer_out_host, int32_t n_peer, int64_t peer_row0, int64_t peer_ld,
                                         rgcn_stream_t stream) {
  RGCN_CHECK_ARG(out_rows && n_list >= 0 && n_list <= n_rows, "transform_fwd_w_rows: bad row list");
  return transform_fwd_w_impl(A_hi, A_lo, lda, K, w_planes, bias, relu, n_rows, d_out, out, ldo, mode, 0.f, 0u, nullptr, 0,
                              peer_out_host, n_peer, peer_row0, peer_ld, nullptr, 0, out_rows, n_list, slot, stream);
}

extern "C" int rgcn_transform_dgrad_w(const void* G_hi, const void* G_lo, int64_t ldg, int32_t d_out, const void* w_planes,
                                      int32_t K, int64_t n_rows, float* gA, int64_t ldga, int32_t mode, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n_rows >= 0 && n_rows < (1ll << 31) && K > 0 && K % 4 == 0 && d_out > 0 && d_out % 4 == 0, "transform_dgrad_w: bad sizes");
  RGCN_CHECK_ARG(mode == 0 || mode == 1, "transform_dgrad_w: mode must be 0 (fp32) or 1 (bf16)");
  RGCN_CHECK_ARG(w_planes && ((uintptr_t)w_planes & 255) == 0, "transform_dgrad_w: w_planes must come from rgcn_prepare_weights");
  int rc = check_plane(G_hi, ldg, "G_hi"); if (rc) return rc;
  if (mode == 0) { rc = check_plane(G_lo, ldg, "G_lo"); if (rc) return rc; }
  RGCN_CHECK_ARG(gA && ((uintptr_t)gA & 15) == 0 && ldga % 4 == 0, "transform_dgrad_w: gA must be 16-byte aligned, ld %% 4 == 0");
  if (n_rows == 0) return RGCN_OK;
  const Tiling t = tile_n(K, 32, K > KBN ? wide_bn() : KBN);
  const __nv_bfloat16* bhi = (const __nv_bfloat16*)w_planes;
  const __nv_bfloat16* blo = (const __nv_bfloat16*)((const char*)w_planes + wplane_bytes(K, d_out));
  GemmKParams p{};
  p.M = n_rows; p.N = K; p.BN = t.BN; p.num_kb = round_up(d_out, BK) / BK;
  p.out = gA; p.ldo = ldga;
  return launch_kmajor(p, G_hi, G_lo, ldg, d_out, bhi, blo, K, d_out, wplane_ld(d_out), false, t.n_tiles, mode == 0, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// All-pairs scoring WITHOUT the score matrix: the tcgen05 kernel's epilogue consumes the accumulator.
//   queries   : bf16 hi / lo planes [n_q, d] (rgcn_split_planes of the prepared rows, csrc/rank.cu rows_prepare)
//   candidates: rgcn_prepare_weights planes of the fp32 candidate rows [n_cand, d] (K-major operand)
//   rgcn_scores_diag_w : thr[i] = <q_i, c_i>  — the diagonal tiles of Q x C'^T with C' = the true tails gathered per query;
//                        same K order and products as the full sweep, so thr[i] carries the bits the sweep computes for
//                        (i, true_pos[i]) and exact ties with other candidates are counted as ties
//   rgcn_scores_rank_w : greater[i] / equal[i] += #{j != true_pos[i] : s_ij > / == thr[i]}   (zero them first)
//   rgcn_scores_topk_w : per query the k <= 16 best candidates (alpha * s + beta, index), sorted by value then index;
//                        every epilogue lane keeps a 16-entry list per row across its run of column tiles and stores it
//                        in one of the row's n_slots partial lists (rgcn_scores_topk_slots: one per CTA run and column
//                        half that touches the row, uncapped); a second small kernel merges them 256 candidates at a time
// Replaces score_all_tails + the per-row argsort of src/evaluate.py:260-276 and the cosine sweeps + top-k / threshold
// filters of src/compare_methods.py:384-397, src/medical_validation.py:222-239, src/case_studies.py:260-274.
// ------------------------------------------------------------------------------------------------
namespace rgcn {
__global__ void __launch_bounds__(256) topk_merge_kernel(const float* __restrict__ cand_val, const int32_t* __restrict__ cand_idx,
                                                         const int32_t* __restrict__ slot_ctr, int n_slots, int64_t n_q, int k,
                                                         float alpha, float beta, float* __restrict__ out_val,
                                                         int64_t* __restrict__ out_idx) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_q) return;
  int used = slot_ctr[row];
  if (used > n_slots) used = n_slots;
  const int total = used * kTopK;
  const float* cv = cand_val + (size_t)row * n_slots * kTopK;
  const int32_t* ci = cand_idx + (size_t)row * n_slots * kTopK;
  constexpr int PER = 8;                              // candidates per lane and pass: the partial lists in chunks of 256
  // running top-k of the chunks merged so far: lane j < k holds entry j (value descending, then index ascending)
  float lv = -INFINITY;
  int li = -1;
  for (int base = 0; base < total; base += PER * 32) {
    float v[PER];
    int id[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int e = base + u * 32 + lane;
      const bool ok = e < total;
      v[u] = ok ? cv[e] : -INFINITY;
      id[u] = ok ? ci[e] : -1;
      if (id[u] < 0) v[u] = -INFINITY;
    }
    float nv = -INFINITY;
    int ni = -1;
    for (int j = 0; j < k; ++j) {
      // warp arg-max over the chunk and the running list by (value desc, index asc)
      float bv = -INFINITY;
      int bi = 0x7fffffff;
      if (li >= 0 && (lv > bv || (lv == bv && li < bi))) { bv = lv; bi = li; }
#pragma unroll
      for (int u = 0; u < PER; ++u)
        if (id[u] >= 0 && (v[u] > bv || (v[u] == bv && id[u] < bi))) { bv = v[u]; bi = id[u]; }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
      }
      if (bi == 0x7fffffff) break;                    // (warp-uniform) nothing left
      // an index occurs once: the partial lists cover disjoint column ranges
      if (li == bi) { li = -1; lv = -INFINITY; }
#pragma unroll
      for (int u = 0; u < PER; ++u)
        if (id[u] == bi) { id[u] = -1; v[u] = -INFINITY; }
      if (lane == j) { nv = bv; ni = bi; }
    }
    lv = nv;
    li = ni;
  }
  if (lane < k) {
    out_val[row * k + lane] = li >= 0 ? alpha * lv + beta : -INFINITY;
    out_idx[row * k + lane] = li >= 0 ? (int64_t)li : -1;
  }
}
}  // namespace rgcn

static int scores_common(GemmKParams& p, const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                         int64_t n_q, const char* what) {
  RGCN_CHECK_ARG(n_q >= 0 && n_q < (1ll << 31) && d > 0 && d % 4 == 0, "%s: bad sizes", what);
  RGCN_CHECK_ARG(cand_planes && ((uintptr_t)cand_planes & 255) == 0, "%s: candidate planes must come from rgcn_prepare_weights", what);
  int rc = check_plane(Q_hi, ldq, "Q_hi"); if (rc) return rc;
  rc = check_plane(Q_lo, ldq, "Q_lo"); if (rc) return rc;
  p.M = n_q; p.BN = KBN; p.num_kb = round_up(d, BK) / BK;
  return RGCN_OK;
}

extern "C" int rgcn_scores_diag_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* tail_planes,
                                  int64_t n_q, float* thr, rgcn_stream_t stream) {
  GemmKParams p{};
  int rc = scores_common(p, Q_hi, Q_lo, ldq, d, tail_planes, n_q, "scores_diag_w");
  if (rc) return rc;
  RGCN_CHECK_ARG(thr, "scores_diag_w: null output");
  if (n_q == 0) return RGCN_OK;
  p.N = (int)(n_q < KBN ? KBN : KBN); p.diag = 1; p.thr_out = thr;
  const __nv_bfloat16* bhi = (const __nv_bfloat16*)tail_planes;
  const __nv_bfloat16* blo = (const __nv_bfloat16*)((const char*)tail_planes + wplane_bytes((int)n_q, d));
  return launch_kmajor(p, Q_hi, Q_lo, ldq, d, bhi, blo, n_q, d, wplane_ld(d), false, 1, true, (cudaStream_t)stream, EPI_THR);
}

// the exclusion lists come as a triple: all null (no filter) or none
static int check_excl(const int64_t* excl_begin, const int64_t* excl_end, const int32_t* excl_pos, const char* what) {
  const int n_null = (excl_begin == nullptr) + (excl_end == nullptr) + (excl_pos == nullptr);
  RGCN_CHECK_ARG(n_null == 0 || n_null == 3, "%s: excl_begin, excl_end and excl_pos are all null or none is", what);
  return RGCN_OK;
}

extern "C" int rgcn_scores_rank_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                                  int64_t n_cand, int64_t n_q, const float* thr, const int64_t* true_pos, int32_t* greater,
                                  int32_t* equal, rgcn_stream_t stream) {
  return rgcn_scores_rank_excl_w(Q_hi, Q_lo, ldq, d, cand_planes, n_cand, n_q, thr, true_pos, greater, equal, nullptr,
                                 nullptr, nullptr, stream);
}

extern "C" int rgcn_scores_rank_excl_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                                       int64_t n_cand, int64_t n_q, const float* thr, const int64_t* true_pos,
                                       int32_t* greater, int32_t* equal, const int64_t* excl_begin, const int64_t* excl_end,
                                       const int32_t* excl_pos, rgcn_stream_t stream) {
  int rc = check_excl(excl_begin, excl_end, excl_pos, "scores_rank_excl_w");
  if (rc) return rc;
  GemmKParams p{};
  rc = scores_common(p, Q_hi, Q_lo, ldq, d, cand_planes, n_q, "scores_rank_w");
  if (rc) return rc;
  RGCN_CHECK_ARG(n_cand > 0 && n_cand < (1ll << 31) && thr && true_pos && greater && equal, "scores_rank_w: null argument");
  if (n_q == 0) return RGCN_OK;
  p.N = (int)n_cand; p.n_cols_valid = n_cand; p.tile_contig = 1;
  p.thr_in = thr; p.true_pos = true_pos; p.greater = greater; p.equal = equal;
  p.excl_begin = excl_begin; p.excl_end = excl_end; p.excl_pos = excl_pos;
  const int n_tiles = (int)((n_cand + KBN - 1) / KBN);
  const __nv_bfloat16* bhi = (const __nv_bfloat16*)cand_planes;
  const __nv_bfloat16* blo = (const __nv_bfloat16*)((const char*)cand_planes + wplane_bytes((int)n_cand, d));
  return launch_kmajor(p, Q_hi, Q_lo, ldq, d, bhi, blo, n_cand, d, wplane_ld(d), false, n_tiles, true, (cudaStream_t)stream, EPI_RANK);
}

extern "C" int32_t rgcn_scores_topk_slots(int64_t n_q, int64_t n_cand) {
  if (n_q <= 0 || n_cand <= 0) return 0;
  const int64_t n_tiles = (n_cand + KBN - 1) / KBN, m_tiles = (n_q + BM - 1) / BM;
  const int64_t tiles = n_tiles * m_tiles;
  const int64_t grid = tiles < sm_count() ? tiles : sm_count();
  const int64_t per = (tiles + grid - 1) / grid;
  // CTA runs touching one row tile x two column halves: at most 2 (#SMs + 1), whatever the shape
  return (int32_t)(2 * ((n_tiles + per - 1) / per + 1));
}

extern "C" int rgcn_scores_topk_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                                  int64_t n_cand, int64_t n_q, int32_t k, float alpha, float beta, float* cand_val,
                                  int32_t* cand_idx, int32_t* slot_ctr, int32_t n_slots, float* out_val, int64_t* out_idx,
                                  rgcn_stream_t stream) {
  return rgcn_scores_topk_excl_w(Q_hi, Q_lo, ldq, d, cand_planes, n_cand, n_q, k, alpha, beta, cand_val, cand_idx, slot_ctr,
                                 n_slots, out_val, out_idx, nullptr, nullptr, nullptr, stream);
}

extern "C" int rgcn_scores_topk_excl_w(const void* Q_hi, const void* Q_lo, int64_t ldq, int32_t d, const void* cand_planes,
                                       int64_t n_cand, int64_t n_q, int32_t k, float alpha, float beta, float* cand_val,
                                       int32_t* cand_idx, int32_t* slot_ctr, int32_t n_slots, float* out_val,
                                       int64_t* out_idx, const int64_t* excl_begin, const int64_t* excl_end,
                                       const int32_t* excl_pos, rgcn_stream_t stream) {
  int rc = check_excl(excl_begin, excl_end, excl_pos, "scores_topk_excl_w");
  if (rc) return rc;
  GemmKParams p{};
  rc = scores_common(p, Q_hi, Q_lo, ldq, d, cand_planes, n_q, "scores_topk_w");
  if (rc) return rc;
  RGCN_CHECK_ARG(n_cand > 0 && n_cand < (1ll << 31) && k >= 1 && k <= kTopK && alpha > 0.f, "scores_topk_w: 1 <= k <= %d, alpha > 0", kTopK);
  RGCN_CHECK_ARG(cand_val && cand_idx && slot_ctr && out_val && out_idx, "scores_topk_w: null argument");
  RGCN_CHECK_ARG(n_slots >= rgcn_scores_topk_slots(n_q, n_cand), "scores_topk_w: too few slots (rgcn_scores_topk_slots)");
  if (n_q == 0) return RGCN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  RGCN_CUDA(cudaMemsetAsync(slot_ctr, 0, (size_t)n_q * sizeof(int32_t), st));
  p.N = (int)n_cand; p.n_cols_valid = n_cand; p.tile_contig = 1;
  p.alpha = alpha; p.beta = beta; p.cand_val = cand_val; p.cand_idx = cand_idx; p.slot_ctr = slot_ctr; p.n_slots = n_slots;
  p.excl_begin = excl_begin; p.excl_end = excl_end; p.excl_pos = excl_pos;
  const int n_tiles = (int)((n_cand + KBN - 1) / KBN);
  const __nv_bfloat16* bhi = (const __nv_bfloat16*)cand_planes;
  const __nv_bfloat16* blo = (const __nv_bfloat16*)((const char*)cand_planes + wplane_bytes((int)n_cand, d));
  rc = launch_kmajor(p, Q_hi, Q_lo, ldq, d, bhi, blo, n_cand, d, wplane_ld(d), false, n_tiles, true, st, EPI_TOPK);
  if (rc) return rc;
  RGCN_CUDA(launch_pdl(topk_merge_kernel, dim3((unsigned)((n_q + 7) / 8)), dim3(256), 0, st, (const float*)cand_val,
                       (const int32_t*)cand_idx, (const int32_t*)slot_ctr, (int)n_slots, n_q, (int)k, alpha, beta, out_val, out_idx));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}
