// One RGCN layer forward in ONE kernel: the neighbourhood walk feeds the tensor cores through shared memory.
//
//   O[i, :] = relu?( sum_r mean_{j in N_r(i)} x[j] @ W_r  +  x[i] @ root  +  bias )          (reference call sites
//   src/models/rgcn.py:123, :128 — RGCNConv's loop path, aggregate-then-transform order)
//
// The unfused path (aggregate.cu -> transform.cu) writes the operand A = [H | X] as bf16 planes to memory and reads it
// back by TMA: 126 MB each way per layer-2 call at cfg2, 19.8 GB per layer and GPU at cfg5 — and the L2-bound walk and
// the tensor-pipe-bound GEMM run back to back.  Here a CTA owns a tile of 128 destination rows and never materialises A:
//
//   table warp         : per (tile, relation) the 128 segment bounds and their prefix sums, one block ahead
//   producer warps (25): the block's edges form ONE stream (segment after segment in slot order); every warp takes an
//                        equal share of it, whatever rows that cuts — a power-law graph has 100-edge segments next to
//                        empty ones, and the tensor core can only start a block when ALL its rows are there.  Sums run
//                        left to right in CSR order with a true division by the segment length; a row cut between
//                        warps is combined from its pieces in stream order; hub segments come from the chunk partials.
//                        Finished row slices go as bf16 hi / lo straight into the 128B-swizzled K-major operand layout
//                        of tcgen05.mma (fence.proxy.async, mbarrier arrive)
//   TMA warp           : streams the weight planes [K, d_out] (MN-major B operand) in 32-row stages
//   MMA warp           : tcgen05.mma.cta_group::1.kind::f16 (M = 128, N = d_out <= 256), hi*hi + hi*lo + lo*hi in the
//                        fp32 mode, accumulating in TMEM; tcgen05.commit frees the A block and the B stage
//   epilogue warps (4) : tcgen05.ld -> + bias -> ReLU -> counter-based dropout -> row stores (rows may be permuted:
//                        every lane owns one row); two TMEM accumulators, so tile i drains under the walk of tile i+1
//
// K order: the operand columns are visited in slices of CW = min(d_in, 128) feature columns — for d_in = 256 the
// sequence is r = 0..R, h = 0, 1 with block (r, h) = columns [r d_in + h CW, + CW) of [H | X] — so one
// A block is 128 rows x CW columns (64 KB as hi + lo at CW = 128) and two of them fit beside the B ring: the producers
// fill block b + 1 while the tensor core consumes block b.  Any K order gives the same sum up to fp32 accumulation order.
//
// Row tiles: on graphs with a global degree order (csr->row_order, L2-resident graphs) the sorted rows are DEALT to
// the tiles (rank k -> tile k mod T, T a multiple of the grid), so every tile carries the same number of edges, the
// heavy rows of a tile come first (slot order), and every CTA runs the same number of equal tiles — no wave
// quantisation.  Otherwise tiles are consecutive row ranges.
//
// The saved-for-backward planes are still written when the caller passes them (A_hi != NULL): the producers have the
// row slice in registers anyway.  What disappears is the read-back, the second kernel and the serialisation.
#include <stdlib.h>

#include "common.cuh"
#include "gemm_common.cuh"
#include "tc05.cuh"

namespace rgcn {
using namespace tc05;

constexpr int FL_BM = 128;                    // rows per tile = UMMA M
constexpr int FL_KB = 32;                     // k rows per B stage
constexpr int FL_NPW = 25;                    // producer warps
constexpr int FL_EPW = 4;                     // epilogue warps (warps 0..3: one per TMEM lane quarter)
constexpr int FL_THREADS = (FL_NPW + FL_EPW + 3) * 32;      // + TMA warp, MMA warp, segment-table warp
constexpr int FL_NMETA = 2;                   // segment tables in flight (one per (tile, relation))
constexpr int FL_ROWRING = 4;                 // tiles whose row ids are kept in shared memory
constexpr int FL_MAXPEERS = 8;
static_assert(FL_THREADS <= 1024, "one CTA per SM, at most 1024 threads");

struct FusedParams {
  // graph (destination, relation) CSR
  const int32_t* rowptr; const int32_t* idx;
  const int32_t* hub_keys; const int32_t* hub_chunk_ptr; const int32_t* row_order;
  int32_t hub_threshold, n_hubs, R;
  int64_t n_rows;
  const float* partials;                      // [n_chunks, d_in] chunk sums of the hub segments (hub_partial_kernel)
  // features
  const float* x_src; int64_t ld_src;
  const float* x_root; int64_t ld_root;
  int32_t d_in;
  // row tiles
  int32_t n_tiles, deal;
  // optional saved-for-backward planes [n_rows, lda]
  __nv_bfloat16* A_hi; __nv_bfloat16* A_lo; int64_t lda;
  // transform + epilogue
  int32_t N, BN;                              // d_out and the UMMA N (d_out rounded up to 16)
  const float* bias; int32_t relu;
  float* out; int64_t ldo;
  __nv_bfloat16* out16; int64_t ldo16;
  uint32_t drop_thresh; float drop_scale; uint32_t drop_seed; const unsigned long long* drop_ctr;
  int64_t drop_row0;                          // layer-output row of local row 0 (a shard's first node): dropout index
  float* peer_out[FL_MAXPEERS]; int32_t n_peer; int64_t peer_row0; int64_t peer_ld;
};

template <int CW, bool SPLIT>
struct FLCfg {
  static constexpr int UNITS = CW / 64;                       // 64-column swizzle units per plane of a block
  static constexpr int A_PLANE = UNITS * FL_BM * 128;          // 128 rows x CW bf16
  static constexpr int A_BLOCK = (SPLIT ? 2 : 1) * A_PLANE;
  static constexpr int NBUF = (131072 / A_BLOCK) > 4 ? 4 : (131072 / A_BLOCK);
  static constexpr int B_PLANE = 4 * FL_KB * 128;              // 4 chunks of 64 columns x 32 k rows
  static constexpr int B_STAGE = (SPLIT ? 2 : 1) * B_PLANE;
  static constexpr int NSB = SPLIT ? 2 : 4;
  static constexpr int G = CW / 4;                             // lanes per worker (16 B of fp32 per lane)
  static constexpr int NW = FL_NPW * (32 / G);                 // workers: lane groups that each take a share of the edges
  static constexpr int SCRATCH = 2 * NW * G * 16;              // one fp32 piece per worker, double buffered by block parity
  static constexpr int SMEM = NBUF * A_BLOCK + NSB * B_STAGE + SCRATCH + 1024;
};

// segment table of one (tile, relation): slot m of the tile owns stream positions [pre[m], pre[m + 1]) of the block's
// edge stream = CSR positions beg[m] ...; len = the segment's true length (hub segments and padding slots stream nothing)
struct FLMeta {
  int32_t pre[FL_BM + 4];
  int32_t beg[FL_BM];
  int32_t len[FL_BM];
};

__device__ __forceinline__ int64_t fl_tile_row(const FusedParams& p, int64_t t, int m) {
  const int64_t pos = p.deal ? (int64_t)m * p.n_tiles + t : t * FL_BM + m;
  if (pos >= p.n_rows) return -1;
  return p.deal ? (int64_t)__ldg(p.row_order + pos) : pos;
}


// One finished row slice of a block: mean, bf16 hi / lo, into the swizzled operand block (and the saved planes).
// Out of line on purpose: the stream loop below reaches it from every unrolled batch slot, and inlined copies of the
// IEEE divisions and conversions made the kernel larger than the instruction cache.
__device__ __noinline__ void fl_finish_row(float4 acc, int len, uint8_t* s_hi, uint32_t lo_plane_off,
                                           __nv_bfloat16* g_hi, __nv_bfloat16* g_lo) {
  if (len > 1) acc = div4(acc, (float)len);                // s / clamp(cnt, 1): a true division, like the reference
  uint2 vhi, vlo;
  split4(acc, vhi, vlo);
  *reinterpret_cast<uint2*>(s_hi) = vhi;
  if (lo_plane_off) *reinterpret_cast<uint2*>(s_hi + lo_plane_off) = vlo;
  if (g_hi) {
    *reinterpret_cast<uint2*>(g_hi) = vhi;
    if (g_lo) *reinterpret_cast<uint2*>(g_lo) = vlo;
  }
}

// Hub segments (longer than the hub threshold): hub_partial_kernel has reduced their 128-edge chunks into `partials`;
// this pass adds each segment's chunk partials IN CHUNK ORDER (the order aggregate_rows_kernel adds them, so the sums are
// the same bits) and leaves the segment's total in the slot of its first chunk.  One block per hub segment, one thread
// per 128-bit column, 16 independent loads in flight: a 12,000-edge hub (94 chunks) takes 6 dependent steps here; read
// chunk by chunk inside the fused kernel it was a 24-step chain in ONE producer warp that held up its whole CTA.
__global__ void __launch_bounds__(256) hub_reduce_kernel(float* __restrict__ partials, const int32_t* __restrict__ hub_chunk_ptr,
                                                         int d) {
  pdl_enter();
  const int h = blockIdx.x;
  const int c0 = __ldg(hub_chunk_ptr + h), c1 = __ldg(hub_chunk_ptr + h + 1);
  constexpr int UR = 16;
  for (int col = threadIdx.x * 4; col < d; col += blockDim.x * 4) {
    float* pp = partials + col;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int c = c0;
    for (; c + UR <= c1; c += UR) {
      float4 v[UR];
#pragma unroll
      for (int u = 0; u < UR; ++u) v[u] = *reinterpret_cast<const float4*>(pp + (size_t)(c + u) * d);
#pragma unroll
      for (int u = 0; u < UR; ++u) add4(acc, v[u]);
    }
    for (; c < c1; ++c) add4(acc, *reinterpret_cast<const float4*>(pp + (size_t)c * d));
    *reinterpret_cast<float4*>(pp + (size_t)c0 * d) = acc;
  }
}

// total of a hub segment (this lane's 4 columns): hub_reduce_kernel left it in the slot of the segment's first chunk
__device__ __noinline__ float4 fl_hub_sum(const FusedParams& p, int key, int col0) {
  int lo = 0, hi = p.n_hubs;
  while (hi - lo > 1) {                       // (hub_keys: a few KB, L1 resident)
    const int mid = (lo + hi) >> 1;
    if (__ldg(p.hub_keys + mid) <= key) lo = mid; else hi = mid;
  }
  const int c0 = __ldg(p.hub_chunk_ptr + lo);
  return *reinterpret_cast<const float4*>(p.partials + (size_t)c0 * p.d_in + col0);
}

template <int CW, bool SPLIT>
__global__ void __launch_bounds__(FL_THREADS, 1)
fused_layer_fwd_kernel(const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                       const __grid_constant__ FusedParams p) {
  using C = FLCfg<CW, SPLIT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + (size_t)C::NBUF * C::A_BLOCK;
  float4* scratch = reinterpret_cast<float4*>(smem_b + (size_t)C::NSB * C::B_STAGE);      // [2][NW][G]
  __shared__ uint64_t a_full[C::NBUF], a_empty[C::NBUF], b_full[C::NSB], b_empty[C::NSB], tfull[2], tempty[2];
  __shared__ uint64_t meta_full[FL_NMETA], meta_empty[FL_NMETA];
  __shared__ FLMeta meta[FL_NMETA];
  __shared__ int32_t tile_rows[FL_ROWRING][FL_BM];
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float s_bias[256];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = p.R;
  const int passes = p.d_in / CW;
  const int blocks_per_tile = passes * (R + 1);
  const uint32_t acc_cols = p.BN <= 32 ? 32 : p.BN <= 64 ? 64 : p.BN <= 128 ? 128 : 256;
  const uint32_t tmem_cols = 2 * acc_cols;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::NBUF; ++s) { mbar_init(&a_full[s], FL_NPW); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < C::NSB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], FL_EPW); }
    for (int s = 0; s < FL_NMETA; ++s) { mbar_init(&meta_full[s], 1); mbar_init(&meta_empty[s], FL_NPW); }
    fence_barrier_init();
  }
  if (warp == FL_EPW && lane == 0) {
    tma_prefetch_desc(&tm_b_hi);
    if (SPLIT) tma_prefetch_desc(&tm_b_lo);
  }
  if (warp == 0) tmem_alloc(&tmem_base_smem, tmem_cols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_launch_dependents();
  pdl_wait();
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_bias[i] = (p.bias && i < p.N) ? p.bias[i] : 0.f;
  __syncthreads();

  if (warp < FL_EPW) {
    // ===================== epilogue: lane l of warp w owns tile slot 32 w + l =====================
    uint32_t drop_key = 0;
    if (p.drop_thresh) {
      const unsigned long long ctr = *p.drop_ctr;
      drop_key = pcg_hash(p.drop_seed ^ (uint32_t)ctr) + (uint32_t)(ctr >> 32);
    }
    int iter = 0;
    for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++iter) {
      const int a = iter & 1;
      const int64_t row = fl_tile_row(p, t, warp * 32 + lane);
      mbar_wait_parked(&tfull[a], (uint32_t)((iter >> 1) & 1));
      fence_after_sync();
      const uint32_t t_lane = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)a * acc_cols;
      for (int cc = 0; cc < p.BN; cc += 16) {
        uint32_t r[16];
        tmem_ld_32x16(t_lane + cc, r);
        tmem_ld_wait();
        if (row >= 0) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const int col = cc + j;
          if (col >= p.N) break;
          const float4 b = *reinterpret_cast<const float4*>(s_bias + col);
          float4 v = make_float4(__uint_as_float(r[j]) + b.x, __uint_as_float(r[j + 1]) + b.y,
                                 __uint_as_float(r[j + 2]) + b.z, __uint_as_float(r[j + 3]) + b.w);
          if (p.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
          if (p.drop_thresh) {
            // the same hash of the GLOBAL element index as the unfused epilogue (transform.cu): identical masks
            const uint64_t e0 = (uint64_t)(row + p.drop_row0) * (uint64_t)p.N + (uint64_t)col;
            const uint32_t bk = drop_block_key(drop_key, e0), e32 = (uint32_t)e0;
            const uint32_t h0 = pcg_hash(e32 ^ bk), h1 = pcg_hash((e32 + 2) ^ bk);
            v.x = (h0 & 0xffffu) >= p.drop_thresh ? v.x * p.drop_scale : 0.f;
            v.y = (h0 >> 16) >= p.drop_thresh ? v.y * p.drop_scale : 0.f;
            v.z = (h1 & 0xffffu) >= p.drop_thresh ? v.z * p.drop_scale : 0.f;
            v.w = (h1 >> 16) >= p.drop_thresh ? v.w * p.drop_scale : 0.f;
          }
          *reinterpret_cast<float4*>(p.out + row * p.ldo + col) = v;
          if (p.out16) {
            __nv_bfloat162 b01 = __floats2bfloat162_rn(v.x, v.y), b23 = __floats2bfloat162_rn(v.z, v.w);
            uint2 o;
            o.x = *reinterpret_cast<uint32_t*>(&b01);
            o.y = *reinterpret_cast<uint32_t*>(&b23);
            *reinterpret_cast<uint2*>(p.out16 + row * p.ldo16 + col) = o;
          }
          for (int q = 0; q < p.n_peer; ++q)
            *reinterpret_cast<float4*>(p.peer_out[q] + (p.peer_row0 + row) * p.peer_ld + col) = v;
        }
        }
        __syncwarp();                          // tcgen05.ld is warp-collective: reconverge before the next one
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[a]);
    }
  } else if (warp == FL_EPW) {
    // ===================== TMA: weight planes, 32 k rows per stage =====================
    if (lane == 0) {
      const int b_chunks = (p.BN + 63) / 64;
      const uint32_t bytes = (uint32_t)b_chunks * (uint32_t)(FL_KB * 128) * (SPLIT ? 2u : 1u);
      uint32_t it = 0;
      for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        for (int r = 0; r <= R; ++r) {
          for (int h = 0; h < passes; ++h) {
            for (int kk = 0; kk < CW / FL_KB; ++kk, ++it) {
              const int s = it % C::NSB;
              mbar_wait_parked(&b_empty[s], ((it / C::NSB) & 1) ^ 1);
              uint8_t* st = smem_b + (size_t)s * C::B_STAGE;
              const int k0 = r * p.d_in + h * CW + kk * FL_KB;
              mbar_arrive_expect_tx(&b_full[s], bytes);
              for (int ch = 0; ch < b_chunks; ++ch) {
                tma_load_2d(st + ch * (FL_KB * 128), &tm_b_hi, &b_full[s], ch * 64, k0);
                if (SPLIT) tma_load_2d(st + C::B_PLANE + ch * (FL_KB * 128), &tm_b_lo, &b_full[s], ch * 64, k0);
              }
            }
          }
        }
      }
    }
  } else if (warp == FL_EPW + 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = idesc_bf16(FL_BM, p.BN, 0, 1);
      uint32_t blk = 0, sb_it = 0;
      int iter = 0;
      for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++iter) {
        const int a = iter & 1;
        mbar_wait_parked(&tempty[a], (uint32_t)(((iter >> 1) & 1) ^ 1));
        fence_after_sync();
        const uint32_t tacc = tmem_base + (uint32_t)a * acc_cols;
        for (int b = 0; b < blocks_per_tile; ++b, ++blk) {
          const int buf = blk % C::NBUF;
          mbar_wait_parked(&a_full[buf], (blk / C::NBUF) & 1);
          fence_after_sync();
          const uint32_t abase = smem_u32(smem_a + (size_t)buf * C::A_BLOCK);
          uint32_t bbase = 0;
          int s = 0;
#pragma unroll
          for (int ks = 0; ks < CW / 16; ++ks) {
            if ((ks & 1) == 0) {
              s = sb_it % C::NSB;
              mbar_wait(&b_full[s], (sb_it / C::NSB) & 1);
              fence_after_sync();
              bbase = smem_u32(smem_b + (size_t)s * C::B_STAGE);
            }
            const uint64_t adv_a = (uint64_t)(((ks & 3) * 32) >> 4);
            const uint64_t da_hi = smem_desc_sw128(abase + (ks >> 2) * (FL_BM * 128), 16, 1024) + adv_a;
            const uint64_t da_lo = smem_desc_sw128(abase + C::A_PLANE + (ks >> 2) * (FL_BM * 128), 16, 1024) + adv_a;
            const uint64_t adv_b = (uint64_t)(((ks & 1) * 2048) >> 4);
            const uint64_t db_hi = smem_desc_sw128(bbase, FL_KB * 128, 1024) + adv_b;
            const uint64_t db_lo = smem_desc_sw128(bbase + C::B_PLANE, FL_KB * 128, 1024) + adv_b;
            mma_bf16_ss(tacc, da_hi, db_hi, idesc, (b | ks) ? 1u : 0u);
            if (SPLIT) {
              mma_bf16_ss(tacc, da_hi, db_lo, idesc, 1u);
              mma_bf16_ss(tacc, da_lo, db_hi, idesc, 1u);
            }
            if (ks & 1) { mma_commit(&b_empty[s]); ++sb_it; }
          }
          mma_commit(&a_empty[buf]);
        }
        mma_commit(&tfull[a]);
      }
    }
  } else if (warp == FL_EPW + 2) {
    // ===================== segment tables: row ids per tile, (begin, length, stream offset) per (tile, relation) ========
    const int thr = p.hub_threshold;
    uint32_t mi = 0;
    int ti = 0;
    for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++ti) {
      int32_t* rows_s = tile_rows[ti & (FL_ROWRING - 1)];
      int rowv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        rowv[j] = (int)fl_tile_row(p, t, j * 32 + lane);
        rows_s[j * 32 + lane] = rowv[j];
      }
      for (int r = 0; r < R; ++r, ++mi) {
        const int s = mi % FL_NMETA;
        mbar_wait_parked(&meta_empty[s], ((mi / FL_NMETA) & 1) ^ 1);
        FLMeta& M = meta[s];
        int eff[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int beg = 0, len = 0;
          if (rowv[j] >= 0) {
            const int32_t* rp = p.rowptr + (int64_t)rowv[j] * R + r;
            beg = __ldg(rp);
            len = __ldg(rp + 1) - beg;
          }
          M.beg[j * 32 + lane] = beg;
          M.len[j * 32 + lane] = len;
          eff[j] = len > thr ? 0 : len;       // hub segments come from the chunk partials, not from the stream
        }
        int carry = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {         // exclusive prefix sums in slot order m = 32 j + lane
          int x = eff[j];
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
          }
          M.pre[j * 32 + lane] = carry + x - eff[j];
          carry += __shfl_sync(0xffffffffu, x, 31);
        }
        if (lane == 0) M.pre[FL_BM] = carry;
        __syncwarp();
        if (lane == 0) mbar_arrive(&meta_full[s]);
      }
    }
  } else {
    // ===================== producers: the block's edge stream, an equal share per worker =====================
    constexpr int G = C::G;                   // lanes per worker
    constexpr int RPW = 32 / G;               // workers per warp
    constexpr int NW = C::NW;
    constexpr int SELF_ROUNDS = (FL_BM + NW - 1) / NW;
    constexpr int U = 8;                      // independent 128-bit row loads in flight per lane
    const int pw = warp - (FL_EPW + 3);
    const int sub = lane / G, gl = lane % G;
    const int wk = pw * RPW + sub;            // worker id
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (sub * G));
    const int32_t* __restrict__ idx = p.idx;
    const int d_in = p.d_in;
    const int thr = p.hub_threshold;
    // position of this lane's 4 columns inside a block: swizzle unit, 16-byte chunk, half of the chunk
    const uint32_t unit_off = (uint32_t)(gl >> 4) * (FL_BM * 128);
    const uint32_t chunk = (uint32_t)(gl & 15) >> 1, half8 = (uint32_t)(gl & 1) * 8u;
    uint32_t blk = 0, mi = 0;
    int ti = 0;
    for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++ti) {
      const int32_t* rows_s = tile_rows[ti & (FL_ROWRING - 1)];
      for (int r = 0; r <= R; ++r) {
        const int ms = mi % FL_NMETA;
        const FLMeta& M = meta[ms];
        if (r < R) mbar_wait_parked(&meta_full[ms], (mi / FL_NMETA) & 1);     // (also orders the reads of rows_s after its writes)
        for (int h = 0; h < passes; ++h, ++blk) {
          const int col0 = h * CW + gl * 4;   // this lane's feature columns
          const int buf = blk % C::NBUF;
          mbar_wait_parked(&a_empty[buf], ((blk / C::NBUF) & 1) ^ 1);
          uint8_t* ab = smem_a + (size_t)buf * C::A_BLOCK;
          // finish slot m (node `row`, < 0: a padding slot of the tile) with the segment sum `val` of `len` edges
          auto finish = [&](int m, int row, int len, const float4& val) {
            uint8_t* s_hi = ab + unit_off + sw128_offset((uint32_t)m, chunk) + half8;
            __nv_bfloat16* g_hi = nullptr;
            __nv_bfloat16* g_lo = nullptr;
            if (p.A_hi && row >= 0) {
              const int64_t o = (int64_t)row * p.lda + (int64_t)r * d_in + col0;
              g_hi = p.A_hi + o;
              if (SPLIT) g_lo = p.A_lo + o;
            }
            fl_finish_row(val, len, s_hi, SPLIT ? (uint32_t)C::A_PLANE : 0u, g_hi, g_lo);
          };
          if (r == R) {
            // self-loop block: the rows themselves, slots wk, wk + NW, ...
            float4 v[SELF_ROUNDS];
            int rws[SELF_ROUNDS];
#pragma unroll
            for (int i = 0; i < SELF_ROUNDS; ++i) {
              const int m = wk + i * NW;
              rws[i] = m < FL_BM ? rows_s[m] : -1;
              v[i] = rws[i] >= 0 ? ldg4(p.x_root + (int64_t)rws[i] * p.ld_root + col0) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < SELF_ROUNDS; ++i)
              if (wk + i * NW < FL_BM) finish(wk + i * NW, rws[i], 1, v[i]);
          } else {
            const float* __restrict__ Fb = p.x_src + col0;
            const int64_t ldf = p.ld_src;
            const int Ltot = M.pre[FL_BM];
            const int S = (((Ltot + NW - 1) / NW) + U - 1) & ~(U - 1);          // share per worker, whole batches
            const int q0 = min(wk * S, Ltot), q1 = min(q0 + S, Ltot);
            float4* piece = scratch + ((size_t)(blk & 1) * NW) * G;             // [NW][G] of this block parity
            // slots that stream nothing: empty segments and padding slots (zeros), hub segments (their total)
            for (int m = wk; m < FL_BM; m += NW) {
              if (M.pre[m + 1] != M.pre[m]) continue;
              const int row = rows_s[m], len = M.len[m];
              float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
              if (row >= 0 && len > thr) val = fl_hub_sum(p, row * R + r, col0);
              finish(m, row, len, val);
            }
            int cur = -1;                     // slot that owns `acc`
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            int own_m = -1;                   // slot whose first piece is mine and whose end lies in a later worker
            float4 own_acc = make_float4(0.f, 0.f, 0.f, 0.f);
            auto close_row = [&]() {
              if (cur >= 0) {
                const int rs = M.pre[cur], re = M.pre[cur + 1];
                if (rs < q0) piece[(size_t)wk * G + gl] = acc;                 // began in an earlier worker: my piece
                else if (re > q1) { own_m = cur; own_acc = acc; }              // continues: combined after the barrier
                else finish(cur, rows_s[cur], M.len[cur], acc);
              }
              acc = make_float4(0.f, 0.f, 0.f, 0.f);
            };
            // stream position -> (slot, source row): the last slot whose start <= q (empty slots share a start)
            auto resolve = [&](int wbase, int& o_m, int& o_j) {
              const int q = wbase + gl;
              int lo = 0, hi = FL_BM;
#pragma unroll
              for (int it = 0; it < 7; ++it) {
                const int mid = (lo + hi) >> 1;
                if (M.pre[mid] <= q) lo = mid; else hi = mid;
              }
              o_m = lo;
              o_j = q < q1 ? __ldg(idx + M.beg[lo] + (q - M.pre[lo])) : 0;
            };
            int nm = 0, nj = 0;
            if (q0 < q1) resolve(q0, nm, nj);
            const uint32_t ldf32 = (uint32_t)ldf;
            for (int wbase = q0; wbase < q1; wbase += G) {
              const int my_m = nm, my_j = nj;
              if (wbase + G < q1) resolve(wbase + G, nm, nj);                  // the next window's indices, under the gathers
              const int n = min(G, q1 - wbase);
              // bit o of `starts`: window position o belongs to another slot than position o - 1 (position 0: than `cur`)
              const int prev_m = __shfl_up_sync(gmask, my_m, 1, G);
              const unsigned starts = (__ballot_sync(gmask, gl == 0 ? my_m != cur : my_m != prev_m) >> (sub * G)) &
                                      ((n >= 32) ? 0xffffffffu : ((1u << n) - 1u));
              for (int e = 0; e < n; e += U) {
                float4 v[U];
                if (e + U <= n) {
#pragma unroll
                  for (int u = 0; u < U; ++u) {
                    const int j = __shfl_sync(gmask, my_j, e + u, G);
                    v[u] = ldg4(Fb + (uint64_t)(uint32_t)j * ldf32);
                  }
                } else {
#pragma unroll
                  for (int u = 0; u < U; ++u) {
                    const int j = __shfl_sync(gmask, my_j, (e + u) & (G - 1), G);
                    v[u] = (e + u < n) ? ldg4(Fb + (uint64_t)(uint32_t)j * ldf32) : make_float4(0.f, 0.f, 0.f, 0.f);
                  }
                }
                const unsigned bits = (starts >> e) & ((1u << U) - 1u);
                if (bits == 0u) {
#pragma unroll
                  for (int u = 0; u < U; ++u) add4(acc, v[u]);                  // (masked slots add exact zeros)
                } else {
#pragma unroll
                  for (int u = 0; u < U; ++u) {
                    if (bits & (1u << u)) { close_row(); cur = __shfl_sync(gmask, my_m, e + u, G); }
                    add4(acc, v[u]);
                  }
                }
              }
            }
            close_row();
            // every worker's piece is in shared memory: the owner of a cut row adds the later pieces in stream order
            __syncwarp();
            asm volatile("bar.sync 1, %0;" ::"n"(FL_NPW * 32) : "memory");
            if (own_m >= 0) {
              const int re = M.pre[own_m + 1];
              for (int w2 = wk + 1; w2 < NW; ++w2) {
                add4(own_acc, piece[(size_t)w2 * G + gl]);
                if (re <= (w2 + 1) * S) break;
              }
              finish(own_m, rows_s[own_m], M.len[own_m], own_acc);
            }
          }
          fence_proxy_async();                 // generic-proxy smem writes -> visible to the tensor core's reads
          __syncwarp();
          if (lane == 0) mbar_arrive(&a_full[buf]);
        }
        if (r < R) {
          if (lane == 0) mbar_arrive(&meta_empty[ms]);   // (after the __syncwarp above: all lanes are done with M)
          ++mi;
        }
      }
    }
  }
  __syncthreads();
  if (warp == 0) {
    fence_after_sync();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

static int fused_env() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RGCN_FUSED_FWD");
    v = !e ? 2 : (e[0] == '0' ? 0 : 1);
  }
  return v;
}

// 0: not eligible.  The fused kernel serves the unmixed forward with fp32 gathers: d_in a multiple of 64, d_out <= 256.
int fused_layer_fwd_eligible(const rgcn_layer_fwd_args* a) {
  // a->pipeline selects the schedule of the call: 0 = the library decides, 1 = walk then transform (two kernels),
  // 2 = row chunks pipelined on two streams, 3 = this kernel
  const int env = a->pipeline == 3 ? 1 : fused_env();
  if (env == 0 || !a->w_planes || a->pipeline == 1 || a->pipeline == 2) return 0;
  const rgcn_csr_t* g = a->csr;
  if (g->w || g->n_rows <= 0) return 0;
  if (a->d_in < 64 || a->d_in % 64 || a->d_in > 1024) return 0;
  if (a->d_out < 16 || a->d_out % 16 || a->d_out > 256) return 0;
  if (a->mode == 1 && a->x_bf16 && a->x_src == a->x_root) return 0;        // bf16 gathers: the unfused walk
  if (((uintptr_t)a->x_src & 15) || a->ld_x_src % 4 || ((uintptr_t)a->x_root & 15) || a->ld_x_root % 4) return 0;
  if (((uintptr_t)a->out & 15) || a->ldo % 4) return 0;
  if (a->n_peer > FL_MAXPEERS) return 0;
  // Library default (env unset, schedule 0): NOT used.  Measured on the B200 (profiles/r2_fused_layer_*): correct, but
  // 372 us against 136 us for the two-kernel path on cfg2's layer 2.  The producers are bound by the latency of their own
  // control flow (27.7 cycles per issued instruction, no eligible warp in 71 % of the cycles; every row slice is finished
  // — divided, converted, stored — eight times per tile, and 18 % of the warp samples wait at the per-block barrier), not
  // by the gathers: with the gathers, the MMAs and the output stores all switched off the kernel still took 376 us.
  // RGCN_FUSED_FWD=1 or schedule 3 opt in.
  if (env == 2) return 0;
  return 1;
}

template <int CW, bool SPLIT>
static int launch_fused(const FusedParams& p, const CUtensorMap& mhi, const CUtensorMap& mlo, unsigned grid, cudaStream_t st) {
  using C = FLCfg<CW, SPLIT>;
  int rc = set_smem(fused_layer_fwd_kernel<CW, SPLIT>, C::SMEM);
  if (rc) return rc;
  RGCN_CUDA(launch_pdl(fused_layer_fwd_kernel<CW, SPLIT>, dim3(grid), dim3(FL_THREADS), (size_t)C::SMEM, st, mhi, mlo, p));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

// weights already converted (rgcn_prepare_weights), hub chunk partials already in a->agg_workspace (reduced per segment here)
int fused_layer_fwd_launch(const rgcn_layer_fwd_args* a, cudaStream_t st) {
  const rgcn_csr_t* g = a->csr;
  if (g->n_hubs > 0) {
    const int thr = a->d_in / 4 < 256 ? a->d_in / 4 : 256;
    RGCN_CUDA(launch_pdl(hub_reduce_kernel, dim3((unsigned)g->n_hubs), dim3((unsigned)thr), 0, st, (float*)a->agg_workspace,
                         g->hub_chunk_ptr, (int)a->d_in));
    RGCN_LAUNCH_CHECK();
  }
  const int R = g->R;
  const int K = (R + 1) * a->d_in;
  FusedParams p{};
  p.rowptr = g->rowptr; p.idx = g->idx; p.hub_keys = g->hub_keys; p.hub_chunk_ptr = g->hub_chunk_ptr;
  p.hub_threshold = g->hub_threshold; p.n_hubs = g->n_hubs; p.R = R; p.n_rows = g->n_rows;
  p.partials = (const float*)a->agg_workspace;
  p.x_src = a->x_src; p.ld_src = a->ld_x_src; p.x_root = a->x_root; p.ld_root = a->ld_x_root; p.d_in = a->d_in;
  const int64_t t0 = (g->n_rows + FL_BM - 1) / FL_BM;
  const unsigned grid = (unsigned)(t0 < sm_count() ? t0 : sm_count());
  // any row permutation may be dealt; a degree order (global, or inside blocks of order_chunk_rows) balances the tiles
  p.deal = g->row_order ? 1 : 0;
  p.row_order = g->row_order;
  p.n_tiles = (int32_t)(p.deal ? (t0 + grid - 1) / grid * grid : t0);
  p.A_hi = (__nv_bfloat16*)a->A_hi; p.A_lo = (__nv_bfloat16*)a->A_lo; p.lda = a->lda;
  p.N = a->d_out; p.BN = round_up(a->d_out, 16);
  p.bias = a->bias; p.relu = a->relu; p.out = a->out; p.ldo = a->ldo;
  p.out16 = (__nv_bfloat16*)a->out_bf16; p.ldo16 = a->ld_out_bf16;
  if (a->dropout_p > 0.f) {
    const double th = (double)a->dropout_p * 65536.0 + 0.5;
    p.drop_thresh = th >= 65535.0 ? 65535u : (th < 1.0 ? 1u : (uint32_t)th);
    p.drop_scale = 1.f / (1.f - a->dropout_p);
    p.drop_seed = a->dropout_seed; p.drop_ctr = a->dropout_counter; p.drop_row0 = a->dropout_row0;
  }
  p.n_peer = a->n_peer; p.peer_row0 = a->peer_row0; p.peer_ld = a->peer_ld;
  for (int q = 0; q < a->n_peer; ++q) p.peer_out[q] = a->peer_out_host[q];
  const __nv_bfloat16* bhi = (const __nv_bfloat16*)a->w_planes;
  const __nv_bfloat16* blo = (const __nv_bfloat16*)((const char*)a->w_planes + wplane_bytes(K, a->d_out));
  const bool split = a->mode == 0;
  CUtensorMap mhi, mlo;
  int rc = make_map(&mhi, bhi, K, a->d_out, wplane_ld(a->d_out), FL_KB);
  if (rc) return rc;
  rc = make_map(&mlo, split ? blo : bhi, K, a->d_out, wplane_ld(a->d_out), FL_KB);
  if (rc) return rc;
  if (a->d_in % 128 == 0)
    return split ? launch_fused<128, true>(p, mhi, mlo, grid, st) : launch_fused<128, false>(p, mhi, mlo, grid, st);
  return split ? launch_fused<64, true>(p, mhi, mlo, grid, st) : launch_fused<64, false>(p, mhi, mlo, grid, st);
}

}  // namespace rgcn
