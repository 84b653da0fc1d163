// Segmented gather + reduce over a relation-keyed CSR: the neighbourhood aggregation of RGCNConv
// (reference call sites src/models/rgcn.py:123, :128) and its transpose for backward.
//
// One family of kernels serves forward and backward:
//   s(i, r)  = sum_{e in seg(i, r)} w(e) * F[idx[e], r * src_rel_stride : +d]     (w = 1 when edge_w == NULL)
//   h(i, r)  = s / max(len, 1)                       when edge_w == NULL  (scatter-MEAN)
//            = s                                     otherwise
//   MIX_NONE : O[i, r*d : (r+1)*d] = h(i, r)                                   forward, full weights
//   MIX_SUM  : O[i, :]             = init[i, :] + sum_r h(i, r)                backward (grad-X)
//   MIX_BASIS: O[i, b*d : (b+1)*d] = sum_r comp[r, b] * h(i, r)                basis decomposition
//
// Mapping: a group of G = min(32, d/4) lanes owns one row i and walks its R segments; every lane
// holds VPL float4 of the d-wide accumulator, issues U independent 128-bit row loads per step and
// adds them left to right, i.e. in the CSR's (= original) edge order.  No atomics anywhere.
// Segments longer than kHubThreshold ("hubs", power-law graphs have rows with 10^4 edges) are cut
// into kHubChunk-edge chunks that whole blocks reduce beforehand (hub_partial_kernel) into a
// partial buffer; the row kernel then adds the chunk partials in chunk order.  Everything is
// deterministic: same bits on every run.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace rgcn {

enum { MIX_NONE = 0, MIX_SUM = 1, MIX_BASIS = 2 };
#ifndef RGCN_TAILPRED_MAX_VPL
#define RGCN_TAILPRED_MAX_VPL 1     // feature widths (in 128-bit vectors per lane) that take one predicated tail batch
#endif
constexpr int kMaxBasis = 8;

struct AggParams {
  const int32_t* rowptr;
  const int32_t* idx;
  const float* edge_w;       // nullable
  const int32_t* hub_keys;   // sorted keys of hub segments
  const int32_t* hub_chunk_ptr;
  const int32_t* chunk_table;  // [n_chunks][4]: {segment key, first chunk of the segment, -, -}
  const int32_t* row_order;    // nullable: rows in the order the groups take them (longest first)
  int32_t hub_threshold;
  int32_t skip_hubs;           // the row walk leaves hub segments out (hub_finish_kernel adds them afterwards)
  int32_t n_hubs;
  int64_t n_rows;
  int32_t range_mode;          // 0: the launch walks all rows; 1: positions [row_begin, row_end) of the row order only
  int64_t row_begin, row_end;
  int32_t no_hub_pass;         // the chunk partials are already in `partials` (an earlier launch of the same call made them)
  int32_t R;
  const float* F;            // gathered feature matrix
  int64_t ldf;
  int32_t src_rel_stride;    // column offset per relation inside a gathered row (0 forward, d backward)
  int32_t d;
  int32_t block_stride;      // columns between consecutive relation / basis blocks of the output (= d unless the
                             // feature columns are processed in slices)
  const float* comp;         // [R, ldcomp] (MIX_BASIS)
  int32_t ldcomp;
  int32_t B;
  const float* init;         // nullable (MIX_SUM)
  int64_t ld_init;
  const float* root_rows;    // nullable (MIX_NONE): row i of this matrix is appended as block R of output row i — the
  int64_t ld_root;           // self-loop operand [H | X] of the transform is then complete after one kernel
  void* O;
  void* O_lo;                // second bf16 plane (out_mode 2)
  int64_t ldo;
  int32_t out_mode;          // 0: fp32, 1: bf16 (hi plane only), 2: bf16 hi + lo planes (hi + lo = value to 2^-17)
  float* partials;           // [n_chunks, d]
  // MIX_BASIS side output (gradient of the basis coefficients): gc[r, b] += <h(i, r), dotP[i, b*d : (b+1)*d]>,
  // written as one [R * B] partial per block, reduced afterwards in block order
  const float* dotP;         // nullable, [n_rows, B * d]
  int64_t ld_dotP;
  float* gc_partial;         // [gridDim.x, R * B]
  // Row-sparse gathered matrix (backward of a layer whose output gradient is zero outside a short row list, e.g. the
  // 2 * batch rows a link-prediction loss touches): F holds only the listed rows, slot[j] is the compact row of node j
  // or zero_row (an all-zero row of F) for every other node.  Absent edges are skipped; since they would add exact
  // zeros, the result equals the dense walk bit for bit.
  const int32_t* slot;       // nullable, [number of gatherable nodes]
  int32_t zero_row;
  // MIX_SUM second output (nullable): the result masked for the layer UPSTREAM — v = (mask > 0 ? O * mp_scale : 0) with
  // mask = that layer's ReLU / dropout output — written as the bf16 operand planes its backward GEMMs read, plus the
  // per-block column sums (its bias gradient).  Saves the separate conversion pass over O.
  const float* mp_mask; int64_t ld_mp_mask; float mp_scale;
  void* mp_hi; void* mp_lo; int64_t ld_mp;
  float* mp_colsum;          // nullable, [gridDim.x, d]
  // Listed-rows forward (LIST instantiations; the last layer of a link-prediction step is only read at the 2 * batch
  // head / tail rows): position c of the launch walks row list[c] and writes OUTPUT row c of a compact [m_c, ...] matrix;
  // positions >= n_list (padding up to a multiple of 128) get all-zero rows.
  const int64_t* list;
  int64_t n_list;
  // the listed walk is latency bound (few, long rows): gridDim.y column slices of d columns each (d = slice width, the
  // output blocks stay block_stride apart) x gridDim.z relation ranges per row shorten every dependent chain of loads;
  // sums per (row, relation, column) keep their edge order, so the bits do not change
  int32_t list_slices, list_rsplit;
  // groups [0, list_walkers) walk: by ROWS (list_by_rows: group i takes row row_order[i] — longest first — and leaves at
  // once unless slot[row] lists it; its output row is slot[row]) or by POSITIONS (group c takes row list[c] if it is the
  // row's first position); groups [list_walkers, list_walkers + m_c) zero-fill the duplicate and padding positions.
  // Either way a row that the list names several times is walked once.
  int64_t list_walkers;
  int32_t list_by_rows;
  int32_t list_overlap_hubs;   // hub chunks on a side stream beside the listed walk (which skips the hub segments) + finish kernel
  int32_t stream_rel;        // backward walk: stream a row's edges across relation boundaries (short segments, many relations)
  // row-sparse backward on large graphs (nullable): row_flag[j] != 0 iff some edge of source row j gathers a LISTED row
  // (marked beforehand from the forward-orientation CSR of the listed rows, mark_sources_kernel); the other rows leave at
  // once with their init row — the walk then costs per marked row, not per row of the graph
  const uint8_t* row_flag;
  // hub pass filter (nullable): node -> first list position map; chunks of rows with hub_filter[row] == hub_unlisted are skipped
  const int32_t* hub_filter;
  int32_t hub_unlisted;
};

// ---- hub chunks: one block per chunk --------------------------------------------------------
template <int G, int VPL, bool W, bool SLOT = false>
__global__ void __launch_bounds__(256) hub_partial_kernel(const AggParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  __shared__ float4 red[GROUPS][G * VPL];
  const int chunk = blockIdx.x;
  // one table load instead of a search through the hub list (a chain of dependent loads in front of every block)
  const int4 t = __ldg(reinterpret_cast<const int4*>(p.chunk_table) + chunk);
  const int key = t.x;
  const int r = key % p.R;
  if (p.hub_filter && __ldg(p.hub_filter + key / p.R) == p.hub_unlisted) return;     // (block-uniform) nobody reads this row
  const int seg_beg = __ldg(p.rowptr + key), seg_end = __ldg(p.rowptr + key + 1);
  const int c_beg = seg_beg + (chunk - t.y) * kHubChunk;
  const int c_end = min(c_beg + kHubChunk, seg_end);
  const int nvec = p.d >> 2;
  const int lane = threadIdx.x % G, grp = threadIdx.x / G;
  // each group sums a contiguous slice of the chunk, left to right
  constexpr int PER = kHubChunk / GROUPS;
  const int g_beg = c_beg + grp * PER, g_end = min(g_beg + PER, c_end);
  float4 acc[VPL];
  int vcol[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int vi = k * G + lane;
    vcol[k] = vi < nvec ? vi * 4 : 0;
  }
  const float* __restrict__ Fb = p.F + (size_t)r * p.src_rel_stride;
  const int32_t* __restrict__ idx = p.idx;
  const float* __restrict__ ew = p.edge_w;
  const int64_t ldf = p.ldf;
  constexpr int U0 = (VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8);
  constexpr int U = U0 < PER ? U0 : PER;
  // the group's PER (<= G) edge indices, slots and weights in ONE coalesced load per array, handed out by shuffle: the
  // gathers of all batches then depend on a single index latency instead of one per batch
  static_assert(PER <= G, "a group's slice of a hub chunk must fit its lanes");
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G));
  const bool mine = lane < PER && g_beg + lane < g_end;
  int my_j = mine ? __ldg(idx + g_beg + lane) : 0;
  if (SLOT) my_j = mine ? __ldg(p.slot + my_j) : p.zero_row;
  const float my_w = (W && mine) ? __ldg(ew + g_beg + lane) : 0.f;
  int e = g_beg;
  for (; e + U <= g_end; e += U) {
    float4 v[U][VPL];
    float w[U];
    int js[U];
    bool any = !SLOT;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      js[u] = __shfl_sync(gmask, my_j, e + u - g_beg, G);
      if (W) w[u] = __shfl_sync(gmask, my_w, e + u - g_beg, G);
      if (SLOT) any |= js[u] != p.zero_row;
    }
    if (!any) continue;                            // (group-uniform) every edge of the batch points at a zero row
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = js[u];
      const float* __restrict__ rp = Fb + (size_t)j * ldf;
      const bool on = !SLOT || j != p.zero_row;
#pragma unroll
      for (int k = 0; k < VPL; ++k) v[u][k] = on ? ldg4(rp + vcol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int k = 0; k < VPL; ++k) {
        if (W) fma4(acc[k], w[u], v[u][k]); else add4(acc[k], v[u][k]);
      }
  }
  for (; e < g_end; ++e) {                         // (group-uniform trip count)
    const int j = __shfl_sync(gmask, my_j, e - g_beg, G);
    const float wv = W ? __shfl_sync(gmask, my_w, e - g_beg, G) : 1.f;
    if (SLOT && j == p.zero_row) continue;
    const float* __restrict__ rp = Fb + (size_t)j * ldf;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const float4 v = ldg4(rp + vcol[k]);
      if (W) fma4(acc[k], wv, v); else add4(acc[k], v);
    }
  }
#pragma unroll
  for (int k = 0; k < VPL; ++k) red[grp][k * G + lane] = acc[k];
  __syncthreads();
  // fixed-order reduce over the groups, one thread per float4 column
  for (int vi = threadIdx.x; vi < nvec; vi += 256) {
    float4 s = red[0][vi];
    for (int g = 1; g < GROUPS; ++g) add4(s, red[g][vi]);
    reinterpret_cast<float4*>(p.partials + (size_t)chunk * p.d)[vi] = s;
  }
}

__device__ __forceinline__ void store_vec_to(void* O, void* O_lo, int64_t ldo, int out_mode, int64_t row, int col,
                                             const float4& v) {
  if (out_mode == 0) {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(O) + row * ldo + col) = v;
    return;
  }
  // packed conversions (F2FP); the bf16 planes are the TMA-loadable operand format of the tensor-core kernels
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 hi;
  hi.x = *reinterpret_cast<uint32_t*>(&a);
  hi.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(O) + row * ldo + col) = hi;
  if (out_mode == 2) {
    const float hx = __uint_as_float(hi.x << 16), hy = __uint_as_float(hi.x & 0xffff0000u);
    const float hz = __uint_as_float(hi.y << 16), hw = __uint_as_float(hi.y & 0xffff0000u);
    a = __floats2bfloat162_rn(v.x - hx, v.y - hy);
    b = __floats2bfloat162_rn(v.z - hz, v.w - hw);
    uint2 lo;
    lo.x = *reinterpret_cast<uint32_t*>(&a);
    lo.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(O_lo) + row * ldo + col) = lo;
  }
}
__device__ __forceinline__ void store_vec(const AggParams& p, int64_t row, int col, const float4& v) {
  store_vec_to(p.O, p.O_lo, p.ldo, p.out_mode, row, col, v);
}

// ---- rows: one G-lane group per row ----------------------------------------------------------
// The inner loop is instruction-issue sensitive (16 B per lane per edge): parameters are hoisted into registers,
// the edge weights are a template flag, full batches of U edges run without any predicate, inactive lanes of a
// ragged feature width read column 0 instead of being masked, and only the tail batch is guarded.
// resident blocks per SM the register allocation aims at: the walk is latency bound, occupancy is its throughput
constexpr int agg_min_blocks(int G, int vpl, int mix, bool w) {
  // measured on the B200 (scripts/bench_agg.py, scripts/bench_cfg.py cfg1 / cfg2)
  if (mix == MIX_BASIS || vpl > 2) return 1;
  if (vpl == 2) return (mix == MIX_NONE && !w) ? 5 : 4;          // d = 256: forward 48 registers, backward 64
  if (G == 32) return mix == MIX_NONE ? 6 : 5;                    // d = 128
  // d <= 64: the walk's time does not move with this choice (3 .. 6 blocks measured the same): 256-byte rows top out at
  // ~7 TB/s of gathered bytes whatever the occupancy, lane-group width or prefetch depth (DESIGN.md §5)
  return (mix == MIX_SUM && w) ? 3 : 4;
}

// MP: the masked-planes second output (MIX_SUM only) is compiled in; one resident block less buys it the registers
// MARK (row-sparse backward only): rows whose row_flag byte is zero leave at once — a separate instantiation, so that the
// unmarked walk keeps its register allocation (with the test compiled in, the d = 256 row-sparse walk spilled: 33 -> 66 us)
template <int G, int VPL, int MIX, bool W, bool SLOT = false, bool MP = false, bool LIST = false, bool MARK = false>
__global__ void __launch_bounds__(256, LIST ? (VPL > 2 ? 1 : (W ? 2 : 3)) : agg_min_blocks(G, VPL, MIX, W) - (((MP || MARK) && agg_min_blocks(G, VPL, MIX, W) > 1) ? 1 : 0))
aggregate_rows_kernel(const AggParams p) {
  static_assert(!MARK || (SLOT && !MP && MIX == MIX_SUM), "marked sources serve the row-sparse backward walk");
  static_assert(!LIST || (MIX == MIX_NONE && !SLOT && !MP), "the listed-rows walk is the unmixed forward form");
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  constexpr int NB = (MIX == MIX_BASIS) ? kMaxBasis : 1;
  constexpr int U0 = (VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8);
  constexpr int U = U0 < G ? U0 : G;             // a batch never exceeds the index window
  constexpr bool TAILPRED = MIX != MIX_BASIS && VPL <= RGCN_TAILPRED_MAX_VPL;
  constexpr bool CHAIN = MIX == MIX_SUM && W;    // backward walk: weighted sums, all relations into one accumulator
  extern __shared__ float s_comp[];   // [R * B] for MIX_BASIS, then [GROUPS][R * B] coefficient-gradient sums
  const bool with_gc = MIX == MIX_BASIS && p.dotP != nullptr;
  const bool with_cs = MP && MIX == MIX_SUM && p.mp_colsum != nullptr;       // s_comp then holds [GROUPS][d] column-sum rows
  float* s_gc = s_comp + p.R * p.B;
  if (MIX == MIX_BASIS) {
    for (int t = threadIdx.x; t < p.R * p.B; t += 256) s_comp[t] = p.comp[(t / p.B) * p.ldcomp + (t % p.B)];
    if (with_gc)
      for (int t = threadIdx.x; t < GROUPS * p.R * p.B; t += 256) s_gc[t] = 0.f;
    __syncthreads();
  }
  const int lane = threadIdx.x % G, grp = threadIdx.x / G;
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G));
  int64_t row = p.row_begin + (int64_t)blockIdx.x * GROUPS + grp;
  if (row >= p.row_end) {
    if (!with_gc && !with_cs) return;
    if (with_cs)
      for (int t = lane; t < p.d; t += G) s_comp[grp * p.d + t] = 0.f;
  } else {
  int64_t orow = row;                            // LIST: the output row is the row's first list position
  if (LIST) {
    if (row >= p.list_walkers) {
      // duplicate or padding position: an all-zero operand row (stale memory could hold NaN patterns)
      const int64_t c = row - p.list_walkers;
      const bool fill = c >= p.n_list || __ldg(p.hub_filter + __ldg(p.list + c)) != (int32_t)c;
      if (fill && blockIdx.y == 0 && blockIdx.z == 0) {
        const int nblk = p.R + (p.root_rows ? 1 : 0);
        for (int b = 0; b < nblk; ++b)
          for (int vi = lane; vi < ((p.d * (int)gridDim.y) >> 2); vi += G)
            store_vec(p, c, b * p.block_stride + vi * 4, make_float4(0.f, 0.f, 0.f, 0.f));
      }
      return;
    }
    if (p.list_by_rows) {
      if (p.row_order) row = __ldg(p.row_order + row);
      orow = __ldg(p.hub_filter + row);
      if (orow == p.hub_unlisted) return;
    } else {
      row = __ldg(p.list + orow);
      if (__ldg(p.hub_filter + row) != (int32_t)orow) return;          // a later duplicate: the first position has the row
    }
  } else if (p.row_order) {
    // longest rows first: neighbouring groups get rows of similar length and the long walks start at time zero
    row = __ldg(p.row_order + row);
  }
  if (MARK && !__ldg(p.row_flag + row)) {
    // (group-uniform) none of this row's edges gathers a listed row: every term of its sum is an exact zero, the result is
    // the init row alone.  Kept ahead of everything else so that the walk below compiles exactly as without the test.
    const float* __restrict__ ir = p.init ? p.init + (int64_t)__ldg(p.slot + row) * p.ld_init : nullptr;
    for (int vi = lane; vi < (p.d >> 2); vi += G)
      store_vec(p, row, vi * 4, ir ? ldg4(ir + vi * 4) : make_float4(0.f, 0.f, 0.f, 0.f));
    return;
  }
  const int R = p.R, d = p.d, nvec = p.d >> 2;
  const int64_t key0 = row * R;
  const int32_t* __restrict__ rowptr = p.rowptr + key0;
  const int32_t* __restrict__ idx = p.idx;
  const float* __restrict__ ew = p.edge_w;
  const int coff = LIST ? (int)blockIdx.y * p.d : 0;                        // this block's column slice
  const int pstride = LIST ? p.d * (int)gridDim.y : p.d;                    // row stride of the hub partials (full width)
  int r_lo = 0, r_hi = p.R;                                                 // this block's relation range
  if (LIST) {
    const int per = (p.R + (int)gridDim.z - 1) / (int)gridDim.z;
    r_lo = (int)blockIdx.z * per;
    r_hi = min(p.R, r_lo + per);
  }
  const float* __restrict__ F = p.F + coff;
  const int64_t ldf = p.ldf;
  const int rel_stride = p.src_rel_stride;
  bool act[VPL];
  int vcol[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    act[k] = vi < nvec;
    vcol[k] = act[k] ? vi * 4 : 0;               // inactive lanes gather column 0; their sums are never stored
  }

  if (MIX == MIX_NONE && p.root_rows && (!LIST || blockIdx.z == 0)) {
#pragma unroll
    for (int k = 0; k < VPL; ++k)
      if (act[k]) store_vec(p, LIST ? orow : row, R * p.block_stride + coff + vcol[k], ldg4(p.root_rows + row * p.ld_root + coff + vcol[k]));
  }
  float4 mix[NB][VPL];
  if (MIX != MIX_NONE) {
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
      for (int k = 0; k < VPL; ++k) mix[b][k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (MIX == MIX_SUM && p.init) {
      const int64_t irow = SLOT ? (int64_t)__ldg(p.slot + row) : row;      // compact row of this node (or the zero row)
#pragma unroll
      for (int k = 0; k < VPL; ++k) mix[0][k] = ldg4(p.init + irow * p.ld_init + vcol[k]);
    }
  }

  // A row's edges are contiguous in the CSR (sorted by (row, relation)).  The group keeps a window of 2*G edge
  // indices (and weights) in registers — two coalesced loads issued back to back — and hands them out by shuffle.
  const int row_end = __ldg(rowptr + R);
  int wbase = -(1 << 30), wi0 = 0, wi1 = 0;
  float ww0 = 1.f, ww1 = 1.f;
  unsigned long long present = 0ull;     // SLOT: bit o = edge wbase + o of the window gathers a listed row
  auto refill = [&](int e) {
    wbase = e;
    const bool in0 = e + lane < row_end, in1 = e + G + lane < row_end;
    wi0 = in0 ? __ldg(idx + e + lane) : 0;
    wi1 = in1 ? __ldg(idx + e + G + lane) : 0;
    if (SLOT) {
      wi0 = in0 ? __ldg(p.slot + wi0) : p.zero_row;
      wi1 = in1 ? __ldg(p.slot + wi1) : p.zero_row;
      const int sh = (G == 32) ? 0 : (int)((threadIdx.x & 31) / G * G);
      const unsigned b0 = (__ballot_sync(gmask, wi0 != p.zero_row) & gmask) >> sh;
      const unsigned b1 = (__ballot_sync(gmask, wi1 != p.zero_row) & gmask) >> sh;
      present = ((unsigned long long)b1 << G) | (unsigned long long)b0;
    }
    if (W) {
      ww0 = in0 ? __ldg(ew + e + lane) : 0.f;
      ww1 = in1 ? __ldg(ew + e + G + lane) : 0.f;
    }
  };

  for (int rbase = r_lo; rbase < r_hi; rbase += G) {
    // the group's lanes fetch G consecutive (beg, end) pairs with two coalesced loads
    const int rl = rbase + lane;
    const int my_beg = (rl < r_hi) ? __ldg(rowptr + rl) : 0;
    const int my_end = (rl < r_hi) ? __ldg(rowptr + rl + 1) : 0;
    const int rcount = min(G, r_hi - rbase);
    if (CHAIN && !SLOT && p.stream_rel) {
      // Backward (summed relations, weighted edges): the row's sum does not care where one relation ends and the next
      // begins, only the column block of the gathered slice does.  So the edges of the G relations this pass covers are
      // streamed as ONE list, U loads in flight across segment boundaries — a graph with 30 relations has mostly one- and
      // two-edge segments, and a batch per segment leaves the memory system idle.  The relation of an edge is the number
      // of segments that end at or before it (one ballot over the lanes' segment ends).  Same additions in the same
      // (edge) order as the per-relation loop below, which serves the passes that contain a hub segment.
      const bool lane_hub = rl < r_hi && my_end - my_beg > p.hub_threshold;
      const int cbeg = __shfl_sync(gmask, my_beg, 0, G);
      const int cend = __shfl_sync(gmask, my_end, rcount - 1, G);
      // ... where it pays: passes whose non-empty segments average fewer than four edges (stream_rel = 1; 3 = always).  A
      // power-law row is mostly a few long segments, whose batches are full anyway (cfg3: streaming everything costs 7 %)
      const int n_seg = __popc(__ballot_sync(gmask, rl < r_hi && my_end > my_beg) & gmask);
      if ((__ballot_sync(gmask, lane_hub) & gmask) == 0u && (p.stream_rel == 3 || cend - cbeg < 4 * n_seg)) {
        const int endk = rl < r_hi ? my_end : 0x7fffffff;          // lanes beyond the pass never count
        const float* __restrict__ Fb = F + (size_t)rbase * rel_stride;
        int e = cbeg;
        auto fbatch = [&](auto ub, const bool pred) {
          constexpr int UB = decltype(ub)::value;
          if (e + UB > wbase + 2 * G) refill(e);
          float4 v[UB][VPL];
          float w[UB];
#pragma unroll
          for (int u = 0; u < UB; ++u) {
            const int off = e + u - wbase;             // uniform across the group, < 2 * G
            const int j = __shfl_sync(gmask, (off & G) ? wi1 : wi0, off & (G - 1), G);
            const float wv = __shfl_sync(gmask, (off & G) ? ww1 : ww0, off & (G - 1), G);
            const int rel = __popc(__ballot_sync(gmask, endk <= e + u) & gmask);
            const bool on = !pred || e + u < cend;
            w[u] = on ? wv : 0.f;
            const float* __restrict__ rp = Fb + (size_t)j * ldf + (size_t)rel * rel_stride;
#pragma unroll
            for (int k = 0; k < VPL; ++k) v[u][k] = on ? ldg4(rp + vcol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int u = 0; u < UB; ++u)
#pragma unroll
            for (int k = 0; k < VPL; ++k) fma4(mix[0][k], w[u], v[u][k]);
          e += UB;
        };
        while (e + U <= cend) fbatch(std::integral_constant<int, U>{}, false);
        const int n_left = cend - e;
        if (n_left == 1) fbatch(std::integral_constant<int, 1>{}, false);
        else if (n_left == 2) fbatch(std::integral_constant<int, (U >= 2 ? 2 : 1)>{}, U < 2);
        else if (n_left > 0 && n_left <= 4 && U > 4) fbatch(std::integral_constant<int, (U > 4 ? 4 : 1)>{}, true);
        else if (n_left > 0) fbatch(std::integral_constant<int, U>{}, true);
        continue;
      }
    }
    for (int rr = 0; rr < rcount; ++rr) {
      const int r = rbase + rr;
      const int beg = __shfl_sync(gmask, my_beg, rr, G);
      const int end = __shfl_sync(gmask, my_end, rr, G);
      const int len = end - beg;
      if (len == 0 && MIX != MIX_NONE) continue;
      if (MIX != MIX_BASIS && p.skip_hubs && len > p.hub_threshold) continue;   // added by hub_finish_kernel
      float4 acc[VPL];
      // CHAIN: the weighted sums of the non-hub segments continue the row's accumulator itself (one chain of additions in
      // edge order, whichever of the three code paths — streamed, per relation, row-sparse — walks the row)
      const bool chained = CHAIN && len <= p.hub_threshold;
#pragma unroll
      for (int k = 0; k < VPL; ++k) acc[k] = chained ? mix[0][k] : make_float4(0.f, 0.f, 0.f, 0.f);
      if (len > p.hub_threshold) {
        // hub: add the chunk partials in chunk order
        const int key = (int)(key0 + r);
        int lo = 0, hi = p.n_hubs;
        while (hi - lo > 1) {
          int mid = (lo + hi) >> 1;
          if (__ldg(p.hub_keys + mid) <= key) lo = mid; else hi = mid;
        }
        const int c0 = __ldg(p.hub_chunk_ptr + lo), c1 = __ldg(p.hub_chunk_ptr + lo + 1);
        // loads U chunks ahead (a 10^4-edge hub has ~100 partials: one dependent load each would be a long chain),
        // adds strictly in chunk order
        int c = c0;
        for (; c + U <= c1; c += U) {
          float4 v[U][VPL];
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < VPL; ++k) v[u][k] = *reinterpret_cast<const float4*>(p.partials + (size_t)(c + u) * pstride + coff + vcol[k]);
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < VPL; ++k) add4(acc[k], v[u][k]);
        }
        for (; c < c1; ++c) {
#pragma unroll
          for (int k = 0; k < VPL; ++k) add4(acc[k], *reinterpret_cast<const float4*>(p.partials + (size_t)c * pstride + coff + vcol[k]));
        }
      } else if (SLOT && len > 0) {
        // only the edges whose gathered row is listed, in edge order: the window's presence mask is walked bit by bit,
        // one 32-bit half at a time (G <= 32), batches of 4 — or 2 when no more bits are left, since a segment of a
        // PrimeKG row has two or three listed edges on average and every unrolled slot costs issue cycles
        const float* __restrict__ Fb = F + (size_t)r * rel_stride;
        int e = beg;
        auto run = [&](unsigned m, int wsel, int obase) {
          auto batch = [&](auto ub) {
            constexpr int UB = decltype(ub)::value;
            float4 v[UB][VPL];
            float w[UB];
#pragma unroll
            for (int u = 0; u < UB; ++u) {
              const bool on = m != 0u;
              const int off = on ? __ffs((int)m) - 1 : obase;
              m &= m - 1u;
              const int j = __shfl_sync(gmask, wsel ? wi1 : wi0, off, G);
              const float wv = __shfl_sync(gmask, wsel ? ww1 : ww0, off, G);
              w[u] = on ? wv : 0.f;
              const float* __restrict__ rp = Fb + (size_t)j * ldf;
#pragma unroll
              for (int k = 0; k < VPL; ++k) v[u][k] = on ? ldg4(rp + vcol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < UB; ++u)
#pragma unroll
              for (int k = 0; k < VPL; ++k) fma4(acc[k], w[u], v[u][k]);
          };
          while (m) {
            if (U >= 4 && __popc(m) > 2) batch(std::integral_constant<int, (U >= 4 ? 4 : 2)>{});
            else batch(std::integral_constant<int, 2>{});
          }
        };
        while (e < end) {
          if (e >= wbase + 2 * G) refill(e);
          const int o0 = e - wbase;                       // < 2 G
          const int lim = min(end - wbase, 2 * G);
          const unsigned full = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);
          if (o0 < G) {
            const int hi = min(lim, G);
            unsigned m = ((unsigned)present & full) >> o0 << o0;
            if (hi < G) m &= (1u << hi) - 1u;
            run(m, 0, o0);
          }
          if (lim > G) {
            const int lo = max(o0 - G, 0), hi = lim - G;
            unsigned m = ((unsigned)(present >> G) & full) >> lo << lo;
            if (hi < G) m &= (1u << hi) - 1u;
            run(m, 1, lo);
          }
          e = wbase + lim;
        }
      } else if (len > 0) {
        const float* __restrict__ Fb = F + (size_t)r * rel_stride;
        // full batches of U edges, then power-of-two remainders: every batch is straight-line code with
        // unconditional loads, nothing is gathered twice and nothing is masked
        int e = beg;
        auto batch = [&](auto ub) {
          constexpr int UB = decltype(ub)::value;
          if (e + UB > wbase + 2 * G) refill(e);
          float4 v[UB][VPL];
          float w[UB];
#pragma unroll
          for (int u = 0; u < UB; ++u) {
            const int off = e + u - wbase;         // uniform across the group, < 2 * G
            const int j = __shfl_sync(gmask, (off & G) ? wi1 : wi0, off & (G - 1), G);
            if (W) w[u] = __shfl_sync(gmask, (off & G) ? ww1 : ww0, off & (G - 1), G);
            const float* __restrict__ rp = Fb + (size_t)j * ldf;
#pragma unroll
            for (int k = 0; k < VPL; ++k) v[u][k] = ldg4(rp + vcol[k]);
          }
#pragma unroll
          for (int u = 0; u < UB; ++u)
#pragma unroll
            for (int k = 0; k < VPL; ++k) {
              if (W) fma4(acc[k], w[u], v[u][k]); else add4(acc[k], v[u][k]);
            }
          e += UB;
        };
        while (e + U <= end) batch(std::integral_constant<int, U>{});
        if (TAILPRED) {
          // narrow rows: ONE predicated batch for the < U remaining edges instead of up to three dependent
          // power-of-two batches, of the smallest width (1, 2, 4, U) that holds them — a graph with many relations has
          // mostly one- and two-edge segments, and every unrolled slot costs issue cycles.  Masked edges add exact
          // zeros, the order of the sum is unchanged.
          auto tail = [&](auto ub) {
            constexpr int UB = decltype(ub)::value;
            if (e + UB > wbase + 2 * G) refill(e);
            const int n = end - e;
            float4 v[UB][VPL];
            float w[UB];
#pragma unroll
            for (int u = 0; u < UB; ++u) {
              const int off = e + u - wbase;
              const int j = __shfl_sync(gmask, (off & G) ? wi1 : wi0, off & (G - 1), G);
              if (W) w[u] = __shfl_sync(gmask, (off & G) ? ww1 : ww0, off & (G - 1), G);
              const float* __restrict__ rp = Fb + (size_t)j * ldf;
#pragma unroll
              for (int k = 0; k < VPL; ++k) v[u][k] = (u < n) ? ldg4(rp + vcol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < UB; ++u)
#pragma unroll
              for (int k = 0; k < VPL; ++k) {
                if (W) fma4(acc[k], (u < n) ? w[u] : 0.f, v[u][k]); else add4(acc[k], v[u][k]);
              }
            e = end;
          };
          const int n_left = end - e;
          if (n_left == 1) batch(std::integral_constant<int, 1>{});
          else if (n_left == 2) batch(std::integral_constant<int, (U >= 2 ? 2 : 1)>{});
          else if (n_left > 0 && n_left <= 4 && U > 4) tail(std::integral_constant<int, (U > 4 ? 4 : 1)>{});
          else if (n_left > 0) tail(std::integral_constant<int, U>{});
        } else {
          if (U > 4 && e + 4 <= end) batch(std::integral_constant<int, (U > 4 ? 4 : 1)>{});
          if (U > 2 && e + 2 <= end) batch(std::integral_constant<int, (U > 2 ? 2 : 1)>{});
          if (e < end) batch(std::integral_constant<int, 1>{});
        }
      }
      if (!W && len > 1) {
        const float c = (float)len;   // s / clamp(cnt, 1): a true division, like the reference
#pragma unroll
        for (int k = 0; k < VPL; ++k) acc[k] = div4(acc[k], c);
      }
      if (MIX == MIX_NONE) {
#pragma unroll
        for (int k = 0; k < VPL; ++k)
          if (act[k]) store_vec(p, LIST ? orow : row, r * p.block_stride + coff + vcol[k], acc[k]);
      } else if (MIX == MIX_SUM) {
#pragma unroll
        for (int k = 0; k < VPL; ++k) {
          if (chained) mix[0][k] = acc[k]; else add4(mix[0][k], acc[k]);
        }
      } else {
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          if (b < p.B) {
            const float c = s_comp[r * p.B + b];
#pragma unroll
            for (int k = 0; k < VPL; ++k) fma4(mix[b][k], c, acc[k]);
          }
        }
        if (with_gc) {
          // <h(i, r), P_b[i]> for every basis b: lane-partial dots, one fixed butterfly per b, lane 0 accumulates
          const float* __restrict__ Pr = p.dotP + row * p.ld_dotP;
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            if (b < p.B) {
              float dot = 0.f;
#pragma unroll
              for (int k = 0; k < VPL; ++k) {
                if (act[k]) {
                  const float4 q = ldg4(Pr + (size_t)b * p.block_stride + vcol[k]);
                  dot = fmaf(acc[k].x, q.x, dot); dot = fmaf(acc[k].y, q.y, dot);
                  dot = fmaf(acc[k].z, q.z, dot); dot = fmaf(acc[k].w, q.w, dot);
                }
              }
#pragma unroll
              for (int o = G >> 1; o; o >>= 1) dot += __shfl_xor_sync(gmask, dot, o, G);
              if (lane == 0) s_gc[(grp * R + r) * p.B + b] += dot;
            }
          }
        }
      }
    }
  }
  if (MIX != MIX_NONE) {
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      if (b < p.B) {
#pragma unroll
        for (int k = 0; k < VPL; ++k)
          if (act[k]) store_vec(p, row, b * p.block_stride + vcol[k], mix[b][k]);
      }
    }
    if (MP && MIX == MIX_SUM && p.mp_hi) {
      // the same row once more, masked and scaled, as the upstream layer's G planes (+ column sums)
#pragma unroll
      for (int k = 0; k < VPL; ++k) {
        if (act[k]) {
          const float4 m = ldg4(p.mp_mask + row * p.ld_mp_mask + vcol[k]);
          float4 v = scale4(mix[0][k], p.mp_scale);
          if (!(m.x > 0.f)) v.x = 0.f;
          if (!(m.y > 0.f)) v.y = 0.f;
          if (!(m.z > 0.f)) v.z = 0.f;
          if (!(m.w > 0.f)) v.w = 0.f;
          store_vec_to(p.mp_hi, p.mp_lo, p.ld_mp, p.mp_lo ? 2 : 1, row, vcol[k], v);
          if (with_cs) *reinterpret_cast<float4*>(s_comp + grp * d + vcol[k]) = v;
        }
      }
    }
  }
  }  // row < n_rows
  if (with_cs) {
    // the block's column sums = its groups' rows in group order (deterministic)
    __syncthreads();
    for (int t = threadIdx.x; t < p.d; t += 256) {
      float sum = s_comp[t];
      for (int g = 1; g < GROUPS; ++g) sum += s_comp[g * p.d + t];
      p.mp_colsum[(size_t)blockIdx.x * p.d + t] = sum;
    }
  }
  if (with_gc) {
    // the block's partial = its groups' sums in group order (deterministic)
    __syncthreads();
    const int RB = p.R * p.B;
    for (int t = threadIdx.x; t < RB; t += 256) {
      float sum = s_gc[t];
      for (int g = 1; g < GROUPS; ++g) sum += s_gc[g * RB + t];
      p.gc_partial[(size_t)blockIdx.x * RB + t] = sum;
    }
  }
}

// ---- hub finish: one G-lane group per hub ROW (led by the row's first hub segment) -------------------------
// Runs after hub_partial_kernel (chunk partials) and after the row walk (which skipped the hub segments): sums each
// hub segment's partials in chunk order and writes its block (MIX_NONE) or adds the row's hub segments to the row the
// walk already wrote (MIX_SUM).  Fixed order everywhere: deterministic.
template <int G, int VPL, int MIX, bool W>
__global__ void __launch_bounds__(256) hub_finish_kernel(const AggParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  const int lane = threadIdx.x % G;
  const int h0 = blockIdx.x * GROUPS + threadIdx.x / G;
  if (h0 >= p.n_hubs) return;
  const int R = p.R, d = p.d, nvec = p.d >> 2;
  const int key0 = __ldg(p.hub_keys + h0);
  const int64_t row = key0 / R;
  if (h0 > 0 && __ldg(p.hub_keys + h0 - 1) / R == row) return;      // not the row's first hub segment
  bool act[VPL];
  int vcol[VPL];
  float4 total[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    act[k] = vi < nvec;
    vcol[k] = act[k] ? vi * 4 : 0;
    total[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  constexpr int U = (VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8);
  for (int h = h0; h < p.n_hubs; ++h) {
    const int key = __ldg(p.hub_keys + h);
    if (key / R != row) break;
    const int r = key - (int)row * R;
    float4 acc[VPL];
#pragma unroll
    for (int k = 0; k < VPL; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int c0 = __ldg(p.hub_chunk_ptr + h), c1 = __ldg(p.hub_chunk_ptr + h + 1);
    int c = c0;
    for (; c + U <= c1; c += U) {                    // loads U chunks ahead, adds strictly in chunk order
      float4 v[U][VPL];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int k = 0; k < VPL; ++k) v[u][k] = *reinterpret_cast<const float4*>(p.partials + (size_t)(c + u) * d + vcol[k]);
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int k = 0; k < VPL; ++k) add4(acc[k], v[u][k]);
    }
    for (; c < c1; ++c) {
#pragma unroll
      for (int k = 0; k < VPL; ++k) add4(acc[k], *reinterpret_cast<const float4*>(p.partials + (size_t)c * d + vcol[k]));
    }
    if (!W) {
      const float len = (float)(__ldg(p.rowptr + key + 1) - __ldg(p.rowptr + key));
#pragma unroll
      for (int k = 0; k < VPL; ++k) acc[k] = div4(acc[k], len);
    }
    if (MIX == MIX_NONE) {
#pragma unroll
      for (int k = 0; k < VPL; ++k)
        if (act[k]) store_vec(p, row, r * p.block_stride + vcol[k], acc[k]);
    } else {
#pragma unroll
      for (int k = 0; k < VPL; ++k) add4(total[k], acc[k]);
    }
  }
  if (MIX == MIX_SUM) {
    float* o = reinterpret_cast<float*>(p.O) + row * p.ldo;      // fp32 output (checked by the host)
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      if (act[k]) {
        float4 cur = *reinterpret_cast<const float4*>(o + vcol[k]);
        add4(cur, total[k]);
        *reinterpret_cast<float4*>(o + vcol[k]) = cur;
      }
    }
  }
}

// ---- hub finish of the LISTED walk: one G-lane group per hub segment of a listed row ---------------------------------
// The listed walk is latency bound and so is its hub pass (few long rows / a few hundred chunks): run side by side they
// overlap almost completely.  The walk then skips the hub segments (skip_hubs) and this kernel adds them afterwards — the
// same additions in the same order as the walk's own hub branch (chunk partials in chunk order, one true division).
template <int G, int VPL>
__global__ void __launch_bounds__(256) hub_finish_list_kernel(const AggParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  const int lane = threadIdx.x % G;
  const int h = blockIdx.x * GROUPS + threadIdx.x / G;
  if (h >= p.n_hubs) return;
  const int key = __ldg(p.hub_keys + h);
  const int64_t row = key / p.R;
  const int r = key - (int)row * p.R;
  const int64_t orow = __ldg(p.hub_filter + row);
  if (orow == p.hub_unlisted) return;
  const int d = p.d, nvec = p.d >> 2;
  const int c0 = __ldg(p.hub_chunk_ptr + h), c1 = __ldg(p.hub_chunk_ptr + h + 1);
  const float len = (float)(__ldg(p.rowptr + key + 1) - __ldg(p.rowptr + key));
  constexpr int U = (VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8);
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    if (vi >= nvec) continue;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int c = c0;
    for (; c + U <= c1; c += U) {                    // loads U chunks ahead, adds strictly in chunk order
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = *reinterpret_cast<const float4*>(p.partials + (size_t)(c + u) * d + vi * 4);
#pragma unroll
      for (int u = 0; u < U; ++u) add4(acc, v[u]);
    }
    for (; c < c1; ++c) add4(acc, *reinterpret_cast<const float4*>(p.partials + (size_t)c * d + vi * 4));
    acc = div4(acc, len);
    store_vec(p, orow, r * p.block_stride + vi * 4, acc);
  }
}

// ---- bf16 features (the "bf16-transform" mode gathers a bf16 copy of the layer input: half the L2 / HBM bytes of the
// dominant kernel; sums, means and hub partials stay fp32) -------------------------------------------------------------
// Forward, unmixed form only.  A lane holds VPL vectors of EIGHT columns (one 128-bit load = 8 bf16), so a 256-wide row is
// one load per lane; the result goes straight into the bf16 hi plane of the transform's operand (16-byte stores).
struct f8 { float v[8]; };
__device__ __forceinline__ void ld_bf8(const __nv_bfloat16* p, uint4& raw) { raw = __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void acc_bf8(f8& a, const uint4& r) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    unsigned long long acc2 = pack2(a.v[2 * i], a.v[2 * i + 1]);
    const unsigned long long x2 = pack2(__uint_as_float(w[i] << 16), __uint_as_float(w[i] & 0xffff0000u));
    asm("add.rn.f32x2 %0, %0, %1;" : "+l"(acc2) : "l"(x2));
    unpack2(acc2, a.v[2 * i], a.v[2 * i + 1]);
  }
}
__device__ __forceinline__ uint4 pack_bf8(const f8& a) {
  uint4 o;
  __nv_bfloat162 t;
  t = __floats2bfloat162_rn(a.v[0], a.v[1]); o.x = *reinterpret_cast<uint32_t*>(&t);
  t = __floats2bfloat162_rn(a.v[2], a.v[3]); o.y = *reinterpret_cast<uint32_t*>(&t);
  t = __floats2bfloat162_rn(a.v[4], a.v[5]); o.z = *reinterpret_cast<uint32_t*>(&t);
  t = __floats2bfloat162_rn(a.v[6], a.v[7]); o.w = *reinterpret_cast<uint32_t*>(&t);
  return o;
}

// fma of 8 bf16 features by an edge weight (the weighted form: unit weights of a sum layer give the sum's bits)
__device__ __forceinline__ void fma_bf8(f8& a, float w, const uint4& r) {
  const uint32_t x[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    a.v[2 * i] = fmaf(w, __uint_as_float(x[i] << 16), a.v[2 * i]);
    a.v[2 * i + 1] = fmaf(w, __uint_as_float(x[i] & 0xffff0000u), a.v[2 * i + 1]);
  }
}

template <int G, int VPL, bool W = false>
__global__ void __launch_bounds__(256) hub_partial_bf16_kernel(const AggParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  __shared__ float red[GROUPS][G * VPL * 8];
  const __nv_bfloat16* __restrict__ F = reinterpret_cast<const __nv_bfloat16*>(p.F);
  const int chunk = blockIdx.x;
  const int4 t = __ldg(reinterpret_cast<const int4*>(p.chunk_table) + chunk);
  const int key = t.x;
  if (p.hub_filter && __ldg(p.hub_filter + key / p.R) == p.hub_unlisted) return;     // (block-uniform) nobody reads this row
  const int seg_beg = __ldg(p.rowptr + key), seg_end = __ldg(p.rowptr + key + 1);
  const int c_beg = seg_beg + (chunk - t.y) * kHubChunk;
  const int c_end = min(c_beg + kHubChunk, seg_end);
  const int nvec = p.d >> 3;
  const int lane = threadIdx.x % G, grp = threadIdx.x / G;
  constexpr int PER = kHubChunk / GROUPS;
  const int g_beg = c_beg + grp * PER, g_end = min(g_beg + PER, c_end);
  f8 acc[VPL];
  int vcol[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[k].v[i] = 0.f;
    const int vi = k * G + lane;
    vcol[k] = vi < nvec ? vi * 8 : 0;
  }
  constexpr int U0 = VPL >= 2 ? 4 : 8;
  constexpr int U = U0 < PER ? U0 : PER;
  static_assert(PER <= G, "a group's slice of a hub chunk must fit its lanes");
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G));
  const int my_j = (lane < PER && g_beg + lane < g_end) ? __ldg(p.idx + g_beg + lane) : 0;     // one coalesced index load
  const float my_w = (W && lane < PER && g_beg + lane < g_end) ? __ldg(p.edge_w + g_beg + lane) : 0.f;
  int e = g_beg;
  for (; e + U <= g_end; e += U) {
    uint4 v[U][VPL];
    float w[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = __shfl_sync(gmask, my_j, e + u - g_beg, G);
      if (W) w[u] = __shfl_sync(gmask, my_w, e + u - g_beg, G);
#pragma unroll
      for (int k = 0; k < VPL; ++k) ld_bf8(F + (size_t)j * p.ldf + vcol[k], v[u][k]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int k = 0; k < VPL; ++k) {
        if (W) fma_bf8(acc[k], w[u], v[u][k]); else acc_bf8(acc[k], v[u][k]);
      }
  }
  for (; e < g_end; ++e) {
    const int j = __shfl_sync(gmask, my_j, e - g_beg, G);
    const float wv = W ? __shfl_sync(gmask, my_w, e - g_beg, G) : 1.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      uint4 r; ld_bf8(F + (size_t)j * p.ldf + vcol[k], r);
      if (W) fma_bf8(acc[k], wv, r); else acc_bf8(acc[k], r);
    }
  }
#pragma unroll
  for (int k = 0; k < VPL; ++k)
#pragma unroll
    for (int i = 0; i < 8; ++i) red[grp][(k * G + lane) * 8 + i] = acc[k].v[i];
  __syncthreads();
  for (int c = threadIdx.x; c < p.d; c += 256) {
    float sum = red[0][c];
    for (int g = 1; g < GROUPS; ++g) sum += red[g][c];       // fixed order over the groups
    p.partials[(size_t)chunk * p.d + c] = sum;
  }
}

template <int G, int VPL, bool LIST = false, bool W = false>
__global__ void __launch_bounds__(256, (VPL == 1 ? 4 : 3) - (W ? 1 : 0)) aggregate_rows_bf16_kernel(const AggParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  constexpr int U0 = VPL >= 2 ? 4 : 8;
  constexpr int U = U0 < G ? U0 : G;
  const __nv_bfloat16* __restrict__ F = reinterpret_cast<const __nv_bfloat16*>(p.F);
  __nv_bfloat16* __restrict__ O = reinterpret_cast<__nv_bfloat16*>(p.O);
  const int lane = threadIdx.x % G, grp = threadIdx.x / G;
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G));
  int64_t row = p.row_begin + (int64_t)blockIdx.x * GROUPS + grp;
  if (row >= p.row_end) return;
  int64_t orow = row;                                 // LIST: the output row is the row's first list position
  if (LIST) {
    if (row >= p.list_walkers) {                      // duplicate or padding position: an all-zero operand row
      const int64_t c = row - p.list_walkers;
      const bool fill = c >= p.n_list || __ldg(p.hub_filter + __ldg(p.list + c)) != (int32_t)c;
      if (fill && blockIdx.y == 0 && blockIdx.z == 0) {
        const int nblk = p.R + (p.root_rows ? 1 : 0);
        for (int b = 0; b < nblk; ++b)
          for (int vi = lane; vi < ((p.d * (int)gridDim.y) >> 3); vi += G)
            *reinterpret_cast<uint4*>(O + c * p.ldo + b * p.block_stride + vi * 8) = make_uint4(0u, 0u, 0u, 0u);
      }
      return;
    }
    if (p.list_by_rows) {
      if (p.row_order) row = __ldg(p.row_order + row);
      orow = __ldg(p.hub_filter + row);
      if (orow == p.hub_unlisted) return;
    } else {
      row = __ldg(p.list + orow);
      if (__ldg(p.hub_filter + row) != (int32_t)orow) return;
    }
  } else if (p.row_order) {
    row = __ldg(p.row_order + row);
  }
  const int R = p.R, nvec = p.d >> 3;
  const int coff = LIST ? (int)blockIdx.y * p.d : 0;                        // this block's column slice
  const int pstride = LIST ? p.d * (int)gridDim.y : p.d;                    // row stride of the hub partials (full width)
  int r_lo = 0, r_hi = R;                                                   // this block's relation range
  if (LIST) {
    const int per = (R + (int)gridDim.z - 1) / (int)gridDim.z;
    r_lo = (int)blockIdx.z * per;
    r_hi = min(R, r_lo + per);
  }
  F += coff;
  const int64_t key0 = row * R;
  const int32_t* __restrict__ rowptr = p.rowptr + key0;
  const int32_t* __restrict__ idx = p.idx;
  const int64_t ldf = p.ldf;
  bool act[VPL];
  int vcol[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    act[k] = vi < nvec;
    vcol[k] = act[k] ? vi * 8 : 0;
  }
  if (p.root_rows && (!LIST || blockIdx.z == 0)) {    // self-loop block: the bf16 copy of x[row] as it is
    const __nv_bfloat16* __restrict__ xr = reinterpret_cast<const __nv_bfloat16*>(p.root_rows) + row * p.ld_root + coff;
#pragma unroll
    for (int k = 0; k < VPL; ++k)
      if (act[k]) *reinterpret_cast<uint4*>(O + (LIST ? orow : row) * p.ldo + R * p.block_stride + coff + vcol[k]) = __ldg(reinterpret_cast<const uint4*>(xr + vcol[k]));
  }
  const int row_end = __ldg(rowptr + R);
  int wbase = -(1 << 30), wi0 = 0, wi1 = 0;
  float ww0 = 1.f, ww1 = 1.f;
  auto refill = [&](int e) {
    wbase = e;
    wi0 = (e + lane < row_end) ? __ldg(idx + e + lane) : 0;
    wi1 = (e + G + lane < row_end) ? __ldg(idx + e + G + lane) : 0;
    if (W) {
      ww0 = (e + lane < row_end) ? __ldg(p.edge_w + e + lane) : 0.f;
      ww1 = (e + G + lane < row_end) ? __ldg(p.edge_w + e + G + lane) : 0.f;
    }
  };
  for (int rbase = r_lo; rbase < r_hi; rbase += G) {
    const int rl = rbase + lane;
    const int my_beg = (rl < r_hi) ? __ldg(rowptr + rl) : 0;
    const int my_end = (rl < r_hi) ? __ldg(rowptr + rl + 1) : 0;
    const int rcount = min(G, r_hi - rbase);
    for (int rr = 0; rr < rcount; ++rr) {
      const int r = rbase + rr;
      const int beg = __shfl_sync(gmask, my_beg, rr, G);
      const int end = __shfl_sync(gmask, my_end, rr, G);
      const int len = end - beg;
      f8 acc[VPL];
#pragma unroll
      for (int k = 0; k < VPL; ++k)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[k].v[i] = 0.f;
      if (len > p.hub_threshold) {
        const int key = (int)(key0 + r);
        int lo = 0, hi = p.n_hubs;
        while (hi - lo > 1) {
          int mid = (lo + hi) >> 1;
          if (__ldg(p.hub_keys + mid) <= key) lo = mid; else hi = mid;
        }
        const int c0 = __ldg(p.hub_chunk_ptr + lo), c1 = __ldg(p.hub_chunk_ptr + lo + 1);
        for (int c = c0; c < c1; ++c) {               // chunk partials (fp32), strictly in chunk order
#pragma unroll
          for (int k = 0; k < VPL; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(p.partials + (size_t)c * pstride + coff + vcol[k]);
            const float4 b = *reinterpret_cast<const float4*>(p.partials + (size_t)c * pstride + coff + vcol[k] + 4);
            acc[k].v[0] += a.x; acc[k].v[1] += a.y; acc[k].v[2] += a.z; acc[k].v[3] += a.w;
            acc[k].v[4] += b.x; acc[k].v[5] += b.y; acc[k].v[6] += b.z; acc[k].v[7] += b.w;
          }
        }
      } else if (len > 0) {
        int e = beg;
        auto batch = [&](auto ub) {
          constexpr int UB = decltype(ub)::value;
          if (e + UB > wbase + 2 * G) refill(e);
          uint4 v[UB][VPL];
          float w[UB];
#pragma unroll
          for (int u = 0; u < UB; ++u) {
            const int off = e + u - wbase;
            const int j = __shfl_sync(gmask, (off & G) ? wi1 : wi0, off & (G - 1), G);
            if (W) w[u] = __shfl_sync(gmask, (off & G) ? ww1 : ww0, off & (G - 1), G);
#pragma unroll
            for (int k = 0; k < VPL; ++k) ld_bf8(F + (size_t)j * ldf + vcol[k], v[u][k]);
          }
#pragma unroll
          for (int u = 0; u < UB; ++u)
#pragma unroll
            for (int k = 0; k < VPL; ++k) {
              if (W) fma_bf8(acc[k], w[u], v[u][k]); else acc_bf8(acc[k], v[u][k]);
            }
          e += UB;
        };
        while (e + U <= end) batch(std::integral_constant<int, U>{});
        if (U > 4 && e + 4 <= end) batch(std::integral_constant<int, (U > 4 ? 4 : 1)>{});
        if (U > 2 && e + 2 <= end) batch(std::integral_constant<int, (U > 2 ? 2 : 1)>{});
        if (e < end) batch(std::integral_constant<int, 1>{});
      }
      if (!W && len > 1) {
        const float c = (float)len;                   // s / clamp(cnt, 1): a true division, like the reference
        const float rc = __frcp_rn(c);
#pragma unroll
        for (int k = 0; k < VPL; ++k)
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[k].v[i] = div_by(acc[k].v[i], c, rc);
      }
#pragma unroll
      for (int k = 0; k < VPL; ++k)
        if (act[k]) *reinterpret_cast<uint4*>(O + (LIST ? orow : row) * p.ldo + r * p.block_stride + coff + vcol[k]) = pack_bf8(acc[k]);
    }
  }
}

template <int G, int VPL>
static int launch_agg_bf16(AggParams p, int n_chunks, cudaStream_t st) {
  constexpr int GROUPS = 256 / G;
  if (!p.range_mode) { p.row_begin = 0; p.row_end = p.n_rows; }
  if (n_chunks > 0 && !p.no_hub_pass) {
    if (p.edge_w) RGCN_CUDA(launch_pdl(hub_partial_bf16_kernel<G, VPL, true>, dim3(n_chunks), dim3(256), 0, st, p));
    else RGCN_CUDA(launch_pdl(hub_partial_bf16_kernel<G, VPL>, dim3(n_chunks), dim3(256), 0, st, p));
    RGCN_LAUNCH_CHECK();
  }
  const int64_t n_walk = p.row_end - p.row_begin;
  if (n_walk <= 0) return RGCN_OK;
  const dim3 lgrid((unsigned)((n_walk + GROUPS - 1) / GROUPS), (unsigned)(p.list_slices > 0 ? p.list_slices : 1),
                   (unsigned)(p.list_rsplit > 0 ? p.list_rsplit : 1));
  const dim3 grid((unsigned)((n_walk + GROUPS - 1) / GROUPS));
  // a weighted CSR (RGCNConv(aggr='sum'): unit weights) takes the weighted instantiations, the mean's are unchanged
  if (p.list && p.edge_w) RGCN_CUDA(launch_pdl(aggregate_rows_bf16_kernel<G, VPL, true, true>, lgrid, dim3(256), 0, st, p));
  else if (p.list) RGCN_CUDA(launch_pdl(aggregate_rows_bf16_kernel<G, VPL, true>, lgrid, dim3(256), 0, st, p));
  else if (p.edge_w) RGCN_CUDA(launch_pdl(aggregate_rows_bf16_kernel<G, VPL, false, true>, grid, dim3(256), 0, st, p));
  else RGCN_CUDA(launch_pdl(aggregate_rows_bf16_kernel<G, VPL>, grid, dim3(256), 0, st, p));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

// side stream + events for the fork / join of the hub pass (one set per device, created on first use)
struct ForkJoin {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
static ForkJoin* fork_join() {
  static ForkJoin fj[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  ForkJoin& f = fj[dev];
  if (!f.side) {
    if (cudaStreamCreateWithFlags(&f.side, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&f.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&f.join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
  }
  return &f;
}
// the side stream if it exists already or may be created now (never while a stream capture is in progress)
static ForkJoin* fork_join_existing(cudaStream_t st) {
  static ForkJoin* made[64] = {nullptr};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (made[dev]) return made[dev];
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return nullptr;
  made[dev] = fork_join();
  return made[dev];
}
// Opt-in (RGCN_OVERLAP_HUBS=1).  Measured on the B200 it LOSES against the plain order hub pass -> row walk
// (cfg2 d = 256 forward 93 vs 75 us, step 0.595 vs 0.533 ms): the two latency-bound kernels slow each other down and
// the finish kernel adds a serial tail, so the default stays the single-stream order.
static bool overlap_hubs_enabled() {
  const char* e = getenv("RGCN_OVERLAP_HUBS");
  return e && e[0] == '1';
}

template <int G, int VPL, int MIX, bool W>
static int launch_agg_overlapped(AggParams p, int n_chunks, cudaStream_t st) {
  if (!p.range_mode) { p.row_begin = 0; p.row_end = p.n_rows; }
  // hub chunks on a side stream, concurrently with the row walk (which skips the hub segments); then the finish
  // kernel.  Inside a stream capture the fork / join becomes two parallel branches of the graph.
  constexpr int GROUPS = 256 / G;
  ForkJoin* fj = fork_join();
  if (!fj) { set_error("aggregate: could not create the side stream for the hub pass"); return RGCN_ECUDA; }
  p.skip_hubs = 1;
  RGCN_CUDA(cudaEventRecord(fj->fork, st));
  RGCN_CUDA(cudaStreamWaitEvent(fj->side, fj->fork, 0));
  hub_partial_kernel<G, VPL, W><<<n_chunks, 256, 0, fj->side>>>(p);
  RGCN_LAUNCH_CHECK();
  RGCN_CUDA(cudaEventRecord(fj->join, fj->side));
  const unsigned grid = (unsigned)((p.n_rows + GROUPS - 1) / GROUPS);
  RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX, W>, dim3(grid), dim3(256), 0, st, p));
  RGCN_LAUNCH_CHECK();
  RGCN_CUDA(cudaStreamWaitEvent(st, fj->join, 0));
  hub_finish_kernel<G, VPL, MIX, W><<<(unsigned)((p.n_hubs + GROUPS - 1) / GROUPS), 256, 0, st>>>(p);
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

template <int G, int VPL>
static int launch_agg(const AggParams& p_in, int mix, int n_chunks, cudaStream_t st) {
  constexpr int GROUPS = 256 / G;
  AggParams p = p_in;
  if (!p.range_mode) { p.row_begin = 0; p.row_end = p.n_rows; }
  if (p.no_hub_pass) n_chunks = 0;
  const int64_t n_walk = p.row_end - p.row_begin;
  if (!p.list && !p.slot && !p.mp_hi && n_chunks > 0 && p.n_rows > 0 && n_walk == p.n_rows && mix != MIX_BASIS && overlap_hubs_enabled() && (mix == MIX_NONE || p.out_mode == 0)) {
    const bool w = p.edge_w != nullptr;
    if (mix == MIX_NONE)
      return w ? launch_agg_overlapped<G, VPL, MIX_NONE, true>(p, n_chunks, st) : launch_agg_overlapped<G, VPL, MIX_NONE, false>(p, n_chunks, st);
    return w ? launch_agg_overlapped<G, VPL, MIX_SUM, true>(p, n_chunks, st) : launch_agg_overlapped<G, VPL, MIX_SUM, false>(p, n_chunks, st);
  }
  if (p.list) {
    // listed-rows walk: forward, unmixed (the last layer of a link-prediction step); a weighted CSR (RGCNConv(aggr='sum'):
    // unit weights) takes the weighted instantiations, the mean's are unchanged
    if (mix != MIX_NONE || p.slot || p.mp_hi) { set_error("aggregate: the listed-rows walk serves the unmixed forward only"); return RGCN_EINVAL; }
    const dim3 lgrid((unsigned)((n_walk + GROUPS - 1) / GROUPS), (unsigned)(p.list_slices > 0 ? p.list_slices : 1),
                     (unsigned)(p.list_rsplit > 0 ? p.list_rsplit : 1));
    ForkJoin* fj = (p.list_overlap_hubs && !p.edge_w && n_chunks > 0 && n_walk > 0 && p.list_slices <= 1) ? fork_join_existing(st) : nullptr;
    if (fj) {
      // hub chunks on the side stream, the walk (without the hub segments) on this one, then the finish kernel
      RGCN_CUDA(cudaEventRecord(fj->fork, st));
      RGCN_CUDA(cudaStreamWaitEvent(fj->side, fj->fork, 0));
      hub_partial_kernel<G, VPL, false><<<n_chunks, 256, 0, fj->side>>>(p);
      RGCN_LAUNCH_CHECK();
      RGCN_CUDA(cudaEventRecord(fj->join, fj->side));
      p.skip_hubs = 1;
      RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_NONE, false, false, false, true>, lgrid, dim3(256), 0, st, p));
      RGCN_LAUNCH_CHECK();
      RGCN_CUDA(cudaStreamWaitEvent(st, fj->join, 0));
      hub_finish_list_kernel<G, VPL><<<(unsigned)((p.n_hubs + GROUPS - 1) / GROUPS), 256, 0, st>>>(p);
      RGCN_LAUNCH_CHECK();
      return RGCN_OK;
    }
    if (n_chunks > 0) {
      if (p.edge_w) RGCN_CUDA(launch_pdl(hub_partial_kernel<G, VPL, true>, dim3(n_chunks), dim3(256), 0, st, p));
      else RGCN_CUDA(launch_pdl(hub_partial_kernel<G, VPL, false>, dim3(n_chunks), dim3(256), 0, st, p));
      RGCN_LAUNCH_CHECK();
    }
    if (n_walk <= 0) return RGCN_OK;
    if (p.edge_w) RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_NONE, true, false, false, true>, lgrid, dim3(256), 0, st, p));
    else RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_NONE, false, false, false, true>, lgrid, dim3(256), 0, st, p));
    RGCN_LAUNCH_CHECK();
    return RGCN_OK;
  }
  if (p.slot) {
    // row-sparse gather: backward form only (summed relations, weighted edges)
    if (mix != MIX_SUM || !p.edge_w) { set_error("aggregate: the row-sparse gather serves the backward walk only"); return RGCN_EINVAL; }
    if (n_chunks > 0) {
      RGCN_CUDA(launch_pdl(hub_partial_kernel<G, VPL, true, true>, dim3(n_chunks), dim3(256), 0, st, p));
      RGCN_LAUNCH_CHECK();
    }
    if (n_walk <= 0) return RGCN_OK;
    const dim3 sgrid((unsigned)((n_walk + GROUPS - 1) / GROUPS));
    if (p.mp_hi) RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_SUM, true, true, true>, sgrid, dim3(256),
                                      p.mp_colsum ? (size_t)GROUPS * p.d * sizeof(float) : 0, st, p));
    else if (p.row_flag) RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_SUM, true, true, false, false, true>, sgrid, dim3(256), 0, st, p));
    else RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_SUM, true, true>, sgrid, dim3(256), 0, st, p));
    RGCN_LAUNCH_CHECK();
    return RGCN_OK;
  }
  if (n_chunks > 0) {
    if (p.edge_w) RGCN_CUDA(launch_pdl(hub_partial_kernel<G, VPL, true>, dim3(n_chunks), dim3(256), 0, st, p));
    else RGCN_CUDA(launch_pdl(hub_partial_kernel<G, VPL, false>, dim3(n_chunks), dim3(256), 0, st, p));
    RGCN_LAUNCH_CHECK();
  }
  if (n_walk <= 0) return RGCN_OK;
  const unsigned grid = (unsigned)((n_walk + GROUPS - 1) / GROUPS);
  const bool w = p.edge_w != nullptr;
  const size_t sm = (size_t)p.R * p.B * sizeof(float) * (p.dotP ? 1 + GROUPS : 1);
  if (mix == MIX_NONE) {
    if (w) RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_NONE, true>, dim3(grid), dim3(256), 0, st, p));
    else RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_NONE, false>, dim3(grid), dim3(256), 0, st, p));
  } else if (mix == MIX_SUM) {
    if (p.mp_hi) {
      if (!w) { set_error("aggregate: the masked-planes output serves the weighted (backward) walk"); return RGCN_EINVAL; }
      RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_SUM, true, false, true>, dim3(grid), dim3(256),
                           p.mp_colsum ? (size_t)GROUPS * p.d * sizeof(float) : 0, st, p));
    } else if (w) RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_SUM, true>, dim3(grid), dim3(256), 0, st, p));
    else RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_SUM, false>, dim3(grid), dim3(256), 0, st, p));
  } else {
    if (w) RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_BASIS, true>, dim3(grid), dim3(256), sm, st, p));
    else RGCN_CUDA(launch_pdl(aggregate_rows_kernel<G, VPL, MIX_BASIS, false>, dim3(grid), dim3(256), sm, st, p));
  }
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

static int dispatch_agg(const AggParams& p, int mix, int n_chunks, cudaStream_t st) {
  const int nvec = p.d >> 2;
  if (nvec <= 4) return launch_agg<4, 1>(p, mix, n_chunks, st);
  if (nvec <= 8) return launch_agg<8, 1>(p, mix, n_chunks, st);
  if (nvec <= 16) return launch_agg<16, 1>(p, mix, n_chunks, st);
  if (nvec <= 32) return launch_agg<32, 1>(p, mix, n_chunks, st);
  if (nvec <= 64) return launch_agg<32, 2>(p, mix, n_chunks, st);
  if (nvec <= 128) return launch_agg<32, 4>(p, mix, n_chunks, st);
  return launch_agg<32, 8>(p, mix, n_chunks, st);
}

static int check_common(const rgcn_csr_t* g, const float* F, int64_t ldf, int32_t d, const void* ws,
                        size_t ws_bytes) {
  RGCN_CHECK_ARG(g && g->rowptr && (g->idx || g->E == 0), "aggregate: null CSR arrays");
  RGCN_CHECK_ARG(g->R >= 1 && g->n_rows >= 0, "aggregate: bad n_rows/R");
  RGCN_CHECK_ARG(g->hub_threshold >= 1, "aggregate: hub_threshold must be the (positive) threshold the hub plan was made with");
  RGCN_CHECK_ARG(d >= 4 && d <= 1024 && d % 4 == 0, "aggregate: feature width d=%d must be a multiple of 4 in [4,1024]", d);
  RGCN_CHECK_ARG(F && ldf % 4 == 0 && ((uintptr_t)F & 15) == 0, "aggregate: feature matrix must be 16-byte aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(g->n_chunks == 0 || (g->hub_keys && g->hub_chunk_ptr && g->n_hubs > 0 && g->chunk_table &&
                                      ((uintptr_t)g->chunk_table & 15) == 0), "aggregate: hub plan missing");
  if (g->n_chunks > 0 && (!ws || ws_bytes < (size_t)g->n_chunks * d * sizeof(float))) {
    set_error("aggregate: workspace too small (%zu < %zu)", ws_bytes, (size_t)g->n_chunks * d * sizeof(float));
    return RGCN_EWORKSPACE;
  }
  return RGCN_OK;
}

}  // namespace rgcn

using namespace rgcn;

extern "C" size_t rgcn_aggregate_workspace_bytes(const rgcn_csr_t* g, int32_t d) {
  if (!g) return 0;
  return align_up((size_t)g->n_chunks * (size_t)d * sizeof(float), 256);
}

// The basis-mixing walk keeps B accumulators per lane.  With the coefficient-gradient side output it runs once per
// slice of kBasisSlice feature columns (one 128-bit vector per lane and basis): measured on cfg3, d = 256, that walk is
// faster in two slices (2 x 1.35 ms) than in one with 150 registers, while the plain mixing walk is faster unsliced
// (1.04 ms against 2 x 0.78 ms).
constexpr int kBasisSlice = 128;

static int64_t agg_blocks(int64_t n_rows, int d) {
  const int nvec = d >> 2;
  const int G = nvec <= 4 ? 4 : nvec <= 8 ? 8 : nvec <= 16 ? 16 : 32;
  const int groups = 256 / G;
  return (n_rows + groups - 1) / groups;
}

// rows of R * B floats the coefficient-gradient side output of rgcn_aggregate_fwd writes
extern "C" int64_t rgcn_aggregate_blocks(const rgcn_csr_t* g, int32_t d) {
  if (!g || d < 4) return 0;
  int64_t total = 0;
  for (int c0 = 0; c0 < d; c0 += kBasisSlice) total += agg_blocks(g->n_rows, d - c0 < kBasisSlice ? d - c0 : kBasisSlice);
  return total;
}

extern "C" int rgcn_aggregate_fwd(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d,
                                  const float* comp, int32_t B, void* H, void* H_lo, int64_t ldh, int32_t out_mode,
                                  const float* dot_p, int64_t ld_dot_p, float* gc_partial,
                                  const float* x_root, int64_t ld_x_root,
                                  void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  int rc = check_common(g, X, ldx, d, workspace, workspace_bytes);
  if (rc) return rc;
  RGCN_CHECK_ARG(!x_root || (!comp && ((uintptr_t)x_root & 15) == 0 && ld_x_root % 4 == 0),
                 "aggregate_fwd: x_root (appended self-loop block) needs the unmixed form and 16-byte aligned rows");
  RGCN_CHECK_ARG(!dot_p || (comp && B <= kMaxBasis && gc_partial && ((uintptr_t)dot_p & 15) == 0 && ld_dot_p % 4 == 0),
                 "aggregate_fwd: the coefficient-gradient side output needs comp, B <= %d, aligned P and a partial buffer", kMaxBasis);
  RGCN_CHECK_ARG(out_mode >= 0 && out_mode <= 2, "aggregate_fwd: out_mode must be 0 (fp32), 1 (bf16) or 2 (bf16 hi+lo)");
  RGCN_CHECK_ARG(H && ((uintptr_t)H & (out_mode ? 7 : 15)) == 0 && ldh % 4 == 0, "aggregate_fwd: output must be aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(out_mode != 2 || (H_lo && ((uintptr_t)H_lo & 7) == 0), "aggregate_fwd: out_mode 2 needs the lo plane");
  RGCN_CHECK_ARG(!comp || (B >= 1), "aggregate_fwd: bad number of bases");
  AggParams p{};
  p.rowptr = g->rowptr; p.idx = g->idx; p.edge_w = g->w;
  p.hub_keys = g->hub_keys; p.hub_chunk_ptr = g->hub_chunk_ptr; p.n_hubs = g->n_hubs; p.chunk_table = g->chunk_table;
  p.row_order = g->row_order; p.hub_threshold = g->hub_threshold;
  p.n_rows = g->n_rows; p.R = g->R;
  p.F = X; p.ldf = ldx; p.src_rel_stride = 0; p.d = d; p.block_stride = d;
  p.O = H; p.O_lo = H_lo; p.ldo = ldh; p.out_mode = out_mode; p.partials = (float*)workspace;
  p.dotP = dot_p; p.ld_dotP = ld_dot_p; p.gc_partial = gc_partial;
  p.root_rows = x_root; p.ld_root = ld_x_root;
  cudaStream_t st = (cudaStream_t)stream;
  if (!comp) return dispatch_agg(p, MIX_NONE, g->n_chunks, st);
  // basis blocks are produced kMaxBasis at a time (registers hold the B accumulators), feature columns in slices
  // of kBasisSlice; every (basis group, slice) launch has its own region of the partial buffers
  int64_t gc_row = 0;
  const int slice = dot_p ? kBasisSlice : d;
  for (int b0 = 0; b0 < B; b0 += kMaxBasis) {
    for (int c0 = 0; c0 < d; c0 += slice) {
      const int dc = d - c0 < slice ? d - c0 : slice;
      AggParams q = p;
      q.comp = comp + b0; q.ldcomp = B; q.B = (B - b0 < kMaxBasis) ? (B - b0) : kMaxBasis;
      q.F = X + c0; q.d = dc;
      const size_t off = (size_t)b0 * d + c0;
      q.O = out_mode ? (void*)((__nv_bfloat16*)H + off) : (void*)((float*)H + off);
      if (out_mode == 2) q.O_lo = (void*)((__nv_bfloat16*)H_lo + off);
      q.partials = (float*)workspace + (size_t)g->n_chunks * c0;
      if (dot_p) {
        q.dotP = dot_p + c0;
        q.gc_partial = gc_partial + (size_t)gc_row * g->R * B;
        gc_row += agg_blocks(g->n_rows, dc);
      }
      rc = dispatch_agg(q, MIX_BASIS, g->n_chunks, st);   // (chunk partials are simply reduced again per basis group)
      if (rc) return rc;
    }
  }
  return RGCN_OK;
}

// Row-range form of the (unmixed) forward walk: positions [row_begin, row_end) of the walk order only; hub_pass = 0 when
// an earlier call of the same layer has already reduced the hub chunks into `workspace`.  rgcn_layer_fwd uses it to
// pipeline the walk of row chunk c + 1 with the transform of chunk c.
extern "C" int rgcn_aggregate_fwd_rows(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d, void* H, void* H_lo,
                                       int64_t ldh, int32_t out_mode, const float* x_root, int64_t ld_x_root,
                                       int64_t row_begin, int64_t row_end, int32_t hub_pass, void* workspace,
                                       size_t workspace_bytes, rgcn_stream_t stream) {
  int rc = check_common(g, X, ldx, d, workspace, workspace_bytes);
  if (rc) return rc;
  RGCN_CHECK_ARG(!x_root || (((uintptr_t)x_root & 15) == 0 && ld_x_root % 4 == 0), "aggregate_fwd_rows: x_root misaligned");
  RGCN_CHECK_ARG(out_mode >= 0 && out_mode <= 2, "aggregate_fwd_rows: out_mode must be 0 (fp32), 1 (bf16) or 2 (bf16 hi+lo)");
  RGCN_CHECK_ARG(H && ((uintptr_t)H & (out_mode ? 7 : 15)) == 0 && ldh % 4 == 0, "aggregate_fwd_rows: output must be aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(out_mode != 2 || (H_lo && ((uintptr_t)H_lo & 7) == 0), "aggregate_fwd_rows: out_mode 2 needs the lo plane");
  RGCN_CHECK_ARG(0 <= row_begin && row_begin <= row_end && row_end <= g->n_rows, "aggregate_fwd_rows: bad row range");
  RGCN_CHECK_ARG(!g->row_order || g->order_chunk_rows == 0 ||
                 ((row_begin % g->order_chunk_rows == 0) && (row_end % g->order_chunk_rows == 0 || row_end == g->n_rows)),
                 "aggregate_fwd_rows: with a chunk-wise row order the range must consist of whole order chunks");
  RGCN_CHECK_ARG(!g->row_order || g->order_chunk_rows > 0 || (row_begin == 0 && row_end == g->n_rows) || row_begin == row_end,
                 "aggregate_fwd_rows: a global row order cannot be walked in ranges");
  AggParams p{};
  p.rowptr = g->rowptr; p.idx = g->idx; p.edge_w = g->w;
  p.hub_keys = g->hub_keys; p.hub_chunk_ptr = g->hub_chunk_ptr; p.n_hubs = g->n_hubs; p.chunk_table = g->chunk_table;
  p.row_order = g->row_order; p.hub_threshold = g->hub_threshold;
  p.n_rows = g->n_rows; p.R = g->R;
  p.F = X; p.ldf = ldx; p.src_rel_stride = 0; p.d = d; p.block_stride = d;
  p.O = H; p.O_lo = H_lo; p.ldo = ldh; p.out_mode = out_mode; p.partials = (float*)workspace;
  p.root_rows = x_root; p.ld_root = ld_x_root;
  p.range_mode = 1; p.row_begin = row_begin; p.row_end = row_end; p.no_hub_pass = hub_pass ? 0 : 1;
  if (row_end == row_begin && !hub_pass) return RGCN_OK;            // (an empty range with hub_pass = the hub pass alone)
  return dispatch_agg(p, MIX_NONE, g->n_chunks, (cudaStream_t)stream);
}

// bf16 features -> bf16 hi plane (the bf16-transform mode): X16 [n_src, d] and x_root16 [n_rows, d] are bf16 matrices
// (leading dimensions in ELEMENTS, multiples of 8, 16-byte aligned rows); H_hi as in out_mode 1.  Row range / hub_pass as in
// rgcn_aggregate_fwd_rows (row_begin = 0, row_end = n_rows, hub_pass = 1: everything).
extern "C" int rgcn_aggregate_fwd_bf16(const rgcn_csr_t* g, const void* X16, int64_t ldx, int32_t d, void* H_hi, int64_t ldh,
                                       const void* x_root16, int64_t ld_x_root, int64_t row_begin, int64_t row_end,
                                       int32_t hub_pass, void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(g && g->rowptr && (g->idx || g->E == 0) && g->R >= 1 && g->n_rows >= 0 && g->hub_threshold >= 1, "aggregate_fwd_bf16: bad CSR");
  RGCN_CHECK_ARG(d >= 8 && d <= 1024 && d % 8 == 0, "aggregate_fwd_bf16: d=%d must be a multiple of 8 in [8, 1024]", d);
  RGCN_CHECK_ARG(X16 && ((uintptr_t)X16 & 15) == 0 && ldx % 8 == 0, "aggregate_fwd_bf16: features must be 16-byte aligned rows");
  RGCN_CHECK_ARG(H_hi && ((uintptr_t)H_hi & 15) == 0 && ldh % 8 == 0, "aggregate_fwd_bf16: output plane must be 16-byte aligned, ld %% 8 == 0");
  RGCN_CHECK_ARG(!x_root16 || (((uintptr_t)x_root16 & 15) == 0 && ld_x_root % 8 == 0), "aggregate_fwd_bf16: x_root misaligned");
  RGCN_CHECK_ARG(0 <= row_begin && row_begin <= row_end && row_end <= g->n_rows, "aggregate_fwd_bf16: bad row range");
  RGCN_CHECK_ARG(g->n_chunks == 0 || (g->hub_keys && g->hub_chunk_ptr && g->n_hubs > 0 && g->chunk_table), "aggregate_fwd_bf16: hub plan missing");
  if (g->n_chunks > 0 && (!workspace || workspace_bytes < (size_t)g->n_chunks * d * sizeof(float))) {
    set_error("aggregate_fwd_bf16: workspace too small"); return RGCN_EWORKSPACE;
  }
  const bool whole = row_begin == 0 && row_end == g->n_rows;
  RGCN_CHECK_ARG(whole || !g->row_order || (g->order_chunk_rows > 0 && row_begin % g->order_chunk_rows == 0 &&
                                            (row_end % g->order_chunk_rows == 0 || row_end == g->n_rows)),
                 "aggregate_fwd_bf16: with a row order the range must consist of whole order chunks");
  AggParams p{};
  p.rowptr = g->rowptr; p.idx = g->idx; p.edge_w = g->w;
  p.hub_keys = g->hub_keys; p.hub_chunk_ptr = g->hub_chunk_ptr; p.n_hubs = g->n_hubs; p.chunk_table = g->chunk_table;
  p.row_order = g->row_order; p.hub_threshold = g->hub_threshold;
  p.n_rows = g->n_rows; p.R = g->R;
  p.F = (const float*)X16; p.ldf = ldx; p.d = d; p.block_stride = d;
  p.O = H_hi; p.ldo = ldh; p.out_mode = 1; p.partials = (float*)workspace;
  p.root_rows = (const float*)x_root16; p.ld_root = ld_x_root;
  p.range_mode = 1; p.row_begin = row_begin; p.row_end = row_end; p.no_hub_pass = hub_pass ? 0 : 1;
  cudaStream_t st = (cudaStream_t)stream;
  const int nvec = d >> 3;
  if (nvec <= 4) return launch_agg_bf16<4, 1>(p, g->n_chunks, st);
  if (nvec <= 8) return launch_agg_bf16<8, 1>(p, g->n_chunks, st);
  if (nvec <= 16) return launch_agg_bf16<16, 1>(p, g->n_chunks, st);
  if (nvec <= 32) return launch_agg_bf16<32, 1>(p, g->n_chunks, st);
  if (nvec <= 64) return launch_agg_bf16<32, 2>(p, g->n_chunks, st);
  return launch_agg_bf16<32, 4>(p, g->n_chunks, st);
}

static int aggregate_bwd_impl(const rgcn_csr_t* gt, const float* gH, int64_t ldg, int32_t d, const int32_t* slot,
                              int32_t zero_row, const float* init, int64_t ld_init, float* gX, int64_t ldgx,
                              const rgcn_masked_planes_out* mp, void* workspace, size_t workspace_bytes, rgcn_stream_t stream,
                              const uint8_t* row_flag = nullptr);

// grid of the (unmixed / summed) row walk = rows of the column-sum partials of rgcn_masked_planes_out
extern "C" int64_t rgcn_aggregate_row_blocks(const rgcn_csr_t* g, int32_t d) {
  if (!g || d < 4) return 0;
  return agg_blocks(g->n_rows, d);
}

extern "C" int rgcn_aggregate_bwd(const rgcn_csr_t* gt, const float* gH, int64_t ldg, int32_t d,
                                  const float* init, int64_t ld_init, float* gX, int64_t ldgx,
                                  const rgcn_masked_planes_out* mp,
                                  void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  return aggregate_bwd_impl(gt, gH, ldg, d, nullptr, 0, init, ld_init, gX, ldgx, mp, workspace, workspace_bytes, stream);
}

extern "C" int rgcn_aggregate_bwd_rows(const rgcn_csr_t* gt, const float* gH_rows, int64_t ldg, int32_t d,
                                       const int32_t* slot, int32_t zero_row, const float* init_rows, int64_t ld_init,
                                       float* gX, int64_t ldgx, const rgcn_masked_planes_out* mp,
                                       void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(slot && zero_row >= 0, "aggregate_bwd_rows: slot map and zero row are required");
  return aggregate_bwd_impl(gt, gH_rows, ldg, d, slot, zero_row, init_rows, ld_init, gX, ldgx, mp, workspace, workspace_bytes, stream);
}

namespace rgcn {
// one warp per list position (first positions only): flag every source of the listed row's in-edges
__global__ void __launch_bounds__(256) mark_sources_kernel(const int32_t* __restrict__ rowptr_f, const int32_t* __restrict__ idx_f,
                                                           int32_t R, const int64_t* __restrict__ rows, int64_t n_list,
                                                           const int32_t* __restrict__ slot, uint8_t* __restrict__ flag) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int64_t c = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (c >= n_list) return;
  const int64_t row = rows[c];
  if (__ldg(slot + row) != (int32_t)c) return;
  const int beg = __ldg(rowptr_f + row * R), end = __ldg(rowptr_f + row * R + R);
  for (int e = beg + lane; e < end; e += 32) flag[__ldg(idx_f + e)] = 1;
}
}  // namespace rgcn

// Row-sparse backward walk on a graph much larger than the row list: src_flag [gt->n_rows] (scratch) is cleared, the
// sources of the listed rows' in-edges are marked from the FORWARD-orientation CSR g_fwd, and unmarked rows leave the walk
// at once.  Same results as rgcn_aggregate_bwd_rows (the skipped rows only ever add exact zeros).
extern "C" int rgcn_aggregate_bwd_rows_marked(const rgcn_csr_t* gt, const rgcn_csr_t* g_fwd, const int64_t* rows, int64_t n_list,
                                              uint8_t* src_flag, const float* gH_rows, int64_t ldg, int32_t d,
                                              const int32_t* slot, int32_t zero_row, const float* init_rows, int64_t ld_init,
                                              float* gX, int64_t ldgx, void* workspace, size_t workspace_bytes,
                                              rgcn_stream_t stream) {
  RGCN_CHECK_ARG(gt && g_fwd && rows && n_list > 0 && src_flag && slot && zero_row >= 0, "aggregate_bwd_rows_marked: null argument");
  RGCN_CHECK_ARG(g_fwd->R == gt->R && g_fwd->rowptr && (g_fwd->idx || g_fwd->E == 0), "aggregate_bwd_rows_marked: the two orientations disagree");
  cudaStream_t st = (cudaStream_t)stream;
  RGCN_CUDA(cudaMemsetAsync(src_flag, 0, (size_t)gt->n_rows, st));
  RGCN_CUDA(launch_pdl(mark_sources_kernel, dim3((unsigned)((n_list + 7) / 8)), dim3(256), 0, st, g_fwd->rowptr, g_fwd->idx, g_fwd->R,
                       rows, n_list, slot, src_flag));
  RGCN_LAUNCH_CHECK();
  return aggregate_bwd_impl(gt, gH_rows, ldg, d, slot, zero_row, init_rows, ld_init, gX, ldgx, nullptr, workspace, workspace_bytes,
                            stream, src_flag);
}

static int aggregate_bwd_impl(const rgcn_csr_t* gt, const float* gH, int64_t ldg, int32_t d, const int32_t* slot,
                              int32_t zero_row, const float* init, int64_t ld_init, float* gX, int64_t ldgx,
                              const rgcn_masked_planes_out* mp, void* workspace, size_t workspace_bytes, rgcn_stream_t stream,
                              const uint8_t* row_flag) {
  int rc = check_common(gt, gH, ldg, d, workspace, workspace_bytes);
  if (rc) return rc;
  RGCN_CHECK_ARG(!mp || (mp->mask && mp->hi && ((uintptr_t)mp->mask & 15) == 0 && mp->ld_mask % 4 == 0 &&
                         ((uintptr_t)mp->hi & 7) == 0 && (!mp->lo || ((uintptr_t)mp->lo & 7) == 0) && mp->ldp % 4 == 0 &&
                         (!mp->colsum_partial || ((uintptr_t)mp->colsum_partial & 15) == 0)),
                 "aggregate_bwd: masked-planes output needs a 16-byte aligned mask and 8-byte aligned planes");
  RGCN_CHECK_ARG(gX && ((uintptr_t)gX & 15) == 0 && ldgx % 4 == 0, "aggregate_bwd: output must be 16-byte aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(!init || (((uintptr_t)init & 15) == 0 && ld_init % 4 == 0), "aggregate_bwd: init must be 16-byte aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(gt->w || gt->E == 0, "aggregate_bwd: the transposed CSR needs per-edge weights w_t");
  AggParams p{};
  p.rowptr = gt->rowptr; p.idx = gt->idx; p.edge_w = gt->w;
  p.hub_keys = gt->hub_keys; p.hub_chunk_ptr = gt->hub_chunk_ptr; p.n_hubs = gt->n_hubs; p.chunk_table = gt->chunk_table;
  p.row_order = gt->row_order; p.hub_threshold = gt->hub_threshold;
  p.n_rows = gt->n_rows; p.R = gt->R;
  p.F = gH; p.ldf = ldg; p.src_rel_stride = d; p.d = d; p.block_stride = d;
  p.init = init; p.ld_init = ld_init; p.B = 1;
  p.O = gX; p.ldo = ldgx; p.out_mode = 0; p.partials = (float*)workspace;
  p.slot = slot; p.zero_row = zero_row; p.row_flag = row_flag;
  // RGCN_STREAM_REL: 0 = never, 3 = every hub-free pass, 1 = per pass where the non-empty segments average fewer than
  // four edges, 2 (default) = 3 on graphs whose segments average fewer than four edges and whose hub segments hold less
  // than 1/16 of the edges, else 0.  Measured on the B200, everything streamed: the partitioned shard (1.25 M rows /
  // 50 M edges / 30 relations, uniform; 1 GPU) 57.5 -> 54.8 ms per step (backward walks 7.84 + 5.96 -> 6.12 + 4.36 ms),
  // but cfg3 (30 relations, power law: most edges sit in long segments whose batches are full anyway) 2.79 -> 2.99 ms;
  // the per-pass rule (1) gives cfg3 2.80 ms but lets the two lane groups of a warp take different paths.
  static int env_stream = -1;
  if (env_stream < 0) { const char* e = getenv("RGCN_STREAM_REL"); env_stream = e ? atoi(e) : 2; }
  p.stream_rel = env_stream != 2 ? env_stream
                                 : ((gt->E < 4 * gt->n_rows * (int64_t)gt->R && (int64_t)gt->n_chunks * kHubChunk * 16 < gt->E) ? 3 : 0);
  if (mp) {
    p.mp_mask = mp->mask; p.ld_mp_mask = mp->ld_mask; p.mp_scale = mp->scale;
    p.mp_hi = mp->hi; p.mp_lo = mp->lo; p.ld_mp = mp->ldp; p.mp_colsum = mp->colsum_partial;
  }
  return dispatch_agg(p, MIX_SUM, gt->n_chunks, (cudaStream_t)stream);
}

// ---- listed-rows forward walk --------------------------------------------------------------------------------------------
// The last layer of the reference's training step is only read at the 2 * batch head / tail rows of its output
// (src/models/rgcn.py:325-326): the walk visits the listed rows only and writes a COMPACT operand [m_c, (R+1) d]
// (m_c = rgcn_rows_compact_size(n_list); position c = row rows[c], duplicates are simply computed twice, padding positions
// are zero rows).  slot (nullable): node -> first list position or m_c, used to skip the hub chunks of unlisted rows.
static int aggregate_fwd_list_impl(const rgcn_csr_t* g, const void* X, int64_t ldx, int32_t d, bool x_bf16, void* H, void* H_lo,
                                   int64_t ldh, int32_t out_mode, const void* x_root, int64_t ld_x_root, const int64_t* rows,
                                   int64_t n_list, const int32_t* slot, void* workspace, size_t workspace_bytes,
                                   rgcn_stream_t stream) {
  RGCN_CHECK_ARG(g && g->rowptr && (g->idx || g->E == 0) && g->R >= 1 && g->n_rows >= 0 && g->hub_threshold >= 1, "aggregate_fwd_list: bad CSR");
  RGCN_CHECK_ARG(rows && slot && n_list > 0 && n_list < (1ll << 30), "aggregate_fwd_list: bad row list / slot map");
  const int64_t m_c = rgcn_rows_compact_size(n_list);
  RGCN_CHECK_ARG(g->n_chunks == 0 || (g->hub_keys && g->hub_chunk_ptr && g->n_hubs > 0 && g->chunk_table), "aggregate_fwd_list: hub plan missing");
  if (g->n_chunks > 0 && (!workspace || workspace_bytes < (size_t)g->n_chunks * d * sizeof(float))) {
    set_error("aggregate_fwd_list: workspace too small"); return RGCN_EWORKSPACE;
  }
  AggParams p{};
  p.rowptr = g->rowptr; p.idx = g->idx;
  p.hub_keys = g->hub_keys; p.hub_chunk_ptr = g->hub_chunk_ptr; p.n_hubs = g->n_hubs; p.chunk_table = g->chunk_table;
  p.hub_threshold = g->hub_threshold;
  p.n_rows = g->n_rows; p.R = g->R;
  p.F = (const float*)X; p.ldf = ldx; p.src_rel_stride = 0; p.d = d; p.block_stride = d;
  p.O = H; p.O_lo = H_lo; p.ldo = ldh; p.out_mode = out_mode; p.partials = (float*)workspace;
  p.root_rows = (const float*)x_root; p.ld_root = ld_x_root;
  p.edge_w = g->w;                                   // unit weights of a sum layer: the weighted instantiations
  p.list = rows; p.n_list = n_list; p.hub_filter = slot; p.hub_unlisted = (int32_t)m_c;
  // by rows (degree order, unlisted rows leave at once) while the row count is moderate; by list positions beyond
  static int env_by_rows = -1;
  // (measured equal on cfg2, 58.2 against 57.6 us, so the cheaper launch — by positions — is the default; 2 = by rows
  // when n_rows <= 16 n_list)
  if (env_by_rows < 0) { const char* e = getenv("RGCN_LIST_BY_ROWS"); env_by_rows = e ? atoi(e) : 0; }
  p.list_by_rows = env_by_rows == 2 ? (g->n_rows <= 16 * n_list ? 1 : 0) : (env_by_rows ? 1 : 0);
  p.row_order = p.list_by_rows ? g->row_order : nullptr;
  p.list_walkers = p.list_by_rows ? g->n_rows : n_list;
  p.range_mode = 1; p.row_begin = 0; p.row_end = p.list_walkers + m_c;
  cudaStream_t st = (cudaStream_t)stream;
  auto run = [&](const AggParams& q, int n_chunks) {
    if (!x_bf16) return dispatch_agg(q, MIX_NONE, n_chunks, st);
    const int nvec = q.d >> 3;
    if (nvec <= 4) return launch_agg_bf16<4, 1>(q, n_chunks, st);
    if (nvec <= 8) return launch_agg_bf16<8, 1>(q, n_chunks, st);
    if (nvec <= 16) return launch_agg_bf16<16, 1>(q, n_chunks, st);
    if (nvec <= 32) return launch_agg_bf16<32, 1>(q, n_chunks, st);
    if (nvec <= 64) return launch_agg_bf16<32, 2>(q, n_chunks, st);
    return launch_agg_bf16<32, 4>(q, n_chunks, st);
  };
  // RGCN_LIST_OVERLAP_HUBS: 0 (default) never, 1 always, 2 while capturing.  OPT-IN: measured on the B200 the hub pass beside
  // the listed walk LOSES like it does for the dense walk — cfg2 layer 2 listed forward 54.8 against 51.6 us, step 0.300
  // against 0.293 ms (two latency-bound kernels sharing the L2 queues, plus the finish kernel's serial tail)
  static int env_overlap = -1;
  if (env_overlap < 0) { const char* e = getenv("RGCN_LIST_OVERLAP_HUBS"); env_overlap = e ? atoi(e) : 0; }
  static int env_slice0 = -1;
  if (env_slice0 < 0) { const char* e = getenv("RGCN_LIST_SLICE"); env_slice0 = e ? atoi(e) : 0; }
  if (!x_bf16 && !g->w && env_overlap && env_slice0 == 0 && g->n_chunks > 0) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    const bool capturing = cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive;
    if (!capturing) (void)fork_join_existing(st);   // (the side stream is made by the first eager call: GraphedTrainStep and
                                                    //  the module's own capture both warm up eagerly before they capture)
    if (env_overlap == 1 || capturing) {
      // one dispatch: hub chunks beside the walk (side stream; two branches of a captured graph), then the finish kernel
      static int env_rs = -1;
      if (env_rs < 0) { const char* e = getenv("RGCN_LIST_RSPLIT"); env_rs = e ? atoi(e) : 1; }
      p.list_overlap_hubs = 1; p.list_slices = 1;
      p.list_rsplit = env_rs < 1 ? 1 : (env_rs > g->R ? g->R : env_rs);
      return run(p, g->n_chunks);
    }
  }
  // hub chunks (full width, only the listed rows' chunks), then the walk in column slices x relation ranges
  if (g->n_chunks > 0) {
    AggParams h = p;
    h.row_end = h.row_begin;                         // hub pass alone
    int rc = run(h, g->n_chunks);
    if (rc) return rc;
  }
  static int env_slice = -1, env_rsplit = -1;
  // measured on the B200 (scripts/ab_listed.py, cfg2 layer 2, 4,096 listed rows of which 2,748 distinct): the whole layer
  // 58 us unsplit, 66 us with two column slices, 97 us with slices x three relation ranges — once duplicates are walked
  // only once the split buys nothing, so both default to off
  if (env_slice < 0) { const char* e = getenv("RGCN_LIST_SLICE"); env_slice = e ? atoi(e) : 0; }
  if (env_rsplit < 0) { const char* e = getenv("RGCN_LIST_RSPLIT"); env_rsplit = e ? atoi(e) : 1; }
  const int unit = x_bf16 ? 8 : 4;
  int slice = d;
  if (env_slice >= unit && env_slice % unit == 0 && env_slice < d && d % env_slice == 0) slice = env_slice;
  p.d = slice; p.list_slices = d / slice;
  p.list_rsplit = env_rsplit < 1 ? 1 : (env_rsplit > g->R ? g->R : env_rsplit);
  p.no_hub_pass = 1;
  return run(p, 0);
}

extern "C" int rgcn_aggregate_fwd_list(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d, void* H, void* H_lo,
                                       int64_t ldh, int32_t out_mode, const float* x_root, int64_t ld_x_root,
                                       const int64_t* rows, int64_t n_list, const int32_t* slot, void* workspace,
                                       size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(d >= 4 && d <= 1024 && d % 4 == 0, "aggregate_fwd_list: feature width d=%d must be a multiple of 4 in [4,1024]", d);
  RGCN_CHECK_ARG(X && ldx % 4 == 0 && ((uintptr_t)X & 15) == 0, "aggregate_fwd_list: feature matrix must be 16-byte aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(!x_root || (((uintptr_t)x_root & 15) == 0 && ld_x_root % 4 == 0), "aggregate_fwd_list: x_root misaligned");
  RGCN_CHECK_ARG(out_mode >= 0 && out_mode <= 2, "aggregate_fwd_list: out_mode must be 0 (fp32), 1 (bf16) or 2 (bf16 hi+lo)");
  RGCN_CHECK_ARG(H && ((uintptr_t)H & (out_mode ? 7 : 15)) == 0 && ldh % 4 == 0, "aggregate_fwd_list: output must be aligned with ld %% 4 == 0");
  RGCN_CHECK_ARG(out_mode != 2 || (H_lo && ((uintptr_t)H_lo & 7) == 0), "aggregate_fwd_list: out_mode 2 needs the lo plane");
  return aggregate_fwd_list_impl(g, X, ldx, d, false, H, H_lo, ldh, out_mode, x_root, ld_x_root, rows, n_list, slot, workspace,
                                 workspace_bytes, stream);
}

extern "C" int rgcn_aggregate_fwd_bf16_list(const rgcn_csr_t* g, const void* X16, int64_t ldx, int32_t d, void* H_hi, int64_t ldh,
                                            const void* x_root16, int64_t ld_x_root, const int64_t* rows, int64_t n_list,
                                            const int32_t* slot, void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(d >= 8 && d <= 1024 && d % 8 == 0, "aggregate_fwd_bf16_list: d=%d must be a multiple of 8 in [8, 1024]", d);
  RGCN_CHECK_ARG(X16 && ((uintptr_t)X16 & 15) == 0 && ldx % 8 == 0, "aggregate_fwd_bf16_list: features must be 16-byte aligned rows");
  RGCN_CHECK_ARG(H_hi && ((uintptr_t)H_hi & 15) == 0 && ldh % 8 == 0, "aggregate_fwd_bf16_list: output plane must be 16-byte aligned, ld %% 8 == 0");
  RGCN_CHECK_ARG(!x_root16 || (((uintptr_t)x_root16 & 15) == 0 && ld_x_root % 8 == 0), "aggregate_fwd_bf16_list: x_root misaligned");
  return aggregate_fwd_list_impl(g, X16, ldx, d, true, H_hi, nullptr, ldh, 1, x_root16, ld_x_root, rows, n_list, slot, workspace,
                                 workspace_bytes, stream);
}
