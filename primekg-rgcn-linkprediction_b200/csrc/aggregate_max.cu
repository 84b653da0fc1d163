// Max aggregation of RGCNConv(aggr='max') and its backward, kept apart from the tuned mean / sum walks of
// aggregate.cu so that those never branch on the aggregation.
//
// Forward, over the (dst, rel) CSR:  per (i, r, column)
//   m = max_{e in seg(i, r)} x[col[e]]   (NaN propagates; 0 for an empty segment)
//   c = |{e : x[col[e]] == m}| + [m == 0]
// i.e. torch's  zeros(..).scatter_reduce_(0, idx, src, 'amax', include_self=False)  and the divisor its backward uses:
// the gradient of h = m is split evenly over the tied sources, and the zero initial value counts as one more tie when
// the maximum is exactly 0.  m is written as the transform's operand planes (block r of row i, x appended as block R),
// and in fp32 with c for the backward (the bf16 planes do not reproduce m exactly, the equality test needs fp32).
//
// Backward, over the transposed (src, rel) CSR:
//   gX[j] = init[j] + sum_r sum_{e: j -> i in seg_t(j, r)} t(e),   t = [x[j] == m(i, r)] * gH[i, r] / c(i, r)
// and t = NaN where m(i, r) is NaN: torch's backward multiplies the zero mask by gH / 0 there.
//
// Mapping and hub treatment as the mean walks (aggregate.cu): a group of G = min(32, d/4) lanes owns one row, each lane
// VPL float4 of it, and U gathers are in flight per batch.  Segments longer than the hub threshold are cut into the
// chunks of the orientation's hub plan, which whole blocks reduce beforehand: forward into (m, c) chunk partials — they
// combine exactly, in any order — backward into sums of t, added by the row walk in chunk order.  Every run gives the
// same bits; no atomics.
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace rgcn {

namespace {

__device__ __forceinline__ void store_planes(void* O, void* O_lo, int64_t ldo, int out_mode, int64_t row, int col,
                                             const float4& v) {
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

// (m, c) <- (m, c) combined with (v, n): the larger value wins, equal values add their counts, NaN absorbs everything
__device__ __forceinline__ void mc_combine(float& m, float& c, float v, float n) {
  if (m != m) return;
  if (v != v || v > m) { m = v; c = n; }
  else if (v == m) c += n;
}
__device__ __forceinline__ void mc4(float4& m, float4& c, const float4& v, const float4& n) {
  mc_combine(m.x, c.x, v.x, n.x); mc_combine(m.y, c.y, v.y, n.y);
  mc_combine(m.z, c.z, v.z, n.z); mc_combine(m.w, c.w, v.w, n.w);
}
__device__ __forceinline__ void mc4(float4& m, float4& c, const float4& v) { mc4(m, c, v, make_float4(1.f, 1.f, 1.f, 1.f)); }

__device__ __forceinline__ float grad_term(float x, float m, float c, float g) {
  if (m != m) return __int_as_float(0x7fffffff);
  return x == m ? g / c : 0.f;
}
__device__ __forceinline__ void add_grad4(float4& acc, const float4& x, const float4& m, const float4& c, const float4& g) {
  acc.x += grad_term(x.x, m.x, c.x, g.x); acc.y += grad_term(x.y, m.y, c.y, g.y);
  acc.z += grad_term(x.z, m.z, c.z, g.z); acc.w += grad_term(x.w, m.w, c.w, g.w);
}

constexpr int batch_edges(int vpl) { return vpl >= 4 ? 2 : (vpl == 2 ? 4 : 8); }
// backward: three gathers per edge (maxima, counts, gradient) — fewer edges per batch keep the loads in registers
constexpr int batch_edges_bwd(int vpl) { return vpl >= 8 ? 1 : (vpl >= 2 ? 2 : 4); }

// position of the hub segment `key` in the plan (it is one: its length exceeds the threshold)
__device__ __forceinline__ int hub_index(const int32_t* hub_keys, int n_hubs, int key) {
  int lo = 0, hi = n_hubs;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(hub_keys + mid) <= key) lo = mid; else hi = mid;
  }
  return lo;
}

}  // namespace

struct MaxParams {
  const int32_t* rowptr;
  const int32_t* idx;
  int64_t n_rows;
  int32_t R, d;
  int32_t hub_threshold, n_hubs;
  const int32_t* hub_keys;
  const int32_t* hub_chunk_ptr;
  const int32_t* chunk_table;
  int32_t n_chunks;
  float* partials;             // forward: [n_chunks, d] maxima then [n_chunks, d] counts; backward: [n_chunks, d] sums
  const float* X; int64_t ldx;
  // forward
  const float* x_root; int64_t ld_root;
  void* O; void* O_lo; int64_t ldo; int32_t out_mode;
  float* Hmax_w; float* Hcnt_w;
  // backward (Hmax / Hcnt / gH indexed by the gathered row i)
  const float* Hmax; const float* Hcnt; int64_t ldm;
  const float* gH; int64_t ldg;
  const float* init; int64_t ld_init;
  float* gX; int64_t ldgx;
};

// ---- hub chunks: one block per chunk of a long segment -------------------------------------------------------------
template <int G, int VPL, bool BWD>
__global__ void __launch_bounds__(256, 1) aggregate_max_hub_kernel(const MaxParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  constexpr int PER = kHubChunk / GROUPS;
  constexpr int U0 = BWD ? batch_edges_bwd(VPL) : batch_edges(VPL);
  constexpr int U = U0 < PER ? U0 : PER;
  __shared__ float4 red[GROUPS][G * VPL];
  const int chunk = blockIdx.x;
  const int4 t = __ldg(reinterpret_cast<const int4*>(p.chunk_table) + chunk);
  const int key = t.x, r = key % p.R;
  const int64_t row = key / p.R;
  const int seg_beg = __ldg(p.rowptr + key), seg_end = __ldg(p.rowptr + key + 1);
  const int c_beg = seg_beg + (chunk - t.y) * kHubChunk;
  const int c_end = min(c_beg + kHubChunk, seg_end);
  const int nvec = p.d >> 2;
  const int lane = threadIdx.x % G, grp = threadIdx.x / G;
  const int g_beg = c_beg + grp * PER, g_end = min(g_beg + PER, c_end);
  int vcol[VPL];
  float4 a[VPL], c[VPL], xj[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    vcol[k] = vi < nvec ? vi * 4 : 0;
    if (BWD) {
      a[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      xj[k] = ldg4(p.X + row * p.ldx + vcol[k]);
    } else {
      a[k] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    c[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  int e = g_beg;
  auto batch = [&](auto ub) {
    constexpr int UB = decltype(ub)::value;
    int j[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) j[u] = __ldg(p.idx + e + u);
    if (BWD) {
      float4 m[UB][VPL], n[UB][VPL], g[UB][VPL];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int64_t om = (int64_t)j[u] * p.ldm + (int64_t)r * p.d, og = (int64_t)j[u] * p.ldg + (int64_t)r * p.d;
#pragma unroll
        for (int k = 0; k < VPL; ++k) {
          m[u][k] = ldg4(p.Hmax + om + vcol[k]); n[u][k] = ldg4(p.Hcnt + om + vcol[k]); g[u][k] = ldg4(p.gH + og + vcol[k]);
        }
      }
#pragma unroll
      for (int u = 0; u < UB; ++u)
#pragma unroll
        for (int k = 0; k < VPL; ++k) add_grad4(a[k], xj[k], m[u][k], n[u][k], g[u][k]);
    } else {
      float4 v[UB][VPL];
#pragma unroll
      for (int u = 0; u < UB; ++u)
#pragma unroll
        for (int k = 0; k < VPL; ++k) v[u][k] = ldg4(p.X + (int64_t)j[u] * p.ldx + vcol[k]);
#pragma unroll
      for (int u = 0; u < UB; ++u)
#pragma unroll
        for (int k = 0; k < VPL; ++k) mc4(a[k], c[k], v[u][k]);
    }
    e += UB;
  };
  while (e + U <= g_end) batch(std::integral_constant<int, U>{});
  while (e < g_end) batch(std::integral_constant<int, 1>{});
#pragma unroll
  for (int k = 0; k < VPL; ++k) red[grp][k * G + lane] = a[k];
  __syncthreads();
  if (BWD) {
    for (int vi = threadIdx.x; vi < nvec; vi += 256) {         // fixed order over the groups
      float4 s = red[0][vi];
      for (int gi = 1; gi < GROUPS; ++gi) add4(s, red[gi][vi]);
      reinterpret_cast<float4*>(p.partials + (size_t)chunk * p.d)[vi] = s;
    }
    return;
  }
  // the chunk's maxima (exact in any order), then the ties of the groups whose maximum equals it
  for (int vi = threadIdx.x; vi < nvec; vi += 256) {
    float4 m = red[0][vi], n = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int gi = 1; gi < GROUPS; ++gi) mc4(m, n, red[gi][vi]);
    red[0][vi] = m;                                            // (only this thread touches column vi)
    reinterpret_cast<float4*>(p.partials + (size_t)chunk * p.d)[vi] = m;
  }
  __syncthreads();
  float4 mine[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const float4 m = red[0][k * G + lane];
    mine[k] = make_float4(a[k].x == m.x ? c[k].x : 0.f, a[k].y == m.y ? c[k].y : 0.f,
                          a[k].z == m.z ? c[k].z : 0.f, a[k].w == m.w ? c[k].w : 0.f);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < VPL; ++k) red[grp][k * G + lane] = mine[k];
  __syncthreads();
  for (int vi = threadIdx.x; vi < nvec; vi += 256) {
    float4 s = red[0][vi];
    for (int gi = 1; gi < GROUPS; ++gi) add4(s, red[gi][vi]);  // integer counts: exact
    reinterpret_cast<float4*>(p.partials + ((size_t)p.n_chunks + chunk) * p.d)[vi] = s;
  }
}

// ---- rows: one G-lane group per row --------------------------------------------------------------------------------
template <int G, int VPL>
__global__ void __launch_bounds__(256) aggregate_max_fwd_kernel(const MaxParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  constexpr int U = batch_edges(VPL);
  const int lane = threadIdx.x % G;
  const int64_t row = (int64_t)blockIdx.x * GROUPS + threadIdx.x / G;
  if (row >= p.n_rows) return;
  const int nvec = p.d >> 2;
  bool act[VPL];
  int vcol[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    act[k] = vi < nvec;
    vcol[k] = act[k] ? vi * 4 : 0;               // inactive lanes gather column 0; their results are never stored
  }
  if (p.x_root) {
#pragma unroll
    for (int k = 0; k < VPL; ++k)
      if (act[k]) store_planes(p.O, p.O_lo, p.ldo, p.out_mode, row, p.R * p.d + vcol[k], ldg4(p.x_root + row * p.ld_root + vcol[k]));
  }
  const int32_t* __restrict__ rowptr = p.rowptr + row * p.R;
  for (int r = 0; r < p.R; ++r) {
    const int beg = __ldg(rowptr + r), end = __ldg(rowptr + r + 1);
    float4 m[VPL], c[VPL];
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      m[k] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      c[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (end - beg > p.hub_threshold) {
      const int h = hub_index(p.hub_keys, p.n_hubs, (int)(row * p.R + r));
      const int c0 = __ldg(p.hub_chunk_ptr + h), c1 = __ldg(p.hub_chunk_ptr + h + 1);
      for (int ch = c0; ch < c1; ++ch) {
#pragma unroll
        for (int k = 0; k < VPL; ++k)
          mc4(m[k], c[k], *reinterpret_cast<const float4*>(p.partials + (size_t)ch * p.d + vcol[k]),
              *reinterpret_cast<const float4*>(p.partials + ((size_t)p.n_chunks + ch) * p.d + vcol[k]));
      }
    } else {
      int e = beg;
      auto batch = [&](auto ub) {
        constexpr int UB = decltype(ub)::value;
        int j[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) j[u] = __ldg(p.idx + e + u);
        float4 v[UB][VPL];
#pragma unroll
        for (int u = 0; u < UB; ++u)
#pragma unroll
          for (int k = 0; k < VPL; ++k) v[u][k] = ldg4(p.X + (int64_t)j[u] * p.ldx + vcol[k]);
#pragma unroll
        for (int u = 0; u < UB; ++u)
#pragma unroll
          for (int k = 0; k < VPL; ++k) mc4(m[k], c[k], v[u][k]);
        e += UB;
      };
      while (e + U <= end) batch(std::integral_constant<int, U>{});
      if (U > 2 && e + 2 <= end) batch(std::integral_constant<int, (U > 2 ? 2 : 1)>{});
      while (e < end) batch(std::integral_constant<int, 1>{});
    }
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      if (!act[k]) continue;
      if (end == beg) {
        m[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        c[k].x += m[k].x == 0.f ? 1.f : 0.f; c[k].y += m[k].y == 0.f ? 1.f : 0.f;
        c[k].z += m[k].z == 0.f ? 1.f : 0.f; c[k].w += m[k].w == 0.f ? 1.f : 0.f;
      }
      const int64_t off = row * p.ldm + (int64_t)r * p.d + vcol[k];
      *reinterpret_cast<float4*>(p.Hmax_w + off) = m[k];
      *reinterpret_cast<float4*>(p.Hcnt_w + off) = c[k];
      store_planes(p.O, p.O_lo, p.ldo, p.out_mode, row, r * p.d + vcol[k], m[k]);
    }
  }
}

template <int G, int VPL>
__global__ void __launch_bounds__(256, 1) aggregate_max_bwd_kernel(const MaxParams p) {
  pdl_enter();
  constexpr int GROUPS = 256 / G;
  constexpr int U = batch_edges_bwd(VPL);
  const int lane = threadIdx.x % G;
  const int64_t row = (int64_t)blockIdx.x * GROUPS + threadIdx.x / G;
  if (row >= p.n_rows) return;
  const int nvec = p.d >> 2;
  bool act[VPL];
  int vcol[VPL];
  float4 xj[VPL], acc[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int vi = k * G + lane;
    act[k] = vi < nvec;
    vcol[k] = act[k] ? vi * 4 : 0;
    xj[k] = ldg4(p.X + row * p.ldx + vcol[k]);
    acc[k] = p.init ? ldg4(p.init + row * p.ld_init + vcol[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int32_t* __restrict__ rowptr = p.rowptr + row * p.R;
  for (int r = 0; r < p.R; ++r) {
    const int beg = __ldg(rowptr + r), end = __ldg(rowptr + r + 1);
    if (end - beg > p.hub_threshold) {
      const int h = hub_index(p.hub_keys, p.n_hubs, (int)(row * p.R + r));
      const int c0 = __ldg(p.hub_chunk_ptr + h), c1 = __ldg(p.hub_chunk_ptr + h + 1);
      float4 s[VPL];
#pragma unroll
      for (int k = 0; k < VPL; ++k) s[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int ch = c0; ch < c1; ++ch) {                       // chunk partials in chunk order
#pragma unroll
        for (int k = 0; k < VPL; ++k) add4(s[k], *reinterpret_cast<const float4*>(p.partials + (size_t)ch * p.d + vcol[k]));
      }
#pragma unroll
      for (int k = 0; k < VPL; ++k) add4(acc[k], s[k]);
      continue;
    }
    int e = beg;
    auto batch = [&](auto ub) {
      constexpr int UB = decltype(ub)::value;
      int i[UB];
#pragma unroll
      for (int u = 0; u < UB; ++u) i[u] = __ldg(p.idx + e + u);
      float4 m[UB][VPL], n[UB][VPL], g[UB][VPL];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int64_t om = (int64_t)i[u] * p.ldm + (int64_t)r * p.d, og = (int64_t)i[u] * p.ldg + (int64_t)r * p.d;
#pragma unroll
        for (int k = 0; k < VPL; ++k) {
          m[u][k] = ldg4(p.Hmax + om + vcol[k]); n[u][k] = ldg4(p.Hcnt + om + vcol[k]); g[u][k] = ldg4(p.gH + og + vcol[k]);
        }
      }
#pragma unroll
      for (int u = 0; u < UB; ++u)
#pragma unroll
        for (int k = 0; k < VPL; ++k) add_grad4(acc[k], xj[k], m[u][k], n[u][k], g[u][k]);
      e += UB;
    };
    while (e + U <= end) batch(std::integral_constant<int, U>{});
    while (e < end) batch(std::integral_constant<int, 1>{});
  }
#pragma unroll
  for (int k = 0; k < VPL; ++k)
    if (act[k]) *reinterpret_cast<float4*>(p.gX + row * p.ldgx + vcol[k]) = acc[k];
}

template <int G, int VPL, bool BWD>
static int launch_max(const MaxParams& p, cudaStream_t st) {
  if (p.n_chunks > 0) {
    RGCN_CUDA(launch_pdl(aggregate_max_hub_kernel<G, VPL, BWD>, dim3((unsigned)p.n_chunks), dim3(256), 0, st, p));
    RGCN_LAUNCH_CHECK();
  }
  const unsigned grid = (unsigned)((p.n_rows + 256 / G - 1) / (256 / G));
  if (BWD) RGCN_CUDA(launch_pdl(aggregate_max_bwd_kernel<G, VPL>, dim3(grid), dim3(256), 0, st, p));
  else RGCN_CUDA(launch_pdl(aggregate_max_fwd_kernel<G, VPL>, dim3(grid), dim3(256), 0, st, p));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

template <bool BWD>
static int dispatch_max(const MaxParams& p, cudaStream_t st) {
  const int nvec = p.d >> 2;
  if (nvec <= 4) return launch_max<4, 1, BWD>(p, st);
  if (nvec <= 8) return launch_max<8, 1, BWD>(p, st);
  if (nvec <= 16) return launch_max<16, 1, BWD>(p, st);
  if (nvec <= 32) return launch_max<32, 1, BWD>(p, st);
  if (nvec <= 64) return launch_max<32, 2, BWD>(p, st);
  if (nvec <= 128) return launch_max<32, 4, BWD>(p, st);
  return launch_max<32, 8, BWD>(p, st);
}

static int max_params(const rgcn_csr_t* g, int32_t d, void* ws, size_t ws_bytes, int parts, const char* who, MaxParams* p) {
  RGCN_CHECK_ARG(g && g->rowptr && (g->idx || g->E == 0) && g->R >= 1 && g->n_rows >= 0 && g->hub_threshold >= 1,
                 "%s: bad CSR", who);
  RGCN_CHECK_ARG(d >= 4 && d <= 1024 && d % 4 == 0, "%s: feature width d=%d must be a multiple of 4 in [4,1024]", who, d);
  RGCN_CHECK_ARG(g->n_chunks == 0 || (g->hub_keys && g->hub_chunk_ptr && g->n_hubs > 0 && g->chunk_table &&
                                      ((uintptr_t)g->chunk_table & 15) == 0), "%s: hub plan missing", who);
  const size_t need = (size_t)g->n_chunks * parts * d * sizeof(float);
  if (g->n_chunks > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 15))) {
    set_error("%s: workspace too small or misaligned (%zu < %zu)", who, ws_bytes, need);
    return RGCN_EWORKSPACE;
  }
  *p = MaxParams{};
  p->rowptr = g->rowptr; p->idx = g->idx; p->n_rows = g->n_rows; p->R = g->R; p->d = d;
  p->hub_threshold = g->hub_threshold; p->n_hubs = g->n_hubs; p->hub_keys = g->hub_keys;
  p->hub_chunk_ptr = g->hub_chunk_ptr; p->chunk_table = g->chunk_table; p->n_chunks = g->n_chunks;
  p->partials = (float*)ws;
  return RGCN_OK;
}

}  // namespace rgcn

using namespace rgcn;

extern "C" size_t rgcn_aggregate_max_workspace_bytes(const rgcn_csr_t* g, int32_t d, int32_t backward) {
  if (!g) return 0;
  return align_up((size_t)g->n_chunks * (backward ? 1 : 2) * (size_t)d * sizeof(float), 256);
}

extern "C" int rgcn_aggregate_max_fwd(const rgcn_csr_t* g, const float* X, int64_t ldx, int32_t d, void* H, void* H_lo,
                                      int64_t ldh, int32_t out_mode, const float* x_root, int64_t ld_x_root, float* Hmax,
                                      float* Hcnt, int64_t ldm, void* workspace, size_t workspace_bytes,
                                      rgcn_stream_t stream) {
  MaxParams p;
  int rc = max_params(g, d, workspace, workspace_bytes, 2, "aggregate_max_fwd", &p);
  if (rc) return rc;
  RGCN_CHECK_ARG(!g->w, "aggregate_max_fwd: walks the forward (unweighted) orientation");
  RGCN_CHECK_ARG(X && ldx % 4 == 0 && ((uintptr_t)X & 15) == 0, "aggregate_max_fwd: features must be 16-byte aligned rows");
  RGCN_CHECK_ARG(!x_root || (((uintptr_t)x_root & 15) == 0 && ld_x_root % 4 == 0), "aggregate_max_fwd: x_root misaligned");
  RGCN_CHECK_ARG(out_mode == 1 || out_mode == 2, "aggregate_max_fwd: out_mode must be 1 (bf16) or 2 (bf16 hi+lo)");
  RGCN_CHECK_ARG(H && ((uintptr_t)H & 7) == 0 && ldh % 4 == 0 && ldh >= (int64_t)(g->R + (x_root ? 1 : 0)) * d,
                 "aggregate_max_fwd: operand planes must be 8-byte aligned, ld %% 4 == 0 and R (+1) blocks wide");
  RGCN_CHECK_ARG(out_mode != 2 || (H_lo && ((uintptr_t)H_lo & 7) == 0), "aggregate_max_fwd: out_mode 2 needs the lo plane");
  RGCN_CHECK_ARG(Hmax && Hcnt && ((uintptr_t)Hmax & 15) == 0 && ((uintptr_t)Hcnt & 15) == 0 && ldm % 4 == 0 &&
                 ldm >= (int64_t)g->R * d, "aggregate_max_fwd: fp32 maxima / counts must be 16-byte aligned [n_rows, >= R*d]");
  if (g->n_rows == 0) return RGCN_OK;
  p.X = X; p.ldx = ldx; p.x_root = x_root; p.ld_root = ld_x_root;
  p.O = H; p.O_lo = H_lo; p.ldo = ldh; p.out_mode = out_mode; p.Hmax_w = Hmax; p.Hcnt_w = Hcnt; p.ldm = ldm;
  return dispatch_max<false>(p, (cudaStream_t)stream);
}

extern "C" int rgcn_aggregate_max_bwd(const rgcn_csr_t* gt, const float* gH, int64_t ldg, const float* Hmax,
                                      const float* Hcnt, int64_t ldm, const float* X, int64_t ldx, int32_t d,
                                      const float* init, int64_t ld_init, float* gX, int64_t ldgx, void* workspace,
                                      size_t workspace_bytes, rgcn_stream_t stream) {
  MaxParams p;
  int rc = max_params(gt, d, workspace, workspace_bytes, 1, "aggregate_max_bwd", &p);
  if (rc) return rc;
  RGCN_CHECK_ARG(gH && ((uintptr_t)gH & 15) == 0 && ldg % 4 == 0 && ldg >= (int64_t)gt->R * d,
                 "aggregate_max_bwd: gH must be 16-byte aligned [n_dst, >= R*d]");
  RGCN_CHECK_ARG(Hmax && Hcnt && ((uintptr_t)Hmax & 15) == 0 && ((uintptr_t)Hcnt & 15) == 0 && ldm % 4 == 0 &&
                 ldm >= (int64_t)gt->R * d, "aggregate_max_bwd: fp32 maxima / counts must be 16-byte aligned [n_dst, >= R*d]");
  RGCN_CHECK_ARG(X && ((uintptr_t)X & 15) == 0 && ldx % 4 == 0, "aggregate_max_bwd: x must be 16-byte aligned rows");
  RGCN_CHECK_ARG(!init || (((uintptr_t)init & 15) == 0 && ld_init % 4 == 0), "aggregate_max_bwd: init misaligned");
  RGCN_CHECK_ARG(gX && ((uintptr_t)gX & 15) == 0 && ldgx % 4 == 0, "aggregate_max_bwd: output must be 16-byte aligned rows");
  if (gt->n_rows == 0) return RGCN_OK;
  p.X = X; p.ldx = ldx; p.Hmax = Hmax; p.Hcnt = Hcnt; p.ldm = ldm; p.gH = gH; p.ldg = ldg;
  p.init = init; p.ld_init = ld_init; p.gX = gX; p.ldgx = ldgx;
  return dispatch_max<true>(p, (cudaStream_t)stream);
}
