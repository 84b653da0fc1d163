// Fused DistMult decoder: row gathers node_embeddings[head], [tail] (reference
// src/models/rgcn.py:325-326) + LinkPredictor.forward (src/models/rgcn.py:207-211) in one kernel,
// and its backward.  One warp per (head, relation, tail) pair, 128-bit loads, shuffle reduction.
#include "common.cuh"

namespace rgcn {

__global__ void __launch_bounds__(256) distmult_fwd_kernel(const float* __restrict__ emb_h, int64_t ld_h,
                                                           const float* __restrict__ emb_t, int64_t ld_t,
                                                           const int64_t* __restrict__ head,
                                                           const int64_t* __restrict__ tail,
                                                           const int64_t* __restrict__ rel,
                                                           const float* __restrict__ rel_table,
                                                           const float* __restrict__ rel_rows,
                                                           const float* __restrict__ rel_scale, int64_t n_pairs,
                                                           int32_t d, float* __restrict__ score) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int64_t p = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (p >= n_pairs) return;
  const float* h = emb_h + (head ? head[p] : p) * ld_h;
  const float* t = emb_t + (tail ? tail[p] : p) * ld_t;
  const float* r = rel_rows ? rel_rows + p * d : rel_table + rel[p] * d;
  float s = 0.f;
  for (int vi = lane; vi < (d >> 2); vi += 32) {
    const float4 a = ldg4(h + vi * 4), c = ldg4(t + vi * 4);
    float4 b = ldg4(r + vi * 4);
    if (rel_scale) {   // dropout on the relation row: mask / (1 - p), drawn by the caller
      const float4 m = ldg4(rel_scale + p * d + vi * 4);
      b.x *= m.x; b.y *= m.y; b.z *= m.z; b.w *= m.w;
    }
    // (h * r) * t, summed in element order inside the lane like torch.sum's pairwise tree is not
    // reproduced bit for bit; the tolerance of the parity tests covers the reduction order
    s += a.x * b.x * c.x;
    s += a.y * b.y * c.y;
    s += a.z * b.z * c.z;
    s += a.w * b.w * c.w;
  }
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) score[p] = s;
}

__global__ void __launch_bounds__(256) distmult_bwd_kernel(const float* __restrict__ emb_h, int64_t ld_h,
                                                           const float* __restrict__ emb_t, int64_t ld_t,
                                                           const int64_t* __restrict__ head,
                                                           const int64_t* __restrict__ tail,
                                                           const int64_t* __restrict__ rel,
                                                           const float* __restrict__ rel_table,
                                                           const float* __restrict__ rel_rows,
                                                           const float* __restrict__ rel_scale,
                                                           const float* __restrict__ g_score, int64_t n_pairs,
                                                           int32_t d, float* __restrict__ g_h, int64_t ld_gh,
                                                           float* __restrict__ g_t, int64_t ld_gt,
                                                           float* __restrict__ g_rel_table,
                                                           float* __restrict__ g_rel_rows) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int64_t p = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (p >= n_pairs) return;
  const int64_t hi = head ? head[p] : p, ti = tail ? tail[p] : p;
  const float* h = emb_h + hi * ld_h;
  const float* t = emb_t + ti * ld_t;
  const float* r = rel_rows ? rel_rows + p * d : rel_table + rel[p] * d;
  const float g = g_score[p];
  for (int vi = lane; vi < (d >> 2); vi += 32) {
    const float4 a = ldg4(h + vi * 4), c = ldg4(t + vi * 4);
    float4 b = ldg4(r + vi * 4);
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (rel_scale) {
      m = ldg4(rel_scale + p * d + vi * 4);
      b.x *= m.x; b.y *= m.y; b.z *= m.z; b.w *= m.w;
    }
    const float4 gh = make_float4(g * b.x * c.x, g * b.y * c.y, g * b.z * c.z, g * b.w * c.w);
    const float4 gt = make_float4(g * a.x * b.x, g * a.y * b.y, g * a.z * b.z, g * a.w * b.w);
    const float4 gr = make_float4(g * a.x * c.x * m.x, g * a.y * c.y * m.y, g * a.z * c.z * m.z, g * a.w * c.w * m.w);
    // gathered rows may repeat => fp32 atomics; identity rows are written exactly once => plain stores
    if (head) atomicAdd(reinterpret_cast<float4*>(g_h + hi * ld_gh + vi * 4), gh);
    else *reinterpret_cast<float4*>(g_h + hi * ld_gh + vi * 4) = gh;
    if (tail) atomicAdd(reinterpret_cast<float4*>(g_t + ti * ld_gt + vi * 4), gt);
    else *reinterpret_cast<float4*>(g_t + ti * ld_gt + vi * 4) = gt;
    if (g_rel_rows) *reinterpret_cast<float4*>(g_rel_rows + p * d + vi * 4) = gr;
    if (g_rel_table) atomicAdd(reinterpret_cast<float4*>(g_rel_table + rel[p] * d + vi * 4), gr);
  }
}

// The accuracy decision of reference src/train.py:321-322, sigmoid(x) > 0.5 in fp32, given e = expf(-|x|): not the same
// as x > 0, since 1 / (1 + expf(-x)) rounds to 0.5 for 0 < x < ~9e-8.  False for x <= 0 and for NaN.
__device__ __forceinline__ bool sigmoid_above_half(float x, float e) { return x > 0.f && 1.f / (1.f + e) > 0.5f; }

// loss = mean_i [ max(x,0) - x*y + log1p(exp(-|x|)) ]   (= torch BCEWithLogitsLoss, reference src/train.py:139, :300)
// one block, fixed-order tree => deterministic; also counts sigmoid(x) > 0.5 == y (the accuracy of src/train.py:321-322)
__global__ void __launch_bounds__(1024) bce_logits_fwd_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                              int64_t n, float* __restrict__ loss,
                                                              int32_t* __restrict__ n_correct) {
  pdl_enter();
  __shared__ float sl[32];
  __shared__ int sc[32];
  float acc = 0.f;
  int cor = 0;
  for (int64_t i = threadIdx.x; i < n; i += 1024) {
    const float v = x[i], t = y[i];
    const float e = expf(-fabsf(v));
    acc += fmaxf(v, 0.f) - v * t + log1pf(e);
    cor += (sigmoid_above_half(v, e) ? 1.f : 0.f) == t;
  }
  for (int o = 16; o; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    cor += __shfl_xor_sync(0xffffffffu, cor, o);
  }
  if ((threadIdx.x & 31) == 0) { sl[threadIdx.x >> 5] = acc; sc[threadIdx.x >> 5] = cor; }
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = sl[threadIdx.x]; cor = sc[threadIdx.x];
    for (int o = 16; o; o >>= 1) {
      acc += __shfl_xor_sync(0xffffffffu, acc, o);
      cor += __shfl_xor_sync(0xffffffffu, cor, o);
    }
    if (threadIdx.x == 0) {
      *loss = acc / (float)n;
      if (n_correct) *n_correct = cor;
    }
  }
}

// g_x[i] = g_loss * (sigmoid(x_i) - y_i) / n
__global__ void bce_logits_bwd_kernel(const float* __restrict__ x, const float* __restrict__ y, int64_t n,
                                      const float* __restrict__ g_loss, float* __restrict__ g_x) {
  pdl_enter();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = 1.f / (1.f + expf(-x[i]));
  g_x[i] = (*g_loss) * (s - y[i]) / (float)n;
}

// ---- fused training-step tail (SURVEY §8f row 2): sampler, and DistMult + BCE-with-logits + accuracy in one pair ----
__device__ __forceinline__ uint32_t pcg32(uint32_t x) {
  uint32_t state = x * 747796405u + 2891336453u;
  uint32_t word = ((state >> ((state >> 28u) + 4u)) ^ state) * 277803737u;
  return (word >> 22u) ^ word;
}
// two independent 32-bit draws for item i of step `ctr`
__device__ __forceinline__ uint2 draw2(uint32_t seed, unsigned long long ctr, uint32_t i) {
  const uint32_t k = pcg32(seed ^ (uint32_t)ctr) + (uint32_t)(ctr >> 32) * 0x9E3779B9u;
  const uint32_t a = pcg32(i ^ k);
  return make_uint2(a, pcg32(a + 0x85EBCA6Bu + i));
}

// entity draw of attempt j >= 1 of negative i: a re-hash of attempt 0's side word x (itself a hash of seed, counter
// value and i) with j — a pure function of (seed, counter value, i, j)
__device__ __forceinline__ uint32_t redraw(uint32_t x, uint32_t i, uint32_t j) {
  return pcg32(pcg32(x ^ (j * 0x9E3779B9u)) + i);
}

// (key, t) in the lexicographically sorted pairs (keys[k], tails[k]), k < n: one binary search over both columns,
// the two loads of a step issued together
__device__ __forceinline__ bool known_triple(const int64_t* __restrict__ keys, const int32_t* __restrict__ tails,
                                             int64_t n, int64_t key, int32_t t) {
  int64_t lo = 0, len = n;
  while (len > 0) {
    const int64_t half = len >> 1, m = lo + half;
    const int64_t km = __ldg(keys + m);
    const int32_t tm = __ldg(tails + m);
    if (km < key || (km == key && tm < t)) { lo = m + 1; len -= half + 1; }
    else len = half;
  }
  return lo < n && __ldg(keys + lo) == key && __ldg(tails + lo) == t;
}

// Negative sampling of reference src/train.py:59-97 + the concatenation / labels of :281-288 on device: out[0 .. n_pos)
// = the positives (label 1); out[n_pos + i * num_neg + k] = positive i with its head (probability head_prob[r], default
// 1/2) or else its tail replaced (label 0) by a node drawn uniformly from the relation's admissible list for that side
// (default: all nodes), redrawn while the corrupted triple is a known one (rgcn_link_batch_ex).  Every thread reads the
// step counter first; one block: thread 0 then advances it, several blocks: the last block to finish does — a captured
// graph draws fresh negatives on every replay.
__global__ void __launch_bounds__(1024) link_batch_kernel(const rgcn_link_batch_args a) {
  pdl_enter();
  const unsigned long long c = *a.counter;
  __syncthreads();
  const bool one_block = gridDim.x == 1;
  if (one_block && threadIdx.x == 0) *a.counter = c + 1ull;
  const int64_t n_neg = a.n_pos * a.num_neg, n_out = a.n_pos + n_neg;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += stride) {
    if (i < a.n_pos) {
      a.heads[i] = a.pos_head[i]; a.tails[i] = a.pos_tail[i]; a.rels[i] = a.pos_rel[i]; a.labels[i] = 1.f;
      continue;
    }
    const int64_t q = (i - a.n_pos) / a.num_neg;
    const uint32_t ni = (uint32_t)(i - a.n_pos);
    const uint2 r = draw2(a.seed, c, ni);
    const int64_t hq = a.pos_head[q], tq = a.pos_tail[q], rq = a.pos_rel[q];
    const bool rel_ok = rq >= 0 && rq < (int64_t)a.num_rel;      // else: no table is read
    // head with probability p: x >= (1 - p) 2^32, which for p = 1/2 is the top bit and is exact for p = 0 and 1
    unsigned long long thr = 1ull << 31;
    if (a.head_prob && rel_ok) thr = (unsigned long long)((1.0 - (double)a.head_prob[rq]) * 4294967296.0);
    const bool corrupt_head = (unsigned long long)r.x >= thr;
    const int64_t* offs = corrupt_head ? a.head_offsets : a.tail_offsets;
    const int32_t* nodes = corrupt_head ? a.head_nodes : a.tail_nodes;
    int64_t base = 0, len = 0;                                    // len 0: all nodes
    if (offs && rel_ok) { base = offs[rq]; len = offs[rq + 1] - base; }
    const int64_t kept = corrupt_head ? tq : hq;
    const bool filtered = a.filter_keys && rel_ok && kept >= 0 && kept < a.num_nodes;
    uint32_t y = r.y;
    int64_t ent;
    for (int32_t j = 0;;) {
      // uniform in [0, len): multiply-shift of a 32-bit draw (bias < len / 2^32)
      ent = len > 0 ? (int64_t)__ldg(nodes + base + (int64_t)(((unsigned long long)y * (unsigned long long)len) >> 32))
                    : (int64_t)(((unsigned long long)y * (unsigned long long)a.num_nodes) >> 32);
      if (!filtered ||
          !known_triple(a.filter_keys, a.filter_tails, a.n_filter, (corrupt_head ? ent : hq) * a.num_rel + rq,
                        (int32_t)(corrupt_head ? tq : ent)))
        break;
      if (++j == a.max_tries) {                                   // keep the last draw
        if (a.exhausted) atomicAdd(a.exhausted, 1ull);
        break;
      }
      y = redraw(r.x, ni, (uint32_t)j);
    }
    a.heads[i] = corrupt_head ? ent : hq;
    a.tails[i] = corrupt_head ? tq : ent;
    a.rels[i] = rq; a.labels[i] = 0.f;
  }
  if (!one_block) {
    // every thread of this block has read the counter; the last block to arrive advances it
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(a.ticket, 1u) == gridDim.x - 1) {
        *a.ticket = 0u;                               // ready for the next launch (graph replay)
        *a.counter = c + 1ull;
      }
    }
  }
}

// keep-mask of the decoder's dropout on the relation row (reference src/models/rgcn.py:207-208): 16 hash bits per
// element of pair p; returns the four multipliers (0 or 1 / (1 - p)) of float4 number vi of the row
__device__ __forceinline__ float4 rel_drop4(uint32_t key, int64_t p, int d, int vi, uint32_t thresh, float scale) {
  const uint32_t e = (uint32_t)(p * d + vi * 4);
  const uint32_t h0 = pcg32(e ^ key), h1 = pcg32((e + 2u) ^ key);
  return make_float4((h0 & 0xffffu) >= thresh ? scale : 0.f, (h0 >> 16) >= thresh ? scale : 0.f,
                     (h1 & 0xffffu) >= thresh ? scale : 0.f, (h1 >> 16) >= thresh ? scale : 0.f);
}

struct LinkLossParams {
  const float* emb; int64_t ld;
  const int64_t* head; const int64_t* tail; const int64_t* rel;
  const float* rel_table; const float* labels;
  int64_t n_pairs; int32_t d;
  uint32_t drop_thresh; float drop_scale; uint32_t seed;     // drop_thresh == 0: no dropout
  unsigned long long* ctr;           // dropout step counter (forward: read by all, advanced by the last block)
  unsigned long long* state;         // forward: out, the counter value used; backward: in
  float* score; float* loss; int32_t* n_correct;
  float* part_loss; int32_t* part_correct; unsigned int* ticket;   // [gridDim.x], [gridDim.x], [1] (zero before launch)
  // index range (n_nodes <= 0: unchecked).  A pair with an out-of-range head / tail / relation is SKIPPED — its score
  // and the loss become NaN, it contributes no gradient — and bit 0 of *status is set (the reference's nn.Embedding
  // raises a device assert there; here the caller polls the flag, see ops.raise_on_bad_pairs)
  int64_t n_nodes; int32_t n_rel; int32_t* status;
};

__device__ __forceinline__ bool pair_ok(const LinkLossParams& q, int64_t hi, int64_t ti, int64_t ri) {
  return q.n_nodes <= 0 || (hi >= 0 && hi < q.n_nodes && ti >= 0 && ti < q.n_nodes && ri >= 0 && ri < (int64_t)q.n_rel);
}

// scores, mean BCE-with-logits loss and the number of correct sigmoid > 0.5 predictions (src/train.py:300, :321-322)
// in ONE kernel: a warp per pair, per-block partials, the last block to finish reduces them in block order.
__global__ void __launch_bounds__(256) link_loss_fwd_kernel(const LinkLossParams q) {
  pdl_enter();
  __shared__ float s_l[8];
  __shared__ int s_c[8];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t p = (int64_t)blockIdx.x * 8 + warp;
  const unsigned long long c = q.drop_thresh ? *q.ctr : 0ull;
  const uint32_t key = pcg32(q.seed ^ (uint32_t)c) + (uint32_t)(c >> 32) * 0x9E3779B9u;
  float l = 0.f;
  int ok = 0;
  if (p < q.n_pairs) {
    const int64_t hi = q.head[p], ti = q.tail[p], ri = q.rel[p];
    const bool in_range = pair_ok(q, hi, ti, ri);
    const float* h = q.emb + (in_range ? hi : 0) * q.ld;
    const float* t = q.emb + (in_range ? ti : 0) * q.ld;
    const float* r = q.rel_table + (in_range ? ri : 0) * q.d;
    float s = 0.f;
    for (int vi = lane; vi < (q.d >> 2); vi += 32) {
      const float4 a = ldg4(h + vi * 4), cc = ldg4(t + vi * 4);
      float4 b = ldg4(r + vi * 4);
      if (q.drop_thresh) {
        const float4 m = rel_drop4(key, p, q.d, vi, q.drop_thresh, q.drop_scale);
        b.x *= m.x; b.y *= m.y; b.z *= m.z; b.w *= m.w;
      }
      s += a.x * b.x * cc.x; s += a.y * b.y * cc.y; s += a.z * b.z * cc.z; s += a.w * b.w * cc.w;
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (!in_range) {
      s = __int_as_float(0x7fc00000);                // NaN: visible in the scores and in the loss
      if (lane == 0 && q.status) atomicOr(q.status, 1);
    }
    if (q.labels) {                                  // NULL: scores only (LinkPredictor.score_pairs)
      const float y = q.labels[p];
      const float e = expf(-fabsf(s));
      l = fmaxf(s, 0.f) - s * y + log1pf(e);
      ok = ((sigmoid_above_half(s, e) ? 1.f : 0.f) == y) ? 1 : 0;
    }
    if (lane == 0) q.score[p] = s;
  }
  if (lane == 0) { s_l[warp] = l; s_c[warp] = ok; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float bl = 0.f; int bc = 0;
    for (int w = 0; w < 8; ++w) { bl += s_l[w]; bc += s_c[w]; }
    q.part_loss[blockIdx.x] = bl; q.part_correct[blockIdx.x] = bc;
    __threadfence();
    s_last = atomicAdd(q.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  // last block: every block has read the counter and published its partial
  __threadfence();
  float acc = 0.f; int cor = 0;
  if (threadIdx.x < 32) {
    // fixed order: lane-strided partials, then a fixed butterfly => same bits on every run
    for (int b = threadIdx.x; b < (int)gridDim.x; b += 32) {
      acc += *((volatile float*)q.part_loss + b);
      cor += *((volatile int*)q.part_correct + b);
    }
    for (int o = 16; o; o >>= 1) {
      acc += __shfl_xor_sync(0xffffffffu, acc, o);
      cor += __shfl_xor_sync(0xffffffffu, cor, o);
    }
    if (threadIdx.x == 0) {
      if (q.loss) *q.loss = acc / (float)q.n_pairs;
      if (q.n_correct) *q.n_correct = cor;
      *q.ticket = 0u;                               // ready for the next launch (graph replay)
      if (q.state) *q.state = c;
      if (q.drop_thresh) *q.ctr = c + 1ull;
    }
  }
}

// g_score[p] = g_loss * (sigmoid(s_p) - y_p) / n folded into the DistMult backward: node-row gradients scattered into
// the dense [N, d] buffer (zeroed by the caller), relation-table gradient accumulated
__global__ void __launch_bounds__(256) link_loss_bwd_kernel(const LinkLossParams q, const float* __restrict__ g_loss,
                                                            const float* __restrict__ g_score,
                                                            float* __restrict__ g_emb, int64_t ld_g,
                                                            float* __restrict__ g_rel_table, int32_t n_rel_smem) {
  pdl_enter();
  // the relation table has few rows that every pair hits: the block's 8 pairs are pre-reduced in shared memory
  // (n_rel_smem rows, 0 = table too large: straight global atomics) and flushed with one atomic per touched element
  extern __shared__ float s_tab[];
  const int lane = threadIdx.x & 31;
  const int64_t p = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const bool tab_smem = g_rel_table && n_rel_smem > 0;
  if (tab_smem) {
    for (int i = threadIdx.x; i < n_rel_smem * q.d; i += 256) s_tab[i] = 0.f;
    __syncthreads();
  }
  if (p < q.n_pairs) {
    const unsigned long long c = q.drop_thresh ? *q.state : 0ull;
    const uint32_t key = pcg32(q.seed ^ (uint32_t)c) + (uint32_t)(c >> 32) * 0x9E3779B9u;
    const int64_t hi = q.head[p], ti = q.tail[p], ri = q.rel[p];
    const bool in_range = pair_ok(q, hi, ti, ri);
    const float* h = q.emb + (in_range ? hi : 0) * q.ld;
    const float* t = q.emb + (in_range ? ti : 0) * q.ld;
    const float* r = q.rel_table + (in_range ? ri : 0) * q.d;
    float g;
    if (g_score) {
      g = g_score[p];                                // scores-only form: the incoming gradient of score[p]
    } else {
      const float s = q.score[p];
      g = (*g_loss) * (1.f / (1.f + expf(-s)) - q.labels[p]) / (float)q.n_pairs;
    }
    for (int vi = lane; in_range && vi < (q.d >> 2); vi += 32) {
      const float4 a = ldg4(h + vi * 4), cc = ldg4(t + vi * 4);
      float4 b = ldg4(r + vi * 4);
      float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
      if (q.drop_thresh) {
        m = rel_drop4(key, p, q.d, vi, q.drop_thresh, q.drop_scale);
        b.x *= m.x; b.y *= m.y; b.z *= m.z; b.w *= m.w;
      }
      const float4 gh = make_float4(g * b.x * cc.x, g * b.y * cc.y, g * b.z * cc.z, g * b.w * cc.w);
      const float4 gt = make_float4(g * a.x * b.x, g * a.y * b.y, g * a.z * b.z, g * a.w * b.w);
      atomicAdd(reinterpret_cast<float4*>(g_emb + hi * ld_g + vi * 4), gh);
      atomicAdd(reinterpret_cast<float4*>(g_emb + ti * ld_g + vi * 4), gt);
      if (g_rel_table) {
        const float4 gr = make_float4(g * a.x * cc.x * m.x, g * a.y * cc.y * m.y, g * a.z * cc.z * m.z, g * a.w * cc.w * m.w);
        if (tab_smem) {
          float* dst = s_tab + ri * q.d + vi * 4;
          atomicAdd(dst, gr.x); atomicAdd(dst + 1, gr.y); atomicAdd(dst + 2, gr.z); atomicAdd(dst + 3, gr.w);
        } else {
          atomicAdd(reinterpret_cast<float4*>(g_rel_table + ri * q.d + vi * 4), gr);
        }
      }
    }
  }
  if (tab_smem) {
    __syncthreads();
    for (int i = threadIdx.x; i < n_rel_smem * (q.d >> 2); i += 256) {
      const float4 v = *reinterpret_cast<const float4*>(s_tab + i * 4);
      if (v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f) atomicAdd(reinterpret_cast<float4*>(g_rel_table) + i, v);
    }
  }
}


// ---- deterministic backward of the fused decoder (no atomics on floating-point data) --------------------------------
// The 2 n gathered rows (positions 0 .. n-1 = the heads, n .. 2n-1 = the tails) repeat: a hub gene is the head or tail
// of dozens of pairs of one batch.  Instead of fp32 atomics (whose order differs from run to run):
//   1. link_contrib_kernel, one warp per POSITION (fully parallel): C[q] = the contribution of position q to its node's
//      gradient row, T[p] = the contribution of pair p to its relation's row; the same launch writes rows[q] and finds
//      every listed node's OWNER — its first position, slot[node] — with an integer atomicMin;
//   2. link_gather_kernel: the owner's warp collects the positions that list its node (a scan of the position list in
//      shared memory), then adds their C rows in ascending position order, eight loads in flight; rows nobody lists are
//      zero-filled by other blocks of the same launch — every row of the dense [N, d] gradient is written exactly once, no
//      memset; further blocks add T rows per relation over 32-pair chunks in pair order (partials), which
//   3. rgcn_reduce_partials sums in a fixed order.
// slot / rows are handed to the last encoder layer's row-sparse backward (csrc/rowsparse.cu) as they are.
struct LinkBwdRows {
  const float* g_loss; const float* g_score;
  float* g_emb; int64_t ld_g; int64_t n_rows;       // [n_rows, d]
  int32_t* slot; int64_t* rows; int32_t unlisted;
  float* C;                                         // [2 n, d] position contributions
  float* T;                                         // [n, d] pair contributions to the relation table, nullable
  float* tab_partial;                               // [n_tab_blocks, n_rel * d], nullable
  int32_t n_owner_blocks, n_zero_blocks, n_tab_blocks;
  int32_t rows_in_smem;                             // the launch has 2 n ints of dynamic shared memory for the position list
};
constexpr int kLinkZeroRows = 64;                    // rows per zero-fill block
constexpr int kLinkTabPairs = 32;                    // pairs per relation-table partial
constexpr int kLinkList = 128;                        // positions of one node collected before they are added

__device__ __forceinline__ float link_pair_grad(const LinkLossParams& q, const LinkBwdRows& b, int64_t p) {
  if (b.g_score) return b.g_score[p];
  const float s = q.score[p];
  return (*b.g_loss) * (1.f / (1.f + expf(-s)) - q.labels[p]) / (float)q.n_pairs;
}

__global__ void __launch_bounds__(256) link_contrib_kernel(const LinkLossParams q, const LinkBwdRows b) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int nv = q.d >> 2;
  const int64_t n = q.n_pairs;
  const int64_t pos = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (pos >= 2 * n) return;
  const bool is_head = pos < n;
  const int64_t p = is_head ? pos : pos - n;
  const int64_t hi = q.head[p], ti = q.tail[p], ri = q.rel[p];
  const bool ok = pair_ok(q, hi, ti, ri);
  if (lane == 0) {
    b.rows[pos] = ok ? (is_head ? hi : ti) : 0;      // an invalid pair parks on row 0, which it never owns
    if (ok) atomicMin(b.slot + (is_head ? hi : ti), (int32_t)pos);
    else if (q.status) atomicOr(q.status, 1);
  }
  float* __restrict__ crow = b.C + pos * q.d;
  float* __restrict__ trow = (b.T && is_head) ? b.T + p * q.d : nullptr;
  if (!ok) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int vi = lane; vi < nv; vi += 32) {
      *reinterpret_cast<float4*>(crow + vi * 4) = z;
      if (trow) *reinterpret_cast<float4*>(trow + vi * 4) = z;
    }
    return;
  }
  const unsigned long long c = q.drop_thresh ? *q.state : 0ull;
  const uint32_t key = pcg32(q.seed ^ (uint32_t)c) + (uint32_t)(c >> 32) * 0x9E3779B9u;
  const float g = link_pair_grad(q, b, p);
  const float* __restrict__ h = q.emb + hi * q.ld;
  const float* __restrict__ t = q.emb + ti * q.ld;
  const float* __restrict__ r = q.rel_table + ri * q.d;
  for (int vi = lane; vi < nv; vi += 32) {
    const float4 a = ldg4(h + vi * 4), cc = ldg4(t + vi * 4);
    float4 w = ldg4(r + vi * 4);
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (q.drop_thresh) {
      m = rel_drop4(key, p, q.d, vi, q.drop_thresh, q.drop_scale);
      w.x *= m.x; w.y *= m.y; w.z *= m.z; w.w *= m.w;
    }
    const float4 o = is_head ? cc : a;               // the partner row
    *reinterpret_cast<float4*>(crow + vi * 4) = make_float4(g * w.x * o.x, g * w.y * o.y, g * w.z * o.z, g * w.w * o.w);
    if (trow)
      *reinterpret_cast<float4*>(trow + vi * 4) =
          make_float4(g * a.x * cc.x * m.x, g * a.y * cc.y * m.y, g * a.z * cc.z * m.z, g * a.w * cc.w * m.w);
  }
}

constexpr int kLinkInFlight = 12;
__global__ void __launch_bounds__(256, 2) link_gather_kernel(const LinkLossParams q, const LinkBwdRows b) {
  pdl_enter();
  extern __shared__ int s_rows[];                    // [2 n rounded up to 128] node of every position (owner blocks)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nv = q.d >> 2;
  const int64_t n = q.n_pairs, n2 = 2 * q.n_pairs;
  int blk = blockIdx.x;
  if (blk < b.n_owner_blocks) {
    // ---- one warp per position; only the node's first position (its owner) works ----
    const int64_t n2p = (n2 + 127) & ~int64_t(127);
    if (b.rows_in_smem) {
      for (int64_t i = threadIdx.x; i < n2p; i += 256) s_rows[i] = i < n2 ? (int)b.rows[i] : -1;
      __syncthreads();
    }
    const int64_t pos = (int64_t)blk * 8 + warp;
    if (pos >= n2) return;
    const int64_t v = b.rows[pos];
    if (__ldg(b.slot + v) != (int32_t)pos) return;
    __shared__ int s_list[8][kLinkList];
    int* list = s_list[warp];
    for (int v0 = 0; v0 < nv; v0 += 64) {            // column passes of two 128-bit vectors per lane
      const int vi0 = v0 + lane, vi1 = v0 + 32 + lane;
      const bool on0 = vi0 < nv, on1 = vi1 < nv;
      const int c0 = on0 ? vi0 * 4 : 0, c1 = on1 ? vi1 * 4 : 0;
      float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
      auto flush = [&](int count) {
        __syncwarp();
        // kLinkInFlight rows in flight, added strictly in list (= position) order: a hub gene heads or tails dozens of
        // pairs of one batch, and its owner's chain of dependent load rounds is what the kernel's duration is
        for (int j = 0; j < count; j += kLinkInFlight) {
          float4 x0[kLinkInFlight], x1[kLinkInFlight];
#pragma unroll
          for (int u = 0; u < kLinkInFlight; ++u) {
            const int e = min(j + u, count - 1);
            const float* __restrict__ row = b.C + (int64_t)list[e] * q.d;
            x0[u] = *reinterpret_cast<const float4*>(row + c0);
            x1[u] = *reinterpret_cast<const float4*>(row + c1);
          }
#pragma unroll
          for (int u = 0; u < kLinkInFlight; ++u) {
            if (j + u < count) { add4(acc0, x0[u]); add4(acc1, x1[u]); }
          }
        }
        __syncwarp();
      };
      int cnt = 0;
      const int vi = (int)v;
      if (b.rows_in_smem) {
        // windows of 128 positions, four per lane (one 128-bit shared-memory load); a window without a match — nearly
        // all of them — costs one vote
        for (int64_t base = pos & ~int64_t(127); base < n2p; base += 128) {
          const int4 w = *reinterpret_cast<const int4*>(s_rows + base + lane * 4);
          const int64_t p0 = base + lane * 4;
          const unsigned mk = (unsigned)(w.x == vi && p0 >= pos) | ((unsigned)(w.y == vi && p0 + 1 >= pos) << 1) |
                              ((unsigned)(w.z == vi && p0 + 2 >= pos) << 2) | ((unsigned)(w.w == vi && p0 + 3 >= pos) << 3);
          if (!__any_sync(0xffffffffu, mk != 0u)) continue;
          // ascending positions = lane-major, then the lane's four: exclusive prefix of the lanes' match counts
          int mine = __popc(mk), before = mine;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, before, o);
            if (lane >= o) before += up;
          }
          const int total = __shfl_sync(0xffffffffu, before, 31);
          before -= mine;
          if (cnt + total > kLinkList) { flush(cnt); cnt = 0; }
          int at = cnt + before;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (mk & (1u << j)) list[at++] = (int)(p0 + j);
          cnt += total;
        }
      } else {
        for (int64_t base = pos & ~int64_t(31); base < n2; base += 32) {
          const int64_t pp = base + lane;
          const bool match = pp >= pos && pp < n2 && b.rows[pp] == v;
          const unsigned m = __ballot_sync(0xffffffffu, match);
          if (!m) continue;
          const int k = __popc(m);
          if (cnt + k > kLinkList) { flush(cnt); cnt = 0; }
          if (match) list[cnt + __popc(m & ((1u << lane) - 1u))] = (int)pp;
          cnt += k;
        }
      }
      flush(cnt);
      if (on0) *reinterpret_cast<float4*>(b.g_emb + v * b.ld_g + c0) = acc0;
      if (on1) *reinterpret_cast<float4*>(b.g_emb + v * b.ld_g + c1) = acc1;
    }
    return;
  }
  blk -= b.n_owner_blocks;
  if (blk < b.n_zero_blocks) {
    // ---- rows nobody lists: zeros ----
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < kLinkZeroRows / 8; ++k) {
      const int64_t row = (int64_t)blk * kLinkZeroRows + k * 8 + warp;
      if (row < b.n_rows && __ldg(b.slot + row) == b.unlisted)
        for (int vi = lane; vi < nv; vi += 32) *reinterpret_cast<float4*>(b.g_emb + row * b.ld_g + vi * 4) = z;
    }
    return;
  }
  blk -= b.n_zero_blocks;
  // ---- relation-table gradient: partial of kLinkTabPairs consecutive pairs, their T rows added in pair order ----
  __shared__ int s_r[kLinkTabPairs];
  const int64_t p0 = (int64_t)blk * kLinkTabPairs;
  if (threadIdx.x < kLinkTabPairs) {
    const int64_t p = p0 + threadIdx.x;
    int r = -1;
    if (p < n) {
      const int64_t hi = q.head[p], ti = q.tail[p], ri = q.rel[p];
      if (pair_ok(q, hi, ti, ri)) r = (int)ri;
    }
    s_r[threadIdx.x] = r;
  }
  __syncthreads();
  float* __restrict__ part = b.tab_partial + (size_t)blk * q.n_rel * q.d;
  const int np = (int)min((int64_t)kLinkTabPairs, n - p0);
  for (int o = threadIdx.x; o < q.n_rel * nv; o += 256) {
    const int r = o / nv, vi = o % nv;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k0 = 0; k0 < np; k0 += 8) {
      float4 x[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int k = min(k0 + u, np - 1);
        x[u] = *reinterpret_cast<const float4*>(b.T + (p0 + k) * q.d + vi * 4);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (k0 + u < np && s_r[k0 + u] == r) add4(acc, x[u]);
    }
    *reinterpret_cast<float4*>(part + (size_t)r * q.d + vi * 4) = acc;
  }
}

// 1 when any index is out of range
__global__ void check_pairs_kernel(const int64_t* head, const int64_t* tail, const int64_t* rel, int64_t n_pairs,
                                   int64_t n_nodes, int32_t n_rel, int32_t* flag) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pairs) return;
  if (head[p] < 0 || head[p] >= n_nodes || tail[p] < 0 || tail[p] >= n_nodes || (rel && (rel[p] < 0 || rel[p] >= n_rel)))
    atomicOr(flag, 1);
}

}  // namespace rgcn

using namespace rgcn;

static int check_dm(const float* emb_h, int64_t ld_h, const float* emb_t, int64_t ld_t, const int64_t* rel,
                    const float* rel_table, const float* rel_rows, int64_t n_pairs, int32_t d) {
  RGCN_CHECK_ARG(n_pairs >= 0 && d >= 4 && d % 4 == 0, "distmult: d=%d must be a positive multiple of 4", d);
  RGCN_CHECK_ARG(n_pairs == 0 || (emb_h && emb_t), "distmult: null embeddings");
  RGCN_CHECK_ARG(ld_h % 4 == 0 && ld_t % 4 == 0 && (((uintptr_t)emb_h | (uintptr_t)emb_t) & 15) == 0,
                 "distmult: embeddings must be 16-byte aligned rows");
  RGCN_CHECK_ARG(rel_rows || (rel_table && rel), "distmult: need rel_rows or (rel_table, rel)");
  RGCN_CHECK_ARG((((uintptr_t)rel_rows | (uintptr_t)rel_table) & 15) == 0, "distmult: relation rows must be 16-byte aligned");
  return RGCN_OK;
}
#define CHECK_SCALE(s) RGCN_CHECK_ARG((((uintptr_t)(s)) & 15) == 0, "distmult: rel_scale must be 16-byte aligned")

extern "C" int rgcn_distmult_fwd(const float* emb_h, int64_t ld_h, const float* emb_t, int64_t ld_t,
                                 const int64_t* head, const int64_t* tail, const int64_t* rel,
                                 const float* rel_table, const float* rel_rows, const float* rel_scale,
                                 int64_t n_pairs, int32_t d, float* score, rgcn_stream_t stream) {
  int rc = check_dm(emb_h, ld_h, emb_t, ld_t, rel, rel_table, rel_rows, n_pairs, d);
  if (rc) return rc;
  if (n_pairs == 0) return RGCN_OK;
  CHECK_SCALE(rel_scale);
  RGCN_CHECK_ARG(score, "distmult_fwd: null output");
  RGCN_CUDA(launch_pdl(distmult_fwd_kernel, dim3((unsigned)((n_pairs + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, 
      emb_h, ld_h, emb_t, ld_t, head, tail, rel, rel_table, rel_rows, rel_scale, n_pairs, d, score));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_distmult_bwd(const float* emb_h, int64_t ld_h, const float* emb_t, int64_t ld_t,
                                 const int64_t* head, const int64_t* tail, const int64_t* rel,
                                 const float* rel_table, const float* rel_rows, const float* rel_scale,
                                 const float* g_score, int64_t n_pairs, int32_t d, float* g_h, int64_t ld_gh, float* g_t, int64_t ld_gt,
                                 float* g_rel_table, float* g_rel_rows, rgcn_stream_t stream) {
  int rc = check_dm(emb_h, ld_h, emb_t, ld_t, rel, rel_table, rel_rows, n_pairs, d);
  if (rc) return rc;
  if (n_pairs == 0) return RGCN_OK;
  RGCN_CHECK_ARG(g_score && g_h && g_t && ld_gh % 4 == 0 && ld_gt % 4 == 0 &&
                 (((uintptr_t)g_h | (uintptr_t)g_t) & 15) == 0, "distmult_bwd: bad gradient buffers");
  CHECK_SCALE(rel_scale);
  RGCN_CHECK_ARG(!g_rel_table || rel, "distmult_bwd: g_rel_table needs rel");
  RGCN_CUDA(launch_pdl(distmult_bwd_kernel, dim3((unsigned)((n_pairs + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, 
      emb_h, ld_h, emb_t, ld_t, head, tail, rel, rel_table, rel_rows, rel_scale, g_score, n_pairs, d, g_h, ld_gh, g_t, ld_gt,
      g_rel_table, g_rel_rows));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}
extern "C" int rgcn_check_pairs(const int64_t* head, const int64_t* tail, const int64_t* rel, int64_t n_pairs,
                                int64_t n_nodes, int32_t n_rel, int32_t* flag, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(flag && (n_pairs == 0 || (head && tail)), "check_pairs: null argument");
  RGCN_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), (cudaStream_t)stream));
  if (n_pairs == 0) return RGCN_OK;
  check_pairs_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(head, tail, rel, n_pairs,
                                                                                          n_nodes, n_rel, flag);
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_bce_logits_fwd(const float* logits, const float* labels, int64_t n, float* loss, int32_t* n_correct,
                                   rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n > 0 && logits && labels && loss, "bce_logits_fwd: bad arguments");
  RGCN_CUDA(launch_pdl(bce_logits_fwd_kernel, dim3(1), dim3(1024), 0, (cudaStream_t)stream, logits, labels, n, loss, n_correct));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_bce_logits_bwd(const float* logits, const float* labels, int64_t n, const float* g_loss,
                                   float* g_logits, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(n > 0 && logits && labels && g_loss && g_logits, "bce_logits_bwd: bad arguments");
  RGCN_CUDA(launch_pdl(bce_logits_bwd_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, logits, labels, n, g_loss, g_logits));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_link_batch_ex(const rgcn_link_batch_args* args_host, rgcn_stream_t stream) {
  RGCN_CHECK_ARG(args_host, "link_batch: null args");
  const rgcn_link_batch_args& a = *args_host;
  RGCN_CHECK_ARG(a.n_pos >= 0 && a.num_neg >= 0 && a.num_nodes > 0 && a.num_nodes < (1ll << 32) && a.num_rel >= 0 &&
                 a.n_filter >= 0, "link_batch: bad sizes");
  RGCN_CHECK_ARG(a.num_neg == 0 || a.n_pos <= (int64_t)0xffffffffll / a.num_neg,
                 "link_batch: bad sizes (more than 2^32 - 1 negatives)");
  RGCN_CHECK_ARG(a.max_tries >= 1, "link_batch: max_tries must be >= 1");
  RGCN_CHECK_ARG(!a.filter_keys == !a.filter_tails && (a.n_filter == 0 || a.filter_keys),
                 "link_batch: filter_keys and filter_tails must both be null or both be set");
  const int n_type_tables = !!a.head_offsets + !!a.head_nodes + !!a.tail_offsets + !!a.tail_nodes;
  RGCN_CHECK_ARG(n_type_tables == 0 || n_type_tables == 4,
                 "link_batch: the four type-constraint tables must all be null or all be set");
  const bool tables = a.head_prob || a.filter_keys || n_type_tables;
  RGCN_CHECK_ARG(!tables || a.num_rel > 0, "link_batch: head_prob / filter / type tables need num_rel > 0");
  RGCN_CHECK_ARG(!(a.filter_keys || n_type_tables) || a.num_nodes < (1ll << 31),
                 "link_batch: filter / type tables hold int32 node ids: num_nodes must be < 2^31");
  RGCN_CHECK_ARG(a.n_pos == 0 || (a.pos_head && a.pos_tail && a.pos_rel && a.heads && a.tails && a.rels && a.labels &&
                                  a.counter), "link_batch: null argument");
  if (a.n_pos == 0) return RGCN_OK;
  // with a ticket: one thread per output entry, so that num_neg = 16 batches do not queue behind one block
  const int64_t n_out = a.n_pos * (1 + (int64_t)a.num_neg);
  const unsigned grid = a.ticket ? (unsigned)((n_out + 255) / 256) : 1u;
  RGCN_CUDA(launch_pdl(link_batch_kernel, dim3(grid), dim3(a.ticket ? 256 : 1024), 0, (cudaStream_t)stream, a));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_link_batch(const int64_t* pos_head, const int64_t* pos_tail, const int64_t* pos_rel, int64_t n_pos,
                               int32_t num_neg, int64_t num_nodes, uint32_t seed, unsigned long long* counter,
                               int64_t* heads, int64_t* tails, int64_t* rels, float* labels, rgcn_stream_t stream) {
  rgcn_link_batch_args a{};
  a.pos_head = pos_head; a.pos_tail = pos_tail; a.pos_rel = pos_rel; a.n_pos = n_pos; a.num_neg = num_neg;
  a.num_nodes = num_nodes; a.seed = seed; a.max_tries = 1; a.counter = counter;
  a.heads = heads; a.tails = tails; a.rels = rels; a.labels = labels;
  return rgcn_link_batch_ex(&a, stream);
}

static int fill_link_params(LinkLossParams& q, const float* emb, int64_t ld, const int64_t* head, const int64_t* tail,
                            const int64_t* rel, const float* rel_table, const float* labels, int64_t n_pairs, int32_t d,
                            float dropout_p, uint32_t seed, int64_t n_nodes, int32_t n_rel, int32_t* status) {
  RGCN_CHECK_ARG(n_pairs > 0 && d >= 4 && d % 4 == 0, "link_loss: n_pairs must be positive and d a multiple of 4");
  RGCN_CHECK_ARG(emb && head && tail && rel && rel_table, "link_loss: null argument");
  RGCN_CHECK_ARG(ld % 4 == 0 && (((uintptr_t)emb | (uintptr_t)rel_table) & 15) == 0, "link_loss: rows must be 16-byte aligned");
  RGCN_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, "link_loss: dropout_p must be in [0, 1)");
  RGCN_CHECK_ARG(n_pairs * (int64_t)d < (1ll << 32), "link_loss: batch too large for the 32-bit dropout index");
  q.emb = emb; q.ld = ld; q.head = head; q.tail = tail; q.rel = rel; q.rel_table = rel_table; q.labels = labels;
  q.n_pairs = n_pairs; q.d = d; q.seed = seed;
  q.n_nodes = n_nodes; q.n_rel = n_rel; q.status = status;
  q.drop_thresh = 0; q.drop_scale = 1.f;
  if (dropout_p > 0.f) {
    const double th = (double)dropout_p * 65536.0 + 0.5;
    q.drop_thresh = th < 1.0 ? 1u : (uint32_t)th;
    q.drop_scale = 1.f / (1.f - dropout_p);
  }
  return RGCN_OK;
}

extern "C" size_t rgcn_link_loss_workspace_bytes(int64_t n_pairs) {
  const size_t blocks = (size_t)((n_pairs + 7) / 8);
  return align_up(blocks * 8 + 16, 256);
}

extern "C" int rgcn_link_loss_fwd(const float* emb, int64_t ld, const int64_t* head, const int64_t* tail, const int64_t* rel,
                                  const float* rel_table, const float* labels, int64_t n_pairs, int32_t d, float dropout_p,
                                  uint32_t seed, unsigned long long* counter, unsigned long long* state, float* score,
                                  float* loss, int32_t* n_correct, int64_t n_nodes, int32_t n_rel, int32_t* status,
                                  void* workspace, size_t workspace_bytes, rgcn_stream_t stream) {
  LinkLossParams q{};
  int rc = fill_link_params(q, emb, ld, head, tail, rel, rel_table, labels, n_pairs, d, dropout_p, seed, n_nodes, n_rel, status);
  if (rc) return rc;
  RGCN_CHECK_ARG(score && (loss || !labels), "link_loss_fwd: null outputs");
  RGCN_CHECK_ARG(dropout_p == 0.f || (counter && state), "link_loss_fwd: dropout needs the counter and a state slot");
  const size_t blocks = (size_t)((n_pairs + 7) / 8);
  if (!workspace || workspace_bytes < rgcn_link_loss_workspace_bytes(n_pairs)) {
    set_error("link_loss_fwd: workspace too small"); return RGCN_EWORKSPACE;
  }
  q.ctr = counter; q.state = state; q.score = score; q.loss = loss; q.n_correct = n_correct;
  q.part_loss = (float*)workspace; q.part_correct = (int32_t*)((char*)workspace + blocks * 4);
  q.ticket = (unsigned int*)((char*)workspace + blocks * 8);
  RGCN_CUDA(launch_pdl(link_loss_fwd_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, q));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

extern "C" int rgcn_link_loss_bwd(const float* emb, int64_t ld, const int64_t* head, const int64_t* tail, const int64_t* rel,
                                  const float* rel_table, const float* labels, const float* score, const float* g_loss,
                                  const float* g_score,
                                  int64_t n_pairs, int32_t d, float dropout_p, uint32_t seed, const unsigned long long* state,
                                  float* g_emb, int64_t ld_g, float* g_rel_table, int32_t n_rel, int64_t n_nodes,
                                  rgcn_stream_t stream) {
  LinkLossParams q{};
  int rc = fill_link_params(q, emb, ld, head, tail, rel, rel_table, labels, n_pairs, d, dropout_p, seed, n_nodes, n_rel, nullptr);
  if (rc) return rc;
  RGCN_CHECK_ARG(g_emb && ld_g % 4 == 0 && ((uintptr_t)g_emb & 15) == 0, "link_loss_bwd: bad buffers");
  RGCN_CHECK_ARG(g_score || (score && g_loss && labels), "link_loss_bwd: need g_score, or score + labels + g_loss");
  RGCN_CHECK_ARG(dropout_p == 0.f || state, "link_loss_bwd: dropout needs the state the forward wrote");
  RGCN_CHECK_ARG(!g_rel_table || ((uintptr_t)g_rel_table & 15) == 0, "link_loss_bwd: g_rel_table misaligned");
  q.state = const_cast<unsigned long long*>(state); q.score = const_cast<float*>(score);
  const int32_t n_rel_smem = (g_rel_table && n_rel > 0 && (size_t)n_rel * d * 4 <= 40 * 1024) ? n_rel : 0;
  RGCN_CUDA(launch_pdl(link_loss_bwd_kernel, dim3((unsigned)((n_pairs + 7) / 8)), dim3(256), (size_t)n_rel_smem * d * 4,
                       (cudaStream_t)stream, q, g_loss, g_score, g_emb, ld_g, g_rel_table, n_rel_smem));
  RGCN_LAUNCH_CHECK();
  return RGCN_OK;
}

// ---- deterministic form of the backward (link_rows_kernel / link_bwd_rows_kernel above) ----
namespace rgcn {
__global__ void __launch_bounds__(256) link_slot_fill_kernel(int32_t* __restrict__ slot, int64_t n, int32_t unlisted) {
  pdl_enter();
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) slot[i] = unlisted;
}
}

static size_t link_ws_C(int64_t n_pairs, int32_t d) { return align_up((size_t)(2 * n_pairs) * d * sizeof(float), 256); }
static size_t link_ws_T(int64_t n_pairs, int32_t d) { return align_up((size_t)n_pairs * d * sizeof(float), 256); }

extern "C" size_t rgcn_link_bwd_rows_workspace_bytes(int64_t n_pairs, int32_t n_rel, int32_t d) {
  if (n_pairs <= 0 || n_rel <= 0 || d <= 0) return 256;
  const size_t chunks = (size_t)((n_pairs + kLinkTabPairs - 1) / kLinkTabPairs);
  return link_ws_C(n_pairs, d) + link_ws_T(n_pairs, d) + align_up(chunks * (size_t)n_rel * (size_t)d * sizeof(float), 256) + 256;
}

extern "C" int rgcn_link_loss_bwd_rows(const float* emb, int64_t ld, const int64_t* head, const int64_t* tail,
                                       const int64_t* rel, const float* rel_table, const float* labels, const float* score,
                                       const float* g_loss, const float* g_score, int64_t n_pairs, int32_t d,
                                       float dropout_p, uint32_t seed, const unsigned long long* state, int64_t n_nodes,
                                       int32_t n_rel, float* g_emb, int64_t ld_g, float* g_rel_table, int32_t* slot,
                                       int64_t* rows, int32_t* status, int32_t listed_only, void* workspace,
                                       size_t workspace_bytes, rgcn_stream_t stream) {
  LinkLossParams q{};
  int rc = fill_link_params(q, emb, ld, head, tail, rel, rel_table, labels, n_pairs, d, dropout_p, seed, n_nodes, n_rel, status);
  if (rc) return rc;
  RGCN_CHECK_ARG(n_nodes > 0 && n_nodes < (1ll << 31) && n_rel > 0 && 2 * n_pairs < (1ll << 30), "link_loss_bwd_rows: bad sizes");
  RGCN_CHECK_ARG(g_emb && ld_g % 4 == 0 && ((uintptr_t)g_emb & 15) == 0 && slot && rows, "link_loss_bwd_rows: bad buffers");
  RGCN_CHECK_ARG(g_score || (score && g_loss && labels), "link_loss_bwd_rows: need g_score, or score + labels + g_loss");
  RGCN_CHECK_ARG(dropout_p == 0.f || state, "link_loss_bwd_rows: dropout needs the state the forward wrote");
  RGCN_CHECK_ARG(!g_rel_table || ((uintptr_t)g_rel_table & 15) == 0, "link_loss_bwd_rows: g_rel_table misaligned");
  if (!workspace || ((uintptr_t)workspace & 15) != 0 || workspace_bytes < rgcn_link_bwd_rows_workspace_bytes(n_pairs, n_rel, d)) {
    set_error("link_loss_bwd_rows: workspace missing, misaligned or too small"); return RGCN_EWORKSPACE;
  }
  q.state = const_cast<unsigned long long*>(state); q.score = const_cast<float*>(score);
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t m_c = (int32_t)rgcn_rows_compact_size(2 * n_pairs);
  RGCN_CUDA(launch_pdl(link_slot_fill_kernel, dim3((unsigned)((n_nodes + 255) / 256)), dim3(256), 0, st, slot, n_nodes, m_c));
  RGCN_LAUNCH_CHECK();
  LinkBwdRows b{};
  b.g_loss = g_loss; b.g_score = g_score; b.g_emb = g_emb; b.ld_g = ld_g; b.n_rows = n_nodes;
  b.slot = slot; b.rows = rows; b.unlisted = m_c;
  b.C = (float*)workspace;
  b.T = g_rel_table ? (float*)((char*)workspace + link_ws_C(n_pairs, d)) : nullptr;
  b.tab_partial = g_rel_table ? (float*)((char*)workspace + link_ws_C(n_pairs, d) + link_ws_T(n_pairs, d)) : nullptr;
  b.n_owner_blocks = (int32_t)((2 * n_pairs + 7) / 8);
  // listed_only: the consumer reads the listed rows of g_emb alone (the listed-rows form of the last encoder layer), so
  // the other rows stay as they are instead of being zero-filled (N x d floats less to write)
  b.n_zero_blocks = listed_only ? 0 : (int32_t)((n_nodes + kLinkZeroRows - 1) / kLinkZeroRows);
  b.n_tab_blocks = g_rel_table ? (int32_t)((n_pairs + kLinkTabPairs - 1) / kLinkTabPairs) : 0;
  RGCN_CUDA(launch_pdl(link_contrib_kernel, dim3((unsigned)b.n_owner_blocks), dim3(256), 0, st, q, b));
  RGCN_LAUNCH_CHECK();
  size_t smem = (size_t)((2 * n_pairs + 127) / 128 * 128) * sizeof(int);
  b.rows_in_smem = smem <= 200 * 1024 ? 1 : 0;       // (larger batches scan the list in global memory)
  if (!b.rows_in_smem) smem = 0;
  if (smem > 0) {
    // the default limit is 48 KB of static + dynamic shared memory, and the kernel's own static arrays count against
    // it: ask the runtime what is left rather than comparing with 48 KB.  Cached per device, so that a captured step
    // (whose eager warm-up ran the same batch size first) makes no attribute call.
    static size_t granted[64] = {0};
    int dev = 0;
    RGCN_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && granted[dev] < smem) {
      cudaFuncAttributes fa{};
      RGCN_CUDA(cudaFuncGetAttributes(&fa, link_gather_kernel));
      granted[dev] = (size_t)fa.maxDynamicSharedSizeBytes;
      if (granted[dev] < smem) {
        RGCN_CUDA(cudaFuncSetAttribute(link_gather_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        granted[dev] = 200 * 1024;
      }
    }
  }
  RGCN_CUDA(launch_pdl(link_gather_kernel, dim3((unsigned)(b.n_owner_blocks + b.n_zero_blocks + b.n_tab_blocks)), dim3(256),
                       smem, st, q, b));
  RGCN_LAUNCH_CHECK();
  if (g_rel_table) {
    rc = rgcn_reduce_partials(b.tab_partial, b.n_tab_blocks, n_rel * d, g_rel_table, stream);    // fixed order
    if (rc) return rc;
  }
  return RGCN_OK;
}
