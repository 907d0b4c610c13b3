// Fused BPR + L2 (+ fairness) loss on a batch of (user, pos, neg) triples: forward value and the
// gradients w.r.t. the propagated tables, scattered WITHOUT atomics.
//
// Replaces (reference, /root/reference): score / l2_reg / loss assembly lightgcn_cu.py:450-463,
// 635-648; bpr_loss Version-2/lighgcn_cu_pop.py:495-508; and the index_put-with-accumulate
// backward autograd runs for them.
//
// Scatter scheme: every triple t contributes to three rows (user u, item pos, item neg).  The 3B
// (row, entry) pairs are packed into 64-bit keys and sorted by row (cgx_bpr_plan: a stable
// shared-memory radix sort inside ONE CTA for batches up to 4096 triples, the global radix sort
// above that); one thread group per distinct row then walks its run in entry order and writes
// the row once.  Entry order is fixed by the stable sort, so the result is bitwise reproducible.
// The plan depends on the indices only, so callers may build it on a side stream while the
// forward propagation runs.
#include <atomic>

#include "common.cuh"

namespace cgx {

constexpr int BP_THREADS = 256;

template <int G>
__device__ __forceinline__ unsigned bp_group_mask() {
  if (G == 32) return 0xffffffffu;
  const unsigned lane = threadIdx.x & 31;
  return ((1u << (G & 31)) - 1u) << (lane & ~(G - 1));
}

template <int G>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, G);
  return v;
}

__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
}

__device__ __forceinline__ int64_t clamp_id(int64_t x, int64_t n) { return (x < 0 || x >= n) ? 0 : x; }

// key of entry e (0..3B): row in the high bits (items offset by U), entry id in the low bits; an entry of a triple
// t >= cnt (absent) gets the row U + I, behind every real row
__device__ __forceinline__ uint64_t plan_key(const int64_t* __restrict__ users, const int64_t* __restrict__ pos,
                                             const int64_t* __restrict__ neg, int64_t B, int64_t cnt, int32_t U,
                                             int32_t I, int entry_bits, int64_t e) {
  const int type = int(e / B);
  const int64_t t = e - int64_t(type) * B;
  const int64_t row = t >= cnt ? int64_t(U) + I
                    : type == 0 ? clamp_id(users[t], U) : int64_t(U) + clamp_id(type == 1 ? pos[t] : neg[t], I);
  return (uint64_t(row) << entry_bits) | uint64_t(e);
}

__global__ void k_plan_keys(const int64_t* __restrict__ users, const int64_t* __restrict__ pos,
                            const int64_t* __restrict__ neg, int64_t B, const int64_t* __restrict__ count, int32_t U,
                            int32_t I, int entry_bits, uint64_t* __restrict__ keys) {
  const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t cnt = count != nullptr ? *count : B;
  if (e < 3 * B) keys[e] = plan_key(users, pos, neg, B, cnt, U, I, entry_bits, e);
}

// ---- single-CTA stable radix sort of up to PS_MAX keys on the row bits -------------------------
constexpr int PS_THREADS = 1024;
constexpr int PS_WARPS = PS_THREADS / 32;
constexpr int PS_STEPS = 12;
constexpr int PS_MAX = PS_THREADS * PS_STEPS;  // 12288 keys = 3 * 4096

__global__ void __launch_bounds__(PS_THREADS, 1) k_plan_small(const int64_t* __restrict__ users,
                                                              const int64_t* __restrict__ pos,
                                                              const int64_t* __restrict__ neg, int64_t B,
                                                              const int64_t* __restrict__ count, int32_t U,
                                                              int32_t I, int entry_bits, int row_bits,
                                                              uint64_t* __restrict__ sorted) {
  extern __shared__ __align__(16) unsigned char ps_smem[];
  uint64_t* buf0 = reinterpret_cast<uint64_t*>(ps_smem);
  uint64_t* buf1 = buf0 + PS_MAX;
  uint16_t(*cnt)[256] = reinterpret_cast<uint16_t(*)[256]>(buf1 + PS_MAX);  // [PS_WARPS][256]
  uint32_t* tot = reinterpret_cast<uint32_t*>(cnt + PS_WARPS);              // [256]
  const int n = int(3 * B);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  const int64_t n_real = count != nullptr ? *count : B;
  for (int e = threadIdx.x; e < n; e += PS_THREADS) buf0[e] = plan_key(users, pos, neg, B, n_real, U, I, entry_bits, e);
  __syncthreads();
  uint64_t* src = buf0;
  uint64_t* dst = buf1;
  const int wbase = warp * (PS_STEPS * 32);
  for (int shift = entry_bits; shift < entry_bits + row_bits; shift += 8) {
    for (int b = lane; b < 256; b += 32) cnt[warp][b] = 0;
    __syncwarp();
    uint64_t key[PS_STEPS];
#pragma unroll
    for (int j = 0; j < PS_STEPS; ++j) {
      const int p = wbase + j * 32 + lane;
      const bool valid = p < n;
      key[j] = valid ? src[p] : 0ull;
      const uint32_t d = valid ? uint32_t((key[j] >> shift) & 0xff) : 256u;
      const uint32_t m = __match_any_sync(0xffffffffu, d);
      if (valid && (m & lt) == 0) cnt[warp][d] += uint16_t(__popc(m));
      __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x < 256) {  // digit totals, and per-warp exclusive prefix inside the digit
      uint32_t run = 0;
#pragma unroll 8
      for (int w = 0; w < PS_WARPS; ++w) {
        const uint32_t c = cnt[w][threadIdx.x];
        cnt[w][threadIdx.x] = uint16_t(run);
        run += c;
      }
      tot[threadIdx.x] = run;
    }
    __syncthreads();
    if (warp == 0) {  // exclusive scan of the 256 digit totals: 8 per lane
      uint32_t v[8], s = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { v[q] = tot[lane * 8 + q]; s += v[q]; }
      uint32_t inc = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
      }
      uint32_t ex = inc - s;
#pragma unroll
      for (int q = 0; q < 8; ++q) { tot[lane * 8 + q] = ex; ex += v[q]; }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PS_STEPS; ++j) {
      const int p = wbase + j * 32 + lane;
      const bool valid = p < n;
      const uint32_t d = valid ? uint32_t((key[j] >> shift) & 0xff) : 256u;
      const uint32_t m = __match_any_sync(0xffffffffu, d);
      uint32_t q = 0;
      if (valid) q = tot[d] + cnt[warp][d] + __popc(m & lt);
      __syncwarp();
      if (valid && (m & lt) == 0) cnt[warp][d] += uint16_t(__popc(m));
      __syncwarp();
      if (valid) dst[q] = key[j];
    }
    __syncthreads();
    uint64_t* t = src; src = dst; dst = t;
  }
  for (int e = threadIdx.x; e < n; e += PS_THREADS) sorted[e] = src[e];
}

static size_t plan_small_smem() { return size_t(2) * PS_MAX * 8 + size_t(PS_WARPS) * 256 * 2 + 256 * 4; }

struct BprArgs {
  const int64_t* users;
  const int64_t* pos;
  const int64_t* neg;
  int64_t B;
  int64_t B_total;   // denominator of the means (== B unless the batch is sharded over ranks)
  const int64_t* count;      // nullable: triples t >= *count are absent (padding of a sharded batch)
  const int64_t* total_dev;  // nullable: the denominator read from the device instead of B_total
  int32_t U, I;
  const float4* f_u;
  const float4* f_i;
  const float4* e0_u;
  const float4* e0_i;
  const float* pop;
  float reg, fair;
};

__device__ __forceinline__ int64_t bpr_count(const BprArgs& a) { return a.count != nullptr ? *a.count : a.B; }
__device__ __forceinline__ float bpr_total(const BprArgs& a) {
  return float(a.total_dev != nullptr ? *a.total_dev : a.B_total);
}

// per triple: scores, loss term, coefficients
template <int G, int V>
__global__ void __launch_bounds__(BP_THREADS) k_bpr_triple(BprArgs a, float* __restrict__ coef_pos,
                                                           float* __restrict__ coef_neg,
                                                           float* __restrict__ loss_term,
                                                           unsigned long long* __restrict__ bad) {
  constexpr int ROW4 = G * V;
  const int lane = threadIdx.x & (G - 1);
  const int64_t t = (int64_t(blockIdx.x) * BP_THREADS + threadIdx.x) / G;
  if (t >= a.B) return;
  if (t >= bpr_count(a)) {                 // absent: no term, no index check
    if ((threadIdx.x & (G - 1)) == 0) loss_term[t] = 0.f;
    return;
  }
  const unsigned mask = bp_group_mask<G>();
  int64_t u = a.users[t], p = a.pos[t], n = a.neg[t];
  if (u < 0 || u >= a.U || p < 0 || p >= a.I || n < 0 || n >= a.I) {
    if (lane == 0) atomicAdd(bad, 1ull);
    u = clamp_id(u, a.U); p = clamp_id(p, a.I); n = clamp_id(n, a.I);
  }
  float yp = 0.f, yn = 0.f, l2 = 0.f;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int o = v * G + lane;
    const float4 fu = __ldg(a.f_u + u * ROW4 + o);
    const float4 fp = __ldg(a.f_i + p * ROW4 + o);
    const float4 fn = __ldg(a.f_i + n * ROW4 + o);
    yp += dot4(fu, fp);
    yn += dot4(fu, fn);
    const float4 eu = __ldg(a.e0_u + u * ROW4 + o);
    const float4 ep = __ldg(a.e0_i + p * ROW4 + o);
    const float4 en = __ldg(a.e0_i + n * ROW4 + o);
    l2 += dot4(eu, eu) + dot4(ep, ep) + dot4(en, en);
  }
  yp = group_sum<G>(yp, mask);
  yn = group_sum<G>(yn, mask);
  l2 = group_sum<G>(l2, mask);
  if (lane == 0) {
    const float invB = 1.0f / bpr_total(a);
    const float x = yp - yn;
    const float sig = 1.0f / (1.0f + expf(-x));
    const float term = -logf(sig + 1e-12f);                      // lightgcn_cu.py:637 (epsilon form)
    const float gx = -(sig * (1.0f - sig)) / (sig + 1e-12f) * invB;
    const float pw = (a.pop != nullptr && a.fair != 0.f) ? a.fair * __ldg(a.pop + p) : 0.f;
    coef_pos[t] = gx + pw * invB;
    coef_neg[t] = -gx;
    loss_term[t] = (term + pw * yp + a.reg * l2) * invB;
  }
}

// One group per sorted entry.  The sorted entry list is cut into blocks of BP_SEG entries; a run (= all entries of
// one row) is accumulated in SEGMENTS: from its head to the end of the head's block, then one segment per further
// block.  A run that stays inside one block is written straight to the gradient row by its head; a longer run
// (popularity-weighted negatives put hundreds of entries on one item) leaves one partial sum per segment, which
// k_bpr_combine adds in segment order.  Walking such a run in one group was a chain of ~3 dependent load latencies
// per 4 entries and set the duration of the whole kernel (36 us for a 12 288-entry batch).
// Partial slot of a segment that starts at entry k: 2 * (k / BP_SEG) + (k % BP_SEG != 0) -- per block at most one
// segment starts at the block's first entry and at most one head-started segment continues past the block.
constexpr int BP_SEG = 8;

template <int G, int V>
__global__ void __launch_bounds__(BP_THREADS) k_bpr_scatter(BprArgs a, int entry_bits,
                                                            const uint64_t* __restrict__ keys,
                                                            const float* __restrict__ coef_pos,
                                                            const float* __restrict__ coef_neg,
                                                            float4* __restrict__ g_u, float4* __restrict__ g_i,
                                                            int32_t* __restrict__ ego_rows,
                                                            float* __restrict__ ego_coef, float4* __restrict__ part,
                                                            int32_t* __restrict__ part_cnt) {
  constexpr int ROW4 = G * V;
  const int lane = threadIdx.x & (G - 1);
  const int64_t k = (int64_t(blockIdx.x) * BP_THREADS + threadIdx.x) / G;
  const int64_t n = 3 * a.B;
  if (k >= n) return;
  if (k >= 3 * bpr_count(a)) {             // absent entries sort last: no row
    if (lane == 0) ego_rows[k] = -1;
    return;
  }
  const uint64_t emask = (uint64_t(1) << entry_bits) - 1;
  const uint64_t key = keys[k];
  const int64_t row = int64_t(key >> entry_bits);
  const bool head = (k == 0) || (int64_t(keys[k - 1] >> entry_bits) != row);
  const bool aligned = (k % BP_SEG) == 0;
  if (!head) {
    if (lane == 0) ego_rows[k] = -1;
    if (!aligned) return;                      // an aligned non-head entry starts a continuation segment
  }
  const int64_t bound = (k / BP_SEG + 1) * BP_SEG;   // first entry of the next block
  const int64_t stop = bound < n ? bound : n;
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  int mult = 0;
  // The run is walked four entries at a time: keys, then coefficients / ids, then the embedding rows of all
  // four are loaded before anything is accumulated (popular items give runs of 50+ entries; one dependent
  // load chain per entry would serialise ~1.5 us each).  Accumulation order stays the entry order.
  constexpr int RU = 4;
  for (int64_t q0 = k; q0 < stop; q0 += RU) {
    int64_t e[RU];
    int m = 0;
#pragma unroll
    for (int t = 0; t < RU; ++t) {
      const uint64_t kq = (q0 + t < stop) ? keys[q0 + t] : ~uint64_t(0);
      e[t] = int64_t(kq & emask);
      if (m == t && q0 + t < stop && int64_t(kq >> entry_bits) == row) m = t + 1;
    }
    float c0[RU], c1[RU];
    int64_t r0[RU], r1[RU];
    int type[RU];
#pragma unroll
    for (int t = 0; t < RU; ++t) {
      type[t] = 0; c0[t] = c1[t] = 0.f; r0[t] = r1[t] = 0;
      if (t < m) {
        type[t] = int(e[t] / a.B);
        const int64_t tt = e[t] - int64_t(type[t]) * a.B;
        if (type[t] == 0) {            // user row: cp * f_i[pos] + cn * f_i[neg]
          c0[t] = coef_pos[tt]; c1[t] = coef_neg[tt];
          r0[t] = clamp_id(a.pos[tt], a.I); r1[t] = clamp_id(a.neg[tt], a.I);
        } else {                       // item row: coefficient * f_u[user]
          c0[t] = type[t] == 1 ? coef_pos[tt] : coef_neg[tt];
          r0[t] = clamp_id(a.users[tt], a.U);
        }
      }
    }
    float4 x0[RU][V], x1[RU][V];
#pragma unroll
    for (int t = 0; t < RU; ++t) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        x0[t][v] = x1[t][v] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < m) {
          if (type[t] == 0) {
            x0[t][v] = __ldg(a.f_i + r0[t] * ROW4 + v * G + lane);
            x1[t][v] = __ldg(a.f_i + r1[t] * ROW4 + v * G + lane);
          } else {
            x0[t][v] = __ldg(a.f_u + r0[t] * ROW4 + v * G + lane);
          }
        }
      }
    }
#pragma unroll
    for (int t = 0; t < RU; ++t) {
      if (t < m) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          acc[v].x += c0[t] * x0[t][v].x + c1[t] * x1[t][v].x;
          acc[v].y += c0[t] * x0[t][v].y + c1[t] * x1[t][v].y;
          acc[v].z += c0[t] * x0[t][v].z + c1[t] * x1[t][v].z;
          acc[v].w += c0[t] * x0[t][v].w + c1[t] * x1[t][v].w;
        }
      }
    }
    mult += m;
    if (m < RU) break;
  }
  // the run goes on in the next block iff this segment reached the block's end and the next block starts with the row
  const bool cont = (k + mult == stop) && stop < n && int64_t(keys[stop] >> entry_bits) == row;
  if (head && !cont) {
    float4* dst = row < a.U ? g_u + row * ROW4 : g_i + (row - a.U) * ROW4;
#pragma unroll
    for (int v = 0; v < V; ++v) dst[v * G + lane] = acc[v];
    if (lane == 0) {
      ego_rows[k] = int32_t(row);
      ego_coef[k] = float(mult) * 2.0f * a.reg / bpr_total(a);
    }
    return;
  }
  const int64_t slot = 2 * (k / BP_SEG) + (aligned ? 0 : 1);
#pragma unroll
  for (int v = 0; v < V; ++v) part[slot * ROW4 + v * G + lane] = acc[v];
  if (lane == 0) {
    part_cnt[slot] = mult;
    if (head) ego_rows[k] = -2;                // k_bpr_combine finishes this row
  }
}

// heads of runs that span several blocks: add the segment partials in order and write the gradient row
template <int G, int V>
__global__ void __launch_bounds__(BP_THREADS) k_bpr_combine(BprArgs a, int entry_bits,
                                                            const uint64_t* __restrict__ keys,
                                                            float4* __restrict__ g_u, float4* __restrict__ g_i,
                                                            int32_t* __restrict__ ego_rows,
                                                            float* __restrict__ ego_coef,
                                                            const float4* __restrict__ part,
                                                            const int32_t* __restrict__ part_cnt) {
  constexpr int ROW4 = G * V;
  const int lane = threadIdx.x & (G - 1);
  const int64_t k = (int64_t(blockIdx.x) * BP_THREADS + threadIdx.x) / G;
  const int64_t n = 3 * a.B;
  if (k >= n || ego_rows[k] != -2) return;
  const int64_t row = int64_t(keys[k] >> entry_bits);
  const int64_t slot0 = 2 * (k / BP_SEG) + ((k % BP_SEG) ? 1 : 0);
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = part[slot0 * ROW4 + v * G + lane];
  int mult = part_cnt[slot0];
  constexpr int RU = 4;      // four blocks per pass: keys, counts and partials of all four are loaded before any add
  for (int64_t b0 = (k / BP_SEG + 1) * BP_SEG; b0 < n; b0 += RU * BP_SEG) {
    int m = 0;
#pragma unroll
    for (int t = 0; t < RU; ++t) {
      const int64_t b = b0 + int64_t(t) * BP_SEG;
      if (m == t && b < n && int64_t(keys[b] >> entry_bits) == row) m = t + 1;
    }
    float4 x[RU][V];
    int c[RU];
#pragma unroll
    for (int t = 0; t < RU; ++t) {
      const int64_t s = 2 * (b0 / BP_SEG + t);
      c[t] = t < m ? part_cnt[s] : 0;
#pragma unroll
      for (int v = 0; v < V; ++v)
        x[t][v] = t < m ? part[s * ROW4 + v * G + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int t = 0; t < RU; ++t) {
      if (t < m) {
        mult += c[t];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          acc[v].x += x[t][v].x; acc[v].y += x[t][v].y; acc[v].z += x[t][v].z; acc[v].w += x[t][v].w;
        }
      }
    }
    if (m < RU) break;
  }
  float4* dst = row < a.U ? g_u + row * ROW4 : g_i + (row - a.U) * ROW4;
#pragma unroll
  for (int v = 0; v < V; ++v) dst[v * G + lane] = acc[v];
  if (lane == 0) {
    ego_rows[k] = int32_t(row);
    ego_coef[k] = float(mult) * 2.0f * a.reg / bpr_total(a);
  }
}

// Row bookkeeping of the dense gradient tables g_u / g_i, driven by ego_rows (the head of every distinct row of the
// batch): MARK sets the row flags the adjoint propagation reads (instead of scanning 4 (U + I) d bytes for
// non-zero rows), CLEAR zeroes the rows -- and their flags -- after use, so that the tables are all-zero again
// without a fill of the whole allocation.
template <bool CLEAR>
__global__ void __launch_bounds__(BP_THREADS) k_bpr_rows(const int32_t* __restrict__ ego_rows, int64_t n, int32_t U,
                                                         int32_t row4, float4* __restrict__ g_u,
                                                         float4* __restrict__ g_i, uint8_t* __restrict__ nz_u,
                                                         uint8_t* __restrict__ nz_i) {
  const int64_t k = blockIdx.x;                       // one CTA per plan entry
  if (k >= n) return;
  const int32_t row = ego_rows[k];
  if (row < 0) return;
  const bool user = row < U;
  const int64_t r = user ? row : row - U;
  if (threadIdx.x == 0) (user ? nz_u : nz_i)[r] = CLEAR ? 0 : 1;
  if (CLEAR) {
    float4* dst = (user ? g_u : g_i) + r * row4;
    for (int p = threadIdx.x; p < row4; p += blockDim.x) dst[p] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// deterministic sum of B terms by one CTA (fixed tree); NaN if any index was out of range
__global__ void __launch_bounds__(1024) k_sum_terms(const float* __restrict__ terms, int64_t n,
                                                    const unsigned long long* __restrict__ bad,
                                                    float* __restrict__ out) {
  __shared__ double sh[1024];
  double s = 0.0;
  for (int64_t p = threadIdx.x; p < n; p += 1024) s += double(terms[p]);
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = (*bad != 0ull) ? __int_as_float(0x7fc00000) : float(sh[0]);
}

template <int G, int V>
__global__ void __launch_bounds__(BP_THREADS) k_apply_ego(const int32_t* __restrict__ ego_rows,
                                                          const float* __restrict__ ego_coef, int64_t n,
                                                          int32_t U, const float4* __restrict__ e0_u,
                                                          const float4* __restrict__ e0_i, float4* d_u,
                                                          float4* d_i) {
  constexpr int ROW4 = G * V;
  const int lane = threadIdx.x & (G - 1);
  const int64_t k = (int64_t(blockIdx.x) * BP_THREADS + threadIdx.x) / G;
  if (k >= n) return;
  const int32_t row = ego_rows[k];
  if (row < 0) return;
  const float c = ego_coef[k];
  const float4* src = row < U ? e0_u + int64_t(row) * ROW4 : e0_i + int64_t(row - U) * ROW4;
  float4* dst = row < U ? d_u + int64_t(row) * ROW4 : d_i + int64_t(row - U) * ROW4;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const float4 e = __ldg(src + v * G + lane);
    float4 g = dst[v * G + lane];
    g.x += c * e.x; g.y += c * e.y; g.z += c * e.z; g.w += c * e.w;
    dst[v * G + lane] = g;
  }
}

static size_t plan_ws(int64_t B) {
  const int64_t n = 3 * B;
  if (n <= PS_MAX) return 256;
  return align_up(size_t(n) * 8) + radix_sort_temp_bytes(n) + 256;
}
// coefficients + loss terms + the segment partials of k_bpr_scatter (sized for the widest table, d = 256)
static size_t bpr_part_slots(int64_t B) { return 2 * size_t(ceil_div(3 * B, BP_SEG)); }
static size_t bpr_ws(int64_t B) {
  return 3 * align_up(size_t(B) * 4) + align_up(bpr_part_slots(B) * 256 * 4) + align_up(bpr_part_slots(B) * 4) + 512;
}

template <int G, int V>
static int bpr_run(const BprArgs& a, const uint64_t* plan, float* loss_out, float* g_u, float* g_i,
                   int32_t* ego_rows, float* ego_coef, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream) {
  const int64_t B = a.B, n = 3 * B;
  Arena ws(workspace, workspace_bytes);
  float* coef_pos = ws.take<float>(B);
  float* coef_neg = ws.take<float>(B);
  float* terms = ws.take<float>(B);
  unsigned long long* bad = ws.take<unsigned long long>(1);
  float4* part = ws.take<float4>(bpr_part_slots(B) * G * V);
  int32_t* part_cnt = ws.take<int32_t>(bpr_part_slots(B));
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "bpr: workspace too small");
  constexpr int GROUPS = BP_THREADS / G;
  CGX_CUDA(cudaMemsetAsync(bad, 0, 8, stream));
  k_bpr_triple<G, V><<<(unsigned)ceil_div(B, GROUPS), BP_THREADS, 0, stream>>>(a, coef_pos, coef_neg, terms, bad);
  CGX_LAUNCH_CHECK();
  k_bpr_scatter<G, V><<<(unsigned)ceil_div(n, GROUPS), BP_THREADS, 0, stream>>>(
      a, bits_for(n), plan, coef_pos, coef_neg, reinterpret_cast<float4*>(g_u), reinterpret_cast<float4*>(g_i),
      ego_rows, ego_coef, part, part_cnt);
  CGX_LAUNCH_CHECK();
  k_bpr_combine<G, V><<<(unsigned)ceil_div(n, GROUPS), BP_THREADS, 0, stream>>>(
      a, bits_for(n), plan, reinterpret_cast<float4*>(g_u), reinterpret_cast<float4*>(g_i), ego_rows, ego_coef, part,
      part_cnt);
  CGX_LAUNCH_CHECK();
  k_sum_terms<<<1, 1024, 0, stream>>>(terms, B, bad, loss_out);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

}  // namespace cgx

using namespace cgx;

extern "C" size_t cgx_bpr_plan_workspace_bytes(int64_t batch) { return plan_ws(batch); }

extern "C" int cgx_bpr_plan(const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t batch, int32_t U,
                            int32_t I, uint64_t* plan, void* workspace, size_t workspace_bytes, void* stream_,
                            const int64_t* count) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(users && pos && neg && plan, CGX_ERR_ARG, "bpr_plan: NULL pointer");
  CGX_REQUIRE(batch > 0 && batch < (int64_t(1) << 29), CGX_ERR_ARG, "bpr_plan: bad batch size %lld",
              (long long)batch);
  CGX_REQUIRE(workspace_bytes >= plan_ws(batch), CGX_ERR_WORKSPACE, "bpr_plan: workspace too small");
  const int64_t n = 3 * batch;
  // with a count, absent entries take the row U + I
  const int entry_bits = bits_for(n), row_bits = bits_for(int64_t(U) + I + (count != nullptr ? 1 : 0));
  if (n <= PS_MAX) {
    const size_t smem = plan_small_smem();
    // the shared-memory opt-in is a per-DEVICE attribute: set it once per device (a bit per ordinal), which also
    // keeps the call out of CUDA-graph captures after warm-up
    static std::atomic<unsigned long long> attr_set{0};
    int dev = 0;
    CGX_CUDA(cudaGetDevice(&dev));
    const unsigned long long bit = 1ull << (dev & 63);
    if (!(attr_set.load(std::memory_order_acquire) & bit)) {
      CGX_CUDA(cudaFuncSetAttribute(k_plan_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_set.fetch_or(bit, std::memory_order_release);
    }
    k_plan_small<<<1, PS_THREADS, smem, stream>>>(users, pos, neg, batch, count, U, I, entry_bits, row_bits, plan);
    CGX_LAUNCH_CHECK();
    return CGX_OK;
  }
  Arena ws(workspace, workspace_bytes);
  uint64_t* alt = ws.take<uint64_t>(n);
  size_t sort_bytes = radix_sort_temp_bytes(n);
  void* sort_tmp = ws.take<char>(sort_bytes);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "bpr_plan: workspace too small");
  k_plan_keys<<<(unsigned)ceil_div(n, 256), 256, 0, stream>>>(users, pos, neg, batch, count, U, I, entry_bits, plan);
  CGX_LAUNCH_CHECK();
  uint64_t* sorted = plan;
  CGX_TRY(radix_sort_u64(plan, alt, n, entry_bits + row_bits, sort_tmp, sort_bytes, stream, &sorted));
  if (sorted != plan) CGX_CUDA(cudaMemcpyAsync(plan, sorted, size_t(n) * 8, cudaMemcpyDeviceToDevice, stream));
  return CGX_OK;
}

extern "C" size_t cgx_bpr_workspace_bytes(int64_t batch, int32_t, int32_t) { return bpr_ws(batch); }

extern "C" int cgx_bpr_fwd_bwd(const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t batch,
                               int64_t batch_total, const uint64_t* plan, int32_t U, int32_t I, int32_t d,
                               const float* f_u,
                               const float* f_i, const float* e0_u, const float* e0_i, const float* pop,
                               float reg_weight, float fair_weight, float* loss_out, float* g_u, float* g_i,
                               int32_t* ego_rows, float* ego_coef, void* workspace, size_t workspace_bytes,
                               void* stream_, const int64_t* count, const int64_t* batch_total_dev) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(users && pos && neg && plan && f_u && f_i && e0_u && e0_i && loss_out && g_u && g_i && ego_rows &&
                  ego_coef,
              CGX_ERR_ARG, "bpr: NULL pointer");
  CGX_REQUIRE(batch > 0 && batch < (int64_t(1) << 29), CGX_ERR_ARG, "bpr: bad batch size %lld", (long long)batch);
  CGX_REQUIRE(workspace_bytes >= bpr_ws(batch), CGX_ERR_WORKSPACE, "bpr: workspace too small");
  BprArgs a{users, pos, neg, batch, batch_total > 0 ? batch_total : batch, count, batch_total_dev, U, I,
            reinterpret_cast<const float4*>(f_u),
            reinterpret_cast<const float4*>(f_i), reinterpret_cast<const float4*>(e0_u),
            reinterpret_cast<const float4*>(e0_i), pop, reg_weight, fair_weight};
  switch (d) {
    case 16: return bpr_run<4, 1>(a, plan, loss_out, g_u, g_i, ego_rows, ego_coef, workspace, workspace_bytes, stream);
    case 32: return bpr_run<8, 1>(a, plan, loss_out, g_u, g_i, ego_rows, ego_coef, workspace, workspace_bytes, stream);
    case 64: return bpr_run<16, 1>(a, plan, loss_out, g_u, g_i, ego_rows, ego_coef, workspace, workspace_bytes, stream);
    case 128: return bpr_run<32, 1>(a, plan, loss_out, g_u, g_i, ego_rows, ego_coef, workspace, workspace_bytes, stream);
    case 256: return bpr_run<32, 2>(a, plan, loss_out, g_u, g_i, ego_rows, ego_coef, workspace, workspace_bytes, stream);
    default:
      set_error("bpr: emb_dim %d unsupported (16, 32, 64, 128, 256)", d);
      return CGX_ERR_UNSUPPORTED;
  }
}

extern "C" int cgx_bpr_mark_rows(const int32_t* ego_rows, int64_t n_entries, int32_t U, uint8_t* nz_u, uint8_t* nz_i,
                                 void* stream_) {
  CGX_REQUIRE(ego_rows && nz_u && nz_i && n_entries > 0 && n_entries < (int64_t(1) << 31), CGX_ERR_ARG,
              "bpr_mark_rows: bad argument");
  k_bpr_rows<false><<<(unsigned)n_entries, 32, 0, static_cast<cudaStream_t>(stream_)>>>(ego_rows, n_entries, U, 0,
                                                                                        nullptr, nullptr, nz_u, nz_i);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_bpr_clear_rows(const int32_t* ego_rows, int64_t n_entries, int32_t U, int32_t d, float* g_u,
                                  float* g_i, uint8_t* nz_u, uint8_t* nz_i, void* stream_) {
  CGX_REQUIRE(ego_rows && g_u && g_i && nz_u && nz_i && n_entries > 0 && n_entries < (int64_t(1) << 31) && d > 0 &&
                  d % 4 == 0,
              CGX_ERR_ARG, "bpr_clear_rows: bad argument");
  k_bpr_rows<true><<<(unsigned)n_entries, 64, 0, static_cast<cudaStream_t>(stream_)>>>(
      ego_rows, n_entries, U, d / 4, reinterpret_cast<float4*>(g_u), reinterpret_cast<float4*>(g_i), nz_u, nz_i);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_bpr_apply_ego(const int32_t* ego_rows, const float* ego_coef, int64_t n_entries, int32_t U,
                                 int32_t d, const float* e0_u, const float* e0_i, float* d_e0_u, float* d_e0_i,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(ego_rows && ego_coef && e0_u && e0_i && d_e0_u && d_e0_i && n_entries > 0, CGX_ERR_ARG,
              "apply_ego: bad argument");
#define CGX_EGO(GG, VV)                                                                                        \
  k_apply_ego<GG, VV><<<(unsigned)ceil_div(n_entries, BP_THREADS / GG), BP_THREADS, 0, stream>>>(              \
      ego_rows, ego_coef, n_entries, U, reinterpret_cast<const float4*>(e0_u),                                  \
      reinterpret_cast<const float4*>(e0_i), reinterpret_cast<float4*>(d_e0_u), reinterpret_cast<float4*>(d_e0_i))
  switch (d) {
    case 16: CGX_EGO(4, 1); break;
    case 32: CGX_EGO(8, 1); break;
    case 64: CGX_EGO(16, 1); break;
    case 128: CGX_EGO(32, 1); break;
    case 256: CGX_EGO(32, 2); break;
    default:
      set_error("apply_ego: emb_dim %d unsupported", d);
      return CGX_ERR_UNSUPPORTED;
  }
#undef CGX_EGO
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}
