// On-device triple sampler: uniform positive from the user's train row, negative by rejection
// from either the uniform law or the popularity mixture mix*pop + (1-mix)*uniform.
//
// Replaces (reference, /root/reference): sample_pos_item / sample_neg_item / user_has_item
// lightgcn_cu.py:279-299; sample_neg_item_popmix Version-2/lighgcn_cu_pop.py:349-376 and the law
// pop_i ~ (deg_i + 1)^gamma at lighgcn_cu_pop.py:805-810.  The reference draws from a sequential
// PCG64 stream (O(I) per popularity draw); here every batch slot owns a Philox4x32-10 counter
// stream, and the popularity law is an alias table over DEGREE CLASSES: items of equal degree
// have equal probability, so "pick class c with weight n_c (deg_c+1)^gamma, then an item of the
// class uniformly" is the same distribution with an O(#distinct degrees) table.
#include "common.cuh"

namespace cgx {

constexpr int SM_THREADS = 256;

// ---- Philox4x32-10 (Salmon et al., SC'11) ----------------------------------------------------
struct Philox {
  uint32_t k0, k1;
  __device__ __forceinline__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
    uint32_t ka = k0, kb = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      const uint32_t n0 = hi1 ^ c1 ^ ka, n1 = lo1, n2 = hi0 ^ c3 ^ kb, n3 = lo0;
      c0 = n0; c1 = n1; c2 = n2; c3 = n3;
      ka += 0x9E3779B9u;
      kb += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};

__device__ __forceinline__ uint64_t u64_of(uint32_t hi, uint32_t lo) { return (uint64_t(hi) << 32) | lo; }
// floor(r * n / 2^64): uniform on [0, n) with bias < n / 2^64
__device__ __forceinline__ uint64_t bounded(uint64_t r, uint64_t n) { return __umul64hi(r, n); }
__device__ __forceinline__ float unit_float(uint32_t r) { return float(r >> 8) * (1.0f / 16777216.0f); }

__device__ __forceinline__ bool row_has(const int32_t* __restrict__ idx, int64_t lo, const int64_t end,
                                        int32_t item) {
  int64_t hi = end;
  while (lo < hi) {  // lower bound
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(idx + mid) < item) lo = mid + 1; else hi = mid;
  }
  return lo < end && __ldg(idx + lo) == item;
}

struct SamplerTables {
  const int32_t* items_by_deg;
  const int32_t* class_start;
  const float* class_prob;
  const int32_t* class_alias;
  const int32_t* n_classes;
};

__global__ void __launch_bounds__(SM_THREADS) k_sample(const int64_t* __restrict__ users, int64_t B,
                                                       const int64_t* __restrict__ indptr,
                                                       const int32_t* __restrict__ idx, int32_t I,
                                                       SamplerTables tb, float mix_pop, int32_t max_tries,
                                                       uint64_t seed, uint64_t offset,
                                                       const unsigned long long* __restrict__ offset_dev,
                                                       const int64_t* __restrict__ slots,
                                                       const int64_t* __restrict__ count,
                                                       int64_t* __restrict__ pos_out, int64_t* __restrict__ neg_out) {
  const int64_t i = int64_t(blockIdx.x) * SM_THREADS + threadIdx.x;
  if (i >= B || (count != nullptr && i >= *count)) return;   // past the device count: absent, nothing written
  // the Philox stream of an entry is keyed by its slot of the (global) batch: a rank holding part of a batch draws
  // exactly what a whole-batch call draws for the same user
  const int64_t t = slots != nullptr ? slots[i] : i;
  if (offset_dev != nullptr) offset += *offset_dev;   // device-side step counter (CUDA-graph replay)
  const Philox rng{uint32_t(seed), uint32_t(seed >> 32)};
  const uint32_t o_lo = uint32_t(offset), o_hi = uint32_t(offset >> 32);
  // counter = (slot, draw index, offset.lo, offset.hi); draw 0 is the positive
  const int64_t u = users[i];
  const int64_t lo = __ldg(indptr + u), hi = __ldg(indptr + u + 1);
  if (hi <= lo) {  // caller contract: batch users own >= 1 train item (lightgcn_cu.py:592)
    pos_out[i] = -1;
    neg_out[i] = -1;
    return;
  }
  uint4 r = rng(uint32_t(t), 0u, o_lo, o_hi ^ uint32_t(t >> 32));
  pos_out[i] = int64_t(__ldg(idx + lo + int64_t(bounded(u64_of(r.x, r.y), uint64_t(hi - lo)))));
  const bool popmix = mix_pop >= 0.f;
  const int32_t D = popmix ? __ldg(tb.n_classes) : 0;
  int32_t item = 0;
  for (uint32_t tries = 0; tries < (1u << 20); ++tries) {
    const uint4 a = rng(uint32_t(t), 1u + 2u * tries, o_lo, o_hi ^ uint32_t(t >> 32));
    if (popmix && int32_t(tries) < max_tries && unit_float(a.x) < mix_pop) {
      const uint4 b = rng(uint32_t(t), 2u + 2u * tries, o_lo, o_hi ^ uint32_t(t >> 32));
      int32_t c = int32_t(bounded(u64_of(a.y, a.z), uint64_t(D)));
      if (!(unit_float(a.w) < __ldg(tb.class_prob + c))) c = __ldg(tb.class_alias + c);
      const int32_t s = __ldg(tb.class_start + c), e = __ldg(tb.class_start + c + 1);
      item = __ldg(tb.items_by_deg + s + int32_t(bounded(u64_of(b.x, b.y), uint64_t(e - s))));
    } else {
      item = int32_t(bounded(u64_of(a.y, a.z), uint64_t(I)));
    }
    if (!row_has(idx, lo, hi, item)) break;
  }
  neg_out[i] = int64_t(item);
}

// ---- sampled-evaluation candidates: 1 test positive + n_neg negatives outside test U train ----------
// (lightgcn_cu.py:505-521; one thread per (user, slot), independent Philox streams)
__global__ void __launch_bounds__(SM_THREADS) k_eval_candidates(const int64_t* __restrict__ users, int64_t n_users,
                                                                const int64_t* __restrict__ tr_indptr,
                                                                const int32_t* __restrict__ tr_idx,
                                                                const int64_t* __restrict__ te_indptr,
                                                                const int32_t* __restrict__ te_idx, int32_t I,
                                                                int32_t n_cand, uint64_t seed, int64_t row_base,
                                                                int64_t* __restrict__ cand) {
  const int64_t t = int64_t(blockIdx.x) * SM_THREADS + threadIdx.x;
  if (t >= n_users * n_cand) return;
  const int64_t rl = t / n_cand;
  const int slot = int(t - rl * n_cand);
  const int64_t u = users[rl];
  const int64_t r = row_base + rl;   // streams are keyed by the row of the whole list
  const Philox rng{uint32_t(seed), uint32_t(seed >> 32)};
  const int64_t te_lo = __ldg(te_indptr + u), te_hi = __ldg(te_indptr + u + 1);
  if (slot == 0) {   // the positive: uniform over the user's test items (callers pass users with >= 1 test item)
    const uint4 a = rng(uint32_t(r), 0u, uint32_t(r >> 32), 0x5eedu);
    cand[t] = te_hi > te_lo ? int64_t(__ldg(te_idx + te_lo + int64_t(bounded(u64_of(a.x, a.y), uint64_t(te_hi - te_lo))))) : -1;
    return;
  }
  const int64_t tr_lo = __ldg(tr_indptr + u), tr_hi = __ldg(tr_indptr + u + 1);
  int32_t item = 0;
  for (uint32_t tries = 0; tries < (1u << 20); ++tries) {
    const uint4 a = rng(uint32_t(r), uint32_t(slot), uint32_t(r >> 32) ^ (tries << 8), 0x5eedu);
    item = int32_t(bounded(u64_of(a.x, a.y), uint64_t(I)));
    if (!row_has(te_idx, te_lo, te_hi, item) && !row_has(tr_idx, tr_lo, tr_hi, item)) break;
  }
  cand[t] = int64_t(item);
}

// ---- batch selection of a user-sharded epoch: one CTA per batch ---------------------------------------------------
// Global batch s is perm[s B, min((s + 1) B, n_train)).  The entries whose user lies in [lo, hi) are compacted in
// batch order (a block-wide exclusive scan of per-thread counts), rebased to local ids, and given their slot in the
// global batch -- the slot keys the sampler's Philox stream.
constexpr int BS_THREADS = 1024;
constexpr int BS_PER = 4;
constexpr int64_t BS_MAX = int64_t(BS_THREADS) * BS_PER;

__global__ void __launch_bounds__(BS_THREADS) k_batch_select(const int64_t* __restrict__ perm, int64_t n_train,
                                                             const unsigned long long* __restrict__ step, int64_t B,
                                                             int64_t lo, int64_t hi, int64_t* __restrict__ users,
                                                             int64_t* __restrict__ slots, int64_t* __restrict__ count,
                                                             int64_t* __restrict__ total) {
  __shared__ int warp_tot[BS_THREADS / 32];
  const int64_t start = int64_t(*step) * B;
  const int64_t rem = n_train - start;
  const int64_t n = rem <= 0 ? 0 : (rem < B ? rem : B);
  const int j0 = threadIdx.x * BS_PER;
  int64_t u[BS_PER];
  int c = 0;
#pragma unroll
  for (int q = 0; q < BS_PER; ++q) {
    u[q] = j0 + q < n ? perm[start + j0 + q] : -1;
    if (u[q] >= lo && u[q] < hi) ++c;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int w = warp_tot[lane];
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += v;
    }
    warp_tot[lane] = wi - w;
  }
  __syncthreads();
  int p = warp_tot[warp] + inc - c;
#pragma unroll
  for (int q = 0; q < BS_PER; ++q) {
    if (u[q] >= lo && u[q] < hi) {
      users[p] = u[q] - lo;
      slots[p] = j0 + q;
      ++p;
    }
  }
  if (threadIdx.x == BS_THREADS - 1) {
    *count = p;
    *total = n;
  }
}

// ---- table build -------------------------------------------------------------------------------
__global__ void k_deg_keys(const int32_t* __restrict__ deg, int32_t I, int bits_i, uint64_t* __restrict__ keys) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < I) keys[i] = (uint64_t(uint32_t(deg[i])) << bits_i) | uint64_t(i);
}
__global__ void k_deg_heads(const uint64_t* __restrict__ keys, int32_t I, int bits_i, uint32_t* __restrict__ flags,
                            int32_t* __restrict__ items_by_deg) {
  int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= I) return;
  items_by_deg[k] = int32_t(keys[k] & ((uint64_t(1) << bits_i) - 1));
  flags[k] = (k == 0 || (keys[k] >> bits_i) != (keys[k - 1] >> bits_i)) ? 1u : 0u;
}
__global__ void k_class_fill(const uint64_t* __restrict__ keys, int32_t I, int bits_i,
                             const uint32_t* __restrict__ cls, const uint32_t* __restrict__ n_cls,
                             int32_t* __restrict__ class_start, int32_t* __restrict__ class_deg,
                             int32_t* __restrict__ n_classes) {
  int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k == 0) {
    class_start[*n_cls] = I;
    *n_classes = int32_t(*n_cls);
  }
  if (k >= I) return;
  if (k == 0 || (keys[k] >> bits_i) != (keys[k - 1] >> bits_i)) {
    class_start[cls[k]] = int32_t(k);
    class_deg[cls[k]] = int32_t(keys[k] >> bits_i);
  }
}
// Vose's alias construction over D classes, one thread (D = number of distinct degrees, small).
__global__ void k_vose(const int32_t* __restrict__ class_start, const int32_t* __restrict__ class_deg,
                       const int32_t* __restrict__ n_classes, double gamma, double* __restrict__ scaled,
                       int32_t* __restrict__ small, int32_t* __restrict__ large, float* __restrict__ prob,
                       int32_t* __restrict__ alias) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  const int D = *n_classes;
  double total = 0.0;
  for (int c = 0; c < D; ++c) {
    const double w = double(class_start[c + 1] - class_start[c]) * pow(double(class_deg[c]) + 1.0, gamma);
    scaled[c] = w;
    total += w;
  }
  int ns = 0, nl = 0;
  for (int c = 0; c < D; ++c) {
    scaled[c] = scaled[c] * double(D) / total;
    if (scaled[c] < 1.0) small[ns++] = c; else large[nl++] = c;
  }
  while (ns > 0 && nl > 0) {
    const int s = small[--ns], l = large[--nl];
    prob[s] = float(scaled[s]);
    alias[s] = l;
    scaled[l] = (scaled[l] + scaled[s]) - 1.0;
    if (scaled[l] < 1.0) small[ns++] = l; else large[nl++] = l;
  }
  while (nl > 0) { const int l = large[--nl]; prob[l] = 1.0f; alias[l] = l; }
  while (ns > 0) { const int s = small[--ns]; prob[s] = 1.0f; alias[s] = s; }
}

static size_t sampler_ws(int32_t I) {
  return 2 * align_up(size_t(I) * 8) + align_up(size_t(I) * 4) * 4 + align_up(size_t(I) * 8) +
         radix_sort_temp_bytes(I) + scan_temp_bytes(I) + 1024;
}

}  // namespace cgx

using namespace cgx;

extern "C" size_t cgx_sampler_build_workspace_bytes(int32_t num_items) { return sampler_ws(num_items); }

extern "C" int cgx_sampler_build(const int32_t* deg_i, int32_t I, double gamma, int32_t* items_by_deg,
                                 int32_t* class_start, float* class_prob, int32_t* class_alias,
                                 int32_t* n_classes, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(deg_i && I > 0 && items_by_deg && class_start && class_prob && class_alias && n_classes, CGX_ERR_ARG,
              "sampler_build: bad argument");
  CGX_REQUIRE(workspace_bytes >= sampler_ws(I), CGX_ERR_WORKSPACE, "sampler_build: workspace too small");
  Arena ws(workspace, workspace_bytes);
  uint64_t* keys = ws.take<uint64_t>(I);
  uint64_t* alt = ws.take<uint64_t>(I);
  uint32_t* flags = ws.take<uint32_t>(I);
  int32_t* class_deg = ws.take<int32_t>(I);
  int32_t* small = ws.take<int32_t>(I);
  int32_t* large = ws.take<int32_t>(I);
  double* scaled = ws.take<double>(I);
  size_t sort_bytes = radix_sort_temp_bytes(I);
  void* sort_tmp = ws.take<char>(sort_bytes);
  size_t scan_bytes = scan_temp_bytes(I);
  void* scan_tmp = ws.take<char>(scan_bytes);
  uint32_t* n_cls = ws.take<uint32_t>(1);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "sampler_build: workspace too small");
  const int bits_i = bits_for(I);
  const unsigned grid = (unsigned)ceil_div(I, 256);
  k_deg_keys<<<grid, 256, 0, stream>>>(deg_i, I, bits_i, keys);
  CGX_LAUNCH_CHECK();
  uint64_t* sorted = keys;
  CGX_TRY(radix_sort_u64(keys, alt, I, bits_i + 31, sort_tmp, sort_bytes, stream, &sorted));
  k_deg_heads<<<grid, 256, 0, stream>>>(sorted, I, bits_i, flags, items_by_deg);
  CGX_LAUNCH_CHECK();
  CGX_TRY(exclusive_scan_u32(flags, flags, I, n_cls, scan_tmp, scan_bytes, stream));
  k_class_fill<<<grid, 256, 0, stream>>>(sorted, I, bits_i, flags, n_cls, class_start, class_deg, n_classes);
  CGX_LAUNCH_CHECK();
  k_vose<<<1, 32, 0, stream>>>(class_start, class_deg, n_classes, gamma, scaled, small, large, class_prob,
                               class_alias);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_sample_triples(const int64_t* users, int64_t batch, const int64_t* samp_indptr,
                                  const int32_t* samp_idx, int32_t num_items, const int32_t* items_by_deg,
                                  const int32_t* class_start, const float* class_prob, const int32_t* class_alias,
                                  const int32_t* n_classes, float mix_pop, int32_t max_tries, uint64_t seed,
                                  uint64_t offset, const uint64_t* offset_dev, int64_t* pos_out, int64_t* neg_out,
                                  void* stream_, const int64_t* slots, const int64_t* count) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(users && samp_indptr && samp_idx && pos_out && neg_out && batch > 0 && num_items > 0, CGX_ERR_ARG,
              "sample_triples: bad argument");
  if (mix_pop >= 0.f)
    CGX_REQUIRE(items_by_deg && class_start && class_prob && class_alias && n_classes, CGX_ERR_ARG,
                "sample_triples: popularity tables missing");
  SamplerTables tb{items_by_deg, class_start, class_prob, class_alias, n_classes};
  k_sample<<<(unsigned)ceil_div(batch, SM_THREADS), SM_THREADS, 0, stream>>>(
      users, batch, samp_indptr, samp_idx, num_items, tb, mix_pop, max_tries, seed, offset,
      reinterpret_cast<const unsigned long long*>(offset_dev), slots, count, pos_out, neg_out);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_eval_candidates(const int64_t* users, int64_t n_users, const int64_t* train_indptr,
                                   const int32_t* train_idx, const int64_t* test_indptr, const int32_t* test_idx,
                                   int32_t num_items, int32_t n_neg, uint64_t seed, int64_t* cand, void* stream_,
                                   int64_t row_base) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(users && train_indptr && train_idx && test_indptr && test_idx && cand && n_users > 0 && num_items > 0 &&
                  n_neg >= 0 && row_base >= 0,
              CGX_ERR_ARG, "eval_candidates: bad argument");
  const int64_t n = n_users * (1 + n_neg);
  k_eval_candidates<<<(unsigned)ceil_div(n, SM_THREADS), SM_THREADS, 0, stream>>>(
      users, n_users, train_indptr, train_idx, test_indptr, test_idx, num_items, 1 + n_neg, seed, row_base, cand);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_batch_select(const int64_t* perm, int64_t n_train, const uint64_t* step, int64_t batch, int64_t lo,
                                int64_t hi, int64_t* users_out, int64_t* slots_out, int64_t* count_out,
                                int64_t* total_out, void* stream_) {
  CGX_REQUIRE(perm && step && users_out && slots_out && count_out && total_out, CGX_ERR_ARG,
              "batch_select: NULL pointer");
  CGX_REQUIRE(n_train > 0 && batch > 0 && batch <= BS_MAX && lo >= 0 && hi >= lo, CGX_ERR_ARG,
              "batch_select: bad argument (n_train %lld, batch %lld <= %lld, range [%lld, %lld))", (long long)n_train,
              (long long)batch, (long long)BS_MAX, (long long)lo, (long long)hi);
  k_batch_select<<<1, BS_THREADS, 0, static_cast<cudaStream_t>(stream_)>>>(
      perm, n_train, reinterpret_cast<const unsigned long long*>(step), batch, lo, hi, users_out, slots_out, count_out,
      total_out);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}
