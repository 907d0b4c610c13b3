// Ranking metrics on the device: precision / recall / NDCG at several cut-offs, item coverage, novelty
// (mean log popularity, mean self-information) and per-credibility-group recall, from the [n, K] matrix of
// ranked item ids that cgx_eval_topk / cgx_rank_candidates leave in HBM.
//
// Replaces (reference, /root/reference): metrics_at_k lightgcn_cu.py:469-484 / Version-2/lighgcn_cu_pop.py:
// 514-530 and the per-user accumulation loops of evaluate_full_ranking (V2:691-752: coverage set, novelty via
// novelty_stats_for_items V2:390-404, high/low credibility recall V2:739-747) and of evaluate_sampled
// (CU:521-546).  The reference accumulates in Python floats (double); so does this file.
//
// Only sums leave the GPU (7 doubles + one count per cut-off): at C5 the ranked matrix is 29 M x 20 ids, which the host
// path would copy and walk.  Everything is deterministic: block partials are combined in a fixed order, the
// coverage bitmap uses integer atomics only.
#include "common.cuh"

namespace cgx {

constexpr int MET_MAX_KS = 8;     // distinct cut-offs per call
constexpr int MET_MAX_K = 4096;   // largest cut-off (the deepest list cgx_eval_topk returns)
constexpr int MET_SUMS = 7;       // precision, recall, ndcg, log-pop, self-information, high-cred recall, low-cred recall
constexpr int MET_THREADS = 256;

struct MetKs {
  int32_t k[MET_MAX_KS];   // ascending
  int32_t n;
};

__device__ __forceinline__ bool met_in_row(const int32_t* __restrict__ idx, int64_t lo, const int64_t end, int32_t item) {
  int64_t hi = end;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(idx + mid) < item) lo = mid + 1; else hi = mid;
  }
  return lo < end && __ldg(idx + lo) == item;
}

// one thread per evaluated user; at every cut-off the block reduces its 7 sums (fixed order) into
// partial[blockIdx][ki][7]
__global__ void __launch_bounds__(MET_THREADS) k_metrics(const int32_t* __restrict__ ranked, int64_t n, int32_t ld,
                                                         const int64_t* __restrict__ users,
                                                         const int64_t* __restrict__ te_indptr,
                                                         const int32_t* __restrict__ te_idx,
                                                         const int32_t* __restrict__ gt_single, int32_t I, MetKs ks,
                                                         const int64_t* __restrict__ item_pop, double pop_denom,
                                                         const uint8_t* __restrict__ group,
                                                         uint32_t* __restrict__ bitmaps, int64_t words,
                                                         double* __restrict__ partial) {
  extern __shared__ double met_tab[];   // disc[kmax], idcg[kmax + 1]: sized by the largest cut-off
  __shared__ double red[MET_THREADS / 32][MET_SUMS];
  const int kmax = ks.k[ks.n - 1];
  double* disc = met_tab;
  double* idcg = met_tab + kmax;
  for (int r = threadIdx.x; r < kmax; r += MET_THREADS) disc[r] = 1.0 / log2(double(r) + 2.0);
  __syncthreads();
  if (threadIdx.x == 0) {
    idcg[0] = 0.0;
    for (int r = 0; r < kmax; ++r) idcg[r + 1] = idcg[r] + disc[r];   // np.cumsum order
  }
  __syncthreads();

  const int64_t r = int64_t(blockIdx.x) * MET_THREADS + threadIdx.x;
  const bool live = r < n;
  int64_t lo = 0, hi = 0, n_gt = 1;
  int32_t single = -1;
  uint8_t grp = 0;
  if (live) {
    if (gt_single) {
      single = gt_single[r];
    } else {
      const int64_t u = users[r];
      lo = __ldg(te_indptr + u);
      hi = __ldg(te_indptr + u + 1);
      n_gt = hi - lo;
    }
    if (group) grp = group[r];
  }
  const double inv_gt = 1.0 / double(n_gt > 1 ? n_gt : 1);
  int nh = 0;
  double dcg = 0.0, lp = 0.0, si = 0.0;
  int ki = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int j = 0; j < kmax; ++j) {
    if (live) {
      const int32_t id = ranked[r * ld + j];
      if (id >= 0 && id < I) {
        const bool hit = gt_single ? id == single : met_in_row(te_idx, lo, hi, id);
        if (hit) { ++nh; dcg += disc[j]; }
        if (item_pop) {
          const double p = double(__ldg(item_pop + id)) + 1.0;
          lp += log(p);
          si -= log2(p / pop_denom);
        }
        if (bitmaps) atomicOr(bitmaps + int64_t(ki) * words + (id >> 5), 1u << (id & 31));
      }
    }
    if (j + 1 == ks.k[ki]) {   // cut-off reached (uniform over the block)
      const int K = ks.k[ki];
      double v[MET_SUMS];
#pragma unroll
      for (int m = 0; m < MET_SUMS; ++m) v[m] = 0.0;
      if (live) {
        const double recall = double(nh) * inv_gt;
        const double ideal = idcg[n_gt < K ? n_gt : K];
        v[0] = double(nh) / double(K);
        v[1] = recall;
        v[2] = ideal > 0.0 ? dcg / ideal : 0.0;
        v[3] = lp / double(K);
        v[4] = si / double(K);
        v[5] = (grp & 1) ? recall : 0.0;
        v[6] = (grp & 2) ? recall : 0.0;
      }
#pragma unroll
      for (int m = 0; m < MET_SUMS; ++m) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[m] += __shfl_xor_sync(0xffffffffu, v[m], o);
      }
      __syncthreads();   // red[] of the previous cut-off has been consumed
      if (lane == 0) {
#pragma unroll
        for (int m = 0; m < MET_SUMS; ++m) red[warp][m] = v[m];
      }
      __syncthreads();
      if (threadIdx.x < MET_SUMS) {
        double s = 0.0;
        for (int w = 0; w < MET_THREADS / 32; ++w) s += red[w][threadIdx.x];
        partial[(int64_t(blockIdx.x) * ks.n + ki) * MET_SUMS + threadIdx.x] = s;
      }
      ++ki;
    }
  }
}

// distinct items among the first Ks[ki] columns = popcount of the OR of bitmaps 0..ki
__global__ void __launch_bounds__(256) k_metrics_cover(const uint32_t* __restrict__ bitmaps, int64_t words, int n_ks,
                                                       unsigned long long* __restrict__ counts) {
  unsigned long long c[MET_MAX_KS];
#pragma unroll
  for (int ki = 0; ki < MET_MAX_KS; ++ki) c[ki] = 0ull;
  for (int64_t w = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; w < words; w += int64_t(gridDim.x) * blockDim.x) {
    uint32_t u = 0u;
#pragma unroll
    for (int ki = 0; ki < MET_MAX_KS; ++ki) {
      if (ki < n_ks) {
        u |= bitmaps[int64_t(ki) * words + w];
        c[ki] += __popc(u);
      }
    }
  }
#pragma unroll
  for (int ki = 0; ki < MET_MAX_KS; ++ki) {
    if (ki < n_ks) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) c[ki] += __shfl_xor_sync(0xffffffffu, c[ki], o);
      if ((threadIdx.x & 31) == 0 && c[ki]) atomicAdd(counts + ki, c[ki]);   // integer: order-independent
    }
  }
}

// block b = (ki, m): sums partial[:, ki, m] in a fixed order into out[ki][m]
__global__ void __launch_bounds__(256) k_metrics_final(const double* __restrict__ partial, int64_t n_blocks, int n_ks,
                                                       double* __restrict__ out) {
  __shared__ double sh[256];
  const int ki = blockIdx.x / MET_SUMS, m = blockIdx.x % MET_SUMS;
  double s = 0.0;
  for (int64_t b = threadIdx.x; b < n_blocks; b += 256) s += partial[(b * n_ks + ki) * MET_SUMS + m];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[ki * MET_SUMS + m] = sh[0];
}

}  // namespace cgx

using namespace cgx;

extern "C" size_t cgx_eval_metrics_workspace_bytes(int64_t n_users, int32_t n_ks) {
  const int64_t blocks = ceil_div(n_users > 0 ? n_users : 1, MET_THREADS);
  return align_up(size_t(blocks) * n_ks * MET_SUMS * 8) + 256;
}

extern "C" int cgx_eval_metrics(const int32_t* ranked, int64_t n_users, int32_t ld, const int64_t* users,
                                const int64_t* test_indptr, const int32_t* test_idx, const int32_t* gt_single,
                                int32_t num_items, const int32_t* ks_host, int32_t n_ks, const int64_t* item_pop,
                                int64_t total_train, const uint8_t* group, uint32_t* bitmaps, double* out,
                                void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(ranked && out && ks_host && n_users > 0 && num_items > 0, CGX_ERR_ARG, "eval_metrics: bad argument");
  CGX_REQUIRE(gt_single != nullptr || (users && test_indptr && test_idx), CGX_ERR_ARG,
              "eval_metrics: need test rows or gt_single");
  CGX_REQUIRE(n_ks >= 1 && n_ks <= MET_MAX_KS, CGX_ERR_ARG, "eval_metrics: 1..%d cut-offs", MET_MAX_KS);
  MetKs ks;
  ks.n = n_ks;
  for (int i = 0; i < MET_MAX_KS; ++i) ks.k[i] = i < n_ks ? ks_host[i] : 0x7fffffff;
  for (int i = 0; i < n_ks; ++i)
    CGX_REQUIRE(ks.k[i] >= 1 && ks.k[i] <= MET_MAX_K && ks.k[i] <= ld && (i == 0 || ks.k[i] > ks.k[i - 1]), CGX_ERR_ARG,
                "eval_metrics: cut-offs must be ascending, 1..%d and <= ld", MET_MAX_K);
  CGX_REQUIRE(workspace_bytes >= cgx_eval_metrics_workspace_bytes(n_users, n_ks), CGX_ERR_WORKSPACE,
              "eval_metrics: workspace too small");
  const int64_t words = (int64_t(num_items) + 31) / 32;
  const int64_t blocks = ceil_div(n_users, MET_THREADS);
  Arena ws(workspace, workspace_bytes);
  double* partial = ws.take<double>(size_t(blocks) * n_ks * MET_SUMS);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "eval_metrics: workspace too small");
  const size_t tab_smem = size_t(2 * ks.k[n_ks - 1] + 1) * sizeof(double);   // 64 KB at a cut-off of 4096
  CGX_CUDA(cudaFuncSetAttribute(k_metrics, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tab_smem));
  k_metrics<<<(unsigned)blocks, MET_THREADS, tab_smem, stream>>>(ranked, n_users, ld, users, test_indptr, test_idx,
                                                                gt_single, num_items, ks, item_pop,
                                                                double(total_train) + double(num_items), group,
                                                                bitmaps, words, partial);
  CGX_LAUNCH_CHECK();
  k_metrics_final<<<n_ks * MET_SUMS, 256, 0, stream>>>(partial, blocks, n_ks, out);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_eval_coverage(const uint32_t* bitmaps, int32_t num_items, int32_t n_ks, uint64_t* counts,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(bitmaps && counts && num_items > 0 && n_ks >= 1 && n_ks <= MET_MAX_KS, CGX_ERR_ARG,
              "eval_coverage: bad argument");
  const int64_t words = (int64_t(num_items) + 31) / 32;
  CGX_CUDA(cudaMemsetAsync(counts, 0, size_t(n_ks) * 8, stream));
  int64_t blocks = ceil_div(words, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_metrics_cover<<<(unsigned)blocks, 256, 0, stream>>>(bitmaps, words, n_ks,
                                                       reinterpret_cast<unsigned long long*>(counts));
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}
