// Full-rank evaluation: user x item score tiles fused with the train-item mask and a per-row
// running top-K, plus candidate-list scoring for the sampled protocol.  This file holds the exact
// fp32 path (CUDA cores) for K <= 128; the tensor-core path lives in eval_tc.cu and reuses the selection code, and
// K > 128 runs the candidate-buffer kernels of eval_deep.cu.
//
// Replaces (reference, /root/reference): the per-user loop of evaluate_full_ranking,
// Version-2/lighgcn_cu_pop.py:691-704 (mul+sum scores, scores[train] = -1e9, full argsort) and the
// candidate scoring of evaluate_sampled, lightgcn_cu.py:521-527.
//
// The U x I score matrix is never materialised: a CTA owns EV_TU users, streams item tiles of
// EV_TI, and keeps each user's best K as a sorted list in shared memory.  A score only reaches
// the list code when it is >= the user's current K-th best (a monotone lower bound), so after
// the first tiles almost every score is discarded by one compare in registers.
// Total order: higher score first, ties by lower item id (BASELINE.json: "ties broken by index").
#include <float.h>

#include "common.cuh"

namespace cgx {

constexpr int EV_THREADS = 256;
constexpr int EV_TU = 64;    // users per CTA
constexpr int EV_TI = 128;   // items per tile
constexpr int EV_KC = 16;    // embedding columns per shared-memory chunk
constexpr int EV_TIP = EV_TI + 4;
constexpr float EV_MASKED = -1e9f;   // lighgcn_cu_pop.py:702

__device__ __forceinline__ bool better(float sa, int32_t ia, float sb, int32_t ib) {
  return sa > sb || (sa == sb && ia < ib);
}

__device__ __forceinline__ bool in_row(const int32_t* __restrict__ idx, int64_t lo, const int64_t end, int32_t item) {
  int64_t hi = end;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(idx + mid) < item) lo = mid + 1; else hi = mid;
  }
  return lo < end && __ldg(idx + lo) == item;
}

// One warp merges the candidates of one user into that user's sorted list (shared memory).
__device__ __forceinline__ void merge_candidates(int lane, int K, float* ls, int32_t* li, const float* cs,
                                                 const int32_t* ci, int n_cand, const int32_t* __restrict__ tr_idx,
                                                 int64_t tr_lo, int64_t tr_hi, float* thr) {
  for (int j = 0; j < n_cand; ++j) {
    float s = cs[j];
    const int32_t id = ci[j];
    if (in_row(tr_idx, tr_lo, tr_hi, id)) s = EV_MASKED;
    if (!better(s, id, ls[K - 1], li[K - 1])) continue;
    // position = number of list entries that beat the candidate (they form a prefix)
    int pos = 0;
    for (int b = 0; b < K; b += 32) {
      const int p = b + lane;
      const bool w = p < K && better(ls[p], li[p], s, id);
      pos += __popc(__ballot_sync(0xffffffffu, w));
    }
    for (int b = ((K - 1) / 32) * 32; b >= 0; b -= 32) {  // shift the tail down by one, high blocks first
      const int p = b + lane;
      float ms = 0.f;
      int32_t mi = 0;
      const bool mv = p < K && p > pos;
      if (mv) { ms = ls[p - 1]; mi = li[p - 1]; }
      __syncwarp();
      if (mv) { ls[p] = ms; li[p] = mi; }
      __syncwarp();
    }
    if (lane == 0) { ls[pos] = s; li[pos] = id; }
    __syncwarp();
  }
  if (lane == 0) *thr = ls[K - 1];
  __syncwarp();
}

// row_list / n_rows_dev (both optional): evaluate only the rows row_list[0 .. *n_rows_dev) of `users`
// (used to redo the rows the tensor-core path could not prove complete); outputs go to those rows.
__global__ void __launch_bounds__(EV_THREADS) k_eval_fp32(const int64_t* __restrict__ users, int64_t n_users,
                                                          const int32_t* __restrict__ row_list,
                                                          const int32_t* __restrict__ n_rows_dev,
                                                          const float* __restrict__ f_u,
                                                          const float* __restrict__ f_i, int32_t I, int32_t d,
                                                          const int64_t* __restrict__ tr_indptr,
                                                          const int32_t* __restrict__ tr_idx, int32_t K,
                                                          int32_t* __restrict__ out_ids,
                                                          float* __restrict__ out_scores) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Us = reinterpret_cast<float*>(smem_raw);               // [EV_KC][EV_TU]
  float* Is = Us + EV_KC * EV_TU;                               // [EV_KC][EV_TIP]
  float* cand_s = Is + EV_KC * EV_TIP;                          // [EV_TU][EV_TI]
  int32_t* cand_i = reinterpret_cast<int32_t*>(cand_s + EV_TU * EV_TI);
  float* list_s = reinterpret_cast<float*>(cand_i + EV_TU * EV_TI);  // [EV_TU][K]
  int32_t* list_i = reinterpret_cast<int32_t*>(list_s + EV_TU * K);
  float* thr = reinterpret_cast<float*>(list_i + EV_TU * K);    // [EV_TU]
  int* cnt = reinterpret_cast<int*>(thr + EV_TU);               // [EV_TU]
  int64_t* urow = reinterpret_cast<int64_t*>(cnt + EV_TU);      // [EV_TU] global user ids (8-byte aligned by layout)
  int64_t* orow = urow + EV_TU;                                 // [EV_TU] output rows

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ty = tid >> 4, tx = tid & 15;  // 16 x 16 threads: 4 users x 8 items each
  const int64_t u0 = int64_t(blockIdx.x) * EV_TU;
  if (n_rows_dev != nullptr) n_users = *n_rows_dev;
  if (u0 >= n_users) return;

  for (int p = tid; p < EV_TU * K; p += EV_THREADS) { list_s[p] = -FLT_MAX; list_i[p] = INT32_MAX; }
  if (tid < EV_TU) {
    thr[tid] = -FLT_MAX;
    cnt[tid] = 0;
    const int64_t r = (u0 + tid < n_users) ? (row_list ? int64_t(row_list[u0 + tid]) : u0 + tid) : -1;
    orow[tid] = r;
    urow[tid] = r >= 0 ? users[r] : -1;
  }
  __syncthreads();

  for (int32_t i0 = 0; i0 < I; i0 += EV_TI) {
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;

    for (int k0 = 0; k0 < d; k0 += EV_KC) {
      {  // user chunk: 64 rows x 16 cols = 256 float4, one per thread
        const int r = tid >> 2, q = tid & 3;
        const int64_t ur = urow[r];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ur >= 0) v = __ldg(reinterpret_cast<const float4*>(f_u + ur * d + k0) + q);
        Us[(q * 4 + 0) * EV_TU + r] = v.x;
        Us[(q * 4 + 1) * EV_TU + r] = v.y;
        Us[(q * 4 + 2) * EV_TU + r] = v.z;
        Us[(q * 4 + 3) * EV_TU + r] = v.w;
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {  // item chunk: 128 rows x 16 cols = 512 float4, two per thread
        const int f = tid + h * EV_THREADS;
        const int r = f >> 2, q = f & 3;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i0 + r < I) v = __ldg(reinterpret_cast<const float4*>(f_i + int64_t(i0 + r) * d + k0) + q);
        Is[(q * 4 + 0) * EV_TIP + r] = v.x;
        Is[(q * 4 + 1) * EV_TIP + r] = v.y;
        Is[(q * 4 + 2) * EV_TIP + r] = v.z;
        Is[(q * 4 + 3) * EV_TIP + r] = v.w;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < EV_KC; ++k) {
        const float4 uu = *reinterpret_cast<const float4*>(Us + k * EV_TU + ty * 4);
        const float4 ia = *reinterpret_cast<const float4*>(Is + k * EV_TIP + tx * 4);
        const float4 ib = *reinterpret_cast<const float4*>(Is + k * EV_TIP + 64 + tx * 4);
        const float uv[4] = {uu.x, uu.y, uu.z, uu.w};
        const float iv[8] = {ia.x, ia.y, ia.z, ia.w, ib.x, ib.y, ib.z, ib.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(uv[a], iv[b], acc[a][b]);
      }
      __syncthreads();
    }

    // filter against the per-user threshold
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int ul = ty * 4 + a;
      if (urow[ul] < 0) continue;
      const float t = thr[ul];
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const int32_t item = i0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + (b - 4));
        if (item < I && acc[a][b] >= t) {
          const int slot = atomicAdd(&cnt[ul], 1);
          cand_s[ul * EV_TI + slot] = acc[a][b];
          cand_i[ul * EV_TI + slot] = item;
        }
      }
    }
    __syncthreads();
    for (int ul = warp; ul < EV_TU; ul += EV_THREADS / 32) {
      const int c = cnt[ul];
      if (c == 0) continue;
      const int64_t ur = urow[ul];
      merge_candidates(lane, K, list_s + ul * K, list_i + ul * K, cand_s + ul * EV_TI, cand_i + ul * EV_TI, c,
                       tr_idx, __ldg(tr_indptr + ur), __ldg(tr_indptr + ur + 1), thr + ul);
      if (lane == 0) cnt[ul] = 0;
    }
    __syncthreads();
  }

  for (int p = tid; p < EV_TU * K; p += EV_THREADS) {
    const int ul = p / K, r = p % K;
    if (orow[ul] >= 0) {
      out_ids[orow[ul] * K + r] = list_i[p];
      out_scores[orow[ul] * K + r] = list_s[p];
    }
  }
}

static size_t eval_smem_bytes(int K) {
  return size_t(EV_KC * EV_TU + EV_KC * EV_TIP) * 4 + size_t(EV_TU) * EV_TI * 8 + size_t(EV_TU) * K * 8 +
         size_t(EV_TU) * 8 + size_t(EV_TU) * 16 + 64;
}

template <int G, int V>
__global__ void __launch_bounds__(256) k_score_cands(const int64_t* __restrict__ users,
                                                     const int64_t* __restrict__ cand, int64_t n_pairs,
                                                     int32_t n_cand, const float4* __restrict__ f_u,
                                                     const float4* __restrict__ f_i, float* __restrict__ scores) {
  constexpr int ROW4 = G * V;
  const int lane = threadIdx.x & (G - 1);
  const int64_t p = (int64_t(blockIdx.x) * 256 + threadIdx.x) / G;
  if (p >= n_pairs) return;
  unsigned mask = 0xffffffffu;
  if (G < 32) mask = ((1u << (G & 31)) - 1u) << ((threadIdx.x & 31) & ~(G - 1));
  const int64_t u = users[p / n_cand], it = cand[p];
  float s = 0.f;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const float4 a = __ldg(f_u + u * ROW4 + v * G + lane), b = __ldg(f_i + it * ROW4 + v * G + lane);
    s += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(mask, s, o, G);
  if (lane == 0) scores[p] = s;
}

// one warp per user: stable descending sort of C candidate scores by rank counting (np.argsort(-scores, stable))
__global__ void __launch_bounds__(256) k_rank_cands(const float* __restrict__ scores, const int64_t* __restrict__ cand,
                                                    int64_t n_users, int32_t C, int64_t* __restrict__ ranked) {
  const int lane = threadIdx.x & 31;
  const int64_t r = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= n_users) return;
  const float* s = scores + r * C;
  for (int i = lane; i < C; i += 32) {
    const float si = s[i];
    int rank = 0;
    for (int j = 0; j < C; ++j) {
      const float sj = __ldg(s + j);
      rank += (sj > si || (sj == si && j < i)) ? 1 : 0;
    }
    ranked[r * C + rank] = cand[r * C + i];
  }
}

int eval_topk_tc(const int64_t* users, int64_t n_users, const float* f_u, const float* f_i, int32_t I, int32_t d,
                 const int64_t* tr_indptr, const int32_t* tr_idx, int32_t K, int precision, int32_t* out_ids,
                 float* out_scores, void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t eval_topk_tc_workspace(int64_t n_users, int32_t I, int32_t d, int32_t K, int precision);
int eval_topk_deep(const int64_t* users, int64_t n_users, const float* f_u, const float* f_i, int32_t I, int32_t d,
                   const int64_t* tr_indptr, const int32_t* tr_idx, int32_t K, int32_t* out_ids, float* out_scores,
                   void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t eval_topk_deep_workspace(int64_t n_users, int32_t K);
int eval_topk_deep_max_k();

// exact path on (a subset of) the rows; grid sized for max_rows, CTAs past *n_rows_dev exit at once
int eval_fp32_rows(const int64_t* users, const int32_t* row_list, const int32_t* n_rows_dev, int64_t max_rows,
                   const float* f_u, const float* f_i, int32_t I, int32_t d, const int64_t* tr_indptr,
                   const int32_t* tr_idx, int32_t K, int32_t* out_ids, float* out_scores, cudaStream_t stream) {
  const size_t smem = eval_smem_bytes(K);
  CGX_CUDA(cudaFuncSetAttribute(k_eval_fp32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_eval_fp32<<<(unsigned)ceil_div(max_rows, EV_TU), EV_THREADS, smem, stream>>>(
      users, max_rows, row_list, n_rows_dev, f_u, f_i, I, d, tr_indptr, tr_idx, K, out_ids, out_scores);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

}  // namespace cgx

using namespace cgx;

extern "C" size_t cgx_eval_topk_workspace_bytes(int64_t n_users, int32_t num_items, int32_t d, int32_t k,
                                                int precision) {
  if (k > 128) return eval_topk_deep_workspace(n_users, k);   // every precision: exact fp32 (eval_deep.cu)
  if (precision == CGX_SCORE_FP32) return 256;
  return eval_topk_tc_workspace(n_users, num_items, d, k, precision);
}

extern "C" int cgx_eval_topk(const int64_t* users, int64_t n_users, const float* f_u, const float* f_i, int32_t I,
                             int32_t d, const int64_t* train_indptr, const int32_t* train_idx, int32_t k,
                             int precision, int32_t* out_ids, float* out_scores, void* workspace,
                             size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(users && f_u && f_i && train_indptr && out_ids && out_scores, CGX_ERR_ARG, "eval_topk: NULL pointer");
  CGX_REQUIRE(n_users > 0 && I > 0 && k > 0 && k <= eval_topk_deep_max_k() && k <= I, CGX_ERR_ARG,
              "eval_topk: need 0 < k <= min(%d, num_items), got k=%d I=%d", eval_topk_deep_max_k(), k, I);
  CGX_REQUIRE(cgx_emb_dim_supported(d), CGX_ERR_UNSUPPORTED, "eval_topk: emb_dim %d unsupported", d);
  CGX_REQUIRE(precision == CGX_SCORE_FP32 || precision == CGX_SCORE_BF16X3 || precision == CGX_SCORE_BF16,
              CGX_ERR_ARG, "eval_topk: bad precision %d", precision);
  if (k > 128)   // past the shared-memory list of k_eval_fp32: the deep path, exact fp32 for every precision
    return eval_topk_deep(users, n_users, f_u, f_i, I, d, train_indptr, train_idx, k, out_ids, out_scores, workspace,
                          workspace_bytes, stream);
  if (precision != CGX_SCORE_FP32)
    return eval_topk_tc(users, n_users, f_u, f_i, I, d, train_indptr, train_idx, k, precision, out_ids, out_scores,
                        workspace, workspace_bytes, stream);
  return eval_fp32_rows(users, nullptr, nullptr, n_users, f_u, f_i, I, d, train_indptr, train_idx, k, out_ids,
                        out_scores, stream);
}

extern "C" int cgx_score_candidates(const int64_t* users, const int64_t* cand, int64_t n_users, int32_t n_cand,
                                    int32_t d, const float* f_u, const float* f_i, float* scores, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(users && cand && f_u && f_i && scores && n_users > 0 && n_cand > 0, CGX_ERR_ARG,
              "score_candidates: bad argument");
  const int64_t n_pairs = n_users * n_cand;
#define CGX_SC(GG, VV)                                                                                   \
  k_score_cands<GG, VV><<<(unsigned)ceil_div(n_pairs, 256 / GG), 256, 0, stream>>>(                       \
      users, cand, n_pairs, n_cand, reinterpret_cast<const float4*>(f_u), reinterpret_cast<const float4*>(f_i), \
      scores)
  switch (d) {
    case 16: CGX_SC(4, 1); break;
    case 32: CGX_SC(8, 1); break;
    case 64: CGX_SC(16, 1); break;
    case 128: CGX_SC(32, 1); break;
    case 256: CGX_SC(32, 2); break;
    default:
      set_error("score_candidates: emb_dim %d unsupported", d);
      return CGX_ERR_UNSUPPORTED;
  }
#undef CGX_SC
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

extern "C" int cgx_rank_candidates(const float* scores, const int64_t* cand, int64_t n_users, int32_t n_cand,
                                   int64_t* ranked, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(scores && cand && ranked && n_users > 0 && n_cand > 0, CGX_ERR_ARG, "rank_candidates: bad argument");
  k_rank_cands<<<(unsigned)ceil_div(n_users, 8), 256, 0, stream>>>(scores, cand, n_users, n_cand, ranked);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}
