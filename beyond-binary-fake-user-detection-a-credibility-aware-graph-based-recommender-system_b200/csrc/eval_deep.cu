// Full-rank top-K for deep cut-offs, 128 < K <= 4096: exact fp32 scores, train items masked to -1e9, the best K by
// (score desc, item id asc) -- the same contract as k_eval_fp32 (eval.cu), whose per-user shared-memory list stops
// at K = 128 (64 users x K x 8 bytes per CTA).
//
// Scores: the tiling and the per-(user, item) fmaf chain of k_eval_fp32 (one chain, ascending embedding column), so
// every score has the bits the K <= 128 kernels return.  The U x I score matrix is never materialised.
//
// Selection: every user owns a candidate buffer of 2K + one tile in the caller's workspace, holding 64-bit keys
// (order-preserving score bits, ~item id) -- one integer order that is the list order of eval.cu.  A score that
// passes the user's threshold is checked against the train row (binary search), masked scores are tested again, and
// the key is appended.  When the next tile could overflow the buffer, a radix select finds the K-th key, the best K
// are compacted to the front and the threshold becomes the K-th score.  Items stream in ascending id, so after the
// first compaction a later item that ties the K-th score loses to it: the filter is a strict `>`.  Before the first
// compaction every item is kept (the buffer then holds every item seen, masked ones included).  A second kernel
// selects the final K of each buffer and sorts them in shared memory.
//
// Users are processed in chunks whose buffers fit a bounded workspace (DP_WS_BOUND; CGX_OPT_TOPK_CHUNK_USERS forces
// smaller chunks).  Chunks run one after the other on the caller's stream and reuse the same buffers.
#include <float.h>

#include "common.cuh"

namespace cgx {

constexpr int DP_THREADS = 256;
constexpr int DP_TU = 64;    // users per CTA      (as k_eval_fp32)
constexpr int DP_TI = 128;   // items per tile     (as k_eval_fp32)
constexpr int DP_KC = 16;    // embedding columns per shared-memory chunk
constexpr int DP_TIP = DP_TI + 4;
constexpr float DP_MASKED = -1e9f;   // lighgcn_cu_pop.py:702
constexpr int DP_MAX_K = 4096;
constexpr size_t DP_WS_BOUND = size_t(1) << 30;   // candidate buffers of one chunk of users

// Order-preserving key: a larger key is a better (score, id).  -0 is keyed as +0 because the list order compares
// scores as floats, where the two are equal and the lower id wins.
__device__ __forceinline__ uint64_t dp_key(float s, int32_t id) {
  uint32_t b = s == 0.f ? 0u : __float_as_uint(s);
  b ^= (b & 0x80000000u) ? 0xffffffffu : 0x80000000u;
  return (uint64_t(b) << 32) | uint64_t(~uint32_t(id));
}
__device__ __forceinline__ float dp_score(uint64_t key) {
  const uint32_t h = uint32_t(key >> 32);
  return __uint_as_float((h & 0x80000000u) ? (h ^ 0x80000000u) : ~h);
}
__device__ __forceinline__ int32_t dp_id(uint64_t key) { return int32_t(~uint32_t(key)); }

__device__ __forceinline__ bool dp_in_row(const int32_t* __restrict__ idx, int64_t lo, const int64_t end, int32_t item) {
  int64_t hi = end;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(idx + mid) < item) lo = mid + 1; else hi = mid;
  }
  return lo < end && __ldg(idx + lo) == item;
}

struct SelScratch {
  unsigned hist[256];
  unsigned res[3];   // digit, keys in the digit's bin, keys in higher bins
};

template <int GROUP>
__device__ __forceinline__ void group_sync() {
  if (GROUP == 32) __syncwarp(); else __syncthreads();
}

// The K-th largest of the n distinct keys buf[0, n), n >= K, by a group of GROUP threads (one warp, or the whole
// CTA): radix select over 8-bit digits from the top, stopping once the K-th key is alone in its digit bin.  On return
// the best K keys are exactly those with (key & mask) >= prefix, and the K-th is the only one with (key & mask) ==
// prefix.  buf was written by this CTA before the caller's last barrier.
template <int GROUP>
__device__ void select_kth(const uint64_t* buf, int n, int K, SelScratch* sc, int gt, uint64_t& prefix,
                           uint64_t& mask) {
  prefix = 0;
  mask = 0;
  unsigned rank = unsigned(K);
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int b = gt; b < 256; b += GROUP) sc->hist[b] = 0;
    group_sync<GROUP>();
    for (int i0 = gt; i0 < n; i0 += 4 * GROUP) {   // four independent loads in flight per thread
      uint64_t k4[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) k4[q] = (i0 + q * GROUP < n) ? buf[i0 + q * GROUP] : 0ull;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (i0 + q * GROUP < n && (k4[q] & mask) == prefix) atomicAdd(sc->hist + ((k4[q] >> shift) & 255), 1u);
    }
    group_sync<GROUP>();
    if (gt < 32) {   // lane l owns bins 8l .. 8l+7; higher bins are better keys
      const int lane = gt;
      unsigned c[8], s = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { c[j] = sc->hist[lane * 8 + j]; s += c[j]; }
      unsigned suf = s;   // keys in the bins of lanes >= lane
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += t;
      }
      const unsigned above = suf - s;
      if (above < rank && rank <= suf) {
        unsigned acc = above;
        for (int j = 7; j >= 0; --j) {
          if (acc + c[j] >= rank) {
            sc->res[0] = unsigned(lane * 8 + j);
            sc->res[1] = c[j];
            sc->res[2] = acc;
            break;
          }
          acc += c[j];
        }
      }
    }
    group_sync<GROUP>();
    const unsigned digit = sc->res[0], in_bin = sc->res[1];
    rank -= sc->res[2];
    prefix |= uint64_t(digit) << shift;
    mask |= uint64_t(255) << shift;
    group_sync<GROUP>();   // res and hist are read before the next digit overwrites them
    if (in_bin == 1) break;
  }
}

// One CTA = 64 users; streams every item tile and leaves each user's candidates (>= K keys, unordered) in
// buf[row * cap ...] and their number in buf_n[row].
__global__ void __launch_bounds__(DP_THREADS) k_eval_deep(const int64_t* __restrict__ users, int64_t n_users,
                                                          const float* __restrict__ f_u,
                                                          const float* __restrict__ f_i, int32_t I, int32_t d,
                                                          const int64_t* __restrict__ tr_indptr,
                                                          const int32_t* __restrict__ tr_idx, int32_t K, int64_t cap,
                                                          uint64_t* __restrict__ buf, int32_t* __restrict__ buf_n) {
  __shared__ __align__(16) float Us[DP_KC * DP_TU];
  __shared__ __align__(16) float Is[DP_KC * DP_TIP];
  __shared__ float thr[DP_TU];
  __shared__ int cnt[DP_TU];
  __shared__ int closed[DP_TU];   // 1 once the user's buffer has been compacted: thr is then the K-th score
  __shared__ int64_t urow[DP_TU];
  __shared__ SelScratch sel[DP_THREADS / 32];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ty = tid >> 4, tx = tid & 15;  // 16 x 16 threads: 4 users x 8 items each
  const int64_t u0 = int64_t(blockIdx.x) * DP_TU;
  if (u0 >= n_users) return;
  if (tid < DP_TU) {
    thr[tid] = -FLT_MAX;
    cnt[tid] = 0;
    closed[tid] = 0;
    urow[tid] = (u0 + tid < n_users) ? users[u0 + tid] : -1;
  }
  __syncthreads();

  for (int32_t i0 = 0; i0 < I; i0 += DP_TI) {
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;

    for (int k0 = 0; k0 < d; k0 += DP_KC) {
      {  // user chunk: 64 rows x 16 cols = 256 float4, one per thread
        const int r = tid >> 2, q = tid & 3;
        const int64_t ur = urow[r];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ur >= 0) v = __ldg(reinterpret_cast<const float4*>(f_u + ur * d + k0) + q);
        Us[(q * 4 + 0) * DP_TU + r] = v.x;
        Us[(q * 4 + 1) * DP_TU + r] = v.y;
        Us[(q * 4 + 2) * DP_TU + r] = v.z;
        Us[(q * 4 + 3) * DP_TU + r] = v.w;
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {  // item chunk: 128 rows x 16 cols = 512 float4, two per thread
        const int f = tid + h * DP_THREADS;
        const int r = f >> 2, q = f & 3;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i0 + r < I) v = __ldg(reinterpret_cast<const float4*>(f_i + int64_t(i0 + r) * d + k0) + q);
        Is[(q * 4 + 0) * DP_TIP + r] = v.x;
        Is[(q * 4 + 1) * DP_TIP + r] = v.y;
        Is[(q * 4 + 2) * DP_TIP + r] = v.z;
        Is[(q * 4 + 3) * DP_TIP + r] = v.w;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < DP_KC; ++k) {
        const float4 uu = *reinterpret_cast<const float4*>(Us + k * DP_TU + ty * 4);
        const float4 ia = *reinterpret_cast<const float4*>(Is + k * DP_TIP + tx * 4);
        const float4 ib = *reinterpret_cast<const float4*>(Is + k * DP_TIP + 64 + tx * 4);
        const float uv[4] = {uu.x, uu.y, uu.z, uu.w};
        const float iv[8] = {ia.x, ia.y, ia.z, ia.w, ib.x, ib.y, ib.z, ib.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(uv[a], iv[b], acc[a][b]);
      }
      __syncthreads();
    }

    // filter against the per-user threshold; survivors are checked against the train row and appended
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int ul = ty * 4 + a;
      const int64_t ur = urow[ul];
      if (ur < 0) continue;
      const float t = thr[ul];
      const bool open = closed[ul] == 0;
      uint64_t* ub = buf + (u0 + ul) * cap;
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const int32_t item = i0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + (b - 4));
        float s = acc[a][b];
        if (item < I && (open || s > t)) {
          if (dp_in_row(tr_idx, __ldg(tr_indptr + ur), __ldg(tr_indptr + ur + 1), item)) s = DP_MASKED;
          if (open || s > t) ub[atomicAdd(&cnt[ul], 1)] = dp_key(s, item);
        }
      }
    }
    __syncthreads();

    // compaction of every buffer the next tile could overflow: one warp per user
    for (int ul = warp; ul < DP_TU; ul += DP_THREADS / 32) {
      const int n = cnt[ul];
      if (urow[ul] < 0 || n + DP_TI <= cap) continue;
      uint64_t* ub = buf + (u0 + ul) * cap;
      uint64_t prefix, mask;
      select_kth<32>(ub, n, K, sel + warp, lane, prefix, mask);
      int w = 0;
      for (int base = 0; base < n; base += 32) {   // in place: a chunk is loaded by every lane before any writes
        const int i = base + lane;
        const uint64_t key = i < n ? ub[i] : 0ull;
        const bool keep = i < n && (key & mask) >= prefix;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) {
          ub[w + __popc(bal & ((1u << lane) - 1u))] = key;
          if ((key & mask) == prefix) thr[ul] = dp_score(key);
        }
        w += __popc(bal);
      }
      if (lane == 0) {
        cnt[ul] = K;
        closed[ul] = 1;
      }
      __syncwarp();
    }
    __syncthreads();
  }

  if (tid < DP_TU && urow[tid] >= 0) buf_n[u0 + tid] = cnt[tid];
}

// One CTA per user: the best K of the user's buffer, sorted by key (score desc, id asc) with a bitonic sort of P
// (power of two >= K) keys in shared memory.
__global__ void __launch_bounds__(DP_THREADS) k_eval_deep_finish(const uint64_t* __restrict__ buf,
                                                                 const int32_t* __restrict__ buf_n, int64_t cap,
                                                                 int32_t K, int32_t P, int32_t* __restrict__ out_ids,
                                                                 float* __restrict__ out_scores) {
  extern __shared__ uint64_t sk[];   // [P]
  __shared__ SelScratch sel;
  __shared__ int pos;
  const int tid = threadIdx.x;
  const int64_t r = blockIdx.x;
  const uint64_t* ub = buf + r * cap;
  const int n = buf_n[r];
  uint64_t prefix = 0, mask = 0;     // n == K: every key is kept
  if (n > K) select_kth<DP_THREADS>(ub, n, K, &sel, tid, prefix, mask);
  if (tid == 0) pos = 0;
  __syncthreads();
  for (int i = tid; i < n; i += DP_THREADS) {
    const uint64_t key = ub[i];
    if ((key & mask) >= prefix) sk[atomicAdd(&pos, 1)] = key;
  }
  for (int i = K + tid; i < P; i += DP_THREADS) sk[i] = 0ull;   // below every real key
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < P / 2; t += DP_THREADS) {
        const int i = 2 * t - (t & (stride - 1)), j = i + stride;
        const bool desc = (i & size) == 0;
        const uint64_t a = sk[i], b = sk[j];
        if ((a < b) == desc) { sk[i] = b; sk[j] = a; }
      }
      __syncthreads();
    }
  }
  for (int j = tid; j < K; j += DP_THREADS) {
    out_ids[r * K + j] = dp_id(sk[j]);
    out_scores[r * K + j] = dp_score(sk[j]);
  }
}

static int64_t deep_cap(int32_t K) { return 2 * int64_t(K) + DP_TI; }

// users per chunk: as many as the bounded workspace holds (16,128 at K = 4096), a multiple of the CTA's 64 users
static int64_t deep_chunk_users(int64_t n_users, int32_t K) {
  int64_t c = int64_t(DP_WS_BOUND / size_t(deep_cap(K) * 8 + 4)) / DP_TU * DP_TU;
  if (c < DP_TU) c = DP_TU;
  const int64_t forced = option(CGX_OPT_TOPK_CHUNK_USERS);
  if (forced > 0 && forced < c) c = forced;
  return n_users < c ? n_users : c;
}

int eval_topk_deep_max_k() { return DP_MAX_K; }

size_t eval_topk_deep_workspace(int64_t n_users, int32_t K) {
  const int64_t c = deep_chunk_users(n_users > 0 ? n_users : 1, K);
  return align_up(size_t(c) * size_t(deep_cap(K)) * 8) + align_up(size_t(c) * 4) + 256;
}

int eval_topk_deep(const int64_t* users, int64_t n_users, const float* f_u, const float* f_i, int32_t I, int32_t d,
                   const int64_t* tr_indptr, const int32_t* tr_idx, int32_t K, int32_t* out_ids, float* out_scores,
                   void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CGX_REQUIRE(K > 128 && K <= DP_MAX_K, CGX_ERR_ARG, "eval_topk: deep path needs 128 < k <= %d, got %d", DP_MAX_K, K);
  CGX_REQUIRE(workspace_bytes >= eval_topk_deep_workspace(n_users, K), CGX_ERR_WORKSPACE,
              "eval_topk: workspace too small");
  const int64_t chunk = deep_chunk_users(n_users, K), cap = deep_cap(K);
  Arena ws(workspace, workspace_bytes);
  uint64_t* buf = ws.take<uint64_t>(size_t(chunk) * cap);
  int32_t* buf_n = ws.take<int32_t>(chunk);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "eval_topk: workspace too small");
  int P = 1;
  while (P < K) P <<= 1;
  for (int64_t c0 = 0; c0 < n_users; c0 += chunk) {
    const int64_t m = n_users - c0 < chunk ? n_users - c0 : chunk;
    k_eval_deep<<<(unsigned)ceil_div(m, DP_TU), DP_THREADS, 0, stream>>>(users + c0, m, f_u, f_i, I, d, tr_indptr,
                                                                         tr_idx, K, cap, buf, buf_n);
    CGX_LAUNCH_CHECK();
    k_eval_deep_finish<<<(unsigned)m, DP_THREADS, size_t(P) * 8, stream>>>(buf, buf_n, cap, K, P, out_ids + c0 * K,
                                                                          out_scores + c0 * K);
    CGX_LAUNCH_CHECK();
  }
  return CGX_OK;
}

}  // namespace cgx
