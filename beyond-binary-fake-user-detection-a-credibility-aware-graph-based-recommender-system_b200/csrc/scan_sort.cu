// Exclusive scan (three-phase, recursive) and stable LSD radix sort of 64-bit keys.
// Both are memory-bound integer kernels: coalesced 16-byte accesses, warp shuffles for the
// in-block prefix, shared-memory histograms; no library (CUB/Thrust) calls.
#include <stdarg.h>

#include <atomic>

#include "common.cuh"

namespace cgx {

static thread_local char g_err[512] = "";

static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Tuning options (cgx_set_option): the only process-wide mutable state of the library besides the launch tally.
// The library reads no environment variables; the Python binding maps CGX_OPT_<NAME> onto these for experiments.
static const int64_t k_option_defaults[CGX_OPT_COUNT_] = {
    int64_t(96) << 20,  // CGX_OPT_L2_TABLE_BYTES
    1,                  // CGX_OPT_SPARSE_FIRST_ADJOINT
    1,                  // CGX_OPT_PDL
    2,                  // CGX_OPT_P2P_ONESHOT_MAX
    0,                  // CGX_OPT_P2P_TIMING
    20000,              // CGX_OPT_P2P_TIMEOUT_MS
    0,                  // CGX_OPT_EVAL_DEBUG
    1,                  // CGX_OPT_HOT_ROWS
    0,                  // CGX_OPT_EVAL_GROUPS
    0,                  // CGX_OPT_TOPK_CHUNK_USERS
};
static std::atomic<int64_t> g_options[CGX_OPT_COUNT_] = {
    {k_option_defaults[0]}, {k_option_defaults[1]}, {k_option_defaults[2]}, {k_option_defaults[3]},
    {k_option_defaults[4]}, {k_option_defaults[5]}, {k_option_defaults[6]}, {k_option_defaults[7]},
    {k_option_defaults[8]}, {k_option_defaults[9]}};
int64_t option(int which) { return g_options[which].load(std::memory_order_relaxed); }

// --------------------------------------------------------------------------------------------
// scan
// --------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint32_t warp_inclusive(uint32_t v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// exclusive prefix of one value per thread across the block; returns block total through smem
__device__ __forceinline__ uint32_t block_exclusive(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
  __shared__ uint32_t block_total;
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = warp_inclusive(v, lane);
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0u;
    uint32_t winc = warp_inclusive(w, lane);
    if (lane < SCAN_THREADS / 32) warp_sums[lane] = winc - w;
    if (lane == SCAN_THREADS / 32 - 1) block_total = winc;
  }
  __syncthreads();
  uint32_t r = inc - v + warp_sums[warp];
  *total = block_total;
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(const uint32_t* __restrict__ in, int64_t n,
                                                              uint32_t* __restrict__ sums) {
  int64_t base = int64_t(blockIdx.x) * SCAN_TILE;
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; ++j) {
    int64_t p = base + int64_t(j) * SCAN_THREADS + threadIdx.x;
    if (p < n) s += in[p];
  }
  uint32_t total;
  block_exclusive(s, &total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_down(const uint32_t* in, uint32_t* out, int64_t n,
                                                            const uint32_t* __restrict__ offsets,
                                                            uint32_t* total_out) {
  int64_t base = int64_t(blockIdx.x) * SCAN_TILE + int64_t(threadIdx.x) * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; ++j) {
    v[j] = (base + j < n) ? in[base + j] : 0u;
    s += v[j];
  }
  uint32_t total;
  uint32_t ex = block_exclusive(s, &total) + (offsets ? offsets[blockIdx.x] : 0u);
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; ++j) {
    if (base + j < n) {
      out[base + j] = ex;
      if (total_out != nullptr && base + j == n - 1) *total_out = ex + v[j];
    }
    ex += v[j];
  }
}

size_t scan_temp_bytes(int64_t n) {
  size_t total = 0;
  int64_t m = ceil_div(n > 0 ? n : 1, SCAN_TILE);
  while (true) {
    total += align_up(size_t(m) * sizeof(uint32_t));
    if (m <= 1) break;
    m = ceil_div(m, SCAN_TILE);
  }
  return total + 256;
}

int exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* total_out, void* temp,
                       size_t temp_bytes, cudaStream_t stream) {
  if (n <= 0) {
    if (total_out) CGX_CUDA(cudaMemsetAsync(total_out, 0, sizeof(uint32_t), stream));
    return CGX_OK;
  }
  CGX_REQUIRE(temp_bytes >= scan_temp_bytes(n), CGX_ERR_WORKSPACE, "scan: workspace too small");
  int64_t blocks = ceil_div(n, SCAN_TILE);
  if (blocks == 1) {
    k_scan_down<<<1, SCAN_THREADS, 0, stream>>>(in, out, n, nullptr, total_out);
    CGX_LAUNCH_CHECK();
    return CGX_OK;
  }
  uint32_t* sums = static_cast<uint32_t*>(temp);
  size_t used = align_up(size_t(blocks) * sizeof(uint32_t));
  k_scan_reduce<<<(unsigned)blocks, SCAN_THREADS, 0, stream>>>(in, n, sums);
  CGX_LAUNCH_CHECK();
  CGX_TRY(exclusive_scan_u32(sums, sums, blocks, nullptr, static_cast<char*>(temp) + used, temp_bytes - used,
                             stream));
  k_scan_down<<<(unsigned)blocks, SCAN_THREADS, 0, stream>>>(in, out, n, sums, total_out);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

// --------------------------------------------------------------------------------------------
// radix sort: 8-bit digits; per pass  histogram -> scan -> stable scatter
// --------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_STEPS = 16;                       // keys per lane
constexpr int RS_WARP_KEYS = RS_STEPS * 32;        // 512
constexpr int RS_TILE = RS_WARP_KEYS * RS_WARPS;   // 4096 keys per block
constexpr int RS_BINS = 256;

__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const uint64_t* __restrict__ keys, int64_t n, int shift,
                                                        uint32_t* __restrict__ hist, int64_t nblocks) {
  __shared__ uint32_t h[RS_BINS];
  h[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = int64_t(blockIdx.x) * RS_TILE;
#pragma unroll 4
  for (int j = 0; j < RS_TILE / RS_THREADS; ++j) {
    int64_t p = base + int64_t(j) * RS_THREADS + threadIdx.x;
    if (p < n) atomicAdd(&h[(keys[p] >> shift) & 0xff], 1u);
  }
  __syncthreads();
  hist[int64_t(threadIdx.x) * nblocks + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const uint64_t* __restrict__ in, uint64_t* __restrict__ out,
                                                           int64_t n, int shift,
                                                           const uint32_t* __restrict__ offs, int64_t nblocks) {
  __shared__ uint32_t cnt[RS_WARPS][RS_BINS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t wbase = int64_t(blockIdx.x) * RS_TILE + int64_t(warp) * RS_WARP_KEYS;
  uint64_t key[RS_STEPS];
#pragma unroll
  for (int j = 0; j < RS_STEPS; ++j) {
    int64_t p = wbase + j * 32 + lane;
    key[j] = p < n ? in[p] : 0ull;
  }
  for (int b = lane; b < RS_BINS; b += 32) cnt[warp][b] = 0;
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  // per-warp digit counts
#pragma unroll
  for (int j = 0; j < RS_STEPS; ++j) {
    bool valid = wbase + j * 32 + lane < n;
    uint32_t d = valid ? uint32_t((key[j] >> shift) & 0xff) : 256u;
    uint32_t m = __match_any_sync(0xffffffffu, d);
    if (valid && (m & lt) == 0) cnt[warp][d] += __popc(m);
    __syncwarp();
  }
  __syncthreads();
  {  // digit t: global base of this block, then exclusive prefix over the warps of this block
    uint32_t run = offs[int64_t(threadIdx.x) * nblocks + blockIdx.x];
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
      uint32_t c = cnt[w][threadIdx.x];
      cnt[w][threadIdx.x] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < RS_STEPS; ++j) {
    bool valid = wbase + j * 32 + lane < n;
    uint32_t d = valid ? uint32_t((key[j] >> shift) & 0xff) : 256u;
    uint32_t m = __match_any_sync(0xffffffffu, d);
    uint32_t pos = 0;
    if (valid) pos = cnt[warp][d] + __popc(m & lt);
    __syncwarp();
    if (valid && (m & lt) == 0) cnt[warp][d] += __popc(m);
    __syncwarp();
    if (valid) out[pos] = key[j];
  }
}

size_t radix_sort_temp_bytes(int64_t n) {
  int64_t nblocks = ceil_div(n > 0 ? n : 1, RS_TILE);
  return align_up(size_t(nblocks) * RS_BINS * sizeof(uint32_t)) + scan_temp_bytes(nblocks * RS_BINS) + 256;
}

int radix_sort_u64(uint64_t* keys, uint64_t* alt, int64_t n, int bits, void* temp, size_t temp_bytes,
                   cudaStream_t stream, uint64_t** sorted) {
  *sorted = keys;
  if (n <= 1) return CGX_OK;
  CGX_REQUIRE(n < (int64_t(1) << 32), CGX_ERR_ARG, "radix sort: more than 2^32 keys");
  CGX_REQUIRE(temp_bytes >= radix_sort_temp_bytes(n), CGX_ERR_WORKSPACE, "radix sort: workspace too small");
  int64_t nblocks = ceil_div(n, RS_TILE);
  uint32_t* hist = static_cast<uint32_t*>(temp);
  size_t used = align_up(size_t(nblocks) * RS_BINS * sizeof(uint32_t));
  char* scan_tmp = static_cast<char*>(temp) + used;
  uint64_t* src = keys;
  uint64_t* dst = alt;
  for (int shift = 0; shift < bits; shift += 8) {
    k_rs_hist<<<(unsigned)nblocks, RS_THREADS, 0, stream>>>(src, n, shift, hist, nblocks);
    CGX_LAUNCH_CHECK();
    CGX_TRY(exclusive_scan_u32(hist, hist, nblocks * RS_BINS, nullptr, scan_tmp, temp_bytes - used, stream));
    k_rs_scatter<<<(unsigned)nblocks, RS_THREADS, 0, stream>>>(src, dst, n, shift, hist, nblocks);
    CGX_LAUNCH_CHECK();
    uint64_t* t = src;
    src = dst;
    dst = t;
  }
  *sorted = src;
  return CGX_OK;
}

}  // namespace cgx

extern "C" const char* cgx_last_error(void) { return cgx::g_err; }
extern "C" int cgx_version(void) { return 200; }
extern "C" int cgx_set_option(int which, int64_t value, int64_t* previous) {
  CGX_REQUIRE(which >= 0 && which < CGX_OPT_COUNT_, CGX_ERR_ARG, "set_option: unknown option %d", which);
  if (value < 0) value = cgx::k_option_defaults[which];   // negative = restore the default
  const int64_t old = cgx::g_options[which].exchange(value, std::memory_order_relaxed);
  if (previous) *previous = old;
  return CGX_OK;
}
extern "C" int64_t cgx_get_option(int which) {
  return which >= 0 && which < CGX_OPT_COUNT_ ? cgx::option(which) : -1;
}
extern "C" uint64_t cgx_launch_count(void) { return cgx::g_launches.load(std::memory_order_relaxed); }
extern "C" int cgx_emb_dim_supported(int32_t d) {
  return d == 16 || d == 32 || d == 64 || d == 128 || d == 256;
}
