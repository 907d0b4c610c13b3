// CSR SpMM with a fused layer-mean / gradient-seed epilogue, and the K-layer propagation
// schedules (forward and adjoint) built on it.
//
// Replaces (reference, /root/reference): torch.sparse.mm at lightgcn_cu.py:431,434 and
// Version-2/lighgcn_cu_pop.py:483-484, the stack().mean() at lightgcn_cu.py:446-447 /
// lighgcn_cu_pop.py:488-489, and autograd's SparseAddmmBackward for the same calls.
//
// Kernel shape: the path is an HBM/L2-bound gather.  A group of G lanes owns one work item and keeps V float4 of the
// output row per lane (G V = d/4).  Two regimes (cgx_spmm switches on the size of the gathered table,
// CGX_OPT_L2_TABLE_BYTES):
//   * table inside L2 (C2, C3; latency-bound): G = d/4 lanes, one float4 each, 8 gathers in flight per lane;
//   * table beyond L2 (C4, C5; HBM-bound): G = d/8 lanes, 32 contiguous bytes each -- ONE 256-bit access per lane and
//     row (LDG.E.256 / STG.E.256, new on sm_100) -- 4 gathers in flight, and, when the graph carries hot-row hints
//     (cgx_hot_hints: bit 31 of a second column-id array marks the columns of the highest-degree rows), per-row L2
//     eviction priorities: hot rows are loaded evict_last and stay resident, everything else (cold rows, the running
//     sums, both outputs) goes through evict_first and does not displace them.
// Column ids / values are fetched coalesced G at a time (the next batch is prefetched while the current one is
// consumed) and broadcast by shuffle; the gathers of a batch are issued before any FMA.
// Work items follow the schedule built by cgx_row_schedule: first the CGX_CHUNK-sized chunks of the rows longer than
// CGX_LONG_ROW (partials in workspace, summed IN CHUNK ORDER by the chunk that arrives last, or by a finishing kernel
// for rows above CGX_HUGE_ROW), then all other rows in descending degree order; every item is ONE 16-byte descriptor.
// Neighbouring groups therefore carry equal work and the heavy items start first (no tail).
// No floating-point atomics anywhere (the only atomic is an integer arrival counter): results are bitwise
// reproducible, and both regimes / all flag combinations add the same terms in the same order (same bits).
// Measured history of the kernel: DESIGN.md section 4.1 (profiles/r1_spmm_variants.txt, profiles/r2_ncu_spmm_c4.txt).
#include "common.cuh"

namespace cgx {

constexpr int SP_THREADS = 256;

__device__ __forceinline__ void fma4(float4& a, float v, const float4& x) {
  a.x = fmaf(v, x.x, a.x);
  a.y = fmaf(v, x.y, a.y);
  a.z = fmaf(v, x.z, a.z);
  a.w = fmaf(v, x.w, a.w);
}
__device__ __forceinline__ float4 add4(const float4& a, const float4& b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 scale4(const float4& a, float s) {
  return make_float4(a.x * s, a.y * s, a.z * s, a.w * s);
}

// 256-bit global accesses with an L2 eviction priority (sm_100: LDG.E.{EF,EL,EN}L2.256 / STG.E.*.256).  The priority
// is how "hot (high-degree) rows are staged" when the gathered table is larger than the 126 MB L2: rows named hot by
// cgx_hot_hints are loaded evict_last and stay resident, everything else -- cold rows, the streamed column ids /
// values, the epilogue's running sums and outputs -- goes through evict_first and does not displace them.
enum { POL_NORMAL = 0, POL_FIRST = 1, POL_LAST = 2 };
template <int POL>
__device__ __forceinline__ void ld256(const float4* p, float4& a, float4& b) {
  if (POL == POL_LAST) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_last.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
  } else if (POL == POL_FIRST) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
  } else {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
  }
}
// plain (coherent) 256-bit load: ACC_IN may alias ACC_OUT, which this kernel writes -- never through the .nc path
template <int POL>
__device__ __forceinline__ void ld256_rw(const float4* p, float4& a, float4& b) {
  if (POL == POL_FIRST) {
    asm volatile("ld.global.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p)
                 : "memory");
  } else {
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p)
                 : "memory");
  }
}
template <int POL>
__device__ __forceinline__ void st256(float4* p, const float4& a, const float4& b) {
  if (POL == POL_FIRST) {
    asm volatile("st.global.L2::evict_first.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a.x), "f"(a.y),
                 "f"(a.z), "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w)
                 : "memory");
  } else {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w),
                 "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w)
                 : "memory");
  }
}
template <bool STREAM>
__device__ __forceinline__ int32_t ld_idx(const int32_t* p) {
  if (!STREAM) return __ldg(p);
  int32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(v) : "l"(p));   // (L2 priorities need 256-bit accesses)
  return v;
}
template <bool STREAM>
__device__ __forceinline__ float ld_val(const float* p) {
  if (!STREAM) return __ldg(p);
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

template <int G>
__device__ __forceinline__ unsigned group_mask() {
  if (G == 32) return 0xffffffffu;
  const unsigned lane = threadIdx.x & 31;
  return ((1u << (G & 31)) - 1u) << (lane & ~(G - 1));
}

// Lane `lane` of a group owns float4 slots lane*V .. lane*V+V-1 of a row (V = 2: 32 contiguous bytes, one 256-bit
// access; V = 1: 16 bytes).  x[v] = X[row c][lane*V + v].
template <int G, int V, bool HOT>
__device__ __forceinline__ void ld_row(const float4* __restrict__ X, int32_t c, int lane, float4 (&x)[V]) {
  constexpr int ROW4 = G * V;
  if constexpr (V == 2) {
    if constexpr (HOT) {   // bit 31 of a hinted column id = "hot row"
      const float4* p = X + int64_t(c & 0x7fffffff) * ROW4 + 2 * lane;
      if (c < 0) ld256<POL_LAST>(p, x[0], x[1]);
      else ld256<POL_FIRST>(p, x[0], x[1]);
    } else {
      ld256<POL_NORMAL>(X + int64_t(c) * ROW4 + 2 * lane, x[0], x[1]);
    }
  } else {
#pragma unroll
    for (int v = 0; v < V; ++v) x[v] = __ldg(X + int64_t(c) * ROW4 + lane * V + v);
  }
}

// acc[v] (v < V) += sum over nnz in [begin, end) of val * X[idx, :]; one group, lane = 0..G-1.
// NZ: `nz[c] == 0` marks row c of X as all-zero (the loss gradient touches <= 3 * batch rows): its weight is
// forced to 0 and rows of weight 0 are not loaded -- same sum, a fraction of the gather traffic.
// HOT: idx carries the hot-row hint in bit 31 (cgx_hot_hints) and the streams use evict_first.
template <int G, int V, int UNR, bool NZ, bool HOT>
__device__ __forceinline__ void gather_batches(const int32_t* __restrict__ idx, const float* __restrict__ val,
                                               int32_t len, const float4* __restrict__ X, int lane,
                                               unsigned mask, int32_t c_nxt, float w_nxt, float4 (&acc)[V],
                                               const uint8_t* __restrict__ nz) {
  // idx / val point at the work item's first non-zero; len <= CGX_CHUNK, so 32-bit offsets do.
  // (c_nxt, w_nxt) = this lane's column id / value of the first batch, already loaded by the caller
  idx += G + lane;   // this lane's slot of the NEXT batch
  val += G + lane;
  for (int32_t rem = len; rem > 0; rem -= G, idx += G, val += G) {
    const int32_t c = c_nxt;
    float w = w_nxt;
    if (NZ) {
      if (w != 0.f && __ldg(nz + c) == 0) w = 0.f;
    }
    if (G + lane < rem) {                // prefetch the next batch of column ids / values
      c_nxt = ld_idx<HOT>(idx);
      w_nxt = ld_val<HOT>(val);
    }
    const int cnt = rem < G ? rem : G;
    for (int j0 = 0; j0 < cnt; j0 += UNR) {
      float4 x[UNR][V];
      float ww[UNR];
#pragma unroll
      for (int t = 0; t < UNR; ++t) {
        const int j = j0 + t;
        const int src = (j < G) ? j : (G - 1);
        const int32_t cj = __shfl_sync(mask, c, src, G);
        ww[t] = __shfl_sync(mask, w, src, G);
        if (j < cnt && (!NZ || ww[t] != 0.f)) {
          ld_row<G, V, HOT>(X, cj, lane, x[t]);
        } else {
          ww[t] = 0.f;
#pragma unroll
          for (int v = 0; v < V; ++v) x[t][v] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int t = 0; t < UNR; ++t) {
#pragma unroll
        for (int v = 0; v < V; ++v) fma4(acc[v], ww[t], x[t][v]);
      }
    }
  }
}

// Push mode of the user-sharded propagation (cgx_spmm_push): output row r is not stored to Y but straight into the
// staging area of the rank that OWNS row r (rows_per consecutive rows per rank), slot `rank` -- a posted store over
// NVLink, issued row by row while the rest of the product is still being gathered.  The exchange kernel
// (comm.cu, pushed form) then sums the slots with local reads only.
__constant__ char* c_push_base[16];        // peer-mapped communication buffers, index = rank (cgx_spmm_set_push_peers)
struct SpmmPush {
  unsigned long long off;                  // byte offset of the staging area inside every communication buffer
  int32_t rows_per;                        // rows owned by each rank; 0 = push mode off
  int32_t rank;
};

// acc_nz (nullable): acc_nz[row] == 0 promises that ACC_IN[row] is all zero, and it is then not read (the adjoint's
// ACC_IN is the loss gradient: <= 3 * batch non-zero rows of millions).
template <int G, int V, bool STREAM>
__device__ __forceinline__ void epilogue(int64_t row, int lane, const float4 (&y)[V], float4* __restrict__ Y,
                                         const float4* ACC_IN, float4* ACC_OUT, float acc_scale,
                                         const uint8_t* __restrict__ acc_nz, const SpmmPush ps) {
  constexpr int ROW4 = G * V;
  constexpr int POL = STREAM ? POL_FIRST : POL_NORMAL;
  const int64_t o = row * ROW4 + lane * V;
  float4 a[V];
#pragma unroll
  for (int v = 0; v < V; ++v) a[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ACC_OUT != nullptr && ACC_IN != nullptr && (acc_nz == nullptr || __ldg(acc_nz + row) != 0)) {
    if constexpr (V == 2) ld256_rw<POL>(ACC_IN + o, a[0], a[1]);
    else {
#pragma unroll
      for (int v = 0; v < V; ++v) a[v] = ACC_IN[o + v];
    }
  }
  if (ps.rows_per > 0) {
    const int owner = int(row / ps.rows_per);
    float4* ypush = reinterpret_cast<float4*>(c_push_base[owner] + ps.off) +
                    (int64_t(ps.rank) * ps.rows_per + (row - int64_t(owner) * ps.rows_per)) * ROW4 + lane * V;
    // one 32-byte store per lane: the G lanes of the instruction write the row's 32 G contiguous bytes as whole
    // sectors (two strided 16-byte stores per lane leave every sector half-written per instruction, and NVLink
    // carries partial-sector writes at a fraction of its rate)
    if constexpr (V == 2) st256<POL_NORMAL>(ypush, y[0], y[1]);
    else {
#pragma unroll
      for (int v = 0; v < V; ++v) ypush[v] = y[v];
    }
  }
  if (Y != nullptr) {
    if constexpr (V == 2) st256<POL>(Y + o, y[0], y[1]);
    else {
#pragma unroll
      for (int v = 0; v < V; ++v) Y[o + v] = y[v];
    }
  }
  if (ACC_OUT != nullptr) {
#pragma unroll
    for (int v = 0; v < V; ++v) a[v] = scale4(add4(a[v], y[v]), acc_scale);
    if constexpr (V == 2) st256<POL>(ACC_OUT + o, a[0], a[1]);
    else {
#pragma unroll
      for (int v = 0; v < V; ++v) ACC_OUT[o + v] = a[v];
    }
  }
}

struct SpmmSched {
  const int32_t* perm;
  const int32_t* chunk_ptr;
  int32_t* arrive;
  int32_t n_chunks, n_huge;
};

// One group per work item of the flattened schedule (cgx_row_schedule_work): ONE 16-byte descriptor
// {begin, length, row | long-row index} per item -- chunk items first, then rows in descending degree.  A chunk
// stores its partial sum; for rows up to CGX_HUGE_ROW the chunk that arrives last (per-row counter, release /
// acquire through __threadfence) adds the partials IN CHUNK ORDER and runs the epilogue, so the result does not
// depend on which chunk happened to be last.
template <int G, int V, int UNR, int MINB, bool NZ, bool PUSH, bool HOT>
__global__ void __launch_bounds__(SP_THREADS, MINB) k_spmm(const int32_t* __restrict__ idx,
                                                           const float* __restrict__ val, int64_t n_items,
                                                           SpmmSched sc, const float4* __restrict__ X,
                                                           float4* __restrict__ Y, const float4* ACC_IN,
                                                           float4* ACC_OUT, float acc_scale, float4* partial,
                                                           const uint8_t* __restrict__ nz,
                                                           const uint8_t* __restrict__ acc_nz,
                                                           const uint8_t* __restrict__ out_rows,
                                                           const int4* __restrict__ work, const SpmmPush ps_in) {
  // PUSH = false: a compile-time "off", so that the ordinary instantiations carry no trace of the push path
  const SpmmPush ps = PUSH ? ps_in : SpmmPush{0ull, 0, 0};
  constexpr int ROW4 = G * V;
  // Programmatic dependent launch: let the next kernel of the stream start its own prologue now, and run
  // THIS kernel's prologue (descriptor, first batch of column ids / values -- graph constants) while the
  // previous kernel is still draining.  Nothing the previous kernel wrote is read, and nothing is written,
  // before griddepcontrol.wait returns.
  asm volatile("griddepcontrol.launch_dependents;");
  const int lane = threadIdx.x & (G - 1);
  const uint32_t item = (blockIdx.x * uint32_t(SP_THREADS) + threadIdx.x) / G;   // < 2^32 / G items
  const unsigned mask = group_mask<G>();
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (item >= n_items) return;
  const int4 wd = __ldg(work + item);
  const int64_t begin = (int64_t(wd.y) << 32) | uint32_t(wd.x);
  idx += begin;
  val += begin;
  int32_t cf = 0;
  float wf = 0.f;
  if (lane < wd.z) {
    cf = ld_idx<HOT>(idx + lane);
    wf = ld_val<HOT>(val + lane);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // out_rows (nullable; written by an earlier kernel, so read after the wait): a row with out_rows[row] == 0 is not
  // computed and none of its outputs is written.  Every chunk of a long row reads the same flag, so either all of
  // them arrive or none does, and the arrival counter stays 0 between launches.  Only the row-sparse (NZ) products
  // take a mask (spmm_dispatch): in the other instantiations the check would cost registers at the 64-register cap
  // (-Xptxas -v: spills in the d = 64 and d = 128 gather loops).
  if (NZ && !PUSH && out_rows != nullptr &&
      __ldg(out_rows + (item >= sc.n_chunks ? wd.w : __ldg(sc.perm + wd.w))) == 0)
    return;
  gather_batches<G, V, UNR, NZ, HOT>(idx, val, wd.z, X, lane, mask, cf, wf, acc, nz);
  if (item >= sc.n_chunks) {
    // (loading ACC_IN[row] before the gathers, to take it off the dependency chain, was measured SLOWER: the
    // four extra live registers spill at the 64-register cap -- C2 0.514 -> 0.553 ms, C4 155 -> 160 ms)
    epilogue<G, V, HOT>(wd.w, lane, acc, Y, ACC_IN, ACC_OUT, acc_scale, acc_nz, ps);
    return;
  }
  const int32_t k = wd.w;
#pragma unroll
  for (int v = 0; v < V; ++v) __stcg(partial + int64_t(item) * ROW4 + lane * V + v, acc[v]);
  if (k < sc.n_huge) return;            // combined by k_spmm_finish
  const int32_t c0 = __ldg(sc.chunk_ptr + k), c1 = __ldg(sc.chunk_ptr + k + 1);
  __threadfence();                       // release: this group's partial is visible device-wide
  __syncwarp(mask);
  int prev = 0;
  if (lane == 0) prev = atomicAdd(sc.arrive + k, 1);
  prev = __shfl_sync(mask, prev, 0, G);
  if (prev != c1 - c0 - 1) return;
  __threadfence();                       // acquire: every other chunk's partial is visible
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int c = c0; c < c1; ++c) {
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = add4(acc[v], __ldcg(partial + int64_t(c) * ROW4 + lane * V + v));
  }
  epilogue<G, V, HOT>(int64_t(__ldg(sc.perm + k)), lane, acc, Y, ACC_IN, ACC_OUT, acc_scale, acc_nz, ps);
  if (lane == 0) sc.arrive[k] = 0;       // self-resetting for the next launch
}

// one CTA per huge row: groups sum interleaved chunk partials, fixed-order reduction, epilogue
template <int G, int V>
__global__ void __launch_bounds__(SP_THREADS) k_spmm_finish(SpmmSched sc, const float4* __restrict__ partial,
                                                            float4* __restrict__ Y, const float4* ACC_IN,
                                                            float4* ACC_OUT, float acc_scale,
                                                            const uint8_t* __restrict__ acc_nz,
                                                            const uint8_t* __restrict__ out_rows, const SpmmPush ps) {
  constexpr int GROUPS = SP_THREADS / G;
  constexpr int ROW4 = G * V;
  __shared__ float4 red[GROUPS][ROW4];
  const int k = blockIdx.x;
  if (out_rows != nullptr && __ldg(out_rows + __ldg(sc.perm + k)) == 0) return;   // the whole CTA: row not computed
  const int lane = threadIdx.x & (G - 1), grp = threadIdx.x / G;
  const int c0 = __ldg(sc.chunk_ptr + k), c1 = __ldg(sc.chunk_ptr + k + 1);
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int c = c0 + grp; c < c1; c += GROUPS) {
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = add4(acc[v], __ldg(partial + int64_t(c) * ROW4 + lane * V + v));
  }
#pragma unroll
  for (int v = 0; v < V; ++v) red[grp][lane * V + v] = acc[v];
  __syncthreads();
  if (grp == 0) {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float4 s = red[0][lane * V + v];
      for (int g = 1; g < GROUPS; ++g) s = add4(s, red[g][lane * V + v]);
      acc[v] = s;
    }
    epilogue<G, V, false>(int64_t(__ldg(sc.perm + k)), lane, acc, Y, ACC_IN, ACC_OUT, acc_scale, acc_nz, ps);
  }
}

__global__ void k_scale(const float4* __restrict__ in, float4* __restrict__ out, int64_t n4, float s) {
  int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p < n4) out[p] = scale4(in[p], s);
}

// flags[r] = 1 when row r of X (row4 float4 per row) has a non-zero entry (-0 counts as zero); flags pre-zeroed
__global__ void k_row_flags(const uint4* __restrict__ X, int64_t n4, int32_t row4, uint8_t* __restrict__ flags) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= n4) return;
  const uint4 v = X[p];
  if ((v.x | v.y | v.z | v.w) & 0x7fffffffu) flags[p / row4] = 1;
}

static int row_flags(const float* X, int64_t n_rows, int32_t d, uint8_t* flags, cudaStream_t stream) {
  CGX_CUDA(cudaMemsetAsync(flags, 0, size_t(n_rows), stream));
  const int64_t n4 = n_rows * d / 4;
  if (n4 == 0) return CGX_OK;
  k_row_flags<<<(unsigned)ceil_div(n4, 256), 256, 0, stream>>>(reinterpret_cast<const uint4*>(X), n4, d / 4, flags);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

template <int G, int V, int UNR, int MINB, bool NZ, bool PUSH, bool HOT>
static int launch_spmm(const cgx_csr* m, const float* val, const float* X, float* Y, const float* ACC_IN,
                       float* ACC_OUT, float acc_scale, void* workspace, size_t workspace_bytes,
                       cudaStream_t stream, const uint8_t* nz, const uint8_t* acc_nz, const uint8_t* out_rows,
                       const SpmmPush ps) {
  constexpr int GROUPS = SP_THREADS / G;
  float4* partial = nullptr;
  if (m->n_long > 0) {
    size_t need = size_t(m->n_chunks) * G * V * sizeof(float4);
    CGX_REQUIRE(workspace != nullptr && workspace_bytes >= need, CGX_ERR_WORKSPACE,
                "spmm: workspace too small for %d long-row chunks", m->n_chunks);
    partial = static_cast<float4*>(workspace);
  }
  SpmmSched sc{m->perm, m->chunk_ptr, m->arrive, m->n_chunks, m->n_huge};
  const int64_t items = int64_t(m->n_chunks) + (m->n_rows - m->n_long);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ceil_div(items, GROUPS));
  cfg.blockDim = dim3(SP_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = option(CGX_OPT_PDL) != 0 ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CGX_CUDA(cudaLaunchKernelEx(&cfg, k_spmm<G, V, UNR, MINB, NZ, PUSH, HOT>, HOT ? m->idx_hint : m->idx, val, items, sc,
                              reinterpret_cast<const float4*>(X), reinterpret_cast<float4*>(Y),
                              reinterpret_cast<const float4*>(ACC_IN), reinterpret_cast<float4*>(ACC_OUT), acc_scale,
                              partial, nz, acc_nz, out_rows, static_cast<const int4*>(m->work), ps));
  CGX_LAUNCH_CHECK();
  if (m->n_huge > 0) {
    k_spmm_finish<G, V><<<(unsigned)m->n_huge, SP_THREADS, 0, stream>>>(
        sc, partial, reinterpret_cast<float4*>(Y), reinterpret_cast<const float4*>(ACC_IN),
        reinterpret_cast<float4*>(ACC_OUT), acc_scale, acc_nz, out_rows, ps);
    CGX_LAUNCH_CHECK();
  }
  return CGX_OK;
}

#define CGX_SPMM_ARGS m, val, X, Y, ACC_IN, ACC_OUT, acc_scale, ws, ws_bytes, stream, nz, acc_nz, out_rows, ps

// Group geometry by regime (profiles/r1_spmm_variants.txt; the sweep itself lives in the round-1 history).
// Gathered table in L2 (C2/C3: latency-bound): d/4 lanes per row, one float4 per lane, 8 gathers in flight.
// Gathered table beyond L2 (HBM-bound): d/8 lanes per row, 32 contiguous bytes (one 256-bit access) per lane, four
// gathers in flight -- twice the rows in flight per SM at the same bytes in flight per lane (d = 64: 27.3 vs 30.1 ms,
// d = 128: 53.8 vs 58.6 ms on the 64M-edge shape; on C2 the same split LOSES, 0.65 vs 0.43 ms at d = 64) -- and,
// when the graph carries hot-row hints (cgx_hot_hints), per-row L2 eviction priorities.
template <int G, int V, int UNR>
static int spmm_flavour(const cgx_csr* m, const float* val, const float* X, float* Y, const float* ACC_IN,
                        float* ACC_OUT, float acc_scale, void* ws, size_t ws_bytes, cudaStream_t stream,
                        const uint8_t* nz, const uint8_t* acc_nz, const uint8_t* out_rows, const SpmmPush ps,
                        bool hot) {
  const bool push = ps.rows_per > 0;
  if constexpr (V == 2) {
    if (hot && nz == nullptr) {
      if (push) return launch_spmm<G, V, UNR, 4, false, true, true>(CGX_SPMM_ARGS);
      return launch_spmm<G, V, UNR, 4, false, false, true>(CGX_SPMM_ARGS);
    }
  }
  if (push) {
    if (nz) return launch_spmm<G, V, UNR, 4, true, true, false>(CGX_SPMM_ARGS);
    return launch_spmm<G, V, UNR, 4, false, true, false>(CGX_SPMM_ARGS);
  }
  if (nz) return launch_spmm<G, V, UNR, 4, true, false, false>(CGX_SPMM_ARGS);
  return launch_spmm<G, V, UNR, 4, false, false, false>(CGX_SPMM_ARGS);
}

#define CGX_FLAVOUR_ARGS m, val, X, Y, ACC_IN, ACC_OUT, acc_scale, ws, ws_bytes, stream, nz, acc_nz, out_rows, ps, hot

static int spmm_dispatch(const cgx_csr* m, int use_bwd, int32_t d, const float* X, float* Y, const float* ACC_IN,
                         float* ACC_OUT, float acc_scale, void* ws, size_t ws_bytes, cudaStream_t stream,
                         const uint8_t* nz = nullptr, const SpmmPush ps = SpmmPush{0ull, 0, 0},
                         const uint8_t* acc_nz = nullptr, const uint8_t* out_rows = nullptr) {
  CGX_REQUIRE(m && m->perm && m->work && (m->nnz == 0 || (m->idx && m->val_fwd && m->val_bwd)) && X, CGX_ERR_ARG,
              "spmm: NULL pointer (cgx_csr needs idx, both value arrays and the cgx_row_schedule* outputs)");
  CGX_REQUIRE(m->n_long == 0 || (m->chunk_ptr && m->arrive), CGX_ERR_ARG, "spmm: chunk tables missing");
  CGX_REQUIRE(Y || ACC_OUT || ps.rows_per > 0, CGX_ERR_ARG, "spmm: no output requested");
  CGX_REQUIRE(out_rows == nullptr || (nz != nullptr && ps.rows_per == 0), CGX_ERR_ARG,
              "spmm: an output-row mask needs gather flags and no push mode");
  const float* val = use_bwd ? m->val_bwd : m->val_fwd;
  if (m->n_rows == 0) return CGX_OK;
  const bool beyond_l2 = int64_t(m->n_cols) * int64_t(d) * 4 > option(CGX_OPT_L2_TABLE_BYTES);
  const bool hot = beyond_l2 && m->idx_hint != nullptr && option(CGX_OPT_HOT_ROWS) != 0;
  switch (d) {
    case 16: return spmm_flavour<4, 1, 4>(CGX_FLAVOUR_ARGS);
    case 32: return spmm_flavour<8, 1, 8>(CGX_FLAVOUR_ARGS);
    case 64:
      if (beyond_l2) return spmm_flavour<8, 2, 4>(CGX_FLAVOUR_ARGS);
      return spmm_flavour<16, 1, 8>(CGX_FLAVOUR_ARGS);
    case 128:
      if (beyond_l2) return spmm_flavour<16, 2, 4>(CGX_FLAVOUR_ARGS);
      return spmm_flavour<32, 1, 8>(CGX_FLAVOUR_ARGS);
    case 256: return spmm_flavour<32, 2, 4>(CGX_FLAVOUR_ARGS);
    default:
      set_error("spmm: emb_dim %d unsupported (16, 32, 64, 128, 256)", d);
      return CGX_ERR_UNSUPPORTED;
  }
}

// hot[c] = 1 for the first n_hot entries of col_by_degree (the OTHER row order's perm: columns in descending degree)
__global__ void k_hot_flags(const int32_t* __restrict__ col_by_degree, int32_t n_hot, uint8_t* __restrict__ hot) {
  const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n_hot) hot[__ldg(col_by_degree + k)] = 1;
}
__global__ void k_hot_hint(const int32_t* __restrict__ idx, int64_t nnz, const uint8_t* __restrict__ hot,
                           int32_t* __restrict__ out) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  const int32_t c = idx[p];
  out[p] = __ldg(hot + c) ? (c | int32_t(0x80000000u)) : c;
}

static size_t spmm_ws(const cgx_csr* m, int32_t d) { return align_up(size_t(m ? m->n_chunks : 0) * d * 4); }

}  // namespace cgx

using namespace cgx;

extern "C" size_t cgx_spmm_workspace_bytes(const cgx_csr* m, int32_t d) { return spmm_ws(m, d); }

extern "C" int cgx_spmm(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X, float* Y,
                        const float* ACC_IN, float* ACC_OUT, float acc_scale, void* workspace,
                        size_t workspace_bytes, void* stream) {
  return spmm_dispatch(m, use_bwd_values, d, X, Y, ACC_IN, ACC_OUT, acc_scale, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int cgx_spmm_sparse_rows(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X,
                                    const uint8_t* x_row_nonzero, float* Y, const float* ACC_IN, float* ACC_OUT,
                                    float acc_scale, void* workspace, size_t workspace_bytes, void* stream) {
  CGX_REQUIRE(x_row_nonzero != nullptr, CGX_ERR_ARG, "spmm_sparse_rows: NULL flags");
  return spmm_dispatch(m, use_bwd_values, d, X, Y, ACC_IN, ACC_OUT, acc_scale, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream), x_row_nonzero);
}

extern "C" int cgx_spmm_ex(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X, const uint8_t* x_row_nonzero,
                           float* Y, const float* ACC_IN, const uint8_t* acc_row_nonzero, float* ACC_OUT,
                           float acc_scale, void* workspace, size_t workspace_bytes, void* stream) {
  return spmm_dispatch(m, use_bwd_values, d, X, Y, ACC_IN, ACC_OUT, acc_scale, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream), x_row_nonzero, SpmmPush{0ull, 0, 0}, acc_row_nonzero);
}

extern "C" int64_t cgx_spmm_set_l2_table_bytes(int64_t bytes) {
  int64_t old = 0;
  cgx_set_option(CGX_OPT_L2_TABLE_BYTES, bytes, &old);
  return old;
}

extern "C" size_t cgx_hot_hints_workspace_bytes(int32_t n_cols) { return align_up(size_t(n_cols > 0 ? n_cols : 0)) + 256; }

extern "C" int cgx_hot_hints(const int32_t* idx, int64_t nnz, int32_t n_cols, const int32_t* col_by_degree,
                             int32_t n_hot, int32_t* idx_hint, void* workspace, size_t workspace_bytes,
                             void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(nnz >= 0 && n_cols > 0 && col_by_degree && idx_hint && (nnz == 0 || idx) && n_hot >= 0 &&
                  n_hot <= n_cols,
              CGX_ERR_ARG, "hot_hints: bad argument");
  CGX_REQUIRE(workspace != nullptr && workspace_bytes >= cgx_hot_hints_workspace_bytes(n_cols), CGX_ERR_WORKSPACE,
              "hot_hints: workspace too small");
  uint8_t* hot = static_cast<uint8_t*>(workspace);
  CGX_CUDA(cudaMemsetAsync(hot, 0, size_t(n_cols), stream));
  if (n_hot > 0) {
    k_hot_flags<<<(unsigned)ceil_div(n_hot, 256), 256, 0, stream>>>(col_by_degree, n_hot, hot);
    CGX_LAUNCH_CHECK();
  }
  if (nnz > 0) {
    k_hot_hint<<<(unsigned)ceil_div(nnz, 256), 256, 0, stream>>>(idx, nnz, hot, idx_hint);
    CGX_LAUNCH_CHECK();
  }
  return CGX_OK;
}

extern "C" int cgx_spmm_set_push_peers(void* const* peer_bases, int world) {
  CGX_REQUIRE(peer_bases != nullptr && world >= 1 && world <= 16, CGX_ERR_ARG, "spmm_set_push_peers: bad argument");
  char* h[16] = {nullptr};
  for (int p = 0; p < world; ++p) h[p] = static_cast<char*>(peer_bases[p]);
  CGX_CUDA(cudaMemcpyToSymbol(c_push_base, h, sizeof(h)));
  return CGX_OK;
}

extern "C" int cgx_spmm_push(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X,
                             const uint8_t* x_row_nonzero, size_t stage_off, int rank, int world, int32_t rows_per,
                             void* workspace, size_t workspace_bytes, void* stream) {
  CGX_REQUIRE(m != nullptr && world >= 1 && world <= 16 && rank >= 0 && rank < world && rows_per > 0 &&
                  int64_t(rows_per) * world >= m->n_rows && stage_off % 16 == 0,
              CGX_ERR_ARG, "spmm_push: bad rank / world / rows_per");
  const SpmmPush ps{(unsigned long long)stage_off, rows_per, rank};
  return spmm_dispatch(m, use_bwd_values, d, X, nullptr, nullptr, nullptr, 1.0f, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream), x_row_nonzero, ps);
}

extern "C" int cgx_row_flags(const float* X, int64_t n_rows, int32_t d, uint8_t* flags, void* stream) {
  CGX_REQUIRE(X && flags && n_rows >= 0 && d > 0 && d % 4 == 0, CGX_ERR_ARG, "row_flags: bad argument");
  return row_flags(X, n_rows, d, flags, static_cast<cudaStream_t>(stream));
}

// Item frontier of a triple batch: flags[i] = 1 for i in pos, neg and the by_user rows of the batch users, and
// (flags_u nullable) flags_u[u] = 1 for the batch users.  One warp per triple; duplicate users walk their row twice
// (the stores are idempotent).  Out-of-range ids are clamped to 0, as cgx_bpr_plan does, so the frontier covers every
// row that cgx_bpr_mark_rows flags.
__device__ __forceinline__ int64_t clamp_row(int64_t x, int64_t n) { return (x < 0 || x >= n) ? 0 : x; }
__global__ void k_batch_frontier(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx,
                                 const int64_t* __restrict__ users, const int64_t* __restrict__ pos,
                                 const int64_t* __restrict__ neg, int64_t B, int32_t U, int32_t I,
                                 uint8_t* __restrict__ flags, uint8_t* __restrict__ flags_u) {
  const int64_t t = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x & 31;
  if (t >= B) return;
  const int64_t u = clamp_row(users[t], U);
  if (lane == 0) {
    flags[clamp_row(pos[t], I)] = 1;
    flags[clamp_row(neg[t], I)] = 1;
    if (flags_u != nullptr) flags_u[u] = 1;
  }
  const int64_t end = indptr[u + 1];
  for (int64_t j = indptr[u] + lane; j < end; j += 32) flags[idx[j]] = 1;
}

extern "C" int cgx_batch_frontier(const cgx_csr* by_user, const int64_t* users, const int64_t* pos,
                                  const int64_t* neg, int64_t B, uint8_t* flags_i, uint8_t* flags_u,
                                  void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(by_user && by_user->indptr && (by_user->nnz == 0 || by_user->idx) && users && pos && neg && flags_i,
              CGX_ERR_ARG, "batch_frontier: NULL pointer");
  CGX_REQUIRE(B > 0 && B < (int64_t(1) << 29) && by_user->n_rows > 0 && by_user->n_cols > 0, CGX_ERR_ARG,
              "batch_frontier: bad batch size %lld or empty graph", (long long)B);
  CGX_CUDA(cudaMemsetAsync(flags_i, 0, size_t(by_user->n_cols), stream));
  if (flags_u != nullptr) CGX_CUDA(cudaMemsetAsync(flags_u, 0, size_t(by_user->n_rows), stream));
  k_batch_frontier<<<(unsigned)ceil_div(B * 32, 256), 256, 0, stream>>>(
      by_user->indptr, by_user->idx, users, pos, neg, B, by_user->n_rows, by_user->n_cols, flags_i, flags_u);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

// Layer buffers: the Jacobi order reads layer k of BOTH sides while it writes layer k + 1, so it needs two buffers
// per side; in Gauss-Seidel order every buffer is dead by the time it is overwritten (the item product reads u_k
// and writes i_{k+1}, the user product reads i_{k+1} and writes u_{k+1}), so one per side is enough -- 15 GB less
// at the C5 shape.
static size_t propagate_ws(const cgx_csr* by_user, const cgx_csr* by_item, int32_t d, int n_buf) {
  if (!by_user || !by_item) return 0;
  size_t long_ws = spmm_ws(by_user, d) > spmm_ws(by_item, d) ? spmm_ws(by_user, d) : spmm_ws(by_item, d);
  return n_buf * (align_up(size_t(by_user->n_rows) * d * 4) + align_up(size_t(by_item->n_rows) * d * 4)) + long_ws +
         align_up(size_t(by_user->n_rows)) + align_up(size_t(by_item->n_rows)) + 256;
}

extern "C" size_t cgx_propagate_workspace_bytes(const cgx_csr* by_user, const cgx_csr* by_item, int32_t d) {
  return propagate_ws(by_user, by_item, d, 2);
}

extern "C" size_t cgx_propagate_workspace_bytes_for(const cgx_csr* by_user, const cgx_csr* by_item, int32_t d,
                                                    int order) {
  return propagate_ws(by_user, by_item, d, order == CGX_ORDER_GS ? 1 : 2);
}

extern "C" int cgx_propagate_fwd(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t K, int32_t d,
                                 const float* e0_u, const float* e0_i, float* out_u, float* out_i,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  return cgx_propagate_fwd_layers(by_user, by_item, order, K, d, e0_u, e0_i, out_u, out_i, 0, K, nullptr, nullptr,
                                  nullptr, workspace, workspace_bytes, stream);
}

extern "C" int cgx_propagate_fwd_layers(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t K,
                                        int32_t d, const float* e0_u, const float* e0_i, float* out_u, float* out_i,
                                        int32_t layer_begin, int32_t layer_end, const uint8_t* rows_u,
                                        const uint8_t* rows_i, const uint8_t* all_rows, void* workspace,
                                        size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE(by_user && by_item && e0_u && e0_i && out_u && out_i, CGX_ERR_ARG, "propagate_fwd: NULL pointer");
  CGX_REQUIRE(K >= 1, CGX_ERR_ARG, "propagate_fwd: num_layers must be >= 1");
  CGX_REQUIRE(0 <= layer_begin && layer_begin <= layer_end && layer_end <= K, CGX_ERR_ARG,
              "propagate_fwd: layers [%d, %d) outside [0, %d)", layer_begin, layer_end, K);
  CGX_REQUIRE((rows_u == nullptr && rows_i == nullptr) || all_rows != nullptr, CGX_ERR_ARG,
              "propagate_fwd: output-row masks need all_rows");
  CGX_REQUIRE(order == CGX_ORDER_JACOBI || order == CGX_ORDER_GS, CGX_ERR_ARG, "propagate_fwd: bad order");
  CGX_REQUIRE(by_user->n_rows == by_item->n_cols && by_user->n_cols == by_item->n_rows, CGX_ERR_ARG,
              "propagate_fwd: operator shapes disagree");
  CGX_REQUIRE(workspace_bytes >= cgx_propagate_workspace_bytes_for(by_user, by_item, d, order), CGX_ERR_WORKSPACE,
              "propagate_fwd: workspace too small");
  const int64_t U = by_user->n_rows, I = by_item->n_rows;
  Arena ws(workspace, workspace_bytes);
  const bool one = order == CGX_ORDER_GS;   // one layer buffer per side is enough (see propagate_ws)
  float* ub[2];
  float* ib[2];
  ub[0] = ws.take<float>(U * d);
  ub[1] = one ? ub[0] : ws.take<float>(U * d);
  ib[0] = ws.take<float>(I * d);
  ib[1] = one ? ib[0] : ws.take<float>(I * d);
  size_t lws = spmm_ws(by_user, d) > spmm_ws(by_item, d) ? spmm_ws(by_user, d) : spmm_ws(by_item, d);
  void* lw = ws.take<char>(lws);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "propagate_fwd: workspace too small");
  const float s = 1.0f / float(K + 1);
  const SpmmPush nops{0ull, 0, 0};
  // The last layer writes only the output rows its masks flag (rows_u / rows_i, nullable).  A mask needs the
  // row-sparse instantiation (spmm_dispatch); its gather flags are all_rows, all ones, so no entry is dropped and the
  // sum is the unmasked one.  Layer k - 1's buffers are what layer k gathers, and the last layer writes no user
  // buffer (and, in Jacobi order, no item buffer): a later call for the rows left out finds its inputs intact.
  for (int k = layer_begin; k < layer_end; ++k) {
    const bool first = k == 0, last = k == K - 1;
    const float* cu = first ? e0_u : ub[(k - 1) & 1];   // layer k tables
    const float* ci = first ? e0_i : ib[(k - 1) & 1];
    float* nu = ub[k & 1];
    float* ni = ib[k & 1];
    const float sc = last ? s : 1.0f;
    const uint8_t* mu = last ? rows_u : nullptr;
    const uint8_t* mi = last ? rows_i : nullptr;
    // item side: i_{k+1} = C u_k
    const bool need_ni = !last || order == CGX_ORDER_GS;
    CGX_TRY(spmm_dispatch(by_item, 0, d, cu, need_ni ? ni : nullptr, first ? e0_i : out_i, out_i, sc, lw, lws,
                          stream, mi ? all_rows : nullptr, nops, nullptr, mi));
    // user side: u_{k+1} = A i_k (Jacobi) or A i_{k+1} (Gauss-Seidel)
    const float* src = order == CGX_ORDER_JACOBI ? ci : ni;
    CGX_TRY(spmm_dispatch(by_user, 0, d, src, last ? nullptr : nu, first ? e0_u : out_u, out_u, sc, lw, lws,
                          stream, mu ? all_rows : nullptr, nops, nullptr, mu));
  }
  return CGX_OK;
}

// d_e0_i = s * g_i where only flagged rows of g_i are non-zero: zero fill + the flagged rows
__global__ void k_scale_rows(const float4* __restrict__ in, const uint8_t* __restrict__ nz, float4* __restrict__ out,
                             int64_t n_rows, int32_t row4, float s) {
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
  if (r >= n_rows || __ldg(nz + r) == 0) return;
  for (int p = threadIdx.x & 31; p < row4; p += 32) out[r * row4 + p] = scale4(in[r * row4 + p], s);
}

extern "C" int cgx_propagate_bwd(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t K, int32_t d,
                                 const float* g_u, const float* g_i, float* d_e0_u, float* d_e0_i,
                                 void* workspace, size_t workspace_bytes, void* stream_) {
  return cgx_propagate_bwd_flagged(by_user, by_item, order, K, d, g_u, g_i, nullptr, nullptr, d_e0_u, d_e0_i, workspace,
                                   workspace_bytes, stream_);
}

extern "C" int cgx_propagate_bwd_flagged(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t K,
                                         int32_t d, const float* g_u, const float* g_i, const uint8_t* g_u_rows,
                                         const uint8_t* g_i_rows, float* d_e0_u, float* d_e0_i, void* workspace,
                                         size_t workspace_bytes, void* stream_) {
  return cgx_propagate_bwd_frontier(by_user, by_item, order, K, d, g_u, g_i, g_u_rows, g_i_rows, nullptr, d_e0_u,
                                    d_e0_i, workspace, workspace_bytes, stream_);
}

extern "C" int cgx_propagate_bwd_frontier(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t K,
                                          int32_t d, const float* g_u, const float* g_i, const uint8_t* g_u_rows,
                                          const uint8_t* g_i_rows, const uint8_t* front_i, float* d_e0_u,
                                          float* d_e0_i, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CGX_REQUIRE((g_u_rows == nullptr) == (g_i_rows == nullptr), CGX_ERR_ARG,
              "propagate_bwd_flagged: pass both row-flag arrays or neither");
  CGX_REQUIRE(by_user && by_item && g_u && g_i && d_e0_u && d_e0_i, CGX_ERR_ARG, "propagate_bwd: NULL pointer");
  CGX_REQUIRE(K >= 1, CGX_ERR_ARG, "propagate_bwd: num_layers must be >= 1");
  CGX_REQUIRE(order == CGX_ORDER_JACOBI || order == CGX_ORDER_GS, CGX_ERR_ARG, "propagate_bwd: bad order");
  CGX_REQUIRE(workspace_bytes >= cgx_propagate_workspace_bytes_for(by_user, by_item, d, order), CGX_ERR_WORKSPACE,
              "propagate_bwd: workspace too small");
  const int64_t U = by_user->n_rows, I = by_item->n_rows;
  Arena ws(workspace, workspace_bytes);
  const bool one = order == CGX_ORDER_GS;   // bi' and bu' are each dead when they are overwritten
  float* ub[2];
  float* ib[2];
  ub[0] = ws.take<float>(U * d);
  ub[1] = one ? ub[0] : ws.take<float>(U * d);
  ib[0] = ws.take<float>(I * d);
  ib[1] = one ? ib[0] : ws.take<float>(I * d);
  size_t lws = spmm_ws(by_user, d) > spmm_ws(by_item, d) ? spmm_ws(by_user, d) : spmm_ws(by_item, d);
  void* lw = ws.take<char>(lws);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "propagate_bwd: workspace too small");
  const float s = 1.0f / float(K + 1);
  // The incoming gradient has non-zero rows only where the batch touched the tables (<= batch users,
  // <= 2 * batch items): the products that gather g_u / g_i directly skip the zero rows (row flags, 1 byte per
  // row), and every product's ACC_IN -- the gradient seed again -- is only read where its flag is set.  After one
  // product the adjoint itself is dense.  CGX_OPT_SPARSE_FIRST_ADJOINT = 0 switches both off.
  const bool given = g_u_rows != nullptr;                 // the caller already knows the non-zero rows
  const bool sparse = given || option(CGX_OPT_SPARSE_FIRST_ADJOINT) != 0;
  uint8_t* nz_u = given ? const_cast<uint8_t*>(g_u_rows) : ws.take<uint8_t>(U);
  uint8_t* nz_i = given ? const_cast<uint8_t*>(g_i_rows) : ws.take<uint8_t>(I);
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "propagate_bwd: workspace too small");
  // Work with the unscaled adjoints bu' = bu / s, bi' = bi / s (the recurrences are linear):
  //   Jacobi: (bu', bi') <- (g_u + C^T bi', g_i + A^T bu');  Gauss-Seidel: bi' = g_i + A^T bu'; bu' = g_u + C^T bi'
  // and fold s into the last product's epilogue.
  // Item frontier (front_i, nullable): the first item-side adjoint g_i + A^T g_u is non-zero only on front_i.  When
  // that product writes scratch, it computes only the rows of front_i, and the one product that gathers it skips
  // every other row.  Invariant: every row outside front_i of the masked buffer is stale and is never read.  No
  // product that writes d_e0_u / d_e0_i is masked.  (A mask needs the row-sparse first product: spmm_dispatch.)
  const uint8_t* front = sparse ? front_i : nullptr;
  if (order == CGX_ORDER_JACOBI) {
    const float* bu = g_u;
    const float* bi = g_i;
    if (sparse && !given) {
      CGX_TRY(row_flags(g_u, U, d, nz_u, stream));
      CGX_TRY(row_flags(g_i, I, d, nz_i, stream));
    }
    for (int k = 0; k < K; ++k) {
      const bool last = k == K - 1;
      float* nu = last ? d_e0_u : ub[k & 1];
      float* ni = last ? d_e0_i : ib[k & 1];
      const float sc = last ? s : 1.0f;
      const bool sp = sparse && k == 0;
      const SpmmPush nops{0ull, 0, 0};
      // bi of k = 1 is the masked output of k = 0's item product (scratch, K >= 2): gather only its frontier rows
      const uint8_t* bi_nz = sp ? nz_i : (k == 1 ? front : nullptr);
      CGX_TRY(spmm_dispatch(by_user, 1, d, bi, nullptr, g_u, nu, sc, lw, lws, stream, bi_nz, nops,
                            sparse ? nz_u : nullptr));                                             // g_u + C^T bi
      CGX_TRY(spmm_dispatch(by_item, 1, d, bu, nullptr, g_i, ni, sc, lw, lws, stream, sp ? nz_u : nullptr, nops,
                            sparse ? nz_i : nullptr, k == 0 && !last ? front : nullptr));       // g_i + A^T bu
      bu = nu;
      bi = ni;
    }
  } else {
    const float* bu = g_u;
    if (sparse && !given) {
      CGX_TRY(row_flags(g_u, U, d, nz_u, stream));
      CGX_TRY(row_flags(g_i, I, d, nz_i, stream));
    }
    const SpmmPush nops{0ull, 0, 0};
    for (int k = 0; k < K; ++k) {
      const bool last = k == K - 1;
      float* ni = ib[0];   // scratch at every k: d_e0_i = s * g_i is written below
      float* nu = last ? d_e0_u : ub[k & 1];
      const uint8_t* f0 = k == 0 ? front : nullptr;
      CGX_TRY(spmm_dispatch(by_item, 1, d, bu, nullptr, g_i, ni, 1.0f, lw, lws, stream,
                            sparse && k == 0 ? nz_u : nullptr, nops, sparse ? nz_i : nullptr, f0));      // bi'
      CGX_TRY(spmm_dispatch(by_user, 1, d, ni, nullptr, g_u, nu, last ? s : 1.0f, lw, lws, stream, f0, nops,
                            sparse ? nz_u : nullptr));                                                // bu'
      bu = nu;
    }
    const int64_t n4 = I * d / 4;
    if (given) {   // d_e0_i = s * g_i is as row-sparse as g_i: zero fill + the flagged rows (half the traffic)
      CGX_CUDA(cudaMemsetAsync(d_e0_i, 0, size_t(I) * d * 4, stream));
      if (I > 0) {
        k_scale_rows<<<(unsigned)ceil_div(I * 32, 256), 256, 0, stream>>>(
            reinterpret_cast<const float4*>(g_i), nz_i, reinterpret_cast<float4*>(d_e0_i), I, d / 4, s);
        CGX_LAUNCH_CHECK();
      }
    } else {
      k_scale<<<(unsigned)ceil_div(n4, 256), 256, 0, stream>>>(reinterpret_cast<const float4*>(g_i),
                                                               reinterpret_cast<float4*>(d_e0_i), n4, s);
      CGX_LAUNCH_CHECK();
    }
  }
  return CGX_OK;
}
