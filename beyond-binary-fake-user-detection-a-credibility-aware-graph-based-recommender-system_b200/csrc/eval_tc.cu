// Tensor-core score path of the full-rank evaluation: tcgen05.mma (UMMA) user x item score tiles
// with accumulators in TMEM, fused with the train-item mask and a per-row running top-K', then an
// exact fp32 re-scoring of the K' candidates.
//
// Replaces (reference, /root/reference): the per-user score + mask + argsort loop of
// evaluate_full_ranking, Version-2/lighgcn_cu_pop.py:691-704 -- the only dense contraction on the
// path (2 * U_eval * I * d FLOPs).
//
// Numerics.  The reference scores in fp32.  precision = BF16X3 splits every fp32 value into
// hi + lo bf16 parts, stored once as [hi | lo], and accumulates a_hi.b_hi + a_lo.b_hi + a_hi.b_lo (3d
// multiply-adds per score) on the tensor cores: |error| <= ~2^-16 |a||b|.  The tensor-core pass only SELECTS K' = K + margin
// candidates per user; k_rescore then recomputes their scores exactly as the fp32 kernel does (same
// fmaf order -> same bits), sorts by (score desc, id asc) and proves the top K complete:
// if exact_score[K-1] > approx_score[K'-1] + eps(user) no item outside the candidate list can reach
// the top K.  Rows that fail the proof are redone by the exact fp32 kernel (k_eval_redo_rows), and so
// are rows whose lists hold fewer than K real candidates (a user with fewer unseen items than K').  The
// result is therefore identical to CGX_SCORE_FP32.  precision = BF16 is the single-pass variant (error
// ~2^-8 relative, no proof; short lists are still redone) for callers that accept approximate ranking.
//
// Kernel anatomy (one CTA per 128 users, 17 warps with two scanning groups, 13 with one):
//   warp 0      TMEM allocation, then one elected lane (elect.sync) issues tcgen05.mma (M=128, N=128, K=16 per
//               instruction, K'/16 instructions per item tile), tcgen05.commit -> mbarriers
//   warps 1-8   epilogue, two groups of four warps (round 2; one group when the lists of two do not fit shared
//               memory or K > 20): group g scans the item tiles of parity g -- tcgen05.ld 32x32b.x16 -> registers, 16
//               compares -> hit mask, one select tree + one shared store per hit, warp-uniform drain into the row's
//               K' kept candidates (one thread per user and group).  The scan is a chain of dependent ALU latencies:
//               ONE warp per scheduler issued on 23 % of its cycles (profiles/r2_ncu_eval_umma_c2_one_group.txt),
//               two warps overlap each other's stalls: C2 1.52 -> 1.09 ms, C3 4.21 -> 2.85 ms
//               (profiles/r2_eval_variants.jsonl), same ids and score bits.
//   next 4      producer: ONE elected thread issues a TMA tile load (cp.async.bulk.tensor.2d, SWIZZLE_128B tensor
//               map over the bf16 item operand [I, Kp]; rows past I are zero-filled by the unit) per ring stage:
//               one 64-column k-block (128 items x 128 B) lands in the canonical K-major SWIZZLE_128B UMMA layout
//               and completes the stage's mbarrier by transaction bytes -- no register staging, no per-thread
//               address arithmetic, no proxy fence.  The ring (3..8 stages) is k-block granular so that wide tables
//               fit: d = 128 with BF16X3 needs 64 KB per item tile next to 64 KB of users.
//   last 4      mask builders: per user row, 128 "is a train item" bits per item tile, a few tiles ahead
// TMEM: 2 accumulators of 128 columns per scanning group (4 x 128 = all 512 columns with two groups).  Group g owns
// stages g and g + 2: the MMA of its next tile fills one while it scans the other.
#include <cuda.h>        // CUtensorMap + the cuTensorMapEncodeTiled prototype (resolved at run time, no -lcuda)
#include <cuda_bf16.h>
#include <float.h>
#include <stdlib.h>

#include "common.cuh"

namespace cgx {

int eval_fp32_rows(const int64_t* users, const int32_t* row_list, const int32_t* n_rows_dev, int64_t max_rows,
                   const float* f_u, const float* f_i, int32_t I, int32_t d, const int64_t* tr_indptr,
                   const int32_t* tr_idx, int32_t K, int32_t* out_ids, float* out_scores, cudaStream_t stream);

constexpr int TC_M = 128;          // users per CTA
constexpr int TC_N = 128;          // items per tile
constexpr int TC_MAX_STAGES = 8;   // B ring: up to 8 stages of one 64-column k-block (128 items x 128 B = 16 KB)
constexpr int TC_KB_BYTES = TC_N * 128;
constexpr int TC_MASK_RING = 4;    // train-item bitmasks of that many item tiles are built ahead of the epilogue
constexpr int TC_MAX_ACC = 4;      // TMEM accumulator stages of 128 columns: two per epilogue group
constexpr float TC_MASKED = -1e9f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// one lane of a converged warp (the form ptxas recognises as "exactly one thread": operands of the tcgen05
// instructions under it move to uniform registers without a per-operand broadcast loop)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(pred));
  return pred != 0u;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major SWIZZLE_128B operand tile: k-block kb (64 bf16 = 128 B per row) at kb * rows * 128; inside
// a k-block row r occupies bytes [r*128, r*128+128) with its 16-byte chunk c stored at chunk c ^ (r % 8).
// Descriptor: start address >> 4, LBO field 1 (unused for swizzled K-major), SBO = 1024 B (8 rows),
// version 1 (Blackwell), layout type 2 (SWIZZLE_128B).  A K=16 step inside a k-block advances the
// start address by 32 bytes.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFF) >> 4) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int q = 0; q < 16; ++q) v[q] = __uint_as_float(r[q]);   // valid after tmem_wait_ld()
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ bool tc_better(float sa, int32_t ia, float sb, int32_t ib) {
  return sa > sb || (sa == sb && ia < ib);
}
__device__ __forceinline__ bool tc_in_row(const int32_t* __restrict__ idx, int64_t lo, const int64_t end,
                                          int32_t item) {
  int64_t hi = end;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(idx + mid) < item) lo = mid + 1; else hi = mid;
  }
  return lo < end && __ldg(idx + lo) == item;
}

// ---- operand preparation: fp32 rows -> bf16 [hi (Dp columns) | lo (Dp columns)], Dp = d rounded up to 64 ------
__global__ void k_tc_convert(const float* __restrict__ src, const int64_t* __restrict__ rows, int64_t n_rows,
                             int32_t d, int parts, int Dp, __nv_bfloat16* __restrict__ dst,
                             float* __restrict__ norms, unsigned int* __restrict__ max_norm_bits) {
  const int64_t r = int64_t(blockIdx.x) * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  const int64_t sr = rows ? rows[r] : r;
  const int Kp = parts * Dp;
  float ss = 0.f;
  for (int c = lane; c < Dp; c += 32) {
    const float x = c < d ? src[sr * d + c] : 0.f;      // columns d..Dp of every part are zero padding
    ss = fmaf(x, x, ss);
    const __nv_bfloat16 hi = __float2bfloat16_rn(x);
    dst[r * Kp + c] = hi;
    if (parts == 2) dst[r * Kp + Dp + c] = __float2bfloat16_rn(x - __bfloat162float(hi));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (lane == 0) {
    const float nrm = sqrtf(ss);
    if (norms) norms[r] = nrm;
    if (max_norm_bits) atomicMax(max_norm_bits, __float_as_uint(nrm));   // non-negative floats order as uints
  }
}

// ---- the UMMA kernel ---------------------------------------------------------------------------
// KC kept candidates and BC arrival-buffer slots per (user, epilogue group); NG epilogue groups of 4 warps.
// The epilogue, not the MMA, bounds this kernel (d is only 64..128: 768 tensor-pipe cycles per tile with BF16X3
// against ~2000 cycles of scanning even when no score enters a list, profiles/r2_eval_ablation_one_group.json).
template <int KC, int BC, int NG>
__global__ void __launch_bounds__(32 * (9 + 4 * NG), 1) k_eval_umma(const __grid_constant__ CUtensorMap b_map,   // item operand [I, Kp] bf16
                                                             const __nv_bfloat16* __restrict__ Au,   // [n_users, Kp]
                                                             const int64_t* __restrict__ users, int64_t n_users,
                                                             int32_t I, int32_t Kp, int32_t nkb, int32_t S,
                                                             const int64_t* __restrict__ tr_indptr,
                                                             const int32_t* __restrict__ tr_idx,
                                                             int32_t* __restrict__ cand_ids,       // [n_users, cand_stride]
                                                             int32_t cand_stride,
                                                             float* __restrict__ cand_thr,          // [n_users, 2]
                                                             int dbg) {
  constexpr int TC_THREADS = 32 * (9 + 4 * NG);
  extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
  // SWIZZLE_128B atoms must start on 1024-byte boundaries of the shared window
  unsigned char* tc_smem = tc_smem_raw + ((1024u - (smem_u32(tc_smem_raw) & 1023u)) & 1023u);
  const uint32_t a_bytes = uint32_t(TC_M) * Kp * 2;              // the users' operand: Kp / 64 k-blocks, [hi | lo]
  unsigned char* smem_a = tc_smem;
  unsigned char* smem_b = tc_smem + a_bytes;                      // ring of S item k-blocks
  float* list_s_all = reinterpret_cast<float*>(smem_b + S * TC_KB_BYTES);          // [NG][KC][128] unsorted candidates
  int32_t* list_i_all = reinterpret_cast<int32_t*>(list_s_all + NG * KC * TC_M);   // [NG][KC][128]
  uint2* buf_all = reinterpret_cast<uint2*>(list_i_all + NG * KC * TC_M);          // [NG][BC][128] arrivals (score bits, item)
  uint4* mask_all = reinterpret_cast<uint4*>(buf_all + NG * BC * TC_M);            // [TC_MASK_RING][128] train-item bits
  uint64_t* bars = reinterpret_cast<uint64_t*>(mask_all + TC_MASK_RING * TC_M);
  uint64_t* full_bar = bars;                     // [TC_MAX_STAGES]  producers -> MMA
  uint64_t* empty_bar = bars + TC_MAX_STAGES;    // [TC_MAX_STAGES]  MMA (commit) -> producers
  uint64_t* tfull_bar = bars + 2 * TC_MAX_STAGES;                        // [TC_MAX_ACC]  MMA (commit) -> epilogue
  uint64_t* tempty_bar = bars + 2 * TC_MAX_STAGES + TC_MAX_ACC;          // [TC_MAX_ACC]  epilogue -> MMA
  uint64_t* mfull_bar = bars + 2 * TC_MAX_STAGES + 2 * TC_MAX_ACC;                   // [TC_MASK_RING] mask warps -> epilogue
  uint64_t* mempty_bar = bars + 2 * TC_MAX_STAGES + 2 * TC_MAX_ACC + TC_MASK_RING;   // [TC_MASK_RING] epilogue -> mask warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_MAX_STAGES + 2 * TC_MAX_ACC + 2 * TC_MASK_RING);
  // NS accumulator stages of TC_N TMEM columns; tile j lives in stage j % NS.  With two epilogue groups, group g owns
  // the tiles of parity g and therefore stages g and g + 2: while it scans one of them the MMA of its next tile fills
  // the other (with one stage per group the group would idle through the issue + execution of its own next tile).
  constexpr int NS = 2 * NG;
  static_assert(NS <= TC_MAX_ACC, "accumulator stages");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t u0 = int64_t(blockIdx.x) * TC_M;
  const int n_tiles = (I + TC_N - 1) / TC_N;
  // Kp = parts * nkb * 64: hi k-blocks 0..nkb-1, then (BF16X3) lo k-blocks nkb..2 nkb-1 -- both operands.
  // One item tile = n_units k-blocks of B ("units"), streamed through the ring one k-block at a time so that
  // the ring does not have to hold a whole tile (d = 128, BF16X3: 64 KB per tile).  Unit u < nkb is b_hi[u] and
  // multiplies a_hi[u] and a_lo[u]; unit u >= nkb is b_lo[u - nkb] and multiplies a_hi[u - nkb]
  // (a_hi b_hi + a_lo b_hi + a_hi b_lo; the lo*lo term is below the proof's eps).
  const int n_units = Kp / 64;
  const int64_t n_steps = int64_t(n_tiles) * n_units;
  const int chunks = TC_M * n_units * 8;         // 16-byte chunks of the A operand

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_MAX_STAGES; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
    for (int a = 0; a < TC_MAX_ACC; ++a) { mbar_init(tfull_bar + a, 1); mbar_init(tempty_bar + a, 128); }
    for (int m = 0; m < TC_MASK_RING; ++m) { mbar_init(mfull_bar + m, 128); mbar_init(mempty_bar + m, 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(NS * TC_N));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // A tile: this CTA's 128 users, staged once by every thread (rows past n_users are zero)
  for (int q = threadIdx.x; q < chunks; q += TC_THREADS) {
    const int c = q & 7, r = (q >> 3) & (TC_M - 1), kb = q >> 10;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (u0 + r < n_users) v = *reinterpret_cast<const uint4*>(Au + (u0 + r) * Kp + kb * 64 + c * 8);
    *reinterpret_cast<uint4*>(smem_a + kb * (TC_M * 128) + r * 128 + ((c ^ (r & 7)) << 4)) = v;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== MMA issuer =====
    // idesc: c=F32 (1<<4), a=BF16 (1<<7), b=BF16 (1<<10), K-major both, N>>3 at bit 17, M>>4 at bit 24
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(TC_N >> 3) << 17) | (uint32_t(TC_M >> 4) << 24);
    const uint32_t a_addr = smem_u32(smem_a);
    int s = 0;                                      // ring position and its phase bit, advanced without dividing
    uint32_t ph = 0;
    // The leader comes from elect.sync (ptxas then knows that exactly one thread runs the block and moves the
    // descriptors to uniform registers directly; under `lane == 0` every tcgen05.mma was wrapped in a broadcast loop:
    // 175 instructions per k-block against 95, and the issuing warp was busy for half of a tile period), and the
    // descriptors are one base each plus (byte offset >> 4): the address field holds (addr & 0x3FFFF) >> 4 and every
    // operand lies below 256 KB, so the sum never carries out of the field.
    const uint64_t a_desc0 = umma_desc_sw128(a_addr);
    const uint64_t b_desc0 = umma_desc_sw128(smem_u32(smem_b));
    for (int j = 0; j < n_tiles; ++j) {
      const int a = j & (NS - 1);
      mbar_wait(tempty_bar + a, ((j / NS) & 1) ^ 1);
      for (int u = 0; u < n_units; ++u) {
        mbar_wait(full_bar + s, ph);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t bd = b_desc0 + uint64_t(uint32_t(s * TC_KB_BYTES) >> 4);
          const int ka = u < nkb ? u : u - nkb;                       // a_hi k-block paired with this unit
          const uint64_t ad = a_desc0 + uint64_t(uint32_t(ka * (TC_M * 128)) >> 4);
          if (!(dbg & 2)) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)   // a K = 16 step inside a k-block: + 32 bytes
              umma_bf16(tmem_base + a * TC_N, ad + 2 * k4, bd + 2 * k4, idesc, (u | k4) ? 1u : 0u);
            if (u < nkb && n_units > nkb) {                           // BF16X3: a_lo[u] . b_hi[u]
              const uint64_t al = a_desc0 + uint64_t(uint32_t((nkb + u) * (TC_M * 128)) >> 4);
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) umma_bf16(tmem_base + a * TC_N, al + 2 * k4, bd + 2 * k4, idesc, 1u);
            }
          }
          umma_commit(empty_bar + s);                   // ring stage reusable once these MMAs have read it
          if (u == n_units - 1) umma_commit(tfull_bar + a);   // accumulator complete
        }
        __syncwarp();
        if (++s == S) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp >= 5 + 4 * NG) {
    // ===== mask builders: one thread per user row walks the row's sorted train items and leaves, for every
    // item tile, 128 bits "column is a train item" in a ring of TC_MASK_RING tiles.  The walk is a chain of
    // dependent loads; here it runs ahead of, and beside, the epilogue instead of inside it. =====
    const int row = threadIdx.x - (5 + 4 * NG) * 32;
    int64_t cur = 0, hi = 0;
    if (u0 + row < n_users) {
      const int64_t uid = users[u0 + row];
      cur = __ldg(tr_indptr + uid);
      hi = __ldg(tr_indptr + uid + 1);
    }
    int32_t nxt = cur < hi ? __ldg(tr_idx + cur) : INT32_MAX;
    for (int j = 0; j < n_tiles; ++j) {
      const int m = j % TC_MASK_RING;
      mbar_wait(mempty_bar + m, ((j / TC_MASK_RING) & 1) ^ 1);
      uint4 bits = make_uint4(0u, 0u, 0u, 0u);
      const int32_t i0 = j * TC_N;
      while (nxt < i0 + TC_N) {
        const int c = nxt - i0;
        const uint32_t b = 1u << (c & 31);
        if (c < 32) bits.x |= b; else if (c < 64) bits.y |= b; else if (c < 96) bits.z |= b; else bits.w |= b;
        ++cur;
        nxt = cur < hi ? __ldg(tr_idx + cur) : INT32_MAX;
      }
      mask_all[m * TC_M + row] = bits;
      mbar_arrive(mfull_bar + m);
    }
  } else if (warp >= 1 + 4 * NG) {
    // ===== producer: one thread, one TMA tile load per ring stage =====
    if (threadIdx.x == (1 + 4 * NG) * 32) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&b_map)) : "memory");
      int j = 0, u = 0, s = 0;
      uint32_t ph = 1;                                // parity to wait for on empty_bar[s]: 1 on the first lap
      for (int64_t g = 0; g < n_steps; ++g) {
        mbar_wait(empty_bar + s, ph);
        const uint32_t bar = smem_u32(full_bar + s);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(uint32_t(TC_KB_BYTES))
                     : "memory");
        if (!(dbg & 4)) {
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
                  "r"(smem_u32(smem_b + s * TC_KB_BYTES)),
              "l"(reinterpret_cast<uint64_t>(&b_map)), "r"(u * 64), "r"(j * TC_N), "r"(bar)
              : "memory");
        } else {
          asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(uint32_t(TC_KB_BYTES)) : "memory");
        }
        if (++u == n_units) { u = 0; ++j; }
        if (++s == S) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ===== epilogue: one thread per user row =====
    // Scores > the row's threshold are appended (predicated store, no branch) to a BC-slot buffer; when
    // some lane's buffer could overflow in the next 16-column chunk the WARP drains with all lanes
    // active: "replace the weakest of the K' kept candidates and rescan for the new weakest" -- a loop of
    // fixed length, so lanes do not diverge on data.  Train items never arrive: the mask builders' bits
    // clear them from the hit mask.  Batching arrivals over several chunks
    // keeps most lanes busy in a drain (a lane sees ~0.8 arrivals per 128-item tile in steady state).
    // The kept list stays unsorted; k_rescore ranks it.  TMEM loads are software pipelined.
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may read
    const int grp = (warp - 1) >> 2;           // epilogue group: owns the tiles j with j % NG == grp
    float* list_s = list_s_all + grp * KC * TC_M;
    int32_t* list_i = list_i_all + grp * KC * TC_M;
    uint2* buf = buf_all + grp * BC * TC_M;
    const int row = quad * 32 + lane;
    const int64_t ug = u0 + row;
    const bool live = ug < n_users;
    for (int p = 0; p < KC; ++p) { list_s[p * TC_M + row] = -FLT_MAX; list_i[p * TC_M + row] = INT32_MAX; }
    float thr = live ? -FLT_MAX : FLT_MAX;      // score of the weakest kept candidate (dead rows accept nothing)
    int weakest = 0;           // its slot
    uint2* const wr0 = buf + row;   // arrival slot e of this row = wr0[e * 128]
    int cnt = 0;                    // arrivals waiting in the buffer

    auto drain = [&]() {
      for (int e = 0; e < cnt; ++e) {
        const uint2 ent = wr0[e * TC_M];
        const float sc = __uint_as_float(ent.x);
        const int32_t item = int32_t(ent.y);
        if (sc > thr) {
          list_s[weakest * TC_M + row] = sc;
          list_i[weakest * TC_M + row] = item;
          // new weakest: KC independent loads, then a min tree of depth log2(KC) (a sequential scan would be a
          // chain of KC dependent compare+select steps)
          float mv[KC];
          int ms[KC];
#pragma unroll
          for (int p = 0; p < KC; ++p) { mv[p] = list_s[p * TC_M + row]; ms[p] = p; }
#pragma unroll
          for (int w = 1; w < KC; w <<= 1) {
#pragma unroll
            for (int p = 0; p + w < KC; p += 2 * w) {
              const bool lower = mv[p + w] < mv[p];
              mv[p] = lower ? mv[p + w] : mv[p];
              ms[p] = lower ? ms[p + w] : ms[p];
            }
          }
          thr = mv[0];
          weakest = ms[0];
        }
      }
      cnt = 0;
    };

    for (int j = grp; j < n_tiles; j += NG) {
      const int a = j & (NS - 1);
      mbar_wait(tfull_bar + a, (j / NS) & 1);
      tc_fence_after();
      const int32_t i0 = j * TC_N;
      const int valid = I - i0 < TC_N ? I - i0 : TC_N;   // columns of this tile that are real items
      const uint32_t tbase = tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(a * TC_N);
      const int m = j % TC_MASK_RING;
      mbar_wait(mfull_bar + m, (j / TC_MASK_RING) & 1);
      const uint4 tbits = mask_all[m * TC_M + row];
      float v[2][16];
      tmem_ld16(tbase, v[0]);
      tmem_wait_ld();
#pragma unroll   // fully: "unroll 2" (4x less code, fewer instruction-cache misses) measured 8-12 % SLOWER
      for (int ch = 0; ch < TC_N / 16; ++ch) {
        if (ch + 1 < TC_N / 16) tmem_ld16(tbase + (ch + 1) * 16, v[(ch + 1) & 1]);   // in flight during the scan below
        // 16 independent compares -> bit mask -> slot of every hit from a popcount of the lower bits: no
        // loop-carried dependency (a single warp per scheduler cannot hide a 16-long pointer-bump chain)
        const int lim = valid - ch * 16;          // columns of this chunk that are real items (>= 16: all)
        const uint32_t tw = (ch >> 1) == 0 ? tbits.x : (ch >> 1) == 1 ? tbits.y : (ch >> 1) == 2 ? tbits.z : tbits.w;
        const uint32_t keep = (lim >= 16 ? 0xffffu : lim <= 0 ? 0u : (1u << lim) - 1u) & ~(tw >> ((ch & 1) * 16));
        uint32_t hit = 0;
#pragma unroll
        for (int q = 0; q < 16; ++q) hit |= v[ch & 1][q] > thr ? (1u << q) : 0u;
        hit &= keep;
        if (dbg & 1) hit = 0;
        // one hit per lane per pass (a warp sees ~3 hits per chunk early on, < 1 later): the passes are
        // warp-uniform, and a hit costs a 16 -> 1 select tree instead of 16 predicated store sequences
        bool any_hit = __any_sync(0xffffffffu, hit != 0u);
        const bool had_hits = any_hit;
        while (any_hit) {
          if (hit != 0u) {
            const int q = __ffs(hit) - 1;
            hit &= hit - 1u;
            float s8[8], s4[4];
#pragma unroll
            for (int t = 0; t < 8; ++t) s8[t] = (q & 1) ? v[ch & 1][2 * t + 1] : v[ch & 1][2 * t];
#pragma unroll
            for (int t = 0; t < 4; ++t) s4[t] = (q & 2) ? s8[2 * t + 1] : s8[2 * t];
            const float s2a = (q & 4) ? s4[1] : s4[0], s2b = (q & 4) ? s4[3] : s4[2];
            wr0[cnt * TC_M] = make_uint2(__float_as_uint((q & 8) ? s2b : s2a), uint32_t(i0 + ch * 16 + q));
            ++cnt;
          }
          any_hit = __any_sync(0xffffffffu, hit != 0u);
        }
        // the buffers only grow in a chunk with hits: with two groups the overflow vote is skipped otherwise
        if ((NG == 1 || had_hits) && __any_sync(0xffffffffu, cnt > BC - 16)) {
          if (dbg & 8) cnt = 0; else drain();
        }
        if (ch + 1 < TC_N / 16) tmem_wait_ld();
      }
      tc_fence_before();
      mbar_arrive(tempty_bar + a);
      mbar_arrive(mempty_bar + m);
    }
    drain();
    if (live) {
      for (int p = 0; p < KC; ++p) cand_ids[ug * cand_stride + grp * KC + p] = list_i[p * TC_M + row];
      if (grp == 0) for (int p = NG * KC; p < cand_stride; ++p) cand_ids[ug * cand_stride + p] = INT32_MAX;
      cand_thr[ug * 2 + grp] = thr;
      if (NG == 1) cand_thr[ug * 2 + 1] = thr;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(NS * TC_N));
  }
}

// ---- exact re-scoring of the candidates: one warp per user --------------------------------------
template <int KC>
__global__ void __launch_bounds__(256) k_rescore(const int64_t* __restrict__ users, int64_t n_users,
                                                 const float* __restrict__ f_u, const float* __restrict__ f_i,
                                                 int32_t d, const int64_t* __restrict__ tr_indptr,
                                                 const int32_t* __restrict__ tr_idx,
                                                 const int32_t* __restrict__ cand_ids, const float* __restrict__ cand_thr,
                                                 const float* __restrict__ u_norm, const unsigned int* __restrict__ max_norm_bits,
                                                 float eps_rel, bool prove, int32_t K, int32_t* __restrict__ out_ids,
                                                 float* __restrict__ out_scores, int32_t* __restrict__ redo_rows,
                                                 int32_t* __restrict__ n_redo) {
  constexpr int PER = KC / 32;
  const int lane = threadIdx.x & 31;
  const int64_t r = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= n_users) return;
  const int64_t uid = users[r];
  const int64_t lo = __ldg(tr_indptr + uid), hi = __ldg(tr_indptr + uid + 1);
  const float* urow = f_u + uid * d;
  float sc[PER];
  int32_t id[PER];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    id[q] = cand_ids[r * KC + q * 32 + lane];
    if (id[q] == INT32_MAX) { sc[q] = -FLT_MAX; continue; }
    const float4* u4 = reinterpret_cast<const float4*>(urow);                       // d % 16 == 0, rows 16-byte aligned
    const float4* i4 = reinterpret_cast<const float4*>(f_i + int64_t(id[q]) * d);
    float acc = 0.f;
    for (int k4 = 0; k4 < d / 4; ++k4) {   // same fmaf order as k_eval_fp32 (ascending k, one chain)
      const float4 a = __ldg(u4 + k4), b = __ldg(i4 + k4);
      acc = fmaf(a.x, b.x, acc);
      acc = fmaf(a.y, b.y, acc);
      acc = fmaf(a.z, b.z, acc);
      acc = fmaf(a.w, b.w, acc);
    }
    sc[q] = tc_in_row(tr_idx, lo, hi, id[q]) ? TC_MASKED : acc;
  }
  // rank of every candidate under (score desc, id asc)
  int rank[PER];
#pragma unroll
  for (int q = 0; q < PER; ++q) rank[q] = 0;
#pragma unroll
  for (int q2 = 0; q2 < PER; ++q2) {
    for (int l = 0; l < 32; ++l) {
      const float os = __shfl_sync(0xffffffffu, sc[q2], l);
      const int32_t oi = __shfl_sync(0xffffffffu, id[q2], l);
#pragma unroll
      for (int q = 0; q < PER; ++q) rank[q] += tc_better(os, oi, sc[q], id[q]) ? 1 : 0;
    }
  }
  float kth = -FLT_MAX;
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    if (rank[q] < K) {
      out_ids[r * K + rank[q]] = id[q];
      out_scores[r * K + rank[q]] = sc[q];
    }
    if (rank[q] == K - 1) kth = sc[q];
  }
  // real candidates: a user with fewer unseen items than the lists hold leaves (-FLT_MAX, INT32_MAX) slots, which
  // all share one rank; with fewer than K real ones the columns past it are never written above
  int n_real = 0;
#pragma unroll
  for (int q = 0; q < PER; ++q) n_real += __popc(__ballot_sync(0xffffffffu, id[q] != INT32_MAX));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kth = fmaxf(kth, __shfl_xor_sync(0xffffffffu, kth, o));
  if (lane == 0) {
    // a short list goes to the exact redo, which ranks the train items after the unseen ones as the fp32 kernel does
    bool redo = n_real < K;
    if (!redo && prove) {
      // proof of completeness: nothing outside the list can have an exact score >= kth
      // approx score of the weakest kept candidate of either group: nothing outside the lists scores above it
      const float thr = fmaxf(cand_thr[2 * r], cand_thr[2 * r + 1]);
      const float eps = eps_rel * u_norm[r] * __uint_as_float(*max_norm_bits);
      redo = thr > -FLT_MAX && !(kth > thr + eps);
    }
    if (redo) redo_rows[atomicAdd(n_redo, 1)] = int32_t(r);
  }
}

// ---- exact redo of the rows whose proof failed: one CTA per row, items spread over the threads -----------
// The tiled fp32 kernel (eval.cu) streams the whole catalogue through ONE CTA per 64 users: ~3 ms on C2 however
// few of the 64 rows are live, which tripled the evaluation time when 4 rows of 31 668 needed the redo.  Here a
// row's items are scored by 256 threads (same fmaf chain -> same bits), every thread keeps its best K in shared
// memory (replace-the-weakest), and K rounds of a block-wide arg-best emit the row in (score desc, id asc) order.
constexpr int ER_THREADS = 256;

__global__ void __launch_bounds__(ER_THREADS) k_eval_redo_rows(const int64_t* __restrict__ users,
                                                               const int32_t* __restrict__ row_list,
                                                               const int32_t* __restrict__ n_rows_dev,
                                                               const float* __restrict__ f_u,
                                                               const float* __restrict__ f_i, int32_t I, int32_t d,
                                                               const int64_t* __restrict__ tr_indptr,
                                                               const int32_t* __restrict__ tr_idx, int32_t K,
                                                               int32_t* __restrict__ out_ids,
                                                               float* __restrict__ out_scores) {
  extern __shared__ __align__(16) unsigned char er_smem[];
  float* urow = reinterpret_cast<float*>(er_smem);                       // [d]
  float* ls = urow + d;                                                  // [K][ER_THREADS]
  int32_t* li = reinterpret_cast<int32_t*>(ls + size_t(K) * ER_THREADS);  // [K][ER_THREADS]
  __shared__ float red_s[ER_THREADS / 32];
  __shared__ int32_t red_i[ER_THREADS / 32];
  __shared__ int red_t[ER_THREADS / 32];
  __shared__ int win_t;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_rows = *n_rows_dev;
  for (int rr = blockIdx.x; rr < n_rows; rr += gridDim.x) {
    const int64_t r = row_list[rr];
    const int64_t uid = users[r];
    const int64_t lo = __ldg(tr_indptr + uid), hi = __ldg(tr_indptr + uid + 1);
    __syncthreads();                                                     // previous row's lists are consumed
    for (int k = tid; k < d; k += ER_THREADS) urow[k] = f_u[uid * d + k];
    for (int p = 0; p < K; ++p) { ls[p * ER_THREADS + tid] = -FLT_MAX; li[p * ER_THREADS + tid] = INT32_MAX; }
    __syncthreads();
    float thr = -FLT_MAX;                 // weakest kept entry of this thread's list (empty slots: -FLT_MAX / INT32_MAX)
    int32_t thr_id = INT32_MAX;
    int weakest = 0;
    const float4* u4 = reinterpret_cast<const float4*>(urow);
    for (int32_t i = tid; i < I; i += ER_THREADS) {
      const float4* i4 = reinterpret_cast<const float4*>(f_i + int64_t(i) * d);
      float acc = 0.f;
      for (int k4 = 0; k4 < d / 4; ++k4) {   // same fmaf order as k_eval_fp32 / k_rescore
        const float4 a = u4[k4], b = __ldg(i4 + k4);
        acc = fmaf(a.x, b.x, acc);
        acc = fmaf(a.y, b.y, acc);
        acc = fmaf(a.z, b.z, acc);
        acc = fmaf(a.w, b.w, acc);
      }
      const float sc = tc_in_row(tr_idx, lo, hi, i) ? TC_MASKED : acc;
      if (tc_better(sc, i, thr, thr_id)) {
        ls[weakest * ER_THREADS + tid] = sc;
        li[weakest * ER_THREADS + tid] = i;
        thr = sc;
        thr_id = i;
        for (int p = 0; p < K; ++p) {        // new weakest
          const float ps = ls[p * ER_THREADS + tid];
          const int32_t pi = li[p * ER_THREADS + tid];
          if (tc_better(thr, thr_id, ps, pi)) { thr = ps; thr_id = pi; weakest = p; }
        }
      }
    }
    // K rounds: every thread offers the best entry it still holds, the block picks the overall best
    for (int out = 0; out < K; ++out) {
      float bs = -FLT_MAX;
      int32_t bi = INT32_MAX;
      int bp = 0;
      for (int p = 0; p < K; ++p) {
        const float ps = ls[p * ER_THREADS + tid];
        const int32_t pi = li[p * ER_THREADS + tid];
        if (tc_better(ps, pi, bs, bi)) { bs = ps; bi = pi; bp = p; }
      }
      float ws = bs;
      int32_t wi = bi;
      int wt = tid;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float os = __shfl_xor_sync(0xffffffffu, ws, o);
        const int32_t oi = __shfl_xor_sync(0xffffffffu, wi, o);
        const int ot = __shfl_xor_sync(0xffffffffu, wt, o);
        if (tc_better(os, oi, ws, wi)) { ws = os; wi = oi; wt = ot; }
      }
      if (lane == 0) { red_s[warp] = ws; red_i[warp] = wi; red_t[warp] = wt; }
      __syncthreads();
      if (tid == 0) {
        for (int w = 1; w < ER_THREADS / 32; ++w)
          if (tc_better(red_s[w], red_i[w], ws, wi)) { ws = red_s[w]; wi = red_i[w]; wt = red_t[w]; }
        out_ids[r * K + out] = wi;
        out_scores[r * K + out] = ws;
        win_t = wt;
      }
      __syncthreads();
      if (tid == win_t) { ls[bp * ER_THREADS + tid] = -FLT_MAX; li[bp * ER_THREADS + tid] = INT32_MAX; }   // taken
      __syncthreads();
    }
  }
}

struct TcConfig {
  int KC, BC, NG, stride;   // stride = candidates per user handed to k_rescore (32 or 64)
};
constexpr int TC_DEFAULT_GROUPS = 2;   // what CGX_OPT_EVAL_GROUPS = 0 selects
// shared memory with a ring of S k-blocks; tc_stages picks the deepest ring that fits (0: the shape does not fit)
static size_t tc_smem(const TcConfig& c, int Kp, int S) {
  return size_t(TC_M) * Kp * 2 + size_t(S) * TC_KB_BYTES + size_t(c.NG) * (c.KC + c.BC) * TC_M * 8 +
         size_t(TC_MASK_RING) * TC_M * 16 + 512 + 1024;
}
static int tc_stages(const TcConfig& c, int Kp) {
  for (int S = TC_MAX_STAGES; S >= 3; --S)
    if (tc_smem(c, Kp, S) <= 227 * 1024) return S;
  return 0;
}
static TcConfig tc_config(int32_t K, int Kp) {
  // Measured and rejected in round 1 (no longer compiled): K' = 24 with ONE list (margin 4) -- 4 % faster on C2, but
  // on C3 the completeness proof fails for enough rows that the exact redo doubles the time (10.9 vs 5.7 ms).
  // Two epilogue groups (CGX_OPT_EVAL_GROUPS = 2): group g scans the item tiles of parity g into its own K' = 24
  // list, eight scanning warps instead of four -- the scan is a chain of dependent ALU latencies, one warp per
  // scheduler issues on 23 % of its cycles (profiles/r2_ncu_eval_umma_c2.txt).  The proof compares the K-th exact
  // score with the LARGER of the two lists' weakest entries, each about the 48th best of the catalogue, so it
  // holds more often than with one list of 32.  Needs four accumulator stages (see the kernel) and 64 candidates
  // per user in k_rescore.
  if (K + 12 <= 32) {
    const TcConfig two{24, 24, 2, 64};
    const int64_t groups = option(CGX_OPT_EVAL_GROUPS);
    if ((groups == 0 ? TC_DEFAULT_GROUPS : groups) == 2 && K + 4 <= 24 && tc_stages(two, Kp) > 0) return two;
    return {32, 32, 1, 32};
  }
  return {64, 16, 1, 64};
}
static int tc_parts(int precision) { return precision == CGX_SCORE_BF16X3 ? 2 : 1; }   // stored parts: [hi | lo]
static int tc_dp(int32_t d) { return (d + 63) / 64 * 64; }

size_t eval_topk_tc_workspace(int64_t n_users, int32_t I, int32_t d, int32_t K, int precision) {
  const size_t Kp = size_t(tc_parts(precision)) * tc_dp(d);
  return align_up(size_t(n_users) * Kp * 2) + align_up(size_t(I) * Kp * 2) + align_up(size_t(n_users) * 64 * 4) +
         4 * align_up(size_t(n_users) * 4) + 1024;
}

static bool tc_supported(int32_t d, int32_t K, int precision) {
  if (K + 12 > 64) return false;
  const int Kp = tc_parts(precision) * tc_dp(d);
  return tc_stages(tc_config(K, Kp), Kp) > 0;
}

// Tensor map of the bf16 item operand [I rows, Kp columns], box = one ring stage (64 columns x 128 rows), 128-byte
// swizzle (the UMMA K-major layout), out-of-bounds rows read as zero.  cuTensorMapEncodeTiled is a driver entry
// point: resolved through the runtime, so the library does not link libcuda.
static int make_b_map(const __nv_bfloat16* Bi, int32_t I, int Kp, CUtensorMap* map) {
  typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static encode_fn encode = nullptr;
  if (encode == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    CGX_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    CGX_REQUIRE(fn != nullptr && q == cudaDriverEntryPointSuccess, CGX_ERR_CUDA,
                "eval_topk: cuTensorMapEncodeTiled is not available from this driver");
    encode = reinterpret_cast<encode_fn>(fn);
  }
  const cuuint64_t dims[2] = {cuuint64_t(Kp), cuuint64_t(I)};
  const cuuint64_t strides[1] = {cuuint64_t(Kp) * 2};
  const cuuint32_t box[2] = {64, cuuint32_t(TC_N)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(Bi), dims, strides, box,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CGX_REQUIRE(r == CUDA_SUCCESS, CGX_ERR_CUDA, "eval_topk: cuTensorMapEncodeTiled failed (%d)", int(r));
  return CGX_OK;
}

template <int KC, int BC, int NG, int STRIDE>
static int tc_launch(const __nv_bfloat16* Au, const __nv_bfloat16* Bi, const int64_t* users, int64_t n_users,
                     const float* f_u, const float* f_i, int32_t I, int32_t d, int Kp, int nkb, const int64_t* tr_indptr,
                     const int32_t* tr_idx, int32_t K, int32_t* cand, float* thr, const float* unorm,
                     const unsigned int* scal, float eps_rel, bool prove, int32_t* out_ids, float* out_scores,
                     int32_t* redo_rows, int32_t* n_redo, cudaStream_t stream) {
  const int S = tc_stages(TcConfig{KC, BC, NG, STRIDE}, Kp);
  const size_t smem = tc_smem(TcConfig{KC, BC, NG, STRIDE}, Kp, S);
  CGX_CUDA(cudaFuncSetAttribute(k_eval_umma<KC, BC, NG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUtensorMap b_map;
  CGX_TRY(make_b_map(Bi, I, Kp, &b_map));
  k_eval_umma<KC, BC, NG><<<(unsigned)ceil_div(n_users, TC_M), 32 * (9 + 4 * NG), smem, stream>>>(
      b_map, Au, users, n_users, I, Kp, nkb, S, tr_indptr, tr_idx, cand, STRIDE, thr,
      int(option(CGX_OPT_EVAL_DEBUG) >> 1));
  CGX_LAUNCH_CHECK();
  k_rescore<STRIDE><<<(unsigned)ceil_div(n_users, 8), 256, 0, stream>>>(users, n_users, f_u, f_i, d, tr_indptr, tr_idx,
                                                                       cand, thr, unorm, scal, eps_rel, prove, K, out_ids,
                                                                       out_scores, redo_rows, n_redo);
  CGX_LAUNCH_CHECK();
  return CGX_OK;
}

int eval_topk_tc(const int64_t* users, int64_t n_users, const float* f_u, const float* f_i, int32_t I, int32_t d,
                 const int64_t* tr_indptr, const int32_t* tr_idx, int32_t K, int precision, int32_t* out_ids,
                 float* out_scores, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CGX_REQUIRE(precision == CGX_SCORE_BF16X3 || precision == CGX_SCORE_BF16, CGX_ERR_ARG, "eval_topk: bad precision %d",
              precision);
  const int parts = tc_parts(precision), Dp = tc_dp(d);
  if (!tc_supported(d, K, precision)) {   // shapes the UMMA tile cannot hold: the exact kernel is always valid
    return eval_fp32_rows(users, nullptr, nullptr, n_users, f_u, f_i, I, d, tr_indptr, tr_idx, K, out_ids, out_scores,
                          stream);
  }
  CGX_REQUIRE(workspace_bytes >= eval_topk_tc_workspace(n_users, I, d, K, precision), CGX_ERR_WORKSPACE,
              "eval_topk: workspace too small");
  const int Kp = parts * Dp, nkb = Dp / 64;
  const TcConfig cfg = tc_config(K, Kp);
  Arena ws(workspace, workspace_bytes);
  __nv_bfloat16* Au = ws.take<__nv_bfloat16>(size_t(n_users) * Kp);
  __nv_bfloat16* Bi = ws.take<__nv_bfloat16>(size_t(I) * Kp);
  int32_t* cand = ws.take<int32_t>(size_t(n_users) * 64);
  float* thr = ws.take<float>(size_t(n_users) * 2);
  float* unorm = ws.take<float>(n_users);
  int32_t* redo = ws.take<int32_t>(n_users);
  unsigned int* scal = ws.take<unsigned int>(4);   // [0] max item norm bits, [1] redo count
  CGX_REQUIRE(ws.ok, CGX_ERR_WORKSPACE, "eval_topk: workspace too small");
  CGX_CUDA(cudaMemsetAsync(scal, 0, 16, stream));
  k_tc_convert<<<(unsigned)ceil_div(n_users, 8), 256, 0, stream>>>(f_u, users, n_users, d, parts, Dp, Au, unorm, nullptr);
  CGX_LAUNCH_CHECK();
  k_tc_convert<<<(unsigned)ceil_div(I, 8), 256, 0, stream>>>(f_i, nullptr, I, d, parts, Dp, Bi, nullptr, scal);
  CGX_LAUNCH_CHECK();
  // bf16x3: dropped lo*lo term, bf16 rounding of lo, fp32 accumulation inside the MMA: 2^-13 |a||b| is a safe cap
  const float eps_rel = 1.0f / 8192.0f;
  // bf16 selects without the proof (approximate ranking), but a row with fewer than K real candidates is redone for
  // both precisions: its list cannot fill the K columns
  const bool prove = precision == CGX_SCORE_BF16X3;
  int32_t* n_redo = reinterpret_cast<int32_t*>(scal + 1);
#define CGX_TC_ARGS Au, Bi, users, n_users, f_u, f_i, I, d, Kp, nkb, tr_indptr, tr_idx, K, cand, thr, unorm, scal, eps_rel, \
                    prove, out_ids, out_scores, redo, n_redo, stream
  if (cfg.NG == 2) {
    CGX_TRY((tc_launch<24, 24, 2, 64>(CGX_TC_ARGS)));
  } else if (cfg.KC == 32) {
    CGX_TRY((tc_launch<32, 32, 1, 32>(CGX_TC_ARGS)));
  } else {
    CGX_TRY((tc_launch<64, 16, 1, 64>(CGX_TC_ARGS)));
  }
#undef CGX_TC_ARGS
  // rows with a short list or a failed completeness proof: exact kernel, count read on device
  const size_t er_smem = size_t(d) * 4 + size_t(K) * ER_THREADS * 8;
  CGX_CUDA(cudaFuncSetAttribute(k_eval_redo_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)er_smem));
  const int64_t er_grid = n_users < 148 * 2 ? n_users : 148 * 2;   // persistent over the device-side row list
  k_eval_redo_rows<<<(unsigned)er_grid, ER_THREADS, er_smem, stream>>>(users, redo, n_redo, f_u, f_i, I, d, tr_indptr,
                                                                      tr_idx, K, out_ids, out_scores);
  CGX_LAUNCH_CHECK();
  if (option(CGX_OPT_EVAL_DEBUG) & 1) {   // diagnostics only: synchronises
    unsigned int h[2];
    CGX_CUDA(cudaMemcpyAsync(h, scal, 8, cudaMemcpyDeviceToHost, stream));
    CGX_CUDA(cudaStreamSynchronize(stream));
    fprintf(stderr, "[cgx eval] rows=%lld redo=%u (%.3f %%)\n", (long long)n_users, h[1], 100.0 * h[1] / n_users);
  }
  return CGX_OK;
}

}  // namespace cgx

extern "C" int cgx_eval_topk_uses_tensor_cores(int32_t d, int32_t k, int precision) {
  if (precision != CGX_SCORE_BF16X3 && precision != CGX_SCORE_BF16) return 0;
  return cgx::tc_supported(d, k, precision) ? 1 : 0;
}
