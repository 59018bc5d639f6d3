// scan_tc.cu -- K1: brute-force kNN as a tcgen05 (5th-gen tensor core) TF32 contraction with a
// fused in-register top-k candidate filter: the Q x N distance matrix lives only in TMEM.
//
// Replaces, for the float spaces, the same reference functions as scan_exact.cu
// (SeqSearch::Search seqsearch.cc:144-150 + L2SqrSIMD / ScalarProductSIMD /
// NormScalarProductSIMD + KNNQueue), but as "candidates on the tensor cores, exact re-rank
// in fp32":
//   pass 1 (tc_scan_kernel)  rank(q, x) = A'(q) . x + bias(x) on the tensor cores, where
//          l2 / l2sqr : A' = -2 q,  bias = |x|^2     (rank = d^2 - |q|^2)
//          cosinesimil: A' = -q,    x pre-normalised (rank = -|q| * nsp)
//          negdotprod : A' = -q                      (rank = -q.x)
//        Each query keeps the candidates whose rank beats a running threshold in a small
//        per-query buffer (k' > k survivors after each compaction).
//   pass 2 (tc_rerank_kernel) the reference's own fp32 formula on the candidates only, the k
//        best by (distance, position), and a CERTIFICATE: every point that is not a candidate
//        has approximate rank >= thr, hence exact rank >= thr - E, with E a rigorous bound on
//        the TF32 error of pass 1.  If the exact k-th rank + E < thr the answer is provably the
//        exact top-k; otherwise the query is re-run by the exact scan (scan_exact.cu).
//
// Four kernels share the TMA / mbarrier / tcgen05 plumbing:
//   tc_scan_ts_kernel    rows of <= 128 floats (configs 1, 2): the CTA's 256 prepared queries live in TENSOR MEMORY
//                        (TS-mode MMA), one stage = one whole 64-row database tile (+ the |x|^2 k-block), N = 64
//                        accumulators double buffered per 128-query half; 352 threads: TMA producer, TWO MMA issuer
//                        warps (one per half), eight epilogue warps
//   tc_scan_u8_kernel    uint8 rows (config 4) on the INTEGER tensor pipe (kind::i8): byte rows + base-255 norm
//                        digits, three accumulator buffers per half, int32 epilogue; same roles
//   tc_scan_pair_kernel  longer rows (configs 3, 5) on CTA PAIRS: cta_group::2 M256 x N256 MMAs, both operands
//                        through shared memory, the tensor cores read B from both SMs
//   tc_scan_kernel       the single-CTA long-row kernel (SS mode, N = 128), kept behind option tc_pair=0 for A/B
// All: one CTA per SM, warp-specialised -- a TMA producer warp (cp.async.bulk.tensor, 128B swizzle, mbarrier
// complete_tx), MMA issue by one elected lane of a warp-uniform loop, epilogue warps with thread = TMEM lane = query
// row.  The TS / u8 epilogues drain a tile with one tcgen05.ld.x64, reduce the row's 64 values with a 3-input
// min / max tree and take ONE warp-uniform branch; survivors (a per-lane walk over the tile's groups of 8 values, see
// epi_select_tile) go to the row's candidate buffer.  The long-row kernels use the round-1 epilogue (epi_process, 32
// columns at a time).  Thresholds: the exact 16th best in a register list for k <= 12, otherwise tightened by
// warp-cooperative compaction of the buffer; shared between the CTAs of one query through a per-query word.
// Batched range queries (DESIGN.md K5b): the TS and pair kernels have a RANGE variant whose thresholds are fixed per
// query (tc_range_threshold_kernel turns the radius into the pass-1 rank domain, widened by the certificate's error
// band); survivors are kept in position order up to a position cut, and range_scan.cu verifies them.  The u8 kernel's
// RANGE variant does the same on exact integer accumulators (tc_range_threshold_u8_kernel, error bound 1).
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace nb200 {
namespace {

constexpr int TC_BM = 128;          // queries per operand tile (two tiles per CTA)
constexpr int TC_QB = 256;          // queries per CTA
constexpr int TC_BN = 128;          // database rows per tile
constexpr int TC_KB = 32;           // floats per k-block: one 128-byte swizzle row
constexpr int CHUNK_BYTES = TC_BM * TC_KB * 4;  // 16 KB: 128 rows x 128 B
constexpr int TC_THREADS = 320;
constexpr unsigned FULL = 0xffffffffu;

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// one lane of a converged warp (the compiler keeps everything outside the elected region uniform)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, TF32 inputs, fp32 accumulate
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from tensor memory (lanes = rows, one 32-bit column per tf32 element)
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 64 consecutive columns in ONE instruction (tools/tc_peak.cu: the x64 shape drains 15 % faster than two x32)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&v0)[32], uint32_t (&v1)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      : "=r"(v0[0]), "=r"(v0[1]), "=r"(v0[2]), "=r"(v0[3]), "=r"(v0[4]), "=r"(v0[5]), "=r"(v0[6]), "=r"(v0[7]), "=r"(v0[8]), "=r"(v0[9]), "=r"(v0[10]), "=r"(v0[11]), "=r"(v0[12]), "=r"(v0[13]), "=r"(v0[14]), "=r"(v0[15]), "=r"(v0[16]), "=r"(v0[17]), "=r"(v0[18]), "=r"(v0[19]), "=r"(v0[20]), "=r"(v0[21]), "=r"(v0[22]), "=r"(v0[23]), "=r"(v0[24]), "=r"(v0[25]), "=r"(v0[26]), "=r"(v0[27]), "=r"(v0[28]), "=r"(v0[29]), "=r"(v0[30]), "=r"(v0[31]),
        "=r"(v1[0]), "=r"(v1[1]), "=r"(v1[2]), "=r"(v1[3]), "=r"(v1[4]), "=r"(v1[5]), "=r"(v1[6]), "=r"(v1[7]), "=r"(v1[8]), "=r"(v1[9]), "=r"(v1[10]), "=r"(v1[11]), "=r"(v1[12]), "=r"(v1[13]), "=r"(v1[14]), "=r"(v1[15]), "=r"(v1[16]), "=r"(v1[17]), "=r"(v1[18]), "=r"(v1[19]), "=r"(v1[20]), "=r"(v1[21]), "=r"(v1[22]), "=r"(v1[23]), "=r"(v1[24]), "=r"(v1[25]), "=r"(v1[26]), "=r"(v1[27]), "=r"(v1[28]), "=r"(v1[29]), "=r"(v1[30]), "=r"(v1[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 registers per thread -> 32 lanes x 32 consecutive columns (thread = lane = operand row)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (PTX "tcgen05 matrix descriptor"): K-major operand, rows of
// 128 bytes, 128B swizzle (what the TMA box above produces).  start >> 4 in [0,14), LBO >> 4 in
// [16,30) (unused for swizzled K-major: 1), SBO >> 4 in [32,46) = 8 rows * 128 B, version 1 in
// [46,48), layout SWIZZLE_128B (2) in [61,64).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::tf32: D = F32 (1 @4), A = B = TF32 (2 @7, 2 @10), both K-major,
// N >> 3 @17, M >> 4 @24.
__host__ __device__ constexpr uint32_t make_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ float min3(float a, float b, float c) { return fminf(fminf(a, b), c); }

// ---------------------------------------------------------------- candidate buffers
// Warp-cooperative compaction of one query row's buffer.  Keeps the keys whose rank is <= a cut T
// chosen so that between kprime and kprime + slack keys survive, and returns T (ordered bits): every
// key that is dropped, now or later, has rank >= T, which is what the certificate of pass 2 needs.
// The cut is found by bisecting the VALUE range [min, max] of the live ranks and stopping as soon as
// the survivor count lands in the window -- typically 5-8 ballot rounds instead of a 32-step exact
// select: a compaction stalls the TMEM pipeline of the whole CTA, so it has to be short.
template <int KPL>
__device__ __forceinline__ uint32_t compact_row(uint64_t* buf, int cnt, int kprime, int slack, int lane,
                                                int* new_cnt) {
  uint64_t key[KPL];   // (raw float rank bits << 32) | position
  uint32_t ord[KPL];   // order-preserving image of the rank
  bool valid[KPL];
  uint32_t lo = 0xFFFFFFFFu, hi = 0u;
#pragma unroll
  for (int s = 0; s < KPL; ++s) {
    const int i = s * 32 + lane;
    valid[s] = i < cnt;
    key[s] = valid[s] ? buf[i] : KEY_MAX;
    ord[s] = f32_ordered(__uint_as_float((uint32_t)(key[s] >> 32)));
    if (valid[s]) {
      lo = min(lo, ord[s]);
      hi = max(hi, ord[s]);
    }
  }
  lo = __reduce_min_sync(FULL, lo);
  hi = __reduce_max_sync(FULL, hi);
  const int limit = kprime + slack;
  // invariant: #(rank <= hi) >= kprime
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    int c = 0;
#pragma unroll
    for (int s = 0; s < KPL; ++s) c += __popc(__ballot_sync(FULL, valid[s] && ord[s] <= mid));
    if (c < kprime) {
      lo = mid + 1;
    } else {
      hi = mid;
      if (c <= limit) break;
    }
  }
  const uint32_t t = hi;
  __syncwarp();
  int out = 0;
#pragma unroll
  for (int s = 0; s < KPL; ++s) {  // strictly better than the cut
    const bool keep = valid[s] && ord[s] < t;
    const unsigned m = __ballot_sync(FULL, keep);
    const int pos = out + __popc(m & ((1u << lane) - 1));
    if (keep && pos < limit) buf[pos] = key[s];
    out = min(limit, out + __popc(m));
  }
#pragma unroll
  for (int s = 0; s < KPL; ++s) {  // ties at the cut, while there is room
    const bool eq = valid[s] && ord[s] == t;
    const unsigned m = __ballot_sync(FULL, eq);
    const int pos = out + __popc(m & ((1u << lane) - 1));
    if (eq && pos < limit) buf[pos] = key[s];
    out = min(limit, out + __popc(m));
  }
  __syncwarp();
  *new_cnt = out;
  return t;
}

// A row's threshold after a compaction, shared with the other CTAs that scan other tile ranges for the same
// query: any published cut has kprime points at or below it, so it bounds the query's kprime-th best rank over
// the whole shard and every piece may prune with the smallest one seen so far.
__device__ __forceinline__ float publish_thr(uint32_t* gthr, uint32_t t_ord) {
  const uint32_t old = atomicMin(gthr, t_ord);
  return f32_from_ordered(min(old, t_ord));
}

template <int KPL>
__device__ __forceinline__ void compact_lane(int src, uint64_t* buf, int& cnt, float& thr, int kprime, int slack,
                                             uint32_t* gthr, int lane) {
  const unsigned long long bp = __shfl_sync(FULL, (unsigned long long)(uintptr_t)buf, src);
  const int c = __shfl_sync(FULL, cnt, src);
  int kept;
  const uint32_t t = compact_row<KPL>(reinterpret_cast<uint64_t*>((uintptr_t)bp), c, kprime, slack, lane, &kept);
  if (lane == src) {
    cnt = kept;
    thr = publish_thr(gthr, t);
  }
}

// cycle accounting of the warp roles (experiments builds only: NB200_TC_COUNT=1 prints the sums of the previous launch)
#ifdef NB200_EXPERIMENTS
#define NB_T0(var) long long var = clock64()
#define NB_TACC(acc, var)                  \
  do {                                     \
    const long long now_ = clock64();      \
    acc += (unsigned long long)(now_ - var); \
    var = now_;                            \
  } while (0)
#else
#define NB_T0(var) do {} while (0)
#define NB_TACC(acc, var) do {} while (0)
#endif

constexpr int TS_RK = 16;  // register mode: ranks of a row's 16 best candidates, sorted, in registers

// REG (kprime <= 16, i.e. k <= 10 with the default margin): the row's threshold is the exact 16th best rank seen,
// kept as a sorted register list of RANKS only (insertion = a 16-step min/max chain); the (rank, position) keys
// themselves are appended to the row's buffer, which then only ever receives the ~k ln(N) true improvements
// and needs no compaction.  !REG: the threshold tightens when the buffer is compacted (compact_row).
// RANGE (batched range queries): the threshold is the query's fixed T_q; survivors are appended in position order
// until the buffer is full, then the row records the position of its first dropped survivor in *cut and stops.
template <int KPL, bool REG, bool RANGE = false>
__device__ __forceinline__ void epi_process(const uint32_t (&v)[32], uint32_t pos0, int vcols, uint64_t* buf, int& cnt,
                                            float& thr, float (&tk)[TS_RK], int cap, int kprime, int slack,
                                            uint32_t* gthr, int lane, unsigned (&ctr)[4], uint32_t* cut = nullptr) {
  unsigned need = RANGE ? 0u : __ballot_sync(FULL, cnt > cap - 32);
  while (need) {  // about to overflow: compact at once (!REG: normally the deferred path keeps rows far from here)
    ++ctr[2];
    const int src = __ffs(need) - 1;
    need &= need - 1;
    const float keep = thr;
    compact_lane<KPL>(src, buf, cnt, thr, kprime, slack, gthr, lane);
    if (REG) thr = fminf(thr, keep);  // (the cut is never below the 16th best, the list stays authoritative)
  }
  float r[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) r[j] = __uint_as_float(v[j]);
  if (vcols < 32) {  // rows past the end of the shard: never candidates
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j >= vcols) r[j] = __int_as_float(0x7F800000);
  }
  float g[4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
    g[q] = min3(min3(r[8 * q], r[8 * q + 1], r[8 * q + 2]), min3(r[8 * q + 3], r[8 * q + 4], r[8 * q + 5]),
                fminf(r[8 * q + 6], r[8 * q + 7]));
  const float m = fminf(min3(g[0], g[1], g[2]), g[3]);
  if (m < thr) {
    ++ctr[1];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (g[q] < thr) {
        if constexpr (REG) {
          // which of the group's 8 values pass, then ONE copy of the insertion code per group, run per survivor
          unsigned mk = 0;
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) mk |= (r[8 * q + jj] < thr ? 1u : 0u) << jj;
#pragma unroll 1
          while (mk) {
            const int jj = __ffs(mk) - 1;
            mk &= mk - 1;
            const float lo4 = (jj & 2) ? ((jj & 1) ? r[8 * q + 3] : r[8 * q + 2]) : ((jj & 1) ? r[8 * q + 1] : r[8 * q]);
            const float hi4 = (jj & 2) ? ((jj & 1) ? r[8 * q + 7] : r[8 * q + 6]) : ((jj & 1) ? r[8 * q + 5] : r[8 * q + 4]);
            const float x = (jj & 4) ? hi4 : lo4;
            if (x < thr) {
              buf[cnt] = ((uint64_t)__float_as_uint(x) << 32) | (uint64_t)(pos0 + 8 * q + jj);
              ++cnt;
              float t = x;  // sorted insertion: every slot keeps the smaller of (itself, what is carried)
#pragma unroll
              for (int i = 0; i < TS_RK; ++i) {
                const float lo = fminf(tk[i], t);
                t = fmaxf(tk[i], t);
                tk[i] = lo;
              }
              if (tk[TS_RK - 1] < thr) {
                thr = tk[TS_RK - 1];
                atomicMin(gthr, f32_ordered(thr));  // (result unused: a fire-and-forget reduction)
              }
            }
          }
        } else if constexpr (RANGE) {
#pragma unroll
          for (int j = 8 * q; j < 8 * q + 8; ++j) {
            if (r[j] < thr) {
              if (cnt == cap) {  // full: everything kept lies before this position
                *cut = pos0 + j;
                thr = __int_as_float(0xFF800000);
              } else {
                buf[cnt++] = ((uint64_t)__float_as_uint(r[j]) << 32) | (uint64_t)(pos0 + j);
              }
            }
          }
        } else {
#pragma unroll
          for (int j = 8 * q; j < 8 * q + 8; ++j) {
            const bool hit = r[j] < thr;
            if (hit) buf[cnt] = ((uint64_t)__float_as_uint(r[j]) << 32) | (uint64_t)(pos0 + j);
            cnt += hit ? 1 : 0;
          }
        }
      }
    }
  }
}

// ---- tile-at-a-time selection of the TS kernels -------------------------------------------------------------
// The fast path of a tile must be ONE branch: ncu's source page of the round-1 epilogue showed the ~18 FMNMX3 of a
// 32-column chunk surrounded by ~10 small branches (overflow ballot, tail-column mask, threshold refresh, group
// tests), each with its branch-resolving / reconvergence stall -- ~350 clk per chunk for ~40 useful instructions.
// Here a row's 64 values are reduced to their minimum first (group minima kept), and everything else -- refresh of
// the shared threshold, masking of columns past the end of the shard, compaction, selection -- sits behind a single
// warp-uniform test.
__device__ __forceinline__ float group_min8(const float (&r)[32], int q) {
  return min3(min3(r[8 * q], r[8 * q + 1], r[8 * q + 2]), min3(r[8 * q + 3], r[8 * q + 4], r[8 * q + 5]),
              fminf(r[8 * q + 6], r[8 * q + 7]));
}

// Per-lane selection over one 64-column tile whose group minima are g0[0..3], g1[0..3] (divergent: only lanes that
// hold a survivor work).  A lane walks ITS OWN groups with a survivor (bit mask over the tile's 8 groups) and fetches
// the group's 8 values through three levels of selects, so the warp runs max-over-lanes(groups with a survivor) rounds.
// The first version walked the groups warp-uniformly (static register names, one round for every group in which ANY
// lane had a survivor): in a piece's start-up phase and on short shards nearly every tile has a handful of survivors
// scattered over lanes and groups -- 6-8 rounds of ~115 instructions with one or two lanes active each, where this
// shape needs 1-2 rounds of ~170.  Measured (tools/tc_exp.py, release build): 125 K-row shard 0.678 -> 0.526 ms,
// config 2 3.03 -> 2.82 ms, config 1 0.113 -> 0.086 ms.  The path is hot for the instruction cache and has to stay
// small: ONE copy of the insertion code, walked by bit masks (also measured and rejected: fully unrolled over the 64
// registers -- 40 KB of code, 2 x slower, stall_no_inst -- and a per-thread scratch array in local memory walked with
// dynamic indices -- 3 x slower, the stores delay the next tile's tensor-memory drain).
// RANGE: groups and the values within a group are walked in increasing column order, so the keys are appended in
// position order and a full buffer records its first dropped position in *cut (see epi_process).
template <bool REG, bool RANGE = false>
__device__ __forceinline__ void epi_select_tile(const float (&r0)[32], const float (&r1)[32], const float (&g0)[4],
                                                const float (&g1)[4], uint32_t pos0, uint64_t* buf, int& cnt, float& thr,
                                                float (&tk)[TS_RK], uint32_t* gthr, int cap = 0, uint32_t* cut = nullptr) {
  unsigned gm = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    gm |= (g0[q] < thr ? 1u : 0u) << q;
    gm |= (g1[q] < thr ? 1u : 0u) << (q + 4);
  }
#pragma unroll 1
  while (gm) {
    const int q = __ffs(gm) - 1;
    gm &= gm - 1;
    const bool b0 = q & 1, b1 = q & 2, b2 = q & 4;
    float v[8];
    unsigned mk = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float a = b0 ? r0[8 + j] : r0[j], b = b0 ? r0[24 + j] : r0[16 + j];
      const float c = b0 ? r1[8 + j] : r1[j], d = b0 ? r1[24 + j] : r1[16 + j];
      const float ab = b1 ? b : a, cd = b1 ? d : c;
      v[j] = b2 ? cd : ab;
      mk |= (v[j] < thr ? 1u : 0u) << j;
    }
#pragma unroll 1
    while (mk) {
      const int jj = __ffs(mk) - 1;
      mk &= mk - 1;
      const float lo4 = (jj & 2) ? ((jj & 1) ? v[3] : v[2]) : ((jj & 1) ? v[1] : v[0]);
      const float hi4 = (jj & 2) ? ((jj & 1) ? v[7] : v[6]) : ((jj & 1) ? v[5] : v[4]);
      const float x = (jj & 4) ? hi4 : lo4;
      if constexpr (RANGE) {
        if (cnt == cap) {
          *cut = pos0 + 8 * q + jj;
          thr = __int_as_float(0xFF800000);
          gm = 0;
          break;
        }
      }
      if (!REG || x < thr) {  // (REG: the threshold may have moved since the mask was made)
        buf[cnt] = ((uint64_t)__float_as_uint(x) << 32) | (uint64_t)(pos0 + 8 * q + jj);
        ++cnt;
        if constexpr (REG) {
          float prev = __int_as_float(0xFF800000);
#pragma unroll
          for (int i = 0; i < TS_RK; ++i) {
            const float cur = tk[i];
            tk[i] = fmaxf(prev, fminf(cur, x));
            prev = cur;
          }
          if (tk[TS_RK - 1] < thr) {
            thr = tk[TS_RK - 1];
            atomicMin(gthr, f32_ordered(thr));  // (result unused: a fire-and-forget reduction)
          }
        }
      }
    }
  }
}

struct TcParams {
  int n, nq, n_kb;
  int n_tiles;             // 128-row tiles per query block (whole shard)
  int q_blocks;            // 256-query blocks
  int work_per_cta;        // W: linear (query block, tile) items per CTA
  int total_work;          // q_blocks * n_tiles
  int s_max;               // candidate-buffer pieces per query block
  uint32_t pos_base;
  uint64_t* cand;          // [q_blocks][s_max][256][cap]
  int* cand_cnt;           // [q_blocks][s_max][256]   (zeroed by the host before the launch)
  float* cand_thr;         // [q_blocks][s_max][256]   final threshold (rank domain) of a piece that compacted
  uint32_t* cand_cut;      // range mode, instead of cand_thr: position of the first dropped survivor, 0xFFFFFFFF = none
  int cap, kprime;
  int slack, hwm;          // survivors of a compaction = kprime .. kprime + slack; deferred compaction above hwm keys
  uint32_t* gthr;          // [q_pad] best threshold published per query (shared by all CTAs), 0xFF-filled
  int n_stage;             // shared-memory ring depth
  int a_resident;          // 1: both query tiles stay in shared memory while a piece is scanned (D <= 128)
  int use_nb;              // 1: an extra K=8 step adds |x|^2 (three TF32 pieces x 1.0) inside the MMA (l2)
  int aligned;             // 1: CTA = (segment, query block) with common tile boundaries; 0: equal linear ranges
  int debug;               // NB200_TC_DEBUG bit 0: epilogue drains TMEM without selecting (timing experiments only)
  const int4* pieces;      // pair kernel: [pairs][TS_MAXP] {query block, first tile, end tile, slot} (tc_ts_plan)
};

// Work decomposition: the (query block, database tile) grid is cut into `gridDim.x` equal linear
// ranges, so every SM gets the same number of tiles whatever the batch size; a CTA's range may
// cross into the next query block, in which case it finishes one "piece" and starts another
// (its own operand tiles, thresholds and candidate buffers).
template <int KPL>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_scan_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmN, const __grid_constant__ CUtensorMap tmO, const TcParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // carve: [A resident: 2*n_kb chunks] [ones chunk] [stages: n_stage * stage_bytes] [barriers]
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int a_bytes = p.a_resident ? 2 * p.n_kb * CHUNK_BYTES : 0;
  const int ones_bytes = p.use_nb ? CHUNK_BYTES : 0;
  const int stage_bytes = p.a_resident ? CHUNK_BYTES : 3 * CHUNK_BYTES;  // B [+ A0 + A1]
  unsigned char* smem_a = smem;
  unsigned char* smem_ones = smem + a_bytes;
  unsigned char* smem_st = smem_ones + ones_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_st + (size_t)p.n_stage * stage_bytes);
  uint64_t* full_bar = bars;                   // [n_stage]
  uint64_t* empty_bar = bars + p.n_stage;      // [n_stage]
  uint64_t* tfull_bar = bars + 2 * p.n_stage;  // [2]
  uint64_t* tempty_bar = tfull_bar + 2;        // [2]
  uint64_t* afull_bar = tempty_bar + 2;        // [1] resident A tiles of the current piece have landed
  uint64_t* aempty_bar = afull_bar + 1;        // [1] every MMA of the finished piece has read them
  uint64_t* ones_bar = aempty_bar + 1;         // [1]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ones_bar + 1);

  // the warp index is made provably warp-uniform (shfl), so that the single-thread TMA / MMA issue loops keep
  // their descriptors in uniform registers instead of paying an ELECT + R2UR round trip per instruction
  const int tid = threadIdx.x, warp = __shfl_sync(FULL, tid >> 5, 0), lane = tid & 31;
  const int cta = blockIdx.x;
  // aligned mode: CTA = (segment, query block), every query block is cut at the SAME tile boundaries and
  // CTAs of one segment are neighbours in the grid, so co-resident CTAs sweep the same database tiles
  // at the same time and the L2 serves all but one of them (the database is larger than the L2).
  // linear mode (tiny batches): equal linear ranges of the (query block, tile) grid.
  long w_begin, w_end;
  if (p.aligned) {
    const int qb_a = cta % p.q_blocks, seg = cta / p.q_blocks;
    w_begin = (long)qb_a * p.n_tiles + min((long)seg * p.work_per_cta, (long)p.n_tiles);
    w_end = (long)qb_a * p.n_tiles + min((long)(seg + 1) * p.work_per_cta, (long)p.n_tiles);
  } else {
    w_begin = (long)cta * p.work_per_cta;
    w_end = min(w_begin + (long)p.work_per_cta, (long)p.total_work);
  }
  const int n_kb_all = p.n_kb + p.use_nb;

  if (tid == 0) {
    for (int s = 0; s < p.n_stage; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 256);
    }
    mbar_init(afull_bar, 1);
    mbar_init(aempty_bar, 1);
    mbar_init(ones_bar, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (p.use_nb) prefetch_tmap(&tmN);
  }
  if (warp == 1) tmem_alloc(tmem_holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer (whole warp runs the loop, one elected lane issues) =====================
    if (w_begin < w_end) {
      if (p.use_nb && elect_one()) {
        mbar_expect_tx(ones_bar, CHUNK_BYTES);
        tma_load_2d(&tmO, ones_bar, smem_ones, 0, 0);
      }
      __syncwarp();
      int s = 0;
      uint32_t ph = 0;  // ring position and its phase bit (no division in the hot loop)
      int piece = 0;
      for (long w = w_begin; w < w_end; ++piece) {
        const int qb = (int)(w / p.n_tiles);
        const int t_begin = (int)(w - (long)qb * p.n_tiles);
        const int t_end = (int)min((long)p.n_tiles, t_begin + (w_end - w));
        const int q0 = qb * TC_QB;
        if (p.a_resident) {
          if (piece > 0) mbar_wait(aempty_bar, (piece - 1) & 1);
          if (elect_one()) {
            mbar_expect_tx(afull_bar, (uint32_t)a_bytes);
            for (int h = 0; h < 2; ++h)
              for (int kb = 0; kb < p.n_kb; ++kb)
                tma_load_2d(&tmA, afull_bar, smem_a + (size_t)(h * p.n_kb + kb) * CHUNK_BYTES, kb * TC_KB,
                            q0 + h * TC_BM);
          }
          __syncwarp();
        }
        for (int t = t_begin; t < t_end; ++t) {
          for (int kb = 0; kb < n_kb_all; ++kb) {
            mbar_wait(&empty_bar[s], ph ^ 1);
            unsigned char* st = smem_st + (size_t)s * stage_bytes;
            if (elect_one()) {
              if (NB200_DBG(p.debug, 2)) {  // timing experiment: no database traffic, the MMAs read stale shared memory
                mbar_arrive(&full_bar[s]);
              } else if (kb < p.n_kb) {
                mbar_expect_tx(&full_bar[s], (uint32_t)stage_bytes);
                tma_load_2d(&tmB, &full_bar[s], st, kb * TC_KB, t * TC_BN);
                if (!p.a_resident) {
                  tma_load_2d(&tmA, &full_bar[s], st + CHUNK_BYTES, kb * TC_KB, q0);
                  tma_load_2d(&tmA, &full_bar[s], st + 2 * CHUNK_BYTES, kb * TC_KB, q0 + TC_BM);
                }
              } else {  // the |x|^2 block of this tile
                mbar_expect_tx(&full_bar[s], CHUNK_BYTES);
                tma_load_2d(&tmN, &full_bar[s], st, 0, t * TC_BN);
              }
            }
            __syncwarp();
            if (++s == p.n_stage) {
              s = 0;
              ph ^= 1;
            }
          }
        }
        w += t_end - t_begin;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp runs the loop, one elected lane issues) =====================
    if (w_begin < w_end) {
      constexpr uint32_t idesc = make_idesc_tf32(TC_BM, TC_BN);
      // The issuing lane must keep the tensor pipe fed (8 MMAs of 64 cycles per k-block): everything outside
      // the elected region is warp-uniform, so descriptors live in uniform registers (no ELECT/R2UR loop per
      // MMA), and the loop carries ring position / phase incrementally: no division, no rebuild.
      const uint32_t st_base = smem_u32(smem_st);
      const uint32_t a_base = smem_u32(smem_a);
      const uint64_t d_ones = make_smem_desc(smem_u32(smem_ones));
      const bool a_res = p.a_resident != 0;
      if (p.use_nb) mbar_wait(ones_bar, 0);
      int s = 0;
      uint32_t ph = 0;
      int ti = 0, piece = 0;
      for (long w = w_begin; w < w_end; ++piece) {
        const int qb = (int)(w / p.n_tiles);
        const int t_begin = (int)(w - (long)qb * p.n_tiles);
        const int t_end = (int)min((long)p.n_tiles, t_begin + (w_end - w));
        if (a_res) mbar_wait(afull_bar, piece & 1);
        for (int t = t_begin; t < t_end; ++t, ++ti) {
          const int b = ti & 1;
          mbar_wait(&tempty_bar[b], ((ti >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d0 = tmem_base + (uint32_t)(b * 2 * TC_BN);
          for (int kb = 0; kb < p.n_kb; ++kb) {
            mbar_wait(&full_bar[s], ph);
            tc_fence_after();
            const uint32_t sb = st_base + (uint32_t)s * (uint32_t)stage_bytes;
            const uint64_t db = make_smem_desc(sb);
            const uint64_t da0 = make_smem_desc(a_res ? a_base + (uint32_t)kb * CHUNK_BYTES : sb + CHUNK_BYTES);
            const uint64_t da1 =
                make_smem_desc(a_res ? a_base + (uint32_t)(p.n_kb + kb) * CHUNK_BYTES : sb + 2 * CHUNK_BYTES);
            const uint32_t acc = kb != 0;
            if (elect_one()) {
              if (!NB200_DBG(p.debug, 4)) {  // (bit 2 set: timing experiment without the MMAs, TMA traffic only)
                // UMMA_K = 8 tf32 = 32 bytes inside the 128-byte swizzle row: +2 in the (address >> 4) field
                umma_tf32(tmem_d0, da0, db, idesc, acc);
                umma_tf32(tmem_d0, da0 + 2, db + 2, idesc, 1);
                umma_tf32(tmem_d0, da0 + 4, db + 4, idesc, 1);
                umma_tf32(tmem_d0, da0 + 6, db + 6, idesc, 1);
                umma_tf32(tmem_d0 + TC_BN, da1, db, idesc, acc);
                umma_tf32(tmem_d0 + TC_BN, da1 + 2, db + 2, idesc, 1);
                umma_tf32(tmem_d0 + TC_BN, da1 + 4, db + 4, idesc, 1);
                umma_tf32(tmem_d0 + TC_BN, da1 + 6, db + 6, idesc, 1);
              }
              tc_commit(&empty_bar[s]);  // frees the stage once these MMAs have read it
            }
            __syncwarp();
            if (++s == p.n_stage) {
              s = 0;
              ph ^= 1;
            }
          }
          if (p.use_nb) {  // + 1.0 * (hi + mid + lo pieces of |x|^2): one K=8 step per operand half
            mbar_wait(&full_bar[s], ph);
            tc_fence_after();
            const uint64_t db = make_smem_desc(st_base + (uint32_t)s * (uint32_t)stage_bytes);
            if (elect_one()) {
              umma_tf32(tmem_d0, d_ones, db, idesc, 1);
              umma_tf32(tmem_d0 + TC_BN, d_ones, db, idesc, 1);
              tc_commit(&empty_bar[s]);
            }
            __syncwarp();
            if (++s == p.n_stage) {
              s = 0;
              ph ^= 1;
            }
          }
          if (elect_one()) tc_commit(&tfull_bar[b]);  // accumulators of this tile are complete
          __syncwarp();
        }
        if (a_res) {
          if (elect_one()) tc_commit(aempty_bar);  // the resident operand tiles may be overwritten
          __syncwarp();
        }
        w += t_end - t_begin;
      }
    }
  } else {
    // ===================== epilogue: 8 warps (2 per scheduler), thread == one query row ==========
    // Warps 2-5 read operand half 0, warps 6-9 half 1; a warp may only touch the TMEM lane quarter
    // (warp index % 4).  The warps never synchronise with each other.  The accumulator already holds
    // the rank (bias folded into the MMA), so the fast path is: tcgen05.ld, min tree, one compare
    // (epi_process: append buffer + warp-cooperative compaction, thresholds shared between CTAs).
    const int e = warp - 2;
    const int h = e >> 2;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;       // row inside the 128-query half
    const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16);
    float tk_unused[TS_RK] = {};               // (the register list is a mode of the TS kernel only)
    unsigned ctr[4] = {0, 0, 0, 0};

    int ti = 0;
    for (long w = w_begin; w < w_end;) {
      const int qb = (int)(w / p.n_tiles);
      const int t_begin = (int)(w - (long)qb * p.n_tiles);
      const int t_end = (int)min((long)p.n_tiles, t_begin + (w_end - w));
      // piece slot of this CTA inside query block qb
      const int first_cta = (int)(((long)qb * p.n_tiles) / p.work_per_cta);
      const size_t unit = (size_t)qb * p.s_max + (p.aligned ? cta / p.q_blocks : cta - first_cta);
      const bool row_valid = qb * TC_QB + h * TC_BM + row < p.nq;
      uint64_t* buf = p.cand + (unit * TC_QB + h * TC_BM + row) * (size_t)p.cap;
      uint32_t* gthr = p.gthr + (qb * TC_QB + h * TC_BM + row);
      int cnt = 0;
      float thr = row_valid ? __int_as_float(0x7F800000) : __int_as_float(0xFF800000);
      for (int tile = t_begin; tile < t_end; ++tile, ++ti) {
        const int b = ti & 1;
        mbar_wait(&tfull_bar[b], (ti >> 1) & 1);
        tc_fence_after();
        const uint32_t tcol = trow + (uint32_t)((b * 2 + h) * TC_BN);
        const uint32_t pos_tile = p.pos_base + (uint32_t)(tile * TC_BN);
        const int vtile = p.n - tile * TC_BN;  // >= 128 except in the last tile
        uint32_t v0[32], v1[32];
        if (NB200_DBG(p.debug, 1)) {  // timing experiment: touch the accumulators, select nothing
          tmem_ld32(tcol, v0);
          tmem_ld_wait();
          if (__uint_as_float(v0[0]) == 1.2345e-30f) thr = 0.f;
          tc_fence_before();
          mbar_arrive(&tempty_bar[b]);
          continue;
        }
        // what the other pieces of this query have found in the meantime (fminf ignores the NaN of "nothing yet")
        if (((tile - t_begin) & 7) == 0 && row_valid) thr = fminf(thr, f32_from_ordered(*gthr));
        tmem_ld32(tcol, v0);
#pragma unroll 1
        for (int cp = 0; cp < TC_BN / 64; ++cp) {  // two chunks per iteration, next load in flight while computing
          tmem_ld_wait();
          tmem_ld32(tcol + (uint32_t)(cp * 64 + 32), v1);
          epi_process<KPL, false>(v0, pos_tile + cp * 64, vtile - cp * 64, buf, cnt, thr, tk_unused, p.cap, p.kprime,
                                  p.slack, gthr, lane, ctr);
          tmem_ld_wait();
          if (cp + 1 < TC_BN / 64) tmem_ld32(tcol + (uint32_t)(cp * 64 + 64), v0);
          epi_process<KPL, false>(v1, pos_tile + cp * 64 + 32, vtile - cp * 64 - 32, buf, cnt, thr, tk_unused, p.cap,
                                  p.kprime, p.slack, gthr, lane, ctr);
        }
        tc_fence_before();
        mbar_arrive(&tempty_bar[b]);
        // deferred compaction, one row per warp and tile (the TMEM buffer is already released)
        const unsigned pend = __ballot_sync(FULL, cnt > p.hwm);
        if (pend) compact_lane<KPL>(__ffs(pend) - 1, buf, cnt, thr, p.kprime, p.slack, gthr, lane);
      }
      // publish this piece's per-row candidate count and final threshold
      const size_t slot = unit * TC_QB + h * TC_BM + row;
      p.cand_cnt[slot] = row_valid ? cnt : 0;
      p.cand_thr[slot] = thr;
      w += t_end - t_begin;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------- K1 for long rows on CTA PAIRS (cta_group::2)
// Same contract as tc_scan_kernel, for rows of more than 128 floats.  Measured on the config-5 shape
// (profiles/README.md): the single-CTA kernel streams 48 KB (16 KB of database + 32 KB of query tile) through
// the L2 for every 8 M128 x N128 x K8 MMAs, which is what bounds it (~12 TB/s chip-wide), and with both operands
// in shared memory each of those MMAs takes 96 cycles instead of 64 because the operand reads saturate the
// shared-memory port.  A CTA pair (two SMs of one TPC) issues ONE M256 x N256 x K8 MMA for both SMs:
//   * CTA r holds query rows [r*128, r*128+128) of the 256-query block (A) and database rows
//     [t*256 + r*128, +128) of the 256-row tile (its half of B); the tensor cores read B from both SMs, so a
//     k-block costs each SM 16 KB + 16 KB from the L2 instead of 48 KB for the same number of MACs, and each
//     MMA reads 8 KB of shared memory per SM for twice the work;
//   * accumulators: 128 lanes x 256 columns per SM, two buffers = the whole tensor memory;
//   * only the leader (cluster rank 0) issues MMAs; both CTAs issue their own TMA loads, which signal the
//     LEADER's full barrier; the leader's commits are multicast to both CTAs' empty / tfull barriers; the
//     epilogue warps of both CTAs release an accumulator buffer by arriving on the leader's tempty barrier.
// The epilogue is the one of tc_scan_kernel: thread = query row, warps 2-5 select over columns 0-127 and warps
// 6-9 over columns 128-255 of the tile, each (row, column half) with its own candidate list.
constexpr int TP_BN = 256;  // database rows per pair tile
constexpr int TS_MAXP = 8;  // pieces per CTA (or CTA pair) in a plan table (tc_ts_plan)

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
// Remote arrival with the default semantics (.release at CTA scope), as CUTLASS' ClusterBarrier::arrive does: what
// the barriers of this kernel hand over lives in tensor memory / the async proxy and is ordered by the tcgen05
// fences and the TMA transaction counts.  (.release.cluster / .acquire.cluster made every arrival and every wait an
// L1 invalidation -- CCTL.IVALL + ERRBAR were 45 % of all warp samples in the first version's ncu source page.)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// this CTA's box into its own shared memory, completion bytes on the barrier at cluster address `bar_cluster`
__device__ __forceinline__ void tma_load_2d_2sm(const CUtensorMap* map, uint32_t bar_cluster, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void umma_tf32_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// TcParams as for tc_scan_kernel with: pieces = the host-made table of (query block, 256-row tile range, slot) per
// PAIR (blockIdx.x / 2; tc_ts_plan over sm_count / 2 units), s_max = candidate lists per query block = 2 x slots.
// RANGE: batched range queries -- every row's threshold is its query's T_q (p.gthr, filled by tc_range_threshold),
// no compaction; a list whose buffer fills stores the position of its first dropped survivor in p.cand_cut.
template <int KPL, bool RANGE = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
tc_scan_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmN, const __grid_constant__ CUtensorMap tmO, const TcParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // carve: [ones chunk] [stages: n_stage * (B half + A half)] [barriers]  (identical offsets in both CTAs)
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int ones_bytes = p.use_nb ? CHUNK_BYTES : 0;
  constexpr int stage_bytes = 2 * CHUNK_BYTES;
  unsigned char* smem_ones = smem;
  unsigned char* smem_st = smem + ones_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_st + (size_t)p.n_stage * stage_bytes);
  uint64_t* full_bar = bars;                   // [n_stage] leader: both CTAs' loads of the stage have landed
  uint64_t* empty_bar = bars + p.n_stage;      // [n_stage] each CTA: the MMAs have read the stage
  uint64_t* tfull_bar = bars + 2 * p.n_stage;  // [2] each CTA: accumulators of a tile are complete
  uint64_t* tempty_bar = tfull_bar + 2;        // [2] leader: both CTAs' epilogue warps have drained the buffer
  uint64_t* ones_bar = tempty_bar + 2;         // [1]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ones_bar + 1);

  const int tid = threadIdx.x, warp = __shfl_sync(FULL, tid >> 5, 0), lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1;
  const int4* my_pieces = p.pieces + (size_t)pair * TS_MAXP;  // host-made table: every pair gets the same number of tiles
  const int n_kb_all = p.n_kb + p.use_nb;

  if (tid == 0) {
    for (int s = 0; s < p.n_stage; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 16);  // 8 epilogue warps of each CTA
    }
    mbar_init(ones_bar, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (p.use_nb) prefetch_tmap(&tmN);
  }
  __syncthreads();
  cluster_sync_all();  // both CTAs' barriers exist before anything remote touches them
  if (warp == 1) tmem_alloc_2sm(tmem_holder, 512);
  if (warp == 0 && p.use_nb) {  // the constant tile of ones (A operand of the |x|^2 step), one copy per CTA
    if (elect_one()) {
      mbar_expect_tx(ones_bar, CHUNK_BYTES);
      tma_load_2d(&tmO, ones_bar, smem_ones, 0, 0);
    }
    __syncwarp();
    mbar_wait(ones_bar, 0);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // tensor memory allocated and the ones tiles resident in BOTH CTAs before the first MMA
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs; completion bytes go to the leader's full barrier) ==========
    {
      int s = 0;
      uint32_t ph = 0;
      for (int pi = 0; pi < TS_MAXP; ++pi) {
        const int4 pc = my_pieces[pi];
        if (pc.x < 0) break;
        const int qb = pc.x, t_begin = pc.y, t_end = pc.z;
        const int q0 = qb * TC_QB + (int)rank * TC_BM;
        for (int t = t_begin; t < t_end; ++t) {
          const int r0 = t * TP_BN + (int)rank * TC_BM;
          for (int kb = 0; kb < n_kb_all; ++kb) {
            mbar_wait(&empty_bar[s], ph ^ 1);
            unsigned char* st = smem_st + (size_t)s * stage_bytes;
            const uint32_t fb = mapa_cluster(smem_u32(&full_bar[s]), 0);
            if (elect_one()) {
              if (kb < p.n_kb) {
                if (leader) mbar_expect_tx(&full_bar[s], 2u * (uint32_t)stage_bytes);
                tma_load_2d_2sm(&tmB, fb, st, kb * TC_KB, r0);
                tma_load_2d_2sm(&tmA, fb, st + CHUNK_BYTES, kb * TC_KB, q0);
              } else {  // the |x|^2 block of this CTA's half of the tile
                if (leader) mbar_expect_tx(&full_bar[s], 2u * (uint32_t)CHUNK_BYTES);
                tma_load_2d_2sm(&tmN, fb, st, 0, r0);
              }
            }
            __syncwarp();
            if (++s == p.n_stage) {
              s = 0;
              ph ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      constexpr uint32_t idesc = make_idesc_tf32(2 * TC_BM, TP_BN);
      const uint32_t st_base = smem_u32(smem_st);
      const uint64_t d_ones = make_smem_desc(smem_u32(smem_ones));
      int s = 0;
      uint32_t ph = 0;
      int ti = 0;
      for (int pi = 0; pi < TS_MAXP; ++pi) {
        const int4 pc = my_pieces[pi];
        if (pc.x < 0) break;
        const int t_begin = pc.y, t_end = pc.z;
        for (int t = t_begin; t < t_end; ++t, ++ti) {
          const int b = ti & 1;
          mbar_wait(&tempty_bar[b], ((ti >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d0 = tmem_base + (uint32_t)(b * TP_BN);
          for (int kb = 0; kb < p.n_kb; ++kb) {
            mbar_wait(&full_bar[s], ph);
            tc_fence_after();
            const uint32_t sb = st_base + (uint32_t)s * (uint32_t)stage_bytes;
            const uint64_t db = make_smem_desc(sb);
            const uint64_t da = make_smem_desc(sb + CHUNK_BYTES);
            const uint32_t acc = kb != 0;
            if (elect_one()) {
              umma_tf32_2sm(tmem_d0, da, db, idesc, acc);
              umma_tf32_2sm(tmem_d0, da + 2, db + 2, idesc, 1);
              umma_tf32_2sm(tmem_d0, da + 4, db + 4, idesc, 1);
              umma_tf32_2sm(tmem_d0, da + 6, db + 6, idesc, 1);
              tc_commit_2sm(&empty_bar[s], 3);  // frees the stage in both CTAs once these MMAs have read it
            }
            __syncwarp();
            if (++s == p.n_stage) {
              s = 0;
              ph ^= 1;
            }
          }
          if (p.use_nb) {  // + 1.0 * (hi + mid + lo pieces of |x|^2)
            mbar_wait(&full_bar[s], ph);
            tc_fence_after();
            const uint64_t db = make_smem_desc(st_base + (uint32_t)s * (uint32_t)stage_bytes);
            if (elect_one()) {
              umma_tf32_2sm(tmem_d0, d_ones, db, idesc, 1);
              tc_commit_2sm(&empty_bar[s], 3);
            }
            __syncwarp();
            if (++s == p.n_stage) {
              s = 0;
              ph ^= 1;
            }
          }
          if (elect_one()) tc_commit_2sm(&tfull_bar[b], 3);  // accumulators of this tile are complete, in both CTAs
          __syncwarp();
        }
      }
    }
  } else {
    // ===================== epilogue: 8 warps per CTA, thread == one query row x one column half ==========
    const int e = warp - 2;
    const int ch = e >> 2;                     // column half of the 256-row tile
    const int quarter = warp & 3;              // TMEM lane quarter this warp may touch
    const int row = quarter * 32 + lane;       // row inside this CTA's 128 queries
    const int row_in_block = (int)rank * TC_BM + row;
    const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t te_addr0 = mapa_cluster(smem_u32(&tempty_bar[0]), 0), te_addr1 = mapa_cluster(smem_u32(&tempty_bar[1]), 0);
    float tk_unused[TS_RK] = {};
    unsigned ctr[4] = {0, 0, 0, 0};

    int ti = 0;
    for (int pi = 0; pi < TS_MAXP; ++pi) {
      const int4 pc = my_pieces[pi];
      if (pc.x < 0) break;
      const int qb = pc.x, t_begin = pc.y, t_end = pc.z;
      const size_t unit = (size_t)qb * p.s_max + 2 * pc.w + ch;
      const bool row_valid = qb * TC_QB + row_in_block < p.nq;
      uint64_t* buf = p.cand + (unit * TC_QB + row_in_block) * (size_t)p.cap;
      uint32_t* gthr = p.gthr + (qb * TC_QB + row_in_block);
      int cnt = 0;
      float thr = !row_valid ? __int_as_float(0xFF800000) : RANGE ? f32_from_ordered(*gthr) : __int_as_float(0x7F800000);
      uint32_t cut = 0xFFFFFFFFu;
      for (int tile = t_begin; tile < t_end; ++tile, ++ti) {
        const int b = ti & 1;
        mbar_wait(&tfull_bar[b], (ti >> 1) & 1);
        tc_fence_after();
        const uint32_t tcol = trow + (uint32_t)(b * TP_BN + ch * TC_BN);
        const uint32_t pos_tile = p.pos_base + (uint32_t)(tile * TP_BN + ch * TC_BN);
        const int vtile = p.n - tile * TP_BN - ch * TC_BN;  // >= 128 except at the end of the shard
        uint32_t v0[32], v1[32];
        if (NB200_DBG(p.debug, 1)) {  // timing experiment: touch the accumulators, select nothing
          tmem_ld32(tcol, v0);
          tmem_ld_wait();
          if (__uint_as_float(v0[0]) == 1.2345e-30f) thr = 0.f;
        } else {
          if (((tile - t_begin) & 7) == 0 && row_valid) thr = fminf(thr, f32_from_ordered(*gthr));
          tmem_ld32(tcol, v0);
#pragma unroll 1
          for (int cp = 0; cp < TC_BN / 64; ++cp) {
            tmem_ld_wait();
            tmem_ld32(tcol + (uint32_t)(cp * 64 + 32), v1);
            epi_process<KPL, false, RANGE>(v0, pos_tile + cp * 64, vtile - cp * 64, buf, cnt, thr, tk_unused, p.cap,
                                           p.kprime, p.slack, gthr, lane, ctr, &cut);
            tmem_ld_wait();
            if (cp + 1 < TC_BN / 64) tmem_ld32(tcol + (uint32_t)(cp * 64 + 64), v0);
            epi_process<KPL, false, RANGE>(v1, pos_tile + cp * 64 + 32, vtile - cp * 64 - 32, buf, cnt, thr, tk_unused,
                                           p.cap, p.kprime, p.slack, gthr, lane, ctr, &cut);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(b ? te_addr1 : te_addr0);  // this warp is done with the buffer (one arrival per warp)
        if (!RANGE && !NB200_DBG(p.debug, 1)) {
          const unsigned pend = __ballot_sync(FULL, cnt > p.hwm);
          if (pend) compact_lane<KPL>(__ffs(pend) - 1, buf, cnt, thr, p.kprime, p.slack, gthr, lane);
        }
      }
      const size_t slot = unit * TC_QB + row_in_block;
      p.cand_cnt[slot] = row_valid ? cnt : 0;
      if constexpr (RANGE) p.cand_cut[slot] = cut;
      else p.cand_thr[slot] = thr;
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer's MMAs / loads / arrivals that touch this CTA are all done
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ---------------------------------------------------------------- K1 for D <= 128: A operand in tensor memory
// Same contract as tc_scan_kernel, different data path.  Measured on config 2 (profiles/README.md): with both
// operands in shared memory an M=128 x N=128 x K=8 TF32 MMA takes ~96 cycles instead of the 64-cycle floor
// (operand reads saturate the shared-memory port); with A in tensor memory it takes ~76.  So for rows of at
// most 128 floats the CTA's 256 prepared queries live in TMEM for the whole piece:
//   TMEM columns [0,128) A of half 0, [128,256) A of half 1 (thread = lane = query row, one column per
//   float; written by the epilogue threads with tcgen05.st straight from the query rows in HBM, scaled),
//   [256,512) two accumulator buffers x two halves x 64 columns.
// Shared memory then holds nothing but database tiles: one stage = one whole 64-row tile (all k-blocks + the
// |x|^2 block), so there is ONE full/empty handshake per tile and ~200 KB of loads in flight per SM.
// The |x|^2 step keeps its A operand (the constant tile of ones) in shared memory: 2 of 34 MMAs per tile.
constexpr int TS_BN = 64;                 // database rows per tile
constexpr int TS_CHUNK = TS_BN * 128;     // 8 KB: 64 rows x one 128-byte k-block
constexpr int TS_ACC0 = 256;              // first accumulator column
constexpr int TS_THREADS = 352;           // warps: 0 TMA producer, 1 MMA issuer (half 0), 2-9 epilogue, 10 MMA issuer (half 1)
constexpr int TS_MMA_WARP2 = 10;


struct TsParams {
  int n, nq, n_kb;
  int s_max;
  const int4* pieces;      // [n_cta][TS_MAXP] {query block, first tile, end tile, slot}; query block < 0 ends the list
  uint32_t pos_base;
  uint64_t* cand;
  int* cand_cnt;
  float* cand_thr;
  uint32_t* cand_cut;      // range mode (see TcParams)
  int cap, kprime, slack, hwm, n_stage, use_nb, debug;
  int warm_max;            // tiles of the warm start (0 when kprime > 32: the 32 column classes bound only the 32nd best)
  int refresh_mask;        // the shared threshold is re-read every (mask + 1) tiles
  uint32_t* gthr;          // [q_pad] ordered bits of the best threshold any piece has published (0xFFFFFFFF = none)
  const float* q;          // [q_pad][row_words] original queries (zero padded rows)
  int row_words;
  float scale;             // A' = scale * q
  int* inexact_flag;       // set when a valid query row is not TF32-exact
  unsigned long long* counters;  // NB200_TC_COUNT diagnostics: [0] appended keys, [1] hit rounds, [2] compactions,
                                 // [3] deferred compactions, [4] chunks; NULL = off
};

// Warm start of a piece: its first ts_warm_tiles() tiles are scanned twice.  The first time nothing is selected:
// each row only keeps the minimum of every column class (column mod 32) in 32 registers; the largest of these 32
// minima bounds the row's 32nd best rank from above (32 distinct points are at least as good), so it is a valid
// starting threshold -- at about the 3 % quantile after 4096 columns -- bought with min/max instructions only.
// Starting from +inf instead costs ~6 warp-cooperative compactions per row within the first 10 K columns, all
// rows of a warp at the same time, and each of them stalls the two-deep accumulator ring.
__device__ __forceinline__ int ts_warm_tiles(int warm_max, int len) {
  return len >= 64 ? min(warm_max, len >> 3) : 0;
}

// one 32-column chunk of one row: fast path = min tree + one compare; survivors are appended to the row's
// buffer, a full buffer is compacted warp-cooperatively first (see compact_row).
// RANGE: batched range queries (fixed per-query thresholds from p.gthr, no compaction, no warm start: the host sets
// warm_max = 0); a full buffer records its first dropped position in p.cand_cut and stops selecting.
template <int KPL, bool REG, bool RANGE = false>
__global__ void __launch_bounds__(TS_THREADS, 1)
tc_scan_ts_kernel(const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmN,
                  const __grid_constant__ CUtensorMap tmO, const TsParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int ones_bytes = p.use_nb ? CHUNK_BYTES : 0;
  const int stage_bytes = (p.n_kb + p.use_nb) * TS_CHUNK;
  unsigned char* smem_ones = smem;
  unsigned char* smem_st = smem + ones_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_st + (size_t)p.n_stage * stage_bytes);
  uint64_t* full_bar = bars;                   // [n_stage] a whole tile has landed
  uint64_t* empty_bar = bars + p.n_stage;      // [n_stage] every MMA of the tile has read it
  uint64_t* tfull_bar = bars + 2 * p.n_stage;  // [2 buffers][2 halves] a half's accumulators of a tile are complete
  uint64_t* tempty_bar = tfull_bar + 4;        // [2][2] ... drained (the 4 warps of that half): the halves run decoupled,
                                               // a warp that is busy selecting only holds up its own half's issuer
  uint64_t* afull_bar = tempty_bar + 4;        // [1] the piece's query rows are in tensor memory (256 threads)
  uint64_t* ones_bar = afull_bar + 1;          // [1]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(ones_bar + 1);

  const int tid = threadIdx.x, warp = __shfl_sync(FULL, tid >> 5, 0), lane = tid & 31;
  // this CTA's work: a short list of pieces = (query block, tile range) made by the host (tc_ts_plan)
  const int4* my_pieces = p.pieces + (size_t)blockIdx.x * TS_MAXP;

  if (tid == 0) {
    for (int s = 0; s < p.n_stage; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 2);   // one commit from each MMA issuer
    }
    for (int b = 0; b < 2; ++b) {
      for (int hh = 0; hh < 2; ++hh) {
        mbar_init(&tfull_bar[b * 2 + hh], 1);
        mbar_init(&tempty_bar[b * 2 + hh], 4);
      }
    }
    mbar_init(afull_bar, 256);
    mbar_init(ones_bar, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmB);
    if (p.use_nb) prefetch_tmap(&tmN);
  }
  if (warp == 1) tmem_alloc(tmem_holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer: one whole tile per stage =====================
    {
      if (p.use_nb && elect_one()) {
        mbar_expect_tx(ones_bar, CHUNK_BYTES);
        tma_load_2d(&tmO, ones_bar, smem_ones, 0, 0);
      }
      __syncwarp();
      int s = 0;
      uint32_t ph = 0;
      [[maybe_unused]] unsigned long long c_wait = 0, c_all = 0;
      NB_T0(tp);
      for (int pi = 0; pi < TS_MAXP; ++pi) {
        const int4 pc = __ldg(my_pieces + pi);
        if (pc.x < 0) break;
        const int t_begin = pc.y, len = pc.z - pc.y;
        const int wa = ts_warm_tiles(p.warm_max, len);
        for (int idx = -wa; idx < len; ++idx) {
          const int t = t_begin + (idx < 0 ? idx + wa : idx);
          NB_TACC(c_all, tp);
          mbar_wait(&empty_bar[s], ph ^ 1);
          NB_TACC(c_wait, tp);
          unsigned char* st = smem_st + (size_t)s * stage_bytes;
          if (elect_one()) {
            if (NB200_DBG(p.debug, 2)) {  // timing experiment: no database traffic
              mbar_arrive(&full_bar[s]);
            } else {
              mbar_expect_tx(&full_bar[s], (uint32_t)stage_bytes);
              for (int kb = 0; kb < p.n_kb; ++kb)
                tma_load_2d(&tmB, &full_bar[s], st + kb * TS_CHUNK, kb * TC_KB, t * TS_BN);
              if (p.use_nb) tma_load_2d(&tmN, &full_bar[s], st + p.n_kb * TS_CHUNK, 0, t * TS_BN);
            }
          }
          __syncwarp();
          if (++s == p.n_stage) {
            s = 0;
            ph ^= 1;
          }
        }
      }
#ifdef NB200_EXPERIMENTS
      if (p.counters && lane == 0) {
        atomicAdd(p.counters + 8, c_wait);
        atomicAdd(p.counters + 9, c_all + c_wait);
      }
#endif
    }
  } else if (warp == 1 || warp == TS_MMA_WARP2) {
    // ===================== MMA issuers: one warp per 128-query half =====================
    // A single thread cannot issue N = 64 MMAs fast enough: cycle accounting (profiles/README.md, round 2) showed the
    // one issuer busy 84 % of the time at ~40 clk per MMA against the 32 clk the tensor pipe needs (tools/tc_peak.cu
    // reaches 32.0 with a bare loop), while the pipe was active 54 %.  Two issuers on different SM sub-partitions,
    // each owning one half's accumulators, halve the instructions per thread; stage / accumulator barriers count
    // one commit from each.
    {
      constexpr uint32_t idesc = make_idesc_tf32(TC_BM, TS_BN);
      const int hh = warp == 1 ? 0 : 1;
      const uint32_t st_base = smem_u32(smem_st);
      const uint64_t d_ones = make_smem_desc(smem_u32(smem_ones));
      const uint32_t a_half = tmem_base + (uint32_t)(hh * 128);
      if (p.use_nb) mbar_wait(ones_bar, 0);
      int s = 0;
      uint32_t ph = 0;
      int ti = 0;
      [[maybe_unused]] unsigned long long c_afull = 0, c_tempty = 0, c_full = 0, c_issue = 0;
      NB_T0(tm);
      for (int pi = 0; pi < TS_MAXP; ++pi) {
        const int4 pc = __ldg(my_pieces + pi);
        if (pc.x < 0) break;
        const int n_iter = (pc.z - pc.y) + ts_warm_tiles(p.warm_max, pc.z - pc.y);
        NB_TACC(c_issue, tm);
        mbar_wait(afull_bar, pi & 1);
        NB_TACC(c_afull, tm);
        tc_fence_after();
        for (int it = 0; it < n_iter; ++it, ++ti) {
          const int b = ti & 1;
          NB_TACC(c_issue, tm);
          mbar_wait(&tempty_bar[b * 2 + hh], ((ti >> 1) & 1) ^ 1);
          NB_TACC(c_tempty, tm);
          mbar_wait(&full_bar[s], ph);
          NB_TACC(c_full, tm);
          tc_fence_after();
          const uint32_t d = tmem_base + (uint32_t)(TS_ACC0 + (b * 2 + hh) * TS_BN);
          const uint32_t sb = st_base + (uint32_t)s * (uint32_t)stage_bytes;
          if (elect_one()) {
            if (!NB200_DBG(p.debug, 4)) {
              for (int kb = 0; kb < p.n_kb; ++kb) {
                const uint64_t db = make_smem_desc(sb + (uint32_t)kb * TS_CHUNK);
                const uint32_t a = a_half + (uint32_t)(kb * TC_KB);
                // UMMA_K = 8 tf32: 8 TMEM columns of A, 32 bytes (+2 in the descriptor) of B
                umma_tf32_ts(d, a, db, idesc, kb != 0);
                umma_tf32_ts(d, a + 8, db + 2, idesc, 1);
                umma_tf32_ts(d, a + 16, db + 4, idesc, 1);
                umma_tf32_ts(d, a + 24, db + 6, idesc, 1);
              }
              if (p.use_nb && !NB200_DBG(p.debug, 128))  // + 1.0 * (hi + mid + lo pieces of |x|^2)
                umma_tf32(d, d_ones, make_smem_desc(sb + (uint32_t)p.n_kb * TS_CHUNK), idesc, 1);
            }
            tc_commit(&empty_bar[s]);   // the stage may be refilled once both issuers' MMAs have read it
            tc_commit(&tfull_bar[b * 2 + hh]);   // this half's accumulators of the tile are complete
          }
          __syncwarp();
          if (++s == p.n_stage) {
            s = 0;
            ph ^= 1;
          }
        }
      }
#ifdef NB200_EXPERIMENTS
      NB_TACC(c_issue, tm);
      if (p.counters && lane == 0 && hh == 0) {
        atomicAdd(p.counters + 10, c_afull);
        atomicAdd(p.counters + 11, c_tempty);
        atomicAdd(p.counters + 12, c_full);
        atomicAdd(p.counters + 13, c_issue);
      }
#endif
    }
  } else {
    // ===================== epilogue: 8 warps, thread == one query row =====================
    const int e = warp - 2;
    const int h = e >> 2;
    const int quarter = warp & 3;
    [[maybe_unused]] unsigned long long c_twait = 0, c_drain = 0, c_proc = 0, c_setup = 0;
    NB_T0(te);
    const int row = quarter * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16);
    unsigned ctr[4] = {0, 0, 0, 0};
    int ti = 0;
    for (int pi = 0; pi < TS_MAXP; ++pi) {
      const int4 pc = __ldg(my_pieces + pi);
      if (pc.x < 0) break;
      const int qb = pc.x, t_begin = pc.y, t_end = pc.z;
      const size_t unit = (size_t)qb * p.s_max + pc.w;
      const int qrow = qb * TC_QB + h * TC_BM + row;
      const bool row_valid = qrow < p.nq;
      uint64_t* buf = p.cand + (unit * TC_QB + h * TC_BM + row) * (size_t)p.cap;
      uint32_t* gthr = p.gthr + qrow;
      int cnt = 0;
      float thr = !row_valid ? __int_as_float(0xFF800000) : RANGE ? f32_from_ordered(*gthr) : __int_as_float(0x7F800000);
      uint32_t cut = 0xFFFFFFFFu;
      float tk[TS_RK];
#pragma unroll
      for (int i = 0; i < TS_RK; ++i) tk[i] = __int_as_float(0x7F800000);
      {
        // This piece's operand rows: HBM -> registers -> tensor memory.  Every MMA of the previous piece has
        // completed (this thread has seen the tfull of its last tile), so the columns may be overwritten.
        const float4* src = reinterpret_cast<const float4*>(p.q + (size_t)qrow * p.row_words);
        unsigned bad = 0;
        for (int kb = 0; kb < p.n_kb; ++kb) {
          uint32_t v[32];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 f = __ldg(src + kb * 8 + i);
            bad |= (__float_as_uint(f.x) | __float_as_uint(f.y) | __float_as_uint(f.z) | __float_as_uint(f.w)) & 0x1FFFu;
            v[4 * i] = __float_as_uint(f.x * p.scale);
            v[4 * i + 1] = __float_as_uint(f.y * p.scale);
            v[4 * i + 2] = __float_as_uint(f.z * p.scale);
            v[4 * i + 3] = __float_as_uint(f.w * p.scale);
          }
          tmem_st32(trow + (uint32_t)(h * 128 + kb * TC_KB), v);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(afull_bar);
        if (!row_valid) bad = 0;
        if (__any_sync(FULL, bad != 0) && lane == 0) atomicOr(p.inexact_flag, 1);
      }
      const int len = t_end - t_begin;
      const int wa = ts_warm_tiles(p.warm_max, len);
      // wait for a tile's accumulators, pull this row's 64 columns into registers and hand the buffer back to
      // the tensor core at once (a warp inside a compaction must not hold up the other seven and the MMA)
      NB_TACC(c_setup, te);
      auto drain = [&](uint32_t (&v0)[32], uint32_t (&v1)[32]) {
        const int b = ti & 1;
        NB_TACC(c_proc, te);
        mbar_wait(&tfull_bar[b * 2 + h], (ti >> 1) & 1);
        NB_TACC(c_twait, te);
        tc_fence_after();
        const uint32_t tcol = trow + (uint32_t)(TS_ACC0 + (b * 2 + h) * TS_BN);
        tmem_ld64(tcol, v0, v1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[b * 2 + h]);
        ++ti;
        NB_TACC(c_drain, te);
      };
      if (wa > 0) {  // warm start (see ts_warm_tiles)
        float gm[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) gm[j] = __int_as_float(0x7F800000);
        for (int i = 0; i < wa; ++i) {
          uint32_t v0[32], v1[32];
          drain(v0, v1);
          const int vtile = p.n - (t_begin + i) * TS_BN;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float a = j < vtile ? __uint_as_float(v0[j]) : __int_as_float(0x7F800000);
            const float c = j + 32 < vtile ? __uint_as_float(v1[j]) : __int_as_float(0x7F800000);
            gm[j] = min3(gm[j], a, c);
          }
        }
        float t = gm[0];
#pragma unroll
        for (int j = 1; j < 32; ++j) t = fmaxf(t, gm[j]);
        if (row_valid && !NB200_DBG(p.debug, 1)) thr = publish_thr(gthr, f32_ordered(t));
      }
      // a row above this many keys sends its warp to the slow path (RANGE: a full row has stopped selecting)
      const int guard = RANGE ? p.cap : REG ? p.cap - TS_BN - 1 : p.hwm;
      for (int tile = t_begin; tile < t_end; ++tile) {
        uint32_t v0[32], v1[32];
        drain(v0, v1);
        if (NB200_DBG(p.debug, 1)) {  // timing experiment: select nothing
          if (__uint_as_float(v0[0]) == 1.2345e-30f || __uint_as_float(v1[0]) == 1.2345e-30f) thr = 0.f;
          continue;
        }
        float r0[32], r1[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          r0[j] = __uint_as_float(v0[j]);
          r1[j] = __uint_as_float(v1[j]);
        }
        float g0[4], g1[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          g0[q] = group_min8(r0, q);
          g1[q] = group_min8(r1, q);
        }
        const float m = fminf(min3(g0[0], g0[1], g0[2]), min3(g0[3], g1[0], g1[1]));
        const float mm = min3(m, g1[2], g1[3]);
        const int vtile = p.n - tile * TS_BN;
        // warp-uniform reasons to leave the fast path: threshold refresh (every refresh_mask + 1 tiles), the shard's
        // last, partial tile; per-lane reasons: a value below the row's threshold, a buffer close to its limit
        const bool uni = (((tile - t_begin) & p.refresh_mask) == 0) | (vtile < TS_BN) | (NB200_DBG(p.debug, 64) != 0);
        const bool mine = (mm < thr) | (cnt > guard);
        if (!uni && !__any_sync(FULL, mine)) continue;
        // ------------------------------------------------------------------ slow path
        // what the other pieces of this query have found in the meantime (fminf ignores the NaN of "nothing yet")
        if (((tile - t_begin) & p.refresh_mask) == 0 && row_valid) thr = fminf(thr, f32_from_ordered(*gthr));
        if (NB200_DBG(p.debug, 64)) thr = __int_as_float(0xFF800000);  // timing experiment: nothing passes
        if (vtile < TS_BN) {  // rows past the end of the shard: never candidates
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (j >= vtile) r0[j] = __int_as_float(0x7F800000);
            if (j + 32 >= vtile) r1[j] = __int_as_float(0x7F800000);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            g0[q] = group_min8(r0, q);
            g1[q] = group_min8(r1, q);
          }
        }
        unsigned need = RANGE ? 0u : __ballot_sync(FULL, cnt > p.cap - TS_BN - 1);
        while (need) {  // about to overflow: compact at once (!REG: normally the deferred path keeps rows far from here)
          ++ctr[2];
          const int src = __ffs(need) - 1;
          need &= need - 1;
          const float keep = thr;
          compact_lane<KPL>(src, buf, cnt, thr, p.kprime, p.slack, gthr, lane);
          if (REG) thr = fminf(thr, keep);  // (the cut is never below the 16th best, the list stays authoritative)
        }
        ++ctr[1];
        const uint32_t pos_tile = p.pos_base + (uint32_t)(tile * TS_BN);
        if (mm < thr || vtile < TS_BN) {
          epi_select_tile<REG, RANGE>(r0, r1, g0, g1, pos_tile, buf, cnt, thr, tk, gthr, p.cap, &cut);
        }
        if constexpr (REG || RANGE) continue;
        // deferred compaction: a row past the high-water mark is compacted here, at most one row per warp and
        // tile, so the bursts (all rows of a warp fill at the same rate) are spread over the slack that every
        // tile leaves; only a row that is about to overflow is compacted at once (above)
        const unsigned pend = __ballot_sync(FULL, cnt > p.hwm);
        if (pend) {
          ++ctr[3];
          compact_lane<KPL>(__ffs(pend) - 1, buf, cnt, thr, p.kprime, p.slack, gthr, lane);
        }
      }
      const size_t slot = unit * TC_QB + h * TC_BM + row;
      p.cand_cnt[slot] = row_valid ? cnt : 0;
      if constexpr (RANGE) p.cand_cut[slot] = cut;
      else p.cand_thr[slot] = thr;
    }
    if (p.counters && lane == 0) {
      for (int i = 0; i < 4; ++i) atomicAdd(p.counters + i, (unsigned long long)ctr[i]);
      atomicAdd(p.counters + 4, (unsigned long long)ti * 2);
#ifdef NB200_EXPERIMENTS
      NB_TACC(c_proc, te);
      atomicAdd(p.counters + 14, c_twait);
      atomicAdd(p.counters + 15, c_drain);
      atomicAdd(p.counters + 16, c_proc);
      atomicAdd(p.counters + 17, c_setup);
#endif
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------- K1 for uint8 rows: the integer tensor pipe
// l2sqr_sift (config 4; reference: l2SqrSIFTPrecompAVX, distcomp_l2sqr_sift.cc:100-151: n1 + n2 - 2 x.y over 128 bytes
// with the int32 norms kept behind each payload).  Same structure as tc_scan_ts_kernel -- a CTA's 256 queries live in
// tensor memory, one 64-row database tile per stage, two MMA issuers, eight epilogue warps -- on
// tcgen05.mma.kind::i8 (u8 x u8 -> s32, K = 32 per instruction, 4 x the TF32 rate; tools/tc_peak.cu):
//   * rows stay BYTES in HBM and in shared memory: 128 B per row instead of the 512 B of the widened fp32 copy;
//   * the accumulator is made to carry the whole rank: with M = ceil(max |x|^2 / 2) and V(x) = M - ceil(|x|^2 / 2)
//     >= 0 written as 32 base-255 "digits" d_j(x) (one more 32-byte k-block per row, against the constant operand
//     row c = [1, 255, 255, ...]),      acc = q.x + sum_j c_j d_j(x) = q.x + V(x),
//     so that  2 (M - acc) = |x|^2 - 2 q.x + (|x|^2 odd)  is the pass-1 rank: exact up to +1, larger acc = nearer.
//     One extra K = 32 MMA per tile and half; needs max |x|^2 <= 4 032 059 (else the engine keeps the widened path);
//   * tensor memory: [0, 128) operand rows (per half 32 columns of query bytes + 8 columns of constants),
//     [128, 512) THREE accumulator buffers x two halves x 64 columns -- one more than the TF32 kernel has room for,
//     which is what absorbs the epilogue's jitter now that a tile's MMAs take ~320 clk instead of ~1100;
//   * the epilogue works on the raw int32 accumulators (max tree, acc > threshold); survivors become the same
//     (float rank, position) keys as everywhere else (an int below 2^24 is exact in fp32), so re-rank, certificate
//     (error bound: 1) and merge are shared.
constexpr int U8_ACC0 = 128;   // first accumulator column
constexpr int U8_NBUF = 3;     // accumulator buffers
constexpr int U8_ROW = 128;    // bytes per database row (SIFT_DIM, space_l2sqr_sift.h)
constexpr int U8_NROW = 32;    // bytes per row of the norm-digit block
constexpr int U8_STAGE = TS_BN * (U8_ROW + U8_NROW);  // 10 KB per tile

struct U8Params {
  int n, nq, s_max;
  const int4* pieces;
  uint32_t pos_base;
  uint64_t* cand;
  int* cand_cnt;
  float* cand_thr;
  int cap, kprime, slack, hwm, n_stage, refresh_mask, debug;
  uint32_t* gthr;           // [q_pad] ordered float bits of the best rank threshold published per query
  const uint8_t* q;         // [q_pad][128] query bytes (zero rows past nq)
  int m_half;               // M = ceil(max |x|^2 / 2)
  unsigned long long* counters;
  uint32_t* cand_cut;       // range mode, instead of cand_thr (see TcParams)
};

__device__ __forceinline__ void umma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::i8: D = S32 (2 @4), A = B = unsigned 8-bit (0 @7, 0 @10), both K-major, N >> 3 @17, M >> 4 @24
__host__ __device__ constexpr uint32_t make_idesc_u8(int m, int n) {
  return (2u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// K-major tile with rows of 32 bytes, 32B swizzle (the norm-digit block): 8-row atoms of 256 B
__device__ __forceinline__ uint64_t make_smem_desc_sw32(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;
  return d;
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ int max3i(int a, int b, int c) { return max(max(a, b), c); }
__device__ __forceinline__ int group_max8(const int (&r)[32], int q) {
  return max3i(max3i(r[8 * q], r[8 * q + 1], r[8 * q + 2]), max3i(r[8 * q + 3], r[8 * q + 4], r[8 * q + 5]),
               max(r[8 * q + 6], r[8 * q + 7]));
}
// accumulator <-> rank (an even integer, exact in fp32: |2 (M - acc)| < 2^24)
__device__ __forceinline__ float u8_rank_of(int acc, int m_half) { return (float)(2 * (m_half - acc)); }
__device__ __forceinline__ int u8_acc_of_rank(float rank, int m_half) {  // pass iff acc > result  <=>  rank' < rank
  if (!(rank < 3.0e38f)) return -1;          // +inf / NaN ("no threshold yet"): every accumulator (>= 0) passes
  return m_half - (__float2int_rd(rank) >> 1) - ((__float2int_rd(rank) & 1) ? 1 : 0) + 0;
}

// per-lane selection over one 64-column tile (integer twin of epi_select_tile): acc > thr passes.
// RANGE: keys are appended in position order; a full buffer records its first dropped position in *cut and the row
// stops selecting (thr = INT_MAX: no accumulator passes).
template <bool REG, bool RANGE = false>
__device__ __forceinline__ void epi_select_tile_i(const int (&r0)[32], const int (&r1)[32], const int (&g0)[4],
                                                  const int (&g1)[4], uint32_t pos0, uint64_t* buf, int& cnt, int& thr,
                                                  int (&tk)[TS_RK], uint32_t* gthr, int m_half, int cap = 0,
                                                  uint32_t* cut = nullptr) {
  unsigned gm = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    gm |= (g0[q] > thr ? 1u : 0u) << q;
    gm |= (g1[q] > thr ? 1u : 0u) << (q + 4);
  }
#pragma unroll 1
  while (gm) {
    const int q = __ffs(gm) - 1;
    gm &= gm - 1;
    const bool b0 = q & 1, b1 = q & 2, b2 = q & 4;
    int v[8];
    unsigned mk = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int a = b0 ? r0[8 + j] : r0[j], b = b0 ? r0[24 + j] : r0[16 + j];
      const int c = b0 ? r1[8 + j] : r1[j], d = b0 ? r1[24 + j] : r1[16 + j];
      const int ab = b1 ? b : a, cd = b1 ? d : c;
      v[j] = b2 ? cd : ab;
      mk |= (v[j] > thr ? 1u : 0u) << j;
    }
#pragma unroll 1
    while (mk) {
      const int jj = __ffs(mk) - 1;
      mk &= mk - 1;
      const int lo4 = (jj & 2) ? ((jj & 1) ? v[3] : v[2]) : ((jj & 1) ? v[1] : v[0]);
      const int hi4 = (jj & 2) ? ((jj & 1) ? v[7] : v[6]) : ((jj & 1) ? v[5] : v[4]);
      const int x = (jj & 4) ? hi4 : lo4;
      if constexpr (RANGE) {
        if (cnt == cap) {
          *cut = pos0 + 8 * q + jj;
          thr = 0x7FFFFFFF;
          gm = 0;
          break;
        }
      }
      if (!REG || x > thr) {
        buf[cnt] = ((uint64_t)__float_as_uint(u8_rank_of(x, m_half)) << 32) | (uint64_t)(pos0 + 8 * q + jj);
        ++cnt;
        if constexpr (REG) {  // 16 best accumulators, descending; every slot computed independently
          int prev = 0x7FFFFFFF;
#pragma unroll
          for (int i = 0; i < TS_RK; ++i) {
            const int cur = tk[i];
            tk[i] = min(prev, max(cur, x));
            prev = cur;
          }
          if (tk[TS_RK - 1] > thr) {
            thr = tk[TS_RK - 1];
            atomicMin(gthr, f32_ordered(u8_rank_of(thr, m_half)));
          }
        }
      }
    }
  }
}

// RANGE: batched range queries -- every row's threshold is its query's fixed accumulator threshold T_acc (p.gthr, the
// int bits written by tc_range_threshold_u8_kernel), no compaction, no refresh; a list whose buffer fills stores the
// position of its first dropped survivor in p.cand_cut.
template <int KPL, bool REG, bool RANGE = false>
__global__ void __launch_bounds__(TS_THREADS, 1)
tc_scan_u8_kernel(const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmN, const U8Params p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  unsigned char* smem_st = smem;  // stage s: [64 rows x 128 B, 128B swizzle][64 rows x 32 B, 32B swizzle]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_st + (size_t)p.n_stage * U8_STAGE);
  uint64_t* full_bar = bars;                       // [n_stage]
  uint64_t* empty_bar = bars + p.n_stage;          // [n_stage] one commit from each issuer
  uint64_t* tfull_bar = bars + 2 * p.n_stage;      // [3 buffers][2 halves]
  uint64_t* tempty_bar = tfull_bar + 2 * U8_NBUF;  // [3][2] the 4 warps of the half
  uint64_t* afull_bar = tempty_bar + 2 * U8_NBUF;  // [1]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(afull_bar + 1);

  const int tid = threadIdx.x, warp = __shfl_sync(FULL, tid >> 5, 0), lane = tid & 31;
  const int4* my_pieces = p.pieces + (size_t)blockIdx.x * TS_MAXP;

  if (tid == 0) {
    for (int s = 0; s < p.n_stage; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 2);
    }
    for (int b = 0; b < 2 * U8_NBUF; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 4);
    }
    mbar_init(afull_bar, 256);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmN);
  }
  if (warp == 1) tmem_alloc(tmem_holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer: one whole tile (rows + norm digits) per stage =====================
    int s = 0;
    uint32_t ph = 0;
    for (int pi = 0; pi < TS_MAXP; ++pi) {
      const int4 pc = __ldg(my_pieces + pi);
      if (pc.x < 0) break;
      for (int t = pc.y; t < pc.z; ++t) {
        mbar_wait(&empty_bar[s], ph ^ 1);
        unsigned char* st = smem_st + (size_t)s * U8_STAGE;
        if (elect_one()) {
          mbar_expect_tx(&full_bar[s], (uint32_t)U8_STAGE);
          tma_load_2d(&tmB, &full_bar[s], st, 0, t * TS_BN);
          tma_load_2d(&tmN, &full_bar[s], st + TS_BN * U8_ROW, 0, t * TS_BN);
        }
        __syncwarp();
        if (++s == p.n_stage) {
          s = 0;
          ph ^= 1;
        }
      }
    }
  } else if (warp == 1 || warp == TS_MMA_WARP2) {
    // ===================== MMA issuers: one warp per 128-query half =====================
    constexpr uint32_t idesc = make_idesc_u8(TC_BM, TS_BN);
    const int hh = warp == 1 ? 0 : 1;
    const uint32_t st_base = smem_u32(smem_st);
    const uint32_t a_half = tmem_base + (uint32_t)(hh * 64);
    int s = 0;
    uint32_t ph = 0;
    int ti = 0, b = 0;
    uint32_t bph = 0;  // parity of the accumulator ring's current round
    [[maybe_unused]] unsigned long long c_tempty = 0, c_full = 0, c_issue = 0;
    NB_T0(tm);
    for (int pi = 0; pi < TS_MAXP; ++pi) {
      const int4 pc = __ldg(my_pieces + pi);
      if (pc.x < 0) break;
      mbar_wait(afull_bar, pi & 1);
      tc_fence_after();
      for (int t = pc.y; t < pc.z; ++t, ++ti) {
        NB_TACC(c_issue, tm);
        mbar_wait(&tempty_bar[b * 2 + hh], bph ^ 1);
        NB_TACC(c_tempty, tm);
        mbar_wait(&full_bar[s], ph);
        NB_TACC(c_full, tm);
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(U8_ACC0 + (b * 2 + hh) * TS_BN);
        const uint32_t sb = st_base + (uint32_t)s * (uint32_t)U8_STAGE;
        if (elect_one()) {
          const uint64_t db = make_smem_desc(sb);
          // UMMA_K = 32 bytes: 8 TMEM columns of A, +2 in the descriptor of B
          umma_i8_ts(d, a_half, db, idesc, 0);
          umma_i8_ts(d, a_half + 8, db + 2, idesc, 1);
          umma_i8_ts(d, a_half + 16, db + 4, idesc, 1);
          umma_i8_ts(d, a_half + 24, db + 6, idesc, 1);
          umma_i8_ts(d, a_half + 32, make_smem_desc_sw32(sb + TS_BN * U8_ROW), idesc, 1);  // + V(x)
          tc_commit(&empty_bar[s]);
          tc_commit(&tfull_bar[b * 2 + hh]);
        }
        __syncwarp();
        if (++s == p.n_stage) {
          s = 0;
          ph ^= 1;
        }
        if (++b == U8_NBUF) {
          b = 0;
          bph ^= 1;
        }
      }
    }
#ifdef NB200_EXPERIMENTS
    NB_TACC(c_issue, tm);
    if (p.counters && lane == 0 && hh == 0) {
      atomicAdd(p.counters + 11, c_tempty);
      atomicAdd(p.counters + 12, c_full);
      atomicAdd(p.counters + 13, c_issue);
    }
#endif
  } else {
    // ===================== epilogue: 8 warps, thread == one query row =====================
    const int e = warp - 2;
    const int h = e >> 2;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16);
    unsigned ctr[4] = {0, 0, 0, 0};
    int b = 0;
    uint32_t bph = 0;
    [[maybe_unused]] unsigned long long c_twait = 0, c_drain = 0, c_proc = 0;
    NB_T0(te);
    for (int pi = 0; pi < TS_MAXP; ++pi) {
      const int4 pc = __ldg(my_pieces + pi);
      if (pc.x < 0) break;
      const int qb = pc.x, t_begin = pc.y, t_end = pc.z;
      const size_t unit = (size_t)qb * p.s_max + pc.w;
      const int qrow = qb * TC_QB + h * TC_BM + row;
      const bool row_valid = qrow < p.nq;
      uint64_t* buf = p.cand + (unit * TC_QB + h * TC_BM + row) * (size_t)p.cap;
      uint32_t* gthr = p.gthr + qrow;
      int cnt = 0;
      int thr = !row_valid ? 0x7FFFFFFF : RANGE ? (int)*gthr : -1;  // pass iff acc > thr (accumulators are >= 0)
      uint32_t cut = 0xFFFFFFFFu;
      int tk[TS_RK];
#pragma unroll
      for (int i = 0; i < TS_RK; ++i) tk[i] = -1;
      {
        // operand rows -> tensor memory: 128 query bytes = 32 columns (byte k in column k / 4), then the constant
        // k-block [1, 255 x 31] that multiplies the norm digits
        const uint4* src = reinterpret_cast<const uint4*>(p.q + (size_t)qrow * U8_ROW);
        const uint32_t ta = trow + (uint32_t)(h * 64);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint4 u0 = __ldg(src + 2 * c), u1 = __ldg(src + 2 * c + 1);
          const uint32_t v[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
          tmem_st8(ta + (uint32_t)(c * 8), v);
        }
        const uint32_t cv[8] = {0xFFFFFF01u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
        tmem_st8(ta + 32u, cv);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(afull_bar);
      }
      // a row above this many keys sends its warp to the slow path (RANGE: a full row has stopped selecting)
      const int guard = RANGE ? p.cap : REG ? p.cap - TS_BN - 1 : p.hwm;
      for (int tile = t_begin; tile < t_end; ++tile) {
        uint32_t v0[32], v1[32];
        NB_TACC(c_proc, te);
        mbar_wait(&tfull_bar[b * 2 + h], bph);
        NB_TACC(c_twait, te);
        tc_fence_after();
        const uint32_t tcol = trow + (uint32_t)(U8_ACC0 + (b * 2 + h) * TS_BN);
        tmem_ld64(tcol, v0, v1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[b * 2 + h]);
        if (++b == U8_NBUF) {
          b = 0;
          bph ^= 1;
        }
        NB_TACC(c_drain, te);
        if (NB200_DBG(p.debug, 1)) {
          if (v0[0] == 0x12345678u || v1[0] == 0x12345678u) thr = 0;
          continue;
        }
        int r0[32], r1[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          r0[j] = (int)v0[j];
          r1[j] = (int)v1[j];
        }
        int g0[4], g1[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          g0[q] = group_max8(r0, q);
          g1[q] = group_max8(r1, q);
        }
        const int mm = max3i(max(max3i(g0[0], g0[1], g0[2]), max3i(g0[3], g1[0], g1[1])), g1[2], g1[3]);
        const int vtile = p.n - tile * TS_BN;
        // (RANGE: the thresholds are fixed, the only warp-uniform reason is the shard's last, partial tile)
        const bool uni = RANGE ? vtile < TS_BN
                               : ((((tile - t_begin) & p.refresh_mask) == 0) & !NB200_DBG(p.debug, 4)) | (vtile < TS_BN);
        const bool mine = (mm > thr) | (cnt > guard);
        if (!uni && !__any_sync(FULL, mine)) continue;
        if (NB200_DBG(p.debug, 2) && tile - t_begin > 64) continue;  // timing experiment: the fast path only
        // ------------------------------------------------------------------ slow path
        if (!RANGE && ((tile - t_begin) & p.refresh_mask) == 0 && row_valid)
          thr = max(thr, u8_acc_of_rank(f32_from_ordered(*gthr), p.m_half));
        if (vtile < TS_BN) {  // rows past the end of the shard: never candidates
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (j >= vtile) r0[j] = -2;
            if (j + 32 >= vtile) r1[j] = -2;
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            g0[q] = group_max8(r0, q);
            g1[q] = group_max8(r1, q);
          }
        }
        unsigned need = RANGE ? 0u : __ballot_sync(FULL, cnt > p.cap - TS_BN - 1);
        while (need) {
          ++ctr[2];
          const int src = __ffs(need) - 1;
          need &= need - 1;
          float tf = u8_rank_of(thr, p.m_half);
          compact_lane<KPL>(src, buf, cnt, tf, p.kprime, p.slack, gthr, lane);
          if (lane == src) thr = max(thr, u8_acc_of_rank(tf, p.m_half));
        }
        ++ctr[1];
        const uint32_t pos_tile = p.pos_base + (uint32_t)(tile * TS_BN);
        if (mm > thr || vtile < TS_BN) {
          epi_select_tile_i<REG, RANGE>(r0, r1, g0, g1, pos_tile, buf, cnt, thr, tk, gthr, p.m_half, p.cap, &cut);
        }
        if constexpr (REG || RANGE) continue;
        const unsigned pend = __ballot_sync(FULL, cnt > p.hwm);
        if (pend) {
          ++ctr[3];
          const int src = __ffs(pend) - 1;
          float tf = u8_rank_of(thr, p.m_half);
          compact_lane<KPL>(src, buf, cnt, tf, p.kprime, p.slack, gthr, lane);
          if (lane == src) thr = max(thr, u8_acc_of_rank(tf, p.m_half));
        }
      }
      const size_t slot = unit * TC_QB + h * TC_BM + row;
      p.cand_cnt[slot] = row_valid ? cnt : 0;
      if constexpr (RANGE) p.cand_cut[slot] = cut;
      else p.cand_thr[slot] = thr < 0 ? __int_as_float(0x7F800000) : u8_rank_of(thr, p.m_half);
    }
    if (p.counters && lane == 0) {
      for (int i = 0; i < 4; ++i) atomicAdd(p.counters + i, (unsigned long long)ctr[i]);
#ifdef NB200_EXPERIMENTS
      NB_TACC(c_proc, te);
      atomicAdd(p.counters + 14, c_twait);
      atomicAdd(p.counters + 15, c_drain);
      atomicAdd(p.counters + 16, c_proc);
#endif
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------- pass 2: exact re-rank
struct RerankParams {
  const float* db;         // [n_pad][row_words] ORIGINAL vectors
  const float* queries;    // [q_pad][row_words] ORIGINAL queries
  const float* db_norm2;   // [n_pad] |x|^2 (cosine) or NULL
  int nq, row_words, k, n_split, cap, mode;  // mode: SCAN_L2 / SCAN_COSINE / SCAN_NEGDOT
  int q_begin, n_lists;    // this launch serves queries q_begin + blockIdx.x; only the first n_lists slots can be in use
  uint32_t pos_base;
  const uint64_t* cand;
  const int* cand_cnt;
  const float* cand_thr;
  float eps_inexact, eps_exact;   // relative error bounds of pass 1 (see DESIGN.md)
  float x_max;                    // max |B-operand row|
  const int* inexact_flags;       // [2]: nonzero if the database / this query batch is not TF32-exact
  uint64_t* out_keys;             // [nq][k]
  int* out_cert;                  // [nq] 1 = certified exact
  const uint8_t* db_u8;           // uint8 index on byte rows (tc_scan_u8_kernel): [n_pad][128] rows / queries, exact
  const uint8_t* q_u8;            //   int32 arithmetic here; NULL: float rows
  float abs_err;                  // > 0: absolute pass-1 error bound (uint8 on the integer pipe: 1), else eps * norms
  int int_keys;                   // uint8 indexes: out keys carry i32_ordered(int distance) (FIN_INT), like the dp4a scan
  int* fb_count;                  // device-side list of the uncertified queries (count + indices), or NULL:
  int* fb_idx;                    // what the device-predicated exact re-run works from (no host round trip)
  int debug_cert;                 // NB200_TC_DEBUG_CERT: print the certificate inputs of the first queries
};

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// E_q: bound on |pass-1 rank - exact rank| of one query (DESIGN.md "certificate"), shared by the kNN re-rank and the
// range thresholds.  abs_err > 0 is an absolute bound (uint8 on the integer pipe), else eps * (2 for l2) * |q| * x_max.
__device__ __forceinline__ float pass1_error(float abs_err, float eps_inexact, float eps_exact, bool inexact_q, int mode,
                                             float qn2, float x_max) {
  return abs_err > 0.f ? abs_err
                       : (inexact_q ? eps_inexact : eps_exact) * (mode == SCAN_L2 ? 2.f : 1.f) * sqrtf(qn2) * x_max + 1e-30f;
}

__global__ void __launch_bounds__(256) tc_rerank_kernel(const RerankParams p, int items_pow2) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  uint64_t* sk = reinterpret_cast<uint64_t*>(smem_raw);          // [items_pow2] exact keys
  float* srank = reinterpret_cast<float*>(sk + items_pow2);       // [items_pow2] exact rank (certificate domain)
  uint32_t* spos = reinterpret_cast<uint32_t*>(srank);            // (the same words first hold the live positions)
  __shared__ int s_cnt[64];
  __shared__ int s_red[8];
  __shared__ int s_live;
  __shared__ uint32_t s_ak, s_worst;
  __shared__ float s_wmin[2], s_qn2;
  const int q = p.q_begin + blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nwarps = blockDim.x >> 5;  // 4, or 8 for long rows / large k (more candidate rows in flight)
  const int qb = q / TC_QB, row = q % TC_QB;
  const float* qv = p.queries + (size_t)q * p.row_words;

  // one thread per candidate slot of this query (n_split <= 64): its key count and final threshold
  if (tid < 64) {
    float mt = __int_as_float(0x7F800000);
    int c = 0;
    if (tid < p.n_lists) {
      const size_t slot = ((size_t)qb * p.n_split + tid) * TC_QB + row;
      c = p.cand_cnt[slot];   // -1: slot unused (the host fills the array with 0xFF)
      if (c >= 0) mt = p.cand_thr[slot];  // +inf when the piece never dropped anything
      c = max(c, 0);
    }
    s_cnt[tid] = c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mt = fminf(mt, __shfl_xor_sync(FULL, mt, o));
    if (lane == 0) s_wmin[warp] = mt;
  }
  if (tid == 0) {
    s_live = 0;
    s_ak = 0xFFFFFFFFu;
    s_worst = 0u;
  }
  if (warp == 2) {
    float s = 0.f;
    if (p.q_u8) {  // 128 bytes: one uchar4 per lane, exact integer sum
      const uchar4 y = reinterpret_cast<const uchar4*>(p.q_u8 + (size_t)q * U8_ROW)[lane];
      int si = (int)y.x * y.x + (int)y.y * y.y + (int)y.z * y.z + (int)y.w * y.w;
      si = __reduce_add_sync(FULL, si);
      s = (float)si;
    } else {
      for (int c = lane; c < p.row_words; c += 32) s = fmaf(qv[c], qv[c], s);
      s = warp_sum_f(s);
    }
    if (lane == 0) s_qn2 = s;
  }
  __syncthreads();
  const float qn2 = s_qn2;
  const float minthr = fminf(s_wmin[0], s_wmin[1]);
  // Only candidates whose pass-1 rank lies below the smallest threshold any piece ended with can matter: if
  // the certificate below holds, every true neighbour has pass-1 rank < minthr (DESIGN.md), and if it does not
  // hold the query is re-run anyway.  With shared thresholds this is ~k' keys out of the few hundred appended.
  // One warp per slot (round robin), so the slots' lists are read concurrently.
  for (int s = warp; s < p.n_lists; s += nwarps) {
    const size_t slot = ((size_t)qb * p.n_split + s) * TC_QB + row;
    const uint64_t* cb = p.cand + slot * (size_t)p.cap;
    const int c = s_cnt[s];
    for (int i = lane; i < c; i += 32) {
      const uint64_t key = cb[i];
      if (__uint_as_float((uint32_t)(key >> 32)) < minthr) {
        const int at = atomicAdd(&s_live, 1);
        if (at < items_pow2) sk[at] = key;
      }
    }
  }
  __syncthreads();
  const bool overflow = s_live > items_pow2;  // more live keys than the sort buffer holds: not certifiable
  int total = min(s_live, items_pow2);
  // pass-1 error bound of this query (same E as the certificate below)
  const bool inexact_q = p.inexact_flags[0] != 0 || p.inexact_flags[1] != 0;
  const float E_q = pass1_error(p.abs_err, p.eps_inexact, p.eps_exact, inexact_q, p.mode, qn2, p.x_max);
  {
    // Second filter.  Let a_k be the k-th smallest PASS-1 rank among the live keys.  The k keys at or below it
    // have exact rank <= a_k + E, so the true k-th best exact rank is <= a_k + E and every true neighbour has
    // pass-1 rank <= a_k + 2E: only those keys need the exact evaluation (k + a few instead of s_max * k').
    uint32_t* sord = reinterpret_cast<uint32_t*>(srank);
    for (int i = tid; i < total; i += blockDim.x) sord[i] = f32_ordered(__uint_as_float((uint32_t)(sk[i] >> 32)));
    __syncthreads();
    uint32_t cut = 0xFFFFFFFFu;
    if (total > p.k) {
      uint32_t lo = 0u, hi = 0xFFFFFFFFu;
      if (total <= 256) {
        // the usual case, a few dozen live keys: every thread counts the keys below / at its own one -- no barrier per
        // step (the 32-step bisection below, two barriers each, was 42 % of this kernel's stall samples on a short
        // shard, profiles/README.md).  Exactly one VALUE v has #(ord < v) < k <= #(ord <= v).
        for (int i = tid; i < total; i += blockDim.x) {
          const uint32_t v = sord[i];
          int lt = 0, le = 0;
          for (int j = 0; j < total; ++j) {
            const uint32_t u = sord[j];
            lt += u < v ? 1 : 0;
            le += u <= v ? 1 : 0;
          }
          if (lt < p.k && le >= p.k) s_ak = v;
        }
        __syncthreads();
        lo = hi = s_ak;
      }
      while (lo < hi) {  // smallest v with #(ord <= v) >= k
        const uint32_t mid = lo + ((hi - lo) >> 1);
        int c = 0;
        for (int i = tid; i < total; i += blockDim.x) c += sord[i] <= mid ? 1 : 0;
        c = __reduce_add_sync(FULL, c);
        if (lane == 0) s_red[warp] = c;
        __syncthreads();
        c = 0;
        for (int w = 0; w < nwarps; ++w) c += s_red[w];
        __syncthreads();
        if (c >= p.k) hi = mid; else lo = mid + 1;
      }
      const float a_k = f32_from_ordered(lo);
      const float t2 = a_k + 2.f * E_q + fabsf(a_k) * 2e-6f;
      if (t2 < minthr) cut = f32_ordered(t2);
    }
    // compact the positions of the keys at or below the cut (flags first, then an exclusive scan, then the moves:
    // the destination aliases the array the flags are read from)
    unsigned long long mask = 0ull;
    int mine = 0;
    for (int j = 0, i = tid; i < total; ++j, i += blockDim.x)
      if (sord[i] <= cut) {
        mask |= 1ull << j;
        ++mine;
      }
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_red[warp] = incl;
    __syncthreads();
    int off = incl - mine;
    for (int w = 0; w < warp; ++w) off += s_red[w];
    int kept = 0;
    for (int w = 0; w < nwarps; ++w) kept += s_red[w];
    for (int j = 0, i = tid; i < total; ++j, i += blockDim.x)
      if (mask >> j & 1ull) spos[off++] = (uint32_t)sk[i];
    __syncthreads();
    total = kept;
  }
  int p2e = 32;
  while (p2e < total || p2e < p.k) p2e <<= 1;
  if (p2e > items_pow2) p2e = items_pow2;
  for (int t = tid; t < p2e; t += blockDim.x) sk[t] = KEY_MAX;
  __syncthreads();
  const int rw4 = p.row_words >> 2;
  const float4* q4 = reinterpret_cast<const float4*>(qv);

  // exact fp32 distance of every live candidate: one warp per candidate, 128-bit loads
  for (int i0 = warp; i0 < total; i0 += nwarps) {
    const uint32_t pos = spos[i0];
    const size_t local = (size_t)(pos - p.pos_base);
    if (p.db_u8) {  // sum (x - y)^2 over 128 bytes in int32: the reference's n1 + n2 - 2 x.y (distcomp_l2sqr_sift.cc:41-50)
      const uchar4 x = __ldg(reinterpret_cast<const uchar4*>(p.db_u8 + local * U8_ROW) + lane);
      const uchar4 y = reinterpret_cast<const uchar4*>(p.q_u8 + (size_t)q * U8_ROW)[lane];
      const int d0 = (int)x.x - y.x, d1 = (int)x.y - y.y, d2 = (int)x.z - y.z, d3 = (int)x.w - y.w;
      int di = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
      di = __reduce_add_sync(FULL, di);
      __syncwarp();
      if (lane == 0) {
        sk[i0] = make_key(i32_ordered(di), pos);
        srank[i0] = (float)di - qn2;
      }
      continue;
    }
    const float4* x4 = reinterpret_cast<const float4*>(p.db + local * p.row_words);
    float acc = 0.f, nxs = 0.f, nqs = 0.f;
    const bool cosfam = p.mode == SCAN_COSINE || p.mode == SCAN_ANGULAR;
    for (int e = lane; e < rw4; e += 32) {
      const float4 x = __ldg(x4 + e), y = q4[e];
      if (p.mode == SCAN_L2) {
        const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z, d3 = x.w - y.w;
        acc = fmaf(d0, d0, acc);
        acc = fmaf(d1, d1, acc);
        acc = fmaf(d2, d2, acc);
        acc = fmaf(d3, d3, acc);
      } else {
        acc = fmaf(x.x, y.x, acc);
        acc = fmaf(x.y, y.y, acc);
        acc = fmaf(x.z, y.z, acc);
        acc = fmaf(x.w, y.w, acc);
        if (cosfam) {
          // the three sums of NormScalarProductSIMD (distcomp_scalar.cc:84-168) with ONE summation pattern, as
          // in the reference: identical vectors then give x.y == |x|^2 == |y|^2 bit for bit and nsp = 1 +- 1 ulp
          nxs = fmaf(x.x, x.x, nxs);
          nxs = fmaf(x.y, x.y, nxs);
          nxs = fmaf(x.z, x.z, nxs);
          nxs = fmaf(x.w, x.w, nxs);
          nqs = fmaf(y.x, y.x, nqs);
          nqs = fmaf(y.y, y.y, nqs);
          nqs = fmaf(y.z, y.z, nqs);
          nqs = fmaf(y.w, y.w, nqs);
        }
      }
    }
    acc = warp_sum_f(acc);
    if (cosfam) {
      nxs = warp_sum_f(nxs);
      nqs = warp_sum_f(nqs);
    }
    float dist, rank;
    if (p.mode == SCAN_L2) {
      dist = acc;                 // sum (x-y)^2, the reference's formula (distcomp_lp.cc:304-365)
      rank = acc - qn2;           // pass 1 ranks by |x|^2 - 2 q.x
    } else if (p.mode == SCAN_NEGDOT) {
      dist = -acc;
      rank = -acc;
    } else {
      const float nx = nxs;
      const float eps = 2.0f * 1.17549435e-38f;
      float nsp = 0.f;
      if (!(nx < eps || nqs < eps)) nsp = fmaxf(-1.f, fminf(1.f, acc / sqrtf(nx) / sqrtf(nqs)));
      dist = p.mode == SCAN_ANGULAR ? acosf(nsp) : fmaxf(0.f, 1.f - nsp);  // AngularDistance, distcomp_scalar.cc:254-258
      rank = (nx < eps) ? 0.f : -acc * rsqrtf(nx);   // pass 1 ranks by -q.x / |x|
    }
    __syncwarp();  // every lane has read spos[i0] before the slot is reused for the rank
    if (lane == 0) {
      sk[i0] = p.int_keys ? make_key(i32_ordered((int)dist), pos) : make_key(f32_ordered(dist), pos);
      srank[i0] = rank;
    }
  }
  __syncthreads();
  const bool rank_sort = total <= 128;
  if (rank_sort) {
    // few candidates (the usual case after the second filter): a key's place in the answer is the number of keys
    // below it (keys are distinct: the position is part of the key) -- no barriers, where the bitonic network below
    // spends 15 of them on 32 keys
    for (int i = tid; i < total; i += blockDim.x) {
      const uint64_t key = sk[i];
      int r = 0;
      for (int j = 0; j < total; ++j) r += sk[j] < key ? 1 : 0;
      if (r < p.k) {
        p.out_keys[(size_t)q * p.k + r] = key;
        atomicMax(&s_worst, f32_ordered(srank[i]));
      }
    }
    for (int e = total + tid; e < p.k; e += blockDim.x) p.out_keys[(size_t)q * p.k + e] = KEY_MAX;
    __syncthreads();
  }
  for (int t = total + tid; t < p2e && !rank_sort; t += blockDim.x) srank[t] = __int_as_float(0x7F800000);
  __syncthreads();

  // sort (key, rank) ascending by key
  for (int size = 2; size <= p2e && !rank_sort; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < p2e / 2; t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const uint64_t a = sk[lo], b = sk[hi];
        if ((a > b) == up) {
          sk[lo] = b;
          sk[hi] = a;
          const float ra = srank[lo];
          srank[lo] = srank[hi];
          srank[hi] = ra;
        }
      }
      __syncthreads();
    }
  }
  for (int e = tid; e < p.k && !rank_sort; e += blockDim.x) p.out_keys[(size_t)q * p.k + e] = e < p2e ? sk[e] : KEY_MAX;

  if (tid == 0) {
    // certificate: every non-candidate has approximate rank >= s_minthr, exact rank >= s_minthr - E
    int cert;
    if (overflow) {
      cert = 0;
    } else if (minthr == __int_as_float(0x7F800000)) {
      cert = 1;  // nothing was ever dropped in any split: the candidates are the whole shard
    } else if (total < p.k) {
      cert = 0;
    } else {
      const float E = E_q;
      // worst exact rank among the k answers (ranks are not exactly monotone in the key for cosine)
      float worst = __int_as_float(0xFF800000);
      if (rank_sort) worst = f32_from_ordered(s_worst);
      else
        for (int e = 0; e < p.k; ++e) worst = fmaxf(worst, srank[e]);
      cert = (worst + E + fabsf(worst) * 1e-6f < minthr) ? 1 : 0;
    }
    p.out_cert[q] = cert;
    if (!cert && p.fb_idx) p.fb_idx[atomicAdd(p.fb_count, 1)] = q;
    if (NB200_DBG(p.debug_cert, 1) && (q < 2 || (cert == 0 && q < 40))) {
      float worst = __int_as_float(0xFF800000);
      for (int e = 0; e < p.k && e < p2e; ++e) worst = fmaxf(worst, srank[e]);
      printf("rerank q=%d cert=%d live=%d total=%d p2e=%d items=%d minthr=%g worst=%g qn2=%g n_split=%d cnt0=%d\n", q, cert,
             s_live, total, p2e, items_pow2, minthr, worst, qn2, p.n_split, s_cnt[0]);
    }
  }
}

// ---------------------------------------------------------------- batched range queries: radius -> threshold
// One warp per query.  T_q is the radius in the rank domain of pass 1 (see the header of this file), widened so that
// every row whose distance by the verification formula (range_scan.cu: range_row_dist) is <= r has pass-1 rank < T_q
// (DESIGN.md "K5b"): E_q of the re-rank's certificate, plus rel = (D + 16) 2^-22 -- about four times the first-order
// fp32 error of the verification sums and of |q|^2 -- on every term, evaluated in double and rounded up.
__global__ void tc_range_threshold_kernel(const float* __restrict__ q, int nq, int row_words, int mode, int take_sqrt,
                                          const float* __restrict__ radii, float x_max, float eps_inexact,
                                          float eps_exact, int db_inexact, uint32_t* __restrict__ gthr) {
  const int qi = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (qi >= nq) return;
  const float* qv = q + (size_t)qi * row_words;
  float s = 0.f;
  unsigned bad = 0;
  for (int c = lane; c < row_words; c += 32) {
    const float v = qv[c];
    s = fmaf(v, v, s);
    bad |= __float_as_uint(v) & 0x1FFFu;  // not TF32-exact (as the scan kernels test it)
  }
  s = warp_sum_f(s);
  bad = __reduce_or_sync(FULL, bad);
  if (lane != 0) return;
  const float E = pass1_error(0.f, eps_inexact, eps_exact, bad != 0 || db_inexact != 0, mode, s, x_max);
  const double r = radii[qi], qn2 = s, qn = sqrt(qn2), xm = x_max;
  const double rel = (row_words + 16) * 2.384185791015625e-07;
  double t;
  if (mode == SCAN_L2) {  // d^2 <= r^2 (l2sqr: d <= r)  <=>  |x|^2 - 2 q.x <= r^2 - |q|^2
    const double r2 = take_sqrt ? r * r : r;
    t = r2 - qn2 + rel * (r2 + qn2 + xm * xm);
  } else if (mode == SCAN_NEGDOT) {  // -q.x <= r
    t = r + 2.0 * rel * qn * xm;
  } else if (s < 1e-30f) {
    // cosine family, a query of (almost) zero norm: the verification formula takes nsp = 0 when |q|^2 < 2 FLT_MIN
    // (d = 1, or pi / 2) whatever its pass-1 rank -q.x/|x| is, so no rank threshold is valid -- admit every row
    // (1e-30 leaves a margin of ~2^33 over 2 FLT_MIN: the fp32 |q|^2 of the two kernels cannot straddle the test)
    t = INFINITY;
  } else if (mode == SCAN_COSINE) {  // 1 - nsp <= r  <=>  -|q| nsp <= -|q| (1 - r); r >= 2 admits every row
    t = r >= 2.0 ? INFINITY : qn * (r - 1.0) + 4.0 * rel * qn;
  } else {  // SCAN_ANGULAR: acos(nsp) <= r  <=>  nsp >= cos r (acosf is within 2 ulp: < 5e-7 below pi); r >= pi admits all
    const double ra = r + 1e-6;
    t = ra >= 3.14159265358979323846 ? INFINITY : -qn * cos(ra) + 4.0 * rel * qn;
  }
  // rank < T_q is strict: one more ulp above the rounded-up bound
  gthr[qi] = f32_ordered(nextafterf(__double2float_ru(t + (double)E), INFINITY));
}

// uint8 byte rows (tc_scan_u8_kernel): the radius as a threshold in the accumulator domain, one warp per query.
// acc = q.x + M - ceil(|x|^2 / 2), so 2 (M - acc) = d - |q|^2 + (|x|^2 odd) with d = |q|^2 + |x|^2 - 2 q.x, all exact
// integers.  For R = floor(radius), d <= R gives 2 (M - acc) <= R - |q|^2 + 1, i.e. acc > T_acc with
// T_acc = M - floor((R - |q|^2 + 1) / 2) - 1.  Invariant: every row with d <= R passes; the only other rows that pass
// lie at d = R + 1 with |x|^2 even, and verification drops them.  Stored as the int bits of T_acc, clamped to -1 (every
// accumulator passes: R >= 2^24 exceeds every distance of 128 bytes, or R = +inf) and INT_MAX (none can: R < 0 or NaN).
// (u8_acc_of_rank is exact for integral ranks only: the radius in the rank domain is not one.)
__global__ void tc_range_threshold_u8_kernel(const uint8_t* __restrict__ q, int nq, const float* __restrict__ radii,
                                             int m_half, uint32_t* __restrict__ gthr) {
  const int qi = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (qi >= nq) return;
  const uchar4 v = reinterpret_cast<const uchar4*>(q + (size_t)qi * U8_ROW)[lane];
  const int qn2 = __reduce_add_sync(FULL, (int)v.x * v.x + (int)v.y * v.y + (int)v.z * v.z + (int)v.w * v.w);
  if (lane != 0) return;
  const float r = radii[qi];
  long long t;
  if (!(r >= 0.f)) {
    t = 0x7FFFFFFF;
  } else if (r >= 16777216.f) {
    t = -1;
  } else {
    const long long b = (long long)r - qn2 + 1;              // (long long)r = floor(r) for r >= 0
    const long long half = b >= 0 ? b / 2 : -((1 - b) / 2);  // floor(b / 2), also for b < 0
    t = (long long)m_half - half - 1;
  }
  gthr[qi] = (uint32_t)(int)std::max(-1LL, std::min(0x7FFFFFFFLL, t));
}

// ---------------------------------------------------------------- operand preparation
// A' = scale * q (scale = -2 for l2, -1 otherwise) into a buffer padded to 256-row blocks; also
// flags a batch that is not TF32-exact (any of the 13 low mantissa bits set).
__global__ void tc_prep_queries_kernel(const float* __restrict__ q, float* __restrict__ out, size_t words,
                                       float scale, int* __restrict__ inexact_flag) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  unsigned bad = 0;
  for (; i < words; i += stride) {
    const float v = q[i];
    bad |= __float_as_uint(v) & 0x1FFFu;
    out[i] = v * scale;
  }
  bad = __reduce_or_sync(FULL, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicOr(inexact_flag, 1);
}

__global__ void tc_split_rows_kernel(const float* __restrict__ src, size_t rows, int rw, float scale, int layout,
                                     float* __restrict__ dst) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x, total = rows * (size_t)rw;
  for (; i < total; i += stride) {
    const size_t r = i / (size_t)rw;
    const int c = (int)(i - r * (size_t)rw);
    const float v = src[i] * scale;
    const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);   // what the tensor core would keep of v
    const float lo = __uint_as_float(__float_as_uint(v - hi) & 0xFFFFE000u);
    float* d = dst + r * 3 * (size_t)rw;
    d[c] = hi;
    d[rw + c] = layout ? hi : lo;
    d[2 * rw + c] = layout ? lo : hi;
  }
}

// database side: bias[row] (|x|^2 for l2, 0 otherwise; +inf on padding rows), optional normalised copy,
// max operand-row norm, TF32-exactness flag.  One warp per row.
__global__ void tc_prep_db_kernel(const float* __restrict__ db, int n, int n_pad, int row_words, int mode,
                                  float* __restrict__ bias, float* __restrict__ norm2, float* __restrict__ db_unit,
                                  float* __restrict__ nblock, unsigned* __restrict__ max_norm_bits,
                                  int* __restrict__ inexact_flag) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_pad) return;
  if (warp >= n) {
    if (lane == 0) bias[warp] = __int_as_float(0x7F800000);
    if (nblock) nblock[(size_t)warp * TC_KB + lane] = 0.f;
    return;
  }
  const float* r = db + (size_t)warp * row_words;
  float s = 0.f;
  unsigned bad = 0;
  for (int c = lane; c < row_words; c += 32) {
    const float v = r[c];
    s = fmaf(v, v, s);
    bad |= __float_as_uint(v) & 0x1FFFu;
  }
  s = warp_sum_f(s);
  bad = __reduce_or_sync(FULL, bad);
  float op_norm2 = s;
  if (mode == SCAN_COSINE) {
    const float eps = 2.0f * 1.17549435e-38f;
    const float inv = s < eps ? 0.f : rsqrtf(s);
    for (int c = lane; c < row_words; c += 32) db_unit[(size_t)warp * row_words + c] = r[c] * inv;
    op_norm2 = s < eps ? 0.f : 1.0f;
    bad = 1;  // the normalised copy is never TF32-exact
  }
  if (nblock) {
    // |x|^2 as three TF32-exact pieces (11 + 11 + 2 significant bits): hi + mid + lo == s exactly, so the
    // tensor core adds the norm with fp32 accuracy in one K=8 step against a row of ones
    const float hi = __uint_as_float(__float_as_uint(s) & 0xFFFFE000u);
    const float r1 = s - hi;
    const float mid = __uint_as_float(__float_as_uint(r1) & 0xFFFFE000u);
    const float lo = r1 - mid;
    nblock[(size_t)warp * TC_KB + lane] = lane == 0 ? hi : lane == 1 ? mid : lane == 2 ? lo : 0.f;
  }
  if (lane == 0) {
    bias[warp] = (mode == SCAN_L2) ? s : 0.f;
    if (norm2) norm2[warp] = s;
    atomicMax(max_norm_bits, __float_as_uint(sqrtf(op_norm2) * 1.000001f));
    if (bad) atomicOr(inexact_flag, 1);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(ptr);
  return fn;
}

// rows x row_words fp32, row-major; box = 128 rows x 32 floats, 128B swizzle
bool make_tmap(CUtensorMap* map, const void* base, size_t rows, int row_elems, int box_rows = TC_BM) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  const int esz = 4;
  cuuint64_t dims[2] = {(cuuint64_t)row_elems, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)row_elems * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// byte rows [rows][row_bytes] (row_bytes = 128: 128B swizzle; 32: 32B swizzle), boxes of box_rows whole rows
bool make_tmap_u8(CUtensorMap* map, const void* base, size_t rows, int row_bytes, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
  cuuint32_t box[2] = {(cuuint32_t)row_bytes, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// uint8 rows: int32 |x|^2 per row (aux, from launch_row_aux) -> the 32 norm digits of V(x) = m_half - ceil(|x|^2 / 2)
// (rest = floor(V / 255) spread over 31 digits of at most 255, d0 = V - 255 rest); padding rows get V = 0.
// The 31 digits carry at most 31 * 255 * 255, so rest is capped there and d0 takes the remainder: d0 <= 254 except at
// V = 255 + 31 * 255 * 255 (a zero row when max |x|^2 is u8_imma_max_norm2(), M = 2 016 030), where d0 = 255
__global__ void u8_norm_digits_kernel(const int* __restrict__ norm2, int n, int n_pad, int m_half, uint8_t* __restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_pad) return;
  int v = 0;
  if (r < n) v = m_half - ((norm2[r] + 1) >> 1);
  uint32_t w[8];
  int rest = min(v / 255, 31 * 255);
  uint32_t d0 = (uint32_t)(v - 255 * rest);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    uint32_t word = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      uint32_t d;
      if (j == 0 && b == 0) d = d0;
      else {
        d = (uint32_t)min(rest, 255);
        rest -= (int)d;
      }
      word |= d << (8 * b);
    }
    w[j] = word;
  }
  uint4* o = reinterpret_cast<uint4*>(out + (size_t)r * U8_NROW);
  o[0] = make_uint4(w[0], w[1], w[2], w[3]);
  o[1] = make_uint4(w[4], w[5], w[6], w[7]);
}
__global__ void max_int_kernel(const int* __restrict__ v, int n, int* __restrict__ out) {
  int m = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = max(m, v[i]);
  m = __reduce_max_sync(FULL, m);
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

}  // namespace

// ---- uint8 rows on the integer tensor pipe (tc_scan_u8_kernel) ----
int u8_imma_max_norm2() { return 2 * (255 + 31 * 255 * 255) - 1; }  // V(x) <= 255 + 31 * 255 * 255 must hold
cudaError_t launch_u8_max_norm(const int* norm2, int n, int* d_out, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(d_out, 0, 4, stream);
  if (e != cudaSuccess || n <= 0) return e;
  max_int_kernel<<<std::min(296, (n + 255) / 256), 256, 0, stream>>>(norm2, n, d_out);
  return cudaGetLastError();
}
cudaError_t launch_u8_norm_digits(const int* norm2, int n, int n_pad, int m_half, uint8_t* out, cudaStream_t stream) {
  if (n_pad <= 0) return cudaSuccess;
  u8_norm_digits_kernel<<<(n_pad + 255) / 256, 256, 0, stream>>>(norm2, n, n_pad, m_half, out);
  return cudaGetLastError();
}

cudaError_t launch_tc_scan_u8(const uint8_t* q, const uint8_t* db, const uint8_t* digits, size_t n_pad, int n, int nq, int k,
                              int kprime, int m_half, uint32_t pos_base, int n_cta, int s_max, const int* d_pieces,
                              uint64_t* cand, int* cand_cnt, float* cand_thr, uint32_t* gthr, cudaStream_t stream,
                              uint32_t* range_cut) {
  if (n <= 0 || nq <= 0) return cudaSuccess;
  CUtensorMap tmB, tmN;
  if (!make_tmap_u8(&tmB, db, n_pad, U8_ROW, TS_BN) || !make_tmap_u8(&tmN, digits, n_pad, U8_NROW, TS_BN)) return cudaErrorUnknown;
  U8Params p;
  p.n = n;
  p.nq = nq;
  p.s_max = s_max;
  p.pieces = reinterpret_cast<const int4*>(d_pieces);
  p.pos_base = pos_base;
  p.cand = cand;
  p.cand_cnt = cand_cnt;
  p.cand_thr = cand_thr;
  int kp_default;
  tc_candidate_shape(k, &kp_default, &p.cap);
  if (p.cap < 128) return cudaErrorInvalidValue;
  p.kprime = std::max(k + 1, std::min(kprime, kp_default));
  p.slack = std::max(8, p.kprime / 2);
  p.hwm = std::min(p.cap / 2, std::max(64, 3 * p.kprime));
  p.refresh_mask = 15;
  p.gthr = gthr;
  p.q = q;
  p.m_half = m_half;
  p.counters = nullptr;
  p.cand_cut = range_cut;
  if (range_cut) p.cap = tc_range_cap();
  {
    const char* dbg = nb200_env("NB200_TC_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
  }
  const char* count_env = nb200_env("NB200_TC_COUNT");
  if (count_env && count_env[0] == '1') {  // diagnostics only: prints the sums of the previous launch
    static unsigned long long* d_ctr = nullptr;
    if (!d_ctr) {
      cudaMalloc(&d_ctr, 256);
    } else {
      unsigned long long h[18];
      cudaStreamSynchronize(stream);
      cudaMemcpy(h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost);
      const double c = (double)n_cta;
      fprintf(stderr, "tc_scan_u8: slow-path tiles (lane 0s) %llu, forced compactions %llu, deferred %llu | cycles per CTA: mma wait-tempty "
                      "%.0f wait-full %.0f issue %.0f | epilogue (per warp) wait-tfull %.0f drain %.0f process %.0f\n",
              h[1], h[2], h[3], h[11] / c, h[12] / c, h[13] / c, h[14] / c / 8, h[15] / c / 8, h[16] / c / 8);
    }
    cudaMemsetAsync(d_ctr, 0, 256, stream);
    p.counters = d_ctr;
  }
  p.n_stage = 16;
  const size_t smem = 1024 + (size_t)p.n_stage * U8_STAGE + (2 * 16 + 4 * U8_NBUF + 2) * 8 + 16;
  cudaError_t e;
#define NB_U8(KPL, REG, RANGE)                                                                                          \
  e = cudaFuncSetAttribute(tc_scan_u8_kernel<KPL, REG, RANGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
  if (e != cudaSuccess) return e;                                                                                       \
  tc_scan_u8_kernel<KPL, REG, RANGE><<<n_cta, TS_THREADS, smem, stream>>>(tmB, tmN, p);
  if (range_cut) {
    NB_U8(8, false, true);
  } else if (k + 4 <= TS_RK && kprime <= k + 6 && p.cap == 256) {
    p.kprime = TS_RK;
    p.slack = 8;
    NB_U8(8, true, false);
  } else if (p.cap == 256) {
    NB_U8(8, false, false);
  } else {
    NB_U8(16, false, false);
  }
#undef NB_U8
  e = cudaGetLastError();
  if (e != cudaSuccess)
    fprintf(stderr, "nmslib_b200: tc_scan_u8 launch (grid %d, smem %zu) failed: %s\n", n_cta, smem, cudaGetErrorString(e));
  return e;
}

int tc_block_queries() { return TC_QB; }
int tc_block_points() { return TC_BN; }
int tc_kblock_words() { return TC_KB; }

namespace {
__global__ void tc_fill_ones_kernel(float* __restrict__ ones) {  // [128][32]: 1.0 in columns 0..2
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < TC_BM * TC_KB) ones[i] = (i % TC_KB) < 3 ? 1.0f : 0.0f;
}
}  // namespace

cudaError_t launch_tc_prep_db(const float* db, int n, int n_pad, int row_words, int mode, float* bias, float* norm2,
                              float* db_unit, float* nblock, float* ones, unsigned* max_norm_bits,
                              int* inexact_flag, cudaStream_t stream) {
  const int threads = 256;
  const int blocks = (int)(((size_t)n_pad * 32 + threads - 1) / threads);
  tc_prep_db_kernel<<<blocks, threads, 0, stream>>>(db, n, n_pad, row_words, mode, bias, norm2, db_unit, nblock,
                                                    max_norm_bits, inexact_flag);
  if (ones) tc_fill_ones_kernel<<<(TC_BM * TC_KB + 255) / 256, 256, 0, stream>>>(ones);
  return cudaGetLastError();
}

// Decomposition of the (query block x tile) grid over the SMs (one CTA per SM).
//  * aligned: every query block is cut into the same `s` segments; q_blocks * s CTAs.  Chosen when some s
//    fills >= 80 % of the last wave: co-scheduled CTAs then stream the same tiles and share them in L2.
//  * linear (few query blocks): equal linear ranges, `sm_count` CTAs, a CTA may span two query blocks.
void tc_plan(int nq, int n, int k, int sm_count, int bn, int* n_cta, int* work_per_cta, int* s_max, int* aligned) {
  int kprime, cap;
  tc_candidate_shape(k, &kprime, &cap);
  const long q_blocks = (nq + TC_QB - 1) / TC_QB;
  const long n_tiles = (n + bn - 1) / bn;
  const long total = q_blocks * n_tiles;
  // the re-rank sorts s_max * cap keys per query in shared memory: bound the pieces per query block
  const long max_pieces = std::min<long>(std::min<long>(64, std::max<long>(2, 16384 / cap)), std::max<long>(4, 3072 / kprime));
  if (q_blocks * 4 >= sm_count || q_blocks * n_tiles <= sm_count) {
    long best = 1;
    double best_eff = 0;
    for (long sp = 1; sp <= std::min<long>(n_tiles, max_pieces); ++sp) {
      const long ctas = q_blocks * sp;
      const long waves = (ctas + sm_count - 1) / sm_count;
      const double eff = (double)ctas / (double)(waves * sm_count);
      if (eff > best_eff + 1e-9) {
        best_eff = eff;
        best = sp;
      }
      if (eff >= 0.8) break;
    }
    const long w = (n_tiles + best - 1) / best;
    const long segs = (n_tiles + w - 1) / w;
    *n_cta = (int)(q_blocks * segs);
    *work_per_cta = (int)w;
    *s_max = (int)segs;
    *aligned = 1;
    return;
  }
  long g = std::min<long>(sm_count, total);
  for (;; --g) {
    const long w = (total + g - 1) / g;
    long smax = 1;
    for (long qb = 0; qb < q_blocks; ++qb) {
      const long first = (qb * n_tiles) / w, last = ((qb + 1) * n_tiles - 1) / w;
      smax = std::max(smax, last - first + 1);
    }
    if (smax <= max_pieces || g == 1) {
      *n_cta = (int)((total + w - 1) / w);
      *work_per_cta = (int)w;
      *s_max = (int)smax;
      *aligned = 0;
      return;
    }
  }
}

cudaError_t launch_tc_split_rows(const float* src, size_t rows, int row_words, float scale, int layout, float* dst,
                                 cudaStream_t stream) {
  const size_t total = rows * (size_t)row_words;
  if (total == 0) return cudaSuccess;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  tc_split_rows_kernel<<<blocks, 256, 0, stream>>>(src, rows, row_words, scale, layout, dst);
  return cudaGetLastError();
}

cudaError_t launch_tc_prep_queries(const float* q, float* out, size_t words, float scale, int* inexact_flag,
                                   cudaStream_t stream) {
  int blocks = (int)std::min<size_t>((words + 255) / 256, 148 * 8);
  if (blocks < 1) blocks = 1;
  tc_prep_queries_kernel<<<blocks, 256, 0, stream>>>(q, out, words, scale, inexact_flag);
  return cudaGetLastError();
}

// cand capacity per (unit,row) and survivors per compaction for a given k
void tc_candidate_shape(int k, int* kprime, int* cap) {
  int kp = k + 22 < 2 * k ? k + 22 + (k / 4) : 2 * k;  // headroom for the certificate
  if (kp < k + 22) kp = k + 22;
  kp = (kp + 31) / 32 * 32;
  int c = kp <= 96 ? 256 : 512;  // (256 even for k' = 32: half as many compactions as 128, see profiles/README.md)
  if (kp > c - 64) kp = c - 64;
  *kprime = kp;
  *cap = c;
}
int tc_max_k() { return 256; }

cudaError_t launch_tc_scan(const float* qa, size_t q_pad, const float* dbB, size_t n_pad, const float* nblock,
                           const float* ones, int n, int nq, int row_words, int k, uint32_t pos_base, int n_cta,
                           int work_per_cta, int s_max, int aligned, int kprime, uint64_t* cand, int* cand_cnt,
                           float* cand_thr, uint32_t* gthr, cudaStream_t stream) {
  if (n <= 0 || nq <= 0) return cudaSuccess;
  if (row_words % TC_KB) return cudaErrorInvalidValue;
  CUtensorMap tmA, tmB, tmN, tmO;
  if (!make_tmap(&tmA, qa, q_pad, row_words) || !make_tmap(&tmB, dbB, n_pad, row_words)) return cudaErrorUnknown;
  const bool use_nb = nblock != nullptr;
  if (use_nb) {
    if (!make_tmap(&tmN, nblock, n_pad, TC_KB) || !make_tmap(&tmO, ones, TC_BM, TC_KB)) return cudaErrorUnknown;
  } else {
    tmN = tmB;
    tmO = tmA;
  }
  TcParams p;
  p.n = n;
  p.nq = nq;
  p.n_kb = row_words / TC_KB;
  p.n_tiles = (n + TC_BN - 1) / TC_BN;
  p.q_blocks = (nq + TC_QB - 1) / TC_QB;
  p.work_per_cta = work_per_cta;
  p.total_work = p.q_blocks * p.n_tiles;
  p.s_max = s_max;
  p.aligned = aligned;
  p.pos_base = pos_base;
  p.cand = cand;
  p.cand_cnt = cand_cnt;
  p.cand_thr = cand_thr;
  int kp_default;
  tc_candidate_shape(k, &kp_default, &p.cap);
  p.kprime = std::max(k + 1, std::min(kprime, kp_default));
  p.slack = std::max(8, p.kprime / 4);
  p.hwm = std::min(p.cap / 2, std::max(64, 2 * p.kprime));
  p.gthr = gthr;
  p.use_nb = use_nb ? 1 : 0;
  {
    const char* dbg = nb200_env("NB200_TC_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
  }
  p.pieces = nullptr;
  p.a_resident = (2 * p.n_kb * CHUNK_BYTES <= 128 * 1024) ? 1 : 0;
  const int a_bytes = p.a_resident ? 2 * p.n_kb * CHUNK_BYTES : 0;
  const int ones_bytes = use_nb ? CHUNK_BYTES : 0;
  const int stage_bytes = p.a_resident ? CHUNK_BYTES : 3 * CHUNK_BYTES;
  const int budget = 214 * 1024;
  p.n_stage = (budget - a_bytes - ones_bytes) / stage_bytes;
  if (p.n_stage > 8) p.n_stage = 8;
  if (p.n_stage < 2) return cudaErrorInvalidValue;
  const size_t smem = 1024 + (size_t)a_bytes + ones_bytes + (size_t)p.n_stage * stage_bytes + (2 * 8 + 8) * 8 + 16;
  cudaError_t e;
#define NB_TC(KPL)                                                                                        \
  e = cudaFuncSetAttribute(tc_scan_kernel<KPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
  if (e != cudaSuccess) return e;                                                                         \
  tc_scan_kernel<KPL><<<n_cta, TC_THREADS, smem, stream>>>(tmA, tmB, tmN, tmO, p);
  if (p.cap == 256) {
    NB_TC(8);
  } else {
    NB_TC(16);
  }
#undef NB_TC
  e = cudaGetLastError();
  if (e != cudaSuccess)
    fprintf(stderr, "nmslib_b200: tc_scan launch (grid %d, smem %zu, stages %d) failed: %s\n", n_cta, smem, p.n_stage,
            cudaGetErrorString(e));
  return e;
}

bool tc_pair_enabled() { return nb200_option("tc_pair", 1) != 0; }
int tc_pair_block_points() { return TP_BN; }

// CTA-pair kernel for long rows: d_pieces / n_pairs from tc_ts_plan(nq, n, k, sm_count / 2, .., TP_BN, 2);
// s_max = candidate lists per query block = 2 x the plan's slots per block
cudaError_t launch_tc_scan_pair(const float* qa, size_t q_pad, const float* dbB, size_t n_pad, const float* nblock,
                                const float* ones, int n, int nq, int row_words, int k, uint32_t pos_base, int n_pairs,
                                const int* d_pieces, int s_max, int kprime, uint64_t* cand, int* cand_cnt,
                                float* cand_thr, uint32_t* gthr, cudaStream_t stream, uint32_t* range_cut) {
  if (n <= 0 || nq <= 0) return cudaSuccess;
  if (row_words % TC_KB) return cudaErrorInvalidValue;
  CUtensorMap tmA, tmB, tmN, tmO;
  if (!make_tmap(&tmA, qa, q_pad, row_words) || !make_tmap(&tmB, dbB, n_pad, row_words)) return cudaErrorUnknown;
  const bool use_nb = nblock != nullptr;
  if (use_nb) {
    if (!make_tmap(&tmN, nblock, n_pad, TC_KB) || !make_tmap(&tmO, ones, TC_BM, TC_KB)) return cudaErrorUnknown;
  } else {
    tmN = tmB;
    tmO = tmA;
  }
  TcParams p;
  p.n = n;
  p.nq = nq;
  p.n_kb = row_words / TC_KB;
  p.n_tiles = (n + TP_BN - 1) / TP_BN;
  p.q_blocks = (nq + TC_QB - 1) / TC_QB;
  p.work_per_cta = 0;
  p.total_work = p.q_blocks * p.n_tiles;
  p.s_max = s_max;
  p.aligned = 0;
  p.pieces = reinterpret_cast<const int4*>(d_pieces);
  p.pos_base = pos_base;
  p.cand = cand;
  p.cand_cnt = cand_cnt;
  p.cand_thr = cand_thr;
  int kp_default;
  tc_candidate_shape(k, &kp_default, &p.cap);
  p.kprime = std::max(k + 1, std::min(kprime, kp_default));
  p.slack = std::max(8, p.kprime / 4);
  p.hwm = std::min(p.cap / 2, std::max(64, 2 * p.kprime));
  p.gthr = gthr;
  p.cand_cut = range_cut;
  if (range_cut) p.cap = tc_range_cap();
  p.use_nb = use_nb ? 1 : 0;
  {
    const char* dbg = nb200_env("NB200_TC_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
  }
  p.a_resident = 0;
  const int ones_bytes = use_nb ? CHUNK_BYTES : 0;
  const int stage_bytes = 2 * CHUNK_BYTES;
  const int budget = 214 * 1024;
  p.n_stage = (budget - ones_bytes) / stage_bytes;
  if (p.n_stage > 8) p.n_stage = 8;
  const size_t smem = 1024 + (size_t)ones_bytes + (size_t)p.n_stage * stage_bytes + (2 * 8 + 12) * 8 + 16;
  cudaError_t e;
#define NB_TP(KPL, RANGE)                                                                                             \
  e = cudaFuncSetAttribute(tc_scan_pair_kernel<KPL, RANGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
  if (e != cudaSuccess) return e;                                                                                     \
  tc_scan_pair_kernel<KPL, RANGE><<<2 * n_pairs, TC_THREADS, smem, stream>>>(tmA, tmB, tmN, tmO, p);
  if (range_cut) {
    NB_TP(8, true);
  } else if (p.cap == 256) {
    NB_TP(8, false);
  } else {
    NB_TP(16, false);
  }
#undef NB_TP
  e = cudaGetLastError();
  if (e != cudaSuccess)
    fprintf(stderr, "nmslib_b200: tc_scan_pair launch (grid %d, smem %zu, stages %d) failed: %s\n", 2 * n_pairs, smem,
            p.n_stage, cudaGetErrorString(e));
  return e;
}

bool tc_ts_supported(int row_words) {
  static const bool off = [] {
    const char* e = nb200_env("NB200_TC_NO_TS");
    return e && e[0] == '1';
  }();
  return !off && row_words <= 128 && row_words % TC_KB == 0;
}
int tc_ts_block_points() { return TS_BN; }

// Work decomposition of the TS kernel: a table of pieces (query block, tile range, candidate slot) per CTA.
//  * whole waves of query blocks (>= sm_count of them): one CTA = one block over the whole shard; CTAs of a wave
//    sweep the same tiles together, so the L2 serves all but one of them;
//  * the remaining B' < sm_count blocks: g = floor(S / B') aligned segments per block (CTAs of a segment are
//    neighbours and share tiles in L2) covering the first part of the tiles, and the R = S - g*B' CTAs left
//    over take what remains of every block: whole tails first, unit j those of blocks j, R + j, ... (so all
//    left-over units sweep the same tile range at the same time, too), then chunks of the B' mod R tails that
//    remain, cut at common boundaries; the segment length is chosen so that all units finish together.
void tc_ts_plan(int nq, int n, int k, int sm_count, std::vector<int>* table, int* n_cta, int* s_max, int bn,
                int lists_per_piece, std::vector<int>* block_slots) {
  int kprime, cap;
  tc_candidate_shape(k, &kprime, &cap);
  if (bn <= 0) bn = TS_BN;
  const int B = (nq + TC_QB - 1) / TC_QB;
  const int T = (n + bn - 1) / bn;
  const int S = std::max(1, sm_count);
  // pieces per query block: bounded by the re-rank (64 lists) and by k' -- every piece ends with its own k' best
  // below a threshold that is only as tight as the piece is long, and the re-rank sorts at most 8192 live keys
  const int max_pieces =
      std::max(4, std::min(std::min(64, std::max(4, 16384 / cap)), std::max(4, 3072 / kprime)) / std::max(1, lists_per_piece));
  std::vector<std::vector<int4>> ctas;
  std::vector<int> slots(B, 0);
  auto add_piece = [&](std::vector<int4>& c, int qb, int t0, int t1) {
    if (t1 <= t0) return;
    c.push_back(make_int4(qb, t0, t1, slots[qb]++));
  };
  const int full = (B / S) * S;
  for (int qb = 0; qb < full; ++qb) {
    ctas.emplace_back();
    add_piece(ctas.back(), qb, 0, T);
  }
  const int Bp = B - full;
  if (Bp > 0) {
    // (behind whole waves keep the lists per block few: every block's candidate buffers are sized by s_max)
    // (and a piece should be long enough to pay for its start-up: >= 16 tiles unless the shard is tiny)
    int g = std::max(1, std::min(std::min(S / Bp, full > 0 ? 4 : max_pieces - 3), std::max(1, T / 16)));
    int R = (g == S / Bp) ? S - g * Bp : 0;
    // Left-over units take WHOLE tails first (unit j: blocks j, R + j, ...: all units sweep the same tile range of
    // different blocks at the same time, so the L2 serves all but one of them, like the aligned segments), then the
    // Bp mod R tails that remain are cut into c chunks at common boundaries.  f = tails per left-over unit.
    const int whole = R > 0 ? Bp / R : 0, rem = R > 0 ? Bp % R : 0;
    if (R > 0 && whole + (rem > 0 ? 1 : 0) > TS_MAXP - 2) R = 0;   // too many blocks per left-over unit
    int c = (R > 0 && rem > 0) ? std::max(1, std::min(R / rem, std::max(1, max_pieces - g))) : 0;
    const double f = R > 0 ? (double)whole + (c > 0 ? 1.0 / c : 0.0) : 0.0;
    // every unit finishes at the same time: Wa = f * (T - g * Wa)
    long Wa = R > 0 ? (long)std::ceil(f * T / (1.0 + f * g)) : (T + g - 1) / g;
    if (Wa < 1) { Wa = 1; R = 0; }
    if (R > 0 && (long)g * Wa >= T) R = 0;
    if (R == 0) {
      Wa = std::max<long>(1, (T + g - 1) / g);
      g = (int)((T + Wa - 1) / Wa);
    }
    const long Ta = std::min<long>((long)g * Wa, T);
    // aligned part: CTA index = seg * Bp + block, so the CTAs of a segment are launched together
    for (int seg = 0; seg < g; ++seg)
      for (int b = 0; b < Bp; ++b) {
        const long t0 = (long)seg * Wa, t1 = std::min<long>(t0 + Wa, R > 0 ? Ta : T);
        if (t1 <= t0) continue;
        ctas.emplace_back();
        add_piece(ctas.back(), full + b, (int)t0, (int)t1);
      }
    if (R > 0) {
      const long r = T - Ta;
      const long ce = c > 0 ? (r + c - 1) / c : 0;
      for (int j = 0; j < R; ++j) {
        std::vector<int4> u;
        for (int p = 0; p < whole; ++p) add_piece(u, full + p * R + j, (int)Ta, (int)T);
        if (c > 0 && j < rem * c) {  // unit q * rem + b takes chunk q of the b-th remaining tail
          const int q = j / rem, b = j % rem;
          const long t0 = Ta + (long)q * ce, t1 = std::min<long>(t0 + ce, T);
          add_piece(u, full + whole * R + b, (int)t0, (int)t1);
        }
        if (!u.empty()) ctas.push_back(u);
      }
    }
  }
  int smax = 1;
  for (int v : slots) smax = std::max(smax, v);
  table->assign(ctas.size() * TS_MAXP * 4, -1);
  for (size_t c = 0; c < ctas.size(); ++c)
    for (size_t i = 0; i < ctas[c].size() && i < (size_t)TS_MAXP; ++i) {
      int* e = table->data() + (c * TS_MAXP + i) * 4;
      e[0] = ctas[c][i].x;
      e[1] = ctas[c][i].y;
      e[2] = ctas[c][i].z;
      e[3] = ctas[c][i].w;
    }
  *n_cta = (int)ctas.size();
  *s_max = smax;
  if (block_slots) *block_slots = slots;  // pieces (candidate slots in use) of every query block
}

cudaError_t launch_tc_scan_ts(const float* q, const float* dbB, size_t n_pad, const float* nblock, const float* ones,
                              int n, int nq, int row_words, int k, int kprime, float scale, uint32_t pos_base,
                              int n_cta, int s_max, const int* d_pieces, uint64_t* cand, int* cand_cnt,
                              float* cand_thr, uint32_t* gthr, int* inexact_flag, cudaStream_t stream,
                              uint32_t* range_cut) {
  if (n <= 0 || nq <= 0) return cudaSuccess;
  if (!tc_ts_supported(row_words)) return cudaErrorInvalidValue;
  CUtensorMap tmB, tmN, tmO;
  if (!make_tmap(&tmB, dbB, n_pad, row_words, TS_BN)) return cudaErrorUnknown;
  const bool use_nb = nblock != nullptr;
  if (use_nb) {
    if (!make_tmap(&tmN, nblock, n_pad, TC_KB, TS_BN) || !make_tmap(&tmO, ones, TC_BM, TC_KB)) return cudaErrorUnknown;
  } else {
    tmN = tmB;
    tmO = tmB;
  }
  TsParams p;
  p.n = n;
  p.nq = nq;
  p.n_kb = row_words / TC_KB;
  p.s_max = s_max;
  p.pieces = reinterpret_cast<const int4*>(d_pieces);
  p.pos_base = pos_base;
  p.cand = cand;
  p.cand_cnt = cand_cnt;
  p.cand_thr = cand_thr;
  int kp_default;
  tc_candidate_shape(k, &kp_default, &p.cap);
  if (p.cap < 128) return cudaErrorInvalidValue;  // (the register mode of tc_scan_kernel<0> is not built here)
  // survivors of a compaction: kprime .. kprime + slack; rows are compacted (deferred, one per warp and tile)
  // once they hold more than hwm keys -- early, because the threshold only tightens at a compaction
  p.kprime = std::max(k + 1, std::min(kprime, kp_default));
  p.slack = std::max(8, p.kprime / 2);
  p.hwm = std::min(p.cap / 2, std::max(64, 3 * p.kprime));
  p.warm_max = p.kprime <= 32 ? 64 : 0;
  p.refresh_mask = 15;
  if (const char* e = nb200_env("NB200_TC_HWM")) p.hwm = std::max(p.kprime + p.slack + 8, std::min(p.cap - 40, atoi(e)));
  if (const char* e = nb200_env("NB200_TC_WARM")) p.warm_max = p.kprime <= 32 ? std::max(0, atoi(e)) : 0;
  if (const char* e = nb200_env("NB200_TC_REFRESH")) p.refresh_mask = std::max(0, atoi(e));
  p.gthr = gthr;
  p.cand_cut = range_cut;
  if (range_cut) {  // range mode: fixed thresholds, so no warm start
    p.cap = tc_range_cap();
    p.warm_max = 0;
  }
  p.use_nb = use_nb ? 1 : 0;
  {
    const char* dbg = nb200_env("NB200_TC_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
  }
  p.q = q;
  p.row_words = row_words;
  p.scale = scale;
  p.inexact_flag = inexact_flag;
  p.counters = nullptr;
  const char* count_env = nb200_env("NB200_TC_COUNT");
  if (count_env && count_env[0] == '1') {  // diagnostics only: synchronous, prints the epilogue's event counts of the previous launch
    static unsigned long long* d_ctr = nullptr;
    if (!d_ctr) {
      cudaMalloc(&d_ctr, 256);
    } else {
      unsigned long long h[18];
      cudaStreamSynchronize(stream);
      cudaMemcpy(h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost);
      fprintf(stderr, "tc_scan_ts counters: (unused) %llu, slow-path entries %llu, forced compactions %llu, deferred %llu, warp-chunks %llu\n",
              h[0], h[1], h[2], h[3], h[4]);
      const double c = (double)n_cta;
      fprintf(stderr, "  cycles per CTA: producer wait-empty %.0f of %.0f | mma wait-afull %.0f wait-tempty %.0f wait-full %.0f issue %.0f | "
                      "epilogue (per warp) wait-tfull %.0f drain %.0f process %.0f setup %.0f\n",
              h[8] / c, h[9] / c, h[10] / c, h[11] / c, h[12] / c, h[13] / c, h[14] / c / 8, h[15] / c / 8, h[16] / c / 8, h[17] / c / 8);
    }
    cudaMemsetAsync(d_ctr, 0, 256, stream);
    p.counters = d_ctr;
  }
  const int ones_bytes = use_nb ? CHUNK_BYTES : 0;
  const int stage_bytes = (p.n_kb + p.use_nb) * TS_CHUNK;
  const int budget = 225 * 1024;
  p.n_stage = (budget - ones_bytes) / stage_bytes;
  if (p.n_stage > 8) p.n_stage = 8;
  if (p.n_stage < 2) return cudaErrorInvalidValue;
  const size_t smem = 1024 + (size_t)ones_bytes + (size_t)p.n_stage * stage_bytes + (2 * 8 + 12) * 8 + 16;
  cudaError_t e;
#define NB_TS(KPL, REG, RANGE)                                                                                          \
  e = cudaFuncSetAttribute(tc_scan_ts_kernel<KPL, REG, RANGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
  if (e != cudaSuccess) return e;                                                                                       \
  tc_scan_ts_kernel<KPL, REG, RANGE><<<n_cta, TS_THREADS, smem, stream>>>(tmB, tmN, tmO, p);
  static const bool no_reg = [] {
    const char* e2 = nb200_env("NB200_TC_NO_REG");
    return e2 && e2[0] == '1';
  }();
  // register list (16 ranks): k <= 12 leaves the certificate a margin of >= 4 ranks; a margin raised by the
  // engine (certificates failed on inexact data) selects the buffer path with its larger k'
  if (range_cut) {
    NB_TS(8, false, true);
  } else if (k + 4 <= TS_RK && kprime <= k + 6 && p.cap == 256 && !no_reg) {
    p.kprime = TS_RK;  // the register list always holds 16
    p.slack = 8;
    if (!nb200_env("NB200_TC_WARM")) p.warm_max = 0;  // exact thresholds make the cold start cheaper than the re-scan
    NB_TS(8, true, false);
  } else if (p.cap == 256) {
    NB_TS(8, false, false);
  } else {
    NB_TS(16, false, false);
  }
#undef NB_TS
  e = cudaGetLastError();
  if (e != cudaSuccess)
    fprintf(stderr, "nmslib_b200: tc_scan_ts launch (grid %d, smem %zu, stages %d) failed: %s\n", n_cta, smem,
            p.n_stage, cudaGetErrorString(e));
  return e;
}

// Error model of pass 1 (DESIGN.md "certificate"): TF32 operands are fp32 with the low 13 mantissa
// bits dropped (relative 2^-10 each when truncated), products exact, fp32 accumulation over D terms.
static void pass1_eps(int row_words, float* eps_exact, float* eps_inexact) {
  *eps_exact = (float)row_words * 2.384185791015625e-07f;         // D * 2^-22  (accumulation only)
  *eps_inexact = 2.0f * 0.0009765625f * 1.01f + *eps_exact;       // 2 * 2^-10 + accumulation
}

int tc_range_cap() { return 256; }

cudaError_t launch_tc_range_threshold(const float* q, int nq, int row_words, int mode, int take_sqrt, const float* radii,
                                      float x_max, int db_inexact, uint32_t* gthr, cudaStream_t stream) {
  if (nq <= 0) return cudaSuccess;
  float eps_exact, eps_inexact;
  pass1_eps(row_words, &eps_exact, &eps_inexact);
  tc_range_threshold_kernel<<<(nq + 7) / 8, 256, 0, stream>>>(q, nq, row_words, mode, take_sqrt, radii, x_max,
                                                              eps_inexact, eps_exact, db_inexact, gthr);
  return cudaGetLastError();
}

cudaError_t launch_tc_range_threshold_u8(const uint8_t* q, int nq, const float* radii, int m_half, uint32_t* gthr,
                                         cudaStream_t stream) {
  if (nq <= 0) return cudaSuccess;
  tc_range_threshold_u8_kernel<<<(nq + 7) / 8, 256, 0, stream>>>(q, nq, radii, m_half, gthr);
  return cudaGetLastError();
}

// live keys the re-rank's sort buffer must hold for a query with n_lists candidate lists of `cap` keys
int tc_rerank_items(int n_lists, int cap, int k, int n) {
  return std::min(n_lists * cap, std::max(std::max(2048, 4 * k), std::min(n, 8192)));  // (small shards: all rows)
}
int tc_rerank_pow2(int n_lists, int cap, int k, int n) {
  int p2 = 32;
  const int items = tc_rerank_items(n_lists, cap, k, n);
  while (p2 < items || p2 < k) p2 <<= 1;
  return p2;
}

cudaError_t launch_tc_rerank(const float* db, const float* queries, const float* db_norm2, int n, int nq,
                             int row_words, int k, int n_split, int mode, uint32_t pos_base, const uint64_t* cand,
                             const int* cand_cnt, const float* cand_thr, float x_max, const int* inexact_flags,
                             uint64_t* out_keys, int* out_cert, cudaStream_t stream, int q_begin, int q_count,
                             int n_lists, float eps_override, int* fb_count, int* fb_idx, const uint8_t* db_u8,
                             const uint8_t* q_u8, float abs_err, int int_keys) {
  if (nq <= 0) return cudaSuccess;
  if (q_count < 0) q_count = nq - q_begin;
  if (q_count <= 0) return cudaSuccess;
  if (n_lists <= 0 || n_lists > n_split) n_lists = n_split;
  RerankParams p;
  p.q_begin = q_begin;
  p.n_lists = n_lists;
  p.fb_count = fb_count;
  p.fb_idx = fb_idx;
  p.db_u8 = db_u8;
  p.q_u8 = q_u8;
  p.abs_err = abs_err;
  p.int_keys = int_keys;
  p.db = db;
  p.queries = queries;
  p.db_norm2 = db_norm2;
  p.nq = nq;
  p.row_words = row_words;
  p.k = k;
  p.n_split = n_split;
  int kprime;
  tc_candidate_shape(k, &kprime, &p.cap);
  p.mode = mode;
  p.pos_base = pos_base;
  p.cand = cand;
  p.cand_cnt = cand_cnt;
  p.cand_thr = cand_thr;
  pass1_eps(row_words, &p.eps_exact, &p.eps_inexact);
  if (eps_override > 0.f) p.eps_exact = p.eps_inexact = eps_override;  // (split operands: see Engine::enable_split)
  p.x_max = x_max;
  p.inexact_flags = inexact_flags;
  p.out_keys = out_keys;
  p.out_cert = out_cert;
  p.debug_cert = nb200_env("NB200_TC_DEBUG_CERT") != nullptr;
  if (n_split > 64) return cudaErrorInvalidValue;
  // sort buffer: the live keys (pass-1 rank below the final threshold) are a few times k'; a query with more
  // than this many is left uncertified and re-run exactly
  int items = tc_rerank_items(n_lists, p.cap, k, n);
  int p2 = 1;
  while (p2 < items || p2 < k) p2 <<= 1;
  const size_t smem = (size_t)p2 * 12 + 16;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(tc_rerank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    fprintf(stderr, "nmslib_b200: tc_rerank cudaFuncSetAttribute(%zu) failed: %s\n", smem, cudaGetErrorString(e));
    return e;
  }
  // 8 warps when the exact evaluation dominates (long rows, many candidates): twice the candidate rows in flight
  const int rr_threads = (row_words > 128 || k >= 32) ? 256 : 128;  // (256 threads on config 2: 0.066 -> 0.128 ms per launch)
  tc_rerank_kernel<<<q_count, rr_threads, smem, stream>>>(p, p2);
  e = cudaGetLastError();
  if (e != cudaSuccess)
    fprintf(stderr, "nmslib_b200: tc_rerank launch (grid %d, smem %zu, items %d) failed: %s\n", nq, smem, p2,
            cudaGetErrorString(e));
  return e;
}

}  // namespace nb200
