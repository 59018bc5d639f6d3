// scan_exact.cu -- K1x / K2x: exact brute-force kNN on the CUDA cores.
//
// Replaces SeqSearch<dist_t>::Search(KNNQuery*) (src/method/seqsearch.cc:144-150), the
// per-pair distance functions behind it (L2SqrSIMD distcomp_lp.cc:304-365,
// NormScalarProductSIMD / ScalarProductSIMD distcomp_scalar.cc:84-245,
// l2SqrSIFTPrecomp* distcomp_l2sqr_sift.cc:41-151) and the KNNQueue result heap
// (knnqueue.h:55-64) for a whole batch of queries in one launch.
//
// Role in the engine: the l2 / l2sqr path evaluates sum (x-y)^2 directly in fp32 --
// the reference's own formula, no norm expansion, hence no cancellation -- so it is
// (a) the first correct path, (b) the re-run path for queries whose tensor-core
// candidate set could not be certified (scan_tc.cu), and (c) the uint8 dp4a path
// with exact int32 distances.
//
// Shape: CTA = 128 queries x a contiguous range of 128-point tiles; 256 threads, each
// owning an 8x8 register micro-tile; operands staged through a 3-deep cp.async ring
// (row stride padded to 20 words: 128-bit shared loads are conflict free).  The
// distance matrix never leaves registers: every value is compared with its query's
// current k-th best (shared memory); survivors (rare once warm) go through a small
// shared-memory queue into per-query sorted lists of 64-bit (distance, position) keys.
//
// RANGE variant (batched range queries over l1 / linf, DESIGN.md K5b): the same main loop, but every query row has a
// fixed threshold T_q (range_threshold) for the whole scan, and survivors go straight into the query's candidate
// list of this split, in the layout range_verify_kernel (range_scan.cu) reads.
#include "common.cuh"
#include "kernels.h"

namespace nb200 {

namespace {

constexpr int BQ = 128;      // queries per CTA
constexpr int BN = 128;      // points per tile
constexpr int BW = 16;       // 32-bit words of each row per pipeline stage
constexpr int LDW = 20;      // padded shared-memory row stride (words)
constexpr int NT = 256;      // threads
constexpr int NSTAGE = 3;    // cp.async ring depth
constexpr int QCAP = 1024;   // candidate queue entries

template <int MODE>
struct Acc { using type = float; };
template <>
struct Acc<SCAN_SIFT> { using type = int; };

template <int MODE>
__device__ __forceinline__ void accum4(const uint4& a, const uint4& b, typename Acc<MODE>::type& acc) {
  if constexpr (MODE == SCAN_SIFT) {
    unsigned u = (unsigned)acc;
    u = __dp4a(a.x, b.x, u);
    u = __dp4a(a.y, b.y, u);
    u = __dp4a(a.z, b.z, u);
    u = __dp4a(a.w, b.w, u);
    acc = (int)u;
  } else if constexpr (MODE == SCAN_L2) {
    float d0 = __uint_as_float(a.x) - __uint_as_float(b.x);
    float d1 = __uint_as_float(a.y) - __uint_as_float(b.y);
    float d2 = __uint_as_float(a.z) - __uint_as_float(b.z);
    float d3 = __uint_as_float(a.w) - __uint_as_float(b.w);
    acc = fmaf(d0, d0, acc);
    acc = fmaf(d1, d1, acc);
    acc = fmaf(d2, d2, acc);
    acc = fmaf(d3, d3, acc);
  } else if constexpr (MODE == SCAN_L1) {  // L1NormSIMD, distcomp_lp.cc:190-251
    acc += fabsf(__uint_as_float(a.x) - __uint_as_float(b.x));
    acc += fabsf(__uint_as_float(a.y) - __uint_as_float(b.y));
    acc += fabsf(__uint_as_float(a.z) - __uint_as_float(b.z));
    acc += fabsf(__uint_as_float(a.w) - __uint_as_float(b.w));
  } else if constexpr (MODE == SCAN_LINF) {  // LInfNormSIMD, distcomp_lp.cc:77-139
    acc = fmaxf(acc, fmaxf(fmaxf(fabsf(__uint_as_float(a.x) - __uint_as_float(b.x)),
                                 fabsf(__uint_as_float(a.y) - __uint_as_float(b.y))),
                           fmaxf(fabsf(__uint_as_float(a.z) - __uint_as_float(b.z)),
                                 fabsf(__uint_as_float(a.w) - __uint_as_float(b.w)))));
  } else {
    acc = fmaf(__uint_as_float(a.x), __uint_as_float(b.x), acc);
    acc = fmaf(__uint_as_float(a.y), __uint_as_float(b.y), acc);
    acc = fmaf(__uint_as_float(a.z), __uint_as_float(b.z), acc);
    acc = fmaf(__uint_as_float(a.w), __uint_as_float(b.w), acc);
  }
}

// exact cosine distance, data point left / query right (distcomp_scalar.cc:150-167, 268-271)
__device__ __forceinline__ float nsp_exact(float dot, float n_x, float n_q) {
  const float eps = 2.0f * 1.17549435e-38f;
  if (n_x < eps || n_q < eps) return 0.f;
  return fmaxf(-1.f, fminf(1.f, dot / sqrtf(n_x) / sqrtf(n_q)));
}
__device__ __forceinline__ float cosine_exact(float dot, float n_x, float n_q) {
  return fmaxf(0.f, 1.f - nsp_exact(dot, n_x, n_q));
}
// AngularDistance, distcomp_scalar.cc:254-258
__device__ __forceinline__ float angular_exact(float dot, float n_x, float n_q) { return acosf(nsp_exact(dot, n_x, n_q)); }

// Batched range queries: the pass-1 threshold T_q of radius r (a row is a candidate when its pass-1 value <= T_q).
// Invariant: every row whose range_row_dist value is <= r has pass-1 value <= T_q.
// Both sums use the same terms t_i = |fl(x_i - y_i)| (fabsf of the same subtraction; fl(q - x) = -fl(x - q)); pass 1
// adds them sequentially over the row, range_row_dist in lane-strided float4 groups and a butterfly.
//  - linf: the max of one set of terms does not depend on the order, and fmaxf skips NaN terms the same way in
//    both, so the two values are equal bit for bit: T_q = r.
//  - l1: the terms are >= 0, so any summation order of the D = row_words terms (padding words add exact zeros) is
//    within gamma S of the exact sum S, gamma = (D - 1) u / (1 - (D - 1) u), u = 2^-24 (no underflow error: fp32
//    addition is exact in the subnormal range; no overflow below T_q: every partial sum is <= the final sum).
//    verified <= r  =>  S <= r / (1 - gamma)  =>  pass1 <= S (1 + gamma) <= r (1 + gamma) / (1 - gamma), evaluated in
//    double, rounded up to float and raised by one more ulp for the double rounding; an overflow becomes +inf.
// r = +inf admits every row, +inf values included; a NaN radius admits none (value <= NaN is false, as it is for the
// per-query scan); NaN values (a NaN term) are NaN in both sums and never selected.
template <int MODE>
__device__ __forceinline__ float range_threshold(float r, int row_words) {
  if constexpr (MODE == SCAN_LINF) {
    return r;
  } else {
    const double x = (row_words - 1) * 0x1p-24, gamma = x / (1.0 - x);
    if (!(gamma < 1.0)) return INFINITY;  // rows of 2^23 words and more: no bound, verification filters everything
    return nextafterf(__double2float_ru((double)r * (1.0 + gamma) / (1.0 - gamma)), INFINITY);
  }
}

// RANGE (MODE SCAN_L1 / SCAN_LINF only): partial / d_nq / glists unused; k = list capacity; radii[nq] the float radii;
// cand [q_blocks of 256][n_split][256][k] keys (ordered pass-1 value << 32 | position), in arrival order;
// cand_cnt / cut [q_blocks of 256][n_split][256], written for every query row of the CTA (a 128-query CTA fills one
// half of a 256-query block; the split index is the list index).  A full list stores the smallest position it
// dropped in its cut and stops selecting in the next tile, so every survivor below the cut was kept.
template <int MODE, bool RANGE = false>
__global__ void __launch_bounds__(NT, (MODE == SCAN_SIFT) ? 1 : 1)
scan_exact_kernel(const uint32_t* __restrict__ db, const uint32_t* __restrict__ qs,
                  const void* __restrict__ db_aux_v, const void* __restrict__ q_aux_v, int n, int nq,
                  int row_words, int k, int tiles_per_split, uint32_t pos_base,
                  uint64_t* __restrict__ partial, int n_split, const int* __restrict__ d_nq,
                  uint64_t* __restrict__ glists, const float* __restrict__ radii, uint64_t* __restrict__ cand,
                  int* __restrict__ cand_cnt, uint32_t* __restrict__ cut) {
  static_assert(!RANGE || MODE == SCAN_L1 || MODE == SCAN_LINF, "range mode: l1 / linf");
  using acc_t = typename Acc<MODE>::type;
  if (d_nq) {  // query count decided on the device (the re-run of uncertified queries): surplus blocks leave at once
    nq = min(nq, *d_nq);
    if ((int)blockIdx.y * BQ >= nq) return;
  }
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* tiles = reinterpret_cast<uint32_t*>(smem_raw);                     // NSTAGE*(BQ+BN)*LDW
  // per-query sorted lists: BQ * k keys in shared memory, or -- k above scan_exact_smem_k(): the reference's KNNQueue
  // has no capacity limit (knnqueue.h:55-64) -- this block's slice of a global scratch array (slower, but unbounded)
  uint64_t* slists = reinterpret_cast<uint64_t*>(tiles + NSTAGE * (BQ + BN) * LDW);
  uint64_t* lists = glists ? glists + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (size_t)BQ * k : slists;
  uint64_t* thr_key = slists + (glists || RANGE ? 0 : (size_t)BQ * k);         // BQ (RANGE: no lists; k = list cap)
  uint64_t* qkey = thr_key + BQ;                                                // QCAP
  uint32_t* thr_fast = reinterpret_cast<uint32_t*>(qkey + QCAP);                // BQ (bit pattern)
  int* cnt = reinterpret_cast<int*>(thr_fast + BQ);                             // BQ
  uint16_t* qrow = reinterpret_cast<uint16_t*>(cnt + BQ);                       // QCAP
  uint32_t* rcut = reinterpret_cast<uint32_t*>(thr_key);  // RANGE: BQ cuts (thr_key unused); thr_fast = T_q
  __shared__ int qcount;

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int split = blockIdx.x;
  const int q0 = blockIdx.y * BQ;
  const int n_tiles_total = (n + BN - 1) / BN;
  const int t0 = split * tiles_per_split;
  const int t1 = min(t0 + tiles_per_split, n_tiles_total);
  const int n_tiles = max(t1 - t0, 0);
  const int n_kb = row_words / BW;

  if constexpr (RANGE) {
    if (tid < BQ) {  // (padding rows: -inf selects nothing)
      thr_fast[tid] = q0 + tid < nq ? __float_as_uint(range_threshold<MODE>(radii[q0 + tid], row_words)) : 0xFF800000u;
      rcut[tid] = 0xFFFFFFFFu;
      cnt[tid] = 0;
    }
  } else if (tid < BQ) {
    thr_key[tid] = KEY_MAX;
    cnt[tid] = 0;
    if constexpr (MODE == SCAN_SIFT) thr_fast[tid] = 0x7FFFFFFFu;
    else thr_fast[tid] = 0x7F800000u;  // +inf
  }
  if (tid == 0) qcount = 0;
  __syncthreads();

  // per-thread query-side aux (|q|^2 for cosine, int norm for sift)
  float qaux_f[8];
  int qaux_i[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    qaux_f[i] = 0.f;
    qaux_i[i] = 0;
    int q = q0 + ty + 16 * i;
    if (q < nq) {
      if constexpr (MODE == SCAN_COSINE || MODE == SCAN_ANGULAR) qaux_f[i] = static_cast<const float*>(q_aux_v)[q];
      if constexpr (MODE == SCAN_SIFT) qaux_i[i] = static_cast<const int*>(q_aux_v)[q];
    }
  }

  acc_t acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0;

  const int total_it = n_tiles * n_kb;
  // one pipeline stage = 16 words of 128 query rows + 16 words of 128 point rows
  auto issue = [&](int it) {
    const int tile = t0 + it / n_kb;
    const int kb = it % n_kb;
    uint32_t* dstA = tiles + (it % NSTAGE) * (BQ + BN) * LDW;
    uint32_t* dstB = dstA + BQ * LDW;
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      int c = tid + v * NT;  // 0..511
      int row = c >> 2, col4 = c & 3;
      cp_async16(dstA + row * LDW + col4 * 4, qs + (size_t)(q0 + row) * row_words + kb * BW + col4 * 4);
      cp_async16(dstB + row * LDW + col4 * 4,
                 db + (size_t)(tile * BN + row) * row_words + kb * BW + col4 * 4);
    }
  };

  for (int s = 0; s < NSTAGE - 1; ++s) {
    if (s < total_it) issue(s);
    cp_async_commit();
  }

  for (int it = 0; it < total_it; ++it) {
    cp_async_wait<NSTAGE - 2>();
    __syncthreads();
    if (it + NSTAGE - 1 < total_it) issue(it + NSTAGE - 1);
    cp_async_commit();

    const uint32_t* As = tiles + (it % NSTAGE) * (BQ + BN) * LDW;
    const uint32_t* Bs = As + BQ * LDW;
#pragma unroll
    for (int w = 0; w < BW; w += 4) {
      uint4 b[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = *reinterpret_cast<const uint4*>(Bs + (tx + 16 * j) * LDW + w);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        uint4 a = *reinterpret_cast<const uint4*>(As + (ty + 16 * i) * LDW + w);
#pragma unroll
        for (int j = 0; j < 8; ++j) accum4<MODE>(a, b[j], acc[i][j]);
      }
    }

    if ((it % n_kb) != n_kb - 1) continue;

    // ---------------- tile epilogue: filter against the running k-th best ----------------
    const int tile = t0 + it / n_kb;
    float xaux_f[8];
    int xaux_i[8];
    bool pvalid[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int p = tile * BN + tx + 16 * j;
      pvalid[j] = p < n;
      xaux_f[j] = 0.f;
      xaux_i[j] = 0;
      if (pvalid[j]) {
        if constexpr (MODE == SCAN_COSINE || MODE == SCAN_ANGULAR) xaux_f[j] = static_cast<const float*>(db_aux_v)[p];
        if constexpr (MODE == SCAN_SIFT) xaux_i[j] = static_cast<const int*>(db_aux_v)[p];
      }
    }
    float rq[8], rx[8];
    if constexpr (MODE == SCAN_COSINE || MODE == SCAN_ANGULAR) {
      const float eps = 2.0f * 1.17549435e-38f;
#pragma unroll
      for (int i = 0; i < 8; ++i) rq[i] = qaux_f[i] < eps ? 0.f : rsqrtf(qaux_f[i]);
#pragma unroll
      for (int j = 0; j < 8; ++j) rx[j] = xaux_f[j] < eps ? 0.f : rsqrtf(xaux_f[j]);
    }

    uint64_t pend = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint32_t tbits = thr_fast[ty + 16 * i];
      if constexpr (RANGE)  // a list that dropped a survivor in an earlier tile has stopped selecting
        if (rcut[ty + 16 * i] < pos_base + (uint32_t)(tile * BN)) tbits = 0xFF800000u;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        bool pass;
        if constexpr (MODE == SCAN_SIFT) {
          int r = xaux_i[j] + qaux_i[i] - 2 * acc[i][j];
          pass = r <= (int)tbits;
        } else if constexpr (MODE == SCAN_L2 || MODE == SCAN_L1 || MODE == SCAN_LINF) {
          pass = acc[i][j] <= __uint_as_float(tbits);
        } else if constexpr (MODE == SCAN_NEGDOT) {
          pass = -acc[i][j] <= __uint_as_float(tbits);
        } else {
          float r = 1.f - acc[i][j] * rq[i] * rx[j];
          pass = r <= __uint_as_float(tbits);  // thr_fast carries a slack, see below
        }
        if (pass && pvalid[j]) pend |= 1ull << (i * 8 + j);
      }
    }

    // ---------------- RANGE: survivors straight into the query's list of this split ----------------
    // (arrival order: verification sorts by position.)  The stop test above compares the cut with this tile's first
    // position, so a drop in this tile, whether other threads see it yet or not, never stops this tile's selection:
    // every survivor is either kept or folded into the cut, and the cut is the smallest dropped position.
    if constexpr (RANGE) {
      if (pend) {
        const size_t list0 = ((size_t)(blockIdx.y >> 1) * n_split + split) * (2 * BQ) + (blockIdx.y & 1) * BQ;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (pend & (1ull << (i * 8 + j))) {
              const int row = ty + 16 * i;
              const uint32_t pos = pos_base + (uint32_t)(tile * BN + tx + 16 * j);
              const int e = atomicAdd(&cnt[row], 1);
              if (e < k) cand[(list0 + row) * k + e] = make_key(f32_ordered(acc[i][j]), pos);
              else atomicMin(&rcut[row], pos);
            }
          }
        }
      }
    }

    // ---------------- slow path: queue the survivors, drain into sorted lists ----------------
    while (!RANGE) {
      if (!__syncthreads_or(pend != 0ull)) break;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint64_t bit = 1ull << (i * 8 + j);
          if (pend & bit) {
            uint32_t ord;
            if constexpr (MODE == SCAN_SIFT) ord = i32_ordered(xaux_i[j] + qaux_i[i] - 2 * acc[i][j]);
            else if constexpr (MODE == SCAN_L2 || MODE == SCAN_L1 || MODE == SCAN_LINF) ord = f32_ordered(acc[i][j]);
            else if constexpr (MODE == SCAN_NEGDOT) ord = f32_ordered(-acc[i][j]);
            else if constexpr (MODE == SCAN_ANGULAR) ord = f32_ordered(angular_exact(acc[i][j], xaux_f[j], qaux_f[i]));
            else ord = f32_ordered(cosine_exact(acc[i][j], xaux_f[j], qaux_f[i]));
            const int row = ty + 16 * i;
            const uint64_t key = make_key(ord, pos_base + (uint32_t)(tile * BN + tx + 16 * j));
            if (key < thr_key[row]) {
              int slot = atomicAdd(&qcount, 1);
              if (slot < QCAP) {
                qkey[slot] = key;
                qrow[slot] = (uint16_t)row;
                pend &= ~bit;
              }
            } else {
              pend &= ~bit;
            }
          }
        }
      }
      __syncthreads();
      if (tid < BQ) {
        const int m = min(qcount, QCAP);
        uint64_t* my = lists + (size_t)tid * k;
        int c = cnt[tid];
        bool touched = false;
        for (int e = 0; e < m; ++e) {
          if (qrow[e] != tid) continue;
          const uint64_t key = qkey[e];
          if (c == k && key >= my[k - 1]) continue;
          int p = (c < k) ? c : k - 1;
          while (p > 0 && my[p - 1] > key) {
            my[p] = my[p - 1];
            --p;
          }
          my[p] = key;
          if (c < k) ++c;
          touched = true;
        }
        if (touched) {
          cnt[tid] = c;
          if (c == k) {
            const uint64_t worst = my[k - 1];
            thr_key[tid] = worst;
            const uint32_t hi = (uint32_t)(worst >> 32);
            if constexpr (MODE == SCAN_SIFT) thr_fast[tid] = (uint32_t)i32_from_ordered(hi);
            else if constexpr (MODE == SCAN_COSINE)
              thr_fast[tid] = __float_as_uint(f32_from_ordered(hi) + 4e-6f);  // fast formula slack
            else if constexpr (MODE == SCAN_ANGULAR)  // the fast filter works on 1 - nsp: 1 - cos(angle) + slack
              thr_fast[tid] = __float_as_uint(1.f - cosf(f32_from_ordered(hi)) + 2e-5f);
            else thr_fast[tid] = __float_as_uint(f32_from_ordered(hi));
          }
        }
      }
      __syncthreads();
      if (tid == 0) qcount = 0;
    }

#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0;
  }
  cp_async_wait<0>();
  __syncthreads();

  if constexpr (RANGE) {
    if (tid < BQ) {
      const size_t slot = ((size_t)(blockIdx.y >> 1) * n_split + split) * (2 * BQ) + (blockIdx.y & 1) * BQ + tid;
      cand_cnt[slot] = min(cnt[tid], k);
      cut[slot] = rcut[tid];
    }
    return;
  }

  // ---------------- write this split's sorted partial list ----------------
  if (tid < BQ) {
    const int q = q0 + tid;
    if (q < nq) {
      const uint64_t* my = lists + (size_t)tid * k;
      uint64_t* out = partial + ((size_t)q * n_split + split) * k;
      const int c = cnt[tid];
      for (int e = 0; e < k; ++e) out[e] = e < c ? my[e] : KEY_MAX;
    }
  }
}

constexpr int SMEM_K = 144;  // largest k whose lists fit shared memory
size_t scan_exact_smem(int k) {
  return (size_t)NSTAGE * (BQ + BN) * LDW * 4 + (size_t)BQ * (k <= SMEM_K ? k : 0) * 8 + BQ * 8 + QCAP * 8 + BQ * 4 + BQ * 4 +
         QCAP * 2 + 64;
}

}  // namespace

int scan_exact_max_k() { return 8192; }   // (what the finalising merge sorts in one block)
int scan_exact_smem_k() { return SMEM_K; }
size_t scan_exact_glists_bytes(int nq, int k, int n_split) {
  return k <= SMEM_K ? 0 : (size_t)n_split * ((nq + BQ - 1) / BQ) * BQ * (size_t)k * 8;
}

cudaError_t launch_scan_exact(int mode, const void* db, const void* queries, const void* db_aux,
                              const void* q_aux, int n, int nq, int row_words, int k, uint32_t pos_base,
                              uint64_t* partial, int n_split, int tiles_per_split, cudaStream_t stream,
                              const int* d_nq, uint64_t* glists) {
  if (nq <= 0 || n <= 0) return cudaSuccess;
  if (k > SMEM_K && !glists) return cudaErrorInvalidValue;
  if (k <= SMEM_K) glists = nullptr;
  const size_t smem = scan_exact_smem(k);
  dim3 grid(n_split, (nq + BQ - 1) / BQ);
  const uint32_t* d = static_cast<const uint32_t*>(db);
  const uint32_t* q = static_cast<const uint32_t*>(queries);
  cudaError_t e;
#define NB_LAUNCH(M)                                                                                   \
  e = cudaFuncSetAttribute(scan_exact_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
  if (e != cudaSuccess) return e;                                                                      \
  scan_exact_kernel<M><<<grid, NT, smem, stream>>>(d, q, db_aux, q_aux, n, nq, row_words, k,           \
                                                   tiles_per_split, pos_base, partial, n_split, d_nq, glists, \
                                                   nullptr, nullptr, nullptr, nullptr);
  switch (mode) {
    case SCAN_L2: NB_LAUNCH(SCAN_L2); break;
    case SCAN_NEGDOT: NB_LAUNCH(SCAN_NEGDOT); break;
    case SCAN_COSINE: NB_LAUNCH(SCAN_COSINE); break;
    case SCAN_SIFT: NB_LAUNCH(SCAN_SIFT); break;
    case SCAN_L1: NB_LAUNCH(SCAN_L1); break;
    case SCAN_LINF: NB_LAUNCH(SCAN_LINF); break;
    case SCAN_ANGULAR: NB_LAUNCH(SCAN_ANGULAR); break;
    default: return cudaErrorInvalidValue;
  }
#undef NB_LAUNCH
  return cudaGetLastError();
}

cudaError_t launch_scan_exact_range(int mode, const void* db, const void* queries, int n, int nq, int row_words,
                                    uint32_t pos_base, const float* radii, int list_cap, uint64_t* cand, int* cand_cnt,
                                    uint32_t* cut, int n_split, int tiles_per_split, cudaStream_t stream) {
  if (nq <= 0 || n <= 0) return cudaSuccess;
  const size_t smem = scan_exact_smem(0);
  dim3 grid(n_split, (nq + BQ - 1) / BQ);
  const uint32_t* d = static_cast<const uint32_t*>(db);
  const uint32_t* q = static_cast<const uint32_t*>(queries);
  cudaError_t e;
#define NB_LAUNCH(M)                                                                                                  \
  e = cudaFuncSetAttribute(scan_exact_kernel<M, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);        \
  if (e != cudaSuccess) return e;                                                                                     \
  scan_exact_kernel<M, true><<<grid, NT, smem, stream>>>(d, q, nullptr, nullptr, n, nq, row_words, list_cap,          \
                                                         tiles_per_split, pos_base, nullptr, n_split, nullptr, nullptr, \
                                                         radii, cand, cand_cnt, cut);
  switch (mode) {
    case SCAN_L1: NB_LAUNCH(SCAN_L1); break;
    case SCAN_LINF: NB_LAUNCH(SCAN_LINF); break;
    default: return cudaErrorInvalidValue;
  }
#undef NB_LAUNCH
  return cudaGetLastError();
}

int scan_exact_block_queries() { return BQ; }
int scan_exact_block_points() { return BN; }
int scan_exact_stage_words() { return BW; }

// ---------------------------------------------------------------------------------------
// K0: per-row auxiliaries.  float rows: |x|^2 (cosine); uint8 rows: int32 sum of squares,
// the value the reference stores behind each SIFT payload (space_l2sqr_sift.cc:141-148).
// One warp per row, 128-bit loads.
// ---------------------------------------------------------------------------------------
namespace {
__global__ void row_aux_f32_kernel(const float* __restrict__ rows, int n, int row_words, float* __restrict__ out,
                                   const int* __restrict__ d_n) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (d_n) n = min(n, *d_n);
  if (warp >= n) return;
  const float4* r = reinterpret_cast<const float4*>(rows + (size_t)warp * row_words);
  float s = 0.f;
  for (int c = lane; c < row_words / 4; c += 32) {
    float4 v = r[c];
    s = fmaf(v.x, v.x, s);
    s = fmaf(v.y, v.y, s);
    s = fmaf(v.z, v.z, s);
    s = fmaf(v.w, v.w, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[warp] = s;
}
__global__ void row_aux_u8_kernel(const uint32_t* __restrict__ rows, int n, int row_words, int* __restrict__ out,
                                  const int* __restrict__ d_n) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (d_n) n = min(n, *d_n);
  if (warp >= n) return;
  unsigned s = 0;
  for (int c = lane; c < row_words; c += 32) {
    unsigned v = rows[(size_t)warp * row_words + c];
    s = __dp4a(v, v, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[warp] = (int)s;
}
}  // namespace

cudaError_t launch_row_aux(bool is_u8, const void* rows, int n, int row_words, void* out, cudaStream_t stream,
                           const int* d_n) {
  if (n <= 0) return cudaSuccess;
  const int threads = 256;
  const int blocks = (int)(((size_t)n * 32 + threads - 1) / threads);
  if (is_u8)
    row_aux_u8_kernel<<<blocks, threads, 0, stream>>>(static_cast<const uint32_t*>(rows), n, row_words,
                                                      static_cast<int*>(out), d_n);
  else
    row_aux_f32_kernel<<<blocks, threads, 0, stream>>>(static_cast<const float*>(rows), n, row_words,
                                                       static_cast<float*>(out), d_n);
  return cudaGetLastError();
}

}  // namespace nb200
