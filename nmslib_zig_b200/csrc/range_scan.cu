// range_scan.cu -- range query of ONE query object against the whole shard, for seq_search indexes.
//
// Replaces SeqSearch<dist_t>::Search(RangeQuery*) (src/method/seqsearch.cc:108-141) +
// RangeQuery::CheckAndAddToResult (`distance <= radius`, src/rangequery.cc:58-65) as reached through
// nmslib_range_query_fill (nmslib_c.cpp:1051-1153): every object is visited in position order, the
// ones within the radius are reported in that order, truncated to the caller's capacity.
// One pass over the rows (HBM-bound: N * D * 4 bytes), exact fp32 distances with the reference's own
// formulas (the same code as the re-rank of scan_tc.cu), then an ordered collection by one block.
// Also the last step of the batched range queries (DESIGN.md K5b): range_verify_kernel evaluates the candidates the
// tensor-core scan's range mode left, with the same per-row function (range_row_dist), so both paths agree bit for bit.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace nb200 {
namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// distance(row, query) by one warp, the same bits on every lane; mode SCAN_L2 (sqrt when take_sqrt), SCAN_L1,
// SCAN_LINF, SCAN_COSINE, SCAN_ANGULAR, SCAN_NEGDOT, SCAN_SIFT (byte rows of 128, row_words = 32).  The one definition
// of a range query's distance: the per-query scan and the verification of the batched scan both call it, so their
// answers agree bit for bit.
__device__ __forceinline__ float range_row_dist(const float* __restrict__ xrow, const float* __restrict__ q, int row_words,
                                                int mode, int take_sqrt, int lane) {
  if (mode == SCAN_SIFT) {  // exact int32 sum (x - y)^2, reported as a float
    const uchar4 x = __ldg(reinterpret_cast<const uchar4*>(xrow) + lane);
    const uchar4 y = reinterpret_cast<const uchar4*>(q)[lane];
    const int d0 = (int)x.x - y.x, d1 = (int)x.y - y.y, d2 = (int)x.z - y.z, d3 = (int)x.w - y.w;
    const int di = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
    return (float)__reduce_add_sync(FULL, di);
  }
  const int rw4 = row_words >> 2;
  const float4* q4 = reinterpret_cast<const float4*>(q);
  const float4* x4 = reinterpret_cast<const float4*>(xrow);
  float acc = 0.f, nxs = 0.f, nqs = 0.f;
  for (int e = lane; e < rw4; e += 32) {
    const float4 x = __ldg(x4 + e), y = q4[e];
    if (mode == SCAN_L2) {
      const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z, d3 = x.w - y.w;
      acc = fmaf(d0, d0, acc);
      acc = fmaf(d1, d1, acc);
      acc = fmaf(d2, d2, acc);
      acc = fmaf(d3, d3, acc);
    } else if (mode == SCAN_L1) {
      acc += fabsf(x.x - y.x) + fabsf(x.y - y.y) + fabsf(x.z - y.z) + fabsf(x.w - y.w);
    } else if (mode == SCAN_LINF) {
      acc = fmaxf(acc, fmaxf(fmaxf(fabsf(x.x - y.x), fabsf(x.y - y.y)), fmaxf(fabsf(x.z - y.z), fabsf(x.w - y.w))));
    } else {
      acc = fmaf(x.x, y.x, acc);
      acc = fmaf(x.y, y.y, acc);
      acc = fmaf(x.z, y.z, acc);
      acc = fmaf(x.w, y.w, acc);
      if (mode == SCAN_COSINE || mode == SCAN_ANGULAR) {  // one summation pattern for all three sums (see scan_tc.cu)
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
  // (butterfly reductions: every lane ends with the same sum)
  if (mode == SCAN_LINF) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc = fmaxf(acc, __shfl_xor_sync(FULL, acc, o));
  } else {
    acc = warp_sum(acc);
    if (mode == SCAN_COSINE || mode == SCAN_ANGULAR) {
      nxs = warp_sum(nxs);
      nqs = warp_sum(nqs);
    }
  }
  if (mode == SCAN_L2) return take_sqrt ? sqrtf(acc) : acc;
  if (mode == SCAN_L1 || mode == SCAN_LINF) return acc;
  if (mode == SCAN_NEGDOT) return -acc;
  const float eps = 2.0f * 1.17549435e-38f;
  float nsp = 0.f;
  if (!(nxs < eps || nqs < eps)) nsp = fmaxf(-1.f, fminf(1.f, acc / sqrtf(nxs) / sqrtf(nqs)));
  return mode == SCAN_ANGULAR ? acosf(nsp) : fmaxf(0.f, 1.f - nsp);
}

// dist[i] = distance(row i, query).  (db_norm2 is unused: the cosine family recomputes all three sums per pair.)
__global__ void __launch_bounds__(256) range_dist_kernel(const float* __restrict__ db, const float* __restrict__ q,
                                                         const float* __restrict__ db_norm2, int n, int row_words,
                                                         int mode, int take_sqrt, float* __restrict__ dist) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = blockIdx.x * (blockDim.x >> 5) + warp; row < n; row += warps) {
    const float d = range_row_dist(db + (size_t)row * row_words, q, row_words, mode, take_sqrt, lane);
    if (lane == 0) dist[row] = d;
  }
}

// rows with dist <= radius, in position order, at most `capacity` of them; *out_count = how many were written
__global__ void __launch_bounds__(1024) range_collect_kernel(const float* __restrict__ dist,
                                                             const int32_t* __restrict__ ext_ids, int n, float radius,
                                                             int capacity, int32_t* __restrict__ out_ids,
                                                             float* __restrict__ out_dists, int* __restrict__ out_count) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int i0 = 0; i0 < n; i0 += 1024) {
    const int i = i0 + tid;
    const float d = i < n ? dist[i] : 0.f;
    const bool hit = i < n && d <= radius;
    const unsigned m = __ballot_sync(FULL, hit);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    const int at = off + __popc(m & ((1u << lane) - 1));
    if (hit && at < capacity) {
      out_ids[at] = ext_ids[i];
      out_dists[at] = d;
    }
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int w = 0; w < 32; ++w) tot += s_warp[w];
      s_base += tot;
    }
    __syncthreads();
    if (s_base >= capacity) break;  // (uniform: read after the barrier)
  }
  if (tid == 0) *out_count = min(s_base, capacity);
}

struct RangeVerifyParams {
  const float* db;          // [n_pad][row_words] rows
  const float* queries;     // [q_pad][row_words] staged queries
  const int32_t* ext_ids;
  int row_words, mode, take_sqrt;
  uint32_t pos_base;
  const float* radii;       // [nq]
  const int* caps;          // [nq] min(capacity, n)
  const int64_t* out_off;   // [nq] CSR offsets of the outputs
  const uint64_t* cand;     // [q_blocks][s_max][256][list_cap] (rank << 32 | position), position order per list
  const int* cand_cnt;      // [q_blocks][s_max][256], -1 = list not in use
  const uint32_t* cut;      // [q_blocks][s_max][256] first dropped position, 0xFFFFFFFF = none
  int s_max, list_cap, q0;
  int32_t* out_ids;
  float* out_dists;
  int* out_count;
  int* fb_count;
  int* fb_idx;
};

// Batched range queries, last step: one block per query.  P = the smallest cut of the query's lists; every list is
// complete below its own cut, so the candidates below P are every row below P whose pass-1 rank beat T_q, which
// includes every row below P within the radius (scan_tc.cu: tc_range_threshold_kernel).  They are sorted by position
// and evaluated 256 at a time with range_row_dist; hits (d <= radius) are written in position order until the
// capacity is reached.  The answer is the single-query answer when P = infinity (nothing was dropped) or when at
// least `capacity` hits lie below P; otherwise the query goes to the exact per-query scan.
__global__ void __launch_bounds__(256) range_verify_kernel(const RangeVerifyParams p) {
  extern __shared__ uint32_t spos[];  // candidate positions, then sorted (a power of two >= s_max * list_cap)
  __shared__ float sd[256];
  __shared__ int s_warp[8];
  __shared__ int s_total, s_base;
  __shared__ uint32_t s_cut;
  const int q = p.q0 + blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t slot0 = (size_t)(q / 256) * p.s_max * 256 + (q % 256);  // list s of this query: slot0 + s * 256
  if (tid == 0) {
    s_cut = 0xFFFFFFFFu;
    s_total = 0;
    s_base = 0;
  }
  __syncthreads();
  if (tid < p.s_max) {
    const size_t slot = slot0 + (size_t)tid * 256;
    if (p.cand_cnt[slot] >= 0) atomicMin(&s_cut, p.cut[slot]);
  }
  __syncthreads();
  const uint32_t P = s_cut;
  for (int s = warp; s < p.s_max; s += 8) {  // one warp per list
    const size_t slot = slot0 + (size_t)s * 256;
    const int c = p.cand_cnt[slot];
    const uint64_t* cb = p.cand + slot * (size_t)p.list_cap;
    for (int i = lane; i < c; i += 32) {
      const uint32_t pos = (uint32_t)cb[i];
      if (pos < P) spos[atomicAdd(&s_total, 1)] = pos;
    }
  }
  __syncthreads();
  const int total = s_total;
  int p2 = 1;
  while (p2 < total) p2 <<= 1;
  for (int t = total + tid; t < p2; t += 256) spos[t] = 0xFFFFFFFFu;
  __syncthreads();
  for (int size = 2; size <= p2; size <<= 1) {  // bitonic sort, ascending (positions are distinct)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < p2 / 2; t += 256) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const uint32_t a = spos[lo], b = spos[hi];
        if ((a > b) == ((lo & size) == 0)) {
          spos[lo] = b;
          spos[hi] = a;
        }
      }
      __syncthreads();
    }
  }
  const float radius = p.radii[q];
  const int capacity = p.caps[q];
  const float* qv = p.queries + (size_t)q * p.row_words;
  int32_t* oid = p.out_ids + p.out_off[q];
  float* od = p.out_dists + p.out_off[q];
  for (int c0 = 0; c0 < total; c0 += 256) {
    for (int i = warp; i < 256 && c0 + i < total; i += 8) {
      const size_t local = spos[c0 + i] - p.pos_base;
      const float d = range_row_dist(p.db + local * p.row_words, qv, p.row_words, p.mode, p.take_sqrt, lane);
      if (lane == 0) sd[i] = d;
    }
    __syncthreads();
    const int i = c0 + tid;
    const float d = sd[tid];
    const bool hit = i < total && d <= radius;
    const unsigned m = __ballot_sync(FULL, hit);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int at = s_base + __popc(m & ((1u << lane) - 1));
    for (int w = 0; w < warp; ++w) at += s_warp[w];
    if (hit && at < capacity) {
      oid[at] = p.ext_ids[spos[i] - p.pos_base];
      od[at] = d;
    }
    __syncthreads();
    if (tid == 0)
      for (int w = 0; w < 8; ++w) s_base += s_warp[w];
    __syncthreads();
    if (s_base >= capacity) break;  // (uniform: read after the barrier)
  }
  if (tid == 0) {
    p.out_count[q] = min(s_base, capacity);
    if (P != 0xFFFFFFFFu && s_base < capacity) p.fb_idx[atomicAdd(p.fb_count, 1)] = q;
  }
}

}  // namespace

cudaError_t launch_range_scan(const float* db, const float* query, const float* db_norm2, const int32_t* ext_ids, int n,
                              int row_words, int mode, int take_sqrt, float radius, int capacity, float* dist_tmp,
                              int32_t* out_ids, float* out_dists, int* out_count, cudaStream_t stream) {
  if (n <= 0 || capacity <= 0) return cudaErrorInvalidValue;
  if (row_words % 4) return cudaErrorInvalidValue;
  const int blocks = (int)std::min<long>(((long)n + 7) / 8, 148L * 8);
  range_dist_kernel<<<blocks, 256, 0, stream>>>(db, query, db_norm2, n, row_words, mode, take_sqrt, dist_tmp);
  range_collect_kernel<<<1, 1024, 0, stream>>>(dist_tmp, ext_ids, n, radius, capacity, out_ids, out_dists, out_count);
  return cudaGetLastError();
}

cudaError_t launch_range_verify(const float* db, const float* queries, const int32_t* ext_ids, int row_words, int mode,
                                int take_sqrt, uint32_t pos_base, const float* radii, const int* caps,
                                const int64_t* out_off, const uint64_t* cand, const int* cand_cnt, const uint32_t* cut,
                                int s_max, int list_cap, int q0, int count, int32_t* out_ids, float* out_dists,
                                int* out_count, int* fb_count, int* fb_idx, cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  if (s_max > 256 || row_words % 4) return cudaErrorInvalidValue;
  RangeVerifyParams p{db, queries, ext_ids, row_words, mode, take_sqrt, pos_base, radii, caps, out_off, cand, cand_cnt,
                      cut, s_max, list_cap, q0, out_ids, out_dists, out_count, fb_count, fb_idx};
  size_t items = 1;
  while (items < (size_t)s_max * list_cap) items <<= 1;
  const size_t smem = items * 4;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(range_verify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  range_verify_kernel<<<count, 256, smem, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace nb200
