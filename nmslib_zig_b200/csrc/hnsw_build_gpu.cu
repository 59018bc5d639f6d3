// hnsw_build_gpu.cu -- HNSW graph construction on the device (SURVEY.md 8f, row N3).
//
// The reference inserts points one at a time (Hnsw::add, hnsw.cc:534-609): the candidates of a new point
// come from an efConstruction-wide graph search over the points inserted BEFORE it
// (kSearchElementsWithAttemptsLevel, hnsw.cc:611-708), "heuristic 2" keeps at most M of them
// (getNeighborsByHeuristic2, hnsw.h:129-169), and every kept neighbour gets the back link, its list being
// re-pruned with the same heuristic when it overflows maxM0 / maxM (addFriendlevel, hnsw.h:258-314).
// That is a pointer chase per point; on a B200 the candidate search is better done as what it approximates:
//
//   candidates(i) = the efConstruction nearest points among those inserted before i   (prefix kNN)
//
// and a prefix kNN over a batch of new points is ONE dense contraction on the tensor cores -- the seq_search
// scan of this library (scan_tc.cu), run with the new points as the query batch over the first b rows.
// Points are inserted in position order in batches [a, b) of at most a/8 points (so a point misses at most
// the few neighbours that sit in its own batch BEHIND it: the scan runs over [0, b) and candidates with a
// position >= the point's own are dropped).  Per batch:
//   1. scan      rows [a, b) as queries against rows [0, b), k = efConstruction + slack   (tcgen05 scan)
//   2. select    one warp per new point: prefix filter, heuristic 2 -> at most M forward links
//   3. sort      the back links (neighbour, distance, new point) by neighbour, then distance (cub radix sort)
//   4. link      one warp per touched neighbour: append, or merge + heuristic 2 down to the capacity
// Upper levels are built the same way over the gathered rows of their members.  Levels, entry point,
// parameters and the emitted layout are those of the host builder / the reference (hnsw.cc:417-465), so the
// result is searched by hnsw_search.cu, saved by nmslib_save_index and loadable by the reference.
// The graph is NOT the reference's graph (neither is the reference's own from run to run, SURVEY 0.7): it is
// held to recall parity -- recall@10 at a given efSearch at or above a reference-built graph
// (tests/test_hnsw_gpu.py, tools/hnsw_bench.py --build device).  On rows whose distances are exact fp32 values the
// build is deterministic, and tests/test_hnsw_build_exact_gpu.py holds it to a restatement list for list.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cub/cub.cuh>
#include <chrono>
#include <memory>

#include "engine.h"

namespace nb200 {
namespace {

constexpr unsigned FULLW = 0xffffffffu;
inline double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
constexpr int HB_MAXC = 256;    // candidates per new point (<= the scan's max k)
constexpr int HB_MAXKEEP = 64;  // M, maxM, maxM0 <= 64
constexpr int HB_MAXIN = 32;    // back links taken per neighbour and batch (closest first)
constexpr int HB_WARPS = 4;
static_assert(HB_MAXIN <= 32, "hb_link_kernel reads one incoming link per lane");

// distance of the graph: 0 squared L2, 1 cosine on unit rows, 2 negative dot (hnsw_search.cu uses the same kinds)
template <int KIND>
__device__ __forceinline__ float hb_finish(float acc) {
  if (KIND == 0) return acc;
  if (KIND == 1) return fmaxf(0.f, 1.f - fmaxf(-1.f, fminf(1.f, acc)));
  return -acc;
}

__device__ __forceinline__ float hb_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLW, v, o);
  return v;
}

// distances from row x to four rows at once (one pass over x; every lane ends with all four values)
template <int KIND>
__device__ __forceinline__ void hb_dist4(const float4* __restrict__ x, const float4* __restrict__ r0,
                                         const float4* __restrict__ r1, const float4* __restrict__ r2,
                                         const float4* __restrict__ r3, int n4, int lane, float (&out)[4]) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (int i = lane; i < n4; i += 32) {
    const float4 xv = __ldg(x + i);
    const float4 v0 = __ldg(r0 + i), v1 = __ldg(r1 + i), v2 = __ldg(r2 + i), v3 = __ldg(r3 + i);
    if (KIND == 0) {
      float d;
      d = xv.x - v0.x; a0 = fmaf(d, d, a0); d = xv.y - v0.y; a0 = fmaf(d, d, a0);
      d = xv.z - v0.z; a0 = fmaf(d, d, a0); d = xv.w - v0.w; a0 = fmaf(d, d, a0);
      d = xv.x - v1.x; a1 = fmaf(d, d, a1); d = xv.y - v1.y; a1 = fmaf(d, d, a1);
      d = xv.z - v1.z; a1 = fmaf(d, d, a1); d = xv.w - v1.w; a1 = fmaf(d, d, a1);
      d = xv.x - v2.x; a2 = fmaf(d, d, a2); d = xv.y - v2.y; a2 = fmaf(d, d, a2);
      d = xv.z - v2.z; a2 = fmaf(d, d, a2); d = xv.w - v2.w; a2 = fmaf(d, d, a2);
      d = xv.x - v3.x; a3 = fmaf(d, d, a3); d = xv.y - v3.y; a3 = fmaf(d, d, a3);
      d = xv.z - v3.z; a3 = fmaf(d, d, a3); d = xv.w - v3.w; a3 = fmaf(d, d, a3);
    } else {
      a0 = fmaf(xv.x, v0.x, a0); a0 = fmaf(xv.y, v0.y, a0); a0 = fmaf(xv.z, v0.z, a0); a0 = fmaf(xv.w, v0.w, a0);
      a1 = fmaf(xv.x, v1.x, a1); a1 = fmaf(xv.y, v1.y, a1); a1 = fmaf(xv.z, v1.z, a1); a1 = fmaf(xv.w, v1.w, a1);
      a2 = fmaf(xv.x, v2.x, a2); a2 = fmaf(xv.y, v2.y, a2); a2 = fmaf(xv.z, v2.z, a2); a2 = fmaf(xv.w, v2.w, a2);
      a3 = fmaf(xv.x, v3.x, a3); a3 = fmaf(xv.y, v3.y, a3); a3 = fmaf(xv.z, v3.z, a3); a3 = fmaf(xv.w, v3.w, a3);
    }
  }
  out[0] = hb_finish<KIND>(hb_warp_sum(a0));
  out[1] = hb_finish<KIND>(hb_warp_sum(a1));
  out[2] = hb_finish<KIND>(hb_warp_sum(a2));
  out[3] = hb_finish<KIND>(hb_warp_sum(a3));
}

// getNeighborsByHeuristic2 (hnsw.h:129-169): candidates by increasing distance to the base point; one is kept
// unless some already kept neighbour is closer to it than the base point is.  Fewer than NN candidates are all
// kept (the reference returns early, hnsw.h:133-135).  ids / ds / keep_* live in this warp's shared memory.
template <int KIND>
__device__ int hb_heuristic2(const float* __restrict__ rows, int row_words, const int* ids, const float* ds, int m,
                             int NN, int* keep_ids, float* keep_ds, int lane) {
  if (m < NN) {
    for (int j = lane; j < m; j += 32) {
      keep_ids[j] = ids[j];
      keep_ds[j] = ds[j];
    }
    __syncwarp();
    return m;
  }
  const int n4 = row_words >> 2;
  int nk = 0;
  for (int j = 0; j < m && nk < NN; ++j) {
    const int c = ids[j];
    const float dc = ds[j];
    const float4* x = reinterpret_cast<const float4*>(rows + (size_t)c * row_words);
    bool good = true;
    for (int r = 0; r < nk && good; r += 4) {
      const int last = nk - 1;
      const float4* p0 = reinterpret_cast<const float4*>(rows + (size_t)keep_ids[min(r, last)] * row_words);
      const float4* p1 = reinterpret_cast<const float4*>(rows + (size_t)keep_ids[min(r + 1, last)] * row_words);
      const float4* p2 = reinterpret_cast<const float4*>(rows + (size_t)keep_ids[min(r + 2, last)] * row_words);
      const float4* p3 = reinterpret_cast<const float4*>(rows + (size_t)keep_ids[min(r + 3, last)] * row_words);
      float o[4];
      hb_dist4<KIND>(x, p0, p1, p2, p3, n4, lane, o);
      if (o[0] < dc || o[1] < dc || o[2] < dc || o[3] < dc) good = false;  // (clamped duplicates repeat a real test)
    }
    if (good) {
      if (lane == 0) {
        keep_ids[nk] = c;
        keep_ds[nk] = dc;
      }
      ++nk;
      __syncwarp();
    }
  }
  return nk;
}

// ---- step 2: forward links of the new points [a, a + nq) --------------------------------------------------
// keys / dists: [nq][K] scan output of the batch (ascending; low key word = position, KEY_MAX padded).
// rev_key[w * M + j] = neighbour << 32 | ordered(distance) (KEY_MAX when unused), rev_src = the new point.
template <int KIND>
__global__ void __launch_bounds__(HB_WARPS * 32)
hb_select_kernel(const float* __restrict__ rows, int row_words, const uint64_t* __restrict__ keys,
                 const float* __restrict__ dists, int K, int a, int nq, int efc, int M, int cap, int* links,
                 float* ldist, int* cnt, uint64_t* rev_key, int* rev_src) {
  __shared__ int s_ids[HB_WARPS][HB_MAXC];
  __shared__ float s_ds[HB_WARPS][HB_MAXC];
  __shared__ int s_kid[HB_WARPS][HB_MAXKEEP];
  __shared__ float s_kd[HB_WARPS][HB_MAXKEEP];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * HB_WARPS + wib;
  if (w >= nq) return;
  const int i = a + w;
  int* ids = s_ids[wib];
  float* ds = s_ds[wib];
  // prefix filter: only points inserted before i are candidates (this also drops i itself)
  int m = 0;
  for (int base = 0; base < K && m < efc; base += 32) {
    const int e = base + lane;
    uint64_t key = KEY_MAX;
    float v = 0.f;
    if (e < K) {
      key = keys[(size_t)w * K + e];
      v = dists[(size_t)w * K + e];
    }
    const uint32_t pos = (uint32_t)key;
    const bool ok = key != KEY_MAX && pos < (uint32_t)i;
    const unsigned bal = __ballot_sync(FULLW, ok);
    const int at = m + __popc(bal & ((1u << lane) - 1));
    if (ok && at < efc) {
      ids[at] = (int)pos;
      // the scan reports squared L2 / minus the dot product; the graph's cosine is 1 - dot on unit rows
      ds[at] = KIND == 1 ? fmaxf(0.f, 1.f - fmaxf(-1.f, fminf(1.f, -v))) : v;
    }
    m = min(efc, m + __popc(bal));
  }
  __syncwarp();
  const int nk = hb_heuristic2<KIND>(rows, row_words, ids, ds, m, M, s_kid[wib], s_kd[wib], lane);
  __syncwarp();
  for (int j = lane; j < M; j += 32) {
    const bool on = j < nk;
    if (on) {
      links[(size_t)i * cap + j] = s_kid[wib][j];
      ldist[(size_t)i * cap + j] = s_kd[wib][j];
    }
    rev_key[(size_t)w * M + j] = on ? ((uint64_t)(uint32_t)s_kid[wib][j] << 32) | f32_ordered(s_kd[wib][j]) : KEY_MAX;
    rev_src[(size_t)w * M + j] = i;
  }
  if (lane == 0) cnt[i] = nk;
}

// ---- step 3b: first entry of every neighbour's run in the sorted back-link list ------------------------------
__global__ void hb_segments_kernel(const uint64_t* __restrict__ rkey, int total, int* seg_start, int* seg_count) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const uint64_t key = rkey[idx];
  if (key == KEY_MAX) return;
  if (idx == 0 || (uint32_t)(rkey[idx - 1] >> 32) != (uint32_t)(key >> 32)) seg_start[atomicAdd(seg_count, 1)] = idx;
}

// ---- step 4: back links (addFriendlevel, hnsw.h:258-314) --------------------------------------------------------
// One warp per touched neighbour c: its incoming links of this batch (closest HB_MAXIN) are appended while the
// list has room; otherwise old and new links are merged by distance and heuristic 2 keeps at most `cap`
// (the reference shrinks after every single insertion with NN = size - 1 = cap; one shrink per batch is the same
// rule applied to the merged list).  A new point cannot already be in c's list (links only point backwards when
// they are made), and no two warps touch the same list.
template <int KIND>
__global__ void __launch_bounds__(HB_WARPS * 32)
hb_link_kernel(const float* __restrict__ rows, int row_words, const uint64_t* __restrict__ rkey,
               const int* __restrict__ rsrc, int total, const int* __restrict__ seg_start,
               const int* __restrict__ seg_count, int cap, int* links, float* ldist, int* cnt,
               unsigned long long* prunes) {
  constexpr int MAXI = HB_MAXKEEP + HB_MAXIN;
  __shared__ int s_ids[HB_WARPS][MAXI];
  __shared__ float s_ds[HB_WARPS][MAXI];
  __shared__ int s_sid[HB_WARPS][MAXI];
  __shared__ float s_sd[HB_WARPS][MAXI];
  __shared__ int s_kid[HB_WARPS][HB_MAXKEEP];
  __shared__ float s_kd[HB_WARPS][HB_MAXKEEP];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * HB_WARPS + wib;
  if (w >= *seg_count) return;
  const int s0 = seg_start[w];
  const uint32_t c = (uint32_t)(rkey[s0] >> 32);
  // incoming links: the run is sorted by distance, the first HB_MAXIN are the closest (the shared lists above hold
  // no more, whatever the warp width)
  uint64_t key = KEY_MAX;
  if (s0 + lane < total) key = rkey[s0 + lane];
  const bool in_ok = lane < HB_MAXIN && key != KEY_MAX && (uint32_t)(key >> 32) == c;
  const unsigned bal = __ballot_sync(FULLW, in_ok);  // a prefix of the lanes (the run is contiguous)
  const int inc = __popc(bal);
  const int have = cnt[c];
  int* L = links + (size_t)c * cap;
  float* LD = ldist + (size_t)c * cap;
  if (have + inc <= cap) {
    if (in_ok) {
      L[have + lane] = rsrc[s0 + lane];
      LD[have + lane] = f32_from_ordered((uint32_t)key);
    }
    if (lane == 0) cnt[c] = have + inc;
    return;
  }
  // merge: old links + incoming, sorted by (distance, id) through rank counting
  int* ids = s_ids[wib];
  float* ds = s_ds[wib];
  for (int j = lane; j < have; j += 32) {
    ids[j] = L[j];
    ds[j] = LD[j];
  }
  if (in_ok) {
    ids[have + lane] = rsrc[s0 + lane];
    ds[have + lane] = f32_from_ordered((uint32_t)key);
  }
  const int m = have + inc;
  __syncwarp();
  for (int j = lane; j < m; j += 32) {
    const float d = ds[j];
    const int id = ids[j];
    int rank = 0;
    for (int t = 0; t < m; ++t) {
      const float dt = ds[t];
      rank += (dt < d || (dt == d && ids[t] < id)) ? 1 : 0;
    }
    s_sid[wib][rank] = id;
    s_sd[wib][rank] = d;
  }
  __syncwarp();
  const int nk = hb_heuristic2<KIND>(rows, row_words, s_sid[wib], s_sd[wib], m, cap, s_kid[wib], s_kd[wib], lane);
  __syncwarp();
  for (int j = lane; j < nk; j += 32) {
    L[j] = s_kid[wib][j];
    LD[j] = s_kd[wib][j];
  }
  if (lane == 0) {
    cnt[c] = nk;
    atomicAdd(prunes, 1ull);
  }
}

#define HB_CUDA(call, what)                                                                             \
  do {                                                                                                  \
    cudaError_t e__ = (call);                                                                           \
    if (e__ != cudaSuccess) {                                                                           \
      cudaGetLastError();                                                                               \
      return Status::Err(e__ == cudaErrorMemoryAllocation ? 3 : 8,                                      \
                         std::string("hnsw device build: ") + what + ": " + cudaGetErrorString(e__));   \
    }                                                                                                   \
  } while (0)

struct LevelGraph {
  std::vector<int32_t> links;  // [m][cap] local indices
  std::vector<int32_t> cnt;    // [m]
};

// one level: members' rows d_rows_l [m_pad][row_words] (local index = insertion order)
Status build_level(const float* d_rows_l, size_t m, int dim, int row_words, int kind, const HnswBuildParams& bp,
                   int cap, int device, cudaStream_t stream, LevelGraph* out, HnswBuildInfo* info) {
  out->links.assign(m * (size_t)cap, -1);
  out->cnt.assign(m, 0);
  if (m < 2) return Status::OK();
  const int M = std::min(bp.M, cap);  // (a level whose capacity is below M keeps at most its capacity)
  const int efc = std::min(bp.efConstruction, HB_MAXC - 24);  // room for the slack below inside the scan's max k
  int K = std::min(HB_MAXC, efc + efc / 8 + 8);
  if (const char* e = nb200_env("NB200_HNSW_BUILD_K")) K = std::max(M + 1, std::min(HB_MAXC, atoi(e)));  // (experiments)
  // scan engine over the members' rows, in place.  cosine rows are unit vectors: 1 - dot ranks like -dot.
  const double t_setup = now_ms();
  Engine scan(kind == 0 ? SPACE_L2SQR : SPACE_NEGDOT, METHOD_SEQ, false, device);
  Status s = scan.adopt_device_rows(d_rows_l, m, dim, row_words);
  if (!s.ok()) return s;
  scan.set_approx_ok(true);
  if (!(s = scan.prepare()).ok()) return s;

  const size_t max_batch = 32768;
  DevBuf d_links, d_ldist, d_cnt, d_keys, d_dists, d_ids, d_rkey, d_rkey2, d_rsrc, d_rsrc2, d_seg, d_segcnt, d_tmp,
      d_prunes;
  struct Free {
    std::vector<DevBuf*> b;
    ~Free() {
      for (DevBuf* x : b) x->release();
    }
  } guard{{&d_links, &d_ldist, &d_cnt, &d_keys, &d_dists, &d_ids, &d_rkey, &d_rkey2, &d_rsrc, &d_rsrc2, &d_seg, &d_segcnt,
           &d_tmp, &d_prunes}};
  HB_CUDA(d_links.ensure(m * (size_t)cap * 4), "links");
  HB_CUDA(d_ldist.ensure(m * (size_t)cap * 4), "link distances");
  HB_CUDA(d_cnt.ensure(m * 4), "link counts");
  HB_CUDA(cudaMemsetAsync(d_cnt.p, 0, m * 4, stream), "memset");
  HB_CUDA(cudaMemsetAsync(d_links.p, 0xFF, m * (size_t)cap * 4, stream), "memset");
  const size_t bq = std::min(max_batch, m);
  HB_CUDA(d_keys.ensure(bq * K * 8), "scan keys");
  HB_CUDA(d_dists.ensure(bq * K * 4), "scan distances");
  HB_CUDA(d_ids.ensure(bq * K * 4), "scan ids");
  HB_CUDA(d_rkey.ensure(bq * M * 8), "back links");
  HB_CUDA(d_rkey2.ensure(bq * M * 8), "back links");
  HB_CUDA(d_rsrc.ensure(bq * M * 4), "back links");
  HB_CUDA(d_rsrc2.ensure(bq * M * 4), "back links");
  HB_CUDA(d_seg.ensure(bq * M * 4), "segments");
  HB_CUDA(d_segcnt.ensure(4), "segments");
  HB_CUDA(d_prunes.ensure(8), "counters");
  HB_CUDA(cudaMemsetAsync(d_prunes.p, 0, 8, stream), "memset");
  size_t tmp_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_rkey.as<uint64_t>(), d_rkey2.as<uint64_t>(), d_rsrc.as<int>(),
                                  d_rsrc2.as<int>(), (int)(bq * M), 0, 64, stream);
  HB_CUDA(d_tmp.ensure(tmp_bytes), "sort scratch");

  cudaEvent_t ev[4];
  for (auto& e : ev) cudaEventCreate(&e);
  struct EvFree {
    cudaEvent_t* e;
    ~EvFree() {
      for (int i = 0; i < 4; ++i) cudaEventDestroy(e[i]);
    }
  } evguard{ev};

  info->setup_ms += now_ms() - t_setup;
  const double t_reserve = now_ms();
  // The batches grow up to max_batch points against up to m rows: size the scan's scratch once for every batch
  // shape of the schedule (a dry run allocates, launches nothing) instead of regrowing it every few batches.
  {
    scan.set_dry_run(true);
    size_t a2 = 0;
    while (a2 < m) {
      size_t step = std::min(std::max<size_t>(256, (a2 / 8) / 256 * 256), max_batch);
      const size_t b2 = std::min(m, a2 + step);
      if (b2 >= 2) {
        scan.set_scan_rows(b2);
        s = scan.knn_device(d_rows_l + a2 * (size_t)row_words, b2 - a2, dim, K, d_ids.as<int32_t>(), d_dists.as<float>(),
                            d_keys.as<uint64_t>(), nullptr, stream, (size_t)row_words * 4);
        if (!s.ok()) return s;
      }
      a2 = b2;
    }
    scan.set_dry_run(false);
    HB_CUDA(cudaStreamSynchronize(stream), "reserve");
  }
  info->reserve_ms += now_ms() - t_reserve;
  size_t a = 0;
  while (a < m) {
    // batch [a, b): at most a/8 new points (whole 256-query blocks), the first one takes 256
    size_t step = std::max<size_t>(256, (a / 8) / 256 * 256);
    step = std::min(step, max_batch);
    const size_t b = std::min(m, a + step);
    const int nq = (int)(b - a);
    if (b >= 2) {
      scan.set_scan_rows(b);
      cudaEventRecord(ev[0], stream);
      s = scan.knn_device(d_rows_l + a * (size_t)row_words, nq, dim, K, d_ids.as<int32_t>(), d_dists.as<float>(),
                          d_keys.as<uint64_t>(), nullptr, stream, (size_t)row_words * 4);
      if (!s.ok()) return s;
      cudaEventRecord(ev[1], stream);
      const int blocks = (nq + HB_WARPS - 1) / HB_WARPS;
#define HB_SELECT(KD)                                                                                              \
  hb_select_kernel<KD><<<blocks, HB_WARPS * 32, 0, stream>>>(d_rows_l, row_words, d_keys.as<uint64_t>(),           \
                                                             d_dists.as<float>(), K, (int)a, nq, efc, M, cap,      \
                                                             d_links.as<int>(), d_ldist.as<float>(), d_cnt.as<int>(), \
                                                             d_rkey.as<uint64_t>(), d_rsrc.as<int>())
      if (kind == 0) HB_SELECT(0);
      else if (kind == 1) HB_SELECT(1);
      else HB_SELECT(2);
#undef HB_SELECT
      HB_CUDA(cudaGetLastError(), "select");
      cudaEventRecord(ev[2], stream);
      const int total = nq * M;
      size_t tb = tmp_bytes;
      HB_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp.p, tb, d_rkey.as<uint64_t>(), d_rkey2.as<uint64_t>(),
                                              d_rsrc.as<int>(), d_rsrc2.as<int>(), total, 0, 64, stream),
              "sort");
      HB_CUDA(cudaMemsetAsync(d_segcnt.p, 0, 4, stream), "memset");
      hb_segments_kernel<<<(total + 255) / 256, 256, 0, stream>>>(d_rkey2.as<uint64_t>(), total, d_seg.as<int>(),
                                                                  d_segcnt.as<int>());
      HB_CUDA(cudaGetLastError(), "segments");
      // (the grid covers the worst case of one neighbour per back link; warps beyond seg_count exit at once)
      const int lblocks = (total + HB_WARPS - 1) / HB_WARPS;
#define HB_LINK(KD)                                                                                                 \
  hb_link_kernel<KD><<<lblocks, HB_WARPS * 32, 0, stream>>>(d_rows_l, row_words, d_rkey2.as<uint64_t>(),            \
                                                            d_rsrc2.as<int>(), total, d_seg.as<int>(),              \
                                                            d_segcnt.as<int>(), cap, d_links.as<int>(),             \
                                                            d_ldist.as<float>(), d_cnt.as<int>(),                   \
                                                            d_prunes.as<unsigned long long>())
      if (kind == 0) HB_LINK(0);
      else if (kind == 1) HB_LINK(1);
      else HB_LINK(2);
#undef HB_LINK
      HB_CUDA(cudaGetLastError(), "link");
      cudaEventRecord(ev[3], stream);
      HB_CUDA(cudaStreamSynchronize(stream), "batch");
      float t01 = 0, t12 = 0, t23 = 0;
      cudaEventElapsedTime(&t01, ev[0], ev[1]);
      cudaEventElapsedTime(&t12, ev[1], ev[2]);
      cudaEventElapsedTime(&t23, ev[2], ev[3]);
      info->scan_ms += t01;
      info->select_ms += t12;
      info->link_ms += t23;
      info->reverse_edges += (uint64_t)total;
      ++info->batches;
    }
    a = b;
  }
  unsigned long long prunes = 0;
  const double t_down = now_ms();
  HB_CUDA(cudaMemcpyAsync(out->links.data(), d_links.p, m * (size_t)cap * 4, cudaMemcpyDeviceToHost, stream), "D2H");
  HB_CUDA(cudaMemcpyAsync(out->cnt.data(), d_cnt.p, m * 4, cudaMemcpyDeviceToHost, stream), "D2H");
  HB_CUDA(cudaMemcpyAsync(&prunes, d_prunes.p, 8, cudaMemcpyDeviceToHost, stream), "D2H");
  HB_CUDA(cudaStreamSynchronize(stream), "level");
  info->prunes += prunes;
  info->download_ms += now_ms() - t_down;
  return Status::OK();
}

}  // namespace

Status build_hnsw_device(const float* d_rows, size_t n, int dim, int row_words, int dist_func, const int32_t* ext_ids,
                         const HnswBuildParams& bp, int device, HnswGraph* out, HnswBuildInfo* info) {
  if (n == 0) return Status::Err(8, "cannot build an HNSW graph over an empty data set");
  if (n > 0x7FFFFFF0ull) return Status::Err(6, "too many points for an HNSW graph");
  if (bp.M > HB_MAXKEEP || bp.maxM > HB_MAXKEEP || bp.maxM0 > HB_MAXKEEP)
    return Status::Err(8, "device HNSW build supports M, maxM, maxM0 <= 64 (use b200_build=host)");
  if (row_words % 4) return Status::Err(8, "device HNSW build needs rows padded to 16 bytes");
  HnswBuildInfo local;
  if (!info) info = &local;
  *info = HnswBuildInfo();
  HB_CUDA(cudaSetDevice(device), "cudaSetDevice");
  cudaStream_t stream = nullptr;
  HB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "stream");
  struct StreamFree {
    cudaStream_t s;
    ~StreamFree() { cudaStreamDestroy(s); }
  } sguard{stream};
  cudaEvent_t t0, t1;
  cudaEventCreate(&t0);
  cudaEventCreate(&t1);
  cudaEventRecord(t0, stream);

  const int kind = dist_func == 3 ? 1 : dist_func == 4 ? 2 : 0;
  const std::vector<int> level = hnsw_assign_levels(n, bp.mult);
  int maxlevel = 0;
  size_t enterpoint = 0;
  for (size_t i = 0; i < n; ++i)
    if (level[i] > maxlevel) {  // the first point that reaches a new top level becomes the entry point (hnsw.cc:601-604)
      maxlevel = level[i];
      enterpoint = i;
    }

  HnswGraph g;
  g.total = (uint32_t)n;
  g.dim = dim;
  g.maxM = bp.maxM;
  g.M = bp.M;
  g.maxM0 = bp.maxM0;
  g.maxlevel = maxlevel;
  g.levels.assign(level.begin(), level.end());
  g.enterpoint = (uint32_t)enterpoint;
  g.dist_func = dist_func;
  g.ext_ids.assign(ext_ids, ext_ids + n);

  // level 0 over the index rows in place
  LevelGraph l0;
  Status s = build_level(d_rows, n, dim, row_words, kind, bp, bp.maxM0, device, stream, &l0, info);
  if (!s.ok()) return s;
  g.links0.swap(l0.links);
  g.links0_cnt.swap(l0.cnt);
  for (size_t i = 0; i < n; ++i)  // unused slots as the host builder leaves them
    for (int j = g.links0_cnt[i]; j < bp.maxM0; ++j) g.links0[i * (size_t)bp.maxM0 + j] = -1;

  // upper levels over the gathered rows of their members (positions ascending = insertion order)
  std::vector<std::vector<int>> members(maxlevel + 1);
  std::vector<LevelGraph> upper(maxlevel + 1);
  DevBuf d_sub, d_idx;
  struct SubFree {
    DevBuf *a, *b;
    ~SubFree() {
      a->release();
      b->release();
    }
  } subguard{&d_sub, &d_idx};
  for (int l = 1; l <= maxlevel; ++l) {
    std::vector<int>& mem = members[l];
    for (size_t i = 0; i < n; ++i)
      if (level[i] >= l) mem.push_back((int)i);
    const size_t m = mem.size();
    const size_t m_pad = round_up(m, 128);
    HB_CUDA(d_sub.ensure(m_pad * (size_t)row_words * 4), "level rows");
    HB_CUDA(d_idx.ensure(m * 4), "level members");
    HB_CUDA(cudaMemsetAsync(d_sub.p, 0, m_pad * (size_t)row_words * 4, stream), "memset");
    HB_CUDA(cudaMemcpyAsync(d_idx.p, mem.data(), m * 4, cudaMemcpyHostToDevice, stream), "H2D");
    HB_CUDA(launch_gather_rows(reinterpret_cast<const uint32_t*>(d_rows), d_idx.as<int>(), (int)m, row_words,
                               d_sub.as<uint32_t>(), stream),
            "gather");
    HB_CUDA(cudaStreamSynchronize(stream), "gather");
    s = build_level(d_sub.as<float>(), m, dim, row_words, kind, bp, bp.maxM, device, stream, &upper[l], info);
    if (!s.ok()) return s;
  }
  info->levels = maxlevel + 1;

  // flatten the upper levels into the optimized-index layout (hnsw.cc:417-465): per node and level maxM + 1 ints
  g.upper_off.assign(n, -1);
  std::vector<int> local_idx(maxlevel + 1, 0);  // running local index of node i inside level l (members ascend)
  for (size_t i = 0; i < n; ++i) {
    if (level[i] < 1) continue;
    g.upper_off[i] = (int64_t)g.upper.size();
    for (int l = 1; l <= level[i]; ++l) {
      const int li = local_idx[l]++;
      const LevelGraph& lg = upper[l];
      const int cc = lg.cnt[li];
      g.upper.push_back(cc);
      for (int j = 0; j < bp.maxM; ++j)
        g.upper.push_back(j < cc ? members[l][lg.links[(size_t)li * bp.maxM + j]] : 0x01010101);
    }
  }
  cudaEventRecord(t1, stream);
  cudaEventSynchronize(t1);
  float ms = 0;
  cudaEventElapsedTime(&ms, t0, t1);
  info->total_ms = ms;
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  if (nb200_env("NB200_HNSW_BUILD_VERBOSE"))
    fprintf(stderr,
            "[nb200] hnsw device build: n=%zu dim=%d levels=%d batches=%d total %.1f ms (scan %.1f, select %.1f, link %.1f; "
            "host: set-up %.1f, scratch sizing %.1f, download %.1f), %llu back links, %llu prunes\n",
            n, dim, info->levels, info->batches, info->total_ms, info->scan_ms, info->select_ms, info->link_ms,
            info->setup_ms, info->reserve_ms, info->download_ms,
            (unsigned long long)info->reverse_edges, (unsigned long long)info->prunes);
  *out = std::move(g);
  return Status::OK();
}

}  // namespace nb200
