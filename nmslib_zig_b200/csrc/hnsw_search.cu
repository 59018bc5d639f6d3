// hnsw_search.cu -- K3: batched HNSW beam search, one warp per query.
//
// Replaces Hnsw<float>::Search(KNNQuery*) on the optimized flat index: the greedy
// descent through the upper layers and the level-0 best-first beam of
// Hnsw::SearchV1Merge (src/method/hnsw_distfunc_opt.cc:152-283), its SortArrBI beam
// (include/sort_arr_bi.h:30-216), the VisitedList epoch array (include/method/hnsw.h:568-591)
// and the inline distance kernels (hnsw_distfunc_opt_impl_inline.h:42-173, hnsw.cc:70-81).
//
// Beam rule kept from V1Merge: W is an ascending array of capacity max(ef, k) with a
// "used" flag per item; while cur < min(|W|, ef): expand the first unused item; every
// unvisited neighbour is evaluated; it is accepted iff d < worst(W) (frozen at the start
// of the expansion) or |W| < ef; accepted items are merged into W (truncating at the
// capacity); cur rewinds to the smallest insertion index; the answer is W[0..k).
// For ef >= 1000 the reference switches to SearchOld (hnsw.cc:724); for k <= ef that
// algorithm keeps the same ef-closest set and stops at the same point, so this kernel
// serves both (tests/test_hnsw_gpu.py checks ef = 1000 against the live reference).
//
// Memory behaviour: per evaluated neighbour the warp gathers one vector with 128-bit
// loads (lane c reads float4 c, c+32, ...), four neighbours in flight per warp; the
// level-0 adjacency row (maxM0 ints) is one coalesced 128-byte read.  The kernel is
// bound by HBM random-gather bandwidth, not FLOPs.
// uint8 rows (l2sqr_sift, dist_kind 3) stay bytes: a 128-byte row is one word per lane, one coalesced
// load per neighbour, and the distance is an exact integer (dp4a of byte differences, integer warp sum)
// converted to float -- the value the widened fp32 sum gives, bit for bit, since every partial sum there
// is an integer below 2^24.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace nb200 {
namespace {

constexpr int WARPS = 4;          // warps (queries in flight) per block
constexpr int MAX_EF = 6144;      // beam capacity limit: 4 warps x (row + 8 B per beam entry) must fit 227 KB of shared memory
constexpr unsigned FULL = 0xffffffffu;
constexpr int USED_BIT = 0x80000000;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

template <int KIND>
__device__ __forceinline__ void acc4(const float4& x, const float4& q, float& s) {
  if constexpr (KIND == 0) {
    float d0 = x.x - q.x, d1 = x.y - q.y, d2 = x.z - q.z, d3 = x.w - q.w;
    s = fmaf(d0, d0, s);
    s = fmaf(d1, d1, s);
    s = fmaf(d2, d2, s);
    s = fmaf(d3, d3, s);
  } else {
    s = fmaf(x.x, q.x, s);
    s = fmaf(x.y, q.y, s);
    s = fmaf(x.z, q.z, s);
    s = fmaf(x.w, q.w, s);
  }
}
template <int KIND>
__device__ __forceinline__ float fin_dist(float s) {  // (KIND 3 never gets here: evalG returns its integer sum)
  if constexpr (KIND == 0) return s;                                            // L2Sqr(16)Ext
  else if constexpr (KIND == 1) return fmaxf(0.f, 1.f - fmaxf(-1.f, fminf(1.f, s)));  // NormCosine hnsw.cc:78-81
  else return -s;                                                               // NegativeDotProduct :70-73
}

// distances of up to G nodes (t[g] valid for g < cnt) to the query in shared memory: G independent row
// gathers in flight per lane and loop iteration (the kernel waits on these loads ~80 % of the time, ncu)
template <int KIND, int G>
__device__ __forceinline__ void evalG(const void* __restrict__ vectors, int row_words,
                                      const float4* __restrict__ q4, const int (&t)[G], int cnt, int lane,
                                      float (&out)[G]) {
  if constexpr (KIND == 3) {
    // byte rows: word c of a row holds elements 4c..4c+3; |x - q|^2 of one word is dp4a(|x - q|, |x - q|) per byte
    // (at most 4 * 255^2), the row's sum at most 128 * 255^2 < 2^24, so the float conversion is exact
    const uint32_t* xw[G];
    uint32_t s[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      xw[g] = static_cast<const uint32_t*>(vectors) + (size_t)t[g < cnt ? g : 0] * row_words;
      s[g] = 0u;
    }
    const uint32_t* qw = reinterpret_cast<const uint32_t*>(q4);
    for (int c = lane; c < row_words; c += 32) {
      uint32_t a[G];
#pragma unroll
      for (int g = 0; g < G; ++g) a[g] = g < cnt ? __ldg(xw[g] + c) : 0u;
      const uint32_t q = qw[c];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const uint32_t d = __vabsdiffu4(a[g], q);
        s[g] = __dp4a(d, d, s[g]);
      }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) out[g] = (float)__reduce_add_sync(FULL, s[g]);
    return;
  }
  const int rw4 = row_words >> 2;
  const float4* x[G];
  float s[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    x[g] = reinterpret_cast<const float4*>(static_cast<const float*>(vectors) + (size_t)t[g < cnt ? g : 0] * row_words);
    s[g] = 0.f;
  }
  if (cnt == G) {
#pragma unroll 2
    for (int c = lane; c < rw4; c += 32) {
      float4 a[G];
#pragma unroll
      for (int g = 0; g < G; ++g) a[g] = __ldg(x[g] + c);
      const float4 q = q4[c];
#pragma unroll
      for (int g = 0; g < G; ++g) acc4<KIND>(a[g], q, s[g]);
    }
  } else {
#pragma unroll 2
    for (int c = lane; c < rw4; c += 32) {
      const float4 q = q4[c];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (g < cnt) {
          const float4 a = __ldg(x[g] + c);
          acc4<KIND>(a, q, s[g]);
        }
      }
    }
  }
#pragma unroll
  for (int g = 0; g < G; ++g) out[g] = fin_dist<KIND>(warp_sum(s[g]));
}

// ascending bitonic sort of one 64-bit key per lane
__device__ __forceinline__ uint64_t warp_sort64(uint64_t v, int lane) {
#pragma unroll
  for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const uint64_t o = __shfl_xor_sync(FULL, v, stride);
      const bool up = (lane & size) == 0;
      const bool lower = (lane & stride) == 0;
      const bool take_min = (lower == up);
      v = take_min ? (v < o ? v : o) : (v < o ? o : v);
    }
  }
  return v;
}

// ---- pieces shared by the one-warp kernel and the team kernel (one warp executes each of them) ----------------

// stage the query in shared memory (cosine: NormalizeVect, hnsw.h:486-497; byte rows: the words are copied as they are)
template <int KIND>
__device__ __forceinline__ void stage_query(const float* __restrict__ qsrc, float* qv, int row_words, int lane) {
  float ss = 0.f;
  for (int c = lane; c < row_words; c += 32) {
    const float v = qsrc[c];
    qv[c] = v;
    ss = fmaf(v, v, ss);
  }
  if constexpr (KIND == 1) {
    ss = warp_sum(ss);
    if (ss != 0.f) {
      const float sc = 1.f / sqrtf(ss);
      for (int c = lane; c < row_words; c += 32) qv[c] *= sc;
    }
  }
  __syncwarp();
}

// greedy descent through the upper layers (hnsw_distfunc_opt.cc:168-198): ends at the level-0 entry node
template <int KIND, int EVG>
__device__ __forceinline__ void greedy_descent(const HnswDeviceGraph& g, const float4* q4, int lane, int& cur_node,
                                               float& cur_dist, unsigned long long& n_eval) {
  cur_node = g.enterpoint;
  {
    int t[EVG] = {cur_node};
    float d[EVG];
    evalG<KIND, EVG>(g.vectors, g.row_words, q4, t, 1, lane, d);
    cur_dist = d[0];
    ++n_eval;
  }
  for (int level = g.maxlevel; level > 0; --level) {
    bool changed = true;
    while (changed) {
      changed = false;
      const int32_t* lk = g.upper + g.upper_off[cur_node] + (size_t)(level - 1) * (g.maxM + 1);
      const int size = lk[0];
      for (int b0 = 0; b0 < size; b0 += 32) {
        const int nb = (b0 + lane < size) ? lk[1 + b0 + lane] : -1;
        unsigned mask = __ballot_sync(FULL, nb >= 0);
        float my_d = __int_as_float(0x7F800000);
        while (mask) {
          int t[EVG], src[EVG], cnt = 0;
#pragma unroll
          for (int gq = 0; gq < EVG; ++gq) {
            src[gq] = 0;
            t[gq] = 0;
            if (mask) {
              src[gq] = __ffs(mask) - 1;
              mask &= mask - 1;
              ++cnt;
            }
          }
#pragma unroll
          for (int gq = 0; gq < EVG; ++gq) t[gq] = __shfl_sync(FULL, nb, src[gq]);
          float d[EVG];
          evalG<KIND, EVG>(g.vectors, g.row_words, q4, t, cnt, lane, d);
          n_eval += cnt;
#pragma unroll
          for (int gq = 0; gq < EVG; ++gq)
            if (gq < cnt && lane == src[gq]) my_d = d[gq];
        }
        // sequential "if (d < curdist)" over j == first minimum over the list
        uint64_t best = ((uint64_t)f32_ordered(my_d) << 32) | (uint32_t)lane;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const uint64_t other = __shfl_xor_sync(FULL, best, o);
          best = other < best ? other : best;
        }
        const int bl = (int)(best & 31u);
        const float bd = __shfl_sync(FULL, my_d, bl);
        const int bn = __shfl_sync(FULL, nb, bl);
        if (bn >= 0 && bd < cur_dist) {
          cur_dist = bd;
          cur_node = bn;
          changed = true;
        }
      }
    }
  }
}

// merge the accepted neighbours of one adjacency chunk (one per lane) into the beam W: SortArrBI's
// merge_with_sorted_items (sort_arr_bi.h:159-199) -- new items go after equal old ones, the tail shifts up and is
// truncated at the capacity, cur rewinds to the smallest insertion index
__device__ __forceinline__ void beam_insert(bool accept, float my_d, int nb, float* wkey, int* wdat, int* pbuf, int cap,
                                            int lane, int& n_w, int& cur) {
  const int m = __popc(__ballot_sync(FULL, accept));
  if (m == 0) return;
  // sort the accepted candidates; lane i < m ends with the i-th smallest
  uint64_t item = accept ? (((uint64_t)f32_ordered(my_d) << 32) | (uint32_t)nb) : KEY_MAX;
  item = warp_sort64(item, lane);
  const float d_i = f32_from_ordered((uint32_t)(item >> 32));
  const int t_i = (int)(uint32_t)item;
  // p_i = number of beam items with key <= d_i (new items go after equal old ones)
  int p_i = n_w;
  if (lane < m) {
    int lo = 0, hi = n_w;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (wkey[mid] <= d_i) lo = mid + 1; else hi = mid;
    }
    p_i = lo;
  }
  pbuf[lane] = lane < m ? p_i : 0x7FFFFFFF;
  __syncwarp();
  const int p0 = pbuf[0];
  // shift the tail of the beam, highest chunk first
  if (p0 < n_w) {
    for (int cb = ((n_w - 1) >> 5) << 5; cb >= ((p0 >> 5) << 5); cb -= 32) {
      const int a = cb + lane;
      const bool valid = a < n_w && a >= p0;
      float ka = 0.f;
      int da = 0, c = 0;
      if (valid) {
        ka = wkey[a];
        da = wdat[a];
        for (int i = 0; i < m; ++i) c += (pbuf[i] <= a) ? 1 : 0;
      }
      __syncwarp();
      if (valid && a + c < cap) {
        wkey[a + c] = ka;
        wdat[a + c] = da;
      }
      __syncwarp();
    }
  }
  if (lane < m && p_i + lane < cap) {
    wkey[p_i + lane] = d_i;
    wdat[p_i + lane] = t_i;
  }
  n_w = min(cap, n_w + m);
  if (p0 < cur) cur = p0;  // p_0 + 0 is the smallest insertion index (sort_arr_bi.h:159-199)
  __syncwarp();
}

// advance to the first unused item of the beam (hnsw_distfunc_opt.cc:272)
__device__ __forceinline__ void beam_advance(const int* wdat, int n_w, int lane, int& cur) {
  while (cur < n_w) {
    const int a = cur + lane;
    const bool unused = a < n_w && !(wdat[a] & USED_BIT);
    const unsigned um = __ballot_sync(FULL, unused);
    if (um) {
      cur += __ffs(um) - 1;
      break;
    }
    cur += 32;
  }
  if (cur > n_w) cur = n_w;
}

template <int KIND, int EVG, int MINB>  // EVG: neighbour vectors gathered at once per warp
__global__ void __launch_bounds__(WARPS * 32, MINB)
hnsw_search_kernel(HnswDeviceGraph g, const void* __restrict__ queries, int nq, int k, int ef, int cap,
                   int cap_r, uint8_t* __restrict__ visited, size_t visited_stride,
                   int* __restrict__ slot_epoch, uint64_t* __restrict__ out_keys,
                   unsigned long long* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t per_warp = (size_t)g.row_words * 4 + (size_t)cap_r * 8 + 32 * 4;
  unsigned char* base = smem_raw + per_warp * warp;
  float* qv = reinterpret_cast<float*>(base);                       // row_words
  float* wkey = qv + g.row_words;                                   // cap_r
  int* wdat = reinterpret_cast<int*>(wkey + cap_r);                 // cap_r (bit 31 = used)
  int* pbuf = wdat + cap_r;                                         // 32
  const float4* q4 = reinterpret_cast<const float4*>(qv);

  const int slot = blockIdx.x * WARPS + warp;
  uint8_t* vis = visited + (size_t)slot * visited_stride;
  unsigned long long n_eval = 0, n_exp = 0;

  // queries are handed out dynamically (they differ a lot in length): counters[2] is the next query index
  for (;;) {
    int qi = 0;
    if (lane == 0) qi = (int)atomicAdd(&counters[2], 1ull);
    qi = __shfl_sync(FULL, qi, 0);
    if (qi >= nq) break;
    // ---- visited epoch (VisitedList::reset, hnsw.h:575-582) ----
    int epoch = 0;
    if (lane == 0) epoch = slot_epoch[slot] + 1;
    epoch = __shfl_sync(FULL, epoch, 0);
    if (epoch > 255) {
      uint4 z = make_uint4(0, 0, 0, 0);
      for (size_t o = (size_t)lane * 16; o < visited_stride; o += 32 * 16) *reinterpret_cast<uint4*>(vis + o) = z;
      epoch = 1;
    }
    if (lane == 0) slot_epoch[slot] = epoch;
    const uint8_t ep = (uint8_t)epoch;
    __syncwarp();

    stage_query<KIND>(static_cast<const float*>(queries) + (size_t)qi * g.row_words, qv, g.row_words, lane);
    int cur_node;
    float cur_dist;
    greedy_descent<KIND, EVG>(g, q4, lane, cur_node, cur_dist, n_eval);

    // ---- level-0 beam (hnsw_distfunc_opt.cc:200-274) ----
    int n_w = 1, cur = 0;
    if (lane == 0) {
      wkey[0] = cur_dist;
      wdat[0] = cur_node;
      vis[cur_node] = ep;
    }
    __syncwarp();

    while (cur < min(n_w, ef)) {
      const int node = wdat[cur] & ~USED_BIT;
      __syncwarp();
      if (lane == 0) wdat[cur] |= USED_BIT;
      ++cur;
      ++n_exp;
      const float top_key = wkey[n_w - 1];
      const bool grow = n_w < ef;
      __syncwarp();
      const int size = g.links0_cnt[node];
      for (int b0 = 0; b0 < size; b0 += 32) {
        const int nb = (b0 + lane < size) ? g.links0[(size_t)node * g.maxM0 + b0 + lane] : -1;
        bool fresh = false;
        if (nb >= 0) {
          fresh = vis[nb] != ep;
          if (fresh) vis[nb] = ep;
        }
        unsigned mask = __ballot_sync(FULL, fresh);
        float my_d = __int_as_float(0x7F800000);
        while (mask) {
          int t[EVG], src[EVG], cnt = 0;
#pragma unroll
          for (int gq = 0; gq < EVG; ++gq) {
            src[gq] = 0;
            t[gq] = 0;
            if (mask) {
              src[gq] = __ffs(mask) - 1;
              mask &= mask - 1;
              ++cnt;
            }
          }
#pragma unroll
          for (int gq = 0; gq < EVG; ++gq) t[gq] = __shfl_sync(FULL, nb, src[gq]);
          float d[EVG];
          evalG<KIND, EVG>(g.vectors, g.row_words, q4, t, cnt, lane, d);
          n_eval += cnt;
#pragma unroll
          for (int gq = 0; gq < EVG; ++gq)
            if (gq < cnt && lane == src[gq]) my_d = d[gq];
        }
        beam_insert(fresh && (my_d < top_key || grow), my_d, nb, wkey, wdat, pbuf, cap, lane, n_w, cur);
      }
      beam_advance(wdat, n_w, lane, cur);
    }

    // ---- W[0..k) -> keys (hnsw_distfunc_opt.cc:276-281) ----
    __syncwarp();
    for (int e = lane; e < k; e += 32) {
      uint64_t key = KEY_MAX;
      if (e < n_w) key = make_key(f32_ordered(wkey[e]), (uint32_t)(wdat[e] & ~USED_BIT));
      out_keys[(size_t)qi * k + e] = key;
    }
    __syncwarp();
  }
  if (lane == 0) {
    atomicAdd(&counters[0], n_eval);
    atomicAdd(&counters[1], n_exp);
  }
}

// ---------------------------------------------------------------- small batches: a team of 2 or 4 warps per query
// With fewer queries than resident warps (a 10 K batch split over 8 replicas leaves 1 250 per GPU for 3 552 warps)
// the one-warp kernel is a chain of dependent gather rounds per query and most of the machine idles.  Here a team of
// TW warps owns ONE query: the team's warp 0 runs exactly the control flow of hnsw_search_kernel (query staging,
// greedy descent, adjacency + visited check, beam insertion -- so the expansions, their order and every comparison
// are the same), and the distance evaluations of an expansion are dealt out to all TW warps, EVG rows each, through
// shared memory.  A round of up to 4 TW neighbours replaces TW rounds of four.  The per-pair arithmetic is evalG's,
// so the answers are bit-identical to the one-warp kernel's (tests/test_hnsw_gpu.py runs all of them on one graph).
// A block holds WARPS / TW teams; a team synchronises on its own named barrier.
template <int TW>
__device__ __forceinline__ void team_sync(int team) {
  if (TW == WARPS) __syncthreads();
  else asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(TW * 32) : "memory");
}

template <int KIND, int EVG, int TW>
__global__ void __launch_bounds__(WARPS * 32, 6)
hnsw_search_team_kernel(HnswDeviceGraph g, const void* __restrict__ queries, int nq, int k, int ef, int cap,
                        int cap_r, uint8_t* __restrict__ visited, size_t visited_stride,
                        int* __restrict__ slot_epoch, uint64_t* __restrict__ out_keys,
                        unsigned long long* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int team = (threadIdx.x >> 5) / TW, warp = (threadIdx.x >> 5) % TW;  // warp: index inside the team
  const int tthread = warp * 32 + lane;                                     // thread index inside the team
  const size_t per_team = (size_t)g.row_words * 4 + (size_t)cap_r * 8 + 3 * 32 * 4 + 8 * 4;
  float* qv = reinterpret_cast<float*>(smem_raw + per_team * team);  // row_words
  float* wkey = qv + g.row_words;                                   // cap_r
  int* wdat = reinterpret_cast<int*>(wkey + cap_r);                 // cap_r (bit 31 = used)
  int* pbuf = wdat + cap_r;                                         // 32
  int* s_nb = pbuf + 32;                                            // 32: neighbours of the current chunk
  float* s_d = reinterpret_cast<float*>(s_nb + 32);                 // 32: their distances
  int* s_ctl = reinterpret_cast<int*>(s_d + 32);                    // 8: qi, cur, n_w, fresh mask, more-chunks flag
  const float4* q4 = reinterpret_cast<const float4*>(qv);

  const int slot = blockIdx.x * (WARPS / TW) + team;
  uint8_t* vis = visited + (size_t)slot * visited_stride;
  unsigned long long n_eval = 0, n_exp = 0;

  // evaluation service: every warp takes every fourth group of EVG fresh neighbours of the published chunk
  auto team_eval = [&]() {
    unsigned mask = (unsigned)s_ctl[3];
    const int nb = s_nb[lane];
    int grp = 0;
    while (mask) {
      int t[EVG], src[EVG], cnt = 0;
#pragma unroll
      for (int gq = 0; gq < EVG; ++gq) {
        src[gq] = 0;
        t[gq] = 0;
        if (mask) {
          src[gq] = __ffs(mask) - 1;
          mask &= mask - 1;
          ++cnt;
        }
      }
      if ((grp++ % TW) != warp) continue;
#pragma unroll
      for (int gq = 0; gq < EVG; ++gq) t[gq] = __shfl_sync(FULL, nb, src[gq]);
      float d[EVG];
      evalG<KIND, EVG>(g.vectors, g.row_words, q4, t, cnt, lane, d);
#pragma unroll
      for (int gq = 0; gq < EVG; ++gq)
        if (gq < cnt && lane == 0) s_d[src[gq]] = d[gq];
    }
  };

  for (;;) {
    if (tthread == 0) s_ctl[0] = (int)atomicAdd(&counters[2], 1ull);
    team_sync<TW>(team);
    const int qi = s_ctl[0];
    if (qi >= nq) break;
    // ---- visited epoch (VisitedList::reset, hnsw.h:575-582) ----
    int epoch = slot_epoch[slot] + 1;
    team_sync<TW>(team);
    if (epoch > 255) {
      uint4 z = make_uint4(0, 0, 0, 0);
      for (size_t o = (size_t)tthread * 16; o < visited_stride; o += TW * 32 * 16)
        *reinterpret_cast<uint4*>(vis + o) = z;
      epoch = 1;
    }
    if (tthread == 0) slot_epoch[slot] = epoch;
    const uint8_t ep = (uint8_t)epoch;
    team_sync<TW>(team);

    int n_w = 1, cur = 0;
    if (warp == 0) {
      // query staging and greedy descent by the team's warp 0 alone: the one-warp kernel's arithmetic
      stage_query<KIND>(static_cast<const float*>(queries) + (size_t)qi * g.row_words, qv, g.row_words, lane);
      int cur_node;
      float cur_dist;
      greedy_descent<KIND, EVG>(g, q4, lane, cur_node, cur_dist, n_eval);
      if (lane == 0) {
        wkey[0] = cur_dist;
        wdat[0] = cur_node;
        vis[cur_node] = ep;
        s_ctl[1] = 0;  // cur
        s_ctl[2] = 1;  // n_w
      }
    }
    team_sync<TW>(team);

    // ---- level-0 beam (hnsw_distfunc_opt.cc:200-274): warp 0 decides, everybody evaluates ----
    for (;;) {
      cur = s_ctl[1];
      n_w = s_ctl[2];
      if (!(cur < min(n_w, ef))) break;
      int node = 0, size = 0;
      float top_key = 0.f;
      bool grow = false;
      if (warp == 0) {
        node = wdat[cur] & ~USED_BIT;
        __syncwarp();
        if (lane == 0) wdat[cur] |= USED_BIT;
        ++cur;
        ++n_exp;
        top_key = wkey[n_w - 1];
        grow = n_w < ef;
        __syncwarp();
        size = g.links0_cnt[node];
      }
      for (int b0 = 0;; b0 += 32) {
        int nb = -1;
        bool fresh = false;
        if (warp == 0) {
          nb = (b0 + lane < size) ? g.links0[(size_t)node * g.maxM0 + b0 + lane] : -1;
          if (nb >= 0) {
            fresh = vis[nb] != ep;
            if (fresh) vis[nb] = ep;
          }
          const unsigned mask = __ballot_sync(FULL, fresh);
          s_nb[lane] = nb;
          if (lane == 0) {
            s_ctl[3] = (int)mask;
            s_ctl[4] = b0 < size ? 1 : 0;  // 0: no such chunk, the expansion is over
          }
          n_eval += __popc(mask);
        }
        team_sync<TW>(team);
        if (!s_ctl[4]) break;
        team_eval();
        team_sync<TW>(team);
        if (warp == 0) {
          const float my_d = fresh ? s_d[lane] : __int_as_float(0x7F800000);
          beam_insert(fresh && (my_d < top_key || grow), my_d, nb, wkey, wdat, pbuf, cap, lane, n_w, cur);
        }
        // (the next chunk's publication overwrites s_nb / s_ctl[3..4]: everybody has read them before this barrier)
        team_sync<TW>(team);
      }
      if (warp == 0) {
        beam_advance(wdat, n_w, lane, cur);
        if (lane == 0) {
          s_ctl[1] = cur;
          s_ctl[2] = n_w;
        }
      }
      team_sync<TW>(team);
    }

    // ---- W[0..k) -> keys (hnsw_distfunc_opt.cc:276-281) ----
    for (int e = tthread; e < k; e += TW * 32) {
      uint64_t key = KEY_MAX;
      if (e < n_w) key = make_key(f32_ordered(wkey[e]), (uint32_t)(wdat[e] & ~USED_BIT));
      out_keys[(size_t)qi * k + e] = key;
    }
    team_sync<TW>(team);
  }
  if (tthread == 0) {
    atomicAdd(&counters[0], n_eval);
    atomicAdd(&counters[1], n_exp);
  }
}

}  // namespace

int hnsw_max_ef() { return MAX_EF; }
int hnsw_warps_per_block() { return WARPS; }

cudaError_t launch_hnsw_search(const HnswDeviceGraph& g, const void* queries, int nq, int k, int ef,
                               uint8_t* visited, int* slot_epoch, int slots, uint64_t* out_keys,
                               unsigned long long* counters, cudaStream_t stream) {
  if (nq <= 0) return cudaSuccess;
  const int cap = ef > k ? ef : k;
  if (cap > MAX_EF) return cudaErrorInvalidValue;
  const int cap_r = (cap + 31) / 32 * 32;
  const size_t per_warp = (size_t)g.row_words * 4 + (size_t)cap_r * 8 + 32 * 4;
  const size_t smem = per_warp * WARPS;
  if (smem > 227 * 1024) return cudaErrorInvalidValue;  // (rows this long leave no room for a beam this wide)
  int blocks = slots / WARPS;
  const int need = (nq + WARPS - 1) / WARPS;
  if (blocks > need) blocks = need;
  if (blocks < 1) blocks = 1;
  const size_t vstride = round_up((size_t)g.n, 16);
  cudaError_t e;
  static const int evg = [] {
    const char* e2 = nb200_env("NB200_HNSW_G");
    return e2 ? atoi(e2) : 4;
  }();
  static const int minb = [] {
    const char* e2 = nb200_env("NB200_HNSW_MINB");
    return e2 ? atoi(e2) : 6;
  }();
  cudaMemsetAsync(counters + 2, 0, 8, stream);  // next query index
  // few queries: a team of 4 or 2 warps per query (hnsw_search_team_kernel); the one-warp kernel keeps 4 x the
  // resident blocks' worth of queries in flight, so it wins as soon as the batch fills that
  const int team_mode = nb200_option("hnsw_team", -1);  // -1 auto, 0 never, 2 / 4 always that team size (A/B runs)
  {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int resident = 6 * sms;  // blocks of 4 warps per wave at the kernels' occupancy
    int tw = 0;
    if (team_mode == 2 || team_mode == 4) tw = team_mode;
    else if (team_mode == 1) tw = 4;
    else if (team_mode < 0) tw = nq <= resident * 3 / 2 ? 4 : nq <= resident * 3 ? 2 : 0;
    if (tw) {
      const size_t per_team = (size_t)g.row_words * 4 + (size_t)cap_r * 8 + 3 * 32 * 4 + 8 * 4;
      const int teams = WARPS / tw;
      const size_t tsmem = per_team * teams;
#define NB_TEAM(KIND, TWV)                                                                                            \
  {                                                                                                                   \
    e = cudaFuncSetAttribute(hnsw_search_team_kernel<KIND, 4, TWV>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                             (int)tsmem);                                                                             \
    if (e != cudaSuccess) return e;                                                                                   \
    int occ = 0;                                                                                                      \
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, hnsw_search_team_kernel<KIND, 4, TWV>, WARPS * 32, tsmem);    \
    int tb = std::min(slots / teams, std::max(1, occ) * sms); /* one resident wave: a team owns its visited array */  \
    if (tb > (nq + teams - 1) / teams) tb = (nq + teams - 1) / teams;                                                 \
    hnsw_search_team_kernel<KIND, 4, TWV><<<tb, WARPS * 32, tsmem, stream>>>(g, queries, nq, k, ef, cap, cap_r,        \
                                                                             visited, vstride, slot_epoch, out_keys,  \
                                                                             counters);                               \
  }
#define NB_TEAM2(KIND)          \
  if (tw == 4) NB_TEAM(KIND, 4) \
  else NB_TEAM(KIND, 2)
      switch (g.dist_kind) {
        case 0: NB_TEAM2(0); break;
        case 1: NB_TEAM2(1); break;
        case 2: NB_TEAM2(2); break;
        case 3: NB_TEAM2(3); break;
        default: return cudaErrorInvalidValue;
      }
#undef NB_TEAM2
#undef NB_TEAM
      return cudaGetLastError();
    }
  }
#define NB_HNSW3(KIND, G, MB)                                                                                   \
  {                                                                                                             \
    e = cudaFuncSetAttribute(hnsw_search_kernel<KIND, G, MB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if (e != cudaSuccess) return e;                                                                             \
    int occ = 0, dev = 0, sms = 0;                                                                              \
    cudaGetDevice(&dev);                                                                                        \
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);                                          \
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, hnsw_search_kernel<KIND, G, MB>, WARPS * 32, smem);      \
    if (occ > 0 && blocks > occ * sms) blocks = occ * sms; /* one resident wave: a slot owns its visited array */ \
    hnsw_search_kernel<KIND, G, MB><<<blocks, WARPS * 32, smem, stream>>>(g, queries, nq, k, ef, cap, cap_r,      \
                                                                         visited, vstride, slot_epoch, out_keys, \
                                                                         counters);                             \
  }
#define NB_HNSW(KIND)                                  \
  if (evg == 8) NB_HNSW3(KIND, 8, 3)                   \
  else if (evg == 2) NB_HNSW3(KIND, 2, 8)              \
  else if (minb >= 8) NB_HNSW3(KIND, 4, 8)             \
  else NB_HNSW3(KIND, 4, 6)
  switch (g.dist_kind) {
    case 0: NB_HNSW(0); break;
    case 1: NB_HNSW(1); break;
    case 2: NB_HNSW(2); break;
    case 3: NB_HNSW(3); break;
    default: return cudaErrorInvalidValue;
  }
#undef NB_HNSW
#undef NB_HNSW3
  return cudaGetLastError();
}

}  // namespace nb200
