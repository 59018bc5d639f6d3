// hnsw_build.cpp -- host-side HNSW graph construction (index BUILD, not the query path).
//
// The hot path this library replaces is the QUERY side of Hnsw (SURVEY.md 8a); graph construction
// stays on CPU cores, as in the reference.  When the graph comes from the reference itself it is
// imported (hnsw_format.cpp) and searched unchanged.  This builder exists so that the library is a
// usable drop-in on its own: `nmslib_create_index(hnsw)` + `nmslib_add_data_point*` + a query work
// without the reference linked in (that is the call sequence of every test in lib.zig:1273-1558).
//
// Algorithm: the published HNSW insertion (Malkov & Yashunin), with the parameters and defaults of
// the reference -- M=16, efConstruction=200, maxM=M, maxM0=2M, mult=1/ln(M), neighbour selection by
// the "heuristic 2" rule that delaunay_type=2 selects (hnsw.cc:189-204, hnsw.h:129-169): scan the
// candidates by increasing distance and keep one only if it is closer to the new point than to every
// neighbour already kept.  Insertions run on all host threads with one lock per node, like the
// reference's ParallelFor build (hnsw.cc:238-247), so the graph is not bit-reproducible run to run
// (neither is the reference's, SURVEY 0.7); search parity is tested on imported graphs.
// The result is emitted in the reference's optimized-index layout (HnswGraph), so it can be saved
// with nmslib_save_index and loaded by the reference.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <queue>
#include <random>
#include <sstream>
#include <thread>

#include "engine.h"

namespace nb200 {
namespace {

typedef HnswBuildParams BuildParams;

}  // namespace

bool parse_hnsw_build_params(const std::vector<std::string>& params, HnswBuildParams* bp, std::string* err) {
  bool has_maxM = false, has_maxM0 = false, has_mult = false;
  for (const std::string& p : params) {
    const size_t eq = p.find('=');
    if (eq == std::string::npos) continue;
    const std::string name = p.substr(0, eq);
    const std::string val = p.substr(eq + 1);
    std::stringstream ss(val);
    double v = 0;
    ss >> v;
    if (name == "M") bp->M = (int)v;
    else if (name == "efConstruction") bp->efConstruction = (int)v;
    else if (name == "maxM") { bp->maxM = (int)v; has_maxM = true; }
    else if (name == "maxM0") { bp->maxM0 = (int)v; has_maxM0 = true; }
    else if (name == "mult") { bp->mult = v; has_mult = true; }
    else if (name == "delaunay_type") bp->delaunay_type = (int)v;
    else if (name == "indexThreadQty") bp->threads = (int)v;
    else if (name == "b200_build") bp->where = val == "device" || val == "gpu" ? 1 : val == "host" || val == "cpu" ? 0 : -1;
  }
  if (const char* e = nb200_env("NB200_HNSW_BUILD")) {  // A/B switch for the tools
    const std::string v(e);
    if (v == "device" || v == "gpu") bp->where = 1;
    else if (v == "host" || v == "cpu") bp->where = 0;
  }
  if (bp->M < 2 || bp->efConstruction < 1) {
    *err = "HNSW needs M >= 2 and efConstruction >= 1";
    return false;
  }
  if (!has_maxM) bp->maxM = bp->M;          // hnsw.cc:192
  if (!has_maxM0) bp->maxM0 = 2 * bp->M;    // hnsw.cc:193
  if (!has_mult) bp->mult = 1.0 / std::log((double)bp->M);
  if (bp->maxM0 > 4096 || bp->maxM > 4096) {
    *err = "maxM / maxM0 too large";
    return false;
  }
  return true;
}

std::vector<int> hnsw_assign_levels(size_t n, double mult) {
  std::vector<int> level(n);
  std::mt19937 rng(0);  // the reference seeds with 0 as well (init.cc:34)
  std::uniform_real_distribution<double> uni(0.0, 1.0);
  for (size_t i = 0; i < n; ++i) {
    double u = uni(rng);
    if (u < 1e-300) u = 1e-300;
    int l = (int)(-std::log(u) * mult);  // getRandomLevel, hnsw.h:476-480
    if (l > 30) l = 30;
    level[i] = l;
  }
  return level;
}

namespace {

struct Builder {
  const float* data;  // [n][dim] (cosine: unit-normalised copy)
  size_t n;
  int dim;
  int kind;  // 0 squared L2, 1 cosine on unit vectors, 2 negative dot
  BuildParams bp;
  std::vector<int> level;
  std::vector<std::vector<std::vector<int32_t>>> links;  // [node][level] -> neighbours
  std::vector<std::mutex> locks;
  std::mutex ep_lock;
  int maxlevel = -1;
  int64_t enterpoint = -1;

  float dist(const float* a, const float* b) const {
    float s = 0.f;
    if (kind == 0) {
      for (int i = 0; i < dim; ++i) {
        const float d = a[i] - b[i];
        s += d * d;
      }
      return s;
    }
    for (int i = 0; i < dim; ++i) s += a[i] * b[i];
    if (kind == 1) return std::max(0.f, 1.f - std::max(-1.f, std::min(1.f, s)));
    return -s;
  }
  const float* vec(size_t i) const { return data + i * (size_t)dim; }

  typedef std::pair<float, int32_t> Cand;

  // best-first search of one layer (the reference's kSearchElementsWithAttemptsLevel, hnsw.cc:611-708)
  std::vector<Cand> search_layer(const float* q, int32_t ep, float ep_dist, int ef, int lc,
                                 std::vector<uint32_t>& visited, uint32_t tag) {
    std::priority_queue<Cand> top;                                         // worst of the ef best on top
    std::priority_queue<Cand, std::vector<Cand>, std::greater<Cand>> cand;  // closest unexpanded on top
    top.emplace(ep_dist, ep);
    cand.emplace(ep_dist, ep);
    visited[ep] = tag;
    std::vector<int32_t> nbrs;
    while (!cand.empty()) {
      const Cand c = cand.top();
      if (c.first > top.top().first && (int)top.size() >= ef) break;
      cand.pop();
      {
        std::lock_guard<std::mutex> g(locks[c.second]);
        nbrs = links[c.second][lc];
      }
      for (int32_t t : nbrs) {
        if (visited[t] == tag) continue;
        visited[t] = tag;
        const float d = dist(q, vec(t));
        if ((int)top.size() < ef || d < top.top().first) {
          cand.emplace(d, t);
          top.emplace(d, t);
          if ((int)top.size() > ef) top.pop();
        }
      }
    }
    std::vector<Cand> out(top.size());
    for (size_t i = top.size(); i-- > 0;) {
      out[i] = top.top();
      top.pop();
    }
    return out;  // ascending by distance
  }

  // neighbour selection, heuristic 2 (hnsw.h:129-169); delaunay_type 0 keeps the closest
  std::vector<int32_t> select(const std::vector<Cand>& sorted, int m) const {
    std::vector<int32_t> keep;
    if ((int)sorted.size() <= m || bp.delaunay_type == 0) {
      for (size_t i = 0; i < sorted.size() && (int)keep.size() < m; ++i) keep.push_back(sorted[i].second);
      return keep;
    }
    for (const Cand& c : sorted) {
      if ((int)keep.size() >= m) break;
      bool good = true;
      for (int32_t s : keep)
        if (dist(vec(s), vec(c.second)) < c.first) {
          good = false;
          break;
        }
      if (good) keep.push_back(c.second);
    }
    return keep;
  }

  void insert(size_t i, std::vector<uint32_t>& visited, uint32_t& tag, int lvl) {
    const float* q = vec(i);
    int64_t ep;
    int top_level;
    std::unique_lock<std::mutex> epg(ep_lock);
    ep = enterpoint;
    top_level = maxlevel;
    if (ep < 0) {  // first element
      enterpoint = (int64_t)i;
      maxlevel = lvl;
      return;
    }
    if (lvl <= top_level) epg.unlock();  // only a new top level keeps the entry point locked (MaxLevelGuard_, hnsw.cc:539-541)

    int32_t cur = (int32_t)ep;
    float cur_dist = dist(q, vec(cur));
    for (int lc = top_level; lc > lvl; --lc) {  // greedy descent
      bool changed = true;
      while (changed) {
        changed = false;
        std::vector<int32_t> nbrs;
        {
          std::lock_guard<std::mutex> g(locks[cur]);
          nbrs = links[cur][lc];
        }
        for (int32_t t : nbrs) {
          const float d = dist(q, vec(t));
          if (d < cur_dist) {
            cur_dist = d;
            cur = t;
            changed = true;
          }
        }
      }
    }
    for (int lc = std::min(lvl, top_level); lc >= 0; --lc) {
      if (++tag == 0) {
        std::fill(visited.begin(), visited.end(), 0u);
        tag = 1;
      }
      std::vector<Cand> w = search_layer(q, cur, cur_dist, bp.efConstruction, lc, visited, tag);
      const int cap = lc == 0 ? bp.maxM0 : bp.maxM;
      std::vector<int32_t> sel = select(w, bp.M);
      {
        std::lock_guard<std::mutex> g(locks[i]);
        links[i][lc] = sel;
      }
      for (int32_t s : sel) {  // back links, re-pruned to the level's capacity when they overflow
        std::lock_guard<std::mutex> g(locks[s]);
        std::vector<int32_t>& ls = links[s][lc];
        if (std::find(ls.begin(), ls.end(), (int32_t)i) != ls.end()) continue;
        if ((int)ls.size() < cap) {
          ls.push_back((int32_t)i);
        } else {
          std::vector<Cand> all;
          all.reserve(ls.size() + 1);
          all.emplace_back(dist(vec(s), q), (int32_t)i);
          for (int32_t t : ls) all.emplace_back(dist(vec(s), vec(t)), t);
          std::sort(all.begin(), all.end());
          ls = select(all, cap);
        }
      }
      if (!w.empty()) {
        cur = w[0].second;
        cur_dist = w[0].first;
      }
    }
    if (lvl > top_level) {
      enterpoint = (int64_t)i;
      maxlevel = lvl;
    }
  }
};

}  // namespace

Status build_hnsw_host(const float* rows, size_t n, int dim, int dist_func, const int32_t* ext_ids,
                       const std::vector<std::string>& params, HnswGraph* out) {
  BuildParams bp;
  std::string err;
  if (!parse_hnsw_build_params(params, &bp, &err)) return Status::Err(8, err);
  if (n == 0) return Status::Err(8, "cannot build an HNSW graph over an empty data set");
  if (n > 0x7FFFFFF0ull) return Status::Err(6, "too many points for an HNSW graph");
  Builder b;
  b.data = rows;
  b.n = n;
  b.dim = dim;
  b.kind = dist_func == 3 ? 1 : dist_func == 4 ? 2 : 0;
  b.bp = bp;
  b.links.resize(n);
  std::vector<std::mutex> locks(n);
  b.locks.swap(locks);
  b.level = hnsw_assign_levels(n, bp.mult);
  for (size_t i = 0; i < n; ++i) b.links[i].resize(b.level[i] + 1);
  int threads = bp.threads > 0 ? bp.threads : (int)std::thread::hardware_concurrency();
  if (threads < 1) threads = 1;
  if (n < 2048) threads = 1;
  {
    std::vector<uint32_t> visited(n, 0);
    uint32_t tag = 0;
    const size_t serial = std::min<size_t>(n, threads > 1 ? 1024 : n);  // a seed graph before going parallel
    for (size_t i = 0; i < serial; ++i) b.insert(i, visited, tag, b.level[i]);
    if (serial < n) {
      std::atomic<size_t> next(serial);
      std::vector<std::thread> pool;
      for (int t = 0; t < threads; ++t)
        pool.emplace_back([&]() {
          std::vector<uint32_t> vis(n, 0);
          uint32_t tg = 0;
          for (;;) {
            const size_t i = next.fetch_add(1);
            if (i >= n) break;
            b.insert(i, vis, tg, b.level[i]);
          }
        });
      for (auto& th : pool) th.join();
    }
  }
  // flatten into the optimized-index layout (hnsw.cc:417-465)
  HnswGraph g;
  g.total = (uint32_t)n;
  g.dim = dim;
  g.maxM = bp.maxM;
  g.M = bp.M;
  g.maxM0 = bp.maxM0;
  g.maxlevel = b.maxlevel;
  g.levels.assign(b.level.begin(), b.level.end());
  g.enterpoint = (uint32_t)b.enterpoint;
  g.dist_func = dist_func;
  g.ext_ids.assign(ext_ids, ext_ids + n);
  g.links0.assign(n * (size_t)bp.maxM0, -1);
  g.links0_cnt.resize(n);
  g.upper_off.assign(n, -1);
  for (size_t i = 0; i < n; ++i) {
    const std::vector<int32_t>& l0 = b.links[i][0];
    const int c = (int)std::min<size_t>(l0.size(), (size_t)bp.maxM0);
    g.links0_cnt[i] = c;
    std::copy(l0.begin(), l0.begin() + c, g.links0.begin() + i * (size_t)bp.maxM0);
    if (b.level[i] >= 1) {
      g.upper_off[i] = (int64_t)g.upper.size();
      for (int l = 1; l <= b.level[i]; ++l) {
        const std::vector<int32_t>& ll = b.links[i][l];
        const int cc = (int)std::min<size_t>(ll.size(), (size_t)bp.maxM);
        g.upper.push_back(cc);
        for (int j = 0; j < bp.maxM; ++j) g.upper.push_back(j < cc ? ll[j] : 0x01010101);
      }
    }
  }
  *out = std::move(g);
  return Status::OK();
}

}  // namespace nb200
