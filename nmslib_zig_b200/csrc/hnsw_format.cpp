// hnsw_format.cpp -- reader / writer for the reference's optimized HNSW index stream.
//
// This is the graph hand-off between the reference CPU builder and the device engine
// (SURVEY.md 0.7, Appendix B): Hnsw::SaveIndex / SaveOptimizedIndex write it
// (src/method/hnsw.cc:748-806), LoadOptimizedIndex reads it (:1025-1074).  Layout
// (little endian, unpadded):
//   u32 optimized(=1) | u32 total | u64 memoryPerObject | u64 offsetLevel0 | u64 offsetData
//   i32 maxlevel | u32 enterpoint | u64 maxM | u64 maxM0 | i32 dist_func | u64 searchMethod
//   total records of memoryPerObject bytes:
//       [i32 id | i32 label | u64 datalen | float[dim]] [i32 count | i32 nbr[maxM0]]
//   per node: u32 bytes, then `bytes` of upper-level lists ((maxM+1) ints per level)
// The device wants structure-of-arrays, so the records are split here.
#include <cstdio>
#include <cstring>
#include <memory>

#include "engine.h"

namespace nb200 {

namespace {
struct FileCloser {
  void operator()(FILE* f) const {
    if (f) fclose(f);
  }
};
using FilePtr = std::unique_ptr<FILE, FileCloser>;

template <typename T>
bool rd(FILE* f, T* v) {
  return fread(v, sizeof(T), 1, f) == 1;
}
template <typename T>
bool wr(FILE* f, const T& v) {
  return fwrite(&v, sizeof(T), 1, f) == 1;
}
constexpr int kErrIO = 10;  // NMSLIB_ERROR_DATA_IO_FAILED
}  // namespace

namespace {
// Hnsw::SaveRegularIndexBin (hnsw.cc:810-842): total (u32), maxlevel (i32), enterpoint (u32), M / maxM / maxM0 (size_t),
// then per node its level and, per level 0..level, the friend count and the friend ids.  No vectors, no external ids:
// the data set is the caller's (LoadRegularIndexBin CHECKs that the counts agree, hnsw.cc:956-959).  The result has
// dim == 0 and empty vectors / ext_ids; dist_func is filled in by the engine from the index space.
Status read_regular(FILE* f, HnswGraph* out) {
  uint32_t total = 0, enterpoint = 0;
  int32_t maxlevel = 0;
  uint64_t M = 0, maxM = 0, maxM0 = 0;
  if (!(rd(f, &total) && rd(f, &maxlevel) && rd(f, &enterpoint) && rd(f, &M) && rd(f, &maxM) && rd(f, &maxM0)))
    return Status::Err(kErrIO, "truncated regular HNSW header");
  if (maxM0 == 0 || maxM0 > 4096 || maxM == 0 || maxM > 4096 || maxlevel < 0 || maxlevel > 64 ||
      (total > 0 && enterpoint >= total))
    return Status::Err(kErrIO, "inconsistent regular HNSW header");
  HnswGraph g;
  g.total = total;
  g.dim = 0;
  g.maxM = (int)maxM;
  g.maxM0 = (int)maxM0;
  g.maxlevel = maxlevel;
  g.M = (int)M;
  g.enterpoint = enterpoint;
  g.dist_func = 0;
  g.links0.assign((size_t)total * g.maxM0, -1);
  g.links0_cnt.assign(total, 0);
  g.upper_off.assign(total, -1);
  std::vector<int32_t>& levels = g.levels;
  levels.assign(total, 0);
  std::vector<int32_t> ids;
  for (uint32_t i = 0; i < total; ++i) {
    uint32_t level = 0;
    if (!rd(f, &level) || level > 64) return Status::Err(kErrIO, "corrupt regular HNSW node record");
    levels[i] = (int32_t)level;
    if (level > 0) {
      g.upper_off[i] = (int64_t)g.upper.size();
      g.upper.resize(g.upper.size() + (size_t)level * (maxM + 1), 0);
    }
    for (uint32_t l = 0; l <= level; ++l) {
      uint32_t cnt = 0;
      if (!rd(f, &cnt) || cnt > (l == 0 ? maxM0 : maxM)) return Status::Err(kErrIO, "corrupt regular HNSW friend list");
      ids.resize(cnt);
      if (cnt && fread(ids.data(), 4, cnt, f) != cnt) return Status::Err(kErrIO, "truncated regular HNSW friend list");
      for (uint32_t j = 0; j < cnt; ++j)
        if ((uint32_t)ids[j] >= total) return Status::Err(kErrIO, "regular HNSW friend id out of range");
      if (l == 0) {
        g.links0_cnt[i] = (int32_t)cnt;
        for (uint32_t j = 0; j < cnt; ++j) g.links0[(size_t)i * g.maxM0 + j] = ids[j];
      } else {
        int32_t* lk = &g.upper[g.upper_off[i] + (size_t)(l - 1) * (maxM + 1)];
        lk[0] = (int32_t)cnt;
        for (uint32_t j = 0; j < cnt; ++j) lk[1 + j] = ids[j];
      }
    }
  }
  // level consistency (see read_hnsw_file): the descent follows a level-l link only into nodes that have level l
  if (total > 0 && levels[enterpoint] < maxlevel) {
    // (hnsw.cc:824-828 notes that maxlevel_ may exceed the entry node's level; the pointer search starts from
    //  enterpoint_->level, hnsw.cc:1183, so that is the level the descent must use; a save writes the header's)
    g.file_maxlevel = maxlevel;
    g.maxlevel = levels[enterpoint];
  }
  for (uint32_t i = 0; i < total; ++i)
    for (int32_t l = 1; l <= levels[i]; ++l) {
      const int32_t* lk = &g.upper[g.upper_off[i] + (size_t)(l - 1) * (maxM + 1)];
      for (int j = 1; j <= lk[0]; ++j)
        if (levels[lk[j]] < l) return Status::Err(kErrIO, "regular HNSW friend does not reach that level");
    }
  *out = std::move(g);
  return Status::OK();
}
}  // namespace

Status read_hnsw_file(const std::string& path, HnswGraph* out) {
  FilePtr f(fopen(path.c_str(), "rb"));
  if (!f) return Status::Err(kErrIO, "cannot open HNSW index file " + path);
  uint32_t optimized = 0, total = 0, enterpoint = 0;
  uint64_t mem_per_obj = 0, off_level0 = 0, off_data = 0, maxM = 0, maxM0 = 0, search_method = 0;
  int32_t maxlevel = 0, dist_func = 0;
  if (!rd(f.get(), &optimized)) return Status::Err(kErrIO, "truncated HNSW header");
  if (optimized == 0) return read_regular(f.get(), out);  // the pointer graph of Hnsw<int> / skip_optimized_index
  if (optimized != 1) return Status::Err(kErrIO, "not an HNSW index file (hnsw.cc:756 flag)");
  if (!(rd(f.get(), &total) && rd(f.get(), &mem_per_obj) && rd(f.get(), &off_level0) &&
        rd(f.get(), &off_data) && rd(f.get(), &maxlevel) && rd(f.get(), &enterpoint) && rd(f.get(), &maxM) &&
        rd(f.get(), &maxM0) && rd(f.get(), &dist_func) && rd(f.get(), &search_method)))
    return Status::Err(kErrIO, "truncated HNSW header");
  if (off_level0 < 16 || (off_level0 - 16) % 4 != 0 || mem_per_obj != off_level0 + 4 * (maxM0 + 1) ||
      off_data != 0 || maxM0 == 0 || maxM0 > 4096 || maxM > 4096)
    return Status::Err(kErrIO, "inconsistent HNSW header");
  if (dist_func < 1 || dist_func > 4)
    return Status::Err(5, "HNSW dist_func_type " + std::to_string(dist_func) +
                              " (l1/linf) is outside this engine's path");
  if (total > 0 && enterpoint >= total) return Status::Err(kErrIO, "HNSW enterpoint out of range");

  HnswGraph g;
  g.total = total;
  g.dim = (int)((off_level0 - 16) / 4);
  g.maxM = (int)maxM;
  g.maxM0 = (int)maxM0;
  g.maxlevel = maxlevel;
  g.enterpoint = enterpoint;
  g.dist_func = dist_func;
  g.vectors.resize((size_t)total * g.dim);
  g.ext_ids.resize(total);
  g.links0.assign((size_t)total * g.maxM0, -1);
  g.links0_cnt.resize(total);
  g.upper_off.assign(total, -1);

  std::vector<char> rec(mem_per_obj);
  for (uint32_t i = 0; i < total; ++i) {
    if (fread(rec.data(), 1, mem_per_obj, f.get()) != mem_per_obj)
      return Status::Err(kErrIO, "truncated HNSW level-0 section");
    int32_t id;
    memcpy(&id, rec.data(), 4);
    g.ext_ids[i] = id;
    memcpy(&g.vectors[(size_t)i * g.dim], rec.data() + 16, (size_t)g.dim * 4);
    int32_t cnt;
    memcpy(&cnt, rec.data() + off_level0, 4);
    if (cnt < 0 || cnt > g.maxM0) return Status::Err(kErrIO, "corrupt HNSW level-0 list");
    g.links0_cnt[i] = cnt;
    memcpy(&g.links0[(size_t)i * g.maxM0], rec.data() + off_level0 + 4, (size_t)cnt * 4);
    for (int j = 0; j < cnt; ++j)
      if ((uint32_t)g.links0[(size_t)i * g.maxM0 + j] >= total)
        return Status::Err(kErrIO, "HNSW level-0 neighbour out of range");
  }
  for (uint32_t i = 0; i < total; ++i) {
    uint32_t bytes = 0;
    if (!rd(f.get(), &bytes)) return Status::Err(kErrIO, "truncated HNSW upper-level section");
    if (!bytes) continue;
    if (bytes % (4 * (maxM + 1)) != 0) return Status::Err(kErrIO, "corrupt HNSW upper-level list size");
    g.upper_off[i] = (int64_t)g.upper.size();
    const size_t words = bytes / 4;
    g.upper.resize(g.upper.size() + words);
    if (fread(&g.upper[g.upper_off[i]], 4, words, f.get()) != words)
      return Status::Err(kErrIO, "truncated HNSW upper-level section");
    const size_t levels = words / (maxM + 1);
    for (size_t l = 0; l < levels; ++l) {
      const int32_t* lk = &g.upper[g.upper_off[i] + l * (maxM + 1)];
      if (lk[0] < 0 || lk[0] > (int)maxM) return Status::Err(kErrIO, "corrupt HNSW upper-level list");
      for (int j = 1; j <= lk[0]; ++j)
        if ((uint32_t)lk[j] >= total) return Status::Err(kErrIO, "HNSW upper-level neighbour out of range");
    }
  }
  // Level consistency: the greedy descent (hnsw_search.cu) reads the level-l list of every node it reaches at
  // level l without asking how many levels that node has -- the enterpoint at every level up to maxlevel, and each
  // neighbour named in a level-l list at level l.  A truncated or hostile file must not turn into device reads
  // outside the upper-level block.
  if (maxlevel < 0) return Status::Err(kErrIO, "negative HNSW maxlevel");
  {
    std::vector<int32_t>& levels = g.levels;
    levels.assign(total, 0);
    // (the blocks were appended in node order: a node's block ends where the next non-empty one starts)
    int64_t prev = -1;
    uint32_t prev_i = 0;
    for (uint32_t i = 0; i < total; ++i) {
      if (g.upper_off[i] < 0) continue;
      if (prev >= 0) levels[prev_i] = (int32_t)((g.upper_off[i] - prev) / (int64_t)(maxM + 1));
      prev = g.upper_off[i];
      prev_i = i;
    }
    if (prev >= 0) levels[prev_i] = (int32_t)(((int64_t)g.upper.size() - prev) / (int64_t)(maxM + 1));
    if (total > 0 && levels[enterpoint] < maxlevel)
      return Status::Err(kErrIO, "HNSW enterpoint has fewer levels than maxlevel");
    for (uint32_t i = 0; i < total; ++i)
      for (int32_t l = 1; l <= levels[i]; ++l) {
        const int32_t* lk = &g.upper[g.upper_off[i] + (size_t)(l - 1) * (maxM + 1)];
        for (int j = 1; j <= lk[0]; ++j)
          if (levels[lk[j]] < l) return Status::Err(kErrIO, "HNSW upper-level neighbour does not reach that level");
      }
  }
  *out = std::move(g);
  return Status::OK();
}

Status write_regular(const std::string& path, const HnswGraph& g) {
  if (g.levels.size() != g.total || g.M <= 0) return Status::Err(kErrIO, "graph without levels or M: no regular file");
  FilePtr f(fopen(path.c_str(), "wb"));
  if (!f) return Status::Err(kErrIO, "cannot open " + path + " for writing");
  bool ok = wr<uint32_t>(f.get(), 0) && wr<uint32_t>(f.get(), g.total) &&
            wr<int32_t>(f.get(), g.file_maxlevel >= 0 ? g.file_maxlevel : g.maxlevel) &&
            wr<uint32_t>(f.get(), g.enterpoint) && wr<uint64_t>(f.get(), (uint64_t)g.M) &&
            wr<uint64_t>(f.get(), (uint64_t)g.maxM) && wr<uint64_t>(f.get(), (uint64_t)g.maxM0);
  for (uint32_t i = 0; ok && i < g.total; ++i) {
    const uint32_t level = (uint32_t)g.levels[i];
    ok = wr<uint32_t>(f.get(), level);
    for (uint32_t l = 0; ok && l <= level; ++l) {
      const int32_t* lk = l == 0 ? &g.links0[(size_t)i * g.maxM0] : &g.upper[g.upper_off[i] + (size_t)(l - 1) * (g.maxM + 1)] + 1;
      const uint32_t cnt = l == 0 ? (uint32_t)g.links0_cnt[i] : (uint32_t)lk[-1];
      ok = wr<uint32_t>(f.get(), cnt) && (cnt == 0 || fwrite(lk, 4, cnt, f.get()) == cnt);
    }
  }
  if (!ok) return Status::Err(kErrIO, "short write to " + path);
  return Status::OK();
}

Status write_hnsw_file(const std::string& path, const HnswGraph& g, const float* vectors,
                       const int32_t* ext_ids) {
  FilePtr f(fopen(path.c_str(), "wb"));
  if (!f) return Status::Err(kErrIO, "cannot open " + path + " for writing");
  const uint64_t off_level0 = 16 + 4ull * g.dim;
  const uint64_t mem_per_obj = off_level0 + 4ull * (g.maxM0 + 1);
  bool ok = wr<uint32_t>(f.get(), 1) && wr<uint32_t>(f.get(), g.total) && wr<uint64_t>(f.get(), mem_per_obj) &&
            wr<uint64_t>(f.get(), off_level0) && wr<uint64_t>(f.get(), 0) && wr<int32_t>(f.get(), g.maxlevel) &&
            wr<uint32_t>(f.get(), g.enterpoint) && wr<uint64_t>(f.get(), (uint64_t)g.maxM) &&
            wr<uint64_t>(f.get(), (uint64_t)g.maxM0) && wr<int32_t>(f.get(), g.dist_func) &&
            wr<uint64_t>(f.get(), 3);
  std::vector<char> rec(mem_per_obj);
  for (uint32_t i = 0; ok && i < g.total; ++i) {
    memset(rec.data(), 1, mem_per_obj);  // hnsw.cc:428 pre-fills records with 0x01
    const int32_t id = ext_ids[i], label = -1;
    const uint64_t datalen = 4ull * g.dim;
    memcpy(rec.data(), &id, 4);
    memcpy(rec.data() + 4, &label, 4);
    memcpy(rec.data() + 8, &datalen, 8);
    memcpy(rec.data() + 16, vectors + (size_t)i * g.dim, datalen);
    const int32_t cnt = g.links0_cnt[i];
    memcpy(rec.data() + off_level0, &cnt, 4);
    memcpy(rec.data() + off_level0 + 4, &g.links0[(size_t)i * g.maxM0], (size_t)cnt * 4);
    ok = fwrite(rec.data(), 1, mem_per_obj, f.get()) == mem_per_obj;
  }
  for (uint32_t i = 0; ok && i < g.total; ++i) {
    uint32_t bytes = 0;
    if (g.upper_off[i] >= 0) {
      // the list block of node i runs to the next node's block (or the end of the pool)
      int64_t end = (int64_t)g.upper.size();
      for (uint32_t j = i + 1; j < g.total; ++j)
        if (g.upper_off[j] >= 0) {
          end = g.upper_off[j];
          break;
        }
      bytes = (uint32_t)((end - g.upper_off[i]) * 4);
    }
    ok = wr<uint32_t>(f.get(), bytes);
    if (ok && bytes) ok = fwrite(&g.upper[g.upper_off[i]], 1, bytes, f.get()) == bytes;
  }
  if (!ok) return Status::Err(kErrIO, "short write to " + path);
  return Status::OK();
}

}  // namespace nb200
