// engine.cu -- host orchestration of the device query path (see engine.h).
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cctype>
#include <cstring>
#include <map>
#include <sstream>
#include <atomic>
#include <thread>

namespace nb200 {

namespace {
constexpr int kErrInvalid = 2, kErrOOM = 3, kErrIncompat = 5, kErrTooLarge = 6, kErrBuild = 8, kErrQuery = 9;
thread_local int g_default_device = -1;
std::mutex g_opt_mu;
std::map<std::string, int>& option_table() {
  static std::map<std::string, int> t;
  return t;
}
}  // namespace

// Variant selectors (kernels.h).  -DNB200_EXPERIMENTS builds also accept NB200_<NAME> from the environment.
int nb200_option(const char* name, int dflt) {
  {
    std::lock_guard<std::mutex> g(g_opt_mu);
    auto it = option_table().find(name);
    if (it != option_table().end()) return it->second;
  }
#ifdef NB200_EXPERIMENTS
  std::string env = "NB200_";
  for (const char* c = name; *c; ++c) env.push_back((char)toupper(*c));
  if (const char* e = getenv(env.c_str())) return atoi(e);
#endif
  return dflt;
}
void nb200_set_option(const char* name, int value) {
  std::lock_guard<std::mutex> g(g_opt_mu);
  option_table()[name] = value;
}
#ifdef NB200_EXPERIMENTS
const char* nb200_env(const char* name) { return getenv(name); }
#endif

int default_device() {
  if (g_default_device >= 0) return g_default_device;
  const char* lr = getenv("LOCAL_RANK");
  int d = lr ? atoi(lr) : 0;
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) == cudaSuccess && cnt > 0) d = d % cnt;
  return d;
}
void set_default_device(int d) { g_default_device = d; }
bool device_available() {
  int cnt = 0;
  cudaError_t e = cudaGetDeviceCount(&cnt);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return cnt > 0;
}

template <typename T>
bool HostSlab<T>::append(const T* src, size_t count) {
  if (count == 0) return true;
  if (n_ + count > cap_) {
    size_t want = std::max(n_ + count, cap_ + cap_ / 2);
    T* np = static_cast<T*>(realloc(p_, want * sizeof(T)));  // (realloc moves pages instead of copying when it can)
    if (!np) return false;
    p_ = np;
    cap_ = want;
  }
  T* dst = p_ + n_;
  const size_t bytes = count * sizeof(T);
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t threads = bytes < (64u << 20) ? 1 : std::min<size_t>(std::min<unsigned>(hw, 16), bytes / (16u << 20));
  if (threads <= 1) {
    memcpy(dst, src, bytes);
  } else {
    std::vector<std::thread> pool;
    const size_t chunk = (count + threads - 1) / threads;
    for (size_t t = 0; t < threads; ++t) {
      const size_t a = t * chunk, b = std::min(count, a + chunk);
      if (b > a) pool.emplace_back([=] { memcpy(dst + a, src + a, (b - a) * sizeof(T)); });
    }
    for (auto& th : pool) th.join();
  }
  n_ += count;
  return true;
}
template class HostSlab<float>;
template class HostSlab<uint8_t>;

cudaError_t DevBuf::ensure(size_t bytes, bool zero_new, cudaStream_t s) {
  if (bytes <= cap) return cudaSuccess;
  if (borrowed) return cudaErrorInvalidValue;  // a borrowed range cannot grow
  size_t want = round_up(bytes, 256);
  if (p) {
    // a buffer that grows once tends to grow again (batches of rising size): 1.5x steps, not one realloc per call
    want = std::max(want, round_up(cap + cap / 2, 256));
    cudaError_t e = cudaFree(p);
    p = nullptr;
    cap = 0;
    if (e != cudaSuccess) return e;
  }
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    p = nullptr;
    return e;
  }
  cap = want;
  if (zero_new) return cudaMemsetAsync(p, 0, want, s);
  return cudaSuccess;
}
// grow without losing the contents (append-only uploads): new allocation, device copy, old one freed
cudaError_t DevBuf::ensure_keep(size_t bytes, cudaStream_t s) {
  if (bytes <= cap) return cudaSuccess;
  if (borrowed) return cudaErrorInvalidValue;
  if (!p) return ensure(bytes);
  const size_t want = std::max(round_up(bytes, 256), round_up(cap + cap / 2, 256));
  void* np = nullptr;
  cudaError_t e = cudaMalloc(&np, want);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyAsync(np, p, cap, cudaMemcpyDeviceToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    cudaFree(np);
    return e;
  }
  cudaFree(p);
  p = np;
  cap = want;
  return cudaSuccess;
}
void DevBuf::release() {
  if (p && !borrowed) cudaFree(p);
  p = nullptr;
  cap = 0;
  borrowed = false;
}
void DevBuf::borrow(void* ptr, size_t bytes) {
  release();
  p = ptr;
  cap = bytes;
  borrowed = true;
}
cudaError_t PinBuf::ensure(size_t bytes) {
  if (bytes <= cap) return cudaSuccess;
  size_t want = round_up(bytes, 4096);
  if (p) {
    want = std::max(want, round_up(cap + cap / 2, 4096));
    cudaFreeHost(p);
  }
  p = nullptr;
  cap = 0;
  cudaError_t e = cudaMallocHost(&p, want);
  if (e != cudaSuccess) {
    p = nullptr;
    return e;
  }
  cap = want;
  return cudaSuccess;
}
void PinBuf::release() {
  if (p) cudaFreeHost(p);
  p = nullptr;
  cap = 0;
}

Engine::Engine(Space space, Method method, bool is_u8, int device)
    : space_(space), method_(method), is_u8_(is_u8), device_(device) {
  force_exact_ = nb200_option("force_exact", 0) != 0;  // A/B switch: CUDA-core exact scan only
  u8_imma_ = is_u8 && method == METHOD_SEQ && !force_exact_ && nb200_option("u8_imma", 1) != 0;
  if (const char* e = nb200_env("NB200_TC_MARGIN")) tc_margin_ = std::max(1, atoi(e));
}

// Device memory back to the driver; the next prepare() uploads again.  (A group of hnsw replicas uses it on the handle's
// own engine once the graph is built: that engine stays the host store, its device copy would only double device 0's.)
void Engine::release_device() {
  if (stream_ || d_db_.p) {
    cudaSetDevice(device_);
    if (stream_) cudaStreamSynchronize(stream_);
    absorb_async_counts(false);  // (counts of device-resident batches still in the pinned ring)
  }
  for (DevBuf* b : {&d_db_, &d_aux_, &d_ids_, &d_links0_, &d_links0_cnt_, &d_upper_, &d_upper_off_, &d_visited_,
                    &d_epoch_, &d_counters_, &d_q_, &d_qaux_, &d_partial_, &d_keys_, &d_out_ids_, &d_out_dists_,
                    &d_out_counts_, &d_bias_, &d_db_unit_, &d_flags_, &d_qa_, &d_cand_, &d_cand_cnt_, &d_cand_thr_,
                    &d_tc_keys_, &d_cert_, &d_plan_, &d_gthr_, &d_u8tmp_, &d_range_, &d_fb_idx_, &d_fb_q_, &d_fb_keys_, &d_nblock_, &d_ones_,
                    &d_db_split_, &d_q_split_, &d_sp_idx_, &d_sp_q_, &d_sp_keys_})
    b->release();
  d_fb_cnt_.release();
  d_digits_.release();
  d_glists_.release();
  for (DevBuf* b : {&d_rq_, &d_rq_out_, &d_rcand_, &d_rcnt_, &d_rcut_, &d_rthr_, &d_rplan_}) b->release();
  upload_valid_ = false;
  n_up_ = 0;
  n_dev_ = 0;
  d_q_dim_ = 0;
  data_dirty_ = true;
  if (!graph_.empty()) graph_dirty_ = true;
  for (auto& f : fb_pending_) f = false;
  stats_.device_bytes = 0;
}

Engine::~Engine() {
  if (xch_) xch_destroy(xch_);
  xch_ = nullptr;
  release_device();
  for (PinBuf* b : {&h_out_ids_, &h_out_dists_, &h_out_counts_, &h_q_, &h_cert_, &h_fb_cnt_}) b->release();
  for (auto& e : fb_ev_)
    if (e) cudaEventDestroy(e);
  for (auto& e : ev_)
    if (e) cudaEventDestroy(e);
  for (auto& pr : scan_ev_)
    for (auto& e : pr)
      if (e) cudaEventDestroy(e);
  for (auto& e : copy_ev_)
    if (e) cudaEventDestroy(e);
  if (copy_stream_) cudaStreamDestroy(copy_stream_);
  h_stage_.release();
  if (stage_ready_) cudaEventDestroy(stage_ready_);
  for (int t = 0; t < kStageThreads; ++t) {
    for (auto& e : stage_ev_[t])
      if (e) cudaEventDestroy(e);
    if (stage_stream_[t]) cudaStreamDestroy(stage_stream_[t]);
  }
  if (stream_) cudaStreamDestroy(stream_);
}

Status Engine::check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return Status::OK();
  std::string m = std::string("CUDA error in ") + what + ": " + cudaGetErrorString(e);
  cudaGetLastError();
  return Status::Err(e == cudaErrorMemoryAllocation ? kErrOOM : kErrQuery, m);
}

// ------------------------------------------------------------------------------------ ingest
Status Engine::add_rows(const void* rows, size_t count, size_t elem_count, const int32_t* ids) {
  if (!rows || count == 0 || elem_count == 0) return Status::Err(kErrInvalid, "empty batch");
  if (borrowed_rows_) return Status::Err(kErrInvalid, "a shard that borrows its rows cannot grow");
  if (is_u8_ && elem_count != 128)  // space_l2sqr_sift.cc:137 CHECK (SIFT_DIM)
    return Status::Err(13, "SIFT vectors must have 128 elements");
  if (dim_ == 0) dim_ = (int)elem_count;
  if ((size_t)dim_ != elem_count)
    return Status::Err(kErrInvalid, "vector length " + std::to_string(elem_count) + " != index dimension " +
                                        std::to_string(dim_));
  if (n_ + count > 0xFFFFFFF0ull) return Status::Err(kErrTooLarge, "more than 2^32 rows in one shard");
  if (is_u8_) {
    const uint8_t* src = static_cast<const uint8_t*>(rows);
    if (!h_u8_.append(src, count * elem_count)) return Status::Err(kErrOOM, "out of host memory");
  } else {
    const float* src = static_cast<const float*>(rows);
    if (!h_f32_.append(src, count * elem_count)) return Status::Err(kErrOOM, "out of host memory");
  }
  if (ids) h_ids_.insert(h_ids_.end(), ids, ids + count);
  else
    for (size_t i = 0; i < count; ++i) h_ids_.push_back((int32_t)i);  // nmslib_c.cpp:768
  n_ += count;
  ++data_gen_;
  data_dirty_ = true;
  rows_normalized_ = false;
  h_hnsw_rows_.clear();
  if (method_ == METHOD_HNSW && !graph_.empty()) {
    graph_ = HnswGraph();  // the graph no longer describes the data
    graph_dirty_ = true;
  }
  return Status::OK();
}

Status Engine::borrow_host_rows(const void* rows, const int32_t* ids, size_t count, size_t elem_count) {
  if (!rows || !ids || count == 0 || elem_count == 0) return Status::Err(kErrInvalid, "empty shard");
  if (method_ != METHOD_SEQ) return Status::Err(kErrIncompat, "only seq_search shards borrow their rows");
  if (n_ != 0) return Status::Err(kErrInvalid, "borrow_host_rows on a non-empty engine");
  dim_ = (int)elem_count;
  n_ = count;
  borrowed_rows_ = rows;
  borrowed_ids_ = ids;
  data_dirty_ = true;
  ++data_gen_;
  return Status::OK();
}

Status Engine::add_row_ptrs(const void* const* ptrs, size_t count, size_t elem_count, const int32_t* ids) {
  if (!ptrs || count == 0) return Status::Err(kErrInvalid, "empty pointer batch");
  for (size_t i = 0; i < count; ++i) {
    if (!ptrs[i]) return Status::Err(1, "null data pointer in batch");
    int32_t id = ids ? ids[i] : (int32_t)i;
    Status s = add_rows(ptrs[i], 1, elem_count, &id);
    if (!s.ok()) return s;
  }
  return Status::OK();
}

void Engine::reset() {
  h_f32_.clear();
  h_u8_.clear();
  h_ids_.clear();
  borrowed_rows_ = nullptr;
  borrowed_ids_ = nullptr;
  replica_rows_ = false;
  n_ = 0;
  dim_ = 0;
  built_ = false;
  graph_ = HnswGraph();
  data_dirty_ = graph_dirty_ = true;
  n_dev_ = 0;
  rows_normalized_ = false;
  h_hnsw_rows_.clear();
  d_q_dim_ = -1;  // the staged-query buffer is re-zeroed before its next use (stale padding columns)
  upload_valid_ = false;
  n_up_ = 0;
  ++data_gen_;
}

float Engine::host_distance(size_t a, size_t b) const {
  if (is_u8_) {
    const uint8_t *x = row_u8(a), *y = row_u8(b);
    int32_t nx = 0, ny = 0, dot = 0;
    for (int i = 0; i < dim_; ++i) {
      nx += (int)x[i] * x[i];
      ny += (int)y[i] * y[i];
      dot += (int)x[i] * y[i];
    }
    return (float)(nx + ny - 2 * dot);
  }
  const float *x = row_f32(a), *y = row_f32(b);
  float s = 0.f, n1 = 0.f, n2 = 0.f;
  if (space_ == SPACE_L1 || space_ == SPACE_LINF) {
    for (int i = 0; i < dim_; ++i) {
      const float d = std::fabs(x[i] - y[i]);
      s = space_ == SPACE_L1 ? s + d : std::max(s, d);
    }
    return s;
  }
  for (int i = 0; i < dim_; ++i) {
    if (space_ == SPACE_L2 || space_ == SPACE_L2SQR) {
      float d = x[i] - y[i];
      s += d * d;
    } else {
      s += x[i] * y[i];
      n1 += x[i] * x[i];
      n2 += y[i] * y[i];
    }
  }
  switch (space_) {
    case SPACE_L2: return std::sqrt(s);
    case SPACE_L2SQR: return s;
    case SPACE_NEGDOT: return -s;
    default: {
      const float eps = 2.0f * 1.17549435e-38f;
      float nsp = (n1 < eps || n2 < eps) ? 0.f : std::max(-1.f, std::min(1.f, s / std::sqrt(n1) / std::sqrt(n2)));
      if (space_ == SPACE_ANGULAR) return std::acos(nsp);
      return std::max(0.f, 1.f - nsp);
    }
  }
}

// ------------------------------------------------------------------------------------ state
void Engine::mark_built(const std::vector<std::string>& index_params) {
  index_params_ = index_params;
  built_ = true;
}

// Hnsw::SetQueryTimeParams (hnsw.cc:474-507): ef / efSearch are synonyms (default 20 in the
// reference, 200 through its C ABI), algoType in {old, v1merge, hybrid}, searchMethod ignored;
// anything else is an error.  SeqSearch::SetQueryTimeParams is a no-op (seqsearch.h:44).
Status Engine::set_query_params(const std::vector<std::string>& params) {
  if (method_ != METHOD_HNSW) return Status::OK();
  bool has_ef = false, has_efs = false;
  size_t ef = 20;  // the reference's own default once the user sets query-time params
  for (const std::string& p : params) {
    size_t eq = p.find('=');
    if (eq == std::string::npos) return Status::Err(kErrInvalid, "malformed parameter '" + p + "'");
    std::string name = p.substr(0, eq), val = p.substr(eq + 1);
    if (name == "ef" || name == "efSearch") {
      (name == "ef" ? has_ef : has_efs) = true;
      std::stringstream ss(val);
      double v = 0;
      if (!(ss >> v) || v < 1) return Status::Err(kErrInvalid, "bad value for " + name);
      ef = (size_t)v;
    } else if (name == "algoType") {
      std::string low = val;
      std::transform(low.begin(), low.end(), low.begin(), ::tolower);
      if (low != "old" && low != "v1merge" && low != "hybrid")
        return Status::Err(kErrInvalid, "algoType should be one of: old, v1merge, hybrid");
    } else if (name == "searchMethod") {
    } else {
      return Status::Err(kErrInvalid, "unknown query-time parameter '" + name + "'");
    }
  }
  if (has_ef && has_efs) return Status::Err(kErrInvalid, "ef and efSearch are synonyms: specify only one");
  if (ef > (size_t)hnsw_max_ef())
    return Status::Err(kErrTooLarge, "efSearch above " + std::to_string(hnsw_max_ef()) + " is not supported");
  ef_ = ef;
  ef_user_set_ = true;
  return Status::OK();
}

Status Engine::adopt_graph(HnswGraph&& g) {
  if (method_ != METHOD_HNSW) return Status::Err(kErrIncompat, "graph import needs method hnsw");
  if (g.dim == 0 && g.vectors.empty()) {
    // The reference's REGULAR index (SaveRegularIndexBin, hnsw.cc:810-842: what Hnsw<int>, i.e. l2sqr_sift + hnsw,
    // saves): links only.  The data set is this index's own; the search is baseSearchAlgorithmV1Merge / Old
    // (hnsw.cc:1076-1300) -- the same beam rule as the flat index over the space's own distance.
    if (g.total != n_) return Status::Err(kErrIncompat, "regular HNSW index: " + std::to_string(g.total) + " nodes but " +
                                                            std::to_string(n_) + " data points (add the data first)");
    g.dim = dim_;
    g.dist_func = space_ == SPACE_COSINE ? 3 : space_ == SPACE_NEGDOT ? 4 : (dim_ % 16 == 0 ? 1 : 2);
    g.ext_ids = h_ids_;
    graph_ = std::move(g);
    graph_dirty_ = true;
    built_ = true;
    ++data_gen_;  // (replicas of this index, shard_group.cu, are cut again)
    return Status::OK();
  }
  if (is_u8_) return Status::Err(kErrIncompat, "the optimized HNSW index holds float vectors only");
  const int want = (space_ == SPACE_COSINE) ? 3 : (space_ == SPACE_NEGDOT) ? 4 : 0;
  const bool l2 = (space_ == SPACE_L2 || space_ == SPACE_L2SQR) && (g.dist_func == 1 || g.dist_func == 2);
  if (!l2 && g.dist_func != want)
    return Status::Err(kErrIncompat, "HNSW file distance type " + std::to_string(g.dist_func) +
                                         " does not match the index space");
  graph_ = std::move(g);
  // the file carries the (for cosine: normalised) vectors and the external ids
  dim_ = graph_.dim;
  n_ = graph_.total;
  if (!h_f32_.assign(graph_.vectors.data(), graph_.vectors.size())) return Status::Err(kErrOOM, "out of host memory");
  h_ids_ = graph_.ext_ids;
  graph_.vectors.clear();
  graph_.vectors.shrink_to_fit();
  upload_valid_ = false;
  rows_normalized_ = true;  // the file stores cosine rows already normalised
  h_hnsw_rows_.clear();
  data_dirty_ = graph_dirty_ = true;
  built_ = true;
  ++data_gen_;
  return Status::OK();
}

Status Engine::adopt_replica(const HnswGraph& g, const void* search_rows, const int32_t* ids, int dim) {
  if (method_ != METHOD_HNSW) return Status::Err(kErrIncompat, "graph replica needs method hnsw");
  if (g.empty() || !search_rows || !ids) return Status::Err(kErrInvalid, "empty graph replica");
  graph_ = g;
  graph_.vectors.clear();
  dim_ = dim;
  n_ = g.total;
  borrowed_rows_ = search_rows;
  borrowed_ids_ = ids;
  replica_rows_ = true;
  rows_normalized_ = true;
  upload_valid_ = false;
  data_dirty_ = graph_dirty_ = true;
  built_ = true;
  return Status::OK();
}

Status Engine::import_graph(const std::string& path) {
  HnswGraph g;
  Status s = read_hnsw_file(path, &g);
  if (!s.ok()) return s;
  return adopt_graph(std::move(g));
}

void Engine::scan_begin(cudaStream_t s) {
  scan_cur_ = scan_head_;
  scan_head_ = (scan_head_ + 1) % kScanRing;
  if (!scan_ev_[scan_cur_][0]) {
    cudaEventCreate(&scan_ev_[scan_cur_][0]);
    cudaEventCreate(&scan_ev_[scan_cur_][1]);
  }
  scan_pending_[scan_cur_] = false;
  cudaEventRecord(scan_ev_[scan_cur_][0], s);
}
void Engine::scan_end(cudaStream_t s) {
  cudaEventRecord(scan_ev_[scan_cur_][1], s);
  scan_pending_[scan_cur_] = true;
}

Stats Engine::stats() {
  absorb_async_counts(false);
  for (int i = 0; i < kScanRing; ++i) {
    if (!scan_pending_[i] || cudaEventQuery(scan_ev_[i][1]) != cudaSuccess) continue;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, scan_ev_[i][0], scan_ev_[i][1]) == cudaSuccess) {
      stats_.last_scan_ms = ms;
      stats_.scan_ms_sum += ms;
      ++stats_.scan_count;
    }
    scan_pending_[i] = false;
  }
  if (method_ == METHOD_HNSW && d_counters_.p) {  // cumulative device counters (also after device-resident calls)
    unsigned long long c[2] = {0, 0};
    if (cudaSetDevice(device_) == cudaSuccess && cudaMemcpy(c, d_counters_.p, 16, cudaMemcpyDeviceToHost) == cudaSuccess) {
      stats_.distance_evals = c[0];
      stats_.hnsw_expansions = c[1];
    }
  }
  cudaGetLastError();
  return stats_;
}

// Float rows as the HNSW builders and the float kernels want them: unit-normalised for cosine (the reference normalises
// its flat index once at build time, hnsw.cc:441-446); uint8 widened to float for the host build only (the search
// reads the byte rows).
const float* Engine::hnsw_host_rows() {
  if (replica_rows_) return static_cast<const float*>(borrowed_rows_);  // search-ready rows of the engine replicated
  if (!is_u8_ && (space_ != SPACE_COSINE || rows_normalized_)) return base_f32();
  if (h_hnsw_rows_.size() == n_ * (size_t)dim_) return h_hnsw_rows_.data();
  h_hnsw_rows_.resize(n_ * (size_t)dim_);
  for (size_t i = 0; i < n_; ++i) {
    float* dst = &h_hnsw_rows_[i * (size_t)dim_];
    if (is_u8_) {
      const uint8_t* r = row_u8(i);
      for (int j = 0; j < dim_; ++j) dst[j] = (float)r[j];
    } else {
      const float* r = row_f32(i);
      float sum = 0.f;
      for (int j = 0; j < dim_; ++j) sum += r[j] * r[j];
      const float sc = sum != 0.f ? 1.f / std::sqrt(sum) : 1.f;  // NormalizeVect, hnsw.h:486-497
      for (int j = 0; j < dim_; ++j) dst[j] = r[j] * sc;
    }
  }
  return h_hnsw_rows_.data();
}

int Engine::finalize_kind() const {
  if (method_ == METHOD_HNSW) return FIN_FLOAT;  // squared / cosine / negdot / (uint8: exact integers as fp32)
  if (is_u8_) return FIN_INT;  // every uint8 path ends in i32_ordered(int distance) keys (re-rank, dp4a scan)
  // l2 + seq_search reports the root; l2 + hnsw reports the squared distance (SURVEY 0.4)
  if (space_ == SPACE_L2 && method_ == METHOD_SEQ) return FIN_SQRT;
  return FIN_FLOAT;
}

// ------------------------------------------------------------------------------------ upload
Status Engine::prepare() {
  if (!device_available()) return Status::Err(kErrQuery, "no CUDA device available (there is no CPU fallback)");
  Status s = check_cuda(cudaSetDevice(device_), "cudaSetDevice");
  if (!s.ok()) return s;
  if (!stream_) {
    s = check_cuda(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking), "cudaStreamCreate");
    if (!s.ok()) return s;
    for (auto& e : ev_) {
      s = check_cuda(cudaEventCreate(&e), "cudaEventCreate");
      if (!s.ok()) return s;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device_) == cudaSuccess) sm_count_ = prop.multiProcessorCount;
  }
  if (data_dirty_) {
    s = upload_data();
    if (!s.ok()) return s;
  }
  if (method_ == METHOD_HNSW && graph_dirty_) {
    s = upload_graph();
    if (!s.ok()) return s;
  }
  return Status::OK();
}

Status Engine::upload_data() {
  if (n_ == 0) {
    n_dev_ = 0;
    data_dirty_ = false;
    return Status::OK();
  }
  const int stage = scan_exact_stage_words();
  const int bn = scan_exact_block_points();
  // HBM layout: row-major [n_pad][row_words] 32-bit words, rows zero padded to a whole
  // pipeline stage (64 B) and the row count to a whole tile, so no kernel needs edge code.
  // float rows are padded to 128 bytes (one TMA / UMMA swizzle row of the tensor-core scan)
  const bool dev_u8 = dev_u8_rows();
  if (!rows_borrowed_)
    row_words_ = (int)round_up(dev_u8 ? (size_t)dim_ / 4 : (size_t)dim_, dev_u8 ? stage : tc_kblock_words());
  if (dev_u8 && dim_ % 4) return Status::Err(kErrInvalid, "uint8 dimension must be a multiple of 4");
  const size_t n_pad = round_up(n_, bn);
  const size_t row_bytes = (size_t)row_words_ * 4;
  // Append-only upload (SURVEY 8f N2): rows [0, n_up_) of a seq_search index are already in HBM in this layout, only
  // the rows added since travel (the reference copies every point once at add time, nmslib_c.cpp:755-871; round 1
  // re-uploaded the whole database after any add).  Buffers grow keeping their contents.
  const bool append = upload_valid_ && method_ == METHOD_SEQ && !rows_borrowed_ && n_up_ > 0 && n_ > n_up_ &&
                      up_row_words_ == row_words_;
  const size_t r0 = append ? n_up_ : 0;
  auto grow = [&](DevBuf& b, size_t bytes) { return append ? b.ensure_keep(bytes, stream_) : b.ensure(bytes); };
  Status s = check_cuda(grow(d_db_, n_pad * row_bytes), "cudaMalloc(data)");
  if (!s.ok()) return s;
  if (!rows_borrowed_)
    s = check_cuda(cudaMemsetAsync(d_db_.as<char>() + r0 * row_bytes, 0, (n_pad - r0) * row_bytes, stream_), "memset(data)");
  if (!s.ok()) return s;
  const size_t src_row = dev_u8 ? (size_t)dim_ : (size_t)dim_ * 4;
  const void* src = dev_u8 ? (const void*)base_u8() : (const void*)base_f32();
  if (method_ == METHOD_HNSW && !is_u8_) src = hnsw_host_rows();  // cosine: unit-normalised (hnsw.cc:441-446)
  if (rows_borrowed_) {
    // (adopt_device_rows: the padded rows are already in HBM; ids = positions)
  } else if (u8_widened()) {  // bytes up in 1 M-row chunks, widened to fp32 rows on the device
    const size_t chunk = 1u << 20;
    if (!(s = check_cuda(d_u8tmp_.ensure(std::min(n_, chunk) * (size_t)dim_), "cudaMalloc(u8 staging)")).ok()) return s;
    for (size_t c0 = r0; c0 < n_; c0 += chunk) {
      const size_t cnt = std::min(chunk, n_ - c0);
      s = check_cuda(cudaMemcpyAsync(d_u8tmp_.p, base_u8() + c0 * dim_, cnt * dim_, cudaMemcpyHostToDevice, stream_),
                     "H2D(u8 data)");
      if (!s.ok()) return s;
      s = check_cuda(launch_widen_u8(d_u8tmp_.as<uint8_t>(), cnt, dim_, row_words_,
                                     d_db_.as<float>() + c0 * (size_t)row_words_, stream_),
                     "widen_u8");
      if (!s.ok()) return s;
      ++stats_.kernel_launches;
    }
  } else {
    s = upload_rows(d_db_.as<char>() + r0 * row_bytes, row_bytes, static_cast<const char*>(src) + r0 * src_row, src_row, n_ - r0);
    if (!s.ok()) return s;
  }
  if (!rows_borrowed_) {
    s = check_cuda(grow(d_ids_, n_ * 4), "cudaMalloc(ids)");
    if (!s.ok()) return s;
    s = check_cuda(cudaMemcpyAsync(d_ids_.as<int32_t>() + r0, base_ids() + r0, (n_ - r0) * 4, cudaMemcpyHostToDevice, stream_),
                   "H2D(ids)");
    if (!s.ok()) return s;
  }
  stats_.uploaded_rows += n_ - r0;
  const bool cos_family = space_ == SPACE_COSINE || space_ == SPACE_ANGULAR;
  if (method_ == METHOD_SEQ && (cos_family || dev_u8)) {
    s = check_cuda(grow(d_aux_, n_pad * 4), "cudaMalloc(aux)");
    if (!s.ok()) return s;
    s = check_cuda(launch_row_aux(dev_u8, d_db_.as<char>() + r0 * row_bytes, (int)(n_ - r0), row_words_,
                                  d_aux_.as<char>() + r0 * 4, stream_), "row_aux");
    if (!s.ok()) return s;
    ++stats_.kernel_launches;
  }
  if (dev_u8 && u8_imma_) {
    // integer tensor pipe: M = ceil(max |x|^2 / 2) and the rows' norm digits (scan_tc.cu); rows whose norms do not fit
    // the digit block send the whole index back to the widened TF32 path
    if (!(s = check_cuda(d_flags_.ensure(16), "cudaMalloc(flags)")).ok()) return s;
    if (!(s = check_cuda(launch_u8_max_norm(d_aux_.as<int>(), (int)n_, d_flags_.as<int>() + 3, stream_), "u8_max_norm")).ok()) return s;
    int max_norm2 = 0;
    if (!(s = check_cuda(cudaMemcpyAsync(&max_norm2, d_flags_.as<int>() + 3, 4, cudaMemcpyDeviceToHost, stream_), "D2H(max norm)")).ok()) return s;
    if (!(s = check_cuda(cudaStreamSynchronize(stream_), "upload sync")).ok()) return s;
    stats_.kernel_launches += 1;
    if (max_norm2 > u8_imma_max_norm2()) {
      u8_imma_ = false;
      upload_valid_ = false;  // (another row layout: everything travels again)
      return upload_data();
    }
    u8_m_half_ = (max_norm2 + 1) / 2;
    if (!(s = check_cuda(d_digits_.ensure(n_pad * 32), "cudaMalloc(norm digits)")).ok()) return s;
    s = check_cuda(launch_u8_norm_digits(d_aux_.as<int>(), (int)n_, (int)n_pad, u8_m_half_, d_digits_.as<uint8_t>(), stream_), "u8_norm_digits");
    if (!s.ok()) return s;
    stats_.kernel_launches += 1;
  }
  x_max_ = 0.f;
  tc_split_ = false;
  d_db_split_.release();
  if (!dev_u8 && method_ == METHOD_SEQ && space_ != SPACE_L1 && space_ != SPACE_LINF) {
    // operands of the tensor-core scan: bias (|x|^2 or 0, +inf on padding rows), the unit-norm copy
    // for cosine, max operand-row norm and the "is TF32-exact" flag (both feed the certificate)
    const int mode = cos_family ? SCAN_COSINE : space_ == SPACE_NEGDOT ? SCAN_NEGDOT : SCAN_L2;
    if (!(s = check_cuda(grow(d_bias_, n_pad * 4), "cudaMalloc(bias)")).ok()) return s;
    if (!(s = check_cuda(d_flags_.ensure(16), "cudaMalloc(flags)")).ok()) return s;
    // (append: the max norm and the "not TF32-exact" flag of the rows already there keep accumulating)
    if (!append && !(s = check_cuda(cudaMemsetAsync(d_flags_.p, 0, 16, stream_), "memset(flags)")).ok()) return s;
    float* unit = nullptr;
    if (mode == SCAN_COSINE) {
      if (!(s = check_cuda(grow(d_db_unit_, n_pad * row_bytes), "cudaMalloc(unit rows)")).ok()) return s;
      if (!(s = check_cuda(cudaMemsetAsync(d_db_unit_.as<char>() + r0 * row_bytes, 0, (n_pad - r0) * row_bytes, stream_),
                           "memset(unit)")).ok()) return s;
      unit = d_db_unit_.as<float>() + r0 * (size_t)row_words_;
    }
    // flags layout: [0] database inexact, [1] query batch inexact, [2] max-norm bits
    float* nblock = nullptr;
    if (mode == SCAN_L2) {  // |x|^2 as an extra K=8 MMA step: [n_pad][32] TF32 pieces + a constant tile of ones
      if (!(s = check_cuda(grow(d_nblock_, n_pad * (size_t)tc_kblock_words() * 4), "cudaMalloc(nblock)")).ok()) return s;
      if (!(s = check_cuda(d_ones_.ensure((size_t)128 * tc_kblock_words() * 4), "cudaMalloc(ones)")).ok()) return s;
      nblock = d_nblock_.as<float>() + r0 * (size_t)tc_kblock_words();
    }
    s = check_cuda(launch_tc_prep_db(d_db_.as<float>() + r0 * (size_t)row_words_, (int)(n_ - r0), (int)(n_pad - r0), row_words_,
                                     mode, d_bias_.as<float>() + r0,
                                     mode == SCAN_COSINE ? d_aux_.as<float>() + r0 : nullptr, unit, nblock,
                                     nblock ? d_ones_.as<float>() : nullptr, d_flags_.as<unsigned>() + 2,
                                     d_flags_.as<int>(), stream_),
                   "tc_prep_db");
    if (!s.ok()) return s;
    ++stats_.kernel_launches;
    unsigned bits = 0;
    int inexact = 0;
    s = check_cuda(cudaMemcpyAsync(&bits, d_flags_.as<unsigned>() + 2, 4, cudaMemcpyDeviceToHost, stream_), "D2H(xmax)");
    if (!s.ok()) return s;
    s = check_cuda(cudaMemcpyAsync(&inexact, d_flags_.as<int>(), 4, cudaMemcpyDeviceToHost, stream_), "D2H(exact flag)");
    if (!s.ok()) return s;
    s = check_cuda(cudaStreamSynchronize(stream_), "upload sync");
    if (!s.ok()) return s;
    memcpy(&x_max_, &bits, 4);
    db_inexact_ = inexact != 0;
  }
  s = check_cuda(cudaStreamSynchronize(stream_), "upload sync");
  if (!s.ok()) return s;
  n_dev_ = n_;
  n_up_ = n_;
  up_row_words_ = row_words_;
  upload_valid_ = !rows_borrowed_;
  data_dirty_ = false;
  stats_.device_bytes = d_db_.cap + d_ids_.cap + d_aux_.cap + d_bias_.cap + d_db_unit_.cap + d_nblock_.cap;
  return Status::OK();
}

// Host rows -> padded device rows.  The host slab is pageable (it is the index's own copy of the caller's data,
// nmslib_c.cpp:755-871 copies every point as well): a plain cudaMemcpy from it goes through the driver's staging buffer
// on the calling thread, 7-10 GB/s measured (tools/ingest_split.py).  From 256 MB up the rows travel through pinned
// staging buffers instead: kStageThreads host threads each copy 4 MB chunks into their own pair of pinned buffers and
// queue the H2D on their own stream, so the host copies of some chunks overlap the bus transfers of others.
Status Engine::upload_rows(char* dst, size_t dst_pitch, const char* src, size_t src_row, size_t rows) {
  const size_t bytes = rows * src_row;
  if (bytes < (256u << 20) || src_row > kStageBytes)
    return check_cuda(cudaMemcpy2DAsync(dst, dst_pitch, src, src_row, src_row, rows, cudaMemcpyHostToDevice, stream_), "H2D(data)");
  Status s = check_cuda(h_stage_.ensure((size_t)kStageThreads * 2 * kStageBytes), "cudaMallocHost(staging)");
  if (!s.ok()) return s;
  if (!stage_ready_) {
    if (!(s = check_cuda(cudaEventCreateWithFlags(&stage_ready_, cudaEventDisableTiming), "cudaEventCreate")).ok()) return s;
    for (int t = 0; t < kStageThreads; ++t) {
      if (!(s = check_cuda(cudaStreamCreateWithFlags(&stage_stream_[t], cudaStreamNonBlocking), "cudaStreamCreate")).ok()) return s;
      for (auto& e : stage_ev_[t])
        if (!(s = check_cuda(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate")).ok()) return s;
    }
  }
  // the copy streams start behind what stream_ has queued for the destination (the padding memset)
  if (!(s = check_cuda(cudaEventRecord(stage_ready_, stream_), "cudaEventRecord")).ok()) return s;
  const size_t chunk_rows = std::max<size_t>(1, kStageBytes / src_row);
  const size_t n_chunks = (rows + chunk_rows - 1) / chunk_rows;
  std::atomic<size_t> next{0};
  std::atomic<int> err{(int)cudaSuccess};
  std::vector<std::thread> pool;
  for (int t = 0; t < kStageThreads; ++t)
    pool.emplace_back([&, t] {
      cudaError_t e = cudaSetDevice(device_);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(stage_stream_[t], stage_ready_, 0);
      for (int it = 0; e == cudaSuccess; ++it) {
        const size_t c = next.fetch_add(1);
        if (c >= n_chunks) break;
        const int b = it & 1;
        char* st = h_stage_.as<char>() + ((size_t)t * 2 + b) * kStageBytes;
        if (it >= 2) e = cudaEventSynchronize(stage_ev_[t][b]);  // the transfer that last used this buffer
        if (e != cudaSuccess) break;
        const size_t c0 = c * chunk_rows, cnt = std::min(chunk_rows, rows - c0);
        memcpy(st, src + c0 * src_row, cnt * src_row);
        e = cudaMemcpy2DAsync(dst + c0 * dst_pitch, dst_pitch, st, src_row, src_row, cnt, cudaMemcpyHostToDevice, stage_stream_[t]);
        if (e == cudaSuccess) e = cudaEventRecord(stage_ev_[t][b], stage_stream_[t]);
      }
      const cudaError_t e2 = cudaStreamSynchronize(stage_stream_[t]);
      if (e == cudaSuccess) e = e2;
      if (e != cudaSuccess) err.store((int)e);
    });
  for (auto& th : pool) th.join();
  return check_cuda((cudaError_t)err.load(), "H2D(data, staged)");
}

// No imported graph: build one on the host cores (hnsw_build.cpp) with the index-time parameters
// recorded by nmslib_create_index (the reference drops them, SURVEY Q3).  Needs no GPU.
Status Engine::ensure_graph_host() {
  if (method_ != METHOD_HNSW || !graph_.empty()) return Status::OK();
  if (n_ == 0) return Status::Err(kErrBuild, "hnsw index holds no data");
  const int dist_func = space_ == SPACE_COSINE ? 3 : space_ == SPACE_NEGDOT ? 4 : (dim_ % 16 == 0 ? 1 : 2);
  HnswGraph g;
  Status bs = build_hnsw_host(hnsw_host_rows(), n_, dim_, dist_func, h_ids_.data(), index_params_, &g);
  if (is_u8_) std::vector<float>().swap(h_hnsw_rows_);  // (widened for the build only: the search reads the bytes)
  if (!bs.ok()) return bs;
  graph_ = std::move(g);
  graph_dirty_ = true;
  return Status::OK();
}

// Graph construction on the device (hnsw_build_gpu.cu) over the rows upload_data() has just put in HBM.
Status Engine::build_graph_device() {
  HnswBuildParams bp;
  std::string err;
  if (!parse_hnsw_build_params(index_params_, &bp, &err)) return Status::Err(kErrBuild, err);
  const int dist_func = space_ == SPACE_COSINE ? 3 : space_ == SPACE_NEGDOT ? 4 : (dim_ % 16 == 0 ? 1 : 2);
  HnswGraph g;
  Status bs;
  if (is_u8_) {
    // the build scans float rows (TF32 over values 0..255 is exact): widen the byte rows into a temporary buffer
    const int f_words = (int)round_up((size_t)dim_, tc_kblock_words());
    const size_t bytes = round_up(n_, scan_exact_block_points()) * f_words * 4;
    DevBuf wide;
    bs = check_cuda(wide.ensure(bytes), "cudaMalloc(widened rows)");
    if (bs.ok()) bs = check_cuda(cudaMemsetAsync(wide.p, 0, bytes, stream_), "memset(widened rows)");
    if (bs.ok()) bs = check_cuda(launch_widen_u8(d_db_.as<uint8_t>(), n_, dim_, f_words, wide.as<float>(), stream_), "widen_u8");
    if (bs.ok()) bs = check_cuda(cudaStreamSynchronize(stream_), "widen sync");
    if (bs.ok())
      bs = build_hnsw_device(wide.as<float>(), n_, dim_, f_words, dist_func, h_ids_.data(), bp, device_, &g, &build_info_);
    wide.release();
  } else {
    bs = build_hnsw_device(d_db_.as<float>(), n_, dim_, row_words_, dist_func, h_ids_.data(), bp, device_, &g,
                           &build_info_);
  }
  if (!bs.ok()) return bs;
  graph_ = std::move(g);
  graph_dirty_ = true;
  return Status::OK();
}

Status Engine::ensure_graph() {
  if (method_ != METHOD_HNSW || !graph_.empty()) return Status::OK();
  if (device_available()) {  // prepare() uploads the rows and builds on the device when the parameters allow it
    Status s = prepare();
    if (s.ok() || !graph_.empty()) return s;
  }
  return ensure_graph_host();
}

Status Engine::adopt_device_rows(const float* d_rows, size_t n, int dim, int row_words) {
  if (method_ != METHOD_SEQ || is_u8_) return Status::Err(kErrIncompat, "adopt_device_rows: float seq_search only");
  n_ = n;
  dim_ = dim;
  row_words_ = row_words;
  rows_borrowed_ = true;
  d_db_.borrow(const_cast<float*>(d_rows), round_up(n, scan_exact_block_points()) * (size_t)row_words * 4);
  data_dirty_ = true;
  built_ = true;
  return Status::OK();
}

Status Engine::upload_graph() {
  if (graph_.empty() && n_ > 0) {
    HnswBuildParams bp;
    std::string err;
    if (!parse_hnsw_build_params(index_params_, &bp, &err)) return Status::Err(kErrBuild, err);
    const bool on_device = bp.where == 1 || (bp.where < 0 && n_ >= 16384);
    if (on_device && bp.M <= 64 && bp.maxM <= 64 && bp.maxM0 <= 64 && bp.delaunay_type != 0) {
      Status bs = build_graph_device();
      if (!bs.ok()) return bs;
    }
  }
  {
    Status bs = ensure_graph_host();
    if (!bs.ok()) return bs;
  }
  if (graph_.total != n_) return Status::Err(kErrBuild, "HNSW graph / data size mismatch");
  const HnswGraph& g = graph_;
  Status s = check_cuda(d_links0_.ensure(std::max<size_t>(g.links0.size(), 1) * 4), "cudaMalloc(links0)");
  if (!s.ok()) return s;
  s = check_cuda(d_links0_cnt_.ensure((size_t)g.total * 4), "cudaMalloc(links0_cnt)");
  if (!s.ok()) return s;
  s = check_cuda(d_upper_.ensure(std::max<size_t>(g.upper.size(), 1) * 4), "cudaMalloc(upper)");
  if (!s.ok()) return s;
  s = check_cuda(d_upper_off_.ensure((size_t)g.total * 8), "cudaMalloc(upper_off)");
  if (!s.ok()) return s;
  if (!(s = check_cuda(cudaMemcpyAsync(d_links0_.p, g.links0.data(), g.links0.size() * 4, cudaMemcpyHostToDevice, stream_),
                       "H2D(links0)")).ok()) return s;
  if (!(s = check_cuda(cudaMemcpyAsync(d_links0_cnt_.p, g.links0_cnt.data(), (size_t)g.total * 4, cudaMemcpyHostToDevice,
                                       stream_), "H2D(links0_cnt)")).ok()) return s;
  if (!g.upper.empty() &&
      !(s = check_cuda(cudaMemcpyAsync(d_upper_.p, g.upper.data(), g.upper.size() * 4, cudaMemcpyHostToDevice, stream_),
                       "H2D(upper)")).ok()) return s;
  if (!(s = check_cuda(cudaMemcpyAsync(d_upper_off_.p, g.upper_off.data(), (size_t)g.total * 8, cudaMemcpyHostToDevice,
                                       stream_), "H2D(upper_off)")).ok()) return s;
  // visited epoch arrays: one per resident warp slot (VisitedListPool, hnsw.h:598-639)
  hnsw_slots_ = sm_count_ * 32;  // upper bound of warps per SM in flight (the launch uses one resident wave)
  if (const char* e = nb200_env("NB200_HNSW_SLOTS")) hnsw_slots_ = sm_count_ * std::max(4, std::min(64, atoi(e)));
  const size_t vstride = round_up((size_t)g.total, 16);
  s = check_cuda(d_visited_.ensure(vstride * hnsw_slots_), "cudaMalloc(visited)");
  if (!s.ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_visited_.p, 0, vstride * hnsw_slots_, stream_), "memset(visited)")).ok()) return s;
  s = check_cuda(d_epoch_.ensure((size_t)hnsw_slots_ * 4), "cudaMalloc(epoch)");
  if (!s.ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_epoch_.p, 0, (size_t)hnsw_slots_ * 4, stream_), "memset(epoch)")).ok()) return s;
  s = check_cuda(d_counters_.ensure(32), "cudaMalloc(counters)");
  if (!s.ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_counters_.p, 0, 32, stream_), "memset(counters)")).ok()) return s;
  s = check_cuda(cudaStreamSynchronize(stream_), "graph upload sync");
  if (!s.ok()) return s;
  graph_dirty_ = false;
  stats_.device_bytes = d_db_.cap + d_ids_.cap + d_aux_.cap + d_links0_.cap + d_links0_cnt_.cap + d_upper_.cap +
                        d_upper_off_.cap + d_visited_.cap;
  return Status::OK();
}

// ------------------------------------------------------------------------------------ query
Status Engine::stage_queries_device(const void* src, bool src_on_device, size_t nq, size_t elem_count,
                                    cudaStream_t stream, size_t src_pitch) {
  const size_t bq = std::max(scan_exact_block_queries(), tc_block_queries());
  const size_t q_pad = round_up(nq, bq);
  const size_t row_bytes = (size_t)row_words_ * 4;
  const size_t old_cap = d_q_.cap;
  Status s = check_cuda(d_q_.ensure(q_pad * row_bytes), "cudaMalloc(queries)");
  if (!s.ok()) return s;
  if (d_q_.cap != old_cap || d_q_dim_ != dim_) {
    // new buffer, or the index was reset and re-filled with rows of another length that pad to the same row_words:
    // zero it so that the padding columns [dim, row_words) hold no values of earlier queries
    s = check_cuda(cudaMemsetAsync(d_q_.p, 0, d_q_.cap, stream), "memset(queries)");
    if (!s.ok()) return s;
    d_q_dim_ = dim_;
  }
  if (u8_widened()) {  // uint8 queries: bytes to a staging buffer, widened into the padded fp32 rows
    s = check_cuda(d_u8tmp_.ensure(std::max<size_t>(nq * elem_count, d_u8tmp_.cap)), "cudaMalloc(u8 staging)");
    if (!s.ok()) return s;
    s = check_cuda(cudaMemcpyAsync(d_u8tmp_.p, src, nq * elem_count,
                                   src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, stream),
                   "copy(u8 queries)");
    if (!s.ok()) return s;
    ++stats_.kernel_launches;
    return check_cuda(launch_widen_u8(d_u8tmp_.as<uint8_t>(), nq, (int)elem_count, row_words_, d_q_.as<float>(), stream),
                      "widen_u8(queries)");
  }
  const size_t src_row = dev_u8_rows() ? elem_count : elem_count * 4;
  return check_cuda(cudaMemcpy2DAsync(d_q_.p, row_bytes, src, src_pitch ? src_pitch : src_row, src_row, nq,
                                      src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, stream),
                    "copy(queries)");
}

Status Engine::run(const void* dq, size_t nq, size_t k, int32_t* d_ids, float* d_dists, uint64_t* d_keys,
                   int32_t* d_counts, cudaStream_t stream, bool async) {
  Status s;
  if (method_ == METHOD_HNSW) {
    HnswDeviceGraph g;
    g.vectors = d_db_.p;
    g.links0 = d_links0_.as<int32_t>();
    g.links0_cnt = d_links0_cnt_.as<int32_t>();
    g.upper = d_upper_.as<int32_t>();
    g.upper_off = d_upper_off_.as<int64_t>();
    g.ext_ids = d_ids_.as<int32_t>();
    g.n = (int)n_dev_;
    g.dim = dim_;
    g.row_words = row_words_;
    g.maxM = graph_.maxM;
    g.maxM0 = graph_.maxM0;
    g.maxlevel = graph_.maxlevel;
    g.enterpoint = (int)graph_.enterpoint;
    g.dist_kind = is_u8_ ? 3 : graph_.dist_func == 3 ? 1 : graph_.dist_func == 4 ? 2 : 0;
    s = check_cuda(d_keys_.ensure(nq * k * 8), "cudaMalloc(keys)");
    if (!s.ok()) return s;
    uint64_t* keys = d_keys ? d_keys : d_keys_.as<uint64_t>();
    scan_begin(stream);
    s = check_cuda(launch_hnsw_search(g, dq, (int)nq, (int)k, (int)ef_,
                                      d_visited_.as<uint8_t>(), d_epoch_.as<int>(), hnsw_slots_, keys,
                                      d_counters_.as<unsigned long long>(), stream),
                   "hnsw_search");
    scan_end(stream);
    if (!s.ok()) return s;
    // internal positions -> external ids (Object::id of data_rearranged_, hnsw_distfunc_opt.cc:280)
    s = check_cuda(launch_merge_topk(keys, nullptr, 1, 0, k, (int)nq, (int)k, FIN_FLOAT, d_ids_.as<int32_t>(), 0,
                                     nullptr, d_ids, d_dists, d_counts, stream),
                   "finalize");
    stats_.kernel_launches += 2;
    return s;
  }

  // ---- sequential search ----
  if (!(s = check_cuda(d_tc_keys_.ensure(nq * k * 8), "cudaMalloc(keys)")).ok()) return s;
  uint64_t* keys = d_tc_keys_.as<uint64_t>();
  const bool use_tc = ((!dev_u8_rows() && space_ != SPACE_L1 && space_ != SPACE_LINF) || u8_imma_) && !force_exact_ &&
                      k <= (size_t)tc_max_k();  // (l1 / linf have no dot-product form: exact CUDA-core scan)
  s = use_tc ? run_seq_tc(dq, nq, k, keys, stream, true, async) : run_seq_exact(dq, nq, k, keys, stream);
  if (!s.ok()) return s;
  if (dry_run_ && use_tc) return Status::OK();
  if (sharded()) {
    // row-sharded: publish this shard's sorted lists to the peers' view and merge all ranks' lists over NVLink peer
    // memory (exchange.cu) -- the chunk merge of SeqSearch::Search (seqsearch.cc:151-175) with a GPU per chunk
    const size_t q0 = std::min(slice_q0_, nq), q1 = std::min(slice_q1_, nq);
    stats_.kernel_launches += 2;
    s = xch_publish(xch_, keys, d_ids_.as<int32_t>(), pos_base_, nq, k, stream);
    if (s.ok() && xch_hook_) s = xch_hook_(stream);
    if (!s.ok()) return s;
    return xch_merge(xch_, k, finalize_kind(), q0, q1 > q0 ? q1 - q0 : 0, d_keys, d_ids, d_dists, d_counts, stream);
  }
  // sorted (distance, position) keys -> external ids + float distances (extract_knn_results, nmslib_c.cpp:293-328)
  s = check_cuda(launch_merge_topk(keys, nullptr, 1, 0, k, (int)nq, (int)k, finalize_kind(), d_ids_.as<int32_t>(),
                                   pos_base_, d_keys, d_ids, d_dists, d_counts, stream),
                 "finalize");
  ++stats_.kernel_launches;
  return s;
}

Status Engine::shard_export(size_t max_q, size_t max_k, void* blob256) {
  if (method_ != METHOD_SEQ) return Status::Err(kErrIncompat, "only seq_search shards by rows (hnsw: replicas, SURVEY 8e)");
  if (!device_available()) return Status::Err(kErrQuery, "no CUDA device available");
  return xch_export(&xch_, device_, max_q, max_k, blob256);
}
Status Engine::shard_connect(int rank, int world, const void* blobs) {
  if (!xch_) return Status::Err(kErrInvalid, "call nmslib_b200_shard_export first");
  return xch_connect(xch_, rank, world, blobs);
}
void Engine::shard_disconnect() {
  if (xch_) xch_destroy(xch_);
  xch_ = nullptr;
}

// Exact scan on the CUDA cores (uint8 always; float spaces when the tensor-core answer of a query could
// not be certified, or when NB200_FORCE_EXACT is set).  Writes the k best keys per query.
Status Engine::run_seq_exact(const void* dq, size_t nq, size_t k, uint64_t* out_keys, cudaStream_t stream,
                             const int* d_nq) {
  Status s;
  const int bq = scan_exact_block_queries(), bn = scan_exact_block_points();
  const int n_tiles = (int)((n_dev_ + bn - 1) / bn);
  const int q_blocks = (int)((nq + bq - 1) / bq);
  int want = (2 * sm_count_ + q_blocks - 1) / q_blocks;  // aim at >= 2 CTAs per SM worth of work
  int n_split = std::max(1, std::min(want, n_tiles));
  const int max_split = std::max(1, merge_topk_max_items() / (int)k);
  n_split = std::min(n_split, max_split);
  const int tiles_per_split = (n_tiles + n_split - 1) / n_split;
  n_split = (n_tiles + tiles_per_split - 1) / tiles_per_split;

  int mode;
  switch (space_) {
    case SPACE_L2:
    case SPACE_L2SQR: mode = SCAN_L2; break;
    case SPACE_COSINE: mode = SCAN_COSINE; break;
    case SPACE_NEGDOT: mode = SCAN_NEGDOT; break;
    case SPACE_L1: mode = SCAN_L1; break;
    case SPACE_LINF: mode = SCAN_LINF; break;
    case SPACE_ANGULAR: mode = SCAN_ANGULAR; break;
    default: mode = dev_u8_rows() ? SCAN_SIFT : SCAN_L2; break;  // widened uint8 rows: exact integers in fp32
  }
  const void* q_aux = nullptr;
  if (mode == SCAN_COSINE || mode == SCAN_ANGULAR || mode == SCAN_SIFT) {
    s = check_cuda(d_qaux_.ensure(round_up(nq, bq) * 4), "cudaMalloc(qaux)");
    if (!s.ok()) return s;
    s = check_cuda(launch_row_aux(dev_u8_rows(), dq, (int)nq, row_words_, d_qaux_.p, stream, d_nq), "query_aux");
    if (!s.ok()) return s;
    q_aux = d_qaux_.p;
    ++stats_.kernel_launches;
  }
  s = check_cuda(d_partial_.ensure(nq * (size_t)n_split * k * 8), "cudaMalloc(partial)");
  if (!s.ok()) return s;
  const bool dominant = force_exact_ || space_ == SPACE_L1 || space_ == SPACE_LINF || k > (size_t)tc_max_k();
  // k beyond what the shared-memory lists hold: the blocks keep their sorted lists in a global scratch array
  const size_t gl_bytes = scan_exact_glists_bytes((int)nq, (int)k, n_split);
  if (gl_bytes && !(s = check_cuda(d_glists_.ensure(gl_bytes), "cudaMalloc(large-k lists)")).ok()) return s;
  if (dominant) scan_begin(stream);
  s = check_cuda(launch_scan_exact(mode, d_db_.p, dq, d_aux_.p, q_aux, (int)n_dev_, (int)nq, row_words_, (int)k,
                                   pos_base_, d_partial_.as<uint64_t>(), n_split, tiles_per_split, stream, d_nq,
                                   gl_bytes ? d_glists_.as<uint64_t>() : nullptr),
                 "scan_exact");
  if (dominant) scan_end(stream);
  if (!s.ok()) return s;
  s = check_cuda(launch_merge_topk(d_partial_.as<uint64_t>(), nullptr, n_split, k, (size_t)n_split * k, (int)nq,
                                   (int)k, FIN_FLOAT, nullptr, pos_base_, out_keys, nullptr, nullptr, nullptr, stream, d_nq),
                 "merge_topk");
  stats_.kernel_launches += 2;
  return s;
}

// Tensor-core candidates + exact fp32 re-rank + certificate; uncertified queries go to run_seq_exact.
// Split mode (3xTF32): when a batch mostly fails its certificates on data that is not TF32-exact -- neighbours
// closer together than the 2^-9 |q||x| error band of truncated operands, e.g. cosine over concentrated 960-D
// clusters -- the operands are split into TF32-exact halves, q = q_hi + q_lo, x = x_hi + x_lo, and the scan runs on
// rows of three times the length, [q_hi | q_hi | q_lo] . [x_hi | x_lo | x_hi] = q_hi.x_hi + q_hi.x_lo + q_lo.x_hi:
// the same kernels, three times the MMA work, and an error band of D 2^-22 + 3 2^-20 (accumulation + the dropped
// q_lo.x_lo term) instead of 2^-9.  The failed queries of that batch and every later batch use it.
Status Engine::enable_split(cudaStream_t stream) {
  if (tc_split_) return Status::OK();
  if (nb200_option("tc_split", 1) == 0) return Status::Err(kErrQuery, "split mode disabled");
  const size_t n_pad = round_up(n_dev_ < n_ ? n_ : n_dev_, (size_t)tc_block_points());
  const size_t bytes = n_pad * 3 * (size_t)row_words_ * 4;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || bytes + (2ull << 30) > free_b)
    return Status::Err(kErrOOM, "no room for the split operand copy");
  Status s = check_cuda(d_db_split_.ensure(bytes), "cudaMalloc(split rows)");
  if (!s.ok()) return s;
  const bool cos_family = space_ == SPACE_COSINE || space_ == SPACE_ANGULAR;
  s = check_cuda(launch_tc_split_rows(cos_family ? d_db_unit_.as<float>() : d_db_.as<float>(), n_pad, row_words_, 1.0f, 0,
                                      d_db_split_.as<float>(), stream),
                 "tc_split_rows");
  if (!s.ok()) return s;
  ++stats_.kernel_launches;
  tc_split_ = true;
  return Status::OK();
}

Status Engine::run_seq_tc(const void* dq, size_t nq, size_t k, uint64_t* out_keys, cudaStream_t stream,
                          bool allow_split_retry, bool async) {
  Status s;
  absorb_async_counts(false);  // what earlier device-resident batches reported in the meantime (may enable split mode)
  const bool dev_fb = async && !approx_ok_ && !dry_run_;
  if (dev_fb) {
    if (!(s = check_cuda(d_fb_cnt_.ensure(16), "cudaMalloc(fb count)")).ok()) return s;
    if (!(s = check_cuda(d_fb_idx_.ensure(nq * 4), "cudaMalloc(fb idx)")).ok()) return s;
    if (!(s = check_cuda(cudaMemsetAsync(d_fb_cnt_.p, 0, 4, stream), "memset(fb count)")).ok()) return s;
  }
  const bool split = tc_split_;
  const int rw = split ? 3 * row_words_ : row_words_;  // operand row length the scan kernels see
  const int mode = (space_ == SPACE_COSINE || space_ == SPACE_ANGULAR) ? SCAN_COSINE
                   : space_ == SPACE_NEGDOT                             ? SCAN_NEGDOT
                                                                        : SCAN_L2;
  const int qb = tc_block_queries(), bn = tc_block_points();
  const size_t q_pad = round_up(nq, qb);
  const size_t n_pad = round_up(n_dev_, bn);
  const int q_blocks = (int)(q_pad / qb);
  // work decomposition: the host-made piece table (tc_ts_plan) for the TS kernel (rows <= 128 floats, units = SMs,
  // 64-row tiles) and the pair kernel (longer rows, units = CTA pairs, 256-row tiles); tc_plan for the A/B kernel
  const bool ts = tc_ts_supported(rw);  // rows <= 128 floats: queries live in tensor memory
  const bool pair = !ts && tc_pair_enabled() && sm_count_ >= 2;
  int n_cta, work_per_cta = 0, s_max, aligned = 0;
  if (ts || pair) {  // host-made piece table (pair: units are CTA pairs over 256-row tiles, two lists per piece)
    if (plan_key_[0] != nq || plan_key_[1] != n_dev_ || plan_key_[2] != k || plan_key_[3] != (size_t)rw) {
      if (ts) tc_ts_plan((int)nq, (int)n_dev_, (int)k, sm_count_, &h_plan_, &plan_n_cta_, &plan_s_max_, 0, 1, &plan_block_slots_);
      else tc_ts_plan((int)nq, (int)n_dev_, (int)k, sm_count_ / 2, &h_plan_, &plan_n_cta_, &plan_s_max_, tc_pair_block_points(), 2, &plan_block_slots_);
      if (!(s = check_cuda(d_plan_.ensure(h_plan_.size() * 4), "cudaMalloc(plan)")).ok()) return s;
      s = check_cuda(cudaMemcpyAsync(d_plan_.p, h_plan_.data(), h_plan_.size() * 4, cudaMemcpyHostToDevice, stream),
                     "H2D(plan)");
      if (!s.ok()) return s;
      plan_key_[0] = nq;
      plan_key_[1] = n_dev_;
      plan_key_[2] = k;
      plan_key_[3] = (size_t)rw;
    }
    n_cta = plan_n_cta_;
    s_max = pair ? 2 * plan_s_max_ : plan_s_max_;
  } else {
    tc_plan((int)nq, (int)n_dev_, (int)k, sm_count_, bn, &n_cta, &work_per_cta, &s_max, &aligned);
  }
  int kprime, cap;
  tc_candidate_shape((int)k, &kprime, &cap);
  const size_t units = (size_t)q_blocks * s_max;
  if (!(s = check_cuda(d_cand_.ensure(units * qb * (size_t)cap * 8), "cudaMalloc(cand)")).ok()) return s;
  if (!(s = check_cuda(d_cand_cnt_.ensure(units * qb * 4), "cudaMalloc(cand_cnt)")).ok()) return s;
  if (!(s = check_cuda(d_cand_thr_.ensure(units * qb * 4), "cudaMalloc(cand_thr)")).ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_cand_cnt_.p, 0xFF, units * qb * 4, stream), "memset(cand_cnt)")).ok()) return s;
  if (!(s = check_cuda(d_cert_.ensure(nq * 4), "cudaMalloc(cert)")).ok()) return s;
  if (!(s = check_cuda(h_cert_.ensure(nq * 4), "cudaMallocHost(cert)")).ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_flags_.as<int>() + 1, 0, 4, stream), "memset(qflag)")).ok()) return s;
  const float scale = mode == SCAN_L2 ? -2.f : -1.f;
  const float* dbB = split ? d_db_split_.as<float>() : mode == SCAN_COSINE ? d_db_unit_.as<float>() : d_db_.as<float>();
  if (split) stats_.split_queries += nq;
  if (split) {  // prepared A operand [q_hi | q_hi | q_lo], already scaled
    if (!(s = check_cuda(d_q_split_.ensure(q_pad * (size_t)rw * 4), "cudaMalloc(split queries)")).ok()) return s;
    s = check_cuda(launch_tc_split_rows(static_cast<const float*>(dq), q_pad, row_words_, scale, 1,
                                        d_q_split_.as<float>(), stream),
                   "tc_split_rows(queries)");
    if (!s.ok()) return s;
    ++stats_.kernel_launches;
  }
  if (!(s = check_cuda(d_gthr_.ensure(q_pad * 4), "cudaMalloc(gthr)")).ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_gthr_.p, 0xFF, q_pad * 4, stream), "memset(gthr)")).ok()) return s;
  if (dry_run_) {  // (hnsw_build_gpu.cu sizes the scratch buffers for its largest batch once, instead of regrowing
                   //  them -- cudaFree + cudaMalloc of gigabytes -- every few batches)
    if (!ts && !split) return check_cuda(d_qa_.ensure(q_pad * (size_t)row_words_ * 4), "cudaMalloc(qa)");
    return Status::OK();
  }
  // survivors per compaction: k + margin.  Data that is not TF32-exact carries a pass-1 error of ~2^-9 |q||x|,
  // which at k = 100 spans tens of ranks: start with half of k there (the margin doubles when certificates fail)
  // (approx_ok_: graph construction takes the tensor-core ranking as it is -- small margin, no error band in the re-rank)
  const int kprime_req = (int)k + (db_inexact_ && !approx_ok_ && !split ? std::max(tc_margin_, (int)k / 2) : tc_margin_);
  if (u8_imma_) {  // uint8 rows on the integer tensor pipe: byte queries / rows / norm digits, the TS piece table
    scan_begin(stream);
    s = check_cuda(launch_tc_scan_u8(static_cast<const uint8_t*>(dq), d_db_.as<uint8_t>(), d_digits_.as<uint8_t>(), n_pad,
                                     (int)n_dev_, (int)nq, (int)k, kprime_req, u8_m_half_, pos_base_, n_cta, s_max,
                                     d_plan_.as<int>(), d_cand_.as<uint64_t>(), d_cand_cnt_.as<int>(), d_cand_thr_.as<float>(),
                                     d_gthr_.as<uint32_t>(), stream),
                   "tc_scan_u8");
    scan_end(stream);
    if (!s.ok()) return s;
    stats_.kernel_launches += 1;
  } else if (ts) {
    scan_begin(stream);
    s = check_cuda(launch_tc_scan_ts(split ? d_q_split_.as<float>() : static_cast<const float*>(dq), dbB, n_pad,
                                     mode == SCAN_L2 ? d_nblock_.as<float>() : nullptr, d_ones_.as<float>(),
                                     (int)n_dev_, (int)nq, rw, (int)k, kprime_req, split ? 1.0f : scale, pos_base_,
                                     n_cta, s_max, d_plan_.as<int>(), d_cand_.as<uint64_t>(), d_cand_cnt_.as<int>(),
                                     d_cand_thr_.as<float>(), d_gthr_.as<uint32_t>(), d_flags_.as<int>() + 1,
                                     stream),
                   "tc_scan_ts");
    scan_end(stream);
    if (!s.ok()) return s;
    stats_.kernel_launches += 1;  // (the re-rank launches are counted where they are made)
  } else {
    const float* qa = d_q_split_.as<float>();
    if (!split) {
      if (!(s = check_cuda(d_qa_.ensure(q_pad * (size_t)row_words_ * 4), "cudaMalloc(qa)")).ok()) return s;
      s = check_cuda(launch_tc_prep_queries(static_cast<const float*>(dq), d_qa_.as<float>(), q_pad * (size_t)row_words_,
                                            scale, d_flags_.as<int>() + 1, stream),
                     "tc_prep_queries");
      if (!s.ok()) return s;
      qa = d_qa_.as<float>();
    }
    scan_begin(stream);
    const float* nbp = mode == SCAN_L2 ? d_nblock_.as<float>() : nullptr;
    s = check_cuda(pair ? launch_tc_scan_pair(qa, q_pad, dbB, n_pad, nbp, d_ones_.as<float>(), (int)n_dev_,
                                              (int)nq, rw, (int)k, pos_base_, n_cta, d_plan_.as<int>(), s_max,
                                              kprime_req, d_cand_.as<uint64_t>(), d_cand_cnt_.as<int>(),
                                              d_cand_thr_.as<float>(), d_gthr_.as<uint32_t>(), stream)
                        : launch_tc_scan(qa, q_pad, dbB, n_pad, nbp, d_ones_.as<float>(), (int)n_dev_,
                                         (int)nq, rw, (int)k, pos_base_, n_cta, work_per_cta, s_max, aligned,
                                         kprime_req, d_cand_.as<uint64_t>(), d_cand_cnt_.as<int>(),
                                         d_cand_thr_.as<float>(), d_gthr_.as<uint32_t>(), stream),
                   pair ? "tc_scan_pair" : "tc_scan");
    scan_end(stream);
    if (!s.ok()) return s;
    stats_.kernel_launches += 2;
  }
  // The re-rank's sort buffer (and with it how many of its blocks fit an SM) follows the number of candidate lists
  // it may have to read: one launch per run of query blocks with the same number of pieces (whole-wave blocks were
  // scanned as one piece, the blocks behind them in up to s_max).
  {
    const int lpp = pair ? 2 : 1;
    int b0 = 0;
    while (b0 < q_blocks) {
      int lists = s_max, b1 = q_blocks;
      if ((ts || pair) && (int)plan_block_slots_.size() == q_blocks) {
        // (runs are merged while the launches would use the same sort buffer: lists 3 and 4 of config 2 both need
        //  1 024 slots -- one launch instead of two; an unused list has count -1 and is skipped by the kernel)
        lists = std::max(1, plan_block_slots_[b0]) * lpp;
        const int p2 = tc_rerank_pow2(std::min(lists, s_max), cap, (int)k, (int)n_dev_);
        b1 = b0 + 1;
        while (b1 < q_blocks) {
          const int l1 = std::max(1, plan_block_slots_[b1]) * lpp;
          if (tc_rerank_pow2(std::min(l1, s_max), cap, (int)k, (int)n_dev_) != p2) break;
          lists = std::max(lists, l1);
          ++b1;
        }
      }
      const size_t q0 = (size_t)b0 * qb, q1 = std::min(nq, (size_t)b1 * qb);
      if (q1 > q0) {
        s = check_cuda(launch_tc_rerank(d_db_.as<float>(), static_cast<const float*>(dq),
                                        mode == SCAN_COSINE ? d_aux_.as<float>() : nullptr, (int)n_dev_, (int)nq, row_words_,
                                        (int)k, s_max, space_ == SPACE_ANGULAR ? SCAN_ANGULAR : mode, pos_base_,
                                        d_cand_.as<uint64_t>(), d_cand_cnt_.as<int>(), d_cand_thr_.as<float>(),
                                        approx_ok_ ? 0.f : x_max_, d_flags_.as<int>(), out_keys, d_cert_.as<int>(), stream,
                                        (int)q0, (int)(q1 - q0), std::min(lists, s_max),
                                        // split operands: accumulation error + the dropped q_lo.x_lo / re-truncated terms
                                        split ? (float)row_words_ * 2.384185791015625e-07f * 1.01f +
                                                    3.0f * 9.5367431640625e-07f + 1e-6f
                                              : 0.f,
                                        dev_fb ? d_fb_cnt_.as<int>() : nullptr, dev_fb ? d_fb_idx_.as<int>() : nullptr,
                                        u8_imma_ ? d_db_.as<uint8_t>() : nullptr, u8_imma_ ? static_cast<const uint8_t*>(dq) : nullptr,
                                        u8_imma_ ? 1.0f : 0.f, is_u8_ ? 1 : 0),
                       "tc_rerank");
        if (!s.ok()) return s;
        ++stats_.kernel_launches;
      }
      b0 = b1;
    }
  }
  if (dev_fb) {
    // Device-predicated exact re-run of the (normally empty) set of uncertified queries: gather -> exact scan ->
    // merge -> scatter are launched for the worst case (all nq) and leave at once past the count the re-rank left
    // on the device.  Nothing here waits for the host, so a caller's steps queue back to back.
    const int* d_cnt = d_fb_cnt_.as<int>();
    const size_t fb_pad = round_up(nq, (size_t)scan_exact_block_queries());
    if (!(s = check_cuda(d_fb_q_.ensure(fb_pad * (size_t)row_words_ * 4), "cudaMalloc(fb q)")).ok()) return s;
    if (!(s = check_cuda(d_fb_keys_.ensure(nq * k * 8), "cudaMalloc(fb keys)")).ok()) return s;
    s = check_cuda(launch_gather_rows(static_cast<const uint32_t*>(dq), d_fb_idx_.as<int>(), (int)nq, row_words_,
                                      d_fb_q_.as<uint32_t>(), stream, d_cnt, scan_exact_block_queries()),
                   "gather");
    if (!s.ok()) return s;
    if (!(s = run_seq_exact(d_fb_q_.p, nq, k, d_fb_keys_.as<uint64_t>(), stream, d_cnt)).ok()) return s;
    s = check_cuda(launch_scatter_keys(d_fb_keys_.as<uint64_t>(), d_fb_idx_.as<int>(), (int)nq, (int)k, out_keys, stream,
                                       d_cnt, u8_widened() ? 1 : 0),
                   "scatter");
    if (!s.ok()) return s;
    stats_.kernel_launches += 2;
    // the count, for the statistics and for the adaptation of later batches
    if (!(s = check_cuda(h_fb_cnt_.ensure(kFbRing * 4), "cudaMallocHost(fb count)")).ok()) return s;
    const int slot = fb_head_;
    if (fb_pending_[slot]) absorb_async_counts(true);  // (ring full: that copy is kFbRing calls old)
    fb_head_ = (fb_head_ + 1) % kFbRing;
    if (!fb_ev_[slot] && !(s = check_cuda(cudaEventCreateWithFlags(&fb_ev_[slot], cudaEventDisableTiming), "cudaEventCreate")).ok())
      return s;
    s = check_cuda(cudaMemcpyAsync(h_fb_cnt_.as<int>() + slot, d_fb_cnt_.p, 4, cudaMemcpyDeviceToHost, stream), "D2H(fb count)");
    if (!s.ok()) return s;
    if (!(s = check_cuda(cudaEventRecord(fb_ev_[slot], stream), "cudaEventRecord")).ok()) return s;
    fb_nq_[slot] = nq;
    fb_pending_[slot] = true;
    return Status::OK();
  }
  // certificates back to the host; re-run the (normally empty) set of uncertified queries exactly
  s = check_cuda(cudaMemcpyAsync(h_cert_.p, d_cert_.p, nq * 4, cudaMemcpyDeviceToHost, stream), "D2H(cert)");
  if (!s.ok()) return s;
  s = check_cuda(cudaStreamSynchronize(stream), "tc scan");
  if (!s.ok()) return s;
  std::vector<int> fb;
  const int* cert = h_cert_.as<int>();
  for (size_t i = 0; i < nq; ++i)
    if (!cert[i]) fb.push_back((int)i);
  if (fb.empty()) return Status::OK();
  if (approx_ok_) {  // (graph construction: the re-ranked candidates are good enough)
    stats_.fallback_queries += fb.size();
    return Status::OK();
  }
  if (!split && allow_split_retry && db_inexact_ && fb.size() * 4 > nq && enable_split(stream).ok()) {
    // most of the batch sits inside the TF32 error band: give the failed queries the split (3xTF32) scan now
    const size_t nsp = fb.size(), sp_pad = round_up(nsp, (size_t)tc_block_queries());
    if (!(s = check_cuda(d_sp_idx_.ensure(nsp * 4), "cudaMalloc(split idx)")).ok()) return s;
    if (!(s = check_cuda(d_sp_q_.ensure(sp_pad * (size_t)row_words_ * 4), "cudaMalloc(split q)")).ok()) return s;
    if (!(s = check_cuda(d_sp_keys_.ensure(nsp * k * 8), "cudaMalloc(split keys)")).ok()) return s;
    if (!(s = check_cuda(cudaMemsetAsync(d_sp_q_.p, 0, sp_pad * (size_t)row_words_ * 4, stream), "memset(split q)")).ok())
      return s;
    s = check_cuda(cudaMemcpyAsync(d_sp_idx_.p, fb.data(), nsp * 4, cudaMemcpyHostToDevice, stream), "H2D(split idx)");
    if (!s.ok()) return s;
    s = check_cuda(launch_gather_rows(static_cast<const uint32_t*>(dq), d_sp_idx_.as<int>(), (int)nsp, row_words_,
                                      d_sp_q_.as<uint32_t>(), stream),
                   "gather");
    if (!s.ok()) return s;
    if (!(s = check_cuda(cudaStreamSynchronize(stream), "split gather")).ok()) return s;  // (fb is reused below)
    s = run_seq_tc(d_sp_q_.p, nsp, k, d_sp_keys_.as<uint64_t>(), stream, false);
    if (!s.ok()) return s;
    s = check_cuda(launch_scatter_keys(d_sp_keys_.as<uint64_t>(), d_sp_idx_.as<int>(), (int)nsp, (int)k, out_keys, stream),
                   "scatter");
    if (!s.ok()) return s;
    stats_.kernel_launches += 2;
    return check_cuda(cudaStreamSynchronize(stream), "split scan");
  }
  stats_.fallback_queries += fb.size();
  // the thresholds sat too close to the k-th answer for this data's pass-1 error bound: keep more survivors per
  // compaction from the next batch on (costs candidates, buys certificate margin)
  if (fb.size() * 64 > nq && tc_margin_ < 128) tc_margin_ *= 2;
  const size_t nfb = fb.size();
  const size_t fb_pad = round_up(nfb, (size_t)scan_exact_block_queries());
  if (!(s = check_cuda(d_fb_idx_.ensure(nfb * 4), "cudaMalloc(fb idx)")).ok()) return s;
  if (!(s = check_cuda(d_fb_q_.ensure(fb_pad * (size_t)row_words_ * 4), "cudaMalloc(fb q)")).ok()) return s;
  if (!(s = check_cuda(d_fb_keys_.ensure(nfb * k * 8), "cudaMalloc(fb keys)")).ok()) return s;
  if (!(s = check_cuda(cudaMemsetAsync(d_fb_q_.p, 0, fb_pad * (size_t)row_words_ * 4, stream), "memset(fb q)")).ok())
    return s;
  s = check_cuda(cudaMemcpyAsync(d_fb_idx_.p, fb.data(), nfb * 4, cudaMemcpyHostToDevice, stream), "H2D(fb idx)");
  if (!s.ok()) return s;
  s = check_cuda(launch_gather_rows(static_cast<const uint32_t*>(dq), d_fb_idx_.as<int>(), (int)nfb, row_words_,
                                    d_fb_q_.as<uint32_t>(), stream),
                 "gather");
  if (!s.ok()) return s;
  s = run_seq_exact(d_fb_q_.p, nfb, k, d_fb_keys_.as<uint64_t>(), stream);
  if (!s.ok()) return s;
  s = check_cuda(launch_scatter_keys(d_fb_keys_.as<uint64_t>(), d_fb_idx_.as<int>(), (int)nfb, (int)k, out_keys,
                                     stream, nullptr, u8_widened() ? 1 : 0),
                 "scatter");
  if (!s.ok()) return s;
  stats_.kernel_launches += 2;
  // fb (host vector) must outlive the async H2D above
  return check_cuda(cudaStreamSynchronize(stream), "fallback scan");
}

// Counts of uncertified queries that device-resident batches left in pinned memory: into the statistics, and into the
// same adaptation the host entry applies at once -- split (3xTF32) operands when a quarter of a batch failed on data
// that is not TF32-exact, a wider candidate margin when certificates fail in numbers.
void Engine::absorb_async_counts(bool wait) {
  for (int i = 0; i < kFbRing; ++i) {
    if (!fb_pending_[i]) continue;
    if (wait) cudaEventSynchronize(fb_ev_[i]);
    else if (cudaEventQuery(fb_ev_[i]) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    fb_pending_[i] = false;
    const size_t c = (size_t)h_fb_cnt_.as<int>()[i], nq = fb_nq_[i];
    stats_.fallback_queries += c;
    if (!tc_split_ && db_inexact_ && c * 4 > nq) enable_split(stream_);
    if (c * 64 > nq && tc_margin_ < 128) tc_margin_ *= 2;
  }
}

Status Engine::knn_device(const void* d_queries, size_t nq, size_t elem_count, size_t k, int32_t* d_ids,
                          float* d_dists, uint64_t* d_keys, int32_t* d_counts, cudaStream_t stream,
                          size_t src_pitch) {
  if (!built_) return Status::Err(kErrBuild, "Index not built");
  if (nq == 0 || k == 0) return Status::Err(kErrInvalid, "empty query batch or k == 0");
  Status s = prepare();
  if (!s.ok()) return s;
  if (n_dev_ == 0) return Status::Err(kErrQuery, "index holds no data");
  if (elem_count != (size_t)dim_)  // the reference CHECKs equal lengths (space_lp.cc:29) -> error 9
    return Status::Err(kErrQuery, "query length " + std::to_string(elem_count) + " != index dimension " +
                                      std::to_string(dim_));
  // (graph construction: tensor-core candidates are taken as they are, so the exact re-run path and its limit on
  // k never come into play)
  const bool approx_tc = approx_ok_ && !force_exact_ && k <= (size_t)tc_max_k();
  if (method_ == METHOD_SEQ && !approx_tc && k > (size_t)scan_exact_max_k())
    return Status::Err(kErrTooLarge, "k above " + std::to_string(scan_exact_max_k()) + " is not supported");
  if (method_ == METHOD_HNSW && k > (size_t)hnsw_max_ef()) return Status::Err(kErrTooLarge, "k too large for hnsw");
  cudaStream_t st = stream ? stream : stream_;
  s = stage_queries_device(d_queries, true, nq, elem_count, st, src_pitch);
  if (!s.ok()) return s;
  s = run(d_q_.p, nq, k, d_ids, d_dists, d_keys, d_counts, st, /*async=*/true);
  if (s.ok()) stats_.queries += nq;
  if (s.ok() && method_ == METHOD_SEQ) stats_.distance_evals += (uint64_t)nq * n_dev_;
  return s;
}

int Engine::range_mode() const {
  return dev_u8_rows()             ? SCAN_SIFT  // byte rows (128 per row)
         : space_ == SPACE_COSINE  ? SCAN_COSINE
         : space_ == SPACE_ANGULAR ? SCAN_ANGULAR
         : space_ == SPACE_NEGDOT  ? SCAN_NEGDOT
         : space_ == SPACE_L1      ? SCAN_L1
         : space_ == SPACE_LINF    ? SCAN_LINF
                                   : SCAN_L2;
}

// SeqSearch::Search(RangeQuery*) (seqsearch.cc:108-141) through nmslib_range_query_fill (nmslib_c.cpp:1051-1153):
// every object within the radius, in position order, truncated to the caller's capacity.
Status Engine::range_host(const void* query, size_t elem_count, double radius, size_t capacity, int32_t* ids,
                          float* dists, size_t* size) {
  *size = 0;
  if (!built_) return Status::Err(kErrBuild, "Index not built");
  if (method_ != METHOD_SEQ)  // hnsw.cc: "Range search is not supported!" -> SPACE_INCOMPATIBLE (nmslib_c.cpp:1127-1137)
    return Status::Err(kErrIncompat, "Range query not supported by method: Range search is not supported!");
  Status s = prepare();
  if (!s.ok()) return s;
  if (n_dev_ == 0) return Status::OK();
  if (elem_count != (size_t)dim_)
    return Status::Err(kErrQuery, "query length " + std::to_string(elem_count) + " != index dimension " +
                                      std::to_string(dim_));
  const int cap = (int)std::min<size_t>(capacity, n_dev_);
  s = stage_queries_device(query, false, 1, elem_count, stream_);
  if (!s.ok()) return s;
  const size_t tmp_bytes = round_up(n_dev_ * 4, 256), out_bytes = round_up((size_t)cap * 4, 256);
  if (!(s = check_cuda(d_range_.ensure(tmp_bytes + 2 * out_bytes + 256), "cudaMalloc(range)")).ok()) return s;
  float* d_tmp = d_range_.as<float>();
  int32_t* d_ids = reinterpret_cast<int32_t*>(d_range_.as<char>() + tmp_bytes);
  float* d_d = reinterpret_cast<float*>(d_range_.as<char>() + tmp_bytes + out_bytes);
  int* d_cnt = reinterpret_cast<int*>(d_range_.as<char>() + tmp_bytes + 2 * out_bytes);
  const int mode = range_mode();
  // RangeQuery<int> compares with static_cast<int>(radius) (nmslib_c.cpp:1087-1088)
  const float r = is_u8_ ? std::floor((float)radius) : (float)radius;
  s = check_cuda(launch_range_scan(d_db_.as<float>(), d_q_.as<float>(),
                                   (mode == SCAN_COSINE || mode == SCAN_ANGULAR) ? d_aux_.as<float>() : nullptr,
                                   d_ids_.as<int32_t>(), (int)n_dev_, row_words_, mode,
                                   space_ == SPACE_L2 ? 1 : 0, r, cap, d_tmp, d_ids, d_d, d_cnt, stream_),
                 "range_scan");
  if (!s.ok()) return s;
  stats_.kernel_launches += 2;
  int found = 0;
  if (!(s = check_cuda(cudaMemcpyAsync(&found, d_cnt, 4, cudaMemcpyDeviceToHost, stream_), "D2H(range count)")).ok()) return s;
  if (!(s = check_cuda(cudaStreamSynchronize(stream_), "range query")).ok()) return s;
  if (found > 0) {
    if (!(s = check_cuda(cudaMemcpyAsync(ids, d_ids, (size_t)found * 4, cudaMemcpyDeviceToHost, stream_), "D2H(range ids)")).ok())
      return s;
    if (!(s = check_cuda(cudaMemcpyAsync(dists, d_d, (size_t)found * 4, cudaMemcpyDeviceToHost, stream_), "D2H(range dists)")).ok())
      return s;
    if (!(s = check_cuda(cudaStreamSynchronize(stream_), "range query")).ok()) return s;
  }
  *size = (size_t)found;
  stats_.queries += 1;
  stats_.distance_evals += n_dev_;
  return Status::OK();
}

// Batched range queries (K5b, DESIGN.md): the answer of range_host for every query, one device submission per chunk.
// Float spaces with a dot-product form and uint8 run on the tensor cores: radius -> pass-1 threshold T_q (uint8 byte
// rows: an integer accumulator threshold), the TS / pair / u8 scan in range mode (survivors beating the threshold in
// position order, a position cut where a list fills), verification of the candidates with the per-query scan's own
// distance code.  l1 / linf run the same way on the CUDA cores: K2 in range mode (scan_exact.cu, T_q from
// range_threshold), then the same verification.  force_exact, and every query a batched pass cannot certify, take
// the per-query exact scan (launch_range_scan) inside the same submission.
// Outputs are staged in CSR form (min(capacity, n) slots per query); a batch whose staging would exceed
// kRangeStageBytes runs in query chunks.
namespace {
constexpr size_t kRangeStageBytes = 64u << 20;  // ids + distances staged on the device per chunk
constexpr size_t kRangeChunkQueries = 65536;    // bounds the candidate lists of one chunk as well
}  // namespace

Status Engine::range_batch_host(const void* queries, size_t nq, size_t elem_count, const double* radii,
                                const size_t* caps, int32_t* const* ids, float* const* dists, size_t* sizes) {
  for (size_t i = 0; i < nq; ++i) sizes[i] = 0;
  if (!built_) return Status::Err(kErrBuild, "Index not built");
  if (method_ != METHOD_SEQ)
    return Status::Err(kErrIncompat, "Range query not supported by method: Range search is not supported!");
  Status s = prepare();
  if (!s.ok()) return s;
  if (n_dev_ == 0 || nq == 0) return Status::OK();
  if (elem_count != (size_t)dim_)
    return Status::Err(kErrQuery, "query length " + std::to_string(elem_count) + " != index dimension " +
                                      std::to_string(dim_));
  // the radius conversions of range_host (RangeQuery<int> compares with static_cast<int>(radius))
  std::vector<float> r(nq);
  std::vector<int> cap(nq);
  for (size_t i = 0; i < nq; ++i) {
    r[i] = is_u8_ ? std::floor((float)radii[i]) : (float)radii[i];
    cap[i] = (int)std::min<size_t>(caps[i], n_dev_);
  }
  const size_t esz = is_u8_ ? 1 : 4;
  size_t c0 = 0;
  while (c0 < nq) {
    size_t c1 = c0, staged = 0;
    while (c1 < nq && c1 - c0 < kRangeChunkQueries &&
           (c1 == c0 || (staged + (size_t)cap[c1]) * 8 <= kRangeStageBytes))
      staged += (size_t)cap[c1++];
    s = range_chunk(static_cast<const char*>(queries) + c0 * elem_count * esz, c1 - c0, elem_count, r.data() + c0,
                    cap.data() + c0, ids + c0, dists + c0, sizes + c0);
    if (!s.ok()) return s;
    c0 = c1;
  }
  stats_.queries += nq;
  stats_.distance_evals += (uint64_t)nq * n_dev_;
  return Status::OK();
}

Status Engine::range_chunk(const void* queries, size_t nq, size_t elem_count, const float* radii, const int* caps,
                           int32_t* const* ids, float* const* dists, size_t* sizes) {
  const int mode = range_mode();
  const int take_sqrt = space_ == SPACE_L2 ? 1 : 0;
  // the tensor-core pass needs the TS kernel (rows <= 128 floats) or the pair kernel; with option tc_pair=0 longer
  // rows take the per-query exact scan like l1 / linf (not counted as fallbacks: no tensor-core pass was made).
  // uint8: byte rows run the integer-pipe kernel (tc_scan_u8_kernel) over the TS piece table; widened rows (option
  // u8_imma=0, or norms beyond the digit block) are exact integers in fp32 and take the TS kernel like l2sqr
  const bool u8 = u8_imma_;  // (never with force_exact)
  const bool ts = u8 || tc_ts_supported(row_words_);
  const bool pair = !ts && tc_pair_enabled() && sm_count_ >= 2;
  const bool tc = !force_exact_ && (ts || pair) &&
                  (u8 || u8_widened() || space_ == SPACE_L2 || space_ == SPACE_L2SQR || space_ == SPACE_COSINE ||
                   space_ == SPACE_NEGDOT || space_ == SPACE_ANGULAR);
  // l1 / linf: K2 in range mode (scan_exact.cu), whatever the row length
  const bool lp = !force_exact_ && (space_ == SPACE_L1 || space_ == SPACE_LINF);
  Status s = stage_queries_device(queries, false, nq, elem_count, stream_);
  if (!s.ok()) return s;
  // per-query parameters: radii [nq] f32 | caps [nq] i32 | CSR offsets [nq] i64; outputs: counts [nq] | fallback
  // count [1] + list [nq] | ids [total] | distances [total]
  std::vector<int64_t> off(nq);
  int64_t total = 0;
  for (size_t i = 0; i < nq; ++i) {
    off[i] = total;
    total += caps[i];
  }
  const size_t a4 = round_up(nq * 4, 256), a8 = round_up(nq * 8, 256);
  std::vector<char> h_par(2 * a4 + a8);
  memcpy(h_par.data(), radii, nq * 4);
  memcpy(h_par.data() + a4, caps, nq * 4);
  memcpy(h_par.data() + 2 * a4, off.data(), nq * 8);
  if (!(s = check_cuda(d_rq_.ensure(h_par.size()), "cudaMalloc(range params)")).ok()) return s;
  s = check_cuda(cudaMemcpyAsync(d_rq_.p, h_par.data(), h_par.size(), cudaMemcpyHostToDevice, stream_), "H2D(range params)");
  if (!s.ok()) return s;
  const float* d_radii = d_rq_.as<float>();
  const int* d_caps = reinterpret_cast<const int*>(d_rq_.as<char>() + a4);
  const int64_t* d_off = reinterpret_cast<const int64_t*>(d_rq_.as<char>() + 2 * a4);
  const size_t ob = round_up((size_t)total * 4, 256);
  if (!(s = check_cuda(d_rq_out_.ensure(3 * a4 + 256 + 2 * ob), "cudaMalloc(range outputs)")).ok()) return s;
  int* d_counts = d_rq_out_.as<int>();
  int* d_fb_cnt = reinterpret_cast<int*>(d_rq_out_.as<char>() + a4);
  int* d_fb_idx = reinterpret_cast<int*>(d_rq_out_.as<char>() + a4 + 256);
  int32_t* d_oids = reinterpret_cast<int32_t*>(d_rq_out_.as<char>() + 2 * a4 + 256);
  float* d_odists = reinterpret_cast<float*>(d_rq_out_.as<char>() + 2 * a4 + 256 + ob);
  if (!(s = check_cuda(d_range_.ensure(round_up(n_dev_ * 4, 256)), "cudaMalloc(range)")).ok()) return s;
  const float* aux = (mode == SCAN_COSINE || mode == SCAN_ANGULAR) ? d_aux_.as<float>() : nullptr;
  // the per-query exact scan of query i (every query of the chunk, or the uncertified ones)
  auto exact = [&](size_t i) {
    stats_.kernel_launches += 2;
    return check_cuda(launch_range_scan(d_db_.as<float>(), reinterpret_cast<const float*>(d_q_.as<char>() + i * row_words_ * 4),
                                        aux, d_ids_.as<int32_t>(), (int)n_dev_, row_words_, mode, take_sqrt, radii[i],
                                        caps[i], d_range_.as<float>(), d_oids + off[i], d_odists + off[i], d_counts + i,
                                        stream_),
                      "range_scan");
  };
  // the candidate lists of a range-mode scan ([q_pad / 256][s_max][256][list cap]): verification, then the per-query
  // exact scan of every query it could not certify; *n_fb = how many
  auto verify = [&](int s_max, size_t* n_fb) {
    Status v = check_cuda(launch_range_verify(d_db_.as<float>(), d_q_.as<float>(), d_ids_.as<int32_t>(), row_words_, mode,
                                              take_sqrt, pos_base_, d_radii, d_caps, d_off, d_rcand_.as<uint64_t>(),
                                              d_rcnt_.as<int>(), d_rcut_.as<uint32_t>(), s_max, tc_range_cap(), 0,
                                              (int)nq, d_oids, d_odists, d_counts, d_fb_cnt, d_fb_idx, stream_),
                          "range_verify");
    if (!v.ok()) return v;
    ++stats_.kernel_launches;
    int fb_cnt = 0;
    v = check_cuda(cudaMemcpyAsync(&fb_cnt, d_fb_cnt, 4, cudaMemcpyDeviceToHost, stream_), "D2H(range fb count)");
    if (v.ok()) v = check_cuda(cudaStreamSynchronize(stream_), "range batch");
    if (!v.ok()) return v;
    *n_fb = (size_t)fb_cnt;
    if (fb_cnt > 0) {
      std::vector<int> fb(fb_cnt);
      v = check_cuda(cudaMemcpyAsync(fb.data(), d_fb_idx, fb.size() * 4, cudaMemcpyDeviceToHost, stream_), "D2H(range fb list)");
      if (v.ok()) v = check_cuda(cudaStreamSynchronize(stream_), "range batch");
      for (size_t j = 0; j < fb.size() && v.ok(); ++j) v = exact((size_t)fb[j]);
    }
    return v;
  };
  size_t n_fb = 0;
  if (lp) {
    // K2 split like run_seq_exact (>= 2 CTAs per SM worth of work), into at most 2^15 / cap splits: range_verify_kernel
    // sorts s_max * cap positions in a power-of-two shared buffer of at most 200 KB
    const int bq = scan_exact_block_queries(), bn = scan_exact_block_points(), cap = tc_range_cap();
    const int n_tiles = (int)((n_dev_ + bn - 1) / bn);
    const int q_blocks = (int)((nq + bq - 1) / bq);
    const int want = (2 * sm_count_ + q_blocks - 1) / q_blocks;
    const int n_split = std::max(1, std::min({want, n_tiles, (1 << 15) / cap}));
    const int tiles_per_split = (n_tiles + n_split - 1) / n_split;
    const int s_max = (n_tiles + tiles_per_split - 1) / tiles_per_split;
    const size_t lists = round_up(nq, (size_t)tc_block_queries()) * s_max;  // (every list is written by the scan)
    if (!(s = check_cuda(d_rcand_.ensure(lists * cap * 8), "cudaMalloc(range cand)")).ok()) return s;
    if (!(s = check_cuda(d_rcnt_.ensure(lists * 4), "cudaMalloc(range cand_cnt)")).ok()) return s;
    if (!(s = check_cuda(d_rcut_.ensure(lists * 4), "cudaMalloc(range cut)")).ok()) return s;
    if (!(s = check_cuda(cudaMemsetAsync(d_fb_cnt, 0, 4, stream_), "memset(range fb count)")).ok()) return s;
    scan_begin(stream_);
    s = check_cuda(launch_scan_exact_range(mode, d_db_.p, d_q_.p, (int)n_dev_, (int)nq, row_words_, pos_base_, d_radii,
                                           cap, d_rcand_.as<uint64_t>(), d_rcnt_.as<int>(), d_rcut_.as<uint32_t>(), s_max,
                                           tiles_per_split, stream_),
                   "scan_exact(range)");
    scan_end(stream_);
    if (!s.ok()) return s;
    ++stats_.kernel_launches;
    if (!(s = verify(s_max, &n_fb)).ok()) return s;
    stats_.range_fallback_queries += n_fb;
  } else if (!tc) {
    for (size_t i = 0; i < nq && s.ok(); ++i) s = exact(i);
    if (!s.ok()) return s;
  } else {
    const int qb = tc_block_queries();
    const size_t q_pad = round_up(nq, (size_t)qb);
    const size_t n_pad = round_up(n_dev_, (size_t)tc_block_points());
    int n_cta, slots;
    if (ts) tc_ts_plan((int)nq, (int)n_dev_, 1, sm_count_, &h_rplan_, &n_cta, &slots);
    else tc_ts_plan((int)nq, (int)n_dev_, 1, sm_count_ / 2, &h_rplan_, &n_cta, &slots, tc_pair_block_points(), 2);
    const int s_max = pair ? 2 * slots : slots;
    const size_t lists = q_pad / qb * (size_t)s_max * qb, cap = (size_t)tc_range_cap();
    if (!(s = check_cuda(d_rplan_.ensure(h_rplan_.size() * 4), "cudaMalloc(range plan)")).ok()) return s;
    s = check_cuda(cudaMemcpyAsync(d_rplan_.p, h_rplan_.data(), h_rplan_.size() * 4, cudaMemcpyHostToDevice, stream_),
                   "H2D(range plan)");
    if (!s.ok()) return s;
    if (!(s = check_cuda(d_rcand_.ensure(lists * cap * 8), "cudaMalloc(range cand)")).ok()) return s;
    if (!(s = check_cuda(d_rcnt_.ensure(lists * 4), "cudaMalloc(range cand_cnt)")).ok()) return s;
    if (!(s = check_cuda(d_rcut_.ensure(lists * 4), "cudaMalloc(range cut)")).ok()) return s;
    if (!(s = check_cuda(d_rthr_.ensure(q_pad * 4), "cudaMalloc(range thr)")).ok()) return s;
    if (!(s = check_cuda(cudaMemsetAsync(d_rcnt_.p, 0xFF, lists * 4, stream_), "memset(range cand_cnt)")).ok()) return s;
    if (!(s = check_cuda(cudaMemsetAsync(d_fb_cnt, 0, 4, stream_), "memset(range fb count)")).ok()) return s;
    const int tmode = space_ == SPACE_COSINE ? SCAN_COSINE : space_ == SPACE_ANGULAR ? SCAN_ANGULAR
                      : space_ == SPACE_NEGDOT ? SCAN_NEGDOT : SCAN_L2;
    s = u8 ? check_cuda(launch_tc_range_threshold_u8(d_q_.as<uint8_t>(), (int)nq, d_radii, u8_m_half_,
                                                     d_rthr_.as<uint32_t>(), stream_),
                        "tc_range_threshold_u8")
           : check_cuda(launch_tc_range_threshold(d_q_.as<float>(), (int)nq, row_words_, tmode, take_sqrt, d_radii,
                                                  x_max_, db_inexact_ ? 1 : 0, d_rthr_.as<uint32_t>(), stream_),
                        "tc_range_threshold");
    if (!s.ok()) return s;
    // pass 1 on the plain operands (never the split copy): the threshold's error band covers TF32-inexact data
    const bool cosf = tmode == SCAN_COSINE || tmode == SCAN_ANGULAR;
    const float scale = tmode == SCAN_L2 ? -2.f : -1.f;
    const float* dbB = cosf ? d_db_unit_.as<float>() : d_db_.as<float>();
    const float* nbp = tmode == SCAN_L2 ? d_nblock_.as<float>() : nullptr;
    if (pair) {
      if (!(s = check_cuda(d_qa_.ensure(q_pad * (size_t)row_words_ * 4), "cudaMalloc(qa)")).ok()) return s;
      s = check_cuda(launch_tc_prep_queries(d_q_.as<float>(), d_qa_.as<float>(), q_pad * (size_t)row_words_, scale,
                                            d_flags_.as<int>() + 1, stream_),
                     "tc_prep_queries");
      if (!s.ok()) return s;
      ++stats_.kernel_launches;
    }
    scan_begin(stream_);
    s = check_cuda(u8   ? launch_tc_scan_u8(d_q_.as<uint8_t>(), d_db_.as<uint8_t>(), d_digits_.as<uint8_t>(), n_pad,
                                            (int)n_dev_, (int)nq, 1, 0, u8_m_half_, pos_base_, n_cta, s_max,
                                            d_rplan_.as<int>(), d_rcand_.as<uint64_t>(), d_rcnt_.as<int>(), nullptr,
                                            d_rthr_.as<uint32_t>(), stream_, d_rcut_.as<uint32_t>())
                   : ts ? launch_tc_scan_ts(d_q_.as<float>(), dbB, n_pad, nbp, d_ones_.as<float>(), (int)n_dev_, (int)nq,
                                            row_words_, 1, 0, scale, pos_base_, n_cta, s_max, d_rplan_.as<int>(),
                                            d_rcand_.as<uint64_t>(), d_rcnt_.as<int>(), nullptr, d_rthr_.as<uint32_t>(),
                                            d_flags_.as<int>() + 1, stream_, d_rcut_.as<uint32_t>())
                        : launch_tc_scan_pair(d_qa_.as<float>(), q_pad, dbB, n_pad, nbp, d_ones_.as<float>(), (int)n_dev_,
                                              (int)nq, row_words_, 1, pos_base_, n_cta, d_rplan_.as<int>(), s_max, 0,
                                              d_rcand_.as<uint64_t>(), d_rcnt_.as<int>(), nullptr, d_rthr_.as<uint32_t>(),
                                              stream_, d_rcut_.as<uint32_t>()),
                   u8 ? "tc_scan_u8(range)" : ts ? "tc_scan_ts(range)" : "tc_scan_pair(range)");
    scan_end(stream_);
    if (!s.ok()) return s;
    stats_.kernel_launches += 2;
    if (!(s = verify(s_max, &n_fb)).ok()) return s;
    stats_.range_tc_queries += nq - n_fb;
    stats_.range_fallback_queries += n_fb;
  }
  std::vector<int> cnt(nq);
  std::vector<int32_t> h_ids((size_t)total);
  std::vector<float> h_d((size_t)total);
  s = check_cuda(cudaMemcpyAsync(cnt.data(), d_counts, nq * 4, cudaMemcpyDeviceToHost, stream_), "D2H(range counts)");
  if (s.ok() && total > 0)
    s = check_cuda(cudaMemcpyAsync(h_ids.data(), d_oids, (size_t)total * 4, cudaMemcpyDeviceToHost, stream_), "D2H(range ids)");
  if (s.ok() && total > 0)
    s = check_cuda(cudaMemcpyAsync(h_d.data(), d_odists, (size_t)total * 4, cudaMemcpyDeviceToHost, stream_), "D2H(range dists)");
  if (s.ok()) s = check_cuda(cudaStreamSynchronize(stream_), "range batch");
  if (!s.ok()) return s;
  for (size_t i = 0; i < nq; ++i) {
    const size_t c = (size_t)cnt[i];
    memcpy(ids[i], h_ids.data() + off[i], c * 4);
    memcpy(dists[i], h_d.data() + off[i], c * 4);
    sizes[i] = c;
  }
  return Status::OK();
}

// ShardGroup worker: this rank's part of one batch.  Queries come from host memory (pinned when the group staged them),
// the rows [q0, q1) this rank finalises go straight into the group's shared pinned result arrays.
Status Engine::knn_host_slice(const void* queries, size_t nq, size_t elem_count, size_t k, size_t q0, size_t q1,
                              int32_t* h_ids, float* h_dists, int32_t* h_counts) {
  if (!built_) return Status::Err(kErrBuild, "Index not built");
  Status s = prepare();
  if (!s.ok()) return s;
  if (n_dev_ == 0) return Status::Err(kErrQuery, "shard holds no data");
  if (elem_count != (size_t)dim_)
    return Status::Err(kErrQuery, "query length " + std::to_string(elem_count) + " != index dimension " + std::to_string(dim_));
  if (k > (size_t)scan_exact_max_k())
    return Status::Err(kErrTooLarge, "k above " + std::to_string(scan_exact_max_k()) + " is not supported");
  const size_t out_n = nq * k;
  if (!(s = check_cuda(d_out_ids_.ensure(out_n * 4), "cudaMalloc(out ids)")).ok()) return s;
  if (!(s = check_cuda(d_out_dists_.ensure(out_n * 4), "cudaMalloc(out dists)")).ok()) return s;
  if (!(s = check_cuda(d_out_counts_.ensure(nq * 4), "cudaMalloc(out counts)")).ok()) return s;
  if (!(s = stage_queries_device(queries, false, nq, elem_count, stream_)).ok()) return s;
  set_merge_slice(q0, q1);
  s = run(d_q_.p, nq, k, d_out_ids_.as<int32_t>(), d_out_dists_.as<float>(), nullptr, d_out_counts_.as<int32_t>(), stream_);
  if (!s.ok()) return s;
  if (q1 > q0) {
    const size_t cnt = q1 - q0;
    if (!(s = check_cuda(cudaMemcpyAsync(h_ids + q0 * k, d_out_ids_.as<int32_t>() + q0 * k, cnt * k * 4, cudaMemcpyDeviceToHost, stream_), "D2H(ids)")).ok()) return s;
    if (!(s = check_cuda(cudaMemcpyAsync(h_dists + q0 * k, d_out_dists_.as<float>() + q0 * k, cnt * k * 4, cudaMemcpyDeviceToHost, stream_), "D2H(dists)")).ok()) return s;
    if (!(s = check_cuda(cudaMemcpyAsync(h_counts + q0, d_out_counts_.as<int32_t>() + q0, cnt * 4, cudaMemcpyDeviceToHost, stream_), "D2H(counts)")).ok()) return s;
  }
  s = check_cuda(cudaStreamSynchronize(stream_), "sharded query batch");
  if (s.ok() && sharded() && xch_take_error(xch_))
    s = Status::Err(kErrQuery, "shard exchange: a peer did not publish its lists within 10 s (ranks must make the same calls)");
  if (s.ok()) {
    stats_.queries += nq;
    stats_.distance_evals += (uint64_t)nq * n_dev_;
  }
  return s;
}

Status Engine::knn_host(const void* queries, size_t nq, size_t elem_count, size_t k, const int32_t** ids,
                        const float** dists, const int32_t** counts) {
  if (!built_) return Status::Err(kErrBuild, "Index not built");
  if (!queries || nq == 0 || k == 0) return Status::Err(kErrInvalid, "empty query batch or k == 0");
  Status s = prepare();
  if (!s.ok()) return s;
  if (n_dev_ == 0) return Status::Err(kErrQuery, "index holds no data");
  if (elem_count != (size_t)dim_)
    return Status::Err(kErrQuery, "query length " + std::to_string(elem_count) + " != index dimension " +
                                      std::to_string(dim_));
  if (method_ == METHOD_SEQ && k > (size_t)scan_exact_max_k())
    return Status::Err(kErrTooLarge, "k above " + std::to_string(scan_exact_max_k()) + " is not supported");
  if (method_ == METHOD_HNSW && k > (size_t)hnsw_max_ef()) return Status::Err(kErrTooLarge, "k too large for hnsw");

  const size_t out_n = nq * k;
  if (!(s = check_cuda(d_out_ids_.ensure(out_n * 4), "cudaMalloc(out ids)")).ok()) return s;
  if (!(s = check_cuda(d_out_dists_.ensure(out_n * 4), "cudaMalloc(out dists)")).ok()) return s;
  if (!(s = check_cuda(d_out_counts_.ensure(nq * 4), "cudaMalloc(out counts)")).ok()) return s;
  if (!(s = check_cuda(h_out_ids_.ensure(out_n * 4), "cudaMallocHost(ids)")).ok()) return s;
  if (!(s = check_cuda(h_out_dists_.ensure(out_n * 4), "cudaMallocHost(dists)")).ok()) return s;
  if (!(s = check_cuda(h_out_counts_.ensure(nq * 4), "cudaMallocHost(counts)")).ok()) return s;

  cudaEventRecord(ev_[0], stream_);
  // chunks of >= 16 K queries only: the search kernel wants a few queries per resident warp (3 552 of them),
  // four chunks of a 10 K batch ran 17.8 ms against 11.5 ms in one launch (profiles/README.md)
  const int n_chunks = (int)std::min<size_t>(kCopyChunks, nq / 16384);
  if (method_ == METHOD_HNSW && n_chunks >= 2) {
    // Graph search treats queries independently and its input is large (100 K x 960 floats = 384 MB): copy the
    // batch in chunks on a second stream and search chunk i while chunk i + 1 is still on the bus.
    const size_t bq = std::max(scan_exact_block_queries(), tc_block_queries());
    const size_t row_bytes = (size_t)row_words_ * 4, src_row = dev_u8_rows() ? elem_count : elem_count * 4;
    const size_t old_cap = d_q_.cap;
    if (!(s = check_cuda(d_q_.ensure(round_up(nq, bq) * row_bytes), "cudaMalloc(queries)")).ok()) return s;
    if (d_q_.cap != old_cap || d_q_dim_ != dim_) {
      if (!(s = check_cuda(cudaMemsetAsync(d_q_.p, 0, d_q_.cap, stream_), "memset(queries)")).ok()) return s;
      d_q_dim_ = dim_;
    }
    if (!copy_stream_) {
      if (!(s = check_cuda(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking), "cudaStreamCreate")).ok()) return s;
      for (auto& e : copy_ev_)
        if (!(s = check_cuda(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate")).ok()) return s;
    }
    cudaEventRecord(copy_ev_[kCopyChunks], stream_);  // the buffer is ready (and the previous batch is done with it)
    cudaStreamWaitEvent(copy_stream_, copy_ev_[kCopyChunks], 0);
    const size_t chunk = round_up((nq + n_chunks - 1) / n_chunks, 64);
    for (int c = 0; c < kCopyChunks; ++c) {
      const size_t c0 = std::min(nq, (size_t)c * chunk), c1 = std::min(nq, c0 + chunk);
      if (c1 > c0) {
        s = check_cuda(cudaMemcpy2DAsync(d_q_.as<char>() + c0 * row_bytes, row_bytes,
                                         static_cast<const char*>(queries) + c0 * src_row, src_row, src_row, c1 - c0,
                                         cudaMemcpyHostToDevice, copy_stream_),
                       "H2D(query chunk)");
        if (!s.ok()) return s;
      }
      cudaEventRecord(copy_ev_[c], copy_stream_);
    }
    cudaEventRecord(ev_[1], stream_);
    for (int c = 0; c < kCopyChunks; ++c) {
      const size_t c0 = std::min(nq, (size_t)c * chunk), c1 = std::min(nq, c0 + chunk);
      cudaStreamWaitEvent(stream_, copy_ev_[c], 0);
      if (c1 <= c0) continue;
      s = run(d_q_.as<char>() + c0 * row_bytes, c1 - c0, k, d_out_ids_.as<int32_t>() + c0 * k,
              d_out_dists_.as<float>() + c0 * k, nullptr, d_out_counts_.as<int32_t>() + c0, stream_);
      if (!s.ok()) return s;
    }
  } else {
    s = stage_queries_device(queries, false, nq, elem_count, stream_);
    if (!s.ok()) return s;
    cudaEventRecord(ev_[1], stream_);
    s = run(d_q_.p, nq, k, d_out_ids_.as<int32_t>(), d_out_dists_.as<float>(), nullptr, d_out_counts_.as<int32_t>(),
            stream_);
    if (!s.ok()) return s;
  }
  cudaEventRecord(ev_[2], stream_);
  if (!(s = check_cuda(cudaMemcpyAsync(h_out_ids_.p, d_out_ids_.p, out_n * 4, cudaMemcpyDeviceToHost, stream_), "D2H(ids)")).ok())
    return s;
  if (!(s = check_cuda(cudaMemcpyAsync(h_out_dists_.p, d_out_dists_.p, out_n * 4, cudaMemcpyDeviceToHost, stream_), "D2H(dists)")).ok())
    return s;
  if (!(s = check_cuda(cudaMemcpyAsync(h_out_counts_.p, d_out_counts_.p, nq * 4, cudaMemcpyDeviceToHost, stream_), "D2H(counts)")).ok())
    return s;
  cudaEventRecord(ev_[3], stream_);
  s = check_cuda(cudaStreamSynchronize(stream_), "query batch");
  if (!s.ok()) return s;
  if (sharded() && xch_take_error(xch_))
    return Status::Err(kErrQuery, "shard exchange: a peer did not publish its lists within 10 s (ranks must make the same calls)");
  float ms = 0;
  if (cudaEventElapsedTime(&ms, ev_[1], ev_[2]) == cudaSuccess) stats_.last_kernel_ms = ms;
  if (cudaEventElapsedTime(&ms, ev_[0], ev_[3]) == cudaSuccess) stats_.last_total_ms = ms;
  stats_.queries += nq;
  if (method_ == METHOD_SEQ) stats_.distance_evals += (uint64_t)nq * n_dev_;
  else {
    unsigned long long c[2] = {0, 0};
    if (cudaMemcpy(c, d_counters_.p, 16, cudaMemcpyDeviceToHost) == cudaSuccess) {
      stats_.distance_evals = c[0];
      stats_.hnsw_expansions = c[1];
    }
  }
  *ids = h_out_ids_.as<int32_t>();
  *dists = h_out_dists_.as<float>();
  *counts = h_out_counts_.as<int32_t>();
  return Status::OK();
}

}  // namespace nb200
