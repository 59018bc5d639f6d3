// engine.h -- host side of the nmslib_b200 query engine (one Engine per index handle).
//
// The Engine owns the host copy of the data set (what the reference keeps as an
// ObjectVector, nmslib_c.cpp:146), its HBM-resident mirror, the optional HNSW graph and
// the per-batch scratch, and turns one nmslib_knn_query_batch call into ONE device
// submission: H2D queries -> kernels -> D2H (id, distance) lists.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace nb200 {

enum Method : int { METHOD_SEQ = 0, METHOD_HNSW = 1 };

struct Status {
  int code = 0;  // nmslib_error_t value
  std::string msg;
  bool ok() const { return code == 0; }
  static Status OK() { return Status(); }
  static Status Err(int c, std::string m) {
    Status s;
    s.code = c;
    s.msg = std::move(m);
    return s;
  }
};

// growable device / pinned-host buffers
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool borrowed = false;  // memory owned by someone else (hnsw_build_gpu.cu scans the rows of the index in place)
  cudaError_t ensure(size_t bytes, bool zero_new = false, cudaStream_t s = nullptr);
  cudaError_t ensure_keep(size_t bytes, cudaStream_t s);  // grow, contents preserved
  void borrow(void* ptr, size_t bytes);
  void release();
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};
struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes);
  void release();
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// The host store of an index: one slab per element type, grown geometrically, filled by several threads for large
// batches (a 10 M x 768 ingest is 30 GB of first-touch page faults: one thread manages ~2 GB/s of that).  Replaces
// the reference's per-point `new Object` + memcpy (nmslib_c.cpp:228-291, 755-871).
template <typename T>
class HostSlab {
 public:
  HostSlab() = default;
  ~HostSlab() { free(p_); }
  HostSlab(const HostSlab&) = delete;
  HostSlab& operator=(const HostSlab&) = delete;
  const T* data() const { return p_; }
  T* data() { return p_; }
  size_t size() const { return n_; }
  bool empty() const { return n_ == 0; }
  void clear() {
    free(p_);
    p_ = nullptr;
    n_ = cap_ = 0;
  }
  bool append(const T* src, size_t count);             // false: out of memory
  bool assign(const T* src, size_t count) {
    clear();
    return append(src, count);
  }

 private:
  T* p_ = nullptr;
  size_t n_ = 0, cap_ = 0;
};

// Host image of the reference's optimized HNSW index (hnsw.cc:774-806; SURVEY Appendix B)
struct HnswGraph {
  uint32_t total = 0;
  int dim = 0;
  int maxM = 0, maxM0 = 0, maxlevel = 0;  // maxlevel: the level the greedy descent starts at
  int M = 0;                              // index-time M (builders, regular files; the optimized stream has none)
  int file_maxlevel = -1;                 // a regular file's maxlevel_ where it exceeds the entry node's level
  uint32_t enterpoint = 0;
  int dist_func = 0;  // 1 L2Sqr16Ext, 2 L2SqrExt, 3 NormCosine, 4 NegativeDotProduct
  std::vector<float> vectors;      // [total][dim] (cosine: unit norm)
  std::vector<int32_t> ext_ids;    // [total]
  std::vector<int32_t> links0;     // [total][maxM0]
  std::vector<int32_t> links0_cnt; // [total]
  std::vector<int32_t> upper;      // concatenated raw upper-level lists
  std::vector<int64_t> upper_off;  // [total], -1 = level 0 only
  std::vector<int32_t> levels;     // [total] top level of every node
  bool empty() const { return total == 0; }
};
Status read_hnsw_file(const std::string& path, HnswGraph* out);
// The reference's regular index file (Hnsw::SaveRegularIndexBin, hnsw.cc:810-842), what Hnsw<int> (l2sqr_sift) saves:
// links only, read back by read_hnsw_file.  Needs M and levels.
Status write_regular(const std::string& path, const HnswGraph& g);
// vectors / ext_ids: [total][dim] and [total] (the Engine keeps them outside the graph)
// host-side graph construction (hnsw_build.cpp): rows are float32 (cosine: unit-normalised)
Status build_hnsw_host(const float* rows, size_t n, int dim, int dist_func, const int32_t* ext_ids,
                       const std::vector<std::string>& params, HnswGraph* out);
Status write_hnsw_file(const std::string& path, const HnswGraph& g, const float* vectors,
                       const int32_t* ext_ids);

// index-time parameters of Hnsw::CreateIndex (hnsw.cc:185-205) + where to build (b200_build=auto|host|device)
struct HnswBuildParams {
  int M = 16, efConstruction = 200, maxM = 16, maxM0 = 32, delaunay_type = 2, threads = 0;
  double mult = 0;
  int where = -1;  // -1 auto (device for >= 16384 points when a GPU is present), 0 host, 1 device
};
bool parse_hnsw_build_params(const std::vector<std::string>& params, HnswBuildParams* bp, std::string* err);
std::vector<int> hnsw_assign_levels(size_t n, double mult);  // getRandomLevel (hnsw.h:476-480), seed 0 (init.cc:34)
struct HnswBuildInfo {
  double scan_ms = 0, select_ms = 0, link_ms = 0, total_ms = 0;
  double setup_ms = 0, reserve_ms = 0, download_ms = 0;  // host wall clock: scan engine set-up, scratch sizing, D2H
  int batches = 0, levels = 0;
  uint64_t reverse_edges = 0, prunes = 0;
};
// device-side graph construction (hnsw_build_gpu.cu): d_rows = [n_pad][row_words] float rows already in HBM
// (cosine: unit-normalised), n_pad = n rounded up to 128 rows.  The graph comes back as a host image.
Status build_hnsw_device(const float* d_rows, size_t n, int dim, int row_words, int dist_func, const int32_t* ext_ids,
                         const HnswBuildParams& bp, int device, HnswGraph* out, HnswBuildInfo* info);

// ---- cross-shard exchange over peer memory (exchange.cu) ----
constexpr int kMaxShardWorld = 16;
struct PeerExchange;
Status xch_export(PeerExchange** out, int device, size_t max_q, size_t max_k, void* blob256);
Status xch_connect(PeerExchange* x, int rank, int world, const void* blobs);
void xch_destroy(PeerExchange* x);
bool xch_connected(const PeerExchange* x);
int xch_world(const PeerExchange* x);
int xch_rank(const PeerExchange* x);
Status xch_publish(PeerExchange* x, const uint64_t* local_keys, const int32_t* ext_ids, uint32_t pos_base, size_t nq, size_t k,
                   cudaStream_t stream);
Status xch_merge(PeerExchange* x, size_t k, int finalize, size_t q_begin, size_t q_count, uint64_t* out_keys,
                 int32_t* out_ids, float* out_dists, int32_t* out_counts, cudaStream_t stream);
bool xch_take_error(PeerExchange* x);

struct Stats {
  uint64_t queries = 0, kernel_launches = 0, distance_evals = 0, hnsw_expansions = 0;
  double last_kernel_ms = 0, last_total_ms = 0, last_scan_ms = 0, scan_ms_sum = 0;
  uint64_t scan_count = 0;
  uint64_t fallback_queries = 0, device_bytes = 0, split_queries = 0, uploaded_rows = 0;
  // batched range queries (range_batch_host): answered by the tensor-core pass / re-run by the per-query exact scan
  // after an uncertified batched pass
  uint64_t range_tc_queries = 0, range_fallback_queries = 0;
};

class Engine {
 public:
  Engine(Space space, Method method, bool is_u8, int device);
  ~Engine();

  // ---- ingest (host copy) ----
  Status add_rows(const void* rows, size_t count, size_t elem_count, const int32_t* ids);
  Status add_row_ptrs(const void* const* ptrs, size_t count, size_t elem_count, const int32_t* ids);
  void reset();
  size_t size() const { return n_; }
  int dim() const { return dim_; }
  bool is_u8() const { return is_u8_; }
  Space space() const { return space_; }
  Method method() const { return method_; }
  const float* row_f32(size_t pos) const { return base_f32() + pos * (size_t)dim_; }
  const uint8_t* row_u8(size_t pos) const { return base_u8() + pos * (size_t)dim_; }
  int32_t ext_id(size_t pos) const { return base_ids()[pos]; }
  const int32_t* ext_id_ptr(size_t pos) const { return base_ids() + pos; }
  // A shard of a ShardGroup does not copy its rows: it borrows [lo, hi) of the group's host store (rows and ids stay
  // valid until the group re-cuts its shards, which drops this engine first)
  Status borrow_host_rows(const void* rows, const int32_t* ids, size_t count, size_t elem_count);
  float host_distance(size_t a, size_t b) const;  // Space::IndexTimeDistance (space.h:136-142)

  // ---- index state ----
  void mark_built(const std::vector<std::string>& index_params);
  bool built() const { return built_; }
  Status set_query_params(const std::vector<std::string>& params);  // hnsw.cc:474-507
  Status import_graph(const std::string& path);
  Status adopt_graph(HnswGraph&& g);
  // replica of another engine's hnsw index (ShardGroup): a copy of the links over BORROWED search-ready rows
  // (float: hnsw_rows_for_save(), cosine already unit-normalised; uint8: the host store's byte rows) and ids
  Status adopt_replica(const HnswGraph& g, const void* search_rows, const int32_t* ids, int dim);
  void release_device();  // frees every device buffer; the next prepare() uploads again
  const HnswGraph& graph() const { return graph_; }
  const float* hnsw_rows_for_save() { return hnsw_host_rows(); }  // float spaces (uint8 graphs save no rows)
  void set_pos_base(uint32_t b) { pos_base_ = b; }
  Status prepare();  // lazy upload; idempotent
  Status ensure_graph_host();  // hnsw: build the graph on the host if none was imported (no GPU needed)
  Status ensure_graph();       // hnsw: build it where the index parameters say (device when one is present)
  const HnswBuildInfo& build_info() const { return build_info_; }
  // ---- internal users (hnsw_build_gpu.cu): a seq_search engine over rows that already live in HBM ----
  Status adopt_device_rows(const float* d_rows, size_t n, int dim, int row_words);
  void set_scan_rows(size_t n) { n_dev_ = n < n_ ? n : n_; }  // scan only the first n rows (prefix kNN)
  void set_approx_ok(bool v) { approx_ok_ = v; }              // keep uncertified tensor-core answers (no exact re-run)
  void set_dry_run(bool v) { dry_run_ = v; }                  // size every scratch buffer of a batch shape, launch nothing

  // ---- queries ----
  // host in / host out: ids/dists are [nq][k] staging arrays owned by the engine
  Status knn_host(const void* queries, size_t nq, size_t elem_count, size_t k, const int32_t** ids,
                  const float** dists, const int32_t** counts);
  // range query of one object (seq_search only, like the reference): ids/dists are caller buffers of `capacity`
  Status range_host(const void* query, size_t elem_count, double radius, size_t capacity, int32_t* ids, float* dists,
                    size_t* size);
  // a batch of range queries: for every i the answer range_host gives with radii[i] and caps[i], written to the
  // caller buffers ids[i] / dists[i] (caps[i] entries), sizes[i] = entries written
  Status range_batch_host(const void* queries, size_t nq, size_t elem_count, const double* radii, const size_t* caps,
                          int32_t* const* ids, float* const* dists, size_t* sizes);
  // device in / device out
  // src_pitch: bytes between query rows (0 = dense rows of elem_count elements)
  Status knn_device(const void* d_queries, size_t nq, size_t elem_count, size_t k, int32_t* d_ids,
                    float* d_dists, uint64_t* d_keys, int32_t* d_counts, cudaStream_t stream, size_t src_pitch = 0);

  // ---- row-sharded search: this engine is rank `rank` of `world` (exchange.cu).  Once connected, every knn call
  // returns the GLOBAL top-k (all ranks' lists merged); merge_slice restricts the finalised rows to [q0, q1) of the
  // batch (a ShardGroup lets device g finalise slice g only).
  Status shard_export(size_t max_q, size_t max_k, void* blob256);
  Status shard_connect(int rank, int world, const void* blobs);
  void shard_disconnect();
  bool sharded() const { return xch_connected(xch_); }
  void set_merge_slice(size_t q0, size_t q1) { slice_q0_ = q0; slice_q1_ = q1; }
  // called between publish and merge with the engine's stream (ShardGroup: the devices of one process meet at a host
  // barrier and order their streams with events, so no kernel of the group ever spins on a kernel not yet launched)
  void set_exchange_hook(std::function<Status(cudaStream_t)> h) { xch_hook_ = std::move(h); }
  // host in, host out for the rows [q0, q1) this rank finalises: h_* are [nq][k] / [nq] pinned arrays shared by a group
  Status knn_host_slice(const void* queries, size_t nq, size_t elem_count, size_t k, size_t q0, size_t q1,
                        int32_t* h_ids, float* h_dists, int32_t* h_counts);
  uint64_t data_generation() const { return data_gen_; }

  Stats stats();  // also resolves the dominant-kernel event pair if it has completed
  int device() const { return device_; }
  std::mutex& mutex() { return mu_; }
  size_t ef() const { return ef_; }
  int finalize_kind() const;
  // uint8 + seq_search normally runs on the tensor cores: rows widened to fp32 on upload (0..255 is TF32-exact
  // and every partial sum stays an integer below 2^24, so the fp32 pipeline returns the int32 distances bit
  // for bit).  NB200_FORCE_EXACT=1 keeps the byte rows and the dp4a scan (K2) instead.
  // Default since round 2: BYTE rows on the integer tensor pipe (tcgen05.mma.kind::i8, tc_scan_u8_kernel) when the
  // rows' norms fit its digit block; the widened TF32 path remains for data beyond that and as option u8_imma=0.
  // uint8 + hnsw always keeps byte rows: the beam search evaluates them with dp4a (hnsw_search.cu, dist_kind 3).
  bool dev_u8_rows() const { return is_u8_ && (method_ == METHOD_HNSW || force_exact_ || u8_imma_); }
  bool u8_widened() const { return is_u8_ && method_ == METHOD_SEQ && !force_exact_ && !u8_imma_; }
  bool u8_imma() const { return u8_imma_; }

 private:
  Status check_cuda(cudaError_t e, const char* what);
  const float* hnsw_host_rows();
  Status upload_data();
  Status upload_graph();
  // d_nq: the query count lives on the device (<= nq): kernels are launched for nq and leave early past *d_nq
  Status run_seq_exact(const void* dq, size_t nq, size_t k, uint64_t* out_keys, cudaStream_t stream,
                       const int* d_nq = nullptr);
  // async: no host round trip -- uncertified queries are listed and re-run exactly by device-predicated launches, the
  // count reaches the host later (stats / adaptation of the next batches); !async (host entry, which synchronises
  // anyway): the host reads the certificates and can re-run a mostly-failed batch with split operands at once
  Status run_seq_tc(const void* dq, size_t nq, size_t k, uint64_t* out_keys, cudaStream_t stream,
                    bool allow_split_retry = true, bool async = false);
  void absorb_async_counts(bool wait);
  Status enable_split(cudaStream_t stream);
  Status run(const void* d_queries_padded, size_t nq, size_t k, int32_t* d_ids, float* d_dists,
             uint64_t* d_keys, int32_t* d_counts, cudaStream_t stream, bool async = false);
  Status stage_queries_device(const void* src, bool src_on_device, size_t nq, size_t elem_count,
                              cudaStream_t stream, size_t src_pitch = 0);
  Status build_graph_device();
  int range_mode() const;  // distance code of range_scan.cu for this index
  // one chunk of range_batch_host: queries [0, nq) of `queries`, per-query float radii / capacities (<= n)
  Status range_chunk(const void* queries, size_t nq, size_t elem_count, const float* radii, const int* caps,
                     int32_t* const* ids, float* const* dists, size_t* sizes);

  Space space_;
  Method method_;
  bool is_u8_;
  int device_;
  int dim_ = 0;        // elements per vector
  int d_q_dim_ = -1;   // dim_ the staged-query buffer d_q_ was last zeroed for
  int row_words_ = 0;  // padded 32-bit words per device row
  uint32_t pos_base_ = 0;
  size_t n_ = 0;
  bool built_ = false;
  bool data_dirty_ = true, graph_dirty_ = true;
  bool upload_valid_ = false;  // rows [0, n_up_) are in HBM in the layout of up_row_words_ (append-only uploads)
  size_t n_up_ = 0;
  int up_row_words_ = 0;
  std::vector<std::string> index_params_;
  size_t ef_ = 200;  // nmslib_c.cpp:330 default through the C ABI
  bool ef_user_set_ = false;

  HostSlab<float> h_f32_;
  HostSlab<uint8_t> h_u8_;
  std::vector<int32_t> h_ids_;
  const void* borrowed_rows_ = nullptr;    // set by borrow_host_rows: the rows / ids live in another engine's host store
  const int32_t* borrowed_ids_ = nullptr;
  bool replica_rows_ = false;              // adopt_replica: borrowed_rows_ are the search-ready rows of an hnsw replica
  const float* base_f32() const { return borrowed_rows_ ? static_cast<const float*>(borrowed_rows_) : h_f32_.data(); }
  const uint8_t* base_u8() const { return borrowed_rows_ ? static_cast<const uint8_t*>(borrowed_rows_) : h_u8_.data(); }
  const int32_t* base_ids() const { return borrowed_ids_ ? borrowed_ids_ : h_ids_.data(); }
  std::vector<float> h_hnsw_rows_;  // float rows for hnsw: cosine normalised; uint8 widened while the host builds
  bool rows_normalized_ = false;
  HnswGraph graph_;

  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_[4] = {nullptr, nullptr, nullptr, nullptr};
  // ring of (start, stop) event pairs around the dominant kernel; resolved lazily in stats()
  static constexpr int kScanRing = 64;
  cudaEvent_t scan_ev_[kScanRing][2] = {};
  bool scan_pending_[kScanRing] = {};
  int scan_head_ = 0;
  int scan_cur_ = 0;
  void scan_begin(cudaStream_t s);
  void scan_end(cudaStream_t s);
  DevBuf d_db_, d_aux_, d_ids_;
  // tensor-core scan operands / scratch
  static constexpr int kCopyChunks = 4;  // query chunks of a large HNSW batch (copy / search overlap)
  cudaStream_t copy_stream_ = nullptr;
  cudaEvent_t copy_ev_[kCopyChunks + 1] = {};
  DevBuf d_range_;                      // per-row distances of a range query + its outputs
  // batched range queries: per-query parameters + CSR outputs, and the range-mode candidate lists of the scan
  DevBuf d_rq_, d_rq_out_, d_rcand_, d_rcnt_, d_rcut_, d_rthr_, d_rplan_;
  std::vector<int> h_rplan_;
  DevBuf d_u8tmp_;                      // staging for uint8 rows / queries before they are widened
  DevBuf d_gthr_;                       // per-query threshold shared by the CTAs of one scan
  bool db_inexact_ = false;             // the uploaded rows are not TF32-exact (read back once at upload)
  int tc_margin_ = 6;                   // survivors per compaction = k + margin (doubles when certificates fail)
  DevBuf d_plan_;                       // piece table of the TS scan (tc_ts_plan), cached per (nq, n, k)
  std::vector<int> h_plan_;
  size_t plan_key_[4] = {0, 0, 0, 0};
  bool tc_split_ = false;               // 3xTF32: operands split into TF32-exact halves (see run_seq_tc)
  DevBuf d_db_split_, d_q_split_, d_sp_idx_, d_sp_q_, d_sp_keys_;
  int plan_n_cta_ = 0, plan_s_max_ = 0;
  std::vector<int> plan_block_slots_;   // pieces per query block of the cached plan
  DevBuf d_bias_, d_db_unit_, d_flags_, d_qa_, d_cand_, d_cand_cnt_, d_cand_thr_, d_tc_keys_, d_cert_, d_fb_idx_,
      d_fb_q_, d_fb_keys_, d_nblock_, d_ones_;
  PinBuf h_cert_;
  // device-predicated re-run of uncertified queries (knn_device): count + index list on the device, the count is
  // copied to a ring of pinned words and absorbed into the statistics / the adaptation later
  DevBuf d_fb_cnt_;
  static constexpr int kFbRing = 16;
  PinBuf h_fb_cnt_;
  cudaEvent_t fb_ev_[kFbRing] = {};
  size_t fb_nq_[kFbRing] = {};
  bool fb_pending_[kFbRing] = {};
  int fb_head_ = 0;
  float x_max_ = 0.f;
  bool force_exact_ = false;
  bool u8_imma_ = false;   // uint8 + seq_search on the integer tensor pipe (decided at upload from the rows' norms)
  int u8_m_half_ = 0;      // M = ceil(max |x|^2 / 2) of the uploaded rows
  DevBuf d_digits_;        // [n_pad][32] norm digits (scan_tc.cu: u8_norm_digits_kernel)
  DevBuf d_glists_;        // exact scan with k > 144: the blocks' sorted lists (scan_exact.cu)
  bool approx_ok_ = false, rows_borrowed_ = false, dry_run_ = false;
  HnswBuildInfo build_info_;
  size_t n_dev_ = 0;
  DevBuf d_links0_, d_links0_cnt_, d_upper_, d_upper_off_, d_visited_, d_epoch_, d_counters_;
  int hnsw_slots_ = 0;
  DevBuf d_q_, d_qaux_, d_partial_, d_keys_, d_out_ids_, d_out_dists_, d_out_counts_;
  PinBuf h_out_ids_, h_out_dists_, h_out_counts_, h_q_;
  // large uploads: pinned staging, kStageThreads host threads x 2 buffers each, one copy stream per thread
  static constexpr int kStageThreads = 4;
  static constexpr size_t kStageBytes = 4u << 20;  // (pinning memory is slow, ~0.5 GB/s: 32 MB in all)
  PinBuf h_stage_;
  cudaStream_t stage_stream_[kStageThreads] = {};
  cudaEvent_t stage_ev_[kStageThreads][2] = {};
  cudaEvent_t stage_ready_ = nullptr;
  Status upload_rows(char* dst, size_t dst_pitch, const char* src, size_t src_row, size_t rows);
  Stats stats_;
  PeerExchange* xch_ = nullptr;
  std::function<Status(cudaStream_t)> xch_hook_;
  uint64_t data_gen_ = 0;
  size_t slice_q0_ = 0, slice_q1_ = (size_t)-1;
  std::mutex mu_;
  int sm_count_ = 148;
};

int default_device();
void set_default_device(int d);
bool device_available();

}  // namespace nb200
