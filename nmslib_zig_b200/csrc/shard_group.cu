// shard_group.cu -- one process, several GPUs behind ONE index handle (SURVEY 8e, VERDICT r1 #3).
//
// An index created with the parameter b200_devices=0,1,2,3 (or "all") keeps its rows on the host as usual (the
// handle's own Engine is the host store: add / get / save work unchanged) and, at the first query, cuts them into
// contiguous row shards -- the same split the reference's multi-threaded SeqSearch makes over its threads
// (seqsearch.cc:73-85) -- one child Engine per device.  A query batch goes to all devices at once (a worker thread
// per device): every device scans its shard for ALL queries, publishes its sorted (distance, global position) lists
// into its exchange window, and finalises 1/G of the queries by merging all devices' lists over NVLink peer memory
// (exchange.cu); the slices land in one pinned result array.  An unmodified caller of nmslib_add_data_point_batch +
// nmslib_knn_query_batch therefore uses G GPUs and gets bit-identical answers to the one-GPU index.
//
// method hnsw: one graph does not shard without changing its answers (SURVEY 8e), so the group holds one REPLICA per
// device -- the graph is built (or imported) once by the handle's own engine, every replica copies the links and
// borrows the search-ready rows and ids from the host store -- and every device takes a contiguous slice of each
// batch; no exchange.  The handle's engine frees its own device copy once the graph exists.
#include <cuda_runtime.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>

#include "engine.h"
#include "shard_group.h"

namespace nb200 {

namespace {
constexpr int kErrInvalid = 2, kErrQuery = 9;

// reusable barrier for the worker threads of one group
class HostBarrier {
 public:
  explicit HostBarrier(int n) : n_(n) {}
  // false: a member of the group failed before it got here (poison) -- nobody waits for it
  bool wait() {
    std::unique_lock<std::mutex> lk(mu_);
    if (poisoned_) return false;
    const uint64_t gen = gen_;
    if (++count_ == n_) {
      count_ = 0;
      ++gen_;
      cv_.notify_all();
    } else {
      cv_.wait(lk, [&] { return gen_ != gen || poisoned_; });
    }
    return !poisoned_;
  }
  void poison() {
    std::lock_guard<std::mutex> lk(mu_);
    poisoned_ = true;
    cv_.notify_all();
  }
  void reset() {
    std::lock_guard<std::mutex> lk(mu_);
    poisoned_ = false;
    count_ = 0;
  }

 private:
  std::mutex mu_;
  std::condition_variable cv_;
  int n_, count_ = 0;
  uint64_t gen_ = 0;
  bool poisoned_ = false;
};
}  // namespace

struct ShardGroup::Impl {
  Space space;
  Method method = METHOD_SEQ;
  bool is_u8;
  std::vector<std::string> query_params;
  bool query_params_set = false;
  std::vector<int> devices;
  int active = 0;                      // shards in use (1 when the index holds fewer than two rows per device)
  std::vector<std::unique_ptr<Engine>> shards;
  std::vector<cudaEvent_t> published;  // per device: its lists of the current step are in its window
  std::unique_ptr<HostBarrier> barrier;
  // worker threads
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_job, cv_done;
  std::function<Status(int)> job;
  uint64_t job_gen = 0;
  int pending = 0;
  bool stop = false;
  std::vector<Status> results;
  // state
  uint64_t built_gen = (uint64_t)-1;
  size_t win_q = 0, win_k = 0;
  PinBuf h_ids, h_dists, h_counts, h_q;
  std::vector<std::string> index_params;
  Stats stats;

  void worker(int g) {
    cudaSetDevice(devices[g]);
    uint64_t seen = 0;
    for (;;) {
      std::function<Status(int)> fn;
      {
        std::unique_lock<std::mutex> lk(mu);
        cv_job.wait(lk, [&] { return stop || job_gen != seen; });
        if (stop) return;
        seen = job_gen;
        fn = job;
      }
      Status s;
      try {
        s = g < active ? fn(g) : Status::OK();
      } catch (const std::bad_alloc&) {
        s = Status::Err(3, "out of host memory in a shard worker");
      } catch (const std::exception& e) {
        s = Status::Err(kErrQuery, std::string("shard worker: ") + e.what());
      } catch (...) {
        s = Status::Err(kErrQuery, "shard worker: unknown error");
      }
      if (!s.ok() && barrier) barrier->poison();  // (peers waiting for this device at the exchange must not hang)
      {
        std::lock_guard<std::mutex> lk(mu);
        results[g] = s;
        if (--pending == 0) cv_done.notify_all();
      }
    }
  }
  // run fn(g) on every worker; first error wins
  Status run_all(std::function<Status(int)> fn) {
    if (barrier) barrier->reset();
    {
      std::lock_guard<std::mutex> lk(mu);
      job = std::move(fn);
      pending = (int)devices.size();
      ++job_gen;
    }
    cv_job.notify_all();
    std::unique_lock<std::mutex> lk(mu);
    cv_done.wait(lk, [&] { return pending == 0; });
    for (const Status& s : results)
      if (!s.ok()) return s;
    return Status::OK();
  }
};

ShardGroup::ShardGroup(Space space, Method method, bool is_u8, const std::vector<int>& devices) : impl_(new Impl()) {
  impl_->space = space;
  impl_->method = method;
  impl_->is_u8 = is_u8;
  impl_->devices = devices;
  impl_->results.resize(devices.size());
  impl_->active = (int)devices.size();
  impl_->published.assign(devices.size(), nullptr);
  for (size_t g = 0; g < devices.size(); ++g) impl_->workers.emplace_back([this, g] { impl_->worker((int)g); });
}

ShardGroup::~ShardGroup() {
  {
    std::lock_guard<std::mutex> lk(impl_->mu);
    impl_->stop = true;
  }
  impl_->cv_job.notify_all();
  for (auto& t : impl_->workers) t.join();
  for (size_t g = 0; g < impl_->devices.size(); ++g) {
    cudaSetDevice(impl_->devices[g]);
    if (impl_->published[g]) cudaEventDestroy(impl_->published[g]);
    if (g < impl_->shards.size()) impl_->shards[g].reset();
  }
  impl_->h_ids.release();
  impl_->h_dists.release();
  impl_->h_counts.release();
  impl_->h_q.release();
  cudaGetLastError();
  delete impl_;
}

size_t ShardGroup::world() const { return impl_->devices.size(); }

Status ShardGroup::parse_devices(const std::string& spec, std::vector<int>* out) {
  out->clear();
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) {
    cudaGetLastError();
    cnt = 0;
  }
  if (spec == "all") {
    for (int d = 0; d < cnt; ++d) out->push_back(d);
  } else {
    size_t i = 0;
    while (i <= spec.size()) {
      size_t j = spec.find_first_of(",;", i);
      if (j == std::string::npos) j = spec.size();
      const std::string tok = spec.substr(i, j - i);
      if (tok.empty()) return Status::Err(kErrInvalid, "b200_devices: empty device entry in '" + spec + "'");
      const size_t dash = tok.find('-');
      char* end = nullptr;
      if (dash != std::string::npos) {  // a range a-b
        const long a = strtol(tok.substr(0, dash).c_str(), &end, 10), b = strtol(tok.substr(dash + 1).c_str(), &end, 10);
        if (dash == 0 || a < 0 || b < a || b > 1024) return Status::Err(kErrInvalid, "b200_devices: bad range '" + tok + "'");
        for (long d = a; d <= b; ++d) out->push_back((int)d);
      } else {
        const long d = strtol(tok.c_str(), &end, 10);
        if (*end != 0 || d < 0) return Status::Err(kErrInvalid, "b200_devices: bad device '" + tok + "'");
        out->push_back((int)d);
      }
      i = j + 1;
    }
  }
  if (out->empty()) return Status::Err(kErrInvalid, "b200_devices names no device");
  if (out->size() > (size_t)kMaxShardWorld) return Status::Err(kErrInvalid, "b200_devices: at most 16 shards");
  if (cnt > 0)
    for (int d : *out)
      if (d >= cnt) return Status::Err(kErrInvalid, "b200_devices: device " + std::to_string(d) + " does not exist");
  return Status::OK();
}

void ShardGroup::set_index_params(const std::vector<std::string>& p) { impl_->index_params = p; }

Status ShardGroup::set_query_params(const std::vector<std::string>& p) {
  impl_->query_params = p;
  impl_->query_params_set = true;
  for (auto& e : impl_->shards)
    if (e) {
      std::lock_guard<std::mutex> lock(e->mutex());
      Status s = e->set_query_params(p);
      if (!s.ok()) return s;
    }
  return Status::OK();
}

// (Re)distribute the host store's rows over the devices and connect the exchange windows.
Status ShardGroup::prepare(Engine* host, size_t nq, size_t k) {
  Impl& m = *impl_;
  if (!device_available()) return Status::Err(kErrQuery, "no CUDA device available (there is no CPU fallback)");
  const size_t n_rows = host->size();
  if (m.method == METHOD_HNSW) {
    // hnsw: one graph does not shard without changing its answers (SURVEY 8e) -- every device holds a REPLICA of the
    // index (links copied, rows and ids borrowed from the host store) and takes 1/G of a batch's queries; no exchange
    if (m.built_gen == host->data_generation() && m.shards.size() == m.devices.size()) return Status::OK();
    if (n_rows == 0) return Status::Err(kErrQuery, "index holds no data");
    Status gs = host->ensure_graph();  // built once (on the device when the parameters say so), or imported
    if (!gs.ok()) return gs;
    host->release_device();            // (the handle's engine stays the host store; the replicas hold the device copies)
    // (float: the search-ready rows, cosine normalised; uint8: the host store's byte rows, which the search reads)
    const void* rows = host->is_u8() ? (const void*)host->row_u8(0) : (const void*)host->hnsw_rows_for_save();
    const size_t G = m.devices.size();
    m.shards.clear();
    m.shards.resize(G);
    m.active = (int)G;
    m.barrier.reset();
    Status s = m.run_all([&](int g) -> Status {
      std::unique_ptr<Engine> e(new Engine(m.space, METHOD_HNSW, m.is_u8, m.devices[g]));
      Status as = e->adopt_replica(host->graph(), rows, host->ext_id_ptr(0), host->dim());
      if (!as.ok()) return as;
      if (m.query_params_set && !(as = e->set_query_params(m.query_params)).ok()) return as;
      m.shards[g] = std::move(e);
      return m.shards[g]->prepare();
    });
    if (!s.ok()) return s;
    m.built_gen = host->data_generation();
    return Status::OK();
  }
  // (an index of fewer than two rows per device is served by the first device alone)
  const size_t G = n_rows >= 2 * m.devices.size() ? m.devices.size() : 1;
  const bool rebuild = m.built_gen != host->data_generation() || m.shards.size() != G;
  const bool regrow = nq > m.win_q || k > m.win_k;
  if (!rebuild && !regrow) return Status::OK();
  const size_t n = host->size();
  if (n == 0) return Status::Err(kErrQuery, "index holds no data");
  if (rebuild) {
    m.shards.clear();
    m.shards.resize(G);
    m.active = (int)G;
    m.barrier.reset(G > 1 ? new HostBarrier((int)G) : nullptr);
    Status s = m.run_all([&](int g) -> Status {
      const size_t lo = n * (size_t)g / G, hi = n * (size_t)(g + 1) / G;
      std::unique_ptr<Engine> e(new Engine(m.space, METHOD_SEQ, m.is_u8, m.devices[g]));
      if (hi > lo) {
        // no second host copy: the shard borrows rows [lo, hi) and their ids from the host store (they stay put until
        // the next add / reset, which re-cuts the shards first); positions are global (lo + local row) so that ties
        // order as on one GPU
        const void* rows = m.is_u8 ? (const void*)host->row_u8(lo) : (const void*)host->row_f32(lo);
        Status as = e->borrow_host_rows(rows, host->ext_id_ptr(lo), hi - lo, (size_t)host->dim());
        if (!as.ok()) return as;
      }
      e->set_pos_base((uint32_t)lo);
      e->mark_built(m.index_params);
      m.shards[g] = std::move(e);
      if (hi > lo) return m.shards[g]->prepare();
      return Status::OK();
    });
    if (!s.ok()) return s;
    m.built_gen = host->data_generation();
    m.win_q = m.win_k = 0;
  }
  if (G == 1) {
    m.win_q = (size_t)-1;
    m.win_k = (size_t)-1;
    return Status::OK();
  }
  // exchange windows: sized for the largest batch seen so far, then connected all-to-all
  const size_t wq = std::max(m.win_q, std::max<size_t>(nq, 1024)), wk = std::max(m.win_k, std::max<size_t>(k, 16));
  std::vector<unsigned char> blobs(G * 256);
  Status s = m.run_all([&](int g) -> Status {
    if (!m.published[g] && cudaEventCreateWithFlags(&m.published[g], cudaEventDisableTiming) != cudaSuccess)
      return Status::Err(kErrQuery, "cudaEventCreate failed");
    return m.shards[g]->shard_export(wq, wk, blobs.data() + (size_t)g * 256);
  });
  if (!s.ok()) return s;
  s = m.run_all([&](int g) -> Status {
    Status cs = m.shards[g]->shard_connect(g, (int)G, blobs.data());
    if (!cs.ok()) return cs;
    // between publish and merge: every device's publish is recorded, the host threads meet, and each stream waits
    // for all the others' events -- the merge kernels then find their flags already set (they never spin on a
    // kernel that is not yet launched, which also makes a group of several shards on ONE device legal)
    m.shards[g]->set_exchange_hook([&m, g, G](cudaStream_t st) -> Status {
      if (cudaEventRecord(m.published[g], st) != cudaSuccess) return Status::Err(kErrQuery, "cudaEventRecord failed");
      if (!m.barrier->wait()) return Status::Err(kErrQuery, "another shard of the group failed");
      for (size_t h = 0; h < G; ++h)
        if ((int)h != g && cudaStreamWaitEvent(st, m.published[h], 0) != cudaSuccess)
          return Status::Err(kErrQuery, "cudaStreamWaitEvent failed");
      return Status::OK();
    });
    return Status::OK();
  });
  if (!s.ok()) return s;
  m.win_q = wq;
  m.win_k = wk;
  return Status::OK();
}

Status ShardGroup::knn_host(Engine* host, const void* queries, size_t nq, size_t elem_count, size_t k, const int32_t** ids,
                            const float** dists, const int32_t** counts) {
  Impl& m = *impl_;
  if (!host->built()) return Status::Err(8, "Index not built");
  if (!queries || nq == 0 || k == 0) return Status::Err(kErrInvalid, "empty query batch or k == 0");
  if (elem_count != (size_t)host->dim())
    return Status::Err(kErrQuery, "query length " + std::to_string(elem_count) + " != index dimension " +
                                      std::to_string(host->dim()));
  Status s = prepare(host, nq, k);
  if (!s.ok()) return s;
  const size_t G = (size_t)m.active;
  cudaSetDevice(m.devices[0]);
  if (cudaSuccess != m.h_ids.ensure(nq * k * 4) || cudaSuccess != m.h_dists.ensure(nq * k * 4) ||
      cudaSuccess != m.h_counts.ensure(nq * 4))
    return Status::Err(3, "cudaMallocHost(results) failed");
  // queries: every device copies the batch from host memory; pageable memory is staged once into a pinned buffer so
  // that the G copies are asynchronous DMA transfers
  const size_t qbytes = nq * elem_count * (m.is_u8 ? 1 : 4);
  const void* src = queries;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, queries) != cudaSuccess || attr.type != cudaMemoryTypeHost) {
    cudaGetLastError();
    if (cudaSuccess != m.h_q.ensure(qbytes)) return Status::Err(3, "cudaMallocHost(queries) failed");
    memcpy(m.h_q.p, queries, qbytes);
    src = m.h_q.p;
  }
  if (m.method == METHOD_HNSW) {
    const size_t esz = m.is_u8 ? 1 : 4;
    s = m.run_all([&](int g) -> Status {
      const size_t q0 = nq * (size_t)g / G, q1 = nq * (size_t)(g + 1) / G;
      if (q1 <= q0) return Status::OK();
      std::lock_guard<std::mutex> lock(m.shards[g]->mutex());
      const int32_t *ri, *rc;
      const float* rd;
      Status rs = m.shards[g]->knn_host(static_cast<const char*>(src) + q0 * elem_count * esz, q1 - q0, elem_count, k, &ri, &rd, &rc);
      if (!rs.ok()) return rs;
      memcpy(m.h_ids.as<int32_t>() + q0 * k, ri, (q1 - q0) * k * 4);
      memcpy(m.h_dists.as<float>() + q0 * k, rd, (q1 - q0) * k * 4);
      memcpy(m.h_counts.as<int32_t>() + q0, rc, (q1 - q0) * 4);
      return Status::OK();
    });
    if (!s.ok()) return s;
    m.stats.queries += nq;
    *ids = m.h_ids.as<int32_t>();
    *dists = m.h_dists.as<float>();
    *counts = m.h_counts.as<int32_t>();
    return Status::OK();
  }
  s = m.run_all([&](int g) -> Status {
    const size_t q0 = nq * (size_t)g / G, q1 = nq * (size_t)(g + 1) / G;
    std::lock_guard<std::mutex> lock(m.shards[g]->mutex());
    return m.shards[g]->knn_host_slice(src, nq, elem_count, k, q0, q1, m.h_ids.as<int32_t>(), m.h_dists.as<float>(),
                                       m.h_counts.as<int32_t>());
  });
  if (!s.ok()) return s;
  m.stats.queries += nq;
  *ids = m.h_ids.as<int32_t>();
  *dists = m.h_dists.as<float>();
  *counts = m.h_counts.as<int32_t>();
  return Status::OK();
}

// Shards hold contiguous position ranges in shard order, so a query's global answer (rows within the radius in
// position order, truncated to the capacity) is the shards' answers -- each truncated to the capacity -- concatenated
// and truncated: a host step, no device exchange.
Status ShardGroup::range_host(Engine* host, const void* queries, size_t nq, size_t elem_count, const double* radii,
                              const size_t* caps, int32_t* const* ids, float* const* dists, size_t* sizes) {
  Impl& m = *impl_;
  for (size_t i = 0; i < nq; ++i) sizes[i] = 0;
  if (!host->built()) return Status::Err(8, "Index not built");
  if (m.method != METHOD_SEQ)
    return Status::Err(5, "Range query not supported by method: Range search is not supported!");
  // (the order of Engine::range_batch_host: no device is an error even for an empty index)
  if (!device_available()) return Status::Err(kErrQuery, "no CUDA device available (there is no CPU fallback)");
  if (host->size() == 0 || nq == 0) return Status::OK();
  Status s = prepare(host, 0, 0);
  if (!s.ok()) return s;
  const size_t G = (size_t)m.active;
  std::vector<size_t> off(nq + 1, 0);
  for (size_t i = 0; i < nq; ++i) off[i + 1] = off[i] + std::min(caps[i], host->size());
  std::vector<std::vector<int32_t>> sid(G, std::vector<int32_t>(off[nq]));
  std::vector<std::vector<float>> sd(G, std::vector<float>(off[nq]));
  std::vector<std::vector<size_t>> ssz(G, std::vector<size_t>(nq));
  s = m.run_all([&](int g) -> Status {
    std::vector<int32_t*> pi(nq);
    std::vector<float*> pd(nq);
    std::vector<size_t> c(nq);
    for (size_t i = 0; i < nq; ++i) {
      pi[i] = sid[g].data() + off[i];
      pd[i] = sd[g].data() + off[i];
      c[i] = off[i + 1] - off[i];
    }
    std::lock_guard<std::mutex> lock(m.shards[g]->mutex());
    return m.shards[g]->range_batch_host(queries, nq, elem_count, radii, c.data(), pi.data(), pd.data(), ssz[g].data());
  });
  if (!s.ok()) return s;
  for (size_t i = 0; i < nq; ++i) {
    size_t at = 0;
    for (size_t g = 0; g < G && at < caps[i]; ++g) {
      const size_t take = std::min(ssz[g][i], caps[i] - at);
      memcpy(ids[i] + at, sid[g].data() + off[i], take * 4);
      memcpy(dists[i] + at, sd[g].data() + off[i], take * 4);
      at += take;
    }
    sizes[i] = at;
  }
  m.stats.queries += nq;
  return Status::OK();
}

Stats ShardGroup::stats() {
  Stats out = impl_->stats;
  for (auto& e : impl_->shards) {
    if (!e) continue;
    std::lock_guard<std::mutex> lock(e->mutex());
    const Stats s = e->stats();
    out.kernel_launches += s.kernel_launches;
    out.distance_evals += s.distance_evals;
    out.hnsw_expansions += s.hnsw_expansions;
    out.fallback_queries += s.fallback_queries;
    out.split_queries += s.split_queries;
    out.range_tc_queries += s.range_tc_queries;
    out.range_fallback_queries += s.range_fallback_queries;
    out.device_bytes += s.device_bytes;
    out.uploaded_rows += s.uploaded_rows;
    out.last_scan_ms = std::max(out.last_scan_ms, s.last_scan_ms);
    out.scan_ms_sum += s.scan_ms_sum;
    out.scan_count += s.scan_count;
    out.last_kernel_ms = std::max(out.last_kernel_ms, s.last_kernel_ms);
  }
  return out;
}

}  // namespace nb200
