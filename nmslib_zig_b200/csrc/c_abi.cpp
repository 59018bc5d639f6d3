// c_abi.cpp -- the extern "C" boundary of libnmslib_b200.so (include/nmslib_b200.h).
//
// Mirrors the observable behaviour of the reference shim nmslib_c.cpp for the dense
// query path: same symbols, argument meaning, ownership rules and error codes
// (citations on each function), with the query dispatch replaced by nb200::Engine.
// No exception crosses the boundary; details go to a thread-local record
// (ref nmslib_c.cpp:36-41) readable through nmslib_get_last_error_detail.
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nmslib_b200.h"
#include "engine.h"
#include "shard_group.h"

using nb200::Engine;
using nb200::Status;

namespace {

struct LastError {
  nmslib_error_t code = NMSLIB_SUCCESS;
  std::string message = "No error";
  std::string file = __FILE__;
  int line = 0;
};
thread_local LastError g_last;

nmslib_error_t set_err(nmslib_error_t code, const std::string& msg, int line) {
  g_last.code = code;
  g_last.message = msg.empty() ? "No error" : msg;
  g_last.file = __FILE__;
  g_last.line = line;
  return code;
}
#define NB_ERR(code, msg) set_err((code), (msg), __LINE__)
#define NB_OK(msg) set_err(NMSLIB_SUCCESS, (msg), __LINE__)
#define NB_STATUS(st) set_err(static_cast<nmslib_error_t>((st).code), (st).msg, __LINE__)

bool alloc_ok(const nmslib_allocator_t* a) { return a && a->alloc && a->free; }

char* dup_string(const std::string& s, const nmslib_allocator_t* a) {  // ref nmslib_c.cpp:64-71
  char* r = static_cast<char*>(a->alloc(s.size() + 1, a->ctx));
  if (!r) return nullptr;
  memcpy(r, s.c_str(), s.size() + 1);
  return r;
}

template <typename F>
nmslib_error_t guarded(F&& f, nmslib_error_t on_throw, const char* what) {
  try {
    return f();
  } catch (const std::bad_alloc& e) {
    return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, std::string(what) + ": " + e.what());
  } catch (const std::exception& e) {
    return NB_ERR(on_throw, std::string(what) + ": " + e.what());
  } catch (...) {
    return NB_ERR(on_throw, std::string(what) + ": unknown error");
  }
}

bool parse_space(const std::string& s, nb200::Space* out) {
  if (s == "l2") *out = nb200::SPACE_L2;
  else if (s == "l2sqr") *out = nb200::SPACE_L2SQR;  // new first-class space (SURVEY Q5)
  else if (s == "cosinesimil" || s == "cosine") *out = nb200::SPACE_COSINE;
  else if (s == "negdotprod") *out = nb200::SPACE_NEGDOT;
  else if (s == "l2sqr_sift") *out = nb200::SPACE_L2SQR_SIFT;
  else if (s == "l1") *out = nb200::SPACE_L1;
  else if (s == "linf") *out = nb200::SPACE_LINF;
  else if (s == "angulardist") *out = nb200::SPACE_ANGULAR;
  else return false;
  return true;
}

}  // namespace

// The index object.  Like the reference's nmslib_internal_index_t (nmslib_c.cpp:136-172) the
// {data_type, dist_type} header is the first field and the object lives in memory obtained
// from the caller's allocator.
struct nmslib_index_t {
  nmslib_index_header_t header;
  Engine* engine;             // the index itself; with a shard group: the host store of the rows
  nb200::ShardGroup* group;   // index parameter b200_devices: row shards on several GPUs of this process
  std::string method;
  std::string space_type;
  nmslib_allocator_t allocator;
  size_t thread_pool_size;
  bool method_served;
};

struct nmslib_params_t {  // ref nmslib_params_wrapper_t, nmslib_c.cpp:131-134
  std::vector<std::string> params;
  nmslib_allocator_t allocator;
};

namespace {
const std::vector<std::string>& params_of(nmslib_params_handle_t p) {
  static const std::vector<std::string> empty;
  return p ? p->params : empty;
}

nmslib_error_t new_index(const std::string& space, const std::string& method, nmslib_data_type_t data_type,
                         nmslib_dist_type_t dist_type, const nmslib_allocator_t* allocator,
                         nmslib_index_handle_t* out) {
  nb200::Space sp;
  if (!parse_space(space, &sp))
    return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE,
                  "space '" + space + "' is outside the B200 dense-vector path (it stays on the reference CPU code)");
  const bool u8 = sp == nb200::SPACE_L2SQR_SIFT;
  if ((u8 && data_type != NMSLIB_DATATYPE_DENSE_UINT8_VECTOR) || (!u8 && data_type != NMSLIB_DATATYPE_DENSE_VECTOR))
    return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "data type does not match space '" + space + "'");
  void* mem = allocator->alloc(sizeof(nmslib_index_t), allocator->ctx);
  if (!mem) return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate index");
  nmslib_index_t* idx = new (mem) nmslib_index_t();
  idx->header.data_type = data_type;
  idx->header.dist_type = dist_type;
  idx->method = method;
  idx->space_type = space;
  idx->allocator = *allocator;
  idx->thread_pool_size = std::thread::hardware_concurrency();
  nb200::Method m = nb200::METHOD_SEQ;
  idx->method_served = true;
  if (method == "hnsw") m = nb200::METHOD_HNSW;
  else if (method != "seq_search" && method != "brute_force") idx->method_served = false;
  // l1 / linf / angulardist are served by the exact scan only (the optimized HNSW index knows l2 / cosine / negdot)
  if (m == nb200::METHOD_HNSW && (sp == nb200::SPACE_L1 || sp == nb200::SPACE_LINF || sp == nb200::SPACE_ANGULAR))
    idx->method_served = false;
  idx->engine = new Engine(sp, m, u8, nb200::default_device());
  idx->group = nullptr;
  *out = idx;
  return NB_OK("Index created");
}
}  // namespace

extern "C" {

void nmslib_init(void) {}  // no global registries to initialise

nmslib_error_t nmslib_index_create(const char* space, nmslib_params_handle_t /*space_params*/, const char* method,
                                   nmslib_data_type_t data_type, nmslib_dist_type_t dist_type,
                                   const nmslib_allocator_t* allocator, nmslib_index_handle_t* out_handle) {
  if (!space || !method || !alloc_ok(allocator) || !out_handle)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid arguments");
  // space params are ignored by the l2 / cosine / negdot creators of the reference as well
  // (factory/space/space_lp.h:38-40, space_scalar.h:27-43).
  return guarded([&] { return new_index(space, method, data_type, dist_type, allocator, out_handle); },
                 NMSLIB_ERROR_RUNTIME, "Failed to create index");
}

void nmslib_index_destroy(nmslib_index_handle_t handle) {
  if (!handle) return;
  nmslib_allocator_t a = handle->allocator;
  delete handle->group;
  delete handle->engine;
  handle->~nmslib_index_t();
  a.free(handle, a.ctx);
}

nmslib_error_t nmslib_create_index(nmslib_index_handle_t index, nmslib_params_handle_t index_params,
                                   int /*print_progress*/) {
  if (!index) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  return guarded(
      [&]() -> nmslib_error_t {
        if (!index->method_served)
          return NB_ERR(NMSLIB_ERROR_INDEX_BUILD_FAILED,
                        "method '" + index->method + "' is not served by the B200 engine (seq_search, brute_force, hnsw)");
        // AnyParamManager::CheckUnused throws on unknown names (params.h:241-251) -> error 8
        static const char* seq_names[] = {"copyMem", "multiThread", "threadQty",  // seqsearch.cc:63-68
                                          "b200_devices"};  // + row shards over several GPUs (extension)
        static const char* hnsw_names[] = {"M", "efConstruction", "maxM", "maxM0", "mult", "delaunay_type", "post",
                                           "indexThreadQty", "skip_optimized_index", "searchMethod",
                                           "b200_build",     // hnsw.cc:189-208 + where to build (extension)
                                           "b200_devices"};  // + replicas on several GPUs, queries split (extension)
        for (const std::string& p : params_of(index_params)) {
          const std::string name = p.substr(0, p.find('='));
          bool known = false;
          if (index->engine->method() == nb200::METHOD_SEQ) {
            for (const char* n : seq_names) known |= name == n;
          } else {
            for (const char* n : hnsw_names) known |= name == n;
          }
          if (!known)
            return NB_ERR(NMSLIB_ERROR_INDEX_BUILD_FAILED, "Failed to create index: unknown parameter '" + name + "'");
        }
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        std::vector<std::string> kept;
        std::string devices;
        for (const std::string& p : params_of(index_params)) {
          if (p.compare(0, 13, "b200_devices=") == 0) devices = p.substr(13);
          else kept.push_back(p);
        }
        delete index->group;
        index->group = nullptr;
        if (!devices.empty()) {
          std::vector<int> devs;
          Status ds = nb200::ShardGroup::parse_devices(devices, &devs);
          if (!ds.ok()) return NB_ERR(NMSLIB_ERROR_INDEX_BUILD_FAILED, "Failed to create index: " + ds.msg);
          if (devs.size() > 1) {
            index->group = new nb200::ShardGroup(index->engine->space(), index->engine->method(), index->engine->is_u8(), devs);
            index->group->set_index_params(kept);
          }
        }
        index->engine->mark_built(kept);
        return NB_OK("Index created successfully");
      },
      NMSLIB_ERROR_INDEX_BUILD_FAILED, "Failed to create index");
}

nmslib_error_t nmslib_reset_index(nmslib_index_handle_t index) {
  if (!index) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  index->engine->reset();
  return NB_OK("Index reset successfully");
}

// Reference: rebuilds the HNSW graph on every call (nmslib_c.cpp:1682-1704, SURVEY 0.6).
// Here: "make sure the device copy exists"; failures surface at the query call.
void nmslib_initialize_pool(nmslib_index_handle_t index) {
  if (!index || !index->engine->built()) return;
  if (index->group) {  // shards are cut (and uploaded) here, like the single-device copy below
    try {
      std::lock_guard<std::mutex> lock(index->engine->mutex());
      Status s = index->group->prepare(index->engine, 1, 1);
      if (!s.ok()) NB_STATUS(s);
    } catch (...) {
    }
    return;
  }
  try {
    std::lock_guard<std::mutex> lock(index->engine->mutex());
    Status s = index->engine->prepare();
    if (!s.ok()) NB_STATUS(s);
  } catch (...) {
  }
}

nmslib_params_handle_t nmslib_create_params(const nmslib_allocator_t* allocator) {
  if (!alloc_ok(allocator)) {
    NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid allocator");
    return nullptr;
  }
  void* mem = allocator->alloc(sizeof(nmslib_params_t), allocator->ctx);
  if (!mem) {
    NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate memory for params");
    return nullptr;
  }
  nmslib_params_t* p = new (mem) nmslib_params_t();
  p->allocator = *allocator;
  NB_OK("Parameters created successfully");
  return p;
}

nmslib_error_t nmslib_add_param(nmslib_params_handle_t params, const char* name, int type, const void* value) {
  if (!params || !name || !value) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid arguments");
  return guarded(
      [&]() -> nmslib_error_t {
        std::string p = std::string(name) + "=";
        switch (type) {  // ref nmslib_c.cpp:576-589
          case 0: p += std::to_string(*static_cast<const int*>(value)); break;
          case 1: p += std::to_string(*static_cast<const double*>(value)); break;
          case 2: p += static_cast<const char*>(value); break;
          default: return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid parameter type");
        }
        params->params.push_back(p);
        return NB_OK("Parameter added successfully");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to add parameter");
}

void nmslib_free_params(nmslib_params_handle_t params) {
  if (!params || !params->allocator.free) {
    NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid params or allocator");
    return;
  }
  nmslib_allocator_t a = params->allocator;
  params->~nmslib_params_t();
  a.free(params, a.ctx);
}

nmslib_error_t nmslib_set_query_time_params(nmslib_index_handle_t index, nmslib_params_handle_t params) {
  if (!index) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  if (!index->engine->built()) return NB_ERR(NMSLIB_ERROR_INDEX_BUILD_FAILED, "Index not built");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->set_query_params(params_of(params));
        if (s.ok() && index->group) s = index->group->set_query_params(params_of(params));
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Query time params set");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to set query time params");
}

nmslib_error_t nmslib_get_space_type(nmslib_index_handle_t index, const char** space_type, size_t* space_type_len,
                                     const nmslib_allocator_t* allocator) {
  if (!index || !space_type || !space_type_len || !alloc_ok(allocator))
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid arguments");
  *space_type_len = index->space_type.size();
  *space_type = dup_string(index->space_type, allocator);
  if (!*space_type) return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate memory for space type");
  return NB_OK("Space type retrieved successfully");
}

nmslib_error_t nmslib_get_method(nmslib_index_handle_t index, const char** method, size_t* method_len,
                                 const nmslib_allocator_t* allocator) {
  if (!index || !method || !method_len || !alloc_ok(allocator))
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid arguments");
  *method_len = index->method.size();
  *method = dup_string(index->method, allocator);
  if (!*method) return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate memory for method");
  return NB_OK("Method retrieved successfully");
}

void nmslib_free_string(char* str, const nmslib_allocator_t* allocator) {
  if (!str || !allocator || !allocator->free) {
    NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid string or allocator");
    return;
  }
  allocator->free(str, allocator->ctx);
}

nmslib_error_t nmslib_get_last_error_detail(nmslib_error_detail_t* detail, const nmslib_allocator_t* allocator) {
  if (!detail || !alloc_ok(allocator)) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid detail or allocator pointer");
  detail->code = g_last.code;
  detail->message = dup_string(g_last.message, allocator);
  if (!detail->message) return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate memory for error message");
  detail->file = dup_string(g_last.file, allocator);
  if (!detail->file) {
    allocator->free(const_cast<char*>(detail->message), allocator->ctx);
    return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate memory for error file");
  }
  detail->line = g_last.line;
  return NB_OK("Error detail retrieved successfully");
}

nmslib_error_t nmslib_set_thread_pool_size(nmslib_index_handle_t index, size_t size) {
  if (!index || size == 0 || size > 1024) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid thread pool size");
  index->thread_pool_size = size;  // accepted and unused, as in the reference (:1507-1535)
  return NB_OK("Thread pool size set");
}
size_t nmslib_get_thread_pool_size(nmslib_index_handle_t index) {
  if (!index) {
    NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
    return std::thread::hardware_concurrency();
  }
  return index->thread_pool_size;
}
size_t nmslib_data_qty(nmslib_index_handle_t index) {
  if (!index) {
    NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
    return 0;
  }
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  return index->engine->size();
}
// ref :1546-1565: sum of object buffers (16-byte header + payload) + n * dim * 4
size_t nmslib_index_memory_usage(nmslib_index_handle_t index) {
  if (!index || !index->engine->built()) return 0;
  const Engine* e = index->engine;
  const size_t payload = e->is_u8() ? (size_t)e->dim() + 4 : (size_t)e->dim() * 4;
  return e->size() * (16 + payload) + e->size() * (size_t)e->dim() * sizeof(float);
}

// ------------------------------------------------------------------------------ ingest
nmslib_error_t nmslib_add_data_point(nmslib_index_handle_t index, const void* data, size_t element_count, int32_t id) {
  if (!index || !data || element_count == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid inputs for adding data point");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->add_rows(data, 1, element_count, &id);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Data point added successfully");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to add data point");
}

nmslib_error_t nmslib_add_data_point_batch(nmslib_index_handle_t index, const void* data, size_t count,
                                           size_t element_count, const int32_t* ids, const size_t* /*num_elements*/) {
  if (!index || !data || count == 0 || element_count == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid batch inputs");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->add_rows(data, count, element_count, ids);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Batch added successfully");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to add batch");
}

nmslib_error_t nmslib_add_data_point_batch_uint8(nmslib_index_handle_t index, const unsigned char* data, size_t count,
                                                 size_t element_count, const int32_t* ids) {
  if (!index || !data || count == 0 || element_count == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid uint8 batch inputs");
  if (index->header.data_type != NMSLIB_DATATYPE_DENSE_UINT8_VECTOR)
    return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "Not uint8 vector space");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->add_rows(data, count, element_count, ids);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("UInt8 batch added successfully");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to add uint8 batch");
}

nmslib_error_t nmslib_add_data_point_batch_string(nmslib_index_handle_t index, const char* const* data, size_t count,
                                                  const int32_t* /*ids*/) {
  if (!index || !data || count == 0) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid string batch inputs");
  return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "Not string space");  // ref :884-887
}

nmslib_error_t nmslib_add_data_point_batch_pointers(nmslib_index_handle_t handle, nmslib_data_mode_t data_mode,
                                                    const void* const* data_ptrs, size_t count, size_t element_count,
                                                    const int32_t* ids, const size_t* /*num_elements*/) {
  if (!handle) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  if (!data_ptrs || count == 0) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid pointer batch");
  if (data_mode == NMSLIB_DATA_MODE_SPARSE)
    return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "sparse vectors stay on the reference CPU code");
  const bool want_u8 = data_mode == NMSLIB_DATA_MODE_UINT8;
  if (want_u8 != handle->engine->is_u8()) return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "data mode does not match index");
  if (element_count == 0) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "element_count == 0");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(handle->engine->mutex());
        Status s = handle->engine->add_row_ptrs(data_ptrs, count, element_count, ids);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Pointer batch added successfully");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to add pointer batch");
}

// ------------------------------------------------------------------------------ the hot path
nmslib_error_t nmslib_knn_query_get_size(nmslib_index_handle_t index, const void* query, size_t /*elem_count*/,
                                         size_t k, size_t* out_size, size_t /*num_elements*/) {
  if (!index || !query || k == 0 || !out_size) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid knn query inputs");
  *out_size = k;  // ref :933
  return NB_OK("KNN size retrieved");
}

nmslib_error_t nmslib_knn_query_batch(nmslib_index_handle_t index, const void* queries, size_t query_count,
                                      size_t elem_count, size_t k, nmslib_result_t* results,
                                      const size_t* /*num_elements*/, size_t /*thread_pool_size*/) {
  if (!index || !queries || query_count == 0 || !results || elem_count == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid batch knn inputs");
  if (k == 0) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "k must be positive");  // SURVEY Q8
  // (two result slabs cut into rows of k, the batch shape INTEGRATION.md gives lib.zig: filled by two copies below)
  bool slabs = true;
  for (size_t i = 0; i < query_count; ++i) {
    if (!results[i].ids || !results[i].distances || results[i].capacity == 0)
      return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Result buffers invalid");
    slabs = slabs && results[i].capacity >= k && results[i].ids == results[0].ids + i * k &&
            results[i].distances == results[0].distances + i * k;
  }
  return guarded(
      [&]() -> nmslib_error_t {
        Engine* e = index->engine;
        std::lock_guard<std::mutex> lock(e->mutex());
        const int32_t *ids, *counts;
        const float* dists;
        Status s = index->group ? index->group->knn_host(e, queries, query_count, elem_count, k, &ids, &dists, &counts)
                                : e->knn_host(queries, query_count, elem_count, k, &ids, &dists, &counts);
        if (!s.ok()) {
          for (size_t i = 0; i < query_count; ++i) results[i].size = 0;
          return NB_STATUS(s);
        }
        if (slabs) {  // (entries past a row's size are the engine's padding: id -1, distance +inf)
          memcpy(results[0].ids, ids, query_count * k * sizeof(int32_t));
          memcpy(results[0].distances, dists, query_count * k * sizeof(float));
          for (size_t i = 0; i < query_count; ++i) results[i].size = (size_t)counts[i];
          return NB_OK("Batch knn query executed");
        }
        bool too_small = false;
        for (size_t i = 0; i < query_count; ++i) {  // extract_knn_results, ref :293-328
          const size_t found = (size_t)counts[i];
          if (found > results[i].capacity) {
            results[i].size = 0;
            too_small = true;
            continue;
          }
          memcpy(results[i].ids, ids + i * k, found * sizeof(int32_t));
          memcpy(results[i].distances, dists + i * k, found * sizeof(float));
          results[i].size = found;
        }
        if (too_small) return NB_ERR(NMSLIB_ERROR_BUFFER_TOO_SMALL, "Result buffers too small");  // SURVEY Q9
        return NB_OK("Batch knn query executed");
      },
      NMSLIB_ERROR_QUERY_EXECUTION_FAILED, "KNN query failed");
}

nmslib_error_t nmslib_knn_query_fill(nmslib_index_handle_t index, const void* query, size_t elem_count, size_t k,
                                     nmslib_result_t* result, size_t num_elements) {
  if (!index || !query || elem_count == 0 || !result)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid KNN query inputs");
  return nmslib_knn_query_batch(index, query, 1, elem_count, k, result, num_elements ? &num_elements : nullptr, 0);
}

void nmslib_free_result(nmslib_result_t* result) {  // results are caller-owned: just forget them
  if (!result) return;
  result->size = 0;
}

// ------------------------------------------------------------------------------ outside the path
nmslib_error_t nmslib_range_query_get_size(nmslib_index_handle_t index, const void* query, size_t, double radius,
                                           size_t* out_size, size_t) {
  if (!index || !query || radius < 0 || !out_size) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid range query inputs");
  *out_size = 128;  // ref :1046
  return NB_OK("Range query size estimated");
}
nmslib_error_t nmslib_range_query_fill(nmslib_index_handle_t index, const void* query, size_t elem_count,
                                       double radius, nmslib_result_t* result, size_t) {
  if (!index || !query || !result || result->capacity == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid range fill inputs");  // ref :1056-1060
  if (!result->ids || !result->distances) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Result buffers invalid");
  return guarded(
      [&]() -> nmslib_error_t {
        Engine* e = index->engine;
        std::lock_guard<std::mutex> lock(e->mutex());
        size_t found = 0;
        Status s = e->range_host(query, elem_count, radius, result->capacity, result->ids, result->distances, &found);
        result->size = s.ok() ? found : 0;
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Range query filled successfully");
      },
      NMSLIB_ERROR_QUERY_EXECUTION_FAILED, "Range query failed");
}
nmslib_error_t nmslib_b200_range_query_batch(nmslib_index_handle_t index, const void* queries, size_t query_count,
                                             size_t elem_count, const double* radii, nmslib_result_t* results) {
  // the whole batch is checked before any work (codes of nmslib_range_query_get_size / _fill)
  if (!index || !queries || query_count == 0 || !radii || !results)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid range batch inputs");
  for (size_t i = 0; i < query_count; ++i) {
    if (radii[i] < 0) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Negative radius in range batch");
    if (!results[i].ids || !results[i].distances || results[i].capacity == 0)
      return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Result buffers invalid");
  }
  return guarded(
      [&]() -> nmslib_error_t {
        Engine* e = index->engine;
        std::lock_guard<std::mutex> lock(e->mutex());
        std::vector<size_t> caps(query_count), sizes(query_count, 0);
        std::vector<int32_t*> ids(query_count);
        std::vector<float*> dists(query_count);
        for (size_t i = 0; i < query_count; ++i) {
          caps[i] = results[i].capacity;
          ids[i] = results[i].ids;
          dists[i] = results[i].distances;
        }
        Status s = index->group ? index->group->range_host(e, queries, query_count, elem_count, radii, caps.data(),
                                                           ids.data(), dists.data(), sizes.data())
                                : e->range_batch_host(queries, query_count, elem_count, radii, caps.data(), ids.data(),
                                                      dists.data(), sizes.data());
        for (size_t i = 0; i < query_count; ++i) results[i].size = s.ok() ? sizes[i] : 0;
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Range query batch executed");
      },
      NMSLIB_ERROR_QUERY_EXECUTION_FAILED, "Range query batch failed");
}
nmslib_error_t nmslib_get_data_point_string(nmslib_index_handle_t index, size_t, const char** data, size_t* data_len,
                                            const nmslib_allocator_t* allocator) {
  if (!index || !data || !data_len || !alloc_ok(allocator)) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid arguments");
  return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "Not a string space");
}
nmslib_error_t nmslib_borrow_data_sparse(nmslib_index_handle_t index, size_t, void** data, size_t* size,
                                         void (**free_fn)(void*)) {
  if (!index || !data || !size || !free_fn) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid arguments");
  return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "Not a sparse space");
}

// ------------------------------------------------------------------------------ data access
nmslib_error_t nmslib_get_distance(nmslib_index_handle_t index, size_t pos1, size_t pos2, float* distance) {
  if (!index || !distance || pos1 >= index->engine->size() || pos2 >= index->engine->size())
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid distance inputs");
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  if (pos1 >= index->engine->size() || pos2 >= index->engine->size())
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid distance inputs");
  *distance = index->engine->host_distance(pos1, pos2);
  return NB_OK("Distance computed");
}

nmslib_error_t nmslib_get_data_point_size(nmslib_index_handle_t index, size_t position, size_t* size) {
  if (!index || !size || position >= index->engine->size())
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid data point request");
  *size = (size_t)index->engine->dim();  // element count (floats or bytes)
  return NB_OK("Data point size retrieved");
}

nmslib_error_t nmslib_get_data_point_fill(nmslib_index_handle_t index, size_t position, void* data, size_t size) {
  if (!index || !data || position >= index->engine->size())
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid data point request");
  Engine* e = index->engine;
  std::lock_guard<std::mutex> lock(e->mutex());  // (a concurrent add_rows may reallocate the host rows)
  if (position >= e->size()) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid data point request");
  if (size < (size_t)e->dim()) return NB_ERR(NMSLIB_ERROR_BUFFER_TOO_SMALL, "Buffer too small for data point");
  if (e->is_u8()) memcpy(data, e->row_u8(position), (size_t)e->dim());
  else memcpy(data, e->row_f32(position), (size_t)e->dim() * sizeof(float));
  return NB_OK("Data point filled");
}

namespace {
// One block [header | payload]; the caller gets the payload pointer and free_fn(payload)
// releases the block.  (The reference hands out a payload pointer whose wrapper cannot be
// reached again, nmslib_c.cpp:1286-1306; lib.zig never calls it, lib.zig:1007-1015.)
struct BorrowHeader {
  nmslib_allocator_t allocator;
  uint64_t magic;
};
void borrowed_free(void* payload) {
  if (!payload) return;
  BorrowHeader* h = reinterpret_cast<BorrowHeader*>(static_cast<char*>(payload) - sizeof(BorrowHeader));
  if (h->magic != 0xB200B0220BB0ull) return;
  nmslib_allocator_t a = h->allocator;
  h->magic = 0;
  a.free(h, a.ctx);
}
}  // namespace

nmslib_error_t nmslib_borrow_data_dense(nmslib_index_handle_t index, size_t position, void** data, size_t* size,
                                        void (**free_fn)(void*)) {
  if (!index || !data || !size || !free_fn || position >= index->engine->size())
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid dense borrow inputs");
  Engine* e = index->engine;
  std::lock_guard<std::mutex> lock(e->mutex());
  if (position >= e->size()) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid dense borrow inputs");
  if (e->is_u8()) return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "Not dense vector");
  const size_t bytes = (size_t)e->dim() * sizeof(float);
  nmslib_allocator_t a = index->allocator;
  char* block = static_cast<char*>(a.alloc(sizeof(BorrowHeader) + bytes, a.ctx));
  if (!block) return NB_ERR(NMSLIB_ERROR_OUT_OF_MEMORY, "Failed to allocate data copy");
  BorrowHeader* h = reinterpret_cast<BorrowHeader*>(block);
  h->allocator = a;
  h->magic = 0xB200B0220BB0ull;
  memcpy(block + sizeof(BorrowHeader), e->row_f32(position), bytes);
  *data = block + sizeof(BorrowHeader);
  *size = bytes;
  *free_fn = borrowed_free;
  return NB_OK("Dense data borrowed");
}

// ------------------------------------------------------------------------------ persistence
nmslib_error_t nmslib_save_index(nmslib_index_handle_t index, const char* path, int save_data) {
  if (!index || !path) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid save inputs");
  if (!index->engine->built()) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Index not built");
  return guarded(
      [&]() -> nmslib_error_t {
        Engine* e = index->engine;
        std::lock_guard<std::mutex> lock(e->mutex());
        if (save_data) {  // Space::WriteObjectVectorBinData, space.cc:90-105
          FILE* f = fopen((std::string(path) + ".dat").c_str(), "wb");
          if (!f) return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, "Failed to save index: cannot open .dat");
          const uint64_t qty = e->size();
          bool ok = fwrite(&qty, 8, 1, f) == 1;
          for (size_t i = 0; ok && i < e->size(); ++i) {
            const uint64_t datalen = e->is_u8() ? (uint64_t)e->dim() + 4 : (uint64_t)e->dim() * 4;
            const uint64_t buflen = 16 + datalen;
            const int32_t id = e->ext_id(i), label = -1;
            ok = fwrite(&buflen, 8, 1, f) == 1 && fwrite(&id, 4, 1, f) == 1 && fwrite(&label, 4, 1, f) == 1 &&
                 fwrite(&datalen, 8, 1, f) == 1;
            if (!ok) break;
            if (e->is_u8()) {
              int32_t sum = 0;
              const uint8_t* r = e->row_u8(i);
              for (int j = 0; j < e->dim(); ++j) sum += (int)r[j] * r[j];
              ok = fwrite(r, 1, e->dim(), f) == (size_t)e->dim() && fwrite(&sum, 4, 1, f) == 1;
            } else {
              ok = fwrite(e->row_f32(i), 4, e->dim(), f) == (size_t)e->dim();
            }
          }
          fclose(f);
          if (!ok) return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, "Failed to save index: short write");
        }
        if (e->method() == nb200::METHOD_HNSW) {
          if (e->graph().empty()) {  // not queried yet: build now (the reference builds at create_index time)
            Status ps = e->ensure_graph();
            if (!ps.ok()) return NB_STATUS(ps);
          }
          // l2sqr_sift is Hnsw<int> in the reference: it saves the regular index (SaveRegularIndexBin), links only
          Status s = e->is_u8() ? nb200::write_regular(path, e->graph())
                                : nb200::write_hnsw_file(path, e->graph(), e->hnsw_rows_for_save(), e->graph().ext_ids.data());
          if (!s.ok()) return NB_STATUS(s);
        } else {
          // SeqSearch has no SaveIndex in the reference (index.h:56-58 throws); we leave a marker
          FILE* f = fopen(path, "wb");
          if (!f) return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, "Failed to save index");
          const std::string tag = "NB200SEQ " + index->space_type + "\n";
          fwrite(tag.data(), 1, tag.size(), f);
          fclose(f);
        }
        return NB_OK("Index saved successfully");
      },
      NMSLIB_ERROR_DATA_IO_FAILED, "Failed to save index");
}

// Space::ReadObjectVectorFromBinData (space.cc:60-88): the rows of `path`.dat appended to h; nullptr, or what failed
static const char* read_dat(const char* path, nmslib_index_handle_t h) {
  FILE* d = fopen((std::string(path) + ".dat").c_str(), "rb");
  if (!d) return "Failed to load index: cannot open .dat";
  uint64_t qty = 0;
  bool ok = fread(&qty, 8, 1, d) == 1;
  std::vector<char> buf;
  for (uint64_t i = 0; ok && i < qty; ++i) {
    uint64_t buflen = 0;
    ok = fread(&buflen, 8, 1, d) == 1 && buflen >= 16 && buflen < (1ull << 32);
    if (!ok) break;
    buf.resize(buflen);
    ok = fread(buf.data(), 1, buflen, d) == buflen;
    if (!ok) break;
    int32_t id;
    memcpy(&id, buf.data(), 4);
    const size_t payload = buflen - 16;
    uint64_t datalen = 0;  // Object header: id, label, datalength (object.h); must describe this record
    memcpy(&datalen, buf.data() + 8, 8);
    ok = datalen == payload && (h->engine->is_u8() ? payload > 4 : (payload >= 4 && payload % 4 == 0));
    if (!ok) break;
    const size_t elems = h->engine->is_u8() ? payload - 4 : payload / 4;
    ok = h->engine->add_rows(buf.data() + 16, 1, elems, &id).ok();
  }
  fclose(d);
  return ok ? nullptr : "Failed to load index: corrupt .dat";
}

nmslib_error_t nmslib_load_index(const char* path, nmslib_data_type_t data_type, nmslib_dist_type_t dist_type,
                                 const nmslib_allocator_t* allocator, int load_data, nmslib_index_handle_t* out_handle) {
  if (!path || !alloc_ok(allocator) || !out_handle) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid load inputs");
  return guarded(
      [&]() -> nmslib_error_t {
        FILE* f = fopen(path, "rb");
        if (!f) return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, "Failed to load index: cannot open file");
        char head[64] = {0};
        const size_t got = fread(head, 1, sizeof(head) - 1, f);
        fclose(f);
        if (got >= 9 && memcmp(head, "NB200SEQ ", 9) == 0) {
          std::string space(head + 9);
          space = space.substr(0, space.find('\n'));
          nmslib_index_handle_t h = nullptr;
          nmslib_error_t rc = new_index(space, "seq_search", data_type, dist_type, allocator, &h);
          if (rc != NMSLIB_SUCCESS) return rc;
          if (const char* err = load_data ? read_dat(path, h) : nullptr) {
            nmslib_index_destroy(h);
            return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, err);
          }
          h->engine->mark_built({});
          *out_handle = h;
          return NB_OK("Index loaded successfully");
        }
        // otherwise: the reference's optimized HNSW stream.  The reference hard-codes "hnsw" + "l2"
        // here (nmslib_c.cpp:1421-1429); we read the distance type from the header (SURVEY Q11).
        // A regular index (flag 0, what l2sqr_sift + hnsw saves) loaded as uint8 is l2sqr_sift over its .dat: the
        // file holds links only (LoadRegularIndexBin CHECKs that the data set has as many points, hnsw.cc:956-959).
        uint32_t flag = 1;
        memcpy(&flag, head, got >= 4 ? 4 : 0);
        const bool regular_u8 = got >= 4 && flag == 0 && data_type == NMSLIB_DATATYPE_DENSE_UINT8_VECTOR;
        if (regular_u8 && !load_data)
          return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, "Failed to load index: a regular HNSW index needs its data (load_data=1)");
        nb200::HnswGraph g;
        Status s = nb200::read_hnsw_file(path, &g);
        if (!s.ok()) return NB_STATUS(s);
        const char* space = regular_u8 ? "l2sqr_sift" : g.dist_func == 3 ? "cosinesimil" : g.dist_func == 4 ? "negdotprod" : "l2";
        nmslib_index_handle_t h = nullptr;
        nmslib_error_t rc = new_index(space, "hnsw", data_type, dist_type, allocator, &h);
        if (rc != NMSLIB_SUCCESS) return rc;
        if (const char* err = regular_u8 ? read_dat(path, h) : nullptr) {
          nmslib_index_destroy(h);
          return NB_ERR(NMSLIB_ERROR_DATA_IO_FAILED, err);
        }
        s = h->engine->adopt_graph(std::move(g));
        if (!s.ok()) {
          nmslib_index_destroy(h);
          return NB_STATUS(s);
        }
        *out_handle = h;
        return NB_OK("Index loaded successfully");
      },
      NMSLIB_ERROR_DATA_IO_FAILED, "Failed to load index");
}

// ------------------------------------------------------------------------------ extensions
int nmslib_b200_set_device(int device) {
  nb200::set_default_device(device);
  return 0;
}
int nmslib_b200_device_available(void) { return nb200::device_available() ? 1 : 0; }

nmslib_error_t nmslib_b200_set_shard(nmslib_index_handle_t index, uint32_t pos_base) {
  if (!index) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  index->engine->set_pos_base(pos_base);
  return NB_OK("Shard base set");
}

nmslib_error_t nmslib_b200_import_hnsw(nmslib_index_handle_t index, const char* path) {
  if (!index || !path) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid import inputs");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->import_graph(path);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("HNSW graph imported");
      },
      NMSLIB_ERROR_DATA_IO_FAILED, "Failed to import HNSW graph");
}

nmslib_error_t nmslib_b200_prepare(nmslib_index_handle_t index) {
  if (!index) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->group ? index->group->prepare(index->engine, 1, 1) : index->engine->prepare();
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Device copy ready");
      },
      NMSLIB_ERROR_QUERY_EXECUTION_FAILED, "Failed to prepare index");
}

nmslib_error_t nmslib_b200_knn_device(nmslib_index_handle_t index, const void* d_queries, size_t query_count,
                                      size_t elem_count, size_t k, int32_t* d_ids, float* d_distances,
                                      uint64_t* d_keys, void* stream) {
  if (!index || !d_queries || query_count == 0 || elem_count == 0 || k == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid device knn inputs");
  if (index->group)
    return NB_ERR(NMSLIB_ERROR_SPACE_INCOMPATIBLE, "device-resident queries address one device: not available on a b200_devices index");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->knn_device(d_queries, query_count, elem_count, k, d_ids, d_distances, d_keys,
                                             nullptr, static_cast<cudaStream_t>(stream));
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Device knn query enqueued");
      },
      NMSLIB_ERROR_QUERY_EXECUTION_FAILED, "Device knn query failed");
}

nmslib_error_t nmslib_b200_merge_topk(nmslib_index_handle_t index, const uint64_t* d_keys, const int32_t* d_ids,
                                      size_t lists, size_t query_count, size_t k, int32_t* d_out_ids,
                                      float* d_out_distances, void* stream) {
  // d_ids == NULL: the ids ARE the global positions the keys carry (default ids of lib.zig's addDenseBatch; what a
  // sharded caller gets when every rank numbers its rows by global position) -- one all-gather per step instead of two
  if (!index || !d_keys || lists == 0 || query_count == 0 || k == 0)
    return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid merge inputs");
  if (lists * k > (size_t)nb200::merge_topk_max_items()) return NB_ERR(NMSLIB_ERROR_QUERY_TOO_LARGE, "lists * k too large");
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  cudaError_t e = cudaSetDevice(index->engine->device());  // launch where the index lives, whatever is current
  if (e == cudaSuccess) e = nb200::launch_merge_topk(d_keys, d_ids, (int)lists, query_count * k, k, (int)query_count, (int)k,
                                           index->engine->finalize_kind(), nullptr, 0, nullptr, d_out_ids,
                                           d_out_distances, nullptr, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return NB_ERR(NMSLIB_ERROR_QUERY_EXECUTION_FAILED, std::string("merge failed: ") + cudaGetErrorString(e));
  return NB_OK("Merged");
}

nmslib_error_t nmslib_b200_get_stats(nmslib_index_handle_t index, nmslib_b200_stats_t* out) {
  if (!index || !out) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid stats request");
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  const nb200::Stats s = index->group ? index->group->stats() : index->engine->stats();
  out->queries = s.queries;
  out->kernel_launches = s.kernel_launches;
  out->distance_evals = s.distance_evals;
  out->hnsw_expansions = s.hnsw_expansions;
  out->last_kernel_ms = s.last_kernel_ms;
  out->last_total_ms = s.last_total_ms;
  out->fallback_queries = s.fallback_queries;
  out->device_bytes = s.device_bytes;
  out->last_scan_ms = s.last_scan_ms;
  out->scan_ms_sum = s.scan_ms_sum;
  out->scan_count = s.scan_count;
  const nb200::HnswBuildInfo& bi = index->engine->build_info();
  out->build_total_ms = bi.total_ms;
  out->build_scan_ms = bi.scan_ms;
  out->build_select_ms = bi.select_ms;
  out->build_link_ms = bi.link_ms;
  out->build_batches = (uint64_t)bi.batches;
  out->build_prunes = bi.prunes;
  out->split_queries = s.split_queries;
  out->uploaded_rows = s.uploaded_rows;
  out->range_tc_queries = s.range_tc_queries;
  out->range_fallback_queries = s.range_fallback_queries;
  out->u8_imma = (!index->group && index->engine->is_u8() && index->engine->method() == nb200::METHOD_SEQ &&
                  index->engine->u8_imma()) ? 1 : 0;
  return NMSLIB_SUCCESS;
}

static size_t scan_plan_impl(size_t query_count, size_t n, size_t k, int units, int tile_rows, int lists_per_piece,
                             int32_t* pieces, size_t capacity, int* n_cta, int* s_max);

size_t nmslib_b200_scan_plan(size_t query_count, size_t n, size_t k, int sm_count, int32_t* pieces, size_t capacity,
                             int* n_cta, int* s_max) {
  return scan_plan_impl(query_count, n, k, sm_count, 0, 1, pieces, capacity, n_cta, s_max);
}

size_t nmslib_b200_scan_plan_pairs(size_t query_count, size_t n, size_t k, int sm_count, int32_t* pieces,
                                   size_t capacity, int* n_pairs, int* s_max) {
  int slots = 0;
  const size_t m = scan_plan_impl(query_count, n, k, sm_count / 2, nb200::tc_pair_block_points(), 2, pieces, capacity,
                                  n_pairs, &slots);
  if (s_max) *s_max = 2 * slots;  // two candidate lists (column halves of the 256-row tile) per piece
  return m;
}

static size_t scan_plan_impl(size_t query_count, size_t n, size_t k, int units, int tile_rows, int lists_per_piece,
                             int32_t* pieces, size_t capacity, int* n_cta, int* s_max) {
  std::vector<int> table;
  int nc = 0, sm = 0;
  nb200::tc_ts_plan((int)query_count, (int)n, (int)k, units, &table, &nc, &sm, tile_rows, lists_per_piece);
  if (n_cta) *n_cta = nc;
  if (s_max) *s_max = sm;
  size_t out = 0;
  for (int c = 0; c < nc; ++c)
    for (int i = 0; i < 8; ++i) {
      const int* e = table.data() + ((size_t)c * 8 + i) * 4;
      if (e[0] < 0) break;
      if (pieces && out < capacity) {
        pieces[out * 5] = c;
        for (int j = 0; j < 4; ++j) pieces[out * 5 + 1 + j] = e[j];
      }
      ++out;
    }
  return out;
}

nmslib_error_t nmslib_b200_shard_export(nmslib_index_handle_t index, size_t max_queries, size_t max_k, void* blob) {
  if (!index || !blob || max_queries == 0 || max_k == 0) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid shard export inputs");
  if (index->group) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "a b200_devices index manages its own shards");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->shard_export(max_queries, max_k, blob);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Exchange window exported");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to export the exchange window");
}

nmslib_error_t nmslib_b200_shard_connect(nmslib_index_handle_t index, int rank, int world, const void* blobs) {
  if (!index || !blobs) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid shard connect inputs");
  return guarded(
      [&]() -> nmslib_error_t {
        std::lock_guard<std::mutex> lock(index->engine->mutex());
        Status s = index->engine->shard_connect(rank, world, blobs);
        if (!s.ok()) return NB_STATUS(s);
        return NB_OK("Shard exchange connected");
      },
      NMSLIB_ERROR_RUNTIME, "Failed to connect the shard exchange");
}

nmslib_error_t nmslib_b200_shard_disconnect(nmslib_index_handle_t index) {
  if (!index) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid index");
  std::lock_guard<std::mutex> lock(index->engine->mutex());
  index->engine->shard_disconnect();
  return NB_OK("Shard exchange closed");
}

nmslib_error_t nmslib_b200_set_option(const char* name, int value) {
  static const char* const known[] = {"tc_pair", "hnsw_team", "force_exact", "tc_split", "u8_imma"};
  if (!name) return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, "Invalid option name");
  for (const char* k : known)
    if (strcmp(k, name) == 0) {
      nb200::nb200_set_option(name, value);
      return NB_OK("Option set");
    }
  return NB_ERR(NMSLIB_ERROR_INVALID_ARGUMENT, std::string("unknown option '") + name + "'");
}

const char* nmslib_b200_version(void) { return "nmslib_b200 0.1 sm_100a"; }

}  // extern "C"
