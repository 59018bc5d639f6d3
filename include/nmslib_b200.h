/* nmslib_b200.h -- C ABI of libnmslib_b200.so, the B200-native k-NN query engine.
 *
 * PART 1 declares, name for name and argument for argument, the C ABI that
 * B-R-P/NMSLIB-ZIG's lib.zig binds through @cImport("nmslib_c.h") (lib.zig:5-8),
 * so that the Zig host can link this library in place of the reference shim for
 * dense-vector indexes.  The type and function NAMES and LAYOUTS are the contract
 * and are therefore identical to the reference's nmslib_c.h (cited per entry as
 * "ref nmslib_c.h:<line>" / "ref nmslib_c.cpp:<line>"); the wording here is ours.
 *
 * What runs where:
 *   data types  DENSE_VECTOR (float32) and DENSE_UINT8_VECTOR (SIFT 128-D)
 *   spaces      l2, l2sqr (new), cosinesimil (alias cosine), negdotprod, l2sqr_sift
 *   methods     seq_search / brute_force  -> sm_100a brute-force kNN kernels
 *               hnsw                      -> sm_100a batched beam search over a graph
 *                                            (imported from the reference's
 *                                            Hnsw::SaveIndex stream, or built on device)
 * Sparse / string spaces and range queries are outside this engine's path: the
 * corresponding entry points exist (all 37 symbols are exported) and return
 * NMSLIB_ERROR_SPACE_INCOMPATIBLE, which lib.zig:29-74 maps to error.SpaceIncompatible.
 * There is no CPU fallback on the query path: if no CUDA device can be opened the
 * query calls fail with NMSLIB_ERROR_QUERY_EXECUTION_FAILED.
 *
 * PART 2 declares the nmslib_b200_* extensions (device-resident queries, shard
 * placement for multi-GPU, top-k list merge, graph import, counters).
 */
#ifndef NMSLIB_B200_H
#define NMSLIB_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ======================================================================== */
/* PART 1 -- the reference ABI (ref nmslib_c.h:12-86)                        */
/* ======================================================================== */

typedef enum { /* ref nmslib_c.h:12-17 */
  NMSLIB_DATATYPE_DENSE_VECTOR = 0,
  NMSLIB_DATATYPE_SPARSE_VECTOR = 1,
  NMSLIB_DATATYPE_DENSE_UINT8_VECTOR = 2,
  NMSLIB_DATATYPE_OBJECT_AS_STRING = 3
} nmslib_data_type_t;

typedef enum { NMSLIB_DISTTYPE_FLOAT = 0, NMSLIB_DISTTYPE_INT = 1 } nmslib_dist_type_t; /* :20 */

typedef enum { /* ref nmslib_c.h:23-39; lib.zig:29-74 maps these to Zig errors */
  NMSLIB_SUCCESS = 0,
  NMSLIB_ERROR_NULL_POINTER = 1,
  NMSLIB_ERROR_INVALID_ARGUMENT = 2,
  NMSLIB_ERROR_OUT_OF_MEMORY = 3,
  NMSLIB_ERROR_BUFFER_TOO_SMALL = 4,
  NMSLIB_ERROR_SPACE_INCOMPATIBLE = 5,
  NMSLIB_ERROR_QUERY_TOO_LARGE = 6,
  NMSLIB_ERROR_INVALID_SPARSE_ELEMENT = 7,
  NMSLIB_ERROR_INDEX_BUILD_FAILED = 8,
  NMSLIB_ERROR_QUERY_EXECUTION_FAILED = 9,
  NMSLIB_ERROR_DATA_IO_FAILED = 10,
  NMSLIB_ERROR_PLUGIN_REGISTRATION_FAILED = 11,
  NMSLIB_ERROR_INTERNAL = 12,
  NMSLIB_ERROR_RUNTIME = 13,
  NMSLIB_ERROR_INDEX_NOT_BUILT = 14
} nmslib_error_t;

typedef enum { /* ref nmslib_c.h:42-46 */
  NMSLIB_DATA_MODE_DENSE_FLOAT = 0,
  NMSLIB_DATA_MODE_SPARSE = 1,
  NMSLIB_DATA_MODE_UINT8 = 2
} nmslib_data_mode_t;

typedef struct { uint32_t id; float value; } nmslib_sparse_elem_float_t; /* :49-52 */

/* Caller-owned result slots (ref nmslib_c.h:55-60): the callee writes
 * ids[0..size) / distances[0..size), size <= capacity, ascending by distance. */
typedef struct {
  int32_t* ids;
  float* distances;
  size_t size;
  size_t capacity;
} nmslib_result_t;

typedef struct { /* ref nmslib_c.h:63-67 */
  void* (*alloc)(size_t size, void* ctx);
  void (*free)(void* ptr, void* ctx);
  void* ctx;
} nmslib_allocator_t;

typedef struct { /* ref nmslib_c.h:70-75 */
  nmslib_error_t code;
  const char* message;
  const char* file;
  int line;
} nmslib_error_detail_t;

/* First field of every index object (ref nmslib_c.h:77-80, nmslib_c.cpp:137-139). */
typedef struct {
  nmslib_data_type_t data_type;
  nmslib_dist_type_t dist_type;
} nmslib_index_header_t;

typedef struct nmslib_index_t* nmslib_index_handle_t;   /* ref :83 */
typedef struct nmslib_params_t* nmslib_params_handle_t; /* ref :86 */

/* -- lifecycle ----------------------------------------------------------- */
void nmslib_init(void); /* ref nmslib_c.cpp:338 */
/* ref nmslib_c.cpp:340-447.  Unknown / unsupported space -> SPACE_INCOMPATIBLE. */
nmslib_error_t nmslib_index_create(const char* space, nmslib_params_handle_t space_params,
                                   const char* method, nmslib_data_type_t data_type,
                                   nmslib_dist_type_t dist_type,
                                   const nmslib_allocator_t* allocator,
                                   nmslib_index_handle_t* out_handle);
void nmslib_index_destroy(nmslib_index_handle_t handle); /* ref :449-477 */
/* ref nmslib_c.cpp:479-517.  Records the index-time params and marks the index
 * built; the device upload (and, for hnsw, the graph) is materialised lazily at
 * the first query / nmslib_initialize_pool, which also covers lib.zig's
 * create-then-add order (lib.zig:629-680). */
nmslib_error_t nmslib_create_index(nmslib_index_handle_t index,
                                   nmslib_params_handle_t index_params, int print_progress);
nmslib_error_t nmslib_reset_index(nmslib_index_handle_t index); /* ref :519-538 */
void nmslib_initialize_pool(nmslib_index_handle_t index);       /* ref :1682-1704 */

/* -- params (ref nmslib_c.cpp:540-614): type 0=int, 1=double, 2=string ------ */
nmslib_params_handle_t nmslib_create_params(const nmslib_allocator_t* allocator);
nmslib_error_t nmslib_add_param(nmslib_params_handle_t params, const char* name, int type,
                                const void* value);
void nmslib_free_params(nmslib_params_handle_t params);
/* ref :1481-1505.  hnsw: ef / efSearch (synonyms; both at once is an error),
 * algoType in {hybrid,v1merge,old}, searchMethod (ignored) -- hnsw.cc:474-507.
 * An explicit value is honoured (the reference clobbers it with 200, SURVEY Q1). */
nmslib_error_t nmslib_set_query_time_params(nmslib_index_handle_t index,
                                            nmslib_params_handle_t params);

/* -- introspection (ref :616-715, :1507-1565) ------------------------------ */
nmslib_error_t nmslib_get_space_type(nmslib_index_handle_t index, const char** space_type,
                                     size_t* space_type_len, const nmslib_allocator_t* allocator);
nmslib_error_t nmslib_get_method(nmslib_index_handle_t index, const char** method,
                                 size_t* method_len, const nmslib_allocator_t* allocator);
void nmslib_free_string(char* str, const nmslib_allocator_t* allocator);
nmslib_error_t nmslib_get_last_error_detail(nmslib_error_detail_t* detail,
                                            const nmslib_allocator_t* allocator);
nmslib_error_t nmslib_set_thread_pool_size(nmslib_index_handle_t index, size_t size);
size_t nmslib_get_thread_pool_size(nmslib_index_handle_t index);
size_t nmslib_data_qty(nmslib_index_handle_t index);
size_t nmslib_index_memory_usage(nmslib_index_handle_t handle);

/* -- ingest (ref :717-918, :1567-1669).  Points are copied (as in the reference). */
nmslib_error_t nmslib_add_data_point(nmslib_index_handle_t index, const void* data,
                                     size_t element_count, int32_t id);
nmslib_error_t nmslib_add_data_point_batch(nmslib_index_handle_t index, const void* data,
                                           size_t count, size_t element_count,
                                           const int32_t* ids, const size_t* num_elements);
nmslib_error_t nmslib_add_data_point_batch_uint8(nmslib_index_handle_t index,
                                                 const unsigned char* data, size_t count,
                                                 size_t element_count, const int32_t* ids);
nmslib_error_t nmslib_add_data_point_batch_string(nmslib_index_handle_t index,
                                                  const char* const* data, size_t count,
                                                  const int32_t* ids);
nmslib_error_t nmslib_add_data_point_batch_pointers(nmslib_index_handle_t handle,
                                                    nmslib_data_mode_t data_mode,
                                                    const void* const* data_ptrs, size_t count,
                                                    size_t element_count, const int32_t* ids,
                                                    const size_t* num_elements);

/* -- THE HOT PATH (ref nmslib_c.cpp:920-1031; lib.zig:799-931) ------------- */
/* *out_size = k (ref :920-939). */
nmslib_error_t nmslib_knn_query_get_size(nmslib_index_handle_t index, const void* query,
                                         size_t query_size_or_elem_count, size_t k,
                                         size_t* out_size, size_t num_elements);
/* One query == a batch of one (ref :941-1001).  k == 0 is INVALID_ARGUMENT (Q8);
 * capacity < found is BUFFER_TOO_SMALL (Q9). */
nmslib_error_t nmslib_knn_query_fill(nmslib_index_handle_t index, const void* query,
                                     size_t query_size_or_elem_count, size_t k,
                                     nmslib_result_t* result, size_t num_elements);
/* ONE device submission for the whole batch (ref :1003-1031 is a serial loop).
 * queries is a flat [query_count][elem_count] array of the index's element type:
 * float32 for DENSE_VECTOR, uint8 for DENSE_UINT8_VECTOR (the reference strides by
 * sizeof(float) for every type, SURVEY Q6).  thread_pool_size is accepted and
 * ignored, as in the reference (:1008). */
nmslib_error_t nmslib_knn_query_batch(nmslib_index_handle_t index, const void* queries,
                                      size_t query_count, size_t query_size_or_elem_count,
                                      size_t k, nmslib_result_t* results,
                                      const size_t* num_elements, size_t thread_pool_size);
void nmslib_free_result(nmslib_result_t* result); /* ref nmslib_c.cpp:1671; lib.zig:8 */

/* -- outside this engine's path: exported, answer SPACE_INCOMPATIBLE ------- */
nmslib_error_t nmslib_range_query_get_size(nmslib_index_handle_t index, const void* query,
                                           size_t query_size_or_elem_count, double radius,
                                           size_t* out_size, size_t num_elements);
nmslib_error_t nmslib_range_query_fill(nmslib_index_handle_t index, const void* query,
                                       size_t query_size_or_elem_count, double radius,
                                       nmslib_result_t* result, size_t num_elements);
nmslib_error_t nmslib_get_data_point_string(nmslib_index_handle_t index, size_t position,
                                            const char** data, size_t* data_len,
                                            const nmslib_allocator_t* allocator);
nmslib_error_t nmslib_borrow_data_sparse(nmslib_index_handle_t index, size_t position,
                                         void** data, size_t* size, void (**free_fn)(void*));

/* -- data access served from the host copy (ref :1155-1367) ---------------- */
nmslib_error_t nmslib_get_distance(nmslib_index_handle_t index, size_t pos1, size_t pos2,
                                   float* distance);
nmslib_error_t nmslib_get_data_point_size(nmslib_index_handle_t index, size_t position,
                                          size_t* size);
nmslib_error_t nmslib_get_data_point_fill(nmslib_index_handle_t index, size_t position,
                                          void* data, size_t size);
nmslib_error_t nmslib_borrow_data_dense(nmslib_index_handle_t index, size_t position,
                                        void** data, size_t* size, void (**free_fn)(void*));

/* -- persistence (ref :1369-1479).  hnsw indexes are written / read in the
 * reference's optimized-index stream (hnsw.cc:774-806) plus the "<path>.dat"
 * dataset (space.cc:90-105), so files are interchangeable with the reference.
 * l2sqr_sift + hnsw (the reference's Hnsw<int>) writes the regular index file
 * instead (SaveRegularIndexBin, hnsw.cc:810-842: links only); loaded with
 * DENSE_UINT8_VECTOR it becomes an l2sqr_sift hnsw index over "<path>.dat",
 * so load_data must be 1 (DATA_IO_FAILED otherwise). */
nmslib_error_t nmslib_save_index(nmslib_index_handle_t index, const char* path, int save_data);
nmslib_error_t nmslib_load_index(const char* path, nmslib_data_type_t data_type,
                                 nmslib_dist_type_t dist_type,
                                 const nmslib_allocator_t* allocator, int load_data,
                                 nmslib_index_handle_t* out_handle);

/* ======================================================================== */
/* PART 2 -- nmslib_b200_* extensions                                         */
/* ======================================================================== */

/* Select the CUDA device used by indexes created afterwards on this thread
 * (default: $LOCAL_RANK if set, else 0).  Returns 0 / cudaError. */
int nmslib_b200_set_device(int device);
/* 1 if a CUDA device can be opened, else 0 (never throws). */
int nmslib_b200_device_available(void);

/* Shard placement for row-wise multi-GPU sharding (SURVEY 8e): positions inside
 * this index are reported as pos_base + local row so that (distance, position)
 * tie-breaking is global.  Call before the first query. */
nmslib_error_t nmslib_b200_set_shard(nmslib_index_handle_t index, uint32_t pos_base);

/* Import a graph written by the reference's Hnsw::SaveIndex (optimized flat index,
 * hnsw.cc:774-806).  The vectors and external ids stored in the file replace the
 * index's data; the search then runs on exactly the reference's graph. */
nmslib_error_t nmslib_b200_import_hnsw(nmslib_index_handle_t index, const char* path);

/* Force the lazy device upload now (idempotent). */
nmslib_error_t nmslib_b200_prepare(nmslib_index_handle_t index);

/* Device-resident batch query: d_queries is [q][elem_count] in device memory
 * (float32, or bytes for uint8 indexes, seq_search and hnsw alike), the outputs are device arrays.  d_keys ([q][k] uint64 = ordered(distance) << 32
 * | position) may be NULL.  Runs on `stream` (a cudaStream_t, may be NULL) and does
 * not synchronise.  Missing results (k > n) are id -1 / distance +inf. */
nmslib_error_t nmslib_b200_knn_device(nmslib_index_handle_t index, const void* d_queries,
                                      size_t query_count, size_t elem_count, size_t k,
                                      int32_t* d_ids, float* d_distances, uint64_t* d_keys,
                                      void* stream);

/* K-way merge of `lists` sorted top-k lists per query ([lists][q][k], as an
 * all-gather lays them out) into [q][k]: the cross-shard step of SURVEY 8e.
 * Ordering is by key (distance, then global position); the index handle supplies
 * the space's final distance transform (sqrt for l2, int->float for l2sqr_sift).
 * All pointers are device pointers (peer-mapped pointers are fine).  d_ids may be NULL when the external ids are
 * the global positions themselves (the low word of every key): the id lists then need not be exchanged at all. */
nmslib_error_t nmslib_b200_merge_topk(nmslib_index_handle_t index, const uint64_t* d_keys,
                                      const int32_t* d_ids, size_t lists, size_t query_count,
                                      size_t k, int32_t* d_out_ids, float* d_out_distances,
                                      void* stream);

typedef struct {
  uint64_t queries;          /* queries answered since creation */
  uint64_t kernel_launches;  /* launches of our own kernels */
  uint64_t distance_evals;   /* hnsw: vectors gathered; brute force: q * n */
  uint64_t hnsw_expansions;  /* hnsw: beam expansions */
  double last_kernel_ms;     /* CUDA-event time of the dominant kernel, last host call */
  double last_total_ms;      /* CUDA-event time h2d + kernels + d2h, last host call */
  uint64_t fallback_queries; /* queries re-run by the exact scan after a failed certificate */
  uint64_t device_bytes;     /* bytes resident in HBM for this index */
  double last_scan_ms;       /* CUDA-event time of the dominant kernel alone (scan / beam search) */
  double scan_ms_sum;        /* sum of that time over all launches resolved so far */
  uint64_t scan_count;       /* number of launches in scan_ms_sum */
  /* device-side HNSW construction (hnsw_build_gpu.cu); all zero when the graph was imported or built on the host */
  double build_total_ms;     /* whole build, CUDA events */
  double build_scan_ms;      /* candidate generation: prefix kNN on the tensor cores */
  double build_select_ms;    /* heuristic-2 neighbour selection of the new points */
  double build_link_ms;      /* back links: sort + append / re-prune */
  uint64_t build_batches;    /* insertion batches over all levels */
  uint64_t build_prunes;     /* neighbour lists re-pruned because they overflowed */
  uint64_t split_queries;    /* queries re-run by the 3xTF32 (split operand) scan after a failed certificate */
  uint64_t u8_imma;          /* 1: uint8 rows are scanned on the integer tensor pipe (tcgen05.mma.kind::i8), 0: widened to TF32 */
  uint64_t uploaded_rows;    /* rows copied host -> device so far (an append uploads only the new rows) */
  /* nmslib_b200_range_query_batch (b200_devices indexes: counted once per shard) */
  uint64_t range_tc_queries;       /* range queries whose answer came from the tensor-core pass (uint8 included) */
  uint64_t range_fallback_queries; /* range queries re-run by the per-query exact scan after an uncertified batched pass */
} nmslib_b200_stats_t;
nmslib_error_t nmslib_b200_get_stats(nmslib_index_handle_t index, nmslib_b200_stats_t* out);

/* Batched range queries (seq_search / brute_force).  `queries` is laid out like the input of
 * nmslib_knn_query_batch (query_count x elem_count floats, or bytes for uint8 indexes); radii[i] is query i's
 * radius and results[i] a caller-owned slot of results[i].capacity entries; results[i].size is set on return.
 * For every query the answer is exactly what nmslib_range_query_fill returns for it with radii[i] and
 * results[i].capacity: the objects within the radius in position order, truncated to the capacity, with the same
 * distance bits and the same radius conversions ((float)radius; floor for l2sqr_sift, RangeQuery<int>).
 * Errors: a negative radius, a NULL pointer or a capacity of 0 anywhere in the batch -> INVALID_ARGUMENT before
 * any work; a query length that does not match the index -> QUERY_EXECUTION_FAILED; hnsw -> SPACE_INCOMPATIBLE
 * (the reference has no range search over hnsw); an index that is not built -> INDEX_BUILD_FAILED, as for
 * nmslib_range_query_fill.  An empty index returns size 0 everywhere.
 * l2, l2sqr, cosinesimil, negdotprod, angulardist and l2sqr_sift run as one tensor-core pass over the rows for the
 * whole batch (a threshold per query, verified with the per-query scan's own distance code; uint8 byte rows on the
 * integer tensor pipe with an exact integer threshold, widened uint8 rows on the TF32 pass); l1 and linf run as one
 * pass of the exact CUDA-core scan with a threshold per query, verified the same way.  force_exact and, under option
 * tc_pair=0, rows of more than 128 floats in the tensor-core spaces use the per-query exact scan, as does any query a
 * batched pass cannot certify (nmslib_b200_stats_t counts the tensor-core answers and those re-runs).  A
 * b200_devices index answers over every shard and concatenates the shards' lists in position order. */
nmslib_error_t nmslib_b200_range_query_batch(nmslib_index_handle_t index, const void* queries,
                                             size_t query_count, size_t elem_count,
                                             const double* radii, nmslib_result_t* results);

/* Diagnostic (needs no device): the work decomposition the tensor-core scan would use for a batch of
 * `query_count` queries against `n` rows of at most 128 floats on a GPU with `sm_count` SMs.
 * Writes up to `capacity` pieces as 5 ints {cta, query block (256 queries), first tile, end tile, slot}
 * (tiles are 64 rows) and returns the number of pieces; *n_cta / *s_max receive the grid size and the
 * number of candidate lists per query block. */
size_t nmslib_b200_scan_plan(size_t query_count, size_t n, size_t k, int sm_count, int32_t* pieces,
                             size_t capacity, int* n_cta, int* s_max);

/* The same for rows of more than 128 floats, which run on CTA pairs (cta_group::2 MMAs): units are sm_count / 2
 * pairs, tiles are 256 rows, every piece fills two candidate lists (*s_max counts lists). */
size_t nmslib_b200_scan_plan_pairs(size_t query_count, size_t n, size_t k, int sm_count, int32_t* pieces,
                                   size_t capacity, int* n_pairs, int* s_max);

/* ---- row-sharded multi-GPU search behind this ABI (SURVEY 8e; the reference's chunk-and-merge, seqsearch.cc:151-175,
 * with a GPU per chunk).  Row shards are for seq_search / brute_force; an hnsw graph does not shard without changing its
 * answers, so under (A) an hnsw index gets one REPLICA of the graph per device and every device takes a contiguous
 * slice of each batch (no exchange; nmslib_set_query_time_params reaches every replica); (B) is seq_search only.
 *
 * (A) ONE process, several devices: pass the index parameter  b200_devices=0,1,2,3  ("0-7", "all") to
 *     nmslib_create_index.  nmslib_add_data_point* and nmslib_knn_query_batch / _fill are used unchanged: the rows are
 *     cut into contiguous shards at the first query, every batch is scanned by all devices concurrently, the per-shard
 *     (distance, global position) lists are exchanged through NVLink peer memory and merged on the devices.  Answers
 *     are bit-identical to the one-device index.
 *
 * (B) one process PER device (torchrun, MPI): every rank creates an ordinary index over its row shard
 *     (nmslib_b200_set_shard(first global row)), then
 *         nmslib_b200_shard_export(index, max_queries, max_k, blob)     allocates this rank's exchange window
 *         ... the caller all-gathers the NMSLIB_B200_SHARD_BLOB_BYTES-byte blobs over any host channel ...
 *         nmslib_b200_shard_connect(index, rank, world, blobs)          maps the peers' windows (CUDA IPC)
 *     after which nmslib_knn_query_batch and nmslib_b200_knn_device return the GLOBAL top-k on every rank: the call
 *     publishes this shard's lists, waits (on the device) for the peers' lists of the same call and merges them.  Like
 *     a collective, every rank must make the same sequence of calls (same query_count and k). */
#define NMSLIB_B200_SHARD_BLOB_BYTES 256
nmslib_error_t nmslib_b200_shard_export(nmslib_index_handle_t index, size_t max_queries, size_t max_k, void* blob);
nmslib_error_t nmslib_b200_shard_connect(nmslib_index_handle_t index, int rank, int world, const void* blobs);
nmslib_error_t nmslib_b200_shard_disconnect(nmslib_index_handle_t index);

/* Process-wide variant selectors (every variant returns the same answers; used for A/B comparisons):
 *   "tc_pair"     1 (default) rows of more than 128 floats on CTA pairs / 0 the single-CTA long-row kernel
 *   "hnsw_team"   -1 (default) auto / 0 one warp per query / 2, 4 teams of that many warps per query
 *   "force_exact" 0 (default) / 1 CUDA-core exact scan only (read when an index is created)
 *   "tc_split"    1 (default) / 0 never switch to split (3xTF32) operands
 *   "u8_imma"     1 (default) uint8 rows on the integer tensor pipe / 0 rows widened to TF32 operands
 * Unknown names are INVALID_ARGUMENT.  The NB200_* timing / debugging environment variables of the tools exist only
 * in -DNB200_EXPERIMENTS builds of the library; the release build never reads the environment for them. */
nmslib_error_t nmslib_b200_set_option(const char* name, int value);

/* Library build / arch string, e.g. "nmslib_b200 0.1 sm_100a". Static storage. */
const char* nmslib_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NMSLIB_B200_H */
