// shard_group.h -- several GPUs of one process behind one index handle (see shard_group.cu).
#pragma once
#include <string>
#include <vector>

#include "engine.h"

namespace nb200 {

class ShardGroup {
 public:
  ShardGroup(Space space, Method method, bool is_u8, const std::vector<int>& devices);
  ~ShardGroup();
  ShardGroup(const ShardGroup&) = delete;
  ShardGroup& operator=(const ShardGroup&) = delete;

  // "0,1,2,3", "0-7" or "all" -> device ordinals (a device may be named twice: two shards on one GPU)
  static Status parse_devices(const std::string& spec, std::vector<int>* out);
  void set_index_params(const std::vector<std::string>& p);
  Status set_query_params(const std::vector<std::string>& p);  // hnsw replicas: efSearch & co. reach every replica
  size_t world() const;
  // host in / host out over all shards: ids / dists / counts point at the group's pinned result arrays
  Status knn_host(Engine* host_store, const void* queries, size_t nq, size_t elem_count, size_t k, const int32_t** ids,
                  const float** dists, const int32_t** counts);
  // batched range queries (seq_search): every shard answers over its rows, the lists are concatenated in shard order
  Status range_host(Engine* host_store, const void* queries, size_t nq, size_t elem_count, const double* radii,
                    const size_t* caps, int32_t* const* ids, float* const* dists, size_t* sizes);
  Status prepare(Engine* host_store, size_t nq, size_t k);
  Stats stats();

 private:
  struct Impl;
  Impl* impl_;
};

}  // namespace nb200
