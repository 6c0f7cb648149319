// Multi-index wrappers of the reference, for several GPUs driven from ONE process:
//   IndexProxy  (reference gpu/IndexProxy.{h,cpp}:24-168): REPLICAS -- train/add go to every sub-index, search splits
//               the queries ceil(n / #indexes) per replica, one thread each, no merge.
//   IndexShards (reference MetaIndexes.{h,cpp}:290-347,486-563): DATABASE SHARDS -- every shard searches all queries,
//               the (nshard, n, k) results are merged; here the merge is the device kernel vlq_merge_topk.
// (The benchmark's multi-GPU path is one process per GPU with NCCL; these classes are the in-process equivalents.)
#pragma once
#include <vector>

#include "Index.h"

namespace faiss {
namespace gpu {

class IndexProxy : public faiss::Index {
 public:
  IndexProxy() : Index(0, faiss::METRIC_L2) {}
  void addIndex(faiss::Index* index);
  void removeIndex(faiss::Index* index);
  void runOnIndex(void (*f)(faiss::Index*, void*), void* arg);
  void reset() override;
  void train(Index::idx_t n, const float* x) override;
  void add(Index::idx_t n, const float* x) override;
  using Index::search;  // the SearchParameters overload: no filtering here (a selector throws)
  void search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const override;
  size_t count() const { return indices_.size(); }

 private:
  std::vector<faiss::Index*> indices_;
};

}  // namespace gpu

class IndexShards : public faiss::Index {
 public:
  /// successive_ids: shard s returns local ids, shifted by the sizes of the shards before it (MetaIndexes.h)
  explicit IndexShards(idx_t d, bool threaded = true, bool successive_ids = true);
  void add_shard(Index* index);
  void train(idx_t n, const float* x) override;
  void add(idx_t n, const float* x) override;  ///< splits the rows evenly over the shards (MetaIndexes.cpp:402-440)
  using Index::search;  // the SearchParameters overload: no filtering here (a selector throws)
  void search(idx_t n, const float* x, idx_t k, float* distances, idx_t* labels) const override;
  void reset() override;
  std::vector<Index*> shard_indexes;
  bool threaded;
  bool successive_ids;

 private:
  /// all shards are GPU indexes: device result buffers + merge kernel reading them over NVLink
  void searchPeers_(const std::vector<int>& dev, idx_t n, const float* x, idx_t k, float* distances, idx_t* labels) const;
};

}  // namespace faiss
