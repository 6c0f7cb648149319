// ID selectors of faiss::Index::remove_ids (reference AuxIndexStructures.h: IDSelector, IDSelectorRange,
// IDSelectorBatch).  The device indexes cannot call a virtual is_member per entry: they recognise these two types and
// hand the range bounds or the sorted id array to the compaction kernels (vlq_remove_ids_plan).  is_member stays for
// host callers.
#pragma once
#include <algorithm>
#include <vector>

#include "Index.h"

namespace faiss {

struct IDSelector {
  typedef Index::idx_t idx_t;
  virtual bool is_member(idx_t id) const = 0;
  virtual ~IDSelector() {}
};

/// the half-open range [imin, imax)
struct IDSelectorRange : IDSelector {
  idx_t imin, imax;
  IDSelectorRange(idx_t imin_, idx_t imax_) : imin(imin_), imax(imax_) {}
  bool is_member(idx_t id) const override { return id >= imin && id < imax; }
};

/// an explicit set of ids, kept sorted and de-duplicated (the array the device search takes; the reference puts a
/// hash set behind a Bloom filter here)
struct IDSelectorBatch : IDSelector {
  std::vector<idx_t> ids;
  IDSelectorBatch(idx_t n, const idx_t* indices) : ids(indices, indices + (n > 0 ? n : 0)) {
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
  }
  bool is_member(idx_t id) const override { return std::binary_search(ids.begin(), ids.end(), id); }
};

}  // namespace faiss
