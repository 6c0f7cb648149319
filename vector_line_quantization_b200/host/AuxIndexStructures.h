// ID selectors of faiss::Index::remove_ids (reference AuxIndexStructures.h: IDSelector, IDSelectorRange,
// IDSelectorBatch) and the result of faiss::Index::range_search (RangeSearchResult).  The device indexes cannot call a virtual is_member per entry: they recognise these two types and
// hand the range bounds or the sorted id array to the compaction kernels (vlq_remove_ids_plan).  is_member stays for
// host callers.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstring>
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

/// the results of range_search for nq queries (reference AuxIndexStructures.h): the results of query i are
/// labels / distances [lims[i], lims[i + 1]).  The index writes the per-query counts into lims[0 .. nq) and calls
/// do_allocation(), which turns them into offsets and allocates the two arrays; the destructor frees them.
struct RangeSearchResult {
  typedef Index::idx_t idx_t;
  size_t nq;
  size_t* lims;       ///< [nq + 1]
  idx_t* labels;      ///< [lims[nq]]
  float* distances;   ///< [lims[nq]]
  size_t buffer_size; ///< kept for source compatibility: the results are assembled in one piece

  explicit RangeSearchResult(idx_t nq_, bool alloc_lims = true)
      : nq((size_t)nq_), lims(nullptr), labels(nullptr), distances(nullptr), buffer_size(1024 * 256) {
    if (alloc_lims) {
      lims = new size_t[nq + 1];
      std::memset(lims, 0, sizeof(size_t) * (nq + 1));
    }
  }
  RangeSearchResult(const RangeSearchResult&) = delete;
  RangeSearchResult& operator=(const RangeSearchResult&) = delete;

  virtual void do_allocation() {
    size_t ofs = 0;
    for (size_t i = 0; i < nq; i++) {
      const size_t n = lims[i];
      lims[i] = ofs;
      ofs += n;
    }
    lims[nq] = ofs;
    delete[] labels;
    delete[] distances;
    labels = new idx_t[ofs];
    distances = new float[ofs];
  }

  virtual ~RangeSearchResult() {
    delete[] labels;
    delete[] distances;
    delete[] lims;
  }
};

}  // namespace faiss
