// ID selectors of faiss::Index::remove_ids and of filtered search (reference AuxIndexStructures.h: IDSelector,
// IDSelectorRange, IDSelectorBatch, IDSelectorBitmap, IDSelectorNot) and the result of faiss::Index::range_search
// (RangeSearchResult).  The device indexes cannot call a virtual is_member per entry: they recognise these types and
// hand the range bounds, the sorted id array or the bitmap to their kernels (vlq_remove_ids_plan takes Range and Batch,
// vlq_filter_kappa all four).  is_member stays for host callers.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>
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

/// bit (id & 7) of bitmap[id >> 3] over n bytes (reference IDSelectorBitmap); ids outside [0, 8 n) are not members.
/// The bitmap is borrowed, in host or device memory (the device search reads either; is_member needs host memory).
struct IDSelectorBitmap : IDSelector {
  size_t n;
  const uint8_t* bitmap;
  IDSelectorBitmap(size_t n_, const uint8_t* bitmap_) : n(n_), bitmap(bitmap_) {}
  bool is_member(idx_t id) const override {
    const uint64_t u = (uint64_t)id;  // a negative id wraps past the end
    return (u >> 3) < n && ((bitmap[u >> 3] >> (u & 7)) & 1);
  }
};

/// the complement of a borrowed selector (reference IDSelectorNot)
struct IDSelectorNot : IDSelector {
  const IDSelector* sel;
  explicit IDSelectorNot(const IDSelector* sel_) : sel(sel_) {}
  bool is_member(idx_t id) const override { return !sel->is_member(id); }
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
