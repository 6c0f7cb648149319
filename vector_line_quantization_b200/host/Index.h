// faiss::Index -- the operator interface the VLQ hot path sits behind (drop-in boundary, SURVEY.md 8b).
// Written from scratch to mirror the reference's public contract (reference Index.h:60-188): same member names,
// argument meaning, padding conventions (-1 labels / FLT_MAX distances) and error behaviour (FaissException for user
// errors).  idx_t = long; matrices are row-major compact float32; pointers may be host or device.
#pragma once
#include <algorithm>
#include <cstdio>
#include <exception>
#include <limits>
#include <string>

namespace faiss {

enum MetricType { METRIC_INNER_PRODUCT = 0, METRIC_L2 = 1 };

struct IDSelector;
struct RangeSearchResult;

/// user-facing errors (reference FaissAssert.h:54-91 throws; invariants abort)
class FaissException : public std::exception {
 public:
  explicit FaissException(const std::string& m) : msg(m) {}
  FaissException(const std::string& m, const char* func, const char* file, int line) {
    char buf[1024];
    snprintf(buf, sizeof(buf), "Error in %s at %s:%d: %s", func, file, line, m.c_str());
    msg = buf;
  }
  const char* what() const noexcept override { return msg.c_str(); }
  std::string msg;
};

#define VLQ_THROW_MSG(MSG) throw ::faiss::FaissException(MSG, __PRETTY_FUNCTION__, __FILE__, __LINE__)
#define VLQ_THROW_IF_NOT_MSG(COND, MSG) \
  do {                                   \
    if (!(COND)) VLQ_THROW_MSG(MSG);     \
  } while (0)
#define VLQ_THROW_IF_NOT(COND) VLQ_THROW_IF_NOT_MSG(COND, "'" #COND "' failed")

struct Index {
  typedef long idx_t;

  int d;
  idx_t ntotal;
  bool verbose;
  bool is_trained;
  MetricType metric_type;

  explicit Index(idx_t d_ = 0, MetricType metric = METRIC_L2)
      : d((int)d_), ntotal(0), verbose(false), is_trained(true), metric_type(metric) {}
  virtual ~Index() {}

  virtual void train(idx_t /*n*/, const float* /*x*/) {}
  virtual void add(idx_t n, const float* x) = 0;
  virtual void add_with_ids(idx_t /*n*/, const float* /*x*/, const long* /*xids*/) {
    VLQ_THROW_MSG("add_with_ids not implemented for this type of index");
  }
  virtual void search(idx_t n, const float* x, idx_t k, float* distances, idx_t* labels) const = 0;
  virtual void reset() = 0;

  /// stored vector `key` (reference Index.h:157; indexes that cannot decode throw, Index.cpp:49-51)
  virtual void reconstruct(idx_t /*key*/, float* /*recons*/) const { VLQ_THROW_MSG("reconstruct not implemented for this type of index"); }
  /// stored vectors [i0, i0 + ni) (reference Index.cpp:54-59: one reconstruct per row unless overridden)
  virtual void reconstruct_n(idx_t i0, idx_t ni, float* recons) const {
    for (idx_t i = 0; i < ni; i++) reconstruct(i0 + i, recons + i * d);
  }
  /// stored vectors of keys[0 .. n) (reference Index.h reconstruct_batch: one reconstruct per key unless overridden)
  virtual void reconstruct_batch(idx_t n, const idx_t* keys, float* recons) const {
    for (idx_t i = 0; i < n; i++) reconstruct(keys[i], recons + i * d);
  }
  /// search, then the stored vector behind every label; rows of label -1 are NaN (reference Index.cpp
  /// search_and_reconstruct).  recons is [n][k][d].
  virtual void search_and_reconstruct(idx_t n, const float* x, idx_t k, float* distances, idx_t* labels,
                                      float* recons) const {
    search(n, x, k, distances, labels);
    for (idx_t i = 0; i < n * k; i++) {
      float* r = recons + i * d;
      if (labels[i] < 0) std::fill(r, r + d, std::numeric_limits<float>::quiet_NaN());
      else reconstruct(labels[i], r);
    }
  }

  /// remove the entries whose id the selector holds; returns how many were removed (reference Index.h remove_ids;
  /// selectors in AuxIndexStructures.h)
  virtual long remove_ids(const IDSelector& /*sel*/) { VLQ_THROW_MSG("remove_ids not implemented for this type of index"); }

  /// every stored vector closer than `radius` to each query (reference Index.h range_search; METRIC_L2: squared
  /// distance < radius).  result->nq == n; the index fills lims, labels and distances (RangeSearchResult,
  /// AuxIndexStructures.h)
  virtual void range_search(idx_t /*n*/, const float* /*x*/, float /*radius*/, RangeSearchResult* /*result*/) const {
    VLQ_THROW_MSG("range_search not implemented for this type of index");
  }

  /// labels of the k nearest neighbours (= search without the distances; reference Index.cpp:23-29)
  void assign(idx_t n, const float* x, idx_t* labels, idx_t k = 1);
};

}  // namespace faiss
