// range_search over the CSR list slab that GpuIndexIVFPQ and GpuIndexIMIPQ share (offsets / codes / lamq / kappa / ids,
// csrc/lists.cu).  Each index supplies its coarse stage (the W lines of every query of a tile with their term1 / term6);
// per query tile the helper then counts the results on the device (vlq_range_count), reads the tile's lims (one host
// synchronisation per tile: the result sizes decide the buffers), gathers the results in query sub-ranges that fit a
// bounded device staging buffer (vlq_range_gather) and downloads them.  The result is assembled through
// RangeSearchResult::do_allocation().
#pragma once
#include <cstddef>
#include <cstdint>
#include <functional>

#include "AuxIndexStructures.h"
#include "GpuResources.h"

namespace faiss {
namespace gpu {

/// the committed slab and the scan tables of an index (device pointers)
struct RangeLists {
  const float* pq;        ///< (M, 256, d / M)
  int M;
  const float* lambdaCb;  ///< [nLambda]
  int nLambda;
  const float* edgeDist;  ///< per-list squared edge length (term5); nullptr = 0 (IMI-PQ)
  int W;                  ///< lines per query
  int cap;                ///< entries scanned per line at most
  const int64_t* offsets;
  const uint8_t* codes;
  const uint8_t* lamq;
  const float* kappa;
  const int64_t* ids;
  size_t nListed;         ///< entries in the slab
  bool addQueryNorm;      ///< term1 excludes ||q||^2 (the VLQ coarse stage): add it back for the full distance
  Index::idx_t tile;      ///< queries per coarse stage at most
};

/// lines / term1 / term6 [m][W] of the m queries at the device pointer dq, on the resource's default stream
using RangeCoarseStage = std::function<void(const float* dq, Index::idx_t m, int* lines, float* term1, float* term6)>;

/// every entry of the selected lines with full squared distance < radius, for the n queries at x (host or device).
/// Staging: at most VLQ_RANGE_STAGING_BYTES (environment, read on every call; default 1 GiB) of results per gather,
/// except that a single query's results always fit.
void rangeSearchLists(GpuResources* res, int d, Index::idx_t n, const float* x, float radius, const RangeLists& lists,
                      const RangeCoarseStage& coarse, RangeSearchResult* result);

}  // namespace gpu
}  // namespace faiss
