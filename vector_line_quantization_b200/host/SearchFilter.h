// Filtered search over the CSR list slab that GpuIndexIVFPQ and GpuIndexIMIPQ share (csrc/lists.cu): the selector of
// SearchParameters becomes a masked copy of the per-entry kappa (vlq_filter_kappa: +inf for every entry whose id the
// selector does not hold), and the unchanged scan / range kernels run on that copy.  A masked entry's distance is +inf,
// so it ranks after every real result; vlq_filter_results turns the (+inf, id) rows a scan may return for a query
// with fewer than k members into the usual (FLT_MAX, -1) padding.
#pragma once
#include <cstddef>
#include <cstdint>

#include "AuxIndexStructures.h"
#include "GpuResources.h"

namespace faiss {
namespace gpu {

/// the selector of params, or nullptr for an unfiltered call
inline const IDSelector* searchSelector(const SearchParameters* params) { return params ? params->sel : nullptr; }

/// throws FaissException unless `sel` is an IDSelectorRange, IDSelectorBatch or IDSelectorBitmap, or an IDSelectorNot
/// (nested any number of times) of one of them -- the types the device mask can evaluate.  Launches nothing.
void checkSearchSelector(const IDSelector* sel);

/// kappa[n] masked by `sel` into `masked` (grow-only, 4 B per entry), on the default stream of `res`: the pointer the
/// scan of a filtered call reads.  A host batch or bitmap is uploaded first; a device bitmap is read in place.  n = 0
/// returns kappa.  Throws (before any launch) for a selector checkSearchSelector rejects.
const float* maskKappa(GpuResources* res, const IDSelector& sel, const int64_t* ids, const float* kappa, size_t n,
                       DeviceBuffer& masked);

}  // namespace gpu
}  // namespace faiss
