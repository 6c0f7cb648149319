// Filtered search over the lists of DeviceLists.h: the selector of SearchParameters becomes a masked copy of the
// per-entry kappa (DeviceLists::kappa: +inf for every entry whose id the selector does not hold), and the unchanged
// scan / range kernels run on that copy.  A masked entry's distance is +inf, so it ranks after every real result;
// vlq_filter_results turns the (+inf, id) rows a scan may return for a query with fewer than k members into the usual
// (FLT_MAX, -1) padding.
#pragma once

#include "AuxIndexStructures.h"

namespace faiss {
namespace gpu {

/// the selector of params, or nullptr for an unfiltered call
inline const IDSelector* searchSelector(const SearchParameters* params) { return params ? params->sel : nullptr; }

/// what vlq_filter_kappa evaluates: one of range / batch / bitmap, and whether the result is negated
struct DeviceSelector {
  const IDSelectorRange* range = nullptr;
  const IDSelectorBatch* batch = nullptr;
  const IDSelectorBitmap* bitmap = nullptr;
  bool invert = false;
};

/// the DeviceSelector of `sel`; throws FaissException unless `sel` is an IDSelectorRange, IDSelectorBatch or
/// IDSelectorBitmap, or an IDSelectorNot (nested any number of times) of one of them -- the types the device mask can
/// evaluate.  Launches nothing.
DeviceSelector checkSearchSelector(const IDSelector* sel);

}  // namespace gpu
}  // namespace faiss
