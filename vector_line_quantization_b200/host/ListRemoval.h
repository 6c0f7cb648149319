// remove_ids over the CSR list slab that GpuIndexIVFPQ and GpuIndexIMIPQ share (offsets / codes / lamq / kappa / ids,
// csrc/lists.cu): the selector becomes a range or a sorted id array, vlq_remove_ids_plan counts the survivors, the new
// slab is allocated at its exact size and vlq_remove_ids_apply fills it.  Peak device memory: old + new slab.
#pragma once
#include <cstddef>
#include <cstdint>

#include "AuxIndexStructures.h"
#include "GpuResources.h"

namespace faiss {
namespace gpu {

struct ListSlab {
  DeviceBuffer& offsets;
  DeviceBuffer& codes;
  DeviceBuffer& lamq;
  DeviceBuffer& kappa;
  DeviceBuffer& ids;
  size_t& nListed;
};

/// removes the selected entries of a committed slab of nlists lists (M code bytes per entry) and returns their number.
/// Throws FaissException for a selector other than IDSelectorRange / IDSelectorBatch: there is no per-entry virtual
/// call on the device and no host path.
long removeFromLists(GpuResources* res, const IDSelector& sel, int64_t nlists, int M, ListSlab slab);

}  // namespace gpu
}  // namespace faiss
