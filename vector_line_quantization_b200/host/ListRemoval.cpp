#include "ListRemoval.h"

#include <algorithm>

namespace faiss {
namespace gpu {

long removeFromLists(GpuResources* res, const IDSelector& sel, int64_t nlists, int M, ListSlab slab) {
  const IDSelectorRange* range = dynamic_cast<const IDSelectorRange*>(&sel);
  const IDSelectorBatch* batch = dynamic_cast<const IDSelectorBatch*>(&sel);
  VLQ_THROW_IF_NOT_MSG(range || batch, "remove_ids: only IDSelectorRange and IDSelectorBatch are supported");
  const int64_t n = (int64_t)slab.nListed;
  if (n == 0 || (range && range->imin >= range->imax) || (batch && batch->ids.empty())) return 0;
  vlq_stream_t st = res->getDefaultStream();
  DeviceBuffer dBatch;
  const int64_t nb = batch ? (int64_t)batch->ids.size() : 0;
  if (batch) {
    dBatch.resize((size_t)nb * sizeof(int64_t));
    VLQ_CALL(vlq_memcpy_h2d(dBatch.get(), batch->ids.data(), dBatch.bytes(), st));
  }
  const int64_t lo = range ? range->imin : 0, hi = range ? range->imax : 0;
  DeviceBuffer ws(vlq_remove_ids_workspace_bytes(n, nlists)), no((size_t)(nlists + 1) * sizeof(int64_t));
  VLQ_CALL(vlq_remove_ids_plan(nlists, n, slab.offsets.as<int64_t>(), slab.ids.as<int64_t>(), lo, hi,
                               dBatch.as<int64_t>(), nb, no.as<int64_t>(), ws.get(), ws.bytes(), st));
  int64_t live = 0;
  VLQ_CALL(vlq_memcpy_d2h(&live, no.as<int64_t>() + nlists, sizeof(int64_t), st));
  res->syncDefaultStream();
  if (live == n) return 0;  // nothing selected: the slab stays as it is
  const size_t keep = std::max<size_t>(1, (size_t)live);
  DeviceBuffer nc(keep * M), nq(keep), nk(keep * sizeof(float)), ni(keep * sizeof(int64_t));
  VLQ_CALL(vlq_remove_ids_apply(nlists, M, n, slab.offsets.as<int64_t>(), slab.codes.as<uint8_t>(),
                                slab.lamq.as<uint8_t>(), slab.kappa.as<float>(), slab.ids.as<int64_t>(),
                                no.as<int64_t>(), nc.as<uint8_t>(), nq.as<uint8_t>(), nk.as<float>(), ni.as<int64_t>(),
                                ws.get(), ws.bytes(), st));
  res->syncDefaultStream();
  slab.offsets.swap(no);
  slab.codes.swap(nc);
  slab.lamq.swap(nq);
  slab.kappa.swap(nk);
  slab.ids.swap(ni);
  slab.nListed = (size_t)live;
  return (long)(n - live);
}

}  // namespace gpu
}  // namespace faiss
