#include "SearchFilter.h"

namespace faiss {
namespace gpu {

namespace {

/// what vlq_filter_kappa evaluates: one of range / batch / bitmap, and whether the result is negated
struct DeviceSelector {
  const IDSelectorRange* range = nullptr;
  const IDSelectorBatch* batch = nullptr;
  const IDSelectorBitmap* bitmap = nullptr;
  bool invert = false;
};

DeviceSelector recognise(const IDSelector* sel) {
  DeviceSelector s;
  while (const IDSelectorNot* no = dynamic_cast<const IDSelectorNot*>(sel)) {  // Not(Not(x)) folds to x
    s.invert = !s.invert;
    sel = no->sel;
  }
  s.range = dynamic_cast<const IDSelectorRange*>(sel);
  s.batch = dynamic_cast<const IDSelectorBatch*>(sel);
  s.bitmap = dynamic_cast<const IDSelectorBitmap*>(sel);
  VLQ_THROW_IF_NOT_MSG(s.range || s.batch || s.bitmap,
                       "search: the selector must be an IDSelectorRange, IDSelectorBatch or IDSelectorBitmap, or an "
                       "IDSelectorNot of one of them");
  VLQ_THROW_IF_NOT_MSG(!s.bitmap || s.bitmap->n == 0 || s.bitmap->bitmap, "search: IDSelectorBitmap has a null bitmap");
  return s;
}

}  // namespace

void checkSearchSelector(const IDSelector* sel) { recognise(sel); }

const float* maskKappa(GpuResources* res, const IDSelector& sel, const int64_t* ids, const float* kappa, size_t n,
                       DeviceBuffer& masked) {
  const DeviceSelector s = recognise(&sel);
  if (n == 0) return kappa;
  vlq_stream_t st = res->getDefaultStream();
  DeviceBuffer dBatch, dBitmap;
  const int64_t nb = s.batch ? (int64_t)s.batch->ids.size() : 0;
  if (nb > 0) {  // IDSelectorBatch keeps its ids sorted and unique on the host
    dBatch.resize((size_t)nb * sizeof(int64_t));
    VLQ_CALL(vlq_memcpy_h2d(dBatch.get(), s.batch->ids.data(), dBatch.bytes(), st));
  }
  const int64_t nbytes = s.bitmap ? (int64_t)s.bitmap->n : 0;
  const uint8_t* bitmap = nbytes > 0 ? s.bitmap->bitmap : nullptr;
  if (nbytes > 0 && vlq_pointer_is_device(bitmap) != 1) {
    dBitmap.resize((size_t)nbytes);
    VLQ_CALL(vlq_memcpy_h2d(dBitmap.get(), bitmap, (size_t)nbytes, st));
    bitmap = dBitmap.as<uint8_t>();
  }
  const int64_t lo = s.range ? s.range->imin : 0, hi = s.range ? s.range->imax : 0;
  masked.reserve(n * sizeof(float));
  VLQ_CALL(vlq_filter_kappa((int64_t)n, ids, kappa, lo, hi, dBatch.as<int64_t>(), nb, bitmap, nbytes, s.invert ? 1 : 0,
                            masked.as<float>(), st));
  if (dBatch.get() || dBitmap.get()) res->syncDefaultStream();  // the uploads outlive the pass that reads them
  return masked.as<float>();
}

}  // namespace gpu
}  // namespace faiss
