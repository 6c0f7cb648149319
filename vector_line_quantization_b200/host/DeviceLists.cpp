#include "DeviceLists.h"

#include <algorithm>
#include <utility>

#include "SearchFilter.h"

namespace faiss {
namespace gpu {

DeviceLists::DeviceLists(GpuResources* res, int64_t nlists, int M, int auxWidth)
    : res_(res), nlists_(nlists), M_(M), auxWidth_(auxWidth) {
  VLQ_THROW_IF_NOT_MSG(auxWidth >= 0 && auxWidth <= 64, "aux column width must be in [0, 64]");
}

DeviceLists::Slots DeviceLists::makeRoom(size_t n) {
  const size_t need = nPending_ + n;
  if (need > capPending_) {
    vlq_stream_t st = res_->getDefaultStream();
    const size_t cap = std::max({need, 2 * capPending_, reserveVecs_, (size_t)1 << 16});
    DeviceBuffer nl(cap * sizeof(int));
    Columns nc(cap, M_, auxWidth_);
    if (nPending_) {
      VLQ_CALL(vlq_memcpy_d2d(nl.get(), pList_.get(), nPending_ * sizeof(int), st));
      VLQ_CALL(vlq_memcpy_d2d(nc.codes.get(), pending_.codes.get(), nPending_ * M_, st));
      VLQ_CALL(vlq_memcpy_d2d(nc.lamq.get(), pending_.lamq.get(), nPending_, st));
      VLQ_CALL(vlq_memcpy_d2d(nc.kappa.get(), pending_.kappa.get(), nPending_ * sizeof(float), st));
      VLQ_CALL(vlq_memcpy_d2d(nc.ids.get(), pending_.ids.get(), nPending_ * sizeof(int64_t), st));
      if (auxWidth_) VLQ_CALL(vlq_memcpy_d2d(nc.aux.get(), pending_.aux.get(), nPending_ * auxWidth_, st));
      res_->syncDefaultStream();
    }
    pList_ = std::move(nl);
    pending_ = std::move(nc);
    capPending_ = cap;
  }
  const size_t o = nPending_;
  return Slots{pList_.as<int>() + o, pending_.codes.as<uint8_t>() + o * M_, pending_.lamq.as<uint8_t>() + o,
               pending_.kappa.as<float>() + o, pending_.ids.as<int64_t>() + o,
               auxWidth_ ? pending_.aux.as<uint8_t>() + o * auxWidth_ : nullptr};
}

void DeviceLists::appended(size_t n) {
  VLQ_THROW_IF_NOT(nPending_ + n <= capPending_);
  nPending_ += n;
}

void DeviceLists::commit(DeviceBuffer& workspace) {
  if (nPending_ == 0 && offsets_.get()) return;
  vlq_stream_t st = res_->getDefaultStream();
  const size_t tot = n_ + nPending_;
  DeviceBuffer no((size_t)(nlists_ + 1) * sizeof(int64_t));
  Columns nc(tot, M_, auxWidth_);
  workspace.reserve(vlq_build_lists_workspace_bytes((int64_t)nPending_, nlists_));
  VLQ_CALL(vlq_build_lists_aux(nlists_, M_, auxWidth_, (int64_t)n_, offsets_.as<int64_t>(), slab_.codes.as<uint8_t>(),
                               slab_.lamq.as<uint8_t>(), slab_.kappa.as<float>(), slab_.ids.as<int64_t>(),
                               slab_.aux.as<uint8_t>(), (int64_t)nPending_, pList_.as<int>(),
                               pending_.codes.as<uint8_t>(), pending_.lamq.as<uint8_t>(), pending_.kappa.as<float>(),
                               pending_.ids.as<int64_t>(), pending_.aux.as<uint8_t>(), no.as<int64_t>(),
                               nc.codes.as<uint8_t>(), nc.lamq.as<uint8_t>(), nc.kappa.as<float>(), nc.ids.as<int64_t>(),
                               nc.aux.as<uint8_t>(), workspace.get(), workspace.bytes(), st));
  // entries the encoder skipped (list id < 0) are not stored: the live count is offsets[nlists]
  int64_t live = 0;
  VLQ_CALL(vlq_memcpy_d2h(&live, no.as<int64_t>() + nlists_, sizeof(int64_t), st));
  res_->syncDefaultStream();
  offsets_ = std::move(no);
  slab_ = std::move(nc);
  n_ = (size_t)live;
  nPending_ = 0;
  if (capPending_ > ((size_t)1 << 21)) {  // keep at most one add-chunk worth of arena
    pList_.release();
    pending_ = Columns();
    capPending_ = 0;
    reserveVecs_ = 0;
  }
}

long DeviceLists::remove(const IDSelector& sel) {
  const IDSelectorRange* range = dynamic_cast<const IDSelectorRange*>(&sel);
  const IDSelectorBatch* batch = dynamic_cast<const IDSelectorBatch*>(&sel);
  VLQ_THROW_IF_NOT_MSG(range || batch, "remove_ids: only IDSelectorRange and IDSelectorBatch are supported");
  const int64_t n = (int64_t)n_;
  if (n == 0 || (range && range->imin >= range->imax) || (batch && batch->ids.empty())) return 0;
  vlq_stream_t st = res_->getDefaultStream();
  DeviceBuffer dBatch;
  const int64_t nb = batch ? (int64_t)batch->ids.size() : 0;
  if (batch) {
    dBatch.resize((size_t)nb * sizeof(int64_t));
    VLQ_CALL(vlq_memcpy_h2d(dBatch.get(), batch->ids.data(), dBatch.bytes(), st));
  }
  const int64_t lo = range ? range->imin : 0, hi = range ? range->imax : 0;
  DeviceBuffer ws(vlq_remove_ids_workspace_bytes(n, nlists_)), no((size_t)(nlists_ + 1) * sizeof(int64_t));
  VLQ_CALL(vlq_remove_ids_plan(nlists_, n, offsets_.as<int64_t>(), slab_.ids.as<int64_t>(), lo, hi, dBatch.as<int64_t>(),
                               nb, no.as<int64_t>(), ws.get(), ws.bytes(), st));
  int64_t live = 0;
  VLQ_CALL(vlq_memcpy_d2h(&live, no.as<int64_t>() + nlists_, sizeof(int64_t), st));
  res_->syncDefaultStream();
  if (live == n) return 0;  // nothing selected: the slab stays as it is
  Columns nc(std::max<size_t>(1, (size_t)live), M_, auxWidth_);
  VLQ_CALL(vlq_remove_ids_apply_aux(nlists_, M_, auxWidth_, n, offsets_.as<int64_t>(), slab_.codes.as<uint8_t>(),
                                    slab_.lamq.as<uint8_t>(), slab_.kappa.as<float>(), slab_.ids.as<int64_t>(),
                                    slab_.aux.as<uint8_t>(), no.as<int64_t>(), nc.codes.as<uint8_t>(),
                                    nc.lamq.as<uint8_t>(), nc.kappa.as<float>(), nc.ids.as<int64_t>(),
                                    nc.aux.as<uint8_t>(), ws.get(), ws.bytes(), st));
  res_->syncDefaultStream();
  offsets_ = std::move(no);
  slab_ = std::move(nc);
  n_ = (size_t)live;
  return (long)(n - live);
}

const float* DeviceLists::kappa(const IDSelector* sel) {
  if (!sel) return slab_.kappa.as<float>();
  const DeviceSelector s = checkSearchSelector(sel);
  if (n_ == 0) return slab_.kappa.as<float>();
  vlq_stream_t st = res_->getDefaultStream();
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
  masked_.reserve(n_ * sizeof(float));
  VLQ_CALL(vlq_filter_kappa((int64_t)n_, slab_.ids.as<int64_t>(), slab_.kappa.as<float>(), lo, hi, dBatch.as<int64_t>(),
                            nb, bitmap, nbytes, s.invert ? 1 : 0, masked_.as<float>(), st));
  if (dBatch.get() || dBitmap.get()) res_->syncDefaultStream();  // the uploads outlive the pass that reads them
  return masked_.as<float>();
}

int64_t DeviceLists::listLength(int64_t l) const {
  VLQ_THROW_IF_NOT(l >= 0 && l < nlists_);
  int64_t o[2];
  VLQ_CALL(vlq_memcpy_d2h(o, offsets_.as<int64_t>() + l, sizeof(o), res_->getDefaultStream()));
  res_->syncDefaultStream();
  return o[1] - o[0];
}

float* DeviceLists::install(const std::vector<int64_t>& offsets, const std::vector<uint8_t>& codes,
                            const std::vector<uint8_t>& lamq, const std::vector<long>& ids) {
  VLQ_THROW_IF_NOT(offsets.size() == (size_t)nlists_ + 1);
  VLQ_THROW_IF_NOT_MSG(auxWidth_ == 0, "lists with an aux column cannot be installed from codes alone");
  const size_t tot = (size_t)offsets.back();
  reset();
  vlq_stream_t st = res_->getDefaultStream();
  offsets_.resize(offsets.size() * sizeof(int64_t));
  slab_ = Columns(std::max<size_t>(1, tot), M_, 0);
  VLQ_CALL(vlq_memcpy_h2d(offsets_.get(), offsets.data(), offsets.size() * sizeof(int64_t), st));
  if (tot) {
    VLQ_CALL(vlq_memcpy_h2d(slab_.codes.get(), codes.data(), codes.size(), st));
    VLQ_CALL(vlq_memcpy_h2d(slab_.lamq.get(), lamq.data(), tot, st));
    VLQ_CALL(vlq_memcpy_h2d(slab_.ids.get(), ids.data(), tot * sizeof(int64_t), st));
  }
  n_ = tot;
  return slab_.kappa.as<float>();
}

void DeviceLists::reset() {
  res_->syncDefaultStream();
  offsets_.release();
  slab_ = Columns();
  pList_.release();
  pending_ = Columns();
  masked_.release();
  n_ = nPending_ = capPending_ = 0;
}

}  // namespace gpu
}  // namespace faiss
