#include "GpuIndexIMIPQ.h"

#include "ListRemoval.h"
#include "RangeSearch.h"
#include "Reconstruct.h"

#include <algorithm>
#include <cstring>

namespace faiss {
namespace gpu {

GpuIndexIMIPQ::GpuIndexIMIPQ(GpuResources* resources, int dims, int nbitsCoarse, int subQuantizers, int bitsPerCode)
    : Index(dims, faiss::METRIC_L2), listCap_(1 << 20), resources_(resources), nbits_(nbitsCoarse), K_(1 << nbitsCoarse),
      M_(subQuantizers), bitsPerCode_(bitsPerCode), nprobe_(1), nListed_(0), nPending_(0), capPending_(0) {
  VLQ_THROW_IF_NOT_MSG(dims % 2 == 0 && dims % subQuantizers == 0 && (dims / 2) % (dims / subQuantizers) == 0,
                       "d must be even and every PQ sub-space must lie inside one half");
  VLQ_THROW_IF_NOT_MSG(bitsPerCode == 8, "only 8-bit PQ codes (as the VLQ index)");
  VLQ_THROW_IF_NOT_MSG(nbitsCoarse >= 1 && nbitsCoarse <= 15, "nbitsCoarse must be in [1, 15]");
  is_trained = false;
  cp_.niter = 10;
  GpuIndexFlatConfig cfg;
  cfg.device = resources->getDevice();
  half_[0] = new GpuIndexFlatL2(resources, dims / 2, cfg);
  half_[1] = new GpuIndexFlatL2(resources, dims / 2, cfg);
  pqHost_.assign((size_t)dims * 256, 0.f);
  DeviceScope scope(resources_->getDevice());
  dLambda_.resize(sizeof(float));
  VLQ_CALL(vlq_memset(dLambda_.get(), 0, sizeof(float), resources_->getDefaultStream()));
}

GpuIndexIMIPQ::~GpuIndexIMIPQ() {
  delete half_[0];
  delete half_[1];
}

void GpuIndexIMIPQ::setNumProbes(int nprobe) {
  VLQ_THROW_IF_NOT_MSG(nprobe >= 1 && nprobe <= VLQ_MAX_K, "nprobe must be in [1, 1024]");
  nprobe_ = nprobe;
}

void GpuIndexIMIPQ::reset() {
  DeviceScope scope(resources_->getDevice());
  lOffsets_.release();
  lCodes_.release();
  lLamq_.release();
  lKappa_.release();
  lIds_.release();
  pCell_.release();
  pCodes_.release();
  pKappa_.release();
  pIds_.release();
  nListed_ = nPending_ = capPending_ = 0;
  ntotal = 0;
}

void GpuIndexIMIPQ::setCodebooks(const float* coarse, const float* pq) {
  DeviceScope scope(resources_->getDevice());
  const size_t h = (size_t)d / 2;
  for (int s = 0; s < 2; s++) {
    half_[s]->reset();
    half_[s]->add(K_, coarse + (size_t)s * K_ * h);
  }
  std::memcpy(pqHost_.data(), pq, pqHost_.size() * sizeof(float));
  dPq_.resize(pqHost_.size() * sizeof(float));
  VLQ_CALL(vlq_memcpy_h2d(dPq_.get(), pqHost_.data(), dPq_.bytes(), resources_->getDefaultStream()));
  resources_->syncDefaultStream();
  is_trained = true;
}

void GpuIndexIMIPQ::getCodebooks(float* coarse, float* pq) const {
  const size_t h = (size_t)d / 2;
  for (int s = 0; s < 2; s++) half_[s]->reconstruct_n(0, K_, coarse + (size_t)s * K_ * h);
  std::memcpy(pq, pqHost_.data(), pqHost_.size() * sizeof(float));
}

// MultiIndexQuantizer::train = ProductQuantizer(d, 2, nbits).train (IndexPQ.cpp:788-802): one k-means per half; then the
// PQ of the index on the residuals to the cell centroids (IndexIVFPQ::train_residual_o, IndexIVFPQ.cpp:95-150)
void GpuIndexIMIPQ::train(Index::idx_t n, const float* x) {
  VLQ_THROW_IF_NOT_MSG(n >= K_, "need at least K training vectors");
  DeviceScope scope(resources_->getDevice());
  vlq_stream_t st = resources_->getDefaultStream();
  const int h = d / 2;
  DeviceBuffer stage, halves((size_t)n * h * sizeof(float)), assign((size_t)n * sizeof(int) * 2);
  const float* dx = static_cast<const float*>(toDevice(x, (size_t)n * d * sizeof(float), stage, st));
  std::vector<float> coarse((size_t)2 * K_ * h);
  for (int s = 0; s < 2; s++) {
    VLQ_CALL(vlq_copy_columns(dx, n, d, s * h, h, halves.as<float>(), st));
    Clustering clus(h, K_, cp_);
    half_[s]->reset();
    clus.train(n, halves.as<float>(), *half_[s]);  // leaves the centroids in half_[s]
    std::memcpy(&coarse[(size_t)s * K_ * h], clus.centroids.data(), (size_t)K_ * h * sizeof(float));
    half_[s]->assignDevice(halves.as<float>(), n, assign.as<int>() + (size_t)s * n, nullptr, false);
  }
  // residuals of (at most 256 * 256, ProductQuantizer's own sub-sampling bound) training vectors, on the host side of the
  // boundary like ProductQuantizer::train
  const Index::idx_t nt = std::min<Index::idx_t>(n, 65536);
  std::vector<int> a((size_t)2 * n);
  std::vector<float> hx((size_t)nt * d);
  VLQ_CALL(vlq_memcpy_d2h(a.data(), assign.get(), a.size() * sizeof(int), st));
  VLQ_CALL(vlq_memcpy_d2h(hx.data(), dx, hx.size() * sizeof(float), st));
  resources_->syncDefaultStream();
  for (Index::idx_t i = 0; i < nt; i++)
    for (int s = 0; s < 2; s++) {
      const float* c = &coarse[((size_t)s * K_ + a[(size_t)s * n + i]) * h];
      for (int t = 0; t < h; t++) hx[(size_t)i * d + s * h + t] -= c[t];
    }
  faiss::ProductQuantizer pq((size_t)d, (size_t)M_, (size_t)bitsPerCode_);
  pq.train((int)nt, hx.data(), resources_);
  pqHost_ = pq.centroids;
  dPq_.resize(pqHost_.size() * sizeof(float));
  VLQ_CALL(vlq_memcpy_h2d(dPq_.get(), pqHost_.data(), dPq_.bytes(), st));
  resources_->syncDefaultStream();
  is_trained = true;
}

void GpuIndexIMIPQ::add(Index::idx_t n, const float* x) {
  std::vector<long> ids((size_t)n);
  for (Index::idx_t i = 0; i < n; i++) ids[i] = ntotal + i;
  add_with_ids(n, x, ids.data());
}

void GpuIndexIMIPQ::add_with_ids(Index::idx_t n, const float* x, const long* xids) {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  if (n == 0) return;
  DeviceScope scope(resources_->getDevice());
  vlq_stream_t st = resources_->getDefaultStream();
  const int h = d / 2;
  if (nPending_ + (size_t)n > capPending_) {  // grow the pending arena (contents preserved)
    const size_t cap = std::max(nPending_ + (size_t)n, 2 * capPending_);
    DeviceBuffer c(cap * sizeof(int)), k(cap * (size_t)M_), kp(cap * sizeof(float)), id(cap * sizeof(int64_t));
    if (nPending_) {
      VLQ_CALL(vlq_memcpy_d2d(c.get(), pCell_.get(), nPending_ * sizeof(int), st));
      VLQ_CALL(vlq_memcpy_d2d(k.get(), pCodes_.get(), nPending_ * (size_t)M_, st));
      VLQ_CALL(vlq_memcpy_d2d(kp.get(), pKappa_.get(), nPending_ * sizeof(float), st));
      VLQ_CALL(vlq_memcpy_d2d(id.get(), pIds_.get(), nPending_ * sizeof(int64_t), st));
      resources_->syncDefaultStream();
    }
    pCell_.swap(c);
    pCodes_.swap(k);
    pKappa_.swap(kp);
    pIds_.swap(id);
    capPending_ = cap;
  }
  const Index::idx_t tile = 1 << 20;
  DeviceBuffer stage, halves((size_t)std::min(tile, n) * h * sizeof(float)), assign((size_t)std::min(tile, n) * sizeof(int) * 2);
  for (Index::idx_t s0 = 0; s0 < n; s0 += tile) {
    const Index::idx_t m = std::min(tile, n - s0);
    const float* dx = static_cast<const float*>(toDevice(x + (size_t)s0 * d, (size_t)m * d * sizeof(float), stage, st));
    int* a1 = assign.as<int>();
    int* a2 = a1 + m;
    for (int s = 0; s < 2; s++) {
      VLQ_CALL(vlq_copy_columns(dx, m, d, s * h, h, halves.as<float>(), st));
      half_[s]->assignDevice(halves.as<float>(), m, s ? a2 : a1, nullptr, false);
    }
    VLQ_CALL(vlq_imi_encode(dx, m, d, a1, a2, half_[0]->deviceVectors(), half_[1]->deviceVectors(), nbits_, dPq_.as<float>(),
                            M_, pCell_.as<int>() + nPending_, pCodes_.as<uint8_t>() + nPending_ * (size_t)M_,
                            pKappa_.as<float>() + nPending_, st));
    VLQ_CALL(vlq_memcpy_h2d(pIds_.as<int64_t>() + nPending_, xids + s0, (size_t)m * sizeof(int64_t), st));
    resources_->syncDefaultStream();
    nPending_ += (size_t)m;
  }
  ntotal += n;
}

// pending entries -> CSR lists over the K^2 cells (stable counting sort, vlq_build_lists; lambda bytes are all zero)
void GpuIndexIMIPQ::commit_() const {
  if (nPending_ == 0 && lOffsets_.bytes()) return;
  vlq_stream_t st = resources_->getDefaultStream();
  const int64_t L = (int64_t)K_ * K_;
  const size_t tot = nListed_ + nPending_;
  DeviceBuffer nOff((size_t)(L + 1) * sizeof(int64_t)), nCodes(std::max<size_t>(1, tot * M_)), nLamq(std::max<size_t>(1, tot)),
      nKappa(std::max<size_t>(1, tot) * sizeof(float)), nIds(std::max<size_t>(1, tot) * sizeof(int64_t));
  DeviceBuffer zeros(std::max<size_t>(1, nPending_));
  VLQ_CALL(vlq_memset(zeros.get(), 0, zeros.bytes(), st));
  DeviceBuffer ws(vlq_build_lists_workspace_bytes((int64_t)nPending_, L));
  VLQ_CALL(vlq_build_lists(L, M_, (int64_t)nListed_, nListed_ ? lOffsets_.as<int64_t>() : nullptr, lCodes_.as<uint8_t>(),
                           lLamq_.as<uint8_t>(), lKappa_.as<float>(), lIds_.as<int64_t>(), (int64_t)nPending_,
                           pCell_.as<int>(), pCodes_.as<uint8_t>(), zeros.as<uint8_t>(), pKappa_.as<float>(),
                           pIds_.as<int64_t>(), nOff.as<int64_t>(), nCodes.as<uint8_t>(), nLamq.as<uint8_t>(),
                           nKappa.as<float>(), nIds.as<int64_t>(), ws.get(), ws.bytes(), st));
  int64_t last = 0;
  VLQ_CALL(vlq_memcpy_d2h(&last, nOff.as<int64_t>() + L, sizeof(int64_t), st));
  resources_->syncDefaultStream();
  lOffsets_.swap(nOff);
  lCodes_.swap(nCodes);
  lLamq_.swap(nLamq);
  lKappa_.swap(nKappa);
  lIds_.swap(nIds);
  nListed_ = (size_t)last;  // rows without a cell (NaN input) are dropped, as in the VLQ index
  nPending_ = 0;
}

// same slab as the VLQ index (zero lambda bytes): the same compaction (host/ListRemoval.cpp)
long GpuIndexIMIPQ::remove_ids(const IDSelector& sel) {
  DeviceScope scope(resources_->getDevice());
  commit_();
  const long removed = removeFromLists(resources_, sel, (int64_t)K_ * K_, M_,
                                       ListSlab{lOffsets_, lCodes_, lLamq_, lKappa_, lIds_, nListed_});
  ntotal -= removed;
  return removed;
}

// the cells of cellsDevice_ are the lines; term1 = ||q - c||^2 already makes the distances full ones (row_add NULL)
void GpuIndexIMIPQ::range_search(Index::idx_t n, const float* x, float radius, RangeSearchResult* result) const {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  DeviceScope scope(resources_->getDevice());
  if (n > 0) commit_();
  vlq_stream_t st = resources_->getDefaultStream();
  const int W = nprobe_;
  RangeLists lists{dPq_.as<float>(), M_, dLambda_.as<float>(), 1, nullptr, W, listCap_, lOffsets_.as<int64_t>(),
                   lCodes_.as<uint8_t>(), lLamq_.as<uint8_t>(), lKappa_.as<float>(), lIds_.as<int64_t>(), nListed_, false,
                   4096};
  rangeSearchLists(resources_, d, n, x, radius, lists,
                   [&](const float* dq, Index::idx_t m, int* cells, float* t1, float* t6) {
                     cellsDevice_(dq, m, W, cells, t1);
                     VLQ_CALL(vlq_memset(t6, 0, (size_t)m * W * sizeof(float), st));
                   },
                   result);
}

// ------------------------------------------------------------------------------------------------ read-back
void GpuIndexIMIPQ::decode_(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t st) const {
  VLQ_CALL(vlq_imi_decode_entries(n, pos, lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(), lIds_.as<int64_t>(), M_, d,
                                  dPq_.as<float>(), half_[0]->deviceVectors(), half_[1]->deviceVectors(), nbits_, out,
                                  outIds, st));
}

void GpuIndexIMIPQ::readBack_(Index::idx_t n, const Index::idx_t* keys, Index::idx_t i0, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(n == 0 || is_trained, "Index not trained");
  if (n == 0) return;
  DeviceScope scope(resources_->getDevice());
  commit_();
  reconstructIds(resources_, d, SlabIds{lIds_.as<int64_t>(), nListed_}, n, keys, i0, recons,
                 [this](const int64_t* p, int64_t c, float* o, int64_t* oi, vlq_stream_t s) { decode_(p, c, o, oi, s); },
                 recStage_);
}

void GpuIndexIMIPQ::reconstruct(Index::idx_t key, float* recons) const { readBack_(1, &key, 0, recons); }
void GpuIndexIMIPQ::reconstruct_n(Index::idx_t i0, Index::idx_t ni, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(i0 >= 0 && ni >= 0, "reconstruct_n: i0 and ni must be >= 0");
  readBack_(ni, nullptr, i0, recons);
}
void GpuIndexIMIPQ::reconstruct_batch(Index::idx_t n, const Index::idx_t* keys, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(n >= 0 && (n == 0 || keys), "reconstruct_batch: n must be >= 0 and keys non-null");
  readBack_(n, keys, 0, recons);
}

int GpuIndexIMIPQ::getListLength(long cell) const {
  VLQ_THROW_IF_NOT(cell >= 0 && cell < (long)K_ * K_);
  DeviceScope scope(resources_->getDevice());
  commit_();
  int64_t o[2];
  VLQ_CALL(vlq_memcpy_d2h(o, lOffsets_.as<int64_t>() + cell, sizeof(o), resources_->getDefaultStream()));
  resources_->syncDefaultStream();
  return (int)(o[1] - o[0]);
}

// nprobe best cells of m device queries: half tables -> sorted prefixes -> hyperbola merge
void GpuIndexIMIPQ::cellsDevice_(const float* dq, Index::idx_t m, int nprobe, int* dCells, float* dDist) const {
  vlq_stream_t st = resources_->getDefaultStream();
  const int h = d / 2;
  const int L = std::min(nprobe, K_);
  // work: halves [m][h] | table [m][K] | qnorm [m] | v1, v2 [m][L] | i1, i2 [m][L]
  const size_t need = (size_t)m * ((size_t)h + K_ + 1 + 2 * (size_t)L) * sizeof(float) + (size_t)m * 2 * L * sizeof(int);
  scratch_.reserve(need);
  float* halves = scratch_.as<float>();
  float* table = halves + (size_t)m * h;
  float* qn = table + (size_t)m * K_;
  float* v[2] = {qn + m, qn + m + (size_t)m * L};
  int* idx[2] = {reinterpret_cast<int*>(v[1] + (size_t)m * L), reinterpret_cast<int*>(v[1] + (size_t)m * L) + (size_t)m * L};
  for (int s = 0; s < 2; s++) {
    VLQ_CALL(vlq_copy_columns(dq, m, d, s * h, h, halves, st));
    VLQ_CALL(vlq_row_norms(halves, m, h, qn, st));
    half_[s]->distancesDevice(halves, m, table, K_);  // ||c||^2 - 2 q.c ; + ||q_half||^2 for the winners below
    VLQ_CALL(vlq_select_rows(table, m, K_, K_, L, qn, v[s], idx[s], st));
  }
  VLQ_CALL(vlq_imi_top_cells(v[0], idx[0], v[1], idx[1], m, L, nbits_, nprobe, dCells, dDist, st));
}

void GpuIndexIMIPQ::searchCells(Index::idx_t n, const float* x, int nprobe, float* distances, Index::idx_t* labels) const {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  VLQ_THROW_IF_NOT_MSG(nprobe >= 1 && nprobe <= VLQ_MAX_K, "nprobe must be in [1, 1024]");
  if (n == 0) return;
  DeviceScope scope(resources_->getDevice());
  vlq_stream_t st = resources_->getDefaultStream();
  const Index::idx_t tile = 4096;
  DeviceBuffer stage, cells((size_t)tile * nprobe * sizeof(int)), dist((size_t)tile * nprobe * sizeof(float)),
      lab((size_t)tile * nprobe * sizeof(int64_t));
  for (Index::idx_t s = 0; s < n; s += tile) {
    const Index::idx_t m = std::min(tile, n - s);
    const float* dq = static_cast<const float*>(toDevice(x + (size_t)s * d, (size_t)m * d * sizeof(float), stage, st));
    cellsDevice_(dq, m, nprobe, cells.as<int>(), dist.as<float>());
    VLQ_CALL(vlq_i32_to_i64(cells.as<int>(), (int64_t)m * nprobe, lab.as<int64_t>(), st));
    fromDevice(distances + (size_t)s * nprobe, dist.get(), (size_t)m * nprobe * sizeof(float), st);
    fromDevice(labels + (size_t)s * nprobe, lab.get(), (size_t)m * nprobe * sizeof(int64_t), st);
    resources_->syncDefaultStream();
  }
}

// IndexIVFPQ::search with a MultiIndexQuantizer (IndexIVFPQ.cpp:1050-1100): cells -> scan of their lists -> top-k
void GpuIndexIMIPQ::search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const {
  DeviceScope scope(resources_->getDevice());
  searchTiles_(n, x, k, distances, labels, false, nullptr);
}

// as GpuIndexIVFPQ::search_and_reconstruct: the scan reports slab indexes, the decode turns them into ids in place
void GpuIndexIMIPQ::search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances,
                                           Index::idx_t* labels, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(n == 0 || recons != nullptr, "search_and_reconstruct: recons is null");
  DeviceScope scope(resources_->getDevice());
  const TileEpilogue decode = [&](Index::idx_t row0, Index::idx_t m, float*, int64_t* dI, vlq_stream_t st) {
    decodeToOutput(d, dI, (int64_t)m * k, recons + (size_t)row0 * k * d, dI,
                   [this](const int64_t* p, int64_t c, float* o, int64_t* oi, vlq_stream_t s) { decode_(p, c, o, oi, s); },
                   recStage_, st);
  };
  searchTiles_(n, x, k, distances, labels, true, &decode);
}

void GpuIndexIMIPQ::searchTiles_(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                                 bool slabIndex, const TileEpilogue* epilogue) const {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  VLQ_THROW_IF_NOT_MSG(k >= 1 && k <= VLQ_MAX_K, "k must be in [1, 1024]");
  if (n == 0) return;
  commit_();
  vlq_stream_t st = resources_->getDefaultStream();
  const int W = nprobe_;
  const Index::idx_t tile = 4096;
  DeviceBuffer stage;
  work_.reserve((size_t)tile * W * (sizeof(int) + 2 * sizeof(float)) + (size_t)tile * k * (sizeof(float) + sizeof(int64_t)));
  int* cells = work_.as<int>();
  float* t1 = reinterpret_cast<float*>(cells + (size_t)tile * W);
  float* t6 = t1 + (size_t)tile * W;
  float* oD = t6 + (size_t)tile * W;
  int64_t* oI = reinterpret_cast<int64_t*>(oD + (size_t)tile * k);
  t3ws_.reserve(vlq_scan_topk_workspace_bytes(tile, M_));
  VLQ_CALL(vlq_memset(t6, 0, (size_t)tile * W * sizeof(float), st));
  const int hint = (int)std::min<size_t>(nListed_ / std::max<size_t>(1, (size_t)K_ * K_), 1 << 20);
  for (Index::idx_t s = 0; s < n; s += tile) {
    const Index::idx_t m = std::min(tile, n - s);
    const float* dq = static_cast<const float*>(toDevice(x + (size_t)s * d, (size_t)m * d * sizeof(float), stage, st));
    cellsDevice_(dq, m, W, cells, t1);  // term1 = ||q - c||^2 in full: the results are full squared distances
    VLQ_CALL(vlq_scan_topk(dq, m, d, dPq_.as<float>(), M_, dLambda_.as<float>(), 1, cells, t1, t6, nullptr, W,
                           lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(), lLamq_.as<uint8_t>(), lKappa_.as<float>(),
                           slabIndex ? nullptr : lIds_.as<int64_t>(), (int)k, listCap_, hint, oD, oI, t3ws_.get(),
                           t3ws_.bytes(), st));
    if (epilogue) (*epilogue)(s, m, oD, oI, st);
    fromDevice(distances + (size_t)s * k, oD, (size_t)m * k * sizeof(float), st);
    fromDevice(labels + (size_t)s * k, oI, (size_t)m * k * sizeof(int64_t), st);
    resources_->syncDefaultStream();
  }
}

}  // namespace gpu
}  // namespace faiss
