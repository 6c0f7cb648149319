#include "GpuIndexIVFPQ.h"

#include "ListRemoval.h"
#include "RangeSearch.h"
#include "Reconstruct.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <fstream>

namespace faiss {
namespace gpu {

// ================================================================================================ GpuIndexIVF
GpuIndexIVF::GpuIndexIVF(GpuResources* resources, int dims, faiss::MetricType metric, int nlist, GpuIndexIVFConfig config)
    : Index(dims, metric), resources_(resources), ivfConfig_(config), nlist_(nlist), nprobe_(1), quantizer_(nullptr) {
  VLQ_THROW_IF_NOT_MSG(resources != nullptr, "GpuResources must not be null");
  VLQ_THROW_IF_NOT_MSG(nlist > 0, "nlist must be > 0");
  VLQ_THROW_IF_NOT_MSG(metric == faiss::METRIC_L2, "only METRIC_L2 is on the VLQ hot path");
  is_trained = false;
  cp_.niter = 10;  // gpu/GpuIndexIVF.cu:50
  GpuIndexFlatConfig fc = config.flatConfig;
  fc.device = config.device;
  quantizer_ = new GpuIndexFlatL2(resources, dims, fc);
}
GpuIndexIVF::~GpuIndexIVF() { delete quantizer_; }

void GpuIndexIVF::setNumProbes(int nprobe) {
  VLQ_THROW_IF_NOT_MSG(nprobe > 0 && nprobe <= 1024, "nprobe must be from 1 to 1024");
  nprobe_ = nprobe;
}

void GpuIndexIVF::add(Index::idx_t n, const float* x) { add_with_ids(n, x, nullptr); }

void GpuIndexIVF::trainQuantizer_(Index::idx_t n, const float* x) {
  if (n == 0) return;
  if (quantizer_->is_trained && quantizer_->ntotal == nlist_) {
    if (verbose) printf("IVF quantizer does not need training.\n");
    return;
  }
  if (verbose) printf("Training IVF quantizer on %ld vectors in %dD\n", n, d);
  quantizer_->reset();
  Clustering clus(d, nlist_, cp_);
  clus.verbose = verbose;
  clus.train(n, x, *quantizer_);  // leaves the final centroids in the quantizer (Clustering.cpp:187-192)
  quantizer_->is_trained = true;
  VLQ_THROW_IF_NOT(quantizer_->ntotal == nlist_);
}

// ================================================================================================ GpuIndexIVFPQ (VLQ)
GpuIndexIVFPQ::GpuIndexIVFPQ(GpuResources* resources, int dims, int nlist, int subQuantizers, int bitsPerCode,
                             int nedge, int nLambda, faiss::MetricType metric, GpuIndexIVFPQConfig config)
    : GpuIndexIVF(resources, dims, metric, nlist, config), nLambda_(nLambda), numedge_(nedge), begin_(0), end_(nlist),
      w1_(256), edgeInfo_(nullptr), edgeDistInfo_(nullptr), lambdaInfo_(nullptr), constInfo_(nullptr), listCap_(VLQ_LIST_CAP),
      ivfpqConfig_(config), subQuantizers_(subQuantizers), bitsPerCode_(bitsPerCode), reserveVecs_(0), nListed_(0), populatedLists_((size_t)nlist * nedge),
      nPending_(0), capPending_(0) {
  VLQ_THROW_IF_NOT_MSG(bitsPerCode == 8, "the scan kernels are written for 8-bit PQ codes");
  VLQ_THROW_IF_NOT_MSG(subQuantizers > 0 && subQuantizers <= 64 && dims % subQuantizers == 0,
                       "number of sub-quantizers must divide the dimension (and be <= 64)");
  VLQ_THROW_IF_NOT_MSG(nedge >= 1 && nedge <= 64 && nedge < nlist, "nedge must be in [1, 64] and < nlist");
  VLQ_THROW_IF_NOT_MSG(nLambda >= 1 && nLambda <= 256, "nLambda must be in [1, 256]");
  VLQ_THROW_IF_NOT_MSG(dims <= 256, "dims must be <= 256");
  VLQ_THROW_IF_NOT_MSG((int64_t)nlist * nedge <= (int64_t)0x7fffffff, "nlist * nedge must fit in 31 bits");
  edgeInfo_ = new int[(size_t)nlist * nedge]();
  edgeDistInfo_ = new float[(size_t)nlist * nedge]();
  lambdaInfo_ = new float[256]();
  constInfo_ = new float[256]();
  pqHost_.resize((size_t)256 * dims);
}

GpuIndexIVFPQ::~GpuIndexIVFPQ() {
  delete[] edgeInfo_;
  delete[] edgeDistInfo_;
  delete[] lambdaInfo_;
  delete[] constInfo_;
  for (int i = 0; i < 2; i++) {
    vlq_event_destroy(evCoarse_[i]);
    vlq_event_destroy(evScan_[i]);
  }
}

void GpuIndexIVFPQ::reserveMemory(size_t numVecs) { reserveVecs_ = numVecs; }

void GpuIndexIVFPQ::reset() {
  DeviceScope scope(ivfConfig_.device);
  resources_->syncDefaultStream();
  lOffsets_.release();
  lCodes_.release();
  lLamq_.release();
  lKappa_.release();
  lIds_.release();
  nListed_ = 0;
  nPending_ = 0;
  ntotal = 0;
  populatedLists_ = (size_t)nlist_ * numedge_;
  begin_ = 0;
  end_ = nlist_;
}

void GpuIndexIVFPQ::uploadTables_() {
  vlq_stream_t st = resources_->getDefaultStream();
  const size_t L = (size_t)nlist_ * numedge_;
  dEdge_.resize(L * sizeof(int));
  dEdgeDist_.resize(L * sizeof(float));
  dLambda_.resize((size_t)nLambda_ * sizeof(float));
  dPq_.resize(pqHost_.size() * sizeof(float));
  VLQ_CALL(vlq_memcpy_h2d(dEdge_.get(), edgeInfo_, dEdge_.bytes(), st));
  VLQ_CALL(vlq_memcpy_h2d(dEdgeDist_.get(), edgeDistInfo_, dEdgeDist_.bytes(), st));
  VLQ_CALL(vlq_memcpy_h2d(dLambda_.get(), lambdaInfo_, dLambda_.bytes(), st));
  VLQ_CALL(vlq_memcpy_h2d(dPq_.get(), pqHost_.data(), dPq_.bytes(), st));
  for (int j = 0; j < nLambda_; j++) constInfo_[j] = lambdaInfo_[j] * lambdaInfo_[j] - lambdaInfo_[j];
  resources_->syncDefaultStream();
}

void GpuIndexIVFPQ::buildGraph_() {  // gpu/GpuIndexIVFPQ.cu:937-953
  quantizer_->buildGraph(nlist_, numedge_, edgeDistInfo_, edgeInfo_);
}

void GpuIndexIVFPQ::setCodebooks(const float* coarse, const int* edge, const float* edgeDist, const float* lambdaCb,
                                 const float* pq) {
  DeviceScope scope(ivfConfig_.device);
  quantizer_->reset();
  quantizer_->add(nlist_, coarse);
  quantizer_->is_trained = true;
  const size_t L = (size_t)nlist_ * numedge_;
  std::memcpy(edgeInfo_, edge, L * sizeof(int));
  std::memcpy(edgeDistInfo_, edgeDist, L * sizeof(float));
  std::memcpy(lambdaInfo_, lambdaCb, (size_t)nLambda_ * sizeof(float));
  std::memcpy(pqHost_.data(), pq, pqHost_.size() * sizeof(float));
  uploadTables_();
  is_trained = true;
}

// GpuIndexIVFPQ::train (gpu/GpuIndexIVFPQ.cu:1160-1178) + trainResidualQuantizer_ (:345-403)
void GpuIndexIVFPQ::train(Index::idx_t n, const float* x) {
  DeviceScope scope(ivfConfig_.device);
  if (is_trained) {
    VLQ_THROW_IF_NOT(quantizer_->is_trained && quantizer_->ntotal == nlist_);
    return;
  }
  VLQ_THROW_IF_NOT_MSG(n >= nlist_, "need at least nlist training vectors");
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer xin;
  const float* dxAll = static_cast<const float*>(toDevice(x, (size_t)n * d * sizeof(float), xin, st));
  resources_->syncDefaultStream();
  trainQuantizer_(n, dxAll);
  buildGraph_();

  // residual quantizer on the first min(n, 2^bits * 128) rows (gpu/GpuIndexIVFPQ.cu:345-352)
  const Index::idx_t n2 = std::min<Index::idx_t>(n, ((Index::idx_t)1 << bitsPerCode_) * 128);
  const size_t L = (size_t)nlist_ * numedge_;
  DeviceBuffer de(L * sizeof(int)), ded(L * sizeof(float));
  VLQ_CALL(vlq_memcpy_h2d(de.get(), edgeInfo_, de.bytes(), st));
  VLQ_CALL(vlq_memcpy_h2d(ded.get(), edgeDistInfo_, ded.bytes(), st));
  DeviceBuffer dA((size_t)n2 * sizeof(int)), dList((size_t)n2 * sizeof(int)), dLam((size_t)n2 * sizeof(float));
  quantizer_->assignDevice(dxAll, n2, dA.as<int>(), nullptr, false);
  VLQ_CALL(vlq_line_encode(dxAll, n2, d, dA.as<int>(), quantizer_->deviceVectors(), de.as<int>(), ded.as<float>(),
                           numedge_, nullptr, 0, nullptr, 0, dList.as<int>(), dLam.as<float>(), nullptr, nullptr,
                           nullptr, nullptr, st));
  {  // 1-D lambda codebook: Clustering(1, nLambda, cp_) over a d = 1 flat index (:365-372)
    GpuIndexFlatConfig fc;
    fc.device = ivfConfig_.device;
    GpuIndexFlatL2 lq(resources_, 1, fc);
    Clustering clus(1, nLambda_, cp_);
    clus.train(n2, dLam.as<float>(), lq);
    std::memcpy(lambdaInfo_, clus.centroids.data(), (size_t)nLambda_ * sizeof(float));
  }
  DeviceBuffer dcb((size_t)nLambda_ * sizeof(float)), dLq((size_t)n2), dRes((size_t)n2 * d * sizeof(float));
  VLQ_CALL(vlq_memcpy_h2d(dcb.get(), lambdaInfo_, dcb.bytes(), st));
  VLQ_CALL(vlq_lambda_quantize(dLam.as<float>(), n2, dcb.as<float>(), nLambda_, dLq.as<uint8_t>(), st));
  VLQ_CALL(vlq_line_residual(dxAll, n2, d, dList.as<int>(), dLq.as<uint8_t>(), dcb.as<float>(),
                             quantizer_->deviceVectors(), de.as<int>(), numedge_, dRes.as<float>(), st));
  resources_->syncDefaultStream();
  faiss::ProductQuantizer pq(d, subQuantizers_, bitsPerCode_);  // CPU class in the reference (:383-385); device k-means here
  pq.verbose = verbose;
  pq.train((int)n2, dRes.as<float>(), resources_);
  pqHost_ = pq.centroids;
  uploadTables_();
  is_trained = true;
}

void GpuIndexIVFPQ::ensurePending_(size_t extra) {
  const size_t need = nPending_ + extra;
  if (need <= capPending_) return;
  vlq_stream_t st = resources_->getDefaultStream();
  size_t cap = std::max(std::max(need, capPending_ * 2), std::max<size_t>(reserveVecs_, 1 << 16));
  const int M = subQuantizers_;
  DeviceBuffer nl(cap * sizeof(int)), nc(cap * M), nq(cap), nk(cap * sizeof(float)), ni(cap * sizeof(int64_t));
  if (nPending_) {
    VLQ_CALL(vlq_memcpy_d2d(nl.get(), pList_.get(), nPending_ * sizeof(int), st));
    VLQ_CALL(vlq_memcpy_d2d(nc.get(), pCodes_.get(), nPending_ * M, st));
    VLQ_CALL(vlq_memcpy_d2d(nq.get(), pLamq_.get(), nPending_, st));
    VLQ_CALL(vlq_memcpy_d2d(nk.get(), pKappa_.get(), nPending_ * sizeof(float), st));
    VLQ_CALL(vlq_memcpy_d2d(ni.get(), pIds_.get(), nPending_ * sizeof(int64_t), st));
    resources_->syncDefaultStream();
  }
  pList_.swap(nl);
  pCodes_.swap(nc);
  pLamq_.swap(nq);
  pKappa_.swap(nk);
  pIds_.swap(ni);
  capPending_ = cap;
}

// classifyAndAddVectors (gpu/GpuIndexIVFPQ.cu:577-908), entirely on the device: coarse NN -> fused line stage / lambda
// quantiser / residual / PQ encode -> append to the pending arena.  Tiles of <= 512 Ki vectors like gpu/GpuIndex.cu:75-106.
void GpuIndexIVFPQ::add_with_ids(Index::idx_t n, const float* x, const long* xids) { addTiles_(n, x, false, xids); }

// uint8 input (SIFT1B .bvecs payload): 4x fewer bytes over PCIe, widened to fp32 on the device (exact)
void GpuIndexIVFPQ::add_with_ids_u8(Index::idx_t n, const uint8_t* x, const long* xids) { addTiles_(n, x, true, xids); }

void GpuIndexIVFPQ::addTiles_(Index::idx_t n, const void* xv, bool isU8, const long* xids) {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  if (n == 0) return;
  VLQ_THROW_IF_NOT(n > 0 && xv);
  DeviceScope scope(ivfConfig_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  ensurePending_((size_t)n);
  const Index::idx_t tile = (Index::idx_t)1 << 19;
  const int M = subQuantizers_;
  const size_t esz = isU8 ? 1 : sizeof(float);
  const uint8_t* xb = static_cast<const uint8_t*>(xv);
  const bool onDevice = vlq_pointer_is_device(xv) == 1;
  vlq_stream_t cs = resources_->getAsyncCopyStream();
  DeviceBuffer& dA = addA_;
  // host input: tile i+1 is staged on the copy stream while tile i is encoded on the compute stream
  auto stage = [&](Index::idx_t s, int slot) -> const void* {
    const Index::idx_t m = std::min(tile, n - s);
    if (onDevice) return xb + (size_t)s * d * esz;
    addIn_[slot].reserve((size_t)tile * d * esz);
    VLQ_CALL(vlq_memcpy_h2d(addIn_[slot].get(), xb + (size_t)s * d * esz, (size_t)m * d * esz, cs));
    return addIn_[slot].get();
  };
  const void* cur = stage(0, 0);
  if (!onDevice) VLQ_CALL(vlq_stream_synchronize(cs));
  int slot = 0;
  for (Index::idx_t s = 0; s < n; s += tile) {
    const Index::idx_t m = std::min(tile, n - s);
    const float* dx;
    if (isU8) {
      addF32_.reserve((size_t)tile * d * sizeof(float));
      VLQ_CALL(vlq_u8_to_f32(static_cast<const uint8_t*>(cur), (int64_t)m * d, addF32_.as<float>(), st));
      dx = addF32_.as<float>();
    } else {
      dx = static_cast<const float*>(cur);
    }
    dA.reserve((size_t)m * sizeof(int));
    quantizer_->assignDevice(dx, m, dA.as<int>(), nullptr, false);
    const size_t o = nPending_;
    VLQ_CALL(vlq_line_encode(dx, m, d, dA.as<int>(), quantizer_->deviceVectors(), dEdge_.as<int>(),
                             dEdgeDist_.as<float>(), numedge_, dLambda_.as<float>(), nLambda_, dPq_.as<float>(), M,
                             pList_.as<int>() + o, nullptr, pLamq_.as<uint8_t>() + o, pCodes_.as<uint8_t>() + o * M,
                             pKappa_.as<float>() + o, nullptr, st));
    if (xids) {
      if (vlq_pointer_is_device(xids) == 1)
        VLQ_CALL(vlq_memcpy_d2d(pIds_.as<int64_t>() + o, xids + s, (size_t)m * sizeof(int64_t), st));
      else
        VLQ_CALL(vlq_memcpy_h2d(pIds_.as<int64_t>() + o, xids + s, (size_t)m * sizeof(int64_t), st));
    } else {
      VLQ_CALL(vlq_iota_i64(pIds_.as<int64_t>() + o, m, (int64_t)(ntotal + s), st));
    }
    nPending_ += (size_t)m;
    if (s + tile < n) cur = stage(s + tile, slot ^ 1);  // overlaps the kernels just launched
    if (!onDevice) VLQ_CALL(vlq_stream_synchronize(cs));
    resources_->syncDefaultStream();  // the staging buffer of this tile is reused two tiles later
    slot ^= 1;
  }
  ntotal += n;
}

void GpuIndexIVFPQ::commit_() const {
  const int64_t L = (int64_t)nlist_ * numedge_;
  if (nPending_ == 0 && lOffsets_.get()) return;
  vlq_stream_t st = resources_->getDefaultStream();
  const int M = subQuantizers_;
  const size_t tot = nListed_ + nPending_;
  DeviceBuffer no((size_t)(L + 1) * sizeof(int64_t)), nc(tot * M), nq(tot), nk(tot * sizeof(float)), ni(tot * sizeof(int64_t));
  const size_t wsb = vlq_build_lists_workspace_bytes((int64_t)nPending_, L);
  scratch_.reserve(wsb);
  VLQ_CALL(vlq_build_lists(L, M, (int64_t)nListed_, lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(), lLamq_.as<uint8_t>(),
                           lKappa_.as<float>(), lIds_.as<int64_t>(), (int64_t)nPending_, pList_.as<int>(),
                           pCodes_.as<uint8_t>(), pLamq_.as<uint8_t>(), pKappa_.as<float>(), pIds_.as<int64_t>(),
                           no.as<int64_t>(), nc.as<uint8_t>(), nq.as<uint8_t>(), nk.as<float>(), ni.as<int64_t>(),
                           scratch_.get(), scratch_.bytes(), st));
  // vectors the encoder skipped (list id < 0) are not stored: the live count is offsets[L]
  int64_t live = 0;
  VLQ_CALL(vlq_memcpy_d2h(&live, no.as<int64_t>() + L, sizeof(int64_t), st));
  resources_->syncDefaultStream();
  lOffsets_.swap(no);
  lCodes_.swap(nc);
  lLamq_.swap(nq);
  lKappa_.swap(nk);
  lIds_.swap(ni);
  nListed_ = (size_t)live;
  nPending_ = 0;
  // the pending arena has done its job: keep at most one add-chunk worth of it (a bulk load followed by searches would
  // otherwise hold 33 B per vector next to the 29 B per vector of the lists)
  const size_t keep = (size_t)1 << 21;
  if (capPending_ > keep) {
    pList_.release();
    pCodes_.release();
    pLamq_.release();
    pKappa_.release();
    pIds_.release();
    capPending_ = 0;
    reserveVecs_ = 0;
  }
}

// IndexIVF::remove_ids: pending adds take part, then the slab is compacted on the device (host/ListRemoval.cpp)
long GpuIndexIVFPQ::remove_ids(const IDSelector& sel) {
  DeviceScope scope(ivfConfig_.device);
  commit_();
  const long removed = removeFromLists(resources_, sel, (int64_t)nlist_ * numedge_, subQuantizers_,
                                       ListSlab{lOffsets_, lCodes_, lLamq_, lKappa_, lIds_, nListed_});
  ntotal -= removed;
  return removed;
}

// ------------------------------------------------------------------------------------------------ read-back
void GpuIndexIVFPQ::decode_(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t st) const {
  VLQ_CALL(vlq_decode_entries(n, pos, (int64_t)nlist_ * numedge_, lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(),
                              lLamq_.as<uint8_t>(), lIds_.as<int64_t>(), subQuantizers_, d, dPq_.as<float>(),
                              quantizer_->deviceVectors(), dEdge_.as<int>(), numedge_, dLambda_.as<float>(), nLambda_,
                              out, outIds, st));
}

void GpuIndexIVFPQ::readBack_(Index::idx_t n, const Index::idx_t* keys, Index::idx_t i0, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(n == 0 || is_trained, "Index not trained");
  if (n == 0) return;
  DeviceScope scope(ivfConfig_.device);
  commit_();
  reconstructIds(resources_, d, SlabIds{lIds_.as<int64_t>(), nListed_}, n, keys, i0, recons,
                 [this](const int64_t* p, int64_t c, float* o, int64_t* oi, vlq_stream_t s) { decode_(p, c, o, oi, s); },
                 recStage_);
}

void GpuIndexIVFPQ::reconstruct(Index::idx_t key, float* recons) const { readBack_(1, &key, 0, recons); }
void GpuIndexIVFPQ::reconstruct_n(Index::idx_t i0, Index::idx_t ni, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(i0 >= 0 && ni >= 0, "reconstruct_n: i0 and ni must be >= 0");
  readBack_(ni, nullptr, i0, recons);
}
void GpuIndexIVFPQ::reconstruct_batch(Index::idx_t n, const Index::idx_t* keys, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(n >= 0 && (n == 0 || keys), "reconstruct_batch: n must be >= 0 and keys non-null");
  readBack_(n, keys, 0, recons);
}

// same lines as search(): the coarse stage of a tile is vlq_coarse_lines (host/RangeSearch.cpp runs the rest)
void GpuIndexIVFPQ::range_search(Index::idx_t n, const float* x, float radius, RangeSearchResult* result) const {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  VLQ_THROW_IF_NOT_MSG(w1_ >= 1 && w1_ <= VLQ_MAX_K, "w1_ must be in [1, 1024]");
  DeviceScope scope(ivfConfig_.device);
  if (n > 0) commit_();
  vlq_stream_t st = resources_->getDefaultStream();
  const int P = std::min(nprobe_, nlist_);
  const int W = w1_;
  const Index::idx_t tile = std::max<Index::idx_t>(64, std::min<Index::idx_t>(5120, ((Index::idx_t)5 << 26) / nlist_));
  DeviceBuffer coarseWs;
  RangeLists lists{dPq_.as<float>(), subQuantizers_, dLambda_.as<float>(), nLambda_, dEdgeDist_.as<float>(), W, listCap_,
                   lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(), lLamq_.as<uint8_t>(), lKappa_.as<float>(),
                   lIds_.as<int64_t>(), nListed_, true, tile};
  rangeSearchLists(resources_, d, n, x, radius, lists,
                   [&](const float* dq, Index::idx_t m, int* lines, float* t1, float* t6) {
                     coarseWs.reserve(vlq_coarse_lines_workspace_bytes(m, d, nlist_, P, numedge_, W,
                                                                       quantizer_->devicePack() != nullptr));
                     VLQ_CALL(vlq_coarse_lines(dq, m, d, quantizer_->deviceVectors(), quantizer_->deviceNorms(),
                                               quantizer_->devicePack(), quantizer_->packScale(), nlist_, P,
                                               dEdge_.as<int>(), dEdgeDist_.as<float>(), numedge_, W, nullptr, lines,
                                               t1, t6, coarseWs.get(), coarseWs.bytes(), st));
                   },
                   result);
}

// searchImpl_ -> IVFPQ::queryGraph (gpu/GpuIndexIVFPQ.cu:1400-1464, gpu/impl/IVFPQ.cu:685-775).  The coarse stage of a
// query tile (a11 + a12: the line, term1, term6 of the W best lines of every query) is one vlq_coarse_lines call, which
// picks the route (fp32 matrix, tcgen05 matrix, matrix-free) and lays out its workspace.
void GpuIndexIVFPQ::search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const {
  DeviceScope scope(ivfConfig_.device);
  searchTiles_(n, x, k, distances, labels, false, nullptr);
}

// search() whose scan reports slab indexes: each tile's labels are decoded (vlq_decode_entries turns them into ids in
// place) before the tile's results leave the device, so D and I are search()'s bits
void GpuIndexIVFPQ::search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances,
                                           Index::idx_t* labels, float* recons) const {
  VLQ_THROW_IF_NOT_MSG(n == 0 || recons != nullptr, "search_and_reconstruct: recons is null");
  DeviceScope scope(ivfConfig_.device);
  const TileEpilogue decode = [&](Index::idx_t row0, Index::idx_t m, float*, int64_t* dI, vlq_stream_t st) {
    decodeToOutput(d, dI, (int64_t)m * k, recons + (size_t)row0 * k * d, dI,
                   [this](const int64_t* p, int64_t c, float* o, int64_t* oi, vlq_stream_t s) { decode_(p, c, o, oi, s); },
                   recStage_, st);
  };
  searchTiles_(n, x, k, distances, labels, true, &decode);
}

void GpuIndexIVFPQ::searchTiles_(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                                 bool slabIndex, const TileEpilogue* epilogue) const {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  VLQ_THROW_IF_NOT_MSG(k >= 1 && k <= VLQ_MAX_K, "k must be in [1, 1024]");
  VLQ_THROW_IF_NOT_MSG(w1_ >= 1 && w1_ <= VLQ_MAX_K, "w1_ must be in [1, 1024]");
  if (n == 0) return;
  commit_();
  const int64_t* ids = slabIndex ? nullptr : lIds_.as<int64_t>();
  vlq_stream_t st = resources_->getDefaultStream();
  const int P = std::min(nprobe_, nlist_);
  const int W = w1_;
  const int M = subQuantizers_;
  const Index::idx_t page = 32768;  // gpu/GpuIndex.cu:109-147
  // query tiles: at most 5120 queries / 1.25 GiB of coarse distances, equal sizes within a page (10 000 queries = 2 x 5000)
  const Index::idx_t tileCap = std::max<Index::idx_t>(64, std::min<Index::idx_t>(5120, ((Index::idx_t)5 << 26) / nlist_));
  DeviceBuffer& xin = qIn_;
  DeviceBuffer& outD = outD_;
  DeviceBuffer& outI = outI_;
  // the coarse workspace is only touched by the coarse stages, which run one after the other on the default stream
  DeviceBuffer& coarseWs = scratch_;
  coarseWs.reserve(vlq_coarse_lines_workspace_bytes(tileCap, d, nlist_, P, numedge_, W, quantizer_->devicePack() != nullptr));
  // two slots of per-tile line buffers (line | term1 | term6): the scan of tile i (scan stream) reads slot i & 1 while the
  // coarse stage of tile i + 1 (default stream) fills the other one
  const size_t lineBytes = ((size_t)tileCap * W * sizeof(float) + 255) & ~size_t(255);
  scratchB_.reserve(2 * 3 * lineBytes);
  t3ws_.reserve(vlq_scan_topk_workspace_bytes(tileCap, M));
  // Host buffers: the queries of tile i+1 go up on the copy stream and the results of tile i-1 come down on the download
  // stream while tile i is computed (cross-stream order by vlq_stream_wait: the compute stream only ever waits for
  // uploads); device buffers are used in place (the scan writes straight into the caller's arrays).
  vlq_stream_t cs = resources_->getAsyncCopyStream();
  vlq_stream_t ds = resources_->getAsyncDownloadStream();
  vlq_stream_t sb = resources_->getScanStream();
  const bool overlap = sb != st && getenv("VLQ_SEARCH_NO_OVERLAP") == nullptr;
  if (!overlap) sb = st;
  if (overlap && !evCoarse_[0]) {
    for (int i = 0; i < 2; i++) {
      VLQ_CALL(vlq_event_create(&evCoarse_[i]));
      VLQ_CALL(vlq_event_create(&evScan_[i]));
    }
  }
  const bool xOnDevice = vlq_pointer_is_device(x) == 1;
  const bool dOnDevice = vlq_pointer_is_device(distances) == 1, lOnDevice = vlq_pointer_is_device(labels) == 1;
  for (Index::idx_t p0 = 0; p0 < n; p0 += page) {
    const Index::idx_t pn = std::min(page, n - p0);
    const Index::idx_t ntiles = (pn + tileCap - 1) / tileCap;
    const Index::idx_t tile = std::min<Index::idx_t>(tileCap, (((pn + ntiles - 1) / ntiles) + 255) / 256 * 256);
    const float* xp = x + (size_t)p0 * d;
    const float* dx = xp;
    if (!xOnDevice) {
      xin.reserve((size_t)pn * d * sizeof(float));
      dx = xin.as<float>();
      VLQ_CALL(vlq_stream_wait(cs, st));  // the staging buffer may still be read by the previous page / call
      VLQ_CALL(vlq_memcpy_h2d(xin.get(), xp, (size_t)std::min(tile, pn) * d * sizeof(float), cs));
    }
    outD.reserve((size_t)pn * k * sizeof(float));
    outI.reserve((size_t)pn * k * sizeof(int64_t));
    if (overlap) VLQ_CALL(vlq_stream_wait(sb, st));  // everything before this page (commit, earlier calls)
    Index::idx_t ti = 0;
    for (Index::idx_t s = 0; s < pn; s += tile, ti++) {
      const Index::idx_t m = std::min(tile, pn - s);
      const float* q = dx + (size_t)s * d;
      const int slot = (int)(ti & 1);
      unsigned char* sbase = scratchB_.as<unsigned char>() + slot * 3 * lineBytes;
      int* lline = reinterpret_cast<int*>(sbase);
      float* t1 = reinterpret_cast<float*>(sbase + lineBytes);
      float* t6 = reinterpret_cast<float*>(sbase + 2 * lineBytes);
      if (!xOnDevice) {
        VLQ_CALL(vlq_stream_wait(st, cs));  // this tile's queries have arrived
        if (s + tile < pn) {
          const Index::idx_t m2 = std::min(tile, pn - s - tile);
          VLQ_CALL(vlq_memcpy_h2d(xin.as<float>() + (size_t)(s + tile) * d, xp + (size_t)(s + tile) * d,
                                  (size_t)m2 * d * sizeof(float), cs));
        }
      }
      if (overlap && ti >= 2) VLQ_CALL(vlq_stream_wait_event(st, evScan_[slot]));  // the slot's last scan has finished
      VLQ_CALL(vlq_coarse_lines(q, m, d, quantizer_->deviceVectors(), quantizer_->deviceNorms(), quantizer_->devicePack(),
                                quantizer_->packScale(), nlist_, P, dEdge_.as<int>(), dEdgeDist_.as<float>(), numedge_, W,
                                nullptr, lline, t1, t6, coarseWs.get(), coarseWs.bytes(), st));
      if (overlap) {
        VLQ_CALL(vlq_event_record(evCoarse_[slot], st));
        VLQ_CALL(vlq_stream_wait_event(sb, evCoarse_[slot]));
      }
      float* hD = distances + (size_t)(p0 + s) * k;
      Index::idx_t* hI = labels + (size_t)(p0 + s) * k;
      const bool inPlace = dOnDevice && lOnDevice;
      float* oD = inPlace ? hD : outD.as<float>() + (size_t)s * k;
      int64_t* oI = inPlace ? reinterpret_cast<int64_t*>(hI) : outI.as<int64_t>() + (size_t)s * k;
      VLQ_CALL(vlq_scan_topk(q, m, d, dPq_.as<float>(), M, dLambda_.as<float>(), nLambda_, lline, t1, t6,
                             dEdgeDist_.as<float>(), W, lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(),
                             lLamq_.as<uint8_t>(), lKappa_.as<float>(), ids, (int)k, listCap_,
                             (int)std::min<size_t>(nListed_ / populatedLists_, 1 << 20), oD, oI, t3ws_.get(),
                             t3ws_.bytes(), sb));
      if (epilogue) (*epilogue)(p0 + s, m, oD, oI, sb);
      if (overlap) VLQ_CALL(vlq_event_record(evScan_[slot], sb));
      if (!inPlace) {
        VLQ_CALL(vlq_stream_wait(ds, sb));  // results of this tile are complete
        fromDevice(hD, oD, (size_t)m * k * sizeof(float), ds);
        fromDevice(hI, oI, (size_t)m * k * sizeof(int64_t), ds);
      }
    }
    VLQ_CALL(vlq_stream_synchronize(cs));
    VLQ_CALL(vlq_stream_synchronize(ds));
    if (overlap) VLQ_CALL(vlq_stream_synchronize(sb));
    resources_->syncDefaultStream();
  }
}

// ---------------------------------------------------------------------------------------------- list accessors
int GpuIndexIVFPQ::getListLength(int listId) const {
  VLQ_THROW_IF_NOT(listId >= 0 && listId < nlist_ * numedge_);
  DeviceScope scope(ivfConfig_.device);
  commit_();
  int64_t o[2];
  VLQ_CALL(vlq_memcpy_d2h(o, lOffsets_.as<int64_t>() + listId, sizeof(o), resources_->getDefaultStream()));
  resources_->syncDefaultStream();
  return (int)(o[1] - o[0]);
}

// Device lists keep the M code bytes of the entry at list position pos rotated by pos mod M (csrc/scan.cuh):
// stored[j] = code[(j + pos) mod M].  The accessors and the .dbcodes files use the canonical order.
static void rotateListCodes(uint8_t* codes, size_t len, int M, bool toStored) {
  std::vector<uint8_t> tmp(M);
  for (size_t pos = 0; pos < len; pos++) {
    uint8_t* c = codes + pos * M;
    const int r = (int)(pos % M);
    for (int j = 0; j < M; j++) tmp[j] = toStored ? c[(j + r) % M] : c[(j - r + M) % M];
    std::memcpy(c, tmp.data(), M);
  }
}

template <typename T>
static std::vector<T> fetchList(const DeviceBuffer& offsets, const DeviceBuffer& data, int listId, size_t per,
                                GpuResources* res) {
  int64_t o[2];
  VLQ_CALL(vlq_memcpy_d2h(o, offsets.as<int64_t>() + listId, sizeof(o), res->getDefaultStream()));
  res->syncDefaultStream();
  std::vector<T> out((size_t)(o[1] - o[0]) * per);
  if (!out.empty()) {
    VLQ_CALL(vlq_memcpy_d2h(out.data(), data.as<T>() + (size_t)o[0] * per, out.size() * sizeof(T), res->getDefaultStream()));
    res->syncDefaultStream();
  }
  return out;
}

std::vector<unsigned char> GpuIndexIVFPQ::getListCodes(int listId) const {
  VLQ_THROW_IF_NOT(listId >= 0 && listId < nlist_ * numedge_);
  DeviceScope scope(ivfConfig_.device);
  commit_();
  std::vector<unsigned char> codes = fetchList<unsigned char>(lOffsets_, lCodes_, listId, subQuantizers_, resources_);
  rotateListCodes(codes.data(), codes.size() / subQuantizers_, subQuantizers_, false);
  return codes;
}
std::vector<unsigned char> GpuIndexIVFPQ::getListLambdas(int listId) const {
  VLQ_THROW_IF_NOT(listId >= 0 && listId < nlist_ * numedge_);
  DeviceScope scope(ivfConfig_.device);
  commit_();
  return fetchList<unsigned char>(lOffsets_, lLamq_, listId, 1, resources_);
}
std::vector<long> GpuIndexIVFPQ::getListIndices(int listId) const {
  VLQ_THROW_IF_NOT(listId >= 0 && listId < nlist_ * numedge_);
  DeviceScope scope(ivfConfig_.device);
  commit_();
  return fetchList<long>(lOffsets_, lIds_, listId, 1, resources_);
}

void GpuIndexIVFPQ::merge(faiss::Index::idx_t* nns, float* dist, int k, int nq, int nprocess, float* distances,
                          faiss::Index::idx_t* labels) const {
  VLQ_THROW_IF_NOT(k >= 1 && k <= VLQ_MAX_K && nq >= 0 && nprocess >= 1);
  if (nq == 0) return;
  DeviceScope scope(ivfConfig_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  const size_t cnt = (size_t)nprocess * nq * k;
  DeviceBuffer din, iin, od((size_t)nq * k * sizeof(float)), oi((size_t)nq * k * sizeof(int64_t));
  const float* dD = static_cast<const float*>(toDevice(dist, cnt * sizeof(float), din, st));
  const int64_t* dI = static_cast<const int64_t*>(toDevice(nns, cnt * sizeof(int64_t), iin, st));
  VLQ_CALL(vlq_merge_topk(dD, dI, nprocess, nq, k, od.as<float>(), oi.as<int64_t>(), st));
  fromDevice(distances, od.get(), od.bytes(), st);
  fromDevice(labels, oi.get(), oi.bytes(), st);
  resources_->syncDefaultStream();
}

// ---------------------------------------------------------------------------------------------- reference file formats
void GpuIndexIVFPQ::writeCodebookToFile(const std::string& name) {  // <name>.ppqt, gpu/GpuIndexIVFPQ.cu:1731-1758
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  DeviceScope scope(ivfConfig_.device);
  std::vector<float> cent((size_t)nlist_ * d);
  VLQ_CALL(vlq_memcpy_d2h(cent.data(), quantizer_->deviceVectors(), cent.size() * sizeof(float), resources_->getDefaultStream()));
  resources_->syncDefaultStream();
  std::ofstream f((name + ".ppqt").c_str(), std::ofstream::out | std::ofstream::binary);
  VLQ_THROW_IF_NOT_MSG(f.good(), "cannot open codebook file for writing");
  const size_t L = (size_t)nlist_ * numedge_;
  f.write((const char*)cent.data(), cent.size() * sizeof(float));
  f.write((const char*)pqHost_.data(), pqHost_.size() * sizeof(float));
  f.write((const char*)edgeInfo_, L * sizeof(int));
  f.write((const char*)edgeDistInfo_, L * sizeof(float));
  f.write((const char*)lambdaInfo_, (size_t)nLambda_ * sizeof(float));
  f.write((const char*)constInfo_, (size_t)nLambda_ * sizeof(float));
}

void GpuIndexIVFPQ::readCodebookFromFile(const std::string& name) {  // gpu/GpuIndexIVFPQ.cu:1774-1810
  std::ifstream f((name + ".ppqt").c_str(), std::ifstream::in | std::ifstream::binary);
  VLQ_THROW_IF_NOT_MSG(f.good(), "cannot open codebook file");
  const size_t L = (size_t)nlist_ * numedge_;
  std::vector<float> cent((size_t)nlist_ * d), pq(pqHost_.size()), ed(L), lam(nLambda_), cst(nLambda_);
  std::vector<int> e(L);
  f.read((char*)cent.data(), cent.size() * sizeof(float));
  f.read((char*)pq.data(), pq.size() * sizeof(float));
  f.read((char*)e.data(), L * sizeof(int));
  f.read((char*)ed.data(), L * sizeof(float));
  f.read((char*)lam.data(), lam.size() * sizeof(float));
  f.read((char*)cst.data(), cst.size() * sizeof(float));
  VLQ_THROW_IF_NOT_MSG(f.good(), "codebook file is truncated");
  setCodebooks(cent.data(), e.data(), ed.data(), lam.data(), pq.data());
}

void GpuIndexIVFPQ::writeDbToFile(const std::string& name) {  // .dbIdx .dbcodes .dbcount .dblas, :1813-1844
  DeviceScope scope(ivfConfig_.device);
  commit_();
  vlq_stream_t st = resources_->getDefaultStream();
  const size_t L = (size_t)nlist_ * numedge_;
  std::vector<int64_t> off(L + 1);
  std::vector<long> ids(nListed_);
  std::vector<uint8_t> codes(nListed_ * subQuantizers_), las(nListed_);
  VLQ_CALL(vlq_memcpy_d2h(off.data(), lOffsets_.get(), off.size() * sizeof(int64_t), st));
  if (nListed_) {
    VLQ_CALL(vlq_memcpy_d2h(ids.data(), lIds_.get(), ids.size() * sizeof(long), st));
    VLQ_CALL(vlq_memcpy_d2h(codes.data(), lCodes_.get(), codes.size(), st));
    VLQ_CALL(vlq_memcpy_d2h(las.data(), lLamq_.get(), las.size(), st));
  }
  resources_->syncDefaultStream();
  std::vector<int> counts(L);
  for (size_t l = 0; l < L; l++) {
    counts[l] = (int)(off[l + 1] - off[l]);
    rotateListCodes(codes.data() + (size_t)off[l] * subQuantizers_, (size_t)counts[l], subQuantizers_, false);
  }
  std::ofstream fi((name + ".dbIdx").c_str(), std::ofstream::binary), fc((name + ".dbcodes").c_str(), std::ofstream::binary),
      fn((name + ".dbcount").c_str(), std::ofstream::binary), fl((name + ".dblas").c_str(), std::ofstream::binary);
  VLQ_THROW_IF_NOT_MSG(fi.good() && fc.good() && fn.good() && fl.good(), "cannot open database files for writing");
  fi.write((const char*)ids.data(), ids.size() * sizeof(long));  // list-major, insertion order inside a list
  fc.write((const char*)codes.data(), codes.size());
  fl.write((const char*)las.data(), las.size());
  fn.write((const char*)counts.data(), counts.size() * sizeof(int));
}

void GpuIndexIVFPQ::installLists_(const std::vector<int>& counts, const std::vector<uint8_t>& codes,
                                  const std::vector<uint8_t>& las, const std::vector<long>& ids) {
  vlq_stream_t st = resources_->getDefaultStream();
  const size_t L = (size_t)nlist_ * numedge_;
  std::vector<int64_t> off(L + 1, 0);
  for (size_t l = 0; l < L; l++) off[l + 1] = off[l] + counts[l];
  const size_t tot = (size_t)off[L];
  VLQ_THROW_IF_NOT(ids.size() == tot && las.size() == tot && codes.size() == tot * subQuantizers_);
  reset();
  lOffsets_.resize((L + 1) * sizeof(int64_t));
  lCodes_.resize(std::max<size_t>(1, codes.size()));
  lLamq_.resize(std::max<size_t>(1, tot));
  lKappa_.resize(std::max<size_t>(1, tot) * sizeof(float));
  lIds_.resize(std::max<size_t>(1, tot) * sizeof(int64_t));
  VLQ_CALL(vlq_memcpy_h2d(lOffsets_.get(), off.data(), off.size() * sizeof(int64_t), st));
  std::vector<uint8_t> stored;  // outlives the copy (freed after the stream sync below)
  if (tot) {
    stored = codes;
    for (size_t l = 0; l < L; l++)
      rotateListCodes(stored.data() + (size_t)off[l] * subQuantizers_, (size_t)counts[l], subQuantizers_, true);
    VLQ_CALL(vlq_memcpy_h2d(lCodes_.get(), stored.data(), stored.size(), st));
    VLQ_CALL(vlq_memcpy_h2d(lLamq_.get(), las.data(), tot, st));
    VLQ_CALL(vlq_memcpy_h2d(lIds_.get(), ids.data(), tot * sizeof(int64_t), st));
    VLQ_CALL(vlq_recompute_kappa((int64_t)tot, (int64_t)L, lOffsets_.as<int64_t>(), lCodes_.as<uint8_t>(),
                                 lLamq_.as<uint8_t>(), quantizer_->deviceVectors(), d, dEdge_.as<int>(), numedge_,
                                 dLambda_.as<float>(), dPq_.as<float>(), subQuantizers_, lKappa_.as<float>(), st));
  }
  resources_->syncDefaultStream();
  nListed_ = tot;
  ntotal = (Index::idx_t)tot;
}

void GpuIndexIVFPQ::readDbFromFile(const std::string& name) { readDbFromFile(name, 1, 0); }

// rank keeps the lists [L/P*rank, L/P*(rank+1)) and zeroes the other counts (gpu/GpuIndexIVFPQ.cu:2106-2163)
void GpuIndexIVFPQ::readDbFromFile(const std::string& name, int pronum, int rank) {
  VLQ_THROW_IF_NOT_MSG(is_trained, "read the codebook first");
  VLQ_THROW_IF_NOT(pronum >= 1 && rank >= 0 && rank < pronum);
  DeviceScope scope(ivfConfig_.device);
  const size_t L = (size_t)nlist_ * numedge_;
  std::vector<int> counts(L);
  std::ifstream fn((name + ".dbcount").c_str(), std::ifstream::binary);
  VLQ_THROW_IF_NOT_MSG(fn.good(), "cannot open .dbcount");
  fn.read((char*)counts.data(), L * sizeof(int));
  VLQ_THROW_IF_NOT_MSG(fn.good(), ".dbcount is truncated");
  const size_t per = L / pronum;
  const size_t l0 = per * rank, l1 = (rank == pronum - 1) ? L : per * (rank + 1);
  size_t skip = 0, keep = 0;
  for (size_t l = 0; l < L; l++) {
    if (l < l0) skip += counts[l];
    else if (l < l1) keep += counts[l];
    if (l < l0 || l >= l1) counts[l] = 0;
  }
  std::vector<long> ids(keep);
  std::vector<uint8_t> codes(keep * subQuantizers_), las(keep);
  std::ifstream fi((name + ".dbIdx").c_str(), std::ifstream::binary), fc((name + ".dbcodes").c_str(), std::ifstream::binary),
      fl((name + ".dblas").c_str(), std::ifstream::binary);
  VLQ_THROW_IF_NOT_MSG(fi.good() && fc.good() && fl.good(), "cannot open database files");
  fi.seekg((std::streamoff)(skip * sizeof(long)));
  fc.seekg((std::streamoff)(skip * subQuantizers_));
  fl.seekg((std::streamoff)skip);
  fi.read((char*)ids.data(), keep * sizeof(long));
  fc.read((char*)codes.data(), codes.size());
  fl.read((char*)las.data(), keep);
  VLQ_THROW_IF_NOT_MSG((keep == 0) || (fi.good() && fc.good() && fl.good()), "database files are truncated");
  installLists_(counts, codes, las, ids);
  // The reference also restricts the COARSE search of rank r to its centroid range [begin_, end_]
  // (gpu/GpuIndexIVFPQ.cu:2132-2137 -> queryGraph(..., begin_, end_)), so its R ranks together visit R x w1_ lines and
  // the merged result differs from the single-index result.  Here every rank selects the global top-w1_ lines and
  // scans those it owns: the merge over the ranks IS the single-index result (DESIGN.md, deviations).  begin_ / end_
  // record the slice; populatedLists_ keeps the kernel choice honest (average length of the lists that hold entries).
  begin_ = (nlist_ / pronum) * rank;
  end_ = rank == pronum - 1 ? nlist_ - 1 : begin_ + nlist_ / pronum - 1;
  populatedLists_ = std::max<size_t>(1, l1 - l0);
}

}  // namespace gpu
}  // namespace faiss

namespace faiss {
namespace gpu {

// ---------------------------------------------------------------------------------------------- f4: CPU index exchange
void GpuIndexIVFPQ::copyFrom(const faiss::IndexIVFPQ* index) {
  VLQ_THROW_IF_NOT_MSG(index != nullptr, "null index");
  VLQ_THROW_IF_NOT_MSG(index->metric_type == faiss::METRIC_L2, "inner product unsupported");
  VLQ_THROW_IF_NOT_MSG(index->d == d && (int)index->nlist == nlist_, "copyFrom: d / nlist differ from this index");
  VLQ_THROW_IF_NOT_MSG((int)index->pq.M == subQuantizers_ && (int)index->pq.nbits == bitsPerCode_,
                       "copyFrom: PQ geometry differs from this index");
  VLQ_THROW_IF_NOT_MSG(index->by_residual && index->polysemous_ht == 0 && index->pq.byte_per_idx == 1,
                       "copyFrom: only residual, non-polysemous, one-byte codes (gpu/GpuIndexIVFPQ.cu:185-188)");
  DeviceScope scope(ivfConfig_.device);
  nprobe_ = (int)std::max<size_t>(1, std::min<size_t>(index->nprobe, 1024));
  reset();
  if (!index->is_trained) {  // gpu/GpuIndexIVFPQ.cu:193-196
    is_trained = false;
    return;
  }
  const faiss::IndexFlatL2* coarse = dynamic_cast<const faiss::IndexFlatL2*>(index->quantizer);
  VLQ_THROW_IF_NOT_MSG(coarse && coarse->ntotal == nlist_ && coarse->xb.size() == (size_t)nlist_ * d,
                       "copyFrom: the quantizer must be an IndexFlatL2 holding the nlist centroids");
  VLQ_THROW_IF_NOT_MSG(index->pq.centroids.size() == pqHost_.size(), "copyFrom: PQ codebook size");
  quantizer_->reset();
  quantizer_->add(nlist_, coarse->xb.data());
  quantizer_->is_trained = true;
  buildGraph_();
  for (int j = 0; j < nLambda_; j++) lambdaInfo_[j] = 0.f;  // every entry sits ON its centroid
  pqHost_ = index->pq.centroids;
  uploadTables_();
  is_trained = true;
  const size_t L = (size_t)nlist_ * numedge_;
  std::vector<int> counts(L, 0);
  size_t tot = 0;
  for (int c = 0; c < nlist_; c++) {
    VLQ_THROW_IF_NOT_MSG(index->ids[c].size() * (size_t)subQuantizers_ == index->codes[c].size(), "copyFrom: list sizes");
    counts[(size_t)c * numedge_] = (int)index->ids[c].size();
    tot += index->ids[c].size();
  }
  std::vector<uint8_t> codes;
  std::vector<long> ids;
  codes.reserve(tot * subQuantizers_);
  ids.reserve(tot);
  for (int c = 0; c < nlist_; c++) {
    codes.insert(codes.end(), index->codes[c].begin(), index->codes[c].end());
    ids.insert(ids.end(), index->ids[c].begin(), index->ids[c].end());
  }
  std::vector<uint8_t> las(tot, 0);
  installLists_(counts, codes, las, ids);
}

void GpuIndexIVFPQ::copyTo(faiss::IndexIVFPQ* index) const {
  VLQ_THROW_IF_NOT_MSG(index != nullptr, "null index");
  for (int j = 0; j < nLambda_; j++)
    VLQ_THROW_IF_NOT_MSG(lambdaInfo_[j] == 0.f,
                         "copyTo: entries of a VLQ index are residuals of line points, not of centroids; only an index "
                         "whose lambda codebook is zero (copyFrom) is a stock IVFPQ");
  DeviceScope scope(ivfConfig_.device);
  index->d = d;
  index->metric_type = faiss::METRIC_L2;
  index->nlist = (size_t)nlist_;
  index->nprobe = (size_t)nprobe_;
  index->by_residual = true;
  index->use_precomputed_table = 0;
  index->code_size = (size_t)subQuantizers_;
  index->polysemous_ht = 0;
  index->pq = faiss::PQCodebook((size_t)d, (size_t)subQuantizers_, (size_t)bitsPerCode_);
  index->pq.centroids = pqHost_;
  faiss::IndexFlatL2* coarse = dynamic_cast<faiss::IndexFlatL2*>(index->quantizer);
  VLQ_THROW_IF_NOT_MSG(coarse != nullptr, "copyTo: the target's quantizer must be an IndexFlatL2");
  coarse->reset();
  coarse->d = d;
  std::vector<float> cent((size_t)nlist_ * d);
  quantizer_->reconstruct_n(0, nlist_, cent.data());
  coarse->add(nlist_, cent.data());
  index->ids.assign((size_t)nlist_, std::vector<long>());
  index->codes.assign((size_t)nlist_, std::vector<uint8_t>());
  index->ntotal = 0;
  index->is_trained = is_trained;
  if (!is_trained) return;
  for (int c = 0; c < nlist_; c++) {
    for (int e = 0; e < numedge_; e++) {
      const int l = c * numedge_ + e;
      if (getListLength(l) == 0) continue;
      const std::vector<long> li = getListIndices(l);
      const std::vector<unsigned char> lc = getListCodes(l);
      index->ids[c].insert(index->ids[c].end(), li.begin(), li.end());
      index->codes[c].insert(index->codes[c].end(), lc.begin(), lc.end());
      index->ntotal += (Index::idx_t)li.size();
    }
  }
}

// ---------------------------------------------------------------------------------------------- f4: candidate lists
void GpuIndexIVFPQ::search1(Index::idx_t n, const float* x, Index::idx_t k, float* /*distances*/, Index::idx_t* labels) const {
  VLQ_THROW_IF_NOT_MSG(is_trained, "Index not trained");
  VLQ_THROW_IF_NOT_MSG(k >= 1, "k must be positive");
  VLQ_THROW_IF_NOT_MSG(w1_ >= 1 && w1_ <= VLQ_MAX_K, "w1_ must be in [1, 1024]");
  if (n == 0) return;
  DeviceScope scope(ivfConfig_.device);
  commit_();
  vlq_stream_t st = resources_->getDefaultStream();
  const int P = std::min(nprobe_, nlist_);
  const int W = w1_;
  const Index::idx_t tile = std::max<Index::idx_t>(64, std::min<Index::idx_t>(1000, ((Index::idx_t)1 << 28) / nlist_));
  DeviceBuffer coarseWs(vlq_coarse_lines_workspace_bytes(tile, d, nlist_, P, numedge_, W, quantizer_->devicePack() != nullptr));
  DeviceBuffer lline((size_t)tile * W * sizeof(int)), t1((size_t)tile * W * sizeof(float)), t6((size_t)tile * W * sizeof(float));
  const bool xOnDevice = vlq_pointer_is_device(x) == 1, lOnDevice = vlq_pointer_is_device(labels) == 1;
  DeviceBuffer xin, out;
  if (!xOnDevice) xin.resize((size_t)tile * d * sizeof(float));
  if (!lOnDevice) out.resize((size_t)tile * k * sizeof(int64_t));
  for (Index::idx_t s = 0; s < n; s += tile) {  // tiles of 1000 queries as in the reference (gpu/GpuIndexIVFPQ.cu:1656)
    const Index::idx_t m = std::min(tile, n - s);
    const float* q = x + (size_t)s * d;
    if (!xOnDevice) {
      VLQ_CALL(vlq_memcpy_h2d(xin.get(), q, (size_t)m * d * sizeof(float), st));
      q = xin.as<float>();
    }
    VLQ_CALL(vlq_coarse_lines(q, m, d, quantizer_->deviceVectors(), quantizer_->deviceNorms(), quantizer_->devicePack(),
                              quantizer_->packScale(), nlist_, P, dEdge_.as<int>(), dEdgeDist_.as<float>(), numedge_, W,
                              nullptr, lline.as<int>(), t1.as<float>(), t6.as<float>(), coarseWs.get(), coarseWs.bytes(), st));
    int64_t* o = lOnDevice ? reinterpret_cast<int64_t*>(labels + (size_t)s * k) : out.as<int64_t>();
    VLQ_CALL(vlq_gather_candidates(lline.as<int>(), m, W, lOffsets_.as<int64_t>(), lIds_.as<int64_t>(), (int64_t)k, o, st));
    if (!lOnDevice) VLQ_CALL(vlq_memcpy_d2h(labels + (size_t)s * k, o, (size_t)m * k * sizeof(int64_t), st));
    resources_->syncDefaultStream();
  }
}

// ---------------------------------------------------------------------------------------------- f4: ground truth
void GpuIndexIVFPQ::add_with_ids2(Index::idx_t n, Index::idx_t nq, unsigned kgt, const float* x, const float* xq,
                                  const Index::idx_t* ids, Index::idx_t* nns, float* dists) {
  VLQ_THROW_IF_NOT_MSG(kgt >= 1 && kgt <= VLQ_MAX_K, "kgt must be in [1, 1024]");
  VLQ_THROW_IF_NOT_MSG(n >= 1 && n <= 0x7fffffff, "the chunk must hold 1 .. INT_MAX rows (gpu/GpuIndexFlat.cu:226-232)");
  if (nq == 0) return;
  DeviceScope scope(ivfConfig_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer dx, dq, xn, qn;
  const float* px = x;
  const float* pq_ = xq;
  if (vlq_pointer_is_device(x) != 1) {
    dx.resize((size_t)n * d * sizeof(float));
    VLQ_CALL(vlq_memcpy_h2d(dx.get(), x, dx.bytes(), st));
    px = dx.as<float>();
  }
  if (vlq_pointer_is_device(xq) != 1) {
    dq.resize((size_t)nq * d * sizeof(float));
    VLQ_CALL(vlq_memcpy_h2d(dq.get(), xq, dq.bytes(), st));
    pq_ = dq.as<float>();
  }
  xn.resize((size_t)n * sizeof(float));
  qn.resize((size_t)nq * sizeof(float));
  VLQ_CALL(vlq_row_norms(px, n, d, xn.as<float>(), st));
  VLQ_CALL(vlq_row_norms(pq_, nq, d, qn.as<float>(), st));
  const Index::idx_t tile = std::max<Index::idx_t>(1, std::min<Index::idx_t>(nq, ((Index::idx_t)1 << 28) / n));
  DeviceBuffer dmat((size_t)tile * n * sizeof(float)), oval((size_t)tile * kgt * sizeof(float)), oidx((size_t)tile * kgt * sizeof(int));
  std::vector<int> hidx((size_t)tile * kgt);
  std::vector<long> hids;
  const long* pid = ids;
  if (ids && vlq_pointer_is_device(ids) == 1) {
    hids.resize((size_t)n);
    VLQ_CALL(vlq_memcpy_d2h(hids.data(), ids, (size_t)n * sizeof(long), st));
    pid = hids.data();
  }
  for (Index::idx_t s = 0; s < nq; s += tile) {
    const Index::idx_t m = std::min(tile, nq - s);
    VLQ_CALL(vlq_l2_distances(pq_ + (size_t)s * d, m, d, px, xn.as<float>(), (int)n, dmat.as<float>(), n, st));
    VLQ_CALL(vlq_select_rows(dmat.as<float>(), m, (int)n, n, (int)kgt, qn.as<float>() + s, oval.as<float>(), oidx.as<int>(), st));
    VLQ_CALL(vlq_memcpy_d2h(dists + (size_t)s * kgt, oval.get(), (size_t)m * kgt * sizeof(float), st));
    VLQ_CALL(vlq_memcpy_d2h(hidx.data(), oidx.get(), (size_t)m * kgt * sizeof(int), st));
    resources_->syncDefaultStream();
    for (size_t i = 0; i < (size_t)m * kgt; i++)  // rank inside the chunk -> label (mergekernel1, gpu/GpuIndexIVFPQ.cu:1285-1308)
      nns[(size_t)s * kgt + i] = hidx[i] < 0 ? -1 : (pid ? pid[hidx[i]] : (long)hidx[i]);
  }
}

}  // namespace gpu
}  // namespace faiss
