#include "GpuIndexIVFPQR.h"

#include <algorithm>
#include <cmath>

#include "Reconstruct.h"
#include "SearchFilter.h"

namespace faiss {
namespace gpu {

GpuIndexIVFPQR::GpuIndexIVFPQR(GpuResources* resources, int dims, int nlist, int subQuantizers, int refineSubQuantizers,
                               int bitsPerCode, int nedge, int nLambda, faiss::MetricType metric,
                               GpuIndexIVFPQConfig config)
    : GpuIndexIVFPQ(resources, dims, nlist, subQuantizers, bitsPerCode, nedge, nLambda, metric, config,
                    refineSubQuantizers > 0 && refineSubQuantizers <= 64 ? refineSubQuantizers : 0),
      k_factor(4.f), M2_(refineSubQuantizers) {
  VLQ_THROW_IF_NOT_MSG(refineSubQuantizers > 0 && refineSubQuantizers <= 64 && dims % refineSubQuantizers == 0,
                       "number of refinement sub-quantizers must divide the dimension (and be <= 64)");
}

void GpuIndexIVFPQR::setRefineCodebook(const float* pq2) {
  VLQ_THROW_IF_NOT_MSG(pq2 != nullptr, "null refinement codebook");
  DeviceScope scope(ivfConfig_.device);
  pq2Host_.assign(pq2, pq2 + (size_t)256 * d);
  dPq2_.resize(pq2Host_.size() * sizeof(float));
  VLQ_CALL(vlq_memcpy_h2d(dPq2_.get(), pq2Host_.data(), dPq2_.bytes(), resources_->getDefaultStream()));
  resources_->syncDefaultStream();
}

void GpuIndexIVFPQR::train(Index::idx_t n, const float* x) {
  GpuIndexIVFPQ::train(n, x);
  if (hasRefineCodebook()) return;
  DeviceScope scope(ivfConfig_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  // the rows the first-level residual quantizer was trained on (GpuIndexIVFPQ::train)
  const Index::idx_t n2 = std::min<Index::idx_t>(n, ((Index::idx_t)1 << bitsPerCode_) * 128);
  const int M = subQuantizers_;
  DeviceBuffer xin;
  const float* dx = static_cast<const float*>(toDevice(x, (size_t)n2 * d * sizeof(float), xin, st));
  DeviceBuffer dA((size_t)n2 * sizeof(int)), dList((size_t)n2 * sizeof(int)), dLq((size_t)n2),
      dCodes((size_t)n2 * M), dR2((size_t)n2 * d * sizeof(float));
  quantizer_->assignDevice(dx, n2, dA.as<int>(), nullptr, false);
  VLQ_CALL(vlq_line_encode(dx, n2, d, dA.as<int>(), quantizer_->deviceVectors(), dEdge_.as<int>(), dEdgeDist_.as<float>(),
                           numedge_, dLambda_.as<float>(), nLambda_, dPq_.as<float>(), M, dList.as<int>(), nullptr,
                           dLq.as<uint8_t>(), dCodes.as<uint8_t>(), nullptr, nullptr, st));
  VLQ_CALL(vlq_refine_encode(dx, n2, d, dList.as<int>(), dLq.as<uint8_t>(), dCodes.as<uint8_t>(), M, dPq_.as<float>(),
                             quantizer_->deviceVectors(), dEdge_.as<int>(), numedge_, dLambda_.as<float>(), nLambda_,
                             nullptr, 0, nullptr, dR2.as<float>(), st));
  resources_->syncDefaultStream();
  faiss::ProductQuantizer pq2(d, M2_, bitsPerCode_);
  pq2.verbose = verbose;
  pq2.train((int)n2, dR2.as<float>(), resources_);
  setRefineCodebook(pq2.centroids.data());
}

void GpuIndexIVFPQR::encodeAux_(const float* dx, Index::idx_t m, const DeviceLists::Slots& out, Index::idx_t s,
                                vlq_stream_t st) {
  VLQ_THROW_IF_NOT_MSG(hasRefineCodebook(), "GpuIndexIVFPQR: no refinement codebook (train or setRefineCodebook)");
  const int M = subQuantizers_;
  VLQ_CALL(vlq_refine_encode(dx, m, d, out.list + s, out.lamq + s, out.codes + (size_t)s * M, M, dPq_.as<float>(),
                             quantizer_->deviceVectors(), dEdge_.as<int>(), numedge_, dLambda_.as<float>(), nLambda_,
                             dPq2_.as<float>(), M2_, out.aux + (size_t)s * M2_, nullptr, st));
}

std::vector<unsigned char> GpuIndexIVFPQR::getListRefineCodes(int listId) const { return listAux_(listId); }

void GpuIndexIVFPQR::decode_(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t st) const {
  VLQ_THROW_IF_NOT_MSG(hasRefineCodebook(), "GpuIndexIVFPQR: no refinement codebook (train or setRefineCodebook)");
  VLQ_CALL(vlq_refine_decode(n, pos, lists_.nlists(), lists_.offsets(), lists_.codes(), lists_.lamq(), lists_.ids(),
                             lists_.aux(), subQuantizers_, d, dPq_.as<float>(), quantizer_->deviceVectors(),
                             dEdge_.as<int>(), numedge_, dLambda_.as<float>(), nLambda_, dPq2_.as<float>(), M2_, out,
                             outIds, st));
}

Index::idx_t GpuIndexIVFPQR::candidates_(Index::idx_t k) const {
  VLQ_THROW_IF_NOT_MSG(hasRefineCodebook(), "GpuIndexIVFPQR: no refinement codebook (train or setRefineCodebook)");
  VLQ_THROW_IF_NOT_MSG(k >= 1 && k <= VLQ_MAX_K, "k must be in [1, 1024]");
  VLQ_THROW_IF_NOT_MSG(k_factor >= 1.f, "k_factor must be >= 1");
  const double want = std::floor((double)k * (double)k_factor);
  return std::min<Index::idx_t>(VLQ_MAX_K, std::max<Index::idx_t>(k, want >= VLQ_MAX_K ? VLQ_MAX_K : (Index::idx_t)want));
}

void GpuIndexIVFPQR::rerank_(const float* dq, Index::idx_t m, const int64_t* cand, Index::idx_t kc, Index::idx_t k,
                             bool labels, float* outD, int64_t* outI, vlq_stream_t st) const {
  VLQ_CALL(vlq_refine_topk(dq, m, d, cand, (int)kc, (int)k, lists_.nlists(), lists_.offsets(), lists_.codes(),
                           lists_.lamq(), labels ? lists_.ids() : nullptr, lists_.aux(), subQuantizers_,
                           dPq_.as<float>(), quantizer_->deviceVectors(), dEdge_.as<int>(), numedge_,
                           dLambda_.as<float>(), nLambda_, dPq2_.as<float>(), M2_, outD, outI, st));
}

void GpuIndexIVFPQR::search(Index::idx_t n, const float* x, Index::idx_t k, float* distances,
                            Index::idx_t* labels) const {
  search(n, x, k, distances, labels, nullptr);
}

// the scan reports the slab indexes of kc candidates; the re-rank reads their entries and writes ids
void GpuIndexIVFPQR::search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                            const SearchParameters* params) const {
  DeviceScope scope(ivfConfig_.device);
  const Index::idx_t kc = candidates_(k);
  const TileEpilogue rerank = [&](Index::idx_t, Index::idx_t m, const float* dq, float*, int64_t* sI, float* oD,
                                  int64_t* oI, vlq_stream_t st) { rerank_(dq, m, sI, kc, k, true, oD, oI, st); };
  searchTiles_(n, x, k, kc, distances, labels, true, &rerank, searchSelector(params));
}

void GpuIndexIVFPQR::search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances,
                                            Index::idx_t* labels, float* recons) const {
  search_and_reconstruct(n, x, k, distances, labels, recons, nullptr);
}

// the re-rank keeps slab indexes; the decode of x2 turns them into ids in place
void GpuIndexIVFPQR::search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances,
                                            Index::idx_t* labels, float* recons, const SearchParameters* params) const {
  VLQ_THROW_IF_NOT_MSG(n == 0 || recons != nullptr, "search_and_reconstruct: recons is null");
  DeviceScope scope(ivfConfig_.device);
  const Index::idx_t kc = candidates_(k);
  const TileEpilogue rerank = [&](Index::idx_t row0, Index::idx_t m, const float* dq, float*, int64_t* sI, float* oD,
                                  int64_t* oI, vlq_stream_t st) {
    rerank_(dq, m, sI, kc, k, false, oD, oI, st);
    decodeToOutput(d, oI, (int64_t)m * k, recons + (size_t)row0 * k * d, oI,
                   [this](const int64_t* p, int64_t c, float* o, int64_t* oi, vlq_stream_t s) { decode_(p, c, o, oi, s); },
                   recStage_, st);
  };
  searchTiles_(n, x, k, kc, distances, labels, true, &rerank, searchSelector(params));
}

void GpuIndexIVFPQR::range_search(Index::idx_t, const float*, float, RangeSearchResult*) const {
  VLQ_THROW_MSG("GpuIndexIVFPQR: range_search is not refined; use a GpuIndexIVFPQ");
}
void GpuIndexIVFPQR::range_search(Index::idx_t, const float*, float, RangeSearchResult*, const SearchParameters*) const {
  VLQ_THROW_MSG("GpuIndexIVFPQR: range_search is not refined; use a GpuIndexIVFPQ");
}

}  // namespace gpu
}  // namespace faiss
