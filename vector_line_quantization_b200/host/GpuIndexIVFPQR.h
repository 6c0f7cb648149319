// GpuIndexIVFPQR: GpuIndexIVFPQ plus a refinement stage (faiss IndexIVFPQR, IndexIVFPQR.{h,cpp}).  Every entry also
// carries code2 = PQ2(x - x1), an 8-bit PQ code of M2 sub-quantizers of the residual its first-level code leaves
// (x1 = the first-level decode, GpuIndexIVFPQ::reconstruct).  It is the aux column of the device lists (DeviceLists.h),
// so it follows its entry through commit and remove_ids.
//
// search(k) scans as GpuIndexIVFPQ::search would for kc = min(1024, max(k, floor(k * k_factor))) results (same coarse
// stage, same scan, selector honoured), then re-ranks those kc candidates on the device by ||q - x2||^2,
// x2 = x1 + p2(code2), and returns the k best in ascending order (ties keep the scan's order; (FLT_MAX, -1) padding).
// Unlike GpuIndexIVFPQ::search, whose distances exclude ||q||^2, these are full squared L2 distances (as
// IndexIVFPQR::search, which re-ranks with fvec_L2sqr).  reconstruct* and search_and_reconstruct return x2.
// range_search, copyFrom / copyTo and the .db* file formats throw: none of them carries or uses code2.
#pragma once
#include <vector>

#include "GpuIndexIVFPQ.h"

namespace faiss {
namespace gpu {

class GpuIndexIVFPQR : public GpuIndexIVFPQ {
 public:
  GpuIndexIVFPQR(GpuResources* resources, int dims, int nlist, int subQuantizers, int refineSubQuantizers,
                 int bitsPerCode, int nedge, int nLambda, faiss::MetricType metric,
                 GpuIndexIVFPQConfig config = GpuIndexIVFPQConfig());

  /// candidates per result of the first-level scan (>= 1; faiss' default 4)
  float k_factor;

  /// the first level as GpuIndexIVFPQ::train, then ProductQuantizer(d, M2, 8) trained on the residuals r2 = x - x1 of
  /// the same training rows (the first min(n, 256 * 128)) with the device k-means.  A refinement codebook that is
  /// already installed is kept.
  void train(Index::idx_t n, const float* x) override;
  /// install a refinement codebook (M2, 256, d / M2); entries already stored keep their codes
  void setRefineCodebook(const float* pq2);
  const std::vector<float>& refineCodebook() const { return pq2Host_; }
  bool hasRefineCodebook() const { return !pq2Host_.empty(); }
  int getNumRefineSubQuantizers() const { return M2_; }
  /// code2 of the entries of list listId, in list order, canonical byte order ([len][M2])
  std::vector<unsigned char> getListRefineCodes(int listId) const;

  void search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const override;
  void search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
              const SearchParameters* params) const override;
  /// search() plus x2 of exactly the entry behind every result: distances are ||q - recons||^2 up to rounding
  void search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                              float* recons) const override;
  void search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                              float* recons, const SearchParameters* params) const override;
  /// not refined (IndexIVFPQR does not refine it either): throws
  void range_search(Index::idx_t n, const float* x, float radius, RangeSearchResult* result) const override;
  void range_search(Index::idx_t n, const float* x, float radius, RangeSearchResult* result,
                    const SearchParameters* params) const override;

 protected:
  void decode_(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t st) const override;
  void encodeAux_(const float* dx, Index::idx_t m, const DeviceLists::Slots& out, Index::idx_t s,
                  vlq_stream_t st) override;

 private:
  Index::idx_t candidates_(Index::idx_t k) const;
  /// vlq_refine_topk of m queries: slab-index candidates [m][kc] -> [m][k] (labels: ids, else slab indexes)
  void rerank_(const float* dq, Index::idx_t m, const int64_t* cand, Index::idx_t kc, Index::idx_t k, bool labels,
               float* outD, int64_t* outI, vlq_stream_t st) const;

  int M2_;
  std::vector<float> pq2Host_;  // (M2, 256, d / M2); empty until trained or installed
  DeviceBuffer dPq2_;
};

}  // namespace gpu
}  // namespace faiss
