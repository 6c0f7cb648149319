// IMI-PQ on the GPU: the baseline index of BASELINE configs[4] (SURVEY.md 8f row f3).  The reference builds it on the CPU as
//   MultiIndexQuantizer coarse(d, 2, nbitsCoarse);  IndexIVFPQ index(&coarse, d, 2^(2 nbitsCoarse), M, 8);
//   index.quantizer_trains_alone = true;                       (tests/sift1b_imi_pq.cpp:216-236)
// i.e. two k-means over the halves of the vectors (K = 2^nbitsCoarse centroids each), K^2 cells, residual PQ codes per
// cell and a search that walks the nprobe cells with the smallest d1 + d2 (multi-sequence, IndexPQ.cpp:637-857).
// Here the same index lives on the device: half assignments / half distance tables by the flat kernels, cell selection by
// vlq_imi_top_cells, encode by vlq_imi_encode, lists = the CSR slab of the VLQ index, scan = vlq_scan_topk with a
// zero lambda codebook (the per-entry kappa replaces the use_precomputed_table = 2 tables, IndexIVFPQ.cpp:645-687).
// search() returns full squared distances ||q - c - p||^2 like IndexIVFPQ::search.
#pragma once
#include <functional>
#include <vector>

#include "AuxIndexStructures.h"
#include "GpuIndexFlat.h"
#include "ProductQuantizer.h"

namespace faiss {
namespace gpu {

class GpuIndexIMIPQ : public faiss::Index {
 public:
  GpuIndexIMIPQ(GpuResources* resources, int dims, int nbitsCoarse, int subQuantizers, int bitsPerCode = 8);
  ~GpuIndexIMIPQ() override;

  void train(Index::idx_t n, const float* x) override;  ///< half k-means x 2, then the PQ on the residuals
  void add(Index::idx_t n, const float* x) override;
  void add_with_ids(Index::idx_t n, const float* x, const long* xids) override;
  void search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const override;
  void reset() override;
  /// IndexIVF::remove_ids for IDSelectorRange / IDSelectorBatch, as GpuIndexIVFPQ::remove_ids (survivors keep their order)
  long remove_ids(const IDSelector& sel) override;
  /// Index::range_search: every entry of the nprobe cells (first listCap_ of each) with ||q - x||^2 < radius, cells in
  /// the order of searchCells, then list position; the same distances as search()
  void range_search(Index::idx_t n, const float* x, float radius, RangeSearchResult* result) const override;
  /// reconstruct / reconstruct_n / reconstruct_batch / search_and_reconstruct as GpuIndexIVFPQ's (keys are ids); the
  /// decode is [cb1[i1] | cb2[i2]] + p(code) in fp32, IndexIVFPQ's decode with a MultiIndexQuantizer
  void reconstruct(Index::idx_t key, float* recons) const override;
  void reconstruct_n(Index::idx_t i0, Index::idx_t ni, float* recons) const override;
  void reconstruct_batch(Index::idx_t n, const Index::idx_t* keys, float* recons) const override;
  void search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                              float* recons) const override;

  void setNumProbes(int nprobe);  ///< cells visited per query, 1 .. 1024
  int getNumProbes() const { return nprobe_; }
  /// install externally trained codebooks: coarse is (2, K, d/2), pq is (M, 256, d/M)
  void setCodebooks(const float* coarse, const float* pq);
  void getCodebooks(float* coarse, float* pq) const;
  /// the nprobe cells of every query, ascending by d1 + d2 (MultiIndexQuantizer::search semantics; int64 labels)
  void searchCells(Index::idx_t n, const float* x, int nprobe, float* distances, Index::idx_t* labels) const;
  int getListLength(long cell) const;
  ClusteringParameters cp_;  ///< niter = 10 like the IVF coarse quantizers (gpu/GpuIndexIVF.cu:50)
  int listCap_;              ///< entries scanned per cell at most (1 << 20: the CPU IndexIVFPQ has no cap)

 private:
  void commit_() const;
  /// the tile loop of search(): slabIndex makes the scan report slab indexes instead of ids; `epilogue` (nullable)
  /// runs after each tile's scan on the device results (as GpuIndexIVFPQ::searchTiles_)
  using TileEpilogue = std::function<void(Index::idx_t row0, Index::idx_t m, float* dD, int64_t* dI, vlq_stream_t st)>;
  void searchTiles_(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                    bool slabIndex, const TileEpilogue* epilogue) const;
  void decode_(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t st) const;
  void readBack_(Index::idx_t n, const Index::idx_t* keys, Index::idx_t i0, float* recons) const;
  void cellsDevice_(const float* dq, Index::idx_t m, int nprobe, int* dCells, float* dDist) const;

  GpuResources* resources_;
  int nbits_, K_, M_, bitsPerCode_, nprobe_;
  GpuIndexFlatL2* half_[2];    // the two coarse codebooks (K rows of d/2)
  std::vector<float> pqHost_;  // (M, 256, dsub)
  DeviceBuffer dPq_, dLambda_;
  mutable DeviceBuffer lOffsets_, lCodes_, lLamq_, lKappa_, lIds_;  // CSR lists over the K^2 cells
  mutable size_t nListed_;
  mutable DeviceBuffer pCell_, pCodes_, pKappa_, pIds_;  // pending entries (arrival order)
  mutable size_t nPending_, capPending_;
  mutable DeviceBuffer scratch_, work_, t3ws_, recStage_;
};

}  // namespace gpu
}  // namespace faiss
