// GpuIndexIVFPQ with the vector-line-quantization extension: the index class of the hot path
// (reference gpu/GpuIndexIVF.{h,cu}, gpu/GpuIndexIVFPQ.{h,cu}; VLQ ctor gpu/GpuIndexIVFPQ.h:59-67, public VLQ members
// :69-81).  Same constructor signature, member names and file formats; the implementation underneath is new:
// inverted lists are one CSR slab on the device (codes + lambda byte + per-entry kappa + ids), adds are encoded and
// appended entirely on the device, and search is four kernels per query tile (coarse GEMM, top-P, line selection,
// fused scan + top-k).
#pragma once
#include <cstdint>
#include <functional>
#include <string>
#include <vector>

#include "AuxIndexStructures.h"
#include "GpuIndexFlat.h"
#include "IndexIVFPQ.h"
#include "ProductQuantizer.h"

namespace faiss {
namespace gpu {

enum IndicesOptions { INDICES_CPU = 0, INDICES_IVF = 1, INDICES_32_BIT = 2, INDICES_64_BIT = 3 };

struct GpuIndexIVFConfig {
  GpuIndexIVFConfig() : device(0), indicesOptions(INDICES_64_BIT) {}
  int device;
  IndicesOptions indicesOptions;  ///< accepted for source compatibility; ids are always 64-bit on the device
  GpuIndexFlatConfig flatConfig;
};

struct GpuIndexIVFPQConfig : public GpuIndexIVFConfig {
  GpuIndexIVFPQConfig() : useFloat16LookupTables(false), usePrecomputedTables(true) {}
  bool useFloat16LookupTables;  ///< ignored: the fp32 table path is the parity target (SURVEY Q6)
  bool usePrecomputedTables;    ///< ignored: the per-entry kappa replaces the term-2 tables (DESIGN.md)
};

class GpuIndexIVF : public faiss::Index {
 public:
  GpuIndexIVF(GpuResources* resources, int dims, faiss::MetricType metric, int nlist, GpuIndexIVFConfig config);
  ~GpuIndexIVF() override;
  int getNumLists() const { return nlist_; }
  int getDevice() const { return resources_->getDevice(); }
  GpuIndexFlat* getQuantizer() { return quantizer_; }
  /// nprobe in [1, 1024] (reference gpu/GpuIndexIVF.cu:201-207)
  void setNumProbes(int nprobe);
  int getNumProbes() const { return nprobe_; }
  void add(Index::idx_t n, const float* x) override;  ///< ids = ntotal + i (gpu/GpuIndexIVF.cu:214-223)

  ClusteringParameters cp_;  ///< niter = 10 for the coarse quantizer (gpu/GpuIndexIVF.cu:50)

 protected:
  void trainQuantizer_(Index::idx_t n, const float* x);
  GpuResources* resources_;
  GpuIndexIVFConfig ivfConfig_;
  int nlist_;
  int nprobe_;
  GpuIndexFlatL2* quantizer_;
};

class GpuIndexIVFPQ : public GpuIndexIVF {
 public:
  /// the VLQ constructor (reference gpu/GpuIndexIVFPQ.h:59-67)
  GpuIndexIVFPQ(GpuResources* resources, int dims, int nlist, int subQuantizers, int bitsPerCode, int nedge,
                int nLambda, faiss::MetricType metric, GpuIndexIVFPQConfig config = GpuIndexIVFPQConfig());
  ~GpuIndexIVFPQ() override;

  // public VLQ state, names as in the reference (gpu/GpuIndexIVFPQ.h:69-81)
  int nLambda_;
  int numedge_;
  int begin_;
  int end_;
  int w1_;             ///< number of lines kept per query (W <= 1024)
  int* edgeInfo_;      ///< [nlist][numedge] neighbour centroid ids (host)
  float* edgeDistInfo_;  ///< [nlist][numedge] squared edge lengths (host)
  float* lambdaInfo_;  ///< [nLambda] lambda codebook (host)
  float* constInfo_;   ///< [nLambda] lambda^2 - lambda (host)

  void train(Index::idx_t n, const float* x) override;
  void add_with_ids(Index::idx_t n, const float* x, const long* xids) override;
  /// uint8-valued vectors (the SIFT1B .bvecs payload the reference drivers widen on the host,
  /// gpu/test/sift1b_createdb.cpp:276-289): copied as bytes, widened to fp32 on the device
  void add_with_ids_u8(Index::idx_t n, const uint8_t* x, const long* xids);
  void search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const override;
  void reset() override;
  /// IndexIVF::remove_ids for IDSelectorRange / IDSelectorBatch (any other selector throws), on the device: pending adds
  /// are committed first, then the lists are compacted.  Survivors keep their order inside a list, so the index equals
  /// one that never received the removed vectors (IndexIVF swaps in the last entry of the list instead).
  long remove_ids(const IDSelector& sel) override;
  /// Index::range_search: every entry that search() scans (the first min(len, listCap_) of each of the w1_ lines) with
  /// full squared distance ||q - x||^2 < radius -- unlike search(), whose distances exclude ||q||^2, a radius needs
  /// the full value.  Per query: lines in slot order, then list position.  Pending adds are committed first.
  void range_search(Index::idx_t n, const float* x, float radius, RangeSearchResult* result) const override;
  /// Index::reconstruct / reconstruct_n / reconstruct_batch, decoded on the device: keys are ids (as in
  /// IndexIVFPQ::reconstruct_n, ids i0 .. i0 + ni - 1), in any order, duplicates allowed.  An id stored more than once
  /// decodes the entry with the lowest slab index; a key without an entry throws before recons is written.  The decode
  /// is anchor + p(code), anchor = (1 - lambda) c + lambda s in fp32 (a copyFrom index: c + p, IndexIVFPQ's own decode).
  /// Pending adds are committed first.  keys / recons may be host or device memory.
  void reconstruct(Index::idx_t key, float* recons) const override;
  void reconstruct_n(Index::idx_t i0, Index::idx_t ni, float* recons) const override;
  void reconstruct_batch(Index::idx_t n, const Index::idx_t* keys, float* recons) const override;
  /// search() plus the decode of exactly the entry behind every result (the scan reports slab indexes, so a repeated id
  /// is no ambiguity): distances and labels are bit-identical to search(); rows of label -1 are NaN.  recons [n][k][d].
  void search_and_reconstruct(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                              float* recons) const override;

  void reserveMemory(size_t numVecs);
  void setPrecomputedCodes(bool) {}
  bool getPrecomputedCodes() const { return true; }
  int getNumSubQuantizers() const { return subQuantizers_; }
  int getBitsPerCode() const { return bitsPerCode_; }
  int getCentroidsPerSubQuantizer() const { return 1 << bitsPerCode_; }
  size_t reclaimMemory() { return 0; }

  int getListLength(int listId) const;
  std::vector<unsigned char> getListCodes(int listId) const;
  std::vector<unsigned char> getListLambdas(int listId) const;
  std::vector<long> getListIndices(int listId) const;

  /// k smallest of the nprocess*k candidates per query; nns / dist are [nprocess][nq][k] (gpu/GpuIndexIVFPQ.cu:1519-1591)
  void merge(faiss::Index::idx_t* nns, float* dist, int k, int nq, int nprocess, float* distances,
             faiss::Index::idx_t* labels) const;

  // reference on-disk formats (gpu/GpuIndexIVFPQ.cu:1731-1844, 2106-2242)
  void writeCodebookToFile(const std::string& name);
  void readCodebookFromFile(const std::string& name);
  void writeDbToFile(const std::string& name);
  void readDbFromFile(const std::string& name);
  void readDbFromFile(const std::string& name, int pronum, int rank);  ///< rank keeps lists [L/P*rank, L/P*(rank+1))
  void buildGraph_();

  /// Populate from / export to a CPU IVFPQ index (reference gpu/GpuIndexIVFPQ.cu:169-281).  A stock IVFPQ entry is a VLQ
  /// entry with lambda = 0: copyFrom takes the coarse centroids and the PQ codebook, rebuilds the centroid graph, zeroes
  /// the lambda codebook and files every entry of coarse list c under line (c, edge 0).  With w1_ = nprobe * numedge_
  /// (every line of the probed centroids) search() then returns exactly IndexIVFPQ::search(nprobe), distances without
  /// the ||q||^2 term.  copyTo needs an index whose lambda codebook is all zero (it throws otherwise: entries on a line
  /// are not residuals of a centroid) and merges the numedge_ lines of every centroid back into one list.
  void copyFrom(const faiss::IndexIVFPQ* index);
  void copyTo(faiss::IndexIVFPQ* index) const;
  /// Candidate lists (reference search1 / searchImpl1_, gpu/GpuIndexIVFPQ.cu:1593-1670): labels[q][0..k) = ids of the
  /// entries of the w1_ selected lines of query q in line order, -1 padded; k is not limited to 1024; `distances` is
  /// not written (as in the reference).
  void search1(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const;
  /// Ground-truth builder (reference add_with_ids2 / generateNNs, gpu/GpuIndexIVFPQ.cu:1312-1398): exact kgt nearest
  /// rows of the chunk x (n rows, labels ids) for every query of xq; nns (nq, kgt) labels, dists squared L2.
  void add_with_ids2(Index::idx_t n, Index::idx_t nq, unsigned kgt, const float* x, const float* xq, const Index::idx_t* ids,
                     Index::idx_t* nns, float* dists);

  /// install externally trained codebooks (tests / multi-GPU broadcast): pq is (M, 256, dsub)
  void setCodebooks(const float* coarse, const int* edge, const float* edgeDist, const float* lambdaCb, const float* pq);
  const std::vector<float>& pqCentroids() const { return pqHost_; }
  /// maximum entries scanned per list (reference: 1024, gpu/impl/IVFUtils.cu:87)
  int listCap_;

 private:
  void uploadTables_();
  void commit_() const;  ///< merge pending entries into the CSR lists (lazy: first search / list access after adds)
  /// the query tile pipeline of search(): slabIndex makes the scan report slab indexes instead of ids; `epilogue`
  /// (nullable) runs on the scan stream after each tile's scan with (first row, rows, device D [m][k], device I [m][k],
  /// stream), before the tile's results are copied out
  using TileEpilogue = std::function<void(Index::idx_t row0, Index::idx_t m, float* dD, int64_t* dI, vlq_stream_t st)>;
  void searchTiles_(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                    bool slabIndex, const TileEpilogue* epilogue) const;
  void decode_(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t st) const;
  void readBack_(Index::idx_t n, const Index::idx_t* keys, Index::idx_t i0, float* recons) const;
  void ensurePending_(size_t extra);
  void addTiles_(Index::idx_t n, const void* x, bool isU8, const long* xids);
  void installLists_(const std::vector<int>& counts, const std::vector<uint8_t>& codes, const std::vector<uint8_t>& las,
                     const std::vector<long>& ids);

  GpuIndexIVFPQConfig ivfpqConfig_;
  int subQuantizers_;
  int bitsPerCode_;
  std::vector<float> pqHost_;  // (M, 256, dsub)
  mutable size_t reserveVecs_;  // bulk-load hint of reserveMemory(): consumed by the first commit

  // device tables
  DeviceBuffer dEdge_, dEdgeDist_, dLambda_, dPq_;
  // CSR lists
  mutable DeviceBuffer lOffsets_, lCodes_, lLamq_, lKappa_, lIds_;
  mutable size_t nListed_;
  size_t populatedLists_;  ///< lists that can hold entries (all of them; the slice of readDbFromFile(name, pronum, rank))
  // pending (encoded, arrival order)
  mutable DeviceBuffer pList_, pCodes_, pLamq_, pKappa_, pIds_;
  mutable size_t nPending_, capPending_;
  mutable vlq_event_t evCoarse_[2] = {nullptr, nullptr}, evScan_[2] = {nullptr, nullptr};  // search(): two-stream tile pipeline
  mutable DeviceBuffer scratch_, scratchB_, qIn_, outD_, outI_, addIn_[2], addA_, addF32_, t3ws_, recStage_;  // grow-only staging / workspace
};

}  // namespace gpu
}  // namespace faiss
