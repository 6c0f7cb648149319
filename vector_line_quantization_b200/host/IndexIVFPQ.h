// CPU-side containers with the member names of the reference's faiss::IndexFlatL2 / faiss::IndexIVFPQ
// (IndexFlat.h:21-60, IndexIVFPQ.h:30-130, IndexIVF.h:30-120): what GpuIndexIVFPQ::copyFrom / copyTo exchange
// (gpu/GpuIndexIVFPQ.cu:169-281).  They hold data only -- centroids, the PQ codebook, per-list codes and ids; searching on
// the CPU is not part of this layer (there is no CPU fallback: the reference's own CPU classes live in oracle/_ref as
// the baseline).
#pragma once
#include <cstdint>
#include <vector>

#include "Index.h"

namespace faiss {

struct IndexFlatL2 : Index {
  std::vector<float> xb;  ///< database vectors, ntotal * d
  explicit IndexFlatL2(idx_t d_ = 0) : Index(d_, METRIC_L2) {}
  void add(idx_t n, const float* x) override {
    xb.insert(xb.end(), x, x + (size_t)n * d);
    ntotal += n;
  }
  using Index::search;
  void search(idx_t, const float*, idx_t, float*, idx_t*) const override {
    VLQ_THROW_MSG("IndexFlatL2 is a container here: search with GpuIndexFlatL2");
  }
  void reset() override {
    xb.clear();
    ntotal = 0;
  }
};

struct PQCodebook {  ///< the fields of faiss::ProductQuantizer that copyFrom / copyTo touch
  size_t d, M, nbits, dsub, ksub, byte_per_idx, code_size;
  std::vector<float> centroids;  ///< (M, ksub, dsub)
  PQCodebook(size_t d_ = 0, size_t M_ = 1, size_t nbits_ = 8)
      : d(d_), M(M_), nbits(nbits_), dsub(M_ ? d_ / M_ : 0), ksub((size_t)1 << nbits_), byte_per_idx((nbits_ + 7) / 8),
        code_size(byte_per_idx * M_), centroids(d_ * ((size_t)1 << nbits_)) {}
};

struct IndexIVFPQ : Index {
  Index* quantizer;  ///< IndexFlatL2 with the nlist coarse centroids
  size_t nlist, nprobe;
  bool own_fields;
  bool by_residual;
  int use_precomputed_table;
  size_t code_size;
  PQCodebook pq;
  int polysemous_ht;
  std::vector<std::vector<long>> ids;       ///< [nlist] labels
  std::vector<std::vector<uint8_t>> codes;  ///< [nlist] PQ codes, code_size bytes per entry

  IndexIVFPQ(Index* quantizer_, size_t d_, size_t nlist_, size_t M, size_t nbits)
      : Index((idx_t)d_, METRIC_L2), quantizer(quantizer_), nlist(nlist_), nprobe(1), own_fields(false), by_residual(true),
        use_precomputed_table(0), code_size(M), pq(d_, M, nbits), polysemous_ht(0), ids(nlist_), codes(nlist_) {
    is_trained = false;
  }
  ~IndexIVFPQ() override {
    if (own_fields) delete quantizer;
  }
  void add(idx_t, const float*) override { VLQ_THROW_MSG("IndexIVFPQ is a container here: add through GpuIndexIVFPQ"); }
  using Index::search;
  void search(idx_t, const float*, idx_t, float*, idx_t*) const override {
    VLQ_THROW_MSG("IndexIVFPQ is a container here: search through GpuIndexIVFPQ");
  }
  void reset() override {
    for (auto& v : ids) v.clear();
    for (auto& v : codes) v.clear();
    ntotal = 0;
  }
};

}  // namespace faiss
