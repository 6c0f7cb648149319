// GpuIndexFlatL2: brute-force store on the device + the VLQ helper entry points the reference bolted onto it
// (reference gpu/GpuIndexFlat.h:53-175, gpu/GpuIndexFlat.cu).  It is the coarse quantizer of the VLQ index and the
// assigner Clustering::train drives.  All arithmetic is in the C-ABI kernels; this class owns memory and pages data.
#pragma once
#include <cstdint>
#include <vector>

#include "GpuResources.h"
#include "Index.h"

namespace faiss {
namespace gpu {

struct GpuIndexFlatConfig {
  GpuIndexFlatConfig() : device(0), useTensorCores(true) {}
  int device;
  /// route k = 1 / distance-matrix GEMMs through the tcgen05 kernels when the shape allows (d % 32 == 0, d <= 128)
  bool useTensorCores;
};

class GpuIndexFlat : public faiss::Index {
 public:
  GpuIndexFlat(GpuResources* resources, int dims, faiss::MetricType metric, GpuIndexFlatConfig config = GpuIndexFlatConfig());
  ~GpuIndexFlat() override;

  void train(Index::idx_t, const float*) override {}
  void add(Index::idx_t n, const float* x) override;  ///< host or device pointer
  void reset() override;
  /// k <= 1024 (reference limit gpu/GpuIndexFlat.cu:226-232).  L2 distances include ||x||^2 (exact flag).
  using Index::search;  // the SearchParameters overload: no filtering here (a selector throws)
  void search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const override;

  size_t getNumVecs() const { return (size_t)ntotal; }

  // ---- VLQ surface of the reference (gpu/GpuIndexFlat.h:75-143); host or device pointers
  /// stored rows back to host or device memory (reference gpu/GpuIndexFlat.h:196-204)
  void reconstruct(Index::idx_t key, float* out) const override;
  void reconstruct_n(Index::idx_t i0, Index::idx_t num, float* out) const override;
  /// search with int labels (reference searchInt, gpu/GpuIndexFlat.cu:299-372)
  void searchInt(Index::idx_t n, const float* x, Index::idx_t k, float* distances, int* labels) const;
  /// nearest stored vector per row as int labels (reference assignFlat, gpu/GpuIndexFlat.cu:894-900); k must be 1
  void assignFlat(Index::idx_t n, const float* x, int* labels, Index::idx_t k = 1);
  /// kNN graph of the stored vectors: the k = nedge nearest OTHER vectors (rank 0 dropped) (gpu/GpuIndexFlat.cu:375-429)
  void buildGraph(Index::idx_t n, int k, float* distances, int* labels) const;
  /// line stage: assign (nearest centroid) -> assign1 = A*numedge + e and float lambda (gpu/GpuIndexFlat.cu:606-700)
  void assign1(Index::idx_t n, int d, const float* x, int* assign, int* assign1, float* lamdaf, int* edgeinfo,
               float* edgedistinfo, int nlist, int numedge, int k = 1) const;
  /// lambda -> uint8 code against the 1-D codebook (gpu/GpuIndexFlat.cu:702-752)
  /// device-pointer core of assign1 (reference assign1Base, gpu/GpuIndexFlat.cu:756-807; raw pointers instead of Tensors)
  void assign1Base(Index::idx_t n, const float* dInput, const int* dAssign1, int* dAssign2, float* dLambdaf,
                   const int* dEdgeInfo, const float* dEdgeDistInfo, int numedge, int k = 1) const;
  void assignLambda(int n, float* lambdaf, uint8_t* lambda, float* lambdaInfo, int nlambda) const;
  /// r = x - ((1-l) c_A + l c_s) with l = lambdaInfo[lambda]; assign holds A*numedge + e (gpu/GpuIndexFlat.cu:1194-1258)
  void compute_residual(Index::idx_t n, const float* x, float* residual, int* edgeInfo, uint8_t* lambda,
                        float* lambdaInfo, int numedge, int nlist, int* assign) const;

  // ---- device-side accessors used by the VLQ index (no host round trips on the hot path)
  const float* deviceVectors() const { return vecs_.as<float>(); }
  const float* deviceNorms() const { return norms_.as<float>(); }
  const void* devicePack() const { return pack_.get(); }  ///< nullptr when the tensor-core path is not usable
  float packScale() const { return packScale_; }
  GpuResources* resources() const { return resources_; }
  int device() const { return config_.device; }
  /// nearest stored vector for device rows: device in / device out (the entry the encode path uses)
  void assignDevice(const float* dx, Index::idx_t n, int* dLabels, float* dDist, bool addXnorm) const;
  /// distance matrix D = ||c||^2 - 2 x.c for device rows (no ||x||^2, reference gpu/impl/Distance.cu:287-290)
  void distancesDevice(const float* dx, Index::idx_t n, float* dD, Index::idx_t ldD) const;

 private:
  void refreshDerived_();
  void searchCore_(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                   int* intLabels) const;

  GpuResources* resources_;
  GpuIndexFlatConfig config_;
  DeviceBuffer vecs_;   // [ntotal][d]
  DeviceBuffer norms_;  // [ntotal]
  DeviceBuffer pack_;   // tcgen05 operand tiles of the stored vectors
  float packScale_;
  mutable DeviceBuffer scratch_;  // grow-only workspace
  mutable DeviceBuffer scratch2_;
  size_t capacity_;  // rows allocated in vecs_
};

class GpuIndexFlatL2 : public GpuIndexFlat {
 public:
  GpuIndexFlatL2(GpuResources* resources, int dims, GpuIndexFlatConfig config = GpuIndexFlatConfig())
      : GpuIndexFlat(resources, dims, faiss::METRIC_L2, config) {}
};

/// stage a host-or-device array on the device: returns a device pointer (the input itself when already resident)
const void* toDevice(const void* p, size_t bytes, DeviceBuffer& staging, vlq_stream_t stream);
/// copy a device result to a host-or-device destination
void fromDevice(void* dst, const void* dsrc, size_t bytes, vlq_stream_t stream);

}  // namespace gpu
}  // namespace faiss
