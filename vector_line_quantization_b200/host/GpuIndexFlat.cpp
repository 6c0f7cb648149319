#include "GpuIndexFlat.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>

namespace faiss {

void Index::assign(idx_t n, const float* x, idx_t* labels, idx_t k) {
  std::vector<float> distances((size_t)n * k);
  search(n, x, k, distances.data(), labels);
}

namespace gpu {

// ------------------------------------------------------------------------------------------------ resources
StandardGpuResources::StandardGpuResources(int device)
    : device_(device), stream_(nullptr), copyStream_(nullptr), downStream_(nullptr), scanStream_(nullptr) {
  DeviceScope scope(device_);
  VLQ_CALL(vlq_stream_create(&stream_));
  VLQ_CALL(vlq_stream_create(&copyStream_));
  VLQ_CALL(vlq_stream_create(&downStream_));
  VLQ_CALL(vlq_stream_create(&scanStream_));
}
StandardGpuResources::~StandardGpuResources() {
  if (stream_) {
    vlq_stream_synchronize(stream_);
    vlq_stream_destroy(stream_);
  }
  if (copyStream_) {
    vlq_stream_synchronize(copyStream_);
    vlq_stream_destroy(copyStream_);
  }
  if (downStream_) {
    vlq_stream_synchronize(downStream_);
    vlq_stream_destroy(downStream_);
  }
  if (scanStream_) {
    vlq_stream_synchronize(scanStream_);
    vlq_stream_destroy(scanStream_);
  }
}
void StandardGpuResources::syncDefaultStream() { VLQ_CALL(vlq_stream_synchronize(stream_)); }

DeviceScope::DeviceScope(int device) : prev_(-1) {
  int cur = 0;
  VLQ_CALL(vlq_get_device(&cur));
  if (cur != device) {
    prev_ = cur;
    VLQ_CALL(vlq_set_device(device));
  }
}
DeviceScope::~DeviceScope() {
  if (prev_ >= 0) vlq_set_device(prev_);
}

const void* toDevice(const void* p, size_t bytes, DeviceBuffer& staging, vlq_stream_t stream) {
  if (bytes == 0 || !p) return p;
  if (vlq_pointer_is_device(p) == 1) return p;
  staging.reserve(bytes);
  VLQ_CALL(vlq_memcpy_h2d(staging.get(), p, bytes, stream));
  return staging.get();
}
void fromDevice(void* dst, const void* dsrc, size_t bytes, vlq_stream_t stream) {
  if (bytes == 0) return;
  if (vlq_pointer_is_device(dst) == 1) VLQ_CALL(vlq_memcpy_d2d(dst, dsrc, bytes, stream));
  else VLQ_CALL(vlq_memcpy_d2h(dst, dsrc, bytes, stream));
}

// ------------------------------------------------------------------------------------------------ flat index
GpuIndexFlat::GpuIndexFlat(GpuResources* resources, int dims, faiss::MetricType metric, GpuIndexFlatConfig config)
    : Index(dims, metric), resources_(resources), config_(config), packScale_(1.f), capacity_(0) {
  VLQ_THROW_IF_NOT_MSG(resources != nullptr, "GpuResources must not be null");
  VLQ_THROW_IF_NOT_MSG(metric == faiss::METRIC_L2, "only METRIC_L2 is on the VLQ hot path");
  VLQ_THROW_IF_NOT_MSG(dims > 0, "invalid dimension");
  is_trained = true;
}
GpuIndexFlat::~GpuIndexFlat() {}

void GpuIndexFlat::reset() {
  DeviceScope scope(config_.device);
  resources_->syncDefaultStream();
  ntotal = 0;
  pack_.release();
}

void GpuIndexFlat::reconstruct(Index::idx_t key, float* out) const { reconstruct_n(key, 1, out); }

void GpuIndexFlat::reconstruct_n(Index::idx_t i0, Index::idx_t num, float* out) const {
  VLQ_THROW_IF_NOT_MSG(i0 >= 0 && num >= 0 && i0 + num <= ntotal, "reconstruct: rows out of range");
  if (num == 0) return;
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  fromDevice(out, vecs_.as<float>() + (size_t)i0 * d, (size_t)num * d * sizeof(float), st);
  resources_->syncDefaultStream();
}

void GpuIndexFlat::add(Index::idx_t n, const float* x) {
  if (n == 0) return;
  VLQ_THROW_IF_NOT_MSG(n > 0 && x, "invalid add arguments");
  VLQ_THROW_IF_NOT_MSG((size_t)(ntotal + n) <= (size_t)0x7fffffff, "GPU flat index holds at most INT_MAX vectors");
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  const size_t need = (size_t)(ntotal + n);
  if (need > capacity_) {
    size_t cap = std::max(need, capacity_ * 2);
    DeviceBuffer grown(cap * d * sizeof(float));
    if (ntotal) VLQ_CALL(vlq_memcpy_d2d(grown.get(), vecs_.get(), (size_t)ntotal * d * sizeof(float), st));
    resources_->syncDefaultStream();
    vecs_.swap(grown);
    capacity_ = cap;
  }
  float* dst = vecs_.as<float>() + (size_t)ntotal * d;
  const size_t bytes = (size_t)n * d * sizeof(float);
  if (vlq_pointer_is_device(x) == 1) VLQ_CALL(vlq_memcpy_d2d(dst, x, bytes, st));
  else VLQ_CALL(vlq_memcpy_h2d(dst, x, bytes, st));
  ntotal += n;
  refreshDerived_();
  resources_->syncDefaultStream();  // the caller may free x right after add() returns
}

void GpuIndexFlat::refreshDerived_() {
  vlq_stream_t st = resources_->getDefaultStream();
  resources_->syncDefaultStream();
  norms_.resize((size_t)ntotal * sizeof(float));
  VLQ_CALL(vlq_row_norms(vecs_.as<float>(), ntotal, d, norms_.as<float>(), st));
  pack_.release();
  if (config_.useTensorCores && vlq_tc_supported(d, (int)ntotal)) {
    // exact power-of-two pre-scale: max|c| * scale ~ 2^9 keeps hi and lo parts in fp16's normal range
    std::vector<float> host((size_t)ntotal * d);
    VLQ_CALL(vlq_memcpy_d2h(host.data(), vecs_.get(), host.size() * sizeof(float), st));
    resources_->syncDefaultStream();
    float mx = 0.f;
    for (float v : host) mx = std::max(mx, std::fabs(v));
    packScale_ = (mx > 0.f && std::isfinite(mx)) ? std::ldexp(1.f, 9 - (int)std::ceil(std::log2(mx))) : 1.f;
    pack_.resize(vlq_tc_cent_pack_bytes((int)ntotal, d));
    VLQ_CALL(vlq_tc_pack_centroids(vecs_.as<float>(), norms_.as<float>(), (int)ntotal, d, packScale_, pack_.get(), st));
  }
}

void GpuIndexFlat::assignDevice(const float* dx, Index::idx_t n, int* dLabels, float* dDist, bool addXnorm) const {
  vlq_stream_t st = resources_->getDefaultStream();
  if (pack_.get()) {
    const size_t ws = vlq_l2_tc_workspace_bytes(n, d, (int)ntotal);
    scratch_.reserve(ws);
    VLQ_CALL(vlq_l2_assign_tc(dx, n, d, pack_.get(), packScale_, (int)ntotal, addXnorm ? 1 : 0, dLabels, dDist,
                              scratch_.get(), scratch_.bytes(), st));
  } else {
    VLQ_CALL(vlq_l2_assign(dx, n, d, vecs_.as<float>(), norms_.as<float>(), (int)ntotal, addXnorm ? 1 : 0, dLabels,
                           dDist, st));
  }
}

void GpuIndexFlat::distancesDevice(const float* dx, Index::idx_t n, float* dD, Index::idx_t ldD) const {
  vlq_stream_t st = resources_->getDefaultStream();
  if (pack_.get()) {
    const size_t ws = vlq_l2_tc_workspace_bytes(n, d, (int)ntotal);
    scratch_.reserve(ws);
    VLQ_CALL(vlq_l2_distances_tc(dx, n, d, pack_.get(), packScale_, (int)ntotal, dD, ldD, nullptr, scratch_.get(),
                                 scratch_.bytes(), st));
  } else {
    VLQ_CALL(vlq_l2_distances(dx, n, d, vecs_.as<float>(), norms_.as<float>(), (int)ntotal, dD, ldD, st));
  }
}

void GpuIndexFlat::search(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels) const {
  searchCore_(n, x, k, distances, labels, nullptr);
}

// same search, int labels (reference searchInt, gpu/GpuIndexFlat.cu:299-372)
void GpuIndexFlat::searchInt(Index::idx_t n, const float* x, Index::idx_t k, float* distances, int* labels) const {
  searchCore_(n, x, k, distances, nullptr, labels);
}

void GpuIndexFlat::searchCore_(Index::idx_t n, const float* x, Index::idx_t k, float* distances, Index::idx_t* labels,
                               int* intLabels) const {
  VLQ_THROW_IF_NOT_MSG(k >= 1 && k <= VLQ_MAX_K, "k must be in [1, 1024]");
  VLQ_THROW_IF_NOT_MSG(ntotal > 0, "index is empty");
  if (n == 0) return;
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  // page the queries like the reference (gpu/GpuIndex.cu:109-147); tile so that the distance matrix stays small
  const Index::idx_t tile = k == 1 ? (Index::idx_t)1 << 18
                                   : std::max<Index::idx_t>(1, std::min<Index::idx_t>(4096, ((Index::idx_t)64 << 20) / ntotal));
  DeviceBuffer xin, dmat, outv, outi, outl, xn;
  for (Index::idx_t s = 0; s < n; s += tile) {
    const Index::idx_t m = std::min(tile, n - s);
    const float* dx = static_cast<const float*>(toDevice(x + (size_t)s * d, (size_t)m * d * sizeof(float), xin, st));
    outv.reserve((size_t)m * k * sizeof(float));
    outi.reserve((size_t)m * k * sizeof(int));
    outl.reserve((size_t)m * k * sizeof(int64_t));
    if (k == 1) {
      assignDevice(dx, m, outi.as<int>(), outv.as<float>(), true);
    } else {
      dmat.reserve((size_t)m * ntotal * sizeof(float));
      xn.reserve((size_t)m * sizeof(float));
      distancesDevice(dx, m, dmat.as<float>(), ntotal);
      VLQ_CALL(vlq_row_norms(dx, m, d, xn.as<float>(), st));
      VLQ_CALL(vlq_select_rows(dmat.as<float>(), m, (int)ntotal, ntotal, (int)k, xn.as<float>(), outv.as<float>(),
                               outi.as<int>(), st));
    }
    fromDevice(distances + (size_t)s * k, outv.get(), (size_t)m * k * sizeof(float), st);
    if (labels) {
      VLQ_CALL(vlq_i32_to_i64(outi.as<int>(), (int64_t)m * k, outl.as<int64_t>(), st));
      fromDevice(labels + (size_t)s * k, outl.get(), (size_t)m * k * sizeof(int64_t), st);
    }
    if (intLabels) fromDevice(intLabels + (size_t)s * k, outi.get(), (size_t)m * k * sizeof(int), st);
    resources_->syncDefaultStream();
  }
}

void GpuIndexFlat::assignFlat(Index::idx_t n, const float* x, int* labels, Index::idx_t k) {
  VLQ_THROW_IF_NOT_MSG(k == 1, "assignFlat supports k == 1");
  if (n == 0) return;
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer xin, outi;
  const float* dx = static_cast<const float*>(toDevice(x, (size_t)n * d * sizeof(float), xin, st));
  outi.reserve((size_t)n * sizeof(int));
  assignDevice(dx, n, outi.as<int>(), nullptr, false);
  fromDevice(labels, outi.get(), (size_t)n * sizeof(int), st);
  resources_->syncDefaultStream();
}

void GpuIndexFlat::buildGraph(Index::idx_t n, int k, float* distances, int* labels) const {
  VLQ_THROW_IF_NOT_MSG(n == ntotal, "buildGraph works on the stored vectors");
  VLQ_THROW_IF_NOT_MSG(k >= 1 && k + 1 <= VLQ_MAX_K && k + 1 <= ntotal, "invalid number of edges");
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer de((size_t)n * k * sizeof(int)), dd((size_t)n * k * sizeof(float));
  const size_t ws = vlq_knn_graph_workspace_bytes((int)n, k);
  scratch2_.reserve(ws);
  VLQ_CALL(vlq_knn_graph(vecs_.as<float>(), norms_.as<float>(), (int)n, d, k, de.as<int>(), dd.as<float>(),
                         scratch2_.get(), scratch2_.bytes(), st));
  fromDevice(labels, de.get(), de.bytes(), st);
  fromDevice(distances, dd.get(), dd.bytes(), st);
  resources_->syncDefaultStream();
}

void GpuIndexFlat::assign1(Index::idx_t n, int dd, const float* x, int* assign, int* assign1, float* lamdaf,
                           int* edgeinfo, float* edgedistinfo, int nlist, int numedge, int /*k*/) const {
  VLQ_THROW_IF_NOT(dd == d && nlist == ntotal);
  if (n == 0) return;
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer xin, ain, ein, edin, ol((size_t)n * sizeof(int)), of((size_t)n * sizeof(float));
  const float* dx = static_cast<const float*>(toDevice(x, (size_t)n * d * sizeof(float), xin, st));
  const int* da = static_cast<const int*>(toDevice(assign, (size_t)n * sizeof(int), ain, st));
  const int* de = static_cast<const int*>(toDevice(edgeinfo, (size_t)nlist * numedge * sizeof(int), ein, st));
  const float* ded = static_cast<const float*>(toDevice(edgedistinfo, (size_t)nlist * numedge * sizeof(float), edin, st));
  VLQ_CALL(vlq_line_encode(dx, n, d, da, vecs_.as<float>(), de, ded, numedge, nullptr, 0, nullptr, 0, ol.as<int>(),
                           of.as<float>(), nullptr, nullptr, nullptr, nullptr, st));
  fromDevice(assign1, ol.get(), ol.bytes(), st);
  fromDevice(lamdaf, of.get(), of.bytes(), st);
  resources_->syncDefaultStream();
}

// the device-resident core of assign1 (reference assign1Base takes device Tensors, gpu/GpuIndexFlat.cu:756-807): every
// pointer is a device pointer, nothing is copied or synchronised
void GpuIndexFlat::assign1Base(Index::idx_t n, const float* dInput, const int* dAssign1, int* dAssign2, float* dLambdaf,
                               const int* dEdgeInfo, const float* dEdgeDistInfo, int numedge, int /*k*/) const {
  if (n == 0) return;
  VLQ_THROW_IF_NOT_MSG(vlq_pointer_is_device(dInput) == 1 && vlq_pointer_is_device(dAssign2) == 1,
                       "assign1Base works on device memory (use assign1 for host pointers)");
  DeviceScope scope(config_.device);
  VLQ_CALL(vlq_line_encode(dInput, n, d, dAssign1, vecs_.as<float>(), dEdgeInfo, dEdgeDistInfo, numedge, nullptr, 0,
                           nullptr, 0, dAssign2, dLambdaf, nullptr, nullptr, nullptr, nullptr,
                           resources_->getDefaultStream()));
}

void GpuIndexFlat::assignLambda(int n, float* lambdaf, uint8_t* lambda, float* lambdaInfo, int nlambda) const {
  if (n == 0) return;
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer lin, cin, out((size_t)n);
  const float* dl = static_cast<const float*>(toDevice(lambdaf, (size_t)n * sizeof(float), lin, st));
  const float* dc = static_cast<const float*>(toDevice(lambdaInfo, (size_t)nlambda * sizeof(float), cin, st));
  VLQ_CALL(vlq_lambda_quantize(dl, n, dc, nlambda, out.as<uint8_t>(), st));
  fromDevice(lambda, out.get(), (size_t)n, st);
  resources_->syncDefaultStream();
}

void GpuIndexFlat::compute_residual(Index::idx_t n, const float* x, float* residual, int* edgeInfo, uint8_t* lambda,
                                    float* lambdaInfo, int numedge, int nlist, int* assign) const {
  VLQ_THROW_IF_NOT(nlist == ntotal);
  if (n == 0) return;
  DeviceScope scope(config_.device);
  vlq_stream_t st = resources_->getDefaultStream();
  DeviceBuffer xin, ein, lin, cin, ain, out((size_t)n * d * sizeof(float));
  const float* dx = static_cast<const float*>(toDevice(x, (size_t)n * d * sizeof(float), xin, st));
  const int* de = static_cast<const int*>(toDevice(edgeInfo, (size_t)nlist * numedge * sizeof(int), ein, st));
  const uint8_t* dl = static_cast<const uint8_t*>(toDevice(lambda, (size_t)n, lin, st));
  // the reference signature carries no table length: size the copy by the largest code actually used
  std::vector<uint8_t> hcodes((size_t)n);
  if (vlq_pointer_is_device(lambda) == 1) {
    VLQ_CALL(vlq_memcpy_d2h(hcodes.data(), lambda, (size_t)n, st));
    resources_->syncDefaultStream();
  } else {
    std::memcpy(hcodes.data(), lambda, (size_t)n);
  }
  const int nl = 1 + (int)*std::max_element(hcodes.begin(), hcodes.end());
  const float* dc = static_cast<const float*>(toDevice(lambdaInfo, (size_t)nl * sizeof(float), cin, st));
  const int* da = static_cast<const int*>(toDevice(assign, (size_t)n * sizeof(int), ain, st));
  VLQ_CALL(vlq_line_residual(dx, n, d, da, dl, dc, vecs_.as<float>(), de, numedge, out.as<float>(), st));
  fromDevice(residual, out.get(), out.bytes(), st);
  resources_->syncDefaultStream();
}

}  // namespace gpu
}  // namespace faiss
