#include "vlq_index_c.h"

#include <cstring>
#include <string>
#include <vector>

#include "AuxIndexStructures.h"
#include "Clustering.h"
#include "GpuIndexIMIPQ.h"
#include "GpuIndexIVFPQ.h"
#include "IndexProxy.h"
#include "filehelper.h"

using namespace faiss;
using namespace faiss::gpu;

static thread_local std::string g_err;

#define GUARD(...)                     \
  try {                                \
    __VA_ARGS__;                       \
    return 0;                          \
  } catch (const std::exception& e) {  \
    g_err = e.what();                  \
    return -1;                         \
  } catch (...) {                      \
    g_err = "unknown C++ exception";   \
    return -1;                         \
  }

static Index* I(void* h) { return static_cast<Index*>(h); }
static GpuIndexIVFPQ* V(void* h) {
  GpuIndexIVFPQ* p = dynamic_cast<GpuIndexIVFPQ*>(static_cast<Index*>(h));
  if (!p) throw FaissException("handle is not a VLQ index");
  return p;
}
static GpuIndexFlat* F(void* h) {
  GpuIndexFlat* p = dynamic_cast<GpuIndexFlat*>(static_cast<Index*>(h));
  if (!p) throw FaissException("handle is not a flat index");
  return p;
}

extern "C" {

const char* vlq_host_last_error(void) { return g_err.c_str(); }

int vlq_host_resources_new(int device, void** out) { GUARD(*out = new StandardGpuResources(device)) }
int vlq_host_resources_free(void* res) { GUARD(delete static_cast<StandardGpuResources*>(res)) }
int vlq_host_resources_sync(void* res) { GUARD(static_cast<GpuResources*>(res)->syncDefaultStream()) }

int vlq_host_index_free(void* index) { GUARD(delete I(index)) }
int vlq_host_index_train(void* index, long n, const float* x) { GUARD(I(index)->train(n, x)) }
int vlq_host_index_add(void* index, long n, const float* x) { GUARD(I(index)->add(n, x)) }
int vlq_host_index_add_with_ids(void* index, long n, const float* x, const long* ids) {
  GUARD(I(index)->add_with_ids(n, x, ids))
}
int vlq_host_index_search(void* index, long n, const float* x, long k, float* distances, long* labels) {
  GUARD(I(index)->search(n, x, k, distances, labels))
}
int vlq_host_index_reset(void* index) { GUARD(I(index)->reset()) }
int vlq_host_index_remove_ids_range(void* index, long imin, long imax, long* nremoved) {
  GUARD(*nremoved = I(index)->remove_ids(IDSelectorRange(imin, imax)))
}
int vlq_host_index_remove_ids_batch(void* index, long n, const long* ids, long* nremoved) {
  GUARD({
    VLQ_THROW_IF_NOT_MSG(n >= 0 && (n == 0 || ids), "remove_ids: n must be >= 0 and ids non-null when n > 0");
    std::vector<long> staged;
    if (n > 0 && vlq_pointer_is_device(ids) == 1) {  // IDSelectorBatch sorts on the host
      staged.resize((size_t)n);
      VLQ_CALL(vlq_memcpy_d2h(staged.data(), ids, (size_t)n * sizeof(long), nullptr));
      VLQ_CALL(vlq_stream_synchronize(nullptr));
      ids = staged.data();
    }
    *nremoved = I(index)->remove_ids(IDSelectorBatch(n, ids));
  })
}
int vlq_host_index_range_search(void* index, long n, const float* x, float radius, void** result) {
  GUARD({
    VLQ_THROW_IF_NOT_MSG(result != nullptr && n >= 0, "range_search: n must be >= 0 and result non-null");
    *result = nullptr;
    RangeSearchResult* r = new RangeSearchResult(n);
    try {
      I(index)->range_search(n, x, radius, r);
    } catch (...) {
      delete r;
      throw;
    }
    *result = r;
  })
}
static RangeSearchResult* R(void* h) {
  if (!h) throw FaissException("null range search result");
  return static_cast<RangeSearchResult*>(h);
}
int vlq_host_range_result_total(void* result, long* total) { GUARD(*total = (long)R(result)->lims[R(result)->nq]) }
int vlq_host_range_result_copy(void* result, long* lims, float* distances, long* labels) {
  GUARD({
    const RangeSearchResult* r = R(result);
    const size_t total = r->lims[r->nq];
    if (lims)
      for (size_t i = 0; i <= r->nq; i++) lims[i] = (long)r->lims[i];
    if (distances && total) std::memcpy(distances, r->distances, total * sizeof(float));
    if (labels && total) std::memcpy(labels, r->labels, total * sizeof(long));
  })
}
int vlq_host_range_result_free(void* result) { GUARD(delete static_cast<RangeSearchResult*>(result)) }
long vlq_host_index_ntotal(void* index) { return I(index)->ntotal; }
int vlq_host_index_is_trained(void* index) { return I(index)->is_trained ? 1 : 0; }

int vlq_host_flat_new(void* res, int d, int use_tensor_cores, void** out) {
  GUARD({
    GpuIndexFlatConfig cfg;
    cfg.device = static_cast<GpuResources*>(res)->getDevice();
    cfg.useTensorCores = use_tensor_cores != 0;
    *out = static_cast<Index*>(new GpuIndexFlatL2(static_cast<GpuResources*>(res), d, cfg));
  })
}
int vlq_host_flat_assign(void* flat, long n, const float* x, int* labels) { GUARD(F(flat)->assignFlat(n, x, labels, 1)) }
int vlq_host_index_reconstruct_n(void* index, long i0, long ni, float* recons) { GUARD(I(index)->reconstruct_n(i0, ni, recons)) }
int vlq_host_index_reconstruct_batch(void* index, long n, const long* keys, float* recons) {
  GUARD(I(index)->reconstruct_batch(n, keys, recons))
}
int vlq_host_index_search_and_reconstruct(void* index, long n, const float* x, long k, float* distances, long* labels,
                                          float* recons) {
  GUARD(I(index)->search_and_reconstruct(n, x, k, distances, labels, recons))
}
int vlq_host_flat_search_int(void* flat, long n, const float* x, long k, float* distances, int* labels) {
  GUARD(F(flat)->searchInt(n, x, k, distances, labels))
}
int vlq_host_flat_assign1_base(void* flat, long n, const float* d_input, const int* d_assign1, int* d_assign2,
                               float* d_lambdaf, const int* d_edge, const float* d_edge_dist, int numedge) {
  GUARD(F(flat)->assign1Base(n, d_input, d_assign1, d_assign2, d_lambdaf, d_edge, d_edge_dist, numedge))
}
int vlq_host_flat_build_graph(void* flat, int nedge, float* distances, int* labels) {
  GUARD(F(flat)->buildGraph(F(flat)->ntotal, nedge, distances, labels))
}

int vlq_host_kmeans(void* res, int d, int k, long n, const float* x, int niter, int seed, float* centroids_out) {
  GUARD({
    GpuResources* r = static_cast<GpuResources*>(res);
    ClusteringParameters cp;
    cp.niter = niter;
    cp.seed = seed;
    Clustering clus(d, k, cp);
    GpuIndexFlatConfig cfg;
    cfg.device = r->getDevice();
    GpuIndexFlatL2 assigner(r, d, cfg);
    clus.train(n, x, assigner);
    std::memcpy(centroids_out, clus.centroids.data(), sizeof(float) * (size_t)d * k);
  })
}

int vlq_host_vlq_new(void* res, int d, int nlist, int M, int bits, int nedge, int nlambda, int use_tensor_cores,
                     void** out) {
  GUARD({
    GpuResources* r = static_cast<GpuResources*>(res);
    GpuIndexIVFPQConfig cfg;
    cfg.device = r->getDevice();
    cfg.flatConfig.useTensorCores = use_tensor_cores != 0;
    *out = static_cast<Index*>(new GpuIndexIVFPQ(r, d, nlist, M, bits, nedge, nlambda, METRIC_L2, cfg));
  })
}
int vlq_host_vlq_set_nprobe(void* index, int nprobe) { GUARD(V(index)->setNumProbes(nprobe)) }
int vlq_host_vlq_set_w1(void* index, int w1) {
  GUARD({
    VLQ_THROW_IF_NOT_MSG(w1 >= 1 && w1 <= VLQ_MAX_K, "w1 must be in [1, 1024]");
    V(index)->w1_ = w1;
  })
}
int vlq_host_vlq_set_list_cap(void* index, int cap) {
  GUARD({
    VLQ_THROW_IF_NOT_MSG(cap >= 1, "cap must be >= 1");
    V(index)->listCap_ = cap;
  })
}
int vlq_host_vlq_add_with_ids_u8(void* index, long n, const unsigned char* x, const long* ids) {
  GUARD(V(index)->add_with_ids_u8(n, x, ids))
}
int vlq_host_vlq_reserve_memory(void* index, long num_vecs) { GUARD(V(index)->reserveMemory((size_t)num_vecs)) }
int vlq_host_vlq_set_train_iters(void* index, int niter) { GUARD(V(index)->cp_.niter = niter) }
int vlq_host_vlq_get_codebooks(void* index, float* coarse, int* edge, float* edge_dist, float* lambda_cb, float* pq) {
  GUARD({
    GpuIndexIVFPQ* v = V(index);
    VLQ_THROW_IF_NOT_MSG(v->is_trained, "Index not trained");
    const size_t L = (size_t)v->getNumLists() * v->numedge_;
    GpuIndexFlat* q = v->getQuantizer();
    VLQ_CALL(vlq_memcpy_d2h(coarse, q->deviceVectors(), (size_t)v->getNumLists() * v->d * sizeof(float),
                            q->resources()->getDefaultStream()));
    q->resources()->syncDefaultStream();
    std::memcpy(edge, v->edgeInfo_, L * sizeof(int));
    std::memcpy(edge_dist, v->edgeDistInfo_, L * sizeof(float));
    std::memcpy(lambda_cb, v->lambdaInfo_, (size_t)v->nLambda_ * sizeof(float));
    std::memcpy(pq, v->pqCentroids().data(), v->pqCentroids().size() * sizeof(float));
  })
}
int vlq_host_vlq_set_codebooks(void* index, const float* coarse, const int* edge, const float* edge_dist,
                               const float* lambda_cb, const float* pq) {
  GUARD(V(index)->setCodebooks(coarse, edge, edge_dist, lambda_cb, pq))
}
int vlq_host_vlq_list_length(void* index, int list, int* out) { GUARD(*out = V(index)->getListLength(list)) }
int vlq_host_vlq_get_list(void* index, int list, unsigned char* codes, unsigned char* lambdas, long* ids) {
  GUARD({
    auto c = V(index)->getListCodes(list);
    auto l = V(index)->getListLambdas(list);
    auto i = V(index)->getListIndices(list);
    if (codes && !c.empty()) std::memcpy(codes, c.data(), c.size());
    if (lambdas && !l.empty()) std::memcpy(lambdas, l.data(), l.size());
    if (ids && !i.empty()) std::memcpy(ids, i.data(), i.size() * sizeof(long));
  })
}
int vlq_host_vlq_merge(void* index, long* nns, float* dist, int k, int nq, int nprocess, float* distances, long* labels) {
  GUARD(V(index)->merge(nns, dist, k, nq, nprocess, distances, labels))
}
int vlq_host_vlq_write_codebook(void* index, const char* name) { GUARD(V(index)->writeCodebookToFile(name)) }
int vlq_host_vlq_read_codebook(void* index, const char* name) { GUARD(V(index)->readCodebookFromFile(name)) }
int vlq_host_vlq_write_db(void* index, const char* name) { GUARD(V(index)->writeDbToFile(name)) }
int vlq_host_vlq_read_db(void* index, const char* name, int pronum, int rank) {
  GUARD(V(index)->readDbFromFile(name, pronum, rank))
}

/* host-side pieces of k-means that never touch the GPU (reference utils.cpp:135-160,307-317) */
int vlq_host_rand_perm(int* perm, long n, long seed) { GUARD(rand_perm(perm, (size_t)n, seed)) }

/* dataset formats (reference filehelper.cpp) */
int vlq_host_vecs_header(const char* path, int elem_size, long* n, long* d) {
  GUARD({
    size_t nn = 0, dd = 0;
    vecs_header(path, (size_t)elem_size, &nn, &dd);
    *n = (long)nn;
    *d = (long)dd;
  })
}
int vlq_host_vecs_read(const char* path, int kind, long start, long num, void* out) {
  GUARD({
    size_t n = 0, d = 0;
    if (kind == 0) {
      auto v = fvecs_read(path, &n, &d, (size_t)start, (size_t)num);
      std::memcpy(out, v.data(), v.size() * sizeof(float));
    } else if (kind == 1) {
      auto v = ivecs_read(path, &n, &d, (size_t)start, (size_t)num);
      std::memcpy(out, v.data(), v.size() * sizeof(int32_t));
    } else {
      auto v = bvecs_read(path, &n, &d, (size_t)start, (size_t)num);
      std::memcpy(out, v.data(), v.size());
    }
  })
}
int vlq_host_vecs_write(const char* path, int kind, const void* x, long n, long d) {
  GUARD({
    if (kind == 0) fvecs_write(path, static_cast<const float*>(x), (size_t)n, (size_t)d);
    else if (kind == 1) ivecs_write(path, static_cast<const int32_t*>(x), (size_t)n, (size_t)d);
    else bvecs_write(path, static_cast<const uint8_t*>(x), (size_t)n, (size_t)d);
  })
}
int vlq_host_umem_header(const char* path, long* num, long* dim) {
  GUARD({
    size_t a = 0, b = 0;
    umem_header(path, &a, &b);
    *num = (long)a;
    *dim = (long)b;
  })
}
int vlq_host_umem_write(const char* path, long num, long dim, const void* ptr, int elem_size, long len, long offset) {
  GUARD(umem_write(path, (size_t)num, (size_t)dim, ptr, (size_t)elem_size, (size_t)len, (size_t)offset))
}
int vlq_host_umem_read(const char* path, void* ptr, int elem_size, long len, long offset) {
  GUARD(umem_read(path, ptr, (size_t)elem_size, (size_t)len, (size_t)offset))
}

int vlq_host_proxy_new(void** out) { GUARD(*out = static_cast<Index*>(new IndexProxy())) }
int vlq_host_proxy_add_index(void* proxy, void* index) {
  GUARD({
    IndexProxy* p = dynamic_cast<IndexProxy*>(I(proxy));
    VLQ_THROW_IF_NOT_MSG(p, "handle is not an IndexProxy");
    p->addIndex(I(index));
  })
}
int vlq_host_shards_new(int d, int threaded, int successive_ids, void** out) {
  GUARD(*out = static_cast<Index*>(new IndexShards(d, threaded != 0, successive_ids != 0)))
}
int vlq_host_shards_add_shard(void* shards, void* index) {
  GUARD({
    IndexShards* s = dynamic_cast<IndexShards*>(I(shards));
    VLQ_THROW_IF_NOT_MSG(s, "handle is not an IndexShards");
    s->add_shard(I(index));
  })
}

// ---- f4: CPU IVFPQ container + copyFrom / copyTo, candidate lists, ground-truth builder
static IndexIVFPQ* CPU(void* h) { return static_cast<IndexIVFPQ*>(h); }
int vlq_host_cpu_ivfpq_new(int d, long nlist, int M, int nbits, void** out) {
  GUARD({
    IndexFlatL2* q = new IndexFlatL2(d);
    IndexIVFPQ* ix = new IndexIVFPQ(q, (size_t)d, (size_t)nlist, (size_t)M, (size_t)nbits);
    ix->own_fields = true;
    *out = ix;
  })
}
int vlq_host_cpu_ivfpq_free(void* h) { GUARD(delete CPU(h)) }
int vlq_host_cpu_ivfpq_set_codebooks(void* h, const float* coarse, const float* pq) {
  GUARD({
    IndexIVFPQ* ix = CPU(h);
    ix->quantizer->reset();
    ix->quantizer->add((long)ix->nlist, coarse);
    std::memcpy(ix->pq.centroids.data(), pq, ix->pq.centroids.size() * sizeof(float));
    ix->is_trained = true;
  })
}
int vlq_host_cpu_ivfpq_get_codebooks(void* h, float* coarse, float* pq) {
  GUARD({
    IndexIVFPQ* ix = CPU(h);
    const IndexFlatL2* q = dynamic_cast<const IndexFlatL2*>(ix->quantizer);
    std::memcpy(coarse, q->xb.data(), q->xb.size() * sizeof(float));
    std::memcpy(pq, ix->pq.centroids.data(), ix->pq.centroids.size() * sizeof(float));
  })
}
int vlq_host_cpu_ivfpq_set_list(void* h, long list, long n, const long* ids, const unsigned char* codes) {
  GUARD({
    IndexIVFPQ* ix = CPU(h);
    if (list < 0 || list >= (long)ix->nlist) throw FaissException("list out of range");
    ix->ntotal += n - (long)ix->ids[list].size();
    ix->ids[list].assign(ids, ids + n);
    ix->codes[list].assign(codes, codes + (size_t)n * ix->code_size);
  })
}
long vlq_host_cpu_ivfpq_list_size(void* h, long list) { return (long)CPU(h)->ids[list].size(); }
long vlq_host_cpu_ivfpq_ntotal(void* h) { return CPU(h)->ntotal; }
int vlq_host_cpu_ivfpq_get_list(void* h, long list, long* ids, unsigned char* codes) {
  GUARD({
    IndexIVFPQ* ix = CPU(h);
    std::memcpy(ids, ix->ids[list].data(), ix->ids[list].size() * sizeof(long));
    std::memcpy(codes, ix->codes[list].data(), ix->codes[list].size());
  })
}
int vlq_host_ivfpq_copy_from(void* index, void* cpu_index) { GUARD(V(index)->copyFrom(CPU(cpu_index))) }
int vlq_host_ivfpq_copy_to(void* index, void* cpu_index) { GUARD(V(index)->copyTo(CPU(cpu_index))) }
int vlq_host_ivfpq_search1(void* index, long n, const float* x, long k, long* labels) {
  GUARD(V(index)->search1(n, x, k, nullptr, labels))
}
int vlq_host_ivfpq_add_with_ids2(void* index, long n, long nq, unsigned kgt, const float* x, const float* xq, const long* ids,
                                 long* nns, float* dists) {
  GUARD(V(index)->add_with_ids2(n, nq, kgt, x, xq, ids, nns, dists))
}

// ---- f3: IMI-PQ on the GPU (the baseline index of BASELINE configs[4])
static GpuIndexIMIPQ* IMI(void* h) {
  GpuIndexIMIPQ* p = dynamic_cast<GpuIndexIMIPQ*>(static_cast<Index*>(h));
  if (!p) throw FaissException("handle is not an IMI-PQ index");
  return p;
}
int vlq_host_imipq_new(void* res, int d, int nbits_coarse, int M, int nbits, void** out) {
  GUARD(*out = static_cast<Index*>(new GpuIndexIMIPQ(static_cast<GpuResources*>(res), d, nbits_coarse, M, nbits)))
}
int vlq_host_imipq_set_nprobe(void* index, int nprobe) { GUARD(IMI(index)->setNumProbes(nprobe)) }
int vlq_host_imipq_set_train_iters(void* index, int niter) { GUARD(IMI(index)->cp_.niter = niter) }
int vlq_host_imipq_set_codebooks(void* index, const float* coarse, const float* pq) {
  GUARD(IMI(index)->setCodebooks(coarse, pq))
}
int vlq_host_imipq_get_codebooks(void* index, float* coarse, float* pq) { GUARD(IMI(index)->getCodebooks(coarse, pq)) }
int vlq_host_imipq_search_cells(void* index, long n, const float* x, int nprobe, float* distances, long* labels) {
  GUARD(IMI(index)->searchCells(n, x, nprobe, distances, labels))
}
int vlq_host_imipq_list_length(void* index, long cell, int* out) { GUARD(*out = IMI(index)->getListLength(cell)) }

}  // extern "C"
