/* vlq_index_c.h -- C wrapper over the C++ host layer (vector_line_quantization_b200/host): the faiss::Index-shaped
 * classes GpuIndexFlatL2 / GpuIndexIVFPQ(VLQ) / IndexProxy / IndexShards / Clustering, for ctypes / FFI callers.
 * Every function returns 0 on success and -1 on failure (message: vlq_host_last_error(), thread-local).
 * Data pointers (x, ids, D, I) may be host or device, like the reference's Index API (gpu/utils/CopyUtils.cuh:24-58).
 * Mirrors: faiss::Index::{train,add,add_with_ids,search,reset} (Index.h:89-165), GpuIndexIVF::setNumProbes,
 * GpuIndexIVFPQ::{w1_, merge, write/readCodebookToFile, write/readDbToFile, getList*} (gpu/GpuIndexIVFPQ.h:59-151). */
#ifndef VLQ_INDEX_C_H
#define VLQ_INDEX_C_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

const char* vlq_host_last_error(void);

/* StandardGpuResources */
int vlq_host_resources_new(int device, void** out);
int vlq_host_resources_free(void* res);
int vlq_host_resources_sync(void* res); /* wait for the resource's default stream (syncDefaultStream) */

/* any index handle (flat, VLQ, proxy, shards): the faiss::Index virtual API */
int vlq_host_index_free(void* index);
int vlq_host_index_train(void* index, long n, const float* x);
int vlq_host_index_add(void* index, long n, const float* x);
int vlq_host_index_add_with_ids(void* index, long n, const float* x, const long* ids);
int vlq_host_index_search(void* index, long n, const float* x, long k, float* distances, long* labels);
int vlq_host_index_reset(void* index);
/* Index::remove_ids with IDSelectorRange [imin, imax) / IDSelectorBatch (ids in host or device memory); *nremoved gets
   the number of entries removed.  GpuIndexIVFPQ and GpuIndexIMIPQ implement it; other indexes fail (-1). */
int vlq_host_index_remove_ids_range(void* index, long imin, long imax, long* nremoved);
int vlq_host_index_remove_ids_batch(void* index, long n, const long* ids, long* nremoved);
/* Index::range_search: every stored vector with squared L2 distance < radius for each of the n queries (x host or
   device).  *result receives a RangeSearchResult handle: vlq_host_range_result_total gives lims[n] (the number of
   results), vlq_host_range_result_copy writes any of lims [n + 1], distances and labels [total] (host memory; NULL
   skips one) and vlq_host_range_result_free releases it.  GpuIndexIVFPQ and GpuIndexIMIPQ implement it; other indexes
   fail (-1) and leave *result NULL. */
int vlq_host_index_range_search(void* index, long n, const float* x, float radius, void** result);
int vlq_host_range_result_total(void* result, long* total);
int vlq_host_range_result_copy(void* result, long* lims, float* distances, long* labels);
int vlq_host_range_result_free(void* result);
long vlq_host_index_ntotal(void* index);
int vlq_host_index_is_trained(void* index);

/* GpuIndexFlatL2 + its VLQ helper surface */
int vlq_host_flat_new(void* res, int d, int use_tensor_cores, void** out);
int vlq_host_flat_assign(void* flat, long n, const float* x, int* labels);
int vlq_host_index_reconstruct_n(void* index, long i0, long ni, float* recons); /* Index::reconstruct_n; throws (-1) where undecodable */
/* Index::reconstruct_batch: the stored vectors of keys[0 .. n) (ids, any order) into recons [n][d]; a key without an
   entry fails (-1) and nothing is written.  Index::search_and_reconstruct: search plus the vector behind every label,
   recons [n][k][d], NaN rows for label -1.  Pointers may be host or device memory for GpuIndexIVFPQ / GpuIndexIMIPQ. */
int vlq_host_index_reconstruct_batch(void* index, long n, const long* keys, float* recons);
int vlq_host_index_search_and_reconstruct(void* index, long n, const float* x, long k, float* distances, long* labels,
                                          float* recons);
int vlq_host_flat_search_int(void* flat, long n, const float* x, long k, float* distances, int* labels); /* searchInt */
/* assign1Base: device pointers only; line id (assign2 = A*numedge + e) and float lambda of every row */
int vlq_host_flat_assign1_base(void* flat, long n, const float* d_input, const int* d_assign1, int* d_assign2,
                               float* d_lambdaf, const int* d_edge, const float* d_edge_dist, int numedge);
int vlq_host_flat_build_graph(void* flat, int nedge, float* distances, int* labels);

/* Clustering::train over a GpuIndexFlatL2 assigner */
int vlq_host_kmeans(void* res, int d, int k, long n, const float* x, int niter, int seed, float* centroids_out);

/* GpuIndexIVFPQ with the VLQ constructor (res, d, nlist, M, bits, nedge, nLambda, METRIC_L2) */
int vlq_host_vlq_new(void* res, int d, int nlist, int M, int bits, int nedge, int nlambda, int use_tensor_cores,
                     void** out);
int vlq_host_vlq_set_nprobe(void* index, int nprobe);
int vlq_host_vlq_set_w1(void* index, int w1);
int vlq_host_vlq_set_list_cap(void* index, int cap);
int vlq_host_vlq_set_train_iters(void* index, int niter);
/* uint8-valued vectors: bytes over PCIe, widened on the device (ids may be NULL: sequential) */
int vlq_host_vlq_add_with_ids_u8(void* index, long n, const unsigned char* x, const long* ids);
int vlq_host_vlq_reserve_memory(void* index, long num_vecs); /* GpuIndexIVFPQ::reserveMemory */
/* sizes: coarse nlist*d, edge / edge_dist nlist*nedge, lambda_cb nlambda, pq 256*d */
int vlq_host_vlq_get_codebooks(void* index, float* coarse, int* edge, float* edge_dist, float* lambda_cb, float* pq);
int vlq_host_vlq_set_codebooks(void* index, const float* coarse, const int* edge, const float* edge_dist,
                               const float* lambda_cb, const float* pq);
int vlq_host_vlq_list_length(void* index, int list, int* out);
int vlq_host_vlq_get_list(void* index, int list, unsigned char* codes, unsigned char* lambdas, long* ids);
int vlq_host_vlq_merge(void* index, long* nns, float* dist, int k, int nq, int nprocess, float* distances, long* labels);
int vlq_host_vlq_write_codebook(void* index, const char* name);
int vlq_host_vlq_read_codebook(void* index, const char* name);
int vlq_host_vlq_write_db(void* index, const char* name);
int vlq_host_vlq_read_db(void* index, const char* name, int pronum, int rank);

/* the permutation Clustering::train subsamples and initialises with (rand_perm, utils.cpp:307-317, on the glibc random_r
 * generator of utils.cpp:135-160): host-only, exposed so that CPU tests can pin it against the reference library */
int vlq_host_rand_perm(int* perm, long n, long seed);

/* dataset / matrix formats of the reference drivers (filehelper.cpp:106-345): TexMex .fvecs (kind 0) / .ivecs (1) /
 * .bvecs (2), and the .umem/.imem layout (ASCII "num\ndim\n" header, payload at byte 20) */
int vlq_host_vecs_header(const char* path, int elem_size, long* n, long* d);
int vlq_host_vecs_read(const char* path, int kind, long start, long num, void* out); /* num == 0: to the end */
int vlq_host_vecs_write(const char* path, int kind, const void* x, long n, long d);
int vlq_host_umem_header(const char* path, long* num, long* dim);
int vlq_host_umem_write(const char* path, long num, long dim, const void* ptr, int elem_size, long len, long offset);
int vlq_host_umem_read(const char* path, void* ptr, int elem_size, long len, long offset);

/* IndexProxy (replicas) / IndexShards (database shards); sub-indexes are borrowed */
int vlq_host_proxy_new(void** out);
int vlq_host_proxy_add_index(void* proxy, void* index);
int vlq_host_shards_new(int d, int threaded, int successive_ids, void** out);
int vlq_host_shards_add_shard(void* shards, void* index);

/* ---- f4: exchange with a CPU faiss::IndexIVFPQ (container: centroids, PQ codebook, per-list ids + codes), candidate
   lists and the ground-truth builder (reference gpu/GpuIndexIVFPQ.cu:169-281, 1312-1398, 1646-1670) */
int vlq_host_cpu_ivfpq_new(int d, long nlist, int M, int nbits, void** out);
int vlq_host_cpu_ivfpq_free(void* cpu_index);
int vlq_host_cpu_ivfpq_set_codebooks(void* cpu_index, const float* coarse, const float* pq);
int vlq_host_cpu_ivfpq_get_codebooks(void* cpu_index, float* coarse, float* pq);
int vlq_host_cpu_ivfpq_set_list(void* cpu_index, long list, long n, const long* ids, const unsigned char* codes);
long vlq_host_cpu_ivfpq_list_size(void* cpu_index, long list);
long vlq_host_cpu_ivfpq_ntotal(void* cpu_index);
int vlq_host_cpu_ivfpq_get_list(void* cpu_index, long list, long* ids, unsigned char* codes);
int vlq_host_ivfpq_copy_from(void* index, void* cpu_index);
int vlq_host_ivfpq_copy_to(void* index, void* cpu_index);
int vlq_host_ivfpq_search1(void* index, long n, const float* x, long k, long* labels);
int vlq_host_ivfpq_add_with_ids2(void* index, long n, long nq, unsigned kgt, const float* x, const float* xq, const long* ids,
                                 long* nns, float* dists);

/* ---- f3: GpuIndexIMIPQ = MultiIndexQuantizer(d, 2, nbits_coarse) + IndexIVFPQ over the 2^(2 nbits_coarse) cells on the
   device (reference CPU composition: tests/sift1b_imi_pq.cpp:216-236); train / add / search / reset through the
   vlq_host_index_* calls above; search returns full squared distances like IndexIVFPQ::search */
int vlq_host_imipq_new(void* res, int d, int nbits_coarse, int M, int nbits, void** out);
int vlq_host_imipq_set_nprobe(void* index, int nprobe);
int vlq_host_imipq_set_train_iters(void* index, int niter);
int vlq_host_imipq_set_codebooks(void* index, const float* coarse, const float* pq); /* (2, K, d/2), (M, 256, d/M) */
int vlq_host_imipq_get_codebooks(void* index, float* coarse, float* pq);
/* MultiIndexQuantizer::search: the nprobe cells (label i1 | i2 << nbits_coarse) with the smallest d1 + d2, ascending */
int vlq_host_imipq_search_cells(void* index, long n, const float* x, int nprobe, float* distances, long* labels);
int vlq_host_imipq_list_length(void* index, long cell, int* out);

#ifdef __cplusplus
}
#endif
#endif
