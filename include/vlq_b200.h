/* vlq_b200.h -- C-ABI of the B200-native (sm_100a) VLQ hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): every entry point takes raw DEVICE pointers, explicit sizes, a
 * caller-provided workspace where one is needed (paired with a *_workspace_bytes query) and a cudaStream_t passed as
 * void*.  Functions return 0 on success, a negative VLQ_E* code for invalid arguments, or a positive cudaError_t.
 * They never throw, never allocate device memory and never synchronise the stream (the only exceptions are the
 * explicitly named memory / stream helpers at the bottom, which exist so that a host layer needs no CUDA headers).
 *
 * Each compute entry cites the reference interface it replaces (paths relative to the reference repository).
 * There is no CPU fallback: if the CUDA library cannot be loaded the host layers fail loudly.
 */
#ifndef VLQ_B200_H
#define VLQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLQ_OK 0
#define VLQ_EINVAL (-1)    /* bad argument (null pointer, size out of range, unsupported d / M / k) */
#define VLQ_EWORKSPACE (-2) /* workspace too small */
#define VLQ_EUNSUPPORTED (-3)

#define VLQ_MAX_K 1024      /* k, nprobe (P) and w1 (W) limits of the reference: gpu/GpuIndexFlat.cu:226-232,
                               gpu/GpuIndexIVF.cu:201-207, gpu/impl/IVFPQ.cu:697-698 */
#define VLQ_LIST_CAP 1024   /* lists are truncated to their first 1024 entries at scan time:
                               gpu/impl/IVFUtils.cu:87, gpu/impl/PQScanMultiPassPrecomputed.cu:728 */

typedef void* vlq_stream_t; /* cudaStream_t */

const char* vlq_error_string(int code);
const char* vlq_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
uint64_t vlq_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------------
 * a1  row norms ||x_i||^2.                          replaces runL2Norm, gpu/impl/L2Norm.cu:34-173 (FlatIndex.cu:369-439)
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_row_norms(const float* x, int64_t n, int d, float* out, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a2  nearest centroid per vector (k = 1), exact fp32 CUDA-core path.
 *     replaces runL2Distance(k=1) = runMatrixMult + l2SelectMin1 + sumAlongRows,
 *     gpu/impl/Distance.cu:579-710, gpu/impl/L2Select.cu:25-121, gpu/impl/BroadcastSum.cu:677-698
 *     (CPU twin knn_L2sqr, utils.cpp:833-901).
 *     out_dist (nullable) = ||c||^2 - 2 x.c (+ ||x||^2 when add_xnorm).  Ties -> lowest centroid id.
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_l2_assign(const float* x, int64_t n, int d, const float* cent, const float* cnorm, int C, int add_xnorm,
                  int* out_ids, float* out_dist, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a2 / a11 on the tensor cores (tcgen05 + TMEM): same contracts as vlq_l2_assign / vlq_l2_distances.
 *     replaces cublasSgemm via runMatrixMult (gpu/utils/MatrixMult.cu:90-147; call sites gpu/impl/Distance.cu:356-362,
 *     679-685) + l2SelectMin1 (gpu/impl/L2Select.cu:25-121) -- the distance matrix is never materialised for k = 1.
 *     Arithmetic: operands split into fp16 hi + lo after an exact power-of-two pre-scale, three tcgen05.mma passes
 *     (hi.hi + hi.lo + lo.hi) accumulated in fp32 TMEM: fp32-GEMM-grade results (see DESIGN.md, "precision").
 *     Supported when vlq_tc_supported(d, C): d a multiple of 32, 32 <= d <= 128.  Other shapes use the exact fp32
 *     CUDA-core entry points above (the host layer dispatches; both are CUDA, there is no CPU path).
 *     cent_pack is produced once per codebook by vlq_tc_pack_centroids (packed fp16 tiles + padded ||c||^2);
 *     `scale` (the same power of two in the pack call and the query calls) scales the CENTROIDS: choose it so that
 *     max|c|*scale is about 2^9.  Vectors / queries are scaled per row by their own power of two inside the call
 *     (max|x_row| -> [2^8, 2^9)), so inputs of any magnitude stay inside fp16's range.
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_tc_supported(int d, int C);
size_t vlq_tc_cent_pack_bytes(int C, int d);
int vlq_tc_pack_centroids(const float* cent, const float* cnorm, int C, int d, float scale, void* cent_pack,
                          vlq_stream_t stream);
size_t vlq_l2_tc_workspace_bytes(int64_t n, int d, int C);
/* add_xnorm != 0: out_dist gets ||x||^2 added (true squared distance) */
int vlq_l2_assign_tc(const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, int add_xnorm,
                     int* out_ids, float* out_dist, void* workspace, size_t workspace_bytes, vlq_stream_t stream);
/* bucket_min (nullable): [n][vlq_tc_num_buckets(C)], the minimum of every 32-column bucket of D, produced by the GEMM
 * epilogue for free; vlq_coarse_select_lines uses it to find the top-P centroids from 2*P*32 bytes instead of 4*C. */
int vlq_tc_num_buckets(int C);
int vlq_l2_distances_tc(const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, float* D,
                        int64_t ldD, float* bucket_min, void* workspace, size_t workspace_bytes, vlq_stream_t stream);
/* the same sweep WITHOUT the distance matrix: only bucket_min [n][vlq_tc_num_buckets(C)] is written (the query path
 * re-evaluates the few columns it needs, vlq_coarse_select_lines_exact).  Replaces the nq x C matrix the reference
 * materialises in runL2Distance, gpu/impl/Distance.cu:233-383. */
int vlq_l2_bucket_min_tc(const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, float* bucket_min,
                         void* workspace, size_t workspace_bytes, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a11 coarse distance matrix for a query tile, D[i][j] = ||c_j||^2 - 2 x_i.c_j  (NO ||x||^2, Distance.cu:287-290).
 *     replaces runMatrixMult + the in-place "+||c||^2" of l2SelectMinK, gpu/impl/Distance.cu:352-373.
 *     D is [n][ldD] with ldD >= C.
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_l2_distances(const float* x, int64_t n, int d, const float* cent, const float* cnorm, int C, float* D,
                     int64_t ldD, vlq_stream_t stream);

/* a11/a15 exact top-k per row, ascending, ties by lowest column; pads with (FLT_MAX, -1).  k <= VLQ_MAX_K.
 *     replaces l2SelectMinK / BlockSelect, gpu/impl/L2Select.cu:124-165, gpu/utils/Select.cuh:77-277
 *     (CPU twin Heap.h:89-323).  row_add (nullable) is added to the k winners of each row (sumAlongRows). */
int vlq_select_rows(const float* D, int64_t n, int cols, int64_t ldD, int k, const float* row_add, float* out_val,
                    int* out_idx, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a4  centroid kNN graph: E+1 nearest centroids by GEMM-form exact distance, rank 0 dropped.
 *     replaces GpuIndexFlat::buildGraph / buildGraphNonPaged_, gpu/GpuIndexFlat.cu:375-429,869-893.
 * ---------------------------------------------------------------------------------------------------------------- */
size_t vlq_knn_graph_workspace_bytes(int C, int E);
int vlq_knn_graph(const float* cent, const float* cnorm, int C, int d, int E, int* edge, float* edge_d2,
                  void* workspace, size_t workspace_bytes, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a5-a8 fused line stage + lambda quantiser + residual + PQ encode.
 *     replaces get1BinKernel_nms (gpu/GpuIndexFlat.cu:433-557, gpu/utils/triangle.cuh:54-87),
 *     assignLambdaKernel (gpu/GpuIndexFlat.cu:559-602), calResidual (gpu/GpuIndexFlat.cu:1092-1129) and the PQ
 *     encode of classifyAndAddVectors (gpu/GpuIndexIVFPQ.cu:646-706; CPU twin ProductQuantizer.cpp:311-336).
 *     pq is (M, ksub=256, dsub) fp32.  Outputs (any may be NULL except out_list):
 *       out_list[n]    = A*E + e            out_lambda[n] = float lambda (unquantised)
 *       out_lamq[n]    = argmin_j (lambda - lambda_cb[j])^2
 *       out_codes[n*M] = PQ codes of r = x - ((1-l)c_A + l c_s), l = lambda_cb[lamq]
 *       out_kappa[n]   = ||p||^2 + 2 anchor.p   (query-independent part of the ADC distance, see DESIGN.md)
 *       out_residual[n*d]
 *     If lambda_cb is NULL only out_list / out_lambda are produced (the training-time call assign1).
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_line_encode(const float* x, int64_t n, int d, const int* assign, const float* cent, const int* edge,
                    const float* edge_d2, int E, const float* lambda_cb, int nL, const float* pq, int M,
                    int* out_list, float* out_lambda, uint8_t* out_lamq, uint8_t* out_codes, float* out_kappa,
                    float* out_residual, vlq_stream_t stream);

/* a6 stand-alone: lambda -> uint8 = argmin_j (lambda - lambda_cb[j])^2, lowest j on ties.
 *     replaces assignLambdaKernel, gpu/GpuIndexFlat.cu:559-602 (host wrapper assignLambda :702-752). */
int vlq_lambda_quantize(const float* lambda, int64_t n, const float* lambda_cb, int nL, uint8_t* out,
                        vlq_stream_t stream);
/* a7 stand-alone: r = x - ((1-l) c_A + l c_s), l = lambda_cb[lamq], list = A*E + e (rows with list < 0 give 0).
 *     replaces calResidual, gpu/GpuIndexFlat.cu:1092-1129 (host wrapper compute_residual :1194-1258). */
int vlq_line_residual(const float* x, int64_t n, int d, const int* list, const uint8_t* lamq, const float* lambda_cb,
                      const float* cent, const int* edge, int E, float* residual, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a9  inverted-list construction: stable counting sort of n new entries (arrival order) behind n_old entries that
 *     are already list-major.   replaces the host hash-map / per-byte copies / runUpdateListPointers /
 *     runIVFPQInvertedListAppend of gpu/GpuIndexIVFPQ.cu:741-905, gpu/impl/InvertedListAppend.cu:20-120.
 *     Layout (CSR): offsets[nlists+1] int64; codes[n][M], lamq[n], kappa[n], ids[n] in list-major order, insertion
 *     order preserved inside a list (what the reference's per-list append produces).
 * ---------------------------------------------------------------------------------------------------------------- */
size_t vlq_build_lists_workspace_bytes(int64_t n_new, int64_t nlists);
int vlq_build_lists(int64_t nlists, int M,
                    /* existing lists (may be empty: n_old == 0, pointers NULL) */
                    int64_t n_old, const int64_t* old_offsets, const uint8_t* old_codes, const uint8_t* old_lamq,
                    const float* old_kappa, const int64_t* old_ids,
                    /* new entries in arrival order */
                    int64_t n_new, const int* new_list, const uint8_t* new_codes, const uint8_t* new_lamq,
                    const float* new_kappa, const int64_t* new_ids,
                    /* merged output, sized n_old + n_new */
                    int64_t* out_offsets, uint8_t* out_codes, uint8_t* out_lamq, float* out_kappa, int64_t* out_ids,
                    void* workspace, size_t workspace_bytes, vlq_stream_t stream);

/* a9 (removal): stable compaction of the CSR slab above, the survivors keeping their order inside their list (the
 *     reference's IndexIVF::remove_ids, IndexIVF.cpp, swaps each removed entry with the last of its list instead).
 *     An entry is removed iff range_lo <= id < range_hi OR id is in batch[0 .. n_batch), sorted ascending (duplicates
 *     allowed; range_lo >= range_hi: no range).  offsets[nlists] must equal n.
 *     pass 1 (plan) writes out_offsets[nlists + 1] of the survivors; out_offsets[nlists] = survivor count, which the
 *     caller reads to size the new slab.  pass 2 (apply) gathers the survivors into out_* and re-rotates every code word
 *     to its new list position; it reads the workspace pass 1 wrote, unchanged in between.  out_* must be non-NULL when
 *     n > 0.  The workspace holds the keep mask (n / 8 bytes) and one int64 per 8192 entries; nlists does not enter it. */
size_t vlq_remove_ids_workspace_bytes(int64_t n, int64_t nlists);
int vlq_remove_ids_plan(int64_t nlists, int64_t n, const int64_t* offsets, const int64_t* ids, int64_t range_lo,
                        int64_t range_hi, const int64_t* batch, int64_t n_batch, int64_t* out_offsets, void* workspace,
                        size_t workspace_bytes, vlq_stream_t stream);
int vlq_remove_ids_apply(int64_t nlists, int M, int64_t n, const int64_t* offsets, const uint8_t* codes,
                         const uint8_t* lamq, const float* kappa, const int64_t* ids, const int64_t* out_offsets,
                         uint8_t* out_codes, uint8_t* out_lamq, float* out_kappa, int64_t* out_ids,
                         const void* workspace, size_t workspace_bytes, vlq_stream_t stream);

/* a9 (read-back): id lookup and decode of stored entries (Index::reconstruct / reconstruct_n / search_and_reconstruct,
 *     IndexIVFPQ::reconstruct_from_offset in the reference).
 *     vlq_lookup_ids: one pass over ids[n]; out_pos[slot] = the LOWEST slab index whose id maps to the slot, -1 if none;
 *       *out_found (one int64 on the device) = the number of slots found.  keys == NULL: range mode, slot = id - range_lo
 *       for range_lo <= id < range_lo + nslots.  keys != NULL: batch mode, keys[nslots] sorted ascending and unique, slot
 *       = index of the id in keys.  There is no persistent id -> slab map: every call reads the ids once.
 *     vlq_decode_entries (VLQ) / vlq_imi_decode_entries (IMI-PQ, nlists = 2^(2 nbits), cell l = i1 | i2 << nbits):
 *       out_x[i][j] = anchor_j + pq[m][code_m][j - m dsub], m = j / dsub, of the entry at slab index pos[i] of list l
 *       (offsets[l] <= pos[i] < offsets[l + 1]), its stored code bytes un-rotated by (pos[i] - offsets[l]) mod M;
 *         VLQ anchor = (1 - lh) cent[l / E] + lh cent[edge[l]], lh = lambda_cb[lamq[pos[i]]]   (nlists = C E)
 *         IMI anchor = [cb1[i1] | cb2[i2]]   (cb1, cb2: [2^nbits][d / 2])
 *       fp32, each operation rounded as written (no fma contraction), summed in the order shown: a lambda codebook {0}
 *       gives exactly c + p (IndexIVFPQ's decode).  pos[i] = -1 (or outside the slab) gives a row of NaN (all-ones bits)
 *       and out_ids[i] = -1.  out_ids (nullable) = ids[pos[i]]; it may alias pos (the scan's slab-index output turned
 *       into labels in place).  M <= 64, d % M == 0 (IMI: d even). */
int vlq_lookup_ids(int64_t n, const int64_t* ids, int64_t range_lo, const int64_t* keys, int64_t nslots, int64_t* out_pos,
                   int64_t* out_found, vlq_stream_t stream);
int vlq_decode_entries(int64_t n, const int64_t* pos, int64_t nlists, const int64_t* offsets, const uint8_t* codes,
                       const uint8_t* lamq, const int64_t* ids, int M, int d, const float* pq, const float* cent,
                       const int* edge, int E, const float* lambda_cb, int nL, float* out_x, int64_t* out_ids,
                       vlq_stream_t stream);
int vlq_imi_decode_entries(int64_t n, const int64_t* pos, const int64_t* offsets, const uint8_t* codes,
                           const int64_t* ids, int M, int d, const float* pq, const float* cb1, const float* cb2,
                           int nbits, float* out_x, int64_t* out_ids, vlq_stream_t stream);

/* a9 (loader): per-entry kappa = ||p||^2 + 2 anchor.p for list-major entries that arrive without it, i.e. lists read
 *     from the reference's .dbIdx/.dbcodes/.dbcount/.dblas files (gpu/GpuIndexIVFPQ.cu:1813-2010). */
int vlq_recompute_kappa(int64_t n, int64_t nlists, const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq,
                        const float* cent, int d, const int* edge, int E, const float* lambda_cb, const float* pq, int M,
                        float* kappa, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a12 query-time line selection: the W best of the P*E lines of the P probed centroids.
 *     replaces sumAlongRowsWithOrder2 / runL2SelectMinGraph, gpu/impl/BroadcastSum.cu:477-560,819-860.
 *     D is the coarse matrix of vlq_l2_distances; coarse_ids [nq][P].
 *     Outputs [nq][W]: out_list = c*E+e (-1 padded), out_term1 = D[c], out_term6 = D[s]-D[c].
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_select_lines(const float* D, int64_t nq, int64_t ldD, const int* coarse_ids, int P, const int* edge,
                     const float* edge_d2, int E, int W, int* out_list, float* out_term1, float* out_term6,
                     vlq_stream_t stream);

/* a11 + a12 fused (tensor-core query path): top-P centroids found through the bucket minima of
 *     vlq_l2_distances_tc, then the line selection of vlq_select_lines, in one kernel.  Same outputs as
 *     vlq_select_rows(k=P) + vlq_select_lines; out_coarse (nullable) [nq][P] receives the top-P centroid ids.
 *     replaces l2SelectMinK + sumAlongRowsWithOrder2, gpu/impl/L2Select.cu:124-165, gpu/impl/BroadcastSum.cu:477-560. */
int vlq_coarse_select_lines(const float* D, int64_t nq, int64_t ldD, const float* bucket_min, int nb, int C, int P,
                            const int* edge, const float* edge_d2, int E, int W, int* out_coarse, int* out_list,
                            float* out_term1, float* out_term6, vlq_stream_t stream);

/* a11 + a12 without a distance matrix: the top-P buckets come from bucket_min (vlq_l2_bucket_min_tc), the 32 columns of
 *     each of them and the P*E neighbour centroids of the top-P are re-evaluated in fp32 from cent [C][d] / cnorm [C]
 *     (D[c] = ||c||^2 - 2 q.c, the same definition).  Same outputs as vlq_coarse_select_lines up to the rounding of D
 *     (near-ties only).  vlq_coarse_exact_supported: d % 4 == 0, d <= 128, max(num_buckets, 32 P, P E) <= 4096, W <= 1024;
 *     otherwise VLQ_EUNSUPPORTED (callers fall back to the matrix path).  q, cent, bucket_min 16-byte aligned.
 *     replaces l2SelectMinK + sumAlongRowsWithOrder2, gpu/impl/L2Select.cu:124-165, gpu/impl/BroadcastSum.cu:477-560.
 *     vlq_coarse_exact_preferred: supported AND faster than the matrix route (at most 256 KiB of centroid rows per
 *     query, i.e. small nprobe: P (32 + E) d 4 bytes from L2 against 4 C bytes of D written to HBM). */
int vlq_coarse_exact_supported(int d, int C, int P, int E, int W);
int vlq_coarse_exact_preferred(int d, int C, int P, int E, int W);
int vlq_coarse_select_lines_exact(const float* q, int64_t nq, int d, const float* cent, const float* cnorm,
                                  const float* bucket_min, int nb, int C, int P, const int* edge, const float* edge_d2,
                                  int E, int W, int* out_coarse, int* out_list, float* out_term1, float* out_term6,
                                  vlq_stream_t stream);

/* a11 + a12 for one query tile, the route chosen here: the one entry the index's search and the Python operator layer
 *     call.  Outputs as vlq_coarse_select_lines (out_coarse nullable [nq][P]); 1 <= P <= min(C, VLQ_MAX_K).
 *     vlq_coarse_route (have_pack: cent_pack of vlq_tc_pack_centroids will be passed):
 *       0  no pack:                                        vlq_l2_distances + vlq_select_rows + vlq_select_lines
 *       1  tcgen05 matrix:                                 vlq_l2_distances_tc (+ bucket minima) + vlq_coarse_select_lines
 *       2  matrix-free (vlq_coarse_exact_preferred):       vlq_l2_bucket_min_tc + vlq_coarse_select_lines_exact
 *     The environment switches VLQ_COARSE_MATRIX (route 1) and VLQ_COARSE_EXACT (route 2 wherever supported) are read on
 *     every call (tests and tuning only).  The workspace (vlq_coarse_lines_workspace_bytes, which applies the same rule;
 *     256-byte aligned, as the device allocators return it) holds only what the route uses: the distance tile [nq][C]
 *     (routes 0, 1), the bucket minima and the vlq_l2_tc_workspace_bytes block (routes 1, 2), the top-P of route 0.
 *     Too small: VLQ_EWORKSPACE.  q (routes 1, 2) and cent (route 2) 16-byte aligned.  Every argument is checked before
 *     the first launch. */
int vlq_coarse_route(int d, int C, int P, int E, int W, int have_pack);
size_t vlq_coarse_lines_workspace_bytes(int64_t nq, int d, int C, int P, int E, int W, int have_pack);
int vlq_coarse_lines(const float* q, int64_t nq, int d, const float* cent, const float* cnorm, const void* cent_pack,
                     float scale, int C, int P, const int* edge, const float* edge_d2, int E, int W, int* out_coarse,
                     int* out_list, float* out_term1, float* out_term6, void* workspace, size_t workspace_bytes,
                     vlq_stream_t stream);

/* candidate lists (f4): ids of the entries of the W selected lines of every query in line order, first k of them, -1
   padded -- the recall-of-the-candidate-list tool GpuIndexIVFPQ::search1 / IVFPQ::queryGraph1
   (gpu/GpuIndexIVFPQ.cu:1646-1670, gpu/impl/IVFPQ.cu:778-870: a host loop over listOffsetToUserIndex_ there) */
int vlq_gather_candidates(const int* line_list, int64_t nq, int W, const int64_t* offsets, const int64_t* ids, int64_t k,
                          int64_t* out, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a13-a15 ADC scan of the selected lists fused with exact top-k.
 *     replaces the term3 build (gpu/impl/IVFPQ.cu:1398-1432), pqScanPrecomputedMultiPassGraph
 *     (gpu/impl/PQScanMultiPassPrecomputed.cu:675-881), runCalcListOffsetsGraph (gpu/impl/IVFUtils.cu:133-169),
 *     pass1SelectLists / pass2SelectListsGraph (gpu/impl/IVFUtilsSelect1.cu:28-144, IVFUtilsSelect2.cu:398-569).
 *     dist = term1 + l*term6 + (l*l-l)*term5 + kappa_i - 2 q.p(code_i),  l = lambda_cb[lamq_i]
 *          = ||q - ((1-l)c + l s) - p(code_i)||^2 - ||q||^2              (same value as the reference's formula)
 *     over the first min(len, cap) entries of each selected list; k smallest ascending, padded (FLT_MAX, -1).
 *     edge_d2 is indexed by list id (term5); NULL = 0 (an index whose lambda codebook is {0}: stock IVFPQ / IMI-PQ).
 *     k <= VLQ_MAX_K, W <= VLQ_MAX_K.
 *     ids == NULL: outI receives each result's SLAB index (the entry's position in codes / lamq / kappa) instead of its
 *     id; selection does not depend on ids, so distances and order are unchanged.  search_and_reconstruct decodes the
 *     exact entries found this way (vlq_decode_entries), which ids alone cannot name when an id is stored twice.
 *     list_len_hint: average list length of the index (entries / lists; 0 = unknown).  >= 24 selects the
 *     warp-per-list walk (1B-scale lists), otherwise the flattened entry stream (lists of a few entries).  Results are
 *     identical either way.
 *     workspace (optional, vlq_scan_topk_workspace_bytes): holds the term-3 tables of the batch, built by one
 *     persistent kernel with the PQ codebook in shared memory; with workspace == NULL every query CTA builds its own.
 *     The one exception to "never synchronises": the FIRST call of a process that selects the long-list kernel
 *     (list_len_hint >= 160) runs a one-thread probe kernel and copies 4 bytes back (base address of the dynamic shared
 *     memory, which that kernel folds into its load instructions); later calls only enqueue work.
 * ---------------------------------------------------------------------------------------------------------------- */
size_t vlq_scan_topk_workspace_bytes(int64_t nq, int M);
int vlq_scan_topk(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                  const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                  const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa,
                  const int64_t* ids, int k, int cap, int list_len_hint, float* outD, int64_t* outI, void* workspace,
                  size_t workspace_bytes, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a15-range  radius search over the selected lines: every entry the scan above would look at (the first min(len, cap)
 *     entries of each of the W lines in line_list, -1 slots skipped) whose distance is below `radius` (strict), in
 *     stream order: lines in slot order, then list position.   replaces IndexIVF::range_search (IndexIVF.cpp) for the
 *     line lists, which the reference GPU index lacks.
 *     dist = term1 + l*term6 + (l*l-l)*term5 + kappa_i - 2 q.p(code_i) + row_add[q]   (row_add nullable; pass ||q||^2 for
 *     the full squared L2 when term1 excludes it, as the VLQ coarse stage does; NULL when term1 = ||q - c||^2, IMI-PQ),
 *     evaluated in fp32 from term-3 tables in a fixed order, each operation rounded as written: both passes compute the
 *     same bits, and results do not depend on the list lengths.  edge_d2 NULL = lambda-hat 0.
 *     pass 1 (count) builds the term-3 tables of the nq queries into the workspace, counts the survivors of every query
 *       and writes out_lims[nq + 1] (exclusive prefix; out_lims[nq] = total, which the caller reads to size its output).
 *     pass 2 (gather) reads the workspace pass 1 wrote, unchanged in between, and writes the results of the queries
 *       [q0, q1) to outD / outI at lims[q] - lims[q0]: a large tile can be gathered in parts.
 *     M <= 64, d % M == 0, 1 <= nL <= 256, 1 <= W <= VLQ_MAX_K, 1 <= cap <= 2^20, W * cap < 2^31; a NaN radius is
 *     VLQ_EINVAL; pq and workspace 16-byte aligned.  VLQ_EUNSUPPORTED where the term-3 kernels do not take the shape:
 *     d % 4 != 0, or the codebook plus one query (1028 d bytes) beyond 200 KiB of shared memory, i.e. d > 196 (GloVe-200
 *     is refused).  Every argument is checked before the first launch.
 * ---------------------------------------------------------------------------------------------------------------- */
size_t vlq_range_workspace_bytes(int64_t nq, int M, int W, int cap);
int vlq_range_count(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                    const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                    const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa, int cap,
                    const float* row_add, float radius, int64_t* out_lims, void* workspace, size_t workspace_bytes,
                    vlq_stream_t stream);
int vlq_range_gather(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                     const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                     const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa, int cap,
                     const float* row_add, float radius, const int64_t* ids, const int64_t* lims, int64_t q0, int64_t q1,
                     float* outD, int64_t* outI, const void* workspace, size_t workspace_bytes, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * a16 shard merge: k smallest of R*k candidates per query; D, I are [R][nq][k] (the all-gather layout); shards with
 *     fewer than k results pad with (FLT_MAX, -1), as vlq_scan_topk does.
 *     replaces GpuIndexIVFPQ::merge / mergekernel, gpu/GpuIndexIVFPQ.cu:1467-1591 (CPU twin MetaIndexes.cpp:290-347).
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_merge_topk(const float* D, const int64_t* I, int R, int64_t nq, int k, float* outD, int64_t* outI,
                   vlq_stream_t stream);
/* Same merge with the gather fused in: shard r's (nq,k) results are read where they were produced, from
 * peer_bufs[r] + d_offset_bytes (f32 distances) and + i_offset_bytes (int64 ids).  peer_bufs is a DEVICE array of R
 * device pointers; entries may point into the memory of other GPUs of the NVLink domain (peer-mapped), which turns the
 * MPI_Gather + mergekernel pair of gpu/test/sift1b16_query.cpp / GpuIndexIVFPQ.cu:1467-1591 into one kernel of P2P
 * loads.  The caller orders it after the producers (a cross-GPU barrier); results are identical to vlq_merge_topk. */
int vlq_merge_topk_peers(const void* const* peer_bufs, size_t d_offset_bytes, size_t i_offset_bytes, int R, int64_t nq,
                         int k, float* outD, int64_t* outI, vlq_stream_t stream);
/* Query-split sharding: every rank holds narr (<= 4) row-major arrays of nq rows x row_bytes at arr_offset_bytes[a] of
 * its peer-mapped buffer and has filled the rows [self nq / R, (self + 1) nq / R); this call copies the rows of every
 * other rank r, [r nq / R, (r + 1) nq / R), from peer_bufs[r] into peer_bufs[self] (one kernel of P2P loads).  Offsets
 * and row_bytes are multiples of 16.  The caller orders it after the producers (a cross-GPU barrier).  It is the
 * exchange step of the line lists (12 W bytes per query) where gpu/test/sift1b16_query.cpp broadcasts the queries to
 * every rank and repeats the coarse stage on each of them. */
int vlq_gather_peer_slices(const void* const* peer_bufs, int R, int self, const int64_t* arr_offset_bytes, int narr,
                           int64_t nq, int64_t row_bytes, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * f1 (next row) k-means centroid update on the device: deterministic per-centroid mean in row order + the
 *     reference's empty-cluster split.    replaces km_update_centroids, utils.cpp:1369-1449.
 * ---------------------------------------------------------------------------------------------------------------- */
size_t vlq_km_update_workspace_bytes(int64_t n, int k);
int vlq_km_update(const float* x, int64_t n, int d, const int* assign, int k, float* centroids, int* counts,
                  void* workspace, size_t workspace_bytes, vlq_stream_t stream);


/* ------------------------------------------------------------------------------------------------------------------
 * f3  inverted multi-index (IMI-PQ baseline of BASELINE configs[4]; csrc/imi.cu).
 *     vlq_imi_top_cells: the nprobe cells (label i1 | i2 << nbits) with the smallest d1[i1] + d2[i2] per query, ascending,
 *       ties to the lowest label, padded (-1, FLT_MAX); v1/i1, v2/i2 are the [nq][L] ascending prefixes of the two
 *       half-distance tables (vlq_select_rows), L >= min(nprobe, K).  nprobe <= VLQ_MAX_K.
 *       replaces MultiIndexQuantizer::search / MinSumK, IndexPQ.cpp:637-857 (which may report a cell twice; this does not).
 *     vlq_imi_encode: cell label, residual PQ codes (first minimum wins, ProductQuantizer.cpp:311-336) and
 *       kappa = ||p||^2 + 2 c.p per vector from its two half assignments a1, a2 (-1 -> cell -1).
 *       replaces IndexIVFPQ::add_core_o with a MultiIndexQuantizer (IndexIVFPQ.cpp:160-260) and the per-half
 *       precomputed tables of use_precomputed_table = 2 (IndexIVFPQ.cpp:645-687).
 *     vlq_copy_columns: dst[n][ncols] = src[n][col0 : col0 + ncols] (row stride ld).
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_copy_columns(const float* src, int64_t n, int64_t ld, int col0, int ncols, float* dst, vlq_stream_t stream);
int vlq_imi_top_cells(const float* v1, const int* i1, const float* v2, const int* i2, int64_t nq, int L, int nbits,
                      int nprobe, int* out_cell, float* out_dist, vlq_stream_t stream);
int vlq_imi_encode(const float* x, int64_t n, int d, const int* a1, const int* a2, const float* cb1, const float* cb2,
                   int nbits, const float* pq, int M, int* out_cell, uint8_t* out_codes, float* out_kappa,
                   vlq_stream_t stream);

/* small device utilities used by the host layer */
int vlq_gather_rows(const float* src, int d, const int64_t* rows, int64_t n, float* dst, vlq_stream_t stream);
int vlq_u8_to_f32(const uint8_t* src, int64_t count, float* dst, vlq_stream_t stream);
int vlq_iota_i64(int64_t* dst, int64_t n, int64_t start, vlq_stream_t stream);
int vlq_i32_to_i64(const int* src, int64_t n, int64_t* dst, vlq_stream_t stream);
/* ids[i] += shift for ids[i] >= 0: shard-local -> global labels after a shard search (replaces the host loop of
   IndexShards::search, MetaIndexes.cpp:536-546) */
int vlq_shift_ids(int64_t* ids, int64_t n, int64_t shift, vlq_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Memory / stream helpers (these DO allocate / synchronise; they exist so host layers need no CUDA toolkit).
 * ---------------------------------------------------------------------------------------------------------------- */
int vlq_device_count(int* count);
int vlq_set_device(int device);
int vlq_get_device(int* device);
int vlq_mem_info(size_t* free_bytes, size_t* total_bytes);
int vlq_malloc(void** ptr, size_t bytes);
int vlq_free(void* ptr);
int vlq_malloc_host(void** ptr, size_t bytes); /* pinned */
int vlq_free_host(void* ptr);
int vlq_memcpy_h2d(void* dst, const void* src, size_t bytes, vlq_stream_t stream);
int vlq_memcpy_d2h(void* dst, const void* src, size_t bytes, vlq_stream_t stream);
int vlq_memcpy_d2d(void* dst, const void* src, size_t bytes, vlq_stream_t stream);
int vlq_memset(void* dst, int value, size_t bytes, vlq_stream_t stream);
int vlq_pointer_is_device(const void* ptr); /* 1 device, 0 host, <0 error */
int vlq_pointer_device(const void* ptr, int* device); /* ordinal of the GPU a device pointer lives on (-1: host memory) */
/* let the CURRENT device read `peer_device`'s memory over NVLink (no-op for the same device or when already enabled);
   the in-process shard merge reads the shards' result buffers straight from their GPUs (gpu/test/sift1b16_query.cpp:389-430
   staged them through MPI and host memory) */
int vlq_enable_peer_access(int peer_device);
int vlq_stream_create(vlq_stream_t* stream);
int vlq_stream_destroy(vlq_stream_t stream);
int vlq_stream_synchronize(vlq_stream_t stream);
/* work enqueued on `waiter` after this call starts only when everything enqueued on `producer` so far has finished */
int vlq_stream_wait(vlq_stream_t waiter, vlq_stream_t producer);
/* the same in two halves (record now, wait wherever the dependent work is enqueued later): a plain cudaEvent_t without
   timing.  Used by GpuIndexIVFPQ::search to run the scan of query tile i beside the coarse stage of tile i + 1. */
typedef void* vlq_event_t;
int vlq_event_create(vlq_event_t* ev);
int vlq_event_destroy(vlq_event_t ev);
int vlq_event_record(vlq_event_t ev, vlq_stream_t stream);
int vlq_stream_wait_event(vlq_stream_t waiter, vlq_event_t ev);

#ifdef __cplusplus
}
#endif
#endif /* VLQ_B200_H */
