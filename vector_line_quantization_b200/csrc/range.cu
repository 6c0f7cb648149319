// Radius search over the selected lines (SURVEY.md 8a row a15, range variant of the scan): every entry of the W selected
// lines of a query (the first min(len, cap) of each) whose full squared distance is below the radius, in stream order --
// lines in slot order, entries by list position.  The number of results per query is not known in advance, so the
// entries are walked twice:
//   range_count_kernel<M>  : one CTA per query counts its survivors; one scan turns the counts into lims (lims[nq] = total)
//   range_gather_kernel<M> : one CTA per query recomputes the same distances and writes its survivors at
//                            lims[q] - lims[q0] + their rank in stream order (ballots + warp totals, no atomics)
// Both passes walk the lines as ONE flattened entry stream per query (as scan_topk_kernel<M, false>), so lanes stay busy
// whether a list holds 5 entries or 500, and both compute an entry's distance with range_dist() from the same fp32 term-3
// tables (built into the workspace by the term3 kernels of search.cu): the gather writes exactly what the count counted.
#include <cmath>

#include "scan.cuh"
#include "pq4.cuh"

namespace vlq {

constexpr int R_THREADS = 256;
constexpr int R_WARPS = R_THREADS / kWarp;
constexpr int R_BATCH = 4;  // stream positions per thread and step: the loads of all four are in flight together

struct RangeArgs {
  const float* t3;  // [nq][M][256] term-3 tables of the batch
  int M, nL;
  const float* lambda_cb;
  const int* line_list;
  const float* term1;
  const float* term6;
  const float* edge_d2;
  int W, cap;
  const int64_t* offsets;
  const uint8_t* codes;
  const uint8_t* lamq;
  const float* kappa;
  const int64_t* ids;
  const float* row_add;
  float radius;
  int64_t nq;
  int64_t* counts;      // count pass: [nq + 1]
  const int64_t* lims;  // gather pass
  int64_t q0;
  float* outD;
  int64_t* outI;
};

// Full squared distance of one entry: (kappa + sum_m T3[m][code_m]) + (t1 + l t6 + (l^2 - l) t5) + row_add.  Every
// operation is rounded as written (no contraction into fma), so the two passes, which are separate kernels, agree to the
// bit; the M terms are summed in canonical order m = 0..M-1 over the un-rotated codes (CodeRegs::adc).
template <int M_T>
__device__ __forceinline__ float range_dist(const CodeRegs<M_T>& cr, const float* T3, int M, float la, float kp,
                                            float t1, float t6, float t5, float radd) {
  const float base = __fadd_rn(__fadd_rn(t1, __fmul_rn(la, t6)), __fmul_rn(__fsub_rn(__fmul_rn(la, la), la), t5));
  return __fadd_rn(__fadd_rn(__fadd_rn(kp, cr.adc(T3, M, 256)), base), radd);
}

static size_t range_smem_bytes(int M, int nL, int W) {
  return sizeof(float) * M * 256 + sizeof(float) * ((nL + 3) & ~3) + sizeof(int64_t) * W +
         sizeof(int) * ((W + 1 + 3) & ~3) + sizeof(float) * 3 * W + sizeof(int) * 2 * R_WARPS;
}

template <int M_T, bool GATHER>
__device__ __forceinline__ void range_query(const RangeArgs& a, int64_t qi) {
  extern __shared__ __align__(16) unsigned char smem[];
  // smem: [T3 M*256 f32][lambda nL f32][per line: start i64, prefix i32 (W+1), t1, t6, t5 f32][warp totals 2 x 8 i32]
  const int M = a.M, W = a.W;
  float* T3 = reinterpret_cast<float*>(smem);
  float* lcb = T3 + M * 256;
  int64_t* lstart = reinterpret_cast<int64_t*>(lcb + ((a.nL + 3) & ~3));
  int* prefix = reinterpret_cast<int*>(lstart + W);
  float* lt1 = reinterpret_cast<float*>(prefix + ((W + 1 + 3) & ~3));
  float* lt6 = lt1 + W;
  float* lt5 = lt6 + W;
  int* wtot = reinterpret_cast<int*>(lt5 + W);

  {
    const float4* src = reinterpret_cast<const float4*>(a.t3 + (size_t)qi * M * 256);
    float4* dst = reinterpret_cast<float4*>(T3);
    for (int i = threadIdx.x; i < M * 64; i += R_THREADS) dst[i] = src[i];
  }
  for (int i = threadIdx.x; i < a.nL; i += R_THREADS) lcb[i] = a.lambda_cb[i];
  for (int w = threadIdx.x; w < W; w += R_THREADS) {  // line descriptors, lengths capped as in the scan
    const int list = a.line_list[qi * W + w];
    int len = 0;
    int64_t st = 0;
    float t5 = 0.f;
    if (list >= 0) {
      st = a.offsets[list];
      const int64_t l = a.offsets[list + 1] - st;
      len = (int)(l < a.cap ? l : a.cap);
      t5 = a.edge_d2 ? a.edge_d2[list] : 0.f;
    }
    lstart[w] = st;
    prefix[w + 1] = len;
    lt1[w] = a.term1[qi * W + w];
    lt6[w] = a.term6[qi * W + w];
    lt5[w] = t5;
  }
  if (threadIdx.x == 0) prefix[0] = 0;
  __syncthreads();
  if (threadIdx.x < kWarp) {  // W <= 1024: one warp scans 32 chunks of the lengths
    const int lane = threadIdx.x;
    const int chunk = (W + kWarp - 1) / kWarp;
    const int b = lane * chunk, e = min(W, b + chunk);
    int s = 0;
    for (int w = b; w < e; w++) s += prefix[w + 1];
    int inc = s;
#pragma unroll
    for (int o = 1; o < kWarp; o <<= 1) {
      const int t = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += t;
    }
    int run = inc - s;
    for (int w = b; w < e; w++) {
      run += prefix[w + 1];
      prefix[w + 1] = run;
    }
  }
  __syncthreads();

  const int total = prefix[W];
  const float radd = a.row_add ? a.row_add[qi] : 0.f;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int count = 0;     // count pass: survivors seen by this thread
  int64_t run = 0;   // gather pass: survivors of the query before this step
  int par = 0;       // gather pass: which half of wtot this step uses
  float* oD = nullptr;
  int64_t* oI = nullptr;
  if (GATHER) {
    const int64_t o = a.lims[qi] - a.lims[a.q0];
    oD = a.outD + o;
    oI = a.outI + o;
  }
  for (int base = 0; base < total; base += R_BATCH * R_THREADS) {
    // stream positions are warp-contiguous: warp w owns [base + 128 w, base + 128 w + 128), lane l the positions
    // +l, +32+l, +64+l, +96+l; output rank order = stream order = (warp, step b, lane)
    const int wpos0 = base + warp * (R_BATCH * kWarp);
    int lo = 0;
    if (wpos0 < total) {  // warp-uniform: largest w with prefix[w] <= wpos0
      int hi = W;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (prefix[mid] <= wpos0) lo = mid; else hi = mid;
      }
    }
    int lo_[R_BATCH], pl_[R_BATCH];
    int64_t ent_[R_BATCH];
#pragma unroll
    for (int b = 0; b < R_BATCH; b++) {
      const int pos = wpos0 + b * kWarp + lane;
      if (pos < total) {
        if (total >= 16 * W) {  // long lists: a step or two forward
          while (lo + 1 < W && prefix[lo + 1] <= pos) lo++;
        } else {  // many short lists per warp: bounded binary search, largest w with prefix[w] <= pos
          int hi = W;
          while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (prefix[mid] <= pos) lo = mid; else hi = mid;
          }
        }
      }
      lo_[b] = lo;
      pl_[b] = pos < total ? pos - prefix[lo] : 0;
      ent_[b] = pos < total ? lstart[lo] + pl_[b] : -1;
    }
    CodeRegs<M_T> cr[R_BATCH];
    uint8_t lq[R_BATCH];
    float kp[R_BATCH];
#pragma unroll
    for (int b = 0; b < R_BATCH; b++) {
      lq[b] = 0;
      kp[b] = 0.f;
      if (ent_[b] >= 0) {
        cr[b].load(a.codes + ent_[b] * M, pl_[b]);
        lq[b] = a.lamq[ent_[b]];
        kp[b] = a.kappa[ent_[b]];
      }
    }
    bool keep[R_BATCH];
    float dist[R_BATCH];
#pragma unroll
    for (int b = 0; b < R_BATCH; b++) {
      keep[b] = false;
      dist[b] = 0.f;
      if (ent_[b] >= 0) {
        const int l = lo_[b];
        dist[b] = range_dist<M_T>(cr[b], T3, M, lcb[lq[b]], kp[b], lt1[l], lt6[l], lt5[l], radd);
        keep[b] = dist[b] < a.radius;
      }
    }
    if (!GATHER) {
#pragma unroll
      for (int b = 0; b < R_BATCH; b++) count += keep[b] ? 1 : 0;
    } else {
      unsigned bal[R_BATCH];
      int mine = 0;
#pragma unroll
      for (int b = 0; b < R_BATCH; b++) {
        bal[b] = __ballot_sync(kFull, keep[b]);
        mine += __popc(bal[b]);
      }
      if (lane == 0) wtot[par * R_WARPS + warp] = mine;
      __syncthreads();  // the other half of wtot was last read before this barrier: one barrier per step suffices
      int before = 0, all = 0;
#pragma unroll
      for (int w = 0; w < R_WARPS; w++) {
        const int t = wtot[par * R_WARPS + w];
        before += w < warp ? t : 0;
        all += t;
      }
      const unsigned lt = (1u << lane) - 1u;
#pragma unroll
      for (int b = 0; b < R_BATCH; b++) {
        if (keep[b]) {
          const int64_t at = run + before + __popc(bal[b] & lt);
          oD[at] = dist[b];
          oI[at] = a.ids[ent_[b]];
        }
        before += __popc(bal[b]);
      }
      run += all;
      par ^= 1;
    }
  }
  if (!GATHER) {
    count = __reduce_add_sync(kFull, count);
    if (lane == 0) wtot[warp] = count;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < R_WARPS; w++) s += wtot[w];
      a.counts[qi] = s;
      if (qi == 0) a.counts[a.nq] = 0;  // the exclusive scan leaves the total here
    }
  }
}

template <int M_T>
__global__ void __launch_bounds__(R_THREADS) range_count_kernel(RangeArgs a) {
  range_query<M_T, false>(a, blockIdx.x);
}

template <int M_T>
__global__ void __launch_bounds__(R_THREADS) range_gather_kernel(RangeArgs a) {
  range_query<M_T, true>(a, a.q0 + blockIdx.x);
}

template <int M_T>
static int launch_range(bool gather, const RangeArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  if (gather) {
    VLQ_CUDA_TRY(cudaFuncSetAttribute(range_gather_kernel<M_T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VLQ_LAUNCH(range_gather_kernel<M_T>, grid, R_THREADS, smem, st, a);
  } else {
    VLQ_CUDA_TRY(cudaFuncSetAttribute(range_count_kernel<M_T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VLQ_LAUNCH(range_count_kernel<M_T>, grid, R_THREADS, smem, st, a);
  }
  return last_error();
}

// 16-byte (M = 16) / 8-byte (M = 8) code loads need an aligned slab; other M load bytes
static int dispatch_range(bool gather, const RangeArgs& a, unsigned grid, cudaStream_t st) {
  const size_t smem = range_smem_bytes(a.M, a.nL, a.W);
  const bool al16 = (reinterpret_cast<uintptr_t>(a.codes) & 15) == 0;
  if (a.M == 16 && al16) return launch_range<16>(gather, a, grid, smem, st);
  if (a.M == 8 && al16) return launch_range<8>(gather, a, grid, smem, st);
  return launch_range<0>(gather, a, grid, smem, st);
}

// the term-3 tables of the 8-bit codebook (M, 256, dsub) or the pair tables of the 4-bit one (M, 16, dsub)
static TableBuild range_tables(bool pq4, int d, int M) {
  return pq4 ? TableBuild{launch_pair_tables, true, true} : TableBuild{launch_term3, term3_supported(d, M), true};
}

// the checks both passes share; VLQ_OK with a.nq == 0 means "nothing to launch".  M is the number of sub-quantizers;
// a.M the number of code bytes per entry (M / 2 for 4-bit codes)
static int range_args(RangeArgs& a, bool pq4, const float* q, int64_t nq, int d, const float* pq, int M,
                      const float* lambda_cb, int nL, const int* line_list, const float* term1, const float* term6,
                      const float* edge_d2, int W, const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq,
                      const float* kappa, int cap, const float* row_add, float radius, const void* workspace,
                      size_t workspace_bytes) {
  const bool shape_ok = pq4 ? pq4_shape_ok(d, M) && d <= 256 : d > 0 && M > 0 && M <= 64 && d % M == 0;
  if (nq < 0 || !shape_ok || nL <= 0 || nL > 256 || W <= 0 || W > VLQ_MAX_K ||
      cap <= 0 || cap > (1 << 20) || (int64_t)W * cap > (int64_t)0x7fffffff || std::isnan(radius))
    return VLQ_EINVAL;
  const int Mb = pq4 ? M / 2 : M;
  a = RangeArgs{};
  a.nq = nq;
  if (nq == 0) return VLQ_OK;
  if (!q || !pq || !lambda_cb || !line_list || !term1 || !term6 || !offsets || !codes || !lamq || !kappa || !workspace)
    return VLQ_EINVAL;
  if ((reinterpret_cast<uintptr_t>(pq) | reinterpret_cast<uintptr_t>(workspace)) & 15) return VLQ_EINVAL;
  if (!range_tables(pq4, d, M).supported) return VLQ_EUNSUPPORTED;
  if (workspace_bytes < vlq_range_workspace_bytes(nq, Mb, W, cap)) return VLQ_EWORKSPACE;
  a.t3 = static_cast<const float*>(workspace);
  a.M = Mb; a.nL = nL; a.lambda_cb = lambda_cb; a.line_list = line_list; a.term1 = term1; a.term6 = term6;
  a.edge_d2 = edge_d2; a.W = W; a.cap = cap; a.offsets = offsets; a.codes = codes; a.lamq = lamq; a.kappa = kappa;
  a.row_add = row_add; a.radius = radius;
  return VLQ_OK;
}

}  // namespace vlq

using namespace vlq;

extern "C" {

// the term-3 tables of the batch; W and cap do not enter it
size_t vlq_range_workspace_bytes(int64_t nq, int M, int /*W*/, int /*cap*/) {
  const size_t n = nq > 0 ? (size_t)nq : 0, m = M > 0 ? (size_t)M : 0;
  return (n * m * 256 * sizeof(float) + 255) & ~size_t(255);
}

}  // extern "C"

// both passes of both codebooks: pq4 selects the table build and the code width, nothing else differs
static int range_count(bool pq4, const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb,
                       int nL, const int* line_list, const float* term1, const float* term6, const float* edge_d2,
                       int W, const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa,
                       int cap, const float* row_add, float radius, int64_t* out_lims, void* workspace,
                       size_t workspace_bytes, vlq_stream_t stream) {
  if (!out_lims) return VLQ_EINVAL;
  RangeArgs a;
  const int rc = range_args(a, pq4, q, nq, d, pq, M, lambda_cb, nL, line_list, term1, term6, edge_d2, W, offsets, codes,
                            lamq, kappa, cap, row_add, radius, workspace, workspace_bytes);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  if (nq == 0) {
    VLQ_CUDA_TRY(cudaMemsetAsync(out_lims, 0, sizeof(int64_t), st));
    return VLQ_OK;
  }
  int r = range_tables(pq4, d, M).launch(q, nq, d, pq, a.M, static_cast<float*>(workspace), false, st);
  if (r) return r;
  a.counts = out_lims;
  r = dispatch_range(false, a, (unsigned)nq, st);
  if (r) return r;
  return launch_exclusive_scan_i64(out_lims, nq + 1, st);
}

static int range_gather(bool pq4, const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb,
                        int nL, const int* line_list, const float* term1, const float* term6, const float* edge_d2,
                        int W, const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa,
                        int cap, const float* row_add, float radius, const int64_t* ids, const int64_t* lims,
                        int64_t q0, int64_t q1, float* outD, int64_t* outI, const void* workspace,
                        size_t workspace_bytes, vlq_stream_t stream) {
  RangeArgs a;
  const int rc = range_args(a, pq4, q, nq, d, pq, M, lambda_cb, nL, line_list, term1, term6, edge_d2, W, offsets, codes,
                            lamq, kappa, cap, row_add, radius, workspace, workspace_bytes);
  if (rc) return rc;
  if (q0 < 0 || q1 < q0 || q1 > nq) return VLQ_EINVAL;
  if (q1 == q0) return VLQ_OK;
  if (!ids || !lims || !outD || !outI) return VLQ_EINVAL;
  a.ids = ids;
  a.lims = lims;
  a.q0 = q0;
  a.outD = outD;
  a.outI = outI;
  return dispatch_range(true, a, (unsigned)(q1 - q0), as_stream(stream));
}

extern "C" {

#define VLQ_RANGE_COUNT_ARGS                                                                                          \
  q, nq, d, pq, M, lambda_cb, nL, line_list, term1, term6, edge_d2, W, offsets, codes, lamq, kappa, cap, row_add,    \
      radius, out_lims, workspace, workspace_bytes, stream
#define VLQ_RANGE_GATHER_ARGS                                                                                         \
  q, nq, d, pq, M, lambda_cb, nL, line_list, term1, term6, edge_d2, W, offsets, codes, lamq, kappa, cap, row_add,    \
      radius, ids, lims, q0, q1, outD, outI, workspace, workspace_bytes, stream

int vlq_range_count(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                    const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                    const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa, int cap,
                    const float* row_add, float radius, int64_t* out_lims, void* workspace, size_t workspace_bytes,
                    vlq_stream_t stream) {
  return range_count(false, VLQ_RANGE_COUNT_ARGS);
}

int vlq_range_count_pq4(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                        const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                        const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa, int cap,
                        const float* row_add, float radius, int64_t* out_lims, void* workspace, size_t workspace_bytes,
                        vlq_stream_t stream) {
  return range_count(true, VLQ_RANGE_COUNT_ARGS);
}

int vlq_range_gather(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                     const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                     const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa, int cap,
                     const float* row_add, float radius, const int64_t* ids, const int64_t* lims, int64_t q0, int64_t q1,
                     float* outD, int64_t* outI, const void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  return range_gather(false, VLQ_RANGE_GATHER_ARGS);
}

int vlq_range_gather_pq4(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                         const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                         const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa, int cap,
                         const float* row_add, float radius, const int64_t* ids, const int64_t* lims, int64_t q0,
                         int64_t q1, float* outD, int64_t* outI, const void* workspace, size_t workspace_bytes,
                         vlq_stream_t stream) {
  return range_gather(true, VLQ_RANGE_GATHER_ARGS);
}

#undef VLQ_RANGE_COUNT_ARGS
#undef VLQ_RANGE_GATHER_ARGS

}  // extern "C"
