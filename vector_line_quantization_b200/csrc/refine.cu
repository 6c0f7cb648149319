// Refinement stage of GpuIndexIVFPQR (faiss IndexIVFPQR): a second 8-bit PQ code of the residual left by the first
// level, and the re-rank of a search's candidates by the two-level reconstruction.
//   x1 = anchor + p(code)          the first-level decode (decode.cuh, the same function as vlq_decode_entries)
//   r2 = x - x1                    one fp32 subtraction per component
//   code2[m] = argmin_j ||r2_m - pq2[m][j]||^2, lowest j on ties
//   x2 = x1 + pq2[m][code2_m]      one fp32 add per component (vlq_refine_decode)
// The re-rank distance is the full squared L2 ||q - x2||^2 (faiss IndexIVFPQR::search computes it with fvec_L2sqr).
#include <cfloat>
#include <climits>

#include "decode.cuh"
#include "topk.cuh"

namespace vlq {

constexpr int REF_THREADS = 256;
constexpr int REF_WARPS = REF_THREADS / kWarp;
constexpr int REF_MAX_D = 512;  // shared memory per warp (encode) / per CTA (re-rank) holds one row

// Encode: one warp per row.  The lanes decode x1 and write r2 into the warp's shared row, then each sub-quantizer's 256
// centroids are split over the lanes (lane l: j = l, l + 32, ...; ascending, so a strict < keeps the lowest j) and the
// (distance, j) minimum is taken over the warp.
__global__ void __launch_bounds__(REF_THREADS)
refine_encode_kernel(const float* __restrict__ x, int64_t n, int d, const int* __restrict__ list,
                     const uint8_t* __restrict__ lamq, const uint8_t* __restrict__ codes, int M,
                     const float* __restrict__ pq, const float* __restrict__ cent, const int* __restrict__ edge, int E,
                     const float* __restrict__ lambda_cb, const float* __restrict__ pq2, int M2,
                     uint8_t* __restrict__ out_code2, float* __restrict__ out_r2) {
  extern __shared__ float sres[];  // [REF_WARPS][d]
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  float* r = sres + warp * d;
  const int dsub = d / M;
  const int64_t nwarps = (int64_t)gridDim.x * REF_WARPS;
  for (int64_t i = (int64_t)blockIdx.x * REF_WARPS + warp; i < n; i += nwarps) {
    const int l = list[i];
    if (l < 0) {  // skipped row (NaN input): nothing of it is read
      if (out_r2)
        for (int j = lane; j < d; j += kWarp) out_r2[i * d + j] = 0.f;
      if (pq2)
        for (int m = lane; m < M2; m += kWarp) out_code2[i * M2 + m] = 0;
      continue;
    }
    const float* c = cent + (int64_t)(l / E) * d;
    const float* s = cent + (int64_t)edge[l] * d;
    const float lh = lambda_cb[lamq[i]];
    const float oml = __fsub_rn(1.f, lh);
    const uint8_t* cw = codes + i * M;
    for (int j = lane; j < d; j += kWarp) {
      const float rj = __fsub_rn(x[i * d + j], vlq_decode_component(c, s, lh, oml, pq, cw, M, dsub, 0, j));
      r[j] = rj;
      if (out_r2) out_r2[i * d + j] = rj;
    }
    __syncwarp();
    if (pq2) {
      const int dsub2 = d / M2;
      for (int m = 0; m < M2; m++) {
        const float* rm = r + m * dsub2;
        float best = __int_as_float(0x7f800000);
        int bj = lane;
        for (int j = lane; j < 256; j += kWarp) {
          const float* cj = pq2 + ((int64_t)m * 256 + j) * dsub2;
          float acc = 0.f;
          for (int u = 0; u < dsub2; u++) {
            const float t = rm[u] - cj[u];
            acc = fmaf(t, t, acc);
          }
          if (acc < best) {
            best = acc;
            bj = j;
          }
        }
        const uint64_t key = warp_min_u64(make_key(best, (uint32_t)bj));
        if (lane == 0) out_code2[i * M2 + m] = (uint8_t)key_payload(key);
      }
    }
    __syncwarp();  // the next row overwrites r
  }
}

// Re-rank: one CTA per query, the query row in shared memory.  Warp w evaluates candidates w, w + 8, ...: x2 of the
// candidate's slab entry, component by component (lane j: j, j + 32, ...), and ||q - x2||^2 reduced over the warp in
// fp32.  Key = (distance, candidate index), so ties keep candidate order; a hole (-1, or outside the slab) or a NaN
// distance gets the unique key (0xffffffff, index), above every real distance.  BlockSelect (topk.cuh) keeps the k
// smallest of the kc keys placed directly, sorted.  cand is read before outD / outI are written, so outI may alias cand
// when k == kc.
__global__ void __launch_bounds__(REF_THREADS)
refine_topk_kernel(const float* __restrict__ q, int d, const int64_t* __restrict__ cand, int kc, int k, int cap,
                   int64_t nlists, const int64_t* __restrict__ offsets, const uint8_t* __restrict__ codes,
                   const uint8_t* __restrict__ lamq, const int64_t* __restrict__ ids, const uint8_t* __restrict__ code2,
                   int M, const float* __restrict__ pq, const float* __restrict__ cent, const int* __restrict__ edge, int E,
                   const float* __restrict__ lambda_cb, const float* __restrict__ pq2, int M2, float* __restrict__ outD,
                   int64_t* __restrict__ outI) {
  extern __shared__ __align__(16) unsigned char smem[];
  float* sq = reinterpret_cast<float*>(smem + select_smem_bytes(cap));
  const int64_t qi = blockIdx.x;
  for (int j = threadIdx.x; j < d; j += REF_THREADS) sq[j] = q[qi * d + j];
  BlockSelect<REF_THREADS> sel;
  sel.init(smem, k, cap, 1);  // syncs the block: sq is complete
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  const int dsub = d / M, dsub2 = d / M2;
  const int64_t nslab = offsets[nlists];
  const int64_t* cq = cand + qi * kc;
  for (int ci = warp; ci < kc; ci += REF_WARPS) {
    const int64_t p = cq[ci];
    uint64_t key = (0xffffffffull << 32) | (uint32_t)ci;
    if (p >= 0 && p < nslab) {
      const int64_t l = list_of_warp(offsets, nlists, p);
      const int rot = (int)((p - offsets[l]) % M);
      const float* c = cent + (l / E) * d;
      const float* s = cent + (int64_t)edge[l] * d;
      const float lh = lambda_cb[lamq[p]];
      const float oml = __fsub_rn(1.f, lh);
      const uint8_t* cw = codes + p * M;
      const uint8_t* c2 = code2 + p * M2;
      float acc = 0.f;
      for (int j = lane; j < d; j += kWarp) {
        const float x2 = __fadd_rn(vlq_decode_component(c, s, lh, oml, pq, cw, M, dsub, rot, j),
                                   pq_component(pq2, c2, M2, dsub2, 0, j));
        const float t = __fsub_rn(sq[j], x2);
        acc = fmaf(t, t, acc);
      }
      const float dist = warp_sum(acc);
      if (dist == dist) key = make_key(dist, (uint32_t)ci);
    }
    if (lane == 0) sel.keys[ci] = key;
  }
  sel.placed(kc, false);
  sel.finish();
  // every read of cand before the first write: outI may alias cand when k == kc (the scan's slab indexes re-ranked in
  // place); k <= VLQ_MAX_K = 4 * REF_THREADS
  float dv[VLQ_MAX_K / REF_THREADS];
  int64_t lab[VLQ_MAX_K / REF_THREADS];
#pragma unroll
  for (int t = 0; t < VLQ_MAX_K / REF_THREADS; t++) {
    const int i = threadIdx.x + t * REF_THREADS;
    dv[t] = FLT_MAX;
    lab[t] = -1;
    const uint64_t key = i < k ? sel.keys[i] : kKeyInf;
    if ((key >> 32) != 0xffffffffull) {
      const int64_t p = cq[key_payload(key)];
      dv[t] = key_val(key);
      lab[t] = ids ? ids[p] : p;
    }
  }
  __syncthreads();
#pragma unroll
  for (int t = 0; t < VLQ_MAX_K / REF_THREADS; t++) {
    const int i = threadIdx.x + t * REF_THREADS;
    if (i < k) {
      outD[qi * k + i] = dv[t];
      outI[qi * k + i] = lab[t];
    }
  }
}

static bool refine_tables_ok(int d, int M, int E, int nL, int M2) {
  return d >= 1 && M >= 1 && M <= 64 && d % M == 0 && E >= 1 && nL >= 1 && nL <= 256 && M2 >= 1 && M2 <= 64 &&
         d % M2 == 0;
}

}  // namespace vlq

using namespace vlq;

extern "C" int vlq_refine_encode(const float* x, int64_t n, int d, const int* list, const uint8_t* lamq,
                                 const uint8_t* codes, int M, const float* pq, const float* cent, const int* edge, int E,
                                 const float* lambda_cb, int nL, const float* pq2, int M2, uint8_t* out_code2,
                                 float* out_r2, vlq_stream_t stream) {
  if (n < 0 || d < 1 || M < 1 || M > 64 || d % M != 0 || E < 1 || nL < 1 || nL > 256) return VLQ_EINVAL;
  if (pq2 && (M2 < 1 || M2 > 64 || d % M2 != 0 || !out_code2)) return VLQ_EINVAL;
  if (!pq2 && !out_r2) return VLQ_EINVAL;  // nothing to write
  if (d > REF_MAX_D) return VLQ_EUNSUPPORTED;
  if (n == 0) return VLQ_OK;
  if (!x || !list || !lamq || !codes || !pq || !cent || !edge || !lambda_cb) return VLQ_EINVAL;
  const int64_t g = div_up(n, REF_WARPS);
  const unsigned grid = (unsigned)(g < 148 * 16 ? g : 148 * 16);
  VLQ_LAUNCH(refine_encode_kernel, grid, REF_THREADS, sizeof(float) * REF_WARPS * d, as_stream(stream), x, n, d, list,
             lamq, codes, M, pq, cent, edge, E, lambda_cb, pq2, pq2 ? M2 : 1, out_code2, out_r2);
  return last_error();
}

extern "C" int vlq_refine_topk(const float* q, int64_t nq, int d, const int64_t* cand, int kc, int k, int64_t nlists,
                               const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const int64_t* ids,
                               const uint8_t* code2, int M, const float* pq, const float* cent, const int* edge, int E,
                               const float* lambda_cb, int nL, const float* pq2, int M2, float* outD, int64_t* outI,
                               vlq_stream_t stream) {
  if (nq < 0 || nq > INT_MAX || kc < 1 || kc > VLQ_MAX_K || k < 1 || k > kc || nlists < 1) return VLQ_EINVAL;
  if (!refine_tables_ok(d, M, E, nL, M2) || nlists % E != 0) return VLQ_EINVAL;
  if (d > REF_MAX_D) return VLQ_EUNSUPPORTED;
  if (nq == 0) return VLQ_OK;
  if (!q || !cand || !offsets || !pq || !cent || !edge || !lambda_cb || !pq2 || !outD || !outI) return VLQ_EINVAL;
  const int cap = select_capacity(k, REF_THREADS, 1, kc);
  const size_t smem = select_smem_bytes(cap) + sizeof(float) * d;
  VLQ_LAUNCH(refine_topk_kernel, (unsigned)nq, REF_THREADS, smem, as_stream(stream), q, d, cand, kc, k, cap, nlists,
             offsets, codes, lamq, ids, code2, M, pq, cent, edge, E, lambda_cb, pq2, M2, outD, outI);
  return last_error();
}
