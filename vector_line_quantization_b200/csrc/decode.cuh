// Decode of stored entries, shared by the read-back kernels (lists.cu) and the refinement stage (refine.cu): one
// definition of the first-level reconstruction x1 of a VLQ entry, so that the residual a refinement code encodes and
// the value the re-rank and reconstruct add it to are the same bits.
#pragma once
#include "common.cuh"
#include "pq4.cuh"

namespace vlq {

// largest l in [lo, hi] with offsets[l] <= p (offsets[lo] <= p)
__device__ __forceinline__ int64_t list_of(const int64_t* offsets, int64_t lo, int64_t hi, int64_t p) {
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (offsets[mid] <= p) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// list_of(offsets, 0, nlists - 1, p) by one warp (all lanes, same p, offsets[0] <= p): a 32-way search, so about
// log32(nlists) dependent loads instead of log2(nlists) (5 instead of 21 at 2^21 lists)
__device__ __forceinline__ int64_t list_of_warp(const int64_t* offsets, int64_t nlists, int64_t p) {
  const int lane = threadIdx.x % kWarp;
  int64_t lo = 0, hi = nlists - 1;  // offsets[lo] <= p; the answer is in [lo, hi]
  while (lo < hi) {
    const int64_t step = (hi - lo + kWarp) / kWarp;  // ceil((hi - lo + 1) / 32)
    const int64_t l = lo + lane * step;
    const unsigned le = __ballot_sync(kFull, l <= hi && offsets[l] <= p);
    const int i = 31 - __clz(le);  // lane 0 always holds
    lo += i * step;
    hi = min(hi, lo + step - 1);
  }
  return lo;
}

// pq[m][code_m][j - m dsub], m = j / dsub, of an 8-bit PQ code whose bytes are stored rotated by rot
// (stored[(m - rot) mod M] = code[m]; rot = 0 for canonical, arrival-order codes)
__device__ __forceinline__ float pq_component(const float* __restrict__ pq, const uint8_t* cw, int M, int dsub, int rot,
                                              int j) {
  const int m = j / dsub;
  int sb = m - rot;
  if (sb < 0) sb += M;
  return pq[((int64_t)m * 256 + cw[sb]) * dsub + (j - m * dsub)];
}

// the same for a packed 4-bit code (pq4.cuh): pq is (M, 16, dsub), the Mb = M / 2 stored bytes are rotated by rot
// (stored[(b - rot) mod Mb] = packed[b]), code m is nibble m & 1 of packed byte m / 2
__device__ __forceinline__ float pq4_component(const float* __restrict__ pq, const uint8_t* cw, int M, int dsub, int rot,
                                               int j) {
  const int m = j / dsub, Mb = M / 2;
  int sb = (m >> 1) - rot;
  if (sb < 0) sb += Mb;
  const int code = (cw[sb] >> ((m & 1) * 4)) & 15;
  return pq[((int64_t)m * kPq4Ksub + code) * dsub + (j - m * dsub)];
}

// x1[j] = ((1 - lh) c[j] + lh s[j]) + pq[m][code_m][j - m dsub]: fp32, each operation rounded as written (no fma
// contraction), oml = 1 - lh rounded; lh = 0 gives exactly c + p (IndexIVFPQ's decode).  pq4: cw is a packed 4-bit code
// of M / 2 bytes and rot is taken mod M / 2.
__device__ __forceinline__ float vlq_decode_component(const float* c, const float* s, float lh, float oml,
                                                      const float* __restrict__ pq, const uint8_t* cw, int M, int dsub,
                                                      int rot, int j, bool pq4 = false) {
  const float a = __fadd_rn(__fmul_rn(oml, c[j]), __fmul_rn(lh, s[j]));
  return __fadd_rn(a, pq4 ? pq4_component(pq, cw, M, dsub, rot, j) : pq_component(pq, cw, M, dsub, rot, j));
}

}  // namespace vlq
