// Declarations shared by the scan kernels (search.cu: block-synchronous and warp-autonomous scans; scan_long.cu: the
// long-list scan for 1B-scale list densities; range.cu: the radius scan).
#pragma once
#include "common.cuh"

namespace vlq {

struct ScanArgs {
  const float* q;
  int d;
  const float* pq;
  int M, ksub, dsub;
  const float* lambda_cb;
  int nL;
  const int* line_list;
  const float* term1;
  const float* term6;
  const float* edge_d2;
  int W;
  const int64_t* offsets;
  const uint8_t* codes;
  const uint8_t* lamq;
  const float* kappa;
  const int64_t* ids;
  int k, cap;
  int sel_cap;
  int owner_cap;    // stream positions covered by the shared-memory owner table (0 = always binary search)
  const int* qlist; // scan_topk_kernel: nullptr = query blockIdx.x; else {n, q_0 .. q_n-1}: CTA j < n scans q_j
  const float* t3;  // optional precomputed term-3 tables [nq][M*ksub] (term3_kernel); nullptr = build in the kernel
  float* outD;
  int64_t* outI;
};

// ---- code-byte rotation of the stored lists -------------------------------------------------------------------------
// The inverted lists store the M code bytes of the entry at list position `pos` rotated by pos mod M:
//     stored[j] = code[(j + pos) mod M]
// so that in the bank-skewed scans, where lane l works on sub-quantizer (s + l) mod M at step s and lane l handles the
// entries with pos mod M == l mod M, byte s of the stored word IS the byte the lane needs at step s: no per-entry
// rotation in the inner loop (it used to cost 12 of ~145 instructions per entry).  vlq_build_lists applies the
// rotation; every reader that needs canonical order (the other scan kernels, vlq_recompute_kappa, the host accessors
// and the .dbcodes writer) undoes it with rot = (M - pos mod M) mod M.
__device__ __forceinline__ void rot16(uint32_t (&w)[4], int r) {  // out[j] = in[(j + r) & 15], r in [0, 16)
  uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
  if (r & 4) { const uint32_t t = w0; w0 = w1; w1 = w2; w2 = w3; w3 = t; }
  if (r & 8) { uint32_t t = w0; w0 = w2; w2 = t; t = w1; w1 = w3; w3 = t; }
  const uint32_t selb = 0x3210u + 0x1111u * (uint32_t)(r & 3);
  w[0] = __byte_perm(w0, w1, selb);
  w[1] = __byte_perm(w1, w2, selb);
  w[2] = __byte_perm(w2, w3, selb);
  w[3] = __byte_perm(w3, w0, selb);
}
__device__ __forceinline__ void rot8(uint32_t (&w)[2], int r) {  // out[j] = in[(j + r) & 7], r in [0, 8)
  uint32_t w0 = w[0], w1 = w[1];
  if (r & 4) { const uint32_t t = w0; w0 = w1; w1 = t; }
  const uint32_t selb = 0x3210u + 0x1111u * (uint32_t)(r & 3);
  w[0] = __byte_perm(w0, w1, selb);
  w[1] = __byte_perm(w1, w0, selb);
}

// PQ codes of one entry held in registers (16-byte / 8-byte vector loads for M = 16 / 8; byte loads otherwise)
// `pos` = position of the entry inside its list: the stored bytes are rotated by pos mod M (above) and adc() sums the
// sub-quantizers in canonical order m = 0..M-1, the order of the reference and of the oracle.
template <int M_T>
struct CodeRegs {
  uint32_t w[M_T == 16 ? 4 : (M_T == 8 ? 2 : 1)];
  const uint8_t* ptr;
  int rot;
  __device__ __forceinline__ void load(const uint8_t* __restrict__ code_ptr, int pos) {
    if constexpr (M_T == 16) {
      const uint4 c = ld_nc_v4(code_ptr);
      w[0] = c.x; w[1] = c.y; w[2] = c.z; w[3] = c.w;
      rot = (16 - (pos & 15)) & 15;
    } else if constexpr (M_T == 8) {
      const uint2 c = ld_nc_v2(code_ptr);
      w[0] = c.x; w[1] = c.y;
      rot = (8 - (pos & 7)) & 7;
    } else {
      ptr = code_ptr;
      rot = pos;
    }
  }
  __device__ __forceinline__ float adc(const float* __restrict__ T3, int M, int ksub) const {
    float acc = 0.f;
    if constexpr (M_T == 16) {
      uint32_t r[4] = {w[0], w[1], w[2], w[3]};
      rot16(r, rot);
#pragma unroll
      for (int t = 0; t < 4; t++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc += T3[(t * 4 + b) * 256 + ((r[t] >> (8 * b)) & 0xff)];
    } else if constexpr (M_T == 8) {
      uint32_t r[2] = {w[0], w[1]};
      rot8(r, rot);
#pragma unroll
      for (int t = 0; t < 2; t++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc += T3[(t * 4 + b) * 256 + ((r[t] >> (8 * b)) & 0xff)];
    } else {
      int j = (M - rot % M) % M;  // stored[j] = code[(j + pos) mod M]  =>  code[m] = stored[(m - pos) mod M]
      for (int m = 0; m < M; m++) {
        acc += T3[m * ksub + ptr[j]];
        j = j + 1 == M ? 0 : j + 1;
      }
    }
    return acc;
  }
};

// Long-list scan with TMA bulk prefetch into L2 (scan_long.cu): one CTA per query, four entries per lane.  Returns
// VLQ_EUNSUPPORTED when the configuration does not fit (the caller then uses the kernels of search.cu).
int launch_scan_long(const ScanArgs& a, int64_t nq, cudaStream_t st);
bool scan_long_supported(const ScanArgs& a);

// term-3 tables T3[q][m][j] = -2 q_m . p_mj of a batch of queries into t3 (search.cu: term3_reg_kernel for the two
// production shapes, term3_kernel otherwise; code_major = the [j][M] rows of the bank-skewed scans).  term3_supported:
// the shapes those kernels take (d % 4 == 0, the PQ codebook fits their shared memory); pq and t3 16-byte aligned.
bool term3_supported(int d, int M);
int launch_term3(const float* q, int64_t nq, int d, const float* pq, int M, float* t3, bool code_major, cudaStream_t st);
// the same tables for a 4-bit codebook (M = 2 Mb, 16, dsub): the Mb pair tables of pq4.cuh in either layout, so the scans
// run unmodified with M = Mb.  Any pq4_shape_ok shape with d <= 256; t3 16-byte aligned.
int launch_pair_tables(const float* q, int64_t nq, int d, const float* pq, int Mb, float* t3, bool code_major,
                       cudaStream_t st);
// how a scan or range entry point gets its term-3 tables: the 8-bit kernels above, or the pair tables (`required`: there
// is no in-kernel table build for that codebook, so the workspace must hold the tables)
struct TableBuild {
  int (*launch)(const float* q, int64_t nq, int d, const float* pq, int M, float* t3, bool code_major, cudaStream_t st);
  bool supported;
  bool required;
};

// in-place exclusive scan of n int64 values by one block (lists.cu)
int launch_exclusive_scan_i64(int64_t* v, int64_t n, cudaStream_t st);

}  // namespace vlq
