// The stored format of 4-bit PQ codes, shared by the device code (encode, pair tables, decode, kappa) and the host layer
// (host/GpuIndexIVFPQ.cpp packs and unpacks the one-byte-per-code formats of its accessors and files).
//
// An entry of M 4-bit codes is stored in Mb = M / 2 bytes (M even):
//     byte j = code[2j] | code[2j + 1] << 4                       (faiss's low-nibble-first order)
// The packed word of Mb bytes is handled like an 8-bit code of Mb sub-quantizers by every list routine, rotation by
// pos mod Mb included (scan.cuh).  The scans see it through pair tables of 256 entries per stored byte:
//     T3'[m'][b] = T3[2m'][b & 15] + T3[2m' + 1][b >> 4]          (one fp32 add)
// so their per-entry work and bytes are those of an 8-bit index with Mb sub-quantizers.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define VLQ_PQ4_HD __host__ __device__ __forceinline__
#else
#define VLQ_PQ4_HD inline
#endif

namespace vlq {

constexpr int kPq4Ksub = 16;

// the M 4-bit codes a 4-bit index accepts: even, 2 .. 64, dividing d
VLQ_PQ4_HD bool pq4_shape_ok(int d, int M) { return M >= 2 && M <= 64 && M % 2 == 0 && d > 0 && d % M == 0; }

VLQ_PQ4_HD uint8_t pq4_pack_byte(uint8_t lo, uint8_t hi) { return (uint8_t)((lo & 15) | (hi << 4)); }

// code m of a packed word (canonical byte order)
VLQ_PQ4_HD int pq4_code(const uint8_t* packed, int m) { return (packed[m >> 1] >> ((m & 1) * 4)) & 15; }

// one-byte-per-code rows [n][M] <-> packed rows [n][M / 2]
inline void pq4_pack(const uint8_t* codes, int64_t n, int M, uint8_t* packed) {
  for (int64_t i = 0; i < n * (M / 2); i++) packed[i] = pq4_pack_byte(codes[2 * i], codes[2 * i + 1]);
}
inline void pq4_unpack(const uint8_t* packed, int64_t n, int M, uint8_t* codes) {
  for (int64_t i = 0; i < n * (M / 2); i++) {
    codes[2 * i] = packed[i] & 15;
    codes[2 * i + 1] = packed[i] >> 4;
  }
}

}  // namespace vlq
