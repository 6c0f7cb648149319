// Coarse assignment on the 5th-generation tensor cores (SURVEY.md 8a rows a2 / a11, north_star item 1).
//
//   D[i][j] = ||c_j||^2 - 2 x_i . c_j        i < n vectors,  j < C centroids,  K = d
//
// fp32-grade result from fp16 tensor-core passes: every operand is split x = x_hi + x_lo (two fp16 numbers, 22 bits of
// mantissa together, after an exact power-of-two pre-scale that keeps both parts in fp16's normal range) and the
// product is accumulated in fp32 TMEM as   x_hi.c_hi + x_hi.c_lo + x_lo.c_hi    (the dropped x_lo.c_lo term is
// 2^-22 relative).  Three tcgen05.mma passes into the same accumulator; the error is at the level of an fp32 GEMM with
// a different summation order, which is what north_star's "identical except near-ties < 1e-5" allows.
//
// Kernel (one CTA per SM, persistent over work items = 256-row block x centroid split):
//   warp 0    producer : cp.async.bulk (TMA engine, SASS UBLKCP) of pre-packed operand tiles, mbarrier complete_tx
//   warp 1    MMA issuer (one elected lane): tcgen05.mma.cta_group::1.kind::f16, M=128 x N=128 x K=16, SMEM descriptors
//             on the no-swizzle K-major canonical layout the pack kernel writes; tcgen05.commit releases stages
//   warps 2-9 epilogue : fused per-row arg-min (tcgen05.ld 32x32b.x32, one accumulator row per thread), or bucket minima
//             only, or the D tile of the query path (tcgen05.ld 16x256b fragments, lane-pair exchange, 64-byte row
//             stores straight from registers); TMEM accumulators are double buffered so the epilogue of centroid tile
//             t overlaps the MMAs of tile t+1
//   A (the 256 x d block of vectors, hi+lo) stays resident in SMEM for the whole centroid sweep; B (128 centroids x 32 K,
//   hi+lo = 16 KiB) streams through a 3-stage ring (4 stages: no change).  256 rows per CTA halve the L2->SM operand traffic per vector
//   compared with one 128-row tile (the sweep is otherwise L2-bandwidth bound at ~42 B/clk/SM).
//
// Packed operand layout (written by pack_rows_kernel; shared by A and B):
//   [tile = row/128][part: hi,lo][kb = k/32][rg = (row%128)/8][kg = (k%32)/8][r8 = row%8][8 x fp16]
//   i.e. 8x8 "core matrices" of 128 contiguous bytes; LBO (next core matrix along K) = 128 B, SBO (next 8 rows) = 512 B.
#include <cuda_fp16.h>

#include <cfloat>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace vlq {
namespace tc {

constexpr int TILE_ROWS = 128;               // UMMA M and N
constexpr int KB = 32;                       // K elements per pipeline stage
constexpr int TILE_KB_BYTES = TILE_ROWS * KB * 2;  // 8 KiB: one (tile, part, kb) block
constexpr int STAGES = 3;
constexpr int ROW_TILES = 2;                 // 256 rows per CTA
constexpr int ACC_BUFS = 2;
constexpr int TMEM_COLS = ROW_TILES * ACC_BUFS * TILE_ROWS;  // 512
constexpr int EPI_WARPS = 8;                 // 2 warps per TMEM lane group: each takes one half of the 128 columns
constexpr int THREADS = 64 + EPI_WARPS * 32; // producer warp + MMA warp + epilogue warps
constexpr int MAX_D = 128;

__host__ __device__ inline int64_t packed_bytes(int64_t rows, int d) {
  int64_t tiles = (rows + TILE_ROWS - 1) / TILE_ROWS;
  return tiles * 2 * (d / KB) * TILE_KB_BYTES;
}

// ------------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(addr), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 16 TMEM lanes x 64 columns: thread t, register 4 j + i <- lane t / 4 + 8 (i / 2), column 8 j + 2 (t % 4) + (i % 2)
// (the m16n8 accumulator fragment repeated over 8 column blocks; layout verified on the device with a tcgen05.st.32x32b
// fill).  A quad of threads holds 8 consecutive floats of a row.
__device__ __forceinline__ void tmem_ld16x64(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x8.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// SMEM matrix descriptor, K-major, SWIZZLE_NONE (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4, [32,46) stride byte offset >> 4, [46,48) version = 1,
//   [61,64) layout type = 0
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  constexpr uint64_t LBO = 128 >> 4, SBO = 512 >> 4;
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (LBO << 16) | (SBO << 32) | (1ull << 46);
}
// Instruction descriptor for kind::f16 (cute::UMMA::InstrDescriptor): c_format F32 = 1 @4, a/b format F16 = 0 @7/@10,
// a/b major K = 0 @15/@16, N>>3 @17, M>>4 @24
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(TILE_ROWS >> 3) << 17) | ((uint32_t)(TILE_ROWS >> 4) << 24);

// ------------------------------------------------------------------------------------------------------ pack kernel
// fp32 [rows][d] -> packed fp16 hi/lo tiles.  Rows in [rows, rows_padded) are written as zeros.
// Scaling (always a power of two, hence exact):
//   * centroids (row_inv == nullptr): the caller's fixed `scale` for the whole codebook, chosen from max|c|;
//   * vectors / queries (row_inv != nullptr): a PER-ROW scale 2^e with max|x_row| * 2^e in [2^8, 2^9), so no input can
//     overflow fp16 (65504) or lose its lo part to underflow, whatever its magnitude relative to the centroids;
//     row_inv[row] = 2^-e is folded back in by the GEMM epilogue.  Non-finite rows keep scale 1: their products are
//     NaN / inf and the row gets label -1, as on the exact fp32 path.
// lo_flags (nullable): lo_flags[row / 256] is set when any lo part of that 256-row block is non-zero; blocks whose rows
// are exactly representable in fp16 (e.g. uint8-valued SIFT data) let the MMA issuer skip the x_lo.c_hi pass.
constexpr int PACK_ROWS = 32;      // rows per CTA iteration
constexpr int PACK_THREADS = 256;  // d / 8 <= 16 groups per row: at most two groups per thread and iteration

__global__ void __launch_bounds__(PACK_THREADS)
pack_rows_kernel(const float* __restrict__ x, int64_t rows, int64_t rows_padded, int d, float scale,
                 uint8_t* __restrict__ out, int* __restrict__ lo_flags, float* __restrict__ row_inv) {
  __shared__ unsigned rmax[PACK_ROWS];
  const int g8 = d / 8;  // 8-element groups per row
  const int nkb = d / KB;
  const int items = PACK_ROWS * g8;  // <= 512
  for (int64_t row0 = (int64_t)blockIdx.x * PACK_ROWS; row0 < rows_padded; row0 += (int64_t)gridDim.x * PACK_ROWS) {
    if (threadIdx.x < PACK_ROWS) rmax[threadIdx.x] = 0;
    __syncthreads();
    float v[2][8];
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const int it = threadIdx.x + u * PACK_THREADS;
      const int r = it / g8, kg8 = it % g8;
      const int64_t row = row0 + r;
      unsigned mx = 0;
      if (it < items && row < rows) {
        const float4* p = reinterpret_cast<const float4*>(x + row * d + kg8 * 8);
        const float4 a = p[0], b = p[1];
        v[u][0] = a.x; v[u][1] = a.y; v[u][2] = a.z; v[u][3] = a.w;
        v[u][4] = b.x; v[u][5] = b.y; v[u][6] = b.z; v[u][7] = b.w;
#pragma unroll
        for (int t = 0; t < 8; t++) mx = max(mx, __float_as_uint(v[u][t]) & 0x7fffffffu);  // |v| orders like its bits; NaN > inf
      } else {
#pragma unroll
        for (int t = 0; t < 8; t++) v[u][t] = 0.f;
      }
      if (row_inv && mx) atomicMax(&rmax[r], mx);
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const int it = threadIdx.x + u * PACK_THREADS;
      if (it >= items) break;
      const int r = it / g8, kg8 = it % g8;
      const int64_t row = row0 + r;
      if (row >= rows_padded) break;
      float sc = scale;
      if (row_inv) {
        const unsigned e = rmax[r] >> 23;  // biased exponent of max|x_row| (0: zero / subnormal row, 255: inf or NaN)
        sc = 1.f;
        float inv = 1.f;
        if (e >= 1 && e <= 254) {
          unsigned se = 262u - e;  // 2^(8 - (e - 127))
          se = se > 254u ? 254u : se;
          sc = __uint_as_float(se << 23);
          inv = __uint_as_float((254u - se) << 23);  // 2^-(se - 127); se = 254 -> 2^-127 is subnormal: exact all the same
          if (se == 254u) inv = 0x1.0p-127f;
        }
        if (kg8 == 0 && row < rows) row_inv[row] = inv;
      }
      __align__(16) __half hi[8];
      __align__(16) __half lo[8];
      bool lo_nz = false;
#pragma unroll
      for (int t = 0; t < 8; t++) {
        const float s = v[u][t] * sc;
        const __half h = __float2half_rn(s);
        hi[t] = h;
        const float rem = s - __half2float(h);
        lo[t] = __float2half_rn(rem);
        lo_nz |= rem != 0.f;
      }
      if (lo_flags && lo_nz) {
        int* f = lo_flags + row / (TILE_ROWS * ROW_TILES);
        if (*reinterpret_cast<volatile int*>(f) == 0) atomicOr(f, 1);
      }
      const int64_t tile = row / TILE_ROWS;
      const int rr = (int)(row % TILE_ROWS);
      const int kb = kg8 / (KB / 8), kg = kg8 % (KB / 8);
      const int64_t base = (tile * 2) * (int64_t)nkb * TILE_KB_BYTES;
      const int64_t inner = (int64_t)kb * TILE_KB_BYTES + (rr / 8) * 512 + kg * 128 + (rr % 8) * 16;
      *reinterpret_cast<uint4*>(out + base + inner) = *reinterpret_cast<const uint4*>(hi);
      *reinterpret_cast<uint4*>(out + base + (int64_t)nkb * TILE_KB_BYTES + inner) = *reinterpret_cast<const uint4*>(lo);
    }
    __syncthreads();
  }
}

__global__ void pad_cnorm_kernel(const float* __restrict__ cnorm, int C, int Cpad, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Cpad) out[i] = i < C ? cnorm[i] : __int_as_float(0x7f800000);
}

// ------------------------------------------------------------------------------------------------------ GEMM kernel
struct Params {
  const uint8_t* a_pack;   // packed vectors: row tiles of this launch
  const uint8_t* b_pack;   // packed centroids
  const float* cnorm_pad;  // [Cpad], +inf beyond C
  const int* a_lo_flags;   // [n_row_blocks]: 0 = the lo part of this vector block is identically zero
  int64_t n;               // valid rows
  int C, d;
  int n_row_blocks;        // ceil(n / 256)
  int n_ctiles;            // Cpad / 128
  int csplit;              // work item = (row block, centroid split)
  int tiles_per_split;
  float m2s;               // -2 / scale of the centroids
  const float* row_inv;    // [n] 1 / (per-row scale of the vectors), see pack_rows_kernel
  unsigned long long* keys;  // mode 0: [n] packed (ordered distance << 32 | centroid)
  float* D;                // mode 1: [n][ldD]
  int64_t ldD;
  float* bmin;             // mode 1 (nullable): [n][n_ctiles*4] minimum of every 32-column bucket of D
};

template <int MODE>  // 0 = fused arg-min, 1 = store the distance tile (+ bucket minima), 2 = bucket minima only
__global__ void __launch_bounds__(THREADS, 1) l2_tc_kernel(const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int nkb = p.d / KB;
  const int a_tile_bytes = 2 * nkb * TILE_KB_BYTES;  // one 128-row tile, hi+lo, all of K
  uint8_t* a_s = smem;                                // [ROW_TILES][hi,lo][nkb][8 KiB]
  uint8_t* b_s = a_s + ROW_TILES * a_tile_bytes;      // [STAGES][hi,lo][8 KiB]
  float* cn_s = reinterpret_cast<float*>(b_s + STAGES * 2 * TILE_KB_BYTES);  // [ACC_BUFS][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(cn_s + ACC_BUFS * TILE_ROWS);
  uint64_t* full = bars;                 // [STAGES]
  uint64_t* empty = bars + STAGES;       // [STAGES]
  uint64_t* a_full = bars + 2 * STAGES;  // [1]
  uint64_t* a_empty = a_full + 1;        // [1]
  uint64_t* t_full = a_empty + 1;        // [ACC_BUFS]
  uint64_t* t_empty = t_full + ACC_BUFS; // [ACC_BUFS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + ACC_BUFS);

  const int warp = threadIdx.x / 32;
  const int lane = threadIdx.x % 32;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int b = 0; b < ACC_BUFS; b++) {
      mbar_init(&t_full[b], 1);
      mbar_init(&t_empty[b], EPI_WARPS * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM allocation (whole warp), 512 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t n_rows = p.n;
  const int n_items = p.n_row_blocks * p.csplit;

  if (warp == 0) {
    // ===================================================================== producer
    if (elect_one()) {
      uint32_t stage = 0, phase = 0, item_phase = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int rb = item / p.csplit, cs = item % p.csplit;
        const int t0 = cs * p.tiles_per_split;
        const int t1 = min(p.n_ctiles, t0 + p.tiles_per_split);
        // A block (both row tiles are contiguous in the packed layout)
        mbar_wait(a_empty, item_phase ^ 1);
        mbar_arrive_expect_tx(a_full, ROW_TILES * a_tile_bytes);
        const uint8_t* asrc = p.a_pack + (int64_t)rb * ROW_TILES * a_tile_bytes;
        for (int c = 0; c < ROW_TILES * 2; c++)
          bulk_g2s(a_s + c * (a_tile_bytes / 2), asrc + (int64_t)c * (a_tile_bytes / 2), a_tile_bytes / 2, a_full);
        item_phase ^= 1;
        for (int t = t0; t < t1; t++) {
          const uint8_t* bsrc = p.b_pack + (int64_t)t * a_tile_bytes;
          for (int kb = 0; kb < nkb; kb++) {
            mbar_wait(&empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&full[stage], 2 * TILE_KB_BYTES);
            uint8_t* dst = b_s + stage * 2 * TILE_KB_BYTES;
            bulk_g2s(dst, bsrc + (int64_t)kb * TILE_KB_BYTES, TILE_KB_BYTES, &full[stage]);                       // hi
            bulk_g2s(dst + TILE_KB_BYTES, bsrc + (int64_t)(nkb + kb) * TILE_KB_BYTES, TILE_KB_BYTES, &full[stage]);  // lo
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    uint32_t stage = 0, phase = 0, item_phase = 0, acc_buf = 0, acc_phase = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int cs = item % p.csplit;
      const int t0 = cs * p.tiles_per_split;
      const int t1 = min(p.n_ctiles, t0 + p.tiles_per_split);
      mbar_wait(a_full, item_phase);
      tc_fence_after();
      const int npass = (p.a_lo_flags[item / p.csplit] != 0) ? 3 : 2;  // warp-uniform
      for (int t = t0; t < t1; t++) {
        mbar_wait(&t_empty[acc_buf], acc_phase ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < nkb; kb++) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t b_hi = smem_u32(b_s + stage * 2 * TILE_KB_BYTES);
            const uint32_t b_lo = b_hi + TILE_KB_BYTES;
#pragma unroll
            for (int r = 0; r < ROW_TILES; r++) {
              const uint32_t a_hi = smem_u32(a_s + r * a_tile_bytes + kb * TILE_KB_BYTES);
              const uint32_t a_lo = a_hi + nkb * TILE_KB_BYTES;
              const uint32_t tacc = tmem_base + (acc_buf * ROW_TILES + r) * TILE_ROWS;
#pragma unroll
              for (int pass = 0; pass < 3; pass++) {
                if (pass >= npass) break;
                const uint32_t a0 = pass == 2 ? a_lo : a_hi;  // hi.hi, hi.lo, lo.hi
                const uint32_t b0 = pass == 1 ? b_lo : b_hi;
#pragma unroll
                for (int k16 = 0; k16 < KB / 16; k16++) {
                  umma_f16(tacc, make_desc(a0 + k16 * 256), make_desc(b0 + k16 * 256), kIdesc,
                           (kb | pass | k16) != 0 ? 1u : 0u);
                }
              }
            }
          }
          __syncwarp();
          if (elect_one()) umma_commit(&empty[stage]);  // frees the B stage once these MMAs have read it
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (elect_one()) umma_commit(&t_full[acc_buf]);  // accumulators of this centroid tile are complete
        __syncwarp();
        if (++acc_buf == ACC_BUFS) {
          acc_buf = 0;
          acc_phase ^= 1;
        }
      }
      if (elect_one()) umma_commit(a_empty);  // all MMAs that read A have retired
      __syncwarp();
      item_phase ^= 1;
    }
  } else {
    // ===================================================================== epilogue (warps 2..9, 256 threads)
    const int et = threadIdx.x - 64;                  // 0..255
    const int lane_grp = warp & 3;                    // TMEM lanes this warp may read: [32*lane_grp, +32)
    const int col_half = (warp - 2) >> 2;             // which 64 of the tile's 128 columns this warp handles
    const int row_in_tile = lane_grp * 32 + lane;
    const int nb = p.n_ctiles * 4;
    uint32_t acc_buf = 0, acc_phase = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int rb = item / p.csplit, cs = item % p.csplit;
      const int t0 = cs * p.tiles_per_split;
      const int t1 = min(p.n_ctiles, t0 + p.tiles_per_split);
      float best[ROW_TILES], m2s[ROW_TILES];
      int bidx[ROW_TILES];
#pragma unroll
      for (int r = 0; r < ROW_TILES; r++) {
        best[r] = __int_as_float(0x7f800000);
        bidx[r] = 0x7fffffff;
        const int64_t row = ((int64_t)rb * ROW_TILES + r) * TILE_ROWS + row_in_tile;
        m2s[r] = p.m2s * (row < n_rows ? p.row_inv[row] : 1.f);  // -2 / (centroid scale * this row's scale): exact
      }
      float m2q[ROW_TILES][4];  // MODE 1: the same factor for the four rows of the thread's 16x64 fragments
      if (MODE == 1) {
#pragma unroll
        for (int r = 0; r < ROW_TILES; r++)
#pragma unroll
          for (int hi = 0; hi < 4; hi++) {
            const int64_t row = ((int64_t)rb * ROW_TILES + r) * TILE_ROWS + lane_grp * 32 + (hi >> 1) * 16 + (lane >> 2) + 8 * (hi & 1);
            m2q[r][hi] = p.m2s * (row < n_rows ? p.row_inv[row] : 1.f);
          }
      }
      (void)m2q;
      float cn_next = (et < TILE_ROWS && t0 < t1) ? p.cnorm_pad[t0 * TILE_ROWS + et] : 0.f;
      for (int t = t0; t < t1; t++) {
        // stage ||c||^2 of this centroid tile (safe: every epilogue thread passed the previous use of this slot
        // before arriving on t_empty two tiles ago, and the named barrier below orders the writes before the reads).
        // The value was fetched one tile ahead so that its L2 latency is off the per-tile critical path.
        if (et < TILE_ROWS) {
          cn_s[acc_buf * TILE_ROWS + et] = cn_next;
          if (t + 1 < t1) cn_next = p.cnorm_pad[(t + 1) * TILE_ROWS + et];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        mbar_wait(&t_full[acc_buf], acc_phase);
        tc_fence_after();
        const float* cn = cn_s + acc_buf * TILE_ROWS + col_half * 64;
        if (MODE == 1) {
          // D tile straight from registers.  With the 16x256b fragment a quad of threads owns 8 consecutive columns of a
          // row; one exchange between lanes t and t ^ 1 over a pair of column blocks gives every thread 4 consecutive
          // columns, so a store instruction writes 8 rows x 64 contiguous bytes: the same 64-byte store wavefronts as
          // fully coalesced rows, and 32 shuffles instead of the 128 shared-memory wavefronts of a transpose through
          // shared memory (which kept the L1 data pipe 76 % busy next to the MMA's operand reads: 284 us per 4096
          // queries, now 265).  Measured bounds of this sweep (tools/bench_coarse.py, DESIGN.md 4): no D at all 116 us;
          // stores that all hit L2 230 us; 32-byte-per-row stores or a 128 KiB-contiguous blocked D layout: no gain --
          // the SM's 32 B/clk write path to L2 (128 KiB per 256 x 128 tile = 4096 clk, twice the MMA time of the
          // tile) is what the D tile costs: ncu l1tex__m_l1tex2xbar_write_bytes 64 % of peak where a pure fill kernel
          // reaches 80 %.  16 epilogue warps of 32 columns each instead of 8 x 64: slower (290 us).
          const int qd = lane & 3;
          float2 cnv[8];
#pragma unroll
          for (int j = 0; j < 8; j++) cnv[j] = *reinterpret_cast<const float2*>(cn + 8 * j + 2 * qd);
          const int colq = t * TILE_ROWS + col_half * 64;
          const bool vec_ok = (p.ldD & 3) == 0 && (reinterpret_cast<uintptr_t>(p.D) & 15) == 0 && colq + 64 <= p.C;  // warp-uniform
#pragma unroll
          for (int r = 0; r < ROW_TILES; r++) {
            const uint32_t taddr = tmem_base + ((uint32_t)(lane_grp * 32) << 16) +
                                   (acc_buf * ROW_TILES + r) * TILE_ROWS + col_half * 64;
            uint32_t v[2][32];
            tmem_ld16x64(taddr, v[0]);
            tmem_ld16x64(taddr + (16u << 16), v[1]);
            tmem_ld_wait();
#pragma unroll
            for (int h = 0; h < 2; h++) {
#pragma unroll
              for (int i2 = 0; i2 < 2; i2++) {
                const int64_t row = ((int64_t)rb * ROW_TILES + r) * TILE_ROWS + lane_grp * 32 + h * 16 + (lane >> 2) + 8 * i2;
                const bool row_ok = row < n_rows;
                const float ms = m2q[r][h * 2 + i2];
                float* out = p.D + row * p.ldD + colq;
                float mn[2] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000)};
#pragma unroll
                for (int m = 0; m < 4; m++) {  // column blocks 2 m and 2 m + 1
                  float2 a, b;
                  a.x = fmaf(__uint_as_float(v[h][8 * m + 2 * i2]), ms, cnv[2 * m].x);
                  a.y = fmaf(__uint_as_float(v[h][8 * m + 2 * i2 + 1]), ms, cnv[2 * m].y);
                  b.x = fmaf(__uint_as_float(v[h][8 * m + 4 + 2 * i2]), ms, cnv[2 * m + 1].x);
                  b.y = fmaf(__uint_as_float(v[h][8 * m + 4 + 2 * i2 + 1]), ms, cnv[2 * m + 1].y);
                  mn[m >> 1] = fminf(mn[m >> 1], fminf(fminf(a.x, a.y), fminf(b.x, b.y)));
                  const bool odd = qd & 1;
                  const float s0 = odd ? a.x : b.x, s1 = odd ? a.y : b.y;
                  const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
                  // even lane of the pair: columns 2 qd .. 2 qd + 3 of block 2 m; odd lane: 2 (qd - 1) .. of block 2 m + 1
                  const float4 o = odd ? make_float4(r0, r1, b.x, b.y) : make_float4(a.x, a.y, r0, r1);
                  const int cc = 16 * m + (odd ? 8 + 2 * (qd - 1) : 2 * qd);
                  if (row_ok) {
                    if (vec_ok) {
                      *reinterpret_cast<float4*>(out + cc) = o;
                    } else {
                      if (colq + cc + 0 < p.C) out[cc + 0] = o.x;
                      if (colq + cc + 1 < p.C) out[cc + 1] = o.y;
                      if (colq + cc + 2 < p.C) out[cc + 2] = o.z;
                      if (colq + cc + 3 < p.C) out[cc + 3] = o.w;
                    }
                  }
                }
#pragma unroll
                for (int b = 0; b < 2; b++) {
                  mn[b] = fminf(mn[b], __shfl_xor_sync(0xffffffffu, mn[b], 1));
                  mn[b] = fminf(mn[b], __shfl_xor_sync(0xffffffffu, mn[b], 2));
                }
                // a select, not mn[qd]: indexed by a lane value, mn would live in local memory (8 bytes of stack, 32
                // local loads and stores in the sweep's epilogue; the sweep took 0.69 instead of 0.62 ms per 10 k
                // C2 queries, profiles/r10_overlap.md)
                if (row_ok && p.bmin && qd < 2) p.bmin[row * nb + t * 4 + col_half * 2 + qd] = qd ? mn[1] : mn[0];
              }
            }
          }
        } else {
#pragma unroll
        for (int r = 0; r < ROW_TILES; r++) {
          const uint32_t taddr = tmem_base + ((uint32_t)(lane_grp * 32) << 16) +
                                 (acc_buf * ROW_TILES + r) * TILE_ROWS + col_half * 64;
          const int64_t row = ((int64_t)rb * ROW_TILES + r) * TILE_ROWS + row_in_tile;
          uint32_t v[2][32];
          tmem_ld32(taddr, v[0]);  // both 32-column chunks in flight before the first use
          tmem_ld32(taddr + 32, v[1]);
          tmem_ld_wait();
          float mn_prev = 0.f;
          (void)mn_prev;
#pragma unroll
          for (int c = 0; c < 2; c++) {
            const int col0 = t * TILE_ROWS + col_half * 64 + c * 32;
            if (MODE == 0) {
              // running minimum with ONE min per element; the column is located only when the minimum of the chunk
              // beats the row's best, which happens O(log C) times per row over the whole sweep (compare + two
              // selects per element cost as much as an MMA pass at K = 128).  Same semantics as a strict `<` scan:
              // first column on exact ties, NaN never selected.
              float cmin = best[r];
#pragma unroll
              for (int i = 0; i < 32; i++) cmin = fminf(cmin, fmaf(__uint_as_float(v[c][i]), m2s[r], cn[c * 32 + i]));
              if (cmin < best[r]) {
                int first = 32;
#pragma unroll
                for (int i = 31; i >= 0; i--)
                  if (fmaf(__uint_as_float(v[c][i]), m2s[r], cn[c * 32 + i]) == cmin) first = i;
                best[r] = cmin;
                bidx[r] = col0 + first;
              }
            } else if (MODE == 2) {
              // bucket minima only: the distance matrix never leaves the SM (the query path re-evaluates the few
              // columns it needs exactly, coarse_select.cuh)
              float mn = __int_as_float(0x7f800000);
#pragma unroll
              for (int i = 0; i < 32; i++) mn = fminf(mn, fmaf(__uint_as_float(v[c][i]), m2s[r], cn[c * 32 + i]));
              if (c == 0) mn_prev = mn;
              if (c == 1 && row < n_rows)  // buckets (col0 >> 5) - 1 and col0 >> 5: one 8-byte store (nb is a multiple of 4)
                *reinterpret_cast<float2*>(p.bmin + row * nb + (col0 >> 5) - 1) = make_float2(mn_prev, mn);
            }
          }
        }
        }
        tc_fence_before();
        mbar_arrive(&t_empty[acc_buf]);
        if (++acc_buf == ACC_BUFS) {
          acc_buf = 0;
          acc_phase ^= 1;
        }
      }
      if (MODE == 0) {
#pragma unroll
        for (int r = 0; r < ROW_TILES; r++) {
          const int64_t row = ((int64_t)rb * ROW_TILES + r) * TILE_ROWS + row_in_tile;
          if (row < n_rows && bidx[r] != 0x7fffffff)  // two column halves (and csplit sweeps) combine through the key
            atomicMin(&p.keys[row], make_key(best[r], (uint32_t)bidx[r]));
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

// keys -> ids (+ distances, + ||x||^2)
__global__ void finalize_keys_kernel(const unsigned long long* __restrict__ keys, int64_t n, const float* __restrict__ xnorm,
                                     int* __restrict__ out_ids, float* __restrict__ out_dist) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long k = keys[i];
  const bool ok = k != kKeyInf;
  out_ids[i] = ok ? (int)key_payload(k) : -1;
  if (out_dist) out_dist[i] = ok ? key_val(k) + (xnorm ? xnorm[i] : 0.f) : FLT_MAX;
}

__global__ void row_norms_f32_kernel(const float* __restrict__ x, int64_t n, int d, float* __restrict__ out) {
  int64_t row = (int64_t)blockIdx.x * (blockDim.x / kWarp) + threadIdx.x / kWarp;
  int lane = threadIdx.x % kWarp;
  if (row >= n) return;
  const float* xr = x + row * d;
  float acc = 0.f;
  for (int j = lane; j < d; j += kWarp) acc = fmaf(xr[j], xr[j], acc);
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

static size_t smem_bytes(int d) {
  const int nkb = d / KB;
  return (size_t)ROW_TILES * 2 * nkb * TILE_KB_BYTES + (size_t)STAGES * 2 * TILE_KB_BYTES +
         ACC_BUFS * TILE_ROWS * sizeof(float) + 16 * sizeof(uint64_t) + 16;
}

static inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

constexpr int64_t CHUNK_ROWS = 1 << 18;  // rows packed + swept per launch (bounds the workspace)

static bool supported(int d, int C) { return d >= KB && d <= MAX_D && d % KB == 0 && C >= 1; }

static int num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return sms;
}

template <int MODE>
static int launch(const Params& p, cudaStream_t st) {
  const size_t smem = smem_bytes(p.d);
  cudaError_t e = cudaFuncSetAttribute(l2_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int items = p.n_row_blocks * p.csplit;
  const int grid = items < num_sms() ? items : num_sms();
  VLQ_LAUNCH(l2_tc_kernel<MODE>, grid, THREADS, smem, st, p);
  return last_error();
}

}  // namespace tc
}  // namespace vlq

using namespace vlq;

extern "C" {

int vlq_tc_supported(int d, int C) { return tc::supported(d, C) ? 1 : 0; }

size_t vlq_tc_cent_pack_bytes(int C, int d) {
  if (!tc::supported(d, C)) return 0;
  const int64_t Cpad = div_up(C, tc::TILE_ROWS) * tc::TILE_ROWS;
  return tc::align256((size_t)tc::packed_bytes(Cpad, d)) + tc::align256(sizeof(float) * Cpad);
}

static unsigned pack_grid(int64_t rows_padded) {
  return (unsigned)std::min<int64_t>(div_up(rows_padded, tc::PACK_ROWS), (int64_t)tc::num_sms() * 8);
}

int vlq_tc_pack_centroids(const float* cent, const float* cnorm, int C, int d, float scale, void* cent_pack,
                          vlq_stream_t stream) {
  if (!tc::supported(d, C) || !(scale > 0.f)) return VLQ_EUNSUPPORTED;
  if (!cent || !cnorm || !cent_pack) return VLQ_EINVAL;
  if ((reinterpret_cast<uintptr_t>(cent) & 15) || (reinterpret_cast<uintptr_t>(cent_pack) & 15)) return VLQ_EINVAL;
  const int64_t Cpad = div_up(C, tc::TILE_ROWS) * tc::TILE_ROWS;
  cudaStream_t st = as_stream(stream);
  VLQ_LAUNCH(tc::pack_rows_kernel, pack_grid(Cpad), tc::PACK_THREADS, 0, st, cent, (int64_t)C, Cpad, d, scale,
             static_cast<uint8_t*>(cent_pack), (int*)nullptr, (float*)nullptr);
  float* cn_pad = reinterpret_cast<float*>(static_cast<uint8_t*>(cent_pack) + tc::align256((size_t)tc::packed_bytes(Cpad, d)));
  VLQ_LAUNCH(tc::pad_cnorm_kernel, (unsigned)div_up(Cpad, 256), 256, 0, st, cnorm, C, (int)Cpad, cn_pad);
  return last_error();
}

size_t vlq_l2_tc_workspace_bytes(int64_t n, int d, int C) {
  if (!tc::supported(d, C) || n < 0) return 0;
  const int64_t rows = n < tc::CHUNK_ROWS ? n : tc::CHUNK_ROWS;
  const int64_t rpad = div_up(rows, tc::TILE_ROWS * tc::ROW_TILES) * tc::TILE_ROWS * tc::ROW_TILES;
  return tc::align256((size_t)tc::packed_bytes(rpad, d)) + tc::align256(sizeof(unsigned long long) * rows) +
         2 * tc::align256(sizeof(float) * rows) + tc::align256(sizeof(int) * (rpad / (tc::TILE_ROWS * tc::ROW_TILES))) + 256;
}

static int tc_run(int mode, const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, int add_xnorm,
                  int* out_ids, float* out_dist, float* D, int64_t ldD, float* bmin, void* workspace,
                  size_t workspace_bytes, vlq_stream_t stream) {
  if (!tc::supported(d, C) || !(scale > 0.f)) return VLQ_EUNSUPPORTED;
  if (n < 0) return VLQ_EINVAL;
  if (n == 0) return VLQ_OK;
  if (!x || !cent_pack || !workspace) return VLQ_EINVAL;
  if (mode == 0 && !out_ids) return VLQ_EINVAL;
  if (mode == 1 && (!D || ldD < C)) return VLQ_EINVAL;
  if (mode == 2 && !bmin) return VLQ_EINVAL;
  if (reinterpret_cast<uintptr_t>(x) & 15) return VLQ_EINVAL;
  if (workspace_bytes < vlq_l2_tc_workspace_bytes(n, d, C)) return VLQ_EWORKSPACE;
  cudaStream_t st = as_stream(stream);
  const int64_t Cpad = div_up(C, tc::TILE_ROWS) * tc::TILE_ROWS;
  const uint8_t* b_pack = static_cast<const uint8_t*>(cent_pack);
  const float* cn_pad = reinterpret_cast<const float*>(b_pack + tc::align256((size_t)tc::packed_bytes(Cpad, d)));
  const int64_t chunk = n < tc::CHUNK_ROWS ? n : tc::CHUNK_ROWS;
  const int64_t cpad_rows = div_up(chunk, tc::TILE_ROWS * tc::ROW_TILES) * tc::TILE_ROWS * tc::ROW_TILES;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255));
  uint8_t* a_pack = ws;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + tc::align256((size_t)tc::packed_bytes(cpad_rows, d)));
  float* xnorm = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(keys) + tc::align256(sizeof(unsigned long long) * chunk));
  float* row_inv = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(xnorm) + tc::align256(sizeof(float) * chunk));
  int* lo_flags = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(row_inv) + tc::align256(sizeof(float) * chunk));
  const bool add_xn = (add_xnorm & 1) != 0;
  const int sms = tc::num_sms();
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    const int64_t rows = (n - r0) < chunk ? (n - r0) : chunk;
    const int64_t rpad = div_up(rows, tc::TILE_ROWS * tc::ROW_TILES) * tc::TILE_ROWS * tc::ROW_TILES;
    const int nblocks = (int)(rpad / (tc::TILE_ROWS * tc::ROW_TILES));
    VLQ_CUDA_TRY(cudaMemsetAsync(lo_flags, 0, sizeof(int) * nblocks, st));
    VLQ_LAUNCH(tc::pack_rows_kernel, pack_grid(rpad), tc::PACK_THREADS, 0, st, x + r0 * d, rows, rpad, d, 1.f, a_pack,
               lo_flags, row_inv);
    tc::Params p{};
    p.a_pack = a_pack;
    p.b_pack = b_pack;
    p.cnorm_pad = cn_pad;
    p.a_lo_flags = lo_flags;
    p.n = rows;
    p.C = C;
    p.d = d;
    p.n_row_blocks = nblocks;
    p.n_ctiles = (int)(Cpad / tc::TILE_ROWS);
    // few row blocks (query batches): split the centroid sweep so that every SM has work
    int csplit = 1;
    if (p.n_row_blocks < sms) {
      csplit = sms / p.n_row_blocks;
      if (csplit > p.n_ctiles) csplit = p.n_ctiles;
      if (csplit < 1) csplit = 1;
    }
    p.tiles_per_split = (int)div_up(p.n_ctiles, csplit);
    p.csplit = (int)div_up(p.n_ctiles, p.tiles_per_split);
    p.m2s = -2.f / scale;
    p.row_inv = row_inv;
    p.keys = keys;
    p.D = mode == 1 ? D + r0 * ldD : nullptr;
    p.ldD = ldD;
    p.bmin = (mode != 0 && bmin) ? bmin + r0 * (int64_t)(Cpad / 32) : nullptr;
    int rc;
    if (mode == 0) {
      VLQ_CUDA_TRY(cudaMemsetAsync(keys, 0xff, sizeof(unsigned long long) * rows, st));
      rc = tc::launch<0>(p, st);
      if (rc) return rc;
      const float* xn = nullptr;
      if (add_xn && out_dist) {
        VLQ_LAUNCH(tc::row_norms_f32_kernel, (unsigned)div_up(rows, 8), 256, 0, st, x + r0 * d, rows, d, xnorm);
        xn = xnorm;
      }
      VLQ_LAUNCH(tc::finalize_keys_kernel, (unsigned)div_up(rows, 256), 256, 0, st, keys, rows, xn, out_ids + r0,
                 out_dist ? out_dist + r0 : nullptr);
    } else {
      rc = mode == 1 ? tc::launch<1>(p, st) : tc::launch<2>(p, st);
      if (rc) return rc;
    }
  }
  return last_error();
}

int vlq_l2_assign_tc(const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, int add_xnorm,
                     int* out_ids, float* out_dist, void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  return tc_run(0, x, n, d, cent_pack, scale, C, add_xnorm, out_ids, out_dist, nullptr, 0, nullptr, workspace,
                workspace_bytes, stream);
}

int vlq_l2_distances_tc(const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, float* D,
                        int64_t ldD, float* bucket_min, void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  return tc_run(1, x, n, d, cent_pack, scale, C, 0, nullptr, nullptr, D, ldD, bucket_min, workspace, workspace_bytes,
                stream);
}

int vlq_l2_bucket_min_tc(const float* x, int64_t n, int d, const void* cent_pack, float scale, int C, float* bucket_min,
                         void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  return tc_run(2, x, n, d, cent_pack, scale, C, 0, nullptr, nullptr, nullptr, 0, bucket_min, workspace,
                workspace_bytes, stream);
}

int vlq_tc_num_buckets(int C) { return (int)(div_up(C, tc::TILE_ROWS) * tc::TILE_ROWS / 32); }

}  // extern "C"
