// Long-list ADC scan (SURVEY.md 8a rows a14 + a15, north_star item 4): the kernel for 1B-scale list densities.
//   replaces pqScanPrecomputedMultiPassGraph + pass1/pass2SelectLists
//   (gpu/impl/PQScanMultiPassPrecomputed.cu:675-881, IVFUtilsSelect1.cu:28-144, IVFUtilsSelect2.cu:398-569).
//
// One CTA per query, 12 warps, two CTAs per SM.  ncu (profiles/r02_scan_long.md) shows what bounds this stage: not HBM
// but warp instructions and L1/shared-memory wavefronts per entry (16 table lookups each), so the kernel is built
// around a per-entry budget:
//
//   * bank-skewed term-3 tables (64-word rows, code-major; see search.cu "SKEW"): PRMT + LDS + FADD per lookup, the 32
//     lanes of a warp always hit 32 different banks.  The tables start at the base of the dynamic shared memory, whose
//     shared-window address (1 KB, checked once per process) is folded into the LDS immediate: the PRMT result
//     (code << 8 | 4 * lane) IS the register operand of the load.  The lists store the code bytes pre-rotated by the
//     position in the list (scan.cuh), so there is no per-entry byte shuffling.  The lambda codebook rides in the 16
//     spare words of the same rows (16 replicas: at most a two-way conflict for the per-entry lambda lookup).
//   * a warp owns whole lines and walks them in 128-entry segments, four entries per lane: 4 x (LDG.128 codes, LDG
//     kappa, LDG.U8 lambda) with clamped (never predicated) addresses, then 64 independent lookup chains: 299 SASS
//     instructions per segment.
//   * every line is brought into L2 by the TMA unit ahead of time: the warp that takes line i of the query issues three
//     cp.async.bulk.prefetch.L2 (codes / kappa / lambda ranges of line i + LOOK; SASS UBLKPF.L2).
//   * all warps share ONE candidate buffer and ONE threshold per query.  The first segment of every warp ends in a
//     block-wide exact selection (first threshold); afterwards the warps never meet again: appends reserve slots with one
//     atomicAdd per warp and segment, and every 128 appended candidates one warp tightens the threshold WITHOUT
//     stopping the others (sorted sample of the buffer -> candidate threshold -> verified by counting that at least k
//     buffered keys are below it -> atomicMin).  A blocking single-warp compaction remains as the overflow path.
//
// Tried on the way (all measured on the GPU, tools/bench_scan.py): a producer-warp / cp.async.bulk ring into shared
// memory (three bulk copies per 64-entry chunk serialise in the producer's ELECT loop: 23 ms vs 8.4 ms; and staging
// through shared memory adds ~25 % to the wavefronts of the pipe that is already the limit); per-warp candidate
// buffers (12x more appends); a blocking single-warp compaction (all warps sleep behind it: no gain); register double
// buffering of the segments (fewer resident warps: slower); L2 eviction-policy hints on loads / prefetch (no effect).
//
// Streamed per entry: M + 1 + 4 bytes (codes, lambda byte, kappa); SURVEY 8d counts M + 1 of them as algorithmic.
// The M terms are summed in a lane-dependent order (as in the skewed kernel of search.cu): distances can differ from
// the block-synchronous scans in the last ulp.
#include <cfloat>
#include <cstdlib>

#include "scan.cuh"
#include "topk.cuh"

namespace vlq {
namespace lscan {

constexpr int NT_MAX = 384;
constexpr int ROW_WORDS = 64;   // table row stride in words
constexpr int LCB_W0 = 48;      // words 48..63 of row j: lambda_cb[j]
constexpr int NBUCKET = 16;     // lines are bucketed by min(segments, 15)

struct __align__(16) LDesc {  // one selected line of the query (two 16-byte reads)
  int64_t st;  // first entry of the list
  int len;     // entries scanned (capped like IVFUtils.cu:87)
  int pad0;
  float t1, t6, t5;
  int pad1;
};

// Shared-memory loads with the table base folded into the instruction's immediate.  The tables sit at the start of the
// dynamic shared memory, which (no static shared memory in this kernel) starts right behind the 1 KB the driver
// reserves per CTA; kDynBase is verified once per process by a probe kernel (smem_base_ok) and the kernel falls back to
// ordinary pointer arithmetic (one extra add per lookup) if it ever differs.
constexpr uint32_t kDynBase = 1024;
template <int IMM>
__device__ __forceinline__ float lds_imm(uint32_t addr) {
  float v;
  asm("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(IMM));
  return v;
}
template <int IMM>
__device__ __forceinline__ int lds_imm_i(uint32_t addr) {
  int v;
  asm("ld.shared.s32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(IMM));
  return v;
}
// The term-3 tables are held as FIXED-POINT int32 (value * 2^e, e per query such that 16 terms cannot overflow): the M
// lookups of an entry are then summed with M / 2 three-input integer adds (IADD3) instead of M FADDs, and the sum is
// exact -- the only rounding is the conversion of each table entry, <= 2^-27 of the largest |T3| of the query, which is
// below the fp32 rounding of a float accumulation.  acc + sum over steps S.. of the lane's table word: PRMT (code << 8 |
// 4 * lane) + LDS per step, one IADD3 per two steps.
template <int MS, int S, bool FOLD>
struct Adc {
  static __device__ __forceinline__ int run(const uint32_t* cw, uint32_t lofs, const unsigned char* tbl, int acc) {
    if constexpr (S == MS) {
      return acc;
    } else {
      const uint32_t o0 = __byte_perm(cw[S >> 2], lofs, 0x5504 | ((S & 3) << 4));
      const uint32_t o1 = __byte_perm(cw[(S + 1) >> 2], lofs, 0x5504 | (((S + 1) & 3) << 4));
      int t0, t1;
      if constexpr (FOLD) {
        t0 = lds_imm_i<(int)kDynBase + 4 * S>(o0);
        t1 = lds_imm_i<(int)kDynBase + 4 * (S + 1)>(o1);
      } else {
        t0 = *reinterpret_cast<const int*>(tbl + o0 + 4 * S);
        t1 = *reinterpret_cast<const int*>(tbl + o1 + 4 * (S + 1));
      }
      return Adc<MS, S + 2, FOLD>::run(cw, lofs, tbl, acc + t0 + t1);
    }
  }
};
__global__ void smem_base_probe(uint32_t* out) {
  extern __shared__ __align__(16) unsigned char smem[];
  *out = (uint32_t)__cvta_generic_to_shared(smem);
}

__device__ __forceinline__ void prefetch_l2(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// 16-byte granules fully inside [p + b0, p + b1); p is 16-byte aligned
__device__ __forceinline__ void prefetch_range(const unsigned char* p, int64_t b0, int64_t b1) {
  const int64_t s = b0 & ~int64_t(15), e = b1 & ~int64_t(15);
  if (e > s) prefetch_l2(p + s, (uint32_t)(e - s));
}

template <int MS>
__device__ __forceinline__ void prefetch_line(const ScanArgs& a, const LDesc& d) {
  if (d.len <= 0) return;
  prefetch_range(a.codes, d.st * MS, (d.st + d.len) * MS);
  prefetch_range(reinterpret_cast<const unsigned char*>(a.kappa), d.st * 4, (d.st + d.len) * 4);
  prefetch_range(a.lamq, d.st, d.st + d.len);
}

__host__ __device__ inline size_t smem_bytes(int W) {
  size_t off = sizeof(float) * 256 * ROW_WORDS;
  off += (select_smem_bytes(kSharedSelCap) + 15) & ~size_t(15);
  off += sizeof(LDesc) * W;
  off += ((size_t)W * 2 + 15) & ~size_t(15);
  off += sizeof(int) * 32;  // misc: [0] next line, [1] lines, [2 + b] bucket cursors, [31] max |T3| of the query
  return off;
}

// ---- one candidate buffer per query, shared by the autonomous warps (BlockSelect layout: keys | hist[256] | meta[8]).
// Unused slots always hold kKeyInf, so a reader may look at any prefix of the buffer while other warps append.
constexpr int CAP = kSharedSelCap;
constexpr int STEP = 128;  // a threshold update is attempted every STEP appended candidates
enum : int { M_CUR = 0, M_COMMIT = 4, M_THR = 5, M_LOCK = 6 };  // meta words ([1..3]: BlockSelect scratch)
// M_THR: order-preserving uint32 image (f2ord) of the distance threshold, only ever lowered (atomicMin)

// Non-blocking threshold update by ONE warp (others keep scanning and appending): sort 128 samples of the buffer, pick
// the sample whose rank should cover k keys, VERIFY by counting that at least k buffered keys are <= it (so no member
// of the final top-k can ever be rejected), publish with atomicMin.  Nothing is moved: the buffer stays append-only.
__device__ void update_threshold(uint64_t* keys, int* hist, int* meta, int k, int lane) {
  int got = 0;
  if (lane == 0) got = atomicCAS(&meta[M_LOCK], 0, 1) == 0;
  if (!__shfl_sync(kFull, got, 0)) return;  // a compaction or another update is running
  const int n0 = min(ld_volatile(&meta[M_CUR]), CAP);
  if (n0 > k) {
    uint64_t* smp = reinterpret_cast<uint64_t*>(hist);  // 128 keys (the histogram is only used under the same lock)
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int j = lane + 32 * r;
      smp[j] = keys[(j * n0) >> 7];
    }
    __syncwarp();
    warp_bitonic_sort<4>(smp);
    __syncwarp();
    const float mean = (float)k * 128.f / (float)n0;
    int j = (int)(mean + 2.f * sqrtf(mean * (1.f - (float)k / (float)n0)) + 1.5f);
#pragma unroll 1
    for (int attempt = 0; attempt < 2; attempt++) {
      j = min(j, 127);
      const uint64_t T = smp[j];
      if (T == kKeyInf) break;
      int cnt = 0;
      for (int i = lane; i < n0; i += 32) cnt += keys[i] <= T;
      cnt = __reduce_add_sync(kFull, cnt);
      if (cnt >= k) {
        if (lane == 0) atomicMin(reinterpret_cast<unsigned*>(&meta[M_THR]), (unsigned)(T >> 32));
        break;
      }
      j = 2 * j + 4;
    }
  }
  __syncwarp();
  if (lane == 0) {
    __threadfence_block();
    atomicExch(&meta[M_LOCK], 0);
  }
}

// warp-collective: every lane offers its EPL entries of the segment (pass[u]: valid and not above the threshold the
// caller read).  ONE reservation for the whole warp.  Returns true when the append crossed a multiple of STEP (the
// caller then runs update_threshold once).  Overflow (rare: the sampled threshold keeps the buffer far from full)
// falls back to a blocking compaction by the warp whose reservation crossed the capacity.
template <int EPL>
__device__ __forceinline__ bool offer_n(uint64_t* keys, int* hist, int* meta, int k, const bool (&valid)[EPL],
                                        const float (&dist)[EPL], uint32_t pay0, float thr, int lane) {
  const unsigned lt = (1u << lane) - 1;
  for (;;) {
    unsigned m[EPL];
    int pre[EPL + 1];
    pre[0] = 0;
#pragma unroll
    for (int u = 0; u < EPL; u++) {
      m[u] = __ballot_sync(kFull, valid[u] && dist[u] <= thr);
      pre[u + 1] = pre[u] + __popc(m[u]);
    }
    const int n = pre[EPL];
    if (!n) return false;
    int base = 0;
    if (lane == 0) base = atomicAdd(&meta[M_CUR], n);
    base = __shfl_sync(kFull, base, 0);
    if (base + n <= CAP) {
#pragma unroll
      for (int u = 0; u < EPL; u++)
        if ((m[u] >> lane) & 1) keys[base + pre[u] + __popc(m[u] & lt)] = make_key(dist[u], pay0 + 32u * u);
      __syncwarp();
      if (lane == 0) {
        __threadfence_block();
        atomicAdd(&meta[M_COMMIT], n);
      }
      return ((base ^ (base + n)) & ~(STEP - 1)) != 0;
    }
    if (base <= CAP) {
      // slots [0, base) belong to other warps' appends: wait until they are all written, keep the k smallest, refill
      // the rest with kKeyInf, publish the k-th value as threshold and reopen the buffer
      if (lane == 0)
        while (atomicCAS(&meta[M_LOCK], 0, 1) != 0) __nanosleep(64);
      __syncwarp();
      while (ld_volatile(&meta[M_COMMIT]) != base) __nanosleep(64);
      __threadfence_block();
      int kept = base;
      if (base > k) {
        const uint64_t kth = warp_select_smem(keys, base, k, hist);
        kept = k;
        __syncwarp();
        for (int i = k + lane; i < base; i += 32) keys[i] = kKeyInf;
        if (lane == 0) atomicMin(reinterpret_cast<unsigned*>(&meta[M_THR]), (unsigned)(kth >> 32));
      }
      __syncwarp();
      if (lane == 0) {
        *reinterpret_cast<volatile int*>(&meta[M_COMMIT]) = kept;
        __threadfence_block();
        atomicExch(&meta[M_CUR], kept);
        atomicExch(&meta[M_LOCK], 0);
      }
      __syncwarp();
    } else {
      while (ld_volatile(&meta[M_CUR]) > CAP) __nanosleep(128);  // closed for compaction
    }
    thr = ord2f((uint32_t)ld_volatile(&meta[M_THR]));
  }
}

template <int MS, bool FOLD, int EPL, int NT>
__global__ void __launch_bounds__(NT, 2) scan_long_kernel(ScanArgs a, int look, int lpt) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int SEG = 32 * EPL;  // entries per segment
  static_assert(NT / 32 * SEG <= CAP, "the first segments of all warps must fit the candidate buffer");
  const int W = a.W;
  const int lane = threadIdx.x & 31;
  unsigned char* tbl = smem;
  unsigned char* selmem = smem + sizeof(float) * 256 * ROW_WORDS;
  uint64_t* skeys = reinterpret_cast<uint64_t*>(selmem);
  int* shist = reinterpret_cast<int*>(skeys + CAP);
  int* smeta = shist + 256;
  size_t off = sizeof(float) * 256 * ROW_WORDS + ((select_smem_bytes(CAP) + 15) & ~size_t(15));
  LDesc* desc = reinterpret_cast<LDesc*>(smem + off);
  off += sizeof(LDesc) * W;
  uint16_t* order = reinterpret_cast<uint16_t*>(smem + off);  // non-empty lines in processing order
  off += ((size_t)W * 2 + 15) & ~size_t(15);
  int* misc = reinterpret_cast<int*>(smem + off);  // [0] next line, [1] lines, [2 + b] bucket cursors

  const int64_t qi = blockIdx.x;
  float inv_scale;  // 2^-e of the fixed-point tables
  {  // word c of row `code` = T3[c mod M][code] * 2^e as int32 (a.t3 is code-major); words 48..63 = lambda_cb[code] (float)
    const float4* src4 = reinterpret_cast<const float4*>(a.t3 + (size_t)qi * MS * 256);
    constexpr int Q4 = (31 + MS + 3) / 4, S4 = MS / 4;
    constexpr int NSRC = 256 * S4, PER = (NSRC + NT - 1) / NT;
    static_assert(Q4 * 4 <= LCB_W0, "table words overlap the lambda words");
    float4 v[PER];
    float mx = 0.f;
#pragma unroll
    for (int t = 0; t < PER; t++) {
      const int j = threadIdx.x + t * NT;
      v[t] = j < NSRC ? src4[j] : make_float4(0.f, 0.f, 0.f, 0.f);
      mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v[t].x), fabsf(v[t].y)), fmaxf(fabsf(v[t].z), fabsf(v[t].w))));
    }
    const unsigned mxb = __reduce_max_sync(kFull, __float_as_uint(mx));  // non-negative floats order like their bit patterns
    if (threadIdx.x == 0) misc[31] = 0;
    __syncthreads();
    if (lane == 0) atomicMax(reinterpret_cast<unsigned*>(&misc[31]), mxb);
    __syncthreads();
    const float qmax = __uint_as_float((unsigned)misc[31]);
    // largest power of two with qmax * scale < 2^26 (the M <= 16 terms of an entry then sum below 2^30); NaN / Inf
    // tables (NaN queries) keep scale 1: their entries are never selected anyway
    int e = 0;
    if (qmax > 0.f && qmax < 3.0e38f) e = 25 - ilogbf(qmax);
    e = max(-100, min(100, e));
    const float scale = ldexpf(1.f, e);
    inv_scale = ldexpf(1.f, -e);
    int4* dst4 = reinterpret_cast<int4*>(tbl);
#pragma unroll
    for (int t = 0; t < PER; t++) {
      const int j = threadIdx.x + t * NT;
      if (j < NSRC) {
        const int code = j / S4, part = j % S4;
        const int4 w = make_int4(__float2int_rn(v[t].x * scale), __float2int_rn(v[t].y * scale),
                                 __float2int_rn(v[t].z * scale), __float2int_rn(v[t].w * scale));
#pragma unroll
        for (int q4 = part; q4 < Q4; q4 += S4) dst4[code * (ROW_WORDS / 4) + q4] = w;
      }
    }
    float4* dstf = reinterpret_cast<float4*>(tbl);
    for (int i = threadIdx.x; i < 256 * 4; i += NT) {
      const int code = i >> 2;
      const float lv = code < a.nL ? a.lambda_cb[code] : 0.f;
      dstf[code * (ROW_WORDS / 4) + LCB_W0 / 4 + (i & 3)] = make_float4(lv, lv, lv, lv);
    }
  }
  for (int i = threadIdx.x; i < CAP; i += NT) skeys[i] = kKeyInf;
  if (threadIdx.x < 2 + NBUCKET) misc[threadIdx.x] = 0;
  if (threadIdx.x < 8) smeta[threadIdx.x] = threadIdx.x == M_THR ? (int)0xff800000u /* f2ord(+inf) */ : 0;
  __syncthreads();
  for (int w = threadIdx.x; w < W; w += NT) {
    const int list = a.line_list[qi * W + w];
    LDesc d;
    d.st = 0;
    d.len = 0;
    d.pad0 = d.pad1 = 0;
    d.t5 = 0.f;
    if (list >= 0) {
      d.st = a.offsets[list];
      const int64_t l = a.offsets[list + 1] - d.st;
      d.len = (int)(l < a.cap ? l : a.cap);
      d.t5 = a.edge_d2 ? a.edge_d2[list] : 0.f;
    }
    d.t1 = a.term1[qi * W + w];
    d.t6 = a.term6[qi * W + w];
    desc[w] = d;
    const int b = min((d.len + SEG - 1) / SEG, NBUCKET - 1);
    if (b > 0) atomicAdd(&misc[2 + b], 1);
  }
  __syncthreads();
  int nlines;
  if (lpt) {  // longest first (counting sort by segment count): the tail of the query is a short list
    if (threadIdx.x == 0) {
      int run = 0;
      for (int b = NBUCKET - 1; b >= 1; b--) {
        const int c = misc[2 + b];
        misc[2 + b] = run;
        run += c;
      }
      misc[1] = run;
    }
    __syncthreads();
    for (int w = threadIdx.x; w < W; w += NT) {
      const int b = min((desc[w].len + SEG - 1) / SEG, NBUCKET - 1);
      if (b > 0) order[atomicAdd(&misc[2 + b], 1)] = (uint16_t)w;
    }
    __syncthreads();
    nlines = misc[1];
  } else {  // the order of the line selection (best line first): good candidates early, fewer appends overall
    if (threadIdx.x < 32) {
      int run = 0;
      for (int w0 = 0; w0 < W; w0 += 32) {
        const int w = w0 + lane;
        const bool ne = w < W && desc[w].len > 0;
        const unsigned m = __ballot_sync(kFull, ne);
        if (ne) order[run + __popc(m & ((1u << lane) - 1))] = (uint16_t)w;
        run += __popc(m);
      }
      if (lane == 0) misc[1] = run;
    }
    __syncthreads();
    nlines = misc[1];
  }
  if ((int)threadIdx.x < look && (int)threadIdx.x < nlines) prefetch_line<MS>(a, desc[order[threadIdx.x]]);

  const uint32_t lofs = 4u * (uint32_t)lane;                      // column of the lane in the skewed table rows
  const uint32_t lcbofs = 4u * (uint32_t)(LCB_W0 + (lane & 15));  // its replica of the lambda codebook

  // ---- every warp walks whole lines in segments of SEG = 32 * EPL entries.  (Measured and dropped: a register
  // double buffer -- loads of segment i + 1 in flight while segment i is scored -- costs a third of the resident warps,
  // 8.05 vs 7.5 ms per 10 k queries at 1 B entries; a rolling half-segment pipeline in the same registers spills the
  // in-flight kappa / lambda values at 80 registers, 9.2 ms, and with 10 warps at 96 registers reaches 8.4 ms.)
  bool first = true;  // the first segment of every warp ends in a block-wide rendezvous (see below)
  for (;;) {
    int li = 0;
    if (lane == 0) li = atomicAdd(&misc[0], 1);
    li = __shfl_sync(kFull, li, 0);
    const bool have = li < nlines;
    if (!have && !first) break;
    int len = 0;
    float t1 = 0.f, t6 = 0.f, t5 = 0.f;
    const unsigned char* cb = a.codes;
    const float* kb = a.kappa;
    const unsigned char* lb = a.lamq;
    uint32_t pay_w = 0;
    if (have) {
      if (lane == 0 && look > 0 && li + look < nlines) prefetch_line<MS>(a, desc[order[li + look]]);
      const int w = order[li];
      const int4 d0 = reinterpret_cast<const int4*>(desc + w)[0];
      const int4 d1 = reinterpret_cast<const int4*>(desc + w)[1];
      const int64_t st = ((int64_t)(uint32_t)d0.y << 32) | (uint32_t)d0.x;
      len = d0.z;
      t1 = __int_as_float(d1.x);
      t6 = __int_as_float(d1.y);
      t5 = __int_as_float(d1.z);
      cb = a.codes + st * MS;
      kb = a.kappa + st;
      lb = a.lamq + st;
      pay_w = (uint32_t)w << 20;
    }
    int e0 = 0;
#pragma unroll 1
    do {
      if (have) {
        const int last = len - 1;
        uint32_t cw[EPL][MS / 4];
        float kap[EPL];
        uint32_t lq[EPL];
        if (e0 + SEG - 1 <= last) {  // full segment: one address per array, the four entries at immediate offsets
          const unsigned char* cp = cb + (size_t)(e0 + lane) * MS;
          const float* kp = kb + (e0 + lane);
          const unsigned char* lp = lb + (e0 + lane);
#pragma unroll
          for (int u = 0; u < EPL; u++) {
            if constexpr (MS == 16) {
              const uint4 c = ld_nc_v4(cp + u * 32 * 16);
              cw[u][0] = c.x; cw[u][1] = c.y; cw[u][MS / 4 - 2] = c.z; cw[u][MS / 4 - 1] = c.w;
            } else {
              const uint2 c = ld_nc_v2(cp + u * 32 * 8);
              cw[u][0] = c.x; cw[u][MS / 4 - 1] = c.y;
            }
            kap[u] = __ldg(kp + u * 32);
            lq[u] = __ldg(lp + u * 32);
          }
        } else {
#pragma unroll
          for (int u = 0; u < EPL; u++) {  // clamped, never predicated: duplicates of the last entry are masked below
            const uint32_t i = (uint32_t)min(e0 + u * 32 + lane, last);
            if constexpr (MS == 16) {
              const uint4 c = ld_nc_v4(cb + (size_t)i * 16);
              cw[u][0] = c.x; cw[u][1] = c.y; cw[u][MS / 4 - 2] = c.z; cw[u][MS / 4 - 1] = c.w;
            } else {
              const uint2 c = ld_nc_v2(cb + (size_t)i * 8);
              cw[u][0] = c.x; cw[u][MS / 4 - 1] = c.y;
            }
            kap[u] = __ldg(kb + i);
            lq[u] = __ldg(lb + i);
          }
        }
        const float thr = ord2f((uint32_t)ld_volatile(&smeta[M_THR]));
        float dist[EPL];
        bool valid[EPL];
        bool pass = false;
#pragma unroll
        for (int u = 0; u < EPL; u++) {
          const uint32_t ol = __byte_perm(lq[u], lcbofs, 0x5504);
          float la;
          if constexpr (FOLD) la = lds_imm<(int)kDynBase>(ol);
          else la = *reinterpret_cast<const float*>(tbl + ol);
          const float base_d = t1 + la * t6 + (la * la - la) * t5;
          const float acc = (float)Adc<MS, 0, FOLD>::run(cw[u], lofs, tbl, 0) * inv_scale;
          dist[u] = (kap[u] + acc) + base_d;
          valid[u] = e0 + u * 32 + lane <= last;
          pass |= valid[u] && dist[u] <= thr;
        }
        if (__any_sync(kFull, pass)) {
          const bool crossed =
              offer_n<EPL>(skeys, shist, smeta, a.k, valid, dist, pay_w | (uint32_t)(e0 + lane), thr, lane);
          if (crossed && !first) update_threshold(skeys, shist, smeta, a.k, lane);
        }
      }
      if (first) {
        // Every warp has scored one segment against an infinite threshold (<= NT / 32 * SEG <= CAP candidates in the
        // buffer): one block-wide exact selection gives the first real threshold; from here on the warps never meet
        // again until the end of the query.
        first = false;
        __syncthreads();
        const int n0 = smeta[M_CUR];
        BlockSelect<NT> sel0;
        sel0.attach(selmem, a.k, CAP);
        sel0.compact();
        const int kept = smeta[M_CUR];
        for (int i = kept + (int)threadIdx.x; i < n0; i += NT) skeys[i] = kKeyInf;
        if (threadIdx.x == 0) {
          smeta[M_COMMIT] = kept;
          if (n0 > a.k) smeta[M_THR] = (int)(unsigned)(sel0.thr >> 32);
        }
        __syncthreads();
      }
      e0 += SEG;
    } while (have && e0 < len);
    if (!have) break;
  }
  __syncthreads();
  BlockSelect<NT> sel;
  sel.attach(selmem, a.k, CAP);
  sel.finish();
  for (int i = threadIdx.x; i < a.k; i += NT) {
    const uint64_t key = sel.keys[i];
    float dv = FLT_MAX;
    int64_t id = -1;
    if (key != kKeyInf) {
      const uint32_t pay = key_payload(key);
      dv = key_val(key);
      const int64_t e = desc[pay >> 20].st + (pay & 0xfffffu);
      id = a.ids ? a.ids[e] : e;
    }
    a.outD[qi * a.k + i] = dv;
    a.outI[qi * a.k + i] = id;
  }
}

static int smem_optin() {
  static int v = 0;
  if (!v) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  }
  return v;
}

// one-time check (first launch of the process) that the dynamic shared memory starts at kDynBase
static bool smem_base_ok() {
  static const bool ok = [] {
    uint32_t* d = nullptr;
    uint32_t h = 0;
    if (cudaMalloc(&d, sizeof(uint32_t)) != cudaSuccess) return false;
    smem_base_probe<<<1, 1, 1024>>>(d);
    const bool good = cudaMemcpy(&h, d, sizeof(uint32_t), cudaMemcpyDeviceToHost) == cudaSuccess && h == kDynBase;
    cudaFree(d);
    return good;
  }();
  return ok;
}

template <int MS, bool FOLD, int EPL, int NT>
static int launch_t(const ScanArgs& a, int64_t nq, int look, int lpt, cudaStream_t st) {
  const size_t smem = smem_bytes(a.W);
  VLQ_CUDA_TRY(cudaFuncSetAttribute(scan_long_kernel<MS, FOLD, EPL, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  VLQ_LAUNCH((scan_long_kernel<MS, FOLD, EPL, NT>), (unsigned)nq, NT, smem, st, a, look, lpt);
  return last_error();
}

// four entries per lane and segment (measured at 1 B entries, ms per 10 k queries: 4 -> 7.54, 3 -> 7.81, 2 -> 8.81;
// sixteen warps per CTA at 64 registers: 8.5-9.4)
template <int MS, bool FOLD>
static int launch_epl(const ScanArgs& a, int64_t nq, int look, int lpt, cudaStream_t st) {
  return launch_t<MS, FOLD, 4, 384>(a, nq, look, lpt, st);
}

}  // namespace lscan

bool scan_long_supported(const ScanArgs& a) {
  if (!(a.M == 16 || a.M == 8) || a.ksub != 256 || !a.t3 || a.nL > 256 || a.k > VLQ_MAX_K || a.cap > (1 << 20) ||
      a.W > 1024)
    return false;
  const uintptr_t al = reinterpret_cast<uintptr_t>(a.codes) | reinterpret_cast<uintptr_t>(a.t3);
  if (al & 15) return false;
  return lscan::smem_bytes(a.W) <= (size_t)lscan::smem_optin();
}

int launch_scan_long(const ScanArgs& a, int64_t nq, cudaStream_t st) {
  if (!scan_long_supported(a)) return VLQ_EUNSUPPORTED;
  // lines brought into L2 ahead of the scanning warps (0 = no prefetch); needs 16-byte aligned arrays
  static const int look_env = [] {
    const char* e = getenv("VLQ_SCAN_LOOK");
    return e ? atoi(e) : 4;
  }();
  const uintptr_t al = reinterpret_cast<uintptr_t>(a.kappa) | reinterpret_cast<uintptr_t>(a.lamq);
  const int look = (al & 15) ? 0 : (look_env < 0 ? 0 : (look_env > 256 ? 256 : look_env));
  static const int lpt = [] {  // 1: hand the lines out longest first; 0: in selection order (best line first)
    const char* e = getenv("VLQ_SCAN_LPT");
    return e ? atoi(e) : 0;
  }();
  const bool fold = lscan::smem_base_ok();
  if (a.M == 16)
    return fold ? lscan::launch_epl<16, true>(a, nq, look, lpt, st)
                : lscan::launch_epl<16, false>(a, nq, look, lpt, st);
  return fold ? lscan::launch_epl<8, true>(a, nq, look, lpt, st)
              : lscan::launch_epl<8, false>(a, nq, look, lpt, st);
}

}  // namespace vlq
