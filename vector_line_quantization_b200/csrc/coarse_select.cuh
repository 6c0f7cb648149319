// Fast path of the fused top-P + line selection (SURVEY.md 8a rows a11 + a12; replaces l2SelectMinK + the line scoring and
// BlockSelect of sumAlongRowsWithOrder2: gpu/impl/L2Select.cu:124-165, BroadcastSum.cu:477-560).
//
// The general kernel (search.cu coarse_select_lines_kernel) runs three block-wide selections over 2048 64-bit keys in
// shared memory per query (bucket minima -> candidate columns -> lines) and was the dominant kernel of the C2 step
// (ncu round 1: 158 M warp instructions per 4096 queries, 0.05 of the HBM roofline).  Here the keys of a selection
// live in REGISTERS as 32-bit order-preserving images, R per thread, and only a threshold is computed:
//
//   kth32():   byte-wise radix select of the K-th smallest key -- shared memory only holds the 256-bin histogram; the
//              bytes that do not vary are skipped, a bin that holds a single key ends the search early.  Returns the
//              threshold, how many keys are strictly below it and how many equal it.
//   taking:    key < threshold, plus the lowest-index keys equal to it (a block scan of the per-thread tie counts,
//              only when there are more ties than needed).  Ties are COMMON in the line stage: every line of a
//              centroid whose neighbour lies behind the query's Voronoi side scores exactly b2.
//   ordering:  the few survivors (P columns, W lines) are ordered by counting ranks against (value, index) keys that
//              sit in shared memory (rank = #keys smaller, O(n^2 / threads) broadcast reads, one barrier) up to 128
//              keys; 129 .. 256 keys (the W = 256 lines of the headline configuration) go through block_sort256(), a
//              bitonic network with one key per thread (shuffles below distance 32).
//
// The same file holds the MATRIX-FREE variant (coarse_select_lines_exact_kernel, further down): same selections, but the
// distances it needs are re-evaluated in fp32 from the centroid table instead of being read from a stored matrix.
//
// The candidate columns of stage 2 are the entries of D not above the P-th smallest bucket minimum (at least P of them,
// all inside the P selected buckets, typically 1.2 P), so stage 2 reads P 128-byte lines of D and orders ~80 keys.
// Results are bit-identical to the general kernel and to select_rows + select_lines (lowest index on ties).
#pragma once
#include "topk.cuh"

namespace vlq {
namespace csl {

constexpr int NT = 256;
constexpr uint32_t kInf32 = 0xffffffffu;

struct Kth {
  uint32_t tau;  // K-th smallest key (kInf32: fewer than K valid keys -- take them all)
  int n_lt;      // valid keys < tau
  int n_eq;      // valid keys == tau
};

// Block-wide K-th smallest of the valid (!= kInf32) keys held R per thread.  hist: 256 ints, meta: 8 ints (shared).
// K >= 1.  Every thread returns the same result.
template <int R>
__device__ __forceinline__ Kth kth32(const uint32_t (&key)[R], int K, int* hist, int* meta) {
  const int lane = threadIdx.x & 31;
  uint32_t o = 0, a = kInf32;
  int nv = 0;
#pragma unroll
  for (int r = 0; r < R; r++) {
    if (key[r] != kInf32) {
      o |= key[r];
      a &= key[r];
      nv++;
    }
  }
  o = __reduce_or_sync(kFull, o);
  a = __reduce_and_sync(kFull, a);
  nv = __reduce_add_sync(kFull, nv);
  if (threadIdx.x == 0) {
    meta[0] = 0;
    meta[1] = (int)kInf32;
    meta[2] = 0;
  }
  __syncthreads();
  if (lane == 0) {
    atomicOr(reinterpret_cast<unsigned*>(&meta[0]), o);
    atomicAnd(reinterpret_cast<unsigned*>(&meta[1]), a);
    atomicAdd(&meta[2], nv);
  }
  __syncthreads();
  const uint32_t bor = (uint32_t)meta[0], band = (uint32_t)meta[1];
  const int total = meta[2];
  Kth out;
  if (total < K || total == 0) {  // block-uniform
    out.tau = kInf32;
    out.n_lt = total;
    out.n_eq = 0;
    __syncthreads();
    return out;
  }
  const uint32_t diff = bor ^ band;
  const int top = diff ? (31 - __clz((int)diff)) >> 3 : 0;  // most significant byte that varies
  uint32_t prefix = top == 3 ? 0u : (bor >> ((top + 1) * 8));
  int need = K, in_bin = total;
  bool found = false;
#pragma unroll 1
  for (int pass = top; pass >= 0; pass--) {
    hist[threadIdx.x] = 0;  // NT == 256 bins
    __syncthreads();
    const int shift = pass * 8;
#pragma unroll
    for (int r = 0; r < R; r++) {
      const uint32_t k_ = key[r];
      const bool match = k_ != kInf32 && (pass == 3 || (k_ >> (shift + 8)) == prefix);
      if (match) atomicAdd(&hist[(k_ >> shift) & 255], 1);
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // lane l owns bins [8l, 8l + 8)
      int c[8], s = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        c[j] = hist[lane * 8 + j];
        s += c[j];
      }
      int inc = s;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(kFull, inc, d);
        if (lane >= d) inc += t;
      }
      int before = inc - s;
      if (before < need && need <= inc) {  // exactly one lane
#pragma unroll
        for (int j = 0; j < 8; j++) {
          if (need <= before + c[j]) {
            meta[4] = lane * 8 + j;
            meta[5] = need - before;
            meta[6] = c[j];
            break;
          }
          before += c[j];
        }
      }
    }
    __syncthreads();
    prefix = (prefix << 8) | (uint32_t)meta[4];
    need = meta[5];
    in_bin = meta[6];
    if (in_bin == 1 && pass > 0) {  // the wanted key is alone under this prefix: look it up
#pragma unroll
      for (int r = 0; r < R; r++)
        if (key[r] != kInf32 && (key[r] >> shift) == prefix) meta[7] = (int)key[r];
      __syncthreads();
      prefix = (uint32_t)meta[7];
      found = true;
      break;
    }
  }
  (void)found;
  out.tau = prefix;
  out.n_eq = in_bin;
  out.n_lt = K - need;
  __syncthreads();  // hist / meta may be reused by the caller
  return out;
}

// Which of the thread's keys belong to the K smallest: key < tau, plus the lowest-index ties (thread t holds the
// indices [R t, R t + R), so index order = thread order).  wsum: 8 ints (shared).
template <int R>
__device__ __forceinline__ void take_k(const uint32_t (&key)[R], const Kth& kt, int K, int* wsum, bool (&take)[R]) {
  const int need_eq = K - kt.n_lt;  // ties to take (<= n_eq)
  if (kt.tau == kInf32) {
#pragma unroll
    for (int r = 0; r < R; r++) take[r] = key[r] != kInf32;
    return;
  }
  if (need_eq >= kt.n_eq) {  // block-uniform: all ties are wanted
#pragma unroll
    for (int r = 0; r < R; r++) take[r] = key[r] <= kt.tau;
    return;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int mine = 0;
#pragma unroll
  for (int r = 0; r < R; r++) mine += key[r] == kt.tau;
  int inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(kFull, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  int rank = inc - mine;
  for (int w = 0; w < warp; w++) rank += wsum[w];
#pragma unroll
  for (int r = 0; r < R; r++) {
    const bool eq = key[r] == kt.tau;
    take[r] = key[r] < kt.tau || (eq && rank < need_eq);
    rank += eq;
  }
  __syncthreads();
}

// take_k for keys held STRIDED: key[r] of thread t is index r * NT + t (adjacent threads own adjacent indices, so the
// loads behind the keys coalesce and every thread has work when fewer than R * NT indices exist).  Same rule: key < tau,
// plus the lowest-index ties.  wsum: 8 ints (shared).
template <int R>
__device__ __forceinline__ void take_k_strided(const uint32_t (&key)[R], const Kth& kt, int K, int* wsum, bool (&take)[R]) {
  const int need_eq = K - kt.n_lt;  // ties to take (<= n_eq)
  if (kt.tau == kInf32) {
#pragma unroll
    for (int r = 0; r < R; r++) take[r] = key[r] != kInf32;
    return;
  }
  if (need_eq >= kt.n_eq) {  // block-uniform: all ties are wanted
#pragma unroll
    for (int r = 0; r < R; r++) take[r] = key[r] <= kt.tau;
    return;
  }
  // rare: more ties at the threshold than places left; index order = row r first, then thread
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int before = 0;
#pragma unroll
  for (int r = 0; r < R; r++) {  // (unrolled: key[] and take[] must stay in registers)
    const bool eq = key[r] == kt.tau;
    const unsigned m = __ballot_sync(kFull, eq);
    if (lane == 0) wsum[warp] = __popc(m);
    __syncthreads();
    int rank = before + __popc(m & ((1u << lane) - 1));
    int all = 0;
    for (int w = 0; w < NT / 32; w++) {
      const int c = wsum[w];
      if (w < warp) rank += c;
      all += c;
    }
    take[r] = key[r] < kt.tau || (eq && rank < need_eq);
    before += all;
    __syncthreads();
  }
}

// Ascending bitonic sort of NT = 256 keys, one per thread (unused slots: ~0).  Exchanges at distance < 32 are shuffles, the
// six at distance >= 32 go through xch[NT] (shared).  ~390 instructions per thread where ranking every key against every
// other key costs 5 per pair (1300 at 256 keys: it was 31 % of the line-selection kernel's instructions).  Keys are
// unique, so the result is THE order the rank loop produced.  All threads of the block must call it.
__device__ __forceinline__ uint64_t block_sort256(uint64_t k, uint64_t* xch) {
  const int t = threadIdx.x;
#pragma unroll
  for (int size = 2; size <= NT; size <<= 1) {
    const bool up = (t & size) == 0;
#pragma unroll
    for (int j = size >> 1; j > 0; j >>= 1) {
      uint64_t o;
      if (j >= 32) {
        xch[t] = k;
        __syncthreads();
        o = xch[t ^ j];
        __syncthreads();
      } else {
        o = __shfl_xor_sync(kFull, k, j);
      }
      const bool keep_min = ((t & j) == 0) == up;
      const uint64_t lo = k < o ? k : o, hi = k < o ? o : k;
      k = keep_min ? lo : hi;
    }
  }
  return k;
}

__device__ __forceinline__ uint32_t key32(float v) { return v == v ? f2ord(v) : kInf32; }  // NaN: never selected

struct Smem {  // layout in dynamic shared memory (host and device agree through bytes())
  __host__ __device__ static size_t bytes(int R, int P) {
    return sizeof(uint64_t) * R * NT                 // keys: candidate columns / surviving lines
           + sizeof(float) * 2 * 1024                // t1, t6 of the surviving lines
           + sizeof(int) * 1024                      // list ids of the surviving lines
           + sizeof(int) * (2 * P + 2 * 256 + 64);   // bucket list, top-P, hist, meta / wsum / counters (+ slack)
  }
};

template <int R>
__global__ void __launch_bounds__(NT, R == 8 ? 4 : 2)
coarse_select_lines_fast_kernel(const float* __restrict__ D, int64_t ldD, const float* __restrict__ bmin, int nb, int C,
                                int P, const int* __restrict__ edge, const float* __restrict__ edge_d2, int E, int W,
                                int* __restrict__ out_coarse, int* __restrict__ out_list,
                                float* __restrict__ out_term1, float* __restrict__ out_term6) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(smem);             // [R * NT]
  float* st1 = reinterpret_cast<float*>(keys + (size_t)R * NT);    // [1024]
  float* st6 = st1 + 1024;                                         // [1024]
  int* slist = reinterpret_cast<int*>(st6 + 1024);                 // [1024]
  int* bk_s = slist + 1024;                                        // [P] selected buckets
  int* top_s = bk_s + P;                                           // [P] top-P centroids, ascending
  int* hist = top_s + P;                                           // [256]
  int* meta = hist + 256;                                          // [8]
  int* wsum = meta + 8;                                            // [8]
  int* cnt = wsum + 8;                                             // [4] append cursors
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t q = blockIdx.x;
  const float* Dq = D + q * ldD;
  const float* bq = bmin + q * nb;

  // ---- 1: the P buckets (32 consecutive centroids each) with the smallest minima contain every top-P centroid
  const int Pb = P < nb ? P : nb;
  uint32_t kb[R];
  {
    const int j0 = R * (int)threadIdx.x;
#pragma unroll
    for (int r4 = 0; r4 < R; r4 += 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool in = j0 + r4 + 3 < nb;
      if (in) v = *reinterpret_cast<const float4*>(bq + j0 + r4);
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int r = 0; r < 4; r++) {
        float x = vv[r];
        if (!in) x = j0 + r4 + r < nb ? bq[j0 + r4 + r] : __int_as_float(0x7fc00000);
        kb[r4 + r] = key32(x);
      }
    }
  }
  if (threadIdx.x < 4) cnt[threadIdx.x] = 0;
  const Kth kt1 = kth32<R>(kb, Pb, hist, meta);
  {
    bool take[R];
    take_k<R>(kb, kt1, Pb, wsum, take);
#pragma unroll
    for (int r = 0; r < R; r++)
      if (take[r]) bk_s[atomicAdd(&cnt[0], 1)] = R * (int)threadIdx.x + r;  // <= Pb appends
  }
  __syncthreads();
  const int nbk = cnt[0];
  // ---- 2: candidate columns = entries of the selected buckets not above the P-th bucket minimum (>= P of them)
  // (the bound needs P distinct buckets: with fewer buckets than P every entry of every bucket is a candidate)
  const float tau1 = (kt1.tau == kInf32 || Pb < P) ? __int_as_float(0x7f800000) : ord2f(kt1.tau);
  // A warp requests all of its bucket lines (8 at P = 64) before it looks at the first: the tile has left the L2, and
  // one line at a time cost one DRAM round trip each on the block's critical path.
  constexpr int LB = 8;  // lines in flight per warp
  for (int b0 = warp; b0 < nbk; b0 += LB * (NT / 32)) {
    float v[LB];
    int col[LB];
#pragma unroll
    for (int j = 0; j < LB; j++) {
      const int b = b0 + j * (NT / 32);
      col[j] = b < nbk ? bk_s[b] * 32 + lane : C;
      v[j] = col[j] < C ? Dq[col[j]] : __int_as_float(0x7fc00000);
    }
#pragma unroll
    for (int j = 0; j < LB; j++) {
      const bool pass = v[j] <= tau1;  // NaN never passes
      const unsigned m = __ballot_sync(kFull, pass);
      int base = 0;
      if (lane == 0 && m) base = atomicAdd(&cnt[1], __popc(m));
      base = __shfl_sync(kFull, base, 0);
      if (pass) keys[base + __popc(m & ((1u << lane) - 1))] = make_key(v[j], (uint32_t)col[j]);
    }
  }
  __syncthreads();
  const int nc = cnt[1];  // <= nbk * 32 <= R * NT
  const int Pk = P < C ? P : C;
  // ---- exact top-P: rank of every candidate among the candidates
  for (int i = threadIdx.x; i < P; i += NT) top_s[i] = -1;
  __syncthreads();
  for (int i = threadIdx.x; i < nc; i += NT) {
    const uint64_t mykey = keys[i];
    int rank = 0;
    for (int j = 0; j < nc; j++) rank += keys[j] < mykey;
    if (rank < Pk) top_s[rank] = (int)key_payload(mykey);
  }
  __syncthreads();
  if (out_coarse)
    for (int i = threadIdx.x; i < P; i += NT) out_coarse[q * P + i] = top_s[i];

  // ---- 3: the W best of the P*E lines (BroadcastSum.cu:505-552); thread t scores the lines [R t, R t + R)
  // All R lines' loads are issued before the first score: the IEEE division has a branchy slow path that the compiler
  // does not move loads across, so a fused loop waited out two dependent round trips (edge from L2, then the
  // neighbour's column of D from DRAM) per line, 2 R in a row on the block's critical path.
  const int num = P * E;
  uint32_t kl[R];
  float a2r[R], b2r[R], c2r[R];
  int lid[R], sr[R];
  int cq = R * (int)threadIdx.x / E, ce = R * (int)threadIdx.x % E;  // line R t + r = edge ce of top-P slot cq
#pragma unroll
  for (int r = 0; r < R; r++) {
    lid[r] = -1;
    a2r[r] = b2r[r] = c2r[r] = 0.f;
    if (R * (int)threadIdx.x + r < num) {
      const int c = top_s[cq];
      if (c >= 0) {
        lid[r] = c * E + ce;
        sr[r] = edge[lid[r]];
        b2r[r] = Dq[c];
        c2r[r] = edge_d2[lid[r]];
      }
    }
    if (++ce == E) {
      ce = 0;
      cq++;
    }
  }
#pragma unroll
  for (int r = 0; r < R; r++)
    if (lid[r] >= 0) a2r[r] = Dq[sr[r]];
#pragma unroll
  for (int r = 0; r < R; r++) {
    kl[r] = kInf32;
    if (lid[r] >= 0) {
      const float a2 = a2r[r], b2 = b2r[r], c2 = c2r[r];
      float v = __fsub_rn(a2, b2);
      v = __fsub_rn(v, c2);
      // BroadcastSum.cu:517: (v>0) ? b2 : b2 - 0.25 v^2 / c2
      const float score = (v > 0.f) ? b2 : __fsub_rn(b2, __fdiv_rn(__fmul_rn(__fmul_rn(0.25f, v), v), c2));
      kl[r] = key32(score);
    }
  }
  const Kth kt3 = kth32<R>(kl, W, hist, meta);
  {
    bool take[R];
    take_k<R>(kl, kt3, W, wsum, take);
#pragma unroll
    for (int r = 0; r < R; r++) {
      if (take[r]) {
        const int slot = atomicAdd(&cnt[2], 1);  // <= W appends
        // order = (score, line index); the slot rides in the low 10 bits (line index < 4096, slot < 1024)
        keys[slot] = ((uint64_t)kl[r] << 32) | ((uint32_t)(R * (int)threadIdx.x + r) << 10) | (uint32_t)slot;
        st1[slot] = b2r[r];
        st6[slot] = __fsub_rn(a2r[r], b2r[r]);
        slist[slot] = lid[r];
      }
    }
  }
  for (int w = threadIdx.x; w < W; w += NT) {  // slots the ranks below do not reach
    out_list[q * W + w] = -1;
    out_term1[q * W + w] = 0.f;
    out_term6[q * W + w] = 0.f;
  }
  __syncthreads();
  const int ns = cnt[2];
  if (ns > 128 && ns <= NT) {  // block-uniform: one key per thread, bitonic sort (cheaper than ranking from 128 keys on)
    uint64_t mykey = (int)threadIdx.x < ns ? keys[threadIdx.x] : ~0ull;
    __syncthreads();  // keys[] becomes the exchange buffer
    mykey = block_sort256(mykey, keys);
    if ((int)threadIdx.x < ns) {
      const int slot = (int)(mykey & 1023u);
      out_list[q * W + threadIdx.x] = slist[slot];
      out_term1[q * W + threadIdx.x] = st1[slot];
      out_term6[q * W + threadIdx.x] = st6[slot];
    }
    return;
  }
  for (int i = threadIdx.x; i < ns; i += NT) {
    const uint64_t mykey = keys[i];
    int rank = 0;
    for (int j = 0; j < ns; j++) rank += keys[j] < mykey;
    out_list[q * W + rank] = slist[i];
    out_term1[q * W + rank] = st1[i];
    out_term6[q * W + rank] = st6[i];
  }
}

// ------------------------------------------------------------------------------------------------------------------
// The same selection WITHOUT a distance matrix (north_star: "stop materialising D").  The tensor-core sweep emits only
// the bucket minima (l2_tc_kernel<2>); the few hundred columns a query really needs -- the 32 columns of each of its P
// best buckets and the P*E neighbour centroids of its top-P -- are re-evaluated here in fp32 from the centroid table,
// which (C * d * 4 = 32 MiB at C2) stays L2-resident because nothing streams a gigabyte of D through the L2 any more.
//   per query: (32 P + P E) rows of d floats from L2 instead of 4 C bytes written + ~(P + P E) random DRAM sectors read.
// Every distance is produced by the same routine (dot8: fixed summation tree, independent of the row's slot), so
// D[c] of a centroid that is both a top-P centroid and somebody's neighbour is one number, as with a stored matrix.

// 8 rows at once: p[r] = this lane's share of x . row_r; afterwards every lane of a quad holds the complete sum of row
// ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1)      (9 shuffles for 8 rows)
__device__ __forceinline__ float reduce8(float (&p)[8], int lane) {
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
  float a[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const float send = b4 ? p[j] : p[j + 4];
    const float keep = b4 ? p[j + 4] : p[j];
    a[j] = keep + __shfl_xor_sync(kFull, send, 16);
  }
  float b[2];
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const float send = b3 ? a[j] : a[j + 2];
    const float keep = b3 ? a[j + 2] : a[j];
    b[j] = keep + __shfl_xor_sync(kFull, send, 8);
  }
  const float send = b2 ? b[0] : b[1];
  const float keep = b2 ? b[1] : b[0];
  float c = keep + __shfl_xor_sync(kFull, send, 4);
  c += __shfl_xor_sync(kFull, c, 2);
  c += __shfl_xor_sync(kFull, c, 1);
  return c;
}
__device__ __forceinline__ int reduce8_row(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }

// x . row for 8 rows; qv = the lane's 4 query components (zero beyond d), act = lane * 4 < d
__device__ __forceinline__ float dot8(const float* __restrict__ cent, int d, const int (&rows)[8], const float4& qv,
                                      bool act, int lane) {
  float p[8];
  float4 c[8];
#pragma unroll
  for (int r = 0; r < 8; r++) {
    c[r] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (act) c[r] = __ldg(reinterpret_cast<const float4*>(cent + (size_t)rows[r] * d) + lane);
  }
#pragma unroll
  for (int r = 0; r < 8; r++) p[r] = fmaf(c[r].w, qv.w, fmaf(c[r].z, qv.z, fmaf(c[r].y, qv.y, c[r].x * qv.x)));
  return reduce8(p, lane);
}

struct SmemExact {
  __host__ __device__ static size_t bytes(int R, int P) {
    return Smem::bytes(R, P) + sizeof(float) * ((size_t)R * NT + P);  // + distances of the candidates / lines, top-P values
  }
};

__host__ __device__ inline bool exact_supported(int d, int nb, int P, int E, int W) {
  const int need = nb > P * E ? (nb > P * 32 ? nb : P * 32) : (P * E > P * 32 ? P * E : P * 32);
  return d >= 4 && d <= 128 && d % 4 == 0 && need <= 16 * NT && W <= 1024 && nb % 4 == 0;
}

template <int R>
__global__ void __launch_bounds__(NT, R == 8 ? 4 : 2)
coarse_select_lines_exact_kernel(const float* __restrict__ xq, int d, const float* __restrict__ cent,
                                 const float* __restrict__ cnorm, const float* __restrict__ bmin, int nb, int C, int P,
                                 const int* __restrict__ edge, const float* __restrict__ edge_d2, int E, int W,
                                 int* __restrict__ out_coarse, int* __restrict__ out_list,
                                 float* __restrict__ out_term1, float* __restrict__ out_term6) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(smem);             // [R * NT]
  float* st1 = reinterpret_cast<float*>(keys + (size_t)R * NT);    // [1024]
  float* st6 = st1 + 1024;                                         // [1024]
  int* slist = reinterpret_cast<int*>(st6 + 1024);                 // [1024]
  int* bk_s = slist + 1024;                                        // [P] selected buckets
  int* top_s = bk_s + P;                                           // [P] top-P centroids, ascending
  int* hist = top_s + P;                                           // [256]
  int* meta = hist + 256;                                          // [8]
  int* wsum = meta + 8;                                            // [8]
  int* cnt = wsum + 8;                                             // [4] append cursors, [3] = bound of the candidates
  float* fbuf = reinterpret_cast<float*>(smem + Smem::bytes(R, P));  // [R * NT] candidate / line distances
  float* top_v = fbuf + (size_t)R * NT;                            // [P] distances of the top-P centroids
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t q = blockIdx.x;
  const float* bq = bmin + q * nb;
  const bool act = lane * 4 < d;
  float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (act) qv = __ldg(reinterpret_cast<const float4*>(xq + q * d) + lane);

  // ---- 1: the P buckets (32 consecutive centroids each) with the smallest minima (tensor-core values)
  const int Pb = P < nb ? P : nb;
  {
    uint32_t kb[R];
    const int j0 = R * (int)threadIdx.x;
#pragma unroll
    for (int r4 = 0; r4 < R; r4 += 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool in = j0 + r4 + 3 < nb;
      if (in) v = *reinterpret_cast<const float4*>(bq + j0 + r4);
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int r = 0; r < 4; r++) {
        float x = vv[r];
        if (!in) x = j0 + r4 + r < nb ? bq[j0 + r4 + r] : __int_as_float(0x7fc00000);
        kb[r4 + r] = key32(x);
      }
    }
    if (threadIdx.x < 4) cnt[threadIdx.x] = 0;
    const Kth kt1 = kth32<R>(kb, Pb, hist, meta);
    bool take[R];
    take_k<R>(kb, kt1, Pb, wsum, take);
#pragma unroll
    for (int r = 0; r < R; r++)
      if (take[r]) bk_s[atomicAdd(&cnt[0], 1)] = R * (int)threadIdx.x + r;  // <= Pb appends
  }
  __syncthreads();
  const int nbk = cnt[0];
  // ---- 2: exact distances of the 32 columns of every selected bucket; warp <- groups of 8 consecutive rows
  for (int g = warp; g < nbk * 4; g += NT / 32) {
    const int c0 = bk_s[g >> 2] * 32 + (g & 3) * 8;
    int rows[8];
#pragma unroll
    for (int r = 0; r < 8; r++) rows[r] = min(c0 + r, C - 1);
    const float dot = dot8(cent, d, rows, qv, act, lane);
    if ((lane & 3) == 0) {
      const int r = reduce8_row(lane), c = c0 + r;
      fbuf[(g >> 2) * 32 + (g & 3) * 8 + r] = c < C ? fmaf(-2.f, dot, __ldg(cnorm + c)) : __int_as_float(0x7fc00000);
    }
  }
  __syncthreads();
  // bound: the largest exact bucket minimum.  The P minima are P different columns, so the P-th smallest candidate
  // cannot be above it (with fewer buckets than P every column of every bucket is a candidate).
  for (int i = threadIdx.x; i < nbk * 32; i += NT) {  // NT is a multiple of 32: a warp covers one bucket
    const uint32_t mk = __reduce_min_sync(kFull, key32(fbuf[i]));
    if (lane == 0) atomicMax(reinterpret_cast<unsigned*>(&cnt[3]), mk);
  }
  __syncthreads();
  const uint32_t tau1 = Pb < P ? kInf32 : (uint32_t)cnt[3];
  for (int i = threadIdx.x; i < nbk * 32; i += NT) {
    const float v = fbuf[i];
    const uint32_t kv = key32(v);
    const bool pass = kv != kInf32 && kv <= tau1;
    const unsigned m = __ballot_sync(kFull, pass);
    int base = 0;
    if (lane == 0 && m) base = atomicAdd(&cnt[1], __popc(m));
    base = __shfl_sync(kFull, base, 0);
    if (pass) keys[base + __popc(m & ((1u << lane) - 1))] = make_key(v, (uint32_t)(bk_s[i >> 5] * 32 + (i & 31)));
  }
  __syncthreads();
  const int nc = cnt[1];  // <= nbk * 32 <= R * NT
  const int Pk = P < C ? P : C;
  // ---- exact top-P: rank of every candidate among the candidates
  for (int i = threadIdx.x; i < P; i += NT) top_s[i] = -1;
  __syncthreads();
  for (int i = threadIdx.x; i < nc; i += NT) {
    const uint64_t mykey = keys[i];
    int rank = 0;
    for (int j = 0; j < nc; j++) rank += keys[j] < mykey;
    if (rank < Pk) {
      top_s[rank] = (int)key_payload(mykey);
      top_v[rank] = key_val(mykey);
    }
  }
  __syncthreads();
  if (out_coarse)
    for (int i = threadIdx.x; i < P; i += NT) out_coarse[q * P + i] = top_s[i];

  // ---- 3a: exact distances of the P*E neighbour centroids (line i = centroid i / E, edge i % E)
  const int num = P * E;
  for (int g = warp; g * 8 < num; g += NT / 32) {
    int rows[8];
    int sid = -1;  // lane 4 r' of the quad that ends up with row r' keeps its neighbour id
#pragma unroll
    for (int r = 0; r < 8; r++) {
      const int i = g * 8 + r;
      int s = -1;
      if (i < num) {
        const int c = top_s[i / E];
        if (c >= 0) s = __ldg(edge + (int64_t)c * E + (i % E));
      }
      if (s >= C) s = -1;
      rows[r] = s < 0 ? 0 : s;
      if (r == reduce8_row(lane)) sid = s;
    }
    const float dot = dot8(cent, d, rows, qv, act, lane);
    if ((lane & 3) == 0) {
      const int i = g * 8 + reduce8_row(lane);
      if (i < num) fbuf[i] = sid >= 0 ? fmaf(-2.f, dot, __ldg(cnorm + sid)) : __int_as_float(0x7fc00000);
    }
  }
  __syncthreads();
  // ---- 3b: the W best of the P*E lines (BroadcastSum.cu:505-552); thread t scores the lines [R t, R t + R)
  uint32_t kl[R];
  float a2r[R], b2r[R];
  int lid[R];
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int i = R * (int)threadIdx.x + r;
    kl[r] = kInf32;
    a2r[r] = b2r[r] = 0.f;
    lid[r] = -1;
    if (i < num) {
      const int c = top_s[i / E];
      if (c >= 0) {
        const int e = i % E;
        const float a2 = fbuf[i], b2 = top_v[i / E], c2 = edge_d2[(int64_t)c * E + e];
        float v = __fsub_rn(a2, b2);
        v = __fsub_rn(v, c2);
        // BroadcastSum.cu:517: (v>0) ? b2 : b2 - 0.25 v^2 / c2
        const float score = (v > 0.f) ? b2 : __fsub_rn(b2, __fdiv_rn(__fmul_rn(__fmul_rn(0.25f, v), v), c2));
        kl[r] = key32(score);
        a2r[r] = a2;
        b2r[r] = b2;
        lid[r] = c * E + e;
      }
    }
  }
  const Kth kt3 = kth32<R>(kl, W, hist, meta);
  {
    bool take[R];
    take_k<R>(kl, kt3, W, wsum, take);
#pragma unroll
    for (int r = 0; r < R; r++) {
      if (take[r]) {
        const int slot = atomicAdd(&cnt[2], 1);  // <= W appends
        keys[slot] = ((uint64_t)kl[r] << 32) | (uint32_t)(R * (int)threadIdx.x + r);
        st1[slot] = b2r[r];
        st6[slot] = __fsub_rn(a2r[r], b2r[r]);
        slist[slot] = lid[r];
      }
    }
  }
  for (int w = threadIdx.x; w < W; w += NT) {  // slots the ranks below do not reach
    out_list[q * W + w] = -1;
    out_term1[q * W + w] = 0.f;
    out_term6[q * W + w] = 0.f;
  }
  __syncthreads();
  const int ns = cnt[2];
  for (int i = threadIdx.x; i < ns; i += NT) {
    const uint64_t mykey = keys[i];
    int rank = 0;
    for (int j = 0; j < ns; j++) rank += keys[j] < mykey;
    out_list[q * W + rank] = slist[i];
    out_term1[q * W + rank] = st1[i];
    out_term6[q * W + rank] = st6[i];
  }
}

}  // namespace csl
}  // namespace vlq
