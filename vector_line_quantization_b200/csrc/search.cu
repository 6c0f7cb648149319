// Query-time kernels (SURVEY.md 8a rows a4, a11-a16).
//
//  select_lines_kernel        : one CTA per query; scores the P*E lines of the probed centroids from the coarse matrix D
//                               and keeps the W best (exact block top-k).                 [BroadcastSum.cu:477-560]
//  coarse_select_lines_kernel : the same fused with the exact top-P (through 32-column bucket minima of D).
//                                                                        [Distance.cu:233-383, L2Select.cu:124-165]
//  term3_reg_kernel / term3_kernel : per-query tables -2 q_m.p_mj for a batch of queries.     [IVFPQ.cu:1398-1432]
//  scan_topk_kernel<M, LONG>  : one CTA per query, block-synchronous; LONG = false walks the selected lists as ONE
//                               flattened entry stream (5-entry and 1000-entry lists use the lanes equally), LONG = true
//                               gives every warp whole lists.  16-byte code loads, distance from the per-entry kappa
//                               and the per-line scalars, fused exact top-k -- no intermediate distance array, no
//                               term-2 tables.                 [PQScanMultiPassPrecomputed.cu:675-881, IVFUtils*.cu]
//  scan_async_kernel<M, SKEW> : warp-autonomous scan for long lists (own top-k per warp, software-pipelined chunks);
//                               SKEW = bank-conflict-free table layout (see the comment above the kernel).
//  merge_topk_kernel          : one CTA per query over the [R][nq][k] all-gather layout, or gathering the shards'
//                               results itself from peer-mapped memory.                 [GpuIndexIVFPQ.cu:1467-1518]
//  knn_graph                  : tiled C x C coarse matrix + top-(E+1) + drop rank 0.     [GpuIndexFlat.cu:869-893]
#include <cfloat>
#include <cstdlib>

#include "scan.cuh"
#include "topk.cuh"
#include "coarse_select.cuh"

#include <type_traits>

namespace vlq {

constexpr int Q_THREADS = 256;

// ------------------------------------------------------------------------------------------------ line selection
constexpr int Q_BATCH = 4;

__global__ void __launch_bounds__(Q_THREADS)
select_lines_kernel(const float* __restrict__ D, int64_t ldD, const int* __restrict__ coarse_ids, int P,
                    const int* __restrict__ edge, const float* __restrict__ edge_d2, int E, int W, int cap,
                    int* __restrict__ out_list, float* __restrict__ out_term1, float* __restrict__ out_term6) {
  extern __shared__ __align__(16) unsigned char smem[];
  BlockSelect<Q_THREADS> sel;
  sel.init(smem, W, cap, Q_BATCH);
  const int64_t q = blockIdx.x;
  const float* Dq = D + q * ldD;
  const int* cq = coarse_ids + q * P;
  const int num = P * E;
  for (int base = 0; base < num; base += Q_BATCH * Q_THREADS) {
    bool any = false;
#pragma unroll
    for (int b = 0; b < Q_BATCH; b++) {
      const int i = base + b * Q_THREADS + threadIdx.x;
      bool valid = i < num;
      float score = 0.f;
      if (valid) {
        const int c = cq[i / E];
        valid = c >= 0;
        if (valid) {
          const int e = i % E;
          const int s = edge[(int64_t)c * E + e];
          const float a2 = Dq[s], b2 = Dq[c], c2 = edge_d2[(int64_t)c * E + e];
          float v = __fsub_rn(a2, b2);
          v = __fsub_rn(v, c2);
          // BroadcastSum.cu:517: (v>0) ? b2 : b2 - 0.25 v^2 / c2
          score = (v > 0.f) ? b2 : __fsub_rn(b2, __fdiv_rn(__fmul_rn(__fmul_rn(0.25f, v), v), c2));
        }
      }
      any |= sel.offer_f(valid, score, (uint32_t)i);
    }
    sel.end_batch(any);
  }
  sel.finish();
  for (int w = threadIdx.x; w < W; w += Q_THREADS) {
    const uint64_t key = sel.keys[w];
    int list = -1;
    float t1 = 0.f, t6 = 0.f;
    if (key != kKeyInf) {
      const int i = (int)key_payload(key);
      const int c = cq[i / E], e = i % E;
      const int s = edge[(int64_t)c * E + e];
      list = c * E + e;
      t1 = Dq[c];
      t6 = __fsub_rn(Dq[s], Dq[c]);
    }
    out_list[q * W + w] = list;
    out_term1[q * W + w] = t1;
    out_term6[q * W + w] = t6;
  }
}

// ------------------------------------------------------------------------------------------------ fused top-P + lines
// a11 + a12 in one CTA per query, driven by the bucket minima the GEMM epilogue emits (vlq_l2_distances_tc):
//   1. the P buckets (32 consecutive centroids each) with the smallest minima contain every top-P centroid,
//   2. exact top-P among those P*32 entries of D (one 128-byte line per bucket instead of the whole 4*C-byte row),
//   3. line scoring of the P*E lines and top-W, as select_lines_kernel.
// i / E and i % E for the (line = centroid slot * E + edge) enumeration; E is a power of two in every driver config
struct EdgeDiv {
  int E, shift;
  __device__ __forceinline__ explicit EdgeDiv(int E_) : E(E_), shift(-1) {
    if ((E_ & (E_ - 1)) == 0) {
      shift = 0;
      while ((1 << shift) < E_) shift++;
    }
  }
  __device__ __forceinline__ int div(int i) const { return shift >= 0 ? (i >> shift) : (i / E); }
  __device__ __forceinline__ int mod(int i) const { return shift >= 0 ? (i & (E - 1)) : (i % E); }
};

__global__ void __launch_bounds__(Q_THREADS)
coarse_select_lines_kernel(const float* __restrict__ D, int64_t ldD, const float* __restrict__ bmin, int nb, int C,
                           int P, const int* __restrict__ edge, const float* __restrict__ edge_d2, int E, int W, int cap,
                           int* __restrict__ out_coarse, int* __restrict__ out_list, float* __restrict__ out_term1,
                           float* __restrict__ out_term6) {
  extern __shared__ __align__(16) unsigned char smem[];
  int* bk_s = reinterpret_cast<int*>(smem + ((select_smem_bytes(cap) + 15) & ~size_t(15)));  // [1024] bucket ids
  int* cq_s = bk_s + VLQ_MAX_K;                                                              // [1024] top-P centroids
  BlockSelect<Q_THREADS> sel;
  const EdgeDiv ed(E);
  const int64_t q = blockIdx.x;
  const float* Dq = D + q * ldD;
  const float* bq = bmin + q * nb;
  // ---- 1: P smallest bucket minima
  const int Pb = P < nb ? P : nb;
  sel.init(smem, Pb, cap, Q_BATCH);
  bool direct = false;
  if (nb <= cap) {  // block-uniform: every candidate fits the buffer, see BlockSelect::put
    bool bad = false;
    for (int j = threadIdx.x; j < nb; j += Q_THREADS) bad |= sel.put(j, true, bq[j], (uint32_t)j);
    direct = sel.placed(nb, bad);
    if (!direct) sel.init(smem, Pb, cap, Q_BATCH);
  }
  if (!direct) {
    for (int base = 0; base < nb; base += Q_BATCH * Q_THREADS) {
      float v[Q_BATCH];
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) {
        const int j = base + b * Q_THREADS + threadIdx.x;
        v[b] = j < nb ? bq[j] : 0.f;
      }
      bool any = false;
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) {
        const int j = base + b * Q_THREADS + threadIdx.x;
        any |= sel.offer_f(j < nb, v[b], (uint32_t)j);
      }
      sel.end_batch(any);
    }
  }
  sel.finish(false);  // only the set of buckets matters
  for (int i = threadIdx.x; i < Pb; i += Q_THREADS) {
    const uint64_t key = sel.keys[i];
    bk_s[i] = key != kKeyInf ? (int)key_payload(key) : -1;
  }
  __syncthreads();
  // ---- 2: exact top-P among the candidate buckets
  const int Pk = P < C ? P : C;
  sel.init(smem, Pk, cap, Q_BATCH);
  const int ncand = Pb * 32;
  auto cand2 = [&](int i, int& col, float& v) {  // candidate i: column (i & 31) of bucket slot i >> 5
    col = -1;
    v = 0.f;
    const int bk = bk_s[i >> 5];
    const int c = bk * 32 + (i & 31);
    if (bk >= 0 && c < C) {
      col = c;
      v = Dq[c];
    }
  };
  direct = false;
  if (ncand <= cap) {
    bool bad = false;
    for (int i = threadIdx.x; i < ncand; i += Q_THREADS) {
      int col;
      float v;
      cand2(i, col, v);
      bad |= sel.put(i, col >= 0, v, (uint32_t)col);
    }
    direct = sel.placed(ncand, bad);
    if (!direct) sel.init(smem, Pk, cap, Q_BATCH);
  }
  if (!direct) {
    for (int base = 0; base < ncand; base += Q_BATCH * Q_THREADS) {
      float v[Q_BATCH];
      int col[Q_BATCH];
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) {
        const int i = base + b * Q_THREADS + threadIdx.x;
        col[b] = -1;
        v[b] = 0.f;
        if (i < ncand) cand2(i, col[b], v[b]);
      }
      bool any = false;
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) any |= sel.offer_f(col[b] >= 0, v[b], (uint32_t)col[b]);
      sel.end_batch(any);
    }
  }
  sel.finish();
  for (int i = threadIdx.x; i < P; i += Q_THREADS) {
    const uint64_t key = i < Pk ? sel.keys[i] : kKeyInf;
    const int c = key != kKeyInf ? (int)key_payload(key) : -1;
    cq_s[i] = c;
    if (out_coarse) out_coarse[q * P + i] = c;
  }
  __syncthreads();
  // ---- 3: the W best of the P*E lines (BroadcastSum.cu:505-552)
  sel.init(smem, W, cap, Q_BATCH);
  const int num = P * E;
  auto cand3 = [&](int i, bool& valid, float& score) {  // line i = (centroid slot i / E, edge i % E)
    score = 0.f;
    const int c = cq_s[ed.div(i)];
    valid = c >= 0;
    if (valid) {
      const int e = ed.mod(i);
      const int s = edge[(int64_t)c * E + e];
      const float a2 = Dq[s], b2 = Dq[c], c2 = edge_d2[(int64_t)c * E + e];
      float v = __fsub_rn(a2, b2);
      v = __fsub_rn(v, c2);
      score = (v > 0.f) ? b2 : __fsub_rn(b2, __fdiv_rn(__fmul_rn(__fmul_rn(0.25f, v), v), c2));
    }
  };
  direct = false;
  if (num <= cap) {
    bool bad = false;
    for (int i = threadIdx.x; i < num; i += Q_THREADS) {
      bool valid;
      float score;
      cand3(i, valid, score);
      bad |= sel.put(i, valid, score, (uint32_t)i);
    }
    direct = sel.placed(num, bad);
    if (!direct) sel.init(smem, W, cap, Q_BATCH);
  }
  if (!direct) {
    for (int base = 0; base < num; base += Q_BATCH * Q_THREADS) {
      bool any = false;
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) {
        const int i = base + b * Q_THREADS + threadIdx.x;
        bool valid = false;
        float score = 0.f;
        if (i < num) cand3(i, valid, score);
        any |= sel.offer_f(valid, score, (uint32_t)i);
      }
      sel.end_batch(any);
    }
  }
  sel.finish();
  for (int w = threadIdx.x; w < W; w += Q_THREADS) {
    const uint64_t key = sel.keys[w];
    int list = -1;
    float t1 = 0.f, t6 = 0.f;
    if (key != kKeyInf) {
      const int i = (int)key_payload(key);
      const int c = cq_s[ed.div(i)], e = ed.mod(i);
      const int s = edge[(int64_t)c * E + e];
      list = c * E + e;
      t1 = Dq[c];
      t6 = __fsub_rn(Dq[s], Dq[c]);
    }
    out_list[q * W + w] = list;
    out_term1[q * W + w] = t1;
    out_term6[q * W + w] = t6;
  }
}

// ------------------------------------------------------------------------------------------------ scan + top-k
// LONG = false: the selected lists are walked as ONE flattened entry stream (lists of a handful of entries keep all
//               lanes busy);  LONG = true: every warp owns whole lists (slot w -> warp w % 8) and strides their entries,
//               so the per-list scalars are warp-uniform and nothing has to be searched per entry.
template <int M_T, bool LONG>
__global__ void __launch_bounds__(Q_THREADS, M_T == 16 ? 3 : 2) scan_topk_kernel(ScanArgs a) {  // 3 CTAs per SM (80 registers); measured at C2 before the strided small-query path: 0.86 ms per 10 k queries, 2 CTAs 1.03, 4 CTAs (spills) 1.63 -- now 0.57
  extern __shared__ __align__(16) unsigned char smem[];
  // smem: [topk keys S*8 + 16][T3 M*ksub f32][lambda nL f32][per line: start i64, prefix i32 (W+1), t1, t6, t5 f32]
  const int M = a.M, ksub = a.ksub, dsub = a.dsub, W = a.W;
  BlockSelect<Q_THREADS> sel;
  size_t off = (select_smem_bytes(a.sel_cap) + 15) & ~size_t(15);
  float* T3 = reinterpret_cast<float*>(smem + off);
  off += sizeof(float) * M * ksub;
  float* lcb = reinterpret_cast<float*>(smem + off);
  off += sizeof(float) * ((a.nL + 3) & ~3);
  int64_t* lstart = reinterpret_cast<int64_t*>(smem + off);
  off += sizeof(int64_t) * W;
  int* prefix = reinterpret_cast<int*>(smem + off);
  off += sizeof(int) * ((W + 1 + 3) & ~3);
  float* lt1 = reinterpret_cast<float*>(smem + off);
  off += sizeof(float) * W;
  float* lt6 = reinterpret_cast<float*>(smem + off);
  off += sizeof(float) * W;
  float* lt5 = reinterpret_cast<float*>(smem + off);
  off += sizeof(float) * W;
  uint16_t* owner = reinterpret_cast<uint16_t*>(smem + off);  // [owner_cap] line slot of every stream position

  sel.init(smem, a.k, a.sel_cap, LONG ? 2 : Q_BATCH);
  const int64_t qi = blockIdx.x;
  const float* qv = a.q + qi * a.d;

  // term3 table: T3[m][j] = -2 q_m . p_mj            (gpu/impl/IVFPQ.cu:1409-1432)
  if (a.t3) {  // precomputed by term3_kernel (PQ codebook read once per CTA there instead of once per query here)
    const float4* src = reinterpret_cast<const float4*>(a.t3 + (size_t)qi * M * ksub);
    float4* dst = reinterpret_cast<float4*>(T3);
    for (int i = threadIdx.x; i < (M * ksub) / 4; i += Q_THREADS) dst[i] = src[i];
  } else
  for (int i = threadIdx.x; i < M * ksub; i += Q_THREADS) {
    const int m = i / ksub;
    const float* p = a.pq + (size_t)i * dsub;
    const float* qm = qv + m * dsub;
    float ip = 0.f;
    for (int t = 0; t < dsub; t++) ip = fmaf(qm[t], p[t], ip);
    T3[i] = -2.f * ip;
  }
  for (int i = threadIdx.x; i < a.nL; i += Q_THREADS) lcb[i] = a.lambda_cb[i];
  // line descriptors (lengths capped like gpu/impl/IVFUtils.cu:87)
  for (int w = threadIdx.x; w < W; w += Q_THREADS) {
    const int list = a.line_list[qi * W + w];
    int len = 0;
    int64_t st = 0;
    float t5 = 0.f;
    if (list >= 0) {
      st = a.offsets[list];
      int64_t l = a.offsets[list + 1] - st;
      len = (int)(l < a.cap ? l : a.cap);
      t5 = a.edge_d2 ? a.edge_d2[list] : 0.f;
    }
    lstart[w] = st;
    prefix[w + 1] = len;  // turned into an inclusive scan below
    lt1[w] = a.term1[qi * W + w];
    lt6[w] = a.term6[qi * W + w];
    lt5[w] = t5;
  }
  if (threadIdx.x == 0) prefix[0] = 0;
  __syncthreads();
  if (threadIdx.x < kWarp) {  // W <= 1024: one warp scans 32 chunks
    const int lane = threadIdx.x;
    const int chunk = (W + kWarp - 1) / kWarp;
    const int b = lane * chunk, e = min(W, b + chunk);
    int s = 0;
    for (int w = b; w < e; w++) s += prefix[w + 1];
    int inc = s;
#pragma unroll
    for (int o = 1; o < kWarp; o <<= 1) {
      int t = __shfl_up_sync(kFull, inc, o);
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
  if (LONG) {
    constexpr int NW = Q_THREADS / 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int* rounds_s = reinterpret_cast<int*>(owner);  // scratch (the owner table is unused in this mode)
    if (threadIdx.x == 0) *rounds_s = 0;
    __syncthreads();
    int mine = 0;  // 64-entry rounds this warp needs for its lists
    for (int w = warp + NW * lane; w < W; w += NW * 32) mine += (prefix[w + 1] - prefix[w] + 63) >> 6;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(kFull, mine, o);
    if (lane == 0) atomicMax(rounds_s, mine);
    __syncthreads();
    const int rounds = *rounds_s;
    int li = warp, off_ = 0;
    for (int r = 0; r < rounds; r++) {
      bool any = false;
      while (li < W && off_ >= prefix[li + 1] - prefix[li]) {  // warp-uniform: next non-exhausted list
        li += NW;
        off_ = 0;
      }
      if (li < W) {
        const int p0 = prefix[li], len = prefix[li + 1] - p0;
        const int64_t st = lstart[li];
        const float t1 = lt1[li], t6 = lt6[li], t5 = lt5[li];
        CodeRegs<M_T> cr[2];
        uint8_t lq[2];
        float kp[2];
#pragma unroll
        for (int u = 0; u < 2; u++) {
          const int e = off_ + u * 32 + lane;
          lq[u] = 0;
          kp[u] = 0.f;
          if (e < len) {
            const int64_t ent = st + e;
            cr[u].load(a.codes + ent * M, e);
            lq[u] = a.lamq[ent];
            kp[u] = a.kappa[ent];
          }
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
          const int e = off_ + u * 32 + lane;
          const bool valid = e < len;
          float dist = 0.f;
          if (valid) {
            const float la = lcb[lq[u]];
            const float base_d = t1 + la * t6 + (la * la - la) * t5;
            dist = (kp[u] + cr[u].adc(T3, M, ksub)) + base_d;
          }
          any |= sel.offer_f(valid, dist, (uint32_t)(p0 + e));
        }
        off_ += 64;
      }
      sel.end_batch(any);
    }
  }
  const bool use_owner = !LONG && total <= a.owner_cap;  // block-uniform
  if (use_owner) {  // each line writes its slot over its own range of stream positions (lists are short here)
    for (int w = threadIdx.x; w < W; w += Q_THREADS)
      for (int p = prefix[w]; p < prefix[w + 1]; p++) owner[p] = (uint16_t)w;
    __syncthreads();
  }

  // ---- small queries (a few thousand entries in all, the C2 regime): every distance of the query fits in registers,
  // kSmallR per thread, so the selection is ONE register-resident radix threshold (csl::kth32, coarse_select.cuh) +
  // a rank ordering of the k survivors instead of the append / compact / sort machinery of BlockSelect, which was 80 %
  // of this kernel's instructions at 2.7 k entries per query.  Ties resolve to the lowest stream position exactly as in
  // the general path (take_k_strided); same arithmetic, same bits.
  constexpr int kSmallR = 16, kSmallB = 4;
  if (!LONG && use_owner && !a.no_small && total <= kSmallR * Q_THREADS && a.k <= a.sel_cap) {  // block-uniform
    // stream position of key[r] = r * Q_THREADS + t: adjacent threads read adjacent entries of a list, every thread has
    // work (a C2 query has ~1800 entries: 7 rows of 256), and the loads of kSmallB rows are in flight together
    uint32_t key[kSmallR];
#pragma unroll
    for (int r = 0; r < kSmallR; r++) key[r] = csl::kInf32;
#pragma unroll
    for (int r0 = 0; r0 < kSmallR; r0 += kSmallB) {
      if (r0 * Q_THREADS >= total) break;  // block-uniform
      CodeRegs<M_T> cr[kSmallB];
      uint8_t lq[kSmallB];
      float kp[kSmallB];
      int lo_[kSmallB];
#pragma unroll
      for (int u = 0; u < kSmallB; u++) {
        const int pos = (r0 + u) * Q_THREADS + (int)threadIdx.x;
        lq[u] = 0;
        kp[u] = 0.f;
        lo_[u] = 0;
        if (pos < total) {
          const int lo = owner[pos];
          const int pl = pos - prefix[lo];
          const int64_t ent = lstart[lo] + pl;
          cr[u].load(a.codes + ent * M, pl);
          lq[u] = a.lamq[ent];
          kp[u] = a.kappa[ent];
          lo_[u] = lo;
        }
      }
#pragma unroll
      for (int u = 0; u < kSmallB; u++) {
        const int pos = (r0 + u) * Q_THREADS + (int)threadIdx.x;
        if (pos < total) {
          const int lo = lo_[u];
          const float la = lcb[lq[u]];
          const float base_d = lt1[lo] + la * lt6[lo] + (la * la - la) * lt5[lo];
          const float dist = (kp[u] + cr[u].adc(T3, M, ksub)) + base_d;
          key[r0 + u] = csl::key32(dist);
        }
      }
    }
    uint64_t* skeys = reinterpret_cast<uint64_t*>(smem);  // the BlockSelect key area: <= k survivors
    int* shist = reinterpret_cast<int*>(skeys + a.sel_cap);
    int* smeta = shist + 256;
    int* swsum = reinterpret_cast<int*>(owner + ((a.owner_cap + 1) & ~1));  // 16 ints behind the owner table
    if (threadIdx.x == 0) swsum[8] = 0;
    const csl::Kth kt = csl::kth32<kSmallR>(key, a.k, shist, smeta);
    bool take[kSmallR];
    csl::take_k_strided<kSmallR>(key, kt, a.k, swsum, take);
#pragma unroll
    for (int r = 0; r < kSmallR; r++)
      if (take[r]) skeys[atomicAdd(&swsum[8], 1)] = ((uint64_t)key[r] << 32) | (uint32_t)(r * Q_THREADS + (int)threadIdx.x);
    for (int i = threadIdx.x; i < a.k; i += Q_THREADS) {
      a.outD[qi * a.k + i] = FLT_MAX;
      a.outI[qi * a.k + i] = -1;
    }
    __syncthreads();
    const int ns = swsum[8];  // <= k
    if (ns > 128 && ns <= Q_THREADS) {  // block-uniform: one survivor per thread, bitonic sort (coarse_select.cuh);
                                        // up to 128 survivors the rank loop below is cheaper (4 warps x ns compares)
      uint64_t mykey = (int)threadIdx.x < ns ? skeys[threadIdx.x] : ~0ull;
      __syncthreads();  // skeys[] becomes the exchange buffer (sel_cap >= 256 keys)
      mykey = csl::block_sort256(mykey, skeys);
      if ((int)threadIdx.x < ns) {
        const int pos = (int)key_payload(mykey);
        const int lo = owner[pos];
        a.outD[qi * a.k + threadIdx.x] = ord2f((uint32_t)(mykey >> 32));
        const int64_t e = lstart[lo] + (pos - prefix[lo]);
        a.outI[qi * a.k + threadIdx.x] = a.ids ? a.ids[e] : e;
      }
      return;
    }
    for (int i = threadIdx.x; i < ns; i += Q_THREADS) {
      const uint64_t mykey = skeys[i];
      int rank = 0;
      for (int j = 0; j < ns; j++) rank += skeys[j] < mykey;
      const int pos = (int)key_payload(mykey);
      const int lo = owner[pos];
      a.outD[qi * a.k + rank] = ord2f((uint32_t)(mykey >> 32));
      const int64_t e = lstart[lo] + (pos - prefix[lo]);
      a.outI[qi * a.k + rank] = a.ids ? a.ids[e] : e;
    }
    return;
  }

  for (int base = 0; !LONG && base < total; base += Q_BATCH * Q_THREADS) {
    // phase A: which list / entry each stream position is; phase B: all global loads of the batch in flight;
    // phase C: arithmetic.  (Interleaving them serialises ~3 DRAM latencies per entry.)
    // stream positions are warp-contiguous: warp w owns [base + 128 w, base + 128 w + 128), lane l the positions
    // +l, +32+l, ...  One (warp-uniform) binary search finds the list of the warp's first position; every lane then
    // walks forward from there -- 0-2 steps when lists are long.  Small batches use the owner table instead.
    int lo_[Q_BATCH];
    int pos_[Q_BATCH];  // position inside the list (code rotation)
    int64_t ent_[Q_BATCH];
    const int wpos0 = base + (threadIdx.x >> 5) * (Q_BATCH * 32);
    int wlo = 0;
    if (!use_owner && wpos0 < total) {
      int hi = W;
      while (hi - wlo > 1) {  // largest w with prefix[w] <= wpos0
        int mid = (wlo + hi) >> 1;
        if (prefix[mid] <= wpos0) wlo = mid; else hi = mid;
      }
    }
#pragma unroll
    for (int b = 0; b < Q_BATCH; b++) {
      const int pos = use_owner ? base + b * Q_THREADS + (int)threadIdx.x : wpos0 + b * 32 + (int)(threadIdx.x & 31);
      int lo = wlo;
      if (pos < total) {
        if (use_owner) {
          lo = owner[pos];
        } else if (total >= 16 * W) {  // long lists: a step or two forward from the warp's first list
          while (lo + 1 < W && prefix[lo + 1] <= pos) lo++;
          wlo = lo;  // positions of later sub-batches are larger: continue the walk from here
        } else {  // many short lists per warp: bounded binary search, largest w with prefix[w] <= pos
          int hi = W;
          while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (prefix[mid] <= pos) lo = mid; else hi = mid;
          }
        }
      }
      lo_[b] = lo;
      pos_[b] = pos < total ? pos - prefix[lo] : 0;
      ent_[b] = pos < total ? lstart[lo] + pos_[b] : -1;
    }
    CodeRegs<M_T> cr[Q_BATCH];
    uint8_t lq[Q_BATCH];
    float kp[Q_BATCH];
#pragma unroll
    for (int b = 0; b < Q_BATCH; b++) {
      lq[b] = 0;
      kp[b] = 0.f;
      if (ent_[b] >= 0) {
        cr[b].load(a.codes + ent_[b] * M, pos_[b]);
        lq[b] = a.lamq[ent_[b]];
        kp[b] = a.kappa[ent_[b]];
      }
    }
    bool any = false;
#pragma unroll
    for (int b = 0; b < Q_BATCH; b++) {
      const int pos = use_owner ? base + b * Q_THREADS + (int)threadIdx.x : wpos0 + b * 32 + (int)(threadIdx.x & 31);
      const bool valid = ent_[b] >= 0;
      float dist = 0.f;
      if (valid) {
        const int lo = lo_[b];
        const float la = lcb[lq[b]];
        const float base_d = lt1[lo] + la * lt6[lo] + (la * la - la) * lt5[lo];
        const float acc = cr[b].adc(T3, M, ksub);
        dist = (kp[b] + acc) + base_d;
      }
      any |= sel.offer_f(valid, dist, (uint32_t)pos);
    }
    sel.end_batch(any);
  }
  sel.finish();
  for (int i = threadIdx.x; i < a.k; i += Q_THREADS) {
    const uint64_t key = sel.keys[i];
    float dv = FLT_MAX;
    int64_t id = -1;
    if (key != kKeyInf) {
      const int pos = (int)key_payload(key);
      int lo = 0, hi = W;
      while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (prefix[mid] <= pos) lo = mid; else hi = mid;
      }
      dv = key_val(key);
      const int64_t e = lstart[lo] + (pos - prefix[lo]);
      id = a.ids ? a.ids[e] : e;
    }
    a.outD[qi * a.k + i] = dv;
    a.outI[qi * a.k + i] = id;
  }
}

// term-3 tables for a batch of queries: T3[q][m][j] = -2 q_m . p_mj (gpu/impl/IVFPQ.cu:1409-1432).  Persistent CTAs
// stage the PQ codebook once in shared memory (natural (m, j, t) layout, plain coalesced copy) and walk the queries;
// thread j owns codeword j of every sub-quantizer, so the table rows are written coalesced.  Same fmaf chain (t
// ascending) as the in-kernel build, hence bit-identical tables.
constexpr int T3_THREADS = 256;  // one thread per codeword of a sub-quantizer (ksub = 256)
__global__ void __launch_bounds__(T3_THREADS)
term3_kernel(const float* __restrict__ q, int64_t nq, int d, const float* __restrict__ pq, int M, int dsub,
             float* __restrict__ t3, bool code_major) {
  extern __shared__ __align__(16) float t3s[];
  float* pqs = t3s;                          // [M][256][dsub]
  float* qs = t3s + (size_t)M * 256 * dsub;  // [d]
  const int total4 = (M * 256 * dsub) / 4;   // d % 4 == 0 is checked by the launcher
  for (int i = threadIdx.x; i < total4; i += T3_THREADS)
    reinterpret_cast<float4*>(pqs)[i] = reinterpret_cast<const float4*>(pq)[i];
  for (int64_t qi = blockIdx.x; qi < nq; qi += gridDim.x) {
    __syncthreads();
    for (int j = threadIdx.x; j < d; j += T3_THREADS) qs[j] = q[qi * d + j];
    __syncthreads();
    float* out = t3 + (size_t)qi * M * 256;
    int m = 0;
    for (; m + 4 <= M; m += 4) {  // four independent fmaf chains in flight (one chain per sub-quantizer)
      float ip[4] = {0.f, 0.f, 0.f, 0.f};
      for (int t = 0; t < dsub; t++) {
#pragma unroll
        for (int u = 0; u < 4; u++)
          ip[u] = fmaf(qs[(m + u) * dsub + t], pqs[((size_t)(m + u) * 256 + threadIdx.x) * dsub + t], ip[u]);
      }
      if (code_major) {  // [j][M]: the row of codeword j is what the bank-skewed scan copies (M % 4 == 0 there)
        *reinterpret_cast<float4*>(out + (size_t)threadIdx.x * M + m) =
            make_float4(-2.f * ip[0], -2.f * ip[1], -2.f * ip[2], -2.f * ip[3]);
      } else {
#pragma unroll
        for (int u = 0; u < 4; u++) out[(m + u) * 256 + threadIdx.x] = -2.f * ip[u];
      }
    }
    for (; m < M; m++) {
      const float* pp = pqs + ((size_t)m * 256 + threadIdx.x) * dsub;
      const float* qm = qs + m * dsub;
      float ip = 0.f;
      for (int t = 0; t < dsub; t++) ip = fmaf(qm[t], pp[t], ip);
      out[code_major ? (size_t)threadIdx.x * M + m : (size_t)m * 256 + threadIdx.x] = -2.f * ip;
    }
  }
}

// Register-resident variant for the two production shapes (M x dsub = 16 x 8 and 8 x 12): thread j keeps codeword j of
// EVERY sub-quantizer in registers (d floats) for the whole launch, so a query costs d fused multiply-adds per thread,
// d/4 broadcast 16-byte reads of the query from shared memory and M coalesced stores -- no shared-memory traffic for the
// codebook at all (the shared-memory version above reads it with an 8-way bank conflict: stride dsub words).
// Same fmaf chains (t ascending from 0), hence the same bits.
template <int M_T, int DSUB>
__global__ void __launch_bounds__(T3_THREADS, 1)
term3_reg_kernel(const float* __restrict__ q, int64_t nq, const float* __restrict__ pq, float* __restrict__ t3,
                 bool code_major) {
  constexpr int D = M_T * DSUB;
  __shared__ __align__(16) float qs[2][D];
  float p[D];
#pragma unroll
  for (int m = 0; m < M_T; m++) {
    const float4* src = reinterpret_cast<const float4*>(pq + ((size_t)m * 256 + threadIdx.x) * DSUB);
#pragma unroll
    for (int t4 = 0; t4 < DSUB / 4; t4++) {
      const float4 v = src[t4];
      p[m * DSUB + t4 * 4 + 0] = v.x;
      p[m * DSUB + t4 * 4 + 1] = v.y;
      p[m * DSUB + t4 * 4 + 2] = v.z;
      p[m * DSUB + t4 * 4 + 3] = v.w;
    }
  }
  int buf = 0;
  if ((int64_t)blockIdx.x < nq && threadIdx.x < D) qs[0][threadIdx.x] = q[(int64_t)blockIdx.x * D + threadIdx.x];
  __syncthreads();
  for (int64_t qi = blockIdx.x; qi < nq; qi += gridDim.x) {
    const int64_t nxt = qi + gridDim.x;  // the next query is staged while this one is computed: one barrier per query
    if (nxt < nq && threadIdx.x < D) qs[buf ^ 1][threadIdx.x] = q[nxt * D + threadIdx.x];
    float* out = t3 + (size_t)qi * M_T * 256;
    const float4* q4 = reinterpret_cast<const float4*>(qs[buf]);
    float res[M_T];
#pragma unroll
    for (int m = 0; m < M_T; m++) {
      float ip = 0.f;
#pragma unroll
      for (int t4 = 0; t4 < DSUB / 4; t4++) {
        const float4 qv = q4[(m * DSUB) / 4 + t4];
        ip = fmaf(qv.x, p[m * DSUB + t4 * 4 + 0], ip);
        ip = fmaf(qv.y, p[m * DSUB + t4 * 4 + 1], ip);
        ip = fmaf(qv.z, p[m * DSUB + t4 * 4 + 2], ip);
        ip = fmaf(qv.w, p[m * DSUB + t4 * 4 + 3], ip);
      }
      res[m] = -2.f * ip;
    }
    if (code_major) {
#pragma unroll
      for (int m = 0; m < M_T; m += 4)
        *reinterpret_cast<float4*>(out + (size_t)threadIdx.x * M_T + m) = make_float4(res[m], res[m + 1], res[m + 2], res[m + 3]);
    } else {
#pragma unroll
      for (int m = 0; m < M_T; m++) out[m * 256 + threadIdx.x] = res[m];
    }
    __syncthreads();
    buf ^= 1;
  }
}

static size_t term3_pq_smem_bytes(int d) { return ((size_t)256 * d + d) * sizeof(float); }  // codebook + one query

bool term3_supported(int d, int M) { return d > 0 && M > 0 && d % M == 0 && d % 4 == 0 && term3_pq_smem_bytes(d) <= 200 * 1024; }

// persistent CTAs (at most one per SM) walk the queries of the batch
int launch_term3(const float* q, int64_t nq, int d, const float* pq, int M, float* t3, bool code_major, cudaStream_t st) {
  const unsigned grid = (unsigned)(nq < 148 ? nq : 148);
  const int dsub = d / M;
  if (M == 16 && dsub == 8) {
    VLQ_LAUNCH((term3_reg_kernel<16, 8>), grid, T3_THREADS, 0, st, q, nq, pq, t3, code_major);
  } else if (M == 8 && dsub == 12) {
    VLQ_LAUNCH((term3_reg_kernel<8, 12>), grid, T3_THREADS, 0, st, q, nq, pq, t3, code_major);
  } else {
    const size_t pq_smem = term3_pq_smem_bytes(d);
    VLQ_CUDA_TRY(cudaFuncSetAttribute(term3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pq_smem));
    VLQ_LAUNCH(term3_kernel, grid, T3_THREADS, pq_smem, st, q, nq, d, pq, M, dsub, t3, code_major);
  }
  return VLQ_OK;
}

// ------------------------------------------------------------------------------------------------ asynchronous scan
// The 1B-scale variant of scan_topk_kernel (k <= 128): one CTA per query, but every WARP runs on its own -- it grabs the
// next selected list from a shared counter, strides its entries (2 per lane per step, loads first), and keeps its own
// exact top-k in a WarpSelect.  No block barrier between setup and the final merge, so the loads of eight independent
// list walks per CTA are in flight at any time.  Same results as the other two modes (selection is exact and keys are
// unique stream positions).
// one selected line of a query as the asynchronous scan keeps it in shared memory (two 16-byte reads per line)
struct __align__(16) LineDesc {
  int64_t st;  // first entry of the list
  int p0;      // stream position of its first entry (tie order of the results)
  int len;     // entries scanned (capped like IVFUtils.cu:87)
  float t1, t6, t5;
  int pad;
};

// SKEW (M = 16 or 8): bank-conflict-free lookups.  With the plain [m][256] tables the 32 lanes of a warp read 32 random
// words of one table: ~2.2 shared-memory wavefronts per lookup, and ncu shows the L1/shared data path at 91 % -- that,
// not HBM, bounds the scan.  Here lane l works on sub-quantizer (s + l) % M at step s, and the tables are stored
// code-major with a 64-word row: word c of row `code` holds T3[c % M][code] for c < 31 + M.  Lane l reads word
// M*(l/M) + l%M + s of row code: the 32 lanes always hit 32 different banks whatever their codes are, the row stride of
// 256 bytes turns "extract byte, scale, add lane offset" into ONE byte-permute, and the step offset is an immediate.
// The lists store the code bytes pre-rotated by the position inside the list (scan.cuh), so the lane needs no byte
// shuffling of its own.  Price: the M terms are summed in a lane-dependent order, so a distance can differ from the other scan modes in the last ulp.  64 KB of tables per query:
// 12 warps per CTA, two CTAs per SM; the block select of the final merge reuses the table space.
constexpr int AQ_THREADS_SKEW = 384;
constexpr int kSkewRowWords = 64;

template <int M_T>
struct SkewCodes {
  uint32_t w[M_T / 4];
  __device__ __forceinline__ void load(const uint8_t* __restrict__ p, int /*pos*/) {
    if constexpr (M_T == 16) {
      const uint4 c = ld_nc_v4(p);
      w[0] = c.x; w[1] = c.y; w[2] = c.z; w[3] = c.w;
    } else {
      const uint2 c = ld_nc_v2(p);
      w[0] = c.x; w[1] = c.y;
    }
  }
  // The lists store the code bytes of the entry at position pos rotated by pos mod M (scan.cuh); a chunk starts at a
  // multiple of 64 inside its list, so lane l holds entries with pos mod M == l mod M and byte s of the stored code is
  // the byte of sub-quantizer (s + l) mod M.  tbl: skewed tables (bytes), lofs = 4 * lane.
  __device__ __forceinline__ float adc(const unsigned char* __restrict__ tbl, uint32_t lofs) const {
    float acc = 0.f;
#pragma unroll
    for (int s = 0; s < M_T; s++) {
      const uint32_t o = __byte_perm(w[s >> 2], lofs, 0x5504 | ((s & 3) << 4));  // code << 8 | lofs
      acc += *reinterpret_cast<const float*>(tbl + o + 4 * s);
    }
    return acc;
  }
};

template <int M_T, bool SKEW>
__global__ void __launch_bounds__(SKEW ? AQ_THREADS_SKEW : Q_THREADS, SKEW ? 2 : 1) scan_async_kernel(ScanArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int NT = SKEW ? AQ_THREADS_SKEW : Q_THREADS;
  constexpr int NW = NT / 32;
  constexpr int MS = M_T ? M_T : 4;  // only used when SKEW
  const int M = a.M, ksub = a.ksub, W = a.W;
  const int MM = M_T ? M_T : M;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // smem: [tables | block select of the final merge (SKEW: same space)][NW x warp select][lcb][LineDesc W][misc]
  const size_t sel_bytes = (select_smem_bytes(a.sel_cap) + 15) & ~size_t(15);
  const size_t tbl_bytes = SKEW ? sizeof(float) * 256 * kSkewRowWords : sizeof(float) * M * ksub;
  size_t off = 0;
  float* T3;
  if (SKEW) {
    T3 = reinterpret_cast<float*>(smem);
    off = sel_bytes > tbl_bytes ? sel_bytes : tbl_bytes;
  } else {
    off = sel_bytes;
    T3 = reinterpret_cast<float*>(smem + off);
    off += tbl_bytes;
  }
  unsigned char* wsel = smem + off;
  off += (size_t)NW * kWarpSelSmemBytes;
  float* lcb = reinterpret_cast<float*>(smem + off);
  off += sizeof(float) * ((a.nL + 3) & ~3);
  LineDesc* desc = reinterpret_cast<LineDesc*>(smem + off);
  off += sizeof(LineDesc) * W;
  int* misc = reinterpret_cast<int*>(smem + off);  // [0] next line, [1..NW] per-warp survivor counts

  const int64_t qi = blockIdx.x;
  if (SKEW) {  // a.t3 is code-major here: row `code` = M consecutive floats
    // word c of row `code` = src[code*M + c % M]: whole float4s, (31 + M + 3) / 4 of them per row
    const float4* src4 = reinterpret_cast<const float4*>(a.t3 + (size_t)qi * M * ksub);
    float4* dst4 = reinterpret_cast<float4*>(T3);
    constexpr int Q4 = (31 + MS + 3) / 4, S4 = MS / 4;
    for (int i = threadIdx.x; i < 256 * Q4; i += NT) {
      const int code = i / Q4, q4 = i % Q4;
      dst4[code * (kSkewRowWords / 4) + q4] = src4[code * S4 + (q4 & (S4 - 1))];
    }
  } else {
    const float4* src = reinterpret_cast<const float4*>(a.t3 + (size_t)qi * M * ksub);
    float4* dst = reinterpret_cast<float4*>(T3);
    for (int i = threadIdx.x; i < (M * ksub) / 4; i += NT) dst[i] = src[i];
  }
  for (int i = threadIdx.x; i < a.nL; i += NT) lcb[i] = a.lambda_cb[i];
  for (int w = threadIdx.x; w < W; w += NT) {
    const int list = a.line_list[qi * W + w];
    LineDesc dsc;
    dsc.st = 0;
    dsc.p0 = 0;
    dsc.len = 0;
    dsc.t5 = 0.f;
    dsc.pad = 0;
    if (list >= 0) {
      dsc.st = a.offsets[list];
      const int64_t l = a.offsets[list + 1] - dsc.st;
      dsc.len = (int)(l < a.cap ? l : a.cap);
      dsc.t5 = a.edge_d2 ? a.edge_d2[list] : 0.f;
    }
    dsc.t1 = a.term1[qi * W + w];
    dsc.t6 = a.term6[qi * W + w];
    desc[w] = dsc;
  }
  if (threadIdx.x == 0) misc[0] = 0;
  __syncthreads();
  if (threadIdx.x < kWarp) {  // exclusive scan of the lengths: stream position of every line
    const int chunk = (W + kWarp - 1) / kWarp;
    const int b = lane * chunk, e = min(W, b + chunk);
    int s = 0;
    for (int w = b; w < e; w++) s += desc[w].len;
    int inc = s;
#pragma unroll
    for (int o = 1; o < kWarp; o <<= 1) {
      int t = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += t;
    }
    int run = inc - s;
    for (int w = b; w < e; w++) {
      desc[w].p0 = run;
      run += desc[w].len;
    }
  }
  __syncthreads();

  WarpSelect ws;
  ws.init(wsel + (size_t)warp * kWarpSelSmemBytes, a.k);
  // Software pipeline over 64-entry chunks (possibly of different lists): the loads of chunk i+1 are issued before the
  // arithmetic of chunk i, so every warp keeps two chunks (~2.7 KB) in flight.  (Unrolling by two so that the buffers
  // alternate roles instead of being copied measured 25-40 % slower: the loop body no longer fits the instruction cache.)
  using Codes = typename std::conditional<SKEW, SkewCodes<MS>, CodeRegs<M_T>>::type;
  struct Chunk {
    int p0, nrem;  // stream position of the chunk's first entry, entries of the list left from there
    float t1, t6, t5;
    Codes cr[2];
    uint32_t lq[2];
    float kp[2];
    bool ok;
  };
  const uint32_t lofs = 4u * (uint32_t)lane;  // column of the lane in the skewed table rows
  const unsigned char* tblc = reinterpret_cast<const unsigned char*>(T3);
  LineDesc cur;  // warp-uniform walk state
  cur.len = 0;
  int cur_e0 = 0;
  bool done = false;
  auto fetch = [&](Chunk& c) {
    cur_e0 += 64;
    if (cur_e0 >= cur.len) {
      cur.len = 0;
      while (!done && cur.len == 0) {  // next non-empty line from the shared counter
        int li = 0;
        if (lane == 0) li = atomicAdd(&misc[0], 1);
        li = __shfl_sync(kFull, li, 0);
        if (li >= W) {
          done = true;
        } else {
          const int4* dp = reinterpret_cast<const int4*>(desc + li);
          const int4 d0 = dp[0], d1 = dp[1];
          cur.st = ((int64_t)(uint32_t)d0.y << 32) | (uint32_t)d0.x;
          cur.p0 = d0.z;
          cur.len = d0.w;
          cur.t1 = __int_as_float(d1.x);
          cur.t6 = __int_as_float(d1.y);
          cur.t5 = __int_as_float(d1.z);
        }
      }
      cur_e0 = 0;
    }
    c.ok = cur.len > 0;
    if (!c.ok) return;
    c.p0 = cur.p0 + cur_e0;
    c.nrem = cur.len - cur_e0;
    c.t1 = cur.t1;
    c.t6 = cur.t6;
    c.t5 = cur.t5;
    const int64_t first = cur.st + cur_e0;  // warp-uniform
    const uint8_t* cb = a.codes + first * MM;
    const uint8_t* lb = a.lamq + first;
    const float* kb = a.kappa + first;
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const unsigned i = u * 32 + lane;
      c.lq[u] = 0;
      c.kp[u] = 0.f;
      if ((int)i < c.nrem) {
        c.cr[u].load(cb + i * (unsigned)MM, cur_e0 + (int)i);
        c.lq[u] = lb[i];
        c.kp[u] = kb[i];
      }
    }
  };
  auto score = [&](const Chunk& c) {
    float dist[2];
    bool pass = false;
#pragma unroll
    for (int u = 0; u < 2; u++) {
      dist[u] = __int_as_float(0x7f800000);
      if (u * 32 + lane < c.nrem) {
        const float la = lcb[c.lq[u]];
        const float base_d = c.t1 + la * c.t6 + (la * la - la) * c.t5;
        float adc;
        if constexpr (SKEW) adc = c.cr[u].adc(tblc, lofs);
        else adc = c.cr[u].adc(T3, M, ksub);
        dist[u] = (c.kp[u] + adc) + base_d;
        pass |= dist[u] <= ws.thr_f;
      }
    }
    if (__any_sync(kFull, pass)) {  // rare once the threshold has tightened
#pragma unroll
      for (int u = 0; u < 2; u++) ws.offer(u * 32 + lane < c.nrem, dist[u], (uint32_t)(c.p0 + u * 32 + lane));
    }
  };
  {
    Chunk A, B;
    fetch(A);
    while (A.ok) {
      fetch(B);
      score(A);
      A = B;
    }
  }
  ws.compact();
  if (lane == 0) misc[1 + warp] = ws.cnt;
  __syncthreads();

  // ---- merge the NW warp-local top-k sets
  BlockSelect<NT> sel;
  sel.init(smem, a.k, a.sel_cap, 1);
  for (int w = 0; w < NW; w++) {
    const uint64_t* wk = reinterpret_cast<const uint64_t*>(wsel + (size_t)w * kWarpSelSmemBytes);
    const int n = misc[1 + w];  // <= k <= kWarpSelCap survivors of warp w
    for (int i0 = 0; i0 < n; i0 += NT) {  // n is block-uniform
      const int i = i0 + (int)threadIdx.x;
      const bool valid = i < n;
      const bool any = sel.offer(valid, valid ? wk[i] : kKeyInf);
      sel.end_batch(any);
    }
  }
  sel.finish();
  for (int i = threadIdx.x; i < a.k; i += NT) {
    const uint64_t key = sel.keys[i];
    float dv = FLT_MAX;
    int64_t id = -1;
    if (key != kKeyInf) {
      const int pos = (int)key_payload(key);
      int lo = 0, hi = W;
      while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (desc[mid].p0 <= pos) lo = mid; else hi = mid;
      }
      dv = key_val(key);
      const int64_t e = desc[lo].st + (pos - desc[lo].p0);
      id = a.ids ? a.ids[e] : e;
    }
    a.outD[qi * a.k + i] = dv;
    a.outI[qi * a.k + i] = id;
  }
}

static size_t scan_async_smem_bytes(int sel_cap, int M, int ksub, int nL, int W, bool skew) {
  const size_t sel_bytes = (select_smem_bytes(sel_cap) + 15) & ~size_t(15);
  const size_t tbl_bytes = skew ? sizeof(float) * 256 * kSkewRowWords : sizeof(float) * M * ksub;
  size_t off = skew ? (sel_bytes > tbl_bytes ? sel_bytes : tbl_bytes) : sel_bytes + tbl_bytes;
  off += (size_t)((skew ? AQ_THREADS_SKEW : Q_THREADS) / 32) * kWarpSelSmemBytes;
  off += sizeof(float) * ((nL + 3) & ~3);
  off += sizeof(LineDesc) * W;
  off += sizeof(int) * 16;
  return off;
}

static size_t scan_smem_bytes(int sel_cap, int M, int ksub, int nL, int W, int owner_cap) {
  size_t off = (select_smem_bytes(sel_cap) + 15) & ~size_t(15);
  off += sizeof(float) * M * ksub;
  off += sizeof(float) * ((nL + 3) & ~3);
  off += sizeof(int64_t) * W;
  off += sizeof(int) * ((W + 1 + 3) & ~3);
  off += sizeof(float) * W * 3;
  off += sizeof(uint16_t) * ((owner_cap + 1) & ~1) + sizeof(int) * 16;  // owner table + scratch of the small-query path
  return off;
}

// ------------------------------------------------------------------------------------------------ shard merge
// `peers` != nullptr: shard r's results are read from peers[r] + d_off / + i_off -- buffers that live on the OTHER GPUs of
// the NVLink domain (peer-mapped symmetric memory), so the gather of the exchange step happens inside this kernel as
// plain P2P loads instead of a separate collective.
__global__ void __launch_bounds__(Q_THREADS)
merge_topk_kernel(const float* __restrict__ D, const int64_t* __restrict__ I, const unsigned char* const* __restrict__ peers,
                  size_t d_off, size_t i_off, int R, int64_t nq, int k, int cap, float* __restrict__ outD,
                  int64_t* __restrict__ outI) {
  extern __shared__ __align__(16) unsigned char smem[];
  BlockSelect<Q_THREADS> sel;
  sel.init(smem, k, cap, Q_BATCH);
  const int64_t q = blockIdx.x;
  const int num = R * k;
  auto d_of = [&](int rank) {
    return peers ? reinterpret_cast<const float*>(peers[rank] + d_off) + q * k : D + ((int64_t)rank * nq + q) * k;
  };
  auto i_of = [&](int rank) {
    return peers ? reinterpret_cast<const int64_t*>(peers[rank] + i_off) + q * k : I + ((int64_t)rank * nq + q) * k;
  };
  // Only the distances are read here (4 of the 12 bytes per candidate); the ids of the k winners are fetched at the end.
  // Padding entries carry (FLT_MAX, -1): they lose against every real entry, and where one is selected the output is
  // the same (FLT_MAX, -1) an empty slot gets.
  bool direct = false;
  if (num <= cap) {  // every candidate fits the buffer: no atomics, no per-batch barriers (BlockSelect::put)
    bool bad = false;
    for (int i = threadIdx.x; i < num; i += Q_THREADS) bad |= sel.put(i, true, d_of(i / k)[i % k], (uint32_t)i);
    direct = sel.placed(num, bad);
    if (!direct) sel.init(smem, k, cap, Q_BATCH);
  }
  if (!direct) {
    for (int base = 0; base < num; base += Q_BATCH * Q_THREADS) {
      float v[Q_BATCH];
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) {  // loads of the whole batch first: remote reads are NVLink round trips
        const int i = base + b * Q_THREADS + threadIdx.x;
        v[b] = i < num ? d_of(i / k)[i % k] : 0.f;
      }
      bool any = false;
#pragma unroll
      for (int b = 0; b < Q_BATCH; b++) {
        const int i = base + b * Q_THREADS + threadIdx.x;
        any |= sel.offer_f(i < num, v[b], (uint32_t)i);
      }
      sel.end_batch(any);
    }
  }
  sel.finish();
  for (int i = threadIdx.x; i < k; i += Q_THREADS) {
    const uint64_t key = sel.keys[i];
    float dv = FLT_MAX;
    int64_t id = -1;
    if (key != kKeyInf) {
      const int fi = (int)key_payload(key);
      dv = key_val(key);
      id = i_of(fi / k)[fi % k];
    }
    outD[q * k + i] = dv;
    outI[q * k + i] = id;
  }
}

// ------------------------------------------------------------------------------------------------ graph helper
__global__ void drop_rank0_kernel(const float* __restrict__ val, const int* __restrict__ idx, int64_t rows, int E,
                                  int* __restrict__ edge, float* __restrict__ edge_d2) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * E) return;
  int64_t r = i / E;
  int e = (int)(i % E);
  edge[i] = idx[r * (E + 1) + 1 + e];
  edge_d2[i] = val[r * (E + 1) + 1 + e];
}

static int graph_tile_rows(int C) {
  int64_t tr = (int64_t)(16 << 20) / C;  // 64 MiB of fp32 per tile: stays in the 126 MB L2
  if (tr < 128) tr = 128;
  if (tr > C) tr = C;
  return (int)tr;
}

}  // namespace vlq

using namespace vlq;

// ------------------------------------------------------------------------------------------------ peer slice gather
// Query-split sharding (the strong-scaling protocol): rank r computed the coarse stage of the queries [q0(r), q0(r + 1))
// and left (list, term1, term6) in its peer-mapped buffer.  This kernel pulls every OTHER rank's slice of up to four
// row-major arrays into the same place of the local buffer in ONE launch of P2P loads (was: one peer copy per rank and
// array, 3 (R - 1) launches per step).  blockIdx.y = source rank, blockIdx.z = array.
struct PeerSlices {
  int64_t arr_off[4];  // byte offset of each array inside the buffers
};
__global__ void __launch_bounds__(256)
gather_peer_slices_kernel(const unsigned char* const* __restrict__ peers, int R, int self, PeerSlices ps, int64_t nq,
                          int64_t row_bytes) {
  const int r = blockIdx.y;
  if (r == self) return;
  const int64_t b0 = (int64_t)r * nq / R * row_bytes, b1 = (int64_t)(r + 1) * nq / R * row_bytes;
  const unsigned char* src = peers[r] + ps.arr_off[blockIdx.z];
  unsigned char* dst = const_cast<unsigned char*>(peers[self]) + ps.arr_off[blockIdx.z];
  const int64_t n16 = (b1 - b0) >> 4;  // offsets and row_bytes are multiples of 16 (checked by the caller)
  const uint4* s4 = reinterpret_cast<const uint4*>(src + b0);
  uint4* d4 = reinterpret_cast<uint4*>(dst + b0);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x)
    d4[i] = s4[i];
}

extern "C" {

int vlq_select_lines(const float* D, int64_t nq, int64_t ldD, const int* coarse_ids, int P, const int* edge,
                     const float* edge_d2, int E, int W, int* out_list, float* out_term1, float* out_term6,
                     vlq_stream_t stream) {
  if (nq < 0 || P <= 0 || P > VLQ_MAX_K || E <= 0 || W <= 0 || W > VLQ_MAX_K) return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  if (!D || !coarse_ids || !edge || !edge_d2 || !out_list || !out_term1 || !out_term6) return VLQ_EINVAL;
  const int cap = select_capacity(W, Q_THREADS, Q_BATCH, (long long)P * E);
  const size_t smem = select_smem_bytes(cap);
  VLQ_LAUNCH(select_lines_kernel, (unsigned)nq, Q_THREADS, smem, as_stream(stream), D, ldD, coarse_ids, P, edge,
             edge_d2, E, W, cap, out_list, out_term1, out_term6);
  return last_error();
}

int vlq_coarse_select_lines(const float* D, int64_t nq, int64_t ldD, const float* bucket_min, int nb, int C, int P,
                            const int* edge, const float* edge_d2, int E, int W, int* out_coarse, int* out_list,
                            float* out_term1, float* out_term6, vlq_stream_t stream) {
  if (nq < 0 || P <= 0 || P > VLQ_MAX_K || E <= 0 || W <= 0 || W > VLQ_MAX_K || C <= 0 || nb <= 0 || ldD < C ||
      (int64_t)nb * 32 < C)
    return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  if (!D || !bucket_min || !edge || !edge_d2 || !out_list || !out_term1 || !out_term6) return VLQ_EINVAL;
  const int kmax = P > W ? P : W;
  long long total = (long long)P * E;
  if (total < (long long)P * 32) total = (long long)P * 32;
  if (total < nb) total = nb;
  const int cap = select_capacity(kmax, Q_THREADS, Q_BATCH, total);
  const size_t smem = ((select_smem_bytes(cap) + 15) & ~size_t(15)) + 2 * VLQ_MAX_K * sizeof(int);
  // fast path (coarse_select.cuh): the keys of each selection fit R per thread in registers
  const bool generic_only = getenv("VLQ_COARSE_GENERIC") != nullptr;  // read per call: tests force the general kernel
  const int need = nb > P * E ? (nb > P * 32 ? nb : P * 32) : (P * E > P * 32 ? P * E : P * 32);
  if (!generic_only && need <= 16 * csl::NT && W <= 1024 && nb % 4 == 0 && (reinterpret_cast<uintptr_t>(bucket_min) & 15) == 0) {
    const int R = need <= 8 * csl::NT ? 8 : 16;
    const size_t fsmem = csl::Smem::bytes(R, P);
    if (R == 8) {
      VLQ_CUDA_TRY(cudaFuncSetAttribute(csl::coarse_select_lines_fast_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
      VLQ_LAUNCH(csl::coarse_select_lines_fast_kernel<8>, (unsigned)nq, csl::NT, fsmem, as_stream(stream), D, ldD, bucket_min,
                 nb, C, P, edge, edge_d2, E, W, out_coarse, out_list, out_term1, out_term6);
    } else {
      VLQ_CUDA_TRY(cudaFuncSetAttribute(csl::coarse_select_lines_fast_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
      VLQ_LAUNCH(csl::coarse_select_lines_fast_kernel<16>, (unsigned)nq, csl::NT, fsmem, as_stream(stream), D, ldD, bucket_min,
                 nb, C, P, edge, edge_d2, E, W, out_coarse, out_list, out_term1, out_term6);
    }
    return last_error();
  }
  VLQ_CUDA_TRY(cudaFuncSetAttribute(coarse_select_lines_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  VLQ_LAUNCH(coarse_select_lines_kernel, (unsigned)nq, Q_THREADS, smem, as_stream(stream), D, ldD, bucket_min, nb, C, P,
             edge, edge_d2, E, W, cap, out_coarse, out_list, out_term1, out_term6);
  return last_error();
}

int vlq_coarse_exact_supported(int d, int C, int P, int E, int W) {
  if (d <= 0 || C <= 0 || P <= 0 || E <= 0 || W <= 0) return 0;
  return csl::exact_supported(d, vlq_tc_num_buckets(C), P, E, W) ? 1 : 0;
}

// The matrix-free route reads (32 P + P E) centroid rows per query from L2 where the matrix route reads ~(P + P E) 32-byte
// sectors of D from DRAM but must first write 4 C bytes per query: measured on B200 (tools/bench_coarse.py, C = 65536,
// d = 128, E = 32, per 8192 queries) 0.45 / 0.67 / 0.93 / 2.5 ms against 0.78 / 0.81 / 0.82 / 0.97 ms at P = 1 / 8 / 16 / 64
// -- it wins up to 256 KiB of rows per query.
int vlq_coarse_exact_preferred(int d, int C, int P, int E, int W) {
  if (!vlq_coarse_exact_supported(d, C, P, E, W)) return 0;
  return (int64_t)P * (32 + E) * d * 4 <= (256 << 10) ? 1 : 0;
}

int vlq_coarse_select_lines_exact(const float* q, int64_t nq, int d, const float* cent, const float* cnorm,
                                  const float* bucket_min, int nb, int C, int P, const int* edge, const float* edge_d2,
                                  int E, int W, int* out_coarse, int* out_list, float* out_term1, float* out_term6,
                                  vlq_stream_t stream) {
  if (nq < 0 || d <= 0 || P <= 0 || P > VLQ_MAX_K || E <= 0 || W <= 0 || W > VLQ_MAX_K || C <= 0 || nb <= 0 ||
      (int64_t)nb * 32 < C)
    return VLQ_EINVAL;
  if (!csl::exact_supported(d, nb, P, E, W)) return VLQ_EUNSUPPORTED;
  if (nq == 0) return VLQ_OK;
  if (!q || !cent || !cnorm || !bucket_min || !edge || !edge_d2 || !out_list || !out_term1 || !out_term6)
    return VLQ_EINVAL;
  if ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(cent) | reinterpret_cast<uintptr_t>(bucket_min)) & 15)
    return VLQ_EINVAL;
  const int need = nb > P * E ? (nb > P * 32 ? nb : P * 32) : (P * E > P * 32 ? P * E : P * 32);
  const int R = need <= 8 * csl::NT ? 8 : 16;
  const size_t smem = csl::SmemExact::bytes(R, P);
  if (R == 8) {
    VLQ_CUDA_TRY(cudaFuncSetAttribute(csl::coarse_select_lines_exact_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VLQ_LAUNCH(csl::coarse_select_lines_exact_kernel<8>, (unsigned)nq, csl::NT, smem, as_stream(stream), q, d, cent, cnorm,
               bucket_min, nb, C, P, edge, edge_d2, E, W, out_coarse, out_list, out_term1, out_term6);
  } else {
    VLQ_CUDA_TRY(cudaFuncSetAttribute(csl::coarse_select_lines_exact_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VLQ_LAUNCH(csl::coarse_select_lines_exact_kernel<16>, (unsigned)nq, csl::NT, smem, as_stream(stream), q, d, cent, cnorm,
               bucket_min, nb, C, P, edge, edge_d2, E, W, out_coarse, out_list, out_term1, out_term6);
  }
  return last_error();
}

int vlq_coarse_route(int d, int C, int P, int E, int W, int have_pack) {
  if (!have_pack) return 0;
  if (getenv("VLQ_COARSE_MATRIX")) return 1;
  if (getenv("VLQ_COARSE_EXACT")) return vlq_coarse_exact_supported(d, C, P, E, W) ? 2 : 1;
  return vlq_coarse_exact_preferred(d, C, P, E, W) ? 2 : 1;
}

}  // extern "C"

// Byte offsets of the arrays of the vlq_coarse_lines workspace: only those the route uses, each on a 256-byte boundary.
struct CoarseWorkspace {
  size_t D = 0, bmin = 0, tc = 0, cval = 0, cidx = 0, end = 0;
};

static CoarseWorkspace coarse_workspace(int route, int64_t nq, int d, int C, int P) {
  const size_t n = nq > 0 ? (size_t)nq : 0;
  CoarseWorkspace w;
  auto take = [&w](size_t bytes) {
    const size_t at = w.end;
    w.end += (bytes + 255) & ~size_t(255);
    return at;
  };
  if (route != 2) w.D = take(n * C * sizeof(float));
  if (route != 0) {
    w.bmin = take(n * vlq_tc_num_buckets(C) * sizeof(float));
    w.tc = take(vlq_l2_tc_workspace_bytes(nq, d, C));
  } else {
    w.cval = take(n * P * sizeof(float));
    w.cidx = take(n * P * sizeof(int));
  }
  return w;
}

extern "C" {

size_t vlq_coarse_lines_workspace_bytes(int64_t nq, int d, int C, int P, int E, int W, int have_pack) {
  return coarse_workspace(vlq_coarse_route(d, C, P, E, W, have_pack), nq, d, C, P).end;
}

int vlq_coarse_lines(const float* q, int64_t nq, int d, const float* cent, const float* cnorm, const void* cent_pack,
                     float scale, int C, int P, const int* edge, const float* edge_d2, int E, int W, int* out_coarse,
                     int* out_list, float* out_term1, float* out_term6, void* workspace, size_t workspace_bytes,
                     vlq_stream_t stream) {
  if (nq < 0 || d <= 0 || C <= 0 || P <= 0 || P > VLQ_MAX_K || P > C || E <= 0 || W <= 0 || W > VLQ_MAX_K)
    return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  if (!q || !cent || !cnorm || !edge || !edge_d2 || !out_list || !out_term1 || !out_term6 || !workspace)
    return VLQ_EINVAL;
  const int route = vlq_coarse_route(d, C, P, E, W, cent_pack != nullptr);
  // the tensor-core sweep reads q, the matrix-free select reads q and cent, in 16-byte vectors
  const uintptr_t vec = reinterpret_cast<uintptr_t>(q) | (route == 2 ? reinterpret_cast<uintptr_t>(cent) : 0);
  if ((route != 0 && (vec & 15)) || (reinterpret_cast<uintptr_t>(workspace) & 255)) return VLQ_EINVAL;
  const CoarseWorkspace w = coarse_workspace(route, nq, d, C, P);
  if (workspace_bytes < w.end) return VLQ_EWORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  float* D = reinterpret_cast<float*>(ws + w.D);
  float* bmin = reinterpret_cast<float*>(ws + w.bmin);
  const int nb = vlq_tc_num_buckets(C);
  const size_t tc_bytes = vlq_l2_tc_workspace_bytes(nq, d, C);
  int rc;
  if (route == 2) {
    rc = vlq_l2_bucket_min_tc(q, nq, d, cent_pack, scale, C, bmin, ws + w.tc, tc_bytes, stream);
    if (rc) return rc;
    return vlq_coarse_select_lines_exact(q, nq, d, cent, cnorm, bmin, nb, C, P, edge, edge_d2, E, W, out_coarse,
                                         out_list, out_term1, out_term6, stream);
  }
  if (route == 1) {
    rc = vlq_l2_distances_tc(q, nq, d, cent_pack, scale, C, D, C, bmin, ws + w.tc, tc_bytes, stream);
    if (rc) return rc;
    return vlq_coarse_select_lines(D, nq, C, bmin, nb, C, P, edge, edge_d2, E, W, out_coarse, out_list, out_term1,
                                   out_term6, stream);
  }
  int* cidx = out_coarse ? out_coarse : reinterpret_cast<int*>(ws + w.cidx);
  rc = vlq_l2_distances(q, nq, d, cent, cnorm, C, D, C, stream);
  if (rc) return rc;
  rc = vlq_select_rows(D, nq, C, C, P, nullptr, reinterpret_cast<float*>(ws + w.cval), cidx, stream);
  if (rc) return rc;
  return vlq_select_lines(D, nq, C, cidx, P, edge, edge_d2, E, W, out_list, out_term1, out_term6, stream);
}

// term-3 tables of the batch (+ 256 spare bytes)
size_t vlq_scan_topk_workspace_bytes(int64_t nq, int M) { return (size_t)(nq > 0 ? nq : 0) * M * 256 * sizeof(float) + 256; }

int vlq_scan_topk(const float* q, int64_t nq, int d, const float* pq, int M, const float* lambda_cb, int nL,
                  const int* line_list, const float* term1, const float* term6, const float* edge_d2, int W,
                  const int64_t* offsets, const uint8_t* codes, const uint8_t* lamq, const float* kappa,
                  const int64_t* ids, int k, int cap, int list_len_hint, float* outD, int64_t* outI, void* workspace,
                  size_t workspace_bytes, vlq_stream_t stream) {
  if (nq > 0 && (!q || !pq || !lambda_cb || !line_list || !term1 || !term6 || !offsets || !outD || !outI))
    return VLQ_EINVAL;
  if (nq < 0 || d <= 0 || M <= 0 || M > 64 || d % M != 0 || nL <= 0 || nL > 256 || W <= 0 || W > VLQ_MAX_K ||
      k <= 0 || k > VLQ_MAX_K || cap <= 0 || cap > (1 << 20) / 1 || (int64_t)W * cap > (int64_t)0x7fffffff)
    return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  ScanArgs a{};
  a.q = q; a.d = d; a.pq = pq; a.M = M; a.ksub = 256; a.dsub = d / M; a.lambda_cb = lambda_cb; a.nL = nL;
  a.line_list = line_list; a.term1 = term1; a.term6 = term6; a.edge_d2 = edge_d2; a.W = W; a.offsets = offsets;
  a.codes = codes; a.lamq = lamq; a.kappa = kappa; a.ids = ids; a.k = k; a.cap = cap; a.outD = outD; a.outI = outI;
  a.sel_cap = select_capacity(k, Q_THREADS, Q_BATCH, (long long)W * cap);
  a.t3 = nullptr;
  const size_t t3_bytes = (size_t)nq * M * 256 * sizeof(float);
  const bool long_lists = list_len_hint >= 24;  // average list length of the index: warp-per-list pays off
  const bool al16 = (reinterpret_cast<uintptr_t>(codes) % 16) == 0;
  const bool have_t3 = workspace && workspace_bytes >= t3_bytes + 256 && term3_supported(d, M) &&
                       ((reinterpret_cast<uintptr_t>(workspace) | reinterpret_cast<uintptr_t>(pq)) & 15) == 0;
  const bool use_async = long_lists && k <= kWarpSelMaxK && have_t3 && (M * 256) % 4 == 0;  // warp-autonomous scan
  // bank-skewed tables pay off once the lists are long enough to amortise the 64 KB table fill and the four extra
  // warps per query (measured on the C2 geometry, average list length -> speed-up over the plain tables:
  // 48 -> 0.94x, 60 -> 1.13x, 72 -> 1.15x, 95 -> 1.18x, 143 -> 1.23x, 477 -> 1.26x)
  static const int skew_min_len = [] {
    const char* e = getenv("VLQ_SCAN_SKEW_MIN_LEN");  // tuning knob
    return e ? atoi(e) : 56;
  }();
  // which long-list kernel: scan_long.cu (four entries per lane behind TMA bulk prefetches into L2, any k) for lists of
  // >= long_min_len entries on average, else the register-pipelined warp-autonomous kernel below (k <= 128).  Both use
  // the bank-skewed tables.  Measured, ms per 10 k queries (long / skew): 60 entries per list 2.63 / 2.40,
  // 477 entries per list 7.54 / 8.35.  VLQ_SCAN_KERNEL=skew | long forces one of them (tests, tools/bench_scan.py).
  static const int long_kernel = [] {
    const char* e = getenv("VLQ_SCAN_KERNEL");
    if (e && e[0] == 's') return 1;
    if (e && e[0] == 'l') return 2;
    return 0;
  }();
  static const int long_min_len = [] {
    const char* e = getenv("VLQ_SCAN_LONG_MIN_LEN");
    return e ? atoi(e) : 160;
  }();
  bool use_long = false;
  if (long_lists && have_t3 && list_len_hint >= skew_min_len && long_kernel != 1 &&
      (long_kernel == 2 || list_len_hint >= long_min_len || k > kWarpSelMaxK)) {
    ScanArgs probe = a;
    probe.t3 = static_cast<float*>(workspace);
    use_long = scan_long_supported(probe);
  }
  const bool skew = use_long || (use_async && al16 && (M == 16 || M == 8) && list_len_hint >= skew_min_len);
  if (have_t3) {
    float* t3 = static_cast<float*>(workspace);
    const int rc = launch_term3(q, nq, d, pq, M, t3, skew, as_stream(stream));
    if (rc) return rc;
    a.t3 = t3;
  }
  a.owner_cap = (int)((long long)W * cap < 4096 ? (long long)W * cap : 4096);
  a.no_small = getenv("VLQ_SCAN_NO_SMALL") != nullptr;  // read per call: tests flip it between calls
  if (use_long) return launch_scan_long(a, nq, as_stream(stream));
  if (use_async) {
    cudaStream_t st_ = as_stream(stream);
    const int nt = skew ? AQ_THREADS_SKEW : Q_THREADS;
    const int scap = select_capacity(k, nt, 1, (long long)(nt / 32) * k);  // <= k survivors per warp
    a.sel_cap = scap;
    const size_t smem_a = scan_async_smem_bytes(scap, M, a.ksub, nL, W, skew);
#define VLQ_ASYNC_LAUNCH(MT, SK)                                                                                      \
  do {                                                                                                                \
    VLQ_CUDA_TRY(cudaFuncSetAttribute(scan_async_kernel<MT, SK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a)); \
    VLQ_LAUNCH((scan_async_kernel<MT, SK>), (unsigned)nq, nt, smem_a, st_, a);                                        \
  } while (0)
    if (skew && M == 16) VLQ_ASYNC_LAUNCH(16, true);
    else if (skew) VLQ_ASYNC_LAUNCH(8, true);
    else if (M == 16 && al16) VLQ_ASYNC_LAUNCH(16, false);
    else if (M == 8 && al16) VLQ_ASYNC_LAUNCH(8, false);
    else VLQ_ASYNC_LAUNCH(0, false);
#undef VLQ_ASYNC_LAUNCH
    return last_error();
  }
  if (long_lists) a.sel_cap = select_capacity(k, Q_THREADS, 2, (long long)W * cap);
  size_t smem = scan_smem_bytes(a.sel_cap, M, a.ksub, nL, W, a.owner_cap);
  cudaStream_t st = as_stream(stream);
#define VLQ_SCAN_LAUNCH(MT, LG)                                                                                        \
  do {                                                                                                                 \
    VLQ_CUDA_TRY(cudaFuncSetAttribute(scan_topk_kernel<MT, LG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    VLQ_LAUNCH((scan_topk_kernel<MT, LG>), (unsigned)nq, Q_THREADS, smem, st, a);                                      \
  } while (0)
  if (M == 16 && al16) {
    if (long_lists) VLQ_SCAN_LAUNCH(16, true); else VLQ_SCAN_LAUNCH(16, false);
  } else if (M == 8 && al16) {
    if (long_lists) VLQ_SCAN_LAUNCH(8, true); else VLQ_SCAN_LAUNCH(8, false);
  } else {
    if (long_lists) VLQ_SCAN_LAUNCH(0, true); else VLQ_SCAN_LAUNCH(0, false);
  }
#undef VLQ_SCAN_LAUNCH
  return last_error();
}

int vlq_merge_topk(const float* D, const int64_t* I, int R, int64_t nq, int k, float* outD, int64_t* outI,
                   vlq_stream_t stream) {
  if (R <= 0 || nq < 0 || k <= 0 || k > VLQ_MAX_K) return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  if (!D || !I || !outD || !outI) return VLQ_EINVAL;
  const int cap = select_capacity(k, Q_THREADS, Q_BATCH, (long long)R * k);
  const size_t smem = select_smem_bytes(cap);
  VLQ_LAUNCH(merge_topk_kernel, (unsigned)nq, Q_THREADS, smem, as_stream(stream), D, I,
             (const unsigned char* const*)nullptr, (size_t)0, (size_t)0, R, nq, k, cap, outD, outI);
  return last_error();
}

int vlq_merge_topk_peers(const void* const* peer_bufs, size_t d_offset_bytes, size_t i_offset_bytes, int R, int64_t nq,
                         int k, float* outD, int64_t* outI, vlq_stream_t stream) {
  if (R <= 0 || nq < 0 || k <= 0 || k > VLQ_MAX_K || d_offset_bytes % 4 != 0 || i_offset_bytes % 8 != 0) return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  if (!peer_bufs || !outD || !outI) return VLQ_EINVAL;
  const int cap = select_capacity(k, Q_THREADS, Q_BATCH, (long long)R * k);
  const size_t smem = select_smem_bytes(cap);
  VLQ_LAUNCH(merge_topk_kernel, (unsigned)nq, Q_THREADS, smem, as_stream(stream), (const float*)nullptr,
             (const int64_t*)nullptr, reinterpret_cast<const unsigned char* const*>(peer_bufs), d_offset_bytes,
             i_offset_bytes, R, nq, k, cap, outD, outI);
  return last_error();
}

int vlq_gather_peer_slices(const void* const* peer_bufs, int R, int self, const int64_t* arr_offset_bytes, int narr,
                           int64_t nq, int64_t row_bytes, vlq_stream_t stream) {
  if (R <= 0 || self < 0 || self >= R || narr <= 0 || narr > 4 || nq < 0 || row_bytes <= 0 || (row_bytes & 15)) return VLQ_EINVAL;
  if (nq == 0 || R == 1) return VLQ_OK;
  if (!peer_bufs || !arr_offset_bytes) return VLQ_EINVAL;
  PeerSlices ps{};
  for (int a = 0; a < narr; a++) {
    if (arr_offset_bytes[a] < 0 || (arr_offset_bytes[a] & 15)) return VLQ_EINVAL;
    ps.arr_off[a] = arr_offset_bytes[a];
  }
  const int64_t per = (nq / R + 1) * row_bytes / 16;  // 16-byte words of the largest slice
  unsigned gx = (unsigned)((per + 255) / 256);
  if (gx > 64) gx = 64;
  if (gx < 1) gx = 1;
  VLQ_LAUNCH(gather_peer_slices_kernel, dim3(gx, (unsigned)R, (unsigned)narr), 256, 0, as_stream(stream),
             reinterpret_cast<const unsigned char* const*>(peer_bufs), R, self, ps, nq, row_bytes);
  return last_error();
}

size_t vlq_knn_graph_workspace_bytes(int C, int E) {
  int tr = graph_tile_rows(C);
  size_t b = (size_t)tr * C * sizeof(float);
  b = (b + 255) & ~size_t(255);
  b += ((size_t)tr * (E + 1) * sizeof(float) + 255) & ~size_t(255);
  b += ((size_t)tr * (E + 1) * sizeof(int) + 255) & ~size_t(255);
  return b;
}

int vlq_knn_graph(const float* cent, const float* cnorm, int C, int d, int E, int* edge, float* edge_d2,
                  void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  if (!cent || !cnorm || !edge || !edge_d2 || !workspace || C <= 1 || d <= 0 || E <= 0 || E + 1 > C ||
      E + 1 > VLQ_MAX_K)
    return VLQ_EINVAL;
  if (workspace_bytes < vlq_knn_graph_workspace_bytes(C, E)) return VLQ_EWORKSPACE;
  const int tr = graph_tile_rows(C);
  unsigned char* p = static_cast<unsigned char*>(workspace);
  float* Dt = reinterpret_cast<float*>(p);
  size_t off = ((size_t)tr * C * sizeof(float) + 255) & ~size_t(255);
  float* val = reinterpret_cast<float*>(p + off);
  off += ((size_t)tr * (E + 1) * sizeof(float) + 255) & ~size_t(255);
  int* idx = reinterpret_cast<int*>(p + off);
  for (int r0 = 0; r0 < C; r0 += tr) {
    const int rows = (C - r0) < tr ? (C - r0) : tr;
    int rc = vlq_l2_distances(cent + (size_t)r0 * d, rows, d, cent, cnorm, C, Dt, C, stream);
    if (rc) return rc;
    // exact flag of the reference: + ||c_i||^2 on the winners (sumAlongRows)
    rc = vlq_select_rows(Dt, rows, C, C, E + 1, cnorm + r0, val, idx, stream);
    if (rc) return rc;
    VLQ_LAUNCH(drop_rank0_kernel, (unsigned)div_up((int64_t)rows * E, 256), 256, 0, as_stream(stream), val, idx,
               (int64_t)rows, E, edge + (size_t)r0 * E, edge_d2 + (size_t)r0 * E);
  }
  return last_error();
}

}  // extern "C"
