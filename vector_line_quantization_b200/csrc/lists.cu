// Inverted-list construction on the device (SURVEY.md 8a row a9).
// (Stored layout: the M code bytes of the entry at list position pos are rotated by pos mod M, see scan.cuh.)
//
// The reference keeps one growable array per list and appends on the host with a hash map and per-byte copies
// (gpu/GpuIndexIVFPQ.cu:741-905, gpu/impl/InvertedListAppend.cu:20-120).  Here the lists are one CSR slab
// (offsets[nlists+1]; codes / lamq / kappa / ids list-major, each list 16-byte friendly for the scan) and an add is a
// stable counting sort of the new entries merged behind the existing ones:
//   1. histogram of the new list ids                         (atomics on int32 counters)
//   2. exclusive scan -> new_base; out_offsets = old_offsets + new_base
//   3. scatter of the new entry ordinals with a per-list cursor (arbitrary order inside a list) ...
//   4. ... made deterministic: each list segment is sorted by ordinal = arrival order (what push_back gives)
//   5. old entries are copied to their new place; new entries are gathered behind them.
#include "scan.cuh"

namespace vlq {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void hist_kernel(const int* __restrict__ list, int64_t n, int* __restrict__ counts) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    int l = list[i];
    if (l >= 0) atomicAdd(&counts[l], 1);
  }
}

__device__ __forceinline__ int64_t block_exscan(int64_t v, int64_t* total, int64_t* wsum) {
  // exclusive scan of one value per thread across the block (SCAN_THREADS threads)
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  int64_t inc = v;
#pragma unroll
  for (int o = 1; o < kWarp; o <<= 1) {
    int64_t t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == kWarp - 1) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int64_t w = lane < SCAN_THREADS / kWarp ? wsum[lane] : 0;
    int64_t winc = w;
#pragma unroll
    for (int o = 1; o < kWarp; o <<= 1) {
      int64_t t = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += t;
    }
    if (lane < SCAN_THREADS / kWarp) wsum[lane] = winc - w;
    if (lane == SCAN_THREADS / kWarp - 1) *total = winc;
  }
  __syncthreads();
  int64_t r = inc - v + wsum[warp];
  __syncthreads();
  return r;
}

// pass 1: per-tile totals
__global__ void scan_tile_sums_kernel(const int* __restrict__ counts, int64_t n, int64_t* __restrict__ tile_sums) {
  __shared__ int64_t wsum[SCAN_THREADS / kWarp];
  __shared__ int64_t total;
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int64_t s = 0;
#pragma unroll
  for (int t = 0; t < SCAN_ITEMS; t++)
    if (base + t < n) s += counts[base + t];
  block_exscan(s, &total, wsum);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
// pass 2: exclusive scan of the tile totals by one block
__global__ void scan_tile_offsets_kernel(int64_t* __restrict__ tile_sums, int64_t ntiles) {
  __shared__ int64_t wsum[SCAN_THREADS / kWarp];
  __shared__ int64_t total;
  int64_t carry = 0;
  for (int64_t b = 0; b < ntiles; b += SCAN_THREADS) {
    int64_t i = b + threadIdx.x;
    int64_t v = i < ntiles ? tile_sums[i] : 0;
    int64_t ex = block_exscan(v, &total, wsum);
    if (i < ntiles) tile_sums[i] = carry + ex;
    carry += total;
    __syncthreads();
  }
}
// pass 3: new_base[l] (exclusive), out_offsets[l] = old_offsets[l] + new_base[l]; element nlists gets the totals
__global__ void scan_finish_kernel(const int* __restrict__ counts, int64_t n, const int64_t* __restrict__ tile_sums,
                                   const int64_t* __restrict__ old_offsets, int64_t* __restrict__ new_base,
                                   int64_t* __restrict__ out_offsets) {
  __shared__ int64_t wsum[SCAN_THREADS / kWarp];
  __shared__ int64_t total;
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int64_t v[SCAN_ITEMS];
  int64_t s = 0;
#pragma unroll
  for (int t = 0; t < SCAN_ITEMS; t++) {
    v[t] = base + t < n ? counts[base + t] : 0;
    s += v[t];
  }
  int64_t ex = block_exscan(s, &total, wsum) + tile_sums[blockIdx.x];
#pragma unroll
  for (int t = 0; t < SCAN_ITEMS; t++) {
    int64_t l = base + t;
    if (l < n) {
      new_base[l] = ex;
      out_offsets[l] = (old_offsets ? old_offsets[l] : 0) + ex;
    }
    ex += v[t];
    if (l == n - 1) {
      new_base[n] = ex;
      out_offsets[n] = (old_offsets ? old_offsets[n] : 0) + ex;
    }
  }
}

__global__ void scatter_ordinals_kernel(const int* __restrict__ list, int64_t n, const int64_t* __restrict__ new_base,
                                        int* __restrict__ cursor, uint32_t* __restrict__ perm) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    int l = list[i];
    if (l < 0) continue;
    int pos = atomicAdd(&cursor[l], 1);
    perm[new_base[l] + pos] = (uint32_t)i;
  }
}

// one block per list: sort its segment of ordinals ascending.  Mirrored-merge bitonic network: every
// compare-exchange is ascending, so a virtual +inf tail (indices >= len) never moves and needs no storage.
constexpr int SEG_THREADS = 128;
constexpr int SEG_SMEM = 2048;
template <typename Ptr>
__device__ __forceinline__ void seg_bitonic(Ptr v, int64_t len, int64_t S) {
  for (int64_t k2 = 2; k2 <= S; k2 <<= 1) {
    const int64_t half = k2 >> 1;
    for (int64_t t = threadIdx.x; t < (S >> 1); t += SEG_THREADS) {
      int64_t blk = t / half, off = t % half;
      int64_t i = blk * k2 + off, m = blk * k2 + (k2 - 1 - off);
      if (m < len) {
        uint32_t a = v[i], c = v[m];
        if (a > c) {
          v[i] = c;
          v[m] = a;
        }
      }
    }
    __syncthreads();
    for (int64_t j = k2 >> 2; j > 0; j >>= 1) {
      for (int64_t t = threadIdx.x; t < (S >> 1); t += SEG_THREADS) {
        int64_t i = 2 * t - (t & (j - 1));
        int64_t m = i | j;
        if (m < len) {
          uint32_t a = v[i], c = v[m];
          if (a > c) {
            v[i] = c;
            v[m] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}
__global__ void __launch_bounds__(SEG_THREADS)
seg_sort_kernel(const int64_t* __restrict__ new_base, int64_t nlists, uint32_t* __restrict__ perm) {
  __shared__ uint32_t sk[SEG_SMEM];
  for (int64_t l = blockIdx.x; l < nlists; l += gridDim.x) {
    const int64_t b = new_base[l];
    const int64_t len = new_base[l + 1] - b;
    if (len <= 1) continue;  // uniform across the block
    uint32_t* seg = perm + b;
    int64_t S = 2;
    while (S < len) S <<= 1;
    if (len <= SEG_SMEM) {
      for (int i = threadIdx.x; i < len; i += SEG_THREADS) sk[i] = seg[i];
      __syncthreads();
      seg_bitonic(sk, len, S);
      for (int i = threadIdx.x; i < len; i += SEG_THREADS) seg[i] = sk[i];
    } else {
      __syncthreads();
      seg_bitonic(seg, len, S);  // rare: a single list received > 2048 entries in one commit
    }
    __syncthreads();
  }
}

// canonical code (arrival order arrays) -> stored code of the entry at list position pos: stored[j] = code[(j + pos) mod M]
__device__ __forceinline__ void store_code_rotated(uint8_t* dst, const uint8_t* src, int M, int64_t pos) {
  if (M == 16) {
    const uint4 c = *reinterpret_cast<const uint4*>(src);
    uint32_t w[4] = {c.x, c.y, c.z, c.w};
    rot16(w, (int)(pos & 15));
    *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
  } else if (M == 8) {
    const uint2 c = *reinterpret_cast<const uint2*>(src);
    uint32_t w[2] = {c.x, c.y};
    rot8(w, (int)(pos & 7));
    *reinterpret_cast<uint2*>(dst) = make_uint2(w[0], w[1]);
  } else {
    int j = (int)(pos % M);
    for (int t = 0; t < M; t++) {
      dst[t] = src[j];
      j = j + 1 == M ? 0 : j + 1;
    }
  }
}

__device__ __forceinline__ void copy_code(uint8_t* dst, const uint8_t* src, int M) {
  if (M == 16) {
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
  } else if (M == 8) {
    *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<const uint2*>(src);
  } else if (M % 4 == 0) {
    for (int t = 0; t < M; t += 4) *reinterpret_cast<uint32_t*>(dst + t) = *reinterpret_cast<const uint32_t*>(src + t);
  } else {
    for (int t = 0; t < M; t++) dst[t] = src[t];
  }
}

struct ListArrays {
  uint8_t* codes;
  uint8_t* lamq;
  float* kappa;
  int64_t* ids;
};
struct ConstListArrays {
  const uint8_t* codes;
  const uint8_t* lamq;
  const float* kappa;
  const int64_t* ids;
};

__global__ void gather_new_kernel(const uint32_t* __restrict__ perm, int64_t nlists, const int* __restrict__ new_list,
                                  const int64_t* __restrict__ new_base, const int64_t* __restrict__ old_offsets,
                                  const int64_t* __restrict__ out_offsets, ConstListArrays src, ListArrays dst, int M) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t live = new_base[nlists];  // entries with list id < 0 (invalid vectors) were never scattered
  for (; j < live; j += stride) {
    uint32_t s = perm[j];
    int l = new_list[s];
    int64_t old_len = old_offsets ? old_offsets[l + 1] - old_offsets[l] : 0;
    const int64_t pos = old_len + (j - new_base[l]);  // position inside the list
    int64_t o = out_offsets[l] + pos;
    store_code_rotated(dst.codes + o * M, src.codes + (int64_t)s * M, M, pos);
    dst.lamq[o] = src.lamq[s];
    dst.kappa[o] = src.kappa[s];
    dst.ids[o] = src.ids[s];
  }
}

__global__ void copy_old_kernel(int64_t n_old, int64_t nlists, const int64_t* __restrict__ old_offsets,
                                const int64_t* __restrict__ out_offsets, ConstListArrays src, ListArrays dst, int M) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n_old; i += stride) {
    // list of entry i: largest l with old_offsets[l] <= i
    int64_t lo = 0, hi = nlists;
    while (hi - lo > 1) {
      int64_t mid = (lo + hi) >> 1;
      if (old_offsets[mid] <= i) lo = mid; else hi = mid;
    }
    int64_t o = out_offsets[lo] + (i - old_offsets[lo]);
    copy_code(dst.codes + o * M, src.codes + i * M, M);
    dst.lamq[o] = src.lamq[i];
    dst.kappa[o] = src.kappa[i];
    dst.ids[o] = src.ids[i];
  }
}

struct ListWs {
  int* counts;         // [nlists]
  int* cursor;         // [nlists]
  int64_t* new_base;   // [nlists+1]
  int64_t* tile_sums;  // [ntiles]
  uint32_t* perm;      // [n_new]
  size_t bytes;
};
static ListWs carve(void* ws, int64_t n_new, int64_t nlists) {
  auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
  ListWs w{};
  size_t off = 0;
  unsigned char* p = static_cast<unsigned char*>(ws);
  w.counts = reinterpret_cast<int*>(p + off); off = align(off + sizeof(int) * nlists);
  w.cursor = reinterpret_cast<int*>(p + off); off = align(off + sizeof(int) * nlists);
  w.new_base = reinterpret_cast<int64_t*>(p + off); off = align(off + sizeof(int64_t) * (nlists + 1));
  w.tile_sums = reinterpret_cast<int64_t*>(p + off); off = align(off + sizeof(int64_t) * (div_up(nlists, SCAN_TILE) + 1));
  w.perm = reinterpret_cast<uint32_t*>(p + off); off = align(off + sizeof(uint32_t) * (n_new > 0 ? n_new : 1));
  w.bytes = off;
  return w;
}

// ---------------------------------------------------------------------------------------------- kappa for loaded lists
// kappa = ||p||^2 + 2 anchor.p for entries that arrive without it (lists read from the reference's .db* files).
// Same per-lane order of operations as line_encode_kernel, so a reloaded index scans bit-identically.
__global__ void recompute_kappa_kernel(int64_t n, int64_t nlists, const int64_t* __restrict__ offsets,
                                       const uint8_t* __restrict__ codes, const uint8_t* __restrict__ lamq,
                                       const float* __restrict__ cent, int d, const int* __restrict__ edge, int E,
                                       const float* __restrict__ lambda_cb, const float* __restrict__ pq, int M,
                                       float* __restrict__ kappa) {
  const int lane = threadIdx.x % kWarp;
  const int dsub = d / M;
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x / kWarp) + threadIdx.x / kWarp; i < n;
       i += (int64_t)gridDim.x * (blockDim.x / kWarp)) {
    int64_t lo = 0, hi = nlists;  // list of entry i: largest l with offsets[l] <= i
    while (hi - lo > 1) {
      int64_t mid = (lo + hi) >> 1;
      if (offsets[mid] <= i) lo = mid; else hi = mid;
    }
    const int A = (int)(lo / E);
    const int s = edge[lo];
    const int rot = (int)((i - offsets[lo]) % M);  // stored[j] = code[(j + pos) mod M]
    const float lh = lambda_cb[lamq[i]];
    const float oml = 1.f - lh;
    float kp = 0.f;
    for (int j = lane; j < d; j += kWarp) {
      const float anc = __fadd_rn(__fmul_rn(oml, cent[(int64_t)A * d + j]), __fmul_rn(lh, cent[(int64_t)s * d + j]));
      const int m = j / dsub, tt = j % dsub;
      const float pv = pq[((size_t)m * 256 + codes[i * M + (m - rot + M) % M]) * dsub + tt];
      kp = fmaf(pv, pv, kp);
      kp = fmaf(2.f * anc, pv, kp);
    }
    kp = warp_sum(kp);
    if (lane == 0) kappa[i] = kp;
  }
}

// ---------------------------------------------------------------------------------------------- k-means update (f1)
// Deterministic restatement of km_update_centroids' accumulation (utils.cpp:1385-1417): rows are grouped by centroid
// with the same stable counting sort as the list build, then one warp per centroid adds its rows IN ROW ORDER
// (fp32, lane j owns dimensions j, j+32, ...), and divides by the count.  The empty-cluster split
// (utils.cpp:1419-1446) is sequential RNG logic and stays on the host (host/clustering.cpp).
__global__ void km_mean_kernel(const float* __restrict__ x, int d, const uint32_t* __restrict__ perm,
                               const int64_t* __restrict__ base, int k, float* __restrict__ centroids,
                               int* __restrict__ counts) {
  int c = blockIdx.x * (blockDim.x / kWarp) + threadIdx.x / kWarp;
  if (c >= k) return;
  const int lane = threadIdx.x % kWarp;
  const int64_t b = base[c], e = base[c + 1];
  for (int j0 = 0; j0 < d; j0 += 8 * kWarp) {
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int64_t r = b; r < e; r++) {
      const float* xr = x + (int64_t)perm[r] * d;
#pragma unroll
      for (int t = 0; t < 8; t++) {
        int j = j0 + lane + 32 * t;
        if (j < d) acc[t] = __fadd_rn(acc[t], xr[j]);
      }
    }
    const float ni = (float)(e - b);
#pragma unroll
    for (int t = 0; t < 8; t++) {
      int j = j0 + lane + 32 * t;
      if (j < d) centroids[(int64_t)c * d + j] = (e > b) ? acc[t] / ni : 0.f;
    }
  }
  if (lane == 0) counts[c] = (int)(e - b);
}

// ------------------------------------------------------------------------------------------------ candidate lists
// ids of the entries of the W selected lines of a query, in line order, first k of them (the reference's candidate-recall
// tool IVFPQ::queryGraph1, gpu/impl/IVFPQ.cu:778-870, walks the lists on the host); unused slots get -1
__global__ void __launch_bounds__(256)
gather_candidates_kernel(const int* __restrict__ line_list, int W, const int64_t* __restrict__ offsets,
                         const int64_t* __restrict__ ids, int64_t k, int64_t* __restrict__ out) {
  extern __shared__ int64_t pre[];  // [W + 1] exclusive prefix of the list lengths
  const int64_t q = blockIdx.x;
  const int* lq = line_list + q * W;
  if (threadIdx.x == 0) {
    int64_t run = 0;
    for (int w = 0; w < W; w++) {
      pre[w] = run;
      const int l = lq[w];
      if (l >= 0) run += offsets[l + 1] - offsets[l];
    }
    pre[W] = run;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int w = warp; w < W; w += 8) {
    const int l = lq[w];
    if (l < 0 || pre[w] >= k) continue;
    const int64_t st = offsets[l], n = min(pre[w + 1], k) - pre[w];
    for (int64_t i = lane; i < n; i += 32) out[q * k + pre[w] + i] = ids[st + i];
  }
  const int64_t tot = min(pre[W], k);
  for (int64_t i = tot + threadIdx.x; i < k; i += 256) out[q * k + i] = -1;
}

// ------------------------------------------------------------------------------------------------ entry removal
// Stable stream compaction of the slab (IndexIVF::remove_ids, but the survivors keep their order).  The slab is cut into
// tiles of REM_TILE entries, one block each; word w of a tile is the keep mask of its entries 32 w .. 32 w + 31.  Because
// the slab is list-major, the global survivor prefix of an entry is its destination, and the survivor prefix at
// offsets[l] is the new offsets[l].  Workspace: the keep mask (n / 8 bytes) and one int64 per tile.
constexpr int REM_WORDS = SCAN_THREADS;  // one mask word per thread
constexpr int REM_TILE = REM_WORDS * kWarp;
constexpr int REM_LISTS = 1024;          // list starts a tile of the apply pass keeps in shared memory

// index of id in the sorted batch[0 .. nb), or -1
__device__ __forceinline__ int64_t batch_slot(int64_t id, const int64_t* __restrict__ batch, int64_t nb) {
  if (nb == 0 || id < batch[0] || id > batch[nb - 1]) return -1;
  int64_t a = 0, b = nb;  // lower bound of id in the sorted batch
  while (a < b) {
    const int64_t mid = (a + b) >> 1;
    if (batch[mid] < id) a = mid + 1; else b = mid;
  }
  return batch[a] == id ? a : -1;
}

__device__ __forceinline__ bool removed_id(int64_t id, int64_t lo, int64_t hi, const int64_t* __restrict__ batch,
                                           int64_t nb) {
  if (id >= lo && id < hi) return true;
  return batch_slot(id, batch, nb) >= 0;
}

// largest l in [lo, hi] with offsets[l] <= p (offsets[lo] <= p)
__device__ __forceinline__ int64_t list_of(const int64_t* offsets, int64_t lo, int64_t hi, int64_t p) {
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (offsets[mid] <= p) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// pass 1: keep mask, survivors per tile (tile_sums), and for every list that starts inside the tile its survivor prefix
// relative to the tile (rem_offsets_kernel adds the tile's base once the tile totals are scanned)
__global__ void __launch_bounds__(SCAN_THREADS)
rem_mark_kernel(int64_t n, int64_t nlists, const int64_t* __restrict__ offsets, const int64_t* __restrict__ ids,
                int64_t lo, int64_t hi, const int64_t* __restrict__ batch, int64_t nb, uint32_t* __restrict__ mask,
                int64_t* __restrict__ tile_sums, int64_t* __restrict__ out_offsets) {
  __shared__ uint32_t sword[REM_WORDS];
  __shared__ int64_t spre[REM_WORDS];
  __shared__ int64_t wsum[SCAN_THREADS / kWarp];
  __shared__ int64_t total;
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  const int64_t base = (int64_t)blockIdx.x * REM_TILE;
#pragma unroll 4
  for (int it = 0; it < REM_WORDS / (SCAN_THREADS / kWarp); it++) {
    const int w = it * (SCAN_THREADS / kWarp) + warp;
    const int64_t e = base + (int64_t)w * kWarp + lane;
    const bool keep = e < n && !removed_id(ids[e], lo, hi, batch, nb);
    const uint32_t bits = __ballot_sync(kFull, keep);
    if (lane == 0) {
      sword[w] = bits;
      mask[(int64_t)blockIdx.x * REM_WORDS + w] = bits;
    }
  }
  __syncthreads();
  spre[threadIdx.x] = block_exscan(__popc(sword[threadIdx.x]), &total, wsum);
  if (threadIdx.x == 0) {
    tile_sums[blockIdx.x] = total;
    if (blockIdx.x == 0) tile_sums[gridDim.x] = 0;  // the exclusive scan leaves the survivor count here
  }
  __syncthreads();
  // lists l with base <= offsets[l] < min(base + REM_TILE, n); lists starting at n are finished by rem_offsets_kernel
  const int64_t end = min(base + REM_TILE, n);
  int64_t a = 0, b = nlists;  // first l with offsets[l] >= base
  while (a < b) {
    const int64_t mid = (a + b) >> 1;
    if (offsets[mid] < base) a = mid + 1; else b = mid;
  }
  for (int64_t l = a + threadIdx.x; l < nlists; l += SCAN_THREADS) {
    const int64_t p = offsets[l];
    if (p >= end) break;
    const int r = (int)(p - base);
    out_offsets[l] = spre[r / kWarp] + __popc(sword[r / kWarp] & ((1u << (r % kWarp)) - 1u));
  }
}

// tile_sums holds the exclusive prefix of the tile totals (tile_sums[ntiles] = survivor count)
__global__ void rem_offsets_kernel(int64_t n, int64_t nlists, const int64_t* __restrict__ offsets,
                                   const int64_t* __restrict__ tile_sums, int64_t ntiles,
                                   int64_t* __restrict__ out_offsets) {
  for (int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; l <= nlists; l += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = l < nlists ? offsets[l] : n;
    out_offsets[l] = p < n ? out_offsets[l] + tile_sums[p / REM_TILE] : tile_sums[ntiles];
  }
}

// pass 2: the in-tile prefix is rebuilt from the mask; every survivor is copied to its prefix and its code word re-rotated
// from its old list position p to its new one p' (store_code_rotated by (p' - p) mod M)
__global__ void __launch_bounds__(SCAN_THREADS)
rem_apply_kernel(int64_t n, int64_t nlists, int M, const int64_t* __restrict__ offsets,
                 const int64_t* __restrict__ out_offsets, const uint32_t* __restrict__ mask,
                 const int64_t* __restrict__ tile_sums, ConstListArrays src, ListArrays dst) {
  __shared__ uint32_t sword[REM_WORDS];
  __shared__ int64_t spre[REM_WORDS];
  __shared__ int64_t soff[REM_LISTS], sout[REM_LISTS];
  __shared__ int64_t wsum[SCAN_THREADS / kWarp];
  __shared__ int64_t total;
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  const int64_t base = (int64_t)blockIdx.x * REM_TILE;
  const int64_t last = min(base + REM_TILE, n) - 1;
  const uint32_t mine = mask[(int64_t)blockIdx.x * REM_WORDS + threadIdx.x];
  sword[threadIdx.x] = mine;
  spre[threadIdx.x] = block_exscan(__popc(mine), &total, wsum) + tile_sums[blockIdx.x];  // syncs the block
  if (total == 0) return;  // uniform
  // the lists the tile spans: [l0, l1]
  const int64_t l0 = list_of(offsets, 0, nlists - 1, base);
  const int64_t l1 = list_of(offsets, l0, nlists - 1, last);
  const bool cached = l1 - l0 < REM_LISTS;
  if (cached) {
    for (int64_t i = threadIdx.x; i <= l1 - l0; i += SCAN_THREADS) {
      soff[i] = offsets[l0 + i];
      sout[i] = out_offsets[l0 + i];
    }
  }
  __syncthreads();
#pragma unroll 2
  for (int it = 0; it < REM_WORDS / (SCAN_THREADS / kWarp); it++) {
    const int w = it * (SCAN_THREADS / kWarp) + warp;
    const uint32_t bits = sword[w];
    if (!((bits >> lane) & 1u)) continue;
    const int64_t e = base + (int64_t)w * kWarp + lane;
    const int64_t o = spre[w] + __popc(bits & ((1u << lane) - 1u));
    int64_t ob, nb;
    if (cached) {
      const int64_t i = list_of(soff, 0, l1 - l0, e);
      ob = soff[i];
      nb = sout[i];
    } else {
      const int64_t l = list_of(offsets, l0, l1, e);
      ob = offsets[l];
      nb = out_offsets[l];
    }
    int64_t rot = ((o - nb) - (e - ob)) % M;  // new position - old position (<= 0)
    if (rot < 0) rot += M;
    store_code_rotated(dst.codes + o * M, src.codes + e * M, M, rot);
    dst.lamq[o] = src.lamq[e];
    dst.kappa[o] = src.kappa[e];
    dst.ids[o] = src.ids[e];
  }
}

struct RemWs {
  uint32_t* mask;      // [ntiles * REM_WORDS]
  int64_t* tile_sums;  // [ntiles + 1]
  int64_t ntiles;
  size_t bytes;
};
static RemWs carve_rem(void* ws, int64_t n) {
  auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
  RemWs w{};
  w.ntiles = div_up(n, REM_TILE);
  unsigned char* p = static_cast<unsigned char*>(ws);
  size_t off = 0;
  w.mask = reinterpret_cast<uint32_t*>(p + off); off = align(off + sizeof(uint32_t) * REM_WORDS * w.ntiles);
  w.tile_sums = reinterpret_cast<int64_t*>(p + off); off = align(off + sizeof(int64_t) * (w.ntiles + 1));
  w.bytes = off;
  return w;
}

// ------------------------------------------------------------------------------------------------ entry lookup / decode
// Lookup: one pass over ids[n]; the slot of an id is id - lo (range) or its index in the sorted keys (batch), and the
// slot keeps the lowest slab index that carries it (atomicMin: the result does not depend on the schedule).  There is
// no id -> slab map to keep in step with add / remove_ids: a lookup costs one read of the ids.
constexpr int64_t kNoPos = INT64_MAX;
constexpr int LOOKUP_UNROLL = 4;

__global__ void lookup_init_kernel(int64_t* __restrict__ out_pos, int64_t nslots,
                                   unsigned long long* __restrict__ found) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nslots; i += stride) out_pos[i] = kNoPos;
  if (blockIdx.x == 0 && threadIdx.x == 0) *found = 0;
}

__global__ void __launch_bounds__(SCAN_THREADS)
lookup_mark_kernel(int64_t n, const int64_t* __restrict__ ids, int64_t lo, int64_t nslots,
                   const int64_t* __restrict__ keys, int64_t* __restrict__ out_pos) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e0 < n; e0 += stride * LOOKUP_UNROLL) {
    int64_t id[LOOKUP_UNROLL];
#pragma unroll
    for (int u = 0; u < LOOKUP_UNROLL; u++) {  // the loads of all four entries first
      const int64_t e = e0 + u * stride;
      id[u] = e < n ? ids[e] : 0;
    }
#pragma unroll
    for (int u = 0; u < LOOKUP_UNROLL; u++) {
      const int64_t e = e0 + u * stride;
      if (e >= n) break;
      int64_t slot;
      if (keys) {
        slot = batch_slot(id[u], keys, nslots);
      } else {  // id - lo in unsigned arithmetic: no overflow for any lo <= id
        slot = (id[u] >= lo && (uint64_t)id[u] - (uint64_t)lo < (uint64_t)nslots) ? id[u] - lo : -1;
      }
      if (slot >= 0) atomicMin(reinterpret_cast<long long*>(out_pos + slot), (long long)e);
    }
  }
}

__global__ void __launch_bounds__(SCAN_THREADS)
lookup_finish_kernel(int64_t* __restrict__ out_pos, int64_t nslots, unsigned long long* __restrict__ found) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned long long cnt = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nslots; i += stride) {
    if (out_pos[i] == kNoPos) out_pos[i] = -1;
    else cnt++;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(kFull, cnt, o);
  if ((threadIdx.x % kWarp) == 0 && cnt) atomicAdd(found, cnt);
}

// Decode: x[j] = anchor[j] + pq[m][code_m][j - m dsub], m = j / dsub, one warp per entry with d spread over the lanes
// (coarse rows and codebook rows are gathered through L2; the output row is one coalesced store).  The list of slab
// index p is found by binary search over offsets; the stored code bytes are un-rotated by (p - offsets[l]) mod M.
//   VLQ:    anchor = (1 - lh) c + lh s,  c = cent[l / E], s = cent[edge[l]], lh = lambda_cb[lamq[p]]
//   IMI-PQ: anchor = [cb1[i1] | cb2[i2]],  l = i1 | i2 << nbits
// fp32, every operation rounded as written (no contraction), in the order shown: lh = 0 gives exactly c + p.
struct DecodeAnchor {
  const float* cent;       // VLQ: [C][d]
  const int* edge;         // VLQ: [nlists]
  const uint8_t* lamq;     // VLQ: [n entries]
  const float* lambda_cb;  // VLQ
  int E;
  const float* cb1;        // IMI: [K][d / 2]
  const float* cb2;
  int nbits;
};

template <bool IMI>
__global__ void __launch_bounds__(SCAN_THREADS)
decode_entries_kernel(int64_t n, const int64_t* pos, int64_t nlists, const int64_t* __restrict__ offsets,
                      const uint8_t* __restrict__ codes, const int64_t* __restrict__ ids, int M, int d,
                      const float* __restrict__ pq, DecodeAnchor an, float* __restrict__ out_x, int64_t* out_ids) {
  const int lane = threadIdx.x % kWarp;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) / kWarp;
  const int64_t nslab = offsets[nlists];
  const int dsub = d / M;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kWarp; r < n; r += nwarps) {
    const int64_t p = pos[r];
    __syncwarp();  // out_ids may alias pos: every lane has read pos[r] before lane 0 overwrites it
    float* o = out_x + r * d;
    if (p < 0 || p >= nslab) {
      for (int j = lane; j < d; j += kWarp) o[j] = __uint_as_float(0xffffffffu);
      if (out_ids && lane == 0) out_ids[r] = -1;
      continue;
    }
    const int64_t l = list_of(offsets, 0, nlists - 1, p);
    const int rot = (int)((p - offsets[l]) % M);
    const uint8_t* cw = codes + p * M;
    const float *a0, *a1;
    float lh = 0.f, oml = 1.f;
    if constexpr (IMI) {
      const int h = d / 2;
      a0 = an.cb1 + (l & ((1 << an.nbits) - 1)) * h;
      a1 = an.cb2 + (l >> an.nbits) * h;
    } else {
      a0 = an.cent + (l / an.E) * d;
      a1 = an.cent + (int64_t)an.edge[l] * d;
      lh = an.lambda_cb[an.lamq[p]];
      oml = __fsub_rn(1.f, lh);
    }
    for (int j = lane; j < d; j += kWarp) {
      const int m = j / dsub;
      int sb = m - rot;  // stored[(m - pos) mod M] = code[m]
      if (sb < 0) sb += M;
      const float pv = pq[((int64_t)m * 256 + cw[sb]) * dsub + (j - m * dsub)];
      float a;
      if constexpr (IMI) a = *(j < d / 2 ? a0 + j : a1 + (j - d / 2));
      else a = __fadd_rn(__fmul_rn(oml, a0[j]), __fmul_rn(lh, a1[j]));
      o[j] = __fadd_rn(a, pv);
    }
    if (out_ids && lane == 0) out_ids[r] = ids[p];
  }
}

static unsigned grid_for(int64_t items, int per_block) {
  const int64_t g = div_up(items, per_block);
  return (unsigned)(g < 1 ? 1 : (g < 148 * 16 ? g : 148 * 16));
}

int launch_exclusive_scan_i64(int64_t* v, int64_t n, cudaStream_t st) {
  VLQ_LAUNCH(scan_tile_offsets_kernel, 1, SCAN_THREADS, 0, st, v, n);
  return last_error();
}

}  // namespace vlq

using namespace vlq;

extern "C" int vlq_recompute_kappa(int64_t n, int64_t nlists, const int64_t* offsets, const uint8_t* codes,
                                   const uint8_t* lamq, const float* cent, int d, const int* edge, int E,
                                   const float* lambda_cb, const float* pq, int M, float* kappa, vlq_stream_t stream) {
  if (n < 0 || nlists <= 0 || d <= 0 || E <= 0 || M <= 0 || d % M != 0) return VLQ_EINVAL;
  if (n == 0) return VLQ_OK;
  if (!offsets || !codes || !lamq || !cent || !edge || !lambda_cb || !pq || !kappa) return VLQ_EINVAL;
  VLQ_LAUNCH(recompute_kappa_kernel, 148 * 8, 256, 0, as_stream(stream), n, nlists, offsets, codes, lamq, cent, d, edge,
             E, lambda_cb, pq, M, kappa);
  return last_error();
}

extern "C" size_t vlq_km_update_workspace_bytes(int64_t n, int k) { return carve(nullptr, n, k).bytes; }

extern "C" int vlq_km_update(const float* x, int64_t n, int d, const int* assign, int k, float* centroids, int* counts,
                             void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  if (!x || !assign || !centroids || !counts || !workspace || n <= 0 || d <= 0 || k <= 0) return VLQ_EINVAL;
  if (n >= (int64_t)0xffffffffll) return VLQ_EINVAL;
  ListWs w = carve(workspace, n, k);
  if (workspace_bytes < w.bytes) return VLQ_EWORKSPACE;
  cudaStream_t st = as_stream(stream);
  VLQ_CUDA_TRY(cudaMemsetAsync(w.counts, 0, sizeof(int) * k, st));
  VLQ_CUDA_TRY(cudaMemsetAsync(w.cursor, 0, sizeof(int) * k, st));
  const unsigned wide = 148 * 8;
  VLQ_LAUNCH(hist_kernel, wide, 256, 0, st, assign, n, w.counts);
  const int64_t ntiles = div_up(k, SCAN_TILE);
  VLQ_LAUNCH(scan_tile_sums_kernel, (unsigned)ntiles, SCAN_THREADS, 0, st, w.counts, (int64_t)k, w.tile_sums);
  VLQ_LAUNCH(scan_tile_offsets_kernel, 1, SCAN_THREADS, 0, st, w.tile_sums, ntiles);
  // out_offsets is not needed here: reuse the tail of new_base as a scratch target via tile_sums-sized dummy
  VLQ_LAUNCH(scan_finish_kernel, (unsigned)ntiles, SCAN_THREADS, 0, st, w.counts, (int64_t)k, w.tile_sums,
             (const int64_t*)nullptr, w.new_base, w.new_base);
  VLQ_LAUNCH(scatter_ordinals_kernel, wide, 256, 0, st, assign, n, w.new_base, w.cursor, w.perm);
  unsigned sgrid = (unsigned)(k < 148 * 64 ? k : 148 * 64);
  VLQ_LAUNCH(seg_sort_kernel, sgrid, SEG_THREADS, 0, st, w.new_base, (int64_t)k, w.perm);
  VLQ_LAUNCH(km_mean_kernel, (unsigned)div_up(k, 8), 256, 0, st, x, d, w.perm, w.new_base, k, centroids, counts);
  return last_error();
}

extern "C" size_t vlq_build_lists_workspace_bytes(int64_t n_new, int64_t nlists) {
  return carve(nullptr, n_new, nlists).bytes;
}

extern "C" int vlq_build_lists(int64_t nlists, int M, int64_t n_old, const int64_t* old_offsets,
                               const uint8_t* old_codes, const uint8_t* old_lamq, const float* old_kappa,
                               const int64_t* old_ids, int64_t n_new, const int* new_list, const uint8_t* new_codes,
                               const uint8_t* new_lamq, const float* new_kappa, const int64_t* new_ids,
                               int64_t* out_offsets, uint8_t* out_codes, uint8_t* out_lamq, float* out_kappa,
                               int64_t* out_ids, void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  if (nlists <= 0 || M <= 0 || n_old < 0 || n_new < 0 || !out_offsets || !workspace) return VLQ_EINVAL;
  if (n_new >= (int64_t)0xffffffffll) return VLQ_EINVAL;
  if (n_old > 0 && (!old_offsets || !old_codes || !old_lamq || !old_kappa || !old_ids)) return VLQ_EINVAL;
  if (n_new > 0 && (!new_list || !new_codes || !new_lamq || !new_kappa || !new_ids)) return VLQ_EINVAL;
  if ((n_old + n_new) > 0 && (!out_codes || !out_lamq || !out_kappa || !out_ids)) return VLQ_EINVAL;
  ListWs w = carve(workspace, n_new, nlists);
  if (workspace_bytes < w.bytes) return VLQ_EWORKSPACE;
  cudaStream_t st = as_stream(stream);
  const int64_t* oo = n_old > 0 ? old_offsets : nullptr;

  VLQ_CUDA_TRY(cudaMemsetAsync(w.counts, 0, sizeof(int) * nlists, st));
  VLQ_CUDA_TRY(cudaMemsetAsync(w.cursor, 0, sizeof(int) * nlists, st));
  const unsigned wide = 148 * 8;
  if (n_new > 0) VLQ_LAUNCH(hist_kernel, wide, 256, 0, st, new_list, n_new, w.counts);
  const int64_t ntiles = div_up(nlists, SCAN_TILE);
  VLQ_LAUNCH(scan_tile_sums_kernel, (unsigned)ntiles, SCAN_THREADS, 0, st, w.counts, nlists, w.tile_sums);
  VLQ_LAUNCH(scan_tile_offsets_kernel, 1, SCAN_THREADS, 0, st, w.tile_sums, ntiles);
  VLQ_LAUNCH(scan_finish_kernel, (unsigned)ntiles, SCAN_THREADS, 0, st, w.counts, nlists, w.tile_sums, oo, w.new_base,
             out_offsets);
  ConstListArrays osrc{old_codes, old_lamq, old_kappa, old_ids};
  ConstListArrays nsrc{new_codes, new_lamq, new_kappa, new_ids};
  ListArrays dst{out_codes, out_lamq, out_kappa, out_ids};
  if (n_new > 0) {
    VLQ_LAUNCH(scatter_ordinals_kernel, wide, 256, 0, st, new_list, n_new, w.new_base, w.cursor, w.perm);
    unsigned sgrid = (unsigned)(nlists < 148 * 64 ? nlists : 148 * 64);
    VLQ_LAUNCH(seg_sort_kernel, sgrid, SEG_THREADS, 0, st, w.new_base, nlists, w.perm);
  }
  if (n_old > 0) VLQ_LAUNCH(copy_old_kernel, wide, 256, 0, st, n_old, nlists, oo, out_offsets, osrc, dst, M);
  if (n_new > 0) {
    VLQ_LAUNCH(gather_new_kernel, wide, 256, 0, st, w.perm, nlists, new_list, w.new_base, oo, out_offsets, nsrc, dst, M);
  }
  return last_error();
}

extern "C" size_t vlq_remove_ids_workspace_bytes(int64_t n, int64_t /*nlists*/) {
  return carve_rem(nullptr, n < 0 ? 0 : n).bytes;
}

extern "C" int vlq_remove_ids_plan(int64_t nlists, int64_t n, const int64_t* offsets, const int64_t* ids,
                                   int64_t range_lo, int64_t range_hi, const int64_t* batch, int64_t n_batch,
                                   int64_t* out_offsets, void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  if (nlists < 1 || n < 0 || n_batch < 0 || !offsets || !out_offsets || !workspace) return VLQ_EINVAL;
  if ((n > 0 && !ids) || (n_batch > 0 && !batch)) return VLQ_EINVAL;
  RemWs w = carve_rem(workspace, n);
  if (workspace_bytes < w.bytes) return VLQ_EWORKSPACE;
  cudaStream_t st = as_stream(stream);
  if (n == 0) {
    VLQ_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, sizeof(int64_t) * (nlists + 1), st));
    return VLQ_OK;
  }
  VLQ_LAUNCH(rem_mark_kernel, (unsigned)w.ntiles, SCAN_THREADS, 0, st, n, nlists, offsets, ids, range_lo, range_hi, batch,
             n_batch, w.mask, w.tile_sums, out_offsets);
  VLQ_LAUNCH(scan_tile_offsets_kernel, 1, SCAN_THREADS, 0, st, w.tile_sums, w.ntiles + 1);
  const int64_t lgrid = div_up(nlists + 1, 256);
  const unsigned grid = (unsigned)(lgrid < 148 * 8 ? lgrid : 148 * 8);
  VLQ_LAUNCH(rem_offsets_kernel, grid, 256, 0, st, n, nlists, offsets, w.tile_sums, w.ntiles, out_offsets);
  return last_error();
}

extern "C" int vlq_remove_ids_apply(int64_t nlists, int M, int64_t n, const int64_t* offsets, const uint8_t* codes,
                                    const uint8_t* lamq, const float* kappa, const int64_t* ids, const int64_t* out_offsets,
                                    uint8_t* out_codes, uint8_t* out_lamq, float* out_kappa, int64_t* out_ids,
                                    const void* workspace, size_t workspace_bytes, vlq_stream_t stream) {
  if (nlists < 1 || M < 1 || M > 64 || n < 0 || !offsets || !out_offsets || !workspace) return VLQ_EINVAL;
  if (n > 0 && (!codes || !lamq || !kappa || !ids || !out_codes || !out_lamq || !out_kappa || !out_ids)) return VLQ_EINVAL;
  RemWs w = carve_rem(const_cast<void*>(workspace), n);
  if (workspace_bytes < w.bytes) return VLQ_EWORKSPACE;
  if (n == 0) return VLQ_OK;
  VLQ_LAUNCH(rem_apply_kernel, (unsigned)w.ntiles, SCAN_THREADS, 0, as_stream(stream), n, nlists, M, offsets,
             out_offsets, w.mask, w.tile_sums, ConstListArrays{codes, lamq, kappa, ids},
             ListArrays{out_codes, out_lamq, out_kappa, out_ids});
  return last_error();
}

extern "C" int vlq_lookup_ids(int64_t n, const int64_t* ids, int64_t range_lo, const int64_t* keys, int64_t nslots,
                              int64_t* out_pos, int64_t* out_found, vlq_stream_t stream) {
  if (n < 0 || nslots < 0 || !out_found || (n > 0 && !ids) || (nslots > 0 && !out_pos)) return VLQ_EINVAL;
  if (!keys && range_lo > INT64_MAX - nslots) return VLQ_EINVAL;
  cudaStream_t st = as_stream(stream);
  unsigned long long* found = reinterpret_cast<unsigned long long*>(out_found);
  if (nslots == 0) {
    VLQ_CUDA_TRY(cudaMemsetAsync(out_found, 0, sizeof(int64_t), st));
    return VLQ_OK;
  }
  const unsigned sgrid = grid_for(nslots, SCAN_THREADS);
  VLQ_LAUNCH(lookup_init_kernel, sgrid, SCAN_THREADS, 0, st, out_pos, nslots, found);
  if (n > 0)
    VLQ_LAUNCH(lookup_mark_kernel, grid_for(div_up(n, LOOKUP_UNROLL), SCAN_THREADS), SCAN_THREADS, 0, st, n, ids, range_lo,
               nslots, keys, out_pos);
  VLQ_LAUNCH(lookup_finish_kernel, sgrid, SCAN_THREADS, 0, st, out_pos, nslots, found);
  return last_error();
}

static int decode_launch(bool imi, int64_t n, const int64_t* pos, int64_t nlists, const int64_t* offsets,
                         const uint8_t* codes, const int64_t* ids, int M, int d, const float* pq, const DecodeAnchor& an,
                         float* out_x, int64_t* out_ids, vlq_stream_t stream) {
  if (n < 0 || nlists < 1 || M < 1 || M > 64 || d < 1 || d % M != 0) return VLQ_EINVAL;
  if (n > 0 && (!pos || !offsets || !codes || !pq || !out_x || (out_ids && !ids))) return VLQ_EINVAL;
  if (n == 0) return VLQ_OK;
  const unsigned grid = grid_for(n, SCAN_THREADS / kWarp);
  if (imi)
    VLQ_LAUNCH(decode_entries_kernel<true>, grid, SCAN_THREADS, 0, as_stream(stream), n, pos, nlists, offsets, codes, ids, M,
               d, pq, an, out_x, out_ids);
  else
    VLQ_LAUNCH(decode_entries_kernel<false>, grid, SCAN_THREADS, 0, as_stream(stream), n, pos, nlists, offsets, codes, ids,
               M, d, pq, an, out_x, out_ids);
  return last_error();
}

extern "C" int vlq_decode_entries(int64_t n, const int64_t* pos, int64_t nlists, const int64_t* offsets,
                                  const uint8_t* codes, const uint8_t* lamq, const int64_t* ids, int M, int d,
                                  const float* pq, const float* cent, const int* edge, int E, const float* lambda_cb,
                                  int nL, float* out_x, int64_t* out_ids, vlq_stream_t stream) {
  if (E < 1 || nlists % E != 0 || nL < 1 || nL > 256) return VLQ_EINVAL;
  if (n > 0 && (!lamq || !cent || !edge || !lambda_cb)) return VLQ_EINVAL;
  DecodeAnchor an{};
  an.cent = cent; an.edge = edge; an.lamq = lamq; an.lambda_cb = lambda_cb; an.E = E;
  return decode_launch(false, n, pos, nlists, offsets, codes, ids, M, d, pq, an, out_x, out_ids, stream);
}

extern "C" int vlq_imi_decode_entries(int64_t n, const int64_t* pos, const int64_t* offsets, const uint8_t* codes,
                                      const int64_t* ids, int M, int d, const float* pq, const float* cb1,
                                      const float* cb2, int nbits, float* out_x, int64_t* out_ids, vlq_stream_t stream) {
  if (nbits < 1 || nbits > 15 || d % 2 != 0) return VLQ_EINVAL;
  if (n > 0 && (!cb1 || !cb2)) return VLQ_EINVAL;
  DecodeAnchor an{};
  an.cb1 = cb1; an.cb2 = cb2; an.nbits = nbits;
  return decode_launch(true, n, pos, (int64_t)1 << (2 * nbits), offsets, codes, ids, M, d, pq, an, out_x, out_ids, stream);
}

extern "C" int vlq_gather_candidates(const int* line_list, int64_t nq, int W, const int64_t* offsets, const int64_t* ids,
                                     int64_t k, int64_t* out, vlq_stream_t stream) {
  using namespace vlq;
  if (nq < 0 || W <= 0 || W > VLQ_MAX_K || k <= 0) return VLQ_EINVAL;
  if (nq == 0) return VLQ_OK;
  if (!line_list || !offsets || !ids || !out) return VLQ_EINVAL;
  VLQ_LAUNCH(gather_candidates_kernel, (unsigned)nq, 256, sizeof(int64_t) * (W + 1), as_stream(stream), line_list, W, offsets,
             ids, k, out);
  return last_error();
}
