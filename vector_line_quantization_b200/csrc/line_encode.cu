// VLQ line stage + lambda quantiser + residual + PQ encode, fused (SURVEY.md 8a rows a5-a8).
//
// One warp per vector, persistent CTAs (grid = k x #SMs) with the PQ codebook staged once per CTA in shared memory in
// a [m][t][code] layout (lane j reads word j: conflict free).  Per vector the warp
//   1. keeps x in registers (lane j holds x[j + 32t]),
//   2. gathers the E+1 centroid rows A, s_0..s_{E-1} through L2 (coalesced 128 B per lane-row),
//   3. reduces the E+1 exact squared distances with shuffles, lane e then owns line e:
//        lambda_e = -0.5 (a - b - c2)/c2,  q_e = b + lambda^2 c2 + lambda (a - b - c2)     (triangle.cuh:54-87)
//   4. picks argmin q_e over 0 <= lambda_e <= 1, else the global argmin (ties -> lowest e)   (GpuIndexFlat.cu:517-550,
//      intended semantics, SURVEY Q1), quantises lambda against the 1-D codebook             (GpuIndexFlat.cu:579-596)
//   5. forms r = x - ((1-l) c_A + l c_s) in registers                                        (GpuIndexFlat.cu:1111-1122)
//   6. encodes r with the PQ: per sub-space arg-min over ksub codewords by direct differences, first minimum wins
//      (ProductQuantizer.cpp:311-336), and emits kappa = ||p||^2 + 2 anchor.p for the scan.
// Nothing but the final list id / lambda byte / M code bytes / kappa leaves the SM.
#include "common.cuh"
#include "pq4.cuh"

namespace vlq {

constexpr int LE_WARPS = 24;
constexpr int LE_THREADS = LE_WARPS * kWarp;
constexpr int LE_MAX_E = 64;

struct LineEncodeArgs {
  const float* x;
  int64_t n;
  int d;
  const int* assign;
  const float* cent;
  const int* edge;
  const float* edge_d2;
  int E;
  const float* lambda_cb;
  int nL;
  const float* pq;  // (M, ksub, dsub)
  int M, ksub, dsub;
  int pq_in_smem;
  int* out_list;
  float* out_lambda;
  uint8_t* out_lamq;
  uint8_t* out_codes;
  float* out_kappa;
  float* out_residual;
};

// Reduce 32 per-lane partial sums v[0..32) across the warp so that lane l ends with the total of v[l] (in v[0]):
// 31 shuffles instead of 32 x 5, and the additions pair up exactly like the xor-butterfly of warp_sum (same bits).
__device__ __forceinline__ void warp_transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int j = 0; j < o; j++) {
      const float send = up ? v[j] : v[j + o];
      const float keep = up ? v[j + o] : v[j];
      v[j] = keep + __shfl_xor_sync(kFull, send, o);
    }
  }
}

// A warp takes LE_V consecutive vectors at a time.  Phase A (per vector): line stage, lambda byte, residual -> per-warp
// shared memory.  Phase B (the LE_V vectors together): PQ encode -- every codeword component read from shared memory is
// used for LE_V vectors, which cuts the shared-memory instructions per multiply-add by LE_V (the loop was LSU-bound:
// one LDS per FSUB+FFMA pair).  Phase C (per vector): kappa and the outputs.  The arithmetic of every vector is
// unchanged (same operation order), so the results do not depend on the grouping.
constexpr int LE_V = 4;

template <int NPL>
__global__ void __launch_bounds__(LE_THREADS, 1) line_encode_kernel(LineEncodeArgs a) {
  extern __shared__ __align__(16) float smem[];
  // layout: [pq transposed: M*dsub*ksub floats (optional)] [per-warp r: LE_WARPS*LE_V*d] [per-warp scalars]
  //         [per-warp codes: LE_WARPS*LE_V*64 bytes]
  const int d = a.d, E = a.E, M = a.M, ksub = a.ksub, dsub = a.dsub;
  float* pqs = smem;
  float* rbuf = smem + (a.pq_in_smem ? (size_t)M * dsub * ksub : 0);
  int* sbuf = reinterpret_cast<int*>(rbuf + (size_t)LE_WARPS * LE_V * d);  // per warp, per vector: A, s, lq, lh
  uint8_t* cbuf = reinterpret_cast<uint8_t*>(sbuf + LE_WARPS * LE_V * 4);
  const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
  const bool encode = a.lambda_cb != nullptr;

  if (encode && a.pq_in_smem) {
    // pq[(m*ksub + j)*dsub + t]  ->  pqs[(m*dsub + t)*ksub + j]
    const int total = M * ksub * dsub;
    for (int i = threadIdx.x; i < total; i += LE_THREADS) {
      int t = i % dsub;
      int j = (i / dsub) % ksub;
      int m = i / (dsub * ksub);
      pqs[(m * dsub + t) * ksub + j] = a.pq[i];
    }
  }
  __syncthreads();

  float* r_w = rbuf + (size_t)warp * LE_V * d;
  int* sc_w = sbuf + warp * LE_V * 4;
  uint8_t* code_w = cbuf + warp * LE_V * 64;

  for (int64_t i0 = ((int64_t)blockIdx.x * LE_WARPS + warp) * LE_V; i0 < a.n;
       i0 += (int64_t)gridDim.x * LE_WARPS * LE_V) {
    // ------------------------------------------------------------------ phase A: line stage, lambda byte, residual
#pragma unroll 1
    for (int v = 0; v < LE_V; v++) {
      const int64_t i = i0 + v;
      float* r_s = r_w + v * d;
      if (lane == 0) sc_w[v * 4] = -1;
      if (i >= a.n) continue;  // warp-uniform
      float xv[NPL];
      const float* xr = a.x + i * d;
#pragma unroll
      for (int t = 0; t < NPL; t++) {
        int j = lane + 32 * t;
        xv[t] = j < d ? xr[j] : 0.f;
      }
      const int A = a.assign[i];
      if (A < 0) {  // invalid vector (NaN input): the reference skips it (GpuIndexIVFPQ.cu:751-755)
        if (lane == 0) {
          a.out_list[i] = -1;
          if (a.out_lambda) a.out_lambda[i] = 0.f;
        }
        continue;
      }
      const float* cA = a.cent + (int64_t)A * d;
      float cAv[NPL];
      float bp = 0.f;
#pragma unroll
      for (int t = 0; t < NPL; t++) {
        int j = lane + 32 * t;
        cAv[t] = j < d ? cA[j] : 0.f;
        float df = xv[t] - cAv[t];
        bp = fmaf(df, df, bp);
      }
      const float b = warp_sum(bp);

      // lane e (+32) owns edge e
      int my_s[2] = {0, 0};
      float my_a[2] = {0.f, 0.f};
      float my_c2[2] = {1.f, 1.f};
#pragma unroll
      for (int h = 0; h < 2; h++) {
        int e = lane + 32 * h;
        if (e < E) {
          my_s[h] = a.edge[(int64_t)A * E + e];
          my_c2[h] = a.edge_d2[(int64_t)A * E + e];
        }
      }
      for (int g = 0; g * 32 < E; g++) {  // 32 edges at a time: lane-private partial sums, one transposed reduction
        float part[32];
#pragma unroll
        for (int ee = 0; ee < 32; ee++) {
          const int e = g * 32 + ee;
          const int s = __shfl_sync(kFull, my_s[g], ee);  // edges beyond E read centroid 0 (result unused)
          const float* cs = a.cent + (int64_t)(e < E ? s : 0) * d;
          float ap = 0.f;
#pragma unroll
          for (int t = 0; t < NPL; t++) {
            int j = lane + 32 * t;
            float cv = j < d ? cs[j] : 0.f;
            float df = xv[t] - cv;
            ap = fmaf(df, df, ap);
          }
          part[ee] = ap;
        }
        warp_transpose_reduce32(part, lane);
        my_a[g] = part[0];
      }
      uint64_t kv = kKeyInf, ka = kKeyInf;
      float my_lam[2];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        int e = lane + 32 * h;
        float vv = my_a[h] - b - my_c2[h];
        float lam = -0.5f * vv / my_c2[h];                                 // project()
        float q2 = __fadd_rn(__fadd_rn(b, __fmul_rn(__fmul_rn(lam, lam), my_c2[h])), __fmul_rn(lam, vv));  // dist2()
        my_lam[h] = lam;
        if (e < E) {
          uint64_t key = make_key(q2, (uint32_t)e);
          ka = key < ka ? key : ka;
          if (lam >= 0.f && lam <= 1.f) kv = key < kv ? key : kv;
        }
      }
      kv = warp_min_u64(kv);
      ka = warp_min_u64(ka);
      const uint64_t kbest = kv != kKeyInf ? kv : ka;
      const int ebest = (int)key_payload(kbest);
      const float lam = __shfl_sync(kFull, my_lam[ebest >> 5], ebest & 31);
      const int sbest = __shfl_sync(kFull, my_s[ebest >> 5], ebest & 31);
      if (lane == 0) {
        a.out_list[i] = A * E + ebest;
        if (a.out_lambda) a.out_lambda[i] = lam;
      }
      if (!encode) continue;

      // ---- lambda quantiser: argmin_j (lam - cb[j])^2, lowest j on ties
      uint64_t kl = kKeyInf;
      for (int j = lane; j < a.nL; j += kWarp) {
        float t = lam - a.lambda_cb[j];
        uint64_t key = make_key(__fmul_rn(t, t), (uint32_t)j);
        kl = key < kl ? key : kl;
      }
      kl = warp_min_u64(kl);
      const int lq = (int)key_payload(kl);
      const float lh = a.lambda_cb[lq];

      // ---- residual -> per-warp shared memory for the sub-space walk
      const float* cs = a.cent + (int64_t)sbest * d;
      const float oml = 1.f - lh;
#pragma unroll
      for (int t = 0; t < NPL; t++) {
        int j = lane + 32 * t;
        float sv = j < d ? cs[j] : 0.f;
        const float anc = __fadd_rn(__fmul_rn(oml, cAv[t]), __fmul_rn(lh, sv));
        float rv = __fsub_rn(xv[t], anc);
        if (j < d) {
          r_s[j] = rv;
          if (a.out_residual) a.out_residual[i * d + j] = rv;
        }
      }
      if (lane == 0) {
        sc_w[v * 4 + 0] = A;
        sc_w[v * 4 + 1] = sbest;
        sc_w[v * 4 + 2] = lq;
        sc_w[v * 4 + 3] = __float_as_int(lh);
      }
    }
    if (!encode) continue;
    __syncwarp();

    // ------------------------------------------------------------------ phase B: PQ encode of the LE_V vectors.  Lane
    // owns codewords lane + 32c; distances accumulate over t in order (ProductQuantizer.cpp:311-336).
    for (int m = 0; m < M; m++) {
      uint64_t kc[LE_V];
      if (a.pq_in_smem && ksub == 256) {
        float dis[LE_V][8];
#pragma unroll
        for (int v = 0; v < LE_V; v++)
#pragma unroll
          for (int c = 0; c < 8; c++) dis[v][c] = 0.f;
        const float* pp = pqs + (size_t)m * dsub * ksub + lane;
        for (int t = 0; t < dsub; t++) {
          float pc[8];
#pragma unroll
          for (int c = 0; c < 8; c++) pc[c] = pp[t * ksub + 32 * c];
#pragma unroll
          for (int v = 0; v < LE_V; v++) {
            const float rt = r_w[v * d + m * dsub + t];
#pragma unroll
            for (int c = 0; c < 8; c++) {
              const float df = rt - pc[c];
              dis[v][c] = fmaf(df, df, dis[v][c]);
            }
          }
        }
        // lane-local arg-min on the floats (strict <: the lowest codeword index wins ties), one 64-bit key per lane
#pragma unroll
        for (int v = 0; v < LE_V; v++) {
          float bd = dis[v][0];
          int bc = 0;
#pragma unroll
          for (int c = 1; c < 8; c++) {
            if (dis[v][c] < bd) {
              bd = dis[v][c];
              bc = c;
            }
          }
          kc[v] = make_key(bd, (uint32_t)(lane + 32 * bc));
        }
      } else if (ksub == kPq4Ksub) {
        // 4-bit codebook (pq4_in_smem always holds, 16 d floats): lane = (h, j) scores codeword j = lane & 15 of
        // sub-quantizer m + h, h = lane >> 4, for all LE_V vectors -- two sub-quantizers per pass, no idle lane.  The
        // arg-min over the 16 lanes of a half takes the lowest (distance, j): the lowest codeword wins ties.
        const int h = lane >> 4, j = lane & 15, mh = m + h;
        float dis[LE_V];
#pragma unroll
        for (int v = 0; v < LE_V; v++) dis[v] = 0.f;
        const float* pp = pqs + (size_t)mh * dsub * kPq4Ksub + j;
        for (int t = 0; t < dsub; t++) {
          const float pc = pp[t * kPq4Ksub];
#pragma unroll
          for (int v = 0; v < LE_V; v++) {
            const float df = r_w[v * d + mh * dsub + t] - pc;
            dis[v] = fmaf(df, df, dis[v]);
          }
        }
#pragma unroll
        for (int v = 0; v < LE_V; v++) {
          uint64_t key = make_key(dis[v], (uint32_t)j);
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) {
            const uint64_t other = __shfl_xor_sync(kFull, key, o);
            key = other < key ? other : key;
          }
          if (j == 0) code_w[v * 64 + mh] = (uint8_t)key_payload(key);
        }
        m++;  // the pass covered m and m + 1 (M is even)
        continue;
      } else {
#pragma unroll
        for (int v = 0; v < LE_V; v++) {
          kc[v] = kKeyInf;
          for (int j = lane; j < ksub; j += kWarp) {
            const float* pp = a.pq + ((size_t)m * ksub + j) * dsub;
            float dis = 0.f;
            for (int t = 0; t < dsub; t++) {
              const float df = r_w[v * d + m * dsub + t] - pp[t];
              dis = fmaf(df, df, dis);
            }
            const uint64_t key = make_key(dis, (uint32_t)j);
            kc[v] = key < kc[v] ? key : kc[v];
          }
        }
      }
#pragma unroll
      for (int v = 0; v < LE_V; v++) {
        kc[v] = warp_min_u64(kc[v]);
        if (lane == 0) code_w[v * 64 + m] = (uint8_t)key_payload(kc[v]);
      }
    }
    __syncwarp();

    // ------------------------------------------------------------------ phase C: kappa = ||p||^2 + 2 anchor.p, outputs
#pragma unroll 1
    for (int v = 0; v < LE_V; v++) {
      const int A = sc_w[v * 4 + 0];
      if (A < 0) continue;  // beyond n, or an invalid vector
      const int64_t i = i0 + v;
      const int sbest = sc_w[v * 4 + 1], lq = sc_w[v * 4 + 2];
      const float lh = __int_as_float(sc_w[v * 4 + 3]);
      const float oml = 1.f - lh;
      const float* cA = a.cent + (int64_t)A * d;
      const float* cs = a.cent + (int64_t)sbest * d;
      const uint8_t* code_s = code_w + v * 64;
      float kp = 0.f;
#pragma unroll
      for (int t = 0; t < NPL; t++) {
        int j = lane + 32 * t;
        if (j < d) {
          const float anc = __fadd_rn(__fmul_rn(oml, cA[j]), __fmul_rn(lh, cs[j]));  // same bits as in phase A
          int m = j / dsub, tt = j % dsub;
          int code = code_s[m];
          float pv = a.pq_in_smem ? pqs[(size_t)(m * dsub + tt) * ksub + code] : a.pq[((size_t)m * ksub + code) * dsub + tt];
          kp = fmaf(pv, pv, kp);
          kp = fmaf(2.f * anc, pv, kp);
        }
      }
      kp = warp_sum(kp);
      if (lane == 0) {
        if (a.out_lamq) a.out_lamq[i] = (uint8_t)lq;
        if (a.out_kappa) a.out_kappa[i] = kp;
      }
      if (a.out_codes && ksub == kPq4Ksub) {  // packed, M / 2 bytes (pq4.cuh)
        for (int b = lane; b < M / 2; b += kWarp) a.out_codes[i * (M / 2) + b] = pq4_pack_byte(code_s[2 * b], code_s[2 * b + 1]);
      } else if (a.out_codes) {
        for (int m = lane; m < M; m += kWarp) a.out_codes[i * M + m] = code_s[m];
      }
    }
    __syncwarp();
  }
}

// ---- stand-alone a6 / a7 (the reference exposes them as separate GpuIndexFlat methods; the add path uses the fused kernel)
__global__ void lambda_quantize_kernel(const float* __restrict__ lam, int64_t n, const float* __restrict__ cb, int nL,
                                       uint8_t* __restrict__ out) {
  __shared__ float cbs[256];
  for (int j = threadIdx.x; j < nL; j += blockDim.x) cbs[j] = cb[j];
  __syncthreads();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float l = lam[i];
  float best = 0.f;
  int bj = 0;
  for (int j = 0; j < nL; j++) {  // argmin_j (l - cb[j])^2, lowest j on ties (GpuIndexFlat.cu:579-596)
    const float t = l - cbs[j];
    const float dd = __fmul_rn(t, t);
    if (j == 0 || dd < best) {
      best = dd;
      bj = j;
    }
  }
  out[i] = (uint8_t)bj;
}

__global__ void line_residual_kernel(const float* __restrict__ x, int64_t n, int d, const int* __restrict__ list,
                                     const uint8_t* __restrict__ lamq, const float* __restrict__ cb,
                                     const float* __restrict__ cent, const int* __restrict__ edge, int E,
                                     float* __restrict__ r) {
  int64_t i = (int64_t)blockIdx.x * (blockDim.x / kWarp) + threadIdx.x / kWarp;
  if (i >= n) return;
  const int lane = threadIdx.x % kWarp;
  const int l = list[i];
  if (l < 0) {
    for (int j = lane; j < d; j += kWarp) r[i * d + j] = 0.f;
    return;
  }
  const int A = l / E;
  const int s = edge[l];
  const float lh = cb[lamq[i]];
  const float oml = 1.f - lh;
  for (int j = lane; j < d; j += kWarp) {  // GpuIndexFlat.cu:1111-1122
    const float anchor = __fadd_rn(__fmul_rn(oml, cent[(int64_t)A * d + j]), __fmul_rn(lh, cent[(int64_t)s * d + j]));
    r[i * d + j] = __fsub_rn(x[i * d + j], anchor);
  }
}

__global__ void i32_to_i64_kernel(const int* __restrict__ src, int64_t n, int64_t* __restrict__ dst) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = src[i];
}

}  // namespace vlq

using namespace vlq;

extern "C" int vlq_lambda_quantize(const float* lambda, int64_t n, const float* lambda_cb, int nL, uint8_t* out,
                                   vlq_stream_t stream) {
  if (n < 0 || nL <= 0 || nL > 256) return VLQ_EINVAL;
  if (n == 0) return VLQ_OK;
  if (!lambda || !lambda_cb || !out) return VLQ_EINVAL;
  VLQ_LAUNCH(lambda_quantize_kernel, (unsigned)div_up(n, 256), 256, 0, as_stream(stream), lambda, n, lambda_cb, nL, out);
  return last_error();
}

extern "C" int vlq_line_residual(const float* x, int64_t n, int d, const int* list, const uint8_t* lamq,
                                 const float* lambda_cb, const float* cent, const int* edge, int E, float* residual,
                                 vlq_stream_t stream) {
  if (n < 0 || d <= 0 || E <= 0) return VLQ_EINVAL;
  if (n == 0) return VLQ_OK;
  if (!x || !list || !lamq || !lambda_cb || !cent || !edge || !residual) return VLQ_EINVAL;
  VLQ_LAUNCH(line_residual_kernel, (unsigned)div_up(n, 8), 256, 0, as_stream(stream), x, n, d, list, lamq, lambda_cb,
             cent, edge, E, residual);
  return last_error();
}

extern "C" int vlq_i32_to_i64(const int* src, int64_t n, int64_t* dst, vlq_stream_t stream) {
  if (n < 0) return VLQ_EINVAL;
  if (n == 0) return VLQ_OK;
  if (!src || !dst) return VLQ_EINVAL;
  VLQ_LAUNCH(i32_to_i64_kernel, 148 * 4, 256, 0, as_stream(stream), src, n, dst);
  return last_error();
}

// vlq_line_encode (ksub = 256) and vlq_line_encode_pq4 (ksub = 16: packed output, M even)
static int line_encode(int ksub, const float* x, int64_t n, int d, const int* assign, const float* cent,
                       const int* edge, const float* edge_d2, int E, const float* lambda_cb, int nL, const float* pq,
                       int M, int* out_list, float* out_lambda, uint8_t* out_lamq, uint8_t* out_codes,
                       float* out_kappa, float* out_residual, vlq_stream_t stream) {
  if (n < 0 || d <= 0 || d > 256 || E <= 0 || E > LE_MAX_E) return VLQ_EINVAL;
  if (n > 0 && (!x || !assign || !cent || !edge || !edge_d2 || !out_list)) return VLQ_EINVAL;
  if (ksub == kPq4Ksub && !pq4_shape_ok(d, M)) return VLQ_EINVAL;
  LineEncodeArgs a{};
  a.x = x; a.n = n; a.d = d; a.assign = assign; a.cent = cent; a.edge = edge; a.edge_d2 = edge_d2; a.E = E;
  a.lambda_cb = lambda_cb; a.nL = nL; a.pq = pq; a.M = M; a.ksub = ksub; a.dsub = M > 0 ? d / M : 0;
  a.out_list = out_list; a.out_lambda = out_lambda; a.out_lamq = out_lamq; a.out_codes = out_codes;
  a.out_kappa = out_kappa; a.out_residual = out_residual;
  if (lambda_cb) {
    if (!pq || M <= 0 || M > 64 || d % M != 0 || nL <= 0 || nL > 256) return VLQ_EINVAL;
  }
  if (n == 0) return VLQ_OK;
  size_t pq_bytes = lambda_cb ? (size_t)M * a.dsub * ksub * sizeof(float) : 0;
  size_t tail = (size_t)LE_WARPS * LE_V * (d * sizeof(float) + 4 * sizeof(int) + 64);
  a.pq_in_smem = (lambda_cb && pq_bytes + tail <= 200 * 1024) ? 1 : 0;
  size_t smem = (a.pq_in_smem ? pq_bytes : 0) + tail;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int64_t need = div_up(n, LE_WARPS * LE_V);
  unsigned grid = (unsigned)(need < sms ? need : sms);
  const int npl = (d + 31) / 32;
  cudaStream_t st = as_stream(stream);
#define VLQ_LE_CASE(N)                                                                                       \
  case N: {                                                                                                  \
    VLQ_CUDA_TRY(cudaFuncSetAttribute(line_encode_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize,    \
                                      (int)smem));                                                           \
    VLQ_LAUNCH(line_encode_kernel<N>, grid, LE_THREADS, smem, st, a);                                        \
    break;                                                                                                   \
  }
  switch (npl) {
    VLQ_LE_CASE(1)
    VLQ_LE_CASE(2)
    VLQ_LE_CASE(3)
    VLQ_LE_CASE(4)
    VLQ_LE_CASE(5)
    VLQ_LE_CASE(6)
    VLQ_LE_CASE(7)
    VLQ_LE_CASE(8)
    default:
      return VLQ_EINVAL;
  }
#undef VLQ_LE_CASE
  return last_error();
}

extern "C" int vlq_line_encode(const float* x, int64_t n, int d, const int* assign, const float* cent,
                               const int* edge, const float* edge_d2, int E, const float* lambda_cb, int nL,
                               const float* pq, int M, int* out_list, float* out_lambda, uint8_t* out_lamq,
                               uint8_t* out_codes, float* out_kappa, float* out_residual, vlq_stream_t stream) {
  return line_encode(256, x, n, d, assign, cent, edge, edge_d2, E, lambda_cb, nL, pq, M, out_list, out_lambda, out_lamq,
                     out_codes, out_kappa, out_residual, stream);
}

extern "C" int vlq_line_encode_pq4(const float* x, int64_t n, int d, const int* assign, const float* cent,
                                   const int* edge, const float* edge_d2, int E, const float* lambda_cb, int nL,
                                   const float* pq, int M, int* out_list, float* out_lambda, uint8_t* out_lamq,
                                   uint8_t* out_codes, float* out_kappa, float* out_residual, vlq_stream_t stream) {
  return line_encode(kPq4Ksub, x, n, d, assign, cent, edge, edge_d2, E, lambda_cb, nL, pq, M, out_list, out_lambda,
                     out_lamq, out_codes, out_kappa, out_residual, stream);
}
