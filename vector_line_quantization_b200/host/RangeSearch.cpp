#include "RangeSearch.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace faiss {
namespace gpu {

static int64_t stagingResults() {
  const char* e = getenv("VLQ_RANGE_STAGING_BYTES");  // read per call: tests force tiny sub-ranges
  const long long bytes = e ? atoll(e) : (1ll << 30);
  return std::max<int64_t>(1, bytes / (int64_t)(sizeof(float) + sizeof(int64_t)));
}

void rangeSearchLists(GpuResources* res, int d, Index::idx_t n, const float* x, float radius, const RangeLists& L,
                      const RangeCoarseStage& coarse, RangeSearchResult* result) {
  VLQ_THROW_IF_NOT_MSG(!std::isnan(radius), "range_search: radius is NaN");
  VLQ_THROW_IF_NOT_MSG(result != nullptr && result->lims != nullptr, "range_search: result must hold nq + 1 lims");
  VLQ_THROW_IF_NOT_MSG(n >= 0 && (size_t)n == result->nq, "range_search: result->nq must equal n");
  VLQ_THROW_IF_NOT_MSG(n == 0 || x != nullptr, "range_search: x is null");
  std::fill(result->lims, result->lims + n + 1, (size_t)0);
  std::vector<float> hD;
  std::vector<int64_t> hI;
  if (n > 0 && L.nListed > 0) {
    vlq_stream_t st = res->getDefaultStream();
    const int W = L.W;
    const Index::idx_t tile = std::min(L.tile, n);
    const bool xOnDevice = vlq_pointer_is_device(x) == 1;
    const int64_t budget = stagingResults();
    DeviceBuffer xin, lines((size_t)tile * W * sizeof(int)), t1((size_t)tile * W * sizeof(float)),
        t6((size_t)tile * W * sizeof(float)), qn((size_t)tile * sizeof(float)), lims((size_t)(tile + 1) * sizeof(int64_t)),
        ws(vlq_range_workspace_bytes(tile, L.M, W, L.cap)), stage;
    if (!xOnDevice) xin.resize((size_t)tile * d * sizeof(float));
    std::vector<int64_t> hl((size_t)tile + 1);
    for (Index::idx_t s = 0; s < n; s += tile) {
      const Index::idx_t m = std::min(tile, n - s);
      const float* q = x + (size_t)s * d;
      if (!xOnDevice) {
        VLQ_CALL(vlq_memcpy_h2d(xin.get(), q, (size_t)m * d * sizeof(float), st));
        q = xin.as<float>();
      }
      coarse(q, m, lines.as<int>(), t1.as<float>(), t6.as<float>());
      if (L.addQueryNorm) VLQ_CALL(vlq_row_norms(q, m, d, qn.as<float>(), st));
      const float* rowAdd = L.addQueryNorm ? qn.as<float>() : nullptr;
      VLQ_CALL(vlq_range_count(q, m, d, L.pq, L.M, L.lambdaCb, L.nLambda, lines.as<int>(), t1.as<float>(), t6.as<float>(),
                               L.edgeDist, W, L.offsets, L.codes, L.lamq, L.kappa, L.cap, rowAdd, radius,
                               lims.as<int64_t>(), ws.get(), ws.bytes(), st));
      // the one host synchronisation of a tile: its result sizes decide the sub-ranges and the host arrays
      VLQ_CALL(vlq_memcpy_d2h(hl.data(), lims.get(), (size_t)(m + 1) * sizeof(int64_t), st));
      res->syncDefaultStream();
      for (Index::idx_t i = 0; i < m; i++) result->lims[s + i] = (size_t)(hl[i + 1] - hl[i]);
      // query sub-ranges [q0, q1) of at most `budget` results (a larger single query is one sub-range of its own)
      std::vector<std::pair<Index::idx_t, Index::idx_t>> parts;
      int64_t most = 0;
      for (Index::idx_t q0 = 0; q0 < m;) {
        Index::idx_t q1 = q0 + 1;
        while (q1 < m && hl[q1 + 1] - hl[q0] <= budget) q1++;
        parts.emplace_back(q0, q1);
        most = std::max<int64_t>(most, hl[q1] - hl[q0]);
        q0 = q1;
      }
      if (most == 0) continue;
      const size_t dBytes = ((size_t)most * sizeof(float) + 255) & ~size_t(255);
      stage.reserve(dBytes + (size_t)most * sizeof(int64_t));
      float* sD = stage.as<float>();
      int64_t* sI = reinterpret_cast<int64_t*>(stage.as<unsigned char>() + dBytes);
      const size_t at = hD.size();
      hD.resize(at + (size_t)hl[m]);
      hI.resize(at + (size_t)hl[m]);
      for (const auto& p : parts) {
        const int64_t cnt = hl[p.second] - hl[p.first];
        if (cnt == 0) continue;
        VLQ_CALL(vlq_range_gather(q, m, d, L.pq, L.M, L.lambdaCb, L.nLambda, lines.as<int>(), t1.as<float>(),
                                  t6.as<float>(), L.edgeDist, W, L.offsets, L.codes, L.lamq, L.kappa, L.cap, rowAdd, radius,
                                  L.ids, lims.as<int64_t>(), p.first, p.second, sD, sI, ws.get(), ws.bytes(), st));
        // stream order: the next gather overwrites the staging buffer only after these copies
        VLQ_CALL(vlq_memcpy_d2h(hD.data() + at + hl[p.first], sD, (size_t)cnt * sizeof(float), st));
        VLQ_CALL(vlq_memcpy_d2h(hI.data() + at + hl[p.first], sI, (size_t)cnt * sizeof(int64_t), st));
      }
      res->syncDefaultStream();
    }
  }
  result->do_allocation();
  const size_t total = result->lims[n];
  if (total) {
    std::memcpy(result->distances, hD.data(), total * sizeof(float));
    std::memcpy(result->labels, hI.data(), total * sizeof(int64_t));
  }
}

}  // namespace gpu
}  // namespace faiss
