#include "Reconstruct.h"

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <string>
#include <vector>

namespace faiss {
namespace gpu {

static int64_t stagingRows(int d) {
  const char* e = getenv("VLQ_RECONSTRUCT_STAGING_BYTES");  // read per call: tests force tiny pages
  const long long bytes = e ? atoll(e) : (256ll << 20);
  return std::max<int64_t>(1, bytes / ((int64_t)d * (int64_t)sizeof(float)));
}

void decodeToOutput(int d, const int64_t* pos, int64_t n, float* recons, int64_t* outIds, const EntryDecoder& decode,
                    DeviceBuffer& staging, vlq_stream_t st) {
  if (n == 0) return;
  if (vlq_pointer_is_device(recons) == 1) {
    decode(pos, n, recons, outIds, st);
    return;
  }
  const int64_t rows = std::min(n, stagingRows(d));
  staging.reserve((size_t)rows * d * sizeof(float));
  for (int64_t r0 = 0; r0 < n; r0 += rows) {
    const int64_t m = std::min(rows, n - r0);
    decode(pos + r0, m, staging.as<float>(), outIds ? outIds + r0 : nullptr, st);
    // stream order: the next page's decode overwrites the staging buffer only after this copy
    VLQ_CALL(vlq_memcpy_d2h(recons + (size_t)r0 * d, staging.get(), (size_t)m * d * sizeof(float), st));
  }
}

void reconstructIds(GpuResources* res, int d, const SlabIds& slab, Index::idx_t n, const Index::idx_t* keys,
                    Index::idx_t i0, float* recons, const EntryDecoder& decode, DeviceBuffer& staging) {
  VLQ_THROW_IF_NOT_MSG(n >= 0, "reconstruct: n must be >= 0");
  if (n == 0) return;
  VLQ_THROW_IF_NOT_MSG(recons != nullptr && (keys != nullptr || i0 >= 0), "reconstruct: null output or negative id");
  VLQ_THROW_IF_NOT_MSG(keys != nullptr || i0 <= LONG_MAX - n, "reconstruct_n: i0 + ni overflows");
  vlq_stream_t st = res->getDefaultStream();
  // batch mode: the sorted, de-duplicated keys are the slots of the lookup
  std::vector<int64_t> hk, uk;
  DeviceBuffer dKeys;
  int64_t nslots = n;
  if (keys) {
    hk.resize((size_t)n);
    if (vlq_pointer_is_device(keys) == 1) {
      VLQ_CALL(vlq_memcpy_d2h(hk.data(), keys, (size_t)n * sizeof(int64_t), st));
      res->syncDefaultStream();
    } else {
      std::copy(keys, keys + n, hk.begin());
    }
    uk = hk;
    std::sort(uk.begin(), uk.end());
    uk.erase(std::unique(uk.begin(), uk.end()), uk.end());
    nslots = (int64_t)uk.size();
    dKeys.resize((size_t)nslots * sizeof(int64_t));
    VLQ_CALL(vlq_memcpy_h2d(dKeys.get(), uk.data(), dKeys.bytes(), st));
  }
  DeviceBuffer dPos((size_t)nslots * sizeof(int64_t)), dFound(sizeof(int64_t));
  VLQ_CALL(vlq_lookup_ids((int64_t)slab.nListed, slab.ids, keys ? 0 : i0, dKeys.as<int64_t>(), nslots,
                          dPos.as<int64_t>(), dFound.as<int64_t>(), st));
  int64_t found = 0;
  VLQ_CALL(vlq_memcpy_d2h(&found, dFound.get(), sizeof(int64_t), st));
  res->syncDefaultStream();
  std::vector<int64_t> hp;
  if (found < nslots || keys) {
    hp.resize((size_t)nslots);
    VLQ_CALL(vlq_memcpy_d2h(hp.data(), dPos.get(), dPos.bytes(), st));
    res->syncDefaultStream();
  }
  if (found < nslots) {
    const int64_t s = std::find(hp.begin(), hp.end(), (int64_t)-1) - hp.begin();
    VLQ_THROW_MSG("reconstruct: key " + std::to_string(keys ? uk[s] : i0 + s) + " has no entry");
  }
  const int64_t* pos = dPos.as<int64_t>();
  DeviceBuffer dSel;
  if (keys) {  // slab index of every requested key, in the caller's order
    std::vector<int64_t> sel((size_t)n);
    for (int64_t i = 0; i < n; i++) sel[i] = hp[std::lower_bound(uk.begin(), uk.end(), hk[i]) - uk.begin()];
    dSel.resize((size_t)n * sizeof(int64_t));
    VLQ_CALL(vlq_memcpy_h2d(dSel.get(), sel.data(), dSel.bytes(), st));
    decodeToOutput(d, dSel.as<int64_t>(), n, recons, nullptr, decode, staging, st);
    res->syncDefaultStream();  // sel outlives its upload
    return;
  }
  decodeToOutput(d, pos, n, recons, nullptr, decode, staging, st);
  res->syncDefaultStream();
}

}  // namespace gpu
}  // namespace faiss
