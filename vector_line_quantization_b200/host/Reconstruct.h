// Read-back of stored entries of the lists of DeviceLists.h: reconstruct, reconstruct_n, reconstruct_batch and the
// decode step of search_and_reconstruct.  Ids are found by one pass over the slab's ids on the device (vlq_lookup_ids,
// no persistent id -> entry map); each index supplies the decode of its own anchors (vlq_decode_entries /
// vlq_imi_decode_entries).  Outputs in host memory are decoded in pages through a bounded device staging buffer.
#pragma once
#include <cstddef>
#include <cstdint>
#include <functional>

#include "DeviceLists.h"

namespace faiss {
namespace gpu {

/// decodes the entries at the device slab indexes pos[0 .. n) into the device rows out[n][d], enqueued on `stream`;
/// outIds (nullable, may alias pos) receives their ids.  Slab index -1 gives a NaN row and id -1.
using EntryDecoder =
    std::function<void(const int64_t* pos, int64_t n, float* out, int64_t* outIds, vlq_stream_t stream)>;

/// reconstruct_batch (keys != nullptr: n ids in any order, duplicates allowed, host or device memory) or reconstruct_n
/// (keys == nullptr: the ids i0 .. i0 + n - 1) into recons[n][d] (host or device).  An id stored more than once decodes
/// its entry with the lowest slab index.  Throws FaissException naming the first id without an entry, before anything
/// is written.  `lists` must be committed.
void reconstructIds(GpuResources* res, int d, const DeviceLists& lists, Index::idx_t n, const Index::idx_t* keys,
                    Index::idx_t i0, float* recons, const EntryDecoder& decode, DeviceBuffer& staging);

/// decode of the n device slab indexes pos into recons[n][d] (host or device) on `stream`; with outIds (device, may
/// alias pos) the ids too.  Host outputs go through `staging` in pages of at most VLQ_RECONSTRUCT_STAGING_BYTES
/// (environment, read on every call; default 256 MiB, one row at least).
void decodeToOutput(int d, const int64_t* pos, int64_t n, float* recons, int64_t* outIds, const EntryDecoder& decode,
                    DeviceBuffer& staging, vlq_stream_t stream);

}  // namespace gpu
}  // namespace faiss
