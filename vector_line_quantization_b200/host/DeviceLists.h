// The inverted lists of GpuIndexIVFPQ and GpuIndexIMIPQ: one storage format, owned here.
//
// Committed slab (CSR over nlists lists, csrc/lists.cu): offsets [nlists + 1] (int64) | codes [n][M] | lamq [n] (the
// lambda byte; zero for IMI-PQ) | kappa [n] (fp32, the per-entry term of the scan) | ids [n] (int64).  Entries are
// list-major, in insertion order inside a list.  The M code bytes of the entry at list position pos are stored rotated
// by pos mod M (stored[j] = code[(j + pos) mod M], csrc/scan.cuh).
//
// Optional aux column: auxWidth bytes per entry (GpuIndexIVFPQR's refinement code), in canonical byte order (not
// rotated), beside the other columns in the slab and the arena; it moves with its entry through commit and remove.
// auxWidth = 0 (GpuIndexIVFPQ, GpuIndexIMIPQ): nothing is allocated and the launches are those without the column.
//
// Pending arena: encoded entries in arrival order (list id | codes | lamq | kappa | id | aux), written by the index's
// encoder.
// commit() merges them into the slab with vlq_build_lists (stable counting sort) at the first read after adds; entries
// the encoder skipped (list id < 0: NaN input) are dropped there.
//
// Every call works on the resource's default stream with the caller's device current (DeviceScope).
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "AuxIndexStructures.h"
#include "GpuResources.h"

namespace faiss {
namespace gpu {

class DeviceLists {
 public:
  DeviceLists(GpuResources* res, int64_t nlists, int M, int auxWidth = 0);

  /// device pointers to the next free arena slots (list id, M code bytes, lambda byte, kappa, id, auxWidth aux bytes per
  /// entry; aux is null when auxWidth = 0)
  struct Slots {
    int* list;
    uint8_t* codes;
    uint8_t* lamq;
    float* kappa;
    int64_t* ids;
    uint8_t* aux;
  };
  /// room for n more pending entries: the arena grows to max(need, 2 x capacity, the reserve() hint, 65 536) entries,
  /// keeping its contents
  Slots makeRoom(size_t n);
  /// counts the next n slots of makeRoom() as pending, once the encoder has written them
  void appended(size_t n);
  /// bulk-load hint: the next arena growth makes room for at least numVecs entries
  void reserve(size_t numVecs) { reserveVecs_ = numVecs; }

  /// merges the pending entries into the slab; a no-op when none are pending and a slab exists.  workspace: the
  /// caller's scratch, grown as needed.  Afterwards an arena of more than 2^21 entries is freed (a bulk load followed by
  /// searches would otherwise keep 16 + M bytes per vector next to the lists).
  void commit(DeviceBuffer& workspace);
  /// IndexIVF::remove_ids on the committed slab: the selector becomes a range or a sorted id array,
  /// vlq_remove_ids_plan counts the survivors, the new slab is allocated at its exact size and vlq_remove_ids_apply fills
  /// it (peak device memory: old + new slab).  Survivors keep their order.  Returns the number removed; throws
  /// FaissException for a selector other than IDSelectorRange / IDSelectorBatch (no per-entry virtual call on the device).
  long remove(const IDSelector& sel);
  /// the kappa column the scan of a call reads: the stored one for sel == nullptr, else a masked copy (+inf for every
  /// entry whose id sel does not hold, vlq_filter_kappa) in a grow-only buffer of 4 B per entry.  A host batch or bitmap
  /// is uploaded first; a device bitmap is read in place.  Throws (before any launch) for a selector
  /// checkSearchSelector rejects.
  const float* kappa(const IDSelector* sel);
  /// entries of list l in the committed slab
  int64_t listLength(int64_t l) const;
  /// replaces the lists by a finished slab from host memory: offsets [nlists + 1], stored-order codes, lambda bytes and
  /// ids of offsets[nlists] entries.  Returns the kappa column for the caller to compute (it depends on the index's
  /// tables).  The uploads are enqueued: the host arrays must outlive the caller's next sync of the default stream.
  /// Lists with an aux column cannot be installed (the formats behind install carry no aux bytes): throws.
  float* install(const std::vector<int64_t>& offsets, const std::vector<uint8_t>& codes,
                 const std::vector<uint8_t>& lamq, const std::vector<long>& ids);
  /// syncs the default stream, then frees the slab, the arena and the masked kappa
  void reset();

  int64_t nlists() const { return nlists_; }
  int M() const { return M_; }
  int auxWidth() const { return auxWidth_; }
  size_t size() const { return n_; }  ///< entries in the committed slab
  const int64_t* offsets() const { return offsets_.as<int64_t>(); }
  const uint8_t* codes() const { return slab_.codes.as<uint8_t>(); }
  const uint8_t* lamq() const { return slab_.lamq.as<uint8_t>(); }
  const int64_t* ids() const { return slab_.ids.as<int64_t>(); }
  const uint8_t* aux() const { return slab_.aux.as<uint8_t>(); }

 private:
  struct Columns {  // codes [n][M] | lamq [n] | kappa [n] | ids [n] | aux [n][R]
    DeviceBuffer codes, lamq, kappa, ids, aux;
    Columns() = default;
    Columns(size_t n, int M, int R)
        : codes(n * M), lamq(n), kappa(n * sizeof(float)), ids(n * sizeof(int64_t)), aux(n * R) {}
  };

  GpuResources* res_;
  int64_t nlists_;
  int M_;
  int auxWidth_;
  DeviceBuffer offsets_;  // committed slab: offsets_ + slab_
  Columns slab_;
  size_t n_ = 0;
  DeviceBuffer pList_;  // pending arena: pList_ + pending_
  Columns pending_;
  size_t nPending_ = 0, capPending_ = 0;
  size_t reserveVecs_ = 0;  // reserve() hint; cleared when a commit frees the arena
  DeviceBuffer masked_;     // the masked kappa of a filtered call
};

}  // namespace gpu
}  // namespace faiss
