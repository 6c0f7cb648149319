"""Python mirror of the reference's index classes, backed by the C++ host layer (lib/libvlq_host.so, C wrapper
include/vlq_index_c.h).  Same names and argument meaning as the reference API (faiss::Index train/add/search/reset,
GpuIndexIVFPQ(res, d, nlist, M, bits, nedge, nLambda), setNumProbes, w1_, merge, write/read*ToFile, IndexProxy,
IndexShards).  Arrays may be numpy (host) or torch CUDA tensors (device); results come back in the same kind.
No CPU fallback: constructing anything here without the built CUDA + host libraries raises.
"""
import ctypes as C
import os

import numpy as np

from . import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(HERE, "lib", "libvlq_host.so")

_host = None


class FaissException(RuntimeError):
    pass


def host():
    global _host
    if _host is None:
        _abi.lib()  # the CUDA library first (RTLD_GLOBAL): the host layer links against it
        if not os.path.exists(HOST_LIB_PATH):
            raise RuntimeError("%s is missing: run `python -m vector_line_quantization_b200.build`" % HOST_LIB_PATH)
        h = C.CDLL(HOST_LIB_PATH)
        h.vlq_host_last_error.restype = C.c_char_p
        h.vlq_host_index_ntotal.restype = C.c_long
        _host = h
    return _host


def _call(name, *args):
    rc = getattr(host(), name)(*args)
    if rc != 0:
        raise FaissException(host().vlq_host_last_error().decode())


def _is_torch(a):
    return type(a).__module__.startswith("torch")


def _in(a, dtype):
    """-> (pointer, keepalive, is_device)"""
    if a is None:
        return None, None, False
    if _is_torch(a):
        import torch

        want = {np.float32: torch.float32, np.int64: torch.int64, np.int32: torch.int32}[dtype]
        if a.dtype != want or not a.is_contiguous():
            a = a.to(want).contiguous()
        return C.c_void_p(a.data_ptr()), a, a.is_cuda
    a = np.ascontiguousarray(a, dtype=dtype)
    return C.c_void_p(a.ctypes.data), a, False


class StandardGpuResources:
    def __init__(self, device=0):
        self.h = C.c_void_p()
        _call("vlq_host_resources_new", int(device), C.byref(self.h))
        self.device = device

    def sync(self):
        _call("vlq_host_resources_sync", self.h)

    def __del__(self):
        try:
            if self.h:
                host().vlq_host_resources_free(self.h)
        except Exception:
            pass


class Index:
    """faiss::Index virtual API over an opaque handle"""

    def __init__(self, d):
        self.d = d
        self.h = C.c_void_p()
        self._keep = []

    @property
    def ntotal(self):
        return host().vlq_host_index_ntotal(self.h)

    @property
    def is_trained(self):
        return bool(host().vlq_host_index_is_trained(self.h))

    def train(self, x):
        p, k, _ = _in(x, np.float32)
        _call("vlq_host_index_train", self.h, C.c_long(x.shape[0]), p)

    def add(self, x):
        p, k, _ = _in(x, np.float32)
        _call("vlq_host_index_add", self.h, C.c_long(x.shape[0]), p)

    def add_with_ids(self, x, ids):
        p, k, _ = _in(x, np.float32)
        pi, ki, _ = _in(ids, np.int64)
        _call("vlq_host_index_add_with_ids", self.h, C.c_long(x.shape[0]), p, pi)

    def search(self, x, k, out=None, sel=None):
        """-> (distances [n][k] f32, labels [n][k] i64), numpy for host input, torch CUDA for device input.
        out=(D, I) reuses caller buffers (e.g. pinned torch tensors).  sel: restrict the results to these ids (see
        _Selector; GpuIndexIVFPQ and GpuIndexIMIPQ), missing results padded with (FLT_MAX, -1)."""
        if sel is not None:
            _sync_if_cuda(x)
        p, keep, dev = _in(x, np.float32)
        n = x.shape[0]
        if out is not None:
            D, I = out
        elif dev:
            import torch

            D = torch.empty((n, k), dtype=torch.float32, device=x.device)
            I = torch.empty((n, k), dtype=torch.int64, device=x.device)
        else:
            D = np.empty((n, k), np.float32)
            I = np.empty((n, k), np.int64)
        pd = C.c_void_p(D.data_ptr() if _is_torch(D) else D.ctypes.data)
        pi = C.c_void_p(I.data_ptr() if _is_torch(I) else I.ctypes.data)
        if sel is None:
            _call("vlq_host_index_search", self.h, C.c_long(n), p, C.c_long(k), pd, pi)
        else:
            with _Selector(sel) as hs:
                _call("vlq_host_index_search_sel", self.h, C.c_long(n), p, C.c_long(k), pd, pi, hs)
        return D, I

    def range_search(self, x, radius, sel=None):
        """faiss Index.range_search: every stored vector with squared L2 distance < radius -> (lims int64 [n + 1],
        D f32 [total], I int64 [total]) numpy arrays; the results of query i are D / I[lims[i]:lims[i + 1]].
        x is numpy or torch (host or device).  GpuIndexIVFPQ and GpuIndexIMIPQ implement it.  sel: only these ids
        (see _Selector)."""
        if sel is not None:
            _sync_if_cuda(x)
        p, keep, _ = _in(x, np.float32)
        n = x.shape[0]
        res = C.c_void_p()
        if sel is None:
            _call("vlq_host_index_range_search", self.h, C.c_long(n), p, C.c_float(radius), C.byref(res))
        else:
            with _Selector(sel) as hs:
                _call("vlq_host_index_range_search_sel", self.h, C.c_long(n), p, C.c_float(radius), C.byref(res), hs)
        try:
            total = C.c_long()
            _call("vlq_host_range_result_total", res, C.byref(total))
            lims = np.empty(n + 1, np.int64)
            D = np.empty(total.value, np.float32)
            I = np.empty(total.value, np.int64)
            _call("vlq_host_range_result_copy", res, C.c_void_p(lims.ctypes.data), C.c_void_p(D.ctypes.data),
                  C.c_void_p(I.ctypes.data))
        finally:
            host().vlq_host_range_result_free(res)
        return lims, D, I

    def reset(self):
        _call("vlq_host_index_reset", self.h)

    def remove_ids(self, sel):
        """faiss Index.remove_ids: sel is an IDSelectorRange or an int64 id array (numpy or torch, host or device; any
        order, duplicates allowed).  Returns the number of entries removed.  GpuIndexIVFPQ and GpuIndexIMIPQ implement
        it; the survivors keep their order inside their lists."""
        out = C.c_long()
        if isinstance(sel, IDSelectorRange):
            _call("vlq_host_index_remove_ids_range", self.h, C.c_long(sel.imin), C.c_long(sel.imax), C.byref(out))
            return out.value
        if _is_torch(sel):
            import torch

            sel = sel.reshape(-1)
            if sel.is_cuda:
                torch.cuda.current_stream(sel.device).synchronize()  # the host layer copies it on its own stream
        else:
            sel = np.asarray(sel).reshape(-1)
        p, keep, _ = _in(sel, np.int64)
        _call("vlq_host_index_remove_ids_batch", self.h, C.c_long(sel.shape[0]), p, C.byref(out))
        return out.value

    def __del__(self):
        try:
            if self.h:
                host().vlq_host_index_free(self.h)
        except Exception:
            pass


class IDSelectorRange:
    """the ids imin <= id < imax (faiss IDSelectorRange), for Index.remove_ids and filtered search"""

    def __init__(self, imin, imax):
        self.imin, self.imax = int(imin), int(imax)


class IDSelectorBitmap:
    """the ids whose bit (id & 7) of bitmap[id >> 3] is set (faiss IDSelectorBitmap); ids outside [0, 8 len(bitmap))
    are not members.  bitmap: uint8 bytes, numpy (host) or a torch CUDA tensor (read on the device in place)."""

    def __init__(self, bitmap):
        if _is_torch(bitmap):
            import torch

            assert bitmap.dtype == torch.uint8
            self.bitmap = bitmap.reshape(-1).contiguous()
        else:
            self.bitmap = np.ascontiguousarray(np.asarray(bitmap, np.uint8).reshape(-1))


class IDSelectorNot:
    """the ids `sel` does not hold (faiss IDSelectorNot); sel: any selector that filtered search accepts"""

    def __init__(self, sel):
        self.sel = sel


class _Selector:
    """context manager: a host-layer IDSelector handle for `sel` (IDSelectorRange, IDSelectorBitmap, IDSelectorNot, or
    an int64 id array -- numpy or torch, any order, duplicates allowed: IDSelectorBatch), freed on exit"""

    def __init__(self, sel):
        self.sel = sel
        self.handles = []
        self.keep = []

    def _new(self, fn, *args):
        h = C.c_void_p()
        self.handles.append(h)  # freed on exit even when a later step fails
        _call(fn, *args, C.byref(h))
        return h

    def _make(self, sel):
        if isinstance(sel, IDSelectorRange):
            return self._new("vlq_host_selector_range_new", C.c_long(sel.imin), C.c_long(sel.imax))
        if isinstance(sel, IDSelectorBitmap):
            _sync_if_cuda(sel.bitmap)
            self.keep.append(sel.bitmap)
            return self._new("vlq_host_selector_bitmap_new", C.c_long(sel.bitmap.shape[0]), _ptr_of(sel.bitmap))
        if isinstance(sel, IDSelectorNot):
            return self._new("vlq_host_selector_not_new", self._make(sel.sel))
        if _is_torch(sel) or isinstance(sel, (np.ndarray, list, tuple)):
            ids = sel.reshape(-1) if _is_torch(sel) else np.asarray(sel).reshape(-1)
            if not _is_torch(ids) and ids.size and not np.issubdtype(ids.dtype, np.integer):
                raise TypeError("an id selector array must hold integers, not %s" % ids.dtype)
            _sync_if_cuda(ids)
            p, keep, _ = _in(ids, np.int64)
            self.keep.append(keep)
            return self._new("vlq_host_selector_batch_new", C.c_long(ids.shape[0]), p)
        raise TypeError("unsupported selector %r: use IDSelectorRange, IDSelectorBitmap, IDSelectorNot or an int64 id "
                        "array" % type(sel).__name__)

    def __enter__(self):
        try:
            return self._make(self.sel)
        except BaseException:
            self.__exit__(None, None, None)
            raise

    def __exit__(self, *exc):
        for h in reversed(self.handles):
            if h:
                host().vlq_host_selector_free(h)
        self.handles = []
        return False


def selector_is_member(sel, ids):
    """host-side membership (IDSelector::is_member) of every id in `ids` -> bool numpy array"""
    out = C.c_int()
    res = []
    with _Selector(sel) as hs:
        for i in np.asarray(ids, np.int64).reshape(-1):
            _call("vlq_host_selector_is_member", hs, C.c_long(int(i)), C.byref(out))
            res.append(bool(out.value))
    return np.array(res, bool)


def _sync_if_cuda(a):
    if _is_torch(a) and a.is_cuda:
        import torch

        torch.cuda.current_stream(a.device).synchronize()  # the host layer reads it on its own stream


def _ptr_of(a):
    return C.c_void_p(a.data_ptr() if _is_torch(a) else a.ctypes.data)


class _ReadBack:
    """Decode of stored entries (GpuIndexIVFPQ, GpuIndexIMIPQ): keys are ids; a key without an entry raises
    FaissException and writes nothing; an id stored more than once gives its entry with the lowest slab index.
    numpy for host input, torch CUDA for device input (as Index.search)."""

    def reconstruct_n(self, i0, ni, out=None):
        """stored vectors of the ids i0 .. i0 + ni - 1 -> [ni][d] f32 (numpy, or `out`: a caller array, e.g. CUDA)"""
        if out is None:
            out = np.empty((ni, self.d), np.float32)
        _call("vlq_host_index_reconstruct_n", self.h, C.c_long(i0), C.c_long(ni), _ptr_of(out))
        return out

    def reconstruct(self, key):
        return self.reconstruct_batch(np.array([key], np.int64))[0]

    def reconstruct_batch(self, keys):
        """stored vectors of the ids `keys` (any order, duplicates allowed) -> [n][d] f32"""
        if _is_torch(keys):
            import torch

            keys = keys.reshape(-1)
            _sync_if_cuda(keys)
            out = torch.empty((keys.shape[0], self.d), dtype=torch.float32, device=keys.device)
        else:
            keys = np.asarray(keys).reshape(-1)
            out = np.empty((keys.shape[0], self.d), np.float32)
        p, keep, _ = _in(keys, np.int64)
        _call("vlq_host_index_reconstruct_batch", self.h, C.c_long(keys.shape[0]), p, _ptr_of(out))
        return out

    def search_and_reconstruct(self, x, k, sel=None):
        """-> (D [n][k], I [n][k], R [n][k][d]): search() and the stored vector behind every label (NaN rows for -1).
        sel: as in search()."""
        _sync_if_cuda(x)
        p, keep, dev = _in(x, np.float32)
        n = x.shape[0]
        if dev:
            import torch

            D = torch.empty((n, k), dtype=torch.float32, device=x.device)
            I = torch.empty((n, k), dtype=torch.int64, device=x.device)
            R = torch.empty((n, k, self.d), dtype=torch.float32, device=x.device)
        else:
            D = np.empty((n, k), np.float32)
            I = np.empty((n, k), np.int64)
            R = np.empty((n, k, self.d), np.float32)
        if sel is None:
            _call("vlq_host_index_search_and_reconstruct", self.h, C.c_long(n), p, C.c_long(k), _ptr_of(D), _ptr_of(I),
                  _ptr_of(R))
        else:
            with _Selector(sel) as hs:
                _call("vlq_host_index_search_and_reconstruct_sel", self.h, C.c_long(n), p, C.c_long(k), _ptr_of(D),
                      _ptr_of(I), _ptr_of(R), hs)
        return D, I, R


def _reconstruct_n(self, i0, ni):
    out = np.empty((ni, self.d), np.float32)
    _call("vlq_host_index_reconstruct_n", self.h, C.c_long(i0), C.c_long(ni), C.c_void_p(out.ctypes.data))
    return out


class GpuIndexFlatL2(Index):
    reconstruct_n = _reconstruct_n

    def reconstruct(self, key):
        return _reconstruct_n(self, key, 1)[0]

    def __init__(self, res, d, use_tensor_cores=True):
        super().__init__(d)
        self.res = res
        _call("vlq_host_flat_new", res.h, d, int(use_tensor_cores), C.byref(self.h))

    def assign(self, x):
        p, keep, _ = _in(x, np.float32)
        out = np.empty(x.shape[0], np.int32)
        _call("vlq_host_flat_assign", self.h, C.c_long(x.shape[0]), p, C.c_void_p(out.ctypes.data))
        return out

    def searchInt(self, x, k):
        """search with int32 labels (reference GpuIndexFlat::searchInt)"""
        p, keep, _ = _in(x, np.float32)
        n = x.shape[0]
        D = np.empty((n, k), np.float32)
        I = np.empty((n, k), np.int32)
        _call("vlq_host_flat_search_int", self.h, C.c_long(n), p, C.c_long(k), C.c_void_p(D.ctypes.data),
              C.c_void_p(I.ctypes.data))
        return D, I

    def assign1Base(self, x, assign, edge, edge_d2):
        """device-pointer line stage (reference assign1Base): torch CUDA tensors in, (assign2 int32, lambda f32) out"""
        import torch

        n = x.shape[0]
        a2 = torch.empty(n, dtype=torch.int32, device=x.device)
        lam = torch.empty(n, dtype=torch.float32, device=x.device)
        _call("vlq_host_flat_assign1_base", self.h, C.c_long(n), C.c_void_p(x.data_ptr()), C.c_void_p(assign.data_ptr()),
              C.c_void_p(a2.data_ptr()), C.c_void_p(lam.data_ptr()), C.c_void_p(edge.data_ptr()),
              C.c_void_p(edge_d2.data_ptr()), edge.shape[1])
        self.res.sync()
        return a2, lam

    def buildGraph(self, nedge):
        n = self.ntotal
        D = np.empty((n, nedge), np.float32)
        I = np.empty((n, nedge), np.int32)
        _call("vlq_host_flat_build_graph", self.h, nedge, C.c_void_p(D.ctypes.data), C.c_void_p(I.ctypes.data))
        return D, I


def kmeans(res, x, k, niter=10, seed=1234):
    """Clustering::train over a GpuIndexFlatL2 assigner -> centroids [k][d] (numpy)"""
    p, keep, _ = _in(x, np.float32)
    d = x.shape[1]
    out = np.empty((k, d), np.float32)
    _call("vlq_host_kmeans", res.h, d, k, C.c_long(x.shape[0]), p, niter, seed, C.c_void_p(out.ctypes.data))
    return out


class GpuIndexIVFPQ(_ReadBack, Index):
    """The VLQ index: GpuIndexIVFPQ(res, d, nlist, M, bitsPerCode, nedge, nLambda) (gpu/GpuIndexIVFPQ.h:59-67).
    bits = 8, or 4 with an even M: two codes per stored byte on the device; getList, copyFrom / copyTo and the .db*
    files still see one byte per code."""

    def __init__(self, res, d, nlist, M, bits=8, nedge=32, nLambda=256, use_tensor_cores=True):
        super().__init__(d)
        self.res, self.nlist, self.M, self.nedge, self.nLambda, self.bits = res, nlist, M, nedge, nLambda, bits
        _call("vlq_host_vlq_new", res.h, d, nlist, M, bits, nedge, nLambda, int(use_tensor_cores), C.byref(self.h))
        self._w1 = 256

    def setNumProbes(self, nprobe):
        _call("vlq_host_vlq_set_nprobe", self.h, int(nprobe))

    @property
    def w1_(self):
        return self._w1

    @w1_.setter
    def w1_(self, w):
        _call("vlq_host_vlq_set_w1", self.h, int(w))
        self._w1 = int(w)

    def setListCap(self, cap):
        _call("vlq_host_vlq_set_list_cap", self.h, int(cap))

    def add_with_ids_u8(self, x, ids=None):
        """x: uint8 [n][d] (numpy or torch, host or device)"""
        if _is_torch(x):
            import torch

            assert x.dtype == torch.uint8 and x.is_contiguous()
            px = C.c_void_p(x.data_ptr())
        else:
            x = np.ascontiguousarray(x, np.uint8)
            px = C.c_void_p(x.ctypes.data)
        pi, ki, _ = _in(ids, np.int64)
        _call("vlq_host_vlq_add_with_ids_u8", self.h, C.c_long(x.shape[0]), px, pi)

    def reserveMemory(self, num_vecs):
        _call("vlq_host_vlq_reserve_memory", self.h, C.c_long(int(num_vecs)))

    def setTrainIters(self, niter):
        _call("vlq_host_vlq_set_train_iters", self.h, int(niter))

    def codebooks(self):
        L = self.nlist * self.nedge
        out = dict(cent=np.empty((self.nlist, self.d), np.float32), edge=np.empty((self.nlist, self.nedge), np.int32),
                   edge_d2=np.empty((self.nlist, self.nedge), np.float32), lambda_cb=np.empty(self.nLambda, np.float32),
                   pq=np.empty((self.M, 1 << self.bits, self.d // self.M), np.float32))
        _call("vlq_host_vlq_get_codebooks", self.h, *(C.c_void_p(out[k].ctypes.data) for k in
                                                      ("cent", "edge", "edge_d2", "lambda_cb", "pq")))
        assert out["edge"].size == L
        return out

    def setCodebooks(self, cent, edge, edge_d2, lambda_cb, pq):
        arrs = [np.ascontiguousarray(cent, np.float32), np.ascontiguousarray(edge, np.int32),
                np.ascontiguousarray(edge_d2, np.float32), np.ascontiguousarray(lambda_cb, np.float32),
                np.ascontiguousarray(pq, np.float32)]
        _call("vlq_host_vlq_set_codebooks", self.h, *(C.c_void_p(a.ctypes.data) for a in arrs))

    def getListLength(self, l):
        out = C.c_int()
        _call("vlq_host_vlq_list_length", self.h, int(l), C.byref(out))
        return out.value

    def getList(self, l):
        n = self.getListLength(l)
        codes = np.empty((n, self.M), np.uint8)
        las = np.empty(n, np.uint8)
        ids = np.empty(n, np.int64)
        _call("vlq_host_vlq_get_list", self.h, int(l), C.c_void_p(codes.ctypes.data), C.c_void_p(las.ctypes.data),
              C.c_void_p(ids.ctypes.data))
        return codes, las, ids

    def merge(self, nns, dist):
        """nns, dist: [nprocess][nq][k] -> (distances, labels) [nq][k]"""
        nns = np.ascontiguousarray(nns, np.int64)
        dist = np.ascontiguousarray(dist, np.float32)
        R, nq, k = dist.shape
        D = np.empty((nq, k), np.float32)
        I = np.empty((nq, k), np.int64)
        _call("vlq_host_vlq_merge", self.h, C.c_void_p(nns.ctypes.data), C.c_void_p(dist.ctypes.data), k, nq, R,
              C.c_void_p(D.ctypes.data), C.c_void_p(I.ctypes.data))
        return D, I

    def writeCodebookToFile(self, name):
        _call("vlq_host_vlq_write_codebook", self.h, name.encode())

    def readCodebookFromFile(self, name):
        _call("vlq_host_vlq_read_codebook", self.h, name.encode())

    def writeDbToFile(self, name):
        _call("vlq_host_vlq_write_db", self.h, name.encode())

    def readDbFromFile(self, name, pronum=1, rank=0):
        _call("vlq_host_vlq_read_db", self.h, name.encode(), int(pronum), int(rank))


    # ---- f4 (gpu/GpuIndexIVFPQ.cu:169-281, 1312-1398, 1646-1670)
    def copyFrom(self, cpu_index):
        _call("vlq_host_ivfpq_copy_from", self.h, cpu_index.h)

    def copyTo(self, cpu_index):
        _call("vlq_host_ivfpq_copy_to", self.h, cpu_index.h)

    def search1(self, x, k):
        """candidate lists: ids of the entries of the w1_ selected lines of every query, first k, -1 padded"""
        px, _keep, _ = _in(x, np.float32)
        n = x.shape[0]
        labels = np.empty((n, k), np.int64)
        _call("vlq_host_ivfpq_search1", self.h, C.c_long(n), px, C.c_long(k), C.c_void_p(labels.ctypes.data))
        return labels

    def add_with_ids2(self, x, xq, kgt, ids=None):
        """exact kgt nearest rows of the chunk x for every query of xq: -> (dists, nns)"""
        x = np.ascontiguousarray(x, np.float32)
        xq = np.ascontiguousarray(xq, np.float32)
        ids = np.ascontiguousarray(ids, np.int64) if ids is not None else None
        nns = np.empty((xq.shape[0], kgt), np.int64)
        dists = np.empty((xq.shape[0], kgt), np.float32)
        _call("vlq_host_ivfpq_add_with_ids2", self.h, C.c_long(x.shape[0]), C.c_long(xq.shape[0]), C.c_uint(kgt),
              C.c_void_p(x.ctypes.data), C.c_void_p(xq.ctypes.data), C.c_void_p(ids.ctypes.data) if ids is not None else None,
              C.c_void_p(nns.ctypes.data), C.c_void_p(dists.ctypes.data))
        return dists, nns


class GpuIndexIVFPQR(GpuIndexIVFPQ):
    """GpuIndexIVFPQ plus a refinement stage (faiss IndexIVFPQR, host/GpuIndexIVFPQR.h): every entry also stores an
    8-bit PQ code of M_refine sub-quantizers of the residual its first-level code leaves, and search re-ranks the
    scan's min(1024, max(k, floor(k * k_factor))) candidates by the two-level reconstruction.  search distances are
    FULL squared L2 ||q - x2||^2 (as IndexIVFPQR), not GpuIndexIVFPQ's ||q||^2-less values; reconstruct* return x2.
    range_search, copyFrom / copyTo and the .db* files raise FaissException."""

    def __init__(self, res, d, nlist, M, M_refine, bits=8, nedge=32, nLambda=256, use_tensor_cores=True):
        M_refine = int(M_refine)
        if not 1 <= M_refine <= 64 or d % M_refine != 0:
            raise ValueError("M_refine must be in [1, 64] and divide d = %d, got %d" % (d, M_refine))
        Index.__init__(self, d)
        self.res, self.nlist, self.M, self.nedge, self.nLambda, self.M_refine = res, nlist, M, nedge, nLambda, M_refine
        self.bits = bits
        _call("vlq_host_ivfpqr_new", res.h, d, nlist, M, M_refine, bits, nedge, nLambda, int(use_tensor_cores),
              C.byref(self.h))
        self._w1 = 256

    @property
    def k_factor(self):
        out = C.c_float()
        _call("vlq_host_ivfpqr_get_k_factor", self.h, C.byref(out))
        return out.value

    @k_factor.setter
    def k_factor(self, v):
        _call("vlq_host_ivfpqr_set_k_factor", self.h, C.c_float(v))

    def setRefineCodebook(self, pq2):
        """pq2: (M_refine, 256, d / M_refine) float32"""
        pq2 = np.ascontiguousarray(pq2, np.float32)
        if pq2.size != 256 * self.d:
            raise ValueError("refinement codebook must hold (M_refine, 256, d / M_refine) floats")
        _call("vlq_host_ivfpqr_set_refine_codebook", self.h, C.c_void_p(pq2.ctypes.data))

    def refineCodebook(self):
        out = np.empty((self.M_refine, 256, self.d // self.M_refine), np.float32)
        _call("vlq_host_ivfpqr_get_refine_codebook", self.h, C.c_void_p(out.ctypes.data))
        return out

    def getListRefineCodes(self, l):
        """code2 of the entries of list l in list order -> uint8 [len][M_refine]"""
        out = np.empty((self.getListLength(l), self.M_refine), np.uint8)
        _call("vlq_host_ivfpqr_get_list_refine_codes", self.h, int(l), C.c_void_p(out.ctypes.data))
        return out


class CpuIndexIVFPQ:
    """faiss::IndexIVFPQ as a CONTAINER (host/IndexIVFPQ.h): coarse centroids, PQ codebook, per-list ids + codes -- what
    GpuIndexIVFPQ.copyFrom / copyTo exchange with a CPU index"""

    def __init__(self, d, nlist, M, nbits=8):
        self.d, self.nlist, self.M, self.nbits = d, nlist, M, nbits
        self.h = C.c_void_p()
        _call("vlq_host_cpu_ivfpq_new", d, C.c_long(nlist), M, nbits, C.byref(self.h))

    def set_codebooks(self, coarse, pq):
        coarse = np.ascontiguousarray(coarse, np.float32)
        pq = np.ascontiguousarray(pq, np.float32)
        assert coarse.shape == (self.nlist, self.d) and pq.size == self.d << self.nbits
        _call("vlq_host_cpu_ivfpq_set_codebooks", self.h, C.c_void_p(coarse.ctypes.data), C.c_void_p(pq.ctypes.data))

    def codebooks(self):
        coarse = np.empty((self.nlist, self.d), np.float32)
        pq = np.empty((self.M, 1 << self.nbits, self.d // self.M), np.float32)
        _call("vlq_host_cpu_ivfpq_get_codebooks", self.h, C.c_void_p(coarse.ctypes.data), C.c_void_p(pq.ctypes.data))
        return coarse, pq

    def set_list(self, l, ids, codes):
        ids = np.ascontiguousarray(ids, np.int64)
        codes = np.ascontiguousarray(codes, np.uint8)
        _call("vlq_host_cpu_ivfpq_set_list", self.h, C.c_long(l), C.c_long(len(ids)), C.c_void_p(ids.ctypes.data),
              C.c_void_p(codes.ctypes.data))

    def get_list(self, l):
        host().vlq_host_cpu_ivfpq_list_size.restype = C.c_long
        n = host().vlq_host_cpu_ivfpq_list_size(self.h, C.c_long(l))
        ids = np.empty(n, np.int64)
        codes = np.empty((n, self.M), np.uint8)
        if n:
            _call("vlq_host_cpu_ivfpq_get_list", self.h, C.c_long(l), C.c_void_p(ids.ctypes.data), C.c_void_p(codes.ctypes.data))
        return ids, codes

    @property
    def ntotal(self):
        host().vlq_host_cpu_ivfpq_ntotal.restype = C.c_long
        return host().vlq_host_cpu_ivfpq_ntotal(self.h)

    def __del__(self):
        try:
            if self.h:
                host().vlq_host_cpu_ivfpq_free(self.h)
        except Exception:
            pass


class GpuIndexIMIPQ(_ReadBack, Index):
    """IMI-PQ on the device (host/GpuIndexIMIPQ.h): MultiIndexQuantizer(d, 2, nbits_coarse) + IVFPQ over the K^2 cells"""

    def __init__(self, res, d, nbits_coarse, M, nbits=8):
        super().__init__(d)
        self.res, self.nbits_coarse, self.M, self.nbits = res, nbits_coarse, M, nbits
        _call("vlq_host_imipq_new", res.h, d, nbits_coarse, M, nbits, C.byref(self.h))

    def setNumProbes(self, nprobe):
        _call("vlq_host_imipq_set_nprobe", self.h, int(nprobe))

    def setTrainIters(self, niter):
        _call("vlq_host_imipq_set_train_iters", self.h, int(niter))

    def setCodebooks(self, coarse, pq):
        coarse = np.ascontiguousarray(coarse, np.float32)
        pq = np.ascontiguousarray(pq, np.float32)
        assert coarse.shape == (2, 1 << self.nbits_coarse, self.d // 2) and pq.size == self.d << self.nbits
        _call("vlq_host_imipq_set_codebooks", self.h, C.c_void_p(coarse.ctypes.data), C.c_void_p(pq.ctypes.data))

    def codebooks(self):
        coarse = np.empty((2, 1 << self.nbits_coarse, self.d // 2), np.float32)
        pq = np.empty((self.M, 1 << self.nbits, self.d // self.M), np.float32)
        _call("vlq_host_imipq_get_codebooks", self.h, C.c_void_p(coarse.ctypes.data), C.c_void_p(pq.ctypes.data))
        return coarse, pq

    def searchCells(self, x, nprobe):
        x = np.ascontiguousarray(x, np.float32)
        D = np.empty((x.shape[0], nprobe), np.float32)
        I = np.empty((x.shape[0], nprobe), np.int64)
        _call("vlq_host_imipq_search_cells", self.h, C.c_long(x.shape[0]), C.c_void_p(x.ctypes.data), int(nprobe),
              C.c_void_p(D.ctypes.data), C.c_void_p(I.ctypes.data))
        return D, I

    def getListLength(self, cell):
        out = C.c_int()
        _call("vlq_host_imipq_list_length", self.h, C.c_long(int(cell)), C.byref(out))
        return out.value


class IndexProxy(Index):
    """replicas: queries are split over the sub-indexes (gpu/IndexProxy.cpp:124-168)"""

    def __init__(self):
        super().__init__(0)
        _call("vlq_host_proxy_new", C.byref(self.h))

    def addIndex(self, index):
        self._keep.append(index)
        self.d = index.d
        _call("vlq_host_proxy_add_index", self.h, index.h)


class IndexShards(Index):
    """database shards: every shard searches all queries, results merged (MetaIndexes.cpp:486-563)"""

    def __init__(self, d, threaded=True, successive_ids=True):
        super().__init__(d)
        _call("vlq_host_shards_new", d, int(threaded), int(successive_ids), C.byref(self.h))

    def add_shard(self, index):
        self._keep.append(index)
        _call("vlq_host_shards_add_shard", self.h, index.h)
