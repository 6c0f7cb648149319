"""Argument checks of vlq_filter_kappa / vlq_filter_results, host-side membership of the filtered-search selectors, and
the filtered entries of the C wrapper.  No GPU: the C-ABI entries check every argument before their first CUDA call,
and the pointers below are never dereferenced."""
import ctypes as C

import numpy as np
import pytest

from vector_line_quantization_b200 import _abi

VLQ_EINVAL = -1
P = 1 << 20  # stands for a device pointer


@pytest.fixture(scope="module")
def lib():
    return _abi.lib()


def fk(lib, n=1000, ids=P, kappa=P, lo=0, hi=10, batch=P, nb=5, bitmap=P, nbytes=8, invert=0, out=P):
    return lib.vlq_filter_kappa(n, ids, kappa, lo, hi, batch, nb, bitmap, nbytes, invert, out, None)


def test_filter_kappa_argument_checks(lib):
    n0 = lib.vlq_launch_count()
    for kw in (dict(n=-1), dict(nb=-1), dict(nbytes=-1)):
        assert fk(lib, **kw) == VLQ_EINVAL, kw
    for name in ("ids", "kappa", "out"):
        assert fk(lib, **{name: None}) == VLQ_EINVAL, name
    assert fk(lib, batch=None) == VLQ_EINVAL                # n_batch > 0 needs the batch
    assert fk(lib, bitmap=None) == VLQ_EINVAL               # bitmap_bytes > 0 needs the bitmap
    assert lib.vlq_launch_count() == n0                     # nothing was launched
    # no batch / no bitmap is fine as far as the checks go; n = 0 is a no-op that needs no pointers at all
    assert fk(lib, n=0, ids=None, kappa=None, batch=None, nb=0, bitmap=None, nbytes=0, out=None) == 0
    assert fk(lib, n=0, ids=None, kappa=None, out=None) == 0
    assert lib.vlq_launch_count() == n0


def test_filter_results_argument_checks(lib):
    n0 = lib.vlq_launch_count()
    assert lib.vlq_filter_results(-1, 10, P, P, None) == VLQ_EINVAL
    assert lib.vlq_filter_results(4, 0, P, P, None) == VLQ_EINVAL
    assert lib.vlq_filter_results(4, 10, None, P, None) == VLQ_EINVAL
    assert lib.vlq_filter_results(4, 10, P, None, None) == VLQ_EINVAL
    assert lib.vlq_filter_results(0, 10, None, None, None) == 0
    assert lib.vlq_launch_count() == n0


def test_bitmap_membership_on_the_host():
    from vector_line_quantization_b200 import index as vi

    bm = np.array([0b00000101, 0b10000000, 0], np.uint8)  # ids 0, 2 and 15 (bit id & 7 of byte id >> 3)
    sel = vi.IDSelectorBitmap(bm)
    ids = np.array([0, 1, 2, 3, 7, 8, 15, 16, 23, 24, 1000, -1, -8, -(1 << 62)])
    got = vi.selector_is_member(sel, ids)
    assert got.tolist() == [i in (0, 2, 15) for i in ids.tolist()]
    assert not vi.selector_is_member(vi.IDSelectorBitmap(np.zeros(0, np.uint8)), [0, 1, 7]).any()


def test_not_and_batch_membership_on_the_host():
    from vector_line_quantization_b200 import index as vi

    ids = np.arange(-5, 40)
    rng = vi.IDSelectorRange(3, 17)
    assert (vi.selector_is_member(rng, ids) == ((ids >= 3) & (ids < 17))).all()
    assert (vi.selector_is_member(vi.IDSelectorNot(rng), ids) == ~((ids >= 3) & (ids < 17))).all()
    assert (vi.selector_is_member(vi.IDSelectorNot(vi.IDSelectorNot(rng)), ids) == ((ids >= 3) & (ids < 17))).all()
    batch = np.array([30, 4, 4, -2, 11], np.int64)  # any order, duplicates allowed
    assert (vi.selector_is_member(batch, ids) == np.isin(ids, batch)).all()
    assert (vi.selector_is_member(vi.IDSelectorNot(batch), ids) == ~np.isin(ids, batch)).all()
    bm = np.packbits(np.isin(np.arange(48), [1, 9, 33]), bitorder="little")
    assert (vi.selector_is_member(vi.IDSelectorNot(vi.IDSelectorBitmap(bm)), ids) == ~np.isin(ids, [1, 9, 33])).all()


def test_c_wrapper_errors_without_a_device():
    from vector_line_quantization_b200 import index as vi

    h = vi.host()
    for name in ("vlq_host_index_search_sel", "vlq_host_index_range_search_sel",
                 "vlq_host_index_search_and_reconstruct_sel", "vlq_host_selector_free"):
        assert hasattr(h, name), name
    # IDSelectorNot of nothing
    out = C.c_void_p()
    assert h.vlq_host_selector_not_new(None, C.byref(out)) == -1
    assert b"null selector" in h.vlq_host_last_error()
    assert h.vlq_host_selector_bitmap_new(C.c_long(4), None, C.byref(out)) == -1
    assert h.vlq_host_selector_batch_new(C.c_long(-1), None, C.byref(out)) == -1
    # a non-null selector on an index that cannot filter fails before anything is written
    shards = vi.IndexShards(8)
    x = np.zeros((2, 8), np.float32)
    D = np.full((2, 3), 7.0, np.float32)
    I = np.full((2, 3), 7, np.int64)
    with vi._Selector(vi.IDSelectorRange(0, 10)) as hs:
        assert h.vlq_host_index_search_sel(shards.h, C.c_long(2), C.c_void_p(x.ctypes.data), C.c_long(3),
                                           C.c_void_p(D.ctypes.data), C.c_void_p(I.ctypes.data), hs) == -1
        assert b"search parameters not supported" in h.vlq_host_last_error()
        res = C.c_void_p(P)
        assert h.vlq_host_index_range_search_sel(shards.h, C.c_long(2), C.c_void_p(x.ctypes.data), C.c_float(1.0),
                                                 C.byref(res), hs) == -1
        assert b"search parameters not supported" in h.vlq_host_last_error()
        assert not res.value
    assert (D == 7.0).all() and (I == 7).all()
    with pytest.raises(vi.FaissException, match="search parameters not supported"):
        shards.search(x, 3, sel=np.array([1, 2]))
    # a selector type the wrapper does not know is refused before any call
    with pytest.raises(TypeError, match="unsupported selector"):
        shards.search(x, 3, sel={1, 2})
    with pytest.raises(TypeError, match="integers"):
        shards.search(x, 3, sel=np.array([1.5]))
