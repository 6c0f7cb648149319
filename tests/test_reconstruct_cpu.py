"""Argument checks of vlq_lookup_ids / vlq_decode_entries / vlq_imi_decode_entries and the read-back entries of the C
wrapper.  No GPU: the C-ABI entries check every argument before their first CUDA call, and the pointers below are never
dereferenced."""
import ctypes as C

import numpy as np
import pytest

from vector_line_quantization_b200 import _abi

VLQ_EINVAL = -1
P = 1 << 20  # stands for a device pointer


@pytest.fixture(scope="module")
def lib():
    return _abi.lib()


def lookup(lib, n=1000, ids=P, lo=0, keys=P, nslots=10, pos=P, found=P):
    return lib.vlq_lookup_ids(n, ids, lo, keys, nslots, pos, found, None)


def decode(lib, n=10, pos=P, nlists=64, off=P, codes=P, lamq=P, ids=P, M=16, d=128, pq=P, cent=P, edge=P, E=8, lcb=P,
           nL=256, out=P, oid=P):
    return lib.vlq_decode_entries(n, pos, nlists, off, codes, lamq, ids, M, d, pq, cent, edge, E, lcb, nL, out, oid, None)


def imi_decode(lib, n=10, pos=P, off=P, codes=P, ids=P, M=16, d=128, pq=P, cb1=P, cb2=P, nbits=4, out=P, oid=P):
    return lib.vlq_imi_decode_entries(n, pos, off, codes, ids, M, d, pq, cb1, cb2, nbits, out, oid, None)


def test_lookup_argument_checks(lib):
    assert lookup(lib, n=-1) == VLQ_EINVAL
    assert lookup(lib, nslots=-1) == VLQ_EINVAL
    assert lookup(lib, found=None) == VLQ_EINVAL
    assert lookup(lib, found=None, nslots=0) == VLQ_EINVAL  # the count is always written
    assert lookup(lib, ids=None) == VLQ_EINVAL
    assert lookup(lib, pos=None) == VLQ_EINVAL
    # range mode: lo + nslots must be representable
    assert lookup(lib, keys=None, lo=(1 << 63) - 5, nslots=10) == VLQ_EINVAL


def test_decode_argument_checks(lib):
    for kw in (dict(n=-1), dict(nlists=0), dict(M=0), dict(M=65), dict(d=0), dict(d=100, M=16), dict(E=0),
               dict(nlists=63, E=8), dict(nL=0), dict(nL=257)):
        assert decode(lib, **kw) == VLQ_EINVAL, kw
    for name in ("pos", "off", "codes", "lamq", "pq", "cent", "edge", "lcb", "out"):
        assert decode(lib, **{name: None}) == VLQ_EINVAL, name
    assert decode(lib, ids=None) == VLQ_EINVAL  # out_ids needs the ids
    # n = 0 launches nothing: no inputs needed
    assert decode(lib, n=0, pos=None, off=None, codes=None, lamq=None, ids=None, pq=None, cent=None, edge=None,
                  lcb=None, out=None, oid=None) == 0


def test_imi_decode_argument_checks(lib):
    for kw in (dict(n=-1), dict(M=0), dict(M=65), dict(d=100, M=16), dict(d=15, M=5), dict(nbits=0),
               dict(nbits=16)):
        assert imi_decode(lib, **kw) == VLQ_EINVAL, kw
    for name in ("pos", "off", "codes", "pq", "cb1", "cb2", "out"):
        assert imi_decode(lib, **{name: None}) == VLQ_EINVAL, name
    assert imi_decode(lib, ids=None) == VLQ_EINVAL
    assert imi_decode(lib, n=0, pos=None, off=None, codes=None, ids=None, pq=None, cb1=None, cb2=None, out=None,
                      oid=None) == 0


def test_c_wrapper_read_back_without_a_device():
    """the new C wrapper entries exist, and an index that cannot decode fails through them with the index's message"""
    from vector_line_quantization_b200 import index as vi

    h = vi.host()
    for name in ("vlq_host_index_reconstruct_batch", "vlq_host_index_search_and_reconstruct",
                 "vlq_host_index_reconstruct_n"):
        assert hasattr(h, name), name
    shards = vi.IndexShards(8)
    keys = np.array([3], np.int64)
    out = np.full((1, 8), 7.0, np.float32)
    assert h.vlq_host_index_reconstruct_batch(shards.h, C.c_long(1), C.c_void_p(keys.ctypes.data),
                                              C.c_void_p(out.ctypes.data)) == -1
    assert b"reconstruct not implemented" in h.vlq_host_last_error()
    assert (out == 7.0).all()
