"""Argument checks and workspace size of vlq_range_count / vlq_range_gather, and the range-search calls of the C wrapper
where no device is involved.  No GPU: both entries check every argument before their first CUDA call, and the pointers
below are never dereferenced."""
import ctypes as C

import numpy as np
import pytest

from vector_line_quantization_b200 import _abi

VLQ_EINVAL, VLQ_EWORKSPACE, VLQ_EUNSUPPORTED = -1, -2, -3
P = 1 << 20  # stands for a 256-byte aligned device pointer


@pytest.fixture(scope="module")
def lib():
    return _abi.lib()


def test_workspace_bytes(lib):
    ws = lib.vlq_range_workspace_bytes
    sizes = [ws(n, 16, 256, 1024) for n in (0, 1, 2, 255, 256, 5120, 10 ** 6)]
    assert sizes == sorted(sizes) and sizes[-1] > sizes[0]
    assert all(s % 256 == 0 for s in sizes)
    for M in (8, 16, 32, 64):
        assert ws(5120, M, 256, 1024) >= 5120 * M * 256 * 4  # one fp32 term-3 table per query
        assert [ws(n, M, 1, 1) for n in (1, 7, 100)] == sorted(ws(n, M, 1, 1) for n in (1, 7, 100))
    assert ws(-5, 16, 256, 1024) == 0


def _common(nq=100, d=128, q=P, pq=P, M=16, lcb=P, nL=16, lines=P, t1=P, t6=P, ed2=P, W=64, off=P, codes=P, lamq=P,
            kappa=P, cap=1024, row_add=P, radius=1.5):
    return [q, nq, d, pq, M, lcb, nL, lines, t1, t6, ed2, W, off, codes, lamq, kappa, cap, row_add, float(radius)]


def count(lib, out=P, ws=P, ws_bytes=None, **kw):
    a = _common(**kw)
    if ws_bytes is None:
        ws_bytes = lib.vlq_range_workspace_bytes(max(a[1], 0), a[4], a[11], a[16])
    return lib.vlq_range_count(*a, out, ws, ws_bytes, None)


def gather(lib, ids=P, lims=P, q0=0, q1=None, oD=P, oI=P, ws=P, ws_bytes=None, **kw):
    a = _common(**kw)
    if ws_bytes is None:
        ws_bytes = lib.vlq_range_workspace_bytes(max(a[1], 0), a[4], a[11], a[16])
    return lib.vlq_range_gather(*a, ids, lims, q0, a[1] if q1 is None else q1, oD, oI, ws, ws_bytes, None)


SHAPE_ERRORS = [dict(nq=-1), dict(d=0), dict(M=0), dict(M=65, d=130), dict(d=100, M=16), dict(nL=0), dict(nL=257),
                dict(W=0), dict(W=1025), dict(cap=0), dict(cap=(1 << 20) + 1), dict(radius=float("nan"))]
POINTERS = ["q", "pq", "lcb", "lines", "t1", "t6", "off", "codes", "lamq", "kappa"]


def test_count_argument_checks(lib):
    for kw in SHAPE_ERRORS:
        assert count(lib, **kw) == VLQ_EINVAL, kw
    for name in POINTERS:
        assert count(lib, **{name: None}) == VLQ_EINVAL, name
    assert count(lib, out=None) == VLQ_EINVAL
    assert count(lib, out=None, nq=0) == VLQ_EINVAL  # lims[0] is always written
    assert count(lib, ws=None) == VLQ_EINVAL
    assert count(lib, pq=P + 4) == VLQ_EINVAL and count(lib, ws=P + 8) == VLQ_EINVAL  # 16-byte alignment
    assert count(lib, ws_bytes=lib.vlq_range_workspace_bytes(100, 16, 64, 1024) - 1) == VLQ_EWORKSPACE
    assert count(lib, ws_bytes=0) == VLQ_EWORKSPACE
    # shapes the term-3 kernels do not take
    assert count(lib, d=102, M=2) == VLQ_EUNSUPPORTED  # d % 4
    assert count(lib, d=256, M=32) == VLQ_EUNSUPPORTED  # codebook beyond the kernel's shared memory
    assert count(lib, d=200, M=8) == VLQ_EUNSUPPORTED  # 1028 d = 205 600 B > 200 KiB: d <= 196 only
    # nq = 0 needs no inputs: only lims[0] = 0 is written (that reaches the device, so it is tested on the GPU)


def test_gather_argument_checks(lib):
    for kw in SHAPE_ERRORS:
        assert gather(lib, **kw) == VLQ_EINVAL, kw
    for name in POINTERS:
        assert gather(lib, **{name: None}) == VLQ_EINVAL, name
    for name in ("ids", "lims", "oD", "oI", "ws"):
        assert gather(lib, **{name: None}) == VLQ_EINVAL, name
    for q0, q1 in ((-1, 5), (5, 4), (0, 101)):
        assert gather(lib, q0=q0, q1=q1) == VLQ_EINVAL, (q0, q1)
    assert gather(lib, ws_bytes=lib.vlq_range_workspace_bytes(100, 16, 64, 1024) - 1) == VLQ_EWORKSPACE
    assert gather(lib, d=102, M=2) == VLQ_EUNSUPPORTED
    assert gather(lib, d=200, M=8) == VLQ_EUNSUPPORTED
    # an empty query range launches nothing, so its outputs may be NULL
    assert gather(lib, q0=7, q1=7, ids=None, lims=None, oD=None, oI=None) == 0
    assert gather(lib, nq=0, q=None, pq=None, lcb=None, lines=None, t1=None, t6=None, off=None, codes=None, lamq=None,
                  kappa=None, ids=None, lims=None, oD=None, oI=None, ws=None, q1=0) == 0


def test_c_wrapper_without_a_device():
    """the C wrapper's result handling: an index without range_search fails and leaves no result behind; NULL handles
    are refused by the accessors"""
    from vector_line_quantization_b200 import index as vi

    shards = vi.IndexShards(8)
    res = C.c_void_p(123)
    x = np.zeros((2, 8), np.float32)
    assert vi.host().vlq_host_index_range_search(shards.h, C.c_long(2), C.c_void_p(x.ctypes.data), C.c_float(1.0),
                                                 C.byref(res)) == -1
    assert b"range_search not implemented" in vi.host().vlq_host_last_error()
    assert res.value is None
    with pytest.raises(vi.FaissException, match="range_search not implemented"):
        shards.range_search(x, 1.0)
    with pytest.raises(vi.FaissException, match="range_search not implemented"):
        vi.IndexProxy().range_search(x, 1.0)
    total = C.c_long()
    assert vi.host().vlq_host_range_result_total(None, C.byref(total)) == -1
    assert vi.host().vlq_host_range_result_copy(None, None, None, None) == -1
    assert vi.host().vlq_host_range_result_free(None) == 0
