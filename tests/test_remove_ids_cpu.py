"""Argument checks and workspace size of vlq_remove_ids_plan / vlq_remove_ids_apply.  No GPU: both check every argument
before their first CUDA call, and the pointers below are never dereferenced."""
import pytest

from vector_line_quantization_b200 import _abi

VLQ_EINVAL, VLQ_EWORKSPACE = -1, -2
P = 1 << 20  # stands for a device pointer


@pytest.fixture(scope="module")
def lib():
    return _abi.lib()


def test_workspace_bytes(lib):
    ws = lib.vlq_remove_ids_workspace_bytes
    sizes = [ws(n, 1 << 21) for n in (0, 1, 8192, 8193, 1 << 20, 10 ** 9)]
    assert sizes == sorted(sizes) and sizes[-1] > sizes[-2] > sizes[0]
    for n in (1 << 20, 10 ** 9):
        assert ws(n, 1 << 21) < n + 4096  # a keep bit and 1/1024 byte per entry: below one byte per entry
        assert ws(n, 1 << 21) >= n // 8
    assert ws(1 << 20, 1) == ws(1 << 20, 1 << 21)  # nothing per list
    assert all(s % 256 == 0 for s in sizes)


def plan(lib, nlists=16, n=1000, offsets=P, ids=P, lo=0, hi=10, batch=P, n_batch=4, out=P, ws=P, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.vlq_remove_ids_workspace_bytes(max(n, 0), nlists)
    return lib.vlq_remove_ids_plan(nlists, n, offsets, ids, lo, hi, batch, n_batch, out, ws, ws_bytes, None)


def apply(lib, nlists=16, M=16, n=1000, offsets=P, codes=P, lamq=P, kappa=P, ids=P, out_off=P, oc=P, ol=P, ok=P,
          oi=P, ws=P, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.vlq_remove_ids_workspace_bytes(max(n, 0), nlists)
    return lib.vlq_remove_ids_apply(nlists, M, n, offsets, codes, lamq, kappa, ids, out_off, oc, ol, ok, oi, ws,
                                    ws_bytes, None)


def test_plan_argument_checks(lib):
    assert plan(lib, n=-1) == VLQ_EINVAL
    assert plan(lib, nlists=0) == VLQ_EINVAL
    assert plan(lib, n_batch=-1) == VLQ_EINVAL
    assert plan(lib, batch=None) == VLQ_EINVAL  # n_batch > 0 needs the array
    for name in ("offsets", "ids", "out", "ws"):
        assert plan(lib, **{name: None}) == VLQ_EINVAL, name
    assert plan(lib, ws_bytes=lib.vlq_remove_ids_workspace_bytes(1000, 16) - 1) == VLQ_EWORKSPACE
    assert plan(lib, ws_bytes=0) == VLQ_EWORKSPACE


def test_apply_argument_checks(lib):
    for M in (0, -1, 65, 128):
        assert apply(lib, M=M) == VLQ_EINVAL, M
    assert apply(lib, n=-1) == VLQ_EINVAL
    assert apply(lib, nlists=0) == VLQ_EINVAL
    for name in ("offsets", "codes", "lamq", "kappa", "ids", "out_off", "oc", "ol", "ok", "oi", "ws"):
        assert apply(lib, **{name: None}) == VLQ_EINVAL, name
    assert apply(lib, ws_bytes=lib.vlq_remove_ids_workspace_bytes(1000, 16) - 1) == VLQ_EWORKSPACE
    assert apply(lib, n=0, codes=None, lamq=None, kappa=None, ids=None, oc=None, ol=None, ok=None, oi=None) == 0
