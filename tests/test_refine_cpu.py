"""Argument checks of the refinement entries (vlq_refine_encode / vlq_refine_topk / vlq_refine_decode and the aux-column
variants of the list build and removal) and of the GpuIndexIVFPQR constructor.  No GPU: the C-ABI entries check every
argument before their first CUDA call, and the pointers below are never dereferenced."""
import numpy as np
import pytest

from vector_line_quantization_b200 import _abi

VLQ_EINVAL = -1
VLQ_EUNSUPPORTED = -3
P = 1 << 20  # stands for a device pointer


@pytest.fixture(scope="module")
def lib():
    return _abi.lib()


def enc(lib, x=P, n=100, d=128, lst=P, lamq=P, codes=P, M=16, pq=P, cent=P, edge=P, E=32, lcb=P, nL=256, pq2=P,
        M2=16, code2=P, r2=None):
    return lib.vlq_refine_encode(x, n, d, lst, lamq, codes, M, pq, cent, edge, E, lcb, nL, pq2, M2, code2, r2, None)


def topk(lib, q=P, nq=10, d=128, cand=P, kc=40, k=10, nlists=64, off=P, codes=P, lamq=P, ids=P, code2=P, M=16, pq=P,
         cent=P, edge=P, E=32, lcb=P, nL=256, pq2=P, M2=16, outD=P, outI=P):
    return lib.vlq_refine_topk(q, nq, d, cand, kc, k, nlists, off, codes, lamq, ids, code2, M, pq, cent, edge, E, lcb,
                               nL, pq2, M2, outD, outI, None)


def dec(lib, n=10, pos=P, nlists=64, off=P, codes=P, lamq=P, ids=P, code2=P, M=16, d=128, pq=P, cent=P, edge=P,
        E=32, lcb=P, nL=256, pq2=P, M2=16, out=P, oid=None):
    return lib.vlq_refine_decode(n, pos, nlists, off, codes, lamq, ids, code2, M, d, pq, cent, edge, E, lcb, nL, pq2,
                                 M2, out, oid, None)


def test_refine_encode_argument_checks(lib):
    n0 = lib.vlq_launch_count()
    for kw in (dict(n=-1), dict(d=0), dict(M=0), dict(M=65), dict(M=24), dict(E=0), dict(nL=0), dict(nL=257),
               dict(M2=0), dict(M2=65), dict(M2=24), dict(code2=None), dict(pq2=None, r2=None)):
        assert enc(lib, **kw) == VLQ_EINVAL, kw
    for name in ("x", "lst", "lamq", "codes", "pq", "cent", "edge", "lcb"):
        assert enc(lib, **{name: None}) == VLQ_EINVAL, name
    assert enc(lib, d=1024, M=16, M2=16) == VLQ_EUNSUPPORTED  # one row per warp lives in shared memory
    assert lib.vlq_launch_count() == n0
    # n = 0 is a no-op that needs no data pointers; training mode (pq2 NULL) needs only r2
    assert enc(lib, n=0, x=None, lst=None, lamq=None, codes=None) == 0
    assert enc(lib, n=0, pq2=None, M2=0, code2=None, r2=P) == 0
    assert lib.vlq_launch_count() == n0


def test_refine_topk_argument_checks(lib):
    n0 = lib.vlq_launch_count()
    for kw in (dict(nq=-1), dict(nq=1 << 31), dict(kc=0), dict(kc=1025), dict(k=0), dict(k=41), dict(nlists=0),
               dict(nlists=65), dict(M2=0), dict(M2=65), dict(M2=24), dict(M=24), dict(E=0), dict(nL=257)):
        assert topk(lib, **kw) == VLQ_EINVAL, kw
    for name in ("q", "cand", "off", "pq", "cent", "edge", "lcb", "pq2", "outD", "outI"):
        assert topk(lib, **{name: None}) == VLQ_EINVAL, name
    assert topk(lib, d=1024) == VLQ_EUNSUPPORTED
    assert lib.vlq_launch_count() == n0
    assert topk(lib, nq=0, q=None, cand=None, outD=None, outI=None) == 0
    assert topk(lib, nq=0, kc=1024, k=1024) == 0
    assert lib.vlq_launch_count() == n0


def test_refine_decode_argument_checks(lib):
    n0 = lib.vlq_launch_count()
    for kw in (dict(n=-1), dict(M2=0), dict(M2=65), dict(M2=24), dict(M=65), dict(nlists=65), dict(E=0),
               dict(nL=0), dict(d=0)):
        assert dec(lib, **kw) == VLQ_EINVAL, kw
    for name in ("pos", "off", "codes", "lamq", "code2", "pq", "cent", "edge", "lcb", "pq2", "out"):
        assert dec(lib, **{name: None}) == VLQ_EINVAL, name
    assert dec(lib, ids=None, oid=P) == VLQ_EINVAL  # labels need the ids
    assert dec(lib, n=0) == 0
    assert lib.vlq_launch_count() == n0


def test_aux_list_entries_argument_checks(lib):
    n0 = lib.vlq_launch_count()

    def build(aux_w=16, n_old=5, old_aux=P, n_new=5, new_aux=P, out_aux=P):
        return lib.vlq_build_lists_aux(64, 16, aux_w, n_old, P, P, P, P, P, old_aux, n_new, P, P, P, P, P, new_aux, P, P,
                                       P, P, P, out_aux, P, 1 << 30, None)

    for kw in (dict(aux_w=-1), dict(aux_w=65), dict(old_aux=None), dict(new_aux=None), dict(out_aux=None)):
        assert build(**kw) == VLQ_EINVAL, kw

    def apply(aux_w=16, n=5, aux=P, out_aux=P):
        return lib.vlq_remove_ids_apply_aux(64, 16, aux_w, n, P, P, P, P, P, aux, P, P, P, P, P, out_aux, P, 1 << 30,
                                            None)

    for kw in (dict(aux_w=-1), dict(aux_w=65), dict(aux=None), dict(out_aux=None)):
        assert apply(**kw) == VLQ_EINVAL, kw
    assert apply(n=0, aux=None, out_aux=None) == 0
    assert lib.vlq_launch_count() == n0


@pytest.mark.parametrize("M_refine", [0, -4, 65, 24, 7])
def test_python_constructor_validates_M_refine(M_refine):
    from vector_line_quantization_b200 import index as vi

    with pytest.raises(ValueError):
        vi.GpuIndexIVFPQR(None, 128, 64, 16, M_refine)
