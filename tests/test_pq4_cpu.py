"""4-bit PQ codes without a GPU: the packed byte order, the code-format rule of the index constructors and the argument
checks of the *_pq4 C-ABI entries (every one is checked before the first CUDA call; the pointers below are never
dereferenced)."""
import numpy as np
import pytest
import torch

from vector_line_quantization_b200 import _abi, ops

VLQ_EINVAL = -1
VLQ_EWORKSPACE = -2
P = 1 << 20  # stands for a device pointer (16-byte aligned)


@pytest.fixture(scope="module")
def lib():
    return _abi.lib()


def test_pack_round_trip_and_faiss_byte_order():
    rng = np.random.default_rng(0)
    codes = torch.from_numpy(rng.integers(0, 16, (257, 32), dtype=np.uint8))
    packed = ops.pack_pq4(codes)
    assert packed.shape == (257, 16)
    assert torch.equal(ops.unpack_pq4(packed), codes)
    c = codes.numpy().astype(np.int64)
    # byte j = code[2j] | code[2j + 1] << 4: faiss's packed order (ProductQuantizer.cpp, PQEncoderGeneric at nbits = 4)
    assert np.array_equal(packed.numpy(), (c[:, 0::2] | (c[:, 1::2] << 4)).astype(np.uint8))
    assert ops.pack_pq4(torch.tensor([[1, 2, 15, 0]], dtype=torch.uint8)).tolist() == [[0x21, 0x0F]]
    assert ops.is_pq4(torch.empty(8, 16, 4)) and not ops.is_pq4(torch.empty(8, 256, 4))


def _new(name, *args):
    from vector_line_quantization_b200 import index as vi

    out = __import__("ctypes").c_void_p()
    rc = getattr(vi.host(), name)(*args, __import__("ctypes").byref(out))
    return rc, vi.host().vlq_host_last_error().decode()


# the code format is checked before the resources are used: with res = NULL an accepted format fails on the resources
@pytest.mark.parametrize("bits,M,ok", [(8, 16, True), (4, 16, True), (4, 32, True), (8, 15, True), (4, 15, False),
                                       (4, 7, False), (6, 16, False), (16, 16, False), (2, 16, False), (0, 16, False)])
def test_ivfpq_constructor_code_format(bits, M, ok):
    rc, msg = _new("vlq_host_vlq_new", None, 120, 64, M, bits, 8, 16, 1)
    assert rc != 0
    assert ("GpuResources must not be null" in msg) == ok, msg


@pytest.mark.parametrize("bits,ok", [(8, True), (4, False)])
def test_ivfpqr_and_imipq_take_8_bit_codes_only(bits, ok):
    rc, msg = _new("vlq_host_ivfpqr_new", None, 128, 64, 16, 8, bits, 8, 16, 1)
    assert rc != 0 and ("GpuResources must not be null" in msg) == ok, msg
    if not ok:
        assert "8-bit" in msg
        rc, msg = _new("vlq_host_imipq_new", None, 128, 4, 16, bits)
        assert rc != 0 and "8-bit" in msg, msg


def enc(lib, n=100, d=128, M=16, pq=P, lcb=P, nL=256, codes=P):
    return lib.vlq_line_encode_pq4(P, n, d, P, P, P, P, 32, lcb, nL, pq, M, P, None, P, codes, P, None, None)


def scan(lib, nq=10, d=128, M=16, pq=P, ws=P, wsb=1 << 30, k=10, W=64):
    return lib.vlq_scan_topk_pq4(P, nq, d, pq, M, P, 256, P, P, P, P, W, P, P, P, P, P, k, 1024, 0, P, P, ws, wsb, None)


def rcount(lib, nq=10, d=128, M=16, ws=P, wsb=1 << 30, radius=1.0):
    return lib.vlq_range_count_pq4(P, nq, d, P, M, P, 256, P, P, P, P, 64, P, P, P, P, 1024, None, radius, P, ws, wsb,
                                   None)


def rgather(lib, nq=10, d=128, M=16, ws=P, wsb=1 << 30):
    return lib.vlq_range_gather_pq4(P, nq, d, P, M, P, 256, P, P, P, P, 64, P, P, P, P, 1024, None, 1.0, P, P, 0, nq, P,
                                    P, ws, wsb, None)


def dec(lib, n=10, d=128, M=16):
    return lib.vlq_decode_entries_pq4(n, P, 64, P, P, P, P, M, d, P, P, P, 32, P, 256, P, None, None)


def kappa(lib, n=10, d=128, M=16):
    return lib.vlq_recompute_kappa_pq4(n, 64, P, P, P, P, d, P, 32, P, P, M, P, None)


BAD_SHAPES = [dict(M=15), dict(M=7), dict(M=0), dict(M=66), dict(M=24), dict(d=0)]


def test_pq4_entries_reject_bad_shapes_before_any_launch(lib):
    n0 = lib.vlq_launch_count()
    for kw in BAD_SHAPES:
        for f in (enc, scan, rcount, rgather, dec, kappa):
            assert f(lib, **kw) == VLQ_EINVAL, (f.__name__, kw)
    assert enc(lib, d=512, M=16) == VLQ_EINVAL  # d <= 256
    assert scan(lib, d=512, M=16) == VLQ_EINVAL
    assert enc(lib, nL=0) == VLQ_EINVAL and enc(lib, pq=None) == VLQ_EINVAL
    assert scan(lib, k=0) == VLQ_EINVAL and scan(lib, W=0) == VLQ_EINVAL and scan(lib, pq=P + 4) == VLQ_EINVAL
    assert rcount(lib, radius=float("nan")) == VLQ_EINVAL
    assert lib.vlq_launch_count() == n0


def test_pq4_scan_and_range_require_the_workspace(lib):
    n0 = lib.vlq_launch_count()
    need = lib.vlq_scan_topk_workspace_bytes(10, 8)  # nq = 10, M / 2 = 8 table bytes
    assert need == lib.vlq_scan_topk_workspace_bytes(10, 8) > 10 * 8 * 256 * 4
    assert scan(lib, ws=None) == VLQ_EWORKSPACE
    assert scan(lib, wsb=need - 1) == VLQ_EWORKSPACE
    assert scan(lib, ws=P + 4, wsb=need) == VLQ_EINVAL  # alignment
    rneed = lib.vlq_range_workspace_bytes(10, 8, 64, 1024)
    assert rcount(lib, ws=None) == VLQ_EINVAL
    assert rcount(lib, wsb=rneed - 1) == VLQ_EWORKSPACE
    assert rgather(lib, wsb=rneed - 1) == VLQ_EWORKSPACE
    assert lib.vlq_launch_count() == n0


def test_pq4_entries_accept_empty_batches(lib):
    n0 = lib.vlq_launch_count()
    assert enc(lib, n=0) == 0 and dec(lib, n=0) == 0 and kappa(lib, n=0) == 0
    assert scan(lib, nq=0) == 0
    assert lib.vlq_launch_count() == n0
