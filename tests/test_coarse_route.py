"""The coarse-stage route rule, its workspace size and the argument checks of vlq_coarse_lines.  No GPU: the library
loads without one, and vlq_coarse_lines checks every argument before its first CUDA call."""
import pytest

from vector_line_quantization_b200 import _abi

VLQ_OK, VLQ_EINVAL, VLQ_EWORKSPACE = 0, -1, -2

# (d, C, P, E, W) -> vlq_coarse_exact_supported / vlq_coarse_exact_preferred (test_abi.test_coarse_route_dispatch_rule)
SUPPORTED = [((128, 65536, 64, 32, 256), 1), ((130, 65536, 8, 32, 32), 0), ((256, 65536, 8, 32, 32), 0),
             ((128, 65536, 200, 32, 256), 0), ((128, 1 << 20, 8, 32, 32), 0), ((128, 65536, 0, 32, 32), 0)]
PREFERRED = [((128, 65536, 64, 32, 256), 0), ((128, 65536, 8, 32, 32), 1), ((128, 65536, 16, 32, 64), 0),
             ((96, 65536, 8, 64, 32), 0), ((96, 65536, 4, 64, 16), 1)]


@pytest.fixture
def lib(monkeypatch):
    monkeypatch.delenv("VLQ_COARSE_MATRIX", raising=False)
    monkeypatch.delenv("VLQ_COARSE_EXACT", raising=False)
    return _abi.lib()


def test_route_rule(lib, monkeypatch):
    for row, preferred in PREFERRED:
        assert lib.vlq_coarse_route(*row, 1) == (2 if preferred else 1), row
        assert lib.vlq_coarse_route(*row, 0) == 0, row
    monkeypatch.setenv("VLQ_COARSE_EXACT", "1")  # matrix-free wherever it is supported
    for row, supported in SUPPORTED:
        assert lib.vlq_coarse_route(*row, 1) == (2 if supported else 1), row
        assert lib.vlq_coarse_route(*row, 0) == 0, row
    monkeypatch.setenv("VLQ_COARSE_MATRIX", "1")  # the tensor-core matrix route wins over VLQ_COARSE_EXACT
    assert lib.vlq_coarse_route(128, 65536, 8, 32, 32, 1) == 1
    assert lib.vlq_coarse_route(128, 65536, 8, 32, 32, 0) == 0


def test_switches_are_read_per_call(lib, monkeypatch):
    small, large = (128, 65536, 8, 32, 32, 1), (128, 65536, 64, 32, 256, 1)
    assert lib.vlq_coarse_route(*small) == 2 and lib.vlq_coarse_route(*large) == 1
    monkeypatch.setenv("VLQ_COARSE_MATRIX", "1")
    assert lib.vlq_coarse_route(*small) == 1
    monkeypatch.delenv("VLQ_COARSE_MATRIX")
    assert lib.vlq_coarse_route(*small) == 2
    monkeypatch.setenv("VLQ_COARSE_EXACT", "1")
    assert lib.vlq_coarse_route(*large) == 2
    monkeypatch.delenv("VLQ_COARSE_EXACT")
    assert lib.vlq_coarse_route(*large) == 1


def test_workspace_bytes(lib):
    nq, C = 1000, 65536
    ws = lambda n, P, W, pack: lib.vlq_coarse_lines_workspace_bytes(n, 128, C, P, 32, W, pack)  # noqa: E731
    assert ws(nq, 8, 32, 1) < nq * C * 4  # route 2: no distance tile
    assert ws(nq, 64, 256, 1) >= nq * C * 4  # route 1
    assert ws(nq, 8, 32, 0) >= nq * C * 4  # route 0
    for P, W, pack in ((8, 32, 1), (64, 256, 1), (8, 32, 0)):
        assert ws(2 * nq, P, W, pack) > ws(nq, P, W, pack)
        assert ws(nq, P, W, pack) % 256 == 0


def test_coarse_lines_argument_checks(lib):
    p = 1 << 20  # stands for a device pointer: no call below reaches the device

    def call(nq=64, P=8, W=32, pack=0, q=p, ws_bytes=1):
        return lib.vlq_coarse_lines(q, nq, 128, p, p, pack, 1.0, 65536, P, p, p, 32, W, None, p, p, p, p, ws_bytes, None)

    assert call(nq=0, ws_bytes=0) == VLQ_OK
    for pack in (0, p):  # route 0; route 2 (P = 8, W = 32)
        assert call(pack=pack) == VLQ_EWORKSPACE
    assert call(pack=p, P=64, W=256) == VLQ_EWORKSPACE  # route 1
    assert call(P=1025) == VLQ_EINVAL
    assert call(pack=p, q=p + 4, ws_bytes=1 << 40) == VLQ_EINVAL  # route 2 reads q in 16-byte vectors
