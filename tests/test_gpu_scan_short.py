"""The short-list scan (scan_short_kernel, search.cu) against the general block-synchronous scan (VLQ_SCAN_NO_SMALL=1):
bit-identical distances and ids, on synthetic lists where one launch mixes queries the short kernel holds (<= 4096
stream positions) with queries it hands to the general kernel through the overflow list."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHORT_CAP = 16 * 256  # stream positions scan_short_kernel holds (kShortCap)


@pytest.fixture(scope="module")
def ops():
    from vector_line_quantization_b200 import ops

    return ops


def _index(torch, ops, dev, M, W, nq, seed, ties=False):
    """lists of a short pool (a query of W of them stays under SHORT_CAP) and a long pool (a query over them overflows);
    even queries pick short lines, odd queries long ones; one slot in 16 is empty (-1)"""
    g = np.random.default_rng(seed)
    n_short, n_long = 2048, 512
    avg = max(1, 1500 // W)
    lens = np.concatenate([g.integers(0, 2 * avg + 1, n_short), g.integers(max(40, 6000 // W), max(41, 6000 // W) + 60,
                                                                            n_long)])
    off = np.zeros(len(lens) + 1, np.int64)
    off[1:] = np.cumsum(lens)
    n = int(off[-1])
    if ties:  # a handful of distinct entries (all M code bytes equal: the list-position rotation keeps them equal)
        codes = np.repeat(g.integers(0, 3, (n, 1)), M, axis=1).astype(np.uint8)
        lamq = g.integers(0, 2, n).astype(np.uint8)
        kappa = g.integers(0, 3, n).astype(np.float32)
    else:
        codes = g.integers(0, 256, (n, M)).astype(np.uint8)
        lamq = g.integers(0, 256, n).astype(np.uint8)
        kappa = (g.standard_normal(n) * 100).astype(np.float32)
    lines = np.where(np.arange(nq)[:, None] % 2 == 0, g.integers(0, n_short, (nq, W)),
                     n_short + g.integers(0, n_long, (nq, W))).astype(np.int32)
    lines[g.random((nq, W)) < 1 / 16] = -1
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    lists = ops.Lists(t(off), t(codes), t(lamq), t(kappa), t(g.permutation(n).astype(np.int64)))
    d = 8 * M
    q = t(g.standard_normal((nq, d)).astype(np.float32))
    pq = t(g.standard_normal((M, 256, d // M)).astype(np.float32))
    lcb = t(g.random(256).astype(np.float32))
    if ties:
        t1, t6 = t(np.ones((nq, W), np.float32)), t(np.zeros((nq, W), np.float32))
        ed2 = t(np.ones(len(lens), np.float32))
    else:
        t1 = t((g.random((nq, W)) * 10).astype(np.float32))
        t6 = t(g.standard_normal((nq, W)).astype(np.float32))
        ed2 = t((g.random(len(lens)) * 4 + 0.5).astype(np.float32))
    total = np.where(lines >= 0, np.minimum(lens[np.maximum(lines, 0)], 1024), 0).sum(axis=1)
    return dict(lists=lists, q=q, pq=pq, lcb=lcb, lines=t(lines), t1=t1, t6=t6, ed2=ed2, total=total)


def _both(ops, monkeypatch, r, k, **kw):
    args = (r["q"], r["pq"], r["lcb"], r["lines"], r["t1"], r["t6"], r["ed2"], r["lists"], k, 1024)
    D0, I0 = ops.scan_topk(*args, list_len_hint=0, **kw)
    monkeypatch.setenv("VLQ_SCAN_NO_SMALL", "1")
    D1, I1 = ops.scan_topk(*args, list_len_hint=0, **kw)
    monkeypatch.delenv("VLQ_SCAN_NO_SMALL")
    return D0, I0, D1, I1


@pytest.mark.parametrize("M", [8, 16])
@pytest.mark.parametrize("W", [1, 256, 1024])
@pytest.mark.parametrize("k", [1, 100, 256, 257, 1024])
def test_short_scan_equals_general_scan(ops, cuda, monkeypatch, M, W, k):
    import torch

    r = _index(torch, ops, cuda, M, W, 96, seed=W * 7 + M)
    if W > 1:  # one launch holds short queries and overflowing ones
        assert (r["total"] <= SHORT_CAP).any() and (r["total"] > SHORT_CAP).any()
    D0, I0, D1, I1 = _both(ops, monkeypatch, r, k)
    assert torch.equal(D0, D1) and torch.equal(I0, I1)
    assert bool((I0 >= 0).any())


@pytest.mark.parametrize("M", [8, 16])
@pytest.mark.parametrize("case", ["slab_index", "masked", "nan", "ties"])
def test_short_scan_equals_general_scan_special(ops, cuda, monkeypatch, M, case):
    """ids = NULL (slab indexes), a filter mask (+inf kappa off the 1 % members: +inf keys are valid and follow every
    member), NaN kappa (never selected: queries with fewer than k others get FLT_MAX padding), and an index of exact
    distance ties straddling the k-th place"""
    import torch

    r = _index(torch, ops, cuda, M, 256, 96, seed=11 + M, ties=case == "ties")
    kw = {}
    kap = r["lists"].kappa
    if case == "slab_index":
        kw["slab_index"] = True
    elif case == "masked":
        g = torch.Generator(device=cuda).manual_seed(3)
        member = torch.rand(kap.shape, device=cuda, generator=g) < 0.01
        kw["kappa"] = torch.where(member, kap, torch.full_like(kap, float("inf")))
    elif case == "nan":
        g = torch.Generator(device=cuda).manual_seed(4)
        kw["kappa"] = torch.where(torch.rand(kap.shape, device=cuda, generator=g) < 0.98, torch.full_like(kap, float("nan")), kap)
    D0, I0, D1, I1 = _both(ops, monkeypatch, r, 100, **kw)
    assert torch.equal(D0, D1) and torch.equal(I0, I1)
    assert not bool(torch.isnan(D0).any())
    short = torch.from_numpy(r["total"] <= SHORT_CAP).to(cuda)
    if case == "masked":
        assert bool(torch.isinf(D0[short]).any())
    if case == "nan":
        assert bool((D0[short] == float(np.finfo(np.float32).max)).any()) and bool((I0[short] == -1).any())
    if case == "ties":
        assert int(((D0[:, 1:] == D0[:, :-1]) & (I0[:, 1:] >= 0)).sum()) > 0
