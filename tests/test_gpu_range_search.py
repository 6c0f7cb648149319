"""range_search: the radius kernels against the oracle's scan of the same lines, against search / search1, determinism
(repeat calls, tiny gather sub-ranges, host API against the operator layer), after remove_ids, and GpuIndexIMIPQ."""
import numpy as np
import pytest

from tests.parity_util import REL_DIST

pytestmark = pytest.mark.gpu


def T(a, dev):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def N(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def vi(cuda):
    from vector_line_quantization_b200 import index

    index.host()
    return index


@pytest.fixture(scope="module")
def res(vi):
    return vi.StandardGpuResources(0)


def _data(kind, n, d, seed):
    from vector_line_quantization_b200 import data

    gen = data.sift_like if kind == "sift" else data.deep_like
    return gen(n, d=d, kc=64, seed=seed)


_models = {}


def _model(vi, res, kind, d, M, C, E):
    """codebooks trained by the host index (nL = 16 lambda levels) + base and query vectors"""
    key = (kind, d, M, C, E)
    if key not in _models:
        t = vi.GpuIndexIVFPQ(res, d, C, M, 8, E, 16)
        t.setTrainIters(4)
        t.train(_data(kind, 20000, d, 1))
        m = dict(t.codebooks())
        m.update(kind=kind, d=d, M=M, C=C, E=E, xb=_data(kind, 20000, d, 2), xq=_data(kind, 60, d, 3))
        _models[key] = m
    return _models[key]


def _ops_index(ops, cuda, m):
    import torch

    cent = T(m["cent"], cuda)
    cn = ops.row_norms(cent)
    edge, ed2, lcb, pq = T(m["edge"], cuda), T(m["edge_d2"], cuda), T(m["lambda_cb"], cuda), T(m["pq"], cuda)
    x = T(m["xb"], cuda)
    A, _ = ops.l2_assign(x, cent, cn)
    enc = ops.line_encode(x, A, cent, edge, ed2, lcb, pq)
    lists = ops.build_lists(m["C"] * m["E"], m["M"], enc.list, enc.codes, enc.lamq, enc.kappa,
                            torch.arange(x.shape[0], dtype=torch.int64, device=cuda))
    return dict(cent=cent, cn=cn, edge=edge, ed2=ed2, lcb=lcb, pq=pq, lists=lists)


def _stream(lines, off, ids, cap):
    """ids of every scanned entry of one query in stream order: lines in slot order, then list position"""
    parts = [ids[off[l]:off[l] + min(off[l + 1] - off[l], cap)] for l in lines if l >= 0]
    return np.concatenate(parts) if parts else np.empty(0, np.int64)


def _rows(lims, D, I):
    return [(D[lims[i]:lims[i + 1]], I[lims[i]:lims[i + 1]]) for i in range(len(lims) - 1)]


def _check_sets(got, want, radius, qn, rel=REL_DIST):
    """per query: id sets equal except entries whose reference distance lies within rel (|dist| + ||q||^2) of the radius;
    distances of shared ids agree within rel.  got / want: [(D full, I)] per query"""
    for i, ((dg, ig), (dw, iw)) in enumerate(zip(got, want)):
        scale = np.abs(dw).max(initial=0.0) + qn[i]
        gm, wm = dict(zip(ig.tolist(), dg.tolist())), dict(zip(iw.tolist(), dw.tolist()))
        for k in set(gm) ^ set(wm):
            d = wm.get(k, gm.get(k))
            assert abs(d - radius) <= rel * (abs(d) + qn[i]), (i, k, d, radius)
        for k in set(gm) & set(wm):
            assert abs(gm[k] - wm[k]) <= rel * scale, (i, k, gm[k], wm[k])


# ------------------------------------------------------------------------------------------------ against the oracle
GEOMS = {  # (kind, d, M, C, E): about 5 entries per line, and about 300 (long lists, beyond a cap of 64)
    "d128M16": ("sift", 128, 16, 256, 16), "d96M8": ("deep", 96, 8, 256, 16), "d128M32": ("sift", 128, 32, 256, 16),
    "d128M16_long": ("sift", 128, 16, 16, 4), "d96M8_long": ("deep", 96, 8, 16, 4),
}


@pytest.mark.parametrize("cap", [1024, 64])
@pytest.mark.parametrize("geom", list(GEOMS))
def test_range_vs_oracle(vi, res, cuda, oracle, geom, cap):
    from vector_line_quantization_b200 import ops

    m = _model(vi, res, *GEOMS[geom])
    gi = _ops_index(ops, cuda, m)
    P, W = (16, 128) if m["C"] > 16 else (4, 12)
    q = T(m["xq"], cuda)
    lines = ops.coarse_lines(q, gi["cent"], gi["cn"], gi["edge"], gi["ed2"], P, W)
    lst = N(lines[0])
    off, ids = N(gi["lists"].offsets), N(gi["lists"].ids)
    streams = [_stream(row, off, ids, cap) for row in lst]
    k = max(len(s) for s in streams)
    canon = N(ops.rotate_codes(gi["lists"].offsets, gi["lists"].codes, inverse=True))
    Do, Io = oracle.scan_lines(m["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], off, canon,
                               N(gi["lists"].lamq), ids, lst, k, cap)
    qn = (m["xq"].astype(np.float64) ** 2).sum(1)
    full = Do.astype(np.float64) + qn[:, None]
    # a radius that keeps about 40 entries per query, and +inf (every scanned entry)
    radius = float(np.median(np.sort(np.where(Io >= 0, full, np.inf), axis=1)[:, 40]))
    for r in (radius, float("inf")):
        lims, D, I = ops.range_scan_lines(q, gi["pq"], gi["lcb"], lines, gi["ed2"], gi["lists"], r, cap=cap,
                                          row_add=ops.row_norms(q))
        lims, D, I = N(lims), N(D), N(I)
        got = _rows(lims, D, I)
        want = [(full[i][(Io[i] >= 0) & (full[i] < r)], Io[i][(Io[i] >= 0) & (full[i] < r)]) for i in range(len(qn))]
        _check_sets(got, want, r, qn)
        assert np.all(D < r)
        for (dg, ig), s in zip(got, streams):  # stream order: positions in the query's entry stream strictly increase
            pos = {v: j for j, v in enumerate(s.tolist())}
            assert np.all(np.diff([pos[v] for v in ig.tolist()]) > 0)
        if r == float("inf"):
            assert all(np.array_equal(ig, s) for (_, ig), s in zip(got, streams))
        else:
            assert 10 * len(qn) < lims[-1] < 100 * len(qn)


# ------------------------------------------------------------------------------------------------ index level
def _index(vi, res, m, x=None, ids=None, tc=True):
    idx = vi.GpuIndexIVFPQ(res, m["d"], m["C"], m["M"], 8, m["E"], 16, use_tensor_cores=tc)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    if x is not None:
        for s in range(0, len(x), 7000):
            idx.add_with_ids(x[s:s + 7000], ids[s:s + 7000])
    return idx


def test_range_vs_search_and_search1(vi, res, cuda):
    m = _model(vi, res, *GEOMS["d128M16_long"])
    xb, xq = m["xb"], m["xq"]
    idx = _index(vi, res, m, xb, np.arange(len(xb), dtype=np.int64))
    qn = (xq.astype(np.float64) ** 2).sum(1)
    # the queries that scan <= 1024 entries: search(k = 1024) sees all of them
    idx.setNumProbes(2)
    idx.w1_ = 2
    cand = idx.search1(xq, 4096)
    ok = (cand >= 0).sum(1) <= 1024
    assert ok.sum() >= 10
    D, I = idx.search(xq, 1024)
    full = D.astype(np.float64) + qn[:, None]
    r = float(np.median(np.sort(np.where(I >= 0, full, np.inf), axis=1)[ok, 30]))
    lims, Dr, Ir = idx.range_search(xq, r)
    rows = _rows(lims, Dr, Ir)
    _check_sets([rows[i] for i in np.flatnonzero(ok)],
                [(full[i][(I[i] >= 0) & (full[i] < r)], I[i][(I[i] >= 0) & (full[i] < r)]) for i in np.flatnonzero(ok)],
                r, qn[ok])
    assert lims[-1] > 5 * ok.sum()
    # radius +inf with no list cut by the cap: the candidate lists of search1, in their order, beyond 1024 per query
    idx.setNumProbes(4)
    idx.w1_ = 16
    idx.setListCap(1 << 20)
    cand = idx.search1(xq, 16384)
    assert (cand[:, -1] < 0).all()
    lims, Dr, Ir = idx.range_search(xq, float("inf"))
    for i, (_, ig) in enumerate(_rows(lims, Dr, Ir)):
        assert np.array_equal(ig, cand[i][cand[i] >= 0])
    assert np.median(np.diff(lims)) > 1024
    idx.setListCap(1024)
    # a radius below every distance: empty rows; n = 0: lims = {0}
    lims, Dr, Ir = idx.range_search(xq, -1.0)
    assert np.all(lims == 0) and len(Dr) == 0 and len(Ir) == 0
    lims, Dr, Ir = idx.range_search(xq[:0], 5.0)
    assert lims.tolist() == [0] and len(Dr) == 0
    with pytest.raises(vi.FaissException, match="NaN"):
        idx.range_search(xq, float("nan"))


def test_range_deterministic_tiles_staging_and_host_vs_ops(vi, res, cuda, monkeypatch):
    """n = 12 000 queries (three query tiles of the host layer): repeat calls, gathers in tiny sub-ranges, CUDA query
    arrays and the operator layer all give the same bits"""
    import torch

    from vector_line_quantization_b200 import ops

    m = _model(vi, res, *GEOMS["d128M16"])
    xb = m["xb"]
    xq = _data("sift", 12000, 128, 7)
    P, W = 16, 128
    idx = _index(vi, res, m)
    idx.add(xb)  # ids 0 .. n - 1, one chunk
    idx.setNumProbes(P)
    idx.w1_ = W
    qn = (xq.astype(np.float64) ** 2).sum(1)
    D, I = idx.search(xq[:200], 100)
    r = float(np.median(D[:, 40].astype(np.float64) + qn[:200]))
    a = idx.range_search(xq, r)
    assert a[0][-1] > 10 * len(xq)
    b = idx.range_search(xq, r)
    with monkeypatch.context() as mp:
        mp.setenv("VLQ_RANGE_STAGING_BYTES", "4096")  # about 340 results per gather
        c = idx.range_search(xq, r)
    d = idx.range_search(T(xq, cuda), r)
    for other in (b, c, d):
        for x, y in zip(a, other):
            assert x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))
    # the same index through the operator layer (tensor-core assignment and coarse route, as the host index uses)
    cent = T(m["cent"], cuda)
    pack = ops.CentPack(cent)
    edge, ed2, lcb, pq = T(m["edge"], cuda), T(m["edge_d2"], cuda), T(m["lambda_cb"], cuda), T(m["pq"], cuda)
    x = T(xb, cuda)
    A, _ = ops.l2_assign_tc(x, pack, want_dist=False)
    enc = ops.line_encode(x, A, cent, edge, ed2, lcb, pq)
    lists = ops.build_lists(m["C"] * m["E"], m["M"], enc.list, enc.codes, enc.lamq, enc.kappa,
                            torch.arange(len(xb), dtype=torch.int64, device=cuda))
    for stage in (None, 50):
        o = ops.range_search(T(xq, cuda), cent, pack.cnorm, edge, ed2, lcb, pq, lists, P, W, r, pack=pack,
                             stage_results=stage)
        for x_, y in zip(a, o):
            assert np.array_equal(x_.view(np.uint8), N(y).view(np.uint8))
    o = ops.range_search(T(xq[:0], cuda), cent, pack.cnorm, edge, ed2, lcb, pq, lists, P, W, r, pack=pack)
    assert N(o[0]).tolist() == [0] and o[1].numel() == 0


def test_range_after_remove_ids_equals_index_without(vi, res, cuda):
    m = _model(vi, res, *GEOMS["d96M8_long"])
    xb, xq = m["xb"], m["xq"]
    ids = np.random.RandomState(4).permutation(100000)[:len(xb)].astype(np.int64) * 3 + 5
    gone = np.random.RandomState(5).rand(len(xb)) < 0.3
    a = _index(vi, res, m, xb, ids)
    b = _index(vi, res, m, xb[~gone], ids[~gone])
    assert a.remove_ids(ids[gone]) == int(gone.sum())
    qn = (xq.astype(np.float64) ** 2).sum(1)
    for cap in (1024, 64):
        for idx in (a, b):
            idx.setNumProbes(4)
            idx.w1_ = 12
            idx.setListCap(cap)
        D, _ = b.search(xq, 50)
        for r in (float(np.median(D[:, 20].astype(np.float64) + qn)), float("inf")):
            ra, rb = a.range_search(xq, r), b.range_search(xq, r)
            for x, y in zip(ra, rb):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), cap
            assert ra[0][-1] > 0 and not np.isin(ra[2], ids[gone]).any()


def test_imipq_range_equals_search_below_radius(vi, res, cuda):
    from vector_line_quantization_b200 import data

    xt = data.sift_like(20000, kc=64, seed=21)
    xb = data.sift_like(20000, kc=64, seed=22)
    xq = data.sift_like(50, kc=64, seed=23)
    idx = vi.GpuIndexIMIPQ(res, 128, 4, 16)
    idx.setTrainIters(4)
    idx.train(xt)
    idx.add_with_ids(xb, np.arange(len(xb), dtype=np.int64) * 7 + 3)
    idx.setNumProbes(4)
    D, I = idx.search(xq, 1024)
    ok = I[:, -1] < 0  # the queries whose scanned entries all fit k = 1024
    assert ok.sum() >= 10
    qn = (xq.astype(np.float64) ** 2).sum(1)
    full = D.astype(np.float64)
    r = float(np.median(full[ok, 25]))
    lims, Dr, Ir = idx.range_search(xq, r)
    assert 5 * len(xq) < lims[-1]
    rows = _rows(lims, Dr, Ir)
    _check_sets([rows[i] for i in np.flatnonzero(ok)],
                [(full[i][(I[i] >= 0) & (full[i] < r)], I[i][(I[i] >= 0) & (full[i] < r)]) for i in np.flatnonzero(ok)],
                r, qn[ok])
    lims, Dr, Ir = idx.range_search(xq, float("inf"))
    assert np.array_equal(np.diff(lims)[ok], (I[ok] >= 0).sum(1))
    assert (np.diff(lims)[~ok] >= 1024).all()
