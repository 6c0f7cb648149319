"""GpuIndexIVFPQR: the refinement encode (vlq_refine_encode), the re-rank (vlq_refine_topk) and the refined decode
against numpy restatements, the refinement codes through adds / commit / remove_ids, and the index against a twin
GpuIndexIVFPQ built from the same codebooks and adds."""
from types import SimpleNamespace

import numpy as np
import pytest

from tests.parity_util import REL_DIST, REL_TIE
from tests.test_gpu_reconstruct import _anchors, _assert_bits, _build

pytestmark = pytest.mark.gpu

M2 = 16


def N(t):
    return t.detach().cpu().numpy()


def T(a, dev):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


@pytest.fixture(scope="module")
def ops(cuda):
    from vector_line_quantization_b200 import ops as _ops

    return _ops


@pytest.fixture(scope="module")
def vi(cuda):
    from vector_line_quantization_b200 import index

    index.host()
    return index


@pytest.fixture(scope="module")
def res(vi):
    return vi.StandardGpuResources(0)


# ------------------------------------------------------------------------------------------------ restatements
def _x1(cent, edge, lcb, pq, lst, lamq, codes):
    """first-level decode from canonical codes, numpy float32, each operation rounded as written"""
    M = pq.shape[0]
    pv = pq[np.arange(M)[None, :], codes].reshape(len(lst), -1)
    lh = lcb[lamq]
    c, s = cent[lst // edge.shape[1]], cent[edge.reshape(-1)[lst]]
    return ((np.float32(1) - lh)[:, None] * c + lh[:, None] * s) + pv


def _p2(pq2, code2):
    M = pq2.shape[0]
    return pq2[np.arange(M)[None, :], code2].reshape(len(code2), -1)


def _check_codes(r2, code2, pq2):
    """code2 is the float64 argmin of ||r2_m - pq2[m][j]||^2 per sub-quantizer, up to verified near-ties; returns the
    share of exact argmin matches"""
    M, _, ds = pq2.shape
    c = pq2.astype(np.float64)
    cn = (c ** 2).sum(-1)  # [M][256]
    exact = 0
    for s in range(0, len(r2), 1024):
        r = r2[s:s + 1024].astype(np.float64).reshape(-1, M, ds)
        rn = (r ** 2).sum(-1)
        dist = rn[:, :, None] - 2 * np.einsum("nmd,mjd->nmj", r, c) + cn[None]  # [n][M][256]
        best = dist.min(-1)
        got = np.take_along_axis(dist, code2[s:s + 1024].astype(np.int64)[..., None], -1)[..., 0]
        bad = got - best > REL_TIE * (rn + cn.max(-1)[None])
        assert not bad.any(), (np.argwhere(bad)[:5], got[bad][:5], best[bad][:5])
        exact += (code2[s:s + 1024] == dist.argmin(-1)).sum()
    return exact / code2.size


# ------------------------------------------------------------------------------------------------ encode
@pytest.mark.parametrize("d", [64, 96, 128])
@pytest.mark.parametrize("m2", [8, 16, 32])
def test_refine_encode_matches_restatement(ops, cuda, d, m2):
    rng = np.random.default_rng(d * 100 + m2)
    C, E, M, n = 64, 8, 16, 3000
    cent, edge, lcb, pq = _anchors(rng, d, M, C, E)
    pq2 = (rng.standard_normal((m2, 256, d // m2)) * 2).astype(np.float32)
    lst = rng.integers(0, C * E, n).astype(np.int32)
    lst[::37] = -1  # rows the encoder skipped (NaN input)
    lamq = rng.integers(0, 256, n).astype(np.uint8)
    codes = rng.integers(0, 256, (n, M)).astype(np.uint8)
    safe = np.maximum(lst, 0)
    x1 = _x1(cent, edge, lcb, pq, safe, lamq, codes)
    x = (x1 + rng.standard_normal((n, d)).astype(np.float32) * 3).astype(np.float32)
    x[lst < 0] = np.nan
    tabs = [T(a, cuda) for a in (pq, cent, edge, lcb, pq2)]
    enc = SimpleNamespace(list=T(lst, cuda), lamq=T(lamq, cuda), codes=T(codes, cuda))
    code2, r2 = ops.refine_encode(T(x, cuda), enc, *tabs, want_residual=True)
    code2, r2 = N(code2), N(r2)
    ok = lst >= 0
    _assert_bits(r2[ok], (x - x1)[ok])
    assert (r2[~ok] == 0).all() and (code2[~ok] == 0).all()
    assert _check_codes(r2[ok], code2[ok], pq2) > 0.999
    # training mode: r2 only, the same bits
    none, r2b = ops.refine_encode(T(x, cuda), enc, *tabs[:4], None)
    assert none is None
    _assert_bits(N(r2b), r2)


# ------------------------------------------------------------------------------------------------ re-rank
def _slab(rng, C, E, M, m2, d, twins=True):
    """lists with long members (the code rotation matters), empty lists, canonical codes; entry pairs that decode to
    the same x2 (exact ties between different ids)"""
    nl = C * E
    lens = rng.poisson(6, nl)
    lens[::5] = 0
    lens[3::17] = 40 + rng.integers(0, 30, len(lens[3::17]))
    off = np.zeros(nl + 1, np.int64)
    off[1:] = np.cumsum(lens)
    n = int(off[-1])
    codes = rng.integers(0, 256, (n, M)).astype(np.uint8)
    lamq = rng.integers(0, 256, n).astype(np.uint8)
    code2 = rng.integers(0, 256, (n, m2)).astype(np.uint8)
    ids = rng.permutation(4 * n)[:n].astype(np.int64) + 11
    tw = []
    if twins:
        for l in np.flatnonzero(lens >= 2)[:50]:
            a, b = off[l], off[l] + 1
            codes[b], lamq[b], code2[b] = codes[a], lamq[a], code2[a]
            tw.append((a, b))
    lst = np.searchsorted(off, np.arange(n), side="right") - 1
    return off, codes, lamq, code2, ids, lst, tw


@pytest.mark.parametrize("kc,ks", [(1, [1]), (7, [1, 7]), (100, [1, 10, 100]), (1024, [10, 100, 1024])])
def test_refine_topk_matches_restatement(ops, cuda, kc, ks):
    import torch

    rng = np.random.default_rng(kc)
    d, C, E, M = 128, 64, 8, 16
    cent, edge, lcb, pq = _anchors(rng, d, M, C, E)
    pq2 = (rng.standard_normal((M2, 256, d // M2)) * 2).astype(np.float32)
    off, codes, lamq, code2, ids, lst, tw = _slab(rng, C, E, M, M2, d)
    n = len(ids)
    x2 = _x1(cent, edge, lcb, pq, lst, lamq, codes) + _p2(pq2, code2)
    nq = 24
    q = (x2[rng.integers(0, n, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 4).astype(np.float32)
    cand = rng.integers(0, n, (nq, kc)).astype(np.int64)
    cand[rng.random((nq, kc)) < 0.1] = -1                        # holes
    if kc > 2:
        cand[:, kc // 2] = cand[:, 0]                            # repeated entries
        a, b = tw[0]
        cand[0, 1], cand[0, 2] = b, a                            # an exact tie between two ids: b comes first
    cand[1] = -1                                                 # a query without candidates
    dev = cuda
    lists = ops.Lists(T(off, dev), ops.rotate_codes(T(off, dev), T(codes, dev)), T(lamq, dev), None, T(ids, dev))
    tabs = [T(a, dev) for a in (pq, cent, edge, lcb, pq2)]
    dist64 = ((q.astype(np.float64)[:, None, :] - x2.astype(np.float64)[None]) ** 2).sum(-1)  # [nq][n]
    qn = (q.astype(np.float64) ** 2).sum(-1)
    for k in ks:
        D, I = ops.refine_topk(T(q, dev), T(cand, dev), k, lists, T(code2, dev), *tabs)
        Ds, S = ops.refine_topk(T(q, dev), T(cand, dev), k, lists, T(code2, dev), *tabs, labels=False)
        D, I, Ds, S = N(D), N(I), N(Ds), N(S)
        _assert_bits(Ds, D)
        assert np.array_equal(np.where(S >= 0, ids[np.maximum(S, 0)], -1), I)
        for r in range(nq):
            valid = cand[r][cand[r] >= 0]
            want = np.sort(dist64[r, valid])[:k]
            got = S[r][S[r] >= 0]
            assert len(got) == min(k, len(valid))
            assert (D[r][len(got):] == np.float32(np.finfo(np.float32).max)).all() and (I[r][len(got):] == -1).all()
            tol = REL_DIST * (np.abs(want) + qn[r])
            assert (np.abs(D[r][:len(got)] - dist64[r, got]) <= REL_DIST * (dist64[r, got] + qn[r])).all()
            assert (np.abs(dist64[r, got] - want[:len(got)]) <= tol[:len(got)]).all()  # the k best up to near-ties
            # ascending by (distance, candidate position): each output consumes the first unused position of its entry
            used = set()
            pos = []
            for s in got:
                p = next(i for i in range(kc) if cand[r, i] == s and i not in used)
                used.add(p)
                pos.append(p)
            key = list(zip(D[r][:len(got)].tolist(), pos))
            assert key == sorted(key)
        if kc > 2 and k >= 3:
            got0 = S[0].tolist()
            a, b = tw[0]
            if a in got0 and b in got0:
                assert got0.index(b) < got0.index(a)


def test_refine_topk_in_place(ops, cuda):
    """k == kc: the labels may overwrite the candidates they come from"""
    rng = np.random.default_rng(5)
    d, C, E, M = 64, 32, 4, 8
    cent, edge, lcb, pq = _anchors(rng, d, M, C, E)
    pq2 = (rng.standard_normal((8, 256, d // 8)) * 2).astype(np.float32)
    off, codes, lamq, code2, ids, lst, _ = _slab(rng, C, E, M, 8, d, twins=False)
    q = (rng.standard_normal((50, d)) * 40).astype(np.float32)
    cand = rng.integers(-1, len(ids), (50, 64)).astype(np.int64)
    lists = ops.Lists(T(off, cuda), ops.rotate_codes(T(off, cuda), T(codes, cuda)), T(lamq, cuda), None, T(ids, cuda))
    tabs = [T(a, cuda) for a in (pq, cent, edge, lcb, pq2)]
    D, S = ops.refine_topk(T(q, cuda), T(cand, cuda), 64, lists, T(code2, cuda), *tabs, labels=False)
    from vector_line_quantization_b200 import _abi

    c, qt, c2 = T(cand, cuda), T(q, cuda), T(code2, cuda)  # held: the call reads them after the last reference here
    D2 = c.new_empty((50, 64), dtype=D.dtype)
    pqt, centt, edget, lcbt, pq2t = tabs
    _abi.call("vlq_refine_topk", qt.data_ptr(), 50, d, c.data_ptr(), 64, 64, len(off) - 1, lists.offsets.data_ptr(),
              lists.codes.data_ptr(), lists.lamq.data_ptr(), 0, c2.data_ptr(), M, pqt.data_ptr(), centt.data_ptr(),
              edget.data_ptr(), E, lcbt.data_ptr(), 256, pq2t.data_ptr(), 8, D2.data_ptr(), c.data_ptr(), ops._stream())
    _assert_bits(N(D2), N(D))
    assert np.array_equal(N(c), N(S))


# ------------------------------------------------------------------------------------------------ index
@pytest.fixture(scope="module")
def pq2(vi, res, small_model):
    """the refinement codebook GpuIndexIVFPQR.train learns on the small model's training rows"""
    m = small_model
    idx = vi.GpuIndexIVFPQR(res, m["d"], m["C"], m["M"], M2, 8, m["E"], 256)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    with pytest.raises(vi.FaissException):
        idx.add(m["xb"][:10])  # no refinement codebook yet
    with pytest.raises(vi.FaissException):
        idx.search(m["xq"], 10)
    idx.setTrainIters(8)
    idx.train(m["xt"])
    cb = idx.refineCodebook()
    assert cb.shape == (M2, 256, m["d"] // M2) and np.isfinite(cb).all()
    return cb


def _refine(vi, res, m, pq2, xb, ids=None, chunks=2, k_factor=4.0):
    idx = vi.GpuIndexIVFPQR(res, m["d"], m["C"], m["M"], M2, 8, m["E"], 256)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    idx.setRefineCodebook(pq2)
    idx.k_factor = k_factor
    step = (len(xb) + chunks - 1) // chunks
    for s in range(0, len(xb), step):
        if ids is None:
            idx.add(xb[s:s + step])
        else:
            idx.add_with_ids(xb[s:s + step], ids[s:s + step])
    return idx


def _setup(*idxs):
    for i in idxs:
        i.setNumProbes(16)
        i.w1_ = 128


def _kc(k, kf):
    return min(1024, max(k, int(np.floor(k * np.float64(np.float32(kf))))))


def _lists_of(idx, m):
    """(ids, code2) of every list"""
    return [(idx.getList(l)[2], idx.getListRefineCodes(l)) for l in range(m["C"] * m["E"])]


def test_reconstruct_is_twin_plus_p2_and_codes_match_vectors(vi, res, small_model, pq2):
    m = small_model
    xb = m["xb"]
    idx, twin = _refine(vi, res, m, pq2, xb), _build(vi, res, m, xb)
    n = idx.ntotal
    R, R1 = idx.reconstruct_n(0, n), twin.reconstruct_n(0, n)
    code2 = np.zeros((n, M2), np.uint8)
    for ids, c2 in _lists_of(idx, m):
        code2[ids] = c2
    _assert_bits(R, R1 + _p2(pq2, code2))
    assert _check_codes(xb - R1, code2, pq2) > 0.999  # code2 = PQ2(x - x1) of the stored vector
    keys = np.array([17, 3, 17, 19999], np.int64)
    _assert_bits(idx.reconstruct_batch(keys), R[keys])
    _assert_bits(idx.reconstruct(5)[None], R[5][None])
    # quality on the fixed seed: the second level lowers the reconstruction error
    assert ((xb - R).astype(np.float64) ** 2).sum(1).mean() < ((xb - R1).astype(np.float64) ** 2).sum(1).mean()


def test_aux_column_through_adds_commit_and_removal(vi, res, small_model, pq2):
    m = small_model
    xb = m["xb"][:12000]
    ids = np.arange(len(xb), dtype=np.int64) * 2 + 1
    idx = _refine(vi, res, m, pq2, xb[:8000], ids[:8000], chunks=3)
    idx.getListLength(0)  # commit
    assert idx.remove_ids(vi.IDSelectorRange(1001, 3001)) == 1000
    gone = ids[rng_pick(len(ids[:8000]), 700)]
    removed = idx.remove_ids(gone)
    for s in range(8000, 12000, 1500):
        idx.add_with_ids(xb[s:s + 1500], ids[s:s + 1500])
    keep = ~(((ids >= 1001) & (ids < 3001)) | np.isin(ids, gone))
    keep[8000:] = True
    assert removed == int((~keep[:8000]).sum()) - 1000
    fresh = _refine(vi, res, m, pq2, xb[keep], ids[keep], chunks=1)
    assert idx.ntotal == fresh.ntotal
    for (i1, c1), (i2, c2) in zip(_lists_of(idx, m), _lists_of(fresh, m)):
        assert np.array_equal(i1, i2) and np.array_equal(c1, c2)
    _setup(idx, fresh)
    D1, I1 = idx.search(m["xq"], 20)
    D2, I2 = fresh.search(m["xq"], 20)
    _assert_bits(D1, D2)
    assert np.array_equal(I1, I2)
    assert not np.isin(I1, ids[~keep]).any()  # no removed id comes back


def rng_pick(n, k):
    return np.random.default_rng(7).choice(n, k, replace=False)


def test_search_at_kc_equal_k_returns_the_twin_ids(vi, res, small_model, pq2):
    m = small_model
    idx, twin = _refine(vi, res, m, pq2, m["xb"], k_factor=1.0), _build(vi, res, m, m["xb"])
    _setup(idx, twin)
    for k in (1, 10, 100):
        D, I = idx.search(m["xq"], k)
        Dt, It = twin.search(m["xq"], k)
        for r in range(len(I)):
            assert set(I[r].tolist()) == set(It[r].tolist())
        assert (np.diff(D, axis=1) >= 0).all()


def test_search_matches_refinement_of_twin_candidates(vi, res, small_model, pq2):
    """the refined result is the k best of the twin's kc candidates by ||q - x2||^2, filtered or not"""
    m = small_model
    xq = m["xq"]
    idx, twin = _refine(vi, res, m, pq2, m["xb"]), _build(vi, res, m, m["xb"])
    _setup(idx, twin)
    R = idx.reconstruct_n(0, idx.ntotal).astype(np.float64)
    qn = (xq.astype(np.float64) ** 2).sum(-1)
    for k, kf, sel in [(10, 4.0, None), (5, 2.5, None), (100, 8.0, None), (10, 4.0, vi.IDSelectorRange(0, 6000)),
                       (10, 4.0, np.arange(0, 20000, 3))]:
        idx.k_factor = kf
        kc = _kc(k, kf)
        D, I = idx.search(xq, k, sel=sel)
        _, Ic = twin.search(xq, kc, sel=sel)
        if sel is not None:
            member = vi.selector_is_member(sel, np.arange(20000))
            assert member[I[I >= 0]].all()
        for r in range(len(xq)):
            c = Ic[r][Ic[r] >= 0]
            dc = ((xq[r].astype(np.float64) - R[c]) ** 2).sum(-1)
            want = np.sort(dc)[:k]
            got = I[r][I[r] >= 0]
            assert len(got) == len(want) and np.isin(got, c).all()
            dg = ((xq[r].astype(np.float64) - R[got]) ** 2).sum(-1)
            assert (np.abs(D[r][:len(got)] - dg) <= REL_DIST * (dg + qn[r])).all()
            assert (np.abs(dg - want) <= REL_DIST * (want + qn[r])).all()


def test_search_and_reconstruct_host_device_and_empty(vi, res, cuda, small_model, pq2):
    import torch

    m = small_model
    xq = m["xq"]
    idx = _refine(vi, res, m, pq2, m["xb"])
    _setup(idx)
    D, I = idx.search(xq, 10)
    D2, I2, R2 = idx.search_and_reconstruct(xq, 10)
    _assert_bits(D2, D)
    assert np.array_equal(I2, I)
    _assert_bits(R2.reshape(-1, m["d"]), idx.reconstruct_batch(I.reshape(-1)))
    dq = ((xq.astype(np.float64)[:, None] - R2.astype(np.float64)) ** 2).sum(-1)
    assert (np.abs(dq - D) <= REL_DIST * (dq + (xq.astype(np.float64) ** 2).sum(-1)[:, None])).all()
    Dd, Id = idx.search(torch.from_numpy(xq).to(cuda), 10)
    _assert_bits(N(Dd), D)
    assert np.array_equal(N(Id), I)
    Dd, Id, Rd = idx.search_and_reconstruct(torch.from_numpy(xq).to(cuda), 10, sel=vi.IDSelectorRange(0, 20000))
    _assert_bits(N(Rd), R2)
    E, J = idx.search(xq[:0], 10)
    assert E.shape == (0, 10) and J.shape == (0, 10)


def test_calls_without_refinement_throw(vi, res, small_model, pq2, tmp_path):
    m = small_model
    idx = _refine(vi, res, m, pq2, m["xb"][:2000])
    with pytest.raises(vi.FaissException):
        idx.range_search(m["xq"], 1e5)
    with pytest.raises(vi.FaissException):
        idx.range_search(m["xq"], 1e5, sel=vi.IDSelectorRange(0, 10))
    with pytest.raises(vi.FaissException):
        idx.writeDbToFile(str(tmp_path / "db"))
    twin = _build(vi, res, m, m["xb"][:2000])
    twin.writeCodebookToFile(str(tmp_path / "cb"))
    twin.writeDbToFile(str(tmp_path / "db"))
    with pytest.raises(vi.FaissException):
        idx.readDbFromFile(str(tmp_path / "db"))
    cpu = vi.CpuIndexIVFPQ(m["d"], m["C"], m["M"])
    with pytest.raises(vi.FaissException):
        idx.copyTo(cpu)
    with pytest.raises(vi.FaissException):
        idx.copyFrom(cpu)
    with pytest.raises(vi.FaissException):
        idx.k_factor = 0.5
    assert idx.ntotal == 2000  # nothing above changed the index


def test_proxy_and_shards(vi, res, small_model, pq2):
    import torch

    m = small_model
    single = _refine(vi, res, m, pq2, m["xb"])
    rep = _refine(vi, res, m, pq2, m["xb"])
    _setup(single, rep)
    D0, I0 = single.search(m["xq"], 10)
    proxy = vi.IndexProxy()
    proxy.addIndex(single)
    proxy.addIndex(rep)
    D1, I1 = proxy.search(m["xq"], 10)
    _assert_bits(D1, D0)
    assert np.array_equal(I1, I0)
    if torch.cuda.device_count() < 2:
        pytest.skip("IndexShards over two GPUs needs two GPUs")
    r1 = vi.StandardGpuResources(1)
    subs = [_refine(vi, res, m, pq2, m["xb"][:9000]), _refine(vi, r1, m, pq2, m["xb"][9000:])]
    _setup(*subs)
    shards = vi.IndexShards(m["d"], threaded=True, successive_ids=True)
    for s in subs:
        shards.add_shard(s)
    D2, I2 = shards.search(m["xq"], 10)
    Da, Ia = subs[0].search(m["xq"], 10)
    Db, Ib = subs[1].search(m["xq"], 10)
    Dm = np.concatenate([Da, Db], 1)
    Im = np.concatenate([Ia, np.where(Ib >= 0, Ib + 9000, -1)], 1)
    o = np.argsort(Dm, 1, kind="stable")[:, :10]
    _assert_bits(D2, np.take_along_axis(Dm, o, 1))
    assert (I2 == np.take_along_axis(Im, o, 1)).mean() > 0.999  # up to the order of equal distances


def test_recall_at_1_above_twin(vi, res, small_model, pq2):
    m = small_model
    xb, xq = m["xb"], m["xq"]
    idx, twin = _refine(vi, res, m, pq2, xb, k_factor=8.0), _build(vi, res, m, xb)
    _setup(idx, twin)
    gt = ((xq.astype(np.float64)[:, None] - xb.astype(np.float64)[None]) ** 2).sum(-1).argmin(1)
    _, I = idx.search(xq, 1)
    _, It = twin.search(xq, 1)
    assert (I[:, 0] == gt).mean() > (It[:, 0] == gt).mean()
