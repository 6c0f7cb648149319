"""Decode of stored entries: vlq_lookup_ids / vlq_decode_entries / vlq_imi_decode_entries against torch and numpy
restatements (bit for bit), the scan's slab-index output, and reconstruct / reconstruct_n / reconstruct_batch /
search_and_reconstruct of GpuIndexIVFPQ and GpuIndexIMIPQ (distance identities, bit-identity with search, mutations)."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_shapes import IMI_ROWS, MISALIGNED_ROWS, ROWS, _misaligned, _row, _variant, scan_calls

pytestmark = pytest.mark.gpu

NAN_BITS = np.uint32(0xFFFFFFFF)
REL = 1e-4  # the project's distance bar: |got - want| <= REL (|want| + ||q||^2)


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
def _slab(torch, ops, nlists, mean, M, dev, seed):
    """list-major slab in the stored layout: empty lists, lists longer than 2048, ids in no order, some ids repeated"""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lens = torch.poisson(torch.distributions.Gamma(2.0, 2.0).sample((nlists,)) * mean, generator=g).to(torch.int64)
    lens[::97] = 0
    lens[5::211] = 2500 + torch.randint(0, 1000, (lens[5::211].numel(),), generator=g)
    off = torch.zeros(nlists + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(lens, 0)
    n = int(off[-1])
    codes = torch.randint(0, 256, (n, M), dtype=torch.uint8, generator=g)
    lamq = torch.randint(0, 256, (n,), dtype=torch.uint8, generator=g)
    ids = torch.randperm(2 * n, generator=g)[:n].to(torch.int64) * 3 + 7
    rep = torch.randperm(n, generator=g)[: n // 50]
    ids[rep] = ids[torch.randperm(n, generator=g)[: n // 50]]  # ids stored twice (add_with_ids allows it)
    off, codes = off.to(dev), codes.to(dev)
    return ops.Lists(off, ops.rotate_codes(off, codes), lamq.to(dev), torch.zeros(n, device=dev), ids.to(dev))


def _lookup_ref(torch, ids, keys):
    """lowest slab index holding each key, -1 if none"""
    srt, perm = torch.sort(ids, stable=True)  # equal ids keep slab order: the first of a run is the lowest index
    at = torch.searchsorted(srt, keys).clamp(max=max(ids.numel() - 1, 0))
    hit = srt[at] == keys
    return torch.where(hit, perm[at], torch.full_like(keys, -1))


def _list_and_pv(off, stored, p, pq):
    """list of each slab index and its PQ vector p(code); stored bytes un-rotated: code[m] = stored[(m - pos) mod M]"""
    M = pq.shape[0]
    lst = np.searchsorted(off, p, side="right") - 1
    rot = (p - off[lst]) % M
    code = stored[p[:, None], (np.arange(M)[None, :] - rot[:, None]) % M]
    return lst, pq[np.arange(M)[None, :], code].reshape(len(p), -1)


def _np_decode(off, stored, pos, pq, lamq=None, cent=None, edge=None, lcb=None, cb=None, nbits=None):
    """x = anchor + p(code) in numpy float32, each operation rounded as written; pos -1 -> NaN bits.  Also returns the
    float64 evaluation and the per-component scale |c| + |s| + |p|."""
    ok = pos >= 0
    p = np.where(ok, pos, 0)
    lst, pv = _list_and_pv(off, stored, p, pq)
    if cb is None:
        lh = lcb[lamq[p]]
        c, s = cent[lst // edge.shape[1]], cent[edge.reshape(-1)[lst]]
        x = ((np.float32(1) - lh)[:, None] * c + lh[:, None] * s) + pv
        lh64 = lh.astype(np.float64)[:, None]
        x64 = (1 - lh64) * c + lh64 * s + pv.astype(np.float64)
        scale = np.abs(c) + np.abs(s) + np.abs(pv)
    else:
        K = 1 << nbits
        anchor = np.concatenate([cb[0][lst & (K - 1)], cb[1][lst >> nbits]], axis=1)
        x = anchor + pv
        x64 = anchor.astype(np.float64) + pv
        scale = np.abs(anchor) + np.abs(pv)
    x.view(np.uint32)[~ok] = NAN_BITS
    return x, x64, scale, ok


def _assert_bits(got, want):
    assert got.shape == want.shape
    g, w = got.view(np.uint32), want.view(np.uint32)
    bad = np.flatnonzero((g != w).any(axis=-1) if g.ndim > 1 else g != w)
    assert bad.size == 0, (bad[:5], got[bad[:2]], want[bad[:2]])


def _anchors(rng, d, M, C, E, nL=256):
    cent = (rng.standard_normal((C, d)) * 40).astype(np.float32)
    edge = np.stack([rng.choice(np.setdiff1d(np.arange(C), [c]), E, replace=False) for c in range(C)]).astype(np.int32)
    lcb = np.sort(rng.uniform(-0.3, 1.3, nL)).astype(np.float32)
    pq = (rng.standard_normal((M, 256, d // M)) * 5).astype(np.float32)
    return cent, edge, lcb, pq


# ------------------------------------------------------------------------------------------------ 1. ops level
@pytest.mark.parametrize("M", [16, 8, 32])
def test_lookup_ids_matches_torch(ops, cuda, M):
    import torch

    lists = _slab(torch, ops, 3000, 200.0, M, cuda, seed=M)
    n = lists.ids.numel()
    lens = N(lists.offsets[1:] - lists.offsets[:-1])
    assert (lens == 0).any() and (lens > 2048).any()
    ids = lists.ids
    assert torch.unique(ids).numel() < n  # repeated ids are present
    g = torch.Generator(device="cpu").manual_seed(M + 5)
    pick = ids.cpu()[torch.randperm(n, generator=g)[:20000]]
    absent = torch.tensor([0, 1, 5, 8, 3 * 2 * n + 100], dtype=torch.int64)  # stored ids are 1 mod 3 and >= 7
    keys = torch.unique(torch.cat([pick, absent])).to(cuda)
    pos, found = ops.lookup_ids(lists, keys=keys)
    want = _lookup_ref(torch, ids, keys)
    assert torch.equal(pos, want)
    assert found == int((want >= 0).sum()) == keys.numel() - absent.numel()
    lo = int(ids.min()) + 1000
    pos, found = ops.lookup_ids(lists, id_range=(lo, lo + 300000))
    rk = torch.arange(lo, lo + 300000, dtype=torch.int64, device=cuda)
    want = _lookup_ref(torch, ids, rk)
    assert torch.equal(pos, want) and found == int((want >= 0).sum()) > 0
    for keys in (torch.zeros(0, dtype=torch.int64, device=cuda),):  # no slots: found = 0, nothing launched
        assert ops.lookup_ids(lists, keys=keys)[1] == 0


@pytest.mark.parametrize("M", [16, 8, 32])
@pytest.mark.parametrize("misaligned", [False, True])
def test_decode_entries_matches_numpy(ops, cuda, M, misaligned):
    import torch

    d, C, E = 128 if M != 32 else 96, 64, 8
    rng = np.random.RandomState(M)
    lists = _slab(torch, ops, C * E, 60.0, M, cuda, seed=100 + M)
    if misaligned:
        lists = _misaligned(ops, lists, cuda)
    cent, edge, lcb, pq = _anchors(rng, d, M, C, E)
    n = lists.ids.numel()
    pos = np.concatenate([rng.randint(0, n, 50000), [-1, 0, n - 1, -1]]).astype(np.int64)
    x, oid = ops.decode_entries(lists, T(pos, cuda), T(pq, cuda), cent=T(cent, cuda), edge=T(edge, cuda),
                                lambda_cb=T(lcb, cuda), want_ids=True)
    want, _, _, ok = _np_decode(N(lists.offsets), N(lists.codes), pos, pq, lamq=N(lists.lamq), cent=cent, edge=edge,
                                lcb=lcb)
    _assert_bits(N(x), want)
    assert np.array_equal(N(oid), np.where(ok, N(lists.ids)[np.maximum(pos, 0)], -1))
    # lambda codebook {0} (a copyFrom index): exactly c + p
    z = np.zeros(1, np.float32)
    x0 = ops.decode_entries(ops.Lists(lists.offsets, lists.codes, torch.zeros_like(lists.lamq), lists.kappa, lists.ids),
                            T(pos, cuda), T(pq, cuda), cent=T(cent, cuda), edge=T(edge, cuda), lambda_cb=T(z, cuda))
    want0, _, _, _ = _np_decode(N(lists.offsets), N(lists.codes), pos, pq, lamq=np.zeros(n, np.uint8), cent=cent,
                                edge=edge, lcb=z)
    lst, pv = _list_and_pv(N(lists.offsets), N(lists.codes), np.maximum(pos, 0), pq)
    c_plus_p = cent[lst // E] + pv
    _assert_bits(N(x0)[ok], want0[ok])
    _assert_bits(want0[ok], c_plus_p[ok])
    # out_ids aliasing pos: the scan's slab indexes turned into labels in place
    p2 = T(pos, cuda)
    dq, dc, de, dl = T(pq, cuda), T(cent, cuda), T(edge, cuda), T(lcb, cuda)  # held until the kernel has run
    xo = torch.empty((len(pos), d), device=cuda)
    ops._abi.call("vlq_decode_entries", len(pos), p2.data_ptr(), C * E, lists.offsets.data_ptr(),
                  lists.codes.data_ptr(), lists.lamq.data_ptr(), lists.ids.data_ptr(), M, d, dq.data_ptr(),
                  dc.data_ptr(), de.data_ptr(), E, dl.data_ptr(), 256, xo.data_ptr(), p2.data_ptr(), ops._stream())
    assert torch.equal(p2, oid) and torch.equal(xo.view(torch.int32), x.view(torch.int32))  # NaN rows: compare bits


# ------------------------------------------------------------------------------------------------ 2. every shape
@pytest.mark.parametrize("name", list(ROWS))
def test_decode_every_shape(ops, cuda, oracle, name):
    """the trained model and lists of every shape row (VLQ anchors), and a synthetic IMI slab of the same d / M"""
    import torch

    r = _row(name, ops, cuda, oracle)
    lists, M, d = r["lists"], r["M"], r["d"]
    n = lists.ids.numel()
    rng = np.random.RandomState(7)
    pos = np.concatenate([rng.randint(0, n, 4000), [-1]]).astype(np.int64)
    m = r["m"]
    variants = [lists] + ([_misaligned(ops, lists, cuda)] if name in MISALIGNED_ROWS else [])
    for lv in variants:
        x = N(ops.decode_entries(lv, T(pos, cuda), r["pq"], cent=r["cent"], edge=r["edge"], lambda_cb=r["lcb"]))
        want, x64, scale, ok = _np_decode(r["off"], N(lists.codes), pos, m["pq"], lamq=r["lamq"], cent=m["cent"],
                                          edge=m["edge"], lcb=m["lambda_cb"])
        _assert_bits(x, want)
        assert (np.abs(x[ok] - x64[ok]) <= 1e-6 * scale[ok] + 1e-30).all()
    # IMI anchors: cells i1 | i2 << nbits over two half codebooks
    nbits = 4
    imi = _slab(torch, ops, 1 << (2 * nbits), 40.0, M, cuda, seed=len(name) * 31 + d)
    cb = [(rng.standard_normal((1 << nbits, d // 2)) * 30).astype(np.float32) for _ in range(2)]
    n = imi.ids.numel()
    pos = np.concatenate([rng.randint(0, n, 4000), [-1]]).astype(np.int64)
    x = N(ops.decode_entries(imi, T(pos, cuda), r["pq"], cb=(T(cb[0], cuda), T(cb[1], cuda)), nbits=nbits))
    want, x64, scale, ok = _np_decode(N(imi.offsets), N(imi.codes), pos, m["pq"], cb=cb, nbits=nbits)
    _assert_bits(x, want)
    assert (np.abs(x[ok] - x64[ok]) <= 1e-6 * scale[ok] + 1e-30).all()


# ------------------------------------------------------------------------------------------------ 3. slab-index scan
def _scan_slab_index(ops, cuda, oracle, name, variant):
    r = _row(name, ops, cuda, oracle)
    lists, lcb, lines, ed2, _, _ = _variant(ops, cuda, r, variant)
    ed2f = None if ed2 is None else ed2.reshape(-1)
    calls = scan_calls(name, variant)  # every scan kernel the dispatcher chooses (test_gpu_shapes checks which ran)

    def run(slab):
        return [ops.scan_topk(r["q"], r["pq"], lcb, lines[0], lines[1], lines[2], ed2f, lists, k, cap,
                              use_workspace=ws, list_len_hint=h, slab_index=slab) for h, k, cap, ws in calls]

    normal = run(False)
    slab = run(True)
    lid = r["lid"]
    for (D, I), (Ds, Is) in zip(normal, slab):
        assert np.array_equal(N(D).view(np.uint32), N(Ds).view(np.uint32))
        Is = N(Is)
        assert np.array_equal(np.where(Is >= 0, lid[np.maximum(Is, 0)], -1), N(I))


@pytest.mark.parametrize("name", list(ROWS))
def test_scan_slab_index_mode(ops, cuda, oracle, name):
    _scan_slab_index(ops, cuda, oracle, name, "vlq")


@pytest.mark.parametrize("name", MISALIGNED_ROWS)
def test_scan_slab_index_misaligned(ops, cuda, oracle, name):
    _scan_slab_index(ops, cuda, oracle, name, "misaligned")


@pytest.mark.parametrize("name", IMI_ROWS)
def test_scan_slab_index_imi(ops, cuda, oracle, name):
    _scan_slab_index(ops, cuda, oracle, name, "imi")


# ------------------------------------------------------------------------------------------------ 4. index level
def _build(vi, res, m, xb, ids=None, chunks=2):
    idx = vi.GpuIndexIVFPQ(res, m["d"], m["C"], m["M"], 8, m["E"], 256)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    step = (len(xb) + chunks - 1) // chunks
    for s in range(0, len(xb), step):
        if ids is None:
            idx.add(xb[s:s + step])
        else:
            idx.add_with_ids(xb[s:s + step], ids[s:s + step])
    return idx


def _slab_of(idx, m, tmp_path):
    """(offsets, canonical codes, lamq, ids) of the committed slab, read through the database files"""
    name = str(tmp_path / "db")
    idx.writeDbToFile(name)
    L = m["C"] * m["E"]
    counts = np.fromfile(name + ".dbcount", np.int32, L)
    off = np.zeros(L + 1, np.int64)
    off[1:] = np.cumsum(counts)
    codes = np.fromfile(name + ".dbcodes", np.uint8).reshape(-1, m["M"])
    return off, codes, np.fromfile(name + ".dblas", np.uint8), np.fromfile(name + ".dbIdx", np.int64)


def _restate(m, off, codes, lamq):
    """decode of every slab entry from the canonical codes of the database files"""
    M = m["M"]
    n = len(lamq)
    lst = np.searchsorted(off, np.arange(n), side="right") - 1
    pv = m["pq"][np.arange(M)[None, :], codes].reshape(n, -1)
    lh = m["lambda_cb"][lamq]
    c, s = m["cent"][lst // m["E"]], m["cent"][m["edge"].reshape(-1)[lst]]
    return ((np.float32(1) - lh)[:, None] * c + lh[:, None] * s) + pv, c, s, lh


def _identity(xq, R, D):
    """float64 ||q - x||^2 - ||q||^2 of decoded rows against the VLQ distances D (which exclude ||q||^2)"""
    q = xq.astype(np.float64)[:, None, :]
    qn = (q ** 2).sum(-1)
    got = ((q - R.astype(np.float64)) ** 2).sum(-1) - qn
    return np.abs(got - D) <= REL * (np.abs(D) + qn)


def test_reconstruct_n_matches_restatement_and_distances(vi, res, oracle, small_model, tmp_path):
    m = small_model
    xb, xq = m["xb"], m["xq"]
    idx = _build(vi, res, m, xb)  # the second add is still pending at the first read-back
    R = idx.reconstruct_n(0, idx.ntotal)
    off, codes, lamq, ids = _slab_of(idx, m, tmp_path)
    ref, c, s, lh = _restate(m, off, codes, lamq)
    want = np.empty_like(ref)
    want[ids] = ref
    _assert_bits(R, want)
    # every entry: the decode identity of the oracle for one query, in float64
    q = xq[0]
    got = ((q.astype(np.float64) - R[ids].astype(np.float64)) ** 2).sum(1) - (q.astype(np.float64) ** 2).sum()
    ora = np.array([oracle.decode_distance(q, c[i], s[i], float(lh[i]), m["pq"], codes[i]) for i in range(len(ids))])
    assert (np.abs(got - ora) <= REL * (np.abs(ora) + (q.astype(np.float64) ** 2).sum())).all()
    # and the distance search returns for every result
    idx.setNumProbes(16)
    idx.w1_ = 64
    D, I = idx.search(xq, 50)
    ok = I >= 0
    assert ok.mean() > 0.9
    assert _identity(xq, R[np.maximum(I, 0)], D.astype(np.float64))[ok].all()
    # reconstruct / reconstruct_batch agree with reconstruct_n
    _assert_bits(idx.reconstruct(int(ids[5]))[None], R[ids[5]][None])
    keys = np.array([ids[9], ids[3], ids[9], ids[0]], np.int64)
    _assert_bits(idx.reconstruct_batch(keys), R[keys])


@pytest.mark.parametrize("route", [None, "VLQ_COARSE_EXACT", "VLQ_COARSE_MATRIX"])
def test_search_and_reconstruct_bit_identical_to_search(vi, res, cuda, small_model, monkeypatch, route):
    import torch

    m = small_model
    if route:
        monkeypatch.setenv(route, "1")
    idx = _build(vi, res, m, m["xb"])
    idx.setNumProbes(8)
    idx.w1_ = 32
    rng = np.random.RandomState(5)
    xq = m["xq"][rng.randint(0, len(m["xq"]), 6000)] + rng.randint(-3, 4, (6000, m["d"])).astype(np.float32)
    k = 20
    D, I = idx.search(xq, k)  # 6000 queries: two query tiles
    D2, I2, R = idx.search_and_reconstruct(xq, k)
    assert np.array_equal(D.view(np.uint32), D2.view(np.uint32)) and np.array_equal(I, I2)
    ok = I >= 0
    assert ok.mean() > 0.95
    assert _identity(xq, R, D.astype(np.float64))[ok].all()
    _assert_bits(R[ok], idx.reconstruct_batch(I[ok]))  # ids are unique here
    assert (R[~ok].view(np.uint32) == NAN_BITS).all()
    # device buffers, and host output in many small pages
    qd = T(xq, cuda)
    Dd, Id, Rd = idx.search_and_reconstruct(qd, k)
    assert isinstance(Rd, torch.Tensor) and Rd.is_cuda
    assert np.array_equal(N(Dd).view(np.uint32), D.view(np.uint32)) and np.array_equal(N(Id), I)
    _assert_bits(N(Rd).reshape(-1, m["d"]), R.reshape(-1, m["d"]))
    monkeypatch.setenv("VLQ_RECONSTRUCT_STAGING_BYTES", str(37 * m["d"] * 4))
    _, _, Rp = idx.search_and_reconstruct(xq, k)
    _assert_bits(Rp.reshape(-1, m["d"]), R.reshape(-1, m["d"]))
    Rn = idx.reconstruct_n(0, idx.ntotal)
    monkeypatch.delenv("VLQ_RECONSTRUCT_STAGING_BYTES")
    _assert_bits(Rn, idx.reconstruct_n(0, idx.ntotal))
    out = torch.empty((idx.ntotal, m["d"]), dtype=torch.float32, device=cuda)
    idx.reconstruct_n(0, idx.ntotal, out=out)
    _assert_bits(N(out), Rn)
    _assert_bits(N(idx.reconstruct_batch(T(I[ok][:500], cuda))), R[ok][:500])


# ------------------------------------------------------------------------------------------------ 5. mutations, edges
def test_reconstruct_after_remove_add_and_edge_cases(vi, res, small_model):
    m = small_model
    xb = m["xb"]
    idx = _build(vi, res, m, xb[:12000])
    before = idx.reconstruct_n(0, 12000)
    assert idx.remove_ids(vi.IDSelectorRange(3000, 5000)) == 2000
    with pytest.raises(vi.FaissException, match="key 3000 has no entry"):
        idx.reconstruct(3000)
    with pytest.raises(vi.FaissException, match="key 4999 has no entry"):
        idx.reconstruct_batch(np.array([10, 4999, 20], np.int64))
    keep = np.r_[0:3000, 5000:12000]
    _assert_bits(idx.reconstruct_batch(keep), before[keep])  # survivors moved and were re-rotated: same vectors
    idx.add(xb[12000:15000])  # ids 10000 .. 12999 (ntotal-based), after the removal
    fresh = _build(vi, res, m, xb[12000:15000], ids=np.arange(10000, 13000, dtype=np.int64), chunks=1)
    _assert_bits(idx.reconstruct_batch(np.arange(12000, 13000)), fresh.reconstruct_batch(np.arange(12000, 13000)))
    # missing / out-of-range keys throw and leave the output as it was
    h = vi.host()
    out = np.full((3, m["d"]), 5.0, np.float32)
    keys = np.array([1, 10 ** 12, 2], np.int64)
    assert h.vlq_host_index_reconstruct_batch(idx.h, C.c_long(3), C.c_void_p(keys.ctypes.data),
                                              C.c_void_p(out.ctypes.data)) == -1
    assert b"key 1000000000000 has no entry" in h.vlq_host_last_error()
    assert (out == 5.0).all()
    assert h.vlq_host_index_reconstruct_n(idx.h, C.c_long(12990), C.c_long(20), C.c_void_p(out.ctypes.data)) == -1
    assert (out == 5.0).all()
    with pytest.raises(vi.FaissException):
        idx.reconstruct(-1)
    with pytest.raises(vi.FaissException):
        idx.reconstruct_n(-1, 2)
    # n == 0 is a no-op
    assert idx.reconstruct_batch(np.zeros(0, np.int64)).shape == (0, m["d"])
    assert idx.reconstruct_n(0, 0).shape == (0, m["d"])
    D, I, R = idx.search_and_reconstruct(np.zeros((0, m["d"]), np.float32), 5)
    assert D.shape == (0, 5) and R.shape == (0, 5, m["d"])
    # k beyond the reachable entries: NaN rows for the -1 labels
    idx.setNumProbes(1)
    idx.w1_ = 1
    D, I, R = idx.search_and_reconstruct(m["xq"][:8], 1024)
    assert (I < 0).any() and (I >= 0).any()
    assert (R[I < 0].view(np.uint32) == NAN_BITS).all()
    assert not np.isnan(R[I >= 0]).any()
    idx.reset()
    with pytest.raises(vi.FaissException, match="key 0 has no entry"):
        idx.reconstruct(0)


def test_duplicate_ids_lowest_slab_and_found_entry(vi, res, small_model, tmp_path):
    m = small_model
    xb = m["xb"][:6000]
    rng = np.random.RandomState(11)
    ids = np.arange(6000, dtype=np.int64)
    idx = _build(vi, res, m, xb, ids=ids, chunks=1)
    idx.add_with_ids(xb + rng.uniform(-12, 12, xb.shape).astype(np.float32), ids)  # the same ids, other vectors
    off, codes, lamq, sid = _slab_of(idx, m, tmp_path)
    ref = _restate(m, off, codes, lamq)[0]
    first = {}
    for p, i in enumerate(sid):
        first.setdefault(int(i), p)
    lowest = np.array([first[i] for i in range(6000)])
    _assert_bits(idx.reconstruct_n(0, 6000), ref[lowest])
    idx.setNumProbes(16)
    idx.w1_ = 64
    xq = xb[rng.randint(0, 6000, 200)]
    D, I, R = idx.search_and_reconstruct(xq, 10)
    ok = I >= 0
    assert _identity(xq, R, D.astype(np.float64))[ok].all()  # each row is the entry that was found
    other = ~np.all(R == ref[lowest][np.maximum(I, 0)], axis=-1) & ok
    assert other.sum() > 0  # found entries that are not the lowest-slab copy of their id
    assert not _identity(xq, ref[lowest][np.maximum(I, 0)], D.astype(np.float64))[other].all()


def test_copy_from_decodes_c_plus_p(vi, res):
    """a stock IVFPQ index (lambda codebook {0}) decodes to exactly c + p, the reference IndexIVFPQ's decode"""
    d, nlist, M = 64, 32, 8
    rng = np.random.RandomState(3)
    coarse = (rng.standard_normal((nlist, d)) * 20).astype(np.float32)
    pq = (rng.standard_normal((M, 256, d // M)) * 3).astype(np.float32)
    cpu = vi.CpuIndexIVFPQ(d, nlist, M)
    cpu.set_codebooks(coarse, pq)
    want = {}
    nid = 0
    for l in range(nlist):
        n = int(rng.randint(0, 80))
        codes = rng.randint(0, 256, (n, M)).astype(np.uint8)
        ids = np.arange(nid, nid + n, dtype=np.int64)
        nid += n
        cpu.set_list(l, ids, codes)
        for i, c in zip(ids, codes):
            want[int(i)] = coarse[l] + pq[np.arange(M), c].reshape(-1)
    g = vi.GpuIndexIVFPQ(res, d, nlist, M, 8, 4, 16)
    g.copyFrom(cpu)
    _assert_bits(g.reconstruct_n(0, nid), np.stack([want[i] for i in range(nid)]))


def test_imipq_read_back(vi, res, cuda):
    from vector_line_quantization_b200 import data

    xt = data.sift_like(20000, kc=64, seed=21)
    xb = data.sift_like(20000, kc=64, seed=22)
    xq = data.sift_like(300, kc=64, seed=23)
    idx = vi.GpuIndexIMIPQ(res, 128, 4, 16)
    idx.setTrainIters(4)
    idx.train(xt)
    ids = np.arange(len(xb), dtype=np.int64) * 7 + 3
    idx.add_with_ids(xb[:12000], ids[:12000])
    idx.add_with_ids(xb[12000:], ids[12000:])  # pending at the first read-back
    R = idx.reconstruct_batch(ids)
    err = ((R.astype(np.float64) - xb) ** 2).sum(1)
    assert np.median(err) < 0.2 * np.median((xb.astype(np.float64) ** 2).sum(1))  # a decode, not noise
    idx.setNumProbes(8)
    D, I = idx.search(xq, 30)
    D2, I2, Rs = idx.search_and_reconstruct(xq, 30)
    assert np.array_equal(D.view(np.uint32), D2.view(np.uint32)) and np.array_equal(I, I2)
    ok = I >= 0
    full = ((xq.astype(np.float64)[:, None, :] - Rs.astype(np.float64)) ** 2).sum(-1)  # IMI distances are full
    assert (np.abs(full - D) <= REL * (np.abs(D) + (xq.astype(np.float64) ** 2).sum(1)[:, None]))[ok].all()
    _assert_bits(Rs[ok], R[(I[ok] - 3) // 7])
    _, _, Rd = idx.search_and_reconstruct(T(xq, cuda), 30)
    _assert_bits(N(Rd).reshape(-1, 128), Rs.reshape(-1, 128))
    idx.remove_ids(ids[:100])
    with pytest.raises(vi.FaissException, match="key 3 has no entry"):
        idx.reconstruct(3)
    _assert_bits(idx.reconstruct_n(ids[100], 1), R[100:101])
