"""Filtered search: vlq_filter_kappa against a torch restatement (bit for bit), every scan variant and the range kernels
on the masked kappa against the unfiltered call, and search / range_search / search_and_reconstruct with a selector on
GpuIndexIVFPQ and GpuIndexIMIPQ (against search(), against an index holding only the selected vectors, and against
remove_ids of the complement)."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_shapes import IMI_ROWS, MISALIGNED_ROWS, RANGE_UNSUPPORTED, ROWS, WARP_SEL_MAX_K, _row, _variant, \
    scan_calls

pytestmark = pytest.mark.gpu

FMAX = np.finfo(np.float32).max
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


# ------------------------------------------------------------------------------------------------ 1. mask kernel
def _mask_ref(torch, ids, kappa, lo=0, hi=0, batch=None, bitmap=None, invert=False):
    m = (ids >= lo) & (ids < hi)
    if batch is not None and batch.numel():
        m |= torch.isin(ids, batch)
    if bitmap is not None and bitmap.numel():
        byte = ids >> 3
        inb = (ids >= 0) & (byte < bitmap.numel())
        b = bitmap[byte.clamp(0, bitmap.numel() - 1)].to(torch.int64)
        m |= inb & (((b >> (ids & 7)) & 1) == 1)
    if invert:
        m = ~m
    return torch.where(m, kappa, torch.full_like(kappa, float("inf")))


@pytest.mark.parametrize("n", [0, 1, 255, 257, 1023 * 4 + 5, 3_000_001])
def test_filter_kappa_matches_torch(ops, cuda, n):
    import torch

    g = torch.Generator(device="cpu").manual_seed(n)
    ids = (torch.randperm(max(3 * n, 1), generator=g)[:n] - n // 10).to(torch.int64)  # some negative ids
    kappa = torch.randn(n, generator=g) * 1e3
    kappa[::7] = -0.0
    lists = ops.Lists(None, None, None, kappa.to(cuda), ids.to(cuda))
    ids_d, kap_d = lists.ids, lists.kappa
    batch = ids[torch.randperm(n, generator=g)[: n // 3]] if n else torch.zeros(0, dtype=torch.int64)
    batch = torch.cat([batch, batch[:5], torch.tensor([-7, 10 ** 15])])  # duplicates, ids not stored
    nbytes = max(1, (2 * n) // 8)  # ids past the bitmap's end, and negative ids, are not in it
    bitmap = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, generator=g)
    lo, hi = n // 4, n // 2
    cases = [dict(id_range=(lo, hi)), dict(ids=batch), dict(bitmap=bitmap), dict(id_range=(5, 5)),
             dict(ids=batch, id_range=(lo, hi), bitmap=bitmap)]
    for kw in cases:
        for inv in (False, True):
            got = ops.filter_kappa(lists, invert=inv, **kw)
            ref_kw = dict(lo=kw.get("id_range", (0, 0))[0], hi=kw.get("id_range", (0, 0))[1],
                          batch=kw["ids"].to(cuda) if "ids" in kw else None,
                          bitmap=kw["bitmap"].to(cuda) if "bitmap" in kw else None)
            want = _mask_ref(torch, ids_d, kap_d, invert=inv, **ref_kw)
            assert torch.equal(got.view(torch.int32), want.view(torch.int32)), (kw.keys(), inv)
    if n:
        inf = ops.filter_kappa(lists, id_range=(0, 0))
        assert (N(inf).view(np.uint32) == 0x7F800000).all()  # the +inf bit pattern itself


def test_filter_results_pads_inf_rows(ops, cuda):
    import torch

    D = torch.tensor([[1.0, 2.0, float("inf"), float("inf")], [float("-inf"), 0.0, 3.0, FMAX]], device=cuda)
    I = torch.tensor([[4, 5, 6, 7], [8, 9, 10, -1]], dtype=torch.int64, device=cuda)
    ops.filter_results(D, I)
    assert N(I).tolist() == [[4, 5, -1, -1], [8, 9, 10, -1]]
    assert N(D)[0, 2:].tolist() == [FMAX, FMAX] and N(D)[1, 0] == -np.inf


# ------------------------------------------------------------------------------------------------ 2. scan variants
SELECTIVITY = ("all", "none", "half", "1%", "one")


def _members(lid, kind, rng):
    u = np.unique(lid)
    if kind == "all":
        return u
    if kind == "none":
        return np.zeros(0, np.int64)
    if kind == "one":
        return u[rng.randint(len(u)):][:1]
    frac = 0.5 if kind == "half" else 0.01
    return u[rng.rand(len(u)) < frac]


def _check_filtered_rows(Du, Iu, Df, If, member_of, k):
    """filtered (Df, If) [nq][k] against the unfiltered top-K (Du, Iu) of the same dispatch class: the first k members
    of each unfiltered row, or -- when the unfiltered row holds every candidate -- all its members then padding"""
    checked = 0
    for q in range(Du.shape[0]):
        keep = (Iu[q] >= 0) & member_of(Iu[q])
        md, mi = Du[q][keep], Iu[q][keep]
        if len(mi) >= k:
            wd, wi = md[:k], mi[:k]
        elif Iu[q, -1] < 0:  # fewer than K candidates: the unfiltered row is complete
            wd = np.r_[md, np.full(k - len(mi), FMAX, np.float32)]
            wi = np.r_[mi, np.full(k - len(mi), -1, np.int64)]
        else:
            continue
        assert np.array_equal(Df[q].view(np.uint32), wd.view(np.uint32)), q
        assert np.array_equal(If[q], wi), q
        checked += 1
    return checked


def _scan_filtered(ops, cuda, oracle, monkeypatch, name, variant):
    import torch

    r = _row(name, ops, cuda, oracle)
    lists, lcb, lines, ed2, _, _ = _variant(ops, cuda, r, variant)
    ed2f = None if ed2 is None else ed2.reshape(-1)
    lid = N(lists.ids)
    rng = np.random.RandomState(7)
    calls = scan_calls(name, variant)
    no_small = (False, True) if variant == "vlq" else (False,)
    total = 0
    for kind in SELECTIVITY:
        mem = _members(lid, kind, rng)
        kap = ops.filter_kappa(lists, ids=T(mem, cuda))
        member_of = lambda slab: np.isin(lid[np.maximum(slab, 0)], mem)  # noqa: E731
        for ns in no_small:
            if ns:
                monkeypatch.setenv("VLQ_SCAN_NO_SMALL", "1")
            for h, k, cap, ws in calls:
                K = WARP_SEL_MAX_K if k <= WARP_SEL_MAX_K else 1024  # the same scan kernel as k
                run = lambda kk, kp: ops.scan_topk(r["q"], r["pq"], lcb, lines[0], lines[1], lines[2], ed2f,  # noqa
                                                   lists, kk, cap, use_workspace=ws, list_len_hint=h, slab_index=True,
                                                   kappa=kp)
                Du, Iu = run(K, None)
                Df, If = ops.filter_results(*run(k, kap))
                total += _check_filtered_rows(N(Du), N(Iu), N(Df), N(If), member_of, k)
                if kind == "none":
                    assert (N(If) == -1).all() and (N(Df) == FMAX).all()
            monkeypatch.delenv("VLQ_SCAN_NO_SMALL", raising=False)
        torch.cuda.synchronize()
    assert total > 0


@pytest.mark.parametrize("name", list(ROWS))
def test_scan_variants_on_masked_kappa(ops, cuda, oracle, monkeypatch, name):
    _scan_filtered(ops, cuda, oracle, monkeypatch, name, "vlq")


@pytest.mark.parametrize("name", MISALIGNED_ROWS)
def test_scan_variants_on_masked_kappa_misaligned(ops, cuda, oracle, monkeypatch, name):
    _scan_filtered(ops, cuda, oracle, monkeypatch, name, "misaligned")


@pytest.mark.parametrize("name", IMI_ROWS)
def test_scan_variants_on_masked_kappa_imi(ops, cuda, oracle, monkeypatch, name):
    _scan_filtered(ops, cuda, oracle, monkeypatch, name, "imi")


# ------------------------------------------------------------------------------------------------ 3. range kernels
@pytest.mark.parametrize("name", [n for n in ROWS if n not in RANGE_UNSUPPORTED])
def test_range_kernels_on_masked_kappa(ops, cuda, oracle, name):
    r = _row(name, ops, cuda, oracle)
    lists = r["lists"]
    lid = N(lists.ids)
    rng = np.random.RandomState(3)
    qn = ops.row_norms(r["q"])
    for kind in ("all", "half", "1%", "none"):
        mem = _members(lid, kind, rng)
        kap = ops.filter_kappa(lists, ids=T(mem, cuda))
        for radius in (np.median(r["qn"]) * 0.05, float("inf")):
            for cap in (1024, 7):
                lu, Du, Iu = (N(t) for t in ops.range_scan_lines(r["q"], r["pq"], r["lcb"], r["lines"], r["ed2"], lists,
                                                                radius, cap=cap, row_add=qn))
                lf, Df, If = (N(t) for t in ops.range_scan_lines(r["q"], r["pq"], r["lcb"], r["lines"], r["ed2"],
                                                                lists, radius, cap=cap, row_add=qn, kappa=kap))
                keep = np.isin(Iu, mem)
                want_l = np.r_[0, np.cumsum([keep[lu[i]:lu[i + 1]].sum() for i in range(len(lu) - 1)])]
                assert np.array_equal(lf, want_l)
                assert np.array_equal(If, Iu[keep])
                assert np.array_equal(Df.view(np.uint32), Du[keep].view(np.uint32))


# ------------------------------------------------------------------------------------------------ 4. index level
def _build(vi, res, m, xb, ids, chunks=2):
    idx = vi.GpuIndexIVFPQ(res, m["d"], m["C"], m["M"], 8, m["E"], 256)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    step = (len(xb) + chunks - 1) // chunks
    for s in range(0, len(xb), step):
        idx.add_with_ids(xb[s:s + step], ids[s:s + step])
    idx.setNumProbes(8)
    idx.w1_ = 48
    return idx


def _queries(m, n, seed=5):
    rng = np.random.RandomState(seed)
    return m["xq"][rng.randint(0, len(m["xq"]), n)] + rng.randint(-3, 4, (n, m["d"])).astype(np.float32)


def _same_up_to_ties(D1, I1, D2, I2, qn):
    """two top-k results over the same candidates, possibly from different scan kernels: same padding, distances within
    the distance bar at every rank, ids that differ only where the distances tie within it"""
    assert np.array_equal(I1 < 0, I2 < 0)
    scale = np.abs(D2.astype(np.float64)) + qn[:, None]
    assert (np.abs(D1.astype(np.float64) - D2) <= REL * scale).all()
    assert (I1 == I2).mean() > 0.99


def _bits(a, b):
    assert np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def _selectors(vi, ids, rng):
    """(name, selector, membership of `ids`) for batch, range, bitmap and Not"""
    sub = ids[rng.rand(len(ids)) < 0.3]
    lo, hi = int(np.percentile(ids, 20)), int(np.percentile(ids, 65))
    nbits = int(ids.max()) + 1
    bits = rng.rand(nbits) < 0.4
    bm = np.packbits(bits, bitorder="little")
    return [("batch", sub, np.isin(ids, sub)),
            ("range", vi.IDSelectorRange(lo, hi), (ids >= lo) & (ids < hi)),
            ("bitmap", vi.IDSelectorBitmap(bm), bits[ids]),
            ("not-batch", vi.IDSelectorNot(sub), ~np.isin(ids, sub))]


@pytest.mark.parametrize("route", [None, "VLQ_COARSE_EXACT", "VLQ_COARSE_MATRIX"])
def test_ivfpq_filtered_search(vi, res, cuda, small_model, monkeypatch, route):
    import torch

    m = small_model
    if route:
        monkeypatch.setenv(route, "1")
    xb = m["xb"]
    rng = np.random.RandomState(1)
    ids = rng.permutation(3 * len(xb))[: len(xb)].astype(np.int64)  # ids in no order
    idx = _build(vi, res, m, xb, ids)  # the second add is still pending at the first filtered search
    xq = _queries(m, 6000)  # two query tiles
    qn = (xq.astype(np.float64) ** 2).sum(1)
    k = 20
    D, I = idx.search(xq, k)
    # every id: search() bit for bit; no id: padding only, no range results, NaN rows
    Da, Ia = idx.search(xq, k, sel=vi.IDSelectorRange(-1, 1 << 40))
    _bits(Da, D)
    assert np.array_equal(Ia, I)
    Dn, In = idx.search(xq, k, sel=np.zeros(0, np.int64))
    assert (In == -1).all() and (Dn == FMAX).all()
    lims, Dr, Ir = idx.range_search(xq[:50], float("inf"), sel=vi.IDSelectorNot(vi.IDSelectorRange(-1, 1 << 40)))
    assert (lims == 0).all() and len(Ir) == 0
    _, In2, Rn = idx.search_and_reconstruct(xq[:40], 5, sel=vi.IDSelectorRange(0, 0))
    assert (In2 == -1).all() and (Rn.view(np.uint32) == NAN_BITS).all()
    for name, sel, member in _selectors(vi, ids, np.random.RandomState(2)):
        Df, If = idx.search(xq, k, sel=sel)
        assert np.isin(If[If >= 0], ids[member]).all(), name
        # an index that holds only the selected vectors, added in the same order with the same ids
        sub = _build(vi, res, m, xb[member], ids[member])
        Ds, Is = sub.search(xq, k)
        _same_up_to_ties(Df, If, Ds, Is, qn)
        # the complement removed instead
        rem = _build(vi, res, m, xb, ids)
        rem.remove_ids(ids[~member])
        Dm, Im = rem.search(xq, k)
        _same_up_to_ties(Df, If, Dm, Im, qn)
        # search_and_reconstruct: filtered search's D and I, and the decode of every result
        D3, I3, R3 = idx.search_and_reconstruct(xq, k, sel=sel)
        _bits(D3, Df)
        assert np.array_equal(I3, If)
        ok = I3 >= 0
        _bits(R3[ok], idx.reconstruct_batch(I3[ok]))
        assert (R3[~ok].view(np.uint32) == NAN_BITS).all()
        # range_search: the unfiltered result without the non-members, same bits and order
        radius = float(np.median(D[:, k // 2] + qn))
        lu, Du, Iu = idx.range_search(xq[:500], radius)
        lf, Dg, Ig = idx.range_search(xq[:500], radius, sel=sel)
        keep = np.isin(Iu, ids[member])
        assert np.array_equal(lf, np.r_[0, np.cumsum([keep[lu[i]:lu[i + 1]].sum() for i in range(500)])])
        assert np.array_equal(Ig, Iu[keep])
        _bits(Dg, Du[keep])
    # device queries, device outputs, device id array and device bitmap
    qd = T(xq, cuda)
    sel_ids = ids[::3]
    Dh, Ih = idx.search(xq, k, sel=sel_ids)
    Dd, Id = idx.search(qd, k, sel=T(sel_ids, cuda))
    assert isinstance(Dd, torch.Tensor) and Dd.is_cuda
    _bits(N(Dd), Dh)
    assert np.array_equal(N(Id), Ih)
    bm = np.packbits(np.isin(np.arange(3 * len(xb)), sel_ids), bitorder="little")
    Db, Ib = idx.search(qd, k, sel=vi.IDSelectorBitmap(T(bm, cuda)))
    _bits(N(Db), Dh)
    assert np.array_equal(N(Ib), Ih)
    _, _, Rd = idx.search_and_reconstruct(qd, k, sel=vi.IDSelectorBitmap(T(bm, cuda)))
    _, _, Rh = idx.search_and_reconstruct(xq, k, sel=sel_ids)
    _bits(N(Rd).reshape(-1), Rh.reshape(-1))


def test_ivfpq_filtered_pages_duplicates_and_errors(vi, res, small_model):
    m = small_model
    xb = m["xb"][:8000]
    ids = np.arange(8000, dtype=np.int64)
    idx = _build(vi, res, m, xb, ids, chunks=1)
    idx.add_with_ids(xb[:2000] + 4.0, ids[:2000])  # ids 0 .. 1999 stored twice
    xq = _queries(m, 33000, seed=9)  # two pages of 32768 queries
    k = 10
    sel = np.arange(0, 8000, 2)
    Df, If = idx.search(xq, k, sel=sel)
    assert ((If % 2 == 0) | (If == -1)).all()
    # both copies of a repeated id pass or fail together: Not(even ids) over the duplicates keeps only odd ids
    D2, I2, R2 = idx.search_and_reconstruct(xq[:3000], k, sel=vi.IDSelectorNot(sel))
    assert ((I2 % 2 == 1) | (I2 == -1)).all()
    dup = (I2 >= 0) & (I2 < 2000)
    assert dup.any()
    # the same filtered search in one call and split at an arbitrary row
    Da, Ia = idx.search(xq[:20000], k, sel=sel)
    Db, Ib = idx.search(xq[20000:], k, sel=sel)
    _bits(np.r_[Da, Db], Df)
    assert np.array_equal(np.r_[Ia, Ib], If)
    # unsupported selectors fail before anything is written
    D = np.full((4, k), 7.0, np.float32)
    I = np.full((4, k), 7, np.int64)
    with pytest.raises(TypeError):
        idx.search(xq[:4], k, out=(D, I), sel={1, 2})
    assert (D == 7.0).all() and (I == 7).all()
    # n = 0 with a selector is a no-op; reset releases the mask and the index keeps working
    D0, I0 = idx.search(xq[:0], k, sel=sel)
    assert D0.shape == (0, k)
    idx.reset()
    idx.add_with_ids(xb[:100], ids[:100])
    _, Ir = idx.search(xq[:5], k, sel=np.arange(50))
    assert ((Ir >= 0) & (Ir < 50) | (Ir == -1)).all()
    # a selector on an index that cannot filter throws
    flat = vi.GpuIndexFlatL2(res, m["d"])
    flat.add(xb[:100])
    h = vi.host()
    with vi._Selector(vi.IDSelectorRange(0, 10)) as hs:
        Dx = np.full((1, 3), 7.0, np.float32)
        Ix = np.full((1, 3), 7, np.int64)
        assert h.vlq_host_index_search_sel(flat.h, C.c_long(1), C.c_void_p(xq.ctypes.data), C.c_long(3),
                                           C.c_void_p(Dx.ctypes.data), C.c_void_p(Ix.ctypes.data), hs) == -1
        assert b"search parameters not supported" in h.vlq_host_last_error()
        assert (Dx == 7.0).all()


def test_imipq_filtered_search(vi, res, cuda):
    from vector_line_quantization_b200 import data

    xt = data.sift_like(20000, kc=64, seed=21)
    xb = data.sift_like(20000, kc=64, seed=22)
    xq = data.sift_like(300, kc=64, seed=23)
    qn = (xq.astype(np.float64) ** 2).sum(1)
    idx = vi.GpuIndexIMIPQ(res, 128, 4, 16)
    idx.setTrainIters(4)
    idx.train(xt)
    coarse, pq = idx.codebooks()
    ids = np.arange(len(xb), dtype=np.int64) * 7 + 3
    idx.add_with_ids(xb[:12000], ids[:12000])
    idx.add_with_ids(xb[12000:], ids[12000:])  # pending at the first filtered search
    idx.setNumProbes(8)
    k = 30
    D, I = idx.search(xq, k)
    Da, Ia = idx.search(xq, k, sel=vi.IDSelectorRange(0, 1 << 40))
    _bits(Da, D)
    assert np.array_equal(Ia, I)
    rng = np.random.RandomState(4)
    for name, sel, member in _selectors(vi, ids, rng):
        Df, If = idx.search(xq, k, sel=sel)
        sub = vi.GpuIndexIMIPQ(res, 128, 4, 16)
        sub.setCodebooks(coarse, pq)
        sub.add_with_ids(xb[member], ids[member])
        sub.setNumProbes(8)
        Ds, Is = sub.search(xq, k)
        _same_up_to_ties(Df, If, Ds, Is, qn)
        D3, I3, R3 = idx.search_and_reconstruct(xq, k, sel=sel)
        _bits(D3, Df)
        assert np.array_equal(I3, If)
        ok = I3 >= 0
        _bits(R3[ok], idx.reconstruct_batch(I3[ok]))
        assert (R3[~ok].view(np.uint32) == NAN_BITS).all()
        radius = float(np.median(D[:, k // 2]))
        lu, Du, Iu = idx.range_search(xq, radius)
        lf, Dg, Ig = idx.range_search(xq, radius, sel=sel)
        keep = np.isin(Iu, ids[member])
        assert np.array_equal(Ig, Iu[keep])
        _bits(Dg, Du[keep])
        assert lf[-1] == keep.sum()
    Dd, Id = idx.search(T(xq, cuda), k, sel=T(ids[::5], cuda))
    Dh, Ih = idx.search(xq, k, sel=ids[::5])
    _bits(N(Dd), Dh)
    assert np.array_equal(N(Id), Ih)
