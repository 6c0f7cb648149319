"""remove_ids: the device compaction against a torch restatement, and an index after removal against an index that never
received the removed vectors (same files, same search results: the survivors keep their order)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FLT_MAX = np.finfo(np.float32).max


# ------------------------------------------------------------------------------------------------ ops level
def _slab(torch, ops, nlists, mean, M, dev, seed):
    """list-major slab in the stored layout: empty lists, lists longer than 2048, ids in no particular order"""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lens = torch.poisson(torch.distributions.Gamma(2.0, 2.0).sample((nlists,)) * mean, generator=g).to(torch.int64)
    lens[::97] = 0
    lens[5::211] = 3000 + torch.randint(0, 2000, (lens[5::211].numel(),), generator=g)
    off = torch.zeros(nlists + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(lens, 0)
    n = int(off[-1])
    codes = torch.randint(0, 256, (n, M), dtype=torch.uint8, generator=g)
    lamq = torch.randint(0, 256, (n,), dtype=torch.uint8, generator=g)
    kappa = torch.randn(n, generator=g) * 100.0
    ids = torch.randperm(2 * n, generator=g)[:n].to(torch.int64) * 3 + 7
    off, codes = off.to(dev), codes.to(dev)
    stored = ops.rotate_codes(off, codes)
    return ops.Lists(off, stored, lamq.to(dev), kappa.to(dev), ids.to(dev))


def _reference(torch, ops, lists, batch, id_range):
    """canonical codes -> boolean mask -> stored layout of the new offsets"""
    canon = ops.rotate_codes(lists.offsets, lists.codes, inverse=True)
    gone = torch.zeros_like(lists.ids, dtype=torch.bool)
    if batch is not None:
        gone |= torch.isin(lists.ids, batch)
    if id_range is not None:
        gone |= (lists.ids >= id_range[0]) & (lists.ids < id_range[1])
    keep = ~gone
    nlists = lists.offsets.numel() - 1
    lens = lists.offsets[1:] - lists.offsets[:-1]
    list_of = torch.repeat_interleave(torch.arange(nlists, device=keep.device), lens)
    new_lens = torch.zeros(nlists, dtype=torch.int64, device=keep.device).index_add_(0, list_of, keep.to(torch.int64))
    off = torch.zeros_like(lists.offsets)
    off[1:] = torch.cumsum(new_lens, 0)
    codes = ops.rotate_codes(off, canon[keep].contiguous())
    return ops.Lists(off, codes, lists.lamq[keep], lists.kappa[keep], lists.ids[keep]), int(gone.sum())


@pytest.mark.parametrize("M", [16, 8, 32])
def test_remove_ids_kernel_matches_torch(cuda, M):
    import torch

    from vector_line_quantization_b200 import ops

    lists = _slab(torch, ops, 6000, 500.0, M, cuda, seed=M)
    n = lists.ids.numel()
    assert n > 2_000_000
    lens = (lists.offsets[1:] - lists.offsets[:-1]).cpu()
    assert int((lens == 0).sum()) > 0 and int((lens > 2048).sum()) > 0
    g = torch.Generator(device="cpu").manual_seed(M + 1)
    ids_cpu = lists.ids.cpu()
    pick = ids_cpu[torch.randperm(n, generator=g)[: n // 10]]
    whole = [int(l) for l in torch.nonzero(lens > 0).flatten()[:40:4]]  # lists that lose every entry
    off = lists.offsets.cpu()
    every = torch.cat([ids_cpu[off[l]:off[l + 1]] for l in whole])
    absent = torch.tensor([0, 1, 2, 3 * n * 2 + 100], dtype=torch.int64)  # stored ids are 1 mod 3 and >= 7
    batch = torch.cat([pick, pick[:1000], every, absent])  # duplicates too
    srt = ids_cpu.sort().values
    rng = (int(srt[n // 3]), int(srt[n // 3 + n // 20]))
    for sel_batch, sel_range in ((batch, None), (None, rng), (batch, rng)):
        got, removed = ops.remove_ids(lists, ids=None if sel_batch is None else sel_batch.to(cuda), id_range=sel_range)
        ref, ref_removed = _reference(torch, ops, lists, None if sel_batch is None else sel_batch.to(cuda), sel_range)
        assert removed == ref_removed > 0
        assert torch.equal(got.offsets, ref.offsets)
        for name in ("codes", "lamq", "ids"):
            assert torch.equal(getattr(got, name), getattr(ref, name)), name
        assert torch.equal(got.kappa.view(torch.int32), ref.kappa.view(torch.int32))
        if sel_batch is not None:
            glens = (got.offsets[1:] - got.offsets[:-1]).cpu()
            assert all(int(glens[l]) == 0 for l in whole)
    # nothing selected: a bit-identical slab
    got, removed = ops.remove_ids(lists, ids=absent.to(cuda), id_range=(5, 5))
    assert removed == 0
    for a, b in zip(got, lists):
        assert torch.equal(a, b)
    got, removed = ops.remove_ids(lists, id_range=(-(1 << 62), 1 << 62))  # everything
    assert removed == n and int(got.offsets.abs().sum()) == 0 and got.ids.numel() == 0


# ------------------------------------------------------------------------------------------------ index level
@pytest.fixture(scope="module")
def vi(cuda):
    from vector_line_quantization_b200 import index

    index.host()
    return index


@pytest.fixture(scope="module")
def res(vi):
    return vi.StandardGpuResources(0)


def _data(kind, n, seed):
    from vector_line_quantization_b200 import data

    return data.sift_like(n, kc=64, seed=seed) if kind == "sift" else data.deep_like(n, kc=64, seed=seed)


@pytest.fixture(scope="module", params=[("sift", 128, 16), ("deep", 96, 8)], ids=["d128M16", "d96M8"])
def model(request, vi, res):
    """codebooks of a C = 16, E = 4 index (about 300 entries per line for 20 000 vectors)"""
    kind, d, M = request.param
    xt = _data(kind, 20000, 1)
    t = vi.GpuIndexIVFPQ(res, d, 16, M, 8, 4, 16)
    t.setTrainIters(4)
    t.train(xt)
    rng = np.random.RandomState(d)
    return dict(kind=kind, d=d, M=M, cb=t.codebooks(), xb=_data(kind, 20000, 2), xq=_data(kind, 200, 3),
                ids=rng.permutation(100000)[:20000].astype(np.int64) * 5 + 11)


def _index(vi, res, m, chunks=()):
    idx = vi.GpuIndexIVFPQ(res, m["d"], 16, m["M"], 8, 4, 16)
    cb = m["cb"]
    idx.setCodebooks(cb["cent"], cb["edge"], cb["edge_d2"], cb["lambda_cb"], cb["pq"])
    idx.setNumProbes(4)
    idx.w1_ = 16
    for x, ids in chunks:
        idx.add_with_ids(x, ids)
    return idx


def _chunks(x, ids, k=3):
    step = -(-len(x) // k)
    return [(x[s:s + step], ids[s:s + step]) for s in range(0, len(x), step)]


def _files(idx, path):
    idx.writeDbToFile(str(path))
    return {ext: open(str(path) + ext, "rb").read() for ext in (".dbIdx", ".dbcodes", ".dbcount", ".dblas")}


def _assert_same(a, b, xq, tmp_path, caps=(1024, 64)):
    fa, fb = _files(a, tmp_path / "a"), _files(b, tmp_path / "b")
    for ext in fa:
        assert fa[ext] == fb[ext], ext
    assert a.ntotal == b.ntotal
    for cap in caps:
        a.setListCap(cap)
        b.setListCap(cap)
        Da, Ia = a.search(xq, 20)
        Db, Ib = b.search(xq, 20)
        assert np.array_equal(Ia, Ib) and np.array_equal(Da, Db), cap
    a.setListCap(1024)
    b.setListCap(1024)


def test_index_after_removal_equals_index_without(vi, res, model, tmp_path):
    m = model
    xb, ids = m["xb"], m["ids"]
    rng = np.random.RandomState(5)
    gone = rng.rand(len(xb)) < 0.3
    a = _index(vi, res, m, _chunks(xb, ids))  # adds still pending: the removal commits them first
    b = _index(vi, res, m, _chunks(xb[~gone], ids[~gone]))
    sel = np.concatenate([ids[gone][::-1], ids[gone][:50], [3, 4]])  # any order, duplicates, absent ids
    assert a.remove_ids(sel) == int(gone.sum())
    assert a.ntotal == int((~gone).sum())
    assert max(a.getListLength(l) for l in range(64)) > 128  # longer than the list cap of 64 below
    _assert_same(a, b, m["xq"], tmp_path)
    # a range, then a batch given as a CUDA tensor
    import torch

    lo, hi = np.sort(ids[~gone])[[100, 2000]]
    in_range = (ids >= lo) & (ids < hi) & ~gone
    assert a.remove_ids(vi.IDSelectorRange(lo, hi)) == int(in_range.sum())
    gone |= in_range
    more = (rng.rand(len(xb)) < 0.2) & ~gone
    assert a.remove_ids(torch.from_numpy(ids[more]).to("cuda")) == int(more.sum())
    gone |= more
    c = _index(vi, res, m, _chunks(xb[~gone], ids[~gone], 2))
    _assert_same(a, c, m["xq"], tmp_path)


def test_removal_with_pending_adds_then_add_with_ids(vi, res, model, tmp_path):
    m = model
    xb, ids = m["xb"], m["ids"]
    a = _index(vi, res, m, [(xb[:8000], ids[:8000]), (xb[8000:14000], ids[8000:14000])])
    a.search(m["xq"][:4], 1)  # commits the first two chunks
    a.add_with_ids(xb[14000:], ids[14000:])  # pending
    gone = np.zeros(len(xb), bool)
    gone[np.random.RandomState(7).choice(len(xb), 4000, replace=False)] = True
    assert gone[14000:].any() and gone[:14000].any()
    assert a.remove_ids(ids[gone]) == int(gone.sum())
    b = _index(vi, res, m, _chunks(xb[~gone], ids[~gone]))
    _assert_same(a, b, m["xq"], tmp_path)
    # upsert: re-add a third of the removed vectors under their ids, plus vectors under new ids
    back = np.flatnonzero(gone)[::3]
    xn = _data(m["kind"], 500, 9)
    idn = np.arange(500, dtype=np.int64) + 10 ** 7
    a.add_with_ids(xb[back], ids[back])
    a.add_with_ids(xn, idn)
    b.add_with_ids(xb[back], ids[back])
    b.add_with_ids(xn, idn)
    _assert_same(a, b, m["xq"], tmp_path)


def test_empty_selection_and_remove_everything(vi, res, model, tmp_path):
    m = model
    xb, ids = m["xb"], m["ids"]
    a = _index(vi, res, m, _chunks(xb, ids))
    D0, I0 = a.search(m["xq"], 20)
    f0 = _files(a, tmp_path / "before")
    for sel in (np.empty(0, np.int64), np.array([0, 1, 2], np.int64), vi.IDSelectorRange(5, 5),
                vi.IDSelectorRange(10, 3)):
        assert a.remove_ids(sel) == 0
    assert a.ntotal == len(xb) and _files(a, tmp_path / "after") == f0
    D1, I1 = a.search(m["xq"], 20)
    assert np.array_equal(D0, D1) and np.array_equal(I0, I1)
    # no removed id is ever returned, by search or by the candidate lists of search1
    gone = ids[::4]
    a.remove_ids(gone)
    D, I = a.search(m["xq"], 50)
    cand = a.search1(m["xq"], 4000)
    assert not np.isin(I, gone).any() and not np.isin(cand, gone).any()
    assert (cand >= 0).sum() > 0
    assert a.remove_ids(vi.IDSelectorRange(int(ids.min()), int(ids.max()) + 1)) == len(xb) - len(gone)
    assert a.ntotal == 0
    D, I = a.search(m["xq"], 10)
    assert np.all(I == -1) and np.all(D == FLT_MAX)
    # add() after a removal numbers the new vectors from ntotal, as faiss does
    a.add(xb[:10])
    D, I = a.search(xb[:10], 1)
    assert a.ntotal == 10 and (I >= 0).any() and set(I[I >= 0].tolist()) <= set(range(10))


def test_imipq_after_removal_equals_fresh_index(vi, res, cuda):
    from vector_line_quantization_b200 import data

    xt = data.sift_like(20000, kc=64, seed=21)
    xb = data.sift_like(20000, kc=64, seed=22)
    xq = data.sift_like(100, kc=64, seed=23)
    ids = np.arange(len(xb), dtype=np.int64) * 3 + 1
    t = vi.GpuIndexIMIPQ(res, 128, 4, 16)
    t.setTrainIters(4)
    t.train(xt)
    coarse, pq = t.codebooks()
    gone = np.random.RandomState(3).rand(len(xb)) < 0.25

    def build(x, i):
        idx = vi.GpuIndexIMIPQ(res, 128, 4, 16)
        idx.setCodebooks(coarse, pq)
        idx.setNumProbes(16)
        for s in range(0, len(x), 7000):
            idx.add_with_ids(x[s:s + 7000], i[s:s + 7000])
        return idx

    a = build(xb, ids)
    b = build(xb[~gone], ids[~gone])
    assert a.remove_ids(ids[gone]) == int(gone.sum())
    assert a.ntotal == b.ntotal
    assert [a.getListLength(c) for c in range(256)] == [b.getListLength(c) for c in range(256)]
    Da, Ia = a.search(xq, 20)
    Db, Ib = b.search(xq, 20)
    assert np.array_equal(Ia, Ib) and np.array_equal(Da, Db)
    assert a.remove_ids(vi.IDSelectorRange(0, 3000)) == int(((ids < 3000) & ~gone).sum())
