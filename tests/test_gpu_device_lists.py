"""The inverted lists GpuIndexIVFPQ and GpuIndexIMIPQ share (host/DeviceLists.h): adds in chunks with searches in
between, reset followed by new adds, and remove_ids followed by adds must leave either index exactly where a fresh index
holding the same vectors is -- every list length, distance and label bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K = 20


@pytest.fixture(scope="module")
def vi(cuda):
    from vector_line_quantization_b200 import index

    index.host()
    return index


@pytest.fixture(scope="module")
def res(vi):
    return vi.StandardGpuResources(0)


@pytest.fixture(scope="module", params=["GpuIndexIVFPQ", "GpuIndexIMIPQ"])
def kind(request, vi, res, small_model):
    """(factory of an empty index with trained codebooks, number of lists)"""
    m = small_model
    if request.param == "GpuIndexIVFPQ":
        def new():
            idx = vi.GpuIndexIVFPQ(res, m["d"], m["C"], m["M"], 8, m["E"], 256)
            idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
            idx.setNumProbes(16)
            idx.w1_ = 128
            return idx

        return new, m["C"] * m["E"]
    t = vi.GpuIndexIMIPQ(res, m["d"], 4, m["M"])
    t.setTrainIters(4)
    t.train(m["xt"])
    coarse, pq = t.codebooks()

    def new():
        idx = vi.GpuIndexIMIPQ(res, m["d"], 4, m["M"])
        idx.setCodebooks(coarse, pq)
        idx.setNumProbes(16)
        return idx

    return new, 256


def _fresh(new, x, ids=None):
    idx = new()
    if ids is None:
        idx.add(x)
    else:
        idx.add_with_ids(x, ids)
    return idx


def _assert_same(a, b, nlists, xq):
    assert a.ntotal == b.ntotal
    assert [a.getListLength(l) for l in range(nlists)] == [b.getListLength(l) for l in range(nlists)]
    Da, Ia = a.search(xq, K)
    Db, Ib = b.search(xq, K)
    assert np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32))


def test_chunked_adds_with_searches_equal_one_add(kind, small_model):
    new, nlists = kind
    xb, xq = small_model["xb"], small_model["xq"]
    a = new()
    for end in (6000, 13000, len(xb)):
        a.add(xb[a.ntotal:end])
        a.search(xq, K)  # merges the chunk into the lists
        _assert_same(a, _fresh(new, xb[:end]), nlists, xq)


def test_reset_then_add_equals_fresh_index(kind, small_model):
    from vector_line_quantization_b200 import data

    new, nlists = kind
    xb, xq = small_model["xb"], small_model["xq"]
    a = new()
    a.add(xb[:8000])
    a.search(xq, K)
    a.add(xb[8000:])  # still pending at the reset
    a.reset()
    assert a.ntotal == 0 and all(a.getListLength(l) == 0 for l in range(0, nlists, 7))
    # 80 000 vectors in four adds without a search between them: the pending entries outgrow the first arena
    x = data.sift_like(80000, kc=512, seed=5)
    for s in range(0, len(x), 20000):
        a.add(x[s:s + 20000])
    _assert_same(a, _fresh(new, x), nlists, xq)


def test_remove_then_add_equals_fresh_index(kind, small_model):
    from vector_line_quantization_b200 import data

    new, nlists = kind
    xb, xq = small_model["xb"], small_model["xq"]
    ids = np.arange(len(xb), dtype=np.int64)
    gone = np.random.RandomState(11).rand(len(xb)) < 0.3
    xn = data.sift_like(3000, kc=512, seed=6)
    idn = np.arange(3000, dtype=np.int64) + 10 ** 6
    a = _fresh(new, xb)
    assert a.remove_ids(ids[gone]) == int(gone.sum())
    a.add_with_ids(xn, idn)
    b = _fresh(new, xb[~gone], ids[~gone])
    b.add_with_ids(xn, idn)
    _assert_same(a, b, nlists, xq)
