"""The C++ host layer (faiss::Index-shaped classes, lib/libvlq_host.so) against the oracle: these read like the
reference's own index tests (build an index through train/add/search, compare with a CPU twin)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vi(cuda):
    from vector_line_quantization_b200 import index

    index.host()
    return index


@pytest.fixture(scope="module")
def res(vi):
    return vi.StandardGpuResources(0)


def test_flat_search_matches_oracle(vi, res, oracle):
    from vector_line_quantization_b200 import data

    xb = data.sift_like(5000, seed=1)
    xq = data.sift_like(100, seed=2)
    for use_tc in (True, False):
        flat = vi.GpuIndexFlatL2(res, 128, use_tensor_cores=use_tc)
        flat.add(xb[:3000])
        flat.add(xb[3000:])
        assert flat.ntotal == 5000
        for k in (1, 10):
            D, I = flat.search(xq, k)
            Do, Io = oracle.l2_topk(xq, xb, k, add_xnorm=True)
            assert (I == Io).mean() > 0.995
            np.testing.assert_allclose(D, Do, rtol=2e-4, atol=1.0)
        assert np.array_equal(flat.assign(xq), oracle.l2_topk(xq, xb, 1)[1][:, 0])
    np.testing.assert_array_equal(flat.reconstruct_n(2990, 20), xb[2990:3010])  # rows of both adds, in order
    np.testing.assert_array_equal(flat.reconstruct(4999), xb[4999])
    with pytest.raises(vi.FaissException):
        flat.reconstruct_n(4990, 20)
    with pytest.raises(vi.FaissException):
        flat.search(xq, 2000)  # k <= 1024
    flat.reset()
    assert flat.ntotal == 0


def test_flat_accepts_device_pointers(vi, res, cuda):
    import torch

    from vector_line_quantization_b200 import data

    xb = data.sift_like(2000, seed=3)
    xq = data.sift_like(64, seed=4)
    flat = vi.GpuIndexFlatL2(res, 128)
    flat.add(torch.from_numpy(xb).to(cuda))
    Dh, Ih = flat.search(xq, 5)
    Dd, Id = flat.search(torch.from_numpy(xq).to(cuda), 5)
    assert Dd.is_cuda and np.array_equal(Id.cpu().numpy(), Ih) and np.array_equal(Dd.cpu().numpy(), Dh)


def test_flat_search_int_and_assign1_base(vi, res, cuda, oracle):
    """searchInt == search with int labels; assign1Base (device pointers) == the oracle's line stage"""
    import torch

    from vector_line_quantization_b200 import data

    cent = data.sift_like(512, seed=5)
    x = data.sift_like(700, seed=6)
    flat = vi.GpuIndexFlatL2(res, 128)
    flat.add(cent)
    D, I = flat.search(x[:50], 7)
    Di, Ii = flat.searchInt(x[:50], 7)
    assert Ii.dtype == np.int32 and np.array_equal(Ii, I) and np.array_equal(Di, D)
    E = 16
    edge, ed2 = oracle.knn_graph(cent, E)
    A = oracle.l2_topk(x, cent, 1)[1][:, 0].astype(np.int32)
    a2, lam = flat.assign1Base(torch.from_numpy(x).to(cuda), torch.from_numpy(A).to(cuda),
                               torch.from_numpy(edge).to(cuda), torch.from_numpy(ed2).to(cuda))
    lo, lamo = oracle.line_stage(x, A, cent, edge, ed2)[:2]
    assert (a2.cpu().numpy() == lo).mean() > 0.995
    same = a2.cpu().numpy() == lo
    np.testing.assert_allclose(lam.cpu().numpy()[same], lamo[same], rtol=1e-3, atol=1e-4)
    with pytest.raises(vi.FaissException):
        flat.assign1Base(torch.from_numpy(x), torch.from_numpy(A), torch.from_numpy(edge), torch.from_numpy(ed2))


def test_kmeans_matches_oracle(vi, res, oracle):
    from vector_line_quantization_b200 import data

    x = data.sift_like(6000, kc=64, seed=31)
    co, _ = oracle.kmeans(x, 40, niter=5, seed=1234)
    cg = vi.kmeans(res, x, 40, niter=5, seed=1234)
    np.testing.assert_allclose(cg, co, rtol=2e-3, atol=0.5)
    assert np.mean(np.abs(cg - co) < 1e-2) > 0.95
    # sub-sampling path (n > k * 256) and a non-tensor-core dimension
    x2 = data.sift_like(3000, d=24, kc=16, seed=33)
    co2, _ = oracle.kmeans(x2, 8, niter=4, seed=99)
    cg2 = vi.kmeans(res, x2, 8, niter=4, seed=99)
    np.testing.assert_allclose(cg2, co2, rtol=2e-3, atol=0.5)


def _build(vi, res, m, xb, chunks=2):
    idx = vi.GpuIndexIVFPQ(res, m["d"], m["C"], m["M"], 8, m["E"], 256)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    step = (len(xb) + chunks - 1) // chunks
    for s in range(0, len(xb), step):
        idx.add(xb[s:s + step])
    return idx


def test_vlq_index_matches_oracle(vi, res, oracle, small_model, tmp_path, monkeypatch):
    m = small_model
    idx = _build(vi, res, m, m["xb"], chunks=3)
    assert idx.ntotal == len(m["xb"])
    enc = oracle.encode_all(m["xb"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    off, perm = oracle.build_lists(enc["list"], m["C"] * m["E"])
    # stored lists == oracle encode, list by list (ids in insertion order; codes / lambda bytes identical up to near-ties)
    mism = 0
    for l in list(range(0, m["C"] * m["E"], 97)) + [int(np.argmax(np.diff(off)))]:
        codes, las, ids = idx.getList(l)
        want = perm[off[l]:off[l + 1]]
        if not np.array_equal(ids, want):
            mism += 1
            continue
        if len(want) == 0:
            continue
        assert (codes == enc["codes"][want]).mean() > 0.99 and (las == enc["lamq"][want]).mean() > 0.99
    assert mism <= 2
    # search: the oracle gets the index exactly as the device stored it (dumped through the reference's .db* files), so
    # only the query path differs; every differing id must be a float64 near-tie (tests/parity_util.py).  The coarse
    # route is chosen per call: at C = 256, P = 16, W = 128 the default is the tcgen05 matrix route, and
    # VLQ_COARSE_EXACT selects the matrix-free one
    for switch, route in ((None, 1), ("VLQ_COARSE_MATRIX", 1), ("VLQ_COARSE_EXACT", 2)):
        with monkeypatch.context() as mp:
            if switch:
                mp.setenv(switch, "1")
            assert _coarse_route(m, 16, 128) == route
            _search_vs_oracle_same_index(idx, oracle, m, m["xq"], 16, 128, 20, tmp_path)


def _coarse_route(m, P, W):
    from vector_line_quantization_b200 import _abi

    return _abi.lib().vlq_coarse_route(m["d"], m["C"], P, m["E"], W, 1)


def test_search_matrix_free_odd_tile_cap(vi, res, oracle, small_model, tmp_path):
    """nlist = 100000, nprobe = 1, w1_ = 256: the matrix-free route with a query tile cap of 3355 rows (odd), where
    per-tile buffers carved back to back once put the bucket minima off their 16-byte boundary and search() failed.
    The host search must equal ops.search bit for bit and match the oracle."""
    import torch

    from vector_line_quantization_b200 import data, ops

    d, C, E, M, P, W, k = 128, 100000, 8, 16, 1, 256, 20
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    cent = t(data.sift_like(C, seed=11))
    edge, ed2 = ops.knn_graph(cent, E)
    m = dict(d=d, C=C, E=E, M=M, cent=cent.cpu().numpy(), edge=edge.cpu().numpy(), edge_d2=ed2.cpu().numpy(),
             lambda_cb=small_model["lambda_cb"], pq=small_model["pq"])
    assert _coarse_route(m, P, W) == 2
    xb = data.sift_like(200000, seed=12)
    xq = data.sift_like(32, seed=13)
    idx = vi.GpuIndexIVFPQ(res, d, C, M, 8, E, len(m["lambda_cb"]))
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    idx.add(xb)
    _search_vs_oracle_same_index(idx, oracle, m, xq, P, W, k, tmp_path)
    D, I = idx.search(xq, k)
    # the same index through the operator layer: tensor-core assignment, line encode, list build, search
    pack = ops.CentPack(cent)
    lcb, pq = t(m["lambda_cb"]), t(m["pq"])
    x = t(xb)
    A, _ = ops.l2_assign_tc(x, pack, want_dist=False)
    enc = ops.line_encode(x, A, cent, edge, ed2, lcb, pq)
    lists = ops.build_lists(C * E, M, enc.list, enc.codes, enc.lamq, enc.kappa,
                            torch.arange(len(xb), dtype=torch.int64, device=dev))
    Do, Io = ops.search(t(xq), cent, pack.cnorm, edge, ed2, lcb, pq, lists, P, W, k, pack=pack,
                        list_len_hint=len(xb) // (C * E))
    assert np.array_equal(Do.cpu().numpy(), D) and np.array_equal(Io.cpu().numpy(), I)


def _dump_index(idx, m, tmp_path):
    """(offsets, list-major codes / lambda bytes / ids, per-id entry tables) of the device index, via writeDbToFile"""
    name = str(tmp_path / "dump")
    idx.writeDbToFile(name)
    M, nl = m["M"], m["C"] * m["E"]
    counts = np.fromfile(name + ".dbcount", dtype=np.int32)
    assert len(counts) == nl
    ids = np.fromfile(name + ".dbIdx", dtype=np.int64)
    codes = np.fromfile(name + ".dbcodes", dtype=np.uint8).reshape(-1, M)
    las = np.fromfile(name + ".dblas", dtype=np.uint8)
    off = np.zeros(nl + 1, np.int64)
    off[1:] = np.cumsum(counts)
    n = int(ids.max()) + 1
    e_list = np.full(n, -1, np.int32)
    e_list[ids] = np.repeat(np.arange(nl, dtype=np.int32), counts)
    e_lamq = np.zeros(n, np.uint8)
    e_lamq[ids] = las
    e_codes = np.zeros((n, M), np.uint8)
    e_codes[ids] = codes
    return off, codes, las, ids, e_list, e_lamq, e_codes


def _search_vs_oracle_same_index(idx, oracle, m, xq, P, W, k, tmp_path, model=None):
    from tests.parity_util import check_lines, check_topk

    mm = m if model is None else model
    off, codes, las, ids, e_list, e_lamq, e_codes = _dump_index(idx, m, tmp_path)
    idx.setNumProbes(P)
    idx.w1_ = W
    D, I = idx.search(xq, k)
    Do, Io, _, lines, _ = oracle.search(xq, mm["cent"], mm["edge"], mm["edge_d2"], mm["lambda_cb"], mm["pq"], off, codes,
                                        las, ids, P=P, W=W, k=k, want_debug=True)
    # the line lists the device path selected (same kernels through the operator layer): every difference from the
    # oracle's choice is verified as a float64 line-score near-tie, and the top-k is compared with the oracle's scan of
    # exactly these lines
    import torch

    from vector_line_quantization_b200 import ops

    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    cent = t(mm["cent"])
    pack = ops.CentPack(cent)
    qd = t(xq)
    stage = ops.CoarseStage(cent, pack.cnorm, t(mm["edge"]), t(mm["edge_d2"]), P, W, len(xq), pack)  # the host's route
    lst, _, _ = stage.run(qd)
    same_lines = check_lines(lst.cpu().numpy(), lines, xq, mm)
    # strict for every query: against the oracle's scan of the device's own line choice
    Dl, Il = oracle.scan_lines(xq, mm["cent"], mm["edge"], mm["edge_d2"], mm["lambda_cb"], mm["pq"], off, codes, las, ids,
                               lst.cpu().numpy(), k)
    check_topk(D, I, Dl, Il, xq, mm, e_list, e_lamq, e_codes)
    check_topk(D, I, Do, Io, xq, mm, e_list, e_lamq, e_codes, same_lines)
    return I, Il


def test_search_tile_pipeline_many_tiles(vi, res, cuda, small_model):
    """GpuIndexIVFPQ::search runs the scan of query tile i on a second stream beside the coarse stage of tile i + 1, on two
    alternating sets of line buffers: a batch of many tiles (slot reuse, several 32768-query pages, host and device
    buffers) must return what the same queries return one small batch at a time"""
    import torch

    m = small_model
    idx = _build(vi, res, m, m["xb"])
    idx.setNumProbes(16)
    idx.w1_ = 64
    k = 10
    rng = np.random.RandomState(3)
    xq = m["xq"][rng.randint(0, len(m["xq"]), 40000)] + rng.randint(-2, 3, (40000, m["d"])).astype(np.float32)
    D, I = idx.search(xq, k)  # 40000 queries: pages of 32768, tiles of <= 5120
    for s in range(0, len(xq), 7000):
        Ds, Is = idx.search(xq[s:s + 1500], k)
        assert np.array_equal(Ds, D[s:s + 1500]) and np.array_equal(Is, I[s:s + 1500])
    qd = torch.from_numpy(xq).to(cuda)
    oD = torch.empty((len(xq), k), dtype=torch.float32, device=cuda)
    oI = torch.empty((len(xq), k), dtype=torch.int64, device=cuda)
    idx.search(qd, k, out=(oD, oI))
    assert np.array_equal(oD.cpu().numpy(), D) and np.array_equal(oI.cpu().numpy(), I)


def test_vlq_train_on_device(vi, res, oracle, small_model, tmp_path):
    """train() end to end on the device; quality must match the oracle-trained model (same algorithm, same seeds)"""
    from vector_line_quantization_b200 import data

    m = small_model
    idx = vi.GpuIndexIVFPQ(res, 128, m["C"], m["M"], 8, m["E"], 256)
    assert not idx.is_trained
    with pytest.raises(vi.FaissException):
        idx.add(m["xb"][:10])  # "Index not trained"
    idx.setTrainIters(6)
    idx.train(m["xt"])
    assert idx.is_trained
    cb = idx.codebooks()
    # same k-means as the oracle (identical RNG + update rule): centroids agree up to assignment near-ties
    assert np.mean(np.abs(cb["cent"] - m["cent"]) < 0.05) > 0.9
    eo, _ = oracle.knn_graph(cb["cent"], m["E"])
    assert (cb["edge"] == eo).mean() > 0.999
    idx.add(m["xb"])
    # recall (gpu/test/sift1b_query.cpp:334-347) against the oracle on the SAME index (device-trained codebooks, device-
    # stored lists): within 0.1 pt (north_star) on 2000 queries -- in fact the results are identical up to near-ties
    xq = data.sift_like(2000, kc=512, seed=4)
    cbm = dict(cent=cb["cent"], edge=cb["edge"], edge_d2=cb["edge_d2"], lambda_cb=cb["lambda_cb"], pq=cb["pq"])
    I, Io = _search_vs_oracle_same_index(idx, oracle, m, xq, 32, 256, 100, tmp_path, model=cbm)
    _, gt = oracle.l2_topk(xq, m["xb"], 1)
    for r in (1, 10, 100):
        r_gpu, r_cpu = data.recall_at(I, gt[:, 0], r), data.recall_at(Io, gt[:, 0], r)
        assert abs(r_gpu - r_cpu) <= 0.001, (r, r_gpu, r_cpu)
    assert data.recall_at(I, gt[:, 0], 100) > 0.8  # and the device-trained model is as good as the oracle-trained one


def test_file_formats_roundtrip_and_rank_slices(vi, res, small_model, tmp_path):
    m = small_model
    idx = _build(vi, res, m, m["xb"])
    idx.setNumProbes(16)
    idx.w1_ = 128
    D0, I0 = idx.search(m["xq"], 10)
    name = str(tmp_path / "vlqdb")
    idx.writeCodebookToFile(name)
    idx.writeDbToFile(name)
    L = m["C"] * m["E"]
    n = len(m["xb"])
    assert os.path.getsize(name + ".dbcount") == 4 * L and os.path.getsize(name + ".dbIdx") == 8 * n
    assert os.path.getsize(name + ".dbcodes") == m["M"] * n and os.path.getsize(name + ".dblas") == n
    assert os.path.getsize(name + ".ppqt") == 4 * (m["C"] * 128 + 256 * 128 + 2 * L + 2 * 256)
    idx2 = vi.GpuIndexIVFPQ(res, 128, m["C"], m["M"], 8, m["E"], 256)
    idx2.readCodebookFromFile(name)
    idx2.readDbFromFile(name)
    idx2.setNumProbes(16)
    idx2.w1_ = 128
    D1, I1 = idx2.search(m["xq"], 10)
    assert np.array_equal(I1, I0) and np.array_equal(D1, D0)
    # list-range slices over 3 "ranks" + merge == the whole index (gpu/test/sift1b16_query.cpp:323,405-430)
    Ds, Is = [], []
    for r in range(3):
        part = vi.GpuIndexIVFPQ(res, 128, m["C"], m["M"], 8, m["E"], 256)
        part.readCodebookFromFile(name)
        part.readDbFromFile(name, 3, r)
        part.setNumProbes(16)
        part.w1_ = 128
        d_, i_ = part.search(m["xq"], 10)
        Ds.append(d_)
        Is.append(i_)
    assert sum(1 for _ in Is) == 3
    Dm, Im = idx.merge(np.stack(Is), np.stack(Ds))
    assert np.array_equal(Dm, D0) and (Im == I0).mean() > 0.999


def test_shards_and_proxy(vi, res, small_model):
    m = small_model
    whole = _build(vi, res, m, m["xb"])
    whole.setNumProbes(16)
    whole.w1_ = 128
    whole.setListCap(1 << 20)
    D0, I0 = whole.search(m["xq"], 10)
    shards = vi.IndexShards(128, threaded=True, successive_ids=True)
    subs = []
    for a, b in [(0, 9000), (9000, 20000)]:
        s = _build(vi, res, m, m["xb"][a:b])
        s.setNumProbes(16)
        s.w1_ = 128
        s.setListCap(1 << 20)
        subs.append(s)
        shards.add_shard(s)
    assert shards.ntotal == 20000
    D1, I1 = shards.search(m["xq"], 10)
    assert np.array_equal(D1, D0) and (I1 == I0).mean() > 0.999
    proxy = vi.IndexProxy()
    rep = _build(vi, res, m, m["xb"])
    rep.setNumProbes(16)
    rep.w1_ = 128
    rep.setListCap(1 << 20)
    proxy.addIndex(whole)
    proxy.addIndex(rep)
    D2, I2 = proxy.search(m["xq"], 10)
    assert np.array_equal(D2, D0) and np.array_equal(I2, I0)


def test_shards_on_two_gpus_merge_over_peer_memory(vi, small_model):
    """IndexShards with one GpuIndexIVFPQ per GPU: the merge kernel on GPU 0 reads the other shard's results straight from
    its memory (vlq_enable_peer_access + vlq_merge_topk_peers); equals the single index, host and device buffers"""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    m = small_model
    r0, r1 = vi.StandardGpuResources(0), vi.StandardGpuResources(1)
    whole = _build(vi, r0, m, m["xb"])
    subs = [_build(vi, r0, m, m["xb"][:9000]), _build(vi, r1, m, m["xb"][9000:])]
    shards = vi.IndexShards(128, threaded=True, successive_ids=True)
    for s in [whole] + subs:
        s.setNumProbes(16)
        s.w1_ = 128
        s.setListCap(1 << 20)
    for s in subs:
        shards.add_shard(s)
    D0, I0 = whole.search(m["xq"], 10)
    D1, I1 = shards.search(m["xq"], 10)
    assert np.array_equal(D1, D0) and (I1 == I0).mean() > 0.999
    xq_dev = torch.from_numpy(m["xq"]).to("cuda:0")
    oD = torch.empty((len(m["xq"]), 10), dtype=torch.float32, device="cuda:0")
    oI = torch.empty((len(m["xq"]), 10), dtype=torch.int64, device="cuda:0")
    shards.search(xq_dev, 10, out=(oD, oI))
    assert np.array_equal(oD.cpu().numpy(), D1) and np.array_equal(oI.cpu().numpy(), I1)


def test_add_with_ids_and_reset(vi, res, small_model):
    m = small_model
    idx = vi.GpuIndexIVFPQ(res, 128, m["C"], m["M"], 8, m["E"], 256)
    idx.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    ids = np.arange(5000, dtype=np.int64) * 7 + 3
    idx.add_with_ids(m["xb"][:5000], ids)
    idx.setNumProbes(8)
    idx.w1_ = 64
    _, I = idx.search(m["xb"][:50], 5)  # database vectors as queries
    assert np.all((I[I >= 0] - 3) % 7 == 0)
    assert np.mean(I[:, 0] == ids[:50]) > 0.5
    idx.reset()
    assert idx.ntotal == 0
    D, I = idx.search(m["xq"], 3)
    assert np.all(I == -1) and np.all(D == np.finfo(np.float32).max)


def test_add_u8_equals_add_f32(vi, res, small_model):
    """uint8 ingestion (bytes over PCIe, widened on the device) stores exactly what the fp32 path stores"""
    m = small_model
    xb = m["xb"][:6000]
    assert np.array_equal(xb, xb.astype(np.uint8).astype(np.float32))  # SIFT-shaped data is uint8-valued
    a = _build(vi, res, m, xb, chunks=1)
    b = vi.GpuIndexIVFPQ(res, m["d"], m["C"], m["M"], 8, m["E"], 256)
    b.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    b.add_with_ids_u8(xb.astype(np.uint8), np.arange(6000, dtype=np.int64))
    for idx in (a, b):
        idx.setNumProbes(16)
        idx.w1_ = 128
    Da, Ia = a.search(m["xq"], 10)
    Db, Ib = b.search(m["xq"], 10)
    assert np.array_equal(Ia, Ib) and np.array_equal(Da, Db)


def test_search1_candidate_lists_and_ground_truth_builder(vi, res, small_model):
    """f4: search1 returns the ids of the entries of the selected lines in line order (gpu/GpuIndexIVFPQ.cu:1646-1670);
    add_with_ids2 is the brute-force ground-truth builder (:1354-1398)"""
    m = small_model
    idx = _build(vi, res, m, m["xb"])
    idx.setNumProbes(8)
    idx.w1_ = 32
    idx.setListCap(1 << 20)
    xq = m["xq"][:40]
    kc = 4000  # room for every entry of 32 lines here
    cand = idx.search1(xq, kc)
    D, I = idx.search(xq, 10)
    for q in range(len(xq)):
        c = cand[q]
        n = int((c >= 0).sum())
        assert n > 0 and (c[:n] >= 0).all() and (c[n:] == -1).all() and len(set(c[:n].tolist())) == n
        assert set(I[q][I[q] >= 0].tolist()) <= set(c[:n].tolist())  # the top-k comes out of the candidate list
    short = idx.search1(xq, 7)
    assert np.array_equal(short, cand[:, :7])
    # ground truth of a chunk with its own labels
    x = m["xb"][:3000]
    ids = np.arange(3000, dtype=np.int64) * 3 + 11
    dists, nns = idx.add_with_ids2(x, xq, 5, ids)
    d2 = ((xq.astype(np.float64)[:, None, :] - x.astype(np.float64)[None, :, :]) ** 2).sum(2)
    order = np.argsort(d2, axis=1, kind="stable")[:, :5]
    ref_d = np.take_along_axis(d2, order, axis=1)
    assert np.allclose(dists, ref_d, rtol=1e-4)
    assert (nns == ids[order]).mean() > 0.99
