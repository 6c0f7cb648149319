"""CUDA path against the UNMODIFIED reference library itself (oracle/_ref/libfaiss_ref.so, the reference's CPU
IndexIVFPQ), not just against the oracle restatement.

With a single lambda level equal to 0 the VLQ anchor (1-l)c + l s is the centroid c itself, so a VLQ index whose search
keeps ALL lines of the probed centroids (w1 = nprobe * nedge) is exactly IndexIVFPQ with nprobe probes: same coarse
assignment, same residual PQ codes, same ADC distances (up to ||q||^2, which the GPU search path omits like the
reference's GPU path, gpu/impl/Distance.cu:287-290).
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vlq_small.npz")


@pytest.fixture(scope="module")
def ref(oracle):
    if not oracle.ref_available():
        pytest.skip("oracle/_ref/libfaiss_ref.so not built")
    oracle.ref()
    return oracle


@pytest.mark.parametrize("d,C,E,M,P", [(128, 64, 16, 16, 8), (64, 32, 8, 8, 6)])
def test_gpu_vlq_lambda0_equals_reference_ivfpq(cuda, ref, d, C, E, M, P):
    from vector_line_quantization_b200 import data, index as vi, ops

    k = 10
    xt = data.sift_like(20000, d=d, kc=256, seed=61)
    xb = data.sift_like(30000, d=d, kc=256, seed=62)
    xq = data.sift_like(100, d=d, kc=256, seed=63)
    ivf = ref.RefIVFPQ(d, C, M)           # the reference's own train: Clustering + ProductQuantizer on the CPU
    ivf.train(xt)
    cent, pq = ivf.codebooks()
    ivf.add(xb)
    Dr, Ir = ivf.search(xq, k, P)

    import torch

    edge, ed2 = ops.knn_graph(torch.from_numpy(cent).to(cuda), E)
    res = vi.StandardGpuResources(0)
    idx = vi.GpuIndexIVFPQ(res, d, C, M, 8, E, 1)
    idx.setCodebooks(cent, edge.cpu().numpy(), ed2.cpu().numpy(), np.zeros(1, np.float32), pq)
    idx.add(xb)
    # encode parity: the union of the E line lists of centroid c holds exactly the reference's list c, same PQ codes
    for c in range(C):
        ids_r, codes_r = ivf.get_list(c)
        got = {}
        for e in range(E):
            codes, las, ids = idx.getList(c * E + e)
            assert np.all(las == 0)
            for i, code in zip(ids, codes):
                got[int(i)] = code
        common = [i for i in ids_r if int(i) in got]
        assert len(common) >= len(ids_r) - 2 and len(got) <= len(ids_r) + 2  # coarse near-ties may move a vector
        same = np.mean([np.array_equal(got[int(i)], codes_r[j]) for j, i in enumerate(ids_r) if int(i) in got])
        assert same > 0.995
    # search parity
    idx.setNumProbes(P)
    idx.w1_ = P * E
    idx.setListCap(1 << 20)
    D, I = idx.search(xq, k)
    qn = np.sum(xq.astype(np.float64) ** 2, axis=1, keepdims=True)
    assert (I == Ir).mean() > 0.97
    same = I == Ir
    np.testing.assert_allclose((D + qn)[same], Dr[same], rtol=2e-4)
    overlap = np.mean([len(set(a) & set(b)) / k for a, b in zip(I, Ir)])
    assert overlap > 0.99


def test_gpu_vlq_lambda0_equals_stored_reference_ivfpq(cuda):
    """The same lambda == 0 identity on the golden fixture (tests/golden/vlq_small.npz), where the reference's
    IndexFlatL2 assignment and IndexIVFPQ search results with the fixture's codebooks are stored: runs without the
    reference library."""
    from vector_line_quantization_b200 import index as vi

    g = dict(np.load(GOLD))
    d, C, E, M, P, k = (int(g[key]) for key in ("d", "C", "E", "M", "P", "k"))
    xb, xq = g["xb"].astype(np.float32), g["xq"].astype(np.float32)
    res = vi.StandardGpuResources(0)
    idx = vi.GpuIndexIVFPQ(res, d, C, M, 8, E, 1)
    idx.setCodebooks(g["cent"], g["edge"], g["edge_d2"], np.zeros(1, np.float32), g["pq"])
    idx.add(xb)
    # encode parity: the E line lists of centroid c hold the vectors IndexFlatL2 assigned to c, up to near-ties
    assign = np.full(len(xb), -1, np.int64)
    for c in range(C):
        for e in range(E):
            _, las, ids = idx.getList(c * E + e)
            assert np.all(las == 0)
            assign[ids] = c
    assert np.all(assign >= 0)
    for i in np.nonzero(assign != g["ref_flat_assign_I"])[0]:
        da, db = (np.sum((xb[i].astype(np.float64) - g["cent"][c]) ** 2) for c in (assign[i], g["ref_flat_assign_I"][i]))
        assert abs(da - db) <= 1e-5 * max(da, db), (int(i), da, db)
    idx.setNumProbes(P)
    idx.w1_ = P * E
    idx.setListCap(1 << 20)
    D, I = idx.search(xq, k)
    qn = np.sum(xq.astype(np.float64) ** 2, axis=1, keepdims=True)
    same = I == g["ref_ivfpq_I"]
    assert same.mean() > 0.97
    np.testing.assert_allclose((D + qn)[same], g["ref_ivfpq_D"][same], rtol=2e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("nedge", [1, 4])
def test_copy_from_reference_cpu_index_and_back(cuda, oracle, nedge):
    """f4, no oracle in between: the UNMODIFIED reference CPU IndexIVFPQ (oracle/_ref) is trained and filled on the CPU,
    its codebooks and inverted lists go through GpuIndexIVFPQ::copyFrom, and GpuIndexIVFPQ::search must return what
    IndexIVFPQ::search returns (gpu/GpuIndexIVFPQ.cu:169-232); copyTo gives the same lists back (:234-281)"""
    if not oracle.ref_available():
        pytest.skip("reference library not built")
    from vector_line_quantization_b200 import data, index as vi

    d, nlist, M, k, nprobe = 64, 64, 8, 10, 8
    xt = data.sift_like(20000, d=d, kc=256, seed=1)
    xb = data.sift_like(30000, d=d, kc=256, seed=2)
    xq = data.sift_like(200, d=d, kc=256, seed=3)
    ref = oracle.RefIVFPQ(d, nlist, M, 8)
    ref.train(xt)
    ref.add(xb)
    Dr, Ir = ref.search(xq, k, nprobe)
    coarse, pq = ref.codebooks()
    cpu = vi.CpuIndexIVFPQ(d, nlist, M, 8)
    cpu.set_codebooks(coarse, pq)
    for l in range(nlist):
        cpu.set_list(l, *ref.get_list(l))
    assert cpu.ntotal == len(xb)
    res = vi.StandardGpuResources(0)
    gpu = vi.GpuIndexIVFPQ(res, d, nlist, M, 8, nedge, 16)
    gpu.copyFrom(cpu)
    assert gpu.ntotal == len(xb)
    gpu.setNumProbes(nprobe)
    gpu.w1_ = nprobe * nedge  # every line of the probed centroids: exactly IndexIVFPQ::search(nprobe)
    gpu.setListCap(1 << 20)  # the reference's CPU search has no 1024-entry cap per list
    D, I = gpu.search(xq, k)
    qn = (xq.astype(np.float64) ** 2).sum(1, keepdims=True)  # the GPU path omits ||q||^2
    same = I == Ir
    assert same.mean() > 0.97  # (a coarse near-tie at the nprobe boundary changes which lists a query scans)
    np.testing.assert_allclose((D + qn)[same], Dr[same], rtol=2e-4)
    assert np.mean([len(set(a) & set(b)) / k for a, b in zip(I, Ir)]) > 0.99
    back = vi.CpuIndexIVFPQ(d, nlist, M, 8)
    gpu.copyTo(back)
    c2, p2 = back.codebooks()
    assert np.array_equal(c2, coarse) and np.array_equal(p2, pq) and back.ntotal == len(xb)
    for l in range(nlist):
        i0, k0 = ref.get_list(l)
        i1, k1 = back.get_list(l)
        assert np.array_equal(i0, i1) and np.array_equal(k0, k1)


@pytest.mark.gpu
@pytest.mark.parametrize("d,nbc,M", [(64, 5, 8), (128, 6, 16)])
def test_gpu_imipq_matches_reference_imipq(cuda, oracle, d, nbc, M):
    """f3: GpuIndexIMIPQ with the codebooks of the UNMODIFIED reference IMI-PQ index (MultiIndexQuantizer(d, 2, nbc) +
    IndexIVFPQ, tests/sift1b_imi_pq.cpp:216-236, trained and filled on the CPU) returns the reference's cells
    (MultiIndexQuantizer::search, IndexPQ.cpp:804-857; oracle restatement vlqo_imi_search) and the reference's
    search results (IndexIVFPQ::search, full squared distances)"""
    if not oracle.ref_available():
        pytest.skip("reference library not built")
    from vector_line_quantization_b200 import data, index as vi

    k = 10
    xt = data.sift_like(20000, d=d, kc=256, seed=71)
    xb = data.sift_like(30000, d=d, kc=256, seed=72)
    xq = data.sift_like(150, d=d, kc=256, seed=73)
    ref = oracle.RefIMIPQ(d, nbc, M)
    ref.train(xt)
    ref.add(xb)
    coarse, pq = ref.codebooks()
    res = vi.StandardGpuResources(0)
    gpu = vi.GpuIndexIMIPQ(res, d, nbc, M)
    gpu.setCodebooks(coarse, pq)
    gpu.add(xb)
    assert gpu.ntotal == len(xb)
    K = 1 << nbc
    # ---- coarse cells against the reference MultiIndexQuantizer and the oracle restatement
    for nprobe in (1, 16, 100):
        Dc, Ic = gpu.searchCells(xq, nprobe)
        Dm, Im = oracle.ref_imi_search(xq, coarse, nprobe)
        Do, Io = oracle.imi_search(xq, coarse, nprobe)
        assert np.allclose(Dc, Do, rtol=1e-4) and np.all(np.diff(Dc, axis=1) >= 0)
        for r in range(len(xq)):  # same cell SETS up to near-ties at the boundary (the reference may repeat a cell)
            got, want = set(Ic[r].tolist()), set(Io[r].tolist())
            assert len(got) == nprobe and all(0 <= c < K * K for c in got)
            for c in got ^ want:  # a cell only one side has must tie with the boundary distance
                i1, i2 = c % K, c // K
                dc = ((xq[r, : d // 2].astype(np.float64) - coarse[0, i1]) ** 2).sum() + \
                     ((xq[r, d // 2:].astype(np.float64) - coarse[1, i2]) ** 2).sum()
                assert abs(dc - Do[r, -1]) <= 1e-5 * abs(Do[r, -1]) + 1e-3
        assert np.mean([len(set(a) & set(b)) / len(set(b)) for a, b in zip(Ic, Im)]) > 0.99
    # ---- the lists hold what the reference's lists hold (sizes per cell; coarse near-ties may move a vector)
    _, c1 = gpu.searchCells(xb[:2000], 1)
    assert sum(gpu.getListLength(int(c)) > 0 for c in np.unique(c1)) == len(np.unique(c1))
    # ---- end to end: IndexIVFPQ::search of the reference with nprobe cells
    for nprobe in (8, 64):
        Dr, Ir = ref.search(xq, k, nprobe)
        gpu.setNumProbes(nprobe)
        D, I = gpu.search(xq, k)
        same = I == Ir
        assert same.mean() > 0.97
        np.testing.assert_allclose(D[same], Dr[same], rtol=2e-4)
        assert np.mean([len(set(a) & set(b)) / k for a, b in zip(I, Ir)]) > 0.99


@pytest.mark.gpu
def test_gpu_imipq_trains_on_the_device(cuda):
    """GpuIndexIMIPQ::train (two half k-means + PQ on the residuals, all on the device): a usable index"""
    from vector_line_quantization_b200 import data, index as vi

    d, nbc, M, k = 64, 5, 8, 10
    xt = data.sift_like(20000, d=d, kc=256, seed=81)
    xb = data.sift_like(20000, d=d, kc=256, seed=82)
    res = vi.StandardGpuResources(0)
    gpu = vi.GpuIndexIMIPQ(res, d, nbc, M)
    gpu.train(xt)
    gpu.add(xb)
    gpu.setNumProbes(64)
    D, I = gpu.search(xb[:200], k)  # database vectors as queries: they find themselves
    assert np.mean(I[:, 0] == np.arange(200)) > 0.9 and np.all(np.diff(D, axis=1) >= 0)
