"""4-bit PQ codes on the device (include/vlq_b200.h, "4-bit PQ codes"): encode, pair tables, every scan kernel, range,
filter, removal, read-back, the faiss container exchange and the .db* files, against the oracle (which takes any ksub
with one byte per code, so it is the reference once the packed codes are unpacked) and against the 8-bit kernels.
Geometries: d in {96, 128} x M in {16, 32}, lists of ~117 entries so that the long-list kernels run too."""
import numpy as np
import pytest

from tests.parity_util import REL_TIE, Model64, check_encode, check_lines, check_topk

pytestmark = pytest.mark.gpu

GEOMS = [(128, 16), (128, 32), (96, 16), (96, 32)]  # (d, M): M / 2 = 8 or 16 stored bytes per entry
NLIST, E, NL = 64, 8, 64


def T(a, dev):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def N(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def ops(cuda):
    from vector_line_quantization_b200 import ops as _ops

    return _ops


_models = {}


def model(oracle, d, M):
    """oracle-trained 4-bit model (ProductQuantizer(d, M, 4) on the first 16 * 128 rows) + base + queries"""
    if (d, M) not in _models:
        from vector_line_quantization_b200 import data

        gen = data.sift_like if d == 128 else data.deep_like
        seed = 7 * d + M
        xt = gen(6000, d=d, kc=128, seed=seed)
        m = oracle.train_all(xt, nlist=NLIST, E=E, M=M, nL=NL, nbits=4, niter=5, pq_niter=8)
        assert m["pq"].shape == (M, 16, d // M)
        m.update(xb=gen(60000, d=d, kc=128, seed=seed + 1), xq=gen(40, d=d, kc=128, seed=seed + 2), d=d, C=NLIST, E=E,
                 M=M)
        _models[(d, M)] = m
    return _models[(d, M)]


_indexes = {}


def device_index(ops, cuda, oracle, d, M):
    """device encode (4-bit) + list build; the oracle gets the same entries with their codes unpacked"""
    import torch

    if (d, M) in _indexes:
        return _indexes[(d, M)]
    m = model(oracle, d, M)
    cent = T(m["cent"], cuda)
    cn = ops.row_norms(cent)
    edge, ed2, lcb, pq = T(m["edge"], cuda), T(m["edge_d2"], cuda), T(m["lambda_cb"], cuda), T(m["pq"], cuda)
    x = T(m["xb"], cuda)
    A, _ = ops.l2_assign(x, cent, cn)
    enc = ops.line_encode(x, A, cent, edge, ed2, lcb, pq, want_residual=True)
    assert enc.codes.shape == (x.shape[0], M // 2)
    nl = NLIST * E
    lists = ops.build_lists(nl, M // 2, enc.list, enc.codes, enc.lamq, enc.kappa,
                            torch.arange(x.shape[0], dtype=torch.int64, device=cuda))
    e_list, e_lamq, e_codes = N(enc.list), N(enc.lamq), N(ops.unpack_pq4(enc.codes))
    off, perm = oracle.build_lists(e_list, nl)
    assert np.array_equal(N(lists.offsets), off) and np.array_equal(N(lists.ids), perm)
    gi = dict(cent=cent, cn=cn, edge=edge, ed2=ed2, lcb=lcb, pq=pq, lists=lists, enc=enc, A=N(A), e_list=e_list,
              e_lamq=e_lamq, e_codes=e_codes, off=off, perm=perm, m64=Model64(m))
    _indexes[(d, M)] = gi
    return gi


@pytest.mark.parametrize("d,M", GEOMS)
def test_encode_vs_oracle(ops, cuda, oracle, d, M):
    m = model(oracle, d, M)
    gi = device_index(ops, cuda, oracle, d, M)
    enc = gi["enc"]
    x = m["xb"]
    o = oracle.encode_all(x, m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    # unpacked codes, lambda bytes and lists identical except near-ties, each verified in float64
    same = check_encode(enc._replace(codes=ops.unpack_pq4(enc.codes)), o, x, m)
    # the packing is byte-exact: byte j = code[2j] | code[2j + 1] << 4 of the oracle's codes
    rows = same & (gi["e_codes"] == o["codes"]).all(1)
    c = o["codes"][rows].astype(np.uint8)
    assert np.array_equal(N(enc.codes)[rows], c[:, 0::2] | (c[:, 1::2] << 4))
    # kappa = ||p||^2 + 2 anchor.p within 1e-4 relative (float64 from the device's own line, lambda and codes)
    lst, lq = gi["e_list"], gi["e_lamq"]
    c64 = m["cent"].astype(np.float64)
    lh = m["lambda_cb"].astype(np.float64)[lq][:, None]
    anchor = (1 - lh) * c64[lst // E] + lh * c64[m["edge"][lst // E, lst % E]]
    p = np.concatenate([m["pq"][mm].astype(np.float64)[gi["e_codes"][:, mm]] for mm in range(M)], axis=1)
    k64 = (p * p).sum(1) + 2 * (anchor * p).sum(1)
    kap = N(enc.kappa)
    assert np.all(np.abs(kap - k64) <= 1e-4 * (np.abs(k64) + (p * p).sum(1) + 1e-6))


def _lines(ops, cuda, m, gi, P, W, route):
    import torch

    q = T(m["xq"], cuda)
    if route == "tc":
        pack = ops.CentPack(gi["cent"], gi["cn"])
        bm = torch.empty((q.shape[0], ops.num_buckets(NLIST)), dtype=torch.float32, device=cuda)
        D = ops.l2_distances_tc(q, pack, bucket_min=bm)
        lst, t1, t6 = ops.coarse_select_lines(D, bm, NLIST, P, gi["edge"], gi["ed2"], W)
    else:
        D = ops.l2_distances(q, gi["cent"], gi["cn"])
        _, cid = ops.select_rows(D, P)
        lst, t1, t6 = ops.select_lines(D, cid, gi["edge"], gi["ed2"], W)
    return q, lst, t1, t6


def _tables(ops, q, nq, Mb):
    import torch

    torch.cuda.synchronize()
    ws = ops._scan_ws[q.device]
    return N(ws[: nq * Mb * 256 * 4].view(torch.float32)).reshape(nq, -1).copy()


@pytest.mark.parametrize("d,M", GEOMS)
def test_pair_tables_bit_exact_in_both_layouts(ops, cuda, oracle, d, M):
    """T3'[m'][b] = T3[2m'][b & 15] + T3[2m'+1][b >> 4] in fp32, bit for bit.  The 16-entry tables T3 come from the
    8-bit table kernel run on a 256-entry codebook whose codeword j is 4-bit codeword j & 15 (same fmaf chain)."""
    import torch

    m = model(oracle, d, M)
    gi = device_index(ops, cuda, oracle, d, M)
    Mb = M // 2
    q, lst, t1, t6 = _lines(ops, cuda, m, gi, 8, 64, "simt")
    nq = q.shape[0]
    ed2f = gi["ed2"].reshape(-1)
    pq8 = gi["pq"][:, torch.arange(256, device=cuda) & 15].contiguous()
    ops.scan_topk(q, pq8, gi["lcb"], lst, t1, t6, ed2f, ops.Lists(gi["lists"].offsets, torch.zeros(
        (gi["lists"].ids.shape[0], M), dtype=torch.uint8, device=cuda), *gi["lists"][2:]), 10, list_len_hint=0)
    t16 = _tables(ops, q, nq, M).reshape(nq, M, 256)[:, :, :16]
    b = np.arange(256)
    want = (t16[:, 0::2][:, :, b & 15] + t16[:, 1::2][:, :, b >> 4]).astype(np.float32)  # [nq][Mb][256]
    ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], 10, list_len_hint=0)  # row-major tables
    assert np.array_equal(_tables(ops, q, nq, Mb).reshape(nq, Mb, 256).view(np.uint32), want.view(np.uint32))
    ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], 10, list_len_hint=100)  # bank-skewed: code-major
    assert np.array_equal(_tables(ops, q, nq, Mb).reshape(nq, 256, Mb).view(np.uint32),
                          want.transpose(0, 2, 1).view(np.uint32))


def _oracle_scan(oracle, m, gi, lines, k, cap=1024):
    perm = gi["perm"]
    return oracle.scan_lines(m["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], gi["off"],
                             gi["e_codes"][perm], gi["e_lamq"][perm], perm.astype(np.int64), lines, k, cap)


@pytest.mark.parametrize("route", ["simt", "tc"])
@pytest.mark.parametrize("d,M", GEOMS)
def test_search_vs_oracle_every_scan_kernel(ops, cuda, oracle, monkeypatch, d, M, route):
    from vector_line_quantization_b200 import _abi

    m = model(oracle, d, M)
    gi = device_index(ops, cuda, oracle, d, M)
    perm = gi["perm"]
    ed2f = gi["ed2"].reshape(-1)
    ent = (m["xq"], gi["m64"], gi["e_list"], gi["e_lamq"], gi["e_codes"])
    for P, W, k, cap in ((16, 64, 100, 1024), (8, 32, 10, 50), (32, 128, 200, 1024)):
        Do, Io, _, lines_ref, _ = oracle.search(m["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"],
                                                gi["off"], gi["e_codes"][perm], gi["e_lamq"][perm], perm.astype(np.int64),
                                                P=P, W=W, k=k, cap=cap, want_debug=True)
        q, lst, t1, t6 = _lines(ops, cuda, m, gi, P, W, route)
        same_lines = check_lines(N(lst), lines_ref, m["xq"], gi["m64"])
        Dl, Il = _oracle_scan(oracle, m, gi, N(lst), k, cap)
        # hint 0: short-list kernel (+ general flattened kernel for longer queries); 30: warp-autonomous (k <= 128) or
        # warp-per-list; 100: bank-skewed; 400: the long-list kernel of scan_long.cu
        for hint in (0, 30, 100, 400):
            D, I = ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], k, cap, list_len_hint=hint)
            check_topk(N(D), N(I), Dl, Il, *ent)
            check_topk(N(D), N(I), Do, Io, *ent, same_lines)
        monkeypatch.setenv("VLQ_SCAN_NO_SMALL", "1")  # every short query through the general kernel
        D, I = ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], k, cap, list_len_hint=0)
        monkeypatch.delenv("VLQ_SCAN_NO_SMALL")
        check_topk(N(D), N(I), Dl, Il, *ent)
        # the 4-bit scan has no in-kernel table build
        with pytest.raises(_abi.VlqError):
            ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], k, cap, use_workspace=False)


@pytest.mark.parametrize("d,M", GEOMS[:2])
def test_filter_all_selected_is_bit_identical(ops, cuda, oracle, d, M):
    m = model(oracle, d, M)
    gi = device_index(ops, cuda, oracle, d, M)
    q, lst, t1, t6 = _lines(ops, cuda, m, gi, 16, 64, "simt")
    ed2f = gi["ed2"].reshape(-1)
    kap = ops.filter_kappa(gi["lists"], id_range=(0, len(m["xb"])))
    for hint in (0, 100, 400):
        D0, I0 = ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], 50, list_len_hint=hint)
        D1, I1 = ops.scan_topk(q, gi["pq"], gi["lcb"], lst, t1, t6, ed2f, gi["lists"], 50, list_len_hint=hint, kappa=kap)
        assert np.array_equal(N(D0).view(np.uint32), N(D1).view(np.uint32)) and np.array_equal(N(I0), N(I1))


@pytest.mark.parametrize("d,M", GEOMS)
def test_range_scan_vs_float64_candidates(ops, cuda, oracle, d, M):
    """every entry of the scanned lines below the radius, in stream order; entries within REL_TIE of the radius may go
    either way"""
    from tests.parity_util import scan_candidates

    m = model(oracle, d, M)
    gi = device_index(ops, cuda, oracle, d, M)
    q, lst, t1, t6 = _lines(ops, cuda, m, gi, 8, 32, "simt")
    qn = ops.row_norms(q)
    L = gi["lists"]
    canon = gi["e_codes"][N(L.ids)]  # list-major, canonical order
    cands = scan_candidates(m["xq"], N(lst), N(t1), N(t6), N(gi["ed2"]).reshape(-1), m["lambda_cb"], m["pq"],
                            N(L.offsets), canon, N(L.lamq), N(L.kappa), N(L.ids), 1024)
    qn64 = (m["xq"].astype(np.float64) ** 2).sum(1)
    radius = float(np.median([np.median(dc + qn64[i]) for i, (dc, _) in enumerate(cands)]))
    lims, D, I = ops.range_scan_lines(q, gi["pq"], gi["lcb"], (lst, t1, t6), gi["ed2"], L, radius, row_add=qn)
    lims, D, I = N(lims), N(D), N(I)
    for i, (dc, ic) in enumerate(cands):
        got = I[lims[i]:lims[i + 1]]
        full = dc + qn64[i]
        tie = np.abs(full - radius) <= REL_TIE * (np.abs(full) + qn64[i])
        want = ic[(full < radius) & ~tie]
        assert np.array_equal(got[~np.isin(got, ic[tie])], want), i
        assert np.all(D[lims[i]:lims[i + 1]] < radius)


# ------------------------------------------------------------------------------------------------ the index class
def _gpu_index(m, d, M, res):
    from vector_line_quantization_b200 import index as vi

    g = vi.GpuIndexIVFPQ(res, d, NLIST, M, 4, E, NL)
    g.setCodebooks(m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    g.setNumProbes(16)
    g.w1_ = 64
    return g


@pytest.fixture(scope="module")
def res(cuda):
    from vector_line_quantization_b200 import index as vi

    return vi.StandardGpuResources(0)


@pytest.mark.parametrize("d,M", [(128, 32), (96, 16)])
def test_index_remove_readback_and_files(ops, cuda, oracle, res, tmp_path, d, M):
    from vector_line_quantization_b200 import index as vi

    m = model(oracle, d, M)
    xb, xq = m["xb"][:20000], m["xq"]
    ids = np.arange(len(xb), dtype=np.int64)
    g = _gpu_index(m, d, M, res)
    g.add_with_ids(xb, ids)
    D, I = g.search(xq, 20)
    # search through GpuIndexIVFPQ equals the oracle's search of the same entries (read back one byte per code)
    nl = NLIST * E
    off, codes, las, lids = [0], [], [], []
    for l in range(nl):
        c, la, i = g.getList(l)
        assert c.shape[1] == M and (c < 16).all()
        codes.append(c), las.append(la), lids.append(i)
        off.append(off[-1] + len(i))
    codes, las, lids = np.concatenate(codes), np.concatenate(las), np.concatenate(lids)
    Do, Io = oracle.search(xq, m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], np.array(off), codes, las,
                           lids, P=16, W=64, k=20)
    e_list = np.empty(len(xb), np.int64)
    e_list[lids] = np.repeat(np.arange(nl), np.diff(off))
    e_lamq, e_codes = np.empty_like(las), np.empty_like(codes)
    e_lamq[lids], e_codes[lids] = las, codes
    # every returned distance is the float64 decode distance of its entry; the sets agree with the oracle's search up to
    # line choices at the W boundary (near-ties there are common: both directions of an edge score alike)
    check_topk(D, I, D, I, xq, Model64(m), e_list, e_lamq, e_codes)
    assert np.mean([len(set(a) & set(b)) / 20 for a, b in zip(I, Io)]) > 0.95
    # reconstruct_n: the oracle decode of the unpacked codes, (1 - l) c + l s + p in fp32 as written
    R = g.reconstruct_n(0, len(xb))
    c32 = m["cent"]
    lh = m["lambda_cb"][e_lamq][:, None].astype(np.float32)
    anc = (np.float32(1) - lh) * c32[e_list // E] + lh * c32[m["edge"][e_list // E, e_list % E]]
    p = np.concatenate([m["pq"][mm][e_codes[:, mm]] for mm in range(M)], axis=1)
    assert np.array_equal((anc + p).view(np.uint32), np.asarray(R).view(np.uint32))
    D2, I2, R2 = g.search_and_reconstruct(xq, 20)
    assert np.array_equal(np.asarray(D2).view(np.uint32), D.view(np.uint32)) and np.array_equal(I2, I)
    assert np.array_equal(np.asarray(R2)[I >= 0], np.asarray(R)[I[I >= 0]])
    # remove_ids(S) == an index that never received S
    S = (5000, 12000)
    h = _gpu_index(m, d, M, res)
    keep = (ids < S[0]) | (ids >= S[1])
    h.add_with_ids(xb[keep], ids[keep])
    assert g.remove_ids(vi.IDSelectorRange(*S)) == S[1] - S[0]
    for l in range(0, nl, 7):
        for a, b in zip(g.getList(l), h.getList(l)):
            assert np.array_equal(a, b)
    Dg, Ig = g.search(xq, 20)
    Dh, Ih = h.search(xq, 20)
    assert np.array_equal(Dg.view(np.uint32), Dh.view(np.uint32)) and np.array_equal(Ig, Ih)
    # .db* files: one byte per code on disk; a fresh index reads them back to the same lists and results
    name = str(tmp_path / "pq4")
    g.writeCodebookToFile(name)
    g.writeDbToFile(name)
    assert (tmp_path / "pq4.dbcodes").stat().st_size == g.ntotal * M
    f = vi.GpuIndexIVFPQ(res, d, NLIST, M, 4, E, NL)
    f.readCodebookFromFile(name)
    f.readDbFromFile(name)
    f.setNumProbes(16)
    f.w1_ = 64
    for l in range(0, nl, 7):
        for a, b in zip(g.getList(l), f.getList(l)):
            assert np.array_equal(a, b)
    Df, If = f.search(xq, 20)
    assert np.array_equal(Df.view(np.uint32), Dg.view(np.uint32)) and np.array_equal(If, Ig)


def test_copy_from_and_to_a_4_bit_container(cuda, oracle, res):
    from vector_line_quantization_b200 import index as vi

    d, nlist, M, nedge = 64, 32, 16, 4
    rng = np.random.default_rng(3)
    coarse = rng.standard_normal((nlist, d)).astype(np.float32)
    pq = rng.standard_normal((M, 16, d // M)).astype(np.float32)
    cpu = vi.CpuIndexIVFPQ(d, nlist, M, 4)
    cpu.set_codebooks(coarse, pq)
    nid = 0
    for l in range(nlist):
        n = int(rng.integers(0, 40))
        cpu.set_list(l, np.arange(nid, nid + n), rng.integers(0, 16, (n, M), dtype=np.uint8))
        nid += n
    gpu = vi.GpuIndexIVFPQ(res, d, nlist, M, 4, nedge, 16)
    gpu.copyFrom(cpu)
    assert gpu.ntotal == nid
    back = vi.CpuIndexIVFPQ(d, nlist, M, 4)
    gpu.copyTo(back)
    c2, p2 = back.codebooks()
    assert np.array_equal(c2, coarse) and np.array_equal(p2, pq) and back.ntotal == nid
    for l in range(nlist):
        for a, b in zip(cpu.get_list(l), back.get_list(l)):
            assert np.array_equal(a, b)
    with pytest.raises(vi.FaissException):  # an 8-bit container does not fit a 4-bit index
        gpu.copyFrom(vi.CpuIndexIVFPQ(d, nlist, M, 8))


def test_copy_from_reference_4_bit_ivfpq(cuda, oracle, res):
    """copyFrom of the reference's own IndexIVFPQ(nbits = 4), then search: what the reference's search returns"""
    if not oracle.ref_available():
        pytest.skip("reference library not built")
    from vector_line_quantization_b200 import data, index as vi

    d, nlist, M, k, nprobe, nedge = 64, 64, 16, 10, 8, 4
    xt = data.sift_like(20000, d=d, kc=256, seed=1)
    xb = data.sift_like(30000, d=d, kc=256, seed=2)
    xq = data.sift_like(200, d=d, kc=256, seed=3)
    ref = oracle.RefIVFPQ(d, nlist, M, 4)
    ref.train(xt)
    ref.add(xb)
    Dr, Ir = ref.search(xq, k, nprobe)
    coarse, pq = ref.codebooks()
    cpu = vi.CpuIndexIVFPQ(d, nlist, M, 4)
    cpu.set_codebooks(coarse, pq)
    for l in range(nlist):
        cpu.set_list(l, *ref.get_list(l))
    gpu = vi.GpuIndexIVFPQ(res, d, nlist, M, 4, nedge, 16)
    gpu.copyFrom(cpu)
    gpu.setNumProbes(nprobe)
    gpu.w1_ = nprobe * nedge
    gpu.setListCap(1 << 20)
    D, I = gpu.search(xq, k)
    qn = (xq.astype(np.float64) ** 2).sum(1, keepdims=True)
    same = I == Ir
    assert same.mean() > 0.97
    np.testing.assert_allclose((D + qn)[same], Dr[same], rtol=2e-4)


def test_train_4_bit_index_on_the_device(cuda, res):
    """GpuIndexIVFPQ(bits = 4).train: ProductQuantizer(d, M, 4) on the first min(n, 16 * 128) rows, then add + search"""
    from vector_line_quantization_b200 import data, index as vi

    d, nlist, M = 64, 32, 16
    xt = data.sift_like(8000, d=d, kc=64, seed=11)
    g = vi.GpuIndexIVFPQ(res, d, nlist, M, 4, 4, 16)
    g.train(xt)
    assert g.codebooks()["pq"].shape == (M, 16, d // M)
    g.add(xt)
    g.setNumProbes(8)
    g.w1_ = 32
    D, I = g.search(xt[:50], 10)
    assert (I >= 0).all() and np.all(np.diff(D, axis=1) >= 0)
    assert np.mean([i in row for i, row in enumerate(I)]) > 0.8  # a stored vector finds itself
