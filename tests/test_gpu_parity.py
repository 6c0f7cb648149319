"""Parity of the CUDA path (through the C-ABI, lib/libvlq_b200.so) against the CPU oracle and the golden fixtures.

Bars (north_star): list / lambda / PQ codes identical except documented near-ties (relative distance gap < 1e-5);
top-k distances within 1e-4 relative; integer / index work (list build, merge, select indices) bit-exact.
"""
import os

import numpy as np
import pytest

from tests.parity_util import check_encode

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vlq_small.npz")
REL_TIE = 1e-5
REL_DIST = 1e-4


def T(a, dev, dtype=None):
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t if dtype is None else t.to(dtype)


def N(t):
    return t.detach().cpu().numpy()


def near_tie_rows(ids_a, ids_b, x, cent, rel=REL_TIE):
    bad = np.nonzero(ids_a != ids_b)[0]
    for i in bad:
        da = np.sum((x[i].astype(np.float64) - cent[ids_a[i]]) ** 2)
        db = np.sum((x[i].astype(np.float64) - cent[ids_b[i]]) ** 2)
        assert abs(da - db) <= rel * max(da, db) + 1e-9, (int(i), da, db)
    return len(bad)


@pytest.fixture(scope="module")
def ops(cuda):
    from vector_line_quantization_b200 import ops as _ops

    return _ops


@pytest.fixture(scope="module")
def g():
    return dict(np.load(GOLD))


# ------------------------------------------------------------------------------------------------ assignment (a1,a2)
@pytest.mark.parametrize("n,d,C", [(1, 128, 7), (127, 128, 256), (1000, 96, 300), (4099, 128, 1024), (513, 20, 33),
                                   (300, 1, 16)])
def test_l2_assign_matches_oracle(ops, cuda, oracle, n, d, C):
    rng = np.random.RandomState(n + d + C)
    x = rng.normal(0, 30, (n, d)).astype(np.float32)
    cent = rng.normal(0, 30, (C, d)).astype(np.float32)
    ids, dist = ops.l2_assign(T(x, cuda), T(cent, cuda), add_xnorm=True)
    Do, Io = oracle.l2_topk(x, cent, 1, add_xnorm=True)
    ids, dist = N(ids), N(dist)
    nbad = near_tie_rows(ids, Io[:, 0], x, cent)
    assert nbad <= max(1, n // 1000)
    ok = ids == Io[:, 0]
    scale = np.sum(x.astype(np.float64) ** 2, axis=1)[ok] + 1.0
    assert np.all(np.abs(dist[ok] - Do[ok, 0]) <= REL_DIST * scale)
    cn = N(ops.row_norms(T(cent, cuda)))
    np.testing.assert_allclose(cn, np.sum(cent.astype(np.float64) ** 2, axis=1), rtol=1e-5)


def test_l2_assign_empty(ops, cuda):
    import torch

    x = torch.empty((0, 64), dtype=torch.float32, device=cuda)
    cent = torch.randn((10, 64), device=cuda)
    ids, dist = ops.l2_assign(x, cent)
    assert ids.shape[0] == 0


def test_l2_assign_golden(ops, cuda, g):
    xb = g["xb"].astype(np.float32)
    ids, dist = ops.l2_assign(T(xb, cuda), T(g["cent"], cuda))
    assert near_tie_rows(N(ids), g["A"], xb, g["cent"]) <= 1
    assert near_tie_rows(N(ids), g["ref_flat_assign_I"], xb, g["cent"]) <= 2  # vs the reference's IndexFlatL2


# ------------------------------------------------------------------------------------------------ select (a11, a15)
@pytest.mark.parametrize("n,cols,k", [(5, 10, 1), (37, 1000, 10), (16, 30000, 100), (9, 5000, 1024), (4, 50, 128),
                                      (3, 1, 1)])
def test_select_rows_exact(ops, cuda, n, cols, k):
    """TestGpuSelect.cu:28-187 protocol: values equal the sorted prefix exactly; indices valid and distinct"""
    rng = np.random.RandomState(cols + k)
    D = np.round(rng.rand(n, cols), 3).astype(np.float32)  # 1000 distinct values: plenty of ties
    val, idx = ops.select_rows(T(D, cuda), k)
    val, idx = N(val), N(idx)
    kk = min(k, cols)
    want_order = np.lexsort((np.broadcast_to(np.arange(cols), D.shape), D), axis=1)[:, :kk]
    want = np.take_along_axis(D, want_order, 1)
    assert np.array_equal(val[:, :kk], want)
    assert np.array_equal(idx[:, :kk], want_order)  # our select is deterministic: lowest index on ties
    if k > cols:
        assert np.all(idx[:, cols:] == -1) and np.all(val[:, cols:] == np.finfo(np.float32).max)


def test_coarse_topP_matches_oracle(ops, cuda, oracle, small_model):
    m = small_model
    D = ops.l2_distances(T(m["xq"], cuda), T(m["cent"], cuda))
    val, idx = ops.select_rows(D, 32)
    Do, Io = oracle.l2_topk(m["xq"], m["cent"], 32, add_xnorm=False)
    assert (N(idx) == Io).mean() > 0.995
    scale = np.sum(m["xq"].astype(np.float64) ** 2, axis=1, keepdims=True)
    assert np.all(np.abs(N(val) - Do) <= REL_DIST * scale)


# ------------------------------------------------------------------------------------------------ graph (a4)
def test_knn_graph_matches_oracle(ops, cuda, oracle, small_model, g):
    for cent, E in [(small_model["cent"], 32), (g["cent"], int(g["E"]))]:
        edge, ed2 = ops.knn_graph(T(cent, cuda), E)
        eo, do = oracle.knn_graph(cent, E)
        edge, ed2 = N(edge), N(ed2)
        assert (edge == eo).mean() > 0.999
        same = edge == eo
        np.testing.assert_allclose(ed2[same], do[same], rtol=1e-4, atol=1e-2)
        # mismatches must be distance ties
        for c, e in np.argwhere(~same):
            assert abs(ed2[c, e] - do[c, e]) <= 1e-5 * abs(do[c, e]) + 1e-3
    # the fixture's graph (the loop's last case) against the reference's IndexFlatL2 search of the centroids against
    # themselves, stored in the fixture (column 0 is the centroid itself)
    assert (edge == g["ref_graph_I"][:, 1:]).mean() > 0.995
    np.testing.assert_allclose(ed2, g["ref_graph_D"][:, 1:], rtol=1e-3, atol=1e-2)


# ------------------------------------------------------------------------------------------------ encode (a5-a8)
def _encode_both(ops, cuda, oracle, x, m, use_oracle_assign=True):
    _, A = oracle.l2_topk(x, m["cent"], 1)
    A = A[:, 0].copy()
    enc = ops.line_encode(T(x, cuda), T(A, cuda), T(m["cent"], cuda), T(m["edge"], cuda), T(m["edge_d2"], cuda),
                          T(m["lambda_cb"], cuda), T(m["pq"], cuda), want_residual=True)
    lst, lam = oracle.line_stage(x, A, m["cent"], m["edge"], m["edge_d2"])
    lamq = oracle.lambda_quantize(lam, m["lambda_cb"])
    r = oracle.residual(x, lst, lamq, m["lambda_cb"], m["cent"], m["edge"])
    codes = oracle.pq_encode(r, m["pq"])
    return enc, dict(A=A, list=lst, lam=lam, lamq=lamq, residual=r, codes=codes)


def test_line_encode_matches_oracle(ops, cuda, oracle, small_model):
    m = small_model
    x = m["xb"][:7001]  # ragged: not a multiple of the CTA's 16 warps
    enc, o = _encode_both(ops, cuda, oracle, x, m)
    same = check_encode(enc, o, x, m)
    # kappa = ||p||^2 + 2 anchor.p  (DESIGN.md): check against float64
    kap = N(enc.kappa)
    E, M = m["E"], m["M"]
    dsub = 128 // M
    for i in np.nonzero(same)[0][::501]:
        l = o["list"][i]
        c, s = m["cent"][l // E].astype(np.float64), m["cent"][m["edge"][l // E, l % E]].astype(np.float64)
        lh = float(m["lambda_cb"][o["lamq"][i]])
        anchor = (1 - lh) * c + lh * s
        p = np.concatenate([m["pq"][mm, o["codes"][i, mm]] for mm in range(M)]).astype(np.float64)
        want = np.dot(p, p) + 2 * np.dot(anchor, p)
        assert abs(kap[i] - want) <= 1e-5 * (abs(want) + np.linalg.norm(anchor) * np.linalg.norm(p))


def test_line_encode_golden(ops, cuda, g):
    xb = g["xb"].astype(np.float32)
    enc = ops.line_encode(T(xb, cuda), T(g["A"], cuda), T(g["cent"], cuda), T(g["edge"], cuda), T(g["edge_d2"], cuda),
                          T(g["lambda_cb"], cuda), T(g["pq"], cuda))
    assert (N(enc.list) == g["list"]).mean() > 0.999
    ok = N(enc.list) == g["list"]
    assert (N(enc.lamq)[ok] == g["lamq"][ok]).mean() > 0.998
    ok &= N(enc.lamq) == g["lamq"]
    assert (N(enc.codes)[ok] == g["codes"][ok]).mean() > 0.9995
    assert (N(enc.codes)[ok] == g["ref_pq_codes"][ok]).mean() > 0.998  # the reference's ProductQuantizer::compute_codes


def test_line_stage_only_mode(ops, cuda, oracle, small_model):
    m = small_model
    x = m["xt"][:2000]
    _, A = oracle.l2_topk(x, m["cent"], 1)
    A = A[:, 0].copy()
    enc = ops.line_encode(T(x, cuda), T(A, cuda), T(m["cent"], cuda), T(m["edge"], cuda), T(m["edge_d2"], cuda))
    lst, lam = oracle.line_stage(x, A, m["cent"], m["edge"], m["edge_d2"])
    ok = N(enc.list) == lst
    assert ok.mean() > 0.999
    np.testing.assert_allclose(N(enc.lam)[ok], lam[ok], rtol=1e-3, atol=1e-4)


def test_line_encode_d96_m8_e64(ops, cuda, oracle):
    """DEEP-shaped geometry and the 64-edge graphs of the 1B drivers (SURVEY Q1: the reference kernel is wrong there)"""
    from vector_line_quantization_b200 import data

    xt = data.deep_like(6000, kc=256, seed=5)
    m = oracle.train_all(xt, nlist=128, E=64, M=8, nL=256, niter=5, pq_niter=5)
    x = data.deep_like(3000, kc=256, seed=6)
    enc, o = _encode_both(ops, cuda, oracle, x, m)
    check_encode(enc, o, x, m)


# ------------------------------------------------------------------------------------------------ lists (a9)
def test_build_lists_exact(ops, cuda, oracle):
    import torch

    rng = np.random.RandomState(4)
    nlists, M, n1, n2 = 777, 16, 5000, 3001
    lst = rng.randint(0, nlists, n1 + n2).astype(np.int32)
    lst[rng.rand(n1 + n2) < 0.3] = 5  # one long list (> 2048 entries: global-memory sort path)
    lst[::97] = -1  # invalid vectors are skipped (GpuIndexIVFPQ.cu:751-755)
    codes = rng.randint(0, 256, (n1 + n2, M)).astype(np.uint8)
    lamq = rng.randint(0, 256, n1 + n2).astype(np.uint8)
    kappa = rng.rand(n1 + n2).astype(np.float32)
    ids = (np.arange(n1 + n2) * 3 + 1).astype(np.int64)

    def build(sl, old):
        return ops.build_lists(nlists, M, T(lst[sl], cuda), T(codes[sl], cuda), T(lamq[sl], cuda), T(kappa[sl], cuda),
                               T(ids[sl], cuda), old)

    l1 = build(slice(0, n1), None)
    l2 = build(slice(n1, n1 + n2), l1)
    torch.cuda.synchronize()
    valid = lst >= 0
    offsets, perm = oracle.build_lists(lst[valid], nlists)
    src = np.nonzero(valid)[0][perm]
    nv = int(valid.sum())
    assert np.array_equal(N(l2.offsets), offsets)
    assert np.array_equal(N(l2.ids)[:nv], ids[src])
    assert np.array_equal(N(ops.rotate_codes(l2.offsets, l2.codes, inverse=True))[:nv], codes[src])  # stored rotated
    pos = np.arange(nv) - np.repeat(offsets[:-1], np.diff(offsets))  # position inside the list
    want = np.take_along_axis(codes[src], (np.arange(M)[None, :] + pos[:, None]) % M, axis=1)
    assert np.array_equal(N(l2.codes)[:nv], want)  # stored[j] = code[(j + pos) mod M]
    assert np.array_equal(N(l2.lamq)[:nv], lamq[src])
    assert np.array_equal(N(l2.kappa)[:nv], kappa[src])


def test_build_lists_empty_add(ops, cuda):
    import torch

    e = lambda dt, *s: torch.empty(s, dtype=dt, device=cuda)  # noqa: E731
    l = ops.build_lists(10, 8, e(torch.int32, 0), e(torch.uint8, 0, 8), e(torch.uint8, 0), e(torch.float32, 0),
                        e(torch.int64, 0))
    assert N(l.offsets).tolist() == [0] * 11


# ------------------------------------------------------------------------------------------------ search (a11-a15)
def _gpu_index(ops, cuda, oracle, m, xb):
    """encode + list build entirely on the device; returns resident tensors"""
    import torch

    cent = T(m["cent"], cuda)
    cn = ops.row_norms(cent)
    edge, ed2 = T(m["edge"], cuda), T(m["edge_d2"], cuda)
    lcb, pq = T(m["lambda_cb"], cuda), T(m["pq"], cuda)
    x = T(xb, cuda)
    A, _ = ops.l2_assign(x, cent, cn)
    enc = ops.line_encode(x, A, cent, edge, ed2, lcb, pq)
    M = m["pq"].shape[0]
    ids = torch.arange(xb.shape[0], dtype=torch.int64, device=cuda)
    lists = ops.build_lists(m["cent"].shape[0] * m["edge"].shape[1], M, enc.list, enc.codes, enc.lamq, enc.kappa, ids)
    return dict(cent=cent, cn=cn, edge=edge, ed2=ed2, lcb=lcb, pq=pq, lists=lists, enc=enc)


def _oracle_index(oracle, m, lst, lamq, codes):
    nl = m["cent"].shape[0] * m["edge"].shape[1]
    offsets, perm = oracle.build_lists(lst, nl)
    return offsets, codes[perm], lamq[perm], perm.astype(np.int64)


@pytest.mark.parametrize("P,W,k,cap", [(16, 128, 10, 1024), (32, 256, 100, 1024), (8, 1024, 1024, 1024),
                                       (16, 64, 50, 2), (1, 1, 1, 1024)])
def test_search_matches_oracle(ops, cuda, oracle, small_model, P, W, k, cap):
    """same index on both sides: the device-encoded lists are handed to the oracle, so only the query path differs.
    Every id that differs from the oracle's is verified as a near-tie in float64 (tests/parity_util.py); more
    geometries and every scan kernel: tests/test_gpu_search_parity.py"""
    from tests.parity_util import check_lines, check_topk

    m = small_model
    gi = _gpu_index(ops, cuda, oracle, m, m["xb"])
    enc = gi["enc"]
    e_list, e_lamq, e_codes = N(enc.list), N(enc.lamq), N(enc.codes)
    off, codes_l, lamq_l, ids_l = _oracle_index(oracle, m, e_list, e_lamq, e_codes)
    assert np.array_equal(N(gi["lists"].offsets), off) and np.array_equal(N(gi["lists"].ids), ids_l)
    q = T(m["xq"], cuda)
    D, I = ops.search(q, gi["cent"], gi["cn"], gi["edge"], gi["ed2"], gi["lcb"], gi["pq"], gi["lists"], P, W, k, cap)
    Do, Io, _, lines, _ = oracle.search(m["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], off,
                                        codes_l, lamq_l, ids_l, P=P, W=W, k=k, cap=cap, want_debug=True)
    Dm = ops.l2_distances(q, gi["cent"], gi["cn"])
    _, cid = ops.select_rows(Dm, P)
    lst, _, _ = ops.select_lines(Dm, cid, gi["edge"], gi["ed2"], W)
    same_lines = check_lines(N(lst), lines, m["xq"], m)  # differing lines are float64 line-score near-ties
    Dl, Il = oracle.scan_lines(m["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], off, codes_l, lamq_l,
                               ids_l, N(lst), k, cap)
    check_topk(N(D), N(I), Dl, Il, m["xq"], m, e_list, e_lamq, e_codes)  # every query, same line choice
    check_topk(N(D), N(I), Do, Io, m["xq"], m, e_list, e_lamq, e_codes, same_lines)


def test_search_golden(ops, cuda, g):
    import torch

    perm = g["perm"]
    C, E, M = int(g["C"]), int(g["E"]), int(g["M"])
    cent = T(g["cent"], cuda)
    cn = ops.row_norms(cent)
    pqn = g["pq"]
    # kappa for the golden (oracle-encoded) entries, computed here in float64 from the fixture itself
    lst = g["list"][perm]
    c = g["cent"][lst // E].astype(np.float64)
    s = g["cent"][g["edge"][lst // E, lst % E]].astype(np.float64)
    lh = g["lambda_cb"][g["lamq"][perm]].astype(np.float64)[:, None]
    anchor = (1 - lh) * c + lh * s
    p = np.concatenate([pqn[mm][g["codes"][perm][:, mm]] for mm in range(M)], axis=1).astype(np.float64)
    kappa = (np.sum(p * p, axis=1) + 2 * np.sum(anchor * p, axis=1)).astype(np.float32)
    from vector_line_quantization_b200.ops import Lists

    lists = Lists(T(g["offsets"], cuda), ops.rotate_codes(T(g["offsets"], cuda), T(g["codes"][perm], cuda)),
                  T(g["lamq"][perm], cuda), T(kappa, cuda), T(perm.astype(np.int64), cuda))
    D, I = ops.search(T(g["xq"].astype(np.float32), cuda), cent, cn, T(g["edge"], cuda), T(g["edge_d2"], cuda),
                      T(g["lambda_cb"], cuda), T(g["pq"], cuda), lists, int(g["P"]), int(g["W"]), int(g["k"]))
    D, I = N(D), N(I)
    assert (I == g["search_I"]).mean() > 0.98
    qn = np.sum(g["xq"].astype(np.float64) ** 2, axis=1, keepdims=True)
    assert np.all(np.abs(D - g["search_D"]) <= REL_DIST * (np.abs(g["search_D"]) + qn))
    # lambda == 0 slice vs the reference's IndexIVFPQ is covered on the CPU side (test_oracle_vs_reference.py)
    Dc, Ic = ops.search(T(g["xq"].astype(np.float32), cuda), cent, cn, T(g["edge"], cuda), T(g["edge_d2"], cuda),
                        T(g["lambda_cb"], cuda), T(g["pq"], cuda), lists, int(g["P"]), int(g["W"]), int(g["k"]), cap=3)
    assert (N(Ic) == g["search_cap3_I"]).mean() > 0.98
    torch.cuda.synchronize()


def test_select_lines_matches_oracle(ops, cuda, oracle, small_model):
    m = small_model
    P, W = 16, 128
    D = ops.l2_distances(T(m["xq"], cuda), T(m["cent"], cuda))
    _, cid = ops.select_rows(D, P)
    lst, t1, t6 = ops.select_lines(D, cid, T(m["edge"], cuda), T(m["edge_d2"], cuda), W)
    # an empty index is enough to get the oracle's line choice
    nl = m["C"] * m["E"]
    off = np.zeros(nl + 1, np.int64)
    _, _, coarse, lines, _ = oracle.search(m["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], off,
                                           np.zeros((0, m["M"]), np.uint8), np.zeros(0, np.uint8),
                                           np.zeros(0, np.int64), P=P, W=W, k=1, want_debug=True)
    from tests.parity_util import Model64, check_lines

    m64 = Model64(m)
    cidn = N(cid)
    qi, r = np.nonzero(cidn != coarse)  # top-P differences must be near-ties of the coarse distance (float64)
    if len(qi):
        q64 = m["xq"].astype(np.float64)[qi]
        dg, do = m64.coarse(q64, cidn[qi, r]), m64.coarse(q64, coarse[qi, r])
        assert np.all(np.abs(dg - do) <= REL_TIE * (np.abs(do) + (q64 ** 2).sum(1)))
    same = check_lines(N(lst), lines, m["xq"], m64)  # every differing line is a near-tie of the float64 line score
    assert same.sum() >= len(same) - 2


# ------------------------------------------------------------------------------------------------ merge (a16)
@pytest.mark.parametrize("R,nq,k", [(2, 10, 1), (8, 33, 100), (4, 7, 1024), (1, 5, 16)])
def test_merge_topk_exact(ops, cuda, oracle, R, nq, k):
    rng = np.random.RandomState(R * 100 + k)
    D = np.sort(rng.rand(R, nq, k).astype(np.float32), axis=2)
    D[:, :, ::3] = np.round(D[:, :, ::3], 2)  # cross-shard ties
    D = np.sort(D, axis=2)
    I = rng.randint(0, 1 << 40, size=(R, nq, k)).astype(np.int64)
    # shards with fewer than k results pad with (FLT_MAX, -1)
    D[0, :, k // 2:] = np.finfo(np.float32).max
    I[0, :, k // 2:] = -1
    oD, oI = ops.merge_topk(T(D, cuda), T(I, cuda))
    wD, wI = oracle.merge_topk(D, I)
    assert np.array_equal(N(oD), wD)
    assert np.array_equal(N(oI), wI)


@pytest.mark.parametrize("R,nq,W", [(2, 100, 256), (8, 1001, 64), (3, 2, 4), (4, 10000, 256)])
def test_gather_peer_slices(ops, cuda, R, nq, W):
    """exchange step of the query-split search (vlq_gather_peer_slices): rank r holds rows [r nq / R, (r + 1) nq / R) of
    three (nq, W) arrays; after the call every rank's buffer holds all rows of all arrays.  The R buffers are separate
    allocations of one device here; on an NVLink domain they are peer-mapped memory of R GPUs."""
    import torch

    a256 = lambda v: (v + 255) // 256 * 256
    base = 512
    offs = [base, base + a256(nq * W * 4), base + 2 * a256(nq * W * 4)]
    size = offs[2] + a256(nq * W * 4) + 256
    g = torch.Generator(device="cpu").manual_seed(R * 7 + nq)
    want = [torch.randint(-2 ** 31, 2 ** 31 - 1, (nq, W), generator=g, dtype=torch.int32).to(cuda) for _ in range(3)]
    q0 = [r * nq // R for r in range(R + 1)]
    bufs = []
    for r in range(R):  # own slice filled, everything else poisoned
        b = torch.full((size,), 0x5A, dtype=torch.uint8, device=cuda)
        for a in range(3):
            v = b[offs[a]:offs[a] + nq * W * 4].view(torch.int32).view(nq, W)
            v[q0[r]:q0[r + 1]] = want[a][q0[r]:q0[r + 1]]
        bufs.append(b)
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=cuda)
    before = [b.clone() for b in bufs]
    for r in range(R):
        ops.gather_peer_slices(ptrs.data_ptr(), R, r, offs, nq, W * 4)
    torch.cuda.synchronize()
    mask = torch.ones(size, dtype=torch.bool, device=cuda)
    for a in range(3):
        mask[offs[a]:offs[a] + nq * W * 4] = False
    for r in range(R):
        for a in range(3):
            v = bufs[r][offs[a]:offs[a] + nq * W * 4].view(torch.int32).view(nq, W)
            assert torch.equal(v, want[a])
        assert torch.equal(bufs[r][mask], before[r][mask])  # nothing outside the three arrays is touched


@pytest.mark.parametrize("R,nq,k", [(2, 10, 1), (8, 33, 100), (4, 7, 1024)])
def test_merge_topk_peers_equals_gathered(ops, cuda, R, nq, k):
    """gather fused into the merge (vlq_merge_topk_peers): shard r's results are read from its own buffer through a
    device array of pointers (peer-mapped symmetric memory in the multi-GPU run; R separate allocations here)"""
    import torch

    g = torch.Generator(device="cpu").manual_seed(R * 7 + k)
    D = torch.sort(torch.rand(R, nq, k, generator=g), dim=2).values
    I = torch.randint(0, 1 << 40, (R, nq, k), generator=g)
    D[0, :, k // 2:] = torch.finfo(torch.float32).max
    I[0, :, k // 2:] = -1
    D, I = D.to(cuda), I.to(cuda)
    wD, wI = ops.merge_topk(D, I)
    i_off = (nq * k * 4 + 15) // 16 * 16
    base = 256  # the results sit at an offset inside each buffer (double-buffer slot)
    bufs = []
    for r in range(R):
        b = torch.zeros(base + i_off + nq * k * 8, dtype=torch.uint8, device=cuda)
        b[base:base + 4 * nq * k].view(torch.float32).copy_(D[r].reshape(-1))
        b[base + i_off:base + i_off + 8 * nq * k].view(torch.int64).copy_(I[r].reshape(-1))
        bufs.append(b)
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=cuda)
    oD, oI = ops.merge_topk_peers(ptrs.data_ptr(), base, base + i_off, R, nq, k, device=cuda)
    assert torch.equal(oD, wD) and torch.equal(oI, wI)


def test_sharded_search_equals_single(ops, cuda, oracle, small_model):
    """id-range shards + merge == one index (SURVEY 8e), exact up to ties"""
    m = small_model
    P, W, k = 16, 128, 20
    xq = T(m["xq"], cuda)
    whole = _gpu_index(ops, cuda, oracle, m, m["xb"])
    D1, I1 = ops.search(xq, whole["cent"], whole["cn"], whole["edge"], whole["ed2"], whole["lcb"], whole["pq"],
                        whole["lists"], P, W, k, cap=1 << 20)
    import torch

    Ds, Is = [], []
    bounds = [0, 7000, 13000, 20000]
    for a, b in zip(bounds[:-1], bounds[1:]):
        sh = _gpu_index(ops, cuda, oracle, m, m["xb"][a:b])
        d_, i_ = ops.search(xq, sh["cent"], sh["cn"], sh["edge"], sh["ed2"], sh["lcb"], sh["pq"], sh["lists"], P, W, k,
                            cap=1 << 20)
        Ds.append(d_)
        Is.append(torch.where(i_ >= 0, i_ + a, i_))
    Dm, Im = ops.merge_topk(torch.stack(Ds).contiguous(), torch.stack(Is).contiguous())
    assert np.array_equal(N(Dm), N(D1))
    assert (N(Im) == N(I1)).mean() > 0.999


# ------------------------------------------------------------------------------------------------ k-means update (f1)
def test_km_update_matches_reference_rule(ops, cuda, oracle):
    rng = np.random.RandomState(8)
    n, d, k = 5000, 24, 37
    x = rng.normal(0, 5, (n, d)).astype(np.float32)
    assign = rng.randint(0, k - 2, n).astype(np.int32)  # two empty clusters
    cent, counts = ops.km_update(T(x, cuda), T(assign, cuda), k)
    cent, counts = N(cent), N(counts)
    assert np.array_equal(counts, np.bincount(assign, minlength=k))
    for c in range(k):
        rows = x[assign == c]
        if len(rows) == 0:
            assert np.all(cent[c] == 0)
            continue
        acc = np.zeros(d, np.float32)
        for r in rows:  # row order, fp32 (utils.cpp:1385-1417)
            acc += r
        np.testing.assert_array_equal(cent[c], acc / np.float32(len(rows)))


# ------------------------------------------------------------------------------------------------ size-independent properties
def test_large_encode_roundtrip_properties(ops, cuda):
    """at a size the oracle could not finish quickly: every returned distance equals the decode distance of the stored
    code, results are sorted, and encode is deterministic (idempotent across runs)"""
    import torch

    from vector_line_quantization_b200 import data

    torch.manual_seed(0)
    n, d, C, E, M = 400_000, 128, 2048, 32, 16
    x = data.sift_like_torch(n, d=d, kc=1 << 14, seed=2, device=cuda)
    cent = x[torch.randperm(n, device=cuda)[:C]].contiguous() + 0.5
    cn = ops.row_norms(cent)
    edge, ed2 = ops.knn_graph(cent, E, cn)
    lcb = torch.linspace(-0.2, 1.2, 256, device=cuda)
    pq = (torch.randn((M, 256, d // M), device=cuda) * 12).contiguous()
    A, _ = ops.l2_assign(x, cent, cn)
    enc = ops.line_encode(x, A, cent, edge, ed2, lcb, pq)
    enc2 = ops.line_encode(x, A, cent, edge, ed2, lcb, pq)
    assert torch.equal(enc.codes, enc2.codes) and torch.equal(enc.list, enc2.list) and torch.equal(enc.lamq, enc2.lamq)
    assert torch.equal(enc.list // E, A)
    ids = torch.arange(n, dtype=torch.int64, device=cuda)
    lists = ops.build_lists(C * E, M, enc.list, enc.codes, enc.lamq, enc.kappa, ids)
    assert int(lists.offsets[-1]) == n
    # checksum of checksums: the list-major arrays are a permutation of the arrival-order arrays
    assert int(lists.ids.sum()) == n * (n - 1) // 2
    assert int(lists.codes.to(torch.int64).sum()) == int(enc.codes.to(torch.int64).sum())
    assert torch.equal(enc.lamq[lists.ids], lists.lamq)
    assert torch.equal(enc.codes[lists.ids], ops.rotate_codes(lists.offsets, lists.codes, inverse=True))
    seg = torch.repeat_interleave(torch.arange(C * E, device=cuda), lists.offsets[1:] - lists.offsets[:-1])
    assert torch.equal(enc.list[lists.ids].to(torch.int64), seg)
    q = x[:256].contiguous()
    k = 10
    D, I = ops.search(q, cent, cn, edge, ed2, lcb, pq, lists, 32, 256, k)
    assert bool((I[:, 0] >= 0).all())
    assert bool((D[:, 1:] >= D[:, :-1]).all())
    # decode identity in float64 on the device
    I0 = I.clamp_min(0)
    l = enc.list[I0].to(torch.int64)
    c = cent[l // E].double()
    s = cent[edge.reshape(-1)[l].to(torch.int64)].double()
    lh = lcb[enc.lamq[I0].to(torch.int64)].double().unsqueeze(-1)
    codes = enc.codes[I0].to(torch.int64)  # [nq][k][M]
    p = torch.stack([pq[mm][codes[..., mm]] for mm in range(M)], dim=-2).reshape(q.shape[0], k, d).double()
    y = (1 - lh) * c + lh * s + p
    qd = q.double().unsqueeze(1)
    want = ((qd - y) ** 2).sum(-1) - (qd ** 2).sum(-1)
    err = (D.double() - want).abs()
    tol = REL_DIST * (want.abs() + (qd ** 2).sum(-1))
    assert bool((err[I >= 0] <= tol[I >= 0]).all())
    # querying with database vectors: the vector itself must be among its own candidates almost always
    hit = (I == torch.arange(256, device=cuda).unsqueeze(1)).any(dim=1).float().mean()
    assert float(hit) > 0.5


@pytest.mark.parametrize("P,W,k,cap", [(16, 128, 10, 1024), (32, 1024, 200, 1024), (8, 64, 1024, 3), (32, 1024, 100, 1024),
                                       (32, 1024, 128, 5)])
def test_scan_modes_identical(ops, cuda, oracle, small_model, P, W, k, cap):
    """the flattened-stream scan and the warp-per-list scan (1B-scale lists) return the same bits"""
    import torch

    m = small_model
    gi = _gpu_index(ops, cuda, oracle, m, np.concatenate([m["xb"]] * 3))  # longer lists: every vector three times
    q = T(m["xq"], cuda)
    D = ops.l2_distances(q, gi["cent"], gi["cn"])
    _, cid = ops.select_rows(D, P)
    lst, t1, t6 = ops.select_lines(D, cid, gi["edge"], gi["ed2"], W)
    args = (q, gi["pq"], gi["lcb"], lst, t1, t6, gi["ed2"].reshape(-1), gi["lists"], k, cap)
    D0, I0 = ops.scan_topk(*args, list_len_hint=0)
    D1, I1 = ops.scan_topk(*args, list_len_hint=100)
    D2, I2 = ops.scan_topk(*args, list_len_hint=0, use_workspace=False)
    D3, I3 = ops.scan_topk(*args, list_len_hint=400)  # the long-list kernel (scan_long.cu)
    assert torch.equal(D0, D2) and torch.equal(I0, I2)
    if gi["pq"].shape[0] not in (8, 16):  # the block-synchronous list scan: same summation order, same bits
        assert torch.equal(D0, D1) and torch.equal(I0, I1)
        return
    # the bank-skewed scans sum the M table terms in a lane-dependent order (hint 100) or in fixed point (hint 400, the
    # long-list kernel): last-ulp differences, so ids may only differ where two candidates are closer than that
    D0n, I0n = N(D0), N(I0)
    qn = np.sum(m["xq"].astype(np.float64) ** 2, axis=1, keepdims=True) * np.ones_like(D0n)
    tol = 2e-6 * (np.abs(D0n) + qn)
    for Dx, Ix in ((D1, I1), (D3, I3)):
        D1n, I1n = N(Dx), N(Ix)
        assert np.array_equal(I0n < 0, I1n < 0)
        valid = I0n >= 0
        assert np.all(np.abs(D1n - D0n)[valid] <= tol[valid])
        assert np.all(np.diff(D1n, axis=1) >= 0)
        diff = valid & (I0n != I1n)  # (every vector is stored three times here: exact ties are everywhere)
        for r, c in zip(*np.nonzero(diff)):  # a differing id must be a near-tie: within tolerance in the other result
            near = np.abs(D0n[r] - D1n[r, c]) <= tol[r]
            assert I1n[r, c] in I0n[r][near] or c == k - 1 or near[-1]


@pytest.mark.parametrize("P,W,k,cap", [(8, 32, 10, 1024), (8, 64, 100, 1024), (16, 128, 50, 8), (4, 16, 1024, 1024), (1, 1, 1, 1024)])
def test_small_query_scan_path_equals_general_path(ops, cuda, oracle, small_model, P, W, k, cap, monkeypatch):
    """scan_topk_kernel's register-resident path for queries of <= 4096 entries (strided stream positions, one radix
    threshold, tie ranks in position order) returns the bits of the general BlockSelect path -- on an index that stores
    every vector three times, so exact distance ties straddle the k-th place for most queries"""
    import torch

    m = small_model
    gi = _gpu_index(ops, cuda, oracle, m, np.concatenate([m["xb"][:6000]] * 3))
    q = T(m["xq"], cuda)
    D = ops.l2_distances(q, gi["cent"], gi["cn"])
    _, cid = ops.select_rows(D, P)
    lst, t1, t6 = ops.select_lines(D, cid, gi["edge"], gi["ed2"], W)
    args = (q, gi["pq"], gi["lcb"], lst, t1, t6, gi["ed2"].reshape(-1), gi["lists"], k, cap)
    lens = (gi["lists"].offsets[1:] - gi["lists"].offsets[:-1]).clamp_max(cap)
    total = lens[lst.clamp_min(0).long()].mul(lst >= 0).sum(dim=1)
    assert int((total <= 4096).sum()) > len(q) // 2  # the small path really is the one exercised
    D0, I0 = ops.scan_topk(*args, list_len_hint=0)
    monkeypatch.setenv("VLQ_SCAN_NO_SMALL", "1")
    D1, I1 = ops.scan_topk(*args, list_len_hint=0)
    monkeypatch.delenv("VLQ_SCAN_NO_SMALL")
    assert torch.equal(D0, D1) and torch.equal(I0, I1)
    ties = (D0[:, 1:] == D0[:, :-1]) & (I0[:, 1:] >= 0)
    if k > 1 and k <= 100:
        assert int(ties.sum()) > 0


@pytest.mark.parametrize("M,d,k", [(16, 128, 100), (8, 96, 100), (8, 64, 10), (4, 32, 50), (16, 64, 128)])
def test_scan_modes_random_index(ops, cuda, M, d, k):
    """flattened-stream scan vs the warp-autonomous scans (plain tables: hint 30; bank-skewed tables: hint 100 and the long-list kernel: hint 400, M = 8/16)
    on a random index with lists of 0..400 entries: same top-k up to last-ulp distance differences"""
    import torch

    g = torch.Generator(device="cpu").manual_seed(5)
    nlist, nq, W, nL = 300, 37, 64, 256
    lens = torch.randint(0, 400, (nlist,), generator=g)
    lens[::7] = 0
    off = torch.zeros(nlist + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(lens, 0)
    n = int(off[-1])
    lists = ops.Lists(off.to(cuda), torch.randint(0, 256, (n, M), generator=g, dtype=torch.uint8).to(cuda),
                      torch.randint(0, nL, (n,), generator=g, dtype=torch.uint8).to(cuda),
                      torch.randn(n, generator=g).to(cuda), torch.randperm(n, generator=g).to(cuda))
    q = torch.randn(nq, d, generator=g).to(cuda)
    pq = torch.randn(M, 256, d // M, generator=g).to(cuda)
    lcb = torch.rand(nL, generator=g).to(cuda)
    line = torch.stack([torch.randperm(nlist, generator=g)[:W] for _ in range(nq)]).to(torch.int32)
    line[:, 5] = -1  # unused slot
    line = line.to(cuda)
    t1 = (torch.rand(nq, W, generator=g) * 10).to(cuda)
    t6 = torch.randn(nq, W, generator=g).to(cuda)
    ed2 = (torch.rand(nlist, generator=g) * 4 + 0.5).to(cuda)
    args = (q, pq, lcb, line, t1, t6, ed2, lists, k, 1024)
    D0, I0 = ops.scan_topk(*args, list_len_hint=0)
    for hint in (30, 100, 400):  # warp-autonomous plain tables / bank-skewed tables / long-list kernel (scan_long.cu)
        D1, I1 = ops.scan_topk(*args, list_len_hint=hint)
        if hint == 30 or M not in (8, 16):
            assert torch.equal(D0, D1) and torch.equal(I0, I1)
            continue
        D0n, D1n, I0n, I1n = N(D0), N(D1), N(I0), N(I1)
        assert np.array_equal(I0n < 0, I1n < 0)
        valid = I0n >= 0
        scale = float(q.pow(2).sum(1).max()) + np.abs(D0n[valid]).max()
        assert np.all(np.abs(D1n - D0n)[valid] <= 2e-6 * scale)
        assert (I0n == I1n)[valid].mean() > 0.999
        assert np.all(np.diff(D1n, axis=1) >= 0)


def test_nan_vectors_are_skipped(ops, cuda, oracle, small_model):
    """invalid (NaN) input rows get no centroid (-1) on both assignment paths and never reach the lists
    (the reference drops them at add time, gpu/GpuIndexIVFPQ.cu:751-755)"""
    import torch

    m = small_model
    x = m["xb"][:1000].copy()
    x[7, 5] = np.nan
    x[500, :] = np.nan
    xt = T(x, cuda)
    cent = T(m["cent"], cuda)
    ids_simt, _ = ops.l2_assign(xt, cent)
    ids_tc, _ = ops.l2_assign_tc(xt, ops.CentPack(cent), want_dist=False)
    for ids in (N(ids_simt), N(ids_tc)):
        assert ids[7] == -1 and ids[500] == -1 and (np.delete(ids, [7, 500]) >= 0).all()
    enc = ops.line_encode(xt, ids_tc, cent, T(m["edge"], cuda), T(m["edge_d2"], cuda), T(m["lambda_cb"], cuda),
                          T(m["pq"], cuda))
    assert N(enc.list)[7] == -1 and N(enc.list)[500] == -1
    lists = ops.build_lists(m["C"] * m["E"], m["M"], enc.list, enc.codes, enc.lamq, enc.kappa,
                            torch.arange(1000, dtype=torch.int64, device=cuda))
    assert int(lists.offsets[-1]) == 998
    stored = set(N(lists.ids)[:998].tolist())
    assert 7 not in stored and 500 not in stored and len(stored) == 998
