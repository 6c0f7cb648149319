"""Encode, list build, scan and range search at the shapes the C-ABI accepts beyond the production geometries, each
against a plain float64 reference or the CPU oracle (itself checked against the reference library).

Which kernel runs, and which branch inside it, depends on d, M, E and nL.  Every row of ROWS is chosen for the code
paths it forces; DISPATCH_REQUIRED lists them and test_cases_cover_every_variant checks that the matrix still reaches
each one.  The scan and range tests also read the names of the kernels that actually ran (torch.profiler) and compare
them with scan_dispatch, a restatement of the dispatch of vlq_scan_topk (search.cu).
"""
import numpy as np
import pytest

from tests.parity_util import REL_DIST, check_encode, check_lines, check_scan_topk, scan_candidates

pytestmark = pytest.mark.gpu

NQ = 40
# id: (data, d, M, E, nL, C, n_base, P, W, [(k, cap)])
ROWS = {
    "S1": ("sift", 16, 4, 1, 1, 64, 8000, 16, 16, [(1, 1024), (100, 50)]),     # NPL 1, one edge, one lambda level
    "S2": ("sift", 48, 16, 7, 3, 128, 20000, 16, 64, [(100, 1024), (129, 1024), (128, 1)]),  # NPL 2, M 16, dsub 3
    "S3": ("deep", 100, 25, 33, 17, 64, 20000, 8, 128, [(1024, 1024)]),        # GloVe-100; M % 4 != 0; E in 33..63
    "S4": ("sift", 140, 20, 32, 256, 64, 20000, 8, 128, [(128, 50)]),         # NPL 5; codebook exactly fills smem
    "S5": ("deep", 144, 12, 40, 256, 64, 20000, 8, 128, [(100, 1024)]),       # codebook in global memory
    "S6": ("deep", 196, 28, 64, 64, 96, 20000, 8, 128, [(129, 1024)]),        # NPL 7; largest d with term-3 tables
    "S7": ("sift", 200, 8, 16, 256, 64, 20000, 8, 64, [(100, 1024)]),         # GloVe-200: per-CTA tables, no range
    "S8": ("sift", 256, 64, 64, 256, 96, 20000, 8, 128, [(128, 1)]),          # NPL 8, M 64
    # long lists: E = 8 because the graph needs E < C, and C E must stay small for ~156 entries per list
    "S9": ("sift", 128, 32, 8, 256, 48, 60000, 8, 32, [(100, 1024), (1024, 1024)]),
    "S10": ("deep", 64, 8, 16, 256, 24, 60000, 8, 32, [(100, 1024), (129, 1024), (1, 50)]),
    # the two remaining line_encode widths
    "S11": ("deep", 176, 16, 24, 128, 64, 12000, 8, 64, [(50, 1024)]),       # NPL 6; M 16 with dsub 11
    "S12": ("sift", 72, 24, 48, 8, 64, 12000, 8, 64, [(10, 200)]),           # NPL 3; E 48
}
MISALIGNED_ROWS = ("S2", "S10")  # codes start 8 bytes past a 16-byte boundary (a shard slice at an odd entry)
IMI_ROWS = ("S2", "S10")         # lambda_cb = {0}, no edge_d2, term6 = 0, term1 a full distance (GpuIndexIMIPQ)
RANGE_UNSUPPORTED = ("S7", "S8")  # 1028 d > 200 KiB: no term-3 tables

# ------------------------------------------------------------------------------------------------ dispatch, restated
SKEW_MIN_LEN, LONG_MIN_LEN, WARP_SEL_MAX_K = 56, 160, 128  # search.cu defaults, topk.cuh kWarpSelMaxK
LE_SMEM_LIMIT = 200 * 1024


def term3_supported(d, M):
    """search.cu term3_supported: codebook + one query in 200 KiB of shared memory, d % 4 == 0 (so d <= 196)"""
    return d % M == 0 and d % 4 == 0 and (256 * d + d) * 4 <= 200 * 1024


def scan_dispatch(M, d, hint, k, aligned=True, workspace=True):
    """(term-3 kernel or None, scan kernel) that vlq_scan_topk launches: search.cu:1310-1386 and scan_long_supported
    (scan_long.cu) restated, names as torch.profiler reports them without spaces"""
    long_lists = hint >= 24
    have_t3 = workspace and term3_supported(d, M)
    use_async = long_lists and k <= WARP_SEL_MAX_K and have_t3
    use_long = (long_lists and have_t3 and hint >= SKEW_MIN_LEN and (hint >= LONG_MIN_LEN or k > WARP_SEL_MAX_K)
                and M in (8, 16) and aligned)
    skew = use_long or (use_async and aligned and M in (8, 16) and hint >= SKEW_MIN_LEN)
    mt = M if M in (8, 16) and aligned else 0
    t3 = None
    if have_t3:
        t3 = {(16, 8): "term3_reg_kernel<16,8>", (8, 12): "term3_reg_kernel<8,12>"}.get((M, d // M), "term3_kernel(")
    if use_long:
        scan = "scan_long_kernel<%d," % M
    elif use_async:
        scan = "scan_async_kernel<%d,%s>" % (M if skew else mt, "true" if skew else "false")
    else:
        scan = "scan_topk_kernel<%d,%s>" % (mt, "true" if long_lists else "false")
    return t3, scan


def range_kernel(M, aligned=True):
    return M if M in (8, 16) and aligned else 0


def avg_len(name):
    _, _, _, E, _, C, nb = ROWS[name][:7]
    return nb // (C * E)


def scan_calls(name, variant):
    """(hint, k, cap, use_workspace) of every scan call a row makes in one variant ("vlq", "misaligned", "imi")"""
    out = []
    for k, cap in ROWS[name][9]:
        out += [(h, k, cap, True) for h in (0, 30, 100, 400, avg_len(name))]
        if variant == "vlq":
            out.append((0, k, cap, False))
    return out


def encode_list_tags(d, M, E, nL):
    tags = {"line_encode_kernel<%d>" % (-(-d // 32))}
    smem = 1408 * d + 7680  # line_encode.cu: codebook 1024 d + per-warp tail 384 d + 7680
    tags.add("codebook in shared memory" if smem <= LE_SMEM_LIMIT else "codebook in global memory")
    if smem == LE_SMEM_LIMIT:
        tags.add("codebook in shared memory, at the limit")
    if E == 1:
        tags.add("E = 1")
    if 32 < E < 64:
        tags.add("second edge half partly filled")
    if nL < 32:
        tags.add("nL < 32")
    tags.add({16: "copy_code uint4", 8: "copy_code uint2"}.get(M, "copy_code words" if M % 4 == 0 else "copy_code bytes"))
    tags.add({16: "store_code_rotated rot16", 8: "store_code_rotated rot8"}.get(M, "store_code_rotated generic"))
    return tags


def scan_tag(variant, M, d, hint, k, aligned, workspace):
    t3, scan = scan_dispatch(M, d, hint, k, aligned, workspace)
    if t3 is None:
        t3 = "tables per CTA, workspace passed" if workspace else "tables per CTA"
    return "%s M=%d|%s|%s" % (variant, M, t3, scan)


DISPATCH_REQUIRED = {
    *("line_encode_kernel<%d>" % n for n in range(1, 9)),
    "codebook in global memory", "codebook in shared memory, at the limit", "E = 1", "second edge half partly filled",
    "nL < 32",
    "copy_code uint4", "copy_code uint2", "copy_code words", "copy_code bytes",
    "store_code_rotated rot16", "store_code_rotated rot8", "store_code_rotated generic",
    # the M = 16 / 8 scan templates fed by the generic term3_kernel (dsub 3 and 8)
    *("vlq M=%d|term3_kernel(|%s" % (M, s) for M in (16, 8) for s in (
        "scan_topk_kernel<%d,false>" % M, "scan_topk_kernel<%d,true>" % M, "scan_async_kernel<%d,false>" % M,
        "scan_async_kernel<%d,true>" % M, "scan_long_kernel<%d," % M)),
    "vlq M=32|term3_kernel(|scan_topk_kernel<0,true>", "vlq M=32|term3_kernel(|scan_async_kernel<0,false>",
    "vlq M=8|tables per CTA, workspace passed|scan_topk_kernel<8,true>",
    "vlq M=64|tables per CTA, workspace passed|scan_topk_kernel<0,true>",
    *("misaligned M=%d|term3_kernel(|%s" % (M, s) for M in (16, 8) for s in (
        "scan_topk_kernel<0,false>", "scan_topk_kernel<0,true>", "scan_async_kernel<0,false>")),
    *("imi M=%d|term3_kernel(|%s" % (M, s) for M in (16, 8) for s in (
        "scan_async_kernel<%d,false>" % M, "scan_async_kernel<%d,true>" % M, "scan_long_kernel<%d," % M)),
    "range<0>", "range<8>", "range<16>", "misaligned range<0>", "imi range<8>", "imi range<16>",
    "range unsupported d=200", "range unsupported d=256",
}


def covered_variants():
    cov = set()
    for name, (_, d, M, E, nL, *_rest) in ROWS.items():
        cov |= encode_list_tags(d, M, E, nL)
        for variant in ("vlq",) + (("misaligned",) if name in MISALIGNED_ROWS else ()) + (
                ("imi",) if name in IMI_ROWS else ()):
            aligned = variant != "misaligned"
            for hint, k, cap, ws in scan_calls(name, variant):
                cov.add(scan_tag(variant, M, d, hint, k, aligned, ws))
            if name in RANGE_UNSUPPORTED:
                cov.add("range unsupported d=%d" % d)
            else:
                cov.add(("" if variant == "vlq" else variant + " ") + "range<%d>" % range_kernel(M, aligned))
    return cov


def test_cases_cover_every_variant():
    missing = DISPATCH_REQUIRED - covered_variants()
    assert not missing, sorted(missing)
    # the bound the header states: term-3 tables up to d = 196
    assert term3_supported(196, 28) and not term3_supported(200, 8) and not term3_supported(256, 64)


# ------------------------------------------------------------------------------------------------ fixtures
def T(a, dev):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def N(t):
    return t.detach().cpu().numpy()


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope="module")
def ops(cuda):
    from vector_line_quantization_b200 import ops as _ops

    return _ops


_rows = {}


def _row(name, ops, cuda, oracle):
    """model (oracle-trained, fixed seeds), the device encode of the base (oracle assignment), lists built in two
    commits, and the coarse stage's lines of the queries"""
    if name in _rows:
        return _rows[name]
    import torch

    from vector_line_quantization_b200 import data

    kind, d, M, E, nL, C, nb, P, W, _ = ROWS[name]
    seed = 1000 + 10 * list(ROWS).index(name)
    gen = data.sift_like if kind == "sift" else data.deep_like
    m = oracle.train_all(gen(6000, d=d, kc=256, seed=seed), nlist=C, E=E, M=M, nL=nL, niter=4, pq_niter=4)
    xb, xq = gen(nb, d=d, kc=256, seed=seed + 1), gen(NQ, d=d, kc=256, seed=seed + 2)
    _, A = oracle.l2_topk(xb, m["cent"], 1)
    A = A[:, 0].copy()
    cent, edge, ed2, lcb, pq = (T(m[k], cuda) for k in ("cent", "edge", "edge_d2", "lambda_cb", "pq"))
    x = T(xb, cuda)
    enc = ops.line_encode(x, T(A, cuda), cent, edge, ed2, lcb, pq, want_residual=True)
    ids = torch.arange(nb, dtype=torch.int64, device=cuda)
    nl = C * E
    h = nb // 2 + 1
    old = ops.build_lists(nl, M, enc.list[:h], enc.codes[:h], enc.lamq[:h], enc.kappa[:h], ids[:h])
    lists = ops.build_lists(nl, M, enc.list[h:], enc.codes[h:], enc.lamq[h:], enc.kappa[h:], ids[h:], old)
    cn = ops.row_norms(cent)
    pack = ops.CentPack(cent, cn) if ops._abi.lib().vlq_tc_supported(d, C) else None
    q = T(xq, cuda)
    lines = ops.coarse_lines(q, cent, cn, edge, ed2, P, W, pack=pack)
    torch.cuda.synchronize()
    off = N(lists.offsets)
    canon = N(ops.rotate_codes(lists.offsets, lists.codes, inverse=True))
    r = dict(m=m, d=d, M=M, E=E, nL=nL, C=C, P=P, W=W, xb=xb, xq=xq, A=A, x=x, q=q, cent=cent, cn=cn, edge=edge,
             ed2=ed2, lcb=lcb, pq=pq, enc=enc, ids=ids, lists=lists, lines=lines, off=off, canon=canon,
             lamq=N(lists.lamq), kappa=N(lists.kappa), lid=N(lists.ids), qn=(xq.astype(np.float64) ** 2).sum(1))
    _rows[name] = r
    return r


def _profiled(fn):
    """run fn; return its result and the names (spaces removed) of the scan, term-3 and range kernels it launched, in
    launch order"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    keys = ("scan_topk_kernel", "scan_async_kernel", "scan_long_kernel", "term3", "range_count_kernel",
            "range_gather_kernel")
    ev = [e for e in prof.events() if any(k in e.name for k in keys)]
    ev.sort(key=lambda e: e.time_range.start)
    return out, [e.name.replace(" ", "") for e in ev]


def _check_launched(names, expected):
    assert len(names) == len(expected), (names, expected)
    for got, want in zip(names, expected):
        assert want in got, (got, want, names)


ROW_IDS = list(ROWS)


# ------------------------------------------------------------------------------------------------ a. encode
@pytest.mark.parametrize("name", ROW_IDS)
def test_encode_matches_oracle(ops, cuda, oracle, name):
    r = _row(name, ops, cuda, oracle)
    m = r["m"]
    n = min(len(r["xb"]), 6000)
    x = r["xb"][:n]
    lst, lam = oracle.line_stage(x, r["A"][:n], m["cent"], m["edge"], m["edge_d2"])
    lamq = oracle.lambda_quantize(lam, m["lambda_cb"])
    res = oracle.residual(x, lst, lamq, m["lambda_cb"], m["cent"], m["edge"])
    o = dict(list=lst, lam=lam, lamq=lamq, residual=res, codes=oracle.pq_encode(res, m["pq"]))
    enc = r["enc"]
    head = type(enc)(*(t[:n] for t in enc))
    check_encode(head, o, x, m)
    # kappa = ||p||^2 + 2 anchor.p of EVERY entry, in float64 from the kernel's own list / lambda byte / codes
    E, M, d = r["E"], r["M"], r["d"]
    el, elq, ec, kap = N(enc.list).astype(np.int64), N(enc.lamq), N(enc.codes), N(enc.kappa)
    c64 = m["cent"].astype(np.float64)
    lh = m["lambda_cb"].astype(np.float64)[elq][:, None]
    anchor = (1 - lh) * c64[el // E] + lh * c64[m["edge"][el // E, el % E]]
    p = np.concatenate([m["pq"][mm][ec[:, mm]] for mm in range(M)], axis=1).astype(np.float64)
    want = (p * p).sum(1) + 2 * (anchor * p).sum(1)
    scale = (p * p).sum(1) + 2 * np.abs(anchor * p).sum(1)
    err = np.abs(kap - want)
    assert np.all(err <= 1e-5 * scale), (int(err.argmax()), float(kap[err.argmax()]), float(want[err.argmax()]))
    assert np.array_equal(el // E, r["A"])


# ------------------------------------------------------------------------------------------------ b. stand-alone a6 / a7
@pytest.mark.parametrize("name", ROW_IDS)
def test_standalone_lambda_and_residual_match_fused(ops, cuda, oracle, name):
    """vlq_lambda_quantize / vlq_line_residual state the fused kernel's operation order: same bits (training uses them)"""
    import torch

    r = _row(name, ops, cuda, oracle)
    enc, n, d = r["enc"], len(r["xb"]), r["d"]
    lq = torch.empty(n, dtype=torch.uint8, device=cuda)
    ops._abi.call("vlq_lambda_quantize", _ptr(enc.lam), n, _ptr(r["lcb"]), r["nL"], _ptr(lq), _stream())
    assert torch.equal(lq, enc.lamq)
    lst = enc.list.clone()
    lst[::37] = -1  # rows without a line give zeros
    res = torch.full((n, d), float("nan"), device=cuda)
    ops._abi.call("vlq_line_residual", _ptr(r["x"]), n, d, _ptr(lst), _ptr(enc.lamq), _ptr(r["lcb"]), _ptr(r["cent"]),
                  _ptr(r["edge"]), r["E"], _ptr(res), _stream())
    valid = lst >= 0
    assert torch.equal(res[valid].view(torch.int32), enc.residual[valid].view(torch.int32))
    assert torch.equal(res[~valid].view(torch.int32), torch.zeros_like(res[~valid]).view(torch.int32))


# ------------------------------------------------------------------------------------------------ c. lists
@pytest.mark.parametrize("name", ROW_IDS)
def test_lists_two_commits_and_recompute_kappa(ops, cuda, oracle, name):
    import torch

    r = _row(name, ops, cuda, oracle)
    enc, lists, M = r["enc"], r["lists"], r["M"]
    nl = r["C"] * r["E"]
    e_list, e_codes = N(enc.list), N(enc.codes)
    off, perm = oracle.build_lists(e_list, nl)
    n = len(perm)
    assert n == len(r["xb"])
    assert np.array_equal(r["off"], off) and np.array_equal(r["lid"], perm)
    pos = np.arange(n) - np.repeat(off[:-1], np.diff(off))  # position inside the list
    want = np.take_along_axis(e_codes[perm], (np.arange(M)[None, :] + pos[:, None]) % M, axis=1)
    assert np.array_equal(N(lists.codes), want)  # stored[j] = code[(j + pos) mod M]
    assert np.array_equal(r["lamq"], N(enc.lamq)[perm])
    assert np.array_equal(r["kappa"].view(np.int32), N(enc.kappa)[perm].view(np.int32))
    # the loader's kappa: same bits as line_encode's
    kap = torch.full((n,), float("nan"), device=cuda)
    ops._abi.call("vlq_recompute_kappa", n, nl, _ptr(lists.offsets), _ptr(lists.codes), _ptr(lists.lamq),
                  _ptr(r["cent"]), r["d"], _ptr(r["edge"]), r["E"], _ptr(r["lcb"]), _ptr(r["pq"]), M, _ptr(kap),
                  _stream())
    assert torch.equal(kap.view(torch.int32), lists.kappa.view(torch.int32))


# ------------------------------------------------------------------------------------------------ d. lines
@pytest.mark.parametrize("name", ROW_IDS)
def test_coarse_lines_match_oracle(ops, cuda, oracle, name):
    r = _row(name, ops, cuda, oracle)
    m = r["m"]
    empty = np.zeros(r["C"] * r["E"] + 1, np.int64)  # an empty index is enough for the oracle's line choice
    _, _, _, lines_ref, _ = oracle.search(r["xq"], m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], empty,
                                          np.zeros((0, r["M"]), np.uint8), np.zeros(0, np.uint8), np.zeros(0, np.int64),
                                          P=r["P"], W=r["W"], k=1, want_debug=True)
    check_lines(N(r["lines"][0]), lines_ref, r["xq"], m)


# ------------------------------------------------------------------------------------------------ e-g. scan
def _misaligned(ops, lists, cuda):
    """the same lists with the code array 8 bytes past a 16-byte boundary"""
    import torch

    n, M = lists.codes.shape
    buf = torch.zeros(n * M + 16, dtype=torch.uint8, device=cuda)
    codes = buf[8:8 + n * M].view(n, M)
    codes.copy_(lists.codes)
    assert codes.data_ptr() % 16 == 8
    return ops.Lists(lists.offsets, codes, lists.lamq, lists.kappa, lists.ids)


def _variant(ops, cuda, r, variant):
    """(lists, lambda_cb, lines, edge_d2 or None, row_add, lamq for the reference, ||q||^2 added for full distances)"""
    import torch

    lists, lines = r["lists"], r["lines"]
    if variant == "misaligned":
        return _misaligned(ops, lists, cuda), r["lcb"], lines, r["ed2"], r["lamq"], r["qn"]
    if variant == "imi":
        # GpuIndexIMIPQ: zero lambda bytes, lambda_cb = {0}, no term5, term6 = 0, term1 = ||q - c||^2 of the cell
        lst = N(lines[0])
        c = r["m"]["cent"].astype(np.float64)[np.maximum(lst, 0) // r["E"]]
        t1 = ((r["xq"].astype(np.float64)[:, None, :] - c) ** 2).sum(-1).astype(np.float32)
        imi = ops.Lists(lists.offsets, lists.codes, torch.zeros_like(lists.lamq), lists.kappa, lists.ids)
        return (imi, torch.zeros(1, device=cuda), (lines[0], T(t1, cuda), torch.zeros_like(lines[2])), None,
                np.zeros_like(r["lamq"]), np.zeros(NQ))
    return lists, r["lcb"], lines, r["ed2"], r["lamq"], r["qn"]


def _candidates(r, lcb, lines, ed2, lamq, cap):
    lst, t1, t6 = (N(t) for t in lines)
    return scan_candidates(r["xq"], lst, t1, t6, None if ed2 is None else N(ed2).reshape(-1), N(lcb), r["m"]["pq"],
                           r["off"], r["canon"], lamq, r["kappa"], r["lid"], cap)


def _scan_variant(ops, cuda, oracle, name, variant):
    r = _row(name, ops, cuda, oracle)
    lists, lcb, lines, ed2, lamq, _ = _variant(ops, cuda, r, variant)
    ed2f = None if ed2 is None else ed2.reshape(-1)
    calls = scan_calls(name, variant)
    aligned = variant != "misaligned"
    outs, names = _profiled(lambda: [
        ops.scan_topk(r["q"], r["pq"], lcb, lines[0], lines[1], lines[2], ed2f, lists, k, cap, use_workspace=ws,
                      list_len_hint=h) for h, k, cap, ws in calls])
    expected = []
    for h, k, cap, ws in calls:
        expected += [x for x in scan_dispatch(r["M"], r["d"], h, k, aligned, ws) if x is not None]
    _check_launched(names, expected)
    cands = {}
    for (h, k, cap, ws), (D, I) in zip(calls, outs):
        if cap not in cands:
            cands[cap] = _candidates(r, lcb, lines, ed2, lamq, cap)
        check_scan_topk(N(D), N(I), cands[cap], k, r["qn"])
    assert max(len(c[1]) for c in cands[max(cands)]) > 0


@pytest.mark.parametrize("name", ROW_IDS)
def test_scan_matches_float64(ops, cuda, oracle, name):
    _scan_variant(ops, cuda, oracle, name, "vlq")


@pytest.mark.parametrize("name", MISALIGNED_ROWS)
def test_scan_misaligned_codes(ops, cuda, oracle, name):
    _scan_variant(ops, cuda, oracle, name, "misaligned")


@pytest.mark.parametrize("name", IMI_ROWS)
def test_scan_imi_configuration(ops, cuda, oracle, name):
    _scan_variant(ops, cuda, oracle, name, "imi")


# ------------------------------------------------------------------------------------------------ h. range search
def _range_variant(ops, cuda, oracle, name, variant):
    import torch

    r = _row(name, ops, cuda, oracle)
    lists, lcb, lines, ed2, lamq, add = _variant(ops, cuda, r, variant)
    cap = ROWS[name][9][0][1]
    row_add = None if variant == "imi" else ops.row_norms(r["q"])
    qn = r["qn"]
    full = [(dc + add[i], ic) for i, (dc, ic) in enumerate(_candidates(r, lcb, lines, ed2, lamq, cap))]
    # about the 50th candidate of each query: counts differ per query
    radius = float(np.median([np.sort(fd)[min(49, len(fd) - 1)] for fd, _ in full if len(fd)]))
    (a, b), names = _profiled(lambda: [
        ops.range_scan_lines(r["q"], r["pq"], lcb, lines, ed2, lists, radius, cap=cap, row_add=row_add,
                             stage_results=s) for s in (None, 64)])
    mt = range_kernel(r["M"], variant != "misaligned")
    assert {n[n.index("range_"):n.index(">") + 1] for n in names if "range_" in n} == {
        "range_count_kernel<%d>" % mt, "range_gather_kernel<%d>" % mt}, names
    # a gather split into sub-ranges writes the same bits
    assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))
    assert torch.equal(a[2], b[2])
    lims, D, I = (N(t) for t in a)
    counts = np.diff(lims)
    assert len(np.unique(counts)) > 1 and lims[-1] > NQ
    assert np.all(D < radius)
    for i, (fd, fi) in enumerate(full):
        dg, ig = D[lims[i]:lims[i + 1]], I[lims[i]:lims[i + 1]]
        all64 = dict(zip(fi.tolist(), fd.tolist()))
        assert all(v in all64 for v in ig.tolist()), i
        got = dict(zip(ig.tolist(), dg.tolist()))
        want = set(fi[fd < radius].tolist())
        for v in set(got) ^ want:  # only entries within 1e-4 of the radius may fall on either side
            assert abs(all64[v] - radius) <= 1e-4 * (abs(all64[v]) + qn[i]), (i, v, all64[v], radius)
        for v, dv in got.items():
            assert abs(dv - all64[v]) <= REL_DIST * (abs(all64[v]) + qn[i]), (i, v, dv, all64[v])
        pos = {v: j for j, v in enumerate(fi.tolist())}  # stream order: lines in slot order, then list position
        assert np.all(np.diff([pos[v] for v in ig.tolist()]) > 0), i


def _range_unsupported(ops, cuda, oracle, name):
    """both passes refuse a shape without term-3 tables, before any launch"""
    import torch

    r = _row(name, ops, cuda, oracle)
    lst, t1, t6 = r["lines"]
    lists, lib = r["lists"], ops._abi.lib()
    nq, W, cap = NQ, r["W"], 1024
    wsb = lib.vlq_range_workspace_bytes(nq, r["M"], W, cap)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
    lims = torch.zeros(nq + 1, dtype=torch.int64, device=cuda)
    outD = torch.empty(16, device=cuda)
    outI = torch.empty(16, dtype=torch.int64, device=cuda)
    qn = ops.row_norms(r["q"])
    args = (_ptr(r["q"]), nq, r["d"], _ptr(r["pq"]), r["M"], _ptr(r["lcb"]), r["nL"], _ptr(lst), _ptr(t1), _ptr(t6),
            _ptr(r["ed2"]), W, _ptr(lists.offsets), _ptr(lists.codes), _ptr(lists.lamq), _ptr(lists.kappa), cap,
            _ptr(qn), 1.0e6)
    VLQ_EUNSUPPORTED = -3
    assert lib.vlq_range_count(*args, _ptr(lims), _ptr(ws), wsb, _stream()) == VLQ_EUNSUPPORTED
    assert lib.vlq_range_gather(*args, _ptr(lists.ids), _ptr(lims), 0, nq, _ptr(outD), _ptr(outI), _ptr(ws), wsb,
                                _stream()) == VLQ_EUNSUPPORTED
    with pytest.raises(ops._abi.VlqError, match="unsupported"):
        ops.range_scan_lines(r["q"], r["pq"], r["lcb"], r["lines"], r["ed2"], lists, 1.0e6, row_add=qn)


@pytest.mark.parametrize("name", ROW_IDS)
def test_range_matches_float64(ops, cuda, oracle, name):
    if name in RANGE_UNSUPPORTED:
        _range_unsupported(ops, cuda, oracle, name)
    else:
        _range_variant(ops, cuda, oracle, name, "vlq")


@pytest.mark.parametrize("name", MISALIGNED_ROWS)
def test_range_misaligned_codes(ops, cuda, oracle, name):
    _range_variant(ops, cuda, oracle, name, "misaligned")


@pytest.mark.parametrize("name", IMI_ROWS)
def test_range_imi_configuration(ops, cuda, oracle, name):
    _range_variant(ops, cuda, oracle, name, "imi")
