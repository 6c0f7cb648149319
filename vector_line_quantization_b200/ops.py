"""Device-resident operator layer: torch CUDA tensors in, torch CUDA tensors out, every op one C-ABI call.

torch is plumbing here (device memory + the current stream); all arithmetic happens in lib/libvlq_b200.so.
Each function names the C-ABI entry it calls; the reference interface that entry replaces is cited in
include/vlq_b200.h.
"""
from collections import namedtuple

import torch

from . import _abi

Lists = namedtuple("Lists", "offsets codes lamq kappa ids")  # CSR inverted lists (see csrc/lists.cu)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _chk(t, dtype, name):
    if t is None:
        return None
    if not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor" % name)
    if t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


def launch_count():
    return int(_abi.lib().vlq_launch_count())


def row_norms(x):
    x = _chk(x, torch.float32, "x")
    n, d = x.shape
    out = torch.empty(n, dtype=torch.float32, device=x.device)
    _abi.call("vlq_row_norms", _ptr(x), n, d, _ptr(out), _stream())
    return out


def l2_assign(x, cent, cnorm=None, add_xnorm=True, want_dist=True):
    """nearest centroid per row (a2): -> (ids int32 [n], dist f32 [n] or None)"""
    x = _chk(x, torch.float32, "x")
    cent = _chk(cent, torch.float32, "cent")
    n, d = x.shape
    if cnorm is None:
        cnorm = row_norms(cent)
    ids = torch.empty(n, dtype=torch.int32, device=x.device)
    dist = torch.empty(n, dtype=torch.float32, device=x.device) if want_dist else None
    _abi.call("vlq_l2_assign", _ptr(x), n, d, _ptr(cent), _ptr(cnorm), cent.shape[0], int(add_xnorm), _ptr(ids),
              _ptr(dist), _stream())
    return ids, dist


def l2_distances(x, cent, cnorm=None, out=None):
    """coarse matrix D = ||c||^2 - 2 x.c (a11)"""
    x = _chk(x, torch.float32, "x")
    cent = _chk(cent, torch.float32, "cent")
    n, d = x.shape
    C = cent.shape[0]
    if cnorm is None:
        cnorm = row_norms(cent)
    D = out if out is not None else torch.empty((n, C), dtype=torch.float32, device=x.device)
    _abi.call("vlq_l2_distances", _ptr(x), n, d, _ptr(cent), _ptr(cnorm), C, _ptr(D), D.stride(0), _stream())
    return D


def select_rows(D, k, row_add=None, cols=None):
    """exact top-k per row ascending (a11/a15): -> (val f32 [n][k], idx int32 [n][k])"""
    D = _chk(D, torch.float32, "D")
    n = D.shape[0]
    cols = D.shape[1] if cols is None else cols
    val = torch.empty((n, k), dtype=torch.float32, device=D.device)
    idx = torch.empty((n, k), dtype=torch.int32, device=D.device)
    _abi.call("vlq_select_rows", _ptr(D), n, cols, D.stride(0), k, _ptr(row_add), _ptr(val), _ptr(idx), _stream())
    return val, idx


def knn_graph(cent, E, cnorm=None):
    """centroid kNN graph (a4): -> (edge int32 [C][E], edge_d2 f32 [C][E])"""
    cent = _chk(cent, torch.float32, "cent")
    C, d = cent.shape
    if cnorm is None:
        cnorm = row_norms(cent)
    edge = torch.empty((C, E), dtype=torch.int32, device=cent.device)
    ed2 = torch.empty((C, E), dtype=torch.float32, device=cent.device)
    wsb = _abi.lib().vlq_knn_graph_workspace_bytes(C, E)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cent.device)
    _abi.call("vlq_knn_graph", _ptr(cent), _ptr(cnorm), C, d, E, _ptr(edge), _ptr(ed2), _ptr(ws), wsb, _stream())
    return edge, ed2


Encoded = namedtuple("Encoded", "list lam lamq codes kappa residual")


# 4-bit PQ codes (include/vlq_b200.h, csrc/pq4.cuh): a codebook (M, 16, dsub) selects the *_pq4 entry points of
# line_encode, scan_topk, range_scan_lines and decode_entries, whose lists hold M / 2 packed bytes per entry,
# byte j = code[2j] | code[2j + 1] << 4.
def is_pq4(pq):
    return pq.shape[1] == 16


def pack_pq4(codes):
    """one byte per 4-bit code [n][M] (M even) -> the stored form [n][M / 2]"""
    return (codes[:, 0::2] | (codes[:, 1::2] << 4)).contiguous()


def unpack_pq4(packed):
    """[n][M / 2] packed bytes -> [n][M] codes"""
    return torch.stack((packed & 15, packed >> 4), dim=2).reshape(packed.shape[0], -1).contiguous()


def line_encode(x, assign, cent, edge, edge_d2, lambda_cb=None, pq=None, want_residual=False):
    """fused line stage (+ lambda quantiser + residual + PQ encode when lambda_cb/pq are given) (a5-a8)"""
    x = _chk(x, torch.float32, "x")
    assign = _chk(assign, torch.int32, "assign")
    cent = _chk(cent, torch.float32, "cent")
    edge = _chk(edge, torch.int32, "edge")
    edge_d2 = _chk(edge_d2, torch.float32, "edge_d2")
    n, d = x.shape
    E = edge.shape[1]
    dev = x.device
    out_list = torch.empty(n, dtype=torch.int32, device=dev)
    out_lam = torch.empty(n, dtype=torch.float32, device=dev)
    lamq = codes = kappa = resid = None
    M = nL = 0
    if lambda_cb is not None:
        lambda_cb = _chk(lambda_cb, torch.float32, "lambda_cb")
        pq = _chk(pq, torch.float32, "pq")
        M, nL = pq.shape[0], lambda_cb.shape[0]
        lamq = torch.empty(n, dtype=torch.uint8, device=dev)
        codes = torch.empty((n, M // 2 if is_pq4(pq) else M), dtype=torch.uint8, device=dev)
        kappa = torch.empty(n, dtype=torch.float32, device=dev)
        if want_residual:
            resid = torch.empty((n, d), dtype=torch.float32, device=dev)
    _abi.call("vlq_line_encode_pq4" if pq is not None and is_pq4(pq) else "vlq_line_encode", _ptr(x), n, d, _ptr(assign), _ptr(cent), _ptr(edge), _ptr(edge_d2), E,
              _ptr(lambda_cb), nL, _ptr(pq), M, _ptr(out_list), _ptr(out_lam), _ptr(lamq), _ptr(codes), _ptr(kappa),
              _ptr(resid), _stream())
    return Encoded(out_list, out_lam, lamq, codes, kappa, resid)


def build_lists(nlists, M, new_list, new_codes, new_lamq, new_kappa, new_ids, old=None):
    """stable counting-sort append of new entries behind the existing CSR lists (a9) -> Lists"""
    dev = new_list.device
    n_new = new_list.shape[0]
    n_old = 0 if old is None else old.ids.shape[0]
    tot = n_old + n_new
    out = Lists(
        torch.empty(nlists + 1, dtype=torch.int64, device=dev),
        torch.empty((tot, M), dtype=torch.uint8, device=dev),
        torch.empty(tot, dtype=torch.uint8, device=dev),
        torch.empty(tot, dtype=torch.float32, device=dev),
        torch.empty(tot, dtype=torch.int64, device=dev),
    )
    wsb = _abi.lib().vlq_build_lists_workspace_bytes(n_new, nlists)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    o = old if n_old > 0 else Lists(None, None, None, None, None)
    _abi.call("vlq_build_lists", nlists, M, n_old, _ptr(o.offsets), _ptr(o.codes), _ptr(o.lamq), _ptr(o.kappa),
              _ptr(o.ids), n_new, _ptr(_chk(new_list, torch.int32, "new_list")),
              _ptr(_chk(new_codes, torch.uint8, "new_codes")), _ptr(_chk(new_lamq, torch.uint8, "new_lamq")),
              _ptr(_chk(new_kappa, torch.float32, "new_kappa")), _ptr(_chk(new_ids, torch.int64, "new_ids")),
              _ptr(out.offsets), _ptr(out.codes), _ptr(out.lamq), _ptr(out.kappa), _ptr(out.ids), _ptr(ws), wsb,
              _stream())
    return out


def remove_ids(lists, ids=None, id_range=None):
    """remove the entries whose id is in `ids` (int64, any order, duplicates allowed) or in the half-open
    id_range = (lo, hi) from CSR lists (vlq_remove_ids_plan + vlq_remove_ids_apply) -> (Lists, removed).
    Survivors keep their order inside a list; their code words are re-rotated to their new positions.  The result is
    a new Lists at its exact size (peak memory: old + new slab); `lists` is left as it is."""
    offsets = _chk(lists.offsets, torch.int64, "offsets")
    dev = offsets.device
    nlists = offsets.shape[0] - 1
    n = lists.ids.shape[0]
    M = lists.codes.shape[1]
    batch = None
    if ids is not None:
        batch = torch.unique(torch.as_tensor(ids, dtype=torch.int64).reshape(-1).to(dev))  # sorted, de-duplicated
    lo, hi = (int(id_range[0]), int(id_range[1])) if id_range is not None else (0, 0)
    wsb = _abi.lib().vlq_remove_ids_workspace_bytes(n, nlists)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    out_off = torch.empty(nlists + 1, dtype=torch.int64, device=dev)
    nb = 0 if batch is None else batch.numel()
    _abi.call("vlq_remove_ids_plan", nlists, n, _ptr(offsets), _ptr(_chk(lists.ids, torch.int64, "ids")), lo, hi,
              _ptr(batch) if nb else 0, nb, _ptr(out_off), _ptr(ws), wsb, _stream())
    live = int(out_off[-1])
    # at least one row each: the apply pass takes non-NULL destinations even when nothing survives
    rows = max(live, 1)
    out = Lists(out_off, torch.empty((rows, M), dtype=torch.uint8, device=dev),
                torch.empty(rows, dtype=torch.uint8, device=dev), torch.empty(rows, dtype=torch.float32, device=dev),
                torch.empty(rows, dtype=torch.int64, device=dev))
    _abi.call("vlq_remove_ids_apply", nlists, M, n, _ptr(offsets), _ptr(_chk(lists.codes, torch.uint8, "codes")),
              _ptr(_chk(lists.lamq, torch.uint8, "lamq")), _ptr(_chk(lists.kappa, torch.float32, "kappa")),
              _ptr(lists.ids), _ptr(out_off), _ptr(out.codes), _ptr(out.lamq), _ptr(out.kappa), _ptr(out.ids),
              _ptr(ws), wsb, _stream())
    return Lists(out_off, *(t[:live] for t in out[1:])), n - live


def lookup_ids(lists, keys=None, id_range=None):
    """slab index of every wanted id (vlq_lookup_ids) -> (pos int64 CUDA tensor, found).  keys: sorted unique int64
    keys (batch mode), pos[i] for keys[i]; id_range = (lo, hi): pos[i] for the id lo + i.  pos = the lowest slab index
    holding the id, -1 where none does; found = the number of slots with an entry."""
    offsets = _chk(lists.offsets, torch.int64, "offsets")
    dev = offsets.device
    n = lists.ids.shape[0]
    if (keys is None) == (id_range is None):
        raise ValueError("give exactly one of keys and id_range")
    if keys is not None:
        keys = _chk(torch.as_tensor(keys, dtype=torch.int64).reshape(-1).to(dev).contiguous(), torch.int64, "keys")
        lo, nslots = 0, keys.numel()
    else:
        lo, nslots = int(id_range[0]), int(id_range[1]) - int(id_range[0])
    pos = torch.empty(max(nslots, 0), dtype=torch.int64, device=dev)
    found = torch.empty(1, dtype=torch.int64, device=dev)
    _abi.call("vlq_lookup_ids", n, _ptr(_chk(lists.ids, torch.int64, "ids")) if n else 0, lo,
              _ptr(keys) if keys is not None and nslots else 0, nslots, _ptr(pos), _ptr(found), _stream())
    return pos, int(found)


def decode_entries(lists, pos, pq, cent=None, edge=None, lambda_cb=None, cb=None, nbits=None, want_ids=False):
    """stored vectors of the entries at the slab indexes pos (-1: a NaN row) -> x f32 [n][d] (, ids int64 [n]).
    VLQ lists (vlq_decode_entries): cent [C][d], edge [C][E] (lists = C E), lambda_cb.  IMI-PQ lists
    (vlq_imi_decode_entries): cb = (cb1, cb2), each [2^nbits][d / 2]."""
    offsets = _chk(lists.offsets, torch.int64, "offsets")
    pq = _chk(pq, torch.float32, "pq")
    pos = _chk(pos, torch.int64, "pos")
    M, d = pq.shape[0], pq.shape[0] * pq.shape[2]
    pq4 = is_pq4(pq)
    n = pos.numel()
    out = torch.empty((n, d), dtype=torch.float32, device=offsets.device)
    oid = torch.empty(n, dtype=torch.int64, device=offsets.device) if want_ids else None
    codes = _chk(lists.codes, torch.uint8, "codes")
    ids = _chk(lists.ids, torch.int64, "ids")
    if cb is None:
        edge = _chk(edge, torch.int32, "edge")
        lambda_cb = _chk(lambda_cb, torch.float32, "lambda_cb")
        _abi.call("vlq_decode_entries_pq4" if pq4 else "vlq_decode_entries", n, _ptr(pos), offsets.shape[0] - 1, _ptr(offsets), _ptr(codes),
                  _ptr(_chk(lists.lamq, torch.uint8, "lamq")), _ptr(ids), M, d, _ptr(pq),
                  _ptr(_chk(cent, torch.float32, "cent")), _ptr(edge), edge.shape[-1], _ptr(lambda_cb),
                  lambda_cb.shape[0], _ptr(out), _ptr(oid), _stream())
    else:
        _abi.call("vlq_imi_decode_entries", n, _ptr(pos), _ptr(offsets), _ptr(codes), _ptr(ids), M, d, _ptr(pq),
                  _ptr(_chk(cb[0], torch.float32, "cb1")), _ptr(_chk(cb[1], torch.float32, "cb2")), int(nbits),
                  _ptr(out), _ptr(oid), _stream())
    return (out, oid) if want_ids else out


def _refine_tables(pq, cent, edge, lambda_cb, pq2):
    return (_chk(pq, torch.float32, "pq"), _chk(cent, torch.float32, "cent"), _chk(edge, torch.int32, "edge"),
            _chk(lambda_cb, torch.float32, "lambda_cb"), _chk(pq2, torch.float32, "pq2"))


def refine_encode(x, enc, pq, cent, edge, lambda_cb, pq2=None, want_residual=False):
    """refinement code of rows x from their line_encode outputs enc (list, lamq, canonical codes) (vlq_refine_encode)
    -> (code2 uint8 [n][M2] or None, r2 f32 [n][d] or None); r2 = x - x1, code2 = PQ2(r2).  pq2=None: r2 only."""
    x = _chk(x, torch.float32, "x")
    pq, cent, edge, lambda_cb, pq2 = _refine_tables(pq, cent, edge, lambda_cb, pq2)
    n, d = x.shape
    M2 = pq2.shape[0] if pq2 is not None else 0
    code2 = torch.empty((n, M2), dtype=torch.uint8, device=x.device) if pq2 is not None else None
    r2 = torch.empty((n, d), dtype=torch.float32, device=x.device) if (want_residual or pq2 is None) else None
    _abi.call("vlq_refine_encode", _ptr(x), n, d, _ptr(_chk(enc.list, torch.int32, "list")),
              _ptr(_chk(enc.lamq, torch.uint8, "lamq")), _ptr(_chk(enc.codes, torch.uint8, "codes")), pq.shape[0],
              _ptr(pq), _ptr(cent), _ptr(edge), edge.shape[-1], _ptr(lambda_cb), lambda_cb.shape[0], _ptr(pq2), M2,
              _ptr(code2), _ptr(r2), _stream())
    return code2, r2


def refine_topk(q, cand, k, lists, code2, pq, cent, edge, lambda_cb, pq2, labels=True):
    """re-rank (vlq_refine_topk): cand int64 [nq][kc] slab indexes (-1 = none) -> (D f32 [nq][k] = ||q - x2||^2
    ascending, I int64 [nq][k] ids, or slab indexes with labels=False); ties keep candidate order, (FLT_MAX, -1) pad"""
    q = _chk(q, torch.float32, "q")
    cand = _chk(cand, torch.int64, "cand")
    pq, cent, edge, lambda_cb, pq2 = _refine_tables(pq, cent, edge, lambda_cb, pq2)
    offsets = _chk(lists.offsets, torch.int64, "offsets")
    nq, d = q.shape
    kc = cand.shape[1]
    D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    _abi.call("vlq_refine_topk", _ptr(q), nq, d, _ptr(cand), kc, k, offsets.shape[0] - 1, _ptr(offsets),
              _ptr(lists.codes), _ptr(lists.lamq), _ptr(lists.ids) if labels else 0, _ptr(code2), pq.shape[0], _ptr(pq),
              _ptr(cent), _ptr(edge), edge.shape[-1], _ptr(lambda_cb), lambda_cb.shape[0], _ptr(pq2), pq2.shape[0],
              _ptr(D), _ptr(I), _stream())
    return D, I


def refine_decode(lists, code2, pos, pq, cent, edge, lambda_cb, pq2):
    """x2 = x1 + p2(code2) of the entries at the slab indexes pos (vlq_refine_decode) -> f32 [n][d] (-1: NaN row)"""
    pq, cent, edge, lambda_cb, pq2 = _refine_tables(pq, cent, edge, lambda_cb, pq2)
    offsets = _chk(lists.offsets, torch.int64, "offsets")
    pos = _chk(pos, torch.int64, "pos")
    M, d = pq.shape[0], pq.shape[0] * pq.shape[2]
    pq4 = is_pq4(pq)
    n = pos.numel()
    out = torch.empty((n, d), dtype=torch.float32, device=offsets.device)
    _abi.call("vlq_refine_decode", n, _ptr(pos), offsets.shape[0] - 1, _ptr(offsets), _ptr(lists.codes),
              _ptr(lists.lamq), _ptr(lists.ids), _ptr(_chk(code2, torch.uint8, "code2")), M, d, _ptr(pq), _ptr(cent),
              _ptr(edge), edge.shape[-1], _ptr(lambda_cb), lambda_cb.shape[0], _ptr(pq2), pq2.shape[0], _ptr(out), 0,
              _stream())
    return out


def filter_kappa(lists, id_range=None, ids=None, bitmap=None, invert=False, out=None):
    """masked kappa of filtered search (vlq_filter_kappa) -> f32 CUDA tensor [n]: lists.kappa where the entry's id is a
    member, +inf elsewhere.  member = id in the half-open id_range (lo, hi) OR in `ids` (int64, any order, duplicates
    allowed) OR bit (id & 7) of bitmap[id >> 3] (uint8 tensor), negated with invert=True.  Pass the result as the
    `kappa` of scan_topk / range_scan_lines."""
    kappa = _chk(lists.kappa, torch.float32, "kappa")
    dev = kappa.device
    n = lists.ids.shape[0]
    batch = None
    if ids is not None:
        batch = torch.unique(torch.as_tensor(ids, dtype=torch.int64).reshape(-1).to(dev))  # sorted, de-duplicated
    nb = 0 if batch is None else batch.numel()
    if bitmap is not None:
        bitmap = _chk(torch.as_tensor(bitmap, dtype=torch.uint8).reshape(-1).to(dev).contiguous(), torch.uint8, "bitmap")
    nbytes = 0 if bitmap is None else bitmap.numel()
    lo, hi = (int(id_range[0]), int(id_range[1])) if id_range is not None else (0, 0)
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=dev)
    _abi.call("vlq_filter_kappa", n, _ptr(_chk(lists.ids, torch.int64, "ids")) if n else 0, _ptr(kappa) if n else 0, lo,
              hi, _ptr(batch) if nb else 0, nb, _ptr(bitmap) if nbytes else 0, nbytes, int(bool(invert)),
              _ptr(out) if n else 0, _stream())
    return out


def filter_results(D, I):
    """(+inf, id) results of a scan on masked kappa -> (FLT_MAX, -1) in place (vlq_filter_results); returns (D, I)"""
    D = _chk(D, torch.float32, "D")
    I = _chk(I, torch.int64, "I")
    rows, k = D.shape
    _abi.call("vlq_filter_results", rows, k, _ptr(D), _ptr(I), _stream())
    return D, I


def rotate_codes(offsets, codes, inverse=False):
    """canonical list-major codes [n][M] -> the stored layout (or back with inverse=True): the entry at position pos of
    its list keeps stored[j] = code[(j + pos) mod M] (csrc/scan.cuh).  Plumbing for callers that assemble Lists by hand
    (tests, fixtures); vlq_build_lists produces the stored layout itself."""
    n, M = codes.shape
    lens = offsets[1:] - offsets[:-1]
    live = int(offsets[-1])  # rows beyond the last list (skipped vectors) are left as they are
    pos = torch.zeros(n, dtype=torch.int64, device=codes.device)
    pos[:live] = torch.arange(live, device=codes.device) - torch.repeat_interleave(offsets[:-1], lens)
    j = torch.arange(M, device=codes.device).unsqueeze(0)
    idx = (j + (-pos if inverse else pos).unsqueeze(1)) % M
    return torch.gather(codes, 1, idx).contiguous()


def _lines_out(nq, W, dev, out):
    """(list int32, term1 f32, term6 f32) [nq][W] destinations of a line selection: `out` checked, or new tensors"""
    if out is not None:
        lst, t1, t6 = out
        assert lst.shape == (nq, W) and lst.is_contiguous() and t1.is_contiguous() and t6.is_contiguous()
        return out
    return (torch.empty((nq, W), dtype=torch.int32, device=dev), torch.empty((nq, W), dtype=torch.float32, device=dev),
            torch.empty((nq, W), dtype=torch.float32, device=dev))


def select_lines(D, coarse_ids, edge, edge_d2, W, out=None):
    """query-time line selection (a12): -> (list int32 [nq][W], term1, term6 f32 [nq][W])"""
    D = _chk(D, torch.float32, "D")
    coarse_ids = _chk(coarse_ids, torch.int32, "coarse_ids")
    nq, P = coarse_ids.shape
    E = edge.shape[1]
    lst, t1, t6 = _lines_out(nq, W, D.device, out)
    _abi.call("vlq_select_lines", _ptr(D), nq, D.stride(0), _ptr(coarse_ids), P, _ptr(edge), _ptr(edge_d2), E, W,
              _ptr(lst), _ptr(t1), _ptr(t6), _stream())
    return lst, t1, t6


_scan_ws = {}


def scan_topk(q, pq, lambda_cb, line_list, term1, term6, edge_d2, lists, k, cap=1024, use_workspace=True,
              list_len_hint=None, out=None, slab_index=False, kappa=None):
    """ADC scan of the selected lists fused with exact top-k (a13-a15): -> (D f32 [nq][k], I int64 [nq][k]).
    slab_index=True: I holds each result's slab index (its row in lists.codes) instead of its id (ids = NULL).
    kappa: per-entry kappa to read instead of lists.kappa (filter_kappa's mask).
    A 4-bit codebook (M, 16, dsub) scans packed lists through pair tables (vlq_scan_topk_pq4: use_workspace required)."""
    q = _chk(q, torch.float32, "q")
    pq = _chk(pq, torch.float32, "pq")
    nq, d = q.shape
    M = pq.shape[0]
    pq4 = is_pq4(pq)
    W = line_list.shape[1]
    if out is not None:  # contiguous (nq, k) f32 / int64 destinations (e.g. row slices of the caller's result arrays)
        outD, outI = _chk(out[0], torch.float32, "out D"), _chk(out[1], torch.int64, "out I")
        assert outD.shape == (nq, k) and outI.shape == (nq, k)
    else:
        outD = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        outI = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    hint = list_len_hint if list_len_hint is not None else lists.ids.shape[0] // max(1, lists.offsets.shape[0] - 1)
    ws = None
    wsb = 0
    if use_workspace:  # term-3 tables of the batch (grow-only cache per device)
        wsb = _abi.lib().vlq_scan_topk_workspace_bytes(nq, M // 2 if pq4 else M)
        ws = _scan_ws.get(q.device)
        if ws is None or ws.numel() < wsb:
            ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device=q.device)
            _scan_ws[q.device] = ws
    _abi.call("vlq_scan_topk_pq4" if pq4 else "vlq_scan_topk", _ptr(q), nq, d, _ptr(pq), M, _ptr(lambda_cb), lambda_cb.shape[0],
              _ptr(_chk(line_list, torch.int32, "line_list")), _ptr(term1), _ptr(term6), _ptr(edge_d2), W,
              _ptr(lists.offsets), _ptr(lists.codes), _ptr(lists.lamq),
              _ptr(lists.kappa if kappa is None else _chk(kappa, torch.float32, "kappa")),
              0 if slab_index else _ptr(lists.ids), k, cap, int(hint), _ptr(outD), _ptr(outI), _ptr(ws), wsb, _stream())
    return outD, outI


def range_scan_lines(q, pq, lambda_cb, lines, edge_d2, lists, radius, cap=1024, row_add=None, tile=5120,
                     stage_results=None, kappa=None):
    """Radius search over the selected lines (a15-range, vlq_range_count + vlq_range_gather): every entry the scan would
    look at whose distance (+ row_add[q], e.g. ||q||^2 for the full squared L2) is < radius, per query in stream order
    (lines in slot order, then list position) -> (lims int64 [nq + 1], D f32 [total], I int64 [total]), CUDA tensors.
    stage_results: gather each tile in query sub-ranges of at most this many results (one query at least).
    kappa: per-entry kappa to read instead of lists.kappa (filter_kappa's mask)."""
    if kappa is not None:
        lists = lists._replace(kappa=_chk(kappa, torch.float32, "kappa"))
    q = _chk(q, torch.float32, "q")
    pq = _chk(pq, torch.float32, "pq")
    nq, d = q.shape
    M = pq.shape[0]
    pq4 = is_pq4(pq)
    count, gather = ("vlq_range_count_pq4", "vlq_range_gather_pq4") if pq4 else ("vlq_range_count", "vlq_range_gather")
    lst, t1, t6 = lines
    W = lst.shape[1]
    dev = q.device
    ed2 = None if edge_d2 is None else edge_d2.reshape(-1)
    lims = [torch.zeros(1, dtype=torch.int64, device=dev)]
    outD, outI = [], []
    tile = _tile_rows(nq, tile)
    ws = torch.empty(max(_abi.lib().vlq_range_workspace_bytes(tile, M // 2 if pq4 else M, W, cap), 256), dtype=torch.uint8, device=dev)
    lt = torch.empty(tile + 1, dtype=torch.int64, device=dev)
    done = 0
    for s in range(0, nq, tile):
        e = min(nq, s + tile)
        m = e - s
        args = (_ptr(q[s:e]), m, d, _ptr(pq), M, _ptr(lambda_cb), lambda_cb.shape[0],
                _ptr(_chk(lst[s:e], torch.int32, "line_list")), _ptr(t1[s:e]), _ptr(t6[s:e]), _ptr(ed2), W,
                _ptr(lists.offsets), _ptr(lists.codes), _ptr(lists.lamq), _ptr(lists.kappa), cap,
                _ptr(None if row_add is None else row_add[s:e]), float(radius))
        _abi.call(count, *args, _ptr(lt), _ptr(ws), ws.numel(), _stream())
        hl = lt[:m + 1].cpu()
        total = int(hl[m])
        D = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
        I = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        q0 = 0
        while q0 < m:
            q1 = q0 + 1
            if stage_results is None:
                q1 = m
            while q1 < m and int(hl[q1 + 1] - hl[q0]) <= stage_results:
                q1 += 1
            o = int(hl[q0])
            if int(hl[q1]) == o:  # no results in [q0, q1): nothing to write (and an empty slice has no address)
                q0 = q1
                continue
            _abi.call(gather, *args, _ptr(lists.ids), _ptr(lt), q0, q1, _ptr(D[o:]), _ptr(I[o:]), _ptr(ws),
                      ws.numel(), _stream())
            q0 = q1
        lims.append(hl[1:].to(dev) + done)
        outD.append(D[:total])
        outI.append(I[:total])
        done += total
    return torch.cat(lims), (torch.cat(outD) if outD else torch.empty(0, device=dev)), \
        (torch.cat(outI) if outI else torch.empty(0, dtype=torch.int64, device=dev))


def range_search(q, cent, cnorm, edge, edge_d2, lambda_cb, pq, lists, P, W, radius, cap=1024, tile=5120, pack=None,
                 stage_results=None):
    """Full radius query (a11 + a12 + a15-range) on resident tensors: the lines of ops.search, then every entry of them
    with full squared distance ||q - x||^2 < radius -> (lims int64 [nq + 1], D f32 [total], I int64 [total])"""
    q = _chk(q, torch.float32, "q")
    lines = coarse_lines(q, cent, cnorm, edge, edge_d2, P, W, tile=tile, pack=pack)
    return range_scan_lines(q, pq, lambda_cb, lines, edge_d2, lists, radius, cap=cap, row_add=row_norms(q), tile=tile,
                            stage_results=stage_results)


def merge_topk(D, I):
    """shard merge (a16): D, I are [R][nq][k] -> (nq,k)"""
    D = _chk(D, torch.float32, "D")
    I = _chk(I, torch.int64, "I")
    R, nq, k = D.shape
    outD = torch.empty((nq, k), dtype=torch.float32, device=D.device)
    outI = torch.empty((nq, k), dtype=torch.int64, device=D.device)
    _abi.call("vlq_merge_topk", _ptr(D), _ptr(I), R, nq, k, _ptr(outD), _ptr(outI), _stream())
    return outD, outI


def merge_topk_peers(peer_ptrs_dev, d_off, i_off, R, nq, k, out=None, device=None):
    """shard merge with the gather fused in (a16): peer_ptrs_dev = device address of an array of R buffer pointers
    (symmetric memory), each buffer holding [D f32 (nq,k)] at d_off and [I int64 (nq,k)] at i_off"""
    if out is None:
        out = (torch.empty((nq, k), dtype=torch.float32, device=device), torch.empty((nq, k), dtype=torch.int64, device=device))
    _abi.call("vlq_merge_topk_peers", int(peer_ptrs_dev), d_off, i_off, R, nq, k, _ptr(out[0]), _ptr(out[1]), _stream())
    return out


def gather_peer_slices(peer_ptrs_dev, R, rank, arr_offsets, nq, row_bytes):
    """query-split sharding: pull the other ranks' row slices of the arrays at arr_offsets (bytes inside the symmetric
    buffers) into this rank's buffer, one launch of P2P loads"""
    import ctypes

    offs = (ctypes.c_int64 * len(arr_offsets))(*[int(o) for o in arr_offsets])
    _abi.call("vlq_gather_peer_slices", int(peer_ptrs_dev), R, rank, ctypes.addressof(offs), len(arr_offsets), nq,
              row_bytes, _stream())


def km_update(x, assign, k):
    """k-means mean step, deterministic row order (f1): -> (centroids f32 [k][d], counts int32 [k])"""
    x = _chk(x, torch.float32, "x")
    assign = _chk(assign, torch.int32, "assign")
    n, d = x.shape
    cent = torch.empty((k, d), dtype=torch.float32, device=x.device)
    counts = torch.empty(k, dtype=torch.int32, device=x.device)
    wsb = _abi.lib().vlq_km_update_workspace_bytes(n, k)
    ws = torch.empty(wsb, dtype=torch.uint8, device=x.device)
    _abi.call("vlq_km_update", _ptr(x), n, d, _ptr(assign), k, _ptr(cent), _ptr(counts), _ptr(ws), wsb, _stream())
    return cent, counts


def _tile_rows(nq, tile):
    """equal query tiles of at most `tile` rows, multiples of 256 (GpuIndexIVFPQ::search makes the same split)"""
    if nq <= tile:
        return max(nq, 1)
    nt = -(-nq // tile)
    return min(tile, (-(-nq // nt) + 255) // 256 * 256)


def coarse_lines(q, cent, cnorm, edge, edge_d2, P, W, tile=5120, pack=None, out=None):
    """First half of the query path (a11 + a12) for a batch of queries: -> (list int32, term1, term6 f32), each [nq][W].
    This half does not touch the inverted lists, so shards can split the QUERIES for it (sharding.QuerySplitSearch)."""
    nq = q.shape[0]
    C = cent.shape[0]
    P = min(P, C)
    if out is None:
        out = (torch.empty((nq, W), dtype=torch.int32, device=q.device), torch.empty((nq, W), dtype=torch.float32, device=q.device),
               torch.empty((nq, W), dtype=torch.float32, device=q.device))
    if nq == 0:
        return out
    tile = _tile_rows(nq, tile)
    stage = CoarseStage(cent, cnorm, edge, edge_d2, P, W, tile, pack)
    for s in range(0, nq, tile):
        e = min(nq, s + tile)
        stage.run(q[s:e], out=tuple(t[s:e] for t in out))
    return out


class CoarseStage:
    """a11 + a12 for query tiles of at most `tile` rows through vlq_coarse_lines, the entry GpuIndexIVFPQ::search calls:
    it picks the route (vlq_coarse_route) and lays out the workspace.  .exact: the matrix-free route (route 2)."""

    def __init__(self, cent, cnorm, edge, edge_d2, P, W, tile, pack=None):
        self.cent, self.cnorm, self.edge, self.edge_d2, self.pack = cent, cnorm, edge, edge_d2, pack
        self.C, self.d = cent.shape
        self.P, self.W = min(P, self.C), W
        args = (self.d, self.C, self.P, edge.shape[1], W, int(pack is not None))
        self.exact = _abi.lib().vlq_coarse_route(*args) == 2
        self.ws = torch.empty(_abi.lib().vlq_coarse_lines_workspace_bytes(tile, *args), dtype=torch.uint8,
                              device=cent.device)

    def run(self, qt, out=None, want_coarse=False):
        qt = _chk(qt, torch.float32, "q")
        nq = qt.shape[0]
        lst, t1, t6 = _lines_out(nq, self.W, qt.device, out)
        cid = torch.empty((nq, self.P), dtype=torch.int32, device=qt.device) if want_coarse else None
        pack = self.pack
        _abi.call("vlq_coarse_lines", _ptr(qt), nq, self.d, _ptr(self.cent), _ptr(self.cnorm),
                  0 if pack is None else _ptr(pack.buf), 1.0 if pack is None else pack.scale, self.C, self.P,
                  _ptr(self.edge), _ptr(self.edge_d2), self.edge.shape[1], self.W, _ptr(cid), _ptr(lst), _ptr(t1),
                  _ptr(t6), _ptr(self.ws), self.ws.numel(), _stream())
        return (lst, t1, t6, cid) if want_coarse else (lst, t1, t6)


def scan_lines(q, pq, lambda_cb, lines, edge_d2, lists, k, cap=1024, tile=5120, out=None, list_len_hint=None):
    """Second half of the query path (a13-a15): scan the selected lines of every query on THIS shard's lists"""
    nq = q.shape[0]
    lst, t1, t6 = lines
    if out is None:
        out = (torch.empty((nq, k), dtype=torch.float32, device=q.device), torch.empty((nq, k), dtype=torch.int64, device=q.device))
    ed2_flat = edge_d2.reshape(-1)
    tile = _tile_rows(nq, tile)
    for s in range(0, nq, tile):
        e = min(nq, s + tile)
        scan_topk(q[s:e], pq, lambda_cb, lst[s:e], t1[s:e], t6[s:e], ed2_flat, lists, k, cap, out=(out[0][s:e], out[1][s:e]),
                  list_len_hint=list_len_hint)
    return out


def search(q, cent, cnorm, edge, edge_d2, lambda_cb, pq, lists, P, W, k, cap=1024, tile=5120, pack=None, out=None,
           list_len_hint=None):
    """Full query path on resident tensors (a11-a15), tiled over queries (at most 5120 per tile: 1.25 GiB of coarse distances).
    pack (a CentPack) routes the coarse distances through the tcgen05 kernel."""
    nq = q.shape[0]
    C = cent.shape[0]
    P = min(P, C)
    if out is not None:
        outD, outI = out
    else:
        outD = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        outI = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    tile = _tile_rows(nq, tile)
    stage = CoarseStage(cent, cnorm, edge, edge_d2, P, W, tile, pack)
    ed2_flat = edge_d2.reshape(-1)
    for s in range(0, nq, tile):
        e = min(nq, s + tile)
        qt = q[s:e]
        lst, t1, t6 = stage.run(qt)
        scan_topk(qt, pq, lambda_cb, lst, t1, t6, ed2_flat, lists, k, cap, out=(outD[s:e], outI[s:e]),
                  list_len_hint=list_len_hint)
    return outD, outI


# ------------------------------------------------------------------------------------------------ tensor-core coarse path
class CentPack:
    """Pre-packed centroids for the tcgen05 kernels (vlq_tc_pack_centroids): fp16 hi/lo tiles + padded ||c||^2."""

    def __init__(self, cent, cnorm=None, scale=None):
        cent = _chk(cent, torch.float32, "cent")
        self.C, self.d = cent.shape
        if not _abi.lib().vlq_tc_supported(self.d, self.C):
            raise ValueError("tensor-core path needs d %% 32 == 0 and 32 <= d <= 128 (got d=%d)" % self.d)
        self.cnorm = row_norms(cent) if cnorm is None else cnorm
        if scale is None:
            import math

            mx = float(cent.abs().max())
            scale = 2.0 ** (9 - math.ceil(math.log2(mx))) if mx > 0 else 1.0
        self.scale = float(scale)
        nbytes = _abi.lib().vlq_tc_cent_pack_bytes(self.C, self.d)
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=cent.device)
        _abi.call("vlq_tc_pack_centroids", _ptr(cent), _ptr(self.cnorm), self.C, self.d, self.scale, _ptr(self.buf),
                  _stream())
        self._ws = None

    def workspace(self, n):
        need = _abi.lib().vlq_l2_tc_workspace_bytes(n, self.d, self.C)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.buf.device)
        return self._ws


def l2_assign_tc(x, pack, add_xnorm=True, want_dist=True):
    """nearest centroid per row on the tensor cores (a2): -> (ids int32 [n], dist f32 [n] or None)"""
    x = _chk(x, torch.float32, "x")
    n, d = x.shape
    ids = torch.empty(n, dtype=torch.int32, device=x.device)
    dist = torch.empty(n, dtype=torch.float32, device=x.device) if want_dist else None
    ws = pack.workspace(n)
    _abi.call("vlq_l2_assign_tc", _ptr(x), n, d, _ptr(pack.buf), pack.scale, pack.C,
              1 if add_xnorm else 0, _ptr(ids),
              _ptr(dist), _ptr(ws), ws.numel(), _stream())
    return ids, dist


def l2_distances_tc(x, pack, out=None, bucket_min=None):
    """coarse matrix D = ||c||^2 - 2 x.c on the tensor cores (a11); bucket_min ([n][num_buckets] f32) optionally
    receives the minimum of every 32-column bucket (input of coarse_select_lines)"""
    x = _chk(x, torch.float32, "x")
    n, d = x.shape
    D = out if out is not None else torch.empty((n, pack.C), dtype=torch.float32, device=x.device)
    ws = pack.workspace(n)
    _abi.call("vlq_l2_distances_tc", _ptr(x), n, d, _ptr(pack.buf), pack.scale, pack.C, _ptr(D), D.stride(0),
              _ptr(bucket_min), _ptr(ws), ws.numel(), _stream())
    return D


def l2_bucket_min_tc(x, pack, bucket_min):
    """the tcgen05 sweep without the distance matrix: only the minima of the 32-column buckets are written"""
    x = _chk(x, torch.float32, "x")
    n, d = x.shape
    assert bucket_min.shape == (n, num_buckets(pack.C)) and bucket_min.is_contiguous()
    ws = pack.workspace(n)
    _abi.call("vlq_l2_bucket_min_tc", _ptr(x), n, d, _ptr(pack.buf), pack.scale, pack.C, _ptr(bucket_min), _ptr(ws),
              ws.numel(), _stream())
    return bucket_min


def coarse_select_lines_exact(q, cent, cnorm, bucket_min, P, edge, edge_d2, W, want_coarse=False, out=None):
    """a11 + a12 without a distance matrix (vlq_coarse_select_lines_exact); out = (list, term1, term6) destinations"""
    q = _chk(q, torch.float32, "q")
    nq, d = q.shape
    C, E = cent.shape[0], edge.shape[1]
    lst, t1, t6 = _lines_out(nq, W, q.device, out)
    cid = torch.empty((nq, P), dtype=torch.int32, device=q.device) if want_coarse else None
    _abi.call("vlq_coarse_select_lines_exact", _ptr(q), nq, d, _ptr(cent), _ptr(cnorm), _ptr(bucket_min),
              bucket_min.shape[1], C, P, _ptr(edge), _ptr(edge_d2), E, W, _ptr(cid), _ptr(lst), _ptr(t1), _ptr(t6),
              _stream())
    return (lst, t1, t6, cid) if want_coarse else (lst, t1, t6)


def num_buckets(C):
    return int(_abi.lib().vlq_tc_num_buckets(C))


def coarse_select_lines(D, bucket_min, C, P, edge, edge_d2, W, want_coarse=False, out=None):
    """fused top-P (through the bucket minima) + line selection (a11 + a12); out = (list, term1, term6) destinations"""
    nq = D.shape[0]
    E = edge.shape[1]
    lst, t1, t6 = _lines_out(nq, W, D.device, out)
    cid = torch.empty((nq, P), dtype=torch.int32, device=D.device) if want_coarse else None
    _abi.call("vlq_coarse_select_lines", _ptr(D), nq, D.stride(0), _ptr(bucket_min), bucket_min.shape[1], C, P,
              _ptr(edge), _ptr(edge_d2), E, W, _ptr(cid), _ptr(lst), _ptr(t1), _ptr(t6), _stream())
    return (lst, t1, t6, cid) if want_coarse else (lst, t1, t6)
