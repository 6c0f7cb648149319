"""Per-mismatch near-tie verification for the encode and query paths (north_star: "identical except documented near-ties,
relative distance gap < 1e-5").  Every id / line that differs from the oracle is re-evaluated in float64 from the
codebooks and must be closer to the oracle's choice than REL_TIE; nothing is accepted as a fraction.

The query-time quantities cancel ||q||^2 (distances are ||q - y||^2 - ||q||^2, line scores are built from
||c||^2 - 2 q.c), so gaps are taken relative to the magnitudes that were cancelled: |value| + ||q||^2.
"""
import numpy as np

REL_TIE = 1e-5
REL_DIST = 1e-4


class Model64:
    """float64 evaluation of line scores and decode distances for one model (numpy, vectorised over pairs)"""

    def __init__(self, m):
        self.cent = np.asarray(m["cent"], np.float64)
        self.cn = (self.cent ** 2).sum(1)
        self.edge = np.asarray(m["edge"])
        self.ed2 = np.asarray(m["edge_d2"], np.float64)  # the stored fp32 values ARE the model (term5)
        self.lcb = np.asarray(m["lambda_cb"], np.float64)
        self.pq = np.asarray(m["pq"], np.float64)
        self.E = self.edge.shape[1]
        self.M = self.pq.shape[0]

    def coarse(self, q, c):
        """D[c] = ||c||^2 - 2 q.c   (gpu/impl/Distance.cu:287-290: no ||q||^2)"""
        return self.cn[c] - 2.0 * (self.cent[c] * q).sum(-1)

    def line_score(self, q, line):
        """BroadcastSum.cu:505-520: (v > 0) ? b : b - v^2 / (4 c2)"""
        c, e = line // self.E, line % self.E
        s = self.edge[c, e]
        a2, b2, c2 = self.coarse(q, s), self.coarse(q, c), self.ed2[c, e]
        v = a2 - b2 - c2
        return np.where(v > 0, b2, b2 - 0.25 * v * v / c2)

    def decode_dist(self, q, line, lamq, code):
        """||q - ((1-l)c + l s) - p(code)||^2 - ||q||^2"""
        c, e = line // self.E, line % self.E
        s = self.edge[c, e]
        lh = self.lcb[lamq][..., None]
        p = np.concatenate([self.pq[mm][code[..., mm]] for mm in range(self.M)], axis=-1)
        y = (1.0 - lh) * self.cent[c] + lh * self.cent[s] + p
        return ((q - y) ** 2).sum(-1) - (q ** 2).sum(-1)


def check_lines(lines_gpu, lines_ref, xq, m, rel=REL_TIE):
    """Top-W line lists [nq][W] (rank order).  Returns a bool mask of the queries whose line SETS agree.  Every
    rank-wise difference must be a near-tie in the float64 line score."""
    m64 = m if isinstance(m, Model64) else Model64(m)
    lg, lr = np.asarray(lines_gpu), np.asarray(lines_ref)
    assert lg.shape == lr.shape
    assert np.array_equal(lg < 0, lr < 0), "padding of the line lists differs"
    qi, r = np.nonzero(lg != lr)
    if len(qi):
        q = np.asarray(xq, np.float64)[qi]
        sg, sr = m64.line_score(q, lg[qi, r]), m64.line_score(q, lr[qi, r])
        scale = np.abs(sr) + (q ** 2).sum(1)
        bad = np.abs(sg - sr) > rel * scale
        assert not bad.any(), "unexplained line mismatches: %s" % [
            (int(qi[i]), int(r[i]), int(lg[qi[i], r[i]]), int(lr[qi[i], r[i]]), float(sg[i]), float(sr[i]))
            for i in np.nonzero(bad)[0][:5]]
    same_set = np.array([set(a.tolist()) == set(b.tolist()) for a, b in zip(lg, lr)])
    return same_set


def check_topk(D, I, Do, Io, xq, m, entry_line, entry_lamq, entry_codes, same_lines=None, rel=REL_TIE, rel_dist=REL_DIST):
    """GPU top-k (D, I) against the oracle's (Do, Io) on the same index; ids index the arrival-order arrays entry_*.
    * padding identical; GPU rows ascending;
    * every returned distance equals the float64 decode distance of its id within rel_dist;
    * every rank where the ids differ is a near-tie: the two ids' float64 distances differ by < rel (relative to
      |d| + ||q||^2).  Queries whose selected line sets differ (same_lines False; those line differences were themselves
      verified as near-ties by check_lines) are exempt from the rank-wise id check only.
    Returns (number of differing ranks, number of exempt queries)."""
    m64 = m if isinstance(m, Model64) else Model64(m)
    D, I, Do, Io = np.asarray(D), np.asarray(I), np.asarray(Do), np.asarray(Io)
    q64 = np.asarray(xq, np.float64)
    nq, k = I.shape
    if same_lines is None:
        same_lines = np.ones(nq, bool)
    fmax = np.finfo(np.float32).max
    assert np.all(np.diff(D, axis=1) >= 0), "GPU distances not ascending"
    strict = same_lines[:, None] & np.ones((1, k), bool)
    assert np.array_equal((I < 0) & strict, (Io < 0) & strict), "padding differs"
    assert np.all(D[I < 0] == fmax) and np.all(Do[Io < 0] == fmax)
    qn = (q64 ** 2).sum(1)
    # self-consistency of every GPU entry
    qi, r = np.nonzero(I >= 0)
    ids = I[qi, r]
    d64 = m64.decode_dist(q64[qi], entry_line[ids], entry_lamq[ids], entry_codes[ids])
    err = np.abs(D[qi, r] - d64)
    assert np.all(err <= rel_dist * (np.abs(d64) + qn[qi])), "GPU distance differs from the float64 decode distance"
    # rank-wise id differences must be near-ties
    diff = (I != Io) & (I >= 0) & (Io >= 0) & strict
    qi, r = np.nonzero(diff)
    if len(qi):
        ig, io = I[qi, r], Io[qi, r]
        dg = m64.decode_dist(q64[qi], entry_line[ig], entry_lamq[ig], entry_codes[ig])
        do = m64.decode_dist(q64[qi], entry_line[io], entry_lamq[io], entry_codes[io])
        bad = np.abs(dg - do) > rel * (np.abs(do) + qn[qi])
        assert not bad.any(), "unexplained id mismatches (query, rank, gpu id, oracle id, d64 gpu, d64 oracle): %s" % [
            (int(qi[i]), int(r[i]), int(ig[i]), int(io[i]), float(dg[i]), float(do[i])) for i in np.nonzero(bad)[0][:5]]
    # where ids agree the distances agree within rel_dist
    same = (I == Io) & (I >= 0)
    assert np.all(np.abs(D - Do)[same] <= rel_dist * (np.abs(Do) + qn[:, None])[same])
    return int(diff.sum()), int((~same_lines).sum())


def _np(t):
    return t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)


def check_encode(enc, o, x, m):
    """line_encode's outputs (enc, an ops.Encoded with residual) against the oracle's encode o of the same vectors x and
    assignment: lines, lambda bytes and PQ codes identical except near-ties, each verified in float64; residuals close
    wherever line and lambda byte agree.  Returns the mask of those vectors."""
    lst, lam, lamq, codes = _np(enc.list), _np(enc.lam), _np(enc.lamq), _np(enc.codes)
    n = x.shape[0]
    same_line = lst == o["list"]
    assert same_line.mean() > 0.999, same_line.mean()
    # mismatching lines must be near-ties in point-to-line distance
    x64, c64 = x.astype(np.float64), m["cent"].astype(np.float64)
    E = m["edge"].shape[1]

    def line_q2(i, l):
        a = c64[l // E]
        s = c64[m["edge"][l // E, l % E]]
        t = np.dot(x64[i] - a, s - a) / np.dot(s - a, s - a)
        return np.sum((x64[i] - (a + t * (s - a))) ** 2)

    for i in np.nonzero(~same_line)[0]:
        qa, qb = line_q2(i, lst[i]), line_q2(i, o["list"][i])
        assert abs(qa - qb) <= 1e-4 * max(qa, qb) + 1e-6, (i, qa, qb)
    ok = same_line
    np.testing.assert_allclose(lam[ok], o["lam"][ok], rtol=1e-3, atol=1e-4)
    same_lq = ok & (lamq == o["lamq"])
    assert same_lq.sum() >= ok.sum() - max(2, n // 500)  # lambda exactly between two levels
    # PQ codes identical wherever line and lambda level agree, except sub-space near-ties
    cm = codes[same_lq] != o["codes"][same_lq]
    assert cm.mean() < 2e-4, cm.mean()
    M = codes.shape[1]
    dsub = x.shape[1] // M
    rows = np.nonzero(same_lq)[0]
    for ri, mm in np.argwhere(cm):
        i = rows[ri]
        sub = o["residual"][i, mm * dsub:(mm + 1) * dsub].astype(np.float64)
        da = np.sum((sub - m["pq"][mm, codes[i, mm]]) ** 2)
        db = np.sum((sub - m["pq"][mm, o["codes"][i, mm]]) ** 2)
        assert abs(da - db) <= REL_TIE * max(da, db) + 1e-9
    res = _np(enc.residual)
    np.testing.assert_allclose(res[same_lq], o["residual"][same_lq], rtol=1e-5, atol=1e-3)
    return same_lq


def scan_candidates(q, lines, term1, term6, t5, lambda_cb, pq, offsets, codes, lamq, kappa, ids, cap):
    """float64 restatement of the scan distance of include/vlq_b200.h (vlq_scan_topk) from the kernel's own inputs:
        dist = t1 + l t6 + (l^2 - l) t5 + kappa - 2 q.p(code),   l = lambda_cb[lamq]
    over the entries the scan looks at: the first min(len, cap) entries of every selected line (-1 slots skipped), lines
    in slot order, then list position.  t5: per list id (edge_d2 flattened), or None for 0.  codes: list-major and in
    canonical sub-quantizer order (not rotated).  No VLQ geometry enters, so IMI-PQ inputs (t1 a full distance, t6 = 0,
    no t5) work the same.  Returns per query (dist float64 [n_q], ids int64 [n_q]) in stream order."""
    q = np.asarray(q, np.float64)
    pq = np.asarray(pq, np.float64)
    lcb = np.asarray(lambda_cb, np.float64)
    M, _, dsub = pq.shape
    out = []
    for i in range(q.shape[0]):
        T3 = -2.0 * np.einsum("mjt,mt->mj", pq, q[i].reshape(M, dsub))
        d_parts, i_parts = [], []
        for w, l in enumerate(lines[i]):
            if l < 0:
                continue
            s = int(offsets[l])
            e = s + min(int(offsets[l + 1]) - s, cap)
            la = lcb[lamq[s:e]]
            base = float(term1[i, w]) + la * float(term6[i, w]) + (la * la - la) * (0.0 if t5 is None else float(t5[l]))
            d_parts.append(base + kappa[s:e].astype(np.float64) + T3[np.arange(M), codes[s:e]].sum(1))
            i_parts.append(ids[s:e])
        out.append((np.concatenate(d_parts) if d_parts else np.empty(0), np.concatenate(i_parts).astype(np.int64)
                    if i_parts else np.empty(0, np.int64)))
    return out


def check_scan_topk(D, I, cands, k, qn, rel=REL_TIE, rel_dist=REL_DIST):
    """a scan's top-k (D, I) [nq][k] against the float64 candidates of scan_candidates (qn: ||q||^2, the scale of the
    cancelled term, as in check_topk):
    * min(k, candidates) results, then (FLT_MAX, -1) padding; rows ascending;
    * every returned distance within rel_dist of the float64 distance of its id;
    * every rank whose id differs from the float64 top-k is a near-tie (rel);
    * a float64 top-k id that is missing ties the k-th float64 distance."""
    D, I = np.asarray(D), np.asarray(I)
    fmax = np.finfo(np.float32).max
    assert np.all(np.diff(D, axis=1) >= 0), "distances not ascending"
    for i, (dc, ic) in enumerate(cands):
        nv = min(k, len(ic))
        assert np.all(I[i, :nv] >= 0) and np.all(I[i, nv:] == -1) and np.all(D[i, nv:] == fmax), ("padding", i, nv)
        if nv == 0:
            continue
        scale = qn[i]
        d64 = dict(zip(ic.tolist(), dc.tolist()))
        got = np.array([d64[v] for v in I[i, :nv].tolist()])
        err = np.abs(D[i, :nv] - got)
        assert np.all(err <= rel_dist * (np.abs(got) + scale)), ("distance", i, float(err.max()))
        order = np.argsort(dc, kind="stable")[:nv]
        ref_i, ref_d = ic[order], dc[order]
        r = np.nonzero(I[i, :nv] != ref_i)[0]
        bad = np.abs(got[r] - ref_d[r]) > rel * (np.abs(ref_d[r]) + scale)
        assert not bad.any(), ("unexplained id mismatch (query, rank, id, ref id, d64, ref d64)",
                               [(i, int(x), int(I[i, x]), int(ref_i[x]), got[x], ref_d[x]) for x in r[bad][:5]])
        missing = np.setdiff1d(ref_i, I[i, :nv])
        if len(missing):
            dm = np.array([d64[v] for v in missing.tolist()])
            kth = ref_d[nv - 1]
            assert np.all(np.abs(dm - kth) <= rel * (np.abs(kth) + scale)), ("missing id", i, missing[:5])
