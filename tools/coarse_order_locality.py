#!/usr/bin/env python
"""Go / no-go measurement for a graph-local column order of the coarse distance tile D (BASELINE configs[1]).

The matrix route writes D[q][c] for every centroid c and the fused select (csl::coarse_select_lines_fast_kernel) then
gathers from one row of D per query: the P best 32-column bucket lines, and the P * E neighbour columns edge[c][e] of the
top-P centroids.  In k-means id order those neighbour columns are scattered over the 256 KB row, so each read is its own
DRAM access.  Any permutation of the columns gives the same values (the sweep computes D[q][c] from the same operands
whatever slot c has); this tool asks how much a locality-preserving order would save before any kernel changes.

For each candidate order (identity, recursive balanced bisection along the principal axis down to 32-centroid leaves,
reverse Cuthill-McKee on the symmetrised E-NN graph) it relabels the index (centroid rows, graph, edge_d2) and
  * counts per query, on the device, the distinct 64-byte segments and 128-byte lines of the D row the select touches
    (P bucket lines + neighbour reads), next to the bucket-minimum row it also reads (nb * 4 bytes, the same in every
    order);
  * counts the stage-2 candidates (entries of the P best buckets not above the P-th bucket minimum);
  * times the unmodified select kernel on the relabelled tile (CUDA events, L2 overwritten before every launch): the
    relabelled index has exactly the access pattern a column-order implementation would have;
  * checks D_order[:, col] == D_id[:, col2id[col]] bitwise on the first tile (the invariance the idea rests on).

Codebooks: coarse k-means on the device exactly as bench.py trains them (same generator, seeds and sizes); the PQ part
is not needed here.

  python tools/coarse_order_locality.py [--nq 10000] [--out FILE.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def order_bisection(cent, leaf=32):
    """Recursive balanced bisection along each node's principal axis (power iteration on the d x d scatter matrix from a
    fixed start vector, stable sort of the projections); left parts are multiples of `leaf`, so leaves are buckets."""
    C, d = cent.shape
    x = cent.astype(np.float64)
    order = np.arange(C, dtype=np.int64)
    stack = [(0, C)]
    while stack:
        lo, hi = stack.pop()
        n = hi - lo
        if n <= leaf:
            continue
        idx = order[lo:hi]
        xc = x[idx] - x[idx].mean(axis=0)
        cov = xc.T @ xc
        v = np.ones(d) / np.sqrt(d)
        for _ in range(30):
            v = cov @ v
            nv = np.linalg.norm(v)
            if nv == 0:
                break
            v /= nv
        if v[np.argmax(np.abs(v))] < 0:
            v = -v
        order[lo:hi] = idx[np.argsort(xc @ v, kind="stable")]
        nl = max(leaf, (n // 2) // leaf * leaf)
        stack.append((lo + nl, hi))
        stack.append((lo, lo + nl))
    return order


def order_rcm(edge):
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import reverse_cuthill_mckee

    C, E = edge.shape
    rows = np.repeat(np.arange(C), E)
    A = csr_matrix((np.ones(C * E, dtype=np.int8), (rows, edge.reshape(-1))), shape=(C, C))
    return np.asarray(reverse_cuthill_mckee((A + A.T).tocsr(), symmetric_mode=True), dtype=np.int64)


def distinct_per_row(x):
    s = x.sort(dim=1).values
    return 1 + (s[:, 1:] != s[:, :-1]).sum(dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10_000_000, help="database size bench.py sizes the training set from")
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--nlist", type=int, default=65536)
    ap.add_argument("--nedge", type=int, default=32)
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--nprobe", type=int, default=64)
    ap.add_argument("--w1", type=int, default=256)
    ap.add_argument("--kc", type=int, default=1 << 18)
    ap.add_argument("--train-iters", type=int, default=10)
    ap.add_argument("--tile", type=int, default=5000, help="queries per select launch (GpuIndexIVFPQ::search: 2 x 5000)")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from vector_line_quantization_b200 import _abi, data, ops, train

    _abi.lib()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    C, E, d, P, W, nq = a.nlist, a.nedge, a.d, a.nprobe, a.w1, a.nq
    t0 = time.time()
    gen = data.SyntheticGen("sift", d=d, kc=a.kc, device=dev)
    nt = min(C * 64, 4 * a.n)
    xt = torch.cat([gen.chunk(7000 + i, min(1 << 20, nt - i * (1 << 20))) for i in range((nt + (1 << 20) - 1) >> 20)])
    cent, _ = train.kmeans(xt, C, niter=a.train_iters, exact_perm=False)  # = train_vlq's first step in bench.py
    del xt
    cn = ops.row_norms(cent)
    edge, ed2 = ops.knn_graph(cent, E, cn)
    xq = gen.chunk(3, nq)
    torch.cuda.synchronize()
    print("[locality] trained C=%d in %.1f s" % (C, time.time() - t0), file=sys.stderr, flush=True)
    nb = ops.num_buckets(C)
    scale = ops.CentPack(cent, cn).scale

    cent_h, edge_h = cent.cpu().numpy(), edge.cpu().numpy()
    orders = {"identity": (np.arange(C, dtype=np.int64), 0.0)}
    t0 = time.perf_counter()
    o = order_bisection(cent_h)
    orders["bisection"] = (o, time.perf_counter() - t0)
    t0 = time.perf_counter()
    o = order_rcm(edge_h)
    orders["rcm"] = (o, time.perf_counter() - t0)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    tiles = [(s, min(nq, s + a.tile)) for s in range(0, nq, a.tile)]
    ref_cid = None
    D_id0 = None
    res = {}
    for name, (col2id_h, build_s) in orders.items():
        assert np.array_equal(np.sort(col2id_h), np.arange(C)), name
        col2id = torch.from_numpy(col2id_h).to(dev)
        id2col = torch.empty_like(col2id)
        id2col[col2id] = torch.arange(C, device=dev)
        cent_l, cn_l = cent[col2id].contiguous(), cn[col2id].contiguous()
        edge_l = id2col[edge[col2id].long()].to(torch.int32).contiguous()
        ed2_l = ed2[col2id].contiguous()
        pack_l = ops.CentPack(cent_l, cn_l, scale=scale)
        Ds, bms = [], []
        for s, e in tiles:
            bm = torch.empty((e - s, nb), dtype=torch.float32, device=dev)
            Ds.append(ops.l2_distances_tc(xq[s:e], pack_l, bucket_min=bm))
            bms.append(bm)
        if name == "identity":
            D_id0 = Ds[0][:256].clone()
        invariant = bool(torch.equal(Ds[0][:256], D_id0[:, col2id]))
        # device counts per query
        acc = {k: [] for k in ("nbr_segments", "nbr_lines", "union_segments", "union_lines", "nbr_segments_outside_buckets",
                               "stage2_candidates")}
        cids = []
        for (s, e), D, bm in zip(tiles, Ds, bms):
            n = e - s
            _, _, _, cid = ops.coarse_select_lines(D, bm, C, P, edge_l, ed2_l, W, want_coarse=True)
            cids.append(col2id[cid.long()])
            bv, bk = torch.topk(bm, P, dim=1, largest=False, sorted=True)
            tau1 = bv[:, -1]
            cols = (bk.long() * 32).unsqueeze(2) + torch.arange(32, device=dev)
            valid = cols < C
            vals = D.gather(1, cols.clamp_max(C - 1).view(n, -1)).view(n, P, 32)
            acc["stage2_candidates"].append(((vals <= tau1.view(n, 1, 1)) & valid).sum(dim=(1, 2)))
            nbr = edge_l[cid.long()].long().view(n, P * E)
            seg_b = (bk.long() * 2).unsqueeze(2) + torch.arange(2, device=dev)
            seg_b = seg_b.view(n, 2 * P)
            seg_n = nbr // 16
            acc["nbr_segments"].append(distinct_per_row(seg_n))
            acc["nbr_lines"].append(distinct_per_row(nbr // 32))
            u = distinct_per_row(torch.cat([seg_b, seg_n], dim=1))
            acc["union_segments"].append(u)
            acc["union_lines"].append(distinct_per_row(torch.cat([bk.long(), nbr // 32], dim=1)))
            acc["nbr_segments_outside_buckets"].append(u - 2 * P)
        cid_all = torch.cat(cids)
        if ref_cid is None:
            ref_cid = cid_all
        same_topp = float((cid_all == ref_cid).all(dim=1).float().mean())
        row = {k: float(torch.cat(v).float().mean()) for k, v in acc.items()}
        row["stage2_candidates_max"] = int(torch.cat(acc["stage2_candidates"]).max())
        row["bmin_row_segments"] = (nb * 4 + 63) // 64
        row["total_segments"] = row["union_segments"] + row["bmin_row_segments"]
        row["build_s"] = build_s
        row["D_invariant_bitwise"] = invariant
        row["topP_same_as_identity"] = same_topp
        # the unmodified select kernel on the relabelled tile
        times = []
        for rep in range(a.reps + 1):
            evs = []
            for (s, e), D, bm in zip(tiles, Ds, bms):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ops.coarse_select_lines(D, bm, C, P, edge_l, ed2_l, W)
                e1.record()
                evs.append((e0, e1))
            torch.cuda.synchronize()
            if rep:
                times.append(sum(x.elapsed_time(y) for x, y in evs))
        row["select_ms_per_%d_queries" % nq] = float(np.median(times))
        row["select_ms_min"] = float(min(times))
        row["select_ms_max"] = float(max(times))
        res[name] = row
        print("[locality]", name, json.dumps(row), file=sys.stderr, flush=True)
        del Ds, bms
        torch.cuda.empty_cache()
    base = res["identity"]
    for name, row in res.items():
        row["union_segments_vs_identity"] = row["union_segments"] / base["union_segments"]
        row["total_segments_vs_identity"] = row["total_segments"] / base["total_segments"]
    best = min((n_ for n_ in res if n_ != "identity"), key=lambda n_: res[n_]["union_segments"])
    props = torch.cuda.get_device_properties(0)
    out = {"config": {"nlist": C, "nedge": E, "d": d, "nq": nq, "nprobe": P, "w1": W, "train_iters": a.train_iters,
                      "tile": a.tile, "data": "synthetic SIFT-shaped, bench.py generator"},
           "gpu": props.name, "orders": res, "best": best,
           "go": res[best]["union_segments_vs_identity"] <= 1.0 / 3.0}
    try:
        import subprocess

        out["power_limit_w"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                              capture_output=True, text=True).stdout.strip()
    except Exception:
        pass
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
