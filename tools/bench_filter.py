#!/usr/bin/env python
"""Filtered-search benchmark: the mask pass (vlq_filter_kappa), filtered against unfiltered GpuIndexIVFPQ::search, and
the 1 B-density scan stage on a masked kappa.

Mask pass: SYNTHETIC slabs of 10 M and 1 B entries (ids a random permutation of 0 .. n-1, random kappa), a filter that
keeps about 10 % of the ids, given as a range, as a sorted batch (n / 10 random ids, one binary search per entry) and
as a bitmap (n / 8 bytes).  Between CUDA events, median of --reps after one warm-up call.  Algorithmic bytes: 16 B per
entry (8 B id + 4 B kappa read, 4 B written); the batch and bitmap reads come on top (L2 for the most part).  The ids
and kappa of the 10 M slab (120 MB) fit L2, those of the 1 B slab (12 GB) do not.
Host level: GpuIndexIVFPQ at the bench.py C2 setting (--host-entries vectors, nlist 65536, E 32, nprobe 64, w1 256,
k 100, 10 k device queries): search without a selector and with a random bitmap of 100 / 50 / 10 / 1 / 0.1 % of the
ids, alternated, host wall time around a device synchronise, median of --reps after a warm-up call each.
Scan stage: tools/bench_scan.py's synthetic 1 B-density lists (2 Mi lists, 10 k queries, w1 256, k 100, list length
hint 477: the long-list kernel), vlq_scan_topk per 4096-query tile between CUDA events on the plain kappa and on
random-bitmap masks keeping 10 % and 1 % of the ids, best and mean of --reps with L2 flushed before each.

  python tools/bench_filter.py [--entries 1e9] [--host-entries 1e7] [--out FILE]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_remove import PEAK, card  # noqa: E402


def random_bitmap(n, frac, g):
    """faiss IDSelectorBitmap bytes over the ids 0 .. n-1, each set with probability frac -> (uint8 tensor, members)"""
    bits = torch.zeros(((n + 7) // 8) * 8, dtype=torch.bool, device=g.device)
    bits[:n] = torch.rand(n, device=g.device, generator=g) < frac
    w = torch.arange(8, device=g.device, dtype=torch.int32)
    return (bits.reshape(-1, 8).to(torch.int32) << w).sum(1).to(torch.uint8), int(bits.sum())


def timed(fn, reps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    out = []
    for r in range(reps + 1):  # call 0 warms up
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        if r:
            out.append(ev[0].elapsed_time(ev[1]))
    return float(np.median(out)), out


def mask_pass(a, rows, n):
    from vector_line_quantization_b200 import _abi

    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(3)
    ids = torch.randperm(n, device=dev, generator=g)
    kappa = torch.randn(n, device=dev, generator=g)
    out = torch.empty(n, dtype=torch.float32, device=dev)
    batch = torch.sort(torch.randperm(n, device=dev, generator=g)[: n // 10]).values
    bitmap, _ = random_bitmap(n, 0.1, g)
    st = torch.cuda.current_stream().cuda_stream
    forms = dict(range=(0, n // 10, 0, 0, 0, 0), batch=(0, 0, batch.data_ptr(), batch.numel(), 0, 0),
                 bitmap=(0, 0, 0, 0, bitmap.data_ptr(), bitmap.numel()))
    for form, (lo, hi, bp, nb, mp, nm) in forms.items():
        ms, alls = timed(lambda: _abi.call("vlq_filter_kappa", n, ids.data_ptr(), kappa.data_ptr(), lo, hi, bp, nb, mp,
                                           nm, 0, out.data_ptr(), st), a.reps)
        kept = int(torch.isfinite(out).sum())
        gb = 16.0 * n / 1e9
        rows.append(dict(what="mask pass", form=form, entries=n, kept=kept, ms=ms, ms_all=alls, GBs=gb / ms * 1e3,
                         frac_of_peak=gb / ms * 1e3 / PEAK))
        print(json.dumps(rows[-1]), flush=True)
    del ids, kappa, out, batch, bitmap
    torch.cuda.empty_cache()


def host_level(a, rows):
    from vector_line_quantization_b200 import data, index, ops

    dev = torch.device("cuda:0")
    C, E, M, d, k, nq = 65536, 32, 16, 128, 100, 10000
    cent = data.sift_like_torch(C, d, seed=11, device=dev)
    edge, ed2 = ops.knn_graph(cent, E)
    g = torch.Generator(device=dev).manual_seed(12)
    pq = torch.rand((M, 256, d // M), generator=g, device=dev) * 40.0 - 20.0
    lam = np.linspace(-0.5, 1.5, 256).astype(np.float32)
    res = index.StandardGpuResources(0)
    idx = index.GpuIndexIVFPQ(res, d, C, M, 8, E, 256)
    idx.setCodebooks(cent.cpu().numpy(), edge.cpu().numpy(), ed2.cpu().numpy(), lam, pq.cpu().numpy())
    n = int(a.host_entries)
    for s in range(0, n, 1 << 22):
        idx.add(data.sift_like_torch(min(1 << 22, n - s), d, seed=100 + s, device=dev))
    idx.setNumProbes(64)
    idx.w1_ = 256
    xq = data.sift_like_torch(nq, d, seed=7, device=dev)
    D0, I0 = idx.search(xq, k)  # commits the adds, warms up
    for frac in (1.0, 0.5, 0.1, 0.01, 0.001):
        bm, members = random_bitmap(n, frac, g)
        sel = index.IDSelectorBitmap(bm)
        Df, If = idx.search(xq, k, sel=sel)  # warm-up
        ts, tf = [], []
        for _ in range(a.reps):
            for fn, acc in ((lambda: idx.search(xq, k), ts), (lambda: idx.search(xq, k, sel=sel), tf)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                acc.append((time.perf_counter() - t0) * 1e3)
        found = float((If >= 0).float().sum(1).mean())
        same = bool(torch.equal(Df.view(torch.int32), D0.view(torch.int32)) and torch.equal(If, I0)) if frac == 1.0 \
            else None
        rows.append(dict(what="search filtered vs unfiltered", selector="bitmap", selectivity=frac,
                         members=members, entries=idx.ntotal, nlist=C, nedge=E, nprobe=64, w1=256, k=k, nq=nq,
                         search_ms=float(np.median(ts)), filtered_ms=float(np.median(tf)), search_ms_all=ts,
                         filtered_ms_all=tf, mean_found_per_query=found, all_members_bit_identical=same))
        print(json.dumps(rows[-1]), flush=True)
    del idx
    torch.cuda.empty_cache()


def scan_stage(a, rows):
    from bench_scan import synthetic_lists

    from vector_line_quantization_b200 import ops

    dev = torch.device("cuda:0")
    M, W, k, nq, nlists, tile = 16, 256, 100, 10000, 1 << 21, 4096
    lists, lens, lens_full = synthetic_lists(ops, int(a.entries), nlists, M, dev)
    g = torch.Generator(device=dev).manual_seed(7)
    line = torch.multinomial(lens_full.float() + 1e-3, nq * W, replacement=True, generator=g).reshape(nq, W)
    line = line.to(torch.int32)
    q = torch.randn(nq, 128, device=dev, generator=g)
    pq = torch.randn(M, 256, 128 // M, device=dev, generator=g)
    lcb = torch.rand(256, device=dev, generator=g)
    t1 = torch.rand(nq, W, device=dev, generator=g) * 10
    t6 = torch.randn(nq, W, device=dev, generator=g)
    ed2 = torch.rand(nlists, device=dev, generator=g) * 4 + 0.5
    hint = int(a.entries / nlists)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    outD = torch.empty((nq, k), dtype=torch.float32, device=dev)
    outI = torch.empty((nq, k), dtype=torch.int64, device=dev)
    n = lists.ids.numel()
    for frac in (None, 0.1, 0.01):
        kap = None
        if frac is not None:  # the ids here are slab indexes: a random bitmap spreads the members over every list
            kap = ops.filter_kappa(lists, bitmap=random_bitmap(n, frac, g)[0])

        def run():
            evs = []
            for s in range(0, nq, tile):
                e = min(nq, s + tile)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ops.scan_topk(q[s:e], pq, lcb, line[s:e], t1[s:e], t6[s:e], ed2, lists, k, 1024, list_len_hint=hint,
                              out=(outD[s:e], outI[s:e]), kappa=kap)
                if kap is not None:
                    ops.filter_results(outD[s:e], outI[s:e])
                e1.record()
                evs.append((e0, e1))
            torch.cuda.synchronize()
            return sum(x.elapsed_time(y) for x, y in evs)

        run()
        ms = []
        for _ in range(a.reps):
            flush.fill_(1)
            ms.append(run())
        found = float((outI >= 0).float().sum(1).mean())
        rows.append(dict(what="scan stage", entries=n, nlists=nlists, hint=hint, nq=nq, w1=W, k=k,
                         filter=("none" if frac is None else "random bitmap, %g of the ids" % frac), ms_best=min(ms),
                         ms_mean=sum(ms) / len(ms), ms_all=ms, mean_found_per_query=found))
        print(json.dumps(rows[-1]), flush=True)
    del lists
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=float, default=1e9)
    ap.add_argument("--host-entries", type=float, default=1e7)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_filter.py needs a CUDA device")
    rows = []
    info = dict(card=card(), peak_GBs=PEAK)
    print(json.dumps(info), flush=True)
    mask_pass(a, rows, int(1e7))
    mask_pass(a, rows, int(a.entries))
    host_level(a, rows)
    scan_stage(a, rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(dict(info, results=rows), f, indent=1)


if __name__ == "__main__":
    main()
