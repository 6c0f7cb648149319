#!/usr/bin/env python
"""Read-back micro-benchmark: id lookup, entry decode, and search_and_reconstruct beside search.

Ops level: SYNTHETIC list slabs (tools/bench_scan.py::synthetic_lists, random codes / lambda bytes, ids 0 .. n-1, M = 16,
d = 128) at the C2 geometry (10 M entries over 65536 x 32 lists) and at the BASELINE configs[3] list density (1 B
entries over 2 Mi lists, as tools/bench_remove.py builds it).  vlq_lookup_ids by range and by batch (sorted random
keys) for 1 k and 1 M keys, and vlq_decode_entries of 1 M random slab indexes, each between CUDA events (median of
--reps after one warm-up call).  Algorithmic bytes: the lookup reads 8 B of ids per entry (one pass over the slab's
ids, whatever the number of keys); the decode reads M + 1 + 8 B per row from HBM (code bytes, lambda byte, id) and
writes 4 d B; centroid and codebook rows are gathers that hit L2.  The 1 B slab (29 GB) does not fit L2; the ids of
the 10 M slab (80 MB) do, so its lookup times are L2 numbers.
Host level: GpuIndexIVFPQ at the bench.py C2 setting (--host-entries vectors, nlist 65536, E 32, nprobe 64, w1 256,
k 100, 10 k queries, device buffers): wall time of search and of search_and_reconstruct (1 M decodes), alternated,
median of --reps after one warm-up call each, with the two results compared bit for bit.

  python tools/bench_reconstruct.py [--entries 1e9] [--host-entries 1e7] [--out FILE]
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


def ops_level(a, rows, geom, entries, nlists):
    from bench_scan import synthetic_lists

    from vector_line_quantization_b200 import _abi, data, ops

    dev = torch.device("cuda:0")
    M, d, E = 16, 128, 32
    lists, _, _ = synthetic_lists(ops, entries, nlists, M, dev, seed=1)
    n = lists.ids.numel()
    g = torch.Generator(device=dev).manual_seed(2)
    st = torch.cuda.current_stream().cuda_stream
    pos = torch.empty(1 << 20, dtype=torch.int64, device=dev)
    found = torch.empty(1, dtype=torch.int64, device=dev)
    for nk in (1000, 1 << 20):
        keys = torch.unique(torch.randint(0, n, (nk,), generator=g, device=dev))
        lo = n // 3
        for mode in ("range", "batch"):
            kp, ns = (0, nk) if mode == "range" else (keys.data_ptr(), keys.numel())
            ms, alls = timed(lambda: _abi.call("vlq_lookup_ids", n, lists.ids.data_ptr(), lo, kp, ns, pos.data_ptr(),
                                               found.data_ptr(), st), a.reps)
            gb = 8.0 * n / 1e9
            rows.append(dict(level="ops", what="lookup_ids", geometry=geom, mode=mode, keys=ns, entries=n, nlists=nlists,
                             found=int(found), ms=ms, ms_all=alls, GBs=gb / ms * 1e3, frac_of_peak=gb / ms * 1e3 / PEAK))
            print(json.dumps(rows[-1]), flush=True)
    C = nlists // E
    cent = data.sift_like_torch(C, d, seed=11, device=dev)
    edge = torch.randint(0, C, (C, E), generator=g, device=dev, dtype=torch.int32)
    lcb = torch.linspace(-0.5, 1.5, 256, device=dev)
    pq = torch.rand((M, 256, d // M), generator=g, device=dev) * 40.0 - 20.0
    rpos = torch.randint(0, n, (1 << 20,), generator=g, device=dev)
    out = torch.empty((1 << 20, d), dtype=torch.float32, device=dev)
    oid = torch.empty(1 << 20, dtype=torch.int64, device=dev)
    ms, alls = timed(lambda: _abi.call(
        "vlq_decode_entries", rpos.numel(), rpos.data_ptr(), nlists, lists.offsets.data_ptr(), lists.codes.data_ptr(),
        lists.lamq.data_ptr(), lists.ids.data_ptr(), M, d, pq.data_ptr(), cent.data_ptr(), edge.data_ptr(), E,
        lcb.data_ptr(), 256, out.data_ptr(), oid.data_ptr(), st), a.reps)
    gb = rpos.numel() * (M + 1 + 8 + 4 * d) / 1e9
    rows.append(dict(level="ops", what="decode_entries", geometry=geom, rows=rpos.numel(), entries=n, nlists=nlists,
                     ms=ms, ms_all=alls, GBs=gb / ms * 1e3, frac_of_peak=gb / ms * 1e3 / PEAK))
    print(json.dumps(rows[-1]), flush=True)
    del lists, out
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
    D1, I1, R = idx.search_and_reconstruct(xq, k)
    same = bool(torch.equal(D0.view(torch.int32), D1.view(torch.int32)) and torch.equal(I0, I1))
    ts, tr = [], []
    for _ in range(a.reps):
        for fn, acc in ((lambda: idx.search(xq, k), ts), (lambda: idx.search_and_reconstruct(xq, k), tr)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            acc.append((time.perf_counter() - t0) * 1e3)
    rows.append(dict(level="host", what="search vs search_and_reconstruct", entries=idx.ntotal, nlist=C, nedge=E,
                     nprobe=64, w1=256, k=k, nq=nq, decodes=nq * k, search_ms=float(np.median(ts)),
                     search_and_reconstruct_ms=float(np.median(tr)), search_ms_all=ts,
                     search_and_reconstruct_ms_all=tr, D_I_bit_identical=same,
                     nan_rows=int(torch.isnan(R[..., 0]).sum())))
    print(json.dumps(rows[-1]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=float, default=1e9)
    ap.add_argument("--nlists", type=int, default=1 << 21)
    ap.add_argument("--host-entries", type=float, default=1e7)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_reconstruct.py needs a CUDA device")
    rows = []
    info = dict(card=card(), peak_GBs=PEAK)
    print(json.dumps(info), flush=True)
    ops_level(a, rows, "C2", 1e7, 65536 * 32)
    ops_level(a, rows, "configs[3] density", a.entries, a.nlists)
    host_level(a, rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(dict(info, results=rows), f, indent=1)


if __name__ == "__main__":
    main()
