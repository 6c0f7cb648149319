#!/usr/bin/env python
"""Refinement (GpuIndexIVFPQR) at the bench.py C2 setting: recall and wall time against GpuIndexIVFPQ, and the re-rank
epilogue alone.

Setting: data.SyntheticGen("sift") as bench.py draws it (training rows, 10 M database rows in 1 Mi blocks, 10 k queries),
codebooks trained on the device as bench.py does (train.train_vlq), nlist 65536, E 32, M 16, nLambda 256, nprobe 64,
w1 256; the refinement codebook (M2 16) is GpuIndexIVFPQR.train on the training rows.  Ground truth: the exact 1-NN by
brute force (fp32 l2_assign over database slices, as bench.py).  Both indexes hold the same 10 M vectors.

Host level, device buffers: for k in {10, 100}, GpuIndexIVFPQ.search and GpuIndexIVFPQR.search at k_factor 1, 2, 4, 8
are called in turn, --reps rounds after one warm-up round; each entry is the median wall time (host clock around the
call, which ends in a device synchronise) and R@1/10/100 (R@r = the true 1-NN among the first r labels).

Ops level: vlq_refine_topk alone between CUDA events (median of --reps after one warm-up), on a synthetic slab of the
same geometry (tools/bench_scan.py::synthetic_lists, 10 M entries over 65536 x 32 lists, random codes and refinement
codes, the trained tables) with uniformly random candidate slab indexes, 10 k queries, each (k, kc) of the host runs.
Bytes it must read from HBM per candidate: the 8 B slab index plus one 32 B sector each for the code word, the lambda
byte and the refinement code (random entries: every one is its own sector), 104 B; the table rows it gathers
(2 d fp32 of centroids, d of each codebook: 2 KiB per candidate at d = 128) come from L2 (the 32 MiB centroid table
and the codebooks fit in it).  The share of peak is the HBM bytes over the measured copy bandwidth (tools/bench_remove.py
PEAK), i.e. against the HBM bound; the L2 gather volume is reported beside it.

  python tools/bench_refine.py [--n 1e7] [--reps 5] [--out FILE]
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


def kc_of(k, kf):
    return min(1024, max(k, int(np.floor(k * np.float64(np.float32(kf))))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1e7)
    ap.add_argument("--nlist", type=int, default=65536)
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--train-iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_refine.py needs a CUDA device")
    from bench_scan import synthetic_lists

    from vector_line_quantization_b200 import _abi, data, index, ops, train

    dev = torch.device("cuda:0")
    n, C, E, M, M2, d, nL, P, W, nq = int(a.n), a.nlist, 32, 16, 16, 128, 256, 64, 256, a.nq
    info = dict(card=card(), peak_GBs=PEAK, n=n, nlist=C, nedge=E, M=M, M2=M2, nLambda=nL, nprobe=P, w1=W, nq=nq,
                reps=a.reps)
    print(json.dumps(info), flush=True)
    gen = data.SyntheticGen("sift", d=d, kc=1 << 18, device=dev)
    chunk = 1 << 20
    nt = min(C * 64, 4 * n)
    xt = torch.cat([gen.chunk(7000 + i, min(chunk, nt - i * chunk)) for i in range((nt + chunk - 1) // chunk)])
    t0 = time.time()
    model = train.train_vlq(xt, C, E, M, nL, niter=a.train_iters, pq_niter=10, exact_perm=False)
    cbs = [model[key].cpu().numpy() for key in ("cent", "edge", "edge_d2", "lambda_cb", "pq")]
    res = index.StandardGpuResources(0)
    base = index.GpuIndexIVFPQ(res, d, C, M, 8, E, nL)
    ref = index.GpuIndexIVFPQR(res, d, C, M, M2, 8, E, nL)
    for idx in (base, ref):
        idx.setCodebooks(*cbs)
    xr = xt[:32768].contiguous()
    torch.cuda.synchronize()
    ref.train(xr)
    del xt
    info["train_s"] = time.time() - t0
    for idx in (base, ref):
        idx.reserveMemory(n)
        idx.setNumProbes(P)
        idx.w1_ = W
    xq = gen.chunk(3, nq)
    gt_d = torch.full((nq,), float("inf"), device=dev)
    gt_i = torch.full((nq,), -1, dtype=torch.int64, device=dev)
    for c in range((n + chunk - 1) // chunk):
        xc = gen.chunk(1000003 + c, min(chunk, n - c * chunk))
        ids = torch.arange(c * chunk, c * chunk + xc.shape[0], dtype=torch.int64, device=dev)
        torch.cuda.synchronize()  # the host layer reads the rows on its own stream
        base.add_with_ids(xc, ids)
        ref.add_with_ids(xc, ids)
        for s in range(0, xc.shape[0], 1 << 18):
            i_, d_ = ops.l2_assign(xq, xc[s:s + (1 << 18)], add_xnorm=True)
            better = d_ < gt_d
            gt_d = torch.where(better, d_, gt_d)
            gt_i = torch.where(better, i_.to(torch.int64) + c * chunk + s, gt_i)
    gt = gt_i.cpu().numpy()
    torch.cuda.synchronize()  # xq is read by the host layer's stream below
    # memory per entry: first level M code bytes + lambda byte + 4 B kappa + 8 B id; the refinement adds M2 bytes
    info["bytes_per_entry"] = dict(ivfpq=M + 1 + 4 + 8, ivfpqr=M + 1 + 4 + 8 + M2)
    rows = []
    for k in (10, 100):
        D = torch.empty((nq, k), dtype=torch.float32, device=dev)
        I = torch.empty((nq, k), dtype=torch.int64, device=dev)
        calls = [("GpuIndexIVFPQ", None)] + [("GpuIndexIVFPQR", kf) for kf in (1.0, 2.0, 4.0, 8.0)]
        times = {c: [] for c in calls}
        recall = {}
        for rep in range(a.reps + 1):  # round 0 warms up
            for c in calls:
                idx = base if c[1] is None else ref
                if c[1] is not None:
                    ref.k_factor = c[1]
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                idx.search(xq, k, out=(D, I))
                torch.cuda.synchronize()
                if rep:
                    times[c].append((time.perf_counter() - t1) * 1e3)
                else:
                    In = I.cpu().numpy()
                    recall[c] = {"R@%d" % r: data.recall_at(In, gt, min(r, k)) for r in (1, 10, 100)}
        for c in calls:
            row = dict(level="host", index=c[0], k=k, k_factor=c[1], kc=None if c[1] is None else kc_of(k, c[1]),
                       search_ms=float(np.median(times[c])), search_ms_all=times[c], **recall[c])
            rows.append(row)
            print(json.dumps(row), flush=True)
    # ---- the re-rank alone
    lists, _, _ = synthetic_lists(ops, n, C * E, M, dev, seed=1)
    ne = lists.ids.numel()
    g = torch.Generator(device=dev).manual_seed(5)
    code2 = torch.randint(0, 256, (ne, M2), dtype=torch.uint8, device=dev, generator=g)
    cent, edge, lcb, pq = model["cent"], model["edge"], model["lambda_cb"], model["pq"]
    pq2 = torch.from_numpy(ref.refineCodebook()).to(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for k, kf in [(10, 1.0), (10, 4.0), (10, 8.0), (100, 1.0), (100, 4.0), (100, 8.0)]:
        kc = kc_of(k, kf)
        cand = torch.randint(0, ne, (nq, kc), dtype=torch.int64, device=dev, generator=g)
        ms = []
        for r in range(a.reps + 1):
            ev[0].record()
            ops.refine_topk(xq, cand, k, lists, code2, pq, cent, edge, lcb, pq2)
            ev[1].record()
            torch.cuda.synchronize()
            if r:
                ms.append(ev[0].elapsed_time(ev[1]))
        t = float(np.median(ms))
        hbm = nq * kc * (8 + 32 * 3) + nq * k * (4 + 8 + 8)  # candidates' sectors + outputs and their id reads
        l2 = nq * kc * 4 * 4 * d                              # 2 centroid rows + first- and second-level codebook rows
        row = dict(level="ops", what="vlq_refine_topk", entries=ne, k=k, k_factor=kf, kc=kc, ms=t, ms_all=ms,
                   hbm_bytes=hbm, hbm_GBs=hbm / t / 1e6, share_of_hbm_bound=hbm / t / 1e6 / PEAK, l2_gather_bytes=l2,
                   l2_gather_GBs=l2 / t / 1e6)
        rows.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(dict(info, results=rows), f, indent=1)


if __name__ == "__main__":
    main()
