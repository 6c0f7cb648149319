#!/usr/bin/env python
"""remove_ids micro-benchmark.

Ops level: a SYNTHETIC list slab (tools/bench_scan.py::synthetic_lists, random codes, ids 0 .. n-1) at the C4 list
density (1 B entries over 2 Mi lists, M = 16).  vlq_remove_ids_plan and vlq_remove_ids_apply are timed separately with
CUDA events (median of --reps after one warm-up round), for 0.1 %, 1 % and 10 % of the ids removed by batch (random ids,
sorted beforehand as ops.remove_ids does) and 10 % by range.  Algorithmic bytes: pass 1 reads the ids (8 B per entry);
pass 2 reads and writes 29 B per survivor (16 code bytes, lambda byte, kappa, id).  The slab (29 GB) does not fit L2.
Host level: GpuIndexIVFPQ.remove_ids on an index of --host-entries vectors (setCodebooks + add), the batch a host numpy
array: wall time of each call, i.e. what a user waits for (sort, copies, allocation and both passes); every fraction is
removed --host-rounds times in turn from the shrinking index.

  python tools/bench_remove.py [--entries 1e9] [--nlists 2097152] [--host-entries 1e7] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

PEAK = 6556.8  # GB/s: HBM copy bandwidth measured on the B200 (DESIGN.md, performance)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def time_passes(_abi, lists, batch, lo, hi, reps):
    """-> (plan ms list, apply ms list, survivors): the two C-ABI calls of ops.remove_ids, each between CUDA events"""
    offsets, ids = lists.offsets, lists.ids
    nlists, n, M = offsets.numel() - 1, ids.numel(), lists.codes.shape[1]
    dev = offsets.device
    wsb = _abi.lib().vlq_remove_ids_workspace_bytes(n, nlists)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    out_off = torch.empty(nlists + 1, dtype=torch.int64, device=dev)
    nb = 0 if batch is None else batch.numel()
    st = torch.cuda.current_stream().cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    tp, ta = [], []
    live = n
    for r in range(reps + 1):  # round 0 warms up
        ev[0].record()
        _abi.call("vlq_remove_ids_plan", nlists, n, offsets.data_ptr(), ids.data_ptr(), lo, hi,
                  0 if nb == 0 else batch.data_ptr(), nb, out_off.data_ptr(), ws.data_ptr(), wsb, st)
        ev[1].record()
        live = int(out_off[-1])
        rows = max(live, 1)
        out = [torch.empty((rows, M), dtype=torch.uint8, device=dev), torch.empty(rows, dtype=torch.uint8, device=dev),
               torch.empty(rows, dtype=torch.float32, device=dev), torch.empty(rows, dtype=torch.int64, device=dev)]
        ev[2].record()
        _abi.call("vlq_remove_ids_apply", nlists, M, n, offsets.data_ptr(), lists.codes.data_ptr(),
                  lists.lamq.data_ptr(), lists.kappa.data_ptr(), ids.data_ptr(), out_off.data_ptr(),
                  *(t.data_ptr() for t in out), ws.data_ptr(), wsb, st)
        ev[3].record()
        torch.cuda.synchronize()
        if r:
            tp.append(ev[0].elapsed_time(ev[1]))
            ta.append(ev[2].elapsed_time(ev[3]))
        del out
    return tp, ta, live


def ops_level(a, rows):
    from bench_scan import synthetic_lists

    from vector_line_quantization_b200 import _abi, ops

    dev = torch.device("cuda:0")
    lists, _, _ = synthetic_lists(ops, a.entries, a.nlists, 16, dev, seed=1)
    n = lists.ids.numel()
    g = torch.Generator(device=dev).manual_seed(2)
    cases = [("batch", f) for f in (0.001, 0.01, 0.1)] + [("range", 0.1)]
    for kind, frac in cases:
        k = int(n * frac)
        if kind == "batch":
            batch = torch.randperm(n, generator=g, device=dev)[:k].sort().values
            lo = hi = 0
        else:
            batch, lo, hi = None, n // 3, n // 3 + k
        tp, ta, live = time_passes(_abi, lists, batch, lo, hi, a.reps)
        del batch
        torch.cuda.empty_cache()
        p_ms, a_ms = float(np.median(tp)), float(np.median(ta))
        p_gb, a_gb = 8.0 * n / 1e9, 2 * 29.0 * live / 1e9
        rows.append(dict(level="ops", selector=kind, frac=frac, entries=n, nlists=a.nlists, removed=n - live,
                         plan_ms=p_ms, apply_ms=a_ms, plan_ms_all=tp, apply_ms_all=ta,
                         plan_GBs=p_gb / p_ms * 1e3, apply_GBs=a_gb / a_ms * 1e3,
                         plan_frac_of_peak=p_gb / p_ms * 1e3 / PEAK, apply_frac_of_peak=a_gb / a_ms * 1e3 / PEAK))
        print(json.dumps(rows[-1]), flush=True)
    del lists
    torch.cuda.empty_cache()


def host_level(a, rows):
    from vector_line_quantization_b200 import data, index, ops

    dev = torch.device("cuda:0")
    C, E, M, d = a.host_nlist, 32, 16, 128
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
    idx.search(np.zeros((1, d), np.float32), 1)  # commits the adds
    rng = np.random.RandomState(3)
    alive = np.arange(n, dtype=np.int64)  # add() numbered the vectors 0 .. n-1
    for frac in (0.001, 0.01, 0.1) * a.host_rounds:
        before = idx.ntotal
        pick = np.zeros(len(alive), bool)
        pick[rng.choice(len(alive), int(len(alive) * frac), replace=False)] = True
        sel = rng.permutation(alive[pick])
        alive = alive[~pick]
        t0 = time.perf_counter()
        removed = idx.remove_ids(sel)
        dt = (time.perf_counter() - t0) * 1e3
        rows.append(dict(level="host", selector="batch (host numpy)", frac=frac, entries=before, nlists=C * E,
                         removed=removed, wall_ms=dt))
        print(json.dumps(rows[-1]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=float, default=1e9)
    ap.add_argument("--nlists", type=int, default=1 << 21)
    ap.add_argument("--host-entries", type=float, default=1e7)
    ap.add_argument("--host-nlist", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-rounds", type=int, default=2, help="host level: times each fraction is removed (in turn)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_remove.py needs a CUDA device")
    rows = []
    info = dict(card=card(), peak_GBs=PEAK)
    print(json.dumps(info), flush=True)
    ops_level(a, rows)
    host_level(a, rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(dict(info, results=rows), f, indent=1)


if __name__ == "__main__":
    main()
