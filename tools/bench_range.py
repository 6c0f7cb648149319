#!/usr/bin/env python
"""Radius-search micro-benchmark (vlq_range_count / vlq_range_gather) beside vlq_scan_topk (k = 100) on the same lines,
at two list densities on SYNTHETIC lists (tools/bench_scan.py's generator: random codes / lambda bytes / kappa, Poisson
list lengths with a Gamma(4) spread, size-biased line choice):
  c2  10 M entries over 65536 x 32 lines (the C2 index of bench.py: ~5 entries per line), w1 = 256
  1b  1 B entries over 2^21 lines (~477 entries per line), w1 = 256
For each density two radii are found by bisection on the count pass: one that keeps about 100 results per query and one
that keeps about 10 000 (beyond any k of search; capped at 90 % of the scanned entries where a query scans fewer).
Times are CUDA events around each pass, per query tile, with a 256 MiB buffer overwritten before each timed repetition
(the 10 M slab fits the 126 MB L2; the lines of a tile are read once per pass either way).  Algorithmic bytes: M + 5 per
scanned entry (codes, lambda byte, kappa) in each pass, plus 12 per result in the gather.

  python tools/bench_range.py [--density c2,1b] [--nq 10000] [--out DIR]   -> DIR/r04_range_search.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_PEAK_GBS = 6556.8  # measured on this card type (profiles/README.md)
DENSITIES = {"c2": (10_000_000, 65536 * 32), "1b": (1_000_000_000, 1 << 21)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # the numbers are still labelled with the torch device name
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--density", default="c2,1b")
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--w1", type=int, default=256)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--tile", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", required=True, help="directory that receives r04_range_search.json")
    a = ap.parse_args()
    from bench_scan import synthetic_lists

    from vector_line_quantization_b200 import _abi, ops

    lib = _abi.lib()
    dev = torch.device("cuda:0")
    M, W, d, nq, cap = a.m, a.w1, a.d, a.nq, 1024
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": card(), "hbm_peak_GBs": HBM_PEAK_GBS, "nq": nq, "w1": W, "M": M, "d": d, "tile": a.tile,
              "cap": cap, "lists": "synthetic (tools/bench_scan.py generator)", "runs": []}
    for name in a.density.split(","):
        n_target, nlists = DENSITIES[name]
        lists, lens, lens_full = synthetic_lists(ops, n_target, nlists, M, dev)
        g = torch.Generator(device=dev).manual_seed(7)
        line = torch.multinomial(lens_full.float() + 1e-3, nq * W, replacement=True, generator=g).reshape(nq, W)
        line = line.to(torch.int32).contiguous()
        q = torch.randn(nq, d, device=dev, generator=g)
        pq = torch.randn(M, 256, d // M, device=dev, generator=g)
        lcb = torch.rand(256, device=dev, generator=g)
        t1 = torch.rand(nq, W, device=dev, generator=g) * 10
        t6 = torch.randn(nq, W, device=dev, generator=g)
        ed2 = torch.rand(nlists, device=dev, generator=g) * 4 + 0.5
        scanned_q = lens.clamp_max(cap)[line.to(torch.int64)].sum(dim=1)
        scanned = float(scanned_q.float().mean())
        tiles = [(s, min(nq, s + a.tile)) for s in range(0, nq, a.tile)]
        wsb = lib.vlq_range_workspace_bytes(a.tile, M, W, cap)
        ws = torch.empty(max(wsb, lib.vlq_scan_topk_workspace_bytes(a.tile, M)), dtype=torch.uint8, device=dev)
        lims = torch.empty((len(tiles), a.tile + 1), dtype=torch.int64, device=dev)
        stream = torch.cuda.current_stream().cuda_stream

        def args(s, e, r):
            return (q[s:e].data_ptr(), e - s, d, pq.data_ptr(), M, lcb.data_ptr(), 256, line[s:e].data_ptr(),
                    t1[s:e].data_ptr(), t6[s:e].data_ptr(), ed2.data_ptr(), W, lists.offsets.data_ptr(),
                    lists.codes.data_ptr(), lists.lamq.data_ptr(), lists.kappa.data_ptr(), cap, None, float(r))

        def count(r, ti, lt):
            s, e = tiles[ti]
            _abi.call("vlq_range_count", *args(s, e, r), lt.data_ptr(), ws.data_ptr(), ws.numel(), stream)

        def per_query(r):  # mean results per query on the first tile
            count(r, 0, lims[0])
            return float(lims[0][tiles[0][1] - tiles[0][0]]) / (tiles[0][1] - tiles[0][0])

        def bisect(target):
            lo, hi = -1e4, 1e4
            for _ in range(20):
                if per_query(hi) >= target:
                    break
                hi *= 2
            for _ in range(40):
                mid = 0.5 * (lo + hi)
                if per_query(mid) < target:
                    lo = mid
                else:
                    hi = mid
            return hi

        outD = torch.empty((nq, 100), dtype=torch.float32, device=dev)
        outI = torch.empty((nq, 100), dtype=torch.int64, device=dev)

        def timed(fn):
            ms = []
            for rep in range(a.steps + 2):
                flush.fill_(rep)
                evs = []
                for ti in range(len(tiles)):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn(ti)
                    e1.record()
                    evs.append((e0, e1))
                torch.cuda.synchronize()
                if rep >= 2:  # the first two are warm-up
                    ms.append(sum(x.elapsed_time(y) for x, y in evs))
            return sum(ms) / len(ms), min(ms)

        def scan(ti):
            s, e = tiles[ti]
            _abi.call("vlq_scan_topk", q[s:e].data_ptr(), e - s, d, pq.data_ptr(), M, lcb.data_ptr(), 256,
                      line[s:e].data_ptr(), t1[s:e].data_ptr(), t6[s:e].data_ptr(), ed2.data_ptr(), W,
                      lists.offsets.data_ptr(), lists.codes.data_ptr(), lists.lamq.data_ptr(), lists.kappa.data_ptr(),
                      lists.ids.data_ptr(), 100, cap, int(n_target / nlists), outD[s:e].data_ptr(), outI[s:e].data_ptr(),
                      ws.data_ptr(), ws.numel(), stream)

        scan_ms, scan_best = timed(scan)
        for target in (100, min(10000, 0.9 * scanned)):
            r = bisect(target)
            for ti in range(len(tiles)):
                count(r, ti, lims[ti])
            totals = [int(lims[ti][e - s]) for ti, (s, e) in enumerate(tiles)]
            big = max(max(totals), 1)
            gD = torch.empty(big, dtype=torch.float32, device=dev)
            gI = torch.empty(big, dtype=torch.int64, device=dev)
            count_ms, count_best = timed(lambda ti: count(r, ti, lims[ti]))

            def gather(ti):
                s, e = tiles[ti]
                _abi.call("vlq_range_gather", *args(s, e, r), lists.ids.data_ptr(), lims[ti].data_ptr(), 0, e - s,
                          gD.data_ptr(), gI.data_ptr(), ws.data_ptr(), ws.numel(), stream)

            # the gather reads the tables the count pass left in the workspace: one tile at a time, count then gather
            def both(ti):
                count(r, ti, lims[ti])
                gather(ti)

            both_ms, both_best = timed(both)
            gather_ms = both_ms - count_ms
            results = sum(totals)
            count_bytes = nq * scanned * (M + 5)
            gather_bytes = count_bytes + 12 * results
            run = {
                "density": name, "entries": int(lists.ids.shape[0]), "lines": nlists, "avg_len": n_target / nlists,
                "scanned_per_query": scanned, "radius": r, "results_per_query": results / nq,
                "count_ms": count_ms, "count_ms_best": count_best, "gather_ms": gather_ms,
                "count_plus_gather_ms": both_ms, "scan_topk_k100_ms": scan_ms, "scan_topk_k100_ms_best": scan_best,
                "count_entries_per_s": nq * scanned / (count_ms * 1e-3),
                "gather_entries_per_s": nq * scanned / (gather_ms * 1e-3),
                "count_GBs": count_bytes / (count_ms * 1e-3) / 1e9, "gather_GBs": gather_bytes / (gather_ms * 1e-3) / 1e9,
            }
            run["count_frac_of_hbm_peak"] = run["count_GBs"] / HBM_PEAK_GBS
            run["gather_frac_of_hbm_peak"] = run["gather_GBs"] / HBM_PEAK_GBS
            result["runs"].append(run)
            print(json.dumps(run), flush=True)
        del lists, lens, lens_full
        torch.cuda.empty_cache()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r04_range_search.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
