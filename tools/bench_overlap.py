#!/usr/bin/env python
"""Co-residency of the coarse sweep with line selection and the scan (C2 geometry: C = 65536, d = 128, E = 32, M = 16,
nprobe 64, w1 256, k 100, 10 000 queries in 4 tiles of 2560 / 2320).  It asks whether a search pipeline that runs the
sweep of tile i + 1 on one stream beside line selection and the scan of tile i on another, from two distance-tile
slots, would pay.

CUDA-event times, ms per 10 000 queries, median of --reps runs with a 256 MiB L2 flush before each:
  sweep            vlq_l2_distances_tc of the 4 tiles on one stream (the tensor-core distance tile + bucket minima)
  select_scan      vlq_coarse_select_lines + vlq_scan_topk of the 4 tiles, each from its own swept tile (summed over
                   tiles timed one by one: informational, it carries a launch gap per tile)
  serial           sweep(i), select(i), scan(i) for every tile on one stream between one pair of events
  concurrent       sweep(i) on a high-priority stream, select(i) + scan(i) on a low-priority stream after it, two
                   distance-tile slots, between one pair of events: its span against the serial span
  search_overlap / search_no_overlap   GpuIndexIVFPQ::search on device buffers (a real encode of a 10 M database with
                   these codebooks), with the scan of a tile beside the next tile's coarse stage and with
                   VLQ_SEARCH_NO_OVERLAP set
--baseline-tree DIR: the sweep is also timed with the package of DIR (another revision, built), in a subprocess.
Co-residency shows only as a concurrent span shorter than the serial span.  At the sweep's 168 registers x 320 threads no
256-thread CTA of 64 registers fits beside it, so here `concurrent` measures how much the tails of the kernels overlap,
not co-residency.  Writes --out (.json and .md)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

C, D_, E, M, P, W, K, NQ, NDB = 65536, 128, 32, 16, 64, 256, 100, 10000, 10_000_000
TILE = 2560


def timed(fn, reps, flush):
    import torch

    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1]}


def sweep_only(reps):
    """the sweep through vlq_l2_distances_tc, which every revision has: comparable across register caps"""
    import torch

    from vector_line_quantization_b200 import data, ops

    dev = torch.device("cuda:0")
    cent = torch.from_numpy(data.sift_like(C, d=D_, kc=1024, seed=1)).to(dev)
    q = torch.from_numpy(data.sift_like(NQ, d=D_, kc=1024, seed=2)).to(dev)
    pack = ops.CentPack(cent)
    Db = torch.empty((TILE, C), dtype=torch.float32, device=dev)
    bm = torch.empty((TILE, ops.num_buckets(C)), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run():
        for s in range(0, NQ, TILE):
            m = min(NQ, s + TILE) - s
            ops.l2_distances_tc(q[s:s + m], pack, out=Db[:m], bucket_min=bm[:m])

    return timed(run, reps, flush)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as exc:  # the card is still named by torch below
        return "nvidia-smi unavailable (%s)" % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--sweep-only", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_overlap"))
    a = ap.parse_args()
    if a.sweep_only:  # run from the tree whose package is timed (see --baseline-tree)
        sys.path.insert(0, os.getcwd())
        print(json.dumps(sweep_only(a.reps)))
        return
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import torch

    from bench_scan import synthetic_lists
    from vector_line_quantization_b200 import data, index, ops

    dev = torch.device("cuda:0")
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": gpu_info() + " (name, power limit, SM clock, max SM clock)",
           "geometry": "C=%d d=%d E=%d M=%d nprobe=%d w1=%d k=%d nq=%d, tiles of %d" % (C, D_, E, M, P, W, K, NQ, TILE),
           "unit": "ms per %d queries (median / min / max of %d runs, L2 flushed before each)" % (NQ, a.reps)}
    res["sweep"] = sweep_only(a.reps)
    if a.baseline_tree:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_overlap.py"), "--sweep-only",
                              "--reps", str(a.reps)], capture_output=True, text=True, cwd=os.path.abspath(a.baseline_tree))
        res["sweep_baseline_tree"] = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else out.stderr[-2000:]

    cent = torch.from_numpy(data.sift_like(C, d=D_, kc=1024, seed=1)).to(dev)
    q = torch.from_numpy(data.sift_like(NQ, d=D_, kc=1024, seed=2)).to(dev)
    cn = ops.row_norms(cent)
    pack = ops.CentPack(cent, cn)
    edge, ed2 = ops.knn_graph(cent, E)
    ed2f = ed2.reshape(-1)
    lists, _, _ = synthetic_lists(ops, NDB, C * E, M, dev)
    g = torch.Generator(device=dev).manual_seed(7)
    pq = torch.randn(M, 256, D_ // M, device=dev, generator=g)
    lcb = torch.rand(256, device=dev, generator=g)
    nb = ops.num_buckets(C)
    Db = [torch.empty((TILE, C), dtype=torch.float32, device=dev) for _ in range(2)]
    bm = [torch.empty((TILE, nb), dtype=torch.float32, device=dev) for _ in range(2)]
    tiles = [(s, min(NQ, s + TILE)) for s in range(0, NQ, TILE)]
    ln = [tuple(torch.empty((TILE, W), dtype=dt, device=dev) for dt in (torch.int32, torch.float32, torch.float32))
          for _ in range(2)]
    outD = torch.empty((NQ, K), dtype=torch.float32, device=dev)
    outI = torch.empty((NQ, K), dtype=torch.int64, device=dev)
    hi = torch.cuda.Stream(priority=-1)
    lo = torch.cuda.Stream(priority=0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sweep(i, s, e):
        ops.l2_distances_tc(q[s:e], pack, out=Db[i & 1][:e - s], bucket_min=bm[i & 1][:e - s])

    def select(i, s, e):
        ops.coarse_select_lines(Db[i & 1][:e - s], bm[i & 1][:e - s], C, P, edge, ed2, W,
                                out=tuple(t[:e - s] for t in ln[i & 1]))

    def scan(i, s, e):
        lst, t1, t6 = (t[:e - s] for t in ln[i & 1])
        ops.scan_topk(q[s:e], pq, lcb, lst, t1, t6, ed2f, lists, K, 1024, list_len_hint=4, out=(outD[s:e], outI[s:e]))

    def select_scan(i, s, e):
        select(i, s, e)
        scan(i, s, e)

    def sweeps():
        for i, (s, e) in enumerate(tiles):
            sweep(i, s, e)

    res["sweep_two_slots"] = timed(sweeps, a.reps, flush)
    # select + scan alone, timed tile by tile: each tile is swept first, outside the timed region, so that every select
    # reads its own tile's distances
    ts = []
    for _ in range(a.reps):
        tot = 0.0
        for i, (s, e) in enumerate(tiles):
            sweep(i, s, e)
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            select_scan(i, s, e)
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        ts.append(tot)
    ts.sort()
    res["select_scan"] = {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1]}
    def serial():
        for i, (s, e) in enumerate(tiles):
            sweep(i, s, e)
            select_scan(i, s, e)

    res["serial"] = timed(serial, a.reps, flush)
    serial_ref = outI.clone()

    def concurrent():
        cur = torch.cuda.current_stream()
        hi.wait_stream(cur)
        lo.wait_stream(cur)
        released = [None, None]
        for i, (s, e) in enumerate(tiles):
            with torch.cuda.stream(hi):
                if released[i & 1] is not None:
                    hi.wait_event(released[i & 1])
                sweep(i, s, e)
                swept = torch.cuda.Event()
                swept.record(hi)
            with torch.cuda.stream(lo):
                lo.wait_event(swept)
                select(i, s, e)
                released[i & 1] = torch.cuda.Event()
                released[i & 1].record(lo)
                scan(i, s, e)
        cur.wait_stream(hi)
        cur.wait_stream(lo)

    res["concurrent"] = timed(concurrent, a.reps, flush)
    res["concurrent_matches_serial"] = bool(torch.equal(outI, serial_ref))
    res["saved_ms"] = res["serial"]["median"] - res["concurrent"]["median"]
    del Db, bm, lists
    torch.cuda.empty_cache()

    # whole search on the index (real encode of a 10 M database with these codebooks; the lists differ from the
    # synthetic ones above)
    gen = data.SyntheticGen("sift", d=D_, kc=1 << 18, device=dev)
    ir = index.StandardGpuResources(0)
    idx = index.GpuIndexIVFPQ(ir, D_, C, M, 8, E, 256)
    idx.setCodebooks(cent.cpu().numpy(), edge.cpu().numpy(), ed2.cpu().numpy(), lcb.cpu().numpy(), pq.cpu().numpy())
    for c in range(0, NDB, 1 << 20):
        x = gen.chunk(1000003 + (c >> 20), min(1 << 20, NDB - c))
        idx.add_with_ids(x, torch.arange(c, c + x.shape[0], dtype=torch.int64, device=dev))
    idx.setNumProbes(P)
    idx.w1_ = W
    xq = gen.chunk(3, NQ)
    dD = torch.empty((NQ, K), dtype=torch.float32, device=dev)
    dI = torch.empty((NQ, K), dtype=torch.int64, device=dev)
    out = {}
    searches = ("search_overlap", "search_no_overlap", "search_overlap_2", "search_no_overlap_2")
    for name in searches:
        off = "no_overlap" in name
        if off:
            os.environ["VLQ_SEARCH_NO_OVERLAP"] = "1"
        else:
            os.environ.pop("VLQ_SEARCH_NO_OVERLAP", None)
        res[name] = timed(lambda: idx.search(xq, K, out=(dD, dI)), a.reps, flush)
        out[off] = (dD.clone(), dI.clone())
    os.environ.pop("VLQ_SEARCH_NO_OVERLAP", None)
    res["search_overlap_matches_no_overlap"] = bool(torch.equal(out[False][0], out[True][0]) and
                                                    torch.equal(out[False][1], out[True][1]))
    res["nvidia_smi_after"] = gpu_info()

    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out + ".json", "w") as f:
        json.dump(res, f, indent=1)
    rows = [("sweep (vlq_l2_distances_tc, this revision)", res["sweep"])]
    if isinstance(res.get("sweep_baseline_tree"), dict):
        rows.append(("sweep (vlq_l2_distances_tc, --baseline-tree)", res["sweep_baseline_tree"]))
    rows += [("sweep, two distance-tile slots", res["sweep_two_slots"]), ("select + scan alone", res["select_scan"]),
             ("sweep, select + scan in order, one stream", res["serial"]),
             ("sweep || select + scan, two streams", res["concurrent"])]
    rows += [(n, res[n]) for n in searches]
    with open(a.out + ".md", "w") as f:
        f.write("# Coarse sweep beside line selection and the scan (tools/bench_overlap.py)\n\n")
        f.write("%s; %s.  %s; %s.\n\n" % (res["gpu"], res["nvidia_smi"], res["geometry"], res["unit"]))
        f.write("| what | median | min | max |\n|---|---:|---:|---:|\n")
        for n, r in rows:
            f.write("| %s | %.3f | %.3f | %.3f |\n" % (n, r["median"], r["min"], r["max"]))
        f.write("\nserial span %.3f ms; concurrent span %.3f ms; saved %.3f ms (tail overlap only at 168 registers).  "
                "Concurrent == serial bitwise: %s.  search overlap == no overlap bitwise: %s.\n"
                % (res["serial"]["median"], res["concurrent"]["median"], res["saved_ms"], res["concurrent_matches_serial"],
                   res["search_overlap_matches_no_overlap"]))


if __name__ == "__main__":
    main()
