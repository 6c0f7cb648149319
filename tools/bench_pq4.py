#!/usr/bin/env python
"""4-bit against 8-bit PQ codes at the C2 setting (10 M SIFT-shaped vectors, nlist 65 536, E 32, nprobe 64, w1 256,
k 100, 10 k device queries), for (M 16, 8-bit), (M 8, 8-bit), (M 16, 4-bit) and (M 32, 4-bit): two pairs at equal
bytes per entry.  Per configuration: queries/s through GpuIndexIVFPQ::search (device queries and outputs, CUDA events),
R@1/10/100 against the exact fp32 kNN, the oracle's recall on the same entries for a query subset (the CPU restatement
of the search, oracle/vlq_oracle.c), encode Mvec/s through GpuIndexIVFPQ::add_with_ids (device input) and bytes per
entry.  Then the scan stage alone at 1 B list density (synthetic lists as tools/bench_scan.py) for M 32 x 4-bit against
M 16 x 8-bit: the same kernel on the same 16 code bytes per entry, so the difference is the table build.

  python tools/bench_pq4.py [--n 10000000] [--oracle-queries 100] [--out profiles/r11_pq4.json]

Without --out the result document is printed as the last line; the script writes nothing else.
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

CONFIGS = [(16, 8), (8, 8), (16, 4), (32, 4)]  # (M, bits)


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "unavailable: %s" % e


def exact_knn(xb, xq, k):
    """exact fp32 top-k by ||x||^2 - 2 q.x (the squared L2 without ||q||^2; tiles of the database, no TF32)"""
    torch.backends.cuda.matmul.allow_tf32 = False
    bestD = torch.full((xq.shape[0], k), float("inf"), device=xq.device)
    bestI = torch.full((xq.shape[0], k), -1, dtype=torch.int64, device=xq.device)
    for s in range(0, xb.shape[0], 1 << 17):
        x = xb[s:s + (1 << 17)]
        d = torch.addmm((x * x).sum(1)[None], xq, x.T, alpha=-2.0)
        D = torch.cat([bestD, d], 1)
        I = torch.cat([bestI, torch.arange(s, s + x.shape[0], device=xq.device).expand(xq.shape[0], -1)], 1)
        bestD, j = D.topk(k, dim=1, largest=False)
        bestI = I.gather(1, j)
    return bestI


def recalls(I, gt):
    I, gt = np.asarray(I), np.asarray(gt)
    return {"R@%d" % r: float(np.mean([len(set(a[:r]) & {g[0]}) for a, g in zip(I, gt)])) for r in (1, 10, 100)}


def timed(fn, steps):
    fn()
    ms = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10_000_000)
    ap.add_argument("--nlist", type=int, default=65536)
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--oracle-queries", type=int, default=100)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--scan-entries", type=float, default=1e9)
    ap.add_argument("--out", default=None, help="write the result document (JSON) to this path")
    a = ap.parse_args()
    from vector_line_quantization_b200 import _abi, data, index as vi, ops, train
    from oracle import pyoracle

    _abi.lib()
    dev = torch.device("cuda:0")
    d, C, E, nL, P, W, k = 128, a.nlist, 32, 256, 64, 256, 100
    out = {"gpu": gpu_info(), "setting": dict(n=a.n, d=d, nlist=C, E=E, nprobe=P, w1=W, k=k, nq=a.nq), "configs": []}
    print(out["gpu"], flush=True)
    gen = data.SyntheticGen("sift", d=d, kc=1 << 18, device=dev)
    nt = min(C * 64, 4 * a.n)
    xt = torch.cat([gen.chunk(7000 + i, min(1 << 20, nt - i * (1 << 20))) for i in range((nt + (1 << 20) - 1) >> 20)])
    xb = torch.cat([gen.chunk(i, min(1 << 20, a.n - i * (1 << 20))) for i in range((a.n + (1 << 20) - 1) >> 20)])
    xq = gen.chunk(999_999, a.nq)
    gt = exact_knn(xb, xq, 1).cpu().numpy()
    ids = torch.arange(a.n, dtype=torch.int64, device=dev)
    res = vi.StandardGpuResources(0)
    base = None
    for M, bits in CONFIGS:
        t0 = time.time()
        if base is None:  # one coarse quantizer, graph and lambda codebook for every configuration
            model = base = train.train_vlq(xt, C, E, M, nL, nbits=bits, niter=10, pq_niter=10, exact_perm=False)
        else:  # only the PQ codebook differs: trained as train_vlq does, on the first 2^bits * 128 residuals
            model = dict(base)
            A = ops.l2_assign(xt[:(1 << bits) * 128], base["cent"], base["cnorm"])[0]
            enc = ops.line_encode(xt[:(1 << bits) * 128], A, base["cent"], base["edge"], base["edge_d2"],
                                  base["lambda_cb"], torch.zeros((M, 1 << bits, d // M), device=dev), want_residual=True)
            pq = torch.empty((M, 1 << bits, d // M), device=dev)
            for m in range(M):
                pq[m], _ = train.kmeans(enc.residual[:, m * (d // M):(m + 1) * (d // M)].contiguous(), 1 << bits,
                                        niter=10, exact_perm=False)
            model["pq"] = pq
        cb = {key: model[key].cpu().numpy() for key in ("cent", "edge", "edge_d2", "lambda_cb", "pq")}
        g = vi.GpuIndexIVFPQ(res, d, C, M, bits, E, nL)
        g.setCodebooks(cb["cent"], cb["edge"], cb["edge_d2"], cb["lambda_cb"], cb["pq"])
        g.setNumProbes(P)
        g.w1_ = W
        torch.cuda.synchronize()
        t_train = time.time() - t0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.add_with_ids(xb, ids)
        e1.record()
        torch.cuda.synchronize()
        enc_ms = e0.elapsed_time(e1)
        D = torch.empty((a.nq, k), dtype=torch.float32, device=dev)
        I = torch.empty((a.nq, k), dtype=torch.int64, device=dev)
        ms = timed(lambda: g.search(xq, k, out=(D, I)), a.steps)
        rec = recalls(I.cpu().numpy(), gt)
        # the oracle's recall on the same entries (same kernels, same codebooks) for the first queries
        pack = ops.CentPack(model["cent"], model["cnorm"])  # the index's add path assigns on the tensor cores too
        A = torch.cat([ops.l2_assign_tc(xb[s:s + (1 << 20)], pack, want_dist=False)[0] for s in range(0, a.n, 1 << 20)])
        lst_enc = ops.line_encode(xb, A, model["cent"], model["edge"], model["edge_d2"], model["lambda_cb"], model["pq"])
        codes = ops.unpack_pq4(lst_enc.codes) if bits == 4 else lst_enc.codes
        e_list = lst_enc.list.cpu().numpy()
        off, perm = pyoracle.build_lists(e_list, C * E)
        nqo = a.oracle_queries
        Do, Io = pyoracle.search(xq[:nqo].cpu().numpy(), cb["cent"], cb["edge"], cb["edge_d2"], cb["lambda_cb"], cb["pq"],
                                 off, codes.cpu().numpy()[perm], lst_enc.lamq.cpu().numpy()[perm], perm.astype(np.int64),
                                 P=P, W=W, k=k)
        row = dict(M=M, bits=bits, bytes_per_entry=M * bits // 8 + 1 + 4 + 8, qps=a.nq / (min(ms) * 1e-3),
                   search_ms=ms, encode_mvecs=a.n / (enc_ms * 1e-3) / 1e6, encode_ms=enc_ms, train_s=t_train,
                   recall=rec, recall_gpu_on_oracle_queries=recalls(I[:nqo].cpu().numpy(), gt[:nqo]),
                   recall_oracle=recalls(Io, gt[:nqo]), oracle_queries=nqo)
        print(json.dumps(row), flush=True)
        out["configs"].append(row)
        del g, lst_enc, codes
        torch.cuda.empty_cache()
    del xb, xt
    torch.cuda.empty_cache()
    # ---- the scan stage alone at 1 B list density: M 16 x 8-bit and M 32 x 4-bit read 16 code bytes per entry
    from bench_scan import synthetic_lists

    nlists, nq = 1 << 21, a.nq
    lists, lens, lens_full = synthetic_lists(ops, int(a.scan_entries), nlists, 16, dev)
    gq = torch.Generator(device=dev).manual_seed(7)
    line = torch.multinomial(lens_full.float() + 1e-3, nq * W, replacement=True, generator=gq).reshape(nq, W).int()
    q = torch.randn(nq, d, device=dev, generator=gq)
    lcb = torch.rand(256, device=dev, generator=gq)
    t1 = torch.rand(nq, W, device=dev, generator=gq) * 10
    t6 = torch.randn(nq, W, device=dev, generator=gq)
    ed2 = torch.rand(nlists, device=dev, generator=gq) * 4 + 0.5
    hint = int(a.scan_entries / nlists)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    scan = {}
    pqs = {"M16_8bit": torch.randn(16, 256, d // 16, device=dev, generator=gq),
           "M32_4bit": torch.randn(32, 16, d // 32, device=dev, generator=gq)}
    oD = torch.empty((nq, k), dtype=torch.float32, device=dev)
    oI = torch.empty((nq, k), dtype=torch.int64, device=dev)
    for rep in range(3):  # alternated, so that drift on a shared machine hits both
        for name, pq in pqs.items():
            def run():
                flush.fill_(1)
                for s in range(0, nq, 4096):
                    e = min(nq, s + 4096)
                    ops.scan_topk(q[s:e], pq, lcb, line[s:e], t1[s:e], t6[s:e], ed2, lists, k, 1024,
                                  list_len_hint=hint, out=(oD[s:e], oI[s:e]))
            scan.setdefault(name, []).extend(timed(run, 2))
    out["scan_1B"] = dict(entries=int(lists.ids.shape[0]), nlists=nlists, nq=nq, hint=hint,
                          ms={n_: v for n_, v in scan.items()}, ms_min={n_: min(v) for n_, v in scan.items()},
                          note="each time includes a 256 MiB L2 flush (memset) before the tiles")
    print(json.dumps(out["scan_1B"]), flush=True)
    out["gpu_after"] = gpu_info()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    else:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
