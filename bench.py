#!/usr/bin/env python
"""bench.py -- VLQ hot path on B200: search QPS (+ encode Mvec/s) for BASELINE.json configs[1]
(C=2^16 centroids, 32 neighbour lines, PQ m=16, synthetic SIFT-shaped 10M x 128 per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   our arm (one process per GPU under torchrun for N>1)
  python bench.py --impl reference [...]                          CPU arm: the reference's CPU code (IndexFlatL2 /
                                                                  ProductQuantizer from oracle/_ref) for the stock
                                                                  pieces + the oracle port for the VLQ-only search

A "step" is one pass of the search hot path (coarse top-P -> line selection -> ADC scan + top-k [-> line exchange +
peer merge for N>1]) over one batch of nq queries.  `value` (queries/s, merged, at every N) is timed with the inputs
resident in HBM; `e2e` goes through host (pinned) buffers with the H2D / D2H copies inside the timed region.
N > 1 is STRONG scaling by default: the same --n vector database is sharded N ways (--scaling weak keeps --n vectors
per GPU instead).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline device loop and of the e2e loop (the --sweep points and the "
                         "configs[3]-density scan stage time a fixed 3 and 5 steps)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "imipq"],
                    help="b200: this framework; reference: the CPU arm of the same metric; imipq: the reference's IMI-PQ "
                         "CPU baseline index of BASELINE configs[4] on a bounded sample (host cores only, its own metric)")
    ap.add_argument("--imi-bits", type=int, default=10, help="--impl imipq: bits per coarse sub-quantizer (2^(2*bits) cells)")
    ap.add_argument("--n", "--db-size", dest="n", type=int, default=10_000_000,
                    help="database vectors PER GPU (use --db-size under torchrun: its parser treats --n as ambiguous)")
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--nlist", type=int, default=65536)
    ap.add_argument("--nedge", type=int, default=32)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--nlambda", type=int, default=256)
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--nprobe", type=int, default=64)
    ap.add_argument("--w1", type=int, default=256)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--train-iters", type=int, default=10, help="coarse k-means iterations in the (untimed) setup "
                    "(the reference's default, gpu/GpuIndexIVF.cu:50)")
    ap.add_argument("--scaling", default=None, choices=["strong", "weak"],
                    help="N > 1: strong (default) = the --n database sharded N ways; weak = --n vectors per GPU")
    ap.add_argument("--shard-by", default="auto", choices=["auto", "ids", "lists"],
                    help="N > 1: ids = every rank holds all lists with its 1/N of the entries; lists = rank r owns the lists "
                         "[r L/N, (r+1) L/N) at full length (the reference's readDbFromFile(name, pronum, rank) split; "
                         "entries routed to the owner after the encode); auto = lists once the lists are long")
    ap.add_argument("--no-c4-stage", action="store_true",
                    help="skip the extra scan measurement at BASELINE configs[3] list density (1 B synthetic entries)")
    ap.add_argument("--kc", type=int, default=1 << 18, help="mixture components of the synthetic generator")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU-baseline budget in the default arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tc", action="store_true", help="use the exact fp32 CUDA-core kernels for the coarse stage")
    ap.add_argument("--shape", default="sift", choices=["sift", "deep"], help="sift: d=128 uint8-valued; deep: d=96 unit-norm (use --d 96 --m 8)")
    ap.add_argument("--u8", action="store_true", help="e2e encode ingests uint8 host vectors (add_with_ids_u8), sift shape only")
    ap.add_argument("--sweep", action="store_true",
                    help="also report recall@1/10/100 and QPS over nprobe = 1..64 with w1 = 4*nprobe (BASELINE configs[2])")
    ap.add_argument("--quick", action="store_true", help="small sizes (for debugging the script itself)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the search result of the last step (distances float32, labels "
                         "float64) as DIR/<name>.npy, at most 64 MB in all, to compare two builds output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the result of the GPU search path: --impl b200 only")
    if a.quick:
        a.n, a.nlist, a.nq, a.kc = 400_000, 4096, 2000, 1 << 14
    return a


# ------------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [t.strip() for t in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------------- CPU arm
def cpu_search_baseline(po, model, lists_host, xq, P, W, k, budget_s, gpu_result=None, gt=None, recall_at=None):
    """Times the oracle port of the VLQ search (the reference has no CPU VLQ) on a bounded sample of the queries,
    against the SAME index.  Returns the cpu_baseline object (+ a parity summary against the GPU results)."""
    T2 = po.term2(model["cent"], model["pq"])  # the reference precomputes this at train time (IVFPQ.cu:599-684)
    off, codes, lamq, ids = lists_host
    args = (model["cent"], model["edge"], model["edge_d2"], model["lambda_cb"], model["pq"], off, codes, lamq, ids)
    ncores = po.num_threads()
    probe = min(xq.shape[0], max(2 * ncores, 16))
    t0 = time.time()
    po.search(xq[:probe], *args, P=P, W=W, k=k, T2=T2)
    per_q = (time.time() - t0) / probe
    ns = int(min(xq.shape[0], max(probe, budget_s / max(per_q, 1e-9))))
    t0 = time.time()
    D, I = po.search(xq[:ns], *args, P=P, W=W, k=k, T2=T2)
    dt = time.time() - t0
    out = {"value": ns / dt, "unit": "queries/s", "cores": ncores, "kind": "port",
           "sample": "%d of the %d queries against the same %d-vector index (oracle/vlq_oracle.c:vlqo_search, OpenMP "
                     "over queries; the reference has no CPU implementation of VLQ search)" % (ns, xq.shape[0], len(ids))}
    parity = None
    if gpu_result is not None:
        gD, gI = gpu_result
        gD, gI = gD[:ns], gI[:ns]
        qn = (xq[:ns].astype(np.float64) ** 2).sum(1, keepdims=True)
        valid = (I >= 0) & (gI == I)  # distances compared where both sides return the same entry at the same rank
        rel = np.abs(gD - D)[valid] / (np.abs(D) + qn)[valid]
        parity = {"queries": ns, "id_match": float((gI == I)[I >= 0].mean()), "max_rel_dist_err": float(rel.max()),
                  "set_overlap": float(np.mean([len(set(a) & set(b)) / max(1, len(set(b))) for a, b in zip(gI, I)]))}
        if gt is not None:  # recall of both sides on the SAME queries of the SAME index (north_star: within 0.1 pt)
            rg = {"R@%d" % r: recall_at(gI, gt[:ns], min(r, k)) for r in (1, 10, 100)}
            ro = {"R@%d" % r: recall_at(I, gt[:ns], min(r, k)) for r in (1, 10, 100)}
            parity["recall_gpu"] = rg
            parity["recall_oracle"] = ro
            parity["recall_max_abs_delta"] = max(abs(rg[key] - ro[key]) for key in rg)
            parity["recall_within_0.001"] = parity["recall_max_abs_delta"] <= 1e-3
    return out, parity


class _StdoutToStderr:
    """the reference library printf()s progress lines; keep fd 1 clean for the ONE JSON line"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def _all_host_cores():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arms use every core of the box (must run before the
    OpenMP runtime of the oracle / reference libraries is loaded)"""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    for key in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[key] = str(n)
    return n


def run_reference(a):
    """--impl reference: everything on the host cores; no CUDA library is loaded."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _all_host_cores()
    with _StdoutToStderr():
        line = _run_reference(a)
    print(json.dumps(line))


def run_imipq(a):
    """--impl imipq: BASELINE configs[4] on a bounded sample -- the reference's IMI-PQ baseline index
    (MultiIndexQuantizer(d, 2, bits) + IndexIVFPQ, the UNMODIFIED reference CPU classes through oracle/_ref,
    tests/sift1b_imi_pq.cpp:216-236) on the host cores, beside the SAME index on the GPU (GpuIndexIMIPQ with the
    reference-trained codebooks: identical cells and codes, so equal recall and a like-for-like speed ratio) and the VLQ
    index at (almost) equal bytes per vector (M code bytes + 1 lambda byte) on the same vectors."""
    _all_host_cores()
    with _StdoutToStderr():
        from oracle import pyoracle as po
        from vector_line_quantization_b200 import data

        d, M, k = a.d, a.m, a.k
        nb = min(a.n, 1_000_000)
        nt = min(nb, 200_000)
        nq = min(a.nq, 2000)
        xt = data.sift_like(nt, d=d, kc=a.kc, seed=1)
        xb = data.sift_like(nb, d=d, kc=a.kc, seed=2)
        xq = data.sift_like(nq, d=d, kc=a.kc, seed=3)
        t0 = time.time()
        idx = po.RefIMIPQ(d, a.imi_bits, M)
        idx.train(xt)
        t_train = time.time() - t0
        t0 = time.time()
        idx.add(xb)
        t_add = time.time() - t0
        gt = po.ref_flat_search(xb, xq, 1)[1][:, 0]
        probes = (8, 64, 512)

        def sweep_of(search, reps=1):
            out = []
            for nprobe in probes:
                search(xq[:64], nprobe)
                t0 = time.time()
                for _ in range(reps):
                    D, I = search(xq, nprobe)
                dt = (time.time() - t0) / reps
                out.append({"nprobe": nprobe, "qps": nq / dt, "R@1": data.recall_at(I, gt, 1),
                            "R@10": data.recall_at(I, gt, 10), "R@100": data.recall_at(I, gt, min(100, k))})
                print("[bench] imipq", out[-1], file=sys.stderr, flush=True)
            return out

        cpu_sweep = sweep_of(lambda q, p_: idx.search(q, k, p_))
        gpu_sweep, vlq_sweep, gpu_note = None, None, None
        try:
            import torch

            if torch.cuda.is_available():
                from vector_line_quantization_b200 import _abi, index as vi

                _abi.lib()
                res = vi.StandardGpuResources(0)
                g = vi.GpuIndexIMIPQ(res, d, a.imi_bits, M)
                g.setCodebooks(*idx.codebooks())  # the reference-trained codebooks: the same index on both sides
                t0 = time.time()
                g.add(xb)
                g.search(xq[:8], k)
                t_gadd = time.time() - t0

                def gsearch(q, p_):
                    g.setNumProbes(p_)
                    return g.search(q, k)

                gpu_sweep = sweep_of(gsearch, reps=5)
                gpu_note = {"add_vec_per_s": nb / t_gadd, "api": "GpuIndexIMIPQ::search, host buffers"}
                # VLQ at equal code bytes on the same vectors (device-trained codebooks)
                C_, E_ = min(a.nlist, 16384), a.nedge
                v = vi.GpuIndexIVFPQ(res, d, C_, M, 8, E_, a.nlambda)
                v.setTrainIters(10)
                v.train(xt)
                v.add(xb)

                def vsearch(q, p_):
                    v.setNumProbes(p_)
                    v.w1_ = min(1024, 4 * p_)
                    return v.search(q, k)

                vlq_sweep = sweep_of(vsearch, reps=5)
                for s_, p_ in zip(vlq_sweep, probes):
                    s_["w1"] = min(1024, 4 * p_)
                gpu_note["vlq"] = {"nlist": C_, "nedge": E_, "bytes_per_vector": M + 1}
        except Exception as exc:
            gpu_note = {"error": "%s: %s" % (type(exc).__name__, exc)}
        mid = cpu_sweep[1]
        line = {"impl": "imipq", "metric": "imipq_search_qps", "value": mid["qps"], "unit": "queries/s",
                "higher_is_better": True, "data": "synthetic", "dtype": "f32",
                "config": {"workload": "BASELINE.json configs[4], bounded sample: IMI-PQ "
                                       "(MultiIndexQuantizer(d,2,%d) + IndexIVFPQ m=%d) on %d synthetic SIFT-shaped "
                                       "vectors, %d queries, k=%d" % (a.imi_bits, M, nb, nq, k),
                           "cells": 1 << (2 * a.imi_bits), "bytes_per_vector": M, "db_vectors": nb, "nq": nq},
                "cpu_baseline": {"value": mid["qps"], "unit": "queries/s", "cores": po.ref_num_threads(), "kind": "reference",
                                 "sample": "nprobe 64 of the sweep below"},
                "sweep": cpu_sweep, "gpu_imipq_sweep": gpu_sweep, "gpu_vlq_sweep": vlq_sweep, "gpu": gpu_note,
                "train_s": t_train, "add_vec_per_s": nb / t_add}
    print(json.dumps(line))


def _run_reference(a):
    """CPU arm on the SAME configuration as ours: the index has C x E lists and a.n entries (same list density, so a
    query scans as many entries as on the GPU).  Only `enc` vectors are really encoded on the CPU (the reference encodes
    ~10 k vectors/s on 16 cores); the a.n-entry index is that encoded sample tiled a.n / enc times with fresh ids --
    every list is as long as in the full database and the scan touches a.n-entry arrays."""
    from oracle import pyoracle as po
    from vector_line_quantization_b200 import data

    have_ref = po.ref_available()
    ncores = po.num_threads()
    C, E, M, d = a.nlist, a.nedge, a.m, a.d
    t_setup = time.time()
    enc = min(a.n, 500_000)
    reps = max(1, a.n // enc)
    xt = data.sift_like(max(C, 32768), d=d, kc=min(a.kc, 1 << 16), seed=1)
    xb = data.sift_like(enc, d=d, kc=min(a.kc, 1 << 16), seed=2)
    xq = data.sift_like(a.nq, d=d, kc=min(a.kc, 1 << 16), seed=3)
    # codebooks: untimed setup.  CPU k-means at C=2^16 takes ~1 h on 8 cores, so centroids are a random sample of the
    # training rows (search / encode cost does not depend on centroid quality); everything else follows the train path.
    cent = xt[po.rand_perm(xt.shape[0], 1234)[:C]] + np.float32(0.25)
    if have_ref:
        Dg, Ig = po.ref_flat_search(cent, cent, E + 1)  # reference IndexFlatL2 (BLAS), GpuIndexFlat.cu:869-893
        edge, ed2 = Ig[:, 1:].astype(np.int32).copy(), Dg[:, 1:].copy()
        ed2 = np.maximum(ed2, 1e-3).astype(np.float32)
    else:
        edge, ed2 = po.knn_graph(cent, E)
    x2 = xt[:32768]
    A2 = (po.ref_flat_search(cent, x2, 1)[1][:, 0].astype(np.int32) if have_ref else po.l2_topk(x2, cent, 1)[1][:, 0].copy())
    lst2, lam2 = po.line_stage(x2, A2, cent, edge, ed2)
    lcb, _ = po.kmeans(lam2.reshape(-1, 1), a.nlambda, niter=10)
    lcb = lcb.reshape(-1)
    r2 = po.residual(x2, lst2, po.lambda_quantize(lam2, lcb), lcb, cent, edge)
    pq = po.ref_pq_train(r2, M) if have_ref else np.stack(
        [po.kmeans(r2[:, m * (d // M):(m + 1) * (d // M)], 256, niter=10)[0] for m in range(M)])
    # encode the sample (timed: the CPU encode rate)
    t0 = time.time()
    if have_ref:
        A = po.ref_flat_search(cent, xb, 1)[1][:, 0].astype(np.int32)  # IndexFlatL2::search, the CPU twin of a2
    else:
        A = po.l2_topk(xb, cent, 1)[1][:, 0].copy()
    lst, lam = po.line_stage(xb, A, cent, edge, ed2)
    lamq = po.lambda_quantize(lam, lcb)
    r = po.residual(xb, lst, lamq, lcb, cent, edge)
    codes = po.ref_pq_compute_codes(r, pq) if have_ref else po.pq_encode(r, pq)
    t_enc = time.time() - t0
    # the a.n-entry index: the encoded sample `reps` times over (ids i + j * enc)
    lst_all = np.tile(lst, reps)
    off, perm = po.build_lists(lst_all, C * E)
    src = perm % enc
    T2 = po.term2(cent, pq)
    args = (cent, edge, ed2, lcb, pq, off, codes[src], lamq[src], perm.astype(np.int64))
    nb = int(lst_all.shape[0])
    del lst_all
    t_setup = time.time() - t_setup
    # steps: each a bounded sample of the nq-query batch, sized for ~4 s
    probe = min(a.nq, max(2 * ncores, 16))
    t0 = time.time()
    po.search(xq[:probe], *args, P=a.nprobe, W=a.w1, k=a.k, T2=T2)
    per_q = (time.time() - t0) / probe
    ns = int(min(a.nq, max(probe, 4.0 / max(per_q, 1e-9))))
    for _ in range(a.warmup):
        po.search(xq[:ns], *args, P=a.nprobe, W=a.w1, k=a.k, T2=T2)
    times = []
    for _ in range(a.steps):
        t0 = time.time()
        po.search(xq[:ns], *args, P=a.nprobe, W=a.w1, k=a.k, T2=T2)
        times.append(time.time() - t0)
    tot = sum(times)
    qps = ns * a.steps / tot
    sample = ("%d of %d queries per step against a %d-entry index with the configuration's C x E = %d lists (same list "
              "density as the %d-vector database): %d vectors encoded on the CPU, tiled %d x with fresh ids; centroids = "
              "random training rows (no CPU k-means at C = %d); stock pieces by the reference CPU library = %s"
              % (ns, a.nq, nb, C * E, a.n, enc, reps, C, have_ref))
    cfg = workload_config(a, a.gpus)  # the same object as our arm prints
    line = {
        "impl": "reference", "metric": "vlq_search_qps", "value": qps, "unit": "queries/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True,
        "scaling": "strong" if a.gpus > 1 and a.scaling != "weak" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": ncores, "kind": "port", "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "encode": {"value": enc / t_enc / 1e6, "unit": "Mvec/s", "kind": "reference" if have_ref else "port",
                   "sample": "%d vectors: IndexFlatL2 assign + oracle line stage + ProductQuantizer::compute_codes" % enc},
        "setup_s": t_setup, "db_vectors_searched": nb, "db_vectors_encoded_on_cpu": enc,
    }
    return line


def workload_config(a, n_gpus):
    strong = n_gpus > 1 and a.scaling != "weak"
    total = a.n if (strong or n_gpus == 1) else a.n * n_gpus
    per_gpu = a.n // n_gpus if strong else a.n
    if a.shape == "deep":
        cfg = "configs[2] (DEEP1B shape)"
    elif a.u8 and total >= 1_000_000_000:
        cfg = "configs[3] (SIFT1B shape, uint8 ingest)"
    elif total == 10_000_000:
        cfg = "configs[1]"
    else:
        cfg = "configs[1] geometry at another database size"
    return {
        "workload": "BASELINE.json %s: VLQ C=%d centroids x E=%d lines, PQ m=%d, nLambda=%d, d=%d, synthetic "
                    "%s-shaped %d vectors in total (%d per GPU); search nq=%d nprobe=%d w1=%d k=%d"
                    % (cfg, a.nlist, a.nedge, a.m, a.nlambda, a.d, a.shape.upper(), total, per_gpu, a.nq, a.nprobe, a.w1, a.k),
        "db_vectors_per_gpu": per_gpu, "db_vectors_total": total, "nlist": a.nlist, "nedge": a.nedge, "m": a.m,
        "nq": a.nq, "nprobe": a.nprobe, "w1": a.w1, "k": a.k, "train_iters": a.train_iters,
        "parallelism": ("database shards (%s scaling); coarse stage split by queries, line lists exchanged "
                        "through peer-mapped memory, every shard scans all queries, per-shard top-k merged by query slice "
                        "over NVLink" % ("strong" if strong else "weak")) if n_gpus > 1 else "single GPU",
        "l2": "an L2-sized (256 MiB) buffer is overwritten between timed steps",
    }


DUMP_LIMIT_BYTES = 64_000_000  # all files together, .npy headers included
NPY_HEADER_BYTES = 128  # numpy pads a 2-D float array's header to 128 bytes


def dump_outputs(path, D, I):
    """--dump-outputs: the (distances, labels) a GpuIndexIVFPQ::search caller receives, as float32 / float64 .npy files.
    Labels fit float64 exactly (< 2^53).  A result larger than 64 MB (10^6 bytes each) is cut to a fixed, seeded sample of query rows,
    whose indices go to query_rows.npy."""
    D = D.cpu().numpy().astype(np.float32)
    I = I.cpu().numpy().astype(np.float64)
    nq, k = D.shape
    rows = max(1, (DUMP_LIMIT_BYTES - 3 * NPY_HEADER_BYTES) // (k * (4 + 8) + 8))
    os.makedirs(path, exist_ok=True)
    if nq > rows:
        sel = np.sort(np.random.default_rng(0).choice(nq, rows, replace=False))
        D, I = D[sel], I[sel]
        np.save(os.path.join(path, "query_rows.npy"), sel.astype(np.float64))
    np.save(os.path.join(path, "distances.npy"), D)
    np.save(os.path.join(path, "labels.npy"), I)


# ------------------------------------------------------------------------------------------------------- our arm
def run_b200(a):
    import torch
    import torch.distributed as dist

    from vector_line_quantization_b200 import _abi, data, ops, sharding, train

    _abi.lib()  # fail loudly without the CUDA extension
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (--impl b200) needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    C, E, M, d, P, W, k, nq = a.nlist, a.nedge, a.m, a.d, a.nprobe, a.w1, a.k, a.nq
    strong = world > 1 and a.scaling != "weak"
    n_total = a.n if (strong or world == 1) else a.n * world
    id0, id1 = sharding.shard_range(n_total, world, rank)  # this rank's rows of the global database
    n_loc = id1 - id0

    def log(*s):
        if rank == 0:
            print("[bench]", *s, file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- setup (untimed): codebooks trained on the device; identical on all ranks (rank 0 broadcasts)
    t0 = time.time()
    nt = min(C * 64, 4 * n_total)
    gen = data.SyntheticGen(a.shape, d=d, kc=a.kc, device=dev)
    xt = torch.cat([gen.chunk(7000 + i, min(1 << 20, nt - i * (1 << 20))) for i in range((nt + (1 << 20) - 1) >> 20)])
    model = train.train_vlq(xt, C, E, M, a.nlambda, niter=a.train_iters, pq_niter=10, exact_perm=False)
    del xt
    if world > 1:
        for key in ("cent", "cnorm", "edge", "edge_d2", "lambda_cb", "pq"):
            dist.broadcast(model[key], 0)
    torch.cuda.synchronize()
    log("trained codebooks in %.1f s" % (time.time() - t0))
    cent, cn, edge, ed2, lcb, pq = (model[key] for key in ("cent", "cnorm", "edge", "edge_d2", "lambda_cb", "pq"))
    use_tc = bool(_abi.lib().vlq_tc_supported(d, C)) and not a.no_tc
    pack = ops.CentPack(cent, cn) if use_tc else None  # re-packed after the broadcast so every rank holds the same bits

    def assign(x_):
        if use_tc:
            return ops.l2_assign_tc(x_, pack, want_dist=False)[0]
        return ops.l2_assign(x_, cent, cn, want_dist=False)[0]

    # ---- encode this rank's shard (timed as its own stage: encode Mvec/s).  The database is streamed in 1 Mi-vector
    #      chunks from a deterministic generator (a 1B-scale shard does not fit in one fp32 tensor); generation is
    #      outside the timed events.
    chunk = 1 << 20

    def db_chunk(s):  # rows [s, s + chunk) of this rank's shard = rows id0 + s ... of the GLOBAL database, which is
        # generated in 1 Mi-row blocks (the same database for every N: a shard boundary may fall inside a block)
        g0, g1 = id0 + s, min(id1, id0 + s + chunk)
        parts_ = []
        for c in range(g0 // chunk, (g1 - 1) // chunk + 1):
            blk = gen.chunk(1000003 + c, min(chunk, n_total - c * chunk))
            parts_.append(blk[max(g0 - c * chunk, 0):min(g1 - c * chunk, blk.shape[0])])
        return parts_[0] if len(parts_) == 1 else torch.cat(parts_)

    lists = None
    x0_ = db_chunk(0)[:65536]
    enc_passes = 2 if use_tc and bool(torch.equal(x0_.half().float(), x0_)) else (3 if use_tc else 1)
    del x0_
    barrier()
    prof = os.environ.get("VLQ_PROFILE", "")  # ncu --profile-from-start off: wrap one region in cudaProfilerStart/Stop
    if prof == "encode":
        torch.cuda.profiler.start()
    n_before = ops.launch_count()
    evs = []
    parts = []
    for s in range(0, n_loc, chunk):
        x = db_chunk(s)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        A = assign(x)
        parts.append(ops.line_encode(x, A, cent, edge, ed2, lcb, pq))
        e1.record()
        evs.append((e0, e1))
        parts[-1] = ops.Encoded(parts[-1].list, None, parts[-1].lamq, parts[-1].codes, parts[-1].kappa, None)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    new_list = torch.cat([p.list for p in parts])
    ids = torch.arange(id0, id1, dtype=torch.int64, device=dev)
    all_codes, all_lamq, all_kappa = (torch.cat([getattr(p, f) for p in parts]) for f in ("codes", "lamq", "kappa"))
    shard_by = a.shard_by if a.shard_by != "auto" else ("lists" if world > 1 and n_total / (C * E) >= 64 else "ids")
    if world == 1:
        shard_by = "ids"
    route_s = 0.0
    if shard_by == "lists":  # route every encoded entry to the rank that owns its list (one all-to-all per array);
        # timed on its own (host clock, includes the NCCL calls): it is index distribution, not encode arithmetic
        del parts
        e1.record()
        evs.append((e0, e1))
        torch.cuda.synchronize()
        t_r = time.perf_counter()
        new_list, (all_codes, all_lamq, all_kappa, ids) = sharding.route_by_list(new_list, [all_codes, all_lamq, all_kappa, ids], C * E)
        torch.cuda.synchronize()
        route_s = time.perf_counter() - t_r
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    lists = ops.build_lists(C * E, M, new_list, all_codes, all_lamq, all_kappa, ids)
    # average length of the lists this rank scans (kernel choice): a list-range shard holds 1/N of the lists at full length
    len_hint = int(lists.ids.shape[0] // max(1, (C * E) // (world if shard_by == "lists" else 1)))
    e1.record()
    evs.append((e0, e1))
    barrier()
    if prof == "encode":
        torch.cuda.profiler.stop()
    enc_ms = torch.tensor([sum(x0.elapsed_time(x1) for x0, x1 in evs)], device=dev)
    if world > 1:
        dist.all_reduce(enc_ms, op=dist.ReduceOp.MAX)
    enc_ms = float(enc_ms)
    enc_launches = ops.launch_count() - n_before
    parts = None
    del new_list, ids, all_codes, all_lamq, all_kappa
    torch.cuda.empty_cache()
    n_listed0 = int(lists.ids.shape[0])
    log("encoded %d vectors/GPU in %.1f ms (shards by %s, %d entries on this rank)" % (n_loc, enc_ms, shard_by, n_listed0))
    n_loc_sum = n_total  # vectors encoded by all ranks together

    # ---- queries + exact ground truth (brute force over every shard, for recall)
    xq = gen.chunk(3, nq)
    gt_d = torch.full((nq,), float("inf"), device=dev)
    gt_i = torch.full((nq,), -1, dtype=torch.int64, device=dev)
    gchunk = 1 << 18
    exact_gt = n_total <= 20_000_000  # beyond that the brute force runs on the tensor-core kernel (fp32-grade, see DESIGN.md)
    for s0 in range(0, n_loc, chunk):
        xc = db_chunk(s0)
        for s in range(0, xc.shape[0], gchunk):  # "centroids" = a database slice; argmin per query = exact 1-NN in the slice
            sl = xc[s:s + gchunk]
            if exact_gt or not use_tc:
                i_, d_ = ops.l2_assign(xq, sl, add_xnorm=True)
            else:
                i_, d_ = ops.l2_assign_tc(xq, ops.CentPack(sl), add_xnorm=True)
            better = d_ < gt_d
            gt_d = torch.where(better, d_, gt_d)
            gt_i = torch.where(better, i_.to(torch.int64) + (id0 + s0 + s), gt_i)
        del xc
    if world > 1:
        all_d = [torch.empty_like(gt_d) for _ in range(world)]
        all_i = [torch.empty_like(gt_i) for _ in range(world)]
        dist.all_gather(all_d, gt_d)
        dist.all_gather(all_i, gt_i)
        sd, si = torch.stack(all_d), torch.stack(all_i)
        best = sd.argmin(dim=0, keepdim=True)
        gt_i = si.gather(0, best)[0]

    # ---- the step
    #  N = 1: the product's C++ API, GpuIndexIVFPQ::search with DEVICE pointers (built further down: `hidx`)
    #  N > 1: query-split coarse stage -> line exchange through peer-mapped memory -> every shard scans all queries ->
    #         peer merge by query slice (sharding.QuerySplitSearch); NCCL all-gather + merge kernel when symmetric
    #         memory is unavailable
    gD = torch.empty((world, nq, k), dtype=torch.float32, device=dev) if world > 1 else None
    gI = torch.empty((world, nq, k), dtype=torch.int64, device=dev) if world > 1 else None

    def ops_search(q):  # the whole query path on this rank's lists through the C-ABI (ops = ctypes bindings)
        return ops.search(q, cent, cn, edge, ed2, lcb, pq, lists, P, W, k, pack=pack, list_len_hint=len_hint)

    def step_nccl(q):
        D, I = ops_search(q)
        if world > 1:
            sharding.gather_topk(D, I, gD, gI)
            D, I = ops.merge_topk(gD, gI)
        return D, I

    exchange = "none"
    qss = None
    if world > 1:
        exchange = "replicated coarse stage, nccl all-gather of the per-shard top-k + merge kernel"
        if os.environ.get("VLQ_EXCHANGE", "peer") == "peer":
            try:
                qss = sharding.QuerySplitSearch(nq, k, W, dev)
                exchange = ("coarse stage split by queries; (list, term1, term6) pulled from the peers' symmetric memory "
                            "over NVLink; per-shard top-k merged by query slice straight from peer memory (two device barriers)")
            except Exception as exc:  # symmetric memory unavailable on this box: the NCCL path is the same result
                log("peer-memory exchange unavailable (%s: %s); using NCCL" % (type(exc).__name__, exc))
                qss = None

    def coarse_fn(qs, out):
        return ops.coarse_lines(qs, cent, cn, edge, ed2, P, W, pack=pack, out=out)

    def scan_fn(q, lines, out):
        return ops.scan_lines(q, pq, lcb, lines, ed2, lists, k, out=out, list_len_hint=len_hint)

    def step_peer(q):  # -> (D, I) of this rank's query slice
        return qss.search(q, coarse_fn, scan_fn)

    if qss is not None:  # the query-split exchange must return the same bits as the NCCL exchange
        Dn, In = step_nccl(xq)
        Dp, Ip = step_peer(xq)
        torch.cuda.synchronize()
        qs0, qs1 = qss.my_slice()
        assert torch.equal(Dn[qs0:qs1], Dp) and torch.equal(In[qs0:qs1], Ip), "query-split exchange differs from the NCCL exchange"
        log("query-split peer exchange == NCCL exchange (bitwise)")

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        evs = []
        n0 = ops.launch_count()
        for _ in range(steps):
            flush.fill_(1)  # L2 flush, outside the timed events
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        barrier()
        launches = ops.launch_count() - n0
        ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in evs)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), launches

    # ---- e2e: the reference-facing API (C++ host layer: GpuIndexIVFPQ::add_with_ids / ::search) with HOST buffers;
    #      the host->device copy of the inputs and the device->host copy of the results are inside the timed region
    from vector_line_quantization_b200 import index as vi

    res = vi.StandardGpuResources(local)
    hidx = vi.GpuIndexIVFPQ(res, d, C, M, 8, E, a.nlambda, use_tensor_cores=use_tc)
    hidx.setCodebooks(*(model[key].cpu().numpy() for key in ("cent", "edge", "edge_d2", "lambda_cb", "pq")))
    hidx.setNumProbes(P)
    hidx.w1_ = W
    hidx.reserveMemory(n_loc)  # GpuIndexIVFPQ::reserveMemory, as the reference drivers do before a bulk load
    add_chunk = 2 * chunk  # the reference drivers ingest 2 M vectors per add (gpu/test/sift1b_createdb.cpp:276-289)
    use_u8 = a.u8 and a.shape == "sift"
    hx = torch.empty((min(add_chunk, n_loc), d), dtype=torch.uint8 if use_u8 else torch.float32).pin_memory()
    hids = torch.empty(min(add_chunk, n_loc), dtype=torch.int64).pin_memory()
    enc_e2e_s = 0.0
    xq8 = xq[:8].cpu().numpy()
    hidx.search(xq8, k)  # untimed: a search of the still empty index allocates the query-path scratch (a 1 GB distance tile)
    for s in range(0, n_loc, add_chunk):
        m_ = min(add_chunk, n_loc - s)
        for s2 in range(s, s + m_, chunk):  # staging the synthetic rows on the host is not part of the timed region
            xc = db_chunk(s2)
            hx[s2 - s:s2 - s + xc.shape[0]].copy_(xc.to(torch.uint8) if use_u8 else xc)
        hids[:m_].copy_(torch.arange(id0 + s, id0 + s + m_, dtype=torch.int64))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if use_u8:
            hidx.add_with_ids_u8(hx[:m_], hids[:m_])
        else:
            hidx.add_with_ids(hx[:m_], hids[:m_])
        enc_e2e_s += time.perf_counter() - t0
        log("e2e add of %d vectors: %.1f ms" % (m_, (time.perf_counter() - t0) * 1e3))
    t0 = time.perf_counter()
    hidx.search(xq8, k)  # first search commits the pending entries into the CSR lists
    torch.cuda.synchronize()
    enc_e2e_s += time.perf_counter() - t0
    log("e2e list commit + first search: %.1f ms" % ((time.perf_counter() - t0) * 1e3))
    enc_e2e = torch.tensor([enc_e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(enc_e2e, op=dist.ReduceOp.MAX)
    enc_e2e_s = float(enc_e2e)
    del hx
    torch.cuda.empty_cache()

    # ---- `value`: device-resident step
    dD = torch.empty((nq, k), dtype=torch.float32, device=dev)
    dI = torch.empty((nq, k), dtype=torch.int64, device=dev)
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.5)  # let nvidia-smi come up: the timed region is only tens of milliseconds long
    result = {}

    def dev_step():
        if world == 1:
            hidx.search(xq, k, out=(dD, dI))  # GpuIndexIVFPQ::search, device pointers in and out
            result["DI"] = (dD, dI)
        elif qss is not None:
            result["DI"] = step_peer(xq)
        else:
            result["DI"] = step_nccl(xq)

    if prof == "search":
        torch.cuda.profiler.start()
    total_ms, launches = timed(dev_step, a.steps, a.warmup)
    if prof == "search":
        torch.cuda.profiler.stop()
    D, I = result["DI"]
    if world > 1 and qss is not None:  # assemble the distributed result (outside the timed region) for recall / parity
        qsl = [qss.q0[r + 1] - qss.q0[r] for r in range(world)]
        if len(set(qsl)) == 1:
            fullD = torch.empty((nq, k), dtype=torch.float32, device=dev)
            fullI = torch.empty((nq, k), dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(fullD, D.contiguous())
            dist.all_gather_into_tensor(fullI, I.contiguous())
            D, I = fullD, fullI
        else:
            D, I = step_nccl(xq)
    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, D, I)
    ops_matches = None
    if world == 1:  # the C++ API and the C-ABI tile loop of ops.search must agree bit for bit
        Do_, Io_ = ops_search(xq)
        ops_matches = bool(torch.equal(Do_, D) and torch.equal(Io_, I))

    hq = torch.empty((nq, d), dtype=torch.float32).pin_memory()
    hq.copy_(xq.cpu())
    hD = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    hI = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    dq = torch.empty_like(xq)
    qs0, qs1 = (qss.my_slice() if qss is not None else (0, nq))

    def e2e_step():
        if world == 1:
            hidx.search(hq, k, out=(hD, hI))  # host pointers straight through the C++ API
        else:  # every rank uploads the query batch (the scan needs all of it) and downloads its slice of the result
            dq.copy_(hq, non_blocking=True)
            if qss is not None:
                D_, I_ = step_peer(dq)
                hD[qs0:qs1].copy_(D_, non_blocking=True)
                hI[qs0:qs1].copy_(I_, non_blocking=True)
            else:
                D_, I_ = step_nccl(dq)
                hD.copy_(D_, non_blocking=True)
                hI.copy_(I_, non_blocking=True)
            torch.cuda.synchronize()

    for _ in range(a.warmup):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_step()
    barrier()
    e2e_t = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_t) * 1e3
    host_matches_ops = bool((hI[qs0:qs1].to(dev) == I[qs0:qs1]).all()) and bool((hD[qs0:qs1].to(dev) == D[qs0:qs1]).all())
    if ops_matches is not None:
        host_matches_ops = host_matches_ops and ops_matches
    clk = clocks.stop()  # sampled across the device-timed steps and the e2e steps

    # ---- per-stage device times of one step (CUDA events on the launching stream) -> roofline of the dominant kernel
    def stage_times():
        names = ["l2_distances", "l2_bucket_min", "select_rows", "select_lines", "coarse_select_lines", "scan_topk"]
        acc = dict.fromkeys(names, 0.0)
        cnt = dict.fromkeys(names, 0)
        tile = 4096
        Dbuf = None if coarse_exact else torch.empty((tile, C), dtype=torch.float32, device=dev)
        bbuf = torch.empty((tile, ops.num_buckets(C)), dtype=torch.float32, device=dev)
        ed2f = ed2.reshape(-1)

        def t(name, fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn()
            e1.record()
            pending.append((name, e0, e1))
            return r

        pending = []
        for s in range(0, nq, tile):
            qt = xq[s:s + tile]
            if coarse_exact:  # no distance matrix: bucket minima from the tcgen05 sweep + exact re-evaluation
                bm = bbuf[: qt.shape[0]]
                t("l2_bucket_min", lambda: ops.l2_bucket_min_tc(qt, pack, bm))
                lst, t1, t6 = t("coarse_select_lines",
                                lambda: ops.coarse_select_lines_exact(qt, cent, cn, bm, P, edge, ed2, W))
            elif use_tc:
                bm = bbuf[: qt.shape[0]]
                Dm = t("l2_distances", lambda: ops.l2_distances_tc(qt, pack, out=Dbuf[: qt.shape[0]], bucket_min=bm))
                lst, t1, t6 = t("coarse_select_lines", lambda: ops.coarse_select_lines(Dm, bm, C, P, edge, ed2, W))
            else:
                Dm = t("l2_distances", lambda: ops.l2_distances(qt, cent, cn, out=Dbuf[: qt.shape[0]]))
                _, cid = t("select_rows", lambda: ops.select_rows(Dm, P))
                lst, t1, t6 = t("select_lines", lambda: ops.select_lines(Dm, cid, edge, ed2, W))
            t("scan_topk", lambda: ops.scan_topk(qt, pq, lcb, lst, t1, t6, ed2f, lists, k))
        torch.cuda.synchronize()
        for name, e0, e1 in pending:
            acc[name] += e0.elapsed_time(e1)
            cnt[name] += 1
        return acc, cnt

    coarse_exact = bool(use_tc and ops.CoarseStage(cent, cn, edge, ed2, P, W, 1, pack).exact)
    stage_times()
    st_ms, st_cnt = stage_times()

    # scanned entries per query (algorithmic bytes of the scan: SURVEY 8d)
    lens = (lists.offsets[1:] - lists.offsets[:-1]).clamp_max(1024)
    Dm = ops.l2_distances(xq[:1024].contiguous(), cent, cn)
    _, cid = ops.select_rows(Dm, P)
    lst, _, _ = ops.select_lines(Dm, cid, edge, ed2, W)
    scanned_per_q = float(lens[lst.clamp_min(0).to(torch.int64)].mul(lst >= 0).sum(dim=1).float().mean())

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tc_peak = peaks.get("bf16_tflops", 1590.0)
    peak_src = "measured (MEASURED_PEAKS.json, burst: kernel timed alone)" if peaks else "fallback (B200_PROFILING.md)"
    # DRAM traffic per launch comes from an `ncu --set full` capture of the same command (profiles/, tools/ncu_traffic.py);
    # it is not measurable inside this run, so the line carries null and the committed summaries carry the numbers
    traffic = {}

    def stage_roofline(name):
        """algorithmic work of one launch of the stage (DESIGN.md section 4) over its measured launch time"""
        if not st_cnt.get(name):
            return None
        ms = st_ms[name] / st_cnt[name]
        rows = nq / st_cnt[name]
        if name == "scan_topk":  # SURVEY 8d: codes + lambda of every scanned entry, ids of the k winners
            r = {"bound": "hbm", "achieved": rows * (scanned_per_q * (M + 1) + k * 8) / (ms * 1e-3) / 1e9,
                 "peak": hbm_peak, "unit": "GB/s"}
        elif name == "coarse_select_lines" and coarse_exact:
            # HBM side: bucket minima + the query + W outputs; the (32 P + P E) centroid rows it re-evaluates come from
            # the L2-resident centroid table (C d 4 bytes), reported as l2_GBs
            nbk = ops.num_buckets(C)
            r = {"bound": "hbm", "achieved": rows * (nbk * 4 + d * 4 + W * 12) / (ms * 1e-3) / 1e9,
                 "peak": hbm_peak, "unit": "GB/s", "l2_GBs": rows * (32 * P + P * E) * d * 4.0 / (ms * 1e-3) / 1e9}
        elif name == "coarse_select_lines":  # bucket minima + P 128-byte lines of D + P*E gathers + W outputs
            nbk = ops.num_buckets(C)
            r = {"bound": "hbm", "achieved": rows * (nbk * 4 + P * 128 + P * E * 4 + W * 12) / (ms * 1e-3) / 1e9,
                 "peak": hbm_peak, "unit": "GB/s"}
        elif name == "l2_bucket_min":  # tensor bound: 2 C d flop per query (x 2-3 fp16 passes executed)
            r = {"bound": "tensor", "achieved": rows * 2.0 * C * d / (ms * 1e-3) / 1e12, "peak": tc_peak, "unit": "TFLOP/s",
                 "executed_passes": "2 (integer-valued queries: x_lo = 0) or 3"}
        elif name in ("select_rows", "select_lines"):  # the whole row of D is read
            r = {"bound": "hbm", "achieved": rows * C * 4.0 / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s"}
        else:  # coarse distance tile: the GEMM is cheap next to writing 4*C bytes of distances (+ bucket minima) per query
            r = {"bound": "hbm", "achieved": rows * (C * 4.0 + (ops.num_buckets(C) * 4 if use_tc else 0)) / (ms * 1e-3) / 1e9,
                 "peak": hbm_peak, "unit": "GB/s", "tensor_tflops": rows * 2.0 * C * d / (ms * 1e-3) / 1e12}
        r.update(frac=r["achieved"] / r["peak"], traffic=traffic.get(name), kernel=name, ms_per_launch=ms)
        return r

    dominant = max(st_ms, key=st_ms.get)
    roof = stage_roofline(dominant)
    roof.update(peak_source=peak_src, stage_ms_per_step=st_ms,
                stages=[r for r in (stage_roofline(n_) for n_ in st_ms if n_ != dominant) if r])

    # ---- recall (R@r of the true 1-NN, gpu/test/sift1b_query.cpp:334-347)
    In = I.cpu().numpy()
    gt = gt_i.cpu().numpy()
    recall = {"R@1": data.recall_at(In, gt, 1), "R@10": data.recall_at(In, gt, 10), "R@100": data.recall_at(In, gt, min(100, k))}

    # ---- recall / QPS over nprobe (BASELINE.json configs[2]: "recall@1/10/100 sweep over nprobe")
    sweep = None
    if a.sweep and world == 1:
        sweep = []
        for P_ in (1, 2, 4, 8, 16, 32, 64):
            W_ = min(1024, 4 * P_)

            def sw_step():
                result["sw"] = ops.search(xq, cent, cn, edge, ed2, lcb, pq, lists, P_, W_, k, pack=pack)

            ms_, _ = timed(sw_step, 3, 1)
            Is = result["sw"][1].cpu().numpy()
            sweep.append({"nprobe": P_, "w1": W_, "R@1": data.recall_at(Is, gt, 1), "R@10": data.recall_at(Is, gt, 10),
                          "R@100": data.recall_at(Is, gt, min(100, k)), "qps": nq * 3 / (ms_ * 1e-3)})
            log("sweep", sweep[-1])

    # ---- CPU baseline on rank 0 (N=1 only): oracle port against the same index + parity on the sample
    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        from oracle import pyoracle as po  # checker / baseline only

        mh = {key: model[key].cpu().numpy() for key in ("cent", "edge", "edge_d2", "lambda_cb", "pq")}
        lh = (lists.offsets.cpu().numpy(), ops.rotate_codes(lists.offsets, lists.codes, inverse=True).cpu().numpy(),
              lists.lamq.cpu().numpy(), lists.ids.cpu().numpy())  # canonical code order for the oracle
        cpu_baseline, parity = cpu_search_baseline(po, mh, lh, xq.cpu().numpy(), P, W, k, a.cpu_seconds,
                                                   (D.cpu().numpy(), In), gt=gt, recall_at=data.recall_at)
    # ---- N > 1: the merged result against the oracle's search of the UNION of the shards (sub-sample of the queries)
    if world > 1 and n_total <= 20_000_000 and not a.no_cpu_baseline:
        canon = ops.rotate_codes(lists.offsets, lists.codes, inverse=True)
        lens_r = (lists.offsets[1:] - lists.offsets[:-1]).to(torch.int32)
        szs = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(szs, torch.tensor([int(lists.ids.shape[0])], dtype=torch.int64, device=dev))
        szs = [int(x) for x in szs]
        mx = max(szs)

        def gather_rows(t):  # ragged all-gather of per-entry arrays (padded to the largest shard)
            pad = torch.zeros((mx,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            pad[: t.shape[0]] = t
            outs = [torch.empty_like(pad) for _ in range(world)]
            dist.all_gather(outs, pad)
            return [o[:n_].cpu().numpy() for o, n_ in zip(outs, szs)]

        all_lens = [torch.empty_like(lens_r) for _ in range(world)]
        dist.all_gather(all_lens, lens_r)
        g_codes, g_lamq, g_ids = gather_rows(canon), gather_rows(lists.lamq), gather_rows(lists.ids)
        if rank == 0:
            from oracle import pyoracle as po  # checker only

            lens_np = [x.cpu().numpy().astype(np.int64) for x in all_lens]
            tot_len = sum(lens_np)
            off_u = np.zeros(C * E + 1, dtype=np.int64)
            off_u[1:] = np.cumsum(tot_len)
            nU = int(off_u[-1])
            codes_u = np.empty((nU, M), dtype=np.uint8)
            lamq_u = np.empty(nU, dtype=np.uint8)
            ids_u = np.empty(nU, dtype=np.int64)
            cur = off_u[:-1].copy()
            for r in range(world):  # list-major union, shard order inside a list (= ascending ids: what one index holds)
                offr = np.zeros(C * E + 1, dtype=np.int64)
                offr[1:] = np.cumsum(lens_np[r])
                dst = np.repeat(cur - offr[:-1], lens_np[r]) + np.arange(szs[r])
                codes_u[dst], lamq_u[dst], ids_u[dst] = g_codes[r], g_lamq[r], g_ids[r]
                cur += lens_np[r]
            mh = {key: model[key].cpu().numpy() for key in ("cent", "edge", "edge_d2", "lambda_cb", "pq")}
            ns = min(nq, 512)
            T2 = po.term2(mh["cent"], mh["pq"])
            Do, Io = po.search(xq[:ns].cpu().numpy(), mh["cent"], mh["edge"], mh["edge_d2"], mh["lambda_cb"], mh["pq"], off_u,
                               codes_u, lamq_u, ids_u, P=P, W=W, k=k, T2=T2)
            gD_, gI_ = D[:ns].cpu().numpy(), In[:ns]
            qn = (xq[:ns].cpu().numpy().astype(np.float64) ** 2).sum(1, keepdims=True)
            same = (Io >= 0) & (gI_ == Io)
            rel = np.abs(gD_ - Do)[same] / (np.abs(Do) + qn)[same]
            parity = {"queries": ns, "against": "oracle search of the union of the %d shards (%d entries)" % (world, nU),
                      "id_match": float((gI_ == Io)[Io >= 0].mean()), "max_rel_dist_err": float(rel.max()),
                      "set_overlap": float(np.mean([len(set(x) & set(y)) / max(1, len(set(y))) for x, y in zip(gI_, Io)]))}
        del g_codes, g_lamq, g_ids, canon

    # ---- the scan stage at BASELINE configs[3] list density (1 B entries, 477 per list) on SYNTHETIC lists (random codes /
    #      lambda bytes / kappa: no 36 s encode), N = 1 only: the >= 0.70-of-HBM target of north_star applies to this density
    c4_stage = None
    if world == 1 and not a.no_c4_stage and not a.quick and M in (8, 16):
        try:
            lists = None
            hidx.reset()
            torch.cuda.empty_cache()
            free_b, _ = torch.cuda.mem_get_info()
            n_c4 = 1_000_000_000
            if free_b > n_c4 * (M + 13) * 1.3:
                c4_stage = scan_stage_at_density(ops, dev, n_c4, C * E, M, d, nq, W, k, hbm_peak, peak_src)
                log("C4-density scan stage", c4_stage)
        except Exception as exc:  # the headline line must survive this extra measurement
            log("C4-density scan stage failed: %s: %s" % (type(exc).__name__, exc))
    if c4_stage is not None:
        roof["stages"].append(c4_stage)

    if rank == 0:
        qps = nq * a.steps / (total_ms * 1e-3)
        e2e_qps = nq * a.steps / (e2e_ms * 1e-3)
        line = {
            "metric": "vlq_search_qps", "value": qps, "unit": "queries/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": total_ms / a.steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32 (coarse GEMM: split-fp16 x3 tcgen05, fp32 accumulate)" if use_tc else "f32", "data": "synthetic",
            "config": workload_config(a, world),
            "plumbing": {"exchange": exchange, "shard_by": shard_by, "entries_on_rank0": int(n_listed0),
                         "value_api": "GpuIndexIVFPQ::search (C++ host layer), device pointers" if world == 1 else
                         "sharding.QuerySplitSearch over the C-ABI stage entry points"},
            "e2e": {"value": e2e_qps, "unit": "queries/s",
                    "h2d_bytes_per_step": nq * d * 4 * world, "d2h_bytes_per_step": nq * k * 12},
            "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu_baseline, "clocks": clk, "recall": recall,
            "encode": {"value": n_loc_sum / (enc_ms * 1e-3) / 1e6, "unit": "Mvec/s", "ms": enc_ms,
                       "e2e": {"value": n_loc_sum / enc_e2e_s / 1e6, "unit": "Mvec/s",
                               "h2d_bytes_per_vector": (d if use_u8 else d * 4) + 8,
                               "note": "GpuIndexIVFPQ::add_with_ids%s from pinned host memory in 2 Mi-vector chunks + "
                                       "list commit" % ("_u8" if use_u8 else "")},
                       "gpu_launches": enc_launches, "route_to_list_owner_s": route_s,
                       "tensor_frac": (n_loc * 2.0 * C * d / (enc_ms * 1e-3) / 1e12) / peaks.get("bf16_tflops_sustained", 1400.0),
                       # the split-fp16 scheme EXECUTES 2 passes (fp16-exact vectors: x_lo = 0) or 3: that is the work the
                       # tensor pipe does for one fp32-grade product (the arg-min GEMM is ~2/3 of the encode time)
                       "tensor_passes_executed": enc_passes,
                       "tensor_executed_tflops": enc_passes * n_loc * 2.0 * C * d / (enc_ms * 1e-3) / 1e12},
            "scanned_entries_per_query": scanned_per_q, "parity_vs_oracle": parity,
            "host_api_matches_ops_bitwise": host_matches_ops,
        }
        if world > 1:
            line["shard_queries_per_s"] = qps * world  # (query, shard) searches per second, all ranks
        if sweep is not None:
            line["recall_sweep"] = sweep
    else:
        line = None
    if world > 1:
        dist.destroy_process_group()
    return line


def scan_stage_at_density(ops, dev, n_target, nlists, M, d, nq, W, k, hbm_peak, peak_src):
    """vlq_scan_topk alone on synthetic lists of the given density (see tools/bench_scan.py): list lengths are Poisson
    around n_target / nlists with a Gamma(4) spread, queries pick lists size-biased (dense regions attract both vectors
    and queries in the real index).  Returns a roofline stage object (SURVEY 8d algorithmic bytes / CUDA-event time)."""
    import torch

    g = torch.Generator(device=dev).manual_seed(1)
    mean = n_target / nlists
    spread = torch.distributions.Gamma(4.0, 4.0).sample((nlists,)).to(dev)
    lens = torch.poisson(spread * mean, generator=g).to(torch.int64)
    off = torch.zeros(nlists + 1, dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(lens, 0)
    n = int(off[-1])
    codes = torch.empty((n, M), dtype=torch.uint8, device=dev)
    lamq = torch.empty(n, dtype=torch.uint8, device=dev)
    kappa = torch.empty(n, dtype=torch.float32, device=dev)
    step = 1 << 26
    for s in range(0, n, step):
        e = min(n, s + step)
        codes[s:e] = torch.randint(0, 256, (e - s, M), dtype=torch.uint8, device=dev, generator=g)
        lamq[s:e] = torch.randint(0, 256, (e - s,), dtype=torch.uint8, device=dev, generator=g)
        kappa[s:e] = torch.randn(e - s, device=dev, generator=g) * 100.0
    lists = ops.Lists(off, codes, lamq, kappa, torch.arange(n, dtype=torch.int64, device=dev))
    g2 = torch.Generator(device=dev).manual_seed(7)
    line = torch.multinomial(lens.float() + 1e-3, nq * W, replacement=True, generator=g2).reshape(nq, W).to(torch.int32)
    q = torch.randn(nq, d, device=dev, generator=g2)
    pq = torch.randn(M, 256, d // M, device=dev, generator=g2)
    lcb = torch.rand(256, device=dev, generator=g2)
    t1 = torch.rand(nq, W, device=dev, generator=g2) * 10
    t6 = torch.randn(nq, W, device=dev, generator=g2)
    ed2 = torch.rand(nlists, device=dev, generator=g2) * 4 + 0.5
    scanned = float(lens.clamp_max(1024)[line.to(torch.int64)].sum(dim=1).float().mean())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    outD = torch.empty((nq, k), dtype=torch.float32, device=dev)
    outI = torch.empty((nq, k), dtype=torch.int64, device=dev)
    tile = 4096

    def run():
        evs = []
        for s in range(0, nq, tile):
            e = min(nq, s + tile)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.scan_topk(q[s:e], pq, lcb, line[s:e], t1[s:e], t6[s:e], ed2, lists, k, 1024, list_len_hint=int(mean),
                          out=(outD[s:e], outI[s:e]))
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(x.elapsed_time(y) for x, y in evs), len(evs)

    for _ in range(3):
        run()
    ms = []
    for _ in range(5):
        flush.fill_(1)
        t, nl = run()
        ms.append(t)
    mean_ms = sum(ms) / len(ms)
    alg = nq * (scanned * (M + 1) + 8 * k)
    ach = alg / (mean_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": None,
            "kernel": "scan_topk @ BASELINE configs[3] list density", "ms_per_launch": mean_ms / nl,
            "ms_per_%d_queries" % nq: mean_ms, "peak_source": peak_src,
            "workload": "synthetic lists: %d entries in %d lists (%.0f per list), %d queries x %d lines, %.0f entries scanned "
                        "per query, k=%d; random codes / lambda bytes / kappa" % (n, nlists, n / nlists, nq, W, scanned, k)}


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "imipq":
        if int(os.environ.get("RANK", "0")) == 0:
            run_imipq(a)
    else:
        # libraries (NCCL's version banner, ...) print to fd 1: keep it clean for the ONE JSON line
        with _StdoutToStderr():
            line = run_b200(a)
        if line is not None:
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
