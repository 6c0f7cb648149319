"""Generates the committed golden fixtures.  Run in the build container (needs oracle/_ref/libfaiss_ref.so, i.e. the
reference sources under /root/reference, for the `ref_*` arrays):

    python tests/golden/make_golden.py

Fixtures
  vlq_small.npz   inputs + codebooks + every intermediate of the VLQ path for a tiny configuration.
                  `ref_*` arrays come from the UNMODIFIED reference CPU library (IndexFlatL2, ProductQuantizer,
                  IndexIVFPQ); all other outputs come from the oracle restatement (oracle/vlq_oracle.c) -- the
                  reference has no CPU VLQ and no golden vectors of its own (SURVEY.md 8c).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import pyoracle as po  # noqa: E402
from vector_line_quantization_b200 import data  # noqa: E402


def main():
    if not po.ref_available():
        # the tests compare against the ref_* arrays; a fixture without them would drop the stored reference output
        sys.exit("make_golden.py: oracle/_ref/libfaiss_ref.so is missing (make -C oracle ref); the fixture is kept as is")
    d, C, E, M, nL = 32, 64, 8, 4, 16
    P, W, k = 8, 32, 10
    xt = data.sift_like(6000, d=d, kc=128, seed=101)
    xb = data.sift_like(3000, d=d, kc=128, seed=102)
    xq = data.sift_like(24, d=d, kc=128, seed=103)
    m = po.train_all(xt, nlist=C, E=E, M=M, nL=nL, niter=8, pq_niter=10)
    enc = po.encode_all(xb, m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"])
    offsets, perm = po.build_lists(enc["list"], C * E)
    codes_l, lamq_l, ids_l = enc["codes"][perm], enc["lamq"][perm], perm.astype(np.int64)
    D, I, coarse, lines, nscan = po.search(xq, m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], offsets,
                                           codes_l, lamq_l, ids_l, P=P, W=W, k=k, cap=1024, want_debug=True)
    Dc, Ic, _, _, nscan_c = po.search(xq, m["cent"], m["edge"], m["edge_d2"], m["lambda_cb"], m["pq"], offsets,
                                      codes_l, lamq_l, ids_l, P=P, W=W, k=k, cap=3, want_debug=True)
    out = dict(
        d=d, C=C, E=E, M=M, nL=nL, P=P, W=W, k=k,
        xb=xb.astype(np.uint8), xq=xq.astype(np.uint8),
        cent=m["cent"], edge=m["edge"], edge_d2=m["edge_d2"], lambda_cb=m["lambda_cb"], pq=m["pq"],
        A=enc["A"], list=enc["list"], lam=enc["lam"], lamq=enc["lamq"], codes=enc["codes"],
        offsets=offsets, perm=perm,
        search_D=D, search_I=I, search_coarse=coarse, search_lines=lines, search_nscan=nscan,
        search_cap3_D=Dc, search_cap3_I=Ic, search_cap3_nscan=nscan_c,
    )
    Dr, Ir = po.ref_flat_search(m["cent"], xb, 1)
    out["ref_flat_assign_D"] = Dr[:, 0]
    out["ref_flat_assign_I"] = Ir[:, 0].astype(np.int32)
    Dg, Ig = po.ref_flat_search(m["cent"], m["cent"], E + 1)
    out["ref_graph_D"] = Dg
    out["ref_graph_I"] = Ig.astype(np.int32)
    out["ref_pq_codes"] = po.ref_pq_compute_codes(enc["residual"], m["pq"])
    # lambda == 0 slice against the reference IndexIVFPQ with the same codebooks
    ivf = po.RefIVFPQ(d, C, M, coarse=m["cent"], pq=m["pq"])
    ivf.add(xb)
    Dv, Iv = ivf.search(xq, k, P)
    out["ref_ivfpq_D"] = Dv
    out["ref_ivfpq_I"] = Iv
    path = os.path.join(HERE, "vlq_small.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
