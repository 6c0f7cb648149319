"""Oracle restatement vs the committed golden fixtures (tests/golden/vlq_small.npz).  CPU only.

`ref_*` arrays in the fixture were produced by the UNMODIFIED reference CPU library; the others by the oracle at
fixture-generation time (they guard the oracle against accidental edits and define what the CUDA path must match).
"""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vlq_small.npz")


@pytest.fixture(scope="module")
def g():
    return dict(np.load(GOLD))


def test_assignment_vs_reference_flat(oracle, g):
    xb = g["xb"].astype(np.float32)
    D, I = oracle.l2_topk(xb, g["cent"], 1, add_xnorm=True)
    assert np.array_equal(I[:, 0], g["A"])
    mism = I[:, 0] != g["ref_flat_assign_I"]
    assert mism.sum() <= 2  # near-ties only
    np.testing.assert_allclose(D[~mism, 0], g["ref_flat_assign_D"][~mism], rtol=1e-4)


def test_graph_vs_reference_flat(oracle, g):
    edge, ed2 = oracle.knn_graph(g["cent"], int(g["E"]))
    assert np.array_equal(edge, g["edge"])
    np.testing.assert_array_equal(ed2, g["edge_d2"])
    # the reference's own C-vs-C search (IndexFlatL2) gives the same neighbours
    assert (edge == g["ref_graph_I"][:, 1:]).mean() > 0.995
    np.testing.assert_allclose(ed2, g["ref_graph_D"][:, 1:], rtol=1e-3, atol=1e-2)


def test_encode_pipeline(oracle, g):
    xb = g["xb"].astype(np.float32)
    enc = oracle.encode_all(xb, g["cent"], g["edge"], g["edge_d2"], g["lambda_cb"], g["pq"])
    for key in ("A", "list", "lamq", "codes"):
        assert np.array_equal(enc[key], g[key]), key
    np.testing.assert_array_equal(enc["lam"], g["lam"])
    # ProductQuantizer::compute_codes of the reference on the same residuals
    assert (enc["codes"] == g["ref_pq_codes"]).mean() > 0.999
    offsets, perm = oracle.build_lists(enc["list"], int(g["C"]) * int(g["E"]))
    assert np.array_equal(offsets, g["offsets"]) and np.array_equal(perm, g["perm"])


def test_search(oracle, g):
    perm = g["perm"]
    args = (g["xq"].astype(np.float32), g["cent"], g["edge"], g["edge_d2"], g["lambda_cb"], g["pq"], g["offsets"],
            g["codes"][perm], g["lamq"][perm], perm.astype(np.int64))
    D, I, coarse, lines, nscan = oracle.search(*args, P=int(g["P"]), W=int(g["W"]), k=int(g["k"]), cap=1024,
                                               want_debug=True)
    assert np.array_equal(I, g["search_I"]) and np.array_equal(coarse, g["search_coarse"])
    assert np.array_equal(lines, g["search_lines"]) and np.array_equal(nscan, g["search_nscan"])
    np.testing.assert_array_equal(D, g["search_D"])
    # list cap (IVFUtils.cu:87): scanning only the first 3 entries of every list
    Dc, Ic, _, _, nsc = oracle.search(*args, P=int(g["P"]), W=int(g["W"]), k=int(g["k"]), cap=3, want_debug=True)
    assert np.array_equal(Ic, g["search_cap3_I"]) and np.array_equal(nsc, g["search_cap3_nscan"])
    assert (nsc <= 3 * int(g["W"])).all()


def test_lambda0_search_vs_reference_ivfpq(oracle, g):
    """With a single lambda level == 0 the VLQ anchor is the centroid, so searching all lines of the P probed centroids
    is IndexIVFPQ with nprobe = P: the reference's IndexIVFPQ results with the fixture's codebooks are stored."""
    C, E, P, k = int(g["C"]), int(g["E"]), int(g["P"]), int(g["k"])
    xb, xq = g["xb"].astype(np.float32), g["xq"].astype(np.float32)
    lcb = np.zeros(1, np.float32)
    enc = oracle.encode_all(xb, g["cent"], g["edge"], g["edge_d2"], lcb, g["pq"])
    offsets, perm = oracle.build_lists(enc["list"], C * E)
    D, I = oracle.search(xq, g["cent"], g["edge"], g["edge_d2"], lcb, g["pq"], offsets, enc["codes"][perm],
                         enc["lamq"][perm], perm.astype(np.int64), P=P, W=P * E, k=k, cap=1 << 20)
    qn = np.sum(xq.astype(np.float64) ** 2, axis=1, keepdims=True)
    np.testing.assert_allclose(D + qn, g["ref_ivfpq_D"], rtol=2e-4)
    assert (I == g["ref_ivfpq_I"]).mean() > 0.97
