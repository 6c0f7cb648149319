"""Fused coarse select (csl::coarse_select_lines_fast_kernel) at graph degrees that split a centroid's lines across
threads in every way (E below, above and not a multiple of the per-thread line count), with duplicate centroids for
exact ties, against the two-step path select_rows + select_lines, bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("nq,C,P,W,E,dup", [(17, 3000, 64, 256, 5, False), (11, 2000, 48, 300, 12, False),
                                            (9, 4096, 64, 256, 24, True), (8, 4000, 40, 200, 40, False),
                                            # 16 keys per thread, two batches of bucket lines per warp
                                            (6, 4096, 100, 512, 24, True), (5, 1000, 16, 64, 3, True)])
def test_fused_select_any_degree(cuda, nq, C, P, W, E, dup):
    import torch

    from vector_line_quantization_b200 import ops

    rng = np.random.RandomState(C + E)
    d = 128
    c = np.clip(np.rint(rng.normal(60, 40, (C, d))), 0, 255).astype(np.float32)
    if dup:  # every 7th centroid repeats its predecessor: equal distances, ordered by id
        c[7::7] = c[6:-1:7][: c[7::7].shape[0]]
    x = np.clip(np.rint(rng.normal(60, 40, (nq, d))), 0, 255).astype(np.float32)
    xt, ct = torch.from_numpy(x).to(cuda), torch.from_numpy(c).to(cuda)
    pack = ops.CentPack(ct)
    bm = torch.empty((nq, ops.num_buckets(C)), dtype=torch.float32, device=cuda)
    D = ops.l2_distances_tc(xt, pack, bucket_min=bm)
    g = torch.Generator(device="cpu").manual_seed(E)
    edge = torch.stack([torch.randperm(C, generator=g)[:E] for _ in range(C)]).to(torch.int32).to(cuda)
    ed2 = (torch.rand((C, E), generator=g) * 1000 + 1).to(cuda)
    _, cid = ops.select_rows(D, P)
    l0, a0, b0 = ops.select_lines(D, cid, edge, ed2, W)
    l1, a1, b1, cid1 = ops.coarse_select_lines(D, bm, C, P, edge, ed2, W, want_coarse=True)
    assert torch.equal(cid1, cid)
    assert torch.equal(l1, l0) and torch.equal(a1, a0) and torch.equal(b1, b0)
