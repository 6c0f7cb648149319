"""Device-resident training of the VLQ codebooks on top of the C-ABI ops (torch tensors as plumbing).

Follows GpuIndexIVFPQ::train (gpu/GpuIndexIVFPQ.cu:1160-1178,345-403): coarse k-means (Clustering.cpp:66-206 with
the device assigner), centroid graph, line stage on the first 2^bits*128 rows, 1-D lambda k-means, residuals,
per-sub-space PQ k-means (ProductQuantizer.cpp:236-308).  Every distance / mean is a C-ABI kernel; only the sequential
RNG logic (permutations, empty-cluster split: utils.cpp:1419-1446) runs on the host, like in the reference.
"""
import ctypes
import ctypes.util

import numpy as np
import torch

from . import ops


class _RandomR:
    """glibc random_r on an 8-byte state, as the reference's RandomGenerator (utils.cpp:135-160)."""

    class _Data(ctypes.Structure):
        _fields_ = [("fptr", ctypes.c_void_p), ("rptr", ctypes.c_void_p), ("state", ctypes.c_void_p),
                    ("rand_type", ctypes.c_int), ("rand_deg", ctypes.c_int), ("rand_sep", ctypes.c_int),
                    ("end_ptr", ctypes.c_void_p)]

    def __init__(self, seed):
        self.libc = ctypes.CDLL(ctypes.util.find_library("c") or "libc.so.6")
        self.buf = ctypes.create_string_buffer(8)
        self.data = self._Data()
        self.libc.initstate_r(ctypes.c_uint(seed & 0xFFFFFFFF), self.buf, ctypes.c_size_t(8), ctypes.byref(self.data))
        self.out = ctypes.c_int32()

    def rand_int(self):
        self.libc.random_r(ctypes.byref(self.data), ctypes.byref(self.out))
        return self.out.value

    def rand_float(self):
        return np.float32(self.rand_int()) / np.float32(1 << 31)


def rand_perm(n, seed):
    """Fisher-Yates with random_r (utils.cpp:307-317)"""
    rng = _RandomR(seed)
    perm = np.arange(n, dtype=np.int64)
    for i in range(n - 1):
        i2 = i + rng.rand_int() % (n - i)
        perm[i], perm[i2] = perm[i2], perm[i]
    return perm


def _split_empty(cent, counts, n):
    """empty-cluster split of km_update_centroids (utils.cpp:1419-1446); cent is a device tensor, counts host int64"""
    k = counts.shape[0]
    empties = np.nonzero(counts == 0)[0]
    if len(empties) == 0:
        return 0
    rng = _RandomR(1234)
    eps = 1.0 / 1024.0
    d = cent.shape[1]
    sign = torch.ones(d, device=cent.device)
    sign[1::2] = -1.0
    for ci in empties:
        cj = 0
        while True:
            p = (counts[cj] - 1.0) / float(n - k)
            if rng.rand_float() < p:
                break
            cj = (cj + 1) % k
        cent[ci] = cent[cj] * (1 + eps * sign)
        cent[cj] = cent[cj] * (1 - eps * sign)
        counts[ci] = counts[cj] // 2
        counts[cj] -= counts[ci]
    return len(empties)


def kmeans(x, k, niter=10, seed=1234, max_points_per_centroid=256, exact_perm=True, verbose=False):
    """Clustering::train on the device.  exact_perm=False swaps the reference's sequential random_r permutation for
    torch.randperm (same distribution, not the same sample) -- used by bench.py for multi-million-row training sets."""
    n, d = x.shape
    dev = x.device
    if n > k * max_points_per_centroid:
        nn = k * max_points_per_centroid
        if exact_perm:
            perm = torch.from_numpy(rand_perm(n, seed)[:nn]).to(dev)
        else:
            g = torch.Generator(device=dev)
            g.manual_seed(seed)
            perm = torch.randperm(n, generator=g, device=dev)[:nn]
        x = x[perm].contiguous()
        n = nn
    if exact_perm:
        perm = torch.from_numpy(rand_perm(n, seed + 1)[:k]).to(dev)
    else:
        g = torch.Generator(device=dev)
        g.manual_seed(seed + 1)
        perm = torch.randperm(n, generator=g, device=dev)[:k]
    cent = x[perm].contiguous()
    obj = []
    use_tc = bool(ops._abi.lib().vlq_tc_supported(d, k))
    for it in range(niter):
        if use_tc:  # tcgen05 assignment (fp32-grade split-fp16); other shapes (d=1 lambda, d=8 PQ) use the fp32 kernel
            ids, dist = ops.l2_assign_tc(x, ops.CentPack(cent), add_xnorm=True, want_dist=verbose)
        else:
            ids, dist = ops.l2_assign(x, cent, add_xnorm=True)
        if verbose:
            obj.append(float(dist.sum()))
        cent, counts = ops.km_update(x, ids, k)
        _split_empty(cent, counts.cpu().numpy().astype(np.int64), n)
    return cent, obj


def train_vlq(xt, nlist, E, M, nL, nbits=8, niter=10, pq_niter=25, seed=1234, exact_perm=True, verbose=False):
    """-> dict(cent, cnorm, edge, edge_d2, lambda_cb, pq) of device tensors; pq is (M, 2^nbits, d / M), nbits 8 or 4
    (two codes per stored byte, M even: the ops entry points take the 4-bit form from the codebook's shape)"""
    assert nbits in (4, 8) and (nbits == 8 or M % 2 == 0), "PQ codes are 8-bit, or 4-bit with an even M"
    d = xt.shape[1]
    cent, _ = kmeans(xt, nlist, niter=niter, seed=seed, exact_perm=exact_perm, verbose=verbose)
    cnorm = ops.row_norms(cent)
    edge, ed2 = ops.knn_graph(cent, E, cnorm)
    n2 = min(xt.shape[0], (1 << nbits) * 128)
    x2 = xt[:n2].contiguous()
    pack = ops.CentPack(cent, cnorm) if ops._abi.lib().vlq_tc_supported(d, nlist) else None
    A, _ = ops.l2_assign_tc(x2, pack, want_dist=False) if pack is not None else ops.l2_assign(x2, cent, cnorm)
    st = ops.line_encode(x2, A, cent, edge, ed2)
    lcb, _ = kmeans(st.lam.reshape(-1, 1).contiguous(), nL, niter=niter, seed=seed, exact_perm=exact_perm)
    lcb = lcb.reshape(-1).contiguous()
    # residuals need the PQ argument only formally: encode against a dummy codebook to obtain them
    dsub = d // M
    dummy = torch.zeros((M, 256, dsub), dtype=torch.float32, device=xt.device)
    enc = ops.line_encode(x2, A, cent, edge, ed2, lcb, dummy, want_residual=True)
    r = enc.residual
    ksub = 1 << nbits
    pq = torch.empty((M, ksub, dsub), dtype=torch.float32, device=xt.device)
    for m in range(M):
        sub = r[:, m * dsub:(m + 1) * dsub].contiguous()
        pq[m], _ = kmeans(sub, ksub, niter=pq_niter, seed=seed, exact_perm=exact_perm)
    return dict(cent=cent, cnorm=cnorm, edge=edge, edge_d2=ed2, lambda_cb=lcb, pq=pq, pack=pack)
