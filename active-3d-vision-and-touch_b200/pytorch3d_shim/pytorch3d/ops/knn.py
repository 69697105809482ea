"""pytorch3d.ops.knn_points for 1 <= K <= 64 and pytorch3d.ops.knn_gather, on homogeneous or ragged batches (lengths1 /
lengths2: padded queries, queries whose target cloud is empty and slots k >= lengths2 get dist 0 and idx 0, as in
PyTorch3D).  dists and knn are differentiable w.r.t. p1 and p2, as PyTorch3D's are."""
from collections import namedtuple

import torch

import ptk_b200

_KNN = namedtuple("KNN", "dists idx knn")


def knn_points(p1, p2, lengths1=None, lengths2=None, K=1, version=-1, return_nn=False, return_sorted=True):
    """`version` is ignored; return_sorted=False returns the sorted order too (a valid unsorted order)."""
    if K == 1:
        dists, idx = ptk_b200.ops.knn1(p1, p2, lengths1, lengths2)
        idx = idx.long()[..., None]
        knn = knn_gather(p2, idx, lengths2) if return_nn else None
        return _KNN(dists=dists[..., None], idx=idx, knn=knn)
    if isinstance(K, int) and K >= 2 and not (p1.is_cuda and p2.is_cuda):
        raise NotImplementedError(
            "ptk_b200 ops run on CUDA (sm_100a) tensors only; got a CPU tensor. There is no CPU fallback.")
    dists, idx = ptk_b200.ops.knn(p1, p2, K, lengths1, lengths2)
    idx = idx.long()
    knn = knn_gather(p2, idx, lengths2) if return_nn else None
    return _KNN(dists=dists, idx=idx, knn=knn)


def knn_gather(x, idx, lengths=None):
    """x (N,M,U), idx (N,L,K) int64 -> (N,L,K,U): out[n,l,k] = x[n, idx[n,l,k]], and 0 where k >= lengths[n] (N,), the
    neighbour slots a cloud of lengths[n] points cannot fill.  PyTorch3D's function, except that the mask is applied
    unconditionally instead of after a host-side `lengths.min() < K` check, so the call never synchronises."""
    N, M, U = x.shape
    _N, L, K = idx.shape
    if N != _N:
        raise ValueError("x and idx must have same batch dimension.")
    out = x[:, :, None].expand(-1, -1, K, -1).gather(1, idx[:, :, :, None].expand(-1, -1, -1, U))
    if lengths is None:
        if K <= M:
            return out
        lengths = torch.full((N,), M, dtype=torch.int64, device=x.device)
    mask = lengths.to(device=x.device, non_blocking=True)[:, None] <= torch.arange(K, device=x.device)[None]  # (N, K): slots past the cloud
    return out.masked_fill(mask[:, None, :, None], 0.0)
