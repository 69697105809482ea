"""fp64 restatement of PyTorch3D 0.5.0's Chamfer normal term (loss/chamfer.py, the x_normals / y_normals branch of
chamfer_distance) -- TEST INFRASTRUCTURE: the reference that test_chamfer_normals.py and test_chamfer_normals_gpu.py
compare the kernels against.  Written with the reference's own eager torch ops, independently of the kernels."""
import torch


def chamfer_normals(x_normals, y_normals, idx_x, idx_y, x_lengths=None, y_lengths=None, point_reduction="mean"):
    """The normal term of pytorch3d.loss.chamfer_distance (PyTorch3D 0.5.0 loss/chamfer.py) in fp64, given the
    nearest-neighbour indices: knn_gather with its zero fill of slots k >= lengths, F.cosine_similarity(eps=1e-6),
    padded queries masked to 0, the divisor of "mean" clamped to 1 as cham's is.  Differentiable w.r.t. the normals.
    Returns (cham_normals (B,), term_x (B,P1), term_y (B,P2))."""
    xn, yn = x_normals.double(), y_normals.double()
    N, P1, _ = xn.shape
    P2 = yn.shape[1]
    dev = xn.device

    def lens(l, P):
        return torch.full((N,), P, dtype=torch.int64, device=dev) if l is None else l.to(dev).long().clamp(0, P)

    lx, ly = lens(x_lengths, P1), lens(y_lengths, P2)

    def gather(pts, idx, lengths):  # pytorch3d.ops.knn_gather with K = 1
        out = pts.gather(1, idx.long()[..., None].expand(-1, -1, 3))
        return out.masked_fill((lengths <= 0)[:, None, None], 0.0)

    x_near, y_near = gather(yn, idx_x, ly), gather(xn, idx_y, lx)
    term_x = 1 - torch.abs(torch.nn.functional.cosine_similarity(xn, x_near, dim=2, eps=1e-6))
    term_y = 1 - torch.abs(torch.nn.functional.cosine_similarity(yn, y_near, dim=2, eps=1e-6))
    term_x = term_x.masked_fill(torch.arange(P1, device=dev)[None] >= lx[:, None], 0.0)
    term_y = term_y.masked_fill(torch.arange(P2, device=dev)[None] >= ly[:, None], 0.0)
    sx, sy = term_x.sum(1), term_y.sum(1)
    if point_reduction == "mean":
        sx, sy = sx / lx.clamp(min=1), sy / ly.clamp(min=1)
    return sx + sy, term_x, term_y
