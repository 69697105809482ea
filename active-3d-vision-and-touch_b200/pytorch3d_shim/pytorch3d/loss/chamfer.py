"""pytorch3d.loss.chamfer_distance of PyTorch3D 0.5.0, on homogeneous or ragged batches, with the normal term.

x_lengths / y_lengths (B,) give the number of points of each padded cloud: only x[b, :x_lengths[b]] and
y[b, :y_lengths[b]] take part.  With point_reduction="mean" a pair's value is sum_x / max(lx, 1) + sum_y / max(ly, 1):
an empty cloud contributes 0, as in current PyTorch3D releases, which clamp the lengths to 1 (what PyTorch3D 0.5.0
does for a zero length is not pinned).  point_reduction="sum" gives sum_x + sum_y.

With both x_normals and y_normals the second value is PyTorch3D's normal-consistency term: per valid query
1 - |cos(normal, normal of its nearest neighbour)| (F.cosine_similarity, eps=1e-6; 1 for a query whose target cloud
is empty), reduced like the distances; its gradient reaches the normals only.  With one of the two, PyTorch3D ignores
it and returns None, and so does this function.  weights and batch_reduction apply to both values.
"""
import ptk_b200


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None, weights=None,
                     batch_reduction="mean", point_reduction="mean"):
    if x_normals is not None or y_normals is not None:
        if not all(t.is_cuda for t in (x, y, x_normals, y_normals) if t is not None):
            raise NotImplementedError("ptk_b200 chamfer_distance with normals runs on CUDA (sm_100a) tensors only; got a "
                                      "CPU tensor. There is no CPU fallback.")
    if point_reduction not in ("mean", "sum"):
        raise ValueError('point_reduction must be one of ["mean", "sum"]')
    if batch_reduction not in (None, "mean", "sum"):
        raise ValueError('batch_reduction must be one of ["mean", "sum"] or None')
    if x_normals is not None and y_normals is not None:
        cham, cham_n, _, _ = ptk_b200.ops.chamfer_normals(x, y, x_normals, y_normals, x_lengths, y_lengths,
                                                          point_reduction)
    else:
        (cham, _, _), cham_n = ptk_b200.ops.chamfer(x, y, x_lengths, y_lengths, point_reduction), None
    return _batch_reduce(cham, x, weights, batch_reduction), _batch_reduce(cham_n, x, weights, batch_reduction)


def _batch_reduce(v, x, weights, batch_reduction):
    if v is None:
        return None
    if weights is not None:
        v = v * weights
    if batch_reduction == "sum":
        v = v.sum()
    elif batch_reduction == "mean":
        v = v.sum() / (weights.sum() if weights is not None else max(x.shape[0], 1))
    return v
