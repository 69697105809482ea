"""pytorch3d.loss.chamfer_distance for the call shape the reference uses (utils.py:207,212), plus ragged batches.

x_lengths / y_lengths (B,) give the number of points of each padded cloud: only x[b, :x_lengths[b]] and
y[b, :y_lengths[b]] take part.  With point_reduction="mean" a pair's value is sum_x / max(lx, 1) + sum_y / max(ly, 1):
an empty cloud contributes 0, as in current PyTorch3D releases, which clamp the lengths to 1 (what PyTorch3D 0.5.0
does for a zero length is not pinned).  point_reduction="sum" gives sum_x + sum_y.
"""
import ptk_b200


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None, weights=None,
                     batch_reduction="mean", point_reduction="mean"):
    if x_normals is not None or y_normals is not None:
        raise NotImplementedError("ptk_b200 chamfer_distance supports clouds without normals "
                                  "(the only form pterotactyl calls)")
    if point_reduction not in ("mean", "sum"):
        raise ValueError('point_reduction must be one of ["mean", "sum"]')
    if batch_reduction not in (None, "mean", "sum"):
        raise ValueError('batch_reduction must be one of ["mean", "sum"] or None')
    cham, _, _ = ptk_b200.ops.chamfer(x, y, x_lengths, y_lengths, point_reduction)
    if weights is not None:
        cham = cham * weights
    if batch_reduction == "sum":
        cham = cham.sum()
    elif batch_reduction == "mean":
        cham = cham.sum() / (weights.sum() if weights is not None else max(x.shape[0], 1))
    return cham, None
