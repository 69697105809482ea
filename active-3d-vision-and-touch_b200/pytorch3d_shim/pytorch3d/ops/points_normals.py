"""pytorch3d.ops.estimate_pointcloud_normals and estimate_pointcloud_local_coord_frames of PyTorch3D 0.5.0, over
ptk_b200.ops.estimate_normals / estimate_local_frames (include/ptk.h: ptk_point_frames_fwd).  The input is a (B,P,3)
tensor, as convert_pointclouds_to_tensor accepts it; there is no Pointclouds stand-in.  Differentiable w.r.t. the
points, as PyTorch3D's are."""
import torch

import ptk_b200


def _check(pointclouds, neighborhood_size):
    if not torch.is_tensor(pointclouds):
        raise ValueError("The inputs X, Y should be either Pointclouds objects or tensors.")
    if pointclouds.dim() != 3 or pointclouds.shape[2] != 3:
        raise ValueError("The pointclouds argument has to be of shape (minibatch, N, 3)")
    if isinstance(neighborhood_size, int) and pointclouds.shape[1] <= neighborhood_size:
        raise ValueError("The neighborhood_size argument has to be >= size of each of the point clouds.")
    if not pointclouds.is_cuda:
        raise NotImplementedError(
            "ptk_b200 ops run on CUDA (sm_100a) tensors only; got a CPU tensor. There is no CPU fallback.")


def estimate_pointcloud_normals(pointclouds, neighborhood_size=50, disambiguate_directions=True):
    """normals (B,P,3): the unit eigenvector of the smallest eigenvalue of each point's neighbourhood covariance, signed
    by the majority of its neighbours when disambiguate_directions.  1 <= neighborhood_size <= 64 (more raises
    NotImplementedError) and below the number of points, as in PyTorch3D."""
    _check(pointclouds, neighborhood_size)
    return ptk_b200.ops.estimate_normals(pointclouds, None, neighborhood_size, disambiguate_directions)


def estimate_pointcloud_local_coord_frames(pointclouds, neighborhood_size=50, disambiguate_directions=True):
    """(curvatures (B,P,3), local_coord_frames (B,P,3,3)): the ascending eigenvalues of each point's neighbourhood
    covariance and the frame whose first column is estimate_pointcloud_normals' normal."""
    _check(pointclouds, neighborhood_size)
    return ptk_b200.ops.estimate_local_frames(pointclouds, None, neighborhood_size, disambiguate_directions)
