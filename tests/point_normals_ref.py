"""fp64 restatements of the point-cloud normals and local frames of include/ptk.h (ptk_point_frames_fwd / _bwd), given
the K-NN indices: PyTorch3D 0.5.0's estimate_pointcloud_local_coord_frames, with torch.linalg.eigh in place of the
removed torch.symeig.

  frames_f64     eager torch in float64, differentiable through linalg.eigh: the values and the gradients the kernels
                 approximate in fp32.
  grad_analytic  numpy float64, the backward as the kernels compute it (fold of the upstream gradients into the
                 eigenvectors, linalg.eigh's backward, one term per neighbour slot): checked against frames_f64's
                 autograd without a GPU.
Cloud b has l = lengths[b] valid points (P without lengths) and K' = min(K, l) neighbours per query; padded rows are 0."""
import numpy as np
import torch


def _len(lengths, b, P):
    return P if lengths is None else int(min(max(int(lengths[b]), 0), P))


def _disambiguate(v, df, Kp):
    """v (l,3), df (l,K',3) = q_k - p_i: v negated where fewer than half the neighbours have v . df > 0."""
    n_pos = ((v[:, None] * df).sum(-1) > 0).to(v.dtype).sum(1, keepdim=True)
    return torch.where(n_pos < 0.5 * Kp, -v, v)


def frames_f64(points, idx, lengths=None, disambiguate=True):
    """points (B,P,3) float64 tensor (may require grad), idx (B,P,K) -> curvatures (B,P,3), frames (B,P,3,3)."""
    B, P, _ = points.shape
    K = idx.shape[2]
    curv, frames = [], []
    for b in range(B):
        l = _len(lengths, b, P)
        if l == 0:
            curv.append(points.new_zeros(P, 3))
            frames.append(points.new_zeros(P, 3, 3))
            continue
        Kp = min(K, l)
        p = points[b, :l]
        q = p[idx[b, :l, :Kp].long().cpu()]                       # (l, K', 3)
        e = q - q.mean(1, keepdim=True)
        lam, V = torch.linalg.eigh(e.transpose(1, 2) @ e / Kp)
        if disambiguate:
            df = q - p[:, None]
            n, z = _disambiguate(V[..., 0], df, Kp), _disambiguate(V[..., 2], df, Kp)
            F = torch.stack([n, torch.linalg.cross(n, z, dim=-1), z], -1)
        else:
            F = V
        curv.append(torch.cat([lam, points.new_zeros(P - l, 3)]))
        frames.append(torch.cat([F, points.new_zeros(P - l, 3, 3)]))
    return torch.stack(curv), torch.stack(frames)


def sign_margins(points, idx, lengths, frames, tol):
    """(B,P,2) float64: |n_pos - K'/2| for columns 0 and 2 of the given (undisambiguated) frames, and (B,P,2) the number
    of slots whose projection is within (8 * 2^-24 + tol) |q - p| of 0, tol (B,P,2) the angle error allowed for the
    two columns: a sign is certain where the margin exceeds that count."""
    B, P, K = idx.shape
    margin = torch.zeros(B, P, 2, dtype=torch.float64)
    near = torch.zeros(B, P, 2, dtype=torch.float64)
    for b in range(B):
        l = _len(lengths, b, P)
        if l == 0:
            continue
        Kp = min(K, l)
        p = points[b, :l].double()
        df = p[idx[b, :l, :Kp].long().cpu()] - p[:, None]
        for c, col in enumerate((0, 2)):
            proj = (frames[b, :l, :, col][:, None] * df).sum(-1)
            margin[b, :l, c] = ((proj > 0).double().sum(1) - 0.5 * Kp).abs()
            bound = (8 * 2.0 ** -24 + tol[b, :l, c, None]) * df.norm(dim=-1)
            near[b, :l, c] = (proj.abs() <= bound).double().sum(1)
    return margin, near


def grad_analytic(points, idx, lengths, disambiguate, g_normals=None, g_curv=None, g_frames=None, like=None):
    """numpy float64: the gradient w.r.t. points (B,P,3) under the upstream gradients (any may be None), computed the
    way ptk_point_frames_bwd computes it.  like (B,P,3,3): frames whose eigenvector signs the solver's are aligned to
    (the upstream gradient of an undisambiguated frame depends on the signs it was taken at)."""
    points = np.asarray(points, np.float64)
    B, P, _ = points.shape
    K = idx.shape[2]
    out = np.zeros_like(points)
    for b in range(B):
        l = _len(lengths, b, P)
        for i in range(l):
            Kp = min(K, l)
            j = np.asarray(idx[b, i, :Kp], np.int64)
            q = points[b, j]
            e = q - q.mean(0)
            lam, V = np.linalg.eigh(e.T @ e / Kp)
            if like is not None:
                V = V * np.where((V * np.asarray(like[b, i])).sum(0) < 0, -1.0, 1.0)
            gv = np.zeros((3, 3))                                  # gv[:, m]: gradient of eigenvector m
            if g_frames is not None:
                gv += g_frames[b, i]
            if g_normals is not None:
                gv[:, 0] += g_normals[b, i]
            gl = np.zeros(3) if g_curv is None else np.asarray(g_curv[b, i], np.float64)
            if disambiguate:
                df = q - points[b, i]
                s = [1.0 if 2 * int(((V[:, m] * df).sum(-1) > 0).sum()) >= Kp else -1.0 for m in (0, 2)]
                n, z = s[0] * V[:, 0], s[1] * V[:, 2]
                gn = gv[:, 0] + np.cross(z, gv[:, 1])
                gz = gv[:, 2] + np.cross(gv[:, 1], n)
                gv = np.stack([s[0] * gn, np.zeros(3), s[1] * gz], 1)
            W = V.T @ gv
            M = np.diag(gl)
            for m in range(3):
                for n_ in range(3):
                    if m != n_ and lam[n_] != lam[m]:
                        M[m, n_] = W[m, n_] / (lam[n_] - lam[m])
            S = V @ (M + M.T) @ V.T / Kp
            np.add.at(out[b], j, e @ S.T)
    return out
