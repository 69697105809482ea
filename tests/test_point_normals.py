"""Point-cloud normals without a GPU: the fp64 restatement (tests/point_normals_ref.py) against a per-point numpy loop,
the analytic backward against torch autograd through linalg.eigh, argument checks of ptk_point_frames_*, and the
Python and shim rejections."""
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from ptk_b200 import _lib
import point_normals_ref as ref

D = 16  # a dummy device pointer: never dereferenced, the arguments are validated before any CUDA call


def knn_np(pts, K, lengths=None):
    """(B,P,K) int64: the lexicographic K nearest (distance, index) of every valid point among its cloud's valid points
    (slots past the cloud and padded rows 0), as ptk_knn_fwd_lengths selects them."""
    B, P, _ = pts.shape
    idx = np.zeros((B, P, K), np.int64)
    for b in range(B):
        l = P if lengths is None else int(lengths[b])
        p = pts[b, :l].astype(np.float64)
        d = ((p[:, None] - p[None]) ** 2).sum(-1)
        order = np.argsort(d, axis=1, kind="stable")[:, :K]
        idx[b, :l, :order.shape[1]] = order
    return idx


def cloud(rng, B, P, scale=(1.0, 0.5, 0.1)):
    """anisotropic Gaussian clouds: well separated covariance eigenvalues in most neighbourhoods"""
    return (rng.standard_normal((B, P, 3)) * np.array(scale)).astype(np.float32)


def numpy_loop(pts, idx, lengths, disambiguate):
    B, P, K = idx.shape
    curv, frames = np.zeros((B, P, 3)), np.zeros((B, P, 3, 3))
    for b in range(B):
        l = P if lengths is None else int(lengths[b])
        for i in range(l):
            Kp = min(K, l)
            q = pts[b, idx[b, i, :Kp]].astype(np.float64)
            e = q - q.mean(0)
            lam, V = np.linalg.eigh(e.T @ e / Kp)
            if disambiguate:
                df = q - pts[b, i].astype(np.float64)
                for m in (0, 2):
                    if ((V[:, m] * df).sum(-1) > 0).sum() < 0.5 * Kp:
                        V[:, m] = -V[:, m]
                V[:, 1] = np.cross(V[:, 0], V[:, 2])
            curv[b, i], frames[b, i] = lam, V
    return curv, frames


@pytest.mark.parametrize("disambiguate", [True, False])
def test_restatement_matches_numpy_loop(disambiguate):
    rng = np.random.default_rng(0)
    pts = cloud(rng, 3, 120)
    lengths = np.array([120, 77, 9])                    # ragged, and K' = 9 < K in the last cloud
    pts[1, 77:] = np.nan                                 # padding is never read
    pts[2, 9:] = 1e30
    K = 12
    idx = knn_np(pts, K, lengths)
    curv, frames = ref.frames_f64(torch.from_numpy(pts).double(), torch.from_numpy(idx), torch.from_numpy(lengths),
                                  disambiguate)
    c_np, f_np = numpy_loop(pts, idx, lengths, disambiguate)
    valid = np.arange(120)[None] < lengths[:, None]
    assert np.abs(curv.numpy()[valid] - c_np[valid]).max() < 1e-12
    f = frames.numpy()
    if disambiguate:
        assert np.abs(f[valid] - f_np[valid]).max() < 1e-9
    else:  # solver signs: equal up to the sign of each column
        dots = np.abs((f[valid] * f_np[valid]).sum(1))
        assert np.abs(dots - 1).max() < 1e-9
    assert not np.any(curv.numpy()[~valid]) and not np.any(f[~valid])


def test_restatement_sign_rule_on_a_plane():
    """z = 0 plane, query at a corner of a grid: every neighbour has d_z = 0, so the normal (0, 0, +-1) has n_pos = 0
    and is flipped to whatever the solver did not give; the in-plane axis follows the majority."""
    g = np.stack(np.meshgrid(np.arange(5.0), np.arange(4.0) * 0.5, indexing="ij"), -1).reshape(-1, 2)
    pts = np.concatenate([g, np.zeros((20, 1))], 1)[None].astype(np.float32)
    idx = knn_np(pts, 8)
    _, frames = ref.frames_f64(torch.from_numpy(pts).double(), torch.from_numpy(idx))
    _, f_np = numpy_loop(pts, idx, None, True)
    assert np.allclose(frames.numpy(), f_np, atol=1e-12)
    assert np.allclose(np.abs(frames.numpy()[0, :, 2, 0]), 1.0)


@pytest.mark.parametrize("disambiguate", [True, False])
@pytest.mark.parametrize("which", ["normals", "curvatures", "frames", "all"])
def test_analytic_backward_matches_autograd(disambiguate, which):
    rng = np.random.default_rng(1)
    pts = cloud(rng, 2, 60)
    lengths = np.array([60, 41])
    K = 10
    idx = knn_np(pts, K, lengths)
    x = torch.from_numpy(pts).double().requires_grad_(True)
    curv, frames = ref.frames_f64(x, torch.from_numpy(idx), torch.from_numpy(lengths), disambiguate)
    g = {k: rng.standard_normal(s) for k, s in (("n", (2, 60, 3)), ("c", (2, 60, 3)), ("f", (2, 60, 3, 3)))}
    gn = g["n"] if which in ("normals", "all") else None
    gc = g["c"] if which in ("curvatures", "all") else None
    gf = g["f"] if which in ("frames", "all") else None
    loss = 0
    if gn is not None:
        loss = loss + (frames[..., 0] * torch.from_numpy(gn)).sum()
    if gc is not None:
        loss = loss + (curv * torch.from_numpy(gc)).sum()
    if gf is not None:
        loss = loss + (frames * torch.from_numpy(gf)).sum()
    loss.backward()
    got = ref.grad_analytic(pts, idx, lengths, disambiguate, gn, gc, gf, like=frames.detach().numpy())
    want = x.grad.numpy()
    assert np.abs(got - want).max() <= 1e-9 * max(np.abs(want).max(), 1.0)
    assert not np.any(got[1, 41:])


# ------------------------------------------------------------------------------------- ABI argument checks
def _fwd(pts=D, lengths=None, idx=D, dist=D, B=2, P=100, K=8, n=D, c=None, f=None):
    return _lib.lib().ptk_point_frames_fwd(pts, lengths, idx, dist, B, P, K, 1, n, c, f, None)


def _bwd(pts=D, lengths=None, idx=D, dist=D, B=2, P=100, K=8, gn=D, gc=None, gf=None, gp=D):
    return _lib.lib().ptk_point_frames_bwd(pts, lengths, idx, dist, B, P, K, 1, gn, gc, gf, gp, None)


def _det(pts=D, lengths=None, idx=D, dist=D, B=2, P=100, K=8, gn=D, gc=None, gf=None, gp=D, ws=D, nbytes=1 << 40):
    return _lib.lib().ptk_point_frames_bwd_det(pts, lengths, idx, dist, B, P, K, 1, gn, gc, gf, gp, ws, nbytes, None)


@pytest.mark.parametrize("call,nulls", [(_fwd, ["pts", "idx", "dist", "n"]), (_bwd, ["pts", "idx", "dist", "gp"]),
                                        (_det, ["pts", "idx", "dist", "gp"])])
def test_rejects_null_pointers(call, nulls):
    for null in nulls:
        assert call(**{null: None}) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error(), null


def test_fwd_rejects_half_a_frames_output():
    assert _fwd(n=None, c=D, f=None) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    assert _fwd(n=None, c=None, f=D) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    assert _fwd(n=D, c=D, f=None) == _lib.PTK_ERR_SHAPE


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("shape", [(0, 10), (1, 0), (-1, 10), (1, -3), (65536, 10), (1, 1 << 28)])
def test_rejects_bad_shapes(call, shape):
    B, P = shape
    assert call(B=B, P=P) == _lib.PTK_ERR_SHAPE and "bad sizes" in _lib.last_error()


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("K", [0, -1, 65, 1000])
def test_rejects_k_outside_range(call, K):
    assert call(K=K) == _lib.PTK_ERR_SHAPE and "outside [1, 64]" in _lib.last_error()


def test_rejects_p_times_k_overflow():
    assert _fwd(B=1, P=(1 << 31) // 9 - 1, K=64) == _lib.PTK_ERR_SHAPE and "32-bit" in _lib.last_error()


def test_bwd_det_rejects_missing_small_or_misaligned_workspace():
    need = _lib.lib().ptk_knn1_bwd_det_workspace_bytes(2, 100, 100)
    assert need == 256 + 24 * 2 * 100
    for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
        assert _det(ws=ws, nbytes=nbytes) == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()
    for off in (4, 8):
        assert _det(ws=D + off, nbytes=need) == _lib.PTK_ERR_ALIGN and "aligned" in _lib.last_error()


# ------------------------------------------------------------------------------------- Python and shim rejections
@pytest.mark.parametrize("fn", [ptk_b200.ops.estimate_normals, ptk_b200.ops.estimate_local_frames])
def test_ops_rejections(fn):
    x = torch.rand(2, 100, 3)
    with pytest.raises(NotImplementedError, match="K <= 64"):
        fn(x, neighborhood_size=65)
    for K in (0, -4):
        with pytest.raises(ValueError, match="K must be >= 1"):
            fn(x, neighborhood_size=K)
    with pytest.raises(ValueError, match="K must be an int"):
        fn(x, neighborhood_size=4.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fn(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fn(x, lengths=torch.tensor([100, 50]), neighborhood_size=8)
    with pytest.raises(ValueError, match=r"\(B,P,3\)"):
        fn(torch.rand(100, 3))


@pytest.fixture
def shim(monkeypatch):
    """The pytorch3d shim on sys.path for one test; its modules are dropped afterwards."""
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


@pytest.mark.parametrize("name", ["estimate_pointcloud_normals", "estimate_pointcloud_local_coord_frames"])
def test_shim_rejections(shim, name):
    import pytorch3d.ops
    fn = getattr(pytorch3d.ops, name)
    with pytest.raises(ValueError, match="Pointclouds objects or tensors"):
        fn(np.zeros((1, 100, 3), np.float32))
    with pytest.raises(ValueError, match="Pointclouds objects or tensors"):
        fn([[0.0, 0.0, 0.0]] * 100)
    with pytest.raises(ValueError, match=r"\(minibatch, N, 3\)"):
        fn(torch.rand(1, 100, 2))
    for P, K in ((50, 50), (10, 50), (8, 12)):
        with pytest.raises(ValueError, match="neighborhood_size"):
            fn(torch.rand(2, P, 3), neighborhood_size=K)
    with pytest.raises(NotImplementedError, match="no CPU fallback"):
        fn(torch.rand(2, 100, 3))
    with pytest.raises(NotImplementedError, match="no CPU fallback"):
        fn(torch.rand(2, 100, 3), neighborhood_size=65)
