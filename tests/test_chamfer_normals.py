"""The Chamfer normal term without a GPU: argument checks of ptk_chamfer_normals_*, the Python and shim front ends on
CPU tensors, and the fp64 restatement of PyTorch3D's term (tests/chamfer_normals_ref.py) against a per-query loop."""
import math
import sys

import pytest
import torch

import ptk_b200
from ptk_b200 import _lib
import chamfer_normals_ref

D = 16  # a dummy device pointer: never dereferenced, the arguments are validated before any CUDA call
MEAN, SUM = _lib.REDUCE_MEAN, _lib.REDUCE_SUM


@pytest.fixture
def shim(monkeypatch):
    """The pytorch3d shim on sys.path for one test; its modules are dropped afterwards."""
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


def _fwd(xn=D, yn=D, ix=D, iy=D, B=2, P1=100, P2=50, red=MEAN, cn=D, ws=D, nbytes=1 << 20):
    return _lib.lib().ptk_chamfer_normals_fwd(xn, yn, None, None, ix, iy, B, P1, P2, red, None, None, cn, ws, nbytes, None)


def _bwd(xn=D, yn=D, ix=D, iy=D, g=D, B=2, P1=100, P2=50, red=MEAN, gx=D, gy=D):
    return _lib.lib().ptk_chamfer_normals_bwd(xn, yn, None, None, ix, iy, g, B, P1, P2, red, gx, gy, None)


def _det(xn=D, yn=D, ix=D, iy=D, g=D, B=2, P1=100, P2=50, red=MEAN, gx=D, gy=D, ws=D, nbytes=1 << 20):
    return _lib.lib().ptk_chamfer_normals_bwd_det(xn, yn, None, None, ix, iy, g, B, P1, P2, red, gx, gy, ws, nbytes, None)


@pytest.mark.parametrize("call,nulls", [(_fwd, ["xn", "yn", "ix", "iy", "cn"]), (_bwd, ["xn", "yn", "ix", "iy", "g"]),
                                        (_det, ["xn", "yn", "ix", "iy", "g"])])
def test_rejects_null_pointers(call, nulls):
    for null in nulls:
        assert call(**{null: None}) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error(), null


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("shape", [(0, 10, 10), (1, 0, 10), (1, 10, 0), (-1, 10, 10), (1, 1 << 30, 10), (70000, 10, 10)])
def test_rejects_bad_shapes(call, shape):
    B, P1, P2 = shape
    kw = {} if call is _bwd else {"nbytes": 1 << 40}
    assert call(B=B, P1=P1, P2=P2, **kw) == _lib.PTK_ERR_SHAPE


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("red", [-1, 2, 7])
def test_rejects_unknown_reduction(call, red):
    assert call(red=red) == _lib.PTK_ERR_SHAPE and "reduction" in _lib.last_error()


def test_fwd_workspace_only_for_sliced_clouds():
    L = _lib.lib()
    # up to FIN_SLICE = 16384 points per cloud one CTA per pair writes cham_normals: no workspace
    assert L.ptk_chamfer_normals_workspace_bytes(256, 10000, 10000) == 0
    assert L.ptk_chamfer_normals_workspace_bytes(3, 16384, 7) == 0
    # beyond it: two fp32 partials per slice of every pair, ceil(max(P1, P2) / 16384) slices, at most 64
    assert L.ptk_chamfer_normals_workspace_bytes(3, 16385, 7) == 3 * 2 * 8
    assert L.ptk_chamfer_normals_workspace_bytes(2, 100, 50000) == 2 * 4 * 8
    assert L.ptk_chamfer_normals_workspace_bytes(1, 1 << 21, 5) == 64 * 8
    for shape in ((0, 10, 10), (1, 0, 10), (1, 10, 0), (-1, 10, 10)):
        assert L.ptk_chamfer_normals_workspace_bytes(*shape) == 0


def test_fwd_rejects_missing_small_or_misaligned_workspace():
    need = _lib.lib().ptk_chamfer_normals_workspace_bytes(2, 20000, 50)
    for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
        assert _fwd(P1=20000, ws=ws, nbytes=nbytes) == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()
    assert _fwd(P1=20000, ws=D + 4, nbytes=need) == _lib.PTK_ERR_ALIGN


def test_bwd_det_uses_the_chamfer_det_workspace():
    need = _lib.lib().ptk_chamfer_bwd_det_workspace_bytes(2, 100, 50)
    for gx, gy in ((D, D), (D, None), (None, D)):
        for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
            assert _det(gx=gx, gy=gy, ws=ws, nbytes=nbytes) == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()
    assert _det(ws=D + 4, nbytes=need) == _lib.PTK_ERR_ALIGN


def test_bwd_without_requested_gradients_is_a_no_op():
    assert _bwd(gx=None, gy=None) == 0
    assert _det(gx=None, gy=None, ws=None, nbytes=0) == 0


# ------------------------------------------------------------------------------------- Python front ends, CPU tensors
def test_ops_rejects_normals_of_the_wrong_shape():
    x, y = torch.rand(2, 5, 3), torch.rand(2, 4, 3)
    for xn, yn in ((torch.rand(2, 4, 3), torch.rand(2, 4, 3)), (torch.rand(2, 5, 3), torch.rand(2, 5, 3)),
                   (torch.rand(1, 5, 3), torch.rand(2, 4, 3)), (torch.rand(2, 5), torch.rand(2, 4, 3)),
                   (None, torch.rand(2, 4, 3))):
        with pytest.raises(ValueError, match="normals"):
            ptk_b200.ops.chamfer_normals(x, y, xn, yn)
    with pytest.raises(ValueError, match="point_reduction"):
        ptk_b200.ops.chamfer_normals(x, y, torch.rand(2, 5, 3), torch.rand(2, 4, 3), point_reduction="max")


def test_ops_rejects_cpu_tensors():
    x, y = torch.rand(2, 5, 3), torch.rand(2, 4, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ptk_b200.ops.chamfer_normals(x, y, x, y)


def test_shim_rejects_cpu_normals(shim):
    from pytorch3d.loss import chamfer_distance
    x, y = torch.rand(2, 5, 3), torch.rand(2, 4, 3)
    for kw in ({"x_normals": x}, {"y_normals": y}, {"x_normals": x, "y_normals": y}):
        with pytest.raises(NotImplementedError, match="no CPU fallback"):
            chamfer_distance(x, y, **kw)


# ------------------------------------------------------------------------------------- the fp64 restatement
def _loop_reference(xn, yn, ix, iy, lx, ly, reduction):
    """One query at a time, from the formula: c = sum_k a_k / max(|a|, eps) * n_k / max(|n|, eps), term = 1 - |c|."""
    B, P1, P2 = xn.shape[0], xn.shape[1], yn.shape[1]

    def term(a, n):
        na = max(math.sqrt(sum(v * v for v in a)), 1e-6)
        nn = max(math.sqrt(sum(v * v for v in n)), 1e-6)
        return 1.0 - abs(sum((a[k] / na) * (n[k] / nn) for k in range(3)))

    out, tx, ty = [], torch.zeros(B, P1, dtype=torch.float64), torch.zeros(B, P2, dtype=torch.float64)
    for b in range(B):
        l1, l2 = min(max(int(lx[b]), 0), P1), min(max(int(ly[b]), 0), P2)
        for i in range(l1):
            n = yn[b, int(ix[b, i])].tolist() if l2 > 0 else [0.0, 0.0, 0.0]
            tx[b, i] = term(xn[b, i].tolist(), n)
        for i in range(l2):
            n = xn[b, int(iy[b, i])].tolist() if l1 > 0 else [0.0, 0.0, 0.0]
            ty[b, i] = term(yn[b, i].tolist(), n)
        sx, sy = float(tx[b].sum()), float(ty[b].sum())
        out.append(sx / max(l1, 1) + sy / max(l2, 1) if reduction == "mean" else sx + sy)
    return torch.tensor(out, dtype=torch.float64), tx, ty


@pytest.mark.parametrize("reduction", ["mean", "sum"])
def test_restatement_matches_a_per_query_loop(reduction):
    g = torch.Generator().manual_seed(3)
    B, P1, P2 = 5, 6, 4
    xn = torch.randn(B, P1, 3, generator=g) * torch.rand(B, P1, 1, generator=g) * 3
    yn = torch.randn(B, P2, 3, generator=g)
    xn[0, 1] = 0.0                           # a zero normal: term 1
    yn[1, 2] = torch.tensor([1e-7, 0, 0])    # below eps: its clamped norm is eps
    xn[0, 2] = -3.0 * yn[0, 0]               # flipped and scaled: term 0
    ix = torch.randint(0, P2, (B, P1), generator=g, dtype=torch.int32)
    iy = torch.randint(0, P1, (B, P2), generator=g, dtype=torch.int32)
    ix[0, 2] = 0
    lx = torch.tensor([6, 3, 6, 0, 9])       # an empty x cloud, and a length above P (clamped)
    ly = torch.tensor([4, 4, 0, 2, -1])      # an empty y cloud and a negative length (clamped to 0)
    got, gtx, gty = chamfer_normals_ref.chamfer_normals(xn, yn, ix, iy, lx, ly, reduction)
    want, wtx, wty = _loop_reference(xn.double(), yn.double(), ix, iy, lx, ly, reduction)
    assert torch.allclose(gtx, wtx, atol=1e-12, rtol=0) and torch.allclose(gty, wty, atol=1e-12, rtol=0)
    assert torch.allclose(got, want, atol=1e-12, rtol=1e-12)
    assert gtx[0, 1] == 1.0 and abs(float(gtx[0, 2])) < 1e-12
    assert torch.all(gtx[2, :6] == 1.0)      # valid x queries of a pair with an empty y cloud: 1 each
    assert not gtx[1, 3:].any() and not gtx[3].any() and not gty[2].any() and not gty[4].any()


def test_restatement_gradient_reaches_the_normals_only_and_not_padding():
    g = torch.Generator().manual_seed(4)
    xn = torch.randn(2, 5, 3, generator=g, dtype=torch.float64, requires_grad=True)
    yn = torch.randn(2, 4, 3, generator=g, dtype=torch.float64, requires_grad=True)
    ix = torch.randint(0, 2, (2, 5), generator=g)
    iy = torch.randint(0, 3, (2, 4), generator=g)
    lx, ly = torch.tensor([3, 5]), torch.tensor([2, 0])
    cham_n, _, _ = chamfer_normals_ref.chamfer_normals(xn, yn, ix, iy, lx, ly)
    cham_n.sum().backward()
    assert not xn.grad[0, 3:].any() and not yn.grad[0, 2:].any()
    assert not yn.grad[1].any()              # ly = 0: no y query and nothing gathered from y
    assert xn.grad[0, :3].abs().sum() > 0
