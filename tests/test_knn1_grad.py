"""1-NN backward entry points (ptk_knn1_bwd_lengths, ptk_knn1_bwd_det) and the shim's knn_gather, without a GPU."""
import sys

import pytest
import torch

import ptk_b200
from ptk_b200 import _lib

D = 16  # a dummy device pointer: never dereferenced, the arguments are validated before any CUDA call


@pytest.fixture
def shim(monkeypatch):
    """The pytorch3d shim on sys.path for one test; its modules are dropped afterwards."""
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


def _bwd(p1=D, p2=D, idx=D, g=D, B=2, P1=100, P2=50, g1=D, g2=D):
    return _lib.lib().ptk_knn1_bwd_lengths(p1, p2, None, None, idx, g, B, P1, P2, g1, g2, None)


def _det(p1=D, p2=D, idx=D, g=D, B=2, P1=100, P2=50, g1=D, g2=D, ws=D, nbytes=1 << 20):
    return _lib.lib().ptk_knn1_bwd_det(p1, p2, None, None, idx, g, B, P1, P2, g1, g2, ws, nbytes, None)


@pytest.mark.parametrize("call", [_bwd, _det])
@pytest.mark.parametrize("null", ["p1", "p2", "idx", "g"])
def test_knn1_bwd_rejects_null_pointers(call, null):
    assert call(**{null: None}) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()


@pytest.mark.parametrize("call", [_bwd, _det])
@pytest.mark.parametrize("shape", [(0, 10, 10), (1, 0, 10), (1, 10, 0), (-1, 10, 10), (1, 1 << 30, 10), (70000, 10, 10)])
def test_knn1_bwd_rejects_bad_shapes(call, shape):
    B, P1, P2 = shape
    kw = {"nbytes": 1 << 40} if call is _det else {}
    assert call(B=B, P1=P1, P2=P2, **kw) == _lib.PTK_ERR_SHAPE


def test_knn1_bwd_det_rejects_missing_or_small_workspace():
    need = _lib.lib().ptk_knn1_bwd_det_workspace_bytes(2, 100, 50)
    for g1, g2 in ((D, D), (D, None), (None, D)):
        for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
            assert _det(g1=g1, g2=g2, ws=ws, nbytes=nbytes) == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()


def test_knn1_bwd_without_requested_gradients_is_a_no_op():
    assert _bwd(g1=None, g2=None) == 0
    assert _det(g1=None, g2=None, ws=None, nbytes=0) == 0
    # the no-op comes before the batch-size check (which ptk_knn_bwd_* makes first)
    assert _bwd(B=70000, g1=None, g2=None) == 0
    assert _det(B=70000, g1=None, g2=None, ws=None, nbytes=0) == 0


def test_knn1_bwd_det_workspace_sizes():
    L = _lib.lib()
    # [M_b bits, padded to 256 B][24 B per p2 point]
    assert L.ptk_knn1_bwd_det_workspace_bytes(2, 100, 50) == 256 + 2400
    assert L.ptk_knn1_bwd_det_workspace_bytes(1, 7, 1) == 256 + 24
    assert L.ptk_knn1_bwd_det_workspace_bytes(65, 10, 3) == 512 + 65 * 72
    assert L.ptk_knn1_bwd_det_workspace_bytes(256, 10000, 10000) == 1024 + 256 * 10000 * 24
    for shape in ((0, 10, 10), (1, 0, 10), (1, 10, 0), (-1, 10, 10)):
        assert L.ptk_knn1_bwd_det_workspace_bytes(*shape) == 0


# ------------------------------------------------------------------------------------- shim knn_gather on CPU tensors
def test_knn_gather_gathers_and_masks_slots_past_the_length(shim):
    from pytorch3d.ops import knn_gather
    x = torch.arange(2 * 5 * 3, dtype=torch.float32).reshape(2, 5, 3) + 1  # no zero entries
    idx = torch.tensor([[[4, 0, 2], [1, 1, 3]], [[0, 2, 4], [3, 2, 1]]])
    want = torch.stack([x[b][idx[b]] for b in range(2)])  # (2, 2, 3, 3)
    assert torch.equal(knn_gather(x, idx), want)
    for lens in ([0, 1], [1, 3], [3, 5], [7, 2]):
        got = knn_gather(x, idx, torch.tensor(lens))
        for b in range(2):
            k = min(lens[b], 3)
            assert torch.equal(got[b, :, :k], want[b, :, :k])
            assert not got[b, :, k:].any()


def test_knn_gather_padded_queries_gather_row_zero(shim):
    from pytorch3d.ops import knn_points, knn_gather  # noqa: F401  (knn_points: both names exported)
    x = torch.rand(2, 6, 3) + 1
    idx = torch.zeros(2, 4, 1, dtype=torch.int64)  # what knn_points returns for padded queries
    got = knn_gather(x, idx, torch.tensor([6, 2]))
    assert torch.equal(got, x[:, :1, None].expand(2, 4, 1, 3))
    assert not knn_gather(x, idx, torch.tensor([0, 2]))[0].any()


def test_knn_gather_gradient_reaches_x(shim):
    from pytorch3d.ops import knn_gather
    x = torch.rand(2, 5, 3, dtype=torch.float64, requires_grad=True)
    idx = torch.tensor([[[4, 0], [4, 2]], [[1, 1], [3, 0]]])
    lens = torch.tensor([5, 1])
    w = torch.rand(2, 2, 2, 3, dtype=torch.float64)
    (knn_gather(x, idx, lens) * w).sum().backward()
    want = torch.zeros(2, 5, 3, dtype=torch.float64)
    for b in range(2):
        for i in range(2):
            for k in range(2):
                if k < lens[b]:
                    want[b, idx[b, i, k]] += w[b, i, k]
    assert torch.equal(x.grad, want)
    assert torch.autograd.gradcheck(lambda t: knn_gather(t, idx, lens), (x,))


def test_knn_gather_rejects_a_batch_mismatch(shim):
    from pytorch3d.ops import knn_gather
    with pytest.raises(ValueError):
        knn_gather(torch.rand(2, 5, 3), torch.zeros(3, 4, 1, dtype=torch.int64))


def test_knn_points_still_rejects_k_above_one_and_normals(shim):
    from pytorch3d.loss import chamfer_distance
    from pytorch3d.ops import knn_points
    x = torch.rand(1, 4, 3)
    with pytest.raises(NotImplementedError):
        knn_points(x, x, K=2)
    with pytest.raises(NotImplementedError):
        knn_points(x, x, K=2, return_nn=True)
    with pytest.raises(NotImplementedError):
        chamfer_distance(x, x, x_normals=x, y_normals=x)
