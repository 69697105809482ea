"""Ragged-batch Chamfer / 1-NN entry points: argument checks that run without a GPU."""
import sys

import pytest
import torch

import ptk_b200
from ptk_b200 import _lib


@pytest.fixture
def shim(monkeypatch):
    """The pytorch3d shim on sys.path for one test; its modules are dropped afterwards."""
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


def test_lengths_entry_points_reject_null_clouds_without_gpu():
    L = _lib.lib()
    rc = L.ptk_chamfer_fwd_lengths(None, None, None, None, 1, 10, 10, _lib.REDUCE_MEAN, None, None, None, None, None,
                                   None, 0, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    rc = L.ptk_chamfer_bwd_lengths(None, None, None, None, None, None, None, 1, 10, 10, _lib.REDUCE_SUM, None, None,
                                   None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    rc = L.ptk_knn1_fwd_lengths(None, None, None, None, 1, 10, 10, None, None, None, 0, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()


@pytest.mark.parametrize("reduction", [-1, 2, 7])
def test_unknown_reduction_is_a_shape_error(reduction):
    L = _lib.lib()
    dummy = 16  # never dereferenced: the arguments are validated before any CUDA call
    rc = L.ptk_chamfer_fwd_lengths(dummy, dummy, None, None, 1, 10, 10, reduction, None, dummy, None, dummy, dummy,
                                   dummy, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "reduction" in _lib.last_error()
    rc = L.ptk_chamfer_bwd_lengths(dummy, dummy, None, None, dummy, dummy, dummy, 1, 10, 10, reduction, dummy, None,
                                   None)
    assert rc == _lib.PTK_ERR_SHAPE and "reduction" in _lib.last_error()


def test_shim_still_rejects_normals_and_k_above_one(shim):
    from pytorch3d.loss import chamfer_distance
    from pytorch3d.ops import knn_points
    x = torch.rand(1, 4, 3)
    with pytest.raises(NotImplementedError):
        chamfer_distance(x, x, x_normals=x)
    with pytest.raises(NotImplementedError):
        chamfer_distance(x, x, y_normals=x)
    with pytest.raises(NotImplementedError):
        knn_points(x, x, K=2)
    with pytest.raises(NotImplementedError):
        knn_points(x, x, lengths1=torch.tensor([4]), K=3)


def test_shim_rejects_unknown_point_reduction(shim):
    from pytorch3d.loss import chamfer_distance
    x = torch.rand(1, 4, 3)
    with pytest.raises(ValueError):
        chamfer_distance(x, x, point_reduction="max")
