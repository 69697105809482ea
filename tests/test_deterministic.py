"""Deterministic backward entry points (ptk_*_bwd_det): argument checks and workspace sizes, without a GPU."""
import pytest

from ptk_b200 import _lib

D = 16  # a dummy device pointer: never dereferenced, the arguments are validated before any CUDA call


def test_chamfer_bwd_det_rejects_null_pointers():
    L = _lib.lib()
    rc = L.ptk_chamfer_bwd_det(None, None, None, None, D, D, D, 1, 10, 10, _lib.REDUCE_MEAN, D, D, D, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    rc = L.ptk_chamfer_bwd_det(D, D, None, None, None, D, D, 1, 10, 10, _lib.REDUCE_MEAN, D, D, D, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    rc = L.ptk_chamfer_bwd_det(D, D, None, None, D, D, None, 1, 10, 10, _lib.REDUCE_SUM, D, D, D, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()


@pytest.mark.parametrize("reduction", [-1, 2, 7])
def test_chamfer_bwd_det_rejects_unknown_reduction(reduction):
    rc = _lib.lib().ptk_chamfer_bwd_det(D, D, None, None, D, D, D, 1, 10, 10, reduction, D, D, D, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "reduction" in _lib.last_error()


def test_chamfer_bwd_det_rejects_small_workspace():
    L = _lib.lib()
    need = L.ptk_chamfer_bwd_det_workspace_bytes(2, 100, 50)
    for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
        rc = L.ptk_chamfer_bwd_det(D, D, None, None, D, D, D, 2, 100, 50, _lib.REDUCE_MEAN, D, None, ws, nbytes, None)
        assert rc == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()
    # neither gradient requested: nothing to do, no workspace needed
    assert L.ptk_chamfer_bwd_det(D, D, None, None, D, D, D, 2, 100, 50, _lib.REDUCE_MEAN, None, None, None, 0, None) == 0


def test_sample_bwd_det_rejects_null_pointers_and_small_workspace():
    L = _lib.lib()
    rc = L.ptk_sample_bwd_det(None, D, D, D, 1, 10, 4, 100, D, D, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    rc = L.ptk_sample_bwd_det(D, D, D, D, 1, 10, 4, 100, None, D, 1 << 20, None)
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    need = L.ptk_sample_bwd_det_workspace_bytes(2, 10)
    for ws, nbytes in ((None, need), (D, need - 1)):
        rc = L.ptk_sample_bwd_det(D, D, D, D, 2, 10, 4, 100, D, ws, nbytes, None)
        assert rc == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()


def test_mesh_chamfer_bwd_det_rejects_null_pointers_and_small_workspace():
    L = _lib.lib()
    args = lambda gt, ws, nbytes: (gt, D, D, D, D, D, D, D, 2, 10, 4, 100, 50, 3, D, D, ws, nbytes, None)
    rc = L.ptk_mesh_chamfer_bwd_det(*args(None, D, 1 << 30))
    assert rc == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()
    need = L.ptk_mesh_chamfer_bwd_det_workspace_bytes(2, 10, 4, 100, 50)
    for ws, nbytes in ((None, need), (D, need - 1)):
        rc = L.ptk_mesh_chamfer_bwd_det(*args(D, ws, nbytes))
        assert rc == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()


def test_det_workspace_sizes():
    L = _lib.lib()
    # [M_b bits, padded to 256 B][24 B per x point][24 B per y point]
    assert L.ptk_chamfer_bwd_det_workspace_bytes(2, 100, 50) == 256 + 4864 + 2400
    assert L.ptk_sample_bwd_det_workspace_bytes(2, 10) == 256 + 480
    assert L.ptk_sample_normals_bwd_det_workspace_bytes(2, 10) == 256 + 480
    assert L.ptk_sample_normals_bwd_det_workspace_bytes(65, 3000) == 512 + 65 * 3000 * 24
    # the default workspace of the fused backward, then the two above (each padded to 256 B)
    assert L.ptk_mesh_chamfer_bwd_det_workspace_bytes(2, 10, 4, 100, 50) == \
        L.ptk_mesh_chamfer_workspace_bytes(2, 10, 4, 100, 50) + 256 + 4864 + 2560 + 768
    for shape in ((0, 10, 10), (1, 0, 10), (1, 10, 0), (-1, 10, 10)):
        assert L.ptk_chamfer_bwd_det_workspace_bytes(*shape) == 0
    assert L.ptk_sample_bwd_det_workspace_bytes(0, 10) == 0 and L.ptk_sample_bwd_det_workspace_bytes(3, 0) == 0
    assert L.ptk_sample_normals_bwd_det_workspace_bytes(0, 10) == 0
    assert L.ptk_sample_normals_bwd_det_workspace_bytes(3, 0) == 0
    for shape in ((0, 10, 4, 100, 50), (2, 0, 4, 100, 50), (2, 10, 0, 100, 50), (2, 10, 4, 0, 50), (2, 10, 4, 100, 0)):
        assert L.ptk_mesh_chamfer_bwd_det_workspace_bytes(*shape) == 0


def test_default_workspace_sizes_unchanged():
    L = _lib.lib()
    assert L.ptk_mesh_chamfer_workspace_bytes(2, 10, 4, 100, 50) == \
        sum((n + 255) // 256 * 256 for n in (L.ptk_sample_workspace_bytes(2, 4), L.ptk_chamfer_workspace_bytes(2, 100, 50),
                                             8, 8, 2 * 100 * 12, 2 * 10 * 12, 2 * 50 * 12))
