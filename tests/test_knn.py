"""K-NN entry points (ptk_knn_*), the orc_knn oracle and the shim's argument errors, without a GPU."""
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from oracle import knn_oracle
from oracle import oracle as orc
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


def _fwd(p1=D, p2=D, B=2, P1=100, P2=50, K=8, dist=D, idx=D, ws=D, nbytes=1 << 30):
    return _lib.lib().ptk_knn_fwd_lengths(p1, p2, None, None, B, P1, P2, K, dist, idx, ws, nbytes, None)


def _bwd(p1=D, p2=D, idx=D, g=D, B=2, P1=100, P2=50, K=8, g1=D, g2=D, ws=D, nbytes=1 << 30):
    return _lib.lib().ptk_knn_bwd_lengths(p1, p2, None, None, idx, g, B, P1, P2, K, g1, g2, None)


def _det(p1=D, p2=D, idx=D, g=D, B=2, P1=100, P2=50, K=8, g1=D, g2=D, ws=D, nbytes=1 << 30):
    return _lib.lib().ptk_knn_bwd_det(p1, p2, None, None, idx, g, B, P1, P2, K, g1, g2, ws, nbytes, None)


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("null", ["p1", "p2"])
def test_knn_rejects_null_clouds(call, null):
    assert call(**{null: None}) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()


@pytest.mark.parametrize("null", ["dist", "idx"])
def test_knn_fwd_rejects_null_outputs(null):
    assert _fwd(**{null: None}) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()


@pytest.mark.parametrize("call", [_bwd, _det])
@pytest.mark.parametrize("null", ["idx", "g"])
def test_knn_bwd_rejects_null_index_or_grad(call, null):
    assert call(**{null: None}) == _lib.PTK_ERR_SHAPE and "null" in _lib.last_error()


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("shape", [(0, 10, 10), (1, 0, 10), (1, 10, 0), (-1, 10, 10), (1, 1 << 30, 10), (70000, 10, 10),
                                   (1, 1 << 26, 10)])
def test_knn_rejects_bad_shapes(call, shape):
    B, P1, P2 = shape
    assert call(B=B, P1=P1, P2=P2, K=64, nbytes=1 << 62) == _lib.PTK_ERR_SHAPE


@pytest.mark.parametrize("call", [_fwd, _bwd, _det])
@pytest.mark.parametrize("K", [0, -1, 65, 1000])
def test_knn_rejects_k_outside_1_to_64(call, K):
    assert call(K=K) == _lib.PTK_ERR_SHAPE and "K=" in _lib.last_error()


def test_knn_fwd_rejects_missing_small_or_misaligned_workspace():
    L = _lib.lib()
    need = L.ptk_knn_workspace_bytes(1, 10000, 10000, 8)
    assert need > 0  # a single pair splits its target range
    for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
        assert _fwd(B=1, P1=10000, P2=10000, ws=ws, nbytes=nbytes) == _lib.PTK_ERR_WORKSPACE
        assert "workspace" in _lib.last_error()
    assert _fwd(B=1, P1=10000, P2=10000, ws=D + 4, nbytes=need) == _lib.PTK_ERR_ALIGN


def test_knn_bwd_det_rejects_missing_or_small_workspace():
    need = _lib.lib().ptk_knn1_bwd_det_workspace_bytes(2, 100, 50)
    for g1, g2 in ((D, D), (D, None), (None, D)):
        for ws, nbytes in ((None, need), (D, need - 1), (D, 0)):
            assert _det(g1=g1, g2=g2, ws=ws, nbytes=nbytes) == _lib.PTK_ERR_WORKSPACE and "workspace" in _lib.last_error()


def test_knn_bwd_without_requested_gradients_is_a_no_op():
    assert _bwd(g1=None, g2=None) == 0
    assert _det(g1=None, g2=None, ws=None, nbytes=0) == 0


def test_knn_workspace_pinned_values():
    L = _lib.lib()
    # [B][n_split][P1][K] (dist bits, idx) pairs when the target range is split (csrc/knn.cu knn_plan), else nothing
    assert L.ptk_knn_workspace_bytes(1, 10000, 10000, 8) == 8 * 10000 * 8 * 8  # 8 splits
    assert L.ptk_knn_workspace_bytes(1, 10000, 10000, 64) == 8 * 10000 * 64 * 8
    assert L.ptk_knn_workspace_bytes(16, 1949, 10000, 8) == 16 * 8 * 1949 * 8 * 8  # 128 query blocks: 8 splits
    assert L.ptk_knn_workspace_bytes(3, 500, 2049, 8) == 3 * 3 * 500 * 8 * 8  # 3 splits of >= 1024 targets
    assert L.ptk_knn_workspace_bytes(2, 100, 50, 8) == 0  # too few targets to split
    assert L.ptk_knn_workspace_bytes(256, 10000, 10000, 8) == 0  # enough query blocks: no split
    assert L.ptk_knn_workspace_bytes(1, 100, 1000, 8) == 0  # one split's worth of targets
    for shape in ((0, 10, 10, 2), (1, 0, 10, 2), (1, 10, 0, 2), (1, 10, 10, 0), (1, 10, 10, 65)):
        assert L.ptk_knn_workspace_bytes(*shape) == 0


# ------------------------------------------------------------------------------------- the oracle
def _numpy_knn(p1, p2, K):
    """Non-FMA float32 restatement: d = (dx*dx + dy*dy) + dz*dz, stable sort by (d, j) over finite d, (+inf, 0) for
    unfilled slots, (0, 0) for slots k >= P2."""
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    dist = np.zeros((B, P1, K), np.float32)
    idx = np.zeros((B, P1, K), np.int32)
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(B):
            diff = p1[b][:, None, :] - p2[b][None, :, :]
            d = (diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]) + diff[..., 2] * diff[..., 2]
            for i in range(P1):
                row = d[i]
                ok = np.nonzero(row < np.float32(np.inf))[0]
                order = ok[np.argsort(row[ok], kind="stable")]
                n = min(K, P2)
                dist[b, i, :n] = np.inf
                take = order[:n]
                dist[b, i, :len(take)] = row[take]
                idx[b, i, :len(take)] = take
    return dist, idx


def _tie_clouds(rng, B, P1, P2):
    g1 = rng.integers(-3, 4, (B, P1, 3)).astype(np.float32) * np.float32(0.25)
    g2 = rng.integers(-3, 4, (B, P2, 3)).astype(np.float32) * np.float32(0.25)
    return g1, g2


def _hostile(rng, B, P1, P2):
    p1 = rng.standard_normal((B, P1, 3)).astype(np.float32)
    p2 = rng.standard_normal((B, P2, 3)).astype(np.float32)
    p2[0, 3] = np.nan
    p2[0, 5, 1] = np.inf
    p2[0, 7, 2] = -np.inf
    p1[0, 2, 0] = np.nan
    p1[0, 4] = np.inf
    p2[1 % B, :P2 // 2] = np.nan
    return p1, p2


@pytest.mark.parametrize("K", [1, 2, 5, 8, 33, 70])
@pytest.mark.parametrize("kind", ["ties", "hostile"])
def test_orc_knn_without_fma_equals_numpy_restatement(K, kind):
    rng = np.random.default_rng(K)
    p1, p2 = (_tie_clouds if kind == "ties" else _hostile)(rng, 2, 40, 60)
    got_d, got_i = knn_oracle.knn(p1, p2, K, use_fma=False)
    want_d, want_i = _numpy_knn(p1, p2, K)
    assert np.array_equal(got_d, want_d, equal_nan=True)
    assert np.array_equal(got_i, want_i)


@pytest.mark.parametrize("use_fma", [True, False])
@pytest.mark.parametrize("kind", ["ties", "hostile", "uniform"])
def test_orc_knn_column_zero_is_orc_knn1(use_fma, kind):
    rng = np.random.default_rng(1)
    if kind == "uniform":
        p1, p2 = rng.random((3, 50, 3), np.float32), rng.random((3, 80, 3), np.float32)
    else:
        p1, p2 = (_tie_clouds if kind == "ties" else _hostile)(rng, 3, 50, 80)
    d, i = knn_oracle.knn(p1, p2, 7, use_fma=use_fma)
    d1, i1 = orc.knn1(p1, p2, use_fma=use_fma)
    assert np.array_equal(d[..., 0], d1, equal_nan=True)
    assert np.array_equal(i[..., 0], i1)


def test_orc_knn_pads_slots_past_the_target_cloud():
    rng = np.random.default_rng(2)
    p1, p2 = rng.random((2, 5, 3), np.float32), rng.random((2, 3, 3), np.float32)
    d, i = knn_oracle.knn(p1, p2, 6)
    assert not d[..., 3:].any() and not i[..., 3:].any()
    assert np.array_equal(np.sort(i[..., :3], axis=-1), np.broadcast_to(np.arange(3), (2, 5, 3)))


# ------------------------------------------------------------------------------------- argument errors
def test_ops_knn_rejects_k_out_of_range_and_cpu_tensors():
    x = torch.rand(1, 4, 3)
    for K in (0, -3):
        with pytest.raises(ValueError):
            ptk_b200.ops.knn(x, x, K)
    with pytest.raises(NotImplementedError):
        ptk_b200.ops.knn(x, x, 65)
    with pytest.raises(ValueError):
        ptk_b200.ops.knn(x, x, 2.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ptk_b200.ops.knn(x, x, 4)


def test_shim_knn_points_k_above_one_on_cpu_says_there_is_no_cpu_fallback(shim):
    from pytorch3d.ops import knn_points
    x = torch.rand(1, 4, 3)
    for kw in ({"K": 2}, {"K": 8, "return_nn": True}, {"K": 3, "return_sorted": False}):
        with pytest.raises(NotImplementedError, match="no CPU fallback"):
            knn_points(x, x, **kw)
    with pytest.raises(RuntimeError):  # NotImplementedError is a RuntimeError: the ops' CPU contract holds
        knn_points(x, x, K=2)


def test_shim_knn_points_rejects_bad_k(shim):
    from pytorch3d.ops import knn_points
    x = torch.rand(1, 4, 3)
    with pytest.raises(ValueError):
        knn_points(x, x, K=0)
    with pytest.raises(NotImplementedError):
        knn_points(x, x, K=65)
