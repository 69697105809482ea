"""K-NN (ptk_knn_*, ops.knn, the shim's knn_points with K > 1) on the GPU: the forward against orc_knn bit for bit,
column 0 against ops.knn1 under every scan, ragged batches with hostile padding, the gradient against torch
restatements in both modes, determinism, CUDA-graph replay, no host synchronisation and the shim's outputs."""
import ctypes as C
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from oracle import knn_oracle
from ptk_b200 import _lib

pytestmark = pytest.mark.gpu
TOL = 1e-5
KS = [1, 2, 3, 8, 16, 31, 32, 33, 63, 64]


@pytest.fixture
def det(monkeypatch):
    """torch's determinism flag on for one test; the flag and fill_uninitialized_memory are restored afterwards."""
    was_on, was_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    was_fill = torch.utils.deterministic.fill_uninitialized_memory
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was_on, warn_only=was_warn)
        torch.utils.deterministic.fill_uninitialized_memory = was_fill


@pytest.fixture
def shim(monkeypatch):
    """The pytorch3d shim on sys.path for one test; its modules are dropped afterwards."""
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


@pytest.fixture(params=["filter", "exact", "pruned"])
def algo(request):
    ptk_b200.ops.set_chamfer_algo(request.param)
    yield request.param
    ptk_b200.ops.set_chamfer_algo("auto")


# ------------------------------------------------------------------------------------- helpers
def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def cpu(t):
    return t.detach().cpu().numpy()


def rel_err(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)) if a.size else 0.0


def cloud_pair(kind, B, P1, P2, seed):
    rng = np.random.default_rng(seed)
    if kind == "ties":  # a quantised grid: many exact ties
        p1 = rng.integers(-4, 5, (B, P1, 3)).astype(np.float32) * np.float32(0.125)
        p2 = rng.integers(-4, 5, (B, P2, 3)).astype(np.float32) * np.float32(0.125)
    elif kind == "dup4":  # the touch form: every target four times
        p1 = rng.random((B, P1, 3), np.float32)
        p2 = np.tile(rng.random((B, (P2 + 3) // 4, 3), np.float32), (1, 4, 1))[:, :P2].copy()
    elif kind == "tiny":
        p1 = rng.random((B, P1, 3), np.float32) * np.float32(1e-20)
        p2 = rng.random((B, P2, 3), np.float32) * np.float32(1e-20)
    elif kind == "large":
        p1 = rng.random((B, P1, 3), np.float32)
        p2 = rng.random((B, P2, 3), np.float32)
        p2[:, 0] = 1e4
        p1[:, -1] = -1e4
    elif kind == "nonfinite":
        p1 = rng.standard_normal((B, P1, 3)).astype(np.float32)
        p2 = rng.standard_normal((B, P2, 3)).astype(np.float32)
        p2[:, 1] = np.nan
        p2[:, 2, 0] = np.inf
        p2[:, 4, 1] = -np.inf
        p1[:, 0, 2] = np.nan
        p1[:, 3] = np.inf
        p2[0, P2 // 3:] = np.nan  # a cloud with few finite targets: unfilled slots stay (+inf, 0)
    else:
        p1 = rng.random((B, P1, 3), np.float32)
        p2 = rng.random((B, P2, 3), np.float32)
    return p1, p2


def knn_abi(p1, p2, K, l1=None, l2=None):
    """ptk_knn_fwd_lengths itself (any K, including 1)."""
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    L = _lib.lib()
    d = torch.empty(B, P1, K, dtype=torch.float32, device="cuda")
    i = torch.empty(B, P1, K, dtype=torch.int32, device="cuda")
    ws = torch.empty(max(L.ptk_knn_workspace_bytes(B, P1, P2, K), 16), dtype=torch.uint8, device="cuda")
    _lib.check(L.ptk_knn_fwd_lengths(_p(p1), _p(p2), _p(l1), _p(l2), B, P1, P2, K, _p(d), _p(i), _p(ws), ws.numel(),
                                     _stream()), "ptk_knn_fwd_lengths")
    return d, i


def assert_same(d, i, want_d, want_i):
    d, i = cpu(d), cpu(i)
    assert np.array_equal(d.view(np.uint32), want_d.view(np.uint32))  # bits: NaN never enters, -0 cannot occur
    assert np.array_equal(i, want_i)


# ------------------------------------------------------------------------------------- 1. forward == orc_knn
SHAPES = {"B1_split": (1, 3000, 5003), "B64_nosplit": (64, 301, 777), "P2_below_K": (3, 70, 20)}


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind", ["uniform", "ties", "dup4", "tiny", "large", "nonfinite"])
def test_forward_equals_the_oracle(K, shape, kind):
    B, P1, P2 = SHAPES[shape]
    p1, p2 = cloud_pair(kind, B, P1, P2, K)
    want_d, want_i = knn_oracle.knn(p1, p2, K, use_fma=True)
    d, i = knn_abi(torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda(), K)
    torch.cuda.synchronize()
    assert_same(d, i, want_d, want_i)
    if K > 1:
        d2, i2 = ptk_b200.ops.knn(torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda(), K)
        assert d2.shape == (B, P1, K) and i2.dtype == torch.int32
        assert_same(d2, i2, want_d, want_i)


def test_split_plan_engages_for_one_pair_and_not_for_a_batch():
    L = _lib.lib()
    assert L.ptk_knn_workspace_bytes(*SHAPES["B1_split"], 8) > 0
    assert L.ptk_knn_workspace_bytes(*SHAPES["B64_nosplit"], 8) == 0


# ------------------------------------------------------------------------------------- 2. column 0 == knn1
@pytest.mark.parametrize("K", [2, 8, 64])
@pytest.mark.parametrize("kind", ["uniform", "ties", "dup4", "nonfinite"])
def test_column_zero_is_knn1(algo, K, kind):
    for B, P1, P2 in ((2, 2500, 2200), (1, 21000, 20500)):
        p1, p2 = cloud_pair(kind, B, P1, P2, 5)
        x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
        d1, i1 = ptk_b200.ops.knn1(x, y)
        d, i = knn_abi(x, y, K)
        assert torch.equal(i[..., 0], i1)
        assert np.array_equal(cpu(d[..., 0]), cpu(d1), equal_nan=True)


# ------------------------------------------------------------------------------------- 3. ragged batches
def _sliced_reference(x, y, l1, l2, K):
    """Each pair as a homogeneous call on the sliced pair, with PyTorch3D's zero fill."""
    B, P1, _ = x.shape
    want_d = torch.zeros(B, P1, K, device="cuda")
    want_i = torch.zeros(B, P1, K, dtype=torch.int32, device="cuda")
    for b in range(B):
        n1, n2 = int(min(max(l1[b], 0), P1)), int(min(max(l2[b], 0), y.shape[1]))
        if n1 == 0 or n2 == 0:
            continue
        d, i = knn_abi(x[b:b + 1, :n1].contiguous(), y[b:b + 1, :n2].contiguous(), K)
        want_d[b, :n1, :min(K, n2)] = d[0, :, :min(K, n2)]
        want_i[b, :n1, :min(K, n2)] = i[0, :, :min(K, n2)]
        assert not d[0, :, n2:].any() and not i[0, :, n2:].any()
    return want_d, want_i


@pytest.mark.parametrize("K", [2, 8, 33, 64])
@pytest.mark.parametrize("pad", ["nan", "big"])
def test_ragged_pairs_equal_their_slices(K, pad):
    B, P1, P2 = 6, 1700, 2300
    p1, p2 = cloud_pair("ties", B, P1, P2, 9)
    l1 = np.array([1700, 0, 900, 1, 1650, 1200])
    l2 = np.array([2300, 700, 0, 5, K - 1, 2299])
    for b in range(B):
        p1[b, l1[b]:] = np.nan if pad == "nan" else 1e30
        p2[b, l2[b]:] = np.nan if pad == "nan" else p1[b, 0] if b % 2 else 1e30  # padding that would win
    x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
    tl1, tl2 = torch.from_numpy(l1).cuda(), torch.from_numpy(l2).cuda()
    d, i = ptk_b200.ops.knn(x, y, K, tl1, tl2)
    want_d, want_i = _sliced_reference(x, y, l1, l2, K)
    assert torch.equal(i, want_i)
    assert np.array_equal(cpu(d), cpu(want_d), equal_nan=True)
    assert not d[1].any() and not d[2].any() and not i[2].any()  # l1 = 0, l2 = 0
    assert not d[4, :, K - 1:].any()  # slots k >= l2


@pytest.mark.parametrize("K", [4, 32])
def test_a_pair_alone_equals_the_pair_in_a_batch_of_256(K):
    B, P1, P2 = 256, 1100, 2100  # the batch fills the GPU unsplit; one pair splits its targets
    p1, p2 = cloud_pair("ties", B, P1, P2, 11)
    x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
    d, i = knn_abi(x, y, K)
    for b in (0, 77, 255):
        da, ia = knn_abi(x[b:b + 1].contiguous(), y[b:b + 1].contiguous(), K)  # splits engage alone
        assert torch.equal(ia[0], i[b]) and torch.equal(da[0], d[b])
    assert _lib.lib().ptk_knn_workspace_bytes(1, P1, P2, K) > 0 and _lib.lib().ptk_knn_workspace_bytes(B, P1, P2, K) == 0


# ------------------------------------------------------------------------------------- 4. backward
def _terms(x, y, idx, g, l1, l2):
    """(B,P1,K,3) terms 2 g (p1_i - p2_j) with knn_term's fp32 operations, and the slot mask."""
    B, P1, K = idx.shape
    P2 = y.shape[1]
    l1 = torch.full((B,), P1, device="cuda") if l1 is None else l1.clamp(0, P1)
    l2 = torch.full((B,), P2, device="cuda") if l2 is None else l2.clamp(0, P2)
    valid = (torch.arange(P1, device="cuda")[None, :, None] < l1[:, None, None]) & \
            (torch.arange(K, device="cuda")[None, None, :] < l2[:, None, None])
    yj = torch.gather(y, 1, idx.long().reshape(B, -1, 1).expand(-1, -1, 3)).reshape(B, P1, K, 3)
    s = 2.0 * torch.where(valid, g, torch.zeros_like(g))
    t = s[..., None] * (x[:, :, None, :] - yj)
    return torch.where(valid[..., None], t, torch.zeros_like(t)), valid


def _grad_p1_slot_order(t, valid):
    acc = torch.where(valid[:, :, 0, None], t[:, :, 0], torch.zeros_like(t[:, :, 0]))
    for k in range(1, t.shape[2]):
        acc = torch.where(valid[:, :, k, None], acc + t[:, :, k], acc)
    return acc


def _grad_p2_fp64(t, idx, P2):
    B = t.shape[0]
    out = torch.zeros(B, P2, 3, dtype=torch.float64, device="cuda")
    out.scatter_add_(1, idx.long().reshape(B, -1, 1).expand(-1, -1, 3), -t.double().reshape(B, -1, 3))
    return out


def _run_grad(x, y, K, l1=None, l2=None, g=None):
    xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    d, i = ptk_b200.ops.knn(xr, yr, K, l1, l2)
    if g is None:
        g = torch.rand_like(d) - 0.5
    d.backward(g)
    return xr.grad, yr.grad, i, g


@pytest.mark.parametrize("flag", [False, True])
@pytest.mark.parametrize("K", [2, 8, 31, 64])
@pytest.mark.parametrize("ragged", [False, True])
def test_grad_matches_the_torch_restatements(flag, K, ragged):
    B, P1, P2 = 5, 1300, 900
    p1, p2 = cloud_pair("uniform", B, P1, P2, K)
    x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
    l1 = torch.tensor([1300, 0, 500, 1299, 7], device="cuda") if ragged else None
    l2 = torch.tensor([900, 300, 0, K - 1, 2], device="cuda") if ragged else None
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    try:
        gx, gy, i, g = _run_grad(x, y, K, l1, l2)
    finally:
        torch.use_deterministic_algorithms(was)
    t, valid = _terms(x, y, i, g, l1, l2)
    assert torch.equal(gx, _grad_p1_slot_order(t, valid))
    assert rel_err(cpu(gy).astype(np.float64), cpu(_grad_p2_fp64(t, i, P2))) < TOL
    if ragged:
        for b in range(B):
            n1, n2 = int(l1[b]), int(l2[b])
            assert not gx[b, n1:].any() and not gy[b, n2:].any()
            assert not torch.signbit(gx[b, n1:]).any() and not torch.signbit(gy[b, n2:]).any()  # +0


def test_det_grad_p2_is_reproducible_alone_batched_and_permuted(det):
    K, B, P1, P2 = 8, 16, 1200, 1500
    p1, p2 = cloud_pair("uniform", B, P1, P2, 21)
    x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
    g = torch.rand(B, P1, K, device="cuda") - 0.5
    gx, gy, _, _ = _run_grad(x, y, K, g=g)
    gx2, gy2, _, _ = _run_grad(x, y, K, g=g)
    assert torch.equal(gx, gx2) and torch.equal(gy, gy2)
    for b in (0, 9):
        ax, ay, _, _ = _run_grad(x[b:b + 1].contiguous(), y[b:b + 1].contiguous(), K, g=g[b:b + 1].contiguous())
        assert torch.equal(ax[0], gx[b]) and torch.equal(ay[0], gy[b])
    perm = torch.randperm(P1, device="cuda")
    _, py, _, _ = _run_grad(x[:, perm].contiguous(), y, K, g=g[:, perm].contiguous())
    assert torch.equal(py, gy)


@pytest.mark.parametrize("flag", [False, True])
def test_nan_in_never_read_upstream_gradient_does_not_leak(flag):
    K, B, P1, P2 = 8, 3, 400, 300
    p1, p2 = cloud_pair("uniform", B, P1, P2, 3)
    x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
    l1 = torch.tensor([400, 100, 0], device="cuda")
    l2 = torch.tensor([5, 300, 300], device="cuda")
    g = torch.rand(B, P1, K, device="cuda")
    g[0, :, 5:] = float("nan")  # slots k >= l2
    g[1, 100:] = float("nan")  # padded queries
    g[2] = float("nan")  # l1 = 0
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    try:
        gx, gy, _, _ = _run_grad(x, y, K, l1, l2, g=g)
    finally:
        torch.use_deterministic_algorithms(was)
    assert torch.isfinite(gx).all() and torch.isfinite(gy).all()
    assert not gx[1, 100:].any() and not gx[2].any() and not gy[0, 5:].any()


def test_grad_through_dists_and_return_nn_matches_torch_autograd(shim):
    from pytorch3d.ops import knn_gather, knn_points
    K, B, P1, P2 = 6, 4, 800, 700
    p1, p2 = cloud_pair("uniform", B, P1, P2, 8)
    l2 = torch.tensor([700, 3, 650, 100], device="cuda")
    w = torch.rand(B, P1, K, device="cuda")
    v = torch.rand(B, P1, K, 3, device="cuda")
    xr, yr = torch.from_numpy(p1).cuda().requires_grad_(True), torch.from_numpy(p2).cuda().requires_grad_(True)
    k = knn_points(xr, yr, lengths2=l2, K=K, return_nn=True)
    ((k.dists * w).sum() + (k.knn * v).sum()).backward()
    xe, ye = xr.detach().double().requires_grad_(True), yr.detach().double().requires_grad_(True)
    nn = knn_gather(ye, k.idx, l2)
    valid = (torch.arange(K, device="cuda")[None, None] < l2[:, None, None])[..., None]
    de = (((xe[:, :, None] - nn) ** 2) * valid).sum(-1)
    ((de * w).sum() + (nn * v).sum()).backward()
    assert rel_err(cpu(xr.grad), cpu(xe.grad)) < TOL and rel_err(cpu(yr.grad), cpu(ye.grad)) < TOL


# ------------------------------------------------------------------------------------- 5. CUDA graph, sync
@pytest.mark.parametrize("flag", [False, True])
def test_cuda_graph_replay_with_lengths_changed_in_place(shim, flag):
    from pytorch3d.ops import knn_points
    K, B, P1, P2 = 8, 8, 1500, 1300
    p1, p2 = cloud_pair("uniform", B, P1, P2, 16)
    x, y = torch.from_numpy(p1).cuda().requires_grad_(True), torch.from_numpy(p2).cuda().requires_grad_(True)
    l1 = torch.full((B,), P1, dtype=torch.int64, device="cuda")
    l2 = torch.full((B,), P2, dtype=torch.int64, device="cuda")
    w = torch.rand(B, P1, K, device="cuda")

    def loss_fn(x, y, l1, l2):
        return (knn_points(x, y, lengths1=l1, lengths2=l2, K=K).dists * w).sum()

    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                loss_fn(x, y, l1, l2).backward()
        torch.cuda.current_stream().wait_stream(s)
        x.grad = y.grad = None
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss = loss_fn(x, y, l1, l2)
            loss.backward()
        rng = np.random.default_rng(17)
        for rep in range(4):
            n1, n2 = rng.integers(-10, P1 + 10, B), rng.integers(-10, P2 + 10, B)
            n1[rep % B] = 0
            n2[(rep + 3) % B] = 3
            l1.copy_(torch.from_numpy(n1))
            l2.copy_(torch.from_numpy(n2))
            graph.replay()
            torch.cuda.synchronize()
            xe, ye = x.detach().clone().requires_grad_(True), y.detach().clone().requires_grad_(True)
            le = loss_fn(xe, ye, l1.clone(), l2.clone())
            gxe, gye = torch.autograd.grad(le, (xe, ye))
            if flag:
                assert torch.equal(loss, le) and torch.equal(x.grad, gxe) and torch.equal(y.grad, gye)
            else:
                assert rel_err(cpu(loss), cpu(le)) < TOL
                assert torch.equal(x.grad, gxe) and rel_err(cpu(y.grad), cpu(gye)) < TOL
    finally:
        torch.use_deterministic_algorithms(was)


@pytest.mark.parametrize("flag", [False, True])
def test_forward_and_backward_run_without_host_sync(shim, flag):
    from pytorch3d.ops import knn_points
    K, B, P1, P2 = 8, 5, 700, 600
    p1, p2 = cloud_pair("uniform", B, P1, P2, 18)
    l1 = torch.tensor([700, 1, 0, 350, 699], device="cuda")
    l2 = torch.tensor([600, 600, 20, 0, 1], device="cuda")
    xr, yr = torch.from_numpy(p1).cuda().requires_grad_(True), torch.from_numpy(p2).cuda().requires_grad_(True)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        k = knn_points(xr, yr, lengths1=l1, lengths2=l2, K=K, return_nn=True)
        (k.dists.sum() + (k.knn * xr[:, :, None]).sum()).backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
        torch.use_deterministic_algorithms(was)
    assert xr.grad is not None and yr.grad is not None


# ------------------------------------------------------------------------------------- 6. shim outputs
@pytest.mark.parametrize("return_nn", [False, True])
@pytest.mark.parametrize("return_sorted", [True, False])
def test_shim_outputs_have_pytorch3d_shapes_and_dtypes(shim, return_nn, return_sorted):
    from pytorch3d.ops import knn_points
    K, B, P1, P2 = 5, 3, 200, 4  # K > P2
    p1, p2 = cloud_pair("uniform", B, P1, P2, 2)
    x, y = torch.from_numpy(p1).cuda(), torch.from_numpy(p2).cuda()
    k = knn_points(x, y, K=K, return_nn=return_nn, return_sorted=return_sorted, version=2)
    assert k._fields == ("dists", "idx", "knn")
    assert k.dists.shape == (B, P1, K) and k.dists.dtype == torch.float32
    assert k.idx.shape == (B, P1, K) and k.idx.dtype == torch.int64
    if return_nn:
        assert k.knn.shape == (B, P1, K, 3) and k.knn.dtype == torch.float32
        assert not k.knn[:, :, P2:].any()
    else:
        assert k.knn is None
    want_d, want_i = knn_oracle.knn(p1, p2, K)
    assert np.array_equal(cpu(k.dists), want_d) and np.array_equal(cpu(k.idx), want_i.astype(np.int64))
    k1 = knn_points(x, y, K=1)
    assert torch.equal(k1.dists, k.dists[..., :1]) and torch.equal(k1.idx, k.idx[..., :1])
