"""Differentiable 1-NN (ops.knn1 / the shim's knn_points and knn_gather): the gradient against torch and numpy
restatements under every scan, ragged batches with hostile padding, the Chamfer identity, the deterministic form,
CUDA-graph replay, no host synchronisation, and the unchanged no-grad path."""
import ctypes as C
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from ptk_b200 import _lib

pytestmark = pytest.mark.gpu
TOL = 1e-5


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
    return t.detach().cpu().numpy() if t is not None else None


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.size == 0:
        return 0.0
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def is_plus_zero(a):
    a = np.asarray(a)
    return not a.any() and not np.signbit(a).any()


def clip_len(lengths, b, P):
    return P if lengths is None else int(np.clip(int(lengths[b]), 0, P))


def clouds(B, P1, P2, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((B, P1, 3), np.float32)
    y = (rng.random((B, P2, 3), np.float32) * 0.9 + 0.05).astype(np.float32)
    return torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()


def upstream(B, P1, l1, l2, seed):
    """g (B,P1): normal values with zeros and negatives, NaN wherever the kernels must not read it (padded queries and
    the queries of a pair whose target cloud is empty)."""
    rng = np.random.default_rng(seed)
    g = rng.standard_normal((B, P1)).astype(np.float32)
    g[:, ::7] = 0.0
    for b in range(B):
        L1 = clip_len(l1, b, P1)
        g[b, L1:] = np.nan
        if clip_len(l2, b, 10 ** 9) == 0:
            g[b] = np.nan
    return torch.from_numpy(g).cuda()


def torch_terms(p1, p2, idx, g):
    """The torch restatement of every query's term: (2 g)[..., None] * (p1 - p2[b, idx])."""
    nn = torch.gather(p2, 1, idx.long()[..., None].expand(-1, -1, 3))
    return (2 * g)[..., None] * (p1 - nn)


def check_grads(p1, p2, l1, l2, idx, g, g1, g2):
    """grad_p1 bit-identical to the torch restatement at valid rows, grad_p2 within TOL of the fp64 index_add of the same
    fp32 terms; every other row +0."""
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    t = cpu(torch_terms(p1.detach(), p2.detach(), idx, g))
    ix = cpu(idx).astype(np.int64)
    for b in range(B):
        L1, L2 = clip_len(l1, b, P1), clip_len(l2, b, P2)
        nv = L1 if L2 > 0 else 0
        if g1 is not None:
            assert same_bits(g1[b, :nv], t[b, :nv]), b
            assert is_plus_zero(g1[b, nv:]), b
        if g2 is not None:
            want = np.zeros((P2, 3), np.float64)
            np.add.at(want, ix[b, :nv], -t[b, :nv].astype(np.float64))
            assert rel_err(g2[b, :L2], want[:L2]) < TOL, b
            assert is_plus_zero(g2[b, L2:]) and not want[L2:].any(), b


def knn1_grads(x, y, l1, l2, g, want1=True, want2=True):
    xr = x.detach().clone().requires_grad_(want1)
    yr = y.detach().clone().requires_grad_(want2)
    d, i = ptk_b200.ops.knn1(xr, yr, l1, l2)
    torch.autograd.backward(d, g)
    return d, i, cpu(xr.grad), cpu(yr.grad)


def fill_padding(x, y, l1, l2, kind):
    x, y = x.clone(), y.clone()
    val = {"nan": float("nan"), "inf": float("inf"), "-inf": float("-inf"), "big": 1e30}[kind]
    for b in range(x.shape[0]):
        x[b, clip_len(l1, b, x.shape[1]):] = val
        y[b, clip_len(l2, b, y.shape[1]):] = val
    return x, y


# lengths: 0 and 1 on either side, full, mid-chunk, outside [0, P] (clamped)
B8, P1_, P2_ = 8, 3000, 2500
L1_ = [3000, 0, 100, 1, 3000, 1777, -3, 5000]
L2_ = [2500, 100, 0, 2500, 1, 1033, 40, 2499]


# ------------------------------------------------------------------------------------- 1. against the restatement
@pytest.mark.parametrize("ragged", [False, True])
def test_grad_matches_the_torch_restatement(algo, ragged):
    x, y = clouds(B8, P1_, P2_, 1)
    y[0, :40] = y[0, 0] + 1e-4 * torch.arange(40, device="cuda", dtype=torch.float32)[:, None]  # a shared neighbour
    l1 = torch.tensor(L1_, device="cuda") if ragged else None
    l2 = torch.tensor(L2_, device="cuda") if ragged else None
    g = upstream(B8, P1_, l1, l2, 2)
    for want1, want2 in ((True, True), (True, False), (False, True)):
        _, idx, g1, g2 = knn1_grads(x, y, l1, l2, g, want1, want2)
        check_grads(x, y, l1, l2, idx, g, g1, g2)
        assert (g1 is None) != want1 and (g2 is None) != want2


def test_knn1_of_a_cloud_with_itself_has_zero_gradient(algo):
    x, _ = clouds(2, 2000, 1, 3)
    x[:, 1000:1010] = x[:, 500:510]  # duplicates: the lower index wins, the difference is still 0
    xr = x.clone().requires_grad_(True)
    d, i = ptk_b200.ops.knn1(xr, xr)
    torch.autograd.backward(d, torch.rand_like(d) - 0.5)
    assert not d.any() and not xr.grad.any()


# ------------------------------------------------------------------------------------- 2. ragged against sliced
@pytest.mark.parametrize("kind", ["nan", "inf", "-inf", "big"])
def test_ragged_gradient_equals_the_sliced_pair(kind):
    l1, l2 = torch.tensor(L1_, device="cuda"), torch.tensor(L2_, device="cuda")
    x, y = fill_padding(*clouds(B8, P1_, P2_, 4), L1_, L2_, kind)
    g = upstream(B8, P1_, L1_, L2_, 5)
    _, idx, g1, g2 = knn1_grads(x, y, l1, l2, g)
    check_grads(x, y, l1, l2, idx, g, g1, g2)
    for b in range(B8):
        L1, L2 = clip_len(L1_, b, P1_), clip_len(L2_, b, P2_)
        if L1 == 0 or L2 == 0:
            assert is_plus_zero(g1[b]) and is_plus_zero(g2[b])
            continue
        _, _, s1, s2 = knn1_grads(x[b:b + 1, :L1].contiguous(), y[b:b + 1, :L2].contiguous(), None, None,
                                  g[b:b + 1, :L1].contiguous())
        assert same_bits(g1[b:b + 1, :L1], s1), b
        assert rel_err(g2[b:b + 1, :L2], s2) < TOL, b


# ------------------------------------------------------------------------------------- 3. the Chamfer identity
@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("ragged", [False, True])
def test_two_knn1_terms_give_the_chamfer_gradient(reduction, ragged):
    B, P1, P2 = 5, 2000, 1700
    x, y = clouds(B, P1, P2, 6)
    lx = torch.tensor([2000, 1, 0, 1234, 999], device="cuda") if ragged else None
    ly = torch.tensor([1700, 1700, 50, 1, 1200], device="cuda") if ragged else None
    w = torch.tensor([1.0, -0.5, 2.0, 0.25, 3.0], device="cuda")
    xa, ya = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    cham, _, _ = ptk_b200.ops.chamfer(xa, ya, lx, ly, point_reduction=reduction)
    (cham * w).sum().backward()
    xb, yb = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    dx, _ = ptk_b200.ops.knn1(xb, yb, lx, ly)
    dy, _ = ptk_b200.ops.knn1(yb, xb, ly, lx)
    sx, sy = dx.sum(1), dy.sum(1)
    if reduction == "mean":
        nx = (lx.clamp(0, P1) if ragged else torch.full((B,), P1, device="cuda")).clamp(min=1)
        ny = (ly.clamp(0, P2) if ragged else torch.full((B,), P2, device="cuda")).clamp(min=1)
        sx, sy = sx / nx, sy / ny
    ((sx + sy) * w).sum().backward()
    assert rel_err(cpu(xb.grad), cpu(xa.grad)) < TOL and rel_err(cpu(yb.grad), cpu(ya.grad)) < TOL


# ------------------------------------------------------------------------------------- 4. deterministic form
def _ceil_log2_f32(m):
    mant, ex = np.frexp(np.float64(m))
    return int(ex) - 1 if mant == 0.5 else int(ex)


def _ceil_log2_int(n):
    c = 0
    while (1 << c) < n:
        c += 1
    return c


def det_knn1_grad_p2(p1, p2, l1, l2, idx, g):
    """ptk_knn1_bwd_det's grad_p2 restated: e_b from the pair's largest finite |term| and l1 + 1, int64 sums of
    round_half_even(term * 2^e_b), an int64 -> float32 cast and ldexp; non-finite terms summed outside."""
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    out = np.zeros((B, P2, 3), np.float32)
    for b in range(B):
        L1, L2 = clip_len(l1, b, P1), clip_len(l2, b, P2)
        if L1 == 0 or L2 == 0:
            continue
        j = idx[b, :L1].astype(np.int64)
        with np.errstate(all="ignore"):
            t = ((np.float32(2) * g[b, :L1])[:, None] * (p1[b, :L1] - p2[b, j])).astype(np.float32)
        a = np.abs(t[np.isfinite(t)])
        M = np.float32(a.max()) if a.size else np.float32(0)
        e = 0 if M == 0 else 62 - _ceil_log2_f32(M) - _ceil_log2_int(L1 + 1)
        fin = np.isfinite(t)
        q = np.where(fin, np.rint(np.where(fin, t, 0).astype(np.float64) * 2.0 ** e), 0).astype(np.int64)
        acc, nf = np.zeros((P2, 3), np.int64), np.zeros((P2, 3), np.float32)
        np.add.at(acc, j, -q)
        with np.errstate(all="ignore"):
            np.add.at(nf, j, np.where(fin, 0, -t))
        conv = np.ldexp(acc.astype(np.float32), np.int32(-e))
        out[b] = np.where(np.isfinite(nf), conv, nf).astype(np.float32)
    return out


def knn1_bwd_det_abi(p1, p2, idx, g, l1=None, l2=None, want1=True, want2=True):
    L = _lib.lib()
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    g1 = torch.empty_like(p1) if want1 else None
    g2 = torch.empty_like(p2) if want2 else None
    ws = torch.empty(max(L.ptk_knn1_bwd_det_workspace_bytes(B, P1, P2), 16), dtype=torch.uint8, device=p1.device)
    _lib.check(L.ptk_knn1_bwd_det(_p(p1), _p(p2), _p(l1), _p(l2), _p(idx), _p(g), B, P1, P2, _p(g1), _p(g2), _p(ws),
                                  ws.numel(), _stream()), "ptk_knn1_bwd_det")
    return cpu(g1), cpu(g2)


@pytest.mark.parametrize("ragged", [False, True])
def test_det_matches_the_default_p1_and_the_restatement_p2(det, algo, ragged):
    x, y = clouds(B8, P1_, P2_, 7)
    y[2, :50] = y[2, 0] + 1e-4 * torch.arange(50, device="cuda", dtype=torch.float32)[:, None]
    l1 = torch.tensor(L1_, device="cuda") if ragged else None
    l2 = torch.tensor(L2_, device="cuda") if ragged else None
    g = upstream(B8, P1_, l1, l2, 8)
    torch.use_deterministic_algorithms(False)
    _, idx, d1, _ = knn1_grads(x, y, l1, l2, g)
    torch.use_deterministic_algorithms(True)
    want2 = det_knn1_grad_p2(cpu(x), cpu(y), cpu(l1), cpu(l2), cpu(idx), cpu(g))
    for w1, w2 in ((True, True), (True, False), (False, True)):
        _, _, g1, g2 = knn1_grads(x, y, l1, l2, g, w1, w2)
        if w1:
            assert same_bits(g1, d1)
        if w2:
            assert same_bits(g2, want2)


def test_det_permuted_queries(det):
    B, P1, P2 = 2, 5000, 4000
    x, y = clouds(B, P1, P2, 9)
    g = torch.randn(B, P1, device="cuda")
    perm = torch.from_numpy(np.random.default_rng(10).permutation(P1)).cuda()
    _, _, a1, a2 = knn1_grads(x, y, None, None, g)
    _, _, b1, b2 = knn1_grads(x[:, perm].contiguous(), y, None, None, g[:, perm].contiguous())
    assert same_bits(b1, np.ascontiguousarray(a1[:, cpu(perm)])) and same_bits(b2, a2)


def test_det_pair_alone_equals_the_pair_in_a_batch_of_64(det):
    B, P1, P2, k = 64, 2000, 1500, 17
    x, y = clouds(B, P1, P2, 11)
    g = torch.randn(B, P1, device="cuda")
    _, idx = ptk_b200.ops.knn1(x, y)
    a1, a2 = knn1_bwd_det_abi(x, y, idx, g)
    s = slice(k, k + 1)
    b1, b2 = knn1_bwd_det_abi(x[s].contiguous(), y[s].contiguous(), idx[s].contiguous(), g[s].contiguous())
    assert same_bits(a1[s], b1) and same_bits(a2[s], b2)


def test_det_ragged_pair_equals_its_slice(det):
    l1, l2 = torch.tensor(L1_, device="cuda"), torch.tensor(L2_, device="cuda")
    x, y = fill_padding(*clouds(B8, P1_, P2_, 12), L1_, L2_, "nan")
    g = upstream(B8, P1_, L1_, L2_, 13)
    _, idx = ptk_b200.ops.knn1(x, y, l1, l2)
    a1, a2 = knn1_bwd_det_abi(x, y, idx, g, l1, l2)
    for b in range(B8):
        L1, L2 = clip_len(L1_, b, P1_), clip_len(L2_, b, P2_)
        if L1 == 0 or L2 == 0:
            assert is_plus_zero(a1[b]) and is_plus_zero(a2[b])
            continue
        b1, b2 = knn1_bwd_det_abi(x[b:b + 1, :L1].contiguous(), y[b:b + 1, :L2].contiguous(),
                                  idx[b:b + 1, :L1].contiguous(), g[b:b + 1, :L1].contiguous())
        assert same_bits(a1[b:b + 1, :L1], b1) and same_bits(a2[b:b + 1, :L2], b2), b
        assert is_plus_zero(a1[b, L1:]) and is_plus_zero(a2[b, L2:]), b


def test_det_two_calls_at_full_size(det):
    B, P = 256, 10000
    gen = torch.Generator(device="cuda").manual_seed(14)
    x = torch.rand(B, P, 3, device="cuda", generator=gen)
    y = torch.rand(B, P, 3, device="cuda", generator=gen)
    g = torch.randn(B, P, device="cuda", generator=gen)
    _, idx = ptk_b200.ops.knn1(x, y)
    a, b = knn1_bwd_det_abi(x, y, idx, g), knn1_bwd_det_abi(x, y, idx, g)
    assert same_bits(a[0], b[0]) and same_bits(a[1], b[1]) and np.isfinite(a[1]).all()


def test_det_non_finite_input(det):
    B, P1, P2 = 3, 2000, 1800
    x, y = clouds(B, P1, P2, 15)
    _, idx = ptk_b200.ops.knn1(x, y)  # indices of the clean clouds; the backward then sees hostile values
    ix = cpu(idx)
    g = torch.randn(B, P1, device="cuda")
    g[1] = g[1].abs() + 0.1           # one sign per row of pair 1: its infinite terms cannot cancel to NaN
    x[0, 5, 0] = float("nan")
    x[0, 6, 1] = float("inf")
    y[1, ix[1, 3], 0] = float("inf")
    y[1, ix[1, 4], 0] = float("-inf")
    g[2, 9] = 3e38                     # s = 2 g overflows to inf
    runs = [knn1_bwd_det_abi(x, y, idx, g) for _ in range(2)]
    want = det_knn1_grad_p2(cpu(x), cpu(y), None, None, ix, cpu(g))
    for a, b in ((runs[0][0], runs[1][0]), (runs[0][1], runs[1][1]), (runs[0][1], want)):
        nan = np.isnan(a)
        assert np.array_equal(nan, np.isnan(b)) and same_bits(a[~nan], b[~nan])
    assert np.isnan(runs[0][1]).any() and np.isinf(runs[0][1]).any()


# ------------------------------------------------------------------------------------- 5. CUDA graph
@pytest.mark.parametrize("flag", [False, True])
def test_cuda_graph_replay_with_lengths_changed_in_place(shim, flag):
    from pytorch3d.ops import knn_points
    B, P1, P2 = 8, 1500, 1300
    x, y = clouds(B, P1, P2, 16)
    x.requires_grad_(True)
    y.requires_grad_(True)
    l1 = torch.full((B,), P1, dtype=torch.int64, device="cuda")
    l2 = torch.full((B,), P2, dtype=torch.int64, device="cuda")
    w = torch.rand(B, device="cuda")

    def loss_fn(x, y, l1, l2):  # a one-directional Chamfer term plus a weighted reverse term
        d1 = knn_points(x, y, lengths1=l1, lengths2=l2).dists[..., 0]
        d2 = knn_points(y, x, lengths1=l2, lengths2=l1).dists[..., 0]
        return ((d1.sum(1) / l1.clamp(0, P1).clamp(min=1) + 0.3 * d2.sum(1)) * w).sum()

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
            n2[(rep + 3) % B] = 1
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
                assert rel_err(cpu(x.grad), cpu(gxe)) < TOL and rel_err(cpu(y.grad), cpu(gye)) < TOL
    finally:
        torch.use_deterministic_algorithms(was)


# ------------------------------------------------------------------------------------- 6. no host synchronisation
def test_knn_points_return_nn_runs_without_host_sync(shim):
    from pytorch3d.ops import knn_points
    B, P1, P2 = 5, 700, 600
    x, y = clouds(B, P1, P2, 18)
    l1 = torch.tensor([700, 1, 0, 350, 699], device="cuda")
    l2 = torch.tensor([600, 600, 20, 0, 1], device="cuda")
    xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        k = knn_points(xr, yr, lengths1=l1, lengths2=l2, return_nn=True)
        loss = k.dists.sum() + (k.knn[:, :, 0] * xr).sum()
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert k.knn.shape == (B, P1, 1, 3) and k.dists.shape == (B, P1, 1)
    d, i = ptk_b200.ops.knn1(x, y, l1, l2)
    assert torch.equal(k.dists[..., 0], d) and torch.equal(k.idx[..., 0], i.long())
    want = torch.gather(y, 1, i.long()[..., None].expand(-1, -1, 3)) * (l2 > 0)[:, None, None]
    assert torch.equal(k.knn[:, :, 0], want)  # padded queries gather y[b, 0]; an empty target cloud gathers 0
    # y's gradient: the dists term plus the gathered rows' weights x[b, i]
    yg = y.clone().requires_grad_(True)
    ref = torch.gather(yg, 1, i.long()[..., None].expand(-1, -1, 3)) * (l2 > 0)[:, None, None]
    (gy,) = torch.autograd.grad((ref * x).sum(), yg)
    g = torch.ones(B, P1, device="cuda")
    _, _, _, g2 = knn1_grads(x, y, l1, l2, g, want1=False)
    assert rel_err(cpu(yr.grad), cpu(gy) + g2) < TOL


# ------------------------------------------------------------------------------------- 7. reproducible end to end
def test_loss_with_dists_and_knn_is_bit_reproducible_under_the_flag(det, shim):
    from pytorch3d.ops import knn_points
    B, P1, P2 = 16, 3000, 4000
    x, y = clouds(B, P1, P2, 19)
    l1 = torch.randint(1500, P1 + 1, (B,), device="cuda")
    l2 = torch.randint(2000, P2 + 1, (B,), device="cuda")
    grads = []
    for _ in range(2):
        xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        k = knn_points(xr, yr, lengths1=l1, lengths2=l2, return_nn=True)
        loss = k.dists.mean() + ((k.knn[:, :, 0] - xr) ** 3).sum()
        loss.backward()
        grads.append((xr.grad, yr.grad))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])
    assert torch.isfinite(grads[0][0]).all() and torch.isfinite(grads[0][1]).all()


# ------------------------------------------------------------------------------------- 8. the no-grad path
@pytest.mark.parametrize("mode", ["plain", "no_grad"])
def test_no_grad_path_launches_and_returns_what_the_forward_does(mode):
    B, P1, P2 = 4, 3000, 2000
    x, y = clouds(B, P1, P2, 20)
    l1, l2 = torch.tensor([3000, 10, 0, 2999], device="cuda"), torch.tensor([2000, 0, 5, 1999], device="cuda")
    L = _lib.lib()
    d0 = torch.empty(B, P1, device="cuda")
    i0 = torch.empty(B, P1, dtype=torch.int32, device="cuda")
    ws = torch.empty(L.ptk_chamfer_workspace_bytes(B, P1, P2), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    c0 = _lib.launch_count()
    _lib.check(L.ptk_knn1_fwd_lengths(_p(x), _p(y), _p(l1), _p(l2), B, P1, P2, _p(d0), _p(i0), _p(ws), ws.numel(),
                                      _stream()), "ptk_knn1_fwd_lengths")
    c1 = _lib.launch_count()
    if mode == "no_grad":
        xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        with torch.no_grad():
            d, i = ptk_b200.ops.knn1(xr, yr, l1, l2)
    else:
        d, i = ptk_b200.ops.knn1(x, y, l1, l2)
    c2 = _lib.launch_count()
    assert c2 - c1 == c1 - c0
    assert not d.requires_grad and not i.requires_grad and d.grad_fn is None
    assert same_bits(cpu(d), cpu(d0)) and torch.equal(i, i0)
