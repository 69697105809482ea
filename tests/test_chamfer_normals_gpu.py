"""The Chamfer normal term on the GPU (ops.chamfer_normals, ptk_chamfer_normals_*, the shim's chamfer_distance with
normals): per-query terms and cham_normals against the fp64 restatement of PyTorch3D's term under every scan, edge
cases, pair independence, gradients against fp64 autograd in both backward forms, the deterministic form's bits, the
shim end to end and CUDA-graph replay."""
import ctypes as C
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from ptk_b200 import _lib
from oracle import torch_ref

import chamfer_normals_ref

pytestmark = pytest.mark.gpu


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
    return t.detach().cpu() if t is not None else None


def same_bits(a, b):
    a, b = cpu(a).contiguous(), cpu(b).contiguous()
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def rel_err(a, b):
    a, b = cpu(a).double(), cpu(b).double()
    if a.numel() == 0:
        return 0.0
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def is_plus_zero(t):
    t = cpu(t)
    return not t.any() and not torch.signbit(t).any()


def data(B, P1, P2, seed, unit=False):
    """Clouds and non-unit normals (norms spread over 1e-2 .. 1e2), on the GPU."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(B, P1, 3, device="cuda", generator=g)
    y = torch.rand(B, P2, 3, device="cuda", generator=g)
    xn = torch.randn(B, P1, 3, device="cuda", generator=g)
    yn = torch.randn(B, P2, 3, device="cuda", generator=g)
    if not unit:
        xn = xn * 10.0 ** (4 * torch.rand(B, P1, 1, device="cuda", generator=g) - 2)
        yn = yn * 10.0 ** (4 * torch.rand(B, P2, 1, device="cuda", generator=g) - 2)
    return x, y, xn, yn


def lengths(B, P, seed):
    """Ragged lengths with 0, 1, P and values outside [0, P] (clamped by the kernels)."""
    rng = np.random.default_rng(seed)
    n = rng.integers(1, P + 1, B)
    for k, v in enumerate([0, 1, P, P + 7, -3]):
        n[(k * 3 + seed) % B] = v
    return torch.from_numpy(n).cuda()


def abi_fwd(xn, yn, ix, iy, lx, ly, reduction=_lib.REDUCE_MEAN):
    """ptk_chamfer_normals_fwd with the per-query terms: (cham_normals, term_x, term_y)."""
    B, P1, _ = xn.shape
    P2 = yn.shape[1]
    L = _lib.lib()
    tx = torch.full((B, P1), float("nan"), device="cuda")
    ty = torch.full((B, P2), float("nan"), device="cuda")
    cn = torch.empty(B, device="cuda")
    ws = torch.empty(max(L.ptk_chamfer_normals_workspace_bytes(B, P1, P2), 16), dtype=torch.uint8, device="cuda")
    _lib.check(L.ptk_chamfer_normals_fwd(_p(xn), _p(yn), _p(lx), _p(ly), _p(ix), _p(iy), B, P1, P2, reduction, _p(tx),
                                         _p(ty), _p(cn), _p(ws), ws.numel(), _stream()), "ptk_chamfer_normals_fwd")
    return cn, tx, ty


def reference(xn, yn, ix, iy, lx, ly, reduction="mean"):
    return chamfer_normals_ref.chamfer_normals(cpu(xn), cpu(yn), cpu(ix), cpu(iy), cpu(lx), cpu(ly), reduction)


def check_forward(xn, yn, ix, iy, lx, ly, reduction):
    red = _lib.REDUCE_MEAN if reduction == "mean" else _lib.REDUCE_SUM
    cn, tx, ty = abi_fwd(xn, yn, ix, iy, None if lx is None else lx.long(), None if ly is None else ly.long(), red)
    want, wtx, wty = reference(xn, yn, ix, iy, lx, ly, reduction)
    assert (cpu(tx).double() - wtx).abs().max() <= 1e-6
    assert (cpu(ty).double() - wty).abs().max() <= 1e-6
    assert torch.all((cpu(cn).double() - want).abs() <= 1e-5 * want.abs() + 1e-6)
    return cn, tx, ty


# ------------------------------------------------------------------------------------- forward
@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("ragged", [False, True])
def test_forward_matches_the_restatement(algo, ragged, reduction):
    B, P1, P2 = 10, 700, 500
    x, y, xn, yn = data(B, P1, P2, 1)
    lx, ly = (lengths(B, P1, 2), lengths(B, P2, 3)) if ragged else (None, None)
    cham, cn, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn, lx, ly, reduction)
    got, _, _ = check_forward(xn, yn, ix, iy, lx, ly, reduction)
    assert same_bits(got, cn)


def test_forward_on_sliced_clouds():
    # more than 16384 points: several slices per pair, partials added by the second kernel
    B, P1, P2 = 3, 40000, 17000
    x, y, xn, yn = data(B, P1, P2, 4)
    lx = torch.tensor([40000, 16385, 1], device="cuda")
    ly = torch.tensor([9, 17000, 0], device="cuda")
    for lens in ((None, None), (lx, ly)):
        _, cn, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn, *lens)
        check_forward(xn, yn, ix, iy, *lens, "mean")


# ------------------------------------------------------------------------------------- edge cases
def test_empty_target_and_zero_normal_give_one():
    x, y, xn, yn = data(3, 50, 40, 5, unit=True)
    xn[1, 7] = 0.0
    lx = torch.tensor([50, 50, 0], device="cuda")
    ly = torch.tensor([0, 40, 40], device="cuda")
    _, _, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn, lx, ly, "sum")
    cn, tx, ty = abi_fwd(xn, yn, ix, iy, lx, ly, _lib.REDUCE_SUM)
    assert torch.all(tx[0] == 1.0) and torch.all(ty[2] == 1.0)   # the valid queries of a pair whose other cloud is empty
    assert float(tx[1, 7]) == 1.0
    assert float(cn[0]) == 50.0 and float(cn[2]) == 40.0
    assert is_plus_zero(ty[0]) and is_plus_zero(tx[2])


def test_scaled_and_flipped_normals_give_the_same_term():
    x, y, xn, yn = data(4, 600, 400, 6, unit=True)
    _, _, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn)
    base, btx, bty = abi_fwd(xn, yn, ix, iy, None, None)
    g = torch.Generator(device="cuda").manual_seed(7)
    sx = 10.0 ** (4 * torch.rand(4, 600, 1, device="cuda", generator=g) - 2)
    sy = 10.0 ** (4 * torch.rand(4, 400, 1, device="cuda", generator=g) - 2)
    fx = torch.where(torch.rand(4, 600, 1, device="cuda", generator=g) < 0.5, -1.0, 1.0)
    for a, b in ((xn * sx, yn * sy), (-xn, yn), (xn * fx * sx, -yn)):
        cn, tx, ty = abi_fwd(a.contiguous(), b.contiguous(), ix, iy, None, None)
        assert (tx - btx).abs().max() <= 2e-6 and (ty - bty).abs().max() <= 2e-6
        assert torch.allclose(cn, base, rtol=1e-5, atol=1e-6)


def test_nan_in_padding_is_never_read():
    B, P1, P2 = 6, 300, 200
    x, y, xn, yn = data(B, P1, P2, 8)
    lx, ly = lengths(B, P1, 9), lengths(B, P2, 10)
    _, _, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn, lx, ly)
    clean = abi_fwd(xn, yn, ix, iy, lx, ly)
    pad_x = torch.arange(P1, device="cuda")[None] >= lx.clamp(0, P1)[:, None]
    pad_y = torch.arange(P2, device="cuda")[None] >= ly.clamp(0, P2)[:, None]
    hx, hy = xn.clone(), yn.clone()
    hx[pad_x] = float("nan")
    hy[pad_y] = float("nan")
    hix, hiy = ix.clone(), iy.clone()
    hix[pad_x] = 1 << 30   # a padded query's idx is not read either
    hiy[pad_y] = -(1 << 30)
    for a, b in zip(clean, abi_fwd(hx, hy, hix, hiy, lx, ly)):
        assert same_bits(a, b)


def test_nan_in_a_valid_normal_reaches_only_the_terms_that_read_it():
    B, P1, P2 = 2, 300, 200
    x, y, xn, yn = data(B, P1, P2, 11)
    _, _, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn)
    clean_cn, ctx, cty = abi_fwd(xn, yn, ix, iy, None, None)
    j = int(ix[0, 0])
    bad = yn.clone()
    bad[0, j] = float("nan")
    cn, tx, ty = abi_fwd(xn, bad, ix, iy, None, None)
    read_x = torch.zeros(B, P1, dtype=torch.bool, device="cuda")
    read_x[0] = ix[0] == j
    read_y = torch.zeros(B, P2, dtype=torch.bool, device="cuda")
    read_y[0, j] = True
    assert torch.isnan(tx[read_x]).all() and torch.isnan(ty[read_y]).all()
    assert same_bits(tx[~read_x], ctx[~read_x]) and same_bits(ty[~read_y], cty[~read_y])
    assert torch.isnan(cn[0]) and same_bits(cn[1], clean_cn[1])


# ------------------------------------------------------------------------------------- pair independence
@pytest.mark.parametrize("P1,P2", [(3000, 2000), (20000, 17000)])
def test_a_pair_alone_in_a_batch_and_as_a_ragged_slice_has_the_same_bits(P1, P2):
    Bb, k = 64, 37
    x, y, xn, yn = data(Bb, P1, P2, 12)
    _, alone, _, _ = ptk_b200.ops.chamfer_normals(x[k:k + 1], y[k:k + 1], xn[k:k + 1], yn[k:k + 1])
    _, batch, _, _ = ptk_b200.ops.chamfer_normals(x, y, xn, yn)
    assert same_bits(alone[0], batch[k])
    l1, l2 = P1 * 2 // 3, P2 // 2 + 1
    lx = torch.full((Bb,), P1, device="cuda")
    ly = torch.full((Bb,), P2, device="cuda")
    lx[k], ly[k] = l1, l2
    _, ragged, _, _ = ptk_b200.ops.chamfer_normals(x, y, xn, yn, lx, ly)
    xs, ys = x[k:k + 1, :l1].contiguous(), y[k:k + 1, :l2].contiguous()
    _, sliced, _, _ = ptk_b200.ops.chamfer_normals(xs, ys, xn[k:k + 1, :l1].contiguous(), yn[k:k + 1, :l2].contiguous())
    assert same_bits(ragged[k], sliced[0])


@pytest.mark.parametrize("ragged", [False, True])
def test_cham_has_the_same_bits_with_and_without_normals(algo, ragged):
    B, P1, P2 = 8, 2000, 1500
    x, y, xn, yn = data(B, P1, P2, 13)
    lx, ly = (lengths(B, P1, 14), lengths(B, P2, 15)) if ragged else (None, None)
    cham, _, ix, iy = ptk_b200.ops.chamfer_normals(x, y, xn, yn, lx, ly)
    c0, jx, jy = ptk_b200.ops.chamfer(x, y, lx, ly)
    assert same_bits(cham, c0) and torch.equal(ix, jx) and torch.equal(iy, jy)


# ------------------------------------------------------------------------------------- gradients
def gpu_grads(x, y, xn, yn, lx, ly, reduction, w, need=(True, True)):
    xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    a, b = xn.clone().requires_grad_(need[0]), yn.clone().requires_grad_(need[1])
    _, cn, ix, iy = ptk_b200.ops.chamfer_normals(xr, yr, a, b, lx, ly, reduction)
    (cn * w).sum().backward()
    assert xr.grad is None and yr.grad is None   # the points get no gradient from the normal term
    return a.grad, b.grad, ix, iy


def ref_grads(xn, yn, ix, iy, lx, ly, reduction, w):
    a = cpu(xn).double().requires_grad_(True)
    b = cpu(yn).double().requires_grad_(True)
    cn, tx, ty = chamfer_normals_ref.chamfer_normals(a, b, cpu(ix), cpu(iy), cpu(lx), cpu(ly), reduction)
    (cn * cpu(w).double()).sum().backward()
    return a.grad, b.grad, tx.detach(), ty.detach()


def decided_rows(ix, iy, tx, ty):
    """Rows no query with fp64 |c| < 1e-5 contributes to (rounding decides sign(c) there)."""
    ix, iy = cpu(ix).long(), cpu(iy).long()
    amb_x, amb_y = (1 - tx).abs() < 1e-5, (1 - ty).abs() < 1e-5
    ok_x, ok_y = ~amb_x.clone(), ~amb_y.clone()
    for b in range(ix.shape[0]):
        ok_y[b, ix[b][amb_x[b]]] = False
        ok_x[b, iy[b][amb_y[b]]] = False
    return ok_x, ok_y


@pytest.mark.parametrize("flag", [False, True])
@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("ragged", [False, True])
def test_gradients_match_fp64_autograd(flag, reduction, ragged):
    B, P1, P2 = 6, 900, 700
    x, y, xn, yn = data(B, P1, P2, 16)
    xn[0, :5] *= 1e-4                                   # norms below 1e-3
    yn[1, :5] *= 1e-8                                   # and below eps: the clamped norm
    xn[2, 3] = 0.0                                      # a zero normal: its own part is 0
    lx, ly = (lengths(B, P1, 17), lengths(B, P2, 18)) if ragged else (None, None)
    w = torch.rand(B, device="cuda") + 0.5
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    try:
        gx, gy, ix, iy = gpu_grads(x, y, xn, yn, lx, ly, reduction, w)
    finally:
        torch.use_deterministic_algorithms(was)
    wx, wy, tx, ty = ref_grads(xn, yn, ix, iy, lx, ly, reduction, w)
    ok_x, ok_y = decided_rows(ix, iy, tx, ty)
    gx, gy = cpu(gx), cpu(gy)
    assert rel_err(gx[ok_x], wx[ok_x]) < 1e-5 and rel_err(gy[ok_y], wy[ok_y]) < 1e-5
    # the same bound on the rows of ordinary norms alone, which the tiny-norm rows would dominate
    big_x, big_y = ok_x & (cpu(xn).norm(dim=2) > 1e-2), ok_y & (cpu(yn).norm(dim=2) > 1e-2)
    assert rel_err(gx[big_x], wx[big_x]) < 1e-5 and rel_err(gy[big_y], wy[big_y]) < 1e-5
    if ragged:
        pad_x = torch.arange(P1)[None] >= cpu(lx).clamp(0, P1)[:, None]
        pad_y = torch.arange(P2)[None] >= cpu(ly).clamp(0, P2)[:, None]
        assert is_plus_zero(gx[pad_x]) and is_plus_zero(gy[pad_y])
        # a pair with an empty cloud has no gradient parts at all: every row of both normals is +0
        for b in range(B):
            if int(cpu(lx)[b].clamp(0, P1)) == 0 or int(cpu(ly)[b].clamp(0, P2)) == 0:
                assert is_plus_zero(gx[b]) and is_plus_zero(gy[b])


@pytest.mark.parametrize("flag", [False, True])
def test_one_gradient_alone(flag):
    B, P1, P2 = 4, 800, 600
    x, y, xn, yn = data(B, P1, P2, 19)
    w = torch.rand(B, device="cuda")
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    try:
        gx, gy, _, _ = gpu_grads(x, y, xn, yn, None, None, "mean", w)
        ax, _, _, _ = gpu_grads(x, y, xn, yn, None, None, "mean", w, (True, False))
        _, by, _, _ = gpu_grads(x, y, xn, yn, None, None, "mean", w, (False, True))
    finally:
        torch.use_deterministic_algorithms(was)
    if flag:
        assert same_bits(gx, ax) and same_bits(gy, by)
    else:
        assert rel_err(ax, gx) < 1e-6 and rel_err(by, gy) < 1e-6


# ------------------------------------------------------------------------------------- deterministic backward
def det_grads(x, y, xn, yn, lx=None, ly=None, w=None):
    if w is None:
        w = torch.ones(x.shape[0], device="cuda")
    gx, gy, ix, iy = gpu_grads(x, y, xn, yn, lx, ly, "mean", w)
    return gx, gy


def test_det_two_full_size_calls_have_the_same_bits(det):
    x, y, xn, yn = data(256, 10000, 10000, 20)
    a = det_grads(x, y, xn, yn)
    b = det_grads(x, y, xn, yn)
    assert same_bits(a[0], b[0]) and same_bits(a[1], b[1])


def test_det_pair_alone_in_a_batch_and_as_a_ragged_slice(det):
    Bb, k, P1, P2 = 64, 21, 3000, 2500
    x, y, xn, yn = data(Bb, P1, P2, 21)
    s = slice(k, k + 1)
    ax, ay = det_grads(x[s], y[s], xn[s], yn[s])
    bx, by = det_grads(x, y, xn, yn)
    assert same_bits(ax[0], bx[k]) and same_bits(ay[0], by[k])
    l1, l2 = 1777, 2100
    lx = torch.full((Bb,), P1, device="cuda")
    ly = torch.full((Bb,), P2, device="cuda")
    lx[k], ly[k] = l1, l2
    rx, ry = det_grads(x, y, xn, yn, lx, ly)
    sx, sy = det_grads(x[s, :l1].contiguous(), y[s, :l2].contiguous(), xn[s, :l1].contiguous(), yn[s, :l2].contiguous())
    assert same_bits(rx[k, :l1], sx[0]) and same_bits(ry[k, :l2], sy[0])
    assert is_plus_zero(rx[k, l1:]) and is_plus_zero(ry[k, l2:])


def test_det_permuting_x_queries_permutes_grad_xn_and_keeps_grad_yn(det):
    B, P1, P2 = 4, 3000, 2000
    x, y, xn, yn = data(B, P1, P2, 22)
    ax, ay = det_grads(x, y, xn, yn)
    perm = torch.randperm(P1, generator=torch.Generator().manual_seed(23)).cuda()
    px, py = det_grads(x[:, perm].contiguous(), y, xn[:, perm].contiguous(), yn)
    assert same_bits(px, ax[:, perm]) and same_bits(py, ay)


# ------------------------------------------------------------------------------------- shim and graph capture
@pytest.mark.parametrize("batch_reduction", [None, "mean", "sum"])
@pytest.mark.parametrize("weighted", [False, True])
def test_shim_end_to_end_against_the_restatement(shim, batch_reduction, weighted):
    from pytorch3d.loss import chamfer_distance
    B, P1, P2 = 4, 300, 250
    x, y, xn, yn = data(B, P1, P2, 24)
    weights = torch.rand(B, device="cuda") + 0.5 if weighted else None
    cham, cham_n = chamfer_distance(x, y, x_normals=xn, y_normals=yn, weights=weights, batch_reduction=batch_reduction)
    # the restatement on the oracle's nearest neighbours (the torch restatement of knn_points)
    _, ix = torch_ref.knn1(cpu(x), cpu(y))
    _, iy = torch_ref.knn1(cpu(y), cpu(x))
    want_cd, _, _ = torch_ref.chamfer_distance(cpu(x).double(), cpu(y).double())
    want_cn, _, _ = chamfer_normals_ref.chamfer_normals(cpu(xn), cpu(yn), ix, iy)
    for name, v in (("cd", want_cd), ("cn", want_cn)):
        if weighted:
            v = v * cpu(weights).double()
        if batch_reduction == "sum":
            v = v.sum()
        elif batch_reduction == "mean":
            v = v.sum() / (cpu(weights).double().sum() if weighted else B)
        got = cpu(cham if name == "cd" else cham_n).double()
        assert got.shape == v.shape and torch.all((got - v).abs() <= 1e-5 * v.abs() + 1e-6), name
    # one of the two normals: PyTorch3D ignores it
    c1, none = chamfer_distance(x, y, x_normals=xn, weights=weights, batch_reduction=batch_reduction)
    c2, none2 = chamfer_distance(x, y, y_normals=yn, weights=weights, batch_reduction=batch_reduction)
    assert none is None and none2 is None and same_bits(c1, cham) and same_bits(c2, cham)


@pytest.mark.parametrize("flag", [False, True])
def test_cuda_graph_replay_with_lengths_changed_in_place(shim, flag):
    from pytorch3d.loss import chamfer_distance
    B, P1, P2 = 8, 1500, 1300
    x, y, xn0, yn0 = data(B, P1, P2, 25)
    xn, yn = xn0.clone().requires_grad_(True), yn0.clone().requires_grad_(True)
    x.requires_grad_(True)
    lx = torch.full((B,), P1, dtype=torch.int64, device="cuda")
    ly = torch.full((B,), P2, dtype=torch.int64, device="cuda")
    w = torch.rand(B, device="cuda")

    def loss_fn(x, xn, yn, lx, ly):
        cham, cham_n = chamfer_distance(x, y, lx, ly, x_normals=xn, y_normals=yn, weights=w, batch_reduction="sum")
        return cham + 0.3 * cham_n

    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(flag)
    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                loss_fn(x, xn, yn, lx, ly).backward()
        torch.cuda.current_stream().wait_stream(s)
        x.grad = xn.grad = yn.grad = None
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss = loss_fn(x, xn, yn, lx, ly)
            loss.backward()
        rng = np.random.default_rng(26)
        for rep in range(4):
            n1, n2 = rng.integers(-10, P1 + 10, B), rng.integers(-10, P2 + 10, B)
            n1[rep % B] = 0
            n2[(rep + 3) % B] = 1
            lx.copy_(torch.from_numpy(n1))
            ly.copy_(torch.from_numpy(n2))
            graph.replay()
            torch.cuda.synchronize()
            xe = x.detach().clone().requires_grad_(True)
            ae, be = xn0.clone().requires_grad_(True), yn0.clone().requires_grad_(True)
            le = loss_fn(xe, ae, be, lx.clone(), ly.clone())
            gxe, gae, gbe = torch.autograd.grad(le, (xe, ae, be))
            if flag:
                assert torch.equal(loss, le) and torch.equal(x.grad, gxe)
                assert torch.equal(xn.grad, gae) and torch.equal(yn.grad, gbe)
            else:
                assert rel_err(loss, le) < 1e-5 and rel_err(x.grad, gxe) < 1e-5
                assert rel_err(xn.grad, gae) < 1e-5 and rel_err(yn.grad, gbe) < 1e-5
    finally:
        torch.use_deterministic_algorithms(was)
