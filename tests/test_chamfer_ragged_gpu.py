"""Ragged batches (per-cloud lengths) through every Chamfer / 1-NN scan: valid queries give the bits of a homogeneous
call on the sliced pair, padding is never read, padded rows are zero-filled (include/ptk.h)."""
import ctypes as C
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from ptk_b200 import _lib

pytestmark = pytest.mark.gpu
TOL = 1e-5  # relative, FP32 float atomics (north_star)

FILTER64_SPLIT = 2112  # split length of the 64-target, two-split form below (P2 = 4160, PTK_CH_NSPLIT = 2)


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


# name -> (scan, PTK_CH_NSPLIT or None, P1, P2, (lx, ly) per pair).  The lengths cover 0 and 1 on either side, P,
# values inside a chunk, inside a TMA tile, exactly on a split boundary, and outside [0, P] (clamped).
CONFIGS = {
    # 64-target chunks (aligned clouds, P % 4 == 0), one long split
    "filter64": ("filter", "1", 2500, 2600,
                 [(2500, 2600), (0, 17), (17, 0), (1, 2600), (2500, 1), (1, 1), (37, 2063), (1500, 1030), (-4, 99),
                  (2499, 9999), (1100, 1024), (0, 0)]),
    # 64-target chunks, two splits of FILTER64_SPLIT targets
    "filter64-split": ("filter", "2", 4160, 4160,
                       [(4160, FILTER64_SPLIT), (FILTER64_SPLIT, FILTER64_SPLIT + 1), (FILTER64_SPLIT - 1, 4159),
                        (3000, 2100), (1, 4160), (4160, 0), (777, 3333)]),
    # 16-target chunks (P % 4 != 0: no vector recheck), long and short splits
    "filter16": ("filter", "1", 1001, 1203, [(1001, 1203), (0, 5), (5, 0), (1, 1), (333, 1203), (1001, 17),
                                             (-1, 2000), (513, 514), (15, 16)]),
    "filter16-short": ("filter", "5", 1001, 1203, [(1001, 1203), (1001, 256), (1001, 512), (256, 255), (1, 1203),
                                                   (0, 300), (700, 0), (999, 1024), (1001, 1)]),
    "exact": ("exact", None, 999, 1100, [(999, 1100), (0, 40), (40, 0), (1, 1), (500, 517), (998, 2), (1234, -3)]),
    # compact sort (< 16k points), 16^3 cells
    "pruned": ("pruned", None, 3000, 2900, [(3000, 2900), (0, 100), (100, 0), (1, 2900), (3000, 1), (1, 1),
                                            (1601, 1777), (2999, 33), (5000, -5)]),
    # wide (multi-launch) sort, 16^3 cells
    "pruned-wide": ("pruned", None, 20000, 17000, [(20000, 17000), (16385, 5000), (1, 16999), (0, 77), (12345, 1)]),
    # wide sort on the fine (32^3) grid
    "pruned-fine": ("pruned", None, 40000, 34000, [(40000, 34000), (33000, 40000), (1, 20000), (20000, 0)]),
}


@pytest.fixture(params=list(CONFIGS))
def algo(request, monkeypatch):
    scan, nsplit, P1, P2, lens = CONFIGS[request.param]
    if nsplit is not None:
        monkeypatch.setenv("PTK_CH_NSPLIT", nsplit)
    ptk_b200.ops.set_chamfer_algo(scan)
    yield P1, P2, lens
    ptk_b200.ops.set_chamfer_algo("auto")


def clouds(B, P1, P2, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, P1, 3, generator=g) - 0.5
    y = torch.rand(B, P2, 3, generator=g) - 0.5
    return x.cuda(), y.cuda()


def clamp(v, P):
    return max(0, min(int(v), P))


def fill_padding(x, y, lx, ly, kind):
    """Copies of x, y whose rows past the lengths hold `kind`."""
    x, y = x.clone(), y.clone()
    B, P1, P2 = x.shape[0], x.shape[1], y.shape[1]
    for b in range(B):
        a, c = clamp(lx[b], P1), clamp(ly[b], P2)
        for t, n, other, m in ((x, a, y, c), (y, c, x, a)):
            P = t.shape[1]
            if n == P:
                continue
            if kind == "zero":
                t[b, n:] = 0
            elif kind == "nan":
                t[b, n:] = float("nan")
            elif kind == "inf":
                t[b, n:, 0] = float("inf")
                t[b, n:, 1] = -float("inf")
                t[b, n:, 2] = float("inf")
            elif kind == "big":
                t[b, n:] = 1e30
            elif kind == "impostor":  # the other cloud's queries: every padding point is some query's exact match
                if m > 0:
                    src = other[b, :m]
                    reps = (P - n + m - 1) // m
                    t[b, n:] = src.repeat(reps, 1)[:P - n]
                else:
                    t[b, n:] = 0
    return x, y


def ragged(x, y, lx, ly, reduction="mean"):
    lxt = torch.tensor(lx, dtype=torch.int64, device="cuda")
    lyt = torch.tensor(ly, dtype=torch.int64, device="cuda")
    cham, ix, iy = ptk_b200.ops.chamfer(x, y, lxt, lyt, point_reduction=reduction)
    dx, jx = ptk_b200.ops.knn1(x, y, lxt, lyt)
    dy, jy = ptk_b200.ops.knn1(y, x, lyt, lxt)
    return [t.cpu().numpy() for t in (cham, ix, iy, dx, jx, dy, jy)]


def check_against_pairs(x, y, lx, ly, out):
    cham, ix, iy, dx, jx, dy, jy = out
    B, P1, P2 = x.shape[0], x.shape[1], y.shape[1]
    for b in range(B):
        a, c = clamp(lx[b], P1), clamp(ly[b], P2)
        # padded queries: dist 0, idx 0
        assert (ix[b, a:] == 0).all() and (jx[b, a:] == 0).all() and (dx[b, a:] == 0).all()
        assert (iy[b, c:] == 0).all() and (jy[b, c:] == 0).all() and (dy[b, c:] == 0).all()
        if a == 0 or c == 0:  # no target for the other cloud's queries: zero fill, empty sums
            assert (ix[b] == 0).all() and (iy[b] == 0).all() and (dx[b] == 0).all() and (dy[b] == 0).all()
            assert cham[b] == 0
            continue
        xs, ys = x[b:b + 1, :a], y[b:b + 1, :c]
        rc, rix, riy = (t.cpu().numpy() for t in ptk_b200.ops.chamfer(xs, ys))
        rdx, rjx = (t.cpu().numpy() for t in ptk_b200.ops.knn1(xs, ys))
        rdy, rjy = (t.cpu().numpy() for t in ptk_b200.ops.knn1(ys, xs))
        assert np.array_equal(ix[b, :a], rix[0]) and np.array_equal(iy[b, :c], riy[0]), b
        assert np.array_equal(jx[b, :a], rjx[0]) and np.array_equal(jy[b, :c], rjy[0]), b
        assert np.array_equal(dx[b, :a].view(np.uint32), rdx[0].view(np.uint32)), b
        assert np.array_equal(dy[b, :c].view(np.uint32), rdy[0].view(np.uint32)), b
        assert np.array_equal(cham[b:b + 1].view(np.uint32), rc.view(np.uint32)), b


def test_ragged_equals_per_pair_for_any_padding(algo):
    P1, P2, lens = algo
    lx, ly = [l[0] for l in lens], [l[1] for l in lens]
    x, y = clouds(len(lens), P1, P2, seed=P1 * 7 + P2)
    base = None
    for kind in ("zero", "nan", "inf", "big", "impostor"):
        xp, yp = fill_padding(x, y, lx, ly, kind)
        out = ragged(xp, yp, lx, ly)
        resc = ptk_b200.ops.chamfer_rescued(xp, yp, torch.tensor(lx), torch.tensor(ly))
        if base is None:
            check_against_pairs(xp, yp, lx, ly, out)
            base = (out, resc)
        else:
            for a, b in zip(out, base[0]):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), kind
            assert resc == base[1], kind


def test_full_lengths_equal_the_homogeneous_entry_points(algo):
    P1, P2, lens = algo
    B = 3
    x, y = clouds(B, P1, P2, seed=11)
    L = _lib.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    ws = torch.empty(L.ptk_chamfer_workspace_bytes(B, P1, P2), dtype=torch.uint8, device="cuda")
    g = torch.rand(B, device="cuda")
    res = []
    for full in (False, True):
        ix = torch.empty(B, P1, dtype=torch.int32, device="cuda")
        iy = torch.empty(B, P2, dtype=torch.int32, device="cuda")
        dx, dy = torch.empty(B, P1, device="cuda"), torch.empty(B, P2, device="cuda")
        cham = torch.empty(B, device="cuda")
        gx, gy = torch.empty_like(x), torch.empty_like(y)
        if full:
            lx = torch.full((B,), P1, dtype=torch.int64, device="cuda")
            ly = torch.full((B,), P2, dtype=torch.int64, device="cuda")
            _lib.check(L.ptk_chamfer_fwd_lengths(p(x), p(y), p(lx), p(ly), B, P1, P2, _lib.REDUCE_MEAN, p(dx), p(ix),
                                                 p(dy), p(iy), p(cham), p(ws), ws.numel(), st))
            _lib.check(L.ptk_chamfer_bwd_lengths(p(x), p(y), p(lx), p(ly), p(ix), p(iy), p(g), B, P1, P2,
                                                 _lib.REDUCE_MEAN, p(gx), None, st))
        else:
            _lib.check(L.ptk_chamfer_fwd(p(x), p(y), B, P1, P2, p(dx), p(ix), p(dy), p(iy), p(cham), p(ws), ws.numel(),
                                         st))
            _lib.check(L.ptk_chamfer_bwd(p(x), p(y), p(ix), p(iy), p(g), B, P1, P2, p(gx), None, st))
        torch.cuda.synchronize()
        res.append([t.cpu().numpy() for t in (cham, ix, iy, dx, dy)] + [gx.cpu().numpy()])
    for a, b in zip(res[0][:5], res[1][:5]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert rel_err(res[1][5], res[0][5]) < TOL


def test_gradients_match_the_per_pair_backward(algo):
    P1, P2, lens = algo
    lx, ly = [l[0] for l in lens], [l[1] for l in lens]
    B = len(lens)
    x, y = clouds(B, P1, P2, seed=5)
    x, y = fill_padding(x, y, lx, ly, "big")
    g = torch.rand(B, device="cuda") + 0.5
    for reduction in ("mean", "sum"):
        for need_x in (True, False):  # grad of y only: the autoencoder's call
            xt, yt = x.clone().requires_grad_(need_x), y.clone().requires_grad_(True)
            cham, ix, iy = ptk_b200.ops.chamfer(xt, yt, torch.tensor(lx), torch.tensor(ly, dtype=torch.int32),
                                                point_reduction=reduction)
            (cham * g).sum().backward()
            gx = xt.grad.cpu().numpy() if need_x else None
            gy = yt.grad.cpu().numpy()
            iy_h = iy.cpu().numpy()
            for b in range(B):
                a, c = clamp(lx[b], P1), clamp(ly[b], P2)
                assert (gy[b, c:] == 0).all()
                if need_x:
                    assert (gx[b, a:] == 0).all()
                if a == 0 or c == 0:
                    assert (gy[b] == 0).all() and (not need_x or (gx[b] == 0).all())
                    continue
                xs, ys = x[b:b + 1, :a].clone().requires_grad_(need_x), y[b:b + 1, :c].clone().requires_grad_(True)
                rc, _, _ = ptk_b200.ops.chamfer(xs, ys, point_reduction=reduction)
                (rc * g[b]).sum().backward()
                rgy = ys.grad.cpu().numpy()[0]
                assert rel_err(gy[b, :c], rgy) < TOL, (reduction, b)
                if need_x:
                    rgx = xs.grad.cpu().numpy()[0]
                    assert rel_err(gx[b, :a], rgx) < TOL, (reduction, b)
                    # rows of x that are nobody's nearest neighbour get only the direct term: plain stores, same bits
                    lone = np.setdiff1d(np.arange(a), iy_h[b, :c])
                    assert np.array_equal(gx[b, lone].view(np.uint32), rgx[lone].view(np.uint32)), (reduction, b)


# ------------------------------------------------------------------ PyTorch3D's masked reductions, restated in torch
def torch_chamfer(x, y, lx, ly, reduction, weights=None, batch_reduction="mean"):
    B, P1, P2 = x.shape[0], x.shape[1], y.shape[1]
    lx = lx.clamp(0, P1)
    ly = ly.clamp(0, P2)
    mx = torch.arange(P1, device=x.device)[None] < lx[:, None]
    my = torch.arange(P2, device=x.device)[None] < ly[:, None]
    d = ((x[:, :, None, :] - y[:, None, :, :]) ** 2).sum(-1)
    big = torch.finfo(torch.float32).max
    dxy = d.masked_fill(~my[:, None, :], big).min(2).values
    dyx = d.masked_fill(~mx[:, :, None], big).min(1).values
    dxy = torch.where(mx & (ly[:, None] > 0), dxy, torch.zeros_like(dxy))
    dyx = torch.where(my & (lx[:, None] > 0), dyx, torch.zeros_like(dyx))
    cx, cy = dxy.sum(1), dyx.sum(1)
    if reduction == "mean":
        cx = cx / lx.clamp(min=1)
        cy = cy / ly.clamp(min=1)
    cham = cx + cy
    if weights is not None:
        cham = cham * weights
    if batch_reduction == "sum":
        cham = cham.sum()
    elif batch_reduction == "mean":
        cham = cham.sum() / (weights.sum() if weights is not None else max(B, 1))
    return cham, dxy


@pytest.fixture
def shim(monkeypatch):
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("batch_reduction", [None, "mean", "sum"])
@pytest.mark.parametrize("weighted", [False, True])
def test_shim_chamfer_distance_with_lengths(shim, reduction, batch_reduction, weighted):
    from pytorch3d.loss import chamfer_distance
    B, P1, P2 = 6, 300, 257
    x, y = clouds(B, P1, P2, seed=3)
    lx = torch.tensor([300, 0, 1, 150, 299, 77], device="cuda")
    ly = torch.tensor([257, 40, 1, 0, 128, 300], dtype=torch.int32)
    x, y = fill_padding(x, y, lx.tolist(), ly.tolist(), "big")
    w = torch.rand(B, device="cuda") + 0.5 if weighted else None
    xa, ya = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    xb, yb = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    cd, none = chamfer_distance(xa, ya, x_lengths=lx, y_lengths=ly, weights=w, batch_reduction=batch_reduction,
                                point_reduction=reduction)
    ref, _ = torch_chamfer(xb, yb, lx, ly.cuda().long(), reduction, w, batch_reduction)
    assert none is None and cd.shape == ref.shape
    assert rel_err(cd.detach().cpu().numpy(), ref.detach().cpu().numpy()) < TOL
    cd.sum().backward()
    ref.sum().backward()
    assert rel_err(xa.grad.cpu().numpy(), xb.grad.cpu().numpy()) < TOL
    assert rel_err(ya.grad.cpu().numpy(), yb.grad.cpu().numpy()) < TOL


def test_shim_knn_points_with_lengths(shim):
    from pytorch3d.ops import knn_points
    B, P1, P2 = 5, 400, 333
    x, y = clouds(B, P1, P2, seed=9)
    l1 = torch.tensor([400, 1, 0, 200, 399], device="cuda")
    l2 = torch.tensor([333, 333, 20, 0, 1], device="cuda")
    x, y = fill_padding(x, y, l1.tolist(), l2.tolist(), "nan")
    k = knn_points(x, y, lengths1=l1, lengths2=l2, K=1)
    assert k.dists.shape == (B, P1, 1) and k.idx.shape == (B, P1, 1) and k.idx.dtype == torch.int64
    d, i = ptk_b200.ops.knn1(x, y, l1, l2)
    assert torch.equal(k.dists[..., 0], d) and torch.equal(k.idx[..., 0], i.long())
    _, ref = torch_chamfer(x, y, l1, l2, "sum")
    assert rel_err(k.dists[..., 0].cpu().numpy(), ref.cpu().numpy()) < TOL
    for b in range(B):
        a = int(l1[b])
        assert (k.dists[b, a:] == 0).all() and (k.idx[b, a:] == 0).all()
        if int(l2[b]) == 0:
            assert (k.dists[b] == 0).all() and (k.idx[b] == 0).all()


def test_cuda_graph_replay_with_lengths_changed_in_place():
    B, P1, P2 = 8, 1500, 1300
    x, y = clouds(B, P1, P2, seed=21)
    x.requires_grad_(True)
    y.requires_grad_(True)
    lx = torch.full((B,), P1, dtype=torch.int64, device="cuda")
    ly = torch.full((B,), P2, dtype=torch.int64, device="cuda")
    g = torch.rand(B, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):  # warm-up outside the capture
            cham, _, _ = ptk_b200.ops.chamfer(x, y, lx, ly)
            (cham * g).sum().backward()
    torch.cuda.current_stream().wait_stream(s)
    x.grad = None
    y.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cham, ix, iy = ptk_b200.ops.chamfer(x, y, lx, ly)
        (cham * g).sum().backward()
    rng = np.random.default_rng(4)
    for rep in range(4):
        nx = rng.integers(-10, P1 + 10, B)
        ny = rng.integers(-10, P2 + 10, B)
        nx[rep % B] = 0
        lx.copy_(torch.from_numpy(nx))
        ly.copy_(torch.from_numpy(ny))
        graph.replay()
        torch.cuda.synchronize()
        xe, ye = x.detach().clone().requires_grad_(True), y.detach().clone().requires_grad_(True)
        ce, iex, iey = ptk_b200.ops.chamfer(xe, ye, lx.clone(), ly.clone())
        gxe, gye = torch.autograd.grad((ce * g).sum(), (xe, ye))
        assert torch.equal(cham, ce) and torch.equal(ix, iex) and torch.equal(iy, iey)
        assert rel_err(x.grad.cpu().numpy(), gxe.cpu().numpy()) < TOL
        assert rel_err(y.grad.cpu().numpy(), gye.cpu().numpy()) < TOL


@pytest.mark.parametrize("B,P", [(256, 10000), (2, 100000)])
def test_ragged_pruned_equals_ragged_filter_at_full_size(B, P):
    x, y = clouds(B, P, P, seed=B + P)
    rng = np.random.default_rng(B)
    lx = torch.from_numpy(rng.integers(P // 4, P + 1, B)).cuda()
    ly = torch.from_numpy(rng.integers(P // 4, P + 1, B)).cuda()
    outs = []
    try:
        for name in ("filter", "pruned"):
            ptk_b200.ops.set_chamfer_algo(name)
            cham, ix, iy = ptk_b200.ops.chamfer(x, y, lx, ly)
            d, i = ptk_b200.ops.knn1(x, y, lx, ly)
            outs.append([t.cpu().numpy() for t in (cham, ix, iy, d, i)])
    finally:
        ptk_b200.ops.set_chamfer_algo("auto")
    for a, b in zip(*outs):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
