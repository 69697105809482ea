"""Deterministic backward (torch.use_deterministic_algorithms(True) -> ptk_*_bwd_det): bit-exact against a numpy
restatement of the scheme, order independence, non-finite inputs, the fused mesh Chamfer and a whole training step."""
import copy
import ctypes as C
import types

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
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # any cuBLAS call of the test may then run under the flag
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was_on, warn_only=was_warn)
        torch.utils.deterministic.fill_uninitialized_memory = was_fill


# ------------------------------------------------------------------------------------- numpy restatement (include/ptk.h)
def _ceil_log2_f32(m):
    mant, ex = np.frexp(np.float64(m))  # m = mant * 2^ex, mant in [0.5, 1)
    return int(ex) - 1 if mant == 0.5 else int(ex)


def _ceil_log2_int(n):
    c = 0
    while (1 << c) < n:
        c += 1
    return c


def _exponent(terms, n):
    a = np.abs(np.concatenate([t.ravel() for t in terms]))
    a = a[np.isfinite(a)]
    M = np.float32(a.max()) if a.size else np.float32(0)
    return 0 if M == 0 else 62 - _ceil_log2_f32(M) - _ceil_log2_int(n)


def _quantise(t, e):
    fin = np.isfinite(t)
    return np.where(fin, np.rint(np.where(fin, t, 0).astype(np.float64) * 2.0 ** e), 0).astype(np.int64), fin


def _convert(acc, nonfinite, e):
    g = np.ldexp(acc.astype(np.float32), np.int32(-e))
    assert g.dtype == np.float32
    return np.where(np.isfinite(nonfinite), g, nonfinite).astype(np.float32)


def det_chamfer_bwd(x, y, lx, ly, ix, iy, g, mean):
    """ptk_chamfer_bwd_det restated: the forward's indices, int64 sums, an int64 -> float32 cast and ldexp."""
    B, P1, _ = x.shape
    P2 = y.shape[1]
    gx, gy = np.zeros((B, P1, 3), np.float32), np.zeros((B, P2, 3), np.float32)
    for b in range(B):
        L1 = int(np.clip(lx[b], 0, P1)) if lx is not None else P1
        L2 = int(np.clip(ly[b], 0, P2)) if ly is not None else P2
        if L1 == 0 or L2 == 0:
            continue
        gb = np.float32(g[b])
        jx, jy = ix[b, :L1].astype(np.int64), iy[b, :L2].astype(np.int64)
        with np.errstate(all="ignore"):
            sx = np.float32(2) * (gb / np.float32(L1)) if mean else np.float32(2) * gb
            sy = np.float32(2) * (gb / np.float32(L2)) if mean else np.float32(2) * gb
            tx = (sx * (x[b, :L1] - y[b, jx])).astype(np.float32)
            ty = (sy * (y[b, :L2] - x[b, jy])).astype(np.float32)
        e = _exponent([tx, ty], max(L1, L2) + 1)
        ax, ay = np.zeros((P1, 3), np.int64), np.zeros((P2, 3), np.int64)
        nx, ny = np.zeros((P1, 3), np.float32), np.zeros((P2, 3), np.float32)
        qx, fx = _quantise(tx, e)
        qy, fy = _quantise(ty, e)
        ax[:L1] += qx
        np.add.at(ay, jx, -qx)
        ay[:L2] += qy
        np.add.at(ax, jy, -qy)
        with np.errstate(all="ignore"):
            nx[:L1] += np.where(fx, 0, tx)
            np.add.at(ny, jx, np.where(fx, 0, -tx))
            ny[:L2] += np.where(fy, 0, ty)
            np.add.at(nx, jy, np.where(fy, 0, -ty))
        gx[b], gy[b] = _convert(ax, nx, e), _convert(ay, ny, e)
    return gx, gy


def _bary(uv, b, S):
    with np.errstate(all="ignore"):
        rt = np.sqrt(uv[0, b]).astype(np.float32)
        v = uv[1, b]
        return np.stack([np.float32(1) - rt, rt * (np.float32(1) - v), rt * v], 1).astype(np.float32)  # (S, 3)


def det_sample_bwd(gp, fidx, uv, faces, V):
    """ptk_sample_bwd_det restated."""
    B, S, _ = gp.shape
    out = np.zeros((B, V, 3), np.float32)
    for b in range(B):
        w = _bary(uv, b, S)
        with np.errstate(all="ignore"):
            c = (w[:, :, None] * gp[b][:, None, :]).astype(np.float32)  # (S, k, d)
        e = _exponent([c], 3 * S + 1)
        q, fin = _quantise(c, e)
        acc, nf = np.zeros((V, 3), np.int64), np.zeros((V, 3), np.float32)
        rows = faces[fidx[b].astype(np.int64)]  # (S, 3) vertex of each k
        for k in range(3):
            np.add.at(acc, rows[:, k], q[:, k])
            with np.errstate(all="ignore"):
                np.add.at(nf, rows[:, k], np.where(fin[:, k], 0, c[:, k]))
        out[b] = _convert(acc, nf, e)
    return out


# ------------------------------------------------------------------------------------- helpers
def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def chamfer_bwd_det_abi(x, y, ix, iy, g, lx=None, ly=None, reduction=_lib.REDUCE_MEAN, want_x=True, want_y=True):
    L = _lib.lib()
    B, P1, _ = x.shape
    P2 = y.shape[1]
    gx = torch.empty_like(x) if want_x else None
    gy = torch.empty_like(y) if want_y else None
    ws = torch.empty(max(L.ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2), 16), dtype=torch.uint8, device=x.device)
    _lib.check(L.ptk_chamfer_bwd_det(_p(x), _p(y), _p(lx), _p(ly), _p(ix), _p(iy), _p(g), B, P1, P2, reduction, _p(gx),
                                     _p(gy), _p(ws), ws.numel(), _stream()), "ptk_chamfer_bwd_det")
    return gx, gy


def sample_bwd_det_abi(gp, fidx, uv, faces_i32, V):
    L = _lib.lib()
    B, S, _ = gp.shape
    gv = torch.empty(B, V, 3, device=gp.device)
    ws = torch.empty(L.ptk_sample_bwd_det_workspace_bytes(B, V), dtype=torch.uint8, device=gp.device)
    _lib.check(L.ptk_sample_bwd_det(_p(gp), _p(fidx), _p(uv), _p(faces_i32), B, V, faces_i32.shape[0], S, _p(gv), _p(ws),
                                    ws.numel(), _stream()), "ptk_sample_bwd_det")
    return gv


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def cpu(t):
    return t.detach().cpu().numpy() if t is not None else None


def _clouds(B, P1, P2, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((B, P1, 3), np.float32)
    y = (rng.random((B, P2, 3), np.float32) * 0.9 + 0.05).astype(np.float32)
    g = rng.uniform(0.5, 2.0, B).astype(np.float32)
    return x, y, g


# ------------------------------------------------------------------------------------- 1. bits against the restatement
@pytest.mark.parametrize("algo", ["filter", "exact", "pruned"])
def test_chamfer_bwd_det_matches_the_restatement(det, algo):
    B, P1, P2 = 5, 3000, 2500
    x, y, g = _clouds(B, P1, P2, 1)
    # clusters: a few targets are the nearest neighbour of many queries
    y[0, :40] = y[0, 0] + np.float32(1e-4) * np.arange(40, dtype=np.float32)[:, None]
    cases = [(None, None), (np.array([0, 1, P1, 1234, 2049]), np.array([700, 1, P2, 0, 1777]))]
    xt, yt, gt_ = (torch.from_numpy(a).cuda() for a in (x, y, g))
    try:
        ptk_b200.ops.set_chamfer_algo(algo)
        for lx, ly in cases:
            lxt = torch.from_numpy(lx).cuda() if lx is not None else None
            lyt = torch.from_numpy(ly).cuda() if ly is not None else None
            for red in ("mean", "sum"):
                _, ix, iy = ptk_b200.ops.chamfer(xt, yt, lxt, lyt, point_reduction=red)
                wx, wy = det_chamfer_bwd(x, y, lx, ly, cpu(ix), cpu(iy), g, red == "mean")
                for want_x, want_y in ((True, True), (True, False), (False, True)):
                    xr = xt.clone().requires_grad_(want_x)
                    yr = yt.clone().requires_grad_(want_y)
                    cham, _, _ = ptk_b200.ops.chamfer(xr, yr, lxt, lyt, point_reduction=red)
                    (cham * gt_).sum().backward()
                    if want_x:
                        assert same_bits(cpu(xr.grad), wx), (algo, lx, red, want_x, want_y)
                    if want_y:
                        assert same_bits(cpu(yr.grad), wy), (algo, lx, red, want_x, want_y)
    finally:
        ptk_b200.ops.set_chamfer_algo("auto")


@pytest.mark.parametrize("V", [500, 3000, 6000])
def test_sample_bwd_det_matches_the_restatement(det, V):
    """Meshes below and above the default kernel's shared-memory limit (4096 vertices) and the det kernel's (2048)."""
    rng = np.random.default_rng(V)
    B, S, F = 3, 20000, 2 * V
    faces = rng.integers(0, V, (F, 3)).astype(np.int32)
    faces[0] = [3, 3, 5]  # a degenerate face lists a vertex twice
    fidx = rng.integers(0, F, (B, S)).astype(np.int32)
    fidx[:, :300] = 0  # one face drawn many times
    uv = rng.random((2, B, S), np.float32)
    gp = rng.standard_normal((B, S, 3)).astype(np.float32)
    gv = sample_bwd_det_abi(*(torch.from_numpy(a).cuda() for a in (gp, fidx, uv, faces)), V)
    assert same_bits(cpu(gv), det_sample_bwd(gp, fidx, uv, faces, V))


# ------------------------------------------------------------------------------------- 2. accuracy
def test_det_accuracy_against_the_double_oracle(det, oracle):
    B, P1, P2 = 3, 4000, 3000
    x, y, g = _clouds(B, P1, P2, 2)
    x[1] *= 1e3
    y[1] *= 1e3
    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    yt = torch.from_numpy(y).cuda().requires_grad_(True)
    cham, ix, iy = ptk_b200.ops.chamfer(xt, yt)
    (cham * torch.from_numpy(g).cuda()).sum().backward()
    ox, oy = oracle.chamfer_bwd(x, y, cpu(ix), cpu(iy), g)
    assert rel_err(cpu(xt.grad), ox) < TOL and rel_err(cpu(yt.grad), oy) < TOL
    fx, fy = np.mean(cpu(xt.grad) == ox), np.mean(cpu(yt.grad) == oy)
    print(f"\nchamfer det: bit-equal to the double oracle: grad_x {fx:.6f}, grad_y {fy:.6f}")

    rng = np.random.default_rng(3)
    V, S, F = 1949, 10000, 2464
    faces = rng.integers(0, V, (F, 3)).astype(np.int32)
    fidx = rng.integers(0, F, (B, S)).astype(np.int32)
    uv = rng.random((2, B, S), np.float32)
    gp = rng.standard_normal((B, S, 3)).astype(np.float32)
    gv = cpu(sample_bwd_det_abi(*(torch.from_numpy(a).cuda() for a in (gp, fidx, uv, faces)), V))
    ov = oracle.sample_bwd(gp, fidx, uv, faces, V)
    assert rel_err(gv, ov) < TOL
    print(f"sampler det: bit-equal to the double oracle: {np.mean(gv == ov):.6f}")


# ------------------------------------------------------------------------------------- 3. order independence
def test_permuting_queries_permutes_grad_x_and_keeps_grad_y(det):
    B, P1, P2 = 2, 5000, 4000
    x, y, g = _clouds(B, P1, P2, 4)
    perm = np.random.default_rng(5).permutation(P1)
    outs = []
    for xs in (x, np.ascontiguousarray(x[:, perm])):
        xt = torch.from_numpy(xs).cuda().requires_grad_(True)
        yt = torch.from_numpy(y).cuda().requires_grad_(True)
        cham, ix, iy = ptk_b200.ops.chamfer(xt, yt)
        (cham * torch.from_numpy(g).cuda()).sum().backward()
        outs.append((cpu(xt.grad), cpu(yt.grad), cpu(iy)))
    (gx0, gy0, iy0), (gx1, gy1, iy1) = outs
    inv = np.argsort(perm)
    assert np.array_equal(perm[iy1], iy0), "the clouds have a nearest-neighbour tie"
    assert same_bits(gx1, np.ascontiguousarray(gx0[:, perm])) and same_bits(gy1, gy0)
    assert same_bits(gx0, np.ascontiguousarray(gx1[:, inv]))


def test_permuting_samples_keeps_grad_verts(det):
    rng = np.random.default_rng(6)
    B, S, V, F = 2, 30000, 1949, 2464
    faces = rng.integers(0, V, (F, 3)).astype(np.int32)
    fidx = rng.integers(0, F, (B, S)).astype(np.int32)
    uv = rng.random((2, B, S), np.float32)
    gp = rng.standard_normal((B, S, 3)).astype(np.float32)
    perm = rng.permutation(S)
    a = sample_bwd_det_abi(*(torch.from_numpy(t).cuda() for t in (gp, fidx, uv, faces)), V)
    b = sample_bwd_det_abi(*(torch.from_numpy(np.ascontiguousarray(t)).cuda()
                             for t in (gp[:, perm], fidx[:, perm], uv[:, :, perm], faces)), V)
    assert same_bits(cpu(a), cpu(b))


def test_pair_alone_equals_pair_in_a_batch_of_64(det):
    B, P1, P2, k = 64, 2000, 1500, 17
    x, y, g = _clouds(B, P1, P2, 7)
    xt, yt, gt_ = (torch.from_numpy(a).cuda() for a in (x, y, g))
    _, ix, iy = ptk_b200.ops.chamfer(xt, yt)
    gx, gy = chamfer_bwd_det_abi(xt, yt, ix, iy, gt_)
    gx1, gy1 = chamfer_bwd_det_abi(xt[k:k + 1].contiguous(), yt[k:k + 1].contiguous(), ix[k:k + 1].contiguous(),
                                   iy[k:k + 1].contiguous(), gt_[k:k + 1].contiguous())
    assert same_bits(cpu(gx)[k:k + 1], cpu(gx1)) and same_bits(cpu(gy)[k:k + 1], cpu(gy1))


@pytest.mark.parametrize("reduction", [_lib.REDUCE_MEAN, _lib.REDUCE_SUM])
def test_ragged_pair_equals_the_sliced_pair(det, reduction):
    B, P1, P2 = 4, 3000, 2600
    x, y, g = _clouds(B, P1, P2, 8)
    lx, ly = np.array([3000, 1, 1500, 2222]), np.array([2600, 900, 1, 1017])
    xt, yt, gt_ = (torch.from_numpy(a).cuda() for a in (x, y, g))
    lxt, lyt = torch.from_numpy(lx).cuda(), torch.from_numpy(ly).cuda()
    _, ix, iy = ptk_b200.ops.chamfer(xt, yt, lxt, lyt, point_reduction="mean" if reduction == _lib.REDUCE_MEAN else "sum")
    gx, gy = (cpu(t) for t in chamfer_bwd_det_abi(xt, yt, ix, iy, gt_, lxt, lyt, reduction))
    for b in range(B):
        sx, sy = xt[b:b + 1, :lx[b]].contiguous(), yt[b:b + 1, :ly[b]].contiguous()
        sgx, sgy = chamfer_bwd_det_abi(sx, sy, ix[b:b + 1, :lx[b]].contiguous(), iy[b:b + 1, :ly[b]].contiguous(),
                                       gt_[b:b + 1].contiguous(), reduction=reduction)
        assert same_bits(gx[b:b + 1, :lx[b]], cpu(sgx)) and same_bits(gy[b:b + 1, :ly[b]], cpu(sgy)), b
        assert not gx[b, lx[b]:].any() and not gy[b, ly[b]:].any()
        assert not np.signbit(gx[b, lx[b]:]).any() and not np.signbit(gy[b, ly[b]:]).any()  # +0


def test_two_calls_at_full_size_give_the_same_bits(det):
    B, P = 256, 10000
    gen = torch.Generator(device="cuda").manual_seed(9)
    x = torch.rand(B, P, 3, device="cuda", generator=gen)
    y = torch.rand(B, P, 3, device="cuda", generator=gen)
    g = torch.rand(B, device="cuda", generator=gen)
    _, ix, iy = ptk_b200.ops.chamfer(x, y)
    a = chamfer_bwd_det_abi(x, y, ix, iy, g)
    b = chamfer_bwd_det_abi(x, y, ix, iy, g)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.isfinite(a[0]).all() and torch.isfinite(a[1]).all()


# ------------------------------------------------------------------------------------- 4. non-finite input
@pytest.mark.parametrize("reduction", [_lib.REDUCE_MEAN, _lib.REDUCE_SUM])
def test_non_finite_input(det, reduction):
    B, P1, P2 = 3, 2000, 1800
    x, y, g = _clouds(B, P1, P2, 10)
    xt, yt = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    _, ix, iy = ptk_b200.ops.chamfer(xt, yt)  # indices of the clean clouds; the backward then sees hostile values
    ixn, iyn = cpu(ix), cpu(iy)
    x[0, 5, 0] = np.nan
    x[0, 6, 1] = np.inf
    y[0, iyn[0, 7], 2] = -np.inf  # a target: its scatter row gets -inf and the query's row +inf
    y[1, ixn[1, 3], 0] = np.inf
    y[1, ixn[1, 4], 0] = -np.inf  # both infinities may meet in one row: NaN
    g[2] = np.float32(3e38)       # mean: terms near 1e35 (a negative exponent); sum: s = 2 g overflows to inf
    xt, yt, gt_ = (torch.from_numpy(a).cuda() for a in (x, y, g))
    runs = [tuple(cpu(t) for t in chamfer_bwd_det_abi(xt, yt, ix, iy, gt_, reduction=reduction)) for _ in range(2)]
    want = det_chamfer_bwd(x, y, None, None, ixn, iyn, g, reduction == _lib.REDUCE_MEAN)
    for got in runs[1:] + [want]:
        for a, b in zip(runs[0], got):
            nan = np.isnan(a)
            assert np.array_equal(nan, np.isnan(b))
            assert same_bits(a[~nan], b[~nan])
    assert np.isnan(runs[0][0]).any() and np.isinf(runs[0][0]).any() and np.isinf(runs[0][1]).any()
    assert np.isfinite(runs[0][0][1:]).mean() > 0.99 or reduction == _lib.REDUCE_SUM


# ------------------------------------------------------------------------------------- 5. fused mesh Chamfer
@pytest.mark.parametrize("want_verts", [True, False])
def test_fused_mesh_chamfer_equals_the_per_repeat_composition(det, golden, want_verts):
    m = golden("meshes")
    verts0 = torch.from_numpy(m["obj0_verts"]).cuda()
    faces = torch.from_numpy(m["obj0_faces"].astype(np.int64)).cuda()
    faces_i32 = faces.to(torch.int32)
    B, S, P2, R = 3, 1700, 2100, 3
    verts = (verts0[None] * (1.0 + 0.1 * torch.arange(B, device="cuda")[:, None, None])).contiguous()
    gen = torch.Generator(device="cuda").manual_seed(5)
    gt = torch.rand(B, P2, 3, device="cuda", generator=gen) * 0.2 - 0.1
    uni = [ptk_b200.utils.draw_uniforms(B, S, torch.device("cuda"), gen) for _ in range(R)]
    w = torch.tensor([1.0, -2.0, 0.5], device="cuda")
    vr = verts.clone().requires_grad_(want_verts)
    gr = gt.clone().requires_grad_(True)
    cd = ptk_b200.utils.chamfer_distance(vr, faces, gr, num=S, repeat=R, uniforms=uni)
    (cd * w).sum().backward()

    gc = w * (torch.ones((), device="cuda") / R)  # mc_scale: fl32(1 / repeat) * grad_cd
    acc_v = acc_g = None
    for uf, uv in uni:
        pts, fidx = ptk_b200.ops.sample_points(verts, faces_i32, uf, uv)
        _, ix, iy = ptk_b200.ops.chamfer(pts, gt)
        gx, gy = chamfer_bwd_det_abi(pts, gt, ix, iy, gc, want_x=want_verts)
        acc_g = gy if acc_g is None else acc_g + gy
        if want_verts:
            gv = sample_bwd_det_abi(gx, fidx, uv.contiguous(), faces_i32, verts.shape[1])
            acc_v = gv if acc_v is None else acc_v + gv
    assert torch.equal(gr.grad, acc_g)
    if want_verts:
        assert torch.equal(vr.grad, acc_v)


# ------------------------------------------------------------------------------------- 6. end to end
def test_training_step_is_bit_reproducible_and_graph_replay_equals_eager(det, golden):
    """The ChartDeformer step of test_compat_gpu.py::test_graphed_step_replays_the_eager_step under the flag, with
    fill_uninitialized_memory left on (an output a kernel fails to write would show up as NaN)."""
    from ptk_b200.graph import Graph
    assert torch.utils.deterministic.fill_uninitialized_memory
    adj, meshes = golden("adjacency"), golden("meshes")
    g = Graph.from_csr(adj["p_adj_rowptr"], adj["p_adj_col"], "cuda")
    adj_info = {"origional": Graph.from_csr(adj["p_origional_rowptr"], adj["p_origional_col"], "cuda").dense(),
                "adj": g.dense(), "faces": torch.from_numpy(adj["p_faces"]).cuda().long()}
    args = types.SimpleNamespace(use_img=True, use_touch=True, finger=True, num_grasps=5, num_GCN_layers=5,
                                 hidden_GCN_size=96, cut=0.33)
    B, width, npts = 3, 40, 2000
    torch.manual_seed(0)
    net_e = ptk_b200.recon.ChartDeformer(adj_info, args, width).cuda()
    net_g = copy.deepcopy(net_e)
    gen = torch.Generator(device="cuda").manual_seed(5)
    vision = torch.from_numpy(meshes["vision_verts"]).cuda()[None].repeat(B, 1, 1)
    touch = torch.rand(B, 125, 3, device="cuda", generator=gen) * 0.02 + 0.2
    feats = [torch.rand(B, n, width, device="cuda", generator=gen) for n in (1824, 1949, 1949)]
    gt = torch.nn.functional.normalize(torch.randn(B, npts, 3, device="cuda", generator=gen), dim=-1) * 0.25
    uni = [ptk_b200.utils.draw_uniforms(B, npts, torch.device("cuda"), gen) for _ in range(3)]
    lr = torch.zeros((), device="cuda")

    def make(net):
        opt = torch.optim.Adam(net.parameters(), lr=lr, fused=True, capturable=True)

        def step():
            opt.zero_grad(set_to_none=True)
            verts = net(vision, touch, lambda it, v: feats[it])
            loss, _ = ptk_b200.recon.recon_loss(verts, adj_info["faces"], gt, number_points=npts, uniforms=uni)
            loss.backward()
            opt.step()
            return loss
        return step

    step_e = make(net_e)
    eager = []
    for _ in range(2):
        loss = step_e().detach().clone()
        eager.append((loss, [p.grad.clone() for p in net_e.parameters()]))
    (l0, g0), (l1, g1) = eager
    assert torch.isfinite(l0) and torch.equal(l0, l1)
    for a, b in zip(g0, g1):
        assert torch.isfinite(a).all() and torch.equal(a, b)
    graphed = ptk_b200.recon.GraphedStep(make(net_g), warmup=2)
    for _ in range(2):
        lg = graphed()
    torch.cuda.synchronize()
    assert torch.equal(lg.detach(), l0)
    for a, b in zip(net_g.parameters(), g0):
        assert torch.equal(a.grad, b)


# ------------------------------------------------------------------------------------- 7. flag off
def test_flag_off_keeps_the_default_backward():
    """Without the flag ops.chamfer runs the two default kernels, with the bits of a direct ptk_chamfer_bwd_lengths call
    (y is x moved by a little: every row receives one scatter term, so the fp32 atomics add in one order only)."""
    assert not torch.are_deterministic_algorithms_enabled()
    B, P = 3, 3000
    rng = np.random.default_rng(11)
    x = rng.random((B, P, 3), np.float32)
    y = (x + rng.uniform(-1e-5, 1e-5, x.shape)).astype(np.float32)
    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    yt = torch.from_numpy(y).cuda().requires_grad_(True)
    g = torch.from_numpy(rng.uniform(0.5, 2.0, B).astype(np.float32)).cuda()
    cham, ix, iy = ptk_b200.ops.chamfer(xt, yt)
    assert torch.equal(ix.long(), torch.arange(P, device="cuda").expand(B, P))
    torch.cuda.synchronize()
    before = _lib.launch_count()
    (cham * g).sum().backward()
    assert _lib.launch_count() - before == 2  # own-part stores + near-part scatter (pair_bwd.cuh)
    gx, gy = torch.empty_like(xt), torch.empty_like(yt)
    _lib.check(_lib.lib().ptk_chamfer_bwd_lengths(_p(xt), _p(yt), None, None, _p(ix), _p(iy), _p(g), B, P, P,
                                                  _lib.REDUCE_MEAN, _p(gx), _p(gy), _stream()), "ptk_chamfer_bwd_lengths")
    assert torch.equal(xt.grad, gx) and torch.equal(yt.grad, gy)
