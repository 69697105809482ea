"""Point-cloud normals on the GPU (ops.estimate_normals / estimate_local_frames, the shim's
estimate_pointcloud_normals / estimate_pointcloud_local_coord_frames, ptk_point_frames_*): the forward against the fp64
restatement on the GPU's own K-NN indices, with angle bounds from the eigenvalue gaps and sign checks where the sign
rule's margin is certain; bits across runs, batching and slicing; non-finite input; both backward forms against fp64
autograd; the mesh -> samples -> chamfer_distance(x_normals=, y_normals=estimate_pointcloud_normals(gt)) chain; CUDA-graph
replay and no host synchronisation."""
import sys

import numpy as np
import pytest
import torch

import ptk_b200
from ptk_b200 import ops

import point_normals_ref as ref

pytestmark = pytest.mark.gpu
U = 2.0 ** -24


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
    before = set(sys.modules)
    monkeypatch.syspath_prepend(ptk_b200._SHIM)
    yield
    for name in set(sys.modules) - before:
        if name == "pytorch3d" or name.startswith("pytorch3d."):
            del sys.modules[name]


def same_bits(a, b):
    a, b = a.detach().cpu().contiguous(), b.detach().cpu().contiguous()
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


# ------------------------------------------------------------------------------------- clouds
def surface(golden, B, S, seed=0):
    """samples of the golden object mesh (ops.sample_points), scaled per cloud"""
    m = golden("meshes")
    v = torch.from_numpy(m["obj0_verts"]).cuda()[None].repeat(B, 1, 1).contiguous()
    f = torch.from_numpy(m["obj0_faces"].astype(np.int32)).cuda()
    g = gen(seed)
    pts, _ = ops.sample_points(v, f, torch.rand(B, S, device="cuda", generator=g),
                               torch.rand(2, B, S, device="cuda", generator=g))
    return (pts * torch.linspace(1.0, 3.0, B, device="cuda")[:, None, None]).contiguous()


def cube(B, P, seed=0):
    return torch.rand(B, P, 3, device="cuda", generator=gen(seed))


def plane(B, P, seed=0):
    """exact planes: z = 0 in the first cloud, x = 0.25 in the second"""
    x = torch.rand(B, P, 3, device="cuda", generator=gen(seed))
    x[0, :, 2] = 0.0
    if B > 1:
        x[1, :, 0] = 0.25
    return x


def tiled(B, P, seed=0):
    """every point four times, as the touch loader duplicates points"""
    return cube(B, P // 4, seed).repeat(1, 4, 1).contiguous()


# ------------------------------------------------------------------------------------- forward
def check_forward(x, lengths, K):
    """estimate_local_frames / estimate_normals against the fp64 restatement on the GPU's idx; returns the fraction of
    valid queries whose normal was angle-checked."""
    B, P, _ = x.shape
    curv, frames = ops.estimate_local_frames(x, lengths, K)
    normals = ops.estimate_normals(x, lengths, K)
    assert same_bits(normals, frames[..., 0])
    l = lengths if lengths is not None else torch.full((B,), P, device="cuda")
    _, idx = ops.knn(x, x, K, l, l)
    xc, ic, lc = x.double().cpu(), idx.cpu(), l.cpu()
    lam, V = ref.frames_f64(xc, ic, lc, disambiguate=False)
    _, Fd = ref.frames_f64(xc, ic, lc, disambiguate=True)
    valid = torch.arange(P)[None] < lc.clamp(0, P)[:, None]
    f, c = frames.double().cpu(), curv.double().cpu()
    assert not f[~valid].any() and not c[~valid].any()
    # unit length and orthonormal everywhere
    eye = torch.eye(3, dtype=torch.float64)
    assert (f[valid].transpose(1, 2) @ f[valid] - eye).abs().max() <= 1e-6
    # angle bounds from the gaps of the reference's eigenvalues
    l0, l1, l2 = lam[..., 0], lam[..., 1], lam[..., 2]
    with np.errstate(all="ignore"):
        b0 = 64 * U * l2 / (l1 - l0)
        b2 = 64 * U * l2 / (l2 - l1)
    ok0, ok2 = valid & (b0 < 1e-2), valid & (b2 < 1e-2)
    sin0 = torch.linalg.cross(f[..., 0], V[..., 0], dim=-1).norm(dim=-1)
    sin2 = torch.linalg.cross(f[..., 2], V[..., 2], dim=-1).norm(dim=-1)
    assert (sin0[ok0] <= b0[ok0]).all(), float((sin0[ok0] / b0[ok0]).max())
    assert (sin2[ok2] <= b2[ok2]).all(), float((sin2[ok2] / b2[ok2]).max())
    assert ((c - lam).abs() <= 256 * U * l2[..., None] + 1e-30)[valid].all()
    # signs where the sign rule's margin exceeds the slots within rounding (plus the angle bound) of zero
    margin, near = ref.sign_margins(xc, ic, lc, V, torch.stack([b0, b2], -1).nan_to_num(1.0))
    for col, okc, m in ((0, ok0, 0), (2, ok2, 1)):
        sure = okc & (margin[..., m] > near[..., m])
        agree = (f[..., col] * Fd[..., col]).sum(-1) > 0
        assert agree[sure].all()
    return float(ok0.sum()) / max(float(valid.sum()), 1.0)


@pytest.mark.parametrize("K", [8, 50])
def test_forward_surface_samples(golden, K):
    assert check_forward(surface(golden, 3, 4000), None, K) > 0.9


@pytest.mark.parametrize("K", [1, 2, 8, 50, 64])
def test_forward_cube(K):
    frac = check_forward(cube(2, 3000, seed=K), None, K)
    assert K < 8 or frac > 0.5


@pytest.mark.parametrize("K", [8, 50])
def test_forward_exact_planes(K):
    x = plane(2, 2000)
    assert check_forward(x, None, K) > 0.99
    n = ops.estimate_normals(x, None, K)
    assert (n[0, :, 2].abs() == 1).all() and (n[1, :, 0].abs() == 1).all()


@pytest.mark.parametrize("K", [8, 50])
def test_forward_tiled(K):
    check_forward(tiled(2, 4000), None, K)


@pytest.mark.parametrize("K", [2, 8, 50, 64])
def test_forward_ragged_with_nan_padding(K):
    x = cube(5, 3000, seed=3)
    lengths = torch.tensor([3000, 1700, 40, 1, 0], device="cuda")  # l <= K in the last three clouds
    x[1, 1700:] = float("nan")
    x[2, 40:] = float("nan")
    x[3, 1:] = float("inf")
    x[4] = float("nan")
    check_forward(x, lengths, K)


@pytest.mark.parametrize("K", [8, 50])
def test_forward_clouds_smaller_than_k(K):
    x = cube(3, 40, seed=4)
    check_forward(x, torch.tensor([40, K, K - 1], device="cuda"), K)


def test_forward_bits(golden):
    x = surface(golden, 3, 3000, seed=5)
    K = 50
    c0, f0 = ops.estimate_local_frames(x, None, K)
    c1, f1 = ops.estimate_local_frames(x, None, K)
    assert same_bits(c0, c1) and same_bits(f0, f1)
    # a cloud alone, inside another batch, and as a ragged slice with garbage padding
    ca, fa = ops.estimate_local_frames(x[1:2].contiguous(), None, K)
    assert same_bits(ca[0], c0[1]) and same_bits(fa[0], f0[1])
    pad = torch.cat([x[1:2], torch.full((1, 700, 3), float("nan"), device="cuda")], 1)
    big = torch.cat([torch.cat([x[0:1], x[0:1, :700]], 1), pad], 0).contiguous()
    cs, fs = ops.estimate_local_frames(big, torch.tensor([3700, 3000], device="cuda"), K)
    assert same_bits(cs[1, :3000], c0[1]) and same_bits(fs[1, :3000], f0[1])
    # with requires_grad, and normals against frames[..., 0]
    cg, fg = ops.estimate_local_frames(x.clone().requires_grad_(True), None, K)
    assert same_bits(cg, c0) and same_bits(fg, f0)
    n = ops.estimate_normals(x.clone().requires_grad_(True), None, K)
    assert same_bits(n, f0[..., 0])
    for dis in (True, False):
        c, f = ops.estimate_local_frames(x, None, K, dis)
        assert same_bits(ops.estimate_normals(x, None, K, dis), f[..., 0])


@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_non_finite_point_affects_only_itself(bad):
    x = cube(1, 2000, seed=6)
    far = x.clone()
    far[0, 17] = 1e6   # a finite point no other query picks
    bx = x.clone()
    bx[0, 17] = float(bad)
    cf, ff = ops.estimate_local_frames(far, None, 16)
    cb, fb = ops.estimate_local_frames(bx, None, 16)
    assert torch.isnan(cb[0, 17]).all() and torch.isnan(fb[0, 17]).all()
    assert torch.isnan(ops.estimate_normals(bx, None, 16)[0, 17]).all()
    keep = torch.arange(2000, device="cuda") != 17
    assert same_bits(cf[0, keep], cb[0, keep]) and same_bits(ff[0, keep], fb[0, keep])


# ------------------------------------------------------------------------------------- backward
def masked_grads(x, lengths, K, dis, which, seed=0):
    """upstream gradients (normals, curvatures, frames; None where unused), zero on queries whose gap bound or sign
    margin fails, and the matching gradients for the reference (columns signed as the reference's eigenvectors)."""
    B, P, _ = x.shape
    l = lengths if lengths is not None else torch.full((B,), P, device="cuda")
    _, idx = ops.knn(x, x, K, l, l)
    xc, ic, lc = x.double().cpu(), idx.cpu(), l.cpu()
    lam, V = ref.frames_f64(xc, ic, lc, disambiguate=False)
    _, f = ops.estimate_local_frames(x, lengths, K, dis)
    f = f.double().cpu()
    with np.errstate(all="ignore"):
        b0 = 64 * U * lam[..., 2] / (lam[..., 1] - lam[..., 0])
        b2 = 64 * U * lam[..., 2] / (lam[..., 2] - lam[..., 1])
        b1 = 64 * U * lam[..., 2] / torch.minimum(lam[..., 1] - lam[..., 0], lam[..., 2] - lam[..., 1])
    good = (b1 < 1e-3) if which != "normals" else (b0 < 1e-3)
    if dis:
        margin, near = ref.sign_margins(xc, ic, lc, V, torch.stack([b0, b2], -1).nan_to_num(1.0))
        good &= margin[..., 0] > near[..., 0]
        if which != "normals":
            good &= margin[..., 1] > near[..., 1]
    g = torch.Generator().manual_seed(seed)
    gn = torch.randn(B, P, 3, generator=g, dtype=torch.float64) * good[..., None]
    gc = torch.randn(B, P, 3, generator=g, dtype=torch.float64) * good[..., None]
    gf = torch.randn(B, P, 3, 3, generator=g, dtype=torch.float64) * good[..., None, None]
    s = torch.ones(B, P, 1, 3, dtype=torch.float64)
    if not dis:  # the upstream gradient of an undisambiguated column follows its sign
        s = torch.where((f * V).sum(-2, keepdim=True) < 0, -1.0, 1.0)
    use = {"normals": (gn, None, None), "frames": (None, gc, gf), "curvatures": (None, gc, None)}[which]
    return use, s, float(good.sum()) / float((torch.arange(P)[None] < lc[:, None]).sum())


def gpu_grad(x, lengths, K, dis, which, use):
    xr = x.clone().requires_grad_(True)
    gn, gc, gf = (u.float().cuda() if u is not None else None for u in use)
    if which == "normals":
        loss = (ops.estimate_normals(xr, lengths, K, dis) * gn).sum()
    else:
        c, f = ops.estimate_local_frames(xr, lengths, K, dis)
        loss = (c * gc).sum() + ((f * gf).sum() if gf is not None else 0)
    loss.backward()
    return xr.grad


def ref_grad(x, lengths, K, dis, use, s):
    B, P, _ = x.shape
    l = lengths if lengths is not None else torch.full((B,), P, device="cuda")
    _, idx = ops.knn(x, x, K, l, l)
    xr = x.double().cpu().requires_grad_(True)
    c, f = ref.frames_f64(xr, idx.cpu(), l.cpu(), dis)
    gn, gc, gf = use
    loss = 0
    if gn is not None:
        loss = loss + (f[..., 0] * gn * s[..., 0, 0:1]).sum()
    if gc is not None:
        loss = loss + (c * gc).sum()
    if gf is not None:
        loss = loss + (f * gf * s).sum()
    loss.backward()
    return xr.grad


@pytest.mark.parametrize("flag", ["default", "det"])
@pytest.mark.parametrize("dis", [True, False])
@pytest.mark.parametrize("which", ["normals", "curvatures", "frames"])
def test_backward_against_fp64_autograd(golden, request, flag, dis, which):
    if flag == "det":
        request.getfixturevalue("det")
    x = surface(golden, 2, 1500, seed=7)
    lengths = torch.tensor([1500, 900], device="cuda")
    x[1, 900:] = float("nan")
    K = 16
    use, s, frac = masked_grads(x, lengths, K, dis, which)
    assert frac > 0.1
    got = gpu_grad(x, lengths, K, dis, which, use).double().cpu()
    want = ref_grad(x, lengths, K, dis, use, s)
    assert not got[1, 900:].any()
    err = (got - want).abs().max() / want.abs().max()
    assert err < 2e-3, float(err)


def test_backward_det_bits(golden, det):
    K = 16
    x = cube(2, 2000, seed=8)   # tie-free: no two distances from a query are equal
    g = torch.randn(2, 2000, 3, device="cuda", generator=gen(9))

    def grad(pts, up, lengths=None):
        xr = pts.clone().requires_grad_(True)
        (ops.estimate_normals(xr, lengths, K) * up).sum().backward()
        return xr.grad

    a = grad(x, g)
    assert same_bits(a, grad(x, g))
    # cloud 1 alone, and as a ragged slice with garbage padding
    assert same_bits(grad(x[1:2].contiguous(), g[1:2])[0], a[1])
    xs = torch.cat([x[1:2], torch.full((1, 500, 3), float("nan"), device="cuda")], 1)
    gs = torch.cat([g[1:2], torch.randn(1, 500, 3, device="cuda")], 1)
    sl = grad(xs, gs, torch.tensor([2000], device="cuda"))
    assert same_bits(sl[0, :2000], a[1]) and not sl[0, 2000:].any()
    # a permutation of the points permutes the gradient bit for bit
    perm = torch.randperm(2000, generator=torch.Generator().manual_seed(0)).cuda()
    assert same_bits(grad(x[:, perm].contiguous(), g[:, perm]), a[:, perm])


# ------------------------------------------------------------------------------------- the whole chain
@pytest.mark.parametrize("flag", ["default", "det"])
def test_chain_mesh_samples_chamfer_normals(golden, shim, request, flag):
    if flag == "det":
        request.getfixturevalue("det")
    from pytorch3d.loss import chamfer_distance
    from pytorch3d.ops import estimate_pointcloud_normals
    m = golden("meshes")
    verts = torch.from_numpy(m["obj0_verts"]).cuda()[None].repeat(2, 1, 1).contiguous()
    faces = torch.from_numpy(m["obj0_faces"].astype(np.int32)).cuda()
    gt = surface(golden, 2, 3000, seed=10) * 1.05
    u = torch.rand(2, 2500, device="cuda", generator=gen(11))
    uv = torch.rand(2, 2, 2500, device="cuda", generator=gen(12))

    def run(by_hand):
        v = verts.clone().requires_grad_(True)
        y = gt.clone().requires_grad_(True)
        pts, _, nrm = ops.sample_points(v, faces, u, uv, return_normals=True)
        if by_hand:
            cham, cham_n, _, _ = ops.chamfer_normals(pts, y, nrm, ops.estimate_normals(y, None, 50))
            cham, cham_n = cham.sum() / 2, cham_n.sum() / 2
        else:
            cham, cham_n = chamfer_distance(pts, y, x_normals=nrm, y_normals=estimate_pointcloud_normals(y))
        (cham + 0.1 * cham_n).backward()
        return cham, cham_n, v.grad, y.grad

    a, b = run(False), run(True)
    assert same_bits(a[0], b[0]) and same_bits(a[1], b[1])
    for ga, gb in zip(a[2:], b[2:]):
        assert torch.isfinite(ga).all() and ga.abs().max() > 0
        if flag == "det":
            assert same_bits(ga, gb)
        else:
            assert (ga - gb).abs().max() <= 1e-5 * gb.abs().max()


@pytest.mark.parametrize("flag", ["default", "det"])
def test_cuda_graph_replay_with_lengths_changed_in_place(request, flag):
    if flag == "det":
        request.getfixturevalue("det")
    K = 16
    x = cube(2, 1200, seed=13).requires_grad_(True)
    g = torch.randn(2, 1200, 3, device="cuda", generator=gen(14))
    lengths = torch.tensor([1200, 700], device="cuda")

    def step():
        n = ops.estimate_normals(x, lengths, K)
        gx, = torch.autograd.grad((n * g).sum(), x)
        return n, gx

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        n_out, g_out = step()
    for new in ([1200, 700], [300, 1200], [5, 0]):
        lengths.copy_(torch.tensor(new, device="cuda"))
        graph.replay()
        torch.cuda.synchronize()
        n_ref, g_ref = step()
        assert same_bits(n_out, n_ref)
        if flag == "det":
            assert same_bits(g_out, g_ref)
        else:
            assert (g_out - g_ref).abs().max() <= 1e-5 * max(float(g_ref.abs().max()), 1e-30)


def test_no_host_sync(shim):
    from pytorch3d.ops import estimate_pointcloud_local_coord_frames
    x = cube(2, 1500, seed=15).requires_grad_(True)
    lengths = torch.tensor([1500, 800], device="cuda")
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        n = ops.estimate_normals(x, lengths, 50)
        c, f = estimate_pointcloud_local_coord_frames(x, neighborhood_size=50)
        (n.sum() + c.sum() + f.sum()).backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.isfinite(x.grad).all()
