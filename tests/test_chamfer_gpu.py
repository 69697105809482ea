"""GPU parity of the Chamfer / 1-NN kernels (through the C ABI) against the CPU oracle and the golden
vectors.  Bar: indices bit-exact, values/gradients within 1e-5 relative (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

import ptk_b200

pytestmark = pytest.mark.gpu
TOL = 1e-5  # relative, FP32 (north_star)


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.fixture(params=["filter", "pruned"])
def algo(request):
    """Run the test under the brute-force filter scan and under the pruned (cell-sorted + box hierarchy) scan: both must
    reproduce the oracle bit for bit."""
    ptk_b200.ops.set_chamfer_algo(request.param)
    yield request.param
    ptk_b200.ops.set_chamfer_algo("auto")


def run(x, y, grad=None):
    xt = torch.from_numpy(x).cuda().requires_grad_(grad is not None)
    yt = torch.from_numpy(y).cuda().requires_grad_(grad is not None)
    cham, ix, iy = ptk_b200.ops.chamfer(xt, yt)
    out = [cham.detach().cpu().numpy(), ix.cpu().numpy(), iy.cpu().numpy()]
    if grad is not None:
        (cham * torch.from_numpy(grad).cuda()).sum().backward()
        out += [xt.grad.cpu().numpy(), yt.grad.cpu().numpy()]
    return out


def test_config1_golden(golden, oracle, algo):
    g = golden("chamfer")
    cham, ix, iy = run(g["c1_x"], g["c1_y"])
    assert np.array_equal(ix, g["c1_fma_idx_x"]) and np.array_equal(iy, g["c1_fma_idx_y"])
    assert np.array_equal(ix, g["c1_idx_x"]) and np.array_equal(iy, g["c1_idx_y"])  # torch restatement
    assert rel_err(cham, g["c1_cham"]) < TOL
    # distances are bit-exact against the FMA-order oracle
    d, i = ptk_b200.ops.knn1(torch.from_numpy(g["c1_x"]).cuda(), torch.from_numpy(g["c1_y"]).cuda())
    od, oi = oracle.knn1(g["c1_x"], g["c1_y"], use_fma=True)
    assert np.array_equal(d.cpu().numpy(), od) and np.array_equal(i.cpu().numpy(), oi)


def test_ties_golden(golden, algo):
    g = golden("chamfer")
    cham, ix, iy = run(g["tie_x"], g["tie_y"])
    assert np.array_equal(ix, g["tie_idx_x"]) and np.array_equal(iy, g["tie_idx_y"])
    assert rel_err(cham, g["tie_cham"]) < TOL


def test_unequal_sizes_gradients_golden(golden):
    g = golden("chamfer")
    cham, ix, iy, gx, gy = run(g["ne_x"], g["ne_y"], g["ne_gcham"])
    assert rel_err(cham, g["ne_cham"]) < TOL
    assert rel_err(gx, g["ne_gx"]) < TOL and rel_err(gy, g["ne_gy"]) < TOL


@pytest.mark.parametrize("B,P1,P2", [(1, 1, 1), (1, 1, 37), (2, 255, 257), (3, 2048, 2049), (1, 4097, 1000),
                                     (5, 1000, 4000), (64, 16, 16), (1, 10000, 6400), (2, 30000, 512)])
def test_random_vs_oracle(oracle, algo, B, P1, P2):
    rng = np.random.default_rng(B * 100003 + P1 * 17 + P2)
    x = (rng.random((B, P1, 3), np.float32) - 0.5).astype(np.float32)
    y = (rng.random((B, P2, 3), np.float32) - 0.5).astype(np.float32)
    gc = rng.random(B).astype(np.float32)
    cham, ix, iy, gx, gy = run(x, y, gc)
    ocham, odx, oix, ody, oiy = oracle.chamfer_fwd(x, y, use_fma=True)
    assert np.array_equal(ix, oix) and np.array_equal(iy, oiy)
    assert rel_err(cham, ocham) < TOL
    ogx, ogy = oracle.chamfer_bwd(x, y, oix, oiy, gc)
    assert rel_err(gx, ogx) < TOL and rel_err(gy, ogy) < TOL


def test_duplicate_points_and_grid_ties(oracle, algo):
    # integer lattice: masses of exact ties; lowest index must win everywhere
    rng = np.random.default_rng(7)
    x = rng.integers(0, 4, (2, 3000, 3)).astype(np.float32)
    y = rng.integers(0, 4, (2, 2500, 3)).astype(np.float32)
    cham, ix, iy = run(x, y)
    ocham, _, oix, _, oiy = oracle.chamfer_fwd(x, y, use_fma=True)
    assert np.array_equal(ix, oix) and np.array_equal(iy, oiy)
    assert rel_err(cham, ocham) < TOL


def _clouds(kind, rng, B, P1, P2):
    """Adversarial inputs for the expansion filter (chamfer_scan.cuh)."""
    if kind == "far_from_origin":      # translation to the box centre must absorb the offset
        c = np.array([1000.0, -250.0, 40.0], np.float32)
        return (c + 0.01 * rng.standard_normal((B, P1, 3))).astype(np.float32), \
               (c + 0.01 * rng.standard_normal((B, P2, 3))).astype(np.float32)
    if kind == "tiled_x4":             # data_loaders.py:80-87 tiles short clouds: exact duplicates far apart
        base = rng.random((B, P2 // 4, 3), np.float32)
        return rng.random((B, P1, 3), np.float32), np.concatenate([base] * 4, 1)
    if kind == "thin_rod":             # config-1-like: tiny NN distances compared with the extent
        x = rng.random((B, P1, 3), np.float32) * np.array([0.004, 0.01, 0.19], np.float32)
        y = rng.random((B, P2, 3), np.float32) * np.array([0.004, 0.01, 0.19], np.float32)
        return x.astype(np.float32), y.astype(np.float32)
    if kind == "huge_values":          # squares overflow: filter must switch itself off
        return (rng.standard_normal((B, P1, 3)) * 1e19).astype(np.float32), \
               (rng.standard_normal((B, P2, 3)) * 1e19).astype(np.float32)
    if kind == "tiny_values":          # squares underflow
        return (rng.standard_normal((B, P1, 3)) * 1e-20).astype(np.float32), \
               (rng.standard_normal((B, P2, 3)) * 1e-20).astype(np.float32)
    if kind == "one_outlier":          # a single far point inflates the radius (and the threshold)
        x = rng.random((B, P1, 3), np.float32); y = rng.random((B, P2, 3), np.float32)
        x[:, 0] = 1e4
        return x, y
    if kind == "identical":            # x == y: every query has distance 0 to itself
        x = rng.random((B, P1, 3), np.float32)
        return x, x.copy()
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["far_from_origin", "tiled_x4", "thin_rod", "huge_values", "tiny_values",
                                  "one_outlier", "identical"])
@pytest.mark.parametrize("B,P1,P2", [(2, 1500, 2000), (1, 4000, 4000)])
def test_filter_adversarial_vs_oracle(oracle, algo, kind, B, P1, P2):
    rng = np.random.default_rng(sum(map(ord, kind)) + P1)
    if kind == "identical":
        P2 = P1
    x, y = _clouds(kind, rng, B, P1, P2)
    cham, ix, iy = run(x, y)
    ocham, odx, oix, ody, oiy = oracle.chamfer_fwd(x, y, use_fma=True)
    assert np.array_equal(ix, oix) and np.array_equal(iy, oiy)
    d, i = ptk_b200.ops.knn1(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
    assert np.array_equal(d.cpu().numpy(), odx) and np.array_equal(i.cpu().numpy(), oix)  # distances bit-exact
    if np.isfinite(ocham).all():
        assert rel_err(cham, ocham) < TOL


def test_non_finite_inputs_take_the_exact_path(oracle, algo):
    rng = np.random.default_rng(11)
    x = rng.random((2, 700, 3), np.float32); y = rng.random((2, 900, 3), np.float32)
    x[0, 5, 1] = np.nan; y[0, 17, 0] = np.inf; y[1, 3, 2] = -np.inf
    _, ix, iy = run(x, y)
    _, _, oix, _, oiy = oracle.chamfer_fwd(x, y, use_fma=True)
    assert np.array_equal(ix, oix) and np.array_equal(iy, oiy)


def test_filter_and_exact_algorithms_agree_bitwise():
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand(8, 5000, 3, device="cuda", generator=g) - 0.5
    y = torch.rand(8, 7000, 3, device="cuda", generator=g) - 0.5
    try:
        ptk_b200.ops.set_chamfer_algo("exact")
        c0, ix0, iy0 = ptk_b200.ops.chamfer(x, y)
        d0, i0 = ptk_b200.ops.knn1(x, y)
        ptk_b200.ops.set_chamfer_algo("filter")
        c1, ix1, iy1 = ptk_b200.ops.chamfer(x, y)
        d1, i1 = ptk_b200.ops.knn1(x, y)
        n = ptk_b200.ops.chamfer_rescued(x, y)
    finally:
        ptk_b200.ops.set_chamfer_algo("auto")
    assert torch.equal(ix0, ix1) and torch.equal(iy0, iy1) and torch.equal(c0, c1)
    assert torch.equal(d0, d1) and torch.equal(i0, i1)
    assert 0 < n < 0.05 * 8 * 12000   # uniform clouds: ~1 % of the queries need the exact rescue


def _surface(B, P, g, noise=0.0):
    p = torch.nn.functional.normalize(torch.randn(B, P, 3, device="cuda", generator=g), dim=-1) * 0.25
    return p * (1 + noise * torch.randn(B, P, 1, device="cuda", generator=g)) if noise else p


@pytest.mark.parametrize("kind,B,P1,P2", [("cube", 256, 10000, 10000), ("surface", 64, 10000, 10000), ("surface", 2, 100000, 100000),
                                          ("cube", 1, 70000, 33000), ("clustered", 3, 6000, 9000), ("lattice", 2, 20000, 20000),
                                          ("surface", 66, 33000, 33500),   # > 64 pairs of > 32k points: one CTA per cloud, 32^3 cells
                                          ("cube", 70, 17000, 20000)])     # > 64 pairs, 16k..32k points: cell ranks recomputed
def test_pruned_scan_equals_the_brute_force_scan_at_full_size(kind, B, P1, P2):
    """Sizes the CPU oracle cannot reach (BASELINE config 3 / 5 shapes): the pruned scan must return the brute-force
    scan's indices, distances and Chamfer values bit for bit, whatever the distribution -- volume, surface samples,
    tight clusters (the uniform grid cannot separate them: the scan cap hands those queries to the exact rescue scan)
    and a lattice with thousands of exact ties per query."""
    g = torch.Generator(device="cuda").manual_seed(P1 + B)
    if kind == "cube":
        x, y = torch.rand(B, P1, 3, device="cuda", generator=g) - 0.5, torch.rand(B, P2, 3, device="cuda", generator=g) - 0.5
    elif kind == "surface":
        x, y = _surface(B, P1, g, 0.02), _surface(B, P2, g)
    elif kind == "clustered":
        x = torch.rand(B, P1, 3, device="cuda", generator=g)
        y = torch.rand(B, P2, 3, device="cuda", generator=g) * 0.01
        y[:, ::2] += 0.9
    else:
        x = torch.randint(0, 10, (B, P1, 3), device="cuda", generator=g).float() * 0.125
        y = torch.randint(0, 10, (B, P2, 3), device="cuda", generator=g).float() * 0.125
    out = {}
    try:
        for name in ("filter", "pruned"):
            ptk_b200.ops.set_chamfer_algo(name)
            out[name] = ptk_b200.ops.chamfer(x, y) + ptk_b200.ops.knn1(y, x)
            if name == "pruned":
                rescued = ptk_b200.ops.chamfer_rescued(x, y)
    finally:
        ptk_b200.ops.set_chamfer_algo("auto")
    for a, b in zip(out["filter"], out["pruned"]):
        assert torch.equal(a, b)
    if kind == "clustered":
        assert rescued > 0          # the cap fired: those queries took the exact scan
    elif kind != "lattice":
        assert rescued == 0


def test_auto_picks_the_pruned_scan_for_large_clouds_only():
    """PTK_CHAMFER_AUTO (the default): brute-force filter scan below PTK_CHAMFER_AUTO_MIN_POINTS (20000) points per cloud
    -- the named 10k configs stay on the kernel north_star specifies and the roofline is quoted on -- pruned at and above.
    The filter queues ~0.3 % of its queries for the rescue scan on uniform clouds, the pruned scan none: that tells
    which one ran."""
    assert ptk_b200._lib.lib().ptk_chamfer_get_algo() == ptk_b200._lib.CHAMFER_AUTO
    g = torch.Generator(device="cuda").manual_seed(3)
    small = [torch.rand(2, 12000, 3, device="cuda", generator=g) for _ in range(2)]
    large = [torch.rand(1, 20000, 3, device="cuda", generator=g) for _ in range(2)]
    mixed = [large[0], small[0][:1].contiguous()]
    assert ptk_b200.ops.chamfer_rescued(*small) > 0
    assert ptk_b200.ops.chamfer_rescued(*large) == 0
    assert ptk_b200.ops.chamfer_rescued(*mixed) > 0     # both clouds have to be large


def test_only_y_needs_grad(oracle):
    # autoencoder case (reconstruction/autoencoder/train.py:145-151): sampled cloud detached
    rng = np.random.default_rng(3)
    x = rng.random((2, 500, 3), np.float32)
    y = rng.random((2, 640, 3), np.float32)
    xt = torch.from_numpy(x).cuda()
    yt = torch.from_numpy(y).cuda().requires_grad_(True)
    cham, ix, iy = ptk_b200.ops.chamfer(xt, yt)
    cham.sum().backward()
    _, ogy = oracle.chamfer_bwd(x, y, ix.cpu().numpy(), iy.cpu().numpy(), np.ones(2, np.float32), want_x=False)
    assert rel_err(yt.grad.cpu().numpy(), ogy) < TOL


def test_full_size_properties(algo):
    """BASELINE size (10k x 10k, batch 256): properties that need no oracle run."""
    B, P = 256, 10000
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(B, P, 3, device="cuda", generator=g) - 0.5
    y = torch.rand(B, P, 3, device="cuda", generator=g) - 0.5
    cham, ix, iy = ptk_b200.ops.chamfer(x, y)
    # (1) the reported index reproduces the reported distance: cham == mean |x - y[idx]|^2 + ...
    ar = torch.arange(B, device="cuda")[:, None]
    dx = ((x - y[ar, ix.long()]) ** 2).sum(-1).mean(1)
    dy = ((y - x[ar, iy.long()]) ** 2).sum(-1).mean(1)
    assert torch.allclose(cham, dx + dy, rtol=1e-5)
    # (2) symmetry: swapping the clouds swaps the index sets and keeps the value
    cham2, jx, jy = ptk_b200.ops.chamfer(y, x)
    assert torch.equal(jx, iy) and torch.equal(jy, ix) and torch.allclose(cham, cham2, rtol=1e-6)
    # (3) identity: chamfer(x, x) == 0 with idx == arange
    cham0, kx, _ = ptk_b200.ops.chamfer(x[:8], x[:8])
    assert float(cham0.abs().max()) == 0.0
    assert torch.equal(kx, torch.arange(P, device="cuda", dtype=torch.int32).expand(8, P))
    # (4) batch independence: a slice of the batch gives bit-identical results
    c_s, ix_s, _ = ptk_b200.ops.chamfer(x[100:103].contiguous(), y[100:103].contiguous())
    assert torch.equal(ix_s, ix[100:103]) and torch.equal(c_s, cham[100:103])
    # (5) optimality spot check against a torch brute force on a few query points
    q = x[5, :64]
    d = ((q[:, None, :] - y[5][None]) ** 2).sum(-1)
    assert torch.equal(d.argmin(1).int(), ix[5, :64])


def test_errors():
    with pytest.raises(ValueError):
        ptk_b200.ops.chamfer(torch.rand(2, 10, 2).cuda(), torch.rand(2, 10, 3).cuda())
    with pytest.raises(ValueError):
        ptk_b200.ops.chamfer(torch.rand(2, 10, 3).cuda(), torch.rand(3, 10, 3).cuda())
    with pytest.raises(ValueError):
        ptk_b200.ops.chamfer(torch.rand(2, 0, 3).cuda(), torch.rand(2, 10, 3).cuda())


def test_pytorch3d_shim_call_shape(golden):
    ptk_b200.install_pytorch3d_shim()
    from pytorch3d.loss import chamfer_distance as cuda_cd
    from pytorch3d.ops import knn_points
    g = golden("chamfer")
    x, y = torch.from_numpy(g["ne_x"]).cuda(), torch.from_numpy(g["ne_y"]).cuda()
    cd, none = cuda_cd(x, y, batch_reduction=None)  # utils.py:207 unpacks a tuple
    assert none is None and cd.shape == (3,)
    assert rel_err(cd.cpu().numpy(), g["ne_cham"]) < TOL
    k = knn_points(x, y, K=1)
    assert k.dists.shape == (3, 700, 1) and k.idx.dtype == torch.int64
