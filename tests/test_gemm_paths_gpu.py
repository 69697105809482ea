"""Every GEMM path of the per-vertex linear layers against a scalar reference, at its tile, split and alignment edges.

(a) Exact paths (PTK_GEMM_FFMA forward and dgrad, the fused split forward, the generic kernel): bit-equal
    (torch.equal) to the scalar FMA loop of oracle.gemm_fma_seq on sampled rows that include the first and last row of
    every row tile and the last row of the matrix.
(b) Tensor-core 3xTF32 and split-K paths: element-wise bound |D - D64| <= tau * (|A| . |B|), both in float64.
(c) The stream-K combine protocol: run-to-run bit identity, back-to-back calls on one workspace, CUDA-graph replay.

Shapes are derived from the device's SM count through the plan mirrors of tests/gemm_plans.py, and each test asserts
the path its shape reaches.  Development switches that the library reads once per process (PTK_FWD_NO_TMA,
PTK_FWD_BM, PTK_TG_PAIR) are covered by running this file as a script in a child interpreter:
    python tests/test_gemm_paths_gpu.py exact|tc
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import gemm_plans as gp  # noqa: E402
import ptk_b200  # noqa: E402
from oracle import oracle as orc  # noqa: E402

_lib, ops = ptk_b200._lib, ptk_b200.ops
FFMA, TF32X3, AUTO = ops.GEMM_FFMA, ops.GEMM_TF32X3, ops.GEMM_AUTO
PAIR = int(os.environ.get("PTK_TG_PAIR", "0") or 0) in (1, 3)  # cluster forms of the tensor-core kernel
U = 2.0 ** -24                                                 # unit roundoff of fp32

pytestmark = pytest.mark.gpu


def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ------------------------------------------------------------------------------------------------------ helpers
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def at_offset(a):
    """Device copy of `a` (C-contiguous) whose data pointer is one float past a 16-byte boundary."""
    buf = torch.empty(a.size + 1, dtype=torch.float32, device="cuda")
    v = buf[1:].view(a.shape)
    v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    assert v.data_ptr() % 16 == 4
    return v


def rand(rng, *shape, scale=1.0):
    return (rng.standard_normal(shape) * scale).astype(np.float32)


def _ws(nbytes):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device="cuda")


def fwd(X, W, algo, ws=None, out=None):
    M, K = X.shape
    N = W.shape[1]
    L = _lib.lib()
    H = torch.empty(M, N, device="cuda") if out is None else out
    ws = _ws(L.ptk_gcn_linear_workspace_bytes(M, K, N)) if ws is None else ws
    _lib.check(L.ptk_gcn_linear_fwd(ops._p(X), ops._p(W), M, K, N, ops._p(H), algo, ops._p(ws), ws.numel(),
                                    ops._stream()), "ptk_gcn_linear_fwd")
    return H


def dgrad(gH, W, act, algo, act_bits=None, ws=None, out=None):
    """gX (M, Kin) = gH (M, Nout) . W^T, W (Kin, Nout) as stored, masked by act > 0."""
    M, N = gH.shape
    K = W.shape[0]
    L = _lib.lib()
    gX = torch.empty(M, K, device="cuda") if out is None else out
    ws = _ws(L.ptk_gcn_linear_workspace_bytes(M, K, N)) if ws is None else ws
    _lib.check(L.ptk_gcn_linear_dgrad(ops._p(gH), ops._p(W), ops._p(act), ops._p(act_bits), M, K, N, ops._p(gX), algo,
                                      ops._p(ws), ws.numel(), ops._stream()), "ptk_gcn_linear_dgrad")
    return gX


def wgrad(X, gH, algo):
    return ops._linear_wgrad(X, gH, algo_id=algo)


def fwd_split(X, W, n_split, x_bits=None):
    """ptk_gcn_linear_fwd_split with relu; columns [0, n_split) of `out` are left to the aggregation (NaN here)."""
    M, K = X.shape
    N = W.shape[1]
    head = torch.full((M, n_split), float("nan"), device="cuda")
    out = torch.full((M, N), float("nan"), device="cuda")
    _lib.check(_lib.lib().ptk_gcn_linear_fwd_split(ops._p(X), ops._p(W), M, K, N, n_split, ops._p(head), ops._p(out), 1,
                                                   ops._p(x_bits), ops._stream()), "ptk_gcn_linear_fwd_split")
    return head, out


def launches(fn):
    """(result of fn(), kernels the library launched for it)"""
    n0 = _lib.launch_count()
    r = fn()
    return r, _lib.launch_count() - n0


def pack_bits(act):
    """Packed ReLU mask of include/ptk.h (ptk_gcn_linear_fwd_split): bit (k & 31) of word [m, k >> 5] = act[m, k] > 0,
    bits beyond K zero."""
    M, K = act.shape
    wpr = gp.ceil_div(K, 32)
    b = np.zeros((M, wpr * 32), bool)
    b[:, :K] = act > 0
    return np.packbits(b, axis=1, bitorder="little").view("<u4").reshape(M, wpr)


def sample_rows(M, tiles, rng, extra=48):
    return np.array(gp.tile_edge_rows(M, tiles, rng.integers(0, M, extra)), np.int64)


def tc_tiles(M):
    return [(m0, gp.TG_BM) for m0 in range(0, M, gp.TG_BM)]


def assert_bits(got, want, what):
    """torch.equal (so -0 == +0) between device rows `got` and the oracle's `want`."""
    g = got.cpu() if isinstance(got, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(got))
    w = torch.from_numpy(np.ascontiguousarray(want))
    if not torch.equal(g, w):
        bad = (g != w).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{what}: {bad.shape[0]} of {w.numel()} elements differ from the scalar FMA loop, "
                             f"first at {i}: {g[i].item()!r} vs {w[i].item()!r}")


def tau_tf32x3(k_blocks, adds):
    """Element-wise bound of the 3xTF32 kernels relative to sum_k |a_k| |b_k| (csrc/gemm_tf32x3.cu):
    - split: a_hi = a rounded to TF32 (11 significant bits), so |a_lo| <= 2^-11 |a|; the tensor core truncates a_lo to
      TF32, an error <= 2^-10 |a_lo| <= 2^-21 |a|, and the same for b: 2 * 2^-21 per product; the dropped a_lo b_lo
      is <= 2^-22: 2.5 * 2^-21 per product in all.
    - TMEM accumulation of one 32-wide k-block: 12 MMAs add into an fp32 accumulator that truncates, each add off by
      <= 2^-23 of a partial sum that is itself <= the block's sum |a||b|: 12 * 2^-23 = 3 * 2^-21.
    - drain and combine: `k_blocks` fp32 additions of the chunks into registers plus `adds` more (the stream-K
      combine of a shared tile, or the split-K reduction), each <= 2^-24 of a partial sum <= sum |a||b|.
    Higher-order terms are below 2^-40 and covered by the slack of the first-order terms (e.g. the +0x1000 rounding
    makes |a_lo| <= 2^-11 |a| hold exactly)."""
    return 2.5 * 2.0 ** -21 + 3 * 2.0 ** -21 + (k_blocks + adds) * U


def gamma(n):
    """gamma_n = n u / (1 - n u): bound of any fp32 summation of n products with n roundings on any path."""
    return n * U / (1 - n * U)


def assert_bound(D, A, B, rows, tau, what, mask=None):
    """|D - D64| <= tau * (|A| . |B|) element-wise on `rows`; B is (K, N); mask (M, N) bool zeroes the reference and
    the bound, so masked outputs must be exactly 0.  Returns the largest err / (|A|.|B|) seen."""
    A64 = A[rows].astype(np.float64)
    B64 = B.astype(np.float64)
    ref = A64 @ B64
    mag = np.abs(A64) @ np.abs(B64)
    if mask is not None:
        ref = np.where(mask[rows], ref, 0.0)
        mag = np.where(mask[rows], mag, 0.0)
    got = (D[torch.from_numpy(rows).cuda()] if isinstance(D, torch.Tensor) else D[rows])
    got = (got.cpu().numpy() if isinstance(got, torch.Tensor) else got).astype(np.float64)
    err = np.abs(got - ref)
    ok = err <= tau * mag
    if not ok.all():
        i = np.argwhere(~ok)[0]
        raise AssertionError(f"{what}: {int((~ok).sum())} elements out of bound (tau = {tau:.3g}); at row {rows[i[0]]} "
                             f"col {i[1]}: got {got[tuple(i)]!r}, ref {ref[tuple(i)]!r}, |A||B| {mag[tuple(i)]!r}")
    return float((err / np.where(mag > 0, mag, 1.0)).max())


# ================================================================================ (a) exact paths: scalar FMA loop
def ffma_fwd_shapes(Q):
    """(M, N, K, what): the tail-tile table (rt_tail 1..8 at N = 300 and K = 300, 448), then the M, N and K edges."""
    shapes = [(gp.fwd_rows_for_rt_tail(rt, 300, Q), 300, K, f"rt_tail={rt}") for K in (300, 448) for rt in range(1, 9)]
    shapes += [(M, 164, 20, "M edge") for M in (1, 63, 64, 65)]
    shapes += [(65, N, 300, "N edge") for N in (64, 160, 164, 320)]
    shapes += [(63, 320, K, "K edge") for K in (4, 16, 20, 300, 448)]
    return shapes


def check_ffma_fwd(M, N, K, seed):
    """The exact forward (TMA kernel, or the register-staged kernel under PTK_FWD_NO_TMA / PTK_FWD_BM) on a shape it is
    eligible for: bit-equal to the scalar FMA loop."""
    assert K % 4 == 0 and N % 4 == 0 and N >= 64
    rng = np.random.default_rng(seed)
    X, W = rand(rng, M, K), rand(rng, K, N, scale=0.1)
    H, n = launches(lambda: fwd(dev(X), dev(W), FFMA))
    assert n == 1
    rows = sample_rows(M, gp.fwd_row_tiles(M, N, sm_count()), rng)
    assert_bits(H[torch.from_numpy(rows).cuda()], orc.gemm_fma_seq(X, W, rows=rows), f"FFMA forward {M}x{N}x{K}")


def fwd_split_shapes(Q):
    """(M, N, K, n_split): a 'cut' GCN layer (L = 99 of 300) at two tail heights, the 448-wide input, the narrowest
    eligible output, K = 4 and K beyond the mask's 512."""
    return [(gp.fwd_rows_for_rt_tail(5, 300, Q), 300, 300, 100), (gp.fwd_rows_for_rt_tail(2, 300, Q), 300, 448, 148),
            (65, 64, 20, 4), (1, 68, 4, 64), (200, 300, 516, 100)]


def check_fwd_split(M, N, K, Lp, seed):
    rng = np.random.default_rng(seed)
    X, W = rand(rng, M, K), rand(rng, K, N, scale=0.1)
    X[rng.random(X.shape) < 0.05] = 0.0
    X[0, :4] = [-0.0, 0.0, 1e-40, -1e-40]  # the mask is X > 0: -0 and +0 out, a positive subnormal in
    Xd, Wd = dev(X), dev(W)
    wpr = gp.ceil_div(K, 32)
    bits = torch.full((M, wpr), -1, dtype=torch.int32, device="cuda") if K <= 512 else None
    head, out = fwd_split(Xd, Wd, Lp, bits)
    rows = sample_rows(M, gp.fwd_row_tiles(M, N, sm_count()), rng)
    ri = torch.from_numpy(rows).cuda()
    H = orc.gemm_fma_seq(X, W, rows=rows)
    assert_bits(head[ri], H[:, :Lp], f"fwd_split head {M}x{N}x{K}")
    assert_bits(out[ri][:, Lp:], np.maximum(H[:, Lp:], 0.0), f"fwd_split relu(out) {M}x{N}x{K}")
    assert torch.isnan(out[:, :Lp]).all(), "fwd_split wrote into the columns left to the aggregation"
    if bits is not None:
        assert np.array_equal(bits.cpu().numpy().view(np.uint32), pack_bits(X)), "x_bits != packed X > 0"
    else:
        with pytest.raises(ValueError):
            fwd_split(Xd, Wd, Lp, torch.zeros((M, wpr), dtype=torch.int32, device="cuda"))


def ffma_dgrad_shapes(Q):
    """(M, Kin, Nout): a reconstruction-step layer with tail rows, the 448-wide input, odd and narrow widths, one row."""
    return [(gp.fwd_rows_for_rt_tail(3, 300, Q), 300, 300), (129, 448, 300), (65, 17, 36), (1, 63, 60), (130, 300, 18)]


def check_ffma_dgrad(M, Kin, Nout, seed, act=None):
    rng = np.random.default_rng(seed)
    G, W = rand(rng, M, Nout), rand(rng, Kin, Nout, scale=0.1)
    if act is None:
        act = rand(rng, M, Kin)
    rows = sample_rows(M, [(m0, 128) for m0 in range(0, M, 128)], rng)
    ref = orc.gemm_fma_seq(G, W, rows=rows, b_transposed=True)
    gX, n = launches(lambda: dgrad(dev(G), dev(W), None, FFMA))
    assert n == 1
    assert_bits(gX[torch.from_numpy(rows).cuda()], ref, f"FFMA dgrad {M}x{Kin}x{Nout}")
    gXm = dgrad(dev(G), dev(W), dev(act), FFMA)
    assert_bits(gXm[torch.from_numpy(rows).cuda()], np.where(act[rows] > 0, ref, 0.0).astype(np.float32),
                f"FFMA dgrad masked {M}x{Kin}x{Nout}")


def test_ffma_forward_is_the_scalar_fma_loop():
    Q = sm_count()
    for i, (M, N, K, what) in enumerate(ffma_fwd_shapes(Q)):
        if what.startswith("rt_tail"):
            assert gp.fwd_tma_plan(M, N, Q).rt_tail == int(what.split("=")[1])
        check_ffma_fwd(M, N, K, seed=i)


def test_fwd_split_is_the_scalar_fma_loop_and_packs_the_mask():
    for i, shape in enumerate(fwd_split_shapes(sm_count())):
        check_fwd_split(*shape, seed=100 + i)


@pytest.mark.parametrize("M,N,K,where", [(130, 161, 18, ""), (257, 300, 301, ""), (129, 63, 20, ""), (40, 8, 36, ""),
                                         (300, 300, 300, "X"), (65, 64, 20, "W"), (129, 160, 36, "H")])
def test_generic_forward_is_the_scalar_fma_loop(M, N, K, where):
    """sgemm_kernel: K % 4 != 0, N % 4 != 0 or N < 64 (N > 4), or a pointer one float off a 16-byte boundary."""
    rng = np.random.default_rng(M * N + K)
    X, W = rand(rng, M, K), rand(rng, K, N, scale=0.1)
    Xd = at_offset(X) if where == "X" else dev(X)
    Wd = at_offset(W) if where == "W" else dev(W)
    Hd = at_offset(np.zeros((M, N), np.float32)) if where == "H" else None
    H, n = launches(lambda: fwd(Xd, Wd, FFMA, out=Hd))
    assert n == 1
    assert where or K % 4 or N % 4 or N < 64  # not the TMA forward
    assert_bits(H, orc.gemm_fma_seq(X, W), f"generic forward {M}x{N}x{K} (offset {where or '-'})")
    if where in ("X", "H"):  # the tensor-core path refuses the misaligned pointer, AUTO falls back to the same kernel
        with pytest.raises(ValueError):
            fwd(Xd, Wd, TF32X3, out=Hd)
        if K >= 32 and N >= 16:
            assert_bits(fwd(Xd, Wd, AUTO, out=Hd), orc.gemm_fma_seq(X, W), "AUTO forward, misaligned")


def test_ffma_dgrad_is_the_scalar_fma_loop():
    for i, shape in enumerate(ffma_dgrad_shapes(sm_count())):
        check_ffma_dgrad(*shape, seed=200 + i)


def test_ffma_wgrad_is_the_split_fma_loop():
    """FFMA wgrad (split over rows, partials added in split order): bit-equal to the scalar loop per slab plus the
    fp32 reduction, and within gamma_M of the float64 product.  N <= 4 runs skinny_wgrad_kernel (clamped at 3 CTAs
    per SM), wider N the split sgemm_kernel."""
    Q = sm_count()
    for M, K, N in [(33, 300, 300), (1949, 36, 20), (31184, 64, 20), (7, 300, 1), (1949, 300, 3), (31184, 300, 4)]:
        rng = np.random.default_rng(M + K + N)
        X, G = rand(rng, M, K), rand(rng, M, N)
        gW = wgrad(dev(X), dev(G), FFMA).cpu().numpy()
        slabs = gp.ffma_wgrad_slabs(M, K, N, Q)
        if M == 31184 and N <= 4:
            assert len(slabs) == 3 * Q
        want = np.zeros((K, N), np.float32)
        for r0, r1 in slabs:
            if r1 > r0:
                want = want + orc.gemm_fma_seq(np.ascontiguousarray(X[r0:r1].T), G[r0:r1])
        assert_bits(gW, want, f"FFMA wgrad {M}x{K}x{N} ({len(slabs)} splits)")
        assert_bound(gW, np.ascontiguousarray(X.T), G, np.arange(K), gamma(M), f"FFMA wgrad {M}x{K}x{N}")


def test_skinny_forward_within_gamma():
    """N <= 4: one warp per row, lane-strided FMA chains and a warp reduction -- not k-sequential, bounded by gamma_K."""
    for M in (1, 7, 1949, 31184):
        for N in (1, 3, 4):
            K = 300
            rng = np.random.default_rng(M + N)
            X, W = rand(rng, M, K), rand(rng, K, N)
            for algo in (FFMA, AUTO):  # N < 16: not eligible for the tensor cores either
                H, n = launches(lambda: fwd(dev(X), dev(W), algo))
                assert n == 1
                assert_bound(H, X, W, np.arange(M), gamma(K), f"skinny forward {M}x{N}x{K}")


@pytest.mark.parametrize("env", ["PTK_FWD_NO_TMA=1", "PTK_FWD_BM=32", "PTK_FWD_BM=96", "PTK_FWD_BM=112",
                                 "PTK_FWD_BM=128"])
def test_exact_paths_in_child(env):
    """The register-staged forward (launch_fwd<BM>) and the non-TMA split forward: the same bit-level checks with the
    process-wide switches set in a child interpreter."""
    k, v = env.split("=")
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "exact"], env=dict(os.environ, **{k: v}),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "exact ok" in out.stdout, out.stdout + out.stderr


# ============================================================================= (b) tensor cores: element-wise bound
def tc_table(Q):
    """(M, N, K, name) of the tensor-core fwd / dgrad table: stream-K shapes (tiles below, equal to, one above and 3.3x
    the SM count; an odd row-tile count), then K, N and M edges."""
    sk = gp.tc_streamk_shapes(Q)
    shapes = [(M, N, K, name) for name, (M, N, K) in sk.items()]
    M33 = sk["x3.3"][0]
    shapes += [(M33, 300, 448, "x3.3"), (M33, 448, 300, "x3.3")]
    shapes += [(129, 161, K, "K edge") for K in (32, 36, 60, 300, 448)]
    shapes += [(127, N, 60, "N edge") for N in (16, 17, 63, 159, 160, 161, 300)]
    shapes += [(M, 17, 36, "M edge") for M in (1, 127, 128, 129)]
    seen, out = set(), []
    for s in shapes:
        if s[:3] not in seen:
            seen.add(s[:3])
            out.append(s)
    return out


def assert_tc_path(M, N, K, name, Q):
    """The stream-K plan the kernel runs for this shape shares tiles exactly when there are more tiles than CTAs."""
    plan = gp.tg_plan(M, N, K, Q, PAIR)
    tiles = gp.ceil_div(M, gp.TG_BM) * gp.ceil_div(N, gp.TG_BN)
    shared = gp.tg_shared_tiles(plan)
    if name in ("below", "equal") and not PAIR:
        assert tiles == {"below": Q - 1, "equal": Q}[name] and not shared
    if name in ("above", "odd", "x3.3"):
        assert shared and tiles > Q, (name, tiles, Q)
    if name == "odd":
        assert gp.ceil_div(M, gp.TG_BM) % 2 == 1
    return plan


def check_tc_fwd(M, N, K, name, seed):
    Q = sm_count()
    assert_tc_path(M, N, K, name, Q)
    rng = np.random.default_rng(seed)
    X, W = rand(rng, M, K), rand(rng, K, N, scale=0.1)
    H, n = launches(lambda: fwd(dev(X), dev(W), TF32X3))
    assert n == 2  # weight split + tensor-core GEMM
    rows = sample_rows(M, tc_tiles(M), rng)
    return assert_bound(H, X, W, rows, tau_tf32x3(gp.ceil_div(K, 32), 1), f"3xTF32 forward {M}x{N}x{K} ({name})")


def check_tc_dgrad(M, N, K, name, seed):
    """gX (M, N) = gH (M, K) . W^T with W (N, K): without a mask, and masked by a random act."""
    Q = sm_count()
    assert_tc_path(M, N, K, name, Q)
    rng = np.random.default_rng(seed)
    G, W, act = rand(rng, M, K), rand(rng, N, K, scale=0.1), rand(rng, M, N)
    Gd, Wd = dev(G), dev(W)
    rows = sample_rows(M, tc_tiles(M), rng)
    tau = tau_tf32x3(gp.ceil_div(K, 32), 1)
    gX, n = launches(lambda: dgrad(Gd, Wd, None, TF32X3))
    assert n == 2
    r = assert_bound(gX, G, np.ascontiguousarray(W.T), rows, tau, f"3xTF32 dgrad {M}x{N}x{K} ({name})")
    gXm, n = launches(lambda: dgrad(Gd, Wd, dev(act), TF32X3))
    assert n == 3  # + packing of the mask
    assert_bound(gXm, G, np.ascontiguousarray(W.T), rows, tau, f"3xTF32 dgrad masked {M}x{N}x{K} ({name})",
                 mask=act > 0)
    return r


@pytest.fixture(scope="module")
def tc_shapes():
    return tc_table(sm_count())


def test_tc_forward_within_bound(tc_shapes):
    for i, s in enumerate(tc_shapes):
        check_tc_fwd(*s, seed=300 + i)


def test_tc_dgrad_within_bound(tc_shapes):
    for i, s in enumerate(tc_shapes):
        check_tc_dgrad(*s, seed=400 + i)


def special_act(rng, M, K):
    """Activations with +0, -0, NaN, +-subnormals, +-Inf and ordinary values; numpy's act > 0 is the mask."""
    act = rand(rng, M, K)
    specials = np.array([0.0, -0.0, np.nan, 1e-40, -1e-40, 1.4e-45, np.inf, -np.inf], np.float32)
    pick = rng.random((M, K)) < 0.25
    act[pick] = specials[rng.integers(0, specials.size, int(pick.sum()))]
    act[0, :specials.size] = specials
    act[-1, -specials.size:] = specials
    return act


def check_dgrad_masks(M, Kin, Nout, name, seed):
    """One mask, three ways: packed from act by the tensor-core path, packed by fwd_split as x_bits, and read from act
    by the FFMA dgrad.  Masked outputs are exactly 0, the rest within the bound."""
    Q = sm_count()
    assert_tc_path(M, Kin, Nout, name, Q)
    rng = np.random.default_rng(seed)
    G, W, act = rand(rng, M, Nout), rand(rng, Kin, Nout, scale=0.1), special_act(rng, M, Kin)
    mask = act > 0
    Gd, Wd, actd = dev(G), dev(W), dev(act)
    bits = torch.zeros((M, gp.ceil_div(Kin, 32)), dtype=torch.int32, device="cuda")
    fwd_split(actd, dev(rand(rng, Kin, 64)), 32, bits)  # x_bits of the layer whose input is act
    assert np.array_equal(bits.cpu().numpy().view(np.uint32), pack_bits(act))
    from_act = dgrad(Gd, Wd, actd, TF32X3)
    from_bits, n = launches(lambda: dgrad(Gd, Wd, actd, TF32X3, act_bits=bits))
    assert n == 2  # no packing
    assert torch.equal(from_act, from_bits)
    rows = sample_rows(M, tc_tiles(M), rng)
    Wt = np.ascontiguousarray(W.T)
    assert_bound(from_act, G, Wt, rows, tau_tf32x3(gp.ceil_div(Nout, 32), 1), f"masked dgrad {M}x{Kin}x{Nout}",
                 mask=mask)
    assert ((from_act.cpu().numpy() == 0) | mask).all()
    ffma = dgrad(Gd, Wd, actd, FFMA)
    want = np.where(mask[rows], orc.gemm_fma_seq(G, W, rows=rows, b_transposed=True), 0.0).astype(np.float32)
    assert_bits(ffma[torch.from_numpy(rows).cuda()], want, f"FFMA masked dgrad {M}x{Kin}x{Nout}")


def test_dgrad_masks_agree_at_special_values():
    sk = gp.tc_streamk_shapes(sm_count())
    for i, name in enumerate(("x3.3", "above")):
        M, N, K = sk[name]
        check_dgrad_masks(M, N, K, name, seed=500 + i)
    check_dgrad_masks(129, 20, 36, "M edge", seed=502)


@pytest.mark.parametrize("M,Kin,Nout", [(M, 300, 300) for M in (32, 33, 63, 1949, 31184)] +
                         [(1949, K, 164) for K in (32, 36, 448)] + [(33, 36, N) for N in (16, 20, 164, 300)])
def test_tc_wgrad_within_bound(M, Kin, Nout):
    """wgrad_tf32x3_kernel over row splits + splitk_reduce_kernel (M not a multiple of 32: zero-filled k-block)."""
    Q = sm_count()
    splits, kb_per_split = gp.tc_wgrad_plan(M, Kin, Nout, Q)
    if M >= 1949:
        assert splits > 1
    rng = np.random.default_rng(M * 7 + Kin + Nout)
    X, G = rand(rng, M, Kin), rand(rng, M, Nout)
    gW = wgrad(dev(X), dev(G), TF32X3)
    assert_bound(gW, np.ascontiguousarray(X.T), G, np.arange(Kin), tau_tf32x3(kb_per_split, splits),
                 f"3xTF32 wgrad {M}x{Kin}x{Nout} ({splits} splits)")


def test_dispatch_refusals_and_fallbacks():
    """GEMM_TF32X3 on an ineligible shape or pointer raises ValueError; GEMM_AUTO takes the FFMA path instead (one
    launch), bit-equal to the scalar loop for fwd / dgrad and within gamma_M for wgrad."""
    rng = np.random.default_rng(9)
    for M, K, N, where in [(64, 20, 64, ""), (64, 300, 8, ""), (64, 34, 64, ""), (64, 300, 64, "X"), (64, 300, 64, "H")]:
        X, W = rand(rng, M, K), rand(rng, K, N, scale=0.1)
        Xd = at_offset(X) if where == "X" else dev(X)
        Hd = at_offset(np.zeros((M, N), np.float32)) if where == "H" else None
        with pytest.raises(ValueError):
            fwd(Xd, dev(W), TF32X3, out=Hd)
        H, n = launches(lambda: fwd(Xd, dev(W), AUTO, out=Hd))
        assert n == 1
        assert_bits(H, orc.gemm_fma_seq(X, W), f"AUTO forward fallback {M}x{N}x{K} {where}")
    for M, Kin, Nout, where in [(64, 64, 20, ""), (64, 64, 34, ""), (64, 8, 300, ""), (64, 64, 300, "gH"),
                                (64, 64, 300, "act")]:
        G, W, act = rand(rng, M, Nout), rand(rng, Kin, Nout, scale=0.1), rand(rng, M, Kin)
        Gd = at_offset(G) if where == "gH" else dev(G)
        actd = at_offset(act) if where == "act" else dev(act)
        with pytest.raises(ValueError):
            dgrad(Gd, dev(W), actd, TF32X3)
        gX, n = launches(lambda: dgrad(Gd, dev(W), actd, AUTO))
        assert n == 1
        want = np.where(act > 0, orc.gemm_fma_seq(G, W, b_transposed=True), 0.0).astype(np.float32)
        assert_bits(gX, want, f"AUTO dgrad fallback {M}x{Kin}x{Nout} {where}")
    for M, Kin, Nout, where in [(31, 64, 64, ""), (64, 64, 18, ""), (64, 34, 64, ""), (64, 64, 64, "X")]:
        X, G = rand(rng, M, Kin), rand(rng, M, Nout)
        Xd = at_offset(X) if where == "X" else dev(X)
        with pytest.raises(ValueError):
            wgrad(Xd, dev(G), TF32X3)
        gW = wgrad(Xd, dev(G), AUTO)
        assert_bound(gW, np.ascontiguousarray(X.T), G, np.arange(Kin), gamma(M), f"AUTO wgrad fallback {where}")


def tf32_exact(rng, *shape):
    """Normal values with the last mantissa bit cleared: 23 significant bits, so a_lo = a - tf32_rna(a) has at most 11
    and the tensor core reads it exactly (a truncating split would leave 12)."""
    a = rand(rng, *shape)
    return (a.view(np.uint32) & np.uint32(0xFFFFFFFE)).view(np.float32)


def one_hot_pow2(rng, rows, cols):
    """(rows, cols) with one +-2^j (|j| <= 2) per column at a random row, zeros elsewhere."""
    B = np.zeros((rows, cols), np.float32)
    B[rng.integers(0, rows, cols), np.arange(cols)] = rng.choice([-4.0, -1.0, 0.5, 1.0, 2.0, 0.25], cols)
    return B


def check_tc_split_exact(M, N, K, seed):
    """With one power of two per output, a * b = a_hi b + a_lo b must come out exactly: every product and partial sum
    is representable, so only the split can be wrong -- a_hi must be rounded to nearest, not truncated."""
    rng = np.random.default_rng(seed)
    X, W = tf32_exact(rng, M, K), one_hot_pow2(rng, K, N)
    want = (X.astype(np.float64) @ W.astype(np.float64)).astype(np.float32)
    assert_bits(fwd(dev(X), dev(W), TF32X3), want, f"3xTF32 forward on a scaled selection {M}x{N}x{K}")
    G, Wd = tf32_exact(rng, M, K), np.ascontiguousarray(one_hot_pow2(rng, K, N).T)  # W (N, K): gX = G . W^T
    want = (G.astype(np.float64) @ Wd.T.astype(np.float64)).astype(np.float32)
    assert_bits(dgrad(dev(G), dev(Wd), None, TF32X3), want, f"3xTF32 dgrad on a scaled selection {M}x{N}x{K}")
    Xs, Gs = np.ascontiguousarray(one_hot_pow2(rng, M, K)), tf32_exact(rng, M, N)
    want = (Xs.T.astype(np.float64) @ Gs.astype(np.float64)).astype(np.float32)
    assert_bits(wgrad(dev(Xs), dev(Gs), TF32X3), want, f"3xTF32 wgrad on a scaled selection {M}x{N}x{K}")


def test_tc_split_rounds_to_nearest():
    sk = gp.tc_streamk_shapes(sm_count())
    check_tc_split_exact(*sk["x3.3"], seed=600)
    check_tc_split_exact(129, 164, 60, seed=601)


def test_tc_non_finite_range():
    """tf32_hi maps +-Inf and finite |a| >= 2^128 - 2^116 (within half a TF32 ulp of FLT_MAX) to +-Inf, so a_lo is NaN:
    the tensor-core paths return NaN where fp32 would give +-Inf or a finite value (include/ptk.h).  Just below that
    the result is finite and within the bound."""
    rng = np.random.default_rng(11)
    M, K, N = 8, 64, 32
    X, W = np.zeros((M, K), np.float32), rand(rng, K, N, scale=0.1)
    X[:, 5] = 1.0
    edge = np.float32(2.0 ** 128 - 2.0 ** 116)
    X[0, 3], X[1, 3], X[2, 3], X[3, 3] = np.inf, -np.inf, np.nan, edge
    X[4, 3] = np.nextafter(edge, np.float32(0))
    X[5, 3] = -X[4, 3]
    H = fwd(dev(X), dev(W), TF32X3).cpu().numpy()
    assert not np.isfinite(H[:4]).any()
    assert np.isfinite(H[4:]).all()
    assert_bound(H, X, W, np.arange(4, M), tau_tf32x3(2, 1), "3xTF32 forward near FLT_MAX")
    G = X.copy()
    gX = dgrad(dev(G), dev(np.ascontiguousarray(W.T)), None, TF32X3).cpu().numpy()
    assert not np.isfinite(gX[:4]).any() and np.isfinite(gX[4:]).all()


# ==================================================================================== (c) the stream-K protocol
def test_streamk_bit_identical_run_to_run():
    M, N, K = gp.tc_streamk_shapes(sm_count())["x3.3"]
    rng = np.random.default_rng(12)
    X, W, G, act = dev(rand(rng, M, K)), dev(rand(rng, K, N, scale=0.1)), dev(rand(rng, M, N)), dev(rand(rng, M, K))
    Wd = dev(rand(rng, K, N, scale=0.1))  # dgrad: gX (M, K) = G (M, N) . Wd^T
    assert torch.equal(fwd(X, W, TF32X3), fwd(X, W, TF32X3))
    assert torch.equal(dgrad(G, Wd, act, TF32X3), dgrad(G, Wd, act, TF32X3))
    assert torch.equal(wgrad(X, G, TF32X3), wgrad(X, G, TF32X3))


def test_streamk_back_to_back_on_one_workspace():
    """Two calls on one workspace with no synchronisation between them: each equals its own call on a fresh workspace,
    so the second call's partial-tile flags start from zero again."""
    M, N, K = gp.tc_streamk_shapes(sm_count())["x3.3"]
    rng = np.random.default_rng(13)
    Xs = [dev(rand(rng, M, K)) for _ in range(2)]
    Ws = [dev(rand(rng, K, N, scale=0.1)) for _ in range(2)]
    L = _lib.lib()
    ws = _ws(L.ptk_gcn_linear_workspace_bytes(M, K, N))
    got = [fwd(Xs[i], Ws[i], TF32X3, ws=ws) for i in range(2)]
    torch.cuda.synchronize()
    for i in range(2):
        assert torch.equal(got[i], fwd(Xs[i], Ws[i], TF32X3))
    # dgrad (M, K) = G (M, N) . W^T with W (K, N), masked: the mask area of the workspace is reused too
    Gs = [dev(rand(rng, M, N)) for _ in range(2)]
    acts = [dev(rand(rng, M, K)) for _ in range(2)]
    ws = _ws(L.ptk_gcn_linear_workspace_bytes(M, K, N))
    got = [dgrad(Gs[i], Ws[i], acts[i], TF32X3, ws=ws) for i in range(2)]
    torch.cuda.synchronize()
    for i in range(2):
        assert torch.equal(got[i], dgrad(Gs[i], Ws[i], acts[i], TF32X3))


def test_streamk_cuda_graph_replay():
    """A masked dgrad at a shared-tile shape captured once, replayed three times with its inputs changed in place:
    every replay equals an eager call bit for bit."""
    M, N, K = gp.tc_streamk_shapes(sm_count())["x3.3"]
    rng = np.random.default_rng(14)
    G, W, act = dev(rand(rng, M, N)), dev(rand(rng, K, N, scale=0.1)), dev(rand(rng, M, K))
    ws = _ws(_lib.lib().ptk_gcn_linear_workspace_bytes(M, K, N))
    out = torch.empty(M, K, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dgrad(G, W, act, TF32X3, ws=ws, out=out)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        dgrad(G, W, act, TF32X3, ws=ws, out=out)
    for _ in range(3):
        G.copy_(dev(rand(rng, M, N)))
        W.copy_(dev(rand(rng, K, N, scale=0.1)))
        act.copy_(dev(rand(rng, M, K)))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, dgrad(G, W, act, TF32X3))


@pytest.mark.parametrize("pair", ["1", "3"])
def test_tc_paths_in_cluster_child(pair):
    """PTK_TG_PAIR=1 (2-CTA clusters, multicast weight tiles) and 3 (cta_group::2 MMAs): the tensor-core table, the
    masks, the exact-split check and run-to-run identity under the same bounds, in a child interpreter."""
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "tc"], env=dict(os.environ, PTK_TG_PAIR=pair),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "tc ok" in out.stdout, out.stdout + out.stderr


# ================================================================================ child-interpreter entry point
def _child_exact():
    Q = sm_count()
    # the register-staged kernel has no tail tiles: the edges and two reconstruction-step shapes
    shapes = [s for s in ffma_fwd_shapes(Q) if not s[3].startswith("rt_tail") or s[3] in ("rt_tail=2", "rt_tail=5")]
    for i, (M, N, K, _) in enumerate(shapes):
        check_ffma_fwd(M, N, K, seed=700 + i)
    split = fwd_split_shapes(Q) if os.environ.get("PTK_FWD_NO_TMA") else []  # PTK_FWD_BM leaves the split form alone
    for i, shape in enumerate(split):
        check_fwd_split(*shape, seed=800 + i)
    print("exact ok:", len(shapes), "forward shapes,", len(split), "split shapes")


def _child_tc():
    Q = sm_count()
    worst = 0.0
    for i, s in enumerate(tc_table(Q)):
        worst = max(worst, check_tc_fwd(*s, seed=900 + i), check_tc_dgrad(*s, seed=1000 + i))
    sk = gp.tc_streamk_shapes(Q)
    check_dgrad_masks(*sk["odd"], "odd", seed=1100)
    check_tc_split_exact(*sk["odd"], seed=1101)
    M, N, K = sk["x3.3"]
    rng = np.random.default_rng(1102)
    X, W = dev(rand(rng, M, K)), dev(rand(rng, K, N))
    assert torch.equal(fwd(X, W, TF32X3), fwd(X, W, TF32X3))
    print(f"tc ok: PTK_TG_PAIR={os.environ.get('PTK_TG_PAIR')}, worst err / (|A||B|) {worst:.3g}")


if __name__ == "__main__":
    orc.build()
    {"exact": _child_exact, "tc": _child_tc}[sys.argv[1]]()
