"""CPU checks behind the GEMM path tests (tests/test_gemm_paths_gpu.py): the scalar FMA oracle, and the Python mirrors
of the launch plans (tests/gemm_plans.py) that choose the GPU shapes.  No GPU needed."""
import numpy as np
import pytest

import gemm_plans as gp

QS = (148, 132, 114, 120, 160)


# ------------------------------------------------------------------------------------------------ the oracle
def test_oracle_fma_seq_fuses(oracle):
    """a * b + c with a = b = 1 + 2^-12, c = -(1 + 2^-11): fused 2^-24; unfused a * b rounds to 1 + 2^-11 and gives 0."""
    a = np.float32(1 + 2.0 ** -12)
    c = np.float32(-(1 + 2.0 ** -11))
    assert np.float32(a * a) + c == 0.0  # the unfused value, for contrast
    A = np.array([[c, a]], np.float32)    # acc = fmaf(c, 1, 0) = c, then fmaf(a, a, c)
    B = np.array([[1.0], [a]], np.float32)
    assert oracle.gemm_fma_seq(A, B)[0, 0] == np.float32(2.0 ** -24)
    assert oracle.gemm_fma_seq(A, np.ascontiguousarray(B.T), b_transposed=True)[0, 0] == np.float32(2.0 ** -24)


def test_oracle_fma_seq_is_exact_on_dyadic_inputs(oracle):
    """Small dyadic operands keep every product and partial sum exact in fp32 and fp64: the oracle must equal the
    float64 product, for row subsets and for the transposed-B layout."""
    rng = np.random.default_rng(7)
    M, K, N = 37, 300, 45
    A = (rng.integers(-8, 9, (M, K)) * 2.0 ** -3).astype(np.float32)
    B = (rng.integers(-8, 9, (K, N)) * 2.0 ** -5).astype(np.float32)
    want = A.astype(np.float64) @ B.astype(np.float64)
    assert np.abs(want).max() * 2 ** 8 < 2 ** 24  # every partial sum is an integer multiple of 2^-8 below 2^24
    assert np.array_equal(oracle.gemm_fma_seq(A, B), want.astype(np.float32))
    rows = np.array([36, 0, 5, 5, 17])
    assert np.array_equal(oracle.gemm_fma_seq(A, B, rows=rows), want[rows].astype(np.float32))
    Bt = np.ascontiguousarray(B.T)
    assert np.array_equal(oracle.gemm_fma_seq(A, Bt, rows=rows, b_transposed=True), want[rows].astype(np.float32))
    assert oracle.gemm_fma_seq(A, B, rows=np.zeros(0, np.int64)).shape == (0, N)


def test_oracle_fma_seq_is_k_sequential(oracle):
    """The chain runs k = 0..K-1 in order: 2^24 + 1 - 2^24 gives 0 in that order (the 1 is absorbed), 1 when the
    large terms cancel first."""
    A = np.array([[2.0 ** 24, 1.0, -(2.0 ** 24)], [2.0 ** 24, -(2.0 ** 24), 1.0]], np.float32)
    B = np.ones((3, 1), np.float32)
    assert oracle.gemm_fma_seq(A, B)[:, 0].tolist() == [0.0, 1.0]


# ------------------------------------------------------------------------------------ tensor-core stream-K plan
TG_SHAPES = [(1, 16, 32), (127, 17, 36), (129, 161, 448), (9344, 300, 300), (18945, 160, 300), (19072, 160, 32),
             (31184, 300, 300), (31184, 448, 300), (31184, 300, 448), (100000, 300, 36)]


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("Q", QS)
def test_tg_plan_covers_every_unit_once(Q, pair):
    for M, N, K in TG_SHAPES:
        plan = gp.tg_plan(M, N, K, Q, pair)
        assert plan.workers == gp.tg_num_ctas(M, N, Q, pair) // (2 if pair else 1)
        assert 1 <= plan.workers <= (Q // 2 if pair else Q)
        seen = np.zeros((plan.num_tiles, plan.num_kb), np.int32)
        for mine in plan.pieces:
            for p in mine:
                assert 0 <= p.kb_begin < p.kb_end <= plan.num_kb
                seen[p.tile, p.kb_begin:p.kb_end] += 1
        assert (seen == 1).all(), (M, N, K)


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("Q", QS)
def test_tg_plan_shares_a_tile_between_two_neighbours_at_most(Q, pair):
    """The combine protocol: a tile spans at most two workers, c and c + 1; c holds its first k-blocks and publishes
    them (head), c + 1 holds the rest and combines (tail).  A worker walks its range from the end, so its head piece
    comes first and its tail piece last, and it is a head at most once and a tail at most once."""
    for M, N, K in TG_SHAPES:
        plan = gp.tg_plan(M, N, K, Q, pair)
        owners = {}
        for c, mine in enumerate(plan.pieces):
            heads = [i for i, p in enumerate(mine) if p.head]
            tails = [i for i, p in enumerate(mine) if p.tail]
            assert heads in ([], [0]) and tails in ([], [len(mine) - 1])
            assert all(mine[i].tile > mine[i + 1].tile for i in range(len(mine) - 1))
            for p in mine:
                owners.setdefault(p.tile, []).append((c, p))
        for tile, own in owners.items():
            assert len(own) <= 2
            if len(own) == 2:
                (c0, head), (c1, tail) = own
                assert c1 == c0 + 1 and head.head and tail.tail
                assert head.kb_begin == 0 and head.kb_end == tail.kb_begin and tail.kb_end == plan.num_kb
            else:
                assert not own[0][1].head and not own[0][1].tail


def test_tg_plan_reaches_the_shared_tile_cases():
    """The shapes the GPU tests use: tiles below, equal to, one above and 3.3x the SM count."""
    for Q in QS:
        shapes = gp.tc_streamk_shapes(Q)
        for name, (M, N, K) in shapes.items():
            plan = gp.tg_plan(M, N, K, Q)
            tiles = gp.ceil_div(M, gp.TG_BM) * gp.ceil_div(N, gp.TG_BN)
            assert tiles == {"below": Q - 1, "equal": Q, "above": Q + 1}.get(name, tiles)
            assert bool(gp.tg_shared_tiles(plan)) == (tiles > Q), (Q, name)
        # the odd row-tile count leaves the second CTA of the last pair of the cluster forms wholly beyond M
        M, N, K = shapes["odd"]
        assert gp.ceil_div(M, gp.TG_BM) % 2 == 1
        assert gp.tg_shared_tiles(gp.tg_plan(M, N, K, Q, pair=True))
    M, N, K = gp.tc_streamk_shapes(148)["x3.3"]
    assert gp.ceil_div(M, gp.TG_BM) * gp.ceil_div(N, gp.TG_BN) == 488


# --------------------------------------------------------------------------------- exact forward: tail plan
@pytest.mark.parametrize("Q", QS)
def test_fwd_tail_plan_covers_every_row_once(Q):
    for N in (64, 160, 300, 320):
        for M in list(range(1, 400, 7)) + [4736, 4737, 9473, 29184, 31184, 100003]:
            tiles = gp.fwd_row_tiles(M, N, Q)
            p = gp.fwd_tma_plan(M, N, Q)
            assert 1 <= p.rt_tail <= 8 and (p.rt_tail == 8) == (p.n_tail == 0)
            end = 0
            for m0, h in tiles:
                assert m0 == end and m0 < M
                end = m0 + h
            assert end >= M


@pytest.mark.parametrize("Q", QS)
def test_fwd_tail_shapes_reach_every_tile_height(Q):
    """The GPU shape table reaches rt_tail 1 through 8 at N = 300, each beyond one full round of CTAs and with its
    last tile cut by M."""
    for rt in range(1, 9):
        M = gp.fwd_rows_for_rt_tail(rt, 300, Q)
        p = gp.fwd_tma_plan(M, 300, Q)
        assert p.rt_tail == rt and p.n_main > 0
        if rt < 8:
            assert p.n_tail > 0 and (M - p.n_main * gp.FT_BM) % (rt * 8) != 0
    assert gp.fwd_tma_plan(31184, 300, 148).rt_tail == 5 and gp.fwd_tma_plan(29184, 300, 148).rt_tail == 2


def test_tile_edge_rows():
    assert gp.tile_edge_rows(100, [(0, 64), (64, 40)], extra=[3, 200]) == [0, 3, 63, 64, 99]
    assert gp.tile_edge_rows(1, [(0, 64)]) == [0]


# ------------------------------------------------------------------------------------------ split-K plans
@pytest.mark.parametrize("Q", QS)
def test_wgrad_split_plans(Q):
    assert gp.skinny_wgrad_ctas(31184, Q) == min(3 * Q, 31184 // 16)
    assert gp.skinny_wgrad_ctas(7, Q) == 1
    for M in (32, 33, 63, 1949, 31184):
        for Kin, Nout in ((300, 300), (36, 20), (448, 164)):
            s = gp.tc_wgrad_splits(M, Kin, Nout, Q)
            assert 1 <= s <= max(gp.ceil_div(M, gp.TG_BK) // 4, 1)
            assert 1 <= gp.ffma_wgrad_splits(M, Kin, Nout, Q) <= gp.ceil_div(M, 16)
    assert gp.tc_wgrad_splits(31184, 300, 300, 148) == 24 and gp.tc_wgrad_splits(32, 300, 300, 148) == 1
