"""Python mirrors of the launch plans of the per-vertex linear layers, for a device with Q SMs.

The tests use them to choose shapes that reach a given path (shared stream-K tiles, a given tail-tile height,
split-K reductions) and check the plans' own invariants without a GPU.  Each function restates the host code it
names; a change there has to be made here too, or the path assertions of tests/test_gemm_paths_gpu.py fail.
"""
from collections import namedtuple

TG_BM, TG_BN, TG_BK = 128, 160, 32   # csrc/gemm_tf32x3.cu: tensor-core tile and k-block
FT_BM, FW_BN = 64, 160               # csrc/gcn_linear.cu: exact forward row tile and column tile
SK_MAXN = 4                          # csrc/gcn_linear.cu: widest "skinny" layer


def ceil_div(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------ tensor-core fwd / dgrad (stream-K)
def tg_num_ctas(M, N, Q, pair=False):
    """tg_num_ctas (gemm_tf32x3.cu): one CTA per SM at most; pair forms launch whole clusters of two."""
    tiles_m, tiles_n = ceil_div(M, TG_BM), ceil_div(N, TG_BN)
    if pair:
        return 2 * min(ceil_div(tiles_m, 2) * tiles_n, Q // 2)
    return min(tiles_m * tiles_n, Q)


Piece = namedtuple("Piece", "tile kb_begin kb_end head tail")
TGPlan = namedtuple("TGPlan", "num_tiles num_kb workers pieces")


def tg_plan(M, N, K, Q, pair=False):
    """The (tile, k-block) work split of gemm_tf32x3_kernel / gemm_tf32x3_2sm_kernel: worker c (a CTA, or a cluster
    of two in the pair forms) takes the units [c U / G, (c+1) U / G) and walks them from the end.  pieces[c] lists its
    tiles in that order; head = the tile's last k-blocks belong to worker c+1 (publish the partial), tail = its first
    k-blocks came from worker c-1 (combine)."""
    num_kb = ceil_div(K, TG_BK)
    tiles_m, tiles_n = ceil_div(M, TG_BM), ceil_div(N, TG_BN)
    num_tiles = (ceil_div(tiles_m, 2) if pair else tiles_m) * tiles_n
    workers = tg_num_ctas(M, N, Q, pair) // (2 if pair else 1)
    units = num_tiles * num_kb
    pieces = []
    for me in range(workers):
        u0, u1 = units * me // workers, units * (me + 1) // workers
        mine, hi = [], u1
        while hi > u0:
            tile = (hi - 1) // num_kb
            kb_begin, kb_end = max(u0 - tile * num_kb, 0), hi - tile * num_kb
            hi = tile * num_kb + kb_begin
            mine.append(Piece(tile, kb_begin, kb_end, kb_end < num_kb, kb_begin > 0))
        pieces.append(mine)
    return TGPlan(num_tiles, num_kb, workers, pieces)


def tg_shared_tiles(plan):
    """Tiles whose k-blocks are split between two workers (combined through a workspace slot and a flag)."""
    return sorted(p.tile for mine in plan.pieces for p in mine if p.head)


def tc_streamk_shapes(Q):
    """(M, N, K) with output tiles below, equal to and one above the SM count (one 160-wide column tile, the last
    row tile cut by M), and about 3.3x the SM count (M = 31184, N = 300 on 148 SMs: a reconstruction step's layer).
    "odd": an odd number of 128-row tiles above Q / 2 pairs, so that the cluster forms share tiles and the second
    CTA of the last pair lies wholly beyond M."""
    odd = Q + 1 if Q % 2 == 0 else Q + 2
    return {"below": ((Q - 1) * TG_BM - 5, 160, 300), "equal": (Q * TG_BM - 3, 160, 300),
            "above": (Q * TG_BM + 1, 160, 300), "odd": ((odd - 1) * TG_BM + 1, 160, 300),
            "x3.3": (round(3.3 * Q / 2) * TG_BM - 48, 300, 300)}


# ------------------------------------------------------------------------------ exact forward: TMA tail plan
FwdPlan = namedtuple("FwdPlan", "cx n_main rt_tail n_tail")


def fwd_tma_plan(M, N, Q):
    """Tail plan of launch_fwd_tma (gcn_linear.cu): rows behind the last full round of Q CTAs go into tiles of
    rt_tail * 8 rows (rt_tail = 8: no tail tiles)."""
    cx, tiles64 = ceil_div(N, FW_BN), ceil_div(M, FT_BM)
    n_main, rt_tail = tiles64, 8
    if (cx * tiles64) % Q != 0:
        n_main = (cx * tiles64 // Q) * Q // cx
        rem = M - n_main * FT_BM
        best = 1e30
        for rt in range(8, 0, -1):
            cost = float(ceil_div(cx * ceil_div(rem, rt * 8), Q)) * rt * (1.0 + 0.03 * (8 - rt))
            if cost < best - 1e-9:
                best, rt_tail = cost, rt
        if rt_tail == 8:
            n_main = tiles64
    n_tail = 0 if rt_tail == 8 else ceil_div(M - n_main * FT_BM, rt_tail * 8)
    return FwdPlan(cx, n_main, rt_tail, n_tail)


def fwd_row_tiles(M, N, Q):
    """(first row, height) of every row tile the TMA forward launches."""
    p = fwd_tma_plan(M, N, Q)
    tiles = [(i * FT_BM, FT_BM) for i in range(p.n_main)]
    tiles += [(p.n_main * FT_BM + t * p.rt_tail * 8, p.rt_tail * 8) for t in range(p.n_tail)]
    return tiles


def fwd_rows_for_rt_tail(rt, N, Q):
    """Smallest M beyond one full round of CTAs for which the forward uses tail tiles of rt * 8 rows and the last of
    them is cut by M (rt = 8: the tail plan runs and keeps 64-row tiles, M not a multiple of 64)."""
    cx = ceil_div(N, FW_BN)
    for M in range(Q * FT_BM // cx + 1, 64 * Q * FT_BM):
        p = fwd_tma_plan(M, N, Q)
        if p.rt_tail != rt:
            continue
        if rt < 8 and (M - p.n_main * FT_BM) % (rt * 8) != 0:
            return M
        if rt == 8 and (cx * ceil_div(M, FT_BM)) % Q != 0 and M % FT_BM != 0:
            return M
    raise ValueError(f"no M reaches rt_tail {rt} at N={N}, Q={Q}")


def tile_edge_rows(M, tiles, extra=()):
    """First and last row of every (first row, height) tile inside [0, M), the last row of the matrix and `extra`."""
    rows = {M - 1}
    for m0, h in tiles:
        if m0 < M:
            rows.update((m0, min(m0 + h, M) - 1))
    rows.update(r for r in extra if 0 <= r < M)
    return sorted(rows)


# ------------------------------------------------------------------------------ wgrad split-K plans
def tc_wgrad_plan(M, Kin, Nout, Q):
    """plan_wgrad (gemm_tf32x3.cu): (row splits, 32-row k-blocks per split) of the tensor-core wgrad; the splits'
    partial products are summed by splitk_reduce_kernel."""
    tiles = ceil_div(Kin, TG_BM) * ceil_div(Nout, TG_BN)
    num_kb = ceil_div(M, TG_BK)
    want = max(Q // tiles, 1)
    want = min(want, max(num_kb // 4, 1))
    kb_per_split = ceil_div(num_kb, want)
    return ceil_div(num_kb, kb_per_split), kb_per_split


def tc_wgrad_splits(M, Kin, Nout, Q):
    return tc_wgrad_plan(M, Kin, Nout, Q)[0]


def skinny_wgrad_ctas(M, Q):
    """skinny_wgrad_ctas (gcn_linear.cu): row slabs of the N <= 4 wgrad, clamped at 3 CTAs per SM."""
    return max(min(M // 16, 3 * Q), 1)


def ffma_wgrad_slabs(M, K, N, Q):
    """Row ranges [r0, r1) of the partial products of the FFMA wgrad, in the order splitk_reduce_kernel adds them:
    skinny_wgrad_kernel's CTAs for N <= 4, else wgrad_splits rounded to 16-row slabs (ptk_gcn_linear_wgrad).  Each
    partial is a k-sequential FMA chain over its rows; a range may be empty (a CTA past M adds zeros)."""
    if N <= SK_MAXN:
        n = skinny_wgrad_ctas(M, Q)
        per = ceil_div(M, n)
    else:
        tiles = ceil_div(K, 128) * ceil_div(N, 128)
        want = max(min(ceil_div(2 * Q * 2, tiles), ceil_div(M, 4 * 16)), 1)
        per = ceil_div(ceil_div(M, want), 16) * 16
        n = ceil_div(M, per)
    return [(min(s * per, M), min((s + 1) * per, M)) for s in range(n)]


def ffma_wgrad_splits(M, K, N, Q):
    return len(ffma_wgrad_slabs(M, K, N, Q))
