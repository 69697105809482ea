"""Cost of the 1-NN backward (ptk_knn1_bwd_lengths, ptk_knn1_bwd_det) against what a user would otherwise run and
against the Chamfer backward.  CUDA events after a warm-up; the rows of a shape alternate within each of three rounds.

    python tools/knn1_bwd_bench.py [--rounds 3] [--iters 50]

Rows per shape:
  knn1 bwd default / det    the two entry points alone, on the forward's idx and a per-query upstream gradient
  torch gather+index_add    the restatement in torch: grad_p1 = (2 g)[..., None] * (p1 - gather(p2, idx)),
                            grad_p2 = zeros.index_add_(-grad_p1) over the flattened rows
  chamfer bwd default / det ptk_chamfer_bwd_lengths / ptk_chamfer_bwd_det (both directions: twice the terms)
  1-dir loss fwd+bwd        ops.knn1(p1, p2).dists, mean over the valid queries, backward; flag off / on
Shapes: 256 x 10k x 10k (bench.py's); the same batch ragged, lengths uniform in [2.5k, 10k]; 16 x 1949 x 10k (a
mesh's vertices against a sampled cloud).  At 256 x 10k x 10k the working set (clouds, gradients, idx, g: 143 MB, plus
61 MB of int64 accumulators for det) is larger than the 126 MB L2; the 16 x 1949 x 10k working set fits in it.
"bytes" is the algorithmic traffic of the knn1 backward: p1, idx and g of every valid query, p2 of every valid target
read once, and both gradients written once (padded rows included); "HBM" is that over 7.7 TB/s.
Prints the card's name and power limit first."""
import argparse
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import ptk_b200  # noqa: E402
from ptk_b200 import _lib  # noqa: E402

HBM_BPS = 7.7e12


def timeit(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def run_shape(name, B, P1, P2, ragged, rounds, iters):
    dev = torch.device("cuda")
    L = _lib.lib()
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(B, P1, 3, device=dev, generator=gen)
    y = torch.rand(B, P2, 3, device=dev, generator=gen)
    l1 = l2 = None
    if ragged:
        l1 = torch.randint(P1 // 4, P1 + 1, (B,), device=dev, generator=gen)
        l2 = torch.randint(P2 // 4, P2 + 1, (B,), device=dev, generator=gen)
    n1 = l1.sum().item() if ragged else B * P1
    n2 = l2.sum().item() if ragged else B * P2
    g = torch.randn(B, P1, device=dev, generator=gen) / n1
    _, idx = ptk_b200.ops.knn1(x, y, l1, l2)
    _, ix, iy = ptk_b200.ops.chamfer(x, y, l1, l2)
    gc = torch.ones(B, device=dev) / B
    g1, g2 = torch.empty_like(x), torch.empty_like(y)
    ws = torch.empty(L.ptk_knn1_bwd_det_workspace_bytes(B, P1, P2), dtype=torch.uint8, device=dev)
    wsc = torch.empty(L.ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2), dtype=torch.uint8, device=dev)
    flat = (idx.long() + (torch.arange(B, device=dev) * P2)[:, None]).reshape(-1)
    valid = torch.ones(B, P1, dtype=torch.bool, device=dev)
    if ragged:
        valid = torch.arange(P1, device=dev)[None] < l1[:, None]
    gm = torch.where(valid, g, torch.zeros((), device=dev))

    def knn_default():
        _lib.check(L.ptk_knn1_bwd_lengths(p(x), p(y), p(l1), p(l2), p(idx), p(g), B, P1, P2, p(g1), p(g2), st()))

    def knn_det():
        _lib.check(L.ptk_knn1_bwd_det(p(x), p(y), p(l1), p(l2), p(idx), p(g), B, P1, P2, p(g1), p(g2), p(ws), ws.numel(),
                                      st()))

    def torch_restatement():
        nn = torch.gather(y, 1, idx.long()[..., None].expand(-1, -1, 3))
        t = (2 * gm)[..., None] * (x - nn)
        torch.zeros(B * P2, 3, device=dev).index_add_(0, flat, -t.reshape(-1, 3))

    def cham_default():
        _lib.check(L.ptk_chamfer_bwd_lengths(p(x), p(y), p(l1), p(l2), p(ix), p(iy), p(gc), B, P1, P2, _lib.REDUCE_MEAN,
                                             p(g1), p(g2), st()))

    def cham_det():
        _lib.check(L.ptk_chamfer_bwd_det(p(x), p(y), p(l1), p(l2), p(ix), p(iy), p(gc), B, P1, P2, _lib.REDUCE_MEAN,
                                         p(g1), p(g2), p(wsc), wsc.numel(), st()))

    xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    den = l1.clamp(min=1) if ragged else torch.full((B,), P1, device=dev)

    def loss(flag):
        def fn():
            torch.use_deterministic_algorithms(flag)
            xr.grad = yr.grad = None
            d, _ = ptk_b200.ops.knn1(xr, yr, l1, l2)
            (d.sum(1) / den).mean().backward()
        return fn

    rows = {"knn1 bwd default": (knn_default, iters), "knn1 bwd det": (knn_det, iters),
            "torch gather+index_add": (torch_restatement, iters), "chamfer bwd default": (cham_default, iters),
            "chamfer bwd det": (cham_det, iters), "1-dir loss fwd+bwd default": (loss(False), max(iters // 10, 3)),
            "1-dir loss fwd+bwd det": (loss(True), max(iters // 10, 3))}
    torch.utils.deterministic.fill_uninitialized_memory = False
    res = {r: [] for r in rows}
    for r, (fn, _) in rows.items():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for r, (fn, n) in rows.items():
            res[r].append(timeit(fn, n))
    torch.use_deterministic_algorithms(False)
    nbytes = n1 * (12 + 4 + 4) + n2 * 12 + B * (P1 + P2) * 12
    print(f"{name}: B={B} P1={P1} P2={P2} valid queries {n1} targets {n2}; knn1 bwd bytes {nbytes / 1e6:.1f} MB "
          f"(>= {nbytes / HBM_BPS * 1e3:.4f} ms at 7.7 TB/s)", flush=True)
    for r, ts in res.items():
        med = float(np.median(ts))
        extra = f"   HBM {nbytes / (med * 1e-3) / HBM_BPS:6.1%}" if r.startswith("knn1") else ""
        print(f"  {r:28s} " + " ".join(f"{t:8.4f}" for t in ts) + f"   median {med:8.4f} ms{extra}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("device:", q[0] if q else torch.cuda.get_device_name(), "| torch", torch.__version__, flush=True)
    run_shape("homogeneous", 256, 10000, 10000, False, a.rounds, a.iters)
    run_shape("ragged", 256, 10000, 10000, True, a.rounds, a.iters)
    run_shape("mesh-shaped", 16, 1949, 10000, False, a.rounds, a.iters)


if __name__ == "__main__":
    main()
