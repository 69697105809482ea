"""Cost of the K-NN forward (ptk_knn_fwd_lengths) and backward (ptk_knn_bwd_lengths, ptk_knn_bwd_det) against the
one-direction 1-NN scan and against what a user would otherwise run.  CUDA events after a warm-up; the rows of a shape
alternate within each round.

    python tools/knn_bench.py [--rounds 3] [--iters 5]

Rows per shape:
  knn fwd K=k               ops.knn forward alone (no grad), K in {2, 4, 8, 16, 32, 64}
  knn bwd default / det     ptk_knn_bwd_lengths / ptk_knn_bwd_det at K = 8, on the forward's idx
  knn1 exact                ops.knn1 forward under set_chamfer_algo("exact"): the one-direction 6-op scan, the floor
                            of the arithmetic every K shares
  torch cdist+topk K=8      a chunked torch restatement: the same distances ((dx*dx + dy*dy) + dz*dz, padded targets
                            +inf) and torch.topk(largest=False); for timing only, topk's tie order is not the contract
Shapes: 256 x 10k x 10k (bench.py's; the clouds exceed the 126 MB L2); the same batch ragged, lengths uniform in
[2.5k, 10k]; 16 x 1949 x 10k (a mesh's vertices against a sampled cloud); 1 x 10k x 10k (one pair: the target range
is split across CTAs).  "evals" counts the valid (query, target) pairs; "FP32" is 8 flop per evaluation (DESIGN.md
K1's accounting) over the 74.4 TFLOP/s FP32 figure DESIGN.md K1 uses.  Prints the card's name and power limit first."""
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

FP32_FLOPS = 74.4e12


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
    evals = float((l1.double() * l2.double()).sum().item()) if ragged else float(B) * P1 * P2
    K8 = 8
    _, idx8 = ptk_b200.ops.knn(x, y, K8, l1, l2)
    g8 = torch.randn(B, P1, K8, device=dev, generator=gen) / (B * P1)
    g1, g2 = torch.empty_like(x), torch.empty_like(y)
    ws = torch.empty(L.ptk_knn1_bwd_det_workspace_bytes(B, P1, P2), dtype=torch.uint8, device=dev)

    def fwd(K):
        def fn():
            with torch.no_grad():
                ptk_b200.ops.knn(x, y, K, l1, l2)
        return fn

    def bwd_default():
        _lib.check(L.ptk_knn_bwd_lengths(p(x), p(y), p(l1), p(l2), p(idx8), p(g8), B, P1, P2, K8, p(g1), p(g2), st()))

    def bwd_det():
        _lib.check(L.ptk_knn_bwd_det(p(x), p(y), p(l1), p(l2), p(idx8), p(g8), B, P1, P2, K8, p(g1), p(g2), p(ws),
                                     ws.numel(), st()))

    def knn1_exact():
        ptk_b200.ops.set_chamfer_algo("exact")
        with torch.no_grad():
            ptk_b200.ops.knn1(x, y, l1, l2)
        ptk_b200.ops.set_chamfer_algo("auto")

    chunk = max(1, (1 << 29) // (P1 * P2))  # at most 2 GB per distance temporary

    def torch_topk():
        for b0 in range(0, B, chunk):
            xs, ys = x[b0:b0 + chunk], y[b0:b0 + chunk]
            dx = xs[:, :, None, 0] - ys[:, None, :, 0]
            dy = xs[:, :, None, 1] - ys[:, None, :, 1]
            dz = xs[:, :, None, 2] - ys[:, None, :, 2]
            d = (dx * dx + dy * dy) + dz * dz
            if ragged:
                d.masked_fill_(torch.arange(P2, device=dev)[None, None] >= l2[b0:b0 + chunk, None, None], float("inf"))
            torch.topk(d, K8, dim=2, largest=False, sorted=True)

    rows = {f"knn fwd K={K}": (fwd(K), iters) for K in (2, 4, 8, 16, 32, 64)}
    rows.update({"knn bwd default K=8": (bwd_default, 10 * iters), "knn bwd det K=8": (bwd_det, 10 * iters),
                 "knn1 exact": (knn1_exact, iters), "torch cdist+topk K=8": (torch_topk, max(iters // 2, 1))})
    for fn, _ in rows.values():
        fn()
    torch.cuda.synchronize()
    res = {r: [] for r in rows}
    for _ in range(rounds):
        for r, (fn, n) in rows.items():
            res[r].append(timeit(fn, n))
    print(f"{name}: B={B} P1={P1} P2={P2}; evaluations {evals:.4g}", flush=True)
    med = {r: float(np.median(ts)) for r, ts in res.items()}
    for r, ts in res.items():
        extra = ""
        if not r.startswith("knn bwd"):
            rate = evals / (med[r] * 1e-3)
            extra = f"   {rate / 1e9:9.1f} G evals/s   FP32 {rate * 8 / FP32_FLOPS:6.1%}"
            if r.startswith("knn fwd"):
                extra += f"   x{med[r] / med['knn1 exact']:.2f} knn1 exact"
        print(f"  {r:22s} " + " ".join(f"{t:9.4f}" for t in ts) + f"   median {med[r]:9.4f} ms{extra}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("device:", q[0] if q else torch.cuda.get_device_name(), "| torch", torch.__version__, flush=True)
    run_shape("homogeneous", 256, 10000, 10000, False, a.rounds, a.iters)
    run_shape("ragged", 256, 10000, 10000, True, a.rounds, a.iters)
    run_shape("mesh-shaped", 16, 1949, 10000, False, a.rounds, a.iters)
    run_shape("one pair", 1, 10000, 10000, False, a.rounds, a.iters)


if __name__ == "__main__":
    main()
