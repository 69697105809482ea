"""Ragged Chamfer batches (per-cloud lengths) against the forms a caller had without them: GPU ms of forward + backward.

    python tools/chamfer_ragged_bench.py [--repeats 5] [--out profiles/r04_chamfer_ragged.txt]

Workloads (seeded):
  1. B = 256 clouds padded to 10k points, lengths uniform in [2.5k, 10k]: the ragged call, the padded homogeneous
     call at the same shapes (the work upper bound; it computes a different, wrong loss) and the per-pair loop of
     homogeneous calls on the sliced clouds (the only correct form without lengths).  The work fraction
     sum(lx * ly) / (B * P1 * P2) is printed next to the time fraction ragged / padded.
  2. Touch-shaped clouds: 256 site clouds of 1000..4000 points against 4000-point ground truths.  The touch loader's
     form tiles each site cloud x4 and keeps the first 4000 points (exact duplicates); the ragged form passes the
     untiled clouds padded to 4000 with their lengths.  Time and ops.chamfer_rescued for each.
  3. The pruned scan: B = 4 clouds padded to 100k points, lengths in [30k, 100k].
Every form is timed with CUDA events around `iters` back-to-back fwd+bwd calls after a warm-up, `repeats` times; the
median, min and max per call are printed.  The card name and power limit are read in the same run.
"""
import argparse
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ptk_b200  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.TimeoutExpired):
        power = "unknown"
    return f"{name}, power limit {power}"


def time_ms(fn, iters, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return statistics.median(out), min(out), max(out)


def fwd_bwd(x, y, lx=None, ly=None):
    def run():
        cham, _, _ = ptk_b200.ops.chamfer(x, y, lx, ly)
        torch.autograd.grad(cham.sum(), (x, y))
    return run


def per_pair(xs, ys):
    def run():
        for a, b in zip(xs, ys):
            cham, _, _ = ptk_b200.ops.chamfer(a, b)
            torch.autograd.grad(cham.sum(), (a, b))
    return run


def fmt(t):
    return f"{t[0]:9.3f} ms  (min {t[1]:.3f}, max {t[2]:.3f})"


def padded(clouds, P):
    """(B, P, 3) with the clouds at the front of each row (zero padding) and their lengths."""
    B = len(clouds)
    out = torch.zeros(B, P, 3)
    for b, c in enumerate(clouds):
        out[b, :len(c)] = c
    return out, torch.tensor([len(c) for c in clouds], dtype=torch.int64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_chamfer_ragged.txt"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("chamfer_ragged_bench: needs a CUDA device")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"# tools/chamfer_ragged_bench.py -- {card()}")
    say("# GPU ms per forward + backward call (CUDA events), median of repeats; Chamfer algo 'auto'")
    rng = np.random.default_rng(0)
    dev = "cuda"

    # ---- 1
    B, P = 256, 10000
    lx = rng.integers(2500, P + 1, B)
    ly = rng.integers(2500, P + 1, B)
    x = (torch.from_numpy(rng.random((B, P, 3), np.float32)) - 0.5).to(dev).requires_grad_(True)
    y = (torch.from_numpy(rng.random((B, P, 3), np.float32)) - 0.5).to(dev).requires_grad_(True)
    lxt, lyt = torch.from_numpy(lx).to(dev), torch.from_numpy(ly).to(dev)
    xs = [x[b:b + 1, :lx[b]].detach().contiguous().requires_grad_(True) for b in range(B)]
    ys = [y[b:b + 1, :ly[b]].detach().contiguous().requires_grad_(True) for b in range(B)]
    work = float((lx.astype(np.float64) * ly).sum() / (B * P * P))
    say(f"\n## 1. B = {B}, clouds padded to {P} points, lengths uniform in [2500, {P}] (seed 0)")
    t_rag = time_ms(fwd_bwd(x, y, lxt, lyt), 10, args.repeats)
    t_pad = time_ms(fwd_bwd(x, y), 10, args.repeats)
    t_loop = time_ms(per_pair(xs, ys), 1, args.repeats)
    say(f"ragged call               {fmt(t_rag)}")
    say(f"padded homogeneous call   {fmt(t_pad)}")
    say(f"per-pair loop ({B} calls) {fmt(t_loop)}")
    say(f"work fraction sum(lx*ly)/(B*P*P) = {work:.3f}; time fraction ragged/padded = {t_rag[0] / t_pad[0]:.3f}; "
        f"per-pair loop / ragged = {t_loop[0] / t_rag[0]:.1f}x")
    del x, y, xs, ys

    # ---- 2
    B, N = 256, 4000
    sizes = rng.integers(1000, N + 1, B)
    sites = [torch.from_numpy(rng.random((int(n), 3), np.float32) - 0.5) for n in sizes]
    gt = (torch.from_numpy(rng.random((B, N, 3), np.float32)) - 0.5).to(dev).requires_grad_(True)
    tiled = torch.stack([s.repeat(4, 1)[:N] for s in sites]).to(dev).requires_grad_(True)
    xr, lr = padded(sites, N)
    xr = xr.to(dev).requires_grad_(True)
    lr = lr.to(dev)
    say(f"\n## 2. touch-shaped: B = {B} site clouds of [1000, {N}] points (mean {sizes.mean():.0f}) vs {N}-point "
        f"ground truths")
    t_tile = time_ms(fwd_bwd(tiled, gt), 10, args.repeats)
    t_rr = time_ms(fwd_bwd(xr, gt, lr, None), 10, args.repeats)
    r_tile = ptk_b200.ops.chamfer_rescued(tiled.detach(), gt.detach())
    r_rr = ptk_b200.ops.chamfer_rescued(xr.detach(), gt.detach(), lr, None)
    q_tile, q_rr = B * (N + N), int(lr.sum()) + B * N
    say(f"x4-tiled, cut to {N} points   {fmt(t_tile)}   rescued {r_tile} of {q_tile} queries "
        f"({100.0 * r_tile / q_tile:.1f} %)")
    say(f"ragged, untiled             {fmt(t_rr)}   rescued {r_rr} of {q_rr} valid queries "
        f"({100.0 * r_rr / q_rr:.1f} %)")
    say(f"ragged / tiled = {t_rr[0] / t_tile[0]:.3f}")
    del gt, tiled, xr

    # ---- 3
    B, P = 4, 100000
    lx = rng.integers(30000, P + 1, B)
    ly = rng.integers(30000, P + 1, B)
    x = (torch.from_numpy(rng.random((B, P, 3), np.float32)) - 0.5).to(dev).requires_grad_(True)
    y = (torch.from_numpy(rng.random((B, P, 3), np.float32)) - 0.5).to(dev).requires_grad_(True)
    lxt, lyt = torch.from_numpy(lx).to(dev), torch.from_numpy(ly).to(dev)
    xs = [x[b:b + 1, :lx[b]].detach().contiguous().requires_grad_(True) for b in range(B)]
    ys = [y[b:b + 1, :ly[b]].detach().contiguous().requires_grad_(True) for b in range(B)]
    work = float((lx.astype(np.float64) * ly).sum() / (B * P * P))
    say(f"\n## 3. pruned scan: B = {B}, clouds padded to {P} points, lengths in [30000, {P}] "
        f"({', '.join(f'{a}x{b}' for a, b in zip(lx, ly))})")
    t_rag = time_ms(fwd_bwd(x, y, lxt, lyt), 10, args.repeats)
    t_pad = time_ms(fwd_bwd(x, y), 10, args.repeats)
    t_loop = time_ms(per_pair(xs, ys), 10, args.repeats)
    say(f"ragged call               {fmt(t_rag)}")
    say(f"padded homogeneous call   {fmt(t_pad)}")
    say(f"per-pair loop ({B} calls)   {fmt(t_loop)}")
    say(f"work fraction (brute force) = {work:.3f}; time fraction ragged/padded = {t_rag[0] / t_pad[0]:.3f}")

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
