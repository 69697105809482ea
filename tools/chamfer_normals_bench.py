"""Cost of the Chamfer normal term (ptk_chamfer_normals_fwd / _bwd / _bwd_det) against the eager torch composition a
user would otherwise write, and against the Chamfer distance itself.  CUDA events after a warm-up; the rows of a shape
alternate within each of three rounds.

    python tools/chamfer_normals_bench.py [--rounds 3] [--iters 50]

Rows per shape:
  normals fwd               ptk_chamfer_normals_fwd alone, on the idx of one ops.chamfer call
  normals bwd default / det ptk_chamfer_normals_bwd / ptk_chamfer_normals_bwd_det alone
  torch composition fwd+bwd knn_gather of the nearest normals + F.cosine_similarity + masks + mean, and its backward
                            (torch autograd: gather and index_add with fp32 atomics)
  chamfer fwd+bwd           ops.chamfer(x, y) forward and backward, for scale
Shapes: 256 x 10k x 10k (bench.py's); the same batch ragged, lengths uniform in [2.5k, 10k]; 16 x 1949 x 10k (a
mesh's vertices against a sampled cloud).  "bytes" is the forward's compulsory traffic: per valid query its normal,
its idx and one gathered normal (28 B); "HBM" is that over 7.7 TB/s.  At 256 x 10k x 10k the normals, idx and
gradients (143 MB read by the forward) exceed the 126 MB L2.  Prints the card's name and power limit first."""
import argparse
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

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
    xn = F.normalize(torch.randn(B, P1, 3, device=dev, generator=gen), dim=2)
    yn = F.normalize(torch.randn(B, P2, 3, device=dev, generator=gen), dim=2)
    lx = ly = None
    if ragged:
        lx = torch.randint(P1 // 4, P1 + 1, (B,), device=dev, generator=gen)
        ly = torch.randint(P2 // 4, P2 + 1, (B,), device=dev, generator=gen)
    n1 = lx.sum().item() if ragged else B * P1
    n2 = ly.sum().item() if ragged else B * P2
    _, ix, iy = ptk_b200.ops.chamfer(x, y, lx, ly)
    cn = torch.empty(B, device=dev)
    g = torch.ones(B, device=dev) / B
    gx, gy = torch.empty_like(xn), torch.empty_like(yn)
    wsf = torch.empty(max(L.ptk_chamfer_normals_workspace_bytes(B, P1, P2), 16), dtype=torch.uint8, device=dev)
    wsd = torch.empty(L.ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2), dtype=torch.uint8, device=dev)
    red = _lib.REDUCE_MEAN

    def fwd():
        _lib.check(L.ptk_chamfer_normals_fwd(p(xn), p(yn), p(lx), p(ly), p(ix), p(iy), B, P1, P2, red, None, None, p(cn),
                                             p(wsf), wsf.numel(), st()))

    def bwd_default():
        _lib.check(L.ptk_chamfer_normals_bwd(p(xn), p(yn), p(lx), p(ly), p(ix), p(iy), p(g), B, P1, P2, red, p(gx), p(gy),
                                             st()))

    def bwd_det():
        _lib.check(L.ptk_chamfer_normals_bwd_det(p(xn), p(yn), p(lx), p(ly), p(ix), p(iy), p(g), B, P1, P2, red, p(gx),
                                                 p(gy), p(wsd), wsd.numel(), st()))

    xr, yr = xn.clone().requires_grad_(True), yn.clone().requires_grad_(True)
    ix64, iy64 = ix.long(), iy.long()
    ar1, ar2 = torch.arange(P1, device=dev), torch.arange(P2, device=dev)
    lxf = torch.full((B,), P1, device=dev) if lx is None else lx
    lyf = torch.full((B,), P2, device=dev) if ly is None else ly

    def torch_composition():  # PyTorch3D 0.5.0's lines on knn_points' idx, without its host-side length checks
        near_x = yr.gather(1, ix64[..., None].expand(-1, -1, 3)).masked_fill((lyf <= 0)[:, None, None], 0.0)
        near_y = xr.gather(1, iy64[..., None].expand(-1, -1, 3)).masked_fill((lxf <= 0)[:, None, None], 0.0)
        tx = (1 - F.cosine_similarity(xr, near_x, dim=2, eps=1e-6).abs()).masked_fill(ar1[None] >= lxf[:, None], 0.0)
        ty = (1 - F.cosine_similarity(yr, near_y, dim=2, eps=1e-6).abs()).masked_fill(ar2[None] >= lyf[:, None], 0.0)
        loss = (tx.sum(1) / lxf.clamp(min=1) + ty.sum(1) / lyf.clamp(min=1)).mean()
        xr.grad = yr.grad = None
        loss.backward()

    xc, yc = x.clone().requires_grad_(True), y.clone().requires_grad_(True)

    def chamfer_fwd_bwd():
        xc.grad = yc.grad = None
        c, _, _ = ptk_b200.ops.chamfer(xc, yc, lx, ly)
        c.mean().backward()

    rows = {"normals fwd": (fwd, iters), "normals bwd default": (bwd_default, iters), "normals bwd det": (bwd_det, iters),
            "torch composition fwd+bwd": (torch_composition, max(iters // 5, 3)),
            "chamfer fwd+bwd": (chamfer_fwd_bwd, max(iters // 10, 3))}
    res = {r: [] for r in rows}
    for r, (fn, _) in rows.items():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for r, (fn, n) in rows.items():
            res[r].append(timeit(fn, n))
    nbytes = (n1 + n2) * 28
    print(f"{name}: B={B} P1={P1} P2={P2} valid queries {n1} + {n2}; normals fwd bytes {nbytes / 1e6:.1f} MB "
          f"(>= {nbytes / HBM_BPS * 1e3:.4f} ms at 7.7 TB/s)", flush=True)
    for r, ts in res.items():
        med = float(np.median(ts))
        extra = f"   HBM {nbytes / (med * 1e-3) / HBM_BPS:6.1%}" if r == "normals fwd" else ""
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
