"""Cost of the point-cloud normals (ptk_point_frames_fwd / _bwd / _bwd_det) against the K-NN that feeds them and against
the eager torch composition a user would otherwise write on the same idx.  CUDA events after a warm-up; the rows of a
shape alternate within each round.

    python tools/point_normals_bench.py [--rounds 3] [--iters 20] [--out profiles/r10_point_normals.txt]

Rows per shape (K = 50, PyTorch3D's default neighborhood_size):
  knn fwd                    ptk_knn_fwd_lengths(points, points, K): the idx / dist the normals read
  normals fwd                ptk_point_frames_fwd, normals only
  normals bwd default / det  ptk_point_frames_bwd / ptk_point_frames_bwd_det under a gradient on the normals
  torch composition fwd+bwd  PyTorch3D 0.5.0's lines on the same idx: knn_gather, mean, covariance, linalg.eigh, the
                             sign rule, and torch autograd's backward of them.  linalg.eigh runs on torch's default
                             backend when it accepts the batch, on MAGMA otherwise (the backend is printed): cusolver's
                             batched syev has raised CUSOLVER_STATUS_INVALID_VALUE on these (N,3,3) float32 batches
Shapes: 16 x 10k (the ground-truth clouds of BASELINE config 3), 64 x 4000 (touch clouds), 32 x 6400 (the autoencoder's
output), 256 x 10k (points, idx and dist, 256 x 10k x 412 B = 1.05 GB, far beyond the 126 MB L2).  Prints the card's
name and power limit first; --out also writes what it prints."""
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

OUT = []


def say(s):
    print(s, flush=True)
    OUT.append(s)


def timeit(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def run_shape(name, B, P, K, rounds, iters):
    dev = torch.device("cuda")
    L = _lib.lib()
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    gen = torch.Generator(device=dev).manual_seed(0)
    # points on a bumpy surface patch per cloud (what depth / touch clouds look like), with a little noise
    uv = torch.rand(B, P, 2, device=dev, generator=gen)
    h = 0.1 * torch.sin(6 * uv[..., :1]) * torch.cos(4 * uv[..., 1:])
    pts = (torch.cat([uv, h], -1) + 1e-3 * torch.randn(B, P, 3, device=dev, generator=gen)).contiguous()
    dist = torch.empty(B, P, K, device=dev)
    idx = torch.empty(B, P, K, dtype=torch.int32, device=dev)
    wsk = torch.empty(max(L.ptk_knn_workspace_bytes(B, P, P, K), 16), dtype=torch.uint8, device=dev)
    nrm = torch.empty(B, P, 3, device=dev)
    gn = torch.randn(B, P, 3, device=dev, generator=gen)
    gp = torch.empty(B, P, 3, device=dev)
    wsd = torch.empty(L.ptk_knn1_bwd_det_workspace_bytes(B, P, P), dtype=torch.uint8, device=dev)

    def knn():
        _lib.check(L.ptk_knn_fwd_lengths(p(pts), p(pts), None, None, B, P, P, K, p(dist), p(idx), p(wsk), wsk.numel(),
                                         st()))

    knn()

    def fwd():
        _lib.check(L.ptk_point_frames_fwd(p(pts), None, p(idx), p(dist), B, P, K, 1, p(nrm), None, None, st()))

    def bwd_default():
        _lib.check(L.ptk_point_frames_bwd(p(pts), None, p(idx), p(dist), B, P, K, 1, p(gn), None, None, p(gp), st()))

    def bwd_det():
        _lib.check(L.ptk_point_frames_bwd_det(p(pts), None, p(idx), p(dist), B, P, K, 1, p(gn), None, None, p(gp),
                                              p(wsd), wsd.numel(), st()))

    xr = pts.clone().requires_grad_(True)
    i64 = idx.long()

    def torch_composition():  # estimate_pointcloud_local_coord_frames' lines on the given idx, normals only
        xr.grad = None
        knns = xr[:, :, None].expand(-1, -1, K, -1).gather(1, i64[..., None].expand(-1, -1, -1, 3))
        knns_c = knns - knns.mean(2, keepdim=True)
        cov = (knns_c[..., :, None] * knns_c[..., None, :]).mean(2)
        _, V = torch.linalg.eigh(cov)
        n = V[..., 0]
        df = knns - xr[:, :, None]
        n_pos = ((n[:, :, None] * df).sum(3) > 0).type_as(knns).sum(2, keepdim=True)
        flip = (n_pos < 0.5 * K).type_as(knns)
        ((1.0 - 2.0 * flip) * n).backward(gn)

    torch.backends.cuda.preferred_linalg_library("default")
    try:
        torch_composition()
        backend = "default"
    except RuntimeError:
        torch.backends.cuda.preferred_linalg_library("magma")
        backend = "magma"
    n_eager = max(iters // 5, 2)
    rows = {"knn fwd": (knn, iters), "normals fwd": (fwd, iters), "normals bwd default": (bwd_default, iters),
            "normals bwd det": (bwd_det, iters), "torch composition fwd+bwd": (torch_composition, n_eager)}
    res = {r: [] for r in rows}
    for r, (fn, _) in rows.items():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for r, (fn, n) in rows.items():
            res[r].append(timeit(fn, n))
    say(f"{name}: B={B} P={P} K={K}; torch linalg backend {backend}")
    med = {}
    for r, ts in res.items():
        med[r] = float(np.median(ts))
        say(f"  {r:28s} " + " ".join(f"{t:9.4f}" for t in ts) + f"   median {med[r]:9.4f} ms")
    ours = med["normals fwd"] + med["normals bwd default"]
    say(f"  fwd + default bwd {ours:.4f} ms = {ours / med['knn fwd']:.1%} of the knn fwd; torch composition / "
        f"(fwd + default bwd) = {med['torch composition fwd+bwd'] / ours:.1f} x")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    say("device: " + (q[0] if q else torch.cuda.get_device_name()) + f" | torch {torch.__version__}")
    for name, B, P in (("config 3 ground truth", 16, 10000), ("touch", 64, 4000), ("autoencoder output", 32, 6400),
                       ("256 x 10k", 256, 10000)):
        run_shape(name, B, P, 50, a.rounds, a.iters)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(OUT) + "\n")


if __name__ == "__main__":
    main()
