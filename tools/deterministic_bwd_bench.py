"""Cost of the deterministic backward (torch.use_deterministic_algorithms(True) -> ptk_*_bwd_det) against the default
fp32-atomic backward.  CUDA events; the modes alternate within each of three rounds.

    python tools/deterministic_bwd_bench.py [--rounds 3] [--iters 20]

  chamfer bwd         ptk_chamfer_bwd_lengths vs ptk_chamfer_bwd_det alone, 256 x 10k x 10k (bench.py's shape)
  chamfer fwd+bwd     ops.chamfer + backward at the same shape, flag off / on
  mesh chamfer        utils.chamfer_distance fwd + bwd at the config-3 shape (16 meshes of 1949 vertices, 2464 faces,
                      10k sampled points against 10k, repeat 3), flag off / on
  recon step          bench.py's config-3 reconstruction step (ChartDeformer, 3 GCN passes, Chamfer loss, Adam; synthetic
                      vertex features), flag off / flag on with torch's NaN fill of new tensors / flag on without it
Modes marked "fill" leave torch.utils.deterministic.fill_uninitialized_memory on (torch's default under the flag);
the others switch it off.  Prints the card's name and power limit first."""
import argparse
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # torch's condition for cuBLAS under the flag
import numpy as np  # noqa: E402
import torch  # noqa: E402

import ptk_b200  # noqa: E402
from ptk_b200 import _lib  # noqa: E402


def set_mode(mode):
    torch.use_deterministic_algorithms(mode != "default")
    torch.utils.deterministic.fill_uninitialized_memory = mode == "det+fill"


def timeit(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def compare(name, fns, rounds, iters):
    """fns: mode -> fn.  Warm every mode, then `rounds` rounds with the modes alternating."""
    res = {m: [] for m in fns}
    for m, fn in fns.items():
        set_mode(m)
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
    for _ in range(rounds):
        for m, fn in fns.items():
            set_mode(m)
            res[m].append(timeit(fn, iters))
    set_mode("default")
    base = np.median(res["default"])
    for m, ts in res.items():
        print(f"{name:18s} {m:10s} " + " ".join(f"{t:8.3f}" for t in ts) +
              f"   median {np.median(ts):8.3f} ms   x{np.median(ts) / base:5.2f}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("device:", q[0] if q else torch.cuda.get_device_name(), "| torch", torch.__version__, flush=True)
    dev = torch.device("cuda")
    L = _lib.lib()
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ---- Chamfer backward alone and fwd+bwd, 256 x 10k x 10k
    B, P = 256, 10000
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(B, P, 3, device=dev, generator=gen)
    y = torch.rand(B, P, 3, device=dev, generator=gen)
    g = torch.ones(B, device=dev) / B
    _, ix, iy = ptk_b200.ops.chamfer(x, y)
    gx, gy = torch.empty_like(x), torch.empty_like(y)
    ws = torch.empty(L.ptk_chamfer_bwd_det_workspace_bytes(B, P, P), dtype=torch.uint8, device=dev)

    def bwd_default():
        _lib.check(L.ptk_chamfer_bwd_lengths(p(x), p(y), None, None, p(ix), p(iy), p(g), B, P, P, _lib.REDUCE_MEAN, p(gx),
                                             p(gy), st()))

    def bwd_det():
        _lib.check(L.ptk_chamfer_bwd_det(p(x), p(y), None, None, p(ix), p(iy), p(g), B, P, P, _lib.REDUCE_MEAN, p(gx),
                                         p(gy), p(ws), ws.numel(), st()))
    # the working set (clouds, gradients, 48 B of accumulators per point) is larger than the L2: read from HBM
    compare("chamfer bwd", {"default": bwd_default, "det": bwd_det}, a.rounds, a.iters * 5)
    del ws

    xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)

    def fwd_bwd():
        xr.grad = yr.grad = None
        cham, _, _ = ptk_b200.ops.chamfer(xr, yr)
        cham.mean().backward()
    compare("chamfer fwd+bwd", {"default": fwd_bwd, "det": fwd_bwd, "det+fill": fwd_bwd}, a.rounds, a.iters)
    del x, y, xr, yr, gx, gy, ix, iy

    # ---- fused mesh Chamfer, config-3 shape
    adj = dict(np.load(os.path.join(ROOT, "tests", "golden", "adjacency.npz")))
    faces = torch.from_numpy(adj["p_faces"]).to(dev, torch.int64)
    verts = (torch.rand(16, 1949, 3, device=dev, generator=gen) * 0.5).requires_grad_(True)
    gt = torch.rand(16, 10000, 3, device=dev, generator=gen) * 0.5
    uni = [ptk_b200.utils.draw_uniforms(16, 10000, dev, gen) for _ in range(3)]

    def mesh():
        verts.grad = None
        (9000.0 * ptk_b200.utils.chamfer_distance(verts, faces, gt, num=10000, repeat=3, uniforms=uni).mean()).backward()
    compare("mesh chamfer", {"default": mesh, "det": mesh, "det+fill": mesh}, a.rounds, a.iters)

    # ---- the reconstruction step of bench.py (config 3, synthetic vertex features)
    import bench
    net, adj_info, vision, touch, feats, gtc = bench._recon_setup(torch, ptk_b200, dev, 0, 16)
    opt = torch.optim.Adam(net.parameters(), lr=0.0, fused=True)

    def step():
        opt.zero_grad(set_to_none=True)
        v = net(vision, touch, lambda it, _v: feats[it])
        loss, _ = ptk_b200.recon.recon_loss(v, adj_info["faces"], gtc, number_points=10000)
        loss.backward()
        opt.step()
    compare("recon step", {"default": step, "det": step, "det+fill": step}, a.rounds, max(a.iters // 2, 3))


if __name__ == "__main__":
    main()
