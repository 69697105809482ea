#!/usr/bin/env python
"""bench.py -- headline benchmark of the pterotactyl reconstruction hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): Chamfer pairs/s at 10k x 10k points.  One "step" = Chamfer forward + backward
(both directions, mean reduction, gradients w.r.t. both clouds) over a batch of 256 cloud pairs per GPU
(BASELINE.json north_star: "Chamfer (10k x 10k, batch 256)"; config 5 "fwd+bwd").  Weak scaling: each
rank owns 256 whole pairs, no data-path collective.

One JSON line on stdout (rank 0).  Besides the base contract it carries
  roofline      FP32 roofline of the dominant kernel (chamfer_nn_filter_kernel), timed live with CUDA
                events on the launching stream
  cpu_baseline  the CPU oracle (oracle/ptk_oracle.c, OpenMP) on a bounded sample of the same workload
  e2e           same metric through the host-buffer C ABI (ptk_host_chamfer): pinned host clouds ->
                H2D -> fwd+bwd -> D2H of the per-pair loss, copies inside the timed region
  extra         secondary numbers: GCN reconstruction steps/s (config 3 shape), sampler, aggregate GB/s

`--impl reference` times the reference arm: the CPU restatement of the reference's PyTorch3D path
(oracle port; PyTorch3D itself is not vendored/installable here) on all host threads, bounded sample.

`--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/<name>.npy, float32: the per-pair
Chamfer values and, at a fixed sample of (pair, point) positions, both nearest-neighbour index arrays and both gradient
clouds.  The inputs depend only on the arguments, so two builds can be compared output for output: the Chamfer values
and indices exactly, the gradients to a few ulps (the backward scatters them with float atomics, as PyTorch3D's does).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it
# NCCL_DEBUG is left as the launcher set it: whatever NCCL prints goes to stderr (run_ours dup2()s fd 1 onto fd 2
# while the job runs), stdout carries exactly one JSON line.

P = 10000           # points per cloud
B_PER_GPU = 256     # cloud pairs per GPU per step
NSETS = 4           # rotating input sets: 4 x 61 MB = 246 MB > 126 MB L2
FLOP_PER_EVAL = 8   # algorithmic: 3 sub + 3 mul + 2 add per (query, target) distance (SURVEY.md 8d)
DUMP_SAMPLE = 1 << 20  # (pair, point) positions of the per-point outputs --dump-outputs keeps: 34 MB of 82 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs:
        if a.impl != "ours":
            ap.error("--dump-outputs applies to the GPU path (--impl ours)")
        os.makedirs(a.dump_outputs, exist_ok=True)  # an unusable DIR fails here, before any GPU work
    return a


def dump_outputs(torch, d, cham, idx_x, idx_y, grad_x, grad_y):
    """What one Chamfer fwd+bwd step hands its caller, as float32 .npy files in `d`: the (B,) Chamfer values in full;
    the (B, P) indices and (B, P, 3) gradients at DUMP_SAMPLE (pair, point) positions drawn once with seed 0, in
    ascending flat order, the same for every run (indices < 2^24 are exact in float32)."""
    n = idx_x.numel()
    pos = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_SAMPLE, n), replace=False))
    sel = torch.from_numpy(pos).to(idx_x.device)
    out = {"cham": cham, "idx_x": idx_x.reshape(-1)[sel], "idx_y": idx_y.reshape(-1)[sel],
           "grad_x": grad_x.reshape(-1, 3)[sel], "grad_y": grad_y.reshape(-1, 3)[sel]}
    for name, t in out.items():
        np.save(os.path.join(d, name + ".npy"), t.float().cpu().numpy())


# --------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i",
                 str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_ready(self, timeout=5.0):
        """Block until nvidia-smi has delivered its first row (its start-up can take longer than the whole timed
        region on a fresh box), so that the timed region is guaranteed to be sampled."""
        t_end = time.time() + timeout
        while self.proc is not None and not self.rows and time.time() < t_end and self.proc.poll() is None:
            time.sleep(0.01)

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:  # no row inside the window: fall back to the rows of the warm-up right before it (same load)
            for ts, line in self.rows:
                if ts < t0 - 1.0:
                    continue
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------- CPU legs
def cpu_chamfer_leg(seconds_target, steps=None, warmup=0):
    """Oracle Chamfer fwd+bwd on a bounded sample: `bs` pairs of 10k x 10k per step, all host threads."""
    from oracle import oracle as orc
    orc.build()
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core it can
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    orc.set_num_threads(ncpu)
    threads = orc.num_threads()
    bs = max(2, min(B_PER_GPU, threads))
    rng = np.random.default_rng(0)
    x = (rng.random((bs, P, 3), np.float32) - 0.5).astype(np.float32)
    y = (rng.random((bs, P, 3), np.float32) - 0.5).astype(np.float32)
    g = np.ones(bs, np.float32)

    def step():
        cham, _, ix, _, iy = orc.chamfer_fwd(x, y, use_fma=True)
        orc.chamfer_bwd(x, y, ix, iy, g)
        return cham

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    n = 0
    while True:
        step()
        n += 1
        el = time.perf_counter() - t0
        if steps is not None:
            if n >= steps:
                break
        elif el >= seconds_target or n >= 50:
            break
    el = time.perf_counter() - t0
    return {"value": bs * n / el, "unit": "pairs/s", "cores": threads, "kind": "port",
            "sample": f"{n} step(s) x {bs} pairs of {P}x{P} points, Chamfer fwd+bwd, oracle/ptk_oracle.c "
                      f"(OpenMP, {threads} threads), {el:.1f} s"}, el, n, bs


def cpu_recon_leg(Bc=2):
    """The reference's reconstruction step restated with its own stack on the host (oracle/torch_ref.py: dense
    adjacency matmul exactly as GCN_layer.forward does, torch brute-force Chamfer): `Bc` objects, one step,
    all host threads.  A reported baseline for the GCN-step metric, not a target."""
    import torch
    from oracle import torch_ref as tr
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    gold = os.path.join(ROOT, "tests", "golden")
    adj = dict(np.load(os.path.join(gold, "adjacency.npz")))
    meshes = dict(np.load(os.path.join(gold, "meshes.npz")))

    def dense(tag):
        rp, col = adj[tag + "_rowptr"], adj[tag + "_col"]
        n = len(rp) - 1
        a = torch.zeros(n, n)
        deg = np.diff(rp)
        rows = np.repeat(np.arange(n), deg)
        a[torch.from_numpy(rows), torch.from_numpy(col.astype(np.int64))] = torch.from_numpy(
            np.repeat((1.0 / deg).astype(np.float32), deg))
        return a

    a0, a1 = dense("p_origional"), dense("p_adj")
    faces = torch.from_numpy(adj["p_faces"].astype(np.int64))
    gen = torch.Generator().manual_seed(0)
    sizes = [448] + [300] * 19 + [3]

    def make():
        ws, bs = [], []
        for i in range(20):
            stdv = 0.3 * 6.0 / np.sqrt(sizes[i] + 1)
            ws.append(((torch.rand(1, sizes[i], sizes[i + 1], generator=gen) * 2 - 1) * stdv).requires_grad_(True))
            bs.append(((torch.rand(sizes[i + 1], generator=gen) * 2 - 1) * 0.1).requires_grad_(True))
        return ws, bs

    w1, b1 = make()
    w2, b2 = make()
    vision = torch.from_numpy(meshes["vision_verts"])[None].repeat(Bc, 1, 1)
    touch = torch.rand(Bc, 125, 3, generator=gen) * 0.02 + 0.2
    feats = [torch.rand(Bc, 1824, 448, generator=gen), torch.rand(Bc, 1949, 448, generator=gen),
             torch.rand(Bc, 1949, 448, generator=gen)]
    gt = torch.nn.functional.normalize(torch.randn(Bc, 10000, 3, generator=gen), dim=-1) * 0.25
    t0 = time.perf_counter()
    verts = vision + tr.gcn_dense(feats[0], w1, b1, a0, 0.33)
    verts = torch.cat((verts, touch), 1)
    for it in (1, 2):
        upd = tr.gcn_dense(feats[it], w2, b2, a1, 0.33)
        verts = torch.cat((verts[:, :1824] + upd[:, :1824], verts[:, 1824:]), 1)
    cd = 0
    for _ in range(3):
        pts, _ = tr.batch_sample(verts, faces, torch.rand(Bc, 10000, generator=gen), torch.rand(2, Bc, 10000, generator=gen))
        cd = cd + tr.chamfer_autograd(pts, gt)
    (9000.0 * (cd / 3).mean()).backward()
    el = time.perf_counter() - t0
    return {"objects_per_s": Bc / el, "steps_per_s_at_16_objects": Bc / el / 16.0, "cores": ncpu, "kind": "port",
            "sample": f"1 step x {Bc} objects (fwd + 3 x 10k-point Chamfer loss + bwd), oracle/torch_ref.py "
                      f"(dense adjacency as the reference, torch CPU, {ncpu} threads), {el:.1f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    info, el, n, bs = cpu_chamfer_leg(None, steps=max(args.steps, 1), warmup=max(args.warmup, 0))
    line = {
        "impl": "reference", "metric": "chamfer_pairs_per_s_10k", "value": info["value"], "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": n, "warmup": max(args.warmup, 0), "ms_per_step": 1e3 * el / n,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": info,
        "e2e": {"value": info["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference arm = CPU restatement of the reference's PyTorch3D chamfer path (PyTorch3D 0.5.0 "
                "is not vendored in the reference tree and cannot be installed offline); all host threads",
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus):
    cfg = {"workload": f"Chamfer fwd+bwd, {P}x{P} points, batch {B_PER_GPU} pairs per GPU (BASELINE configs[4] "
                       f"cell P=10k,B=256; north_star target shape)",
           "points": P, "pairs_per_gpu": B_PER_GPU, "global_pairs": B_PER_GPU * n_gpus,
           "parallelism": f"object-sharded x{n_gpus}, no data-path collective",
           "l2_policy": f"rotating {NSETS} input sets ({NSETS * 2 * B_PER_GPU * P * 12 / 1e6:.0f} MB > 126 MB L2)"}
    return cfg


# --------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import ctypes as C

    import torch
    import torch.distributed as dist

    import ptk_b200
    from ptk_b200 import _lib

    # Everything libraries print while the job runs (NCCL banner, warnings) goes to stderr: stdout carries exactly
    # the one JSON line.  File descriptor 1 is restored right before that line is printed.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = ptk_b200.dist.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    info = _lib.device_info(local)
    K, W = args.steps, max(args.warmup, 3)
    B = B_PER_GPU

    def p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    # inputs resident in HBM: NSETS rotating sets of (x, y), x,y ~ U[-0.5, 0.5]^3, per-rank seeds
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    xs = [torch.rand(B, P, 3, device=dev, generator=gen) - 0.5 for _ in range(NSETS)]
    ys = [torch.rand(B, P, 3, device=dev, generator=gen) - 0.5 for _ in range(NSETS)]
    idx_x = torch.empty(B, P, dtype=torch.int32, device=dev)
    idx_y = torch.empty(B, P, dtype=torch.int32, device=dev)
    cham = torch.empty(B, device=dev)
    gcham = torch.full((B,), 1.0 / B, device=dev)
    gx = torch.empty(B, P, 3, device=dev)
    gy = torch.empty(B, P, 3, device=dev)
    ws = torch.empty(L.ptk_chamfer_workspace_bytes(B, P, P), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)

    def fwd(i):
        _lib.check(L.ptk_chamfer_fwd(p(xs[i % NSETS]), p(ys[i % NSETS]), B, P, P, None, p(idx_x), None, p(idx_y),
                                     p(cham), p(ws), ws.numel(), sp), "ptk_chamfer_fwd")

    def bwd(i):
        _lib.check(L.ptk_chamfer_bwd(p(xs[i % NSETS]), p(ys[i % NSETS]), p(idx_x), p(idx_y), p(gcham), B, P, P,
                                     p(gx), p(gy), sp), "ptk_chamfer_bwd")

    sampler = ClockSampler(local) if rank == 0 else None  # started before the warm-up: nvidia-smi needs time to come up
    for i in range(W):
        fwd(i); bwd(i)
    torch.cuda.synchronize()
    if sampler:
        sampler.wait_ready()
        fwd(0); bwd(0)  # untimed: the GPU is under load again when the timed region starts
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    launches0 = _lib.launch_count()
    t_wall0 = time.time()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(stream)
    for i in range(K):
        ev[i][0].record(stream)
        fwd(i)
        ev[i][1].record(stream)
        bwd(i)
        ev[i][2].record(stream)
    stop.record(stream)
    torch.cuda.synchronize()
    t_wall1 = time.time()
    launches = _lib.launch_count() - launches0  # kernels of libptk_b200.so launched inside the timed region, this rank
    if world > 1:
        dist.barrier()
        t = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        launches = int(t.item())
    total_ms = start.elapsed_time(stop)
    fwd_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    bwd_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:  # before the pruned-scan leg below reuses these buffers
        dump_outputs(torch, args.dump_outputs, cham, idx_x, idx_y, gx, gy)
    pairs_per_s = world * B * K / (total_ms * 1e-3)
    rescued = C.c_int64(0)  # queries of the last timed forward that the filter handed to the exact rescue scan
    _lib.check(L.ptk_chamfer_rescued(p(ws), B, P, P, C.byref(rescued), sp), "ptk_chamfer_rescued")

    # ---------------------------------------------------------------- end-to-end through the host ABI
    e2e = None
    hx = [torch.empty(B, P, 3).pin_memory() for _ in range(2)]
    hy = [torch.empty(B, P, 3).pin_memory() for _ in range(2)]
    for t in hx + hy:
        t.uniform_(-0.5, 0.5)
    hg = np.full(B, 1.0 / B, np.float32)
    hcham = torch.empty(B).pin_memory()
    ctx = ptk_b200.host.HostContext(local)
    out = {"cham": hcham.numpy()}
    ke = max(3, min(K, 10))
    for i in range(2):
        ctx.chamfer(hx[i % 2].numpy(), hy[i % 2].numpy(), grad_cham=hg, want_grad_x=False, want_grad_y=False, out=out)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(ke):
        ctx.chamfer(hx[i % 2].numpy(), hy[i % 2].numpy(), grad_cham=hg, want_grad_x=False, want_grad_y=False, out=out)
    e2e_s = time.perf_counter() - t0  # every call ends with a stream synchronise: host clock == device done
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": world * B * ke / e2e_s, "unit": "pairs/s", "h2d_bytes_per_step": 2 * B * P * 12 + B * 4,
           "d2h_bytes_per_step": B * 4, "steps": ke, "ms_per_step": 1e3 * e2e_s / ke,
           "api": "ptk_host_chamfer (C ABI, pinned host buffers; backward on device, loss read back)"}
    # the same call returning BOTH gradient clouds to the host as well (2 x 31 MB more D2H per step)
    hgx, hgy = torch.empty(B, P, 3).pin_memory(), torch.empty(B, P, 3).pin_memory()
    outg = {"cham": hcham.numpy(), "grad_x": hgx.numpy(), "grad_y": hgy.numpy()}
    for i in range(2):
        ctx.chamfer(hx[i % 2].numpy(), hy[i % 2].numpy(), grad_cham=hg, out=outg)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(ke):
        ctx.chamfer(hx[i % 2].numpy(), hy[i % 2].numpy(), grad_cham=hg, out=outg)
    e2eg_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2eg_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2eg_s = float(t.item())
    ctx.close()
    e2e["with_grads"] = {"value": world * B * ke / e2eg_s, "unit": "pairs/s", "ms_per_step": 1e3 * e2eg_s / ke,
                         "h2d_bytes_per_step": 2 * B * P * 12 + B * 4, "d2h_bytes_per_step": B * 4 + 2 * B * P * 12,
                         "note": "loss AND both (B,P,3) gradient clouds copied back to pinned host memory"}

    # ---------------------------------------------------------------- the same workload under the pruned scan
    # (PTK_CHAMFER_PRUNED: cell-sorted clouds + box hierarchy, bit-identical results, csrc/chamfer_pruned.cuh).  The
    # headline above stays on the brute-force scan north_star specifies and the roofline is quoted on (the default
    # PTK_CHAMFER_AUTO switches to the pruned scan only from 20k points per cloud); this is what the switch buys at 10k.
    pruned = None
    if not args.no_extra:
        try:
            ptk_b200.ops.set_chamfer_algo("pruned")
            kp = max(3, min(K, 10))
            for i in range(3):
                fwd(i); bwd(i)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            pe = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            pe[0].record(stream)
            for i in range(kp):
                fwd(i)
            pe[1].record(stream)
            for i in range(kp):
                fwd(i); bwd(i)
            pe[2].record(stream)
            torch.cuda.synchronize()
            p_fwd_ms, p_ms = pe[0].elapsed_time(pe[1]) / kp, pe[1].elapsed_time(pe[2]) / kp
            p_rescued = C.c_int64(0)
            _lib.check(L.ptk_chamfer_rescued(p(ws), B, P, P, C.byref(p_rescued), sp), "ptk_chamfer_rescued")
            ctx = ptk_b200.host.HostContext(local)
            for i in range(2):
                ctx.chamfer(hx[i % 2].numpy(), hy[i % 2].numpy(), grad_cham=hg, want_grad_x=False, want_grad_y=False, out=out)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for i in range(ke):
                ctx.chamfer(hx[i % 2].numpy(), hy[i % 2].numpy(), grad_cham=hg, want_grad_x=False, want_grad_y=False, out=out)
            p_e2e_s = time.perf_counter() - t0
            ctx.close()
            if world > 1:
                t = torch.tensor([p_ms, p_e2e_s], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                p_ms, p_e2e_s = float(t[0].item()), float(t[1].item())
            pruned = {"algo": "PTK_CHAMFER_PRUNED (ops.set_chamfer_algo('pruned')); indices, distances and Chamfer values "
                              "bit-identical to the brute-force scan (tests/test_chamfer_gpu.py)",
                      "ms_per_step": p_ms, "fwd_ms": p_fwd_ms, "value": world * B / (p_ms * 1e-3), "unit": "pairs/s",
                      "speedup_vs_headline": (total_ms / K) / p_ms,
                      "e2e": {"value": world * B * ke / p_e2e_s, "unit": "pairs/s", "ms_per_step": 1e3 * p_e2e_s / ke,
                              "h2d_bytes_per_step": 2 * B * P * 12 + B * 4, "d2h_bytes_per_step": B * 4},
                      "rescued_queries_frac": p_rescued.value / (2.0 * B * P)}
        except Exception as exc:  # secondary numbers must never lose the headline
            pruned = {"error": repr(exc)[:300]}
        finally:
            ptk_b200.ops.set_chamfer_algo("auto")

    recon = policy = None
    if not args.no_extra:  # collective measurements: every rank takes part
        try:
            recon = recon_step_measurement(torch, ptk_b200, dev, rank, world)
        except Exception as exc:  # secondary numbers must never lose the headline
            recon = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()
        try:
            policy = policy_measurement(torch, ptk_b200, dev, rank, world)
        except Exception as exc:
            policy = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------- roofline of the dominant kernel
    evals = 2.0 * B * P * P                      # both directions, per launch
    sm_max_mhz = (clocks or {}).get("sm_max_mhz") or info["clock_khz"] / 1e3
    peak_tflops = 2 * 128 * info["sm_count"] * sm_max_mhz * 1e6 / 1e12   # FP32 FMA peak of the chip
    achieved = FLOP_PER_EVAL * evals / (fwd_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "chamfer_scan_traffic.json")))
        if (tj["pairs"], tj["points"]) == (B, P):
            traffic, traffic_src = float(tj["dram_bytes_read"]) + float(tj["dram_bytes_write"]), tj["source"]
    except Exception:
        pass
    roofline = {
        "kernel": "chamfer_nn_filter_tma_kernel<8,16,128,4,1024> (the event pair also spans chamfer_bounds_kernel, chamfer_prep_kernel, the "
                  "exact rescue pass chamfer_nn_exact2_kernel and chamfer_finalize_kernel, ~2 % together)",
        "bound": "fp32", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s", "frac": achieved / peak_tflops,
        # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the scan kernel at this exact shape, read from the
        # committed summary of an `ncu --set full` capture (profiles/chamfer_scan_traffic.json names the capture);
        # null when that file does not cover this shape.  Algorithmic minimum: two clouds (61 MB) + their SoA copies
        # (82 MB) + 41 MB of keys: HBM is idle in this kernel.
        "traffic": traffic, "traffic_unit": "bytes per launch (ncu)", "traffic_source": traffic_src,
        "evals_per_s": evals / (fwd_ms * 1e-3), "ms_per_launch": fwd_ms,
        "rescued_queries_frac": rescued.value / (2.0 * B * P),
        "peak_source": f"derived, MEASURED_PEAKS.json has no FP32 entry: 2 flop x 128 FP32 lanes x {info['sm_count']} SMs x "
                       f"{sm_max_mhz:.0f} MHz (max SM clock). Algorithmic work = 8 flop x 2*B*P1*P2 distance evaluations "
                       f"per launch; the filter executes 3 FFMA (6 flop) per evaluation, so 100 % FMA-pipe time "
                       f"would read 1.33 here (ncu pipe utilisation: profiles/)",
    }
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak = 6650.0
    hbm_src = "fallback"
    if os.path.exists(peaks_path):
        try:
            hbm_peak = float(json.load(open(peaks_path))["hbm_gbs"]); hbm_src = "measured"
        except Exception:
            pass

    extra = {"fwd_ms": fwd_ms, "bwd_ms": bwd_ms, "bwd_hbm_gbs": (2 * B * P) * (12 + 4 + 12 + 12 + 12) / (bwd_ms * 1e-3) / 1e9,
             "device": torch.cuda.get_device_name(dev), "sm_count": info["sm_count"]}
    if pruned is not None:
        extra["pruned_scan"] = pruned
    if recon is not None:
        extra["recon_step"] = recon
    if policy is not None:
        extra["policy_scoring"] = policy
    if not args.no_extra:
        try:
            extra.update(extra_measurements(torch, ptk_b200, dev, hbm_peak, hbm_src))
        except Exception as exc:  # secondary numbers must never lose the headline
            extra["extra_error"] = repr(exc)

    cpu = None
    if not args.no_cpu:
        cpu, _, _, _ = cpu_chamfer_leg(10.0)
        if not args.no_extra and world == 1 and isinstance(extra.get("recon_step"), dict):
            try:
                extra["recon_step"]["cpu_baseline"] = cpu_recon_leg()
            except Exception as exc:
                extra["recon_step"]["cpu_baseline"] = {"error": repr(exc)[:200]}

    line = {
        "metric": "chamfer_pairs_per_s_10k", "value": pairs_per_s, "unit": "pairs/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic", "config": workload_config(world),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "roofline": roofline, "cpu_baseline": cpu, "extra": extra,
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _timeit_ranks(torch, fn, iters, warm, dev, world):
    """CUDA-event time per call of fn after `warm` untimed calls; barrier first, MAX over ranks."""
    import torch.distributed as dist
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / iters
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def _recon_setup(torch, ptk_b200, dev, rank, Bs, seed=0):
    """Config-3-shaped model + inputs for `Bs` objects on this rank (synthetic vertex features)."""
    import types
    from ptk_b200.graph import Graph
    gold = os.path.join(ROOT, "tests", "golden")
    adj = dict(np.load(os.path.join(gold, "adjacency.npz")))
    meshes = dict(np.load(os.path.join(gold, "meshes.npz")))
    args = types.SimpleNamespace(use_img=True, use_touch=True, finger=True, num_grasps=5, num_GCN_layers=20,
                                 hidden_GCN_size=300, cut=0.33)
    to = lambda a, dt: torch.from_numpy(a).to(dev, dt)
    g0 = Graph.from_csr(adj["p_origional_rowptr"], adj["p_origional_col"], dev)
    g = Graph.from_csr(adj["p_adj_rowptr"], adj["p_adj_col"], dev)
    adj_info = {"origional": g0.dense(), "adj": g.dense(), "faces": to(adj["p_faces"], torch.int64)}
    ptk_b200.graph.register(adj_info["origional"], g0)   # the dense tensors the reference's callers hold are never
    ptk_b200.graph.register(adj_info["adj"], g)          # scanned: their CSR is known (as utils.adj_init does)
    torch.manual_seed(seed)                                   # identical initial weights on every rank
    net = ptk_b200.recon.ChartDeformer(adj_info, args, 448).to(dev)
    gen = torch.Generator(device=dev).manual_seed(100 + rank)   # every rank owns different objects
    vision = to(meshes["vision_verts"], torch.float32)[None].repeat(Bs, 1, 1)
    touch = torch.rand(Bs, 125, 3, device=dev, generator=gen) * 0.02 + 0.2
    feats = [torch.rand(Bs, 1824, 448, device=dev, generator=gen), torch.rand(Bs, 1949, 448, device=dev, generator=gen),
             torch.rand(Bs, 1949, 448, device=dev, generator=gen)]
    gt = torch.nn.functional.normalize(torch.randn(Bs, 10000, 3, device=dev, generator=gen), dim=-1) * 0.25
    return net, adj_info, vision, touch, feats, gt


def _recon_e2e(torch, ptk_b200, dev, net, adj_info, vision, img_feats, Bs, time):
    """The reconstruction step the way the reference's loop runs it (vision/train.py:120-157): per step the batch the
    loader delivers -- touch charts (B,5,25,4: positions + mask token) and ground-truth clouds (B,10000,3) -- is copied
    from pinned host memory, the vertex features come from the fused front (positional MLP + mask-token embedding +
    pooled image features; the image features stand in for the CNN, which is out of scope, and stay on the device), the
    loss is read back (`loss.item()`, train.py:151).  Host clock around K steps."""
    torch.manual_seed(3)
    enc, menc = ptk_b200.Positional_Encoder(448).to(dev), ptk_b200.Mask_Encoder(448).to(dev)
    params = list(net.parameters()) + list(enc.parameters()) + list(menc.parameters())
    opt = torch.optim.Adam(params, lr=3e-4, fused=True)
    h_touch = torch.rand(Bs, 125, 4).pin_memory()
    h_touch[..., :3] = h_touch[..., :3] * 0.02 + 0.2
    h_touch[..., 3] = torch.randint(0, 3, (Bs, 125)).float()
    h_gt = (torch.nn.functional.normalize(torch.randn(Bs, 10000, 3), dim=-1) * 0.25).pin_memory()
    d_touch, d_gt = torch.empty(Bs, 125, 4, device=dev), torch.empty(Bs, 10000, 3, device=dev)
    vmask = 3 * torch.ones(Bs, 1824, 1, device=dev)

    def step():
        d_touch.copy_(h_touch, non_blocking=True)
        d_gt.copy_(h_gt, non_blocking=True)
        masks = [vmask, torch.cat((vmask, d_touch[..., 3:]), dim=1)]
        opt.zero_grad(set_to_none=True)
        verts = net(vision, d_touch[..., :3], lambda it, v: ptk_b200.encoders.vertex_features(
            enc, menc, v, masks[0 if it == 0 else 1], img_feats[it]))
        loss, _ = ptk_b200.recon.recon_loss(verts, adj_info["faces"], d_gt, number_points=10000)
        loss.backward()
        opt.step()
        return float(loss.item())

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    K = 10
    t0 = time.perf_counter()
    for _ in range(K):
        last = step()
    el = time.perf_counter() - t0
    # the same loop body replayed from one CUDA graph (the two host -> device copies are captured with it; the loss is
    # read back after every replay): what recon.GraphedStep, the recommended form of the loop, delivers end to end
    graph = None
    try:
        opt_g = torch.optim.Adam(params, lr=3e-4, fused=True, capturable=True)

        def step_g():
            d_touch.copy_(h_touch, non_blocking=True)
            d_gt.copy_(h_gt, non_blocking=True)
            masks = [vmask, torch.cat((vmask, d_touch[..., 3:]), dim=1)]
            opt_g.zero_grad(set_to_none=True)
            verts = net(vision, d_touch[..., :3], lambda it, v: ptk_b200.encoders.vertex_features(
                enc, menc, v, masks[0 if it == 0 else 1], img_feats[it]))
            loss, _ = ptk_b200.recon.recon_loss(verts, adj_info["faces"], d_gt, number_points=10000)
            loss.backward()
            opt_g.step()
            return loss

        graphed = ptk_b200.recon.GraphedStep(step_g)
        for _ in range(2):
            graphed()
            float(graphed.loss.item())
        t0 = time.perf_counter()
        for _ in range(K):
            graphed()
            last_g = float(graphed.loss.item())
        el_g = time.perf_counter() - t0
        graph = {"ms": 1e3 * el_g / K, "steps_per_s": K / el_g, "objects_per_s": Bs * K / el_g, "loss_last": last_g}
        del graphed
    except Exception as exc:
        graph = {"error": repr(exc)[:300]}
    return {"ms": 1e3 * el / K, "steps_per_s": K / el, "objects_per_s": Bs * K / el,
            "h2d_bytes_per_step": int(h_touch.numel() * 4 + h_gt.numel() * 4), "d2h_bytes_per_step": 4,
            "loss_last": last, "cuda_graph": graph,
            "note": "pinned host batch (touch charts + mask tokens + 10k-point clouds) -> device, fused vertex front "
                    "(positional MLP + mask embedding + resident image features), 3 GCN passes, Chamfer loss, backward, "
                    "Adam, loss.item(); includes the front's forward + backward, which the device-timed step above "
                    "replaces by synthetic features"}


def recon_step_measurement(torch, ptk_b200, dev, rank, world):
    """BASELINE configs[2]-shaped reconstruction step on EVERY rank: 3 GCN passes (448 -> 300 x 18 -> 3,
    N = 1824/1949/1949) + 3 x 10k-point Chamfer loss + backward + Adam; for world > 1 the parameter gradients go
    through the bucketed NCCL all-reduce that overlaps the backward (ptk_b200.dist).  Weak scaling (16 objects per
    GPU) and, for world > 1, strong scaling at the reference's global batch of 16 (16/world objects per GPU), both
    timed at the actual world size with the all-reduce inside.  The CNN/MLP vertex-feature encoders are out of
    scope: vertex features are synthetic."""
    info = ptk_b200._lib.device_info(dev.index or 0)
    fp32_peak = 2 * 128 * info["sm_count"] * info["clock_khz"] * 1e3 / 1e12
    flop_per_object = 3 * 2 * (1824 * (448 * 300 + 18 * 300 * 300 + 300 * 3) + 2 * 1949 * (448 * 300 + 18 * 300 * 300 + 300 * 3))

    def measure(Bs, global_objects):
        net, adj_info, vision, touch, feats, gt = _recon_setup(torch, ptk_b200, dev, rank, Bs)
        opt = torch.optim.Adam(net.parameters(), lr=3e-4, fused=True)
        reducer = ptk_b200.dist.GradReducer(net.parameters(), bucket_mb=4)

        def step():
            opt.zero_grad(set_to_none=True)
            verts = net(vision, touch, lambda it, v: feats[it])
            _, cd = ptk_b200.recon.recon_loss(verts, adj_info["faces"], gt, number_points=10000)
            loss = 9000.0 * cd.sum() / global_objects         # mean over the GLOBAL batch; gradients reduced with SUM
            loss.backward()
            reducer.finish()
            opt.step()
            return loss

        n0 = ptk_b200._lib.launch_count()
        step()
        launches = ptk_b200._lib.launch_count() - n0
        ms = _timeit_ranks(torch, step, 5, 2, dev, world)
        try:  # the same step with the Chamfer loss on the pruned scan (bit-identical loss and gradients; 10k-point clouds
            # are below the PTK_CHAMFER_AUTO threshold, so the numbers above use the brute-force scan)
            ptk_b200.ops.set_chamfer_algo("pruned")
            ms_pr = _timeit_ranks(torch, step, 5, 2, dev, world)
        finally:
            ptk_b200.ops.set_chamfer_algo("auto")
        return ms, launches, len(reducer.buckets), (net, adj_info, vision, touch, feats, gt, reducer), ms_pr

    Bs = 16
    ms, launches, nb, state, ms_pr = measure(Bs, Bs * world)
    out = {"shape": "v_t_p GCN part: 16 objects per GPU, 3 x (448->300x18->3), N=1824/1949/1949, 3 x 10k-point "
                    "Chamfer loss, fwd+bwd+Adam; synthetic vertex features (CNN/MLP encoders out of scope)",
           "n_gpus": world, "ms": ms, "steps_per_s": 1e3 / ms, "objects_per_s": world * Bs * 1e3 / ms,
           "ptk_launches_per_step": launches,
           "grad_allreduce": (f"{nb} NCCL buckets overlapped with backward" if world > 1 else "none (1 GPU)")}
    out["gemm_tflops_per_gpu"] = Bs * flop_per_object / (ms * 1e-3) / 1e12
    # north_star's yardstick for the step: algorithmic GEMM flop (SURVEY 8d: 964 GFLOP per step at 16 objects) over
    # the chip's FP32 FMA peak.  The backward GEMMs run on the tensor cores, so this is a throughput fraction, not a
    # pipe utilisation; aggregation, Chamfer and optimizer time count against it.
    out["fp32_peak_tflops"] = fp32_peak
    out["fp32_roofline_frac"] = out["gemm_tflops_per_gpu"] / fp32_peak
    out["pruned_chamfer"] = {"ms": ms_pr, "steps_per_s": 1e3 / ms_pr, "objects_per_s": world * Bs * 1e3 / ms_pr,
                             "fp32_roofline_frac": Bs * flop_per_object / (ms_pr * 1e-3) / 1e12 / fp32_peak,
                             "note": "ops.set_chamfer_algo('pruned'): the 3 x 10k-point Chamfer losses on the pruned scan, "
                                     "everything else unchanged; loss and gradients are bit-identical"}
    net, adj_info, vision, touch, feats, gt, reducer = state
    graphed = None
    try:  # the same step replayed from one CUDA graph per rank (launch gaps and Python overhead removed); for world > 1
        # the bucketed NCCL all-reduces are captured with it (tools/graph_ddp_check.py: gradients equal the eager step's)
        opt_g = torch.optim.Adam(net.parameters(), lr=3e-4, fused=True, capturable=True)

        def step_g():
            opt_g.zero_grad(set_to_none=True)
            verts = net(vision, touch, lambda it, v: feats[it])
            _, cd = ptk_b200.recon.recon_loss(verts, adj_info["faces"], gt, number_points=10000)
            loss = 9000.0 * cd.sum() / (Bs * world)
            loss.backward()
            reducer.finish()
            opt_g.step()
            return loss

        graphed = ptk_b200.recon.GraphedStep(step_g)
        msg = _timeit_ranks(torch, graphed, 10, 2, dev, world)
        out["ms_cuda_graph"] = msg
        out["steps_per_s_cuda_graph"] = 1e3 / msg
        out["objects_per_s_cuda_graph"] = world * Bs * 1e3 / msg
        out["fp32_roofline_frac_cuda_graph"] = Bs * flop_per_object / (msg * 1e-3) / 1e12 / fp32_peak
    except Exception as exc:
        out["cuda_graph_error"] = repr(exc)[:300]
    finally:
        graphed = None          # a live graph with captured NCCL kernels blocks destroy_process_group()
        torch.cuda.synchronize()
    if world == 1:
        try:  # what bit-level ReLU-mask parity costs: the same step with the tensor-core (3xTF32) training forward
            saved = ptk_b200.ops.algo["fwd_train"]
            ptk_b200.ops.algo["fwd_train"] = ptk_b200.ops.GEMM_AUTO  # tcgen05 wherever the kernel accepts the shape
            opt2 = torch.optim.Adam(net.parameters(), lr=3e-4, fused=True)

            def step_tc():
                opt2.zero_grad(set_to_none=True)
                verts = net(vision, touch, lambda it, v: feats[it])
                loss, _ = ptk_b200.recon.recon_loss(verts, adj_info["faces"], gt, number_points=10000)
                loss.backward()
                opt2.step()
                return loss

            ms_tc = _timeit_ranks(torch, step_tc, 5, 2, dev, world)
            out["tensor_core_forward"] = {
                "ms": ms_tc, "steps_per_s": 1e3 / ms_tc, "fp32_roofline_frac": Bs * flop_per_object / (ms_tc * 1e-3) / 1e12 / fp32_peak,
                "note": "ops.algo['fwd_train'] = GEMM_AUTO: forward GEMMs on tcgen05 (3xTF32, error vs fp64 below "
                        "the FP32 kernels') -- not the default because a 1e-6 perturbation flips individual ReLUs and "
                        "the 1e-5 gradient parity against the reference's fp32 run is then lost (SURVEY H1)"}
        except Exception as exc:
            out["tensor_core_forward"] = {"error": repr(exc)[:300]}
        finally:
            ptk_b200.ops.algo["fwd_train"] = saved
        try:  # end to end: what a data loader delivers starts in pinned host memory, the loss is read back every step
            import time
            out["e2e"] = _recon_e2e(torch, ptk_b200, dev, net, adj_info, vision, feats, Bs, time)
        except Exception as exc:
            out["e2e"] = {"error": repr(exc)[:300]}
    del state, net, adj_info, vision, touch, feats, gt, reducer
    torch.cuda.empty_cache()
    if world > 1 and 16 % world == 0:
        try:
            Bl = 16 // world
            ms_s, launches_s, _, st, _ = measure(Bl, 16)
            del st
            out["strong_scaling_global_16"] = {
                "objects_per_gpu": Bl, "ms": ms_s, "steps_per_s": 1e3 / ms_s, "objects_per_s": 16 * 1e3 / ms_s,
                "note": "the reference's global batch of 16 split over the ranks, NCCL gradient all-reduce inside the "
                        "timed step, max over ranks (SURVEY 8e: kernels are latency-bound below ~8 objects per GPU)"}
        except Exception as exc:
            out["strong_scaling_global_16"] = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()
    return out


def policy_measurement(torch, ptk_b200, dev, rank, world):
    """BASELINE configs[3] as ONE call on every rank: 32 environments x 50 candidate actions -> no-grad deformation GCN
    (3 passes, tensor-core forward) -> 3 x (10k-point sampling + Chamfer) -> masked arg-min, the 1600 candidates
    sharded over the ranks, one all-gather of the score vector (ptk_b200.policy.best_step_batched)."""
    E, A = 32, 50
    chunk = 200
    net, adj_info, vision, touch, feats, _ = _recon_setup(torch, ptk_b200, dev, 0, chunk)  # same candidates on every rank
    net.eval()
    gen = torch.Generator(device=dev).manual_seed(7)
    charts = {"vision_charts": vision[:1].repeat(E, 1, 1),
              "touch_charts": (touch[:1, None].repeat(E, A, 1, 1) + 0.01 * torch.rand(E, A, 1, 3, device=dev, generator=gen))}
    gtp = torch.nn.functional.normalize(torch.randn(E, 10000, 3, device=dev, generator=gen), dim=-1) * 0.25
    maskp = (torch.rand(E, A, device=dev, generator=gen) < 0.1).to(torch.int64)

    def deform(img, ch):
        n = ch["vision_charts"].shape[0]
        return net(ch["vision_charts"], ch["touch_charts"], lambda it, v: feats[it][:n])

    def call():
        return ptk_b200.policy.best_step_batched(deform, None, charts, gtp, adj_info["faces"], mask=maskp, num=10000,
                                                 chunk=chunk, shard=world > 1)

    n0 = ptk_b200._lib.launch_count()
    call()
    launches = ptk_b200._lib.launch_count() - n0
    ms = _timeit_ranks(torch, call, 3, 1, dev, world)
    try:  # the same call with the 3 x 1600 Chamfer evaluations on the pruned scan (same scores, same arg-min)
        ptk_b200.ops.set_chamfer_algo("pruned")
        ms_pr = _timeit_ranks(torch, call, 3, 1, dev, world)
    finally:
        ptk_b200.ops.set_chamfer_algo("auto")
    # scoring alone (candidate meshes given), sharded the same way: what round 1 reported
    cand = torch.cat([vision[:1], touch[:1]], 1).repeat(E * A, 1, 1).reshape(E, A, -1, 3)
    cand = cand * (1.0 + 0.01 * torch.rand(E, A, 1, 1, device=dev, generator=gen))
    ms_score = _timeit_ranks(torch, lambda: ptk_b200.policy.best_actions(
        ptk_b200.policy.score_candidates(cand, adj_info["faces"], gtp, num=10000, shard=world > 1), maskp), 3, 1, dev, world)
    return {"shape": "BASELINE configs[3]: 32 envs x 50 actions = 1600 candidates (V=1949, F=2464): deformation GCN "
                     "(3 x 20 layers, no grad) + 3 x 10k-point samplings + Chamfer each + masked arg-min, one call",
            "n_gpus": world, "sharded": world > 1, "ms": ms, "candidates_per_s": E * A / (ms * 1e-3),
            "ptk_launches_per_call_per_rank": launches,
            "pruned_chamfer": {"ms": ms_pr, "candidates_per_s": E * A / (ms_pr * 1e-3)},
            "scoring_only": {"ms": ms_score, "candidates_per_s": E * A / (ms_score * 1e-3),
                             "note": "sample + Chamfer + arg-min on given candidate meshes (no GCN)"}}


def extra_measurements(torch, ptk_b200, dev, hbm_peak, hbm_src):
    """Secondary numbers (not the headline): config-3-shaped GCN reconstruction step, sampler, aggregate."""
    import types
    from ptk_b200.graph import Graph
    out = {}
    gold = os.path.join(ROOT, "tests", "golden")
    adj = dict(np.load(os.path.join(gold, "adjacency.npz")))
    meshes = dict(np.load(os.path.join(gold, "meshes.npz")))

    def timeit(fn, iters, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    # --- GCN aggregate at a batch that spills L2 (B=256, N=1949, C=300, L=99): HBM roofline
    g = Graph.from_csr(adj["p_adj_rowptr"], adj["p_adj_col"], dev)
    Bh, C_, L_ = 256, 300, 99
    H = torch.rand(Bh, g.n, C_, device=dev)
    bias = torch.rand(C_, device=dev)
    o = torch.empty_like(H)
    ms = timeit(lambda: ptk_b200.ops._aggregate(g, H, L_, bias, True, out=o), 20)
    alg = Bh * g.n * C_ * 4 * 2 + g.nnz * 8 + (g.n + 1) * 4
    out["gcn_aggregate"] = {"shape": f"B={Bh} N={g.n} C={C_} L={L_} (fwd, bias+ReLU fused)", "ms": ms,
                            "achieved_gbs": alg / (ms * 1e-3) / 1e9, "peak_gbs": hbm_peak, "peak_source": hbm_src,
                            "frac": alg / (ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": alg}
    # ... and the full-propagate layer (L = C = 300: output layer of the autoencoder encoder / the DDQN graph model)
    ms_w = timeit(lambda: ptk_b200.ops._aggregate(g, H, C_, bias, False, out=o), 20)
    out["gcn_aggregate"]["wide_layer"] = {"shape": f"B={Bh} N={g.n} C=L={C_}", "ms": ms_w,
                                          "achieved_gbs": alg / (ms_w * 1e-3) / 1e9,
                                          "frac": alg / (ms_w * 1e-3) / 1e9 / hbm_peak}
    del H, o

    # (the config-3-shaped reconstruction step is measured by recon_step_measurement() on every rank)
    args = types.SimpleNamespace(use_img=True, use_touch=True, finger=True, num_grasps=5, num_GCN_layers=20,
                                 hidden_GCN_size=300, cut=0.33)
    to = lambda a, dt: torch.from_numpy(a).to(dev, dt)
    adj_info = {"origional": Graph.from_csr(adj["p_origional_rowptr"], adj["p_origional_col"], dev).dense(),
                "adj": g.dense(), "faces": to(adj["p_faces"], torch.int64)}
    Bs = 16
    vision = to(meshes["vision_verts"], torch.float32)[None].repeat(Bs, 1, 1)
    touch = torch.rand(Bs, 125, 3, device=dev) * 0.02 + 0.2
    # --- sampler (B=16, V=1949, F=2464, S=10000)
    faces32 = adj_info["faces"].to(torch.int32)
    verts = torch.cat([vision, touch], 1)
    uf = torch.rand(Bs, 10000, device=dev)
    uv = torch.rand(2, Bs, 10000, device=dev)
    ms = timeit(lambda: ptk_b200.ops.sample_points(verts, faces32, uf, uv), 20)
    out["sampler"] = {"shape": "B=16 V=1949 F=2464 S=10000", "ms": ms}

    # --- fused vertex-feature front (config-3 shape: 16 x 1949 vertices, input_size 448): positions -> GCN layer-0 input in one
    # launch, next to the same modules on the unfused path (embedding kernel + torch Linear / Embedding / adds = library GEMMs)
    import copy
    torch.manual_seed(1)
    enc, menc = ptk_b200.Positional_Encoder(448).to(dev), ptk_b200.Mask_Encoder(448).to(dev)
    enc_u, menc_u = copy.deepcopy(enc), copy.deepcopy(menc)
    enc_u.fused = False
    pos = verts.clone().requires_grad_(True)
    mask = torch.randint(0, 4, (Bs, 1949, 1), device=dev).float()
    img = torch.rand(Bs, 1949, 448, device=dev)
    w = torch.rand(Bs, 1949, 448, device=dev)

    def front(e, m, train):
        def fn():
            if train:
                pos.grad = None
                e.zero_grad(set_to_none=True)
                m.zero_grad(set_to_none=True)
                (ptk_b200.encoders.vertex_features(e, m, pos, mask, img) * w).sum().backward()
            else:
                with torch.no_grad():
                    ptk_b200.encoders.vertex_features(e, m, pos, mask, img)
        return fn
    torch.backends.cuda.matmul.allow_tf32 = False
    out["vertex_front"] = {
        "shape": "M = 16 x 1949 vertices, 63 -> 112 -> 224 -> 448 (+ mask-token row + image features), FP32",
        "fwd_ms": timeit(front(enc, menc, False), 20), "fwd_bwd_ms": timeit(front(enc, menc, True), 10),
        "unfused_fwd_ms": timeit(front(enc_u, menc_u, False), 20), "unfused_fwd_bwd_ms": timeit(front(enc_u, menc_u, True), 10),
        "note": "fused: ptk_vertex_front_fwd (one launch); unfused: ptk_nerf_embed + three cuBLAS FP32 GEMMs + elementwise kernels"}

    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
