"""Dev tool: Chamfer forward time of the brute-force filter scan for cloud layouts off the aligned fast path.
    python tools/chamfer_layout_bench.py
The exact recheck reads each query's recorded chunk with vector loads only when every cloud of the batch is 16-byte
aligned; these rows time a batch with P not a multiple of 4 (odd clouds start 4 or 8 bytes past a 16-byte boundary)
and a view whose storage starts 4 bytes into its allocation, next to an aligned control."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import ptk_b200

dev = torch.device("cuda")
ptk_b200.ops.set_chamfer_algo("filter")


def timeit(fn, iters):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def clouds(B, P, offset, g):
    buf = torch.rand(B * P * 3 + offset, device=dev, generator=g) - 0.5
    return buf[offset:].view(B, P, 3)


print(f"{'case':<34} {'B':>4} {'P':>6} {'fwd ms':>9}")
for name, B, P, off in (("aligned", 256, 10000, 0), ("P % 4 != 0", 256, 9999, 0), ("storage offset 4 bytes", 256, 10000, 1),
                        ("aligned", 4, 10000, 0), ("P % 4 != 0", 4, 9999, 0), ("storage offset 4 bytes", 4, 10000, 1)):
    g = torch.Generator(device=dev).manual_seed(P + B)
    x, y = clouds(B, P, off, g), clouds(B, P, off, g)
    with torch.no_grad():
        ms = timeit(lambda: ptk_b200.ops.chamfer(x, y), max(3, min(30, int(2e11 / (B * P * P)))))
    print(f"{name:<34} {B:4d} {P:6d} {ms:9.3f}", flush=True)
