"""SHA-256 digests of every deterministic backward (ptk_*_bwd_det) on seeded inputs, plus the plain-store grad_p1 of
the default 1-NN and K-NN backward.  A change to the fixed-point scheme or to a backward kernel that alters one bit of
one gradient changes a digest; tests/test_det_bits_gpu.py reruns these cases against the committed digests and checks
each call's kernel launch count against include/ptk.h.

    python tools/det_bits.py [--out tests/data/det_bits.json]

Inputs come from numpy on the CPU (seeded per case), so the digests depend only on the library.  The indices are
drawn, not computed by a forward: any valid nearest-neighbour index exercises the backward the same way.  Outputs and
workspaces are pre-filled with a fixed garbage pattern, so a row the call failed to overwrite would show as well."""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import ptk_b200  # noqa: E402,F401
from ptk_b200 import _lib  # noqa: E402

OUT = os.path.join(ROOT, "tests", "data", "det_bits.json")
MEAN, SUM = 0, 1  # PTK_REDUCE_MEAN, PTK_REDUCE_SUM


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _i32(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.int32)).cuda()


def _lens(a):
    return None if a is None else torch.from_numpy(np.asarray(a, np.int64)).cuda()


def _out(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


def _ws(nbytes):
    return torch.full((max(int(nbytes), 256),), 0x5A, dtype=torch.uint8, device="cuda")


def _call(what, fn):
    """Run one ABI call; returns its kernel launch count."""
    before = _lib.launch_count()
    _lib.check(fn(), what)
    return _lib.launch_count() - before


def _nn_idx(rng, B, P, L_other, K=None):
    """Indices into the other cloud: < its length (0 when empty); K distinct ones per query for K-NN."""
    if K is None:
        return np.stack([rng.integers(0, max(L_other[b], 1), P) for b in range(B)]).astype(np.int32)
    idx = np.zeros((B, P, K), np.int32)
    for b in range(B):
        n = min(K, L_other[b])
        for i in range(P):
            idx[b, i, :n] = rng.permutation(L_other[b])[:n] if L_other[b] > 0 else []
    return idx


def _full(B, P):
    return [P] * B


# ------------------------------------------------------------------------------------------- Chamfer and its normal term
def _pair_case(entry, seed, B, P1, P2, lx, ly, reduction, want_x=True, want_y=True, nonfinite=False, normals=False):
    def run():
        rng = np.random.default_rng(seed)
        Lx, Ly = lx or _full(B, P1), ly or _full(B, P2)
        x = rng.standard_normal((B, P1, 3)).astype(np.float32)
        y = rng.standard_normal((B, P2, 3)).astype(np.float32)
        if normals:
            x[0, 1] = 0.0  # a zero normal: its norm is clamped
        if nonfinite:
            x[0, 2, 1] = np.inf
            y[B - 1, 0, 0] = np.nan
        ix, iy = _nn_idx(rng, B, P1, Ly), _nn_idx(rng, B, P2, Lx)
        g = rng.uniform(0.5, 2.0, B).astype(np.float32)
        xt, yt, ixt, iyt, gt = _f(x), _f(y), _i32(ix), _i32(iy), _f(g)
        gx, gy = (_out(B, P1, 3) if want_x else None), (_out(B, P2, 3) if want_y else None)
        lxt, lyt = _lens(lx), _lens(ly)
        L = _lib.lib()
        ws = _ws(L.ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2))
        fn = getattr(L, entry)
        n = _call(entry, lambda: fn(_p(xt), _p(yt), _p(lxt), _p(lyt), _p(ixt), _p(iyt), _p(gt), B, P1, P2, reduction,
                                    _p(gx), _p(gy), _p(ws), ws.numel(), _stream()))
        return [t for t in (gx, gy) if t is not None], n
    return run


# --------------------------------------------------------------------------------------------------------- 1-NN, K-NN
def _knn_case(seed, B, P1, P2, l1, l2, K, det=True, want1=True, want2=True, nonfinite=False):
    """K = None: ptk_knn1_bwd_det / ptk_knn1_bwd_lengths; otherwise ptk_knn_bwd_det / ptk_knn_bwd_lengths.  The default
    form's grad_p2 has run-to-run low bits, so only its grad_p1 is digested."""
    def run():
        rng = np.random.default_rng(seed)
        L1, L2 = l1 or _full(B, P1), l2 or _full(B, P2)
        p1 = rng.standard_normal((B, P1, 3)).astype(np.float32)
        p2 = rng.standard_normal((B, P2, 3)).astype(np.float32)
        idx = _nn_idx(rng, B, P1, L2, K)
        g = rng.uniform(-1.0, 1.0, idx.shape).astype(np.float32)
        if nonfinite:
            p1[0, 0, 2] = np.inf
            g[B - 1, 1] = np.nan
        a, b_, it, gt = _f(p1), _f(p2), _i32(idx), _f(g)
        g1, g2 = (_out(B, P1, 3) if want1 else None), (_out(B, P2, 3) if want2 else None)
        L = _lib.lib()
        la, lb = _lens(l1), _lens(l2)
        head = (_p(a), _p(b_), _p(la), _p(lb), _p(it), _p(gt), B, P1, P2)
        if det:
            ws = _ws(L.ptk_knn1_bwd_det_workspace_bytes(B, P1, P2))
            if K is None:
                n = _call("knn1_bwd_det", lambda: L.ptk_knn1_bwd_det(*head, _p(g1), _p(g2), _p(ws), ws.numel(), _stream()))
            else:
                n = _call("knn_bwd_det", lambda: L.ptk_knn_bwd_det(*head, K, _p(g1), _p(g2), _p(ws), ws.numel(), _stream()))
            return [t for t in (g1, g2) if t is not None], n
        if K is None:
            n = _call("knn1_bwd_lengths", lambda: L.ptk_knn1_bwd_lengths(*head, _p(g1), _p(g2), _stream()))
        else:
            n = _call("knn_bwd_lengths", lambda: L.ptk_knn_bwd_lengths(*head, K, _p(g1), _p(g2), _stream()))
        return [g1], n
    return run


# ------------------------------------------------------------------------------------------------------- point frames
def _frames_case(seed, B, P, K, lengths, mode, disambiguate=1, nonfinite=False):
    def run():
        rng = np.random.default_rng(seed)
        Ls = lengths or _full(B, P)
        pts = rng.standard_normal((B, P, 3)).astype(np.float32)
        pts[:, :, 2] *= 0.1  # roughly planar neighbourhoods
        idx = np.zeros((B, P, K), np.int32)
        dist = np.zeros((B, P, K), np.float32)
        for b in range(B):
            q = pts[b, :Ls[b]]
            d = ((q[:, None, :] - q[None, :, :]) ** 2).sum(-1)
            order = np.argsort(d, axis=1, kind="stable")[:, :K]
            n = order.shape[1]
            idx[b, :Ls[b], :n] = order
            dist[b, :Ls[b], :n] = np.take_along_axis(d, order, 1)
        gn = rng.standard_normal((B, P, 3)).astype(np.float32) if mode == "normals" else None
        gc = rng.standard_normal((B, P, 3)).astype(np.float32) if mode == "frames" else None
        gf = rng.standard_normal((B, P, 3, 3)).astype(np.float32) if mode == "frames" else None
        if nonfinite:
            (gn if gn is not None else gf)[0, 3, 0] = np.inf
        t = [None if v is None else _f(v) for v in (pts, dist, gn, gc, gf)]
        it, lt = _i32(idx), _lens(lengths)
        gp = _out(B, P, 3)
        L = _lib.lib()
        ws = _ws(L.ptk_knn1_bwd_det_workspace_bytes(B, P, P))
        n = _call("point_frames_bwd_det", lambda: L.ptk_point_frames_bwd_det(
            _p(t[0]), _p(lt), _p(it), _p(t[1]), B, P, K, disambiguate, _p(t[2]), _p(t[3]), _p(t[4]), _p(gp), _p(ws),
            ws.numel(), _stream()))
        return [gp], n
    return run


# ------------------------------------------------------------------------------------------------------------ samplers
def _mesh(rng, B, V, F):
    verts = rng.standard_normal((B, V, 3)).astype(np.float32)
    faces = np.stack([rng.choice(V, 3, replace=False) for _ in range(F)]).astype(np.int32)
    faces[0, 2] = faces[0, 1]  # a degenerate face lists a vertex twice
    return verts, faces


def _sample_case(seed, B, V, F, S, nonfinite=False):
    def run():
        rng = np.random.default_rng(seed)
        _, faces = _mesh(rng, B, V, F)
        fidx = rng.integers(0, F, (B, S)).astype(np.int32)
        uv = rng.random((2, B, S)).astype(np.float32)
        gp = rng.standard_normal((B, S, 3)).astype(np.float32)
        if nonfinite:
            gp[0, 5, 1] = np.inf
        gpt, ft, uvt, fat = _f(gp), _i32(fidx), _f(uv), _i32(faces)
        gv = _out(B, V, 3)
        L = _lib.lib()
        ws = _ws(L.ptk_sample_bwd_det_workspace_bytes(B, V))
        n = _call("sample_bwd_det", lambda: L.ptk_sample_bwd_det(_p(gpt), _p(ft), _p(uvt), _p(fat), B, V, F, S, _p(gv),
                                                                 _p(ws), ws.numel(), _stream()))
        return [gv], n
    return run


def _sample_normals_case(seed, B, V, F, S, with_pts=True, nonfinite=False):
    def run():
        rng = np.random.default_rng(seed)
        verts, faces = _mesh(rng, B, V, F)
        if nonfinite:
            verts[0, faces[3, 0], 0] = np.nan
        fidx = rng.integers(0, F, (B, S)).astype(np.int32)
        # samples on the degenerate face in mesh 0 only: its terms of size |g| / eps set M_b there and quantise every
        # other term of that mesh to 0, so the other meshes keep faces 1.. to give real sums
        fidx[1:] = rng.integers(1, F, (B - 1, S))
        fidx[0, :4] = 0
        uv = rng.random((2, B, S)).astype(np.float32)
        gp = rng.standard_normal((B, S, 3)).astype(np.float32) if with_pts else None
        gn = rng.standard_normal((B, S, 3)).astype(np.float32)
        vt, fat, ft, uvt, gnt = _f(verts), _i32(faces), _i32(fidx), _f(uv), _f(gn)
        gpt = None if gp is None else _f(gp)
        gv = _out(B, V, 3)
        L = _lib.lib()
        ws = _ws(L.ptk_sample_normals_bwd_det_workspace_bytes(B, V))
        n = _call("sample_normals_bwd_det", lambda: L.ptk_sample_normals_bwd_det(
            _p(vt), _p(fat), _p(ft), _p(uvt), _p(gpt), _p(gnt), B, V, F, S, _p(gv), _p(ws), ws.numel(), _stream()))
        return [gv], n
    return run


def _mesh_chamfer_case(seed, B, V, F, S, P2, repeat, want_verts=True, want_gt=True):
    def run():
        rng = np.random.default_rng(seed)
        _, faces = _mesh(rng, B, V, F)
        gt = rng.standard_normal((B, P2, 3)).astype(np.float32)
        pts = rng.standard_normal((repeat, B, S, 3)).astype(np.float32)
        fidx = rng.integers(0, F, (repeat, B, S)).astype(np.int32)
        ix = rng.integers(0, P2, (repeat, B, S)).astype(np.int32)
        iy = rng.integers(0, S, (repeat, B, P2)).astype(np.int32)
        uv = rng.random((repeat, 2, B, S)).astype(np.float32)
        gcd = rng.uniform(0.5, 2.0, B).astype(np.float32)
        t = [_f(gt), _f(pts), _i32(fidx), _i32(ix), _i32(iy), _f(uv), _i32(faces), _f(gcd)]
        gv, gg = (_out(B, V, 3) if want_verts else None), (_out(B, P2, 3) if want_gt else None)
        L = _lib.lib()
        ws = _ws(L.ptk_mesh_chamfer_bwd_det_workspace_bytes(B, V, F, S, P2))
        n = _call("mesh_chamfer_bwd_det", lambda: L.ptk_mesh_chamfer_bwd_det(
            *[_p(v) for v in t], B, V, F, S, P2, repeat, _p(gv), _p(gg), _p(ws), ws.numel(), _stream()))
        return [v for v in (gv, gg) if v is not None], n
    return run


def cases():
    """name -> (run, launches): run() returns (outputs, kernel launches of the call); `launches` is what include/ptk.h
    documents for that call (a memset is not a kernel launch)."""
    c = {}
    rag1, rag2 = [300, 0, 177, 64], [250, 120, 0, 1]  # pair 1: empty x cloud; pair 2: empty y cloud
    for entry, tag in (("ptk_chamfer_bwd_det", "chamfer"), ("ptk_chamfer_normals_bwd_det", "chamfer_normals")):
        nm = tag == "chamfer_normals"
        for red, rn in ((MEAN, "mean"), (SUM, "sum")):
            c[f"{tag}/full/{rn}"] = (_pair_case(entry, 11, 3, 700, 500, None, None, red, normals=nm), 3)
            c[f"{tag}/ragged/{rn}"] = (_pair_case(entry, 12, 4, 300, 250, rag1, rag2, red, normals=nm), 3)
        c[f"{tag}/ragged/x_only"] = (_pair_case(entry, 12, 4, 300, 250, rag1, rag2, MEAN, want_y=False, normals=nm), 3)
        c[f"{tag}/ragged/y_only"] = (_pair_case(entry, 12, 4, 300, 250, rag1, rag2, MEAN, want_x=False, normals=nm), 3)
        c[f"{tag}/ragged/nonfinite"] = (_pair_case(entry, 13, 4, 300, 250, rag1, rag2, SUM, nonfinite=True,
                                                   normals=nm), 3)
    for K in (None, 1, 2, 16, 64):
        tag = "knn1" if K is None else f"knn/K{K}"
        Kr = 1 if K is None else K
        r1, r2 = [300, 0, 177, 64], [250, 120, 0, max(Kr // 2, 1)]  # the last pair: l2 < K (for K > 1)
        c[f"{tag}/det/full"] = (_knn_case(21 + Kr, 3, 400, 520, None, None, K), 3)
        c[f"{tag}/det/ragged"] = (_knn_case(22 + Kr, 4, 300, 250, r1, r2, K), 3)
        c[f"{tag}/det/ragged/p1_only"] = (_knn_case(22 + Kr, 4, 300, 250, r1, r2, K, want2=False), 1)
        c[f"{tag}/det/ragged/p2_only"] = (_knn_case(22 + Kr, 4, 300, 250, r1, r2, K, want1=False), 3)
        c[f"{tag}/det/nonfinite"] = (_knn_case(23 + Kr, 4, 300, 250, r1, r2, K, nonfinite=True), 3)
        c[f"{tag}/default/ragged/p1"] = (_knn_case(22 + Kr, 4, 300, 250, r1, r2, K, det=False), 2)
        c[f"{tag}/default/ragged/p1_only"] = (_knn_case(22 + Kr, 4, 300, 250, r1, r2, K, det=False, want2=False), 1)
    fl = [400, 5, 0, 260]  # a cloud with l < K, an empty one
    c["point_frames/normals"] = (_frames_case(31, 4, 400, 8, fl, "normals"), 3)
    c["point_frames/frames"] = (_frames_case(32, 4, 400, 8, fl, "frames"), 3)
    c["point_frames/frames/no_disambiguate"] = (_frames_case(33, 3, 300, 16, None, "frames", disambiguate=0), 3)
    c["point_frames/normals/nonfinite"] = (_frames_case(34, 4, 400, 8, fl, "normals", nonfinite=True), 3)
    for V, where in ((500, "smem"), (3000, "global")):
        c[f"sample/{where}"] = (_sample_case(41, 3, V, 2 * V, 9000), 3)
        c[f"sample/{where}/nonfinite"] = (_sample_case(42, 3, V, 2 * V, 9000, nonfinite=True), 3)
        c[f"sample_normals/{where}"] = (_sample_normals_case(43, 3, V, 2 * V, 9000), 3)
        c[f"sample_normals/{where}/normals_only"] = (_sample_normals_case(44, 3, V, 2 * V, 9000, with_pts=False), 3)
        c[f"sample_normals/{where}/nonfinite"] = (_sample_normals_case(45, 3, V, 2 * V, 9000, nonfinite=True), 3)
    # 1 scale + per repeat: chamfer_bwd_det (3) and sample_bwd_det (3), plus one accumulate per gradient after the first
    c["mesh_chamfer/both"] = (_mesh_chamfer_case(51, 2, 600, 1100, 1500, 1200, 2), 1 + 6 + 8)
    c["mesh_chamfer/gt_only"] = (_mesh_chamfer_case(52, 2, 600, 1100, 1500, 1200, 2, want_verts=False), 1 + 3 + 4)
    return c


def digest(outputs):
    return [hashlib.sha256(t.detach().cpu().numpy().tobytes()).hexdigest() for t in outputs]


MIN_COVERAGE = 0.1


def coverage(outputs):
    """The smallest share of finite non-zero elements over the outputs: a digest of an output that is (nearly) all
    zeros would pin nothing of the accumulation it is meant to check."""
    return min(float((torch.isfinite(t) & (t != 0)).float().mean()) for t in outputs)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=OUT)
    args = ap.parse_args()
    torch.cuda.init()
    res, bad = {}, []
    for name, (run, launches) in cases().items():
        outs, n = run()
        torch.cuda.synchronize()
        if n != launches:
            bad.append(f"{name}: {n} kernel launches, include/ptk.h documents {launches}")
        if coverage(outs) < MIN_COVERAGE:
            bad.append(f"{name}: only {coverage(outs):.1%} of an output is finite and non-zero")
        res[name] = digest(outs)
    if bad:
        raise SystemExit("\n".join(bad))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"cases": res}, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"{len(res)} cases -> {args.out}")


if __name__ == "__main__":
    main()
