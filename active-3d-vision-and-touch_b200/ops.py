"""torch.autograd bindings over the C ABI (include/ptk.h).  Tensors are only used for device memory,
streams and autograd bookkeeping; all arithmetic of the hot path runs in libptk_b200.so.

There is NO CPU / eager fallback: CPU tensors are rejected with a RuntimeError.
"""
import ctypes as C

import torch

from . import _lib
from .graph import Graph, graph_of


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "ptk_b200 ops run on CUDA (sm_100a) tensors only; got a CPU tensor. There is no CPU fallback.")


def _f32c(t):
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


# ------------------------------------------------------------------------------------- Chamfer / KNN
def set_chamfer_algo(name):
    """'filter' (3-FFMA expansion filter + exact recheck), 'exact' (6-op scan), 'pruned' (cell-sorted clouds + box
    hierarchy, a few hundred evaluations per query) or 'auto' (the default: pruned when both clouds have >= 20k points,
    filter otherwise); all return the same bits."""
    algo = {"filter": _lib.CHAMFER_FILTER, "exact": _lib.CHAMFER_EXACT, "pruned": _lib.CHAMFER_PRUNED,
            "auto": _lib.CHAMFER_AUTO}[name]
    _lib.check(_lib.lib().ptk_chamfer_set_algo(algo), "ptk_chamfer_set_algo")


_REDUCTIONS = {"mean": _lib.REDUCE_MEAN, "sum": _lib.REDUCE_SUM}


def _lengths(lengths, B, device, name):
    """Per-cloud lengths as a contiguous int64 (B,) device tensor, or None.  No host synchronisation: the values are
    clamped to [0, P] by the kernels."""
    if lengths is None:
        return None
    if not torch.is_tensor(lengths) or lengths.dtype not in (torch.int32, torch.int64):
        raise ValueError(f"{name} must be an int32 or int64 tensor")
    if lengths.shape != (B,):
        raise ValueError(f"{name} must have shape ({B},), got {tuple(lengths.shape)}")
    return lengths.to(device=device, dtype=torch.int64, non_blocking=True).contiguous()


def _check_pair(x, y):
    if x.dim() != 3 or y.dim() != 3 or x.shape[2] != 3 or y.shape[2] != 3:
        raise ValueError(f"Expected (B,P,3) point clouds, got {tuple(x.shape)} and {tuple(y.shape)}")
    if x.shape[0] != y.shape[0]:
        raise ValueError("y must have the same batch dimension as x")


def chamfer_rescued(x, y, x_lengths=None, y_lengths=None):
    """Diagnostics: run the forward NN scan on (x, y) and return how many of the B*(P1+P2) queries the
    filter could not decide (near or exact ties across chunks) and handed to the exact rescue scan.
    x_lengths / y_lengths: a ragged batch, as in chamfer()."""
    _need_cuda(x, y)
    x, y = _f32c(x), _f32c(y)
    B, P1, _ = x.shape
    P2 = y.shape[1]
    lx, ly = _lengths(x_lengths, B, x.device, "x_lengths"), _lengths(y_lengths, B, x.device, "y_lengths")
    L = _lib.lib()
    idx_x = torch.empty(B, P1, dtype=torch.int32, device=x.device)
    idx_y = torch.empty(B, P2, dtype=torch.int32, device=x.device)
    cham = torch.empty(B, dtype=torch.float32, device=x.device)
    ws = _ws(L.ptk_chamfer_workspace_bytes(B, P1, P2), x.device)
    n = C.c_int64(0)
    with torch.cuda.device(x.device):
        _lib.check(L.ptk_chamfer_fwd_lengths(_p(x), _p(y), _p(lx), _p(ly), B, P1, P2, _lib.REDUCE_MEAN, None, _p(idx_x),
                                             None, _p(idx_y), _p(cham), _p(ws), ws.numel(), _stream()),
                   "ptk_chamfer_fwd_lengths")
        _lib.check(L.ptk_chamfer_rescued(_p(ws), B, P1, P2, C.byref(n), _stream()), "ptk_chamfer_rescued")
    return int(n.value)


class _Chamfer(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, lx, ly, reduction):
        _need_cuda(x, y)
        x, y = _f32c(x), _f32c(y)
        _check_pair(x, y)
        B, P1, _ = x.shape
        P2 = y.shape[1]
        lx, ly = _lengths(lx, B, x.device, "x_lengths"), _lengths(ly, B, x.device, "y_lengths")
        L = _lib.lib()
        idx_x = torch.empty(B, P1, dtype=torch.int32, device=x.device)
        idx_y = torch.empty(B, P2, dtype=torch.int32, device=x.device)
        cham = torch.empty(B, dtype=torch.float32, device=x.device)
        nb = L.ptk_chamfer_workspace_bytes(B, P1, P2)
        ws = _ws(nb, x.device)
        with torch.cuda.device(x.device):
            _lib.check(L.ptk_chamfer_fwd_lengths(_p(x), _p(y), _p(lx), _p(ly), B, P1, P2, reduction, None, _p(idx_x),
                                                 None, _p(idx_y), _p(cham), _p(ws), ws.numel(), _stream()),
                       "ptk_chamfer_fwd_lengths")
        ctx.save_for_backward(x, y, idx_x, idx_y, lx, ly)
        ctx.reduction = reduction
        ctx.mark_non_differentiable(idx_x, idx_y)
        return cham, idx_x, idx_y

    @staticmethod
    def backward(ctx, g, _gi, _gj):
        x, y, idx_x, idx_y, lx, ly = ctx.saved_tensors
        B, P1, _ = x.shape
        P2 = y.shape[1]
        g = _f32c(g)
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(y) if ctx.needs_input_grad[1] else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().ptk_chamfer_bwd_lengths(_p(x), _p(y), _p(lx), _p(ly), _p(idx_x), _p(idx_y), _p(g), B,
                                                          P1, P2, ctx.reduction, _p(gx), _p(gy), _stream()),
                       "ptk_chamfer_bwd_lengths")
        return gx, gy, None, None, None


def chamfer(x, y, x_lengths=None, y_lengths=None, point_reduction="mean"):
    """cham (B,), idx_x (B,P1) int32, idx_y (B,P2) int32.  Differentiable w.r.t. x and y.

    x_lengths / y_lengths (B,) int32 or int64, on any device: only x[b, :x_lengths[b]] and y[b, :y_lengths[b]] exist
    (ragged batch, values clamped to [0, P]).  Padded rows get idx 0 and zero gradient; cham[b] is
    sum_x / max(lx, 1) + sum_y / max(ly, 1) for point_reduction="mean", sum_x + sum_y for "sum" (include/ptk.h)."""
    if point_reduction not in _REDUCTIONS:
        raise ValueError('point_reduction must be one of ["mean", "sum"]')
    return _Chamfer.apply(x, y, x_lengths, y_lengths, _REDUCTIONS[point_reduction])


def knn1(p1, p2, lengths1=None, lengths2=None):
    """dists (B,P1) f32, idx (B,P1) int32 -- forward only.  lengths1 / lengths2 as in chamfer(): padded queries and
    queries whose target cloud is empty get dist 0, idx 0."""
    _need_cuda(p1, p2)
    p1, p2 = _f32c(p1), _f32c(p2)
    if p1.dim() != 3 or p2.dim() != 3 or p1.shape[2] != 3 or p2.shape[2] != 3 or p1.shape[0] != p2.shape[0]:
        raise ValueError(f"Expected (B,P,3) point clouds, got {tuple(p1.shape)} and {tuple(p2.shape)}")
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    l1, l2 = _lengths(lengths1, B, p1.device, "lengths1"), _lengths(lengths2, B, p1.device, "lengths2")
    L = _lib.lib()
    dist = torch.empty(B, P1, dtype=torch.float32, device=p1.device)
    idx = torch.empty(B, P1, dtype=torch.int32, device=p1.device)
    ws = _ws(L.ptk_chamfer_workspace_bytes(B, P1, P2), p1.device)
    with torch.cuda.device(p1.device):
        _lib.check(L.ptk_knn1_fwd_lengths(_p(p1), _p(p2), _p(l1), _p(l2), B, P1, P2, _p(dist), _p(idx), _p(ws),
                                          ws.numel(), _stream()), "ptk_knn1_fwd_lengths")
    return dist, idx


# ------------------------------------------------------------------------------------- vertex max-pool
class _VertexMax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats):
        _need_cuda(feats)
        feats = _f32c(feats)
        if feats.dim() != 3:
            raise ValueError(f"Expected (B,N,C) vertex features, got {tuple(feats.shape)}")
        B, Nv, Cc = feats.shape
        out = torch.empty(B, Cc, dtype=torch.float32, device=feats.device)
        arg = torch.empty(B, Cc, dtype=torch.int32, device=feats.device)
        with torch.cuda.device(feats.device):
            _lib.check(_lib.lib().ptk_vertex_maxpool_fwd(_p(feats), B, Nv, Cc, _p(out), _p(arg), _stream()),
                       "ptk_vertex_maxpool_fwd")
        ctx.save_for_backward(arg)
        ctx.shape = (B, Nv, Cc)
        ctx.mark_non_differentiable(arg)
        return out, arg

    @staticmethod
    def backward(ctx, g, _ga):
        (arg,) = ctx.saved_tensors
        B, Nv, Cc = ctx.shape
        gin = torch.empty(B, Nv, Cc, dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            _lib.check(_lib.lib().ptk_vertex_maxpool_bwd(_p(_f32c(g)), _p(arg), B, Nv, Cc, _p(gin), _stream()),
                       "ptk_vertex_maxpool_bwd")
        return gin


def vertex_max(feats):
    """(B,N,C) -> (values (B,C), vertex index (B,C) int32): `features.max(dim=1)` of the autoencoder's GCN
    encoder (autoencoder/model.py:91) and the DDQN graph model (DDQN/model.py:128), differentiable."""
    return _VertexMax.apply(feats)


# ------------------------------------------------------------------------------------- positional embedding
class _NerfEmbed(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos):
        _need_cuda(pos)
        pos = _f32c(pos)
        M = pos.shape[0]
        out = torch.empty(M, 63, dtype=torch.float32, device=pos.device)
        with torch.cuda.device(pos.device):
            _lib.check(_lib.lib().ptk_nerf_embed_fwd(_p(pos), M, _p(out), _stream()), "ptk_nerf_embed_fwd")
        # The reference's Deformation.forward updates `vertices` IN PLACE right after encoding them
        # (vision/model.py:250,270,283), so the input must not be what the backward reads: the positions are the
        # last three columns of the output (model.py:396-397), which nobody writes to.
        ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        pos = out[:, 60:].contiguous()
        gpos = torch.empty_like(pos)
        with torch.cuda.device(pos.device):
            _lib.check(_lib.lib().ptk_nerf_embed_bwd(_p(pos), _p(_f32c(g)), pos.shape[0], _p(gpos), _stream()),
                       "ptk_nerf_embed_bwd")
        return gpos


def nerf_embed(points):
    """(..., 3) positions -> (..., 63): the 60-wide sin/cos NeRF embedding followed by the positions themselves
    (Positional_Encoder.nerf_embedding + cat, vision/model.py:381-397), one launch, differentiable."""
    if points.shape[-1] != 3:
        raise ValueError(f"positions must end in a dimension of 3, got {tuple(points.shape)}")
    return _NerfEmbed.apply(points.reshape(-1, 3)).reshape(*points.shape[:-1], 63)


# ------------------------------------------------------------------------------------- fused vertex-feature front
VERTEX_FRONT_MAX_H1, VERTEX_FRONT_MAX_H2 = 112, 224  # csrc/vertex_front.cu


class _VertexFront(torch.autograd.Function):
    """positions (M,3) [, mask (M,), emb (4,S), add (M,S)] -> (M,S): NeRF embedding, the three Linear layers of
    Positional_Encoder, the mask-token embedding row and the optional additive features in one launch
    (ptk_vertex_front_fwd).  Backward: column sums per mask token (ptk_vertex_front_colsum: embedding-table and last
    bias gradient), the library's own GEMM kernels for the weight / data gradients, ptk_nerf_embed_bwd."""

    @staticmethod
    def forward(ctx, pos, mask, w1, b1, w2, b2, w3, b3, emb, add):
        _need_cuda(pos, mask, w1, b1, w2, b2, w3, b3, emb, add)
        pos, w1, b1, w2, b2, w3, b3 = (_f32c(t) for t in (pos, w1, b1, w2, b2, w3, b3))
        mask = _f32c(mask) if mask is not None else None
        emb = _f32c(emb) if emb is not None else None
        add = _f32c(add) if add is not None else None
        M, h1, h2, S = pos.shape[0], w1.shape[0], w2.shape[0], w3.shape[0]
        if w1.shape[1] != 63 or w2.shape[1] != h1 or w3.shape[1] != h2:
            raise ValueError("vertex_front: weight shapes must be (h1,63), (h2,h1), (S,h2)")
        if emb is not None and (mask is None or tuple(emb.shape) != (4, S) or mask.numel() != M):
            raise ValueError("vertex_front: emb must be (4,S) and come with a mask of M tokens")
        if add is not None and tuple(add.shape) != (M, S):
            raise ValueError("vertex_front: add must be (M,S)")
        train = any(ctx.needs_input_grad)
        out = torch.empty(M, S, dtype=torch.float32, device=pos.device)
        h1s = torch.empty(M, h1, dtype=torch.float32, device=pos.device) if train else None
        h2s = torch.empty(M, h2, dtype=torch.float32, device=pos.device) if train else None
        with torch.cuda.device(pos.device):
            _lib.check(_lib.lib().ptk_vertex_front_fwd(_p(pos), _p(mask), _p(w1), _p(b1), _p(w2), _p(b2), _p(w3), _p(b3),
                                                       _p(emb), _p(add), M, h1, h2, S, _p(out), _p(h1s), _p(h2s),
                                                       _stream()), "ptk_vertex_front_fwd")
        if train:
            # the reference updates `vertices` in place right after encoding them (vision/model.py:250,270,283):
            # keep a private copy of the positions for the backward
            ctx.save_for_backward(pos.clone(), mask, w1, w2, w3, h1s, h2s)
            ctx.has_emb = emb is not None
        return out

    @staticmethod
    def backward(ctx, g):
        pos, mask, w1, w2, w3, h1s, h2s = ctx.saved_tensors
        need = ctx.needs_input_grad
        g = _f32c(g)
        M, S = g.shape
        L = _lib.lib()
        with torch.cuda.device(g.device):
            sums = torch.empty(4, S, dtype=torch.float32, device=g.device)
            ws = _ws(L.ptk_vertex_front_colsum_workspace_bytes(M, S), g.device)
            _lib.check(L.ptk_vertex_front_colsum(_p(g), _p(mask if ctx.has_emb else None), M, S, _p(sums), _p(ws),
                                                 ws.numel(), _stream()), "ptk_vertex_front_colsum")
            gb3 = sums.sum(0)
            gemb = sums if ctx.has_emb else None
            gw3 = _linear_wgrad(g, h2s)                                  # (S, h2): nn.Linear layout
            gh2 = _linear_dgrad(g, w3.t().contiguous(), h2s)            # (M, h2), ReLU mask of hidden 2 fused
            gb2 = _bias_grad(gh2, gh2.shape[1])
            gw2 = _linear_wgrad(gh2, h1s)
            gh1 = _linear_dgrad(gh2, w2.t().contiguous(), h1s)
            gb1 = _bias_grad(gh1, gh1.shape[1])
            x0 = torch.empty(M, 63, dtype=torch.float32, device=g.device)
            _lib.check(L.ptk_nerf_embed_fwd(_p(pos), M, _p(x0), _stream()), "ptk_nerf_embed_fwd")
            gw1 = _linear_wgrad(gh1, x0)
            gpos = None
            if need[0]:
                gx0 = _linear_fwd(gh1, w1, algo_id=GEMM_AUTO)           # (M,h1) . (h1,63)
                gpos = torch.empty_like(pos)
                _lib.check(L.ptk_nerf_embed_bwd(_p(pos), _p(gx0), M, _p(gpos), _stream()), "ptk_nerf_embed_bwd")
        return gpos, None, gw1, gb1, gw2, gb2, gw3, gb3, gemb, (g if need[9] else None)


def vertex_front(positions, mask, w1, b1, w2, b2, w3, b3, emb=None, add=None):
    """(B,N,3) positions [+ (B,N,1) mask tokens, (4,S) embedding table, (B,N,S) additive features] -> (B,N,S):
    Positional_Encoder(positions) + Mask_Encoder(mask) [+ img_features] of Deformation.forward
    (vision/model.py:229-236) in one launch."""
    if positions.shape[-1] != 3:
        raise ValueError(f"positions must end in a dimension of 3, got {tuple(positions.shape)}")
    lead = positions.shape[:-1]
    S = w3.shape[0]
    out = _VertexFront.apply(positions.reshape(-1, 3), mask.reshape(-1) if mask is not None else None, w1, b1, w2, b2,
                             w3, b3, emb, add.reshape(-1, S) if add is not None else None)
    return out.reshape(*lead, S)


def vertex_front_supported(input_size):
    return input_size // 4 >= 1 and input_size // 4 <= VERTEX_FRONT_MAX_H1 and input_size // 2 <= VERTEX_FRONT_MAX_H2


# ------------------------------------------------------------------------------------- surface sampling
class _Sample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, verts, faces_i32, u_face, uv, given_idx):
        _need_cuda(verts, faces_i32, u_face, uv, given_idx)
        verts, uv = _f32c(verts), _f32c(uv)
        if verts.dim() != 3 or verts.shape[2] != 3:
            raise ValueError(f"verts must be (B,V,3), got {tuple(verts.shape)}")
        if faces_i32.dtype != torch.int32 or faces_i32.dim() != 2 or faces_i32.shape[1] != 3:
            raise ValueError("faces must be an (F,3) int32 tensor")
        B, V, _ = verts.shape
        F = faces_i32.shape[0]
        S = uv.shape[2] if uv.dim() == 3 else -1
        if tuple(uv.shape) != (2, B, S):
            raise ValueError("uv must be (2,B,S)")
        faces_i32 = faces_i32.contiguous()
        L = _lib.lib()
        pts = torch.empty(B, S, 3, dtype=torch.float32, device=verts.device)
        if given_idx is None:
            u_face = _f32c(u_face)
            if tuple(u_face.shape) != (B, S):
                raise ValueError("u_face must be (B,S) and uv (2,B,S)")
            fidx = torch.empty(B, S, dtype=torch.int32, device=verts.device)
            ws = _ws(L.ptk_sample_workspace_bytes(B, F), verts.device)
        else:  # faces drawn by the caller: interpolation only
            if tuple(given_idx.shape) != (B, S):
                raise ValueError("face_idx must be (B,S)")
            fidx = given_idx.to(torch.int32).contiguous()
            u_face, ws = None, None
        with torch.cuda.device(verts.device):
            _lib.check(L.ptk_sample_fwd(_p(verts), B, V, _p(faces_i32), F, _p(u_face), _p(uv), S, _p(pts),
                                        _p(fidx), _p(ws), ws.numel() if ws is not None else 0, _stream()),
                       "ptk_sample_fwd")
        ctx.save_for_backward(fidx, uv, faces_i32)
        ctx.dims = (B, V, F, S)
        ctx.mark_non_differentiable(fidx)
        return pts, fidx

    @staticmethod
    def backward(ctx, gpts, _gf):
        fidx, uv, faces_i32 = ctx.saved_tensors
        B, V, F, S = ctx.dims
        gpts = _f32c(gpts)
        gv = torch.empty(B, V, 3, dtype=torch.float32, device=gpts.device)
        with torch.cuda.device(gpts.device):
            _lib.check(_lib.lib().ptk_sample_bwd(_p(gpts), _p(fidx), _p(uv), _p(faces_i32), B, V, F, S, _p(gv),
                                                 _stream()), "ptk_sample_bwd")
        return gv, None, None, None, None


def sample_points(verts, faces_i32, u_face, uv, face_idx=None):
    """pts (B,S,3), face_idx (B,S) for explicit uniforms; differentiable w.r.t. verts.  With `face_idx` given
    (u_face ignored) the faces are the caller's draw and only the barycentric interpolation runs."""
    return _Sample.apply(verts, faces_i32, u_face, uv, face_idx)


class _MeshChamfer(torch.autograd.Function):
    """utils.chamfer_distance as ONE autograd node (ptk_mesh_chamfer_fwd / bwd): `repeat` samplings of the mesh, the
    Chamfer distance of each against gt, the mean -- instead of 2 x repeat + 2 nodes with torch tensors in between."""

    @staticmethod
    def forward(ctx, verts, gt, faces_i32, u_face, uv, given_idx):
        _need_cuda(verts, gt, faces_i32, u_face, uv, given_idx)
        verts, gt, uv = _f32c(verts), _f32c(gt), _f32c(uv)
        if verts.dim() != 3 or verts.shape[2] != 3 or gt.dim() != 3 or gt.shape[2] != 3 or gt.shape[0] != verts.shape[0]:
            raise ValueError(f"Expected verts (B,V,3) and gt (B,P,3), got {tuple(verts.shape)} and {tuple(gt.shape)}")
        if faces_i32.dtype != torch.int32 or faces_i32.dim() != 2 or faces_i32.shape[1] != 3:
            raise ValueError("faces must be an (F,3) int32 tensor")
        B, V, _ = verts.shape
        P2, F = gt.shape[1], faces_i32.shape[0]
        if uv.dim() != 4 or uv.shape[1] != 2 or uv.shape[2] != B:
            raise ValueError("uv must be (repeat,2,B,S)")
        R, S = uv.shape[0], uv.shape[3]
        dev = verts.device
        if given_idx is None:
            u_face = _f32c(u_face)
            if tuple(u_face.shape) != (R, B, S):
                raise ValueError("u_face must be (repeat,B,S)")
            fidx = torch.empty(R, B, S, dtype=torch.int32, device=dev)
        else:
            if tuple(given_idx.shape) != (R, B, S):
                raise ValueError("face_idx must be (repeat,B,S)")
            fidx, u_face = given_idx.to(torch.int32).contiguous(), None
        faces_i32 = faces_i32.contiguous()
        L = _lib.lib()
        cd = torch.empty(B, dtype=torch.float32, device=dev)
        pts = torch.empty(R, B, S, 3, dtype=torch.float32, device=dev)
        idx_x = torch.empty(R, B, S, dtype=torch.int32, device=dev)
        idx_y = torch.empty(R, B, P2, dtype=torch.int32, device=dev)
        ws = _ws(L.ptk_mesh_chamfer_workspace_bytes(B, V, F, S, P2), dev)
        with torch.cuda.device(dev):
            _lib.check(L.ptk_mesh_chamfer_fwd(_p(verts), B, V, _p(faces_i32), F, _p(gt), P2, _p(u_face), _p(uv), S, R,
                                              _p(cd), _p(pts), _p(fidx), _p(idx_x), _p(idx_y), _p(ws), ws.numel(),
                                              _stream()), "ptk_mesh_chamfer_fwd")
        ctx.save_for_backward(gt, pts, fidx, idx_x, idx_y, uv, faces_i32)
        ctx.dims = (B, V, F, S, P2, R)
        return cd

    @staticmethod
    def backward(ctx, g):
        gt, pts, fidx, idx_x, idx_y, uv, faces_i32 = ctx.saved_tensors
        B, V, F, S, P2, R = ctx.dims
        g = _f32c(g)
        dev = g.device
        gv = torch.empty(B, V, 3, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        gg = torch.empty(B, P2, 3, dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        L = _lib.lib()
        ws = _ws(L.ptk_mesh_chamfer_workspace_bytes(B, V, F, S, P2), dev)
        with torch.cuda.device(dev):
            _lib.check(L.ptk_mesh_chamfer_bwd(_p(gt), _p(pts), _p(fidx), _p(idx_x), _p(idx_y), _p(uv), _p(faces_i32), _p(g),
                                              B, V, F, S, P2, R, _p(gv), _p(gg), _p(ws), ws.numel(), _stream()),
                       "ptk_mesh_chamfer_bwd")
        return gv, gg, None, None, None, None


def mesh_chamfer(verts, gt, faces_i32, u_face, uv, face_idx=None):
    """cd (B,): mean over the repeats of chamfer(sample(verts, faces), gt).  u_face (repeat,B,S), uv (repeat,2,B,S);
    with `face_idx` (repeat,B,S) given, u_face is ignored (the caller drew the faces).  Differentiable w.r.t. verts and gt."""
    return _MeshChamfer.apply(verts, gt, faces_i32, u_face, uv, face_idx)


def mesh_face_areas(verts, faces_i32):
    """(B,V,3), (F,3) int32 -> areas (B,F): utils.py:163-164 for a batch sharing one face list (no grad)."""
    _need_cuda(verts, faces_i32)
    verts = _f32c(verts.detach())
    B, V, _ = verts.shape
    F = faces_i32.shape[0]
    out = torch.empty(B, F, dtype=torch.float32, device=verts.device)
    with torch.cuda.device(verts.device):
        _lib.check(_lib.lib().ptk_mesh_face_areas(_p(verts), B, V, _p(faces_i32.contiguous()), F, _p(out), _stream()),
                   "ptk_mesh_face_areas")
    return out


def face_areas_normals(verts_packed, faces_i64):
    _need_cuda(verts_packed, faces_i64)
    v = _f32c(verts_packed)
    f = faces_i64.contiguous().long()
    F = f.shape[0]
    areas = torch.empty(F, dtype=torch.float32, device=v.device)
    normals = torch.empty(F, 3, dtype=torch.float32, device=v.device)
    with torch.cuda.device(v.device):
        _lib.check(_lib.lib().ptk_face_areas_normals(_p(v), v.shape[0], _p(f), F, _p(areas), _p(normals),
                                                     _stream()), "ptk_face_areas_normals")
    return areas, normals


# ------------------------------------------------------------------------------------- GCN primitives
# GEMM algorithm selection (include/ptk.h: PTK_GEMM_*).  The TRAINING forward uses the exact-FP32 FFMA
# kernel: its k-sequential FMA accumulation reproduces a scalar FP32 GEMM almost bit for bit, which keeps
# the ReLU masks of a deep GCN identical to the reference's (a 1e-6 perturbation flips individual ReLUs and
# moves 20-layer gradients by 1e-3 -- measured, see DESIGN.md).  Inference forwards and the backward GEMMs,
# whose errors enter the result smoothly, may use the 3xTF32 tensor-core kernel.
GEMM_AUTO, GEMM_FFMA, GEMM_TF32X3 = 0, 1, 2
algo = {"fwd_train": GEMM_FFMA, "fwd_infer": GEMM_AUTO, "dgrad": GEMM_AUTO, "wgrad": GEMM_AUTO}
batch_bias_grad = True  # one slab + two launches for the bias gradients of a GCN pass (tests flip this)
fuse_layers = True  # training forward of 'cut' layers: split-epilogue GEMM + strided aggregate (tests flip this)
# Form of the vertex aggregation (include/ptk.h: PTK_AGG_*): "auto" lets the library pick the form measured fastest for
# the shape (dense-tile product for wide layers and for the compact head at large batches / on dense graphs, the L2
# gather otherwise); "l2", "dense", "ring" force one.  All forms give identical results (tests flip this).
AGG_FORMS = {"auto": 0, "l2": 1, "dense": 2, "ring": 3}
aggregate_form = "auto"


def _linear_fwd(X2, W2, out=None, algo_id=GEMM_FFMA):
    M, K = X2.shape
    N = W2.shape[1]
    H = out if out is not None else torch.empty(M, N, dtype=torch.float32, device=X2.device)
    L = _lib.lib()
    ws = _ws(L.ptk_gcn_linear_workspace_bytes(M, K, N), X2.device)
    _lib.check(L.ptk_gcn_linear_fwd(_p(X2), _p(W2), M, K, N, _p(H), algo_id, _p(ws), ws.numel(), _stream()),
               "ptk_gcn_linear_fwd")
    return H


def _linear_dgrad(gH2, W2, act2, algo_id=None, act_bits=None, out=None):
    algo_id = algo["dgrad"] if algo_id is None else algo_id
    M, N = gH2.shape
    K = W2.shape[0]
    gX = out if out is not None else torch.empty(M, K, dtype=torch.float32, device=gH2.device)
    L = _lib.lib()
    ws = _ws(L.ptk_gcn_linear_workspace_bytes(M, K, N), gH2.device)
    _lib.check(L.ptk_gcn_linear_dgrad(_p(gH2), _p(W2), _p(act2), _p(act_bits), M, K, N, _p(gX), algo_id, _p(ws),
                                      ws.numel(), _stream()),
               "ptk_gcn_linear_dgrad")
    return gX


def _linear_wgrad(X2, gH2, algo_id=None):
    algo_id = algo["wgrad"] if algo_id is None else algo_id
    M, K = X2.shape
    N = gH2.shape[1]
    L = _lib.lib()
    gW = torch.empty(K, N, dtype=torch.float32, device=X2.device)
    ws = _ws(L.ptk_gcn_linear_wgrad_workspace_bytes(M, K, N), X2.device)
    _lib.check(L.ptk_gcn_linear_wgrad(_p(X2), _p(gH2), M, K, N, _p(gW), algo_id, _p(ws), ws.numel(), _stream()),
               "ptk_gcn_linear_wgrad")
    return gW


def _aggregate(g: Graph, H3, Lc, bias, relu, transpose=False, out=None):
    B, Nv, Cc = H3.shape
    if Nv != g.n:
        raise ValueError(f"features have {Nv} vertices but the adjacency has {g.n}")
    out = out if out is not None else torch.empty_like(H3)
    k = g.bwd_k if transpose else g.fwd_k
    vector_path = Cc % 4 == 0 and 1 <= Lc <= 384 and H3.data_ptr() % 16 == 0 and out.data_ptr() % 16 == 0 and \
        (bias is None or bias.data_ptr() % 16 == 0)
    if vector_path and (k.n_common > 0 or k.tile_uptr is not None):
        # kernel form (hub rows' common set split off when there is one) + the tiles' neighbour unions
        _lib.check(_lib.lib().ptk_gcn_aggregate_tiled(_p(k.rowptr), _p(k.col), _p(k.val), _p(k.hubs), k.n_hubs,
                                                      _p(k.common_col), _p(k.common_w), k.n_common, _p(k.alpha),
                                                      _p(k.row_skip), _p(k.tile_uptr), _p(k.tile_ucol), _p(k.tile_lidx),
                                                      k.max_union, AGG_FORMS[aggregate_form], Nv, _p(H3), B, Cc, Lc,
                                                      _p(bias), int(relu), _p(out), 0, 0, _stream()),
                   "ptk_gcn_aggregate_tiled")
        return out
    if transpose:
        rp, col, val, hubs, nh = g.rowptr_t, g.col_t, g.val_t, g.hubs_t, g.n_hubs_t
    else:
        rp, col, val, hubs, nh = g.rowptr, g.col, g.val, g.hubs, g.n_hubs
    _lib.check(_lib.lib().ptk_gcn_aggregate(_p(rp), _p(col), _p(val), _p(hubs), nh, Nv, _p(H3), B, Cc, Lc,
                                            _p(bias), int(relu), _p(out), _stream()), "ptk_gcn_aggregate")
    return out


def _fused_layer_ok(K, N, Lc, relu):
    """Shapes the fused forward (ptk_gcn_linear_fwd_split + strided aggregate) covers: a 'cut' layer whose
    propagated slice, rounded up to whole float4 groups, is a proper prefix of a >= 64-wide output."""
    Lp = (Lc + 3) // 4 * 4
    return relu and K % 4 == 0 and N % 4 == 0 and N >= 64 and 1 <= Lc and Lp < N and Lp <= 384


def _fused_layer_fwd(g: Graph, X2, W2, Lc, bias, B, Nv, head_buf, x_bits=None):
    """One GCN_layer.forward (vision/model.py:351-363) in two kernels: the exact FFMA2 GEMM writes the
    propagated slice H[:, :Lp] into the compact `head_buf` and relu(H[:, Lp:]) straight into the layer
    output; the aggregation gathers from the head and fills out[:, :, :Lp]."""
    M, K = X2.shape
    N = W2.shape[1]
    Lp = (Lc + 3) // 4 * 4
    out = torch.empty(B, Nv, N, dtype=torch.float32, device=X2.device)
    L = _lib.lib()
    _lib.check(L.ptk_gcn_linear_fwd_split(_p(X2), _p(W2), M, K, N, Lp, _p(head_buf), _p(out), 1, _p(x_bits),
                                          _stream()), "ptk_gcn_linear_fwd_split")
    k = g.fwd_k
    _lib.check(L.ptk_gcn_aggregate_tiled(_p(k.rowptr), _p(k.col), _p(k.val), _p(k.hubs), k.n_hubs, _p(k.common_col),
                                         _p(k.common_w), k.n_common, _p(k.alpha), _p(k.row_skip), _p(k.tile_uptr),
                                         _p(k.tile_ucol), _p(k.tile_lidx), k.max_union, AGG_FORMS[aggregate_form], Nv,
                                         _p(head_buf), B, Lp, Lc, _p(bias), 1, _p(out), Lp, N, _stream()),
               "ptk_gcn_aggregate_tiled")
    return out


def _bias_grad(g2, Lc):
    M, Cc = g2.shape
    L = _lib.lib()
    gb = torch.empty(Cc, dtype=torch.float32, device=g2.device)
    ws = _ws(L.ptk_gcn_bias_grad_workspace_bytes(M, Lc), g2.device)
    _lib.check(L.ptk_gcn_bias_grad(_p(g2), M, Cc, Lc, _p(gb), _p(ws), ws.numel(), _stream()), "ptk_gcn_bias_grad")
    return gb


def _bias_grad_batched(slab, Lc):
    """slab (n, M, C) -> (n, C): the bias gradients of n layers in two launches."""
    n, M, Cc = slab.shape
    L = _lib.lib()
    gb = torch.empty(n, Cc, dtype=torch.float32, device=slab.device)
    ws = _ws(L.ptk_gcn_bias_grad_batched_workspace_bytes(n, M, Lc), slab.device)
    _lib.check(L.ptk_gcn_bias_grad_batched(_p(slab), n, M, Cc, Lc, _p(gb), _p(ws), ws.numel(), _stream()),
               "ptk_gcn_bias_grad_batched")
    return gb


def _relu_mask(g, act):
    out = torch.empty_like(g)
    _lib.check(_lib.lib().ptk_relu_mask(_p(g), _p(act), g.numel(), _p(out), _stream()), "ptk_relu_mask")
    return out


class _GCNLayer(torch.autograd.Function):
    """One GCN_layer.forward (vision/model.py:351-363): linear + aggregate (+bias, +ReLU)."""

    @staticmethod
    def forward(ctx, X, W, bias, graph, Lc, relu, train):
        _need_cuda(X, W, bias)
        X, W, bias = _f32c(X), _f32c(W), _f32c(bias)
        B, Nv, K = X.shape
        W2 = W.reshape(K, -1)
        with torch.cuda.device(X.device):
            H = _linear_fwd(X.reshape(B * Nv, K), W2,
                            algo_id=algo["fwd_train"] if train else algo["fwd_infer"]).reshape(B, Nv, -1)
            out = _aggregate(graph, H, Lc, bias, relu)
        ctx.save_for_backward(X, W2, out if relu else None)
        ctx.graph, ctx.Lc, ctx.relu, ctx.wshape = graph, Lc, relu, W.shape
        return out

    @staticmethod
    def backward(ctx, gout):
        X, W2, out = ctx.saved_tensors
        B, Nv, K = X.shape
        N = W2.shape[1]
        gout = _f32c(gout)
        with torch.cuda.device(X.device):
            if ctx.relu:
                gout = _relu_mask(gout, out)
            gb = _bias_grad(gout.reshape(B * Nv, N), ctx.Lc) if ctx.needs_input_grad[2] else None
            gH = _aggregate(ctx.graph, gout, ctx.Lc, None, False, transpose=True).reshape(B * Nv, N)
            gW = _linear_wgrad(X.reshape(B * Nv, K), gH).reshape(ctx.wshape) if ctx.needs_input_grad[1] else None
            gX = _linear_dgrad(gH, W2, None).reshape(B, Nv, K) if ctx.needs_input_grad[0] else None
        return gX, gW, gb, None, None, None, None


def _will_backprop(*tensors):
    """True when autograd records this call: grad mode on and something requires grad.  (Inside
    autograd.Function.forward grad mode is always off and ctx.needs_input_grad ignores torch.no_grad(), so this is
    decided by the caller and passed in.)"""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def gcn_layer(X, W, bias, adj, Lc, relu):
    return _GCNLayer.apply(X, W, bias, graph_of(adj), int(Lc), bool(relu), _will_backprop(X, W, bias))


native_stack = True  # GCN stacks run through ptk_gcn_stack_fwd/bwd (one C-ABI call per pass); tests flip this


def _ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


class _GCNStackNative(torch.autograd.Function):
    """The whole GCN.forward (vision/model.py:316-331) and its backward, one ptk_gcn_stack_fwd / ptk_gcn_stack_bwd call
    each: the layer loop, buffer reuse, fused layer forward, packed ReLU masks and batched bias gradients of
    _GCNStack below, walked in native code (csrc/gcn_stack.cu) -- identical kernels and results, no Python frame
    between two launches."""

    @staticmethod
    def forward(ctx, X, graph, Ls, relus, train, *params):
        n = len(params) // 2
        _need_cuda(X, *params)
        X = _f32c(X)
        B, Nv, K0 = X.shape
        if Nv != graph.n:
            raise ValueError(f"features have {Nv} vertices but the adjacency has {graph.n}")
        Ws = [_f32c(w) for w in params[:n]]
        bs = [_f32c(b) for b in params[n:]]
        widths = [K0] + [w.shape[-1] for w in Ws]
        for l, w in enumerate(Ws):
            if w.numel() != widths[l] * widths[l + 1]:
                raise ValueError(f"layer {l}: weight {tuple(w.shape)} does not map {widths[l]} -> {widths[l + 1]} channels")
        M = B * Nv
        dev = X.device
        fwd_algo = algo["fwd_train"] if train else algo["fwd_infer"]
        c_widths = (C.c_int64 * (n + 1))(*widths)
        c_Ls = (C.c_int32 * n)(*Ls)
        c_relus = (C.c_uint8 * n)(*[1 if r else 0 for r in relus])
        L = _lib.lib()
        if train:
            acts = [torch.empty(B, Nv, widths[l + 1], dtype=torch.float32, device=dev) for l in range(n)]
            bits = [None] * n
            for l in range(1, n):  # the fused forward of layer l packs the ReLU mask of its input for its own dgrad
                if fuse_layers and fwd_algo == GEMM_FFMA and relus[l - 1] and widths[l] <= 512 and \
                        _fused_layer_ok(widths[l], widths[l + 1], Ls[l], relus[l]):
                    bits[l] = torch.empty(M, (widths[l] + 31) // 32, dtype=torch.int32, device=dev)
        else:  # inference: two alternating buffers, nothing kept
            wmax = max(widths[1:])
            pool = [torch.empty(M * wmax, dtype=torch.float32, device=dev) for _ in range(min(2, n - 1))]
            acts = [pool[l % 2][:M * widths[l + 1]].view(B, Nv, widths[l + 1]) for l in range(n - 1)]
            acts.append(torch.empty(B, Nv, widths[n], dtype=torch.float32, device=dev))  # the result owns its memory
            bits = [None] * n
        ws = _ws(L.ptk_gcn_stack_fwd_workspace_bytes(B, Nv, n, c_widths, c_Ls), dev)
        with torch.cuda.device(dev):
            _lib.check(L.ptk_gcn_stack_fwd(C.byref(graph.csr_struct(False)), B, Nv, n, c_widths, c_Ls, c_relus, _p(X),
                                           _ptr_array(Ws), _ptr_array(bs), _ptr_array(acts), _ptr_array(bits), fwd_algo,
                                           int(fuse_layers), _p(ws), ws.numel(), _stream()), "ptk_gcn_stack_fwd")
        out = acts[-1]
        if not train:
            return out
        ctx.save_for_backward(X, *acts, *Ws)
        ctx.bits = bits
        ctx.graph, ctx.Ls, ctx.relus, ctx.n, ctx.widths = graph, Ls, relus, n, widths
        ctx.wshapes = [w.shape for w in params[:n]]
        return out

    @staticmethod
    def backward(ctx, gout):
        n, widths = ctx.n, ctx.widths
        saved = ctx.saved_tensors
        X, acts, Ws = saved[0], saved[1:n + 1], saved[n + 1:]
        B, Nv, _ = X.shape
        dev = X.device
        gout = _f32c(gout)
        need_gX = ctx.needs_input_grad[0]
        need_gW = [ctx.needs_input_grad[5 + l] for l in range(n)]
        need_gb = [ctx.needs_input_grad[5 + n + l] for l in range(n)]
        gX = torch.empty_like(X) if need_gX else None
        gWs = [torch.empty(widths[l], widths[l + 1], dtype=torch.float32, device=dev) if need_gW[l] else None
               for l in range(n)]
        # bias gradients of the layers that share the hidden width: consecutive rows of one matrix (batched launch)
        gbs = [None] * n
        group = []
        if batch_bias_grad and n >= 3:
            ref = (widths[n - 1], ctx.Ls[n - 2])
            group = [l for l in range(n - 1) if need_gb[l] and (widths[l + 1], ctx.Ls[l]) == ref]
        if len(group) >= 2:
            gb_all = torch.empty(len(group), widths[n - 1], dtype=torch.float32, device=dev)
            for i, l in enumerate(group):
                gbs[l] = gb_all[i]
        for l in range(n):
            if need_gb[l] and gbs[l] is None:
                gbs[l] = torch.empty(widths[l + 1], dtype=torch.float32, device=dev)
        c_widths = (C.c_int64 * (n + 1))(*widths)
        c_Ls = (C.c_int32 * n)(*ctx.Ls)
        c_relus = (C.c_uint8 * n)(*[1 if r else 0 for r in ctx.relus])
        c_need = (C.c_uint8 * n)(*[1 if v else 0 for v in need_gb])
        L = _lib.lib()
        ws = _ws(L.ptk_gcn_stack_bwd_workspace_bytes(B, Nv, n, c_widths, c_Ls, c_need, int(batch_bias_grad)), dev)
        with torch.cuda.device(dev):
            _lib.check(L.ptk_gcn_stack_bwd(C.byref(ctx.graph.csr_struct(True)), B, Nv, n, c_widths, c_Ls, c_relus, _p(X),
                                           _ptr_array(Ws), _ptr_array(acts), _ptr_array(ctx.bits), _p(gout), _p(gX),
                                           _ptr_array(gWs), _ptr_array(gbs), c_need, int(batch_bias_grad), algo["dgrad"],
                                           algo["wgrad"], _p(ws), ws.numel(), _stream()), "ptk_gcn_stack_bwd")
        gWs = [g.reshape(ctx.wshapes[l]) if g is not None else None for l, g in enumerate(gWs)]
        return (gX, None, None, None, None, *gWs, *gbs)


class _GCNStack(torch.autograd.Function):
    """The whole GCN.forward (vision/model.py:316-331): n layers, ReLU on all but the last, the first
    n-1 layers 'cut' (only the first L channels are propagated).  One autograd node so that the ReLU
    backward of layer l is fused into the dgrad epilogue of layer l+1 and H buffers are reused."""

    @staticmethod
    def forward(ctx, X, graph, Ls, relus, train, *params):
        n = len(params) // 2
        Ws, bs = params[:n], params[n:]
        _need_cuda(X, *params)
        X = _f32c(X)
        B, Nv, _ = X.shape
        acts = [X]
        fwd_algo = algo["fwd_train"] if train else algo["fwd_infer"]
        bits = [None] * n
        with torch.cuda.device(X.device):
            Hbuf = {}
            for l in range(n):
                K = acts[-1].shape[2]
                W2 = _f32c(Ws[l]).reshape(K, -1)
                N = W2.shape[1]
                bias = _f32c(bs[l])
                if fuse_layers and fwd_algo == GEMM_FFMA and _fused_layer_ok(K, N, Ls[l], relus[l]) and \
                        bias.data_ptr() % 16 == 0:
                    Lp = (Ls[l] + 3) // 4 * 4
                    head = Hbuf.get(("head", Lp))
                    if head is None:
                        head = Hbuf[("head", Lp)] = torch.empty(B * Nv, Lp, dtype=torch.float32, device=X.device)
                    # the GEMM also packs the ReLU mask of its input (= what layer l's dgrad applies)
                    xb = None
                    if train and l > 0 and relus[l - 1] and K <= 512:
                        xb = torch.empty(B * Nv, (K + 31) // 32, dtype=torch.int32, device=X.device)
                    bits[l] = xb
                    acts.append(_fused_layer_fwd(graph, acts[-1].reshape(B * Nv, K), W2, Ls[l], bias, B, Nv, head, xb))
                    if not train:
                        acts = acts[-1:]
                    continue
                H = Hbuf.get(N)
                if H is None:
                    H = Hbuf[N] = torch.empty(B * Nv, N, dtype=torch.float32, device=X.device)
                _linear_fwd(acts[-1].reshape(B * Nv, K), W2, out=H, algo_id=fwd_algo)
                acts.append(_aggregate(graph, H.reshape(B, Nv, N), Ls[l], bias, relus[l]))
                if not train:
                    acts = acts[-1:]  # inference: nothing is kept for a backward, layer l-1's output is free again
        if not train:
            return acts[-1]
        ctx.save_for_backward(*acts, *[_f32c(w) for w in Ws])
        ctx.bits = bits  # plain int32 buffers, no autograd history
        ctx.graph, ctx.Ls, ctx.relus, ctx.n = graph, Ls, relus, n
        ctx.wshapes = [w.shape for w in Ws]
        return acts[-1]

    @staticmethod
    def backward(ctx, gout):
        n = ctx.n
        saved = ctx.saved_tensors
        acts, Ws = saved[:n + 1], saved[n + 1:]
        B, Nv, _ = acts[0].shape
        M = B * Nv
        gWs, gbs = [None] * n, [None] * n
        g = _f32c(gout)
        # Layers whose output gradient has the same shape and propagated width write it into one slab (the dgrad of
        # the layer above is pointed at its slice), so their bias gradients are two batched launches at the end
        # instead of two per layer.  Costs one (M x N) matrix per such layer until the pass is over.
        need_gb = [ctx.needs_input_grad[5 + n + l] for l in range(n)]
        widths = [Ws[l].reshape(acts[l].shape[2], -1).shape[1] for l in range(n)]
        group = []
        if batch_bias_grad and n >= 3:
            ref = (widths[n - 2], ctx.Ls[n - 2])
            group = [l for l in range(n - 1) if need_gb[l] and (widths[l], ctx.Ls[l]) == ref]
        slot = {l: i for i, l in enumerate(group)}
        slab = None
        if len(group) >= 2:
            slab = torch.empty(len(group), M, widths[group[0]], dtype=torch.float32, device=g.device)
        else:
            slot = {}
        with torch.cuda.device(g.device):
            if ctx.relus[n - 1]:
                g = _relu_mask(g, acts[n])
            for l in range(n - 1, -1, -1):
                K = acts[l].shape[2]
                W2 = Ws[l].reshape(K, -1)
                N = W2.shape[1]
                if need_gb[l] and l not in slot:
                    gbs[l] = _bias_grad(g.reshape(M, N), ctx.Ls[l])
                gH = _aggregate(ctx.graph, g.reshape(B, Nv, N), ctx.Ls[l], None, False, transpose=True).reshape(M, N)
                if ctx.needs_input_grad[5 + l]:
                    gWs[l] = _linear_wgrad(acts[l].reshape(M, K), gH).reshape(ctx.wshapes[l])
                if l > 0 or ctx.needs_input_grad[0]:
                    mask = acts[l].reshape(M, K) if (l > 0 and ctx.relus[l - 1]) else None
                    dst = slab[slot[l - 1]] if (l - 1) in slot else None
                    g = _linear_dgrad(gH, W2, mask, act_bits=ctx.bits[l] if mask is not None else None,
                                      out=dst).reshape(B, Nv, K)
                else:
                    g = None
            if slot:
                gb_all = _bias_grad_batched(slab, ctx.Ls[group[0]])
                for l, i in slot.items():
                    gbs[l] = gb_all[i]
        return (g, None, None, None, None, *gWs, *gbs)


def gcn_stack(X, adj, weights, biases, Ls, relus):
    fn = _GCNStackNative if native_stack else _GCNStack
    return fn.apply(X, graph_of(adj), tuple(int(v) for v in Ls), tuple(bool(r) for r in relus),
                    _will_backprop(X, *weights, *biases), *weights, *biases)
