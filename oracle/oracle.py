"""ctypes wrapper over oracle/libptk_oracle.so -- the CPU ORACLE (test infrastructure).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module.  The product package never does.

All functions take / return numpy arrays (C-contiguous).  See ptk_oracle.c for the
reference file:line each one restates.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libptk_oracle.so")


def build(force=False):
    src = os.path.join(_HERE, "ptk_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_num_threads.restype = C.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def num_threads():
    return int(lib().orc_num_threads())


def set_num_threads(n):
    lib().orc_set_num_threads(C.c_int(int(n)))


def knn1(p1, p2, use_fma=True):
    p1, p2 = _f32(p1), _f32(p2)
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    dist = np.empty((B, P1), np.float32)
    idx = np.empty((B, P1), np.int32)
    lib().orc_knn1(_p(p1), _p(p2), C.c_int64(B), C.c_int64(P1), C.c_int64(P2), _p(dist), _p(idx),
                   C.c_int(int(use_fma)))
    return dist, idx


def chamfer_fwd(x, y, use_fma=True):
    x, y = _f32(x), _f32(y)
    B, P1, _ = x.shape
    P2 = y.shape[1]
    dx = np.empty((B, P1), np.float32)
    ix = np.empty((B, P1), np.int32)
    dy = np.empty((B, P2), np.float32)
    iy = np.empty((B, P2), np.int32)
    cham = np.empty((B,), np.float32)
    lib().orc_chamfer_fwd(_p(x), _p(y), C.c_int64(B), C.c_int64(P1), C.c_int64(P2), _p(dx), _p(ix),
                          _p(dy), _p(iy), _p(cham), C.c_int(int(use_fma)))
    return cham, dx, ix, dy, iy


def chamfer_bwd(x, y, idx_x, idx_y, grad_cham, want_x=True, want_y=True):
    x, y = _f32(x), _f32(y)
    B, P1, _ = x.shape
    P2 = y.shape[1]
    ix = np.ascontiguousarray(idx_x, np.int32)
    iy = np.ascontiguousarray(idx_y, np.int32)
    g = _f32(grad_cham)
    gx = np.empty_like(x) if want_x else None
    gy = np.empty_like(y) if want_y else None
    lib().orc_chamfer_bwd(_p(x), _p(y), _p(ix), _p(iy), _p(g), C.c_int64(B), C.c_int64(P1),
                          C.c_int64(P2), _p(gx), _p(gy))
    return gx, gy


def face_areas(verts, faces):
    verts = _f32(verts)
    faces = np.ascontiguousarray(faces, np.int64)
    B, V, _ = verts.shape
    F = faces.shape[0]
    out = np.empty((B, F), np.float32)
    lib().orc_face_areas(_p(verts), C.c_int64(B), C.c_int64(V), _p(faces), C.c_int64(F), _p(out))
    return out


def face_cumweights(areas):
    areas = _f32(areas)
    B, F = areas.shape
    cum = np.empty((B, F), np.uint64)
    lib().orc_face_cumweights(_p(areas), C.c_int64(B), C.c_int64(F), _p(cum))
    return cum


def sample_fwd(verts, faces, u_face, uv):
    verts = _f32(verts)
    faces = np.ascontiguousarray(faces, np.int64)
    u_face, uv = _f32(u_face), _f32(uv)
    B, V, _ = verts.shape
    F = faces.shape[0]
    S = u_face.shape[1]
    assert uv.shape == (2, B, S)
    pts = np.empty((B, S, 3), np.float32)
    fidx = np.empty((B, S), np.int32)
    lib().orc_sample_fwd(_p(verts), C.c_int64(B), C.c_int64(V), _p(faces), C.c_int64(F), _p(u_face),
                         _p(uv), C.c_int64(S), _p(pts), _p(fidx))
    return pts, fidx


def sample_bwd(grad_pts, face_idx, uv, faces, V):
    g = _f32(grad_pts)
    fi = np.ascontiguousarray(face_idx, np.int32)
    uv = _f32(uv)
    faces = np.ascontiguousarray(faces, np.int64)
    B, S, _ = g.shape
    gv = np.empty((B, V, 3), np.float32)
    lib().orc_sample_bwd(_p(g), _p(fi), _p(uv), _p(faces), C.c_int64(B), C.c_int64(V), C.c_int64(S),
                         _p(gv))
    return gv


def gcn_linear(X, W):
    X, W = _f32(X), _f32(W)
    M, K = X.shape
    N = W.shape[1]
    H = np.empty((M, N), np.float32)
    lib().orc_gcn_linear(_p(X), _p(W), C.c_int64(M), C.c_int64(K), C.c_int64(N), _p(H))
    return H


def gemm_fma_seq(A, B, rows=None, b_transposed=False):
    """C = A[rows] . B as a scalar FP32 loop: per output acc = fmaf(A[i,k], B[k,j], acc) for k = 0..K-1 from 0.0f.
    B is (K, N), or (N, K) read as its transpose without a copy when b_transposed (the dgrad's W)."""
    A, B = _f32(A), _f32(B)
    M, K = A.shape
    N = B.shape[0] if b_transposed else B.shape[1]
    assert B.shape == ((N, K) if b_transposed else (K, N))
    idx = None if rows is None else np.ascontiguousarray(rows, np.int64)
    if idx is not None:
        assert idx.ndim == 1 and (idx.size == 0 or (idx.min() >= 0 and idx.max() < M))
    n_rows = M if idx is None else idx.size
    C_ = np.empty((n_rows, N), np.float32)
    lib().orc_gemm_fma_seq(_p(A), C.c_int64(K), _p(B), C.c_int64(K if b_transposed else N), C.c_int(int(b_transposed)),
                           _p(idx), C.c_int64(n_rows), C.c_int64(K), C.c_int64(N), _p(C_))
    return C_


def gcn_aggregate_fwd(rowptr, col, H, L, bias, relu):
    H = _f32(H)
    B, Nv, Cc = H.shape
    rowptr = np.ascontiguousarray(rowptr, np.int32)
    col = np.ascontiguousarray(col, np.int32)
    bias = _f32(bias)
    out = np.empty_like(H)
    lib().orc_gcn_aggregate_fwd(_p(rowptr), _p(col), C.c_int64(Nv), _p(H), C.c_int64(B),
                                C.c_int64(Cc), C.c_int64(L), _p(bias), C.c_int(int(relu)), _p(out))
    return out


def gcn_aggregate_bwd(rowptr, col, gout, L):
    gout = _f32(gout)
    B, Nv, Cc = gout.shape
    rowptr = np.ascontiguousarray(rowptr, np.int32)
    col = np.ascontiguousarray(col, np.int32)
    gH = np.empty_like(gout)
    gb = np.empty((Cc,), np.float32)
    lib().orc_gcn_aggregate_bwd(_p(rowptr), _p(col), C.c_int64(Nv), _p(gout), C.c_int64(B),
                                C.c_int64(Cc), C.c_int64(L), _p(gH), _p(gb))
    return gH, gb


def gcn_layer_fwd(X, W, bias, rowptr, col, cut, do_cut, relu):
    """GCN_layer.forward (vision/model.py:351-363) on a CSR adjacency."""
    B, Nv, Kin = X.shape
    W2 = np.asarray(W, np.float32).reshape(Kin, -1)
    H = gcn_linear(_f32(X).reshape(B * Nv, Kin), W2).reshape(B, Nv, -1)
    Cc = H.shape[2]
    L = int(round(Cc * cut)) if do_cut else Cc
    return gcn_aggregate_fwd(rowptr, col, H, L, bias, relu)
