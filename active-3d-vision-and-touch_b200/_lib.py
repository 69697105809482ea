"""ctypes binding of libptk_b200.so (include/ptk.h).  No CPU fallback: if the CUDA extension is
missing or a call fails, this raises -- loudly."""
import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libptk_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "ptk.h")

CHAMFER_FILTER, CHAMFER_EXACT, CHAMFER_PRUNED, CHAMFER_AUTO = 0, 1, 2, 3
REDUCE_MEAN, REDUCE_SUM = 0, 1
KNN_MAX_K = 64
PTK_OK, PTK_ERR_SHAPE, PTK_ERR_ALIGN, PTK_ERR_ARCH, PTK_ERR_CUDA, PTK_ERR_WORKSPACE = 0, -1, -2, -3, -4, -5

_vp, _i64, _i32, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_size_t


class GcnCsr(C.Structure):
    """ptk_gcn_csr of include/ptk.h: one direction of the adjacency, plain CSR + kernel form."""
    _fields_ = [("rowptr", _vp), ("col", _vp), ("val", _vp), ("hubs", _vp), ("n_hubs", _i32),
                ("k_rowptr", _vp), ("k_col", _vp), ("k_val", _vp), ("k_hubs", _vp), ("k_n_hubs", _i32),
                ("common_col", _vp), ("common_w", _vp), ("n_common", _i32), ("alpha", _vp), ("row_skip", _vp),
                ("tile_uptr", _vp), ("tile_ucol", _vp), ("tile_lidx", _vp), ("max_union", _i32)]


# name -> (restype, argtypes); mirrors include/ptk.h one to one (tests check the two stay in sync)
SIGNATURES = {
    "ptk_version": (C.c_int, []),
    "ptk_last_error": (C.c_char_p, []),
    "ptk_device_info": (C.c_int, [C.c_int] + [C.POINTER(C.c_int)] * 6),
    "ptk_launch_count": (C.c_uint64, []),
    "ptk_chamfer_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_chamfer_set_algo": (C.c_int, [C.c_int]),
    "ptk_chamfer_get_algo": (C.c_int, []),
    "ptk_chamfer_rescued": (C.c_int, [_vp, _i64, _i64, _i64, C.POINTER(_i64), _vp]),
    "ptk_knn1_fwd": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ptk_chamfer_fwd": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ptk_chamfer_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ptk_chamfer_fwd_lengths": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                          _vp]),
    "ptk_chamfer_bwd_lengths": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp]),
    "ptk_knn1_fwd_lengths": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ptk_chamfer_bwd_det_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_chamfer_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _sz, _vp]),
    "ptk_chamfer_normals_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_chamfer_normals_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _sz,
                                          _vp]),
    "ptk_chamfer_normals_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp]),
    "ptk_chamfer_normals_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp,
                                              _sz, _vp]),
    "ptk_knn1_bwd_lengths":(C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ptk_knn1_bwd_det_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_knn1_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ptk_knn_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64]),
    "ptk_knn_fwd_lengths": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ptk_knn_bwd_lengths": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ptk_knn_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ptk_point_frames_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp]),
    "ptk_point_frames_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "ptk_point_frames_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp, _sz,
                                           _vp]),
    "ptk_sample_workspace_bytes": (_sz, [_i64, _i64]),
    "ptk_sample_fwd": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ptk_sample_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "ptk_sample_bwd_det_workspace_bytes": (_sz, [_i64, _i64]),
    "ptk_sample_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _sz, _vp]),
    "ptk_sample_normals_fwd": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _vp]),
    "ptk_sample_normals_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "ptk_sample_normals_bwd_det_workspace_bytes": (_sz, [_i64, _i64]),
    "ptk_sample_normals_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _sz, _vp]),
    "ptk_face_areas_normals": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "ptk_mesh_face_areas": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp]),
    "ptk_gcn_aggregate": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _vp, _i64, _i64, _i64, _vp, C.c_int, _vp, _vp]),
    "ptk_gcn_aggregate_ex": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _i64, _i64, _i64, _vp,
                                       C.c_int, _vp, _i64, _i64, _vp]),
    "ptk_gcn_aggregate_tiled": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64,
                                          _vp, _i64, _i64, _i64, _vp, C.c_int, _vp, _i64, _i64, _vp]),
    "ptk_gcn_linear_fwd_split": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, C.c_int, _vp, _vp]),
    "ptk_gcn_bias_grad_workspace_bytes": (_sz, [_i64, _i64]),
    "ptk_gcn_bias_grad": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _sz, _vp]),
    "ptk_gcn_bias_grad_batched_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_gcn_bias_grad_batched": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp, _sz, _vp]),
    "ptk_relu_mask": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "ptk_gcn_linear_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_gcn_linear_fwd": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, C.c_int, _vp, _sz, _vp]),
    "ptk_gcn_linear_dgrad": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, C.c_int, _vp, _sz, _vp]),
    "ptk_gcn_linear_wgrad_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ptk_gcn_linear_wgrad": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, C.c_int, _vp, _sz, _vp]),
    "ptk_gcn_stack_fwd_workspace_bytes": (_sz, [_i64, _i64, _i32, _vp, _vp]),
    "ptk_gcn_stack_fwd": (C.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int,
                                    _vp, _sz, _vp]),
    "ptk_gcn_stack_bwd_workspace_bytes": (_sz, [_i64, _i64, _i32, _vp, _vp, _vp, C.c_int]),
    "ptk_gcn_stack_bwd": (C.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                    C.c_int, C.c_int, C.c_int, _vp, _sz, _vp]),
    "ptk_vertex_maxpool_fwd": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ptk_vertex_maxpool_bwd": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "ptk_adj_workspace_bytes": (_sz, [_i64]),
    "ptk_adj_count": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _sz, _vp]),
    "ptk_adj_emit": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ptk_nerf_embed_fwd": (C.c_int, [_vp, _i64, _vp, _vp]),
    "ptk_nerf_embed_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "ptk_vertex_front_fwd": (C.c_int, [_vp] * 10 + [_i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "ptk_vertex_front_colsum_workspace_bytes": (_sz, [_i64, _i32]),
    "ptk_vertex_front_colsum": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "ptk_mesh_chamfer_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64, _i64]),
    "ptk_mesh_chamfer_fwd": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _sz, _vp]),
    "ptk_mesh_chamfer_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp,
                                       _vp, _sz, _vp]),
    "ptk_mesh_chamfer_bwd_det_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64, _i64]),
    "ptk_mesh_chamfer_bwd_det": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp,
                                           _vp, _vp, _sz, _vp]),
    "ptk_host_ctx_create": (_vp, [C.c_int]),
    "ptk_host_ctx_destroy": (None, [_vp]),
    "ptk_host_chamfer": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ptk_host_mesh_chamfer": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64,
                                        _vp, _vp, _vp]),
}


def header_symbols():
    """Every function name include/ptk.h declares."""
    with open(HEADER_PATH) as fh:
        src = fh.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ptk_[a-z0-9_]+)\s*\(", src)))


_lib = None


def lib():
    """The loaded library.  Raises ImportError (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
                "`python active-3d-vision-and-touch_b200/build.py` (nvcc, sm_100a). There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        if handle.ptk_version() != 1:
            raise ImportError("libptk_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def last_error():
    msg = lib().ptk_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what=""):
    """Map a PTK_ERR_* code to the exception the reference's stack would raise."""
    if rc == PTK_OK:
        return
    msg = f"{what}: {last_error()}" if what else last_error()
    if rc == PTK_ERR_SHAPE:
        raise ValueError(msg)  # PyTorch3D raises ValueError on shape errors
    raise RuntimeError(f"libptk_b200 error {rc}: {msg}")


def launch_count():
    """Kernels launched by libptk_b200.so in this process so far."""
    return int(lib().ptk_launch_count())


def device_info(device=0):
    vals = [C.c_int(0) for _ in range(6)]
    check(lib().ptk_device_info(int(device), *[C.byref(v) for v in vals]), "ptk_device_info")
    keys = ["sm_count", "clock_khz", "l2_bytes", "smem_optin", "cc_major", "cc_minor"]
    return {k: v.value for k, v in zip(keys, vals)}
