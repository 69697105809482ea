"""ctypes wrapper over knn_oracle.c, the CPU oracle of the K-NN scan (test infrastructure).

The library is compiled on first use into the system temporary directory, with the flags of oracle/Makefile
(-ffp-contract=off: no multiply-add is fused unless written as fmaf())."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "knn_oracle.c")
_FLAGS = ["-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-std=gnu11", "-shared"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as fh:
            tag = hashlib.sha1(fh.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"ptk_knn_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            try:
                subprocess.check_call(["/usr/bin/gcc"] + _FLAGS + ["-fopenmp", "-o", tmp, _SRC, "-lm"])
            except subprocess.CalledProcessError:  # no OpenMP: single-threaded
                subprocess.check_call(["/usr/bin/gcc"] + _FLAGS + ["-Wno-unknown-pragmas", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def knn(p1, p2, K, use_fma=True):
    """orc_knn: the K nearest p2 points of every p1 point, (B,P1,K) f32 / int32 (include/ptk.h ptk_knn_fwd_lengths)."""
    p1 = np.ascontiguousarray(p1, dtype=np.float32)
    p2 = np.ascontiguousarray(p2, dtype=np.float32)
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    dist = np.empty((B, P1, K), np.float32)
    idx = np.empty((B, P1, K), np.int32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    lib().orc_knn(ptr(p1), ptr(p2), C.c_int64(B), C.c_int64(P1), C.c_int64(P2), C.c_int64(K), ptr(dist), ptr(idx),
                  C.c_int(int(use_fma)))
    return dist, idx
