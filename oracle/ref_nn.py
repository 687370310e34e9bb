"""The reference's own nearest-neighbour launcher, run on the GPU box -- TEST AND BENCHMARK INFRASTRUCTURE ONLY.

`oracle/_ref/libpvnet_refnn.so` is lib/utils/extend_utils/src/nearest_neighborhood.cu compiled verbatim
(oracle/metrics.mk, target `refnn`).  `findNearestPointIdxLauncher` takes host pointers and does, on every call,
three cudaMalloc, the copies in, one launch, a blocking copy out and three cudaFree (:123-163).
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libpvnet_refnn.so")
_lib = None


def available() -> bool:
    if not os.path.exists(LIB_PATH):
        return False
    import torch
    return torch.cuda.is_available()


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(LIB_PATH)
        L.findNearestPointIdxLauncher.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 5
        L.findNearestPointIdxLauncher.restype = None
        _lib = L
    return _lib


def find_nearest_point_idx_batched(ref, que, exclude_self=False):
    """ref [b,pn1,d], que [b,pn2,d] host arrays -> int32 [b,pn2] from the reference kernel."""
    r = np.ascontiguousarray(ref, np.float32)
    q = np.ascontiguousarray(que, np.float32)
    b, pn1, d = r.shape
    pn2 = q.shape[1]
    out = np.zeros([b, pn2], np.int32)
    lib().findNearestPointIdxLauncher(r.ctypes.data, q.ctypes.data, out.ctypes.data, b, pn1, pn2, d,
                                      int(bool(exclude_self)))
    return out


def find_nearest_point_idx(ref_pts, que_pts):
    """extend_utils.py:39-60 on the reference kernel: [pn1,d], [pn2,d] -> int32 [pn2]."""
    return find_nearest_point_idx_batched(ref_pts[None], que_pts[None])[0]
