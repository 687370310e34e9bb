"""ctypes binding of libpvnet_b200.so (the C ABI declared in include/pvnet_b200.h).

There is no fallback: if the library is missing or a call fails, a RuntimeError is
raised.  Nothing here imports oracle/.
"""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libpvnet_b200.so")

_lock = threading.Lock()
_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_float = ctypes.c_float
c_size_t = ctypes.c_size_t
c_int64_p = ctypes.POINTER(ctypes.c_int64)

# name -> (restype, argtypes); must list every symbol include/pvnet_b200.h declares
SIGNATURES = {
    "pvnet_last_error": (ctypes.c_char_p, []),
    "pvnet_version": (c_int, []),
    "pvnet_launch_count": (ctypes.c_longlong, []),
    "pvnet_launch_count_reset": (None, []),
    "pvnet_vote_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_size_t)]),
    "pvnet_mask_foreground_count": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                            c_size_t, c_void_p]),
    "pvnet_ransac_voting_v3": (c_int, [c_void_p, c_int, c_void_p, c_int64_p, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_refit_at_points": (c_int, [c_void_p, c_int, c_void_p, c_int64_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                      c_float, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_ransac_voting_v5": (c_int, [c_void_p, c_int, c_void_p, c_int64_p, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_ransac_voting_v4": (c_int, [c_void_p, c_int, c_void_p, c_int64_p, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_ransac_motion_voting": (c_int, [c_void_p, c_int, c_void_p, c_int64_p, c_int, c_int, c_int, c_int,
                                           c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_vote_cov_with_mean": (c_int, [c_void_p, c_int, c_void_p, c_int64_p, c_void_p, c_void_p, c_void_p,
                                         c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_ransac_voting_pipeline": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int64_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_int,
                                             c_float, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_covariance_to_weights": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "pvnet_uncertainty_pnp": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.POINTER(ctypes.c_double), c_int, c_int,
                                      c_void_p, c_void_p, c_void_p]),
    "pvnet_find_nearest_point_idx": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "pvnet_pose_metrics_workspace_bytes": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_size_t)]),
    "pvnet_pose_metrics": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.POINTER(ctypes.c_double), c_void_p, c_int, c_int,
                                   c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, c_void_p,
                                   c_void_p, c_void_p, c_size_t, c_void_p]),
    "pvnet_generate_hypothesis": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pvnet_voting_for_hypothesis": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                                            c_void_p]),
    "pvnet_generate_hypothesis_vanishing_point": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                                          c_void_p]),
    "pvnet_voting_for_hypothesis_vanishing_point": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                                            c_int, c_float, c_void_p]),
    "pvnet_vote_counts": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p]),
    "pvnet_conv2d_nhwc": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                  c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_int, c_int, c_void_p]),
    "pvnet_conv_set_mode": (c_int, [c_int]),
    "pvnet_conv_set_multicast": (c_int, [c_int]),
    "pvnet_conv_set_persistent": (c_int, [c_int]),
    "pvnet_conv_set_head_epilogue_sets": (c_int, [c_int]),
    "pvnet_backbone_create": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
    "pvnet_backbone_destroy": (None, [c_void_p]),
    "pvnet_backbone_num_convs": (c_int, []),
    "pvnet_backbone_set_conv": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "pvnet_backbone_set_output_layout": (c_int, [c_void_p, c_int]),
    "pvnet_backbone_set_fused_upsample": (c_int, [c_void_p, c_int]),
    "pvnet_backbone_workspace_bytes": (c_int, [c_void_p, c_int, c_int, c_int, ctypes.POINTER(c_size_t)]),
    "pvnet_backbone_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                       c_void_p, c_size_t, c_void_p]),
    "pvnet_backbone_forward_u8": (c_int, [c_void_p, c_void_p, ctypes.POINTER(c_float), ctypes.POINTER(c_float), c_int, c_int,
                                          c_int, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "pvnet_jpeg_available": (c_int, []),
    "pvnet_jpeg_decoder_create": (c_int, [ctypes.POINTER(c_void_p)]),
    "pvnet_jpeg_decoder_destroy": (None, [c_void_p]),
    "pvnet_jpeg_decode_batch": (c_int, [c_void_p, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(c_size_t), c_int, c_int,
                                        c_int, c_void_p, c_void_p]),
    "pvnet_backbone_num_stages": (c_int, []),
    "pvnet_backbone_stage_name": (ctypes.c_char_p, [c_int]),
    "pvnet_backbone_run_stage": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                         c_void_p, c_size_t, c_void_p]),
}


def lib():
    """The loaded library.  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -m pvnet_b200._build` "
                        "(or __graft_entry__.build()).  pvnet_b200 has no CPU or PyTorch fallback.")
                L = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(L, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = L
    return _lib


def check(status: int, what: str):
    if status != 0:
        msg = lib().pvnet_last_error()
        raise RuntimeError(f"{what} failed (status {status}): {msg.decode() if msg else '?'}")


def launch_count() -> int:
    return int(lib().pvnet_launch_count())


def launch_count_reset():
    lib().pvnet_launch_count_reset()
