"""CPU oracle for the reference's pose-accuracy metrics -- TEST INFRASTRUCTURE ONLY.

Restates in numpy, with the reference's dtypes and operation order, the five metric methods of
`Evaluator` (lib/utils/evaluation_utils.py:75-141) and `find_nearest_point_distance` (:54-62), with
`Projector.project_K` (lib/utils/base_utils.py:290-294).  The nearest-neighbour index is
`pvo_find_nearest_point_idx` of nn_oracle.c, the reference kernel's sequence (pinned against the
kernel itself by tests/golden/ref_nn.npz).  Dtypes: a float32 ground-truth pose gives a float32 target
cloud, a float64 predicted pose a float64 one, exactly as numpy promotes them in the reference.

Each metric returns (value, flag) instead of appending to a recorder.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpvnet_nn_oracle.so")
_F32P = ctypes.POINTER(ctypes.c_float)
_I32P = ctypes.POINTER(ctypes.c_int32)
_lib_handle = None


def build(force: bool = False) -> str:
    """Compile nn_oracle.c (oracle/metrics.mk) if the .so is missing or stale."""
    src = os.path.join(_HERE, "nn_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-f", "metrics.mk", "nn_oracle"])
    return _LIB_PATH


def _lib():
    global _lib_handle
    if _lib_handle is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        L.pvo_find_nearest_point_idx.argtypes = [_F32P, _F32P, _I32P] + [ctypes.c_int] * 5
        L.pvo_find_nearest_point_idx.restype = None
        _lib_handle = L
    return _lib_handle


def find_nearest_point_idx_batched(ref, que, exclude_self=False):
    """ref [b,pn1,d], que [b,pn2,d] (cast to float32) -> int32 [b,pn2] (nearest_neighborhood.cu:48-117)."""
    r = np.ascontiguousarray(ref, np.float32)
    q = np.ascontiguousarray(que, np.float32)
    b, pn1, d = r.shape
    pn2 = q.shape[1]
    assert q.shape[0] == b and q.shape[2] == d and d in (2, 3)
    out = np.zeros([b, pn2], np.int32)
    _lib().pvo_find_nearest_point_idx(r.ctypes.data_as(_F32P), q.ctypes.data_as(_F32P), out.ctypes.data_as(_I32P),
                                      b, pn1, pn2, d, int(bool(exclude_self)))
    return out


def find_nearest_point_idx(ref_pts, que_pts):
    """extend_utils.py:39-60: [pn1,d], [pn2,d] -> int32 [pn2]."""
    assert (ref_pts.shape[1] == que_pts.shape[1] and 1 < que_pts.shape[1] <= 3)
    return find_nearest_point_idx_batched(ref_pts[None], que_pts[None])[0]


def find_nearest_point_distance(pts1, pts2):
    """evaluation_utils.py:54-62."""
    idxs = find_nearest_point_idx(pts1, pts2)
    return np.linalg.norm(pts1[idxs] - pts2, 2, 1)


def project_K(pts_3d, RT, K):
    """base_utils.py:290-294."""
    pts_2d = np.matmul(pts_3d, RT[:, :3].T) + RT[:, 3:].T
    pts_2d = np.matmul(pts_2d, K.T)
    return pts_2d[:, :2] / pts_2d[:, 2:]


def projection_2d(pose_pred, pose_targets, model, K, threshold=5):
    """evaluation_utils.py:75-81."""
    d = np.mean(np.linalg.norm(project_K(model, pose_pred, K) - project_K(model, pose_targets, K), axis=-1))
    return d, d < threshold


def projection_2d_sym(pose_pred, pose_targets, model, K, threshold=5):
    """evaluation_utils.py:83-89."""
    d = np.mean(find_nearest_point_distance(project_K(model, pose_pred, K), project_K(model, pose_targets, K)))
    return d, d < threshold


def add_metric(pose_pred, pose_targets, model, diameter, percentage=0.1):
    """evaluation_utils.py:91-117."""
    diameter = diameter * percentage
    model_pred = np.dot(model, pose_pred[:, :3].T) + pose_pred[:, 3]
    model_targets = np.dot(model, pose_targets[:, :3].T) + pose_targets[:, 3]
    d = np.mean(np.linalg.norm(model_pred - model_targets, axis=-1))
    return d, d < diameter


def add_metric_sym(pose_pred, pose_targets, model, diameter, percentage=0.1):
    """evaluation_utils.py:119-130."""
    diameter = diameter * percentage
    model_pred = np.dot(model, pose_pred[:, :3].T) + pose_pred[:, 3]
    model_targets = np.dot(model, pose_targets[:, :3].T) + pose_targets[:, 3]
    d = np.mean(find_nearest_point_distance(model_pred, model_targets))
    return d, d < diameter


def cm_degree_5_metric(pose_pred, pose_targets):
    """evaluation_utils.py:132-141 -> (translation_cm, angle_deg, flag)."""
    translation_distance = np.linalg.norm(pose_pred[:, 3] - pose_targets[:, 3]) * 100
    rotation_diff = np.dot(pose_pred[:, :3], pose_targets[:, :3].T)
    trace = np.trace(rotation_diff)
    trace = trace if trace <= 3 else 3
    angular_distance = np.rad2deg(np.arccos((trace - 1.) / 2.))
    return translation_distance, angular_distance, translation_distance < 5 and angular_distance < 5


def pose_metrics(pose_pred, pose_gt, model, K, diameter, percentage=0.1, sym_add=False, sym_proj=False):
    """One image, the dict pvnet_b200.evaluation.pose_metrics returns per image (numpy scalars)."""
    add, add_ok = (add_metric_sym if sym_add else add_metric)(pose_pred, pose_gt, model, diameter, percentage)
    proj, proj_ok = (projection_2d_sym if sym_proj else projection_2d)(pose_pred, pose_gt, model, K)
    t, r, cm_ok = cm_degree_5_metric(pose_pred, pose_gt)
    return {"add_dist": add, "proj_mean_diff": proj, "trans_cm": t, "rot_deg": r, "add_ok": bool(add_ok),
            "proj_ok": bool(proj_ok), "cm5_ok": bool(cm_ok)}
