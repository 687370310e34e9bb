"""Pose-accuracy metrics on the device: the metric methods of the reference's `Evaluator`
(lib/utils/evaluation_utils.py:64-226) for a batch of images, over the C ABI (`pvnet_pose_metrics`,
`pvnet_find_nearest_point_idx` in include/pvnet_b200.h).

    pose_metrics(pose_pred [b,3,4], pose_gt [b,3,4], model_points [pn,3], K, diameter, ...) -> dict of [b] tensors

    add_dist        add_metric (:91-117), or add_metric_sym (:119-130) with sym_add=True (ADD-S)
    proj_mean_diff  projection_2d (:75-81), or projection_2d_sym (:83-89) with sym_proj=True
    trans_cm, rot_deg                   cm_degree_5_metric (:132-141)
    add_ok, proj_ok, cm5_ok             the recorders' flags (strict `<`)

The clouds keep the reference's dtypes: a float32 pose (the data loader's ground truth) gives a float32 cloud,
a float64 pose (the PnP result) a float64 one; the rest is fp64 with fixed-order sums.  Nothing synchronises, so
a call can be captured into a CUDA graph.  The reference evaluates `evaluate` / `evaluate_uncertainty` with
ADD-S and the plain projection for its symmetric objects ('eggbox', 'glue') and `evaluate_uncertainty_v2` with
both symmetric forms.

`DeviceEvaluator` keeps per-image results on the device and reports the reference's
`average_precision()` triple after one device-to-host copy.  Reading `.ply` models is the caller's job.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native

SYM_ADD, SYM_PROJ, PRED_F32, GT_F32 = 1, 2, 4, 8      # PVNET_METRICS_* in include/pvnet_b200.h


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _poses(p, dev, name):
    t = torch.as_tensor(p, device=dev)
    if t.dim() == 2:
        t = t[None]
    if t.dim() != 3 or tuple(t.shape[1:]) != (3, 4):
        raise ValueError(f"{name} must be [b,3,4], got {tuple(t.shape)}")
    return t.to(torch.float64).contiguous(), t.dtype == torch.float32


def pose_metrics(pose_pred, pose_gt, model_points, camera_matrix, diameter, percentage=0.1, sym_add=False,
                 sym_proj=False, proj_threshold=5.0, cm_threshold=5.0, deg_threshold=5.0):
    """pose_pred, pose_gt [b,3,4] (CUDA tensors; float32 or float64, see the module note); model_points [pn,3]
    float32 CUDA tensor; camera_matrix one 3x3 K (host array or tensor; copied by value) or a [b,3,3] CUDA
    tensor (one K per image); diameter in the model's units.  -> dict of [b] CUDA tensors (float64 values,
    bool flags).  No host synchronisation."""
    if not (isinstance(pose_pred, torch.Tensor) and pose_pred.is_cuda):
        raise RuntimeError("pvnet_b200: pose_metrics needs CUDA tensors (there is no CPU path)")
    dev = pose_pred.device
    pp, pred_f32 = _poses(pose_pred, dev, "pose_pred")
    pg, gt_f32 = _poses(pose_gt, dev, "pose_gt")
    b = pp.shape[0]
    if pg.shape[0] != b:
        raise ValueError(f"pose_pred has {b} poses, pose_gt {pg.shape[0]}")
    X = torch.as_tensor(model_points, device=dev).float().contiguous()
    if X.dim() != 2 or X.shape[1] != 3:
        raise ValueError(f"model_points must be [pn,3], got {tuple(X.shape)}")
    pn = X.shape[0]
    K_host, K_dev = None, None
    if isinstance(camera_matrix, torch.Tensor) and camera_matrix.dim() == 3:
        K_dev = camera_matrix.to(dev, torch.float64).contiguous()
        if tuple(K_dev.shape) != (b, 3, 3):
            raise ValueError(f"per-image camera matrices must be [{b},3,3], got {tuple(K_dev.shape)}")
    else:
        k = camera_matrix.detach().cpu() if isinstance(camera_matrix, torch.Tensor) else camera_matrix
        K_host = (ctypes.c_double * 9)(*np.asarray(k, np.float64).reshape(9).tolist())
    flags = (SYM_ADD if sym_add else 0) | (SYM_PROJ if sym_proj else 0) | (PRED_F32 if pred_f32 else 0) | \
            (GT_F32 if gt_f32 else 0)
    L = _native.lib()
    n = ctypes.c_size_t()
    _native.check(L.pvnet_pose_metrics_workspace_bytes(b, pn, flags, ctypes.byref(n)),
                  "pvnet_pose_metrics_workspace_bytes")
    ws = torch.empty([max(n.value, 1)], dtype=torch.uint8, device=dev)
    values = torch.empty([b, 4], dtype=torch.float64, device=dev)
    ok = torch.empty([b, 3], dtype=torch.uint8, device=dev)
    add_threshold = float(diameter) * float(percentage)            # evaluation_utils.py:96
    with torch.cuda.device(dev):
        _native.check(L.pvnet_pose_metrics(pp.data_ptr(), pg.data_ptr(), X.data_ptr(), K_host,
                                           None if K_dev is None else K_dev.data_ptr(), b, pn, flags, add_threshold,
                                           float(proj_threshold), float(cm_threshold), float(deg_threshold),
                                           values.data_ptr(), ok.data_ptr(), ws.data_ptr(), n.value, _stream(dev)),
                      "pvnet_pose_metrics")
    okb = ok.bool()
    return {"add_dist": values[:, 0], "proj_mean_diff": values[:, 1], "trans_cm": values[:, 2],
            "rot_deg": values[:, 3], "add_ok": okb[:, 0], "proj_ok": okb[:, 1], "cm5_ok": okb[:, 2]}


class DeviceEvaluator:
    """The metric half of the reference's Evaluator for one object: `evaluate_batch` appends a batch's results on
    the device; `average_precision()` returns the reference's (2-D projection, ADD, 5 cm 5 degree) accuracies
    after one device-to-host copy.

    symmetric=True uses ADD-S, as the reference's `evaluate` / `evaluate_uncertainty` do for 'eggbox' and 'glue';
    sym_proj=True adds the symmetric projection metric (`evaluate_uncertainty_v2`)."""

    def __init__(self, model_points, diameter, camera_matrix, symmetric=False, sym_proj=False, percentage=0.1):
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.model_points = torch.as_tensor(np.asarray(model_points, np.float32), device=self.device)
        self.diameter = float(diameter)
        self.camera_matrix = camera_matrix
        self.sym_add = bool(symmetric)
        self.sym_proj = bool(sym_proj)
        self.percentage = percentage
        self._batches = []

    def evaluate_batch(self, pose_pred, pose_gt, K=None):
        """pose_pred, pose_gt [b,3,4] (or [3,4]); K: None for the evaluator's camera, a 3x3 K, or [b,3,3] per
        image.  Returns the pose_metrics dict of this batch; nothing leaves the device."""
        m = pose_metrics(torch.as_tensor(pose_pred, device=self.device), torch.as_tensor(pose_gt, device=self.device),
                         self.model_points, self.camera_matrix if K is None else K, self.diameter,
                         percentage=self.percentage, sym_add=self.sym_add, sym_proj=self.sym_proj)
        self._batches.append(m)
        return m

    def _cat(self, key):
        if not self._batches:
            return torch.empty([0], device=self.device)
        return torch.cat([m[key] for m in self._batches])

    def _host(self):
        keys = ("add_dist", "proj_mean_diff", "add_ok", "proj_ok", "cm5_ok")
        if not self._batches:
            return {k: np.zeros([0]) for k in keys}
        stacked = torch.stack([self._cat(k).double() for k in keys]).cpu().numpy()     # the one copy
        return {k: stacked[i].astype(bool) if k.endswith("_ok") else stacked[i] for i, k in enumerate(keys)}

    @property
    def add_dists(self):
        return list(self._host()["add_dist"])

    @property
    def proj_mean_diffs(self):
        return list(self._host()["proj_mean_diff"])

    def average_precision(self, verbose=True):
        """(mean 2-D projection flag, mean ADD flag, mean 5 cm 5 degree flag), as evaluation_utils.py:218-226
        returns them (without its `tmp.npy` side file)."""
        h = self._host()
        proj, add, cm = np.mean(h["proj_ok"]), np.mean(h["add_ok"]), np.mean(h["cm5_ok"])
        if verbose:
            print('2d projections metric: {}'.format(proj))
            print('ADD metric: {}'.format(add))
            print('5 cm 5 degree metric: {}'.format(cm))
        return proj, add, cm
