"""Device-side uncertainty-driven PnP: the reference's `uncertainty_pnp`
(zju3dv/pvnet lib/utils/extend_utils/extend_utils.py:63-114) and the covariance -> weight step of
`Evaluator.evaluate_uncertainty` (lib/utils/evaluation_utils.py:165-201), over the C ABI
(`pvnet_uncertainty_pnp`, `pvnet_covariance_to_weights` in include/pvnet_b200.h).

    uncertainty_pnp(points_2d [pn,2], weights_2d [pn,3], points_3d [pn,3], camera_matrix [3,3]) -> Rt [3,4]

keeps the reference's signature and return type (numpy float64) for numpy inputs -- the arrays are
moved to the current CUDA device; batched CUDA tensors ([b,pn,2], [b,pn,3]) return a float64 CUDA
tensor [b,3,4] with no host synchronisation, which is what `PoseKeypointPipeline(with_pose=True)` uses so
that poses, not keypoints, are what leaves the GPU.  No CPU path: without the library or a CUDA
device these functions raise.

    find_nearest_point_idx(ref_pts, que_pts)                                          (extend_utils.py:39-60)
    uncertainty_pnp_v2(points_2d, covars, points_3d, camera_matrix, type='single')    (extend_utils.py:116-177)

complete the names lib/utils/evaluation_utils.py:16 imports, with the same numpy-in / numpy-out contract and
batched CUDA forms (`pvnet_find_nearest_point_idx`, and the isotropic weights fed to `pvnet_uncertainty_pnp`).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _camera(camera_matrix):
    k = np.asarray(camera_matrix.detach().cpu() if isinstance(camera_matrix, torch.Tensor) else camera_matrix,
                   dtype=np.float64).reshape(3, 3)
    return (ctypes.c_double * 9)(*k.ravel().tolist())


def covariance_to_weights(cov: torch.Tensor) -> torch.Tensor:
    """cov [...,2,2] CUDA float32 -> weights [...,3] = (wxx, wxy, wyy) of inv(sqrtm(cov))
    (evaluation_utils.py:170-181; zeros where the reference skips the point)."""
    if not cov.is_cuda:
        raise RuntimeError("pvnet_b200: `cov` must be a CUDA tensor (there is no CPU path)")
    c = cov.contiguous().float()
    n = c.numel() // 4
    out = torch.empty(tuple(c.shape[:-2]) + (3,), dtype=torch.float32, device=c.device)
    with torch.cuda.device(c.device):
        _native.check(_native.lib().pvnet_covariance_to_weights(c.data_ptr(), n, out.data_ptr(), _stream(c.device)),
                      "pvnet_covariance_to_weights")
    return out


def uncertainty_pnp_batched(points_2d, points_3d, camera_matrix, weights_2d=None, cov=None, return_info=False):
    """points_2d [b,pn,2] CUDA; weights_2d [b,pn,3] or cov [b,pn,2,2] (exactly one); points_3d [pn,3];
    camera_matrix 3x3 (host).  -> poses float64 [b,3,4] on the device (and info int32 [b,2])."""
    if not points_2d.is_cuda:
        raise RuntimeError("pvnet_b200: `points_2d` must be a CUDA tensor (there is no CPU path)")
    if (weights_2d is None) == (cov is None):
        raise ValueError("pass exactly one of weights_2d / cov")
    dev = points_2d.device
    p2 = points_2d.contiguous().float()
    b, pn, _ = p2.shape
    p3 = torch.as_tensor(points_3d, dtype=torch.float32, device=dev).contiguous()
    if tuple(p3.shape) != (pn, 3):
        raise ValueError(f"points_3d must be [{pn},3], got {tuple(p3.shape)}")
    w = None if weights_2d is None else weights_2d.to(dev).contiguous().float()
    c = None if cov is None else cov.to(dev).contiguous().float()
    out = torch.empty([b, 3, 4], dtype=torch.float64, device=dev)
    info = torch.empty([b, 2], dtype=torch.int32, device=dev) if return_info else None
    with torch.cuda.device(dev):
        _native.check(_native.lib().pvnet_uncertainty_pnp(
            p2.data_ptr(), None if c is None else c.data_ptr(), None if w is None else w.data_ptr(), p3.data_ptr(),
            _camera(camera_matrix), b, pn, out.data_ptr(), None if info is None else info.data_ptr(), _stream(dev)),
            "pvnet_uncertainty_pnp")
    return (out, info) if return_info else out


def uncertainty_pnp(points_2d, weights_2d, points_3d, camera_matrix):
    """Reference signature (extend_utils.py:63): numpy [pn,2], [pn,3] (wxx,wxy,wyy), [pn,3], [3,3] ->
    Rt numpy float64 [3,4].  Batched CUDA tensors are accepted too (see uncertainty_pnp_batched)."""
    if isinstance(points_2d, torch.Tensor) and points_2d.dim() == 3:
        return uncertainty_pnp_batched(points_2d, points_3d, camera_matrix, weights_2d=weights_2d)
    if not torch.cuda.is_available():
        raise RuntimeError("pvnet_b200: uncertainty_pnp needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    p2 = torch.as_tensor(np.asarray(points_2d, np.float32), device=dev)[None]
    w = torch.as_tensor(np.asarray(weights_2d, np.float32), device=dev)[None]
    assert p2.shape[1] == np.asarray(points_3d).shape[0] and p2.shape[1] >= 4          # extend_utils.py:72
    return uncertainty_pnp_batched(p2, np.asarray(points_3d, np.float32), camera_matrix, weights_2d=w)[0].cpu().numpy()


def find_nearest_point_idx_batched(ref_pts: torch.Tensor, que_pts: torch.Tensor, exclude_self: bool = False):
    """ref_pts [b,pn1,d], que_pts [b,pn2,d] CUDA (d = 2 or 3) -> int32 CUDA [b,pn2]: for every query point the
    index of the nearest reference point, exactly the index the reference kernel returns
    (nearest_neighborhood.cu:48-117, see pvnet_find_nearest_point_idx).  No host synchronisation."""
    if not (isinstance(ref_pts, torch.Tensor) and ref_pts.is_cuda and isinstance(que_pts, torch.Tensor)
            and que_pts.is_cuda):
        raise RuntimeError("pvnet_b200: batched find_nearest_point_idx needs CUDA tensors (there is no CPU path)")
    if ref_pts.dim() != 3 or que_pts.dim() != 3 or ref_pts.shape[0] != que_pts.shape[0] \
            or ref_pts.shape[2] != que_pts.shape[2] or ref_pts.shape[2] not in (2, 3):
        raise ValueError(f"expected [b,pn1,d] and [b,pn2,d] with d in (2, 3), got {tuple(ref_pts.shape)}, "
                         f"{tuple(que_pts.shape)}")
    dev = ref_pts.device
    r = ref_pts.contiguous().float()
    q = que_pts.to(dev).contiguous().float()
    b, pn1, d = r.shape
    pn2 = q.shape[1]
    out = torch.empty([b, pn2], dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _native.check(_native.lib().pvnet_find_nearest_point_idx(r.data_ptr(), q.data_ptr(), out.data_ptr(), b, pn1,
                                                                 pn2, d, int(bool(exclude_self)), _stream(dev)),
                      "pvnet_find_nearest_point_idx")
    return out


def find_nearest_point_idx(ref_pts, que_pts):
    """Reference signature (extend_utils.py:39-60): for every point in que_pts [pn2,2|3] the index of the nearest
    point in ref_pts [pn1,2|3] -> numpy int32 [pn2].  Both are rounded to float32 first, as the reference casts
    them.  Batched CUDA tensors [b,pn,d] return an int32 CUDA tensor [b,pn2] (find_nearest_point_idx_batched)."""
    if isinstance(ref_pts, torch.Tensor) and ref_pts.dim() == 3:
        return find_nearest_point_idx_batched(ref_pts, que_pts)
    assert (ref_pts.shape[1] == que_pts.shape[1] and 1 < que_pts.shape[1] <= 3)      # extend_utils.py:46
    if not torch.cuda.is_available():
        raise RuntimeError("pvnet_b200: find_nearest_point_idx needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    r = torch.as_tensor(np.ascontiguousarray(ref_pts, np.float32), device=dev)[None]
    q = torch.as_tensor(np.ascontiguousarray(que_pts, np.float32), device=dev)[None]
    return find_nearest_point_idx_batched(r, q)[0].cpu().numpy()


def covariance_to_isotropic_weights(cov: torch.Tensor) -> torch.Tensor:
    """cov [...,2,2] -> float32 weights [...,3] = (w, 0, w) with w = 1 / lambda_max(cov), or 0 where
    cov[0,0] < 1e-5: the weights of the reference's uncertainty_pnp_v2 (extend_utils.py:130-139, :153-154).
    lambda_max = (a+d)/2 + sqrt(((a-d)/2)^2 + b*c), in float64 on the covariance's device.
    A covariance with a NaN entry gets weight 0 (the point is left out of the fit); the reference's
    np.linalg.eigvals raises LinAlgError on it instead."""
    c = cov.double()
    a, b, cc, d = c[..., 0, 0], c[..., 0, 1], c[..., 1, 0], c[..., 1, 1]
    h = (a - d) / 2
    lam = (a + d) / 2 + torch.sqrt(h * h + b * cc)
    w = torch.where((a < 1e-5) | torch.isnan(c).flatten(-2).any(-1), torch.zeros_like(lam), 1.0 / lam)
    return torch.stack([w, torch.zeros_like(w), w], -1).float()


def uncertainty_pnp_v2(points_2d, covars, points_3d, camera_matrix, type='single'):
    """Reference signature (extend_utils.py:116-177): points_2d [pn,2], covars [pn,2,2], points_3d [pn,3],
    camera_matrix [3,3] -> Rt numpy float64 [3,4].  The isotropic weights (w, 0, w) of
    covariance_to_isotropic_weights feed the device solver of uncertainty_pnp; its P3P start takes the four
    points with the largest wxx + wxy = w, the points `argsort(weights)[-4:]` picks.  `type` is unused, as in
    the reference.  Batched CUDA tensors ([b,pn,2], [b,pn,2,2]) return a float64 CUDA tensor [b,3,4]."""
    if isinstance(points_2d, torch.Tensor) and points_2d.dim() == 3:
        w = covariance_to_isotropic_weights(covars.to(points_2d.device))
        return uncertainty_pnp_batched(points_2d, points_3d, camera_matrix, weights_2d=w)
    pn = points_2d.shape[0]
    assert (points_3d.shape[0] == pn and pn >= 4 and covars.shape[0] == pn)              # extend_utils.py:125
    if not torch.cuda.is_available():
        raise RuntimeError("pvnet_b200: uncertainty_pnp_v2 needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    p2 = torch.as_tensor(np.asarray(points_2d, np.float32), device=dev)[None]
    w = covariance_to_isotropic_weights(torch.as_tensor(np.asarray(covars, np.float64), device=dev))[None]
    return uncertainty_pnp_batched(p2, np.asarray(points_3d, np.float32), camera_matrix, weights_2d=w)[0].cpu().numpy()
