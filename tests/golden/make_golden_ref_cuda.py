"""Regenerates tests/golden/ref_cuda_kernels.npz and tests/golden/ref_cuda_layer.npz: what the
REFERENCE'S OWN CUDA voting kernels compute on the inputs of tests/test_gpu_reference_layer.py and of
the vanishing-point test in tests/test_gpu_variants.py.

Needs a CUDA device, oracle/_ref/libpvnet_refcuda.so (oracle/Makefile, target `ref`: the reference's
ransac_voting_kernel.cu compiled verbatim) and the built product library (the covariance cases start
from the product's v3 keypoints, stored with them):

    python tests/golden/make_golden_ref_cuda.py [OUT_DIR]        (default: tests/golden)

ref_cuda_kernels.npz   per kernel case: the hypotheses and counts the reference kernels returned, and the
                       digest (tests.helpers.digest) of their inlier flags.
ref_cuda_layer.npz     per REF_LAYER_CASES entry: the reference layer's keypoints with its stock fp32 refit
                       (`_kp`) and with the same refit ops in fp64 (`_kp64`), and for every image the digests
                       of the first round's samples, counts and hypotheses (`_tn` = -1 and empty digests where
                       the image has too few pixels); for the covariance cases the mean they start from, the
                       covariances, and the digests of every image's samples and counts.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import pvnet_oracle as po  # noqa: E402
from oracle import ref_cuda  # noqa: E402
from pvnet_b200 import ransac_voting_gpu as rv  # noqa: E402
from pvnet_b200 import synthetic as syn  # noqa: E402
from tests.helpers import (EDGE_THRESHOLDS, REF_LAYER_CASES, cfg1_inputs, digest,  # noqa: E402
                           edge_kernel_inputs, ref_layer_inputs, vp_inputs)

DEV = "cuda:0"


def _digests(rec, key):
    """Digest of one recorded array per image; "" for images the layer skipped (record None)."""
    return np.array(["" if r is None else digest(r[key].cpu().numpy()) for r in rec])


def _dev(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for a in arrays]


def _vote(d, c, hyp, thresh, vp=False):
    inl = torch.zeros([hyp.shape[0], d.shape[1], d.shape[0]], dtype=torch.uint8, device=DEV)
    (ref_cuda.voting_for_hypothesis_vanishing_point if vp else ref_cuda.voting_for_hypothesis)(d, c, hyp, inl, thresh)
    return inl.cpu().numpy()


def kernel_cases():
    out = {}
    for kind in ("random", "planted"):
        mask, field, idxs = cfg1_inputs(kind)
        coords, direct = po.compact(mask.astype(np.uint8), syn.as_reference_view(field[None])[0])
        d, c, i = _dev(direct, coords, idxs)
        hyp = ref_cuda.generate_hypothesis(d, c, i)
        inl = _vote(d, c, hyp, 0.99)
        out[f"cfg1_{kind}_hyp"] = hyp.cpu().numpy()
        out[f"cfg1_{kind}_counts"] = inl.sum(2).astype(np.int32)
        out[f"cfg1_{kind}_inliers8"] = np.array(digest(inl[:8]))
    direct, coords, idxs, extra = edge_kernel_inputs()
    d, c, i = _dev(direct, coords, idxs)
    hyp = ref_cuda.generate_hypothesis(d, c, i)
    out["edge_hyp"] = hyp.cpu().numpy()
    for t, thresh in enumerate(EDGE_THRESHOLDS):
        for j, hp in enumerate((hyp, _dev(extra)[0])):
            out[f"edge_inliers_{t}_{j}"] = np.array(digest(_vote(d, c, hp, thresh)))
    d, c, i = _dev(*vp_inputs(21))
    hyp = ref_cuda.generate_hypothesis_vanishing_point(d, c, i)
    out["vp_hyp"] = hyp.cpu().numpy()
    out["vp_inliers"] = np.array(digest(_vote(d, c, hyp, 0.99, vp=True)))
    return out


def layer_cases():
    out = {}
    for name, case in REF_LAYER_CASES.items():
        masks, fields = ref_layer_inputs(name)
        mask = torch.from_numpy(masks).to(DEV)
        ver = torch.from_numpy(fields).to(DEV)
        b, c2, h, w = ver.shape
        vertex = ver.permute(0, 2, 3, 1).view(b, h, w, c2 // 2, 2)
        if "hn" in case:
            rec = []
            torch.manual_seed(0)
            kp = ref_cuda.layer_v3(mask, vertex, case["hn"], inlier_thresh=0.99, record=rec)
            torch.manual_seed(0)
            kp64 = ref_cuda.layer_v3(mask, vertex, case["hn"], inlier_thresh=0.99, refit_dtype=torch.float64)
            out[f"{name}_kp"] = kp.cpu().numpy()
            out[f"{name}_kp64"] = kp64.cpu().numpy()
            out[f"{name}_tn"] = np.array([-1 if r is None else r["tn"] for r in rec], np.int32)
            for key in ("idxs", "counts", "hyp"):
                out[f"{name}_{key}"] = _digests(rec, key)
        if "cov" in case:
            seed, hn = case["mean"]
            torch.manual_seed(seed)
            mean = rv.ransac_voting_layer_v3(mask, vertex, hn, inlier_thresh=0.99)
            rec = []
            seed, hn, min_hyp = case["cov"]
            torch.manual_seed(seed)
            _, cov = ref_cuda.layer_cov_with_mean(mask, vertex, mean, round_hyp_num=hn, min_hyp_num=min_hyp,
                                                  inlier_thresh=0.99, record=rec)
            assert all(r is not None for r in rec)
            out[f"{name}_mean"] = mean.cpu().numpy()
            out[f"{name}_cov"] = cov.cpu().numpy()
            out[f"{name}_cov_idxs"] = _digests(rec, "idxs")
            out[f"{name}_cov_counts"] = _digests(rec, "counts")
        print(name, {k: v.shape for k, v in out.items() if k.startswith(name + "_")})
    return out


def main():
    if not ref_cuda.available():
        raise SystemExit(f"{ref_cuda.LIB_PATH} and a CUDA device are needed")
    dst = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(dst, exist_ok=True)
    for fname, make in (("ref_cuda_kernels.npz", kernel_cases), ("ref_cuda_layer.npz", layer_cases)):
        path = os.path.join(dst, fname)
        np.savez_compressed(path, **make())
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
