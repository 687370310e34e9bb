"""The reference's OWN CUDA kernels against the oracle and against the product.  What those kernels
(oracle/_ref: the reference's ransac_voting_kernel.cu compiled verbatim by oracle/Makefile, driven by
oracle/ref_cuda.py with the reference's torch ops) computed on the inputs below is stored in
tests/golden/ref_cuda_kernels.npz and ref_cuda_layer.npz by tests/golden/make_golden_ref_cuda.py
(large exact-match arrays as digests: tests.helpers.digest).
This is what pins the oracle (SURVEY.md §8c, CPU) and what measures "within 1e-4 of the reference
CUDA layer" (GPU)."""
import os

import numpy as np
import pytest
import torch

from oracle import pvnet_oracle as po
from pvnet_b200 import ransac_voting_gpu as rv
from pvnet_b200 import synthetic as syn
from tests.helpers import EDGE_THRESHOLDS, REF_LAYER_CASES, cfg1_inputs, digest, edge_kernel_inputs, ref_layer_inputs

DEV = "cuda:0"


@pytest.fixture(scope="module")
def kernels(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_cuda_kernels.npz"))


@pytest.fixture(scope="module")
def layer(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_cuda_layer.npz"))


def _dev_inputs(mask_np, field_np):
    mask = torch.from_numpy(np.ascontiguousarray(mask_np)).to(DEV)
    ver = torch.from_numpy(np.ascontiguousarray(field_np)).to(DEV)
    b, c2, h, w = ver.shape
    return mask, ver.permute(0, 2, 3, 1).view(b, h, w, c2 // 2, 2)


@pytest.mark.parametrize("kind", ["random", "planted"])
def test_reference_kernels_pin_the_oracle(kernels, kind):
    mask, field, idxs = cfg1_inputs(kind)
    coords, direct = po.compact(mask.astype(np.uint8), syn.as_reference_view(field[None])[0])
    hyp = kernels[f"cfg1_{kind}_hyp"]
    ohyp = po.generate_hypothesis_kernel(direct, coords, idxs)
    assert np.array_equal(hyp.view(np.uint32), ohyp.view(np.uint32))
    assert np.array_equal(kernels[f"cfg1_{kind}_counts"], po.vote_counts(direct, coords, ohyp, 0.99))
    assert kernels[f"cfg1_{kind}_inliers8"] == digest(po.voting_for_hypothesis_kernel(direct, coords, ohyp[:8], 0.99))


def test_reference_kernels_pin_the_oracle_on_edge_values(kernels):
    direct, coords, idxs, extra = edge_kernel_inputs()
    ohyp = po.generate_hypothesis_kernel(direct, coords, idxs)
    assert np.array_equal(kernels["edge_hyp"].view(np.uint32), ohyp.view(np.uint32))
    # also hypotheses ON pixels (norm2 == 0) and far away
    for t, thresh in enumerate(EDGE_THRESHOLDS):
        for j, hp in enumerate((ohyp, extra)):
            assert kernels[f"edge_inliers_{t}_{j}"] == digest(po.voting_for_hypothesis_kernel(direct, coords, hp, thresh))


def _product_vs_reference_layer(layer, name, label=""):
    """Runs the product from torch.manual_seed(0) and compares it with the reference layer (its own
    kernels + its torch ops) run from the same seed, with its stock fp32 refit and with the refit ops
    in fp64.  Asserts fixed-seed parity of samples / hypotheses / counts, and that the product is
    within 1e-4 of the reference layer once the reference's fp32 refit rounding is taken out (fp64
    run).  Returns the gaps."""
    mask, vertex = _dev_inputs(*ref_layer_inputs(name))
    torch.manual_seed(0)
    kp, dbg = rv.ransac_voting_layer_v3(mask, vertex, REF_LAYER_CASES[name]["hn"], inlier_thresh=0.99,
                                        max_num=30000, return_debug=True)
    for bi, tn in enumerate(layer[f"{name}_tn"]):
        if tn < 0:
            continue
        # fixed-seed parity: same samples drawn, same counts, same winner
        assert digest(dbg["idxs"][bi].cpu().numpy()) == layer[f"{name}_idxs"][bi], "RNG stream differs from the reference's"
        assert int(dbg["tn"][bi]) == tn
        assert digest(dbg["counts"][bi].cpu().numpy()) == layer[f"{name}_counts"][bi], \
            "inlier counts differ from the reference layer"
        assert digest(dbg["hyp"][bi].cpu().numpy()) == layer[f"{name}_hyp"][bi]
    kp, ref_kp, ref_kp64 = kp.cpu().numpy(), layer[f"{name}_kp"], layer[f"{name}_kp64"]
    gap32 = np.abs(kp - ref_kp).max()
    gap64 = np.abs(kp - ref_kp64).max()
    noise = np.abs(ref_kp - ref_kp64).max()
    print(f"\n[reference-layer gap] {label}: |ours - ref(fp32 refit)| = {gap32:.3e}; "
          f"|ours - ref(fp64 refit)| = {gap64:.3e}; reference's own fp32 noise |ref32 - ref64| = {noise:.3e}")
    assert gap64 <= 1e-4, "product differs from the reference layer beyond its fp32 refit rounding"
    # and the distance to the STOCK fp32 reference is explained by that rounding noise, not hidden behind it
    assert gap32 <= 1.5 * noise + 1e-5, (gap32, noise)
    return gap32, gap64, noise


def _cov_vs_reference_layer(layer, name):
    """The product's estimate_voting_distribution_with_mean against the reference's, from the same torch
    seed and the same mean: samples, counts, covariances.  Returns (ours, the reference's)."""
    mask, vertex = _dev_inputs(*ref_layer_inputs(name))
    seed, hn, min_hyp = REF_LAYER_CASES[name]["cov"]
    mean = torch.from_numpy(layer[f"{name}_mean"]).to(DEV)
    torch.manual_seed(seed)
    _, cov, dbg = rv.estimate_voting_distribution_with_mean(mask, vertex, mean, round_hyp_num=hn, min_hyp_num=min_hyp,
                                                            inlier_thresh=0.99, max_num=30000, return_debug=True)
    for bi in range(mask.shape[0]):
        assert digest(dbg["idxs"][bi].cpu().numpy()) == layer[f"{name}_cov_idxs"][bi], \
            "RNG stream differs from the reference's"
        assert digest(dbg["counts"][bi].cpu().numpy()) == layer[f"{name}_cov_counts"][bi], \
            "inlier counts differ from the reference layer"
    ref_cov = torch.from_numpy(layer[f"{name}_cov"]).to(DEV)
    assert torch.allclose(cov, ref_cov, atol=1e-4, rtol=1e-4), (cov - ref_cov).abs().max().item()
    return cov, ref_cov


@pytest.mark.gpu
def test_fixed_seed_parity_with_reference_layer_config1(layer):
    _product_vs_reference_layer(layer, "config1",
                                label="config1 planted, tn=10000, K=9 (odd keypoints 260 px outside the mask)")


@pytest.mark.gpu
def test_fixed_seed_parity_with_reference_layer_demo(layer):
    """The reference's own demo fixture (well conditioned: keypoints inside the object)."""
    gap32, _, _ = _product_vs_reference_layer(layer, "demo", label="demo fixture, tn=2289")
    assert gap32 <= 1e-3


@pytest.mark.gpu
def test_fixed_seed_parity_near_keypoints(layer):
    """Keypoints inside the mask (R=20 px): the best-conditioned case."""
    gap32, _, _ = _product_vs_reference_layer(layer, "near", label="near keypoints, tn=3000")
    assert gap32 <= 1e-3


@pytest.mark.gpu
def test_fixed_seed_parity_with_subsampling(layer):
    _product_vs_reference_layer(layer, "subsampled", label="subsampled 40000->~30000")


@pytest.mark.gpu
def test_covariance_fixed_seed_parity(layer):
    cov, ref_cov = _cov_vs_reference_layer(layer, "covariance")
    gap = (cov - ref_cov).abs()
    print(f"\n[reference-layer gap] covariance: max abs {gap.max().item():.3e}, "
          f"max rel {(gap / ref_cov.abs().clamp_min(1e-6)).max().item():.3e}, |cov| max {ref_cov.abs().max().item():.3e}")


@pytest.mark.gpu
def test_config4_shape_fixed_seed_vs_reference_layer(layer):
    """BASELINE config 4 per image (K=9, 20000 px, v3(256) + with_mean(256, 4096), thresh 0.99) against the reference's
    own kernels + torch ops under the same torch seed: samples, counts, keypoints, covariances."""
    _product_vs_reference_layer(layer, "config4", label="config 4 shape, tn=20000, K=9, 256 hyp")
    _cov_vs_reference_layer(layer, "config4")


@pytest.mark.gpu
def test_config5_shape_fixed_seed_vs_reference_layer(layer):
    """BASELINE config 5 per image (K=17, 92160 px subsampled to ~30000 by the reference's own uniform_ draw,
    v3(1024) + with_mean(1024, 1024))."""
    _product_vs_reference_layer(layer, "config5", label="config 5 shape, 92160 px -> ~30000, K=17, 1024 hyp")
    _cov_vs_reference_layer(layer, "config5")
