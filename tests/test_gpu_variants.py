"""GPU: the module's other voting variants (SURVEY.md §8 f-3) through the reference's import path,
against (a) tests/golden/ref_variants.npz, outputs of the reference's own Python functions with
the same samples, and (b) the oracle.  Hypotheses and counts: bit-exact.  Means / covariances /
variances: 1e-4-class tolerances (the reference sums in fp32, see DESIGN.md)."""
import os

import numpy as np
import pytest
import torch

from lib.ransac_voting_gpu_layer.ransac_voting_gpu import (estimate_voting_distribution, ransac_motion_voting,
                                                           ransac_voting_hypothesis, ransac_voting_layer,
                                                           ransac_voting_layer_v4)
from oracle import pvnet_oracle as po
from pvnet_b200 import synthetic as syn
from tests.helpers import digest, variant_inputs, vp_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_variants.npz"))


def _dev(mask, vertex):
    # the callers' layout: vertex is the permuted view of an NCHW tensor (tools/demo.py:48-50)
    b, h, w, k, _ = vertex.shape
    nchw = torch.from_numpy(vertex).to(DEV).permute(0, 3, 4, 1, 2).reshape(b, 2 * k, h, w).contiguous()
    return torch.from_numpy(mask).to(DEV), nchw.permute(0, 2, 3, 1).view(b, h, w, k, 2)


def test_v1_against_reference_fixture(gold):
    seed, n, classes = (int(v) for v in gold["v1_seed"])
    mask, vertex, _ = variant_inputs(seed, n, classes)
    m, v = _dev(mask, vertex)
    idxs = torch.from_numpy(gold["v1_idxs"])[:, None].to(DEV)           # [class, b=1, hn, K, 2]
    out = ransac_voting_layer(m, v, classes + 1, 32, inlier_thresh=0.99, idxs=idxs)
    assert out.shape == (1, classes, 5, 2)
    assert np.array_equal(out.cpu().numpy(), gold["v1_out"])


def test_hypothesis_against_reference_fixture(gold):
    seed, n, _ = (int(v) for v in gold["hyp_seed"])
    mask, vertex, _ = variant_inputs(seed, n)
    m, v = _dev(mask, vertex)
    hyp, cnt = ransac_voting_hypothesis(m, v, 48, inlier_thresh=0.99, idxs=torch.from_numpy(gold["hyp_idxs"])[None].to(DEV))
    assert cnt.dtype == torch.int64
    assert np.array_equal(hyp.cpu().numpy(), gold["hyp_out"])
    assert np.array_equal(cnt.cpu().numpy(), gold["hyp_counts"])
    small_m, small_v = _dev(*variant_inputs(5, 3)[:2])
    hyp, cnt = ransac_voting_hypothesis(small_m, small_v, 8)
    assert not hyp.any() and (cnt == 1).all()


def test_distribution_against_reference_fixture(gold):
    seed, n, _ = (int(v) for v in gold["dist_seed"])
    mask, vertex, _ = variant_inputs(seed, n)
    m, v = _dev(mask, vertex)
    idxs = torch.from_numpy(gold["dist_idxs"].reshape(1, 96, 5, 2)).to(DEV)
    mean, cov = estimate_voting_distribution(m, v, 32, 96, 24, inlier_thresh=0.99, idxs=idxs)
    # keypoints with a tie at the top-k cut: torch.topk's pick among equals is unspecified
    ratio = po.estimate_voting_distribution(mask, vertex, 32, 96, 24, inlier_thresh=0.99, idxs=[gold["dist_idxs"]],
                                            return_ratio=True)[2][0]
    srt = -np.sort(-ratio, axis=1)
    ok = srt[:, 23] != srt[:, 24]
    assert ok.sum() >= 2
    assert np.abs(mean.cpu().numpy() - gold["dist_mean"])[0, ok].max() <= 1e-4 * 80
    assert np.abs(cov.cpu().numpy() - gold["dist_cov"])[0, ok].max() <= 1e-4 * max(1.0, np.abs(gold["dist_cov"]).max())


def test_motion_voting(gold):
    seed, n, _ = (int(v) for v in gold["motion_seed"])
    mask, vertex, _ = variant_inputs(seed, n)
    m, v = _dev(mask, vertex)
    out = ransac_motion_voting(m, v).cpu().numpy()
    assert np.abs(out - gold["motion_out"]).max() <= 1e-4
    assert np.abs(out - po.ransac_motion_voting(mask, vertex)).max() <= 1e-5
    assert not ransac_motion_voting(torch.zeros_like(m), v).any()       # empty mask: zeros (:971-973)


def test_motion_voting_full_size_batch():
    """480x640, K=9, batch 3 with different foreground sizes; int64 argmax-style mask."""
    ms, vs = [], []
    for i, n in enumerate((20000, 1, 7777)):
        mask = syn.disc_mask(n)
        ms.append(mask)
        vs.append(syn.planted_field(mask, 9, 50 + i)[0])
    mask = np.stack(ms).astype(np.int64)
    field = np.stack(vs)                                                # [b,18,480,640]
    vertex = syn.as_reference_view(field)
    nchw = torch.from_numpy(field).to(DEV)
    v = nchw.permute(0, 2, 3, 1).view(3, 480, 640, 9, 2)
    out = ransac_motion_voting(torch.from_numpy(mask).to(DEV), v).cpu().numpy()
    ref = po.ransac_motion_voting(mask, vertex)
    assert np.abs(out - ref).max() <= 1e-4


def test_v4_against_oracle():
    mask, vertex, _ = variant_inputs(21, 600)
    rng = np.random.default_rng(0)
    idxs = rng.integers(0, 600, (1, 40, 5, 2), dtype=np.int32)
    m, v = _dev(mask, vertex)
    kp, var = ransac_voting_layer_v4(m, v, 40, idxs=torch.from_numpy(idxs).to(DEV))
    kp_o, var_o = po.ransac_voting_layer_v4(mask, vertex, 40, idxs=[idxs[0]])
    assert np.abs(kp.cpu().numpy() - kp_o).max() <= 1e-4
    assert np.abs(var.cpu().numpy() - var_o).max() <= 1e-4 * max(1.0, np.abs(var_o).max())
    sm, sv = _dev(*variant_inputs(5, 3)[:2])
    kp, var = ransac_voting_layer_v4(sm, sv, 8)
    assert not kp.any() and (var == 1).all()                            # skipped image (:685-689)


def test_v4_full_size():
    mask = syn.disc_mask(20000)
    field = syn.planted_field(mask, 9, 3)[0]
    vertex = syn.as_reference_view(field[None])
    idxs = syn.draw_idxs(20000, 128, 9, seed=5)[None]
    nchw = torch.from_numpy(field[None]).to(DEV)
    v = nchw.permute(0, 2, 3, 1).view(1, 480, 640, 9, 2)
    kp, var = ransac_voting_layer_v4(torch.from_numpy(mask[None].astype(np.int64)).to(DEV), v, 128,
                                     idxs=torch.from_numpy(idxs).to(DEV))
    kp_o, var_o = po.ransac_voting_layer_v4(mask[None], vertex, 128, idxs=[idxs[0]])
    assert np.abs(kp.cpu().numpy() - kp_o).max() <= 1e-4
    assert np.abs(var.cpu().numpy() - var_o).max() <= 1e-4 * max(1.0, np.abs(var_o).max())


# ---------------------------------------------------------------- vanishing-point pair (ransac_voting_kernel.cu:170-351)
def test_vanishing_point_pair_bit_exact_vs_oracle_and_reference_kernels(golden_dir):
    from pvnet_b200 import ransac_voting as ext
    direct, coords, idxs = vp_inputs(21)
    d, c, i = (torch.from_numpy(a).to(DEV) for a in (direct, coords, idxs))
    hyp = ext.generate_hypothesis_vanishing_point(d, c, i)
    ohyp = po.generate_hypothesis_vanishing_point_kernel(direct, coords, idxs)
    assert np.array_equal(hyp.cpu().numpy().view(np.uint32), ohyp.view(np.uint32))
    assert (ohyp == 0).all(axis=2).any() and (ohyp != 0).any()            # both the zeroed and the kept branch occur
    for thresh in (0.99, 0.5):
        inl = torch.zeros([96, 4, 3000], dtype=torch.uint8, device=DEV)
        cnt = ext.voting_for_hypothesis_vanishing_point(d, c, hyp, inl, thresh, return_counts=True)
        oinl = po.voting_for_hypothesis_vanishing_point_kernel(direct, coords, ohyp, thresh)
        assert np.array_equal(inl.cpu().numpy(), oinl)
        assert np.array_equal(cnt.cpu().numpy(), oinl.sum(2))
        assert oinl.sum() > 1000
    # the reference's own kernels pin both (tests/golden/make_golden_ref_cuda.py)
    ref = np.load(os.path.join(golden_dir, "ref_cuda_kernels.npz"))
    assert np.array_equal(ref["vp_hyp"].view(np.int32), hyp.cpu().numpy().view(np.int32))
    inl = torch.zeros([96, 4, 3000], dtype=torch.uint8, device=DEV)
    ext.voting_for_hypothesis_vanishing_point(d, c, hyp, inl, 0.99)
    assert ref["vp_inliers"] == digest(inl.cpu().numpy())


def test_v2_against_reference_fixture(gold):
    """ransac_voting_layer_v2 with two refinement rounds: output of the reference's own function (pinverse
    refits in fp32) vs ours (normal equations in fp64)."""
    from lib.ransac_voting_gpu_layer.ransac_voting_gpu import ransac_voting_layer_v2
    seed, n, classes = (int(v) for v in gold["v2_seed"])
    mask, vertex, _ = variant_inputs(seed, n, classes)
    m, v = _dev(mask, vertex)
    idxs = torch.from_numpy(gold["v2_idxs"])[:, None].to(DEV)           # [class, b=1, hn, K, 2]
    out = ransac_voting_layer_v2(m, v, classes + 1, 32, inlier_thresh=0.99, refine_iter_num=2, idxs=idxs)
    assert out.shape == (1, classes, 5, 2)
    assert np.abs(out.cpu().numpy() - gold["v2_out"]).max() <= 2e-4
    one = ransac_voting_layer_v2(m, v, classes + 1, 32, inlier_thresh=0.99, refine_iter_num=1, idxs=idxs)
    assert np.abs((one - out).cpu().numpy()).max() < 1.0 and not torch.equal(one, out)


def test_class_layers_replay_rng_in_image_class_order():
    """v1/v2 with rng="reference", two images x two classes: the torch RNG calls happen in the reference's
    `for bi: for k:` order (ransac_voting_gpu.py:23-26)."""
    from lib.ransac_voting_gpu_layer.ransac_voting_gpu import ransac_voting_layer_v2
    masks, verts = zip(*[variant_inputs(30 + i, 900, 2)[:2] for i in range(2)])
    m, v = _dev(np.concatenate(masks), np.concatenate(verts))
    torch.manual_seed(9)
    got = ransac_voting_layer_v2(m, v, 3, 24, inlier_thresh=0.99)
    torch.manual_seed(9)
    idxs = torch.zeros([2, 2, 24, 5, 2], dtype=torch.int32, device=DEV)    # [class, b, ...]
    for bi in range(2):
        for k in range(2):
            tn = int((m[bi] == k + 1).sum())
            idxs[k, bi] = torch.zeros([24, 5, 2], dtype=torch.int32, device=DEV).random_(0, tn)
    want = ransac_voting_layer_v2(m, v, 3, 24, inlier_thresh=0.99, idxs=idxs)
    assert torch.equal(got, want)


def test_vanish_point_layer_recovers_a_planted_vanishing_point():
    """The reference layer cannot run as written (undefined `class_num`, :415) and ships no expected
    values: pin behaviour by a known answer -- every pixel's direction points at one finite point per
    keypoint, so the homogeneous result is proportional to (x, y, 1) of that point (the reference's own
    disabled check, :1088-1097)."""
    from lib.ransac_voting_gpu_layer.ransac_voting_gpu import ransac_voting_vanish_point_layer
    H, W, K = 64, 80, 3
    targets = np.array([[100.0, 20.0], [-30.0, 40.0], [45.0, 150.0]])
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    mask = np.zeros((1, H, W), np.int64)
    mask[0, 16:48, 20:60] = 1
    vertex = np.zeros((1, H, W, K, 2), np.float32)
    for k in range(K):
        d = np.stack([targets[k, 0] - xx, targets[k, 1] - yy], -1)
        vertex[0, :, :, k] = (d / np.linalg.norm(d, axis=-1, keepdims=True)) * mask[0, :, :, None]
    m, v = _dev(mask, vertex)
    torch.manual_seed(0)
    out = ransac_voting_vanish_point_layer(m, v, 64, inlier_thresh=0.999)
    assert out.shape == (1, 1, K, 3)
    o = out[0, 0].cpu().numpy().astype(np.float64)
    assert np.abs(np.linalg.norm(o, axis=1) - 1).max() < 1e-5
    assert np.abs(o[:, :2] / o[:, 2:3] - targets).max() < 5e-2
