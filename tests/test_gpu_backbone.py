"""GPU: the native Resnet18_8s (tcgen05 convs) against (a) the golden outputs produced by the
REFERENCE classes on the CPU in true fp32 (a seeded sample of positions in every output plane),
(b) our torch graph on the GPU with TF32 off (every position, full size).

Tolerance.  The native path computes every conv with TF32 inputs (10-bit mantissa) and fp32
accumulation -- what the reference's own cuDNN path does on this GPU under torch's default
`cudnn.allow_tf32=True`.  Through 26 layers this gives ~2e-3 of the output range.  The bound is 3x the
error cuDNN-TF32 itself shows on the same input in the same test (floor 3e-3 of the range, in case cuDNN
picks fp32 kernels for the small test shapes): a dropped K-block or tap in any layer, or a wrong BN fold,
moves the output by far more.  Argmax flips against the fp32 graph are bounded too."""
import os

import numpy as np
import pytest
import torch

from pvnet_b200.model_repository import Resnet18_8s
from tests.helpers import GOLDEN, backbone_input, backbone_sample, digest, seeded_state_dict

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _net(ver, seed=1):
    net = Resnet18_8s(ver, 2)
    net.load_state_dict(seeded_state_dict(net, seed=seed))
    return net.to(DEV).eval()


class _tf32:
    """cudnn / matmul TF32 switches, restored on exit."""

    def __init__(self, on):
        self.on = on

    def __enter__(self):
        self.old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = self.on
        torch.backends.cuda.matmul.allow_tf32 = self.on

    def __exit__(self, *a):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.old


def _cudnn_tf32_error(net, x, ref):
    """max abs deviation of the torch graph under cuDNN-TF32 from `ref` (true fp32) on this input"""
    with torch.no_grad(), _tf32(True):
        t = torch.cat(net._forward_torch(x), 1)
    return (t - ref).abs().max().item()


def _sampled(z, tag, seg, ver):
    """(seg, ver) outputs on the device at the golden file's positions, as numpy [b,c,k]"""
    return (backbone_sample(seg.cpu().numpy(), z[tag + "_seg_pos"]), backbone_sample(ver.cpu().numpy(), z[tag + "_ver_pos"]))


def _cudnn_tf32_error_sampled(net, x, z, tag):
    """max abs deviation of the torch graph under cuDNN-TF32 from the golden (true fp32) samples on this input"""
    with torch.no_grad(), _tf32(True):
        t = _sampled(z, tag, *net._forward_torch(x))
    return max(np.abs(t[0] - z[tag + "_seg"]).max(), np.abs(t[1] - z[tag + "_ver"]).max())


@pytest.mark.parametrize("mode", [0, 1], ids=["auto(column+fused head)", "per-tap only"])
@pytest.mark.parametrize("tag,ver", [("k9", 18), ("k17", 34)])
def test_native_vs_reference_golden(tag, ver, mode):
    from pvnet_b200 import conv as pc
    z = np.load(os.path.join(GOLDEN, "resnet18_8s_ref.npz"))
    pc.set_mode(mode)
    try:
        net = _net(ver)
        x_np = backbone_input(tag)
        assert digest(x_np) == z[tag + "_x_digest"], "the fixture's seeded input changed"
        x = torch.from_numpy(x_np).to(DEV)
        with torch.no_grad():
            seg, v = net(x)
        torch.cuda.synchronize()
    finally:
        pc.set_mode(0)
    e_cudnn = _cudnn_tf32_error_sampled(net, x, z, tag)
    for name, got, ref in zip(("seg", "ver"), _sampled(z, tag, seg, v), (z[tag + "_seg"], z[tag + "_ver"])):
        err = np.abs(got - ref).max()
        scale = np.abs(ref).max()
        print(f"\n[backbone vs reference fp32 golden] {tag} {name}: max abs err {err:.3e}, range {scale:.3f}, "
              f"rel {err / scale:.3e}; cuDNN-TF32 on the same input: {e_cudnn:.3e}")
        assert err <= max(3.0 * e_cudnn, 3e-3 * scale)


def test_native_vs_torch_graph_fullsize_and_mask():
    net = _net(18, seed=3)
    x = torch.from_numpy(np.random.default_rng(0).standard_normal((2, 3, 480, 640), dtype=np.float32)).to(DEV)
    with torch.no_grad():
        with _tf32(False):
            rs, rv = net._forward_torch(x)
        with _tf32(True):
            ts, tv = net._forward_torch(x)
        out, mask = net.forward_native(x, with_mask=True)
        out8, mask8 = net.forward_native(x, with_mask=True, mask_dtype=torch.uint8)
    torch.cuda.synchronize()
    seg, ver = out[:, :2], out[:, 2:]
    e_seg = (seg - rs).abs().max().item() / rs.abs().max().item()
    e_ver = (ver - rv).abs().max().item() / rv.abs().max().item()
    c_seg = (ts - rs).abs().max().item() / rs.abs().max().item()
    c_ver = (tv - rv).abs().max().item() / rv.abs().max().item()
    # bit-exact argmax GIVEN our logits (the fused head's mask == torch.argmax of its own output)
    assert torch.equal(mask, torch.argmax(seg, 1))
    assert torch.equal(out8, out) and torch.equal(mask8.long(), mask)
    flips = (mask != torch.argmax(rs, 1)).float().mean().item()
    flips_cudnn = (torch.argmax(ts, 1) != torch.argmax(rs, 1)).float().mean().item()
    print(f"\n[backbone vs torch fp32 graph] 480x640: rel err seg {e_seg:.3e}, ver {e_ver:.3e} (cuDNN-TF32: {c_seg:.3e}, "
          f"{c_ver:.3e}); argmax pixels differing from the fp32 graph: {flips * 100:.4f}% (cuDNN-TF32: {flips_cudnn * 100:.4f}%)")
    assert e_seg <= max(3 * c_seg, 3e-3) and e_ver <= max(3 * c_ver, 3e-3)
    assert flips <= max(3 * flips_cudnn, 1e-4), "argmax flip rate against the fp32 graph"


def test_native_matches_cudnn_tf32_class():
    """The reference's default numerics on this GPU (cuDNN TF32) deviate from fp32 by about as
    much as the native path does."""
    net = _net(18, seed=5)
    x = torch.from_numpy(np.random.default_rng(1).standard_normal((1, 3, 240, 320), dtype=np.float32)).to(DEV)
    with torch.no_grad():
        with _tf32(False):
            f32 = torch.cat(net._forward_torch(x), 1)
        with _tf32(True):
            tf32 = torch.cat(net._forward_torch(x), 1)
        ours = net.forward_native(x)
    scale = f32.abs().max().item()
    e_cudnn = (tf32 - f32).abs().max().item() / scale
    e_ours = (ours - f32).abs().max().item() / scale
    print(f"\n[tf32 class] rel err vs fp32: cuDNN-TF32 {e_cudnn:.3e}, native {e_ours:.3e}")
    assert e_ours < max(3 * e_cudnn, 3e-3)


def test_reference_view_roundtrip_into_vote():
    """forward -> argmax -> permuted view -> ransac_voting_layer_v3, as tools/demo.py:46-55."""
    from pvnet_b200 import ransac_voting_gpu as rv
    net = _net(18, seed=7)
    x = torch.randn(2, 3, 128, 160, device=DEV)
    with torch.no_grad():
        seg_pred, vertex_pred = net(x)
    vertex = vertex_pred.permute(0, 2, 3, 1)
    b, h, w, vn2 = vertex.shape
    vertex = vertex.view(b, h, w, vn2 // 2, 2)
    mask = torch.argmax(seg_pred, 1)
    kp = rv.ransac_voting_layer_v3(mask, vertex, 64, inlier_thresh=0.99)
    assert kp.shape == (2, 9, 2)


def test_weights_update_is_picked_up():
    net = _net(18, seed=9)
    x = torch.randn(1, 3, 64, 64, device=DEV)
    with torch.no_grad():
        a = net.forward_native(x).clone()
        net.convraw[3].bias.add_(1.0)
        b = net.forward_native(x)
    assert torch.allclose(b - a, torch.ones_like(a), atol=1e-5)


def test_odd_sizes_multiple_of_8():
    net = _net(18, seed=2)
    for h, w in [(72, 104), (256, 264)]:
        x = torch.randn(1, 3, h, w, device=DEV)
        with torch.no_grad():
            with _tf32(False):
                ref = torch.cat(net._forward_torch(x), 1)
            out = net.forward_native(x)
        assert (out - ref).abs().max().item() <= max(3 * _cudnn_tf32_error(net, x, ref), 3e-3 * ref.abs().max().item())


@pytest.mark.parametrize("shape", [(2, 480, 640), (1, 72, 104), (3, 16, 16), (1, 256, 264)], ids=str)
@pytest.mark.parametrize("pixel_major", [False, True], ids=["nchw", "pixel-major"])
@pytest.mark.parametrize("mode", [1, 2], ids=["epilogue warps", "dedicated warps"])
def test_fused_upsample_equals_separate_launch(shape, pixel_major, mode):
    """convraw.0 interpolating its upsampled input itself (pvnet_backbone_set_fused_upsample) against the separate
    k_upsample2x launch it replaces: the same ATen arithmetic on the same conv2s.0 output, so the two forwards agree to the last bit
    (partial tiles, image borders and the last-row rounding case of the align_corners scale included)."""
    b, h, w = shape
    net = _net(18, seed=11)
    x = torch.from_numpy(np.random.default_rng(5).standard_normal((b, 3, h, w), dtype=np.float32)).to(DEV)
    with torch.no_grad():
        net.set_fused_upsample(False)
        launches0 = _launches(lambda: net.forward_native(x, with_mask=True, mask_dtype=torch.uint8, pixel_major=pixel_major))
        sep, msep = net.forward_native(x, with_mask=True, mask_dtype=torch.uint8, pixel_major=pixel_major)
        sep, msep = sep.clone(), msep.clone()
        net.set_fused_upsample(mode)
        launches1 = _launches(lambda: net.forward_native(x, with_mask=True, mask_dtype=torch.uint8, pixel_major=pixel_major))
        fused, mfused = net.forward_native(x, with_mask=True, mask_dtype=torch.uint8, pixel_major=pixel_major)
        net.set_fused_upsample(None)
    torch.cuda.synchronize()
    assert launches1 == launches0 - 1, "the fused form has one launch less (no 1/2 -> 1 k_upsample2x)"
    d = (fused - sep).abs().max().item()
    print(f"\n[fused upsample] {shape} pixel_major={pixel_major}: max abs diff {d:.3e}, launches {launches0} -> {launches1}")
    assert torch.equal(fused, sep), f"fused and separate upsampling differ by {d:.3e}"
    assert torch.equal(mfused, msep)


@pytest.mark.parametrize("fused", [False, True], ids=["separate upsampling", "fused upsampling"])
def test_two_epilogue_sets_equal_one(fused):
    """The fused-head kernel with two epilogue warp sets alternating tiles (tuning knob, 96 registers per thread)
    computes exactly what the default single set does."""
    from pvnet_b200 import conv as pc
    x = torch.from_numpy(np.random.default_rng(6).standard_normal((2, 3, 240, 328), dtype=np.float32)).to(DEV)
    outs = []
    for sets in (1, 2):
        pc.set_head_epilogue_sets(sets)
        try:
            net = _net(18, seed=12).set_fused_upsample(1 if fused else 0)     # a fresh handle: plans are built under the hook
            with torch.no_grad():
                outs.append(net.forward_native(x, with_mask=True, mask_dtype=torch.uint8))
            torch.cuda.synchronize()
        finally:
            pc.set_head_epilogue_sets(0)
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def _launches(fn):
    from pvnet_b200 import _native
    _native.launch_count_reset()
    fn()
    return _native.launch_count()
