"""Shared test helpers (CPU side)."""
import hashlib
import os

import numpy as np

from pvnet_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def demo_fixture():
    """mask int64 [480,640], exact vector field NCHW [18,480,640] f32, points_2d [9,2].
    The field is rebuilt from the fixture with the recipe of the reference's
    tools/demo.py:58-71 (`compute_vertex`): (kp - xy)/norm, norm<1e-3 -> +1e-3."""
    z = np.load(os.path.join(GOLDEN, "demo_cat.npz"))
    h, w = (int(v) for v in z["shape"])
    fg = z["fg_yx"].astype(np.int64)
    pts = z["points_2d"]
    mask = np.zeros((h, w), np.int64)
    mask[fg[:, 0], fg[:, 1]] = 1
    xy = fg[:, [1, 0]].astype(np.float64)
    v = pts[None, :, :2] - xy[:, None, :]
    n = np.linalg.norm(v, axis=2, keepdims=True)
    n[n < 1e-3] += 1e-3
    v = v / n
    field = np.zeros((h, w, pts.shape[0], 2), np.float32)
    field[fg[:, 0], fg[:, 1]] = v
    nchw = np.ascontiguousarray(field.reshape(h, w, -1).transpose(2, 0, 1))
    return mask, nchw, pts


def cfg1_inputs(kind):
    mask = syn.disc_mask(10000)
    field = syn.random_field(mask, 9, 1000) if kind == "random" else syn.planted_field(mask, 9, 1000)[0]
    idxs = syn.draw_idxs(10000, 128, 9, seed=1000)
    return mask, field, idxs


def seeded_state_dict(model, seed=0):
    """Deterministic weights for a Resnet18_8s-shaped module, a pure function of
    (parameter name, shape, seed) -- so the golden generator (which builds the REFERENCE
    classes) and the tests (which build ours) get identical tensors without sharing a file.
    Conv weights ~ N(0, sqrt(2/fan_out)); BN gamma ~ U(0.5,1.5), beta ~ N(0,0.1),
    running_mean ~ N(0,0.1), running_var ~ U(0.5,1.5) so folding is exercised."""
    import hashlib

    import torch
    out = {}
    for name, t in model.state_dict().items():
        h = int(hashlib.sha256(f"{seed}:{name}".encode()).hexdigest()[:8], 16)
        g = torch.Generator().manual_seed(h)
        if name.endswith("num_batches_tracked"):
            out[name] = torch.zeros_like(t)
        elif name.endswith("running_var"):
            out[name] = torch.rand(t.shape, generator=g) + 0.5
        elif name.endswith("running_mean"):
            out[name] = torch.randn(t.shape, generator=g) * 0.1
        elif t.dim() == 4:
            fan = t.shape[0] * t.shape[2] * t.shape[3]
            out[name] = torch.randn(t.shape, generator=g) * (2.0 / fan) ** 0.5
        elif name.endswith(".weight"):          # BN gamma
            out[name] = torch.rand(t.shape, generator=g) + 0.5
        else:                                    # BN beta / conv bias
            out[name] = torch.randn(t.shape, generator=g) * 0.1
    return out


# ---------------------------------------------------------------- tests/golden/resnet18_8s_ref.npz
# tag -> (ver_dim, H, W) of the Resnet18_8s(ver_dim, 2) runs whose outputs the fixture samples
BACKBONE_CASES = {"k9": (18, 64, 96), "k17": (34, 48, 64)}


def backbone_input(tag):
    """The fixture's input [2,3,H,W]; the fixture stores its digest, not the array."""
    _, h, w = BACKBONE_CASES[tag]
    return np.random.default_rng(7).standard_normal((2, 3, h, w), dtype=np.float32)


def backbone_sample(out, pos):
    """out [b,c,H,W] (numpy) at the positions pos [b,c,k] (flat H*W indices of each plane) -> [b,c,k]."""
    b, c = out.shape[:2]
    return np.take_along_axis(out.reshape(b, c, -1), pos.astype(np.int64), axis=2)


# ---------------------------------------------------------------- inputs of tests/golden/ref_variants.npz
VARIANT_HWK = (64, 80, 5)


def variant_inputs(seed, n_fg=900, classes=1):
    """mask [1,H,W] int64 with `classes` disc-shaped regions (values 1..classes), vertex
    [1,H,W,K,2] f32: unit vectors towards K planted keypoints, rotated by N(0, 0.05 rad) noise.
    Shared by tests/golden/make_golden_variants.py (which feeds them to the reference's own
    Python functions) and the tests that replay the recorded samples."""
    H, W, K = VARIANT_HWK
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    mask = np.zeros((H, W), np.int64)
    for c in range(classes):
        cx, cy = W * (c + 1) / (classes + 1), H / 2
        d2 = (xx - cx) ** 2 + (yy - cy) ** 2
        order = np.argsort(d2.ravel(), kind="stable")[:n_fg // classes]
        mask.ravel()[order] = c + 1
    kps = np.stack([W / 2 + 30 * np.cos(2 * np.pi * np.arange(K) / K), H / 2 + 20 * np.sin(2 * np.pi * np.arange(K) / K)], 1)
    d = kps[None, None] - np.stack([xx, yy], -1)[:, :, None, :].astype(np.float64)      # [H,W,K,2]
    ang = np.arctan2(d[..., 1], d[..., 0]) + rng.normal(0, 0.05, d.shape[:-1])
    vertex = np.stack([np.cos(ang), np.sin(ang)], -1).astype(np.float32)
    vertex[mask == 0] = 0
    return mask[None], vertex[None], kps


# ---------------------------------------------------------------- inputs of tests/golden/ref_cuda_*.npz
def edge_kernel_inputs():
    """direct [4096,3,2], coords, idxs [64,3,2] with values around the kernels' 1e-6 norm test, zero
    vectors and near-parallel families; and 40 hypotheses ON pixels (norm2 == 0) and far away."""
    rng = np.random.default_rng(0)
    tn, vn, hn = 4096, 3, 64
    direct = rng.standard_normal((tn, vn, 2)).astype(np.float32)
    direct[:200] *= 1e-6
    direct[200:300] = 0
    direct[300:400, :, 1] = direct[300:400, :, 0]
    coords = np.stack([rng.integers(0, 640, tn), rng.integers(0, 480, tn)], 1).astype(np.float32)
    idxs = rng.integers(0, tn, (hn, vn, 2), dtype=np.int32)
    extra = np.concatenate([coords[:32, None, :].repeat(vn, 1), np.full((8, vn, 2), 3e7, np.float32)]).astype(np.float32)
    return direct, coords, idxs, extra


EDGE_THRESHOLDS = (0.99, 0.5, -0.25)


def vp_inputs(seed, tn=3000, vn=4, hn=96):
    """Inputs of the vanishing-point kernel pair: 1e-6 norms, zero vectors, parallel families (z ~ 0)."""
    rng = np.random.default_rng(seed)
    direct = rng.standard_normal((tn, vn, 2)).astype(np.float32)
    direct[:100] *= 1e-6
    direct[100:150] = 0
    direct[150:300, :, 1] = direct[150:300, :, 0]
    coords = np.stack([rng.integers(0, 640, tn), rng.integers(0, 480, tn)], 1).astype(np.float32)
    idxs = rng.integers(0, tn, (hn, vn, 2), dtype=np.int32)
    return direct, coords, idxs


def _near_keypoints_field(mask):
    """Keypoints inside the mask (R=20 px), directions rotated by N(0, 0.03 rad)."""
    rng = np.random.default_rng(5)
    kps = np.stack([320 + 20 * np.cos(np.arange(9)), 240 + 20 * np.sin(np.arange(9))], 1)
    ys, xs = np.mgrid[0:480, 0:640].astype(np.float64)
    field = np.zeros((18, 480, 640), np.float32)
    for j in range(9):
        dx, dy = kps[j, 0] - xs, kps[j, 1] - ys
        n = np.sqrt(dx * dx + dy * dy) + 1e-3
        eps = rng.normal(0, 0.03, size=dx.shape)
        field[2 * j] = (np.cos(eps) * dx / n - np.sin(eps) * dy / n) * (mask != 0)
        field[2 * j + 1] = (np.sin(eps) * dx / n + np.cos(eps) * dy / n) * (mask != 0)
    return field


# hn: round_hyp_num of the v3 comparison (torch seed 0); cov: (torch seed, round_hyp_num, min_hyp_num) of the
# covariance comparison, which starts from the mean the product's v3 gave under (torch seed, round_hyp_num) `mean`
# (stored in the golden file).  inlier_thresh 0.99, max_num 30000 throughout.
REF_LAYER_CASES = {
    "config1": dict(hn=128),
    "demo": dict(hn=512),
    "near": dict(hn=256),
    "subsampled": dict(hn=256),
    "covariance": dict(mean=(1, 256), cov=(2, 128, 512)),
    "config4": dict(hn=256, mean=(44, 256), cov=(45, 256, 4096)),
    "config5": dict(hn=1024, mean=(55, 1024), cov=(56, 1024, 1024)),
}


def ref_layer_inputs(name):
    """mask [b,480,640] and vector field NCHW [b,2K,480,640] of a REF_LAYER_CASES entry."""
    if name == "config1":
        mask, field, _ = cfg1_inputs("planted")
        return np.stack([mask, mask]), np.stack([field, field])
    if name == "demo":
        mask, field, _ = demo_fixture()
        return mask[None], field[None]
    if name == "near":
        mask = syn.disc_mask(3000)
        return mask[None], _near_keypoints_field(mask)[None]
    if name == "subsampled":
        masks = np.stack([syn.disc_mask(40000), syn.disc_mask(3), syn.disc_mask(9000)])
        return masks, np.stack([syn.planted_field(masks[i], 9, 40 + i)[0] for i in range(3)])
    if name == "covariance":
        masks = np.stack([syn.disc_mask(7000), syn.disc_mask(12000)])
        return masks, np.stack([syn.planted_field(masks[i], 9, 60 + i, sigma=0.05)[0] for i in range(2)])
    if name == "config4":
        masks = np.stack([syn.disc_mask(20000)])
        return masks, np.stack([syn.planted_field(masks[0], 9, 4400, sigma=0.05)[0]])
    if name == "config5":
        masks = np.stack([syn.disc_mask(92160)])
        return masks, np.stack([syn.planted_field(masks[0], 17, 5500, sigma=0.05)[0]])
    raise KeyError(name)


def digest(a):
    """sha256 of an array's shape and values (integers as int64, floats as float32 with -0.0 read as 0.0),
    so that equal digests mean np.array_equal arrays whatever their integer width.  The golden files
    keep large exact-match arrays (samples, counts, inlier flags) as digests."""
    a = np.asarray(a)
    a = a.astype("<f4") + np.float32(0) if a.dtype.kind == "f" else a.astype("<i8")
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()
