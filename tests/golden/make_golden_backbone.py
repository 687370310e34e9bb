"""Regenerates tests/golden/resnet18_8s_ref.npz on the CPU:
    python tests/golden/make_golden_backbone.py REFERENCE_ROOT

Imports the REFERENCE network classes from REFERENCE_ROOT/lib/networks/{resnet,
model_repository}.py (by file path, with `lib.utils.config` stubbed and the ImageNet
download at resnet.py:231 switched off), loads the deterministic weights of
tests/helpers.seeded_state_dict and runs Resnet18_8s(ver_dim, 2).eval() in true fp32 on the
seeded input of tests/helpers.backbone_input for each BACKBONE_CASES entry.  The tests rebuild
the same weights and input and check that our module reproduces these outputs: the graph
(dilation rules, decoder wiring, align_corners upsampling, channel order of the concatenations)
is pinned to the reference's.

Stored per case (the whole outputs would exceed 1 MB): `<tag>_x_digest` (tests.helpers.digest of
the input, so that a changed random stream fails loudly), and for seg and ver a fixed seeded sample
of SAMPLES[name] positions in every (image, channel) plane: `<tag>_<name>_pos` [2,C,k] uint16 flat
H*W indices, sorted, and `<tag>_<name>` [2,C,k] float32 the outputs there.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
# positions sampled per (image, channel) plane, per case and output
SAMPLES = {"k9": {"seg": 512, "ver": 256}, "k17": {"seg": 512, "ver": 128}}


def load_reference_classes(ref):
    saved = {k: sys.modules.get(k) for k in ("lib", "lib.utils", "lib.utils.config", "lib.networks",
                                             "lib.networks.resnet", "lib.networks.model_repository")}
    lib = types.ModuleType("lib"); lib.__path__ = []
    utils = types.ModuleType("lib.utils"); utils.__path__ = []
    cfgm = types.ModuleType("lib.utils.config"); cfgm.cfg = types.SimpleNamespace(MODEL_DIR="/tmp")
    nets = types.ModuleType("lib.networks"); nets.__path__ = []
    sys.modules.update({"lib": lib, "lib.utils": utils, "lib.utils.config": cfgm, "lib.networks": nets})

    def load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    r = load("lib.networks.resnet", os.path.join(ref, "resnet.py"))
    orig = r.resnet18
    r.resnet18 = lambda pretrained=False, **kw: orig(pretrained=False, **kw)   # no network here
    mr = load("lib.networks.model_repository", os.path.join(ref, "model_repository.py"))
    cls = mr.Resnet18_8s
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v
    return cls


def main():
    cls = load_reference_classes(os.path.join(sys.argv[1], "lib", "networks"))
    sys.path.insert(0, ROOT)
    from tests.helpers import BACKBONE_CASES, backbone_input, backbone_sample, digest, seeded_state_dict
    rng = np.random.default_rng(11)
    out = {}
    for tag, (ver, h, w) in BACKBONE_CASES.items():
        net = cls(ver, 2)
        net.load_state_dict(seeded_state_dict(net, seed=1))
        net.eval()
        x = backbone_input(tag)
        with torch.no_grad():
            s, v = net(torch.from_numpy(x))
        out[tag + "_x_digest"] = np.array(digest(x))
        for name, a in (("seg", s.numpy()), ("ver", v.numpy())):
            b, c = a.shape[:2]
            pos = np.sort(np.stack([rng.permutation(h * w)[:SAMPLES[tag][name]] for _ in range(b * c)]), axis=1)
            pos = pos.reshape(b, c, -1).astype(np.uint16)
            out[f"{tag}_{name}_pos"] = pos
            out[f"{tag}_{name}"] = backbone_sample(a, pos)
    path = os.path.join(HERE, "resnet18_8s_ref.npz")
    np.savez_compressed(path, **out)
    print({k: v.shape for k, v in out.items()}, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
