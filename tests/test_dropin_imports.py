"""CPU: the reference's import lines resolve against the shims under lib/, and the public
signatures (parameter names and defaults) equal the reference's.  The expected signatures are
transcribed from lib/ransac_voting_gpu_layer/ransac_voting_gpu.py and compared with the ones
tests/golden/make_golden_signatures.py derived from its source with `ast`
(tests/golden/ref_signatures.json)."""
import inspect
import json
import os

import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

EXPECTED = {
    "ransac_voting_layer": "mask, vertex, class_num, round_hyp_num, inlier_thresh=0.999, confidence=0.99, max_iter=20, min_num=5, max_num=30000",
    "ransac_voting_layer_v2": "mask, vertex, class_num, round_hyp_num, inlier_thresh=0.999, confidence=0.99, max_iter=20, min_num=5, max_num=30000, refine_iter_num=1",
    "ransac_voting_vanish_point_layer": "mask, vertex, round_hyp_num, inlier_thresh=0.999, confidence=0.99, max_iter=20, min_num=5, max_num=30000, refine_iter_num=1",
    "ransac_voting_hypothesis": "mask, vertex, round_hyp_num, inlier_thresh=0.999, min_num=5, max_num=30000",
    "estimate_voting_distribution": "mask, vertex, round_hyp_num=256, min_hyp_num=4096, topk=128, inlier_thresh=0.99, min_num=5, max_num=30000",
    "estimate_voting_distribution_with_mean": "mask, vertex, mean, round_hyp_num=256, min_hyp_num=4096, topk=128, inlier_thresh=0.99, min_num=5, max_num=30000, output_hyp=False",
    "ransac_voting_layer_v3": "mask, vertex, round_hyp_num, inlier_thresh=0.999, confidence=0.99, max_iter=20, min_num=5, max_num=30000",
    "ransac_voting_layer_v4": "mask, vertex, round_hyp_num, inlier_thresh=0.99, confidence=0.999, max_iter=20, min_num=5, max_num=30000",
    "ransac_voting_layer_v5": "mask, vertex, round_hyp_num, inlier_thresh=0.999, confidence=0.99, max_iter=20, min_num=5, max_num=100",
    "ransac_motion_voting": "mask, vertex",
    "generate_hypothesis": "mask, vertex, round_hyp_num, inlier_thresh=0.999, confidence=0.99, max_iter=20, min_num=5, max_num=30000",
}


def _positional_signature(fn):
    parts = []
    for p in inspect.signature(fn).parameters.values():
        if p.kind is not inspect.Parameter.POSITIONAL_OR_KEYWORD:
            continue                      # keyword-only extras (idxs=, selection=, rng=) are ours
        parts.append(p.name if p.default is inspect.Parameter.empty else f"{p.name}={p.default!r}")
    return ", ".join(parts)


def test_reference_import_lines():
    # tools/train_linemod.py:8-10 and tools/demo.py:5,121, verbatim
    from lib.ransac_voting_gpu_layer.ransac_voting_gpu import ransac_voting_layer_v3, \
        estimate_voting_distribution_with_mean, ransac_voting_layer_v5, ransac_motion_voting  # noqa: F401
    from lib.networks.model_repository import Resnet18_8s  # noqa: F401
    from lib.ransac_voting_gpu_layer.ransac_voting_gpu import generate_hypothesis  # noqa: F401
    # lib/utils/extend_utils/extend_utils.py:241
    from lib.ransac_voting_gpu_layer.ransac_voting_gpu import ransac_voting_layer  # noqa: F401


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_signature_equals_reference(name):
    import lib.ransac_voting_gpu_layer.ransac_voting_gpu as shim
    assert _positional_signature(getattr(shim, name)) == EXPECTED[name]


def test_expected_signatures_match_reference_source():
    # pins the transcription EXPECTED to the reference's source; test_signature_equals_reference is what checks the shim
    with open(os.path.join(GOLDEN, "ref_signatures.json")) as f:
        assert json.load(f) == EXPECTED
