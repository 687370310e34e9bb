"""CPU: the reference's evaluation import line resolves against the shims, the new shim functions keep the
reference's signatures, the nearest-neighbour oracle equals the reference kernel (tests/golden/ref_nn.npz) bit
for bit, and the metric oracle reproduces the reference's Evaluator (tests/golden/ref_metrics.npz)."""
import ctypes
import inspect
import json
import os

import numpy as np
import pytest

from oracle import metrics_oracle as mo
from tests.helpers import digest
from tests.metrics_cases import model_points, nn_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_evaluation_utils_import_line():
    # lib/utils/evaluation_utils.py:16, verbatim
    from lib.utils.extend_utils.extend_utils import uncertainty_pnp, find_nearest_point_idx, uncertainty_pnp_v2  # noqa
    assert callable(find_nearest_point_idx) and callable(uncertainty_pnp_v2) and callable(uncertainty_pnp)


def test_shim_signatures_equal_reference():
    import lib.utils.extend_utils.extend_utils as shim
    with open(os.path.join(GOLDEN, "ref_extend_signatures.json")) as f:
        expected = json.load(f)
    assert sorted(expected) == ["find_nearest_point_idx", "uncertainty_pnp_v2"]
    for name, sig in expected.items():
        got = ", ".join(p.name if p.default is inspect.Parameter.empty else f"{p.name}={p.default!r}"
                        for p in inspect.signature(getattr(shim, name)).parameters.values())
        assert got == sig, name


def test_nn_oracle_equals_reference_kernel():
    z = np.load(os.path.join(GOLDEN, "ref_nn.npz"))
    cases = nn_cases()
    assert len(cases) == len([k for k in z.files if k.endswith("_idx")]) - 3
    for name, (ref, que, excl) in cases.items():
        assert str(z[f"{name}_in"]) == digest(np.concatenate([ref.ravel(), que.ravel()])), name
        got = mo.find_nearest_point_idx_batched(ref, que, excl)
        assert got.dtype == np.int32 and np.array_equal(got, z[f"{name}_idx"]), name


def test_nn_oracle_selection_rule():
    ref = np.array([[1, 0, 0], [0, 1, 0], [np.nan, 0, 0], [-1, 0, 0], [1, 0, 0]], np.float32)
    que = np.array([[0, 0, 0], [1, 0, 0], [np.inf, 0, 0]], np.float32)
    # equidistant -> lowest index; exact duplicate -> first copy; all distances inf/NaN -> 0
    assert mo.find_nearest_point_idx(ref, que).tolist() == [0, 0, 0]
    assert mo.find_nearest_point_idx_batched(ref[None], ref[None], exclude_self=True)[0].tolist() == [4, 0, 0, 1, 0]


def _close(a, b, rtol):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.all((np.abs(a - b) <= rtol * np.abs(b)) | (np.isnan(a) & np.isnan(b)))


def test_metric_oracle_reproduces_reference():
    z = np.load(os.path.join(GOLDEN, "ref_metrics.npz"))
    assert len(z["names"]) >= 30
    for i, name in enumerate(z["names"]):
        X, diameter = model_points(str(z["kinds"][i]), int(z["model_sizes"][i]))
        pp, pg = z["pose_pred"][i], z["pose_gt"][i]
        assert pp.dtype == np.float64 and pg.dtype == np.float32
        for sym_add in (False, True):
            for sym_proj in (False, True):
                m = mo.pose_metrics(pp, pg, X, z["K"], diameter, sym_add=sym_add, sym_proj=sym_proj)
                a, p = ("adds" if sym_add else "add"), ("projs" if sym_proj else "proj")
                assert _close(m["add_dist"], z[a][i], 1e-9), (name, a, m["add_dist"], z[a][i])
                assert _close(m["proj_mean_diff"], z[p][i], 1e-9), (name, p, m["proj_mean_diff"], z[p][i])
                assert m["add_ok"] == z[a + "_ok"][i] and m["proj_ok"] == z[p + "_ok"][i], name
                assert m["cm5_ok"] == z["cm_ok"][i], name
    # the fixture reaches both sides of every threshold and the NaN angle
    for key in ("add_ok", "proj_ok", "cm_ok"):
        assert z[key].any() and not z[key].all()
    names = list(z["names"])
    m = mo.pose_metrics(z["pose_pred"][names.index("torus_trace_below_m1")],
                        z["pose_gt"][names.index("torus_trace_below_m1")], *model_points("torus", 3001)[:1], z["K"], 0.2)
    assert np.isnan(m["rot_deg"]) and not m["cm5_ok"]


def test_entry_points_validate_arguments():
    from pvnet_b200 import _native
    L = _native.lib()
    assert L.pvnet_find_nearest_point_idx(None, None, None, 1, 1, 1, 3, 0, None) == -1
    assert b"null" in L.pvnet_last_error()
    p = ctypes.c_void_p(16)
    assert L.pvnet_find_nearest_point_idx(p, p, p, 1, 4, 4, 4, 0, None) == -1
    assert b"dim" in L.pvnet_last_error()
    assert L.pvnet_find_nearest_point_idx(p, p, p, 1, 0, 4, 3, 0, None) == -1
    n = ctypes.c_size_t()
    assert L.pvnet_pose_metrics_workspace_bytes(16, 2048, 0, ctypes.byref(n)) == 0 and n.value == 0
    assert L.pvnet_pose_metrics_workspace_bytes(16, 2048, 3, ctypes.byref(n)) == 0
    assert n.value >= 16 * 2048 * (6 + 4) * 4 + 2 * 16 * 2048 * 4
    K = (ctypes.c_double * 9)()
    assert L.pvnet_pose_metrics(p, p, p, K, p, 1, 8, 0, 1.0, 5.0, 5.0, 5.0, p, p, None, 0, None) == -1
    assert b"exactly one" in L.pvnet_last_error()
    assert L.pvnet_pose_metrics(p, p, p, K, None, 1, 8, 1, 1.0, 5.0, 5.0, 5.0, p, p, p, 16, None) == -2
    assert L.pvnet_pose_metrics(p, p, p, K, None, 1, 8, 64, 1.0, 5.0, 5.0, 5.0, p, p, None, 0, None) == -1


def test_device_paths_refuse_host_tensors():
    import torch
    from pvnet_b200 import evaluation
    from pvnet_b200 import extend_utils as eu
    with pytest.raises(RuntimeError, match="CUDA"):
        eu.find_nearest_point_idx(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        evaluation.pose_metrics(torch.zeros(1, 3, 4), torch.zeros(1, 3, 4), torch.zeros(8, 3), np.eye(3), 0.1)
