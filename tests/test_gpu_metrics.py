"""GPU: pvnet_find_nearest_point_idx against the reference kernel's indices (tests/golden/ref_nn.npz) and the
oracle, bit for bit; pose_metrics / DeviceEvaluator against the reference's Evaluator (tests/golden/ref_metrics.npz)
and oracle/metrics_oracle.py; determinism, CUDA-graph capture, and the numpy entry points.

Tolerance of the metric values: 1e-6 relative.  Two values have an absolute floor: the angle, 1e-5 degree,
because arccos near a trace of 3 turns the last bit of the trace into ~3e-6 degree; and, for the per-image K
comparison with the oracle only, nothing else."""
import os

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as mo
from oracle import pnp_oracle as pno
from pvnet_b200 import evaluation as ev
from pvnet_b200 import extend_utils as eu
from tests.helpers import digest
from tests.metrics_cases import K_LINEMOD, large_nn_case, model_points, nn_cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL, DEG_ATOL = 1e-6, 1e-5
LARGE = {"large3": (7, 4, 8192, 8192, 3), "large2": (8, 4, 8192, 8192, 2), "few_queries3": (9, 1, 200003, 96, 3)}
THRESH = {"add_dist": None, "proj_mean_diff": 5.0, "trans_cm": 5.0, "rot_deg": 5.0}


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def test_nn_equals_reference_kernel():
    z = np.load(os.path.join(GOLDEN, "ref_nn.npz"))
    for name, (ref, que, excl) in nn_cases().items():
        got = eu.find_nearest_point_idx_batched(_dev(ref), _dev(que), exclude_self=bool(excl))
        assert got.dtype == torch.int32
        assert np.array_equal(got.cpu().numpy(), z[f"{name}_idx"]), name
    for name, case in LARGE.items():
        ref, que = large_nn_case(*case)
        assert str(z[f"{name}_in"]) == digest(np.concatenate([ref.ravel(), que.ravel()]))
        got = eu.find_nearest_point_idx_batched(_dev(ref), _dev(que)).cpu().numpy()
        assert digest(got) == str(z[f"{name}_idx"]), name


@pytest.mark.parametrize("dim", [3, 2])
def test_nn_equals_oracle_large(dim):
    ref, que = large_nn_case(100 + dim, 16, 16384, 16384, dim)
    got = eu.find_nearest_point_idx_batched(_dev(ref), _dev(que)).cpu().numpy()
    assert np.array_equal(got, mo.find_nearest_point_idx_batched(ref, que))
    # exclude_self on a batch too small to fill the GPU with four queries per lane (one query per lane)
    got = eu.find_nearest_point_idx_batched(_dev(ref[:2, :3000]), _dev(ref[:2, :3000]), exclude_self=True)
    assert np.array_equal(got.cpu().numpy(), mo.find_nearest_point_idx_batched(ref[:2, :3000], ref[:2, :3000], True))


def test_nn_few_queries_large_reference_set():
    ref, que = large_nn_case(11, 2, 300007, 70, 3)
    got = eu.find_nearest_point_idx_batched(_dev(ref), _dev(que)).cpu().numpy()
    assert np.array_equal(got, mo.find_nearest_point_idx_batched(ref, que))


def _fixture():
    z = np.load(os.path.join(GOLDEN, "ref_metrics.npz"))
    groups = {}
    for i, kind in enumerate(z["kinds"]):
        groups.setdefault((str(kind), int(z["model_sizes"][i])), []).append(i)
    return z, groups


def _check(got, want, what):
    for key, thr in THRESH.items():
        a, b = np.asarray(got[key], np.float64), np.asarray(want[key], np.float64)
        tol = RTOL * np.abs(b) + (DEG_ATOL if key == "rot_deg" else 0.0)
        ok = (np.abs(a - b) <= tol) | (np.isnan(a) & np.isnan(b))
        assert ok.all(), (what, key, a[~ok], b[~ok])


def _flags_agree(got_flag, want_flag, values, thresholds, what):
    """Flags must be equal wherever every value is farther than the tolerance from its threshold."""
    far = np.ones(len(got_flag), bool)
    for v, t in zip(values, thresholds):
        far &= ~(np.abs(v - t) <= RTOL * np.abs(t) + 1e-5)
    assert np.array_equal(np.asarray(got_flag)[far], np.asarray(want_flag)[far]), what


@pytest.mark.parametrize("sym_add", [False, True])
@pytest.mark.parametrize("sym_proj", [False, True])
def test_metrics_match_reference_and_oracle(sym_add, sym_proj):
    z, groups = _fixture()
    a, p = ("adds" if sym_add else "add"), ("projs" if sym_proj else "proj")
    for (kind, n), idx in groups.items():
        X, diameter = model_points(kind, n)
        m = ev.pose_metrics(_dev(z["pose_pred"][idx]), _dev(z["pose_gt"][idx]), _dev(X), z["K"], diameter,
                            sym_add=sym_add, sym_proj=sym_proj)
        h = {k: v.cpu().numpy() for k, v in m.items()}
        ref = {"add_dist": z[a][idx], "proj_mean_diff": z[p][idx]}
        orc = [mo.pose_metrics(z["pose_pred"][i], z["pose_gt"][i], X, z["K"], diameter, sym_add=sym_add,
                               sym_proj=sym_proj) for i in idx]
        orc = {k: np.array([o[k] for o in orc]) for k in orc[0]}
        _check(h, orc, (kind, "oracle"))
        for key in ref:
            b = np.asarray(ref[key], np.float64)
            assert (np.abs(h[key] - b) <= RTOL * np.abs(b)).all(), (kind, key, h[key], b)
        thr_add = 0.1 * diameter
        _flags_agree(h["add_ok"], z[a + "_ok"][idx], [h["add_dist"]], [thr_add], (kind, "add"))
        _flags_agree(h["proj_ok"], z[p + "_ok"][idx], [h["proj_mean_diff"]], [5.0], (kind, "proj"))
        _flags_agree(h["cm5_ok"], z["cm_ok"][idx], [h["trans_cm"], h["rot_deg"]], [5.0, 5.0], (kind, "cm"))
        for key in ("add_ok", "proj_ok", "cm5_ok"):
            assert np.array_equal(h[key], orc[key]), (kind, key)


def test_metrics_per_image_camera():
    z, groups = _fixture()
    (kind, n), idx = next(iter(groups.items()))
    X, diameter = model_points(kind, n)
    rng = np.random.default_rng(5)
    Ks = np.stack([K_LINEMOD * np.array([[rng.uniform(0.8, 1.2)] * 3] * 2 + [[1.0] * 3]) for _ in idx])
    for sym in (False, True):
        m = ev.pose_metrics(_dev(z["pose_pred"][idx]), _dev(z["pose_gt"][idx]), _dev(X), _dev(Ks), diameter,
                            sym_add=sym, sym_proj=sym)
        h = {k: v.cpu().numpy() for k, v in m.items()}
        orc = [mo.pose_metrics(z["pose_pred"][i], z["pose_gt"][i], X, Ks[j], diameter, sym_add=sym, sym_proj=sym)
               for j, i in enumerate(idx)]
        _check(h, {k: np.array([o[k] for o in orc]) for k in orc[0]}, "per-image K")


def _batch():
    z, groups = _fixture()
    (kind, n), idx = next(iter(groups.items()))
    X, diameter = model_points(kind, n)
    return _dev(z["pose_pred"][idx]), _dev(z["pose_gt"][idx]), _dev(X), z["K"], diameter


def test_metrics_deterministic():
    args = _batch()
    m1 = ev.pose_metrics(*args, sym_add=True, sym_proj=True)
    m2 = ev.pose_metrics(*args, sym_add=True, sym_proj=True)
    for k in m1:
        assert torch.equal(m1[k], m2[k]) or (k == "rot_deg" and torch.equal(m1[k].isnan(), m2[k].isnan())
                                             and torch.equal(m1[k].nan_to_num(), m2[k].nan_to_num())), k


def test_metrics_graph_capture():
    pp, pg, X, K, diameter = _batch()
    eager = ev.pose_metrics(pp, pg, X, K, diameter, sym_add=True, sym_proj=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ev.pose_metrics(pp, pg, X, K, diameter, sym_add=True, sym_proj=True)      # warm-up outside capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = ev.pose_metrics(pp, pg, X, K, diameter, sym_add=True, sym_proj=True)
    g.replay()
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(eager[k].nan_to_num(), cap[k].nan_to_num()), k


def test_device_evaluator_average_precision():
    z, groups = _fixture()
    for (kind, n), idx in groups.items():
        X, diameter = model_points(kind, n)
        for sym in (False, True):
            e = ev.DeviceEvaluator(X, diameter, z["K"], symmetric=sym)
            half = len(idx) // 2
            for part in (idx[:half], idx[half:]):
                e.evaluate_batch(_dev(z["pose_pred"][part]), _dev(z["pose_gt"][part]))
            a = "adds" if sym else "add"
            proj, add, cm = e.average_precision(verbose=False)
            assert np.allclose(e.add_dists, z[a][idx], rtol=RTOL, atol=0)
            assert np.allclose(e.proj_mean_diffs, z["proj"][idx], rtol=RTOL, atol=0)
            assert (proj, add, cm) == (np.mean(z["proj_ok"][idx]), np.mean(z[a + "_ok"][idx]),
                                      np.mean(z["cm_ok"][idx]))


def test_numpy_entry_points():
    ref, que, _ = nn_cases()["rand3"]
    idx = eu.find_nearest_point_idx(ref[0].astype(np.float64), que[0])
    assert isinstance(idx, np.ndarray) and idx.dtype == np.int32 and idx.shape == (que.shape[1],)
    assert np.array_equal(idx, mo.find_nearest_point_idx(ref[0], que[0]))
    with pytest.raises(AssertionError):
        eu.find_nearest_point_idx(ref[0], que[0, :, :2])
    z = np.load(os.path.join(GOLDEN, "pnp_cases.npz"))
    pts32 = z["points_3d"].astype(np.float32)
    names = sorted(k[:-5] for k in z.files if k.endswith("_pose"))
    for name in names:
        pose = eu.uncertainty_pnp_v2(z[name + "_kp"], z[name + "_cov"], z["points_3d"], z["K"])
        assert isinstance(pose, np.ndarray) and pose.dtype == np.float64 and pose.shape == (3, 4)
        w = eu.covariance_to_isotropic_weights(torch.from_numpy(z[name + "_cov"])).numpy()
        assert np.array_equal(w[:, 1], np.zeros(len(w))) and np.array_equal(w[:, 0], w[:, 2])
        lam = np.array([np.max(np.linalg.eigvals(c.astype(np.float64))) for c in z[name + "_cov"]])
        want = np.where(z[name + "_cov"][:, 0, 0] < 1e-5, 0.0, 1.0 / lam).astype(np.float32)
        assert np.allclose(w[:, 0], want, rtol=1e-6, atol=0), name
        ref_pose = pno.uncertainty_pnp(z[name + "_kp"], w, pts32, z["K"])
        assert np.abs(pose - ref_pose).max() < 1e-8, (name, np.abs(pose - ref_pose).max())
    # batched form: one device tensor, no host copy
    kp = _dev(np.stack([z[n + "_kp"] for n in names]))
    cov = _dev(np.stack([z[n + "_cov"] for n in names]))
    poses = eu.uncertainty_pnp_v2(kp, cov, z["points_3d"], z["K"])
    assert poses.is_cuda and poses.dtype == torch.float64 and tuple(poses.shape) == (len(names), 3, 4)
