"""Regenerates tests/golden/ref_metrics.npz by running the REFERENCE'S OWN metric methods
(lib/utils/evaluation_utils.py:54-141, Evaluator) with its own Projector (lib/utils/base_utils.py:239-294).

Runs on the CPU in the authoring container:  python tests/golden/make_golden_metrics.py REFERENCE_ROOT

evaluation_utils.py is imported unmodified.  The modules it and base_utils.py import that are not installed
here (plyfile, lmdb, transforms3d, lib.utils.config, lib.utils.data_utils, lib.datasets.linemod_dataset) are
stubbed; `find_nearest_point_idx` is served by the oracle (oracle/metrics_oracle.py, nn_oracle.c: the
reference kernel's sequence, pinned to it by tests/golden/ref_nn.npz).  The Evaluator is built without its
__init__ (which loads LINEMOD models): only the recorders and the projector are set.

Cases (poses stored; models rebuilt by tests/metrics_cases.model_points): identical poses, small
perturbations, poses placed 1e-4 relative either side of each threshold (ADD 0.1 * diameter, 2-D
projection 5 px, 5 cm, 5 degrees) and a predicted rotation whose trace with the target is below -1
(a pose half a turn off whose matrix is 1e-12 off orthonormal), which makes the angle NaN.
Ground-truth poses are float32, as the data loader yields them; predicted poses float64, as the PnP returns.

Stored: model kind and size, `pose_pred` [n,3,4] f64, `pose_gt` [n,3,4] f32, `K` [3,3] and, per case, the
recorders of add_metric, add_metric_sym, projection_2d, projection_2d_sym (value and flag) and the flag of
cm_degree_5_metric.
"""
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import metrics_oracle as mo  # noqa: E402
from tests.metrics_cases import K_LINEMOD, model_points, random_gt_pose, rotation  # noqa: E402

MODELS = {"ellipsoid": 2500, "torus": 3001}
EDGE = 1e-4


def import_reference(ref_root):
    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    for name in ("lib", "lib.utils", "lib.datasets", "lib.utils.extend_utils"):
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(ref_root, *name.split("."))]
        sys.modules[name] = m
    stub("plyfile", PlyData=None)
    stub("lmdb")
    stub("transforms3d")
    stub("transforms3d.euler", mat2euler=None)
    stub("lib.utils.config", cfg=types.SimpleNamespace())
    import lib.utils.base_utils as bu
    stub("lib.utils.data_utils", LineModModelDB=None, Projector=bu.Projector)
    stub("lib.datasets.linemod_dataset", VotingType=types.SimpleNamespace(BB8=0))
    stub("lib.utils.extend_utils.extend_utils", uncertainty_pnp=None, uncertainty_pnp_v2=None,
         find_nearest_point_idx=mo.find_nearest_point_idx)
    import lib.utils.evaluation_utils as eu
    return eu, bu


def _bisect(f, target, lo, hi, iters=200):
    """s in [lo, hi] with f(s) = target (f increasing)."""
    for _ in range(iters):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if f(mid) < target else (lo, mid)
    return 0.5 * (lo + hi)


def _pose(R, t):
    return np.concatenate([R, np.asarray(t, np.float64).reshape(3, 1)], 1)


def cases():
    rng = np.random.default_rng(2024)
    out = []      # (name, kind, pose_pred f64, pose_gt f32)
    for kind, n in MODELS.items():
        X, diameter = model_points(kind, n)
        for i in range(3):
            gt = random_gt_pose(rng)
            out.append((f"{kind}_identical_{i}", kind, gt.astype(np.float64), gt))
        for i in range(6):
            gt = random_gt_pose(rng)
            g = gt.astype(np.float64)
            dR = rotation(rng.standard_normal(3), rng.uniform(0, 0.15))
            out.append((f"{kind}_perturbed_{i}", kind, _pose(dR @ g[:, :3], g[:, 3] + rng.standard_normal(3) * 0.01),
                        gt))
        gt = random_gt_pose(rng)
        g = gt.astype(np.float64)
        u = rng.standard_normal(3)
        u /= np.linalg.norm(u)
        lateral = np.array([1.0, 0.3, 0.0]) / np.linalg.norm([1.0, 0.3, 0.0])
        ax = rng.standard_normal(3)
        for side, s in (("below", 1 - EDGE), ("above", 1 + EDGE)):
            # ADD: a pure translation moves every point by the same vector
            out.append((f"{kind}_add_{side}", kind, _pose(g[:, :3], g[:, 3] + u * 0.1 * diameter * s), gt))
            # 2-D projection: a lateral translation scaled to a mean image distance of 5 px
            proj = lambda a: mo.projection_2d(_pose(g[:, :3], g[:, 3] + a * lateral), gt, X, K_LINEMOD)[0]  # noqa
            a = _bisect(proj, 5.0 * s, 0.0, 0.05)
            out.append((f"{kind}_proj_{side}", kind, _pose(g[:, :3], g[:, 3] + a * lateral), gt))
            out.append((f"{kind}_cm_{side}", kind, _pose(g[:, :3], g[:, 3] + u * 0.05 * s), gt))
            out.append((f"{kind}_deg_{side}", kind, _pose(rotation(ax, np.deg2rad(5.0 * s)) @ g[:, :3], g[:, 3]), gt))
        # half a turn, scaled 1e-12 off orthonormal: trace(R_p R_g^T) = -1 - 1e-12 -> arccos gives NaN
        flip = rotation(ax, np.pi) * (1 + 1e-12)
        out.append((f"{kind}_trace_below_m1", kind, _pose(flip @ g[:, :3], g[:, 3]), gt))
    return out


def main():
    eu, bu = import_reference(sys.argv[1])
    ev = eu.Evaluator.__new__(eu.Evaluator)
    cs = cases()
    rec = {k: [] for k in ("add", "add_ok", "adds", "adds_ok", "proj", "proj_ok", "projs", "projs_ok", "cm_ok")}
    models = {kind: model_points(kind, n) for kind, n in MODELS.items()}
    for name, kind, pp, pg in cs:
        X, diameter = models[kind]
        for method, key, args in (("add_metric", "add", (X, diameter)), ("add_metric_sym", "adds", (X, diameter)),
                                  ("projection_2d", "proj", (X, K_LINEMOD)),
                                  ("projection_2d_sym", "projs", (X, K_LINEMOD))):
            ev.projector = bu.Projector()
            ev.add_recorder, ev.add_dists, ev.projection_2d_recorder, ev.proj_mean_diffs = [], [], [], []
            getattr(ev, method)(pp, pg, *args)
            vals, oks = (ev.add_dists, ev.add_recorder) if key.startswith("add") else \
                (ev.proj_mean_diffs, ev.projection_2d_recorder)
            rec[key].append(float(vals[0]))
            rec[key + "_ok"].append(bool(oks[0]))
        ev.cm_degree_5_recorder = []
        with np.errstate(invalid="ignore"):
            ev.cm_degree_5_metric(pp, pg)
        rec["cm_ok"].append(bool(ev.cm_degree_5_recorder[0]))
        print(f"{name:28s} add {rec['add'][-1]:.6g} adds {rec['adds'][-1]:.6g} proj {rec['proj'][-1]:.6g} "
              f"projs {rec['projs'][-1]:.6g} cm_ok {rec['cm_ok'][-1]}")
    path = os.path.join(HERE, "ref_metrics.npz")
    np.savez_compressed(path, names=np.array([c[0] for c in cs]), kinds=np.array([c[1] for c in cs]),
                        model_sizes=np.array([MODELS[c[1]] for c in cs]), pose_pred=np.stack([c[2] for c in cs]),
                        pose_gt=np.stack([c[3] for c in cs]), K=K_LINEMOD,
                        **{k: np.array(v) for k, v in rec.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
