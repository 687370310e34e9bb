"""Inputs of the nearest-neighbour and pose-metric fixtures (tests/golden/ref_nn.npz, ref_metrics.npz), rebuilt
from seeds by the generators and by the tests alike."""
import numpy as np

# the reference's Projector.intrinsic_matrix['linemod'] (lib/utils/base_utils.py:241-243)
K_LINEMOD = np.array([[572.4114, 0., 325.2611], [0., 573.57043, 242.04899], [0., 0., 1.]])


def _grid_ties(dim, rng):
    """Integer grid references (with duplicates) and queries at cell centres: every query has 2**dim nearest
    points at exactly the same distance, and duplicated points tie at distance 0."""
    g = np.stack(np.meshgrid(*[np.arange(6)] * dim, indexing="ij"), -1).reshape(-1, dim).astype(np.float32)
    ref = np.concatenate([g, g[rng.integers(0, len(g), 50)]])[rng.permutation(len(g) + 50)]
    centres = (g[rng.integers(0, len(g), 200)] + 0.5).astype(np.float32)
    que = np.concatenate([centres, ref[:100]])
    return ref, que


def nn_cases():
    """name -> (ref [b,pn1,d] f32, que [b,pn2,d] f32, exclude_self)."""
    out = {}
    rng = np.random.default_rng(1234)
    for d in (2, 3):
        out[f"rand{d}"] = (rng.standard_normal((1, 1000, d)).astype(np.float32),
                           rng.standard_normal((1, 777, d)).astype(np.float32), 0)
        # pn not a multiple of any tile (1024, 128, 32), b > 1, with and without exclude_self
        pts = (rng.standard_normal((3, 1037, d)) * 0.1).astype(np.float32)
        out[f"b3_{d}"] = (pts, (pts + rng.standard_normal(pts.shape) * 1e-3).astype(np.float32), 0)
        out[f"b3_self_{d}"] = (pts, pts, 1)
        out[f"b2_self_uneven_{d}"] = (pts[:2, :1037], pts[:2, :2053 // 2], 1)
        ref, que = _grid_ties(d, rng)
        out[f"ties_{d}"] = (ref[None], que[None], 0)
        out[f"ties_self_{d}"] = (ref[None], ref[None], 1)
        # squared distances that overflow to +inf: only the near cluster is finite for the first queries,
        # nothing is for the far queries (index 0)
        big = np.concatenate([rng.standard_normal((300, d)) * 1e19, rng.standard_normal((40, d))]).astype(np.float32)
        q = np.concatenate([rng.standard_normal((30, d)), rng.standard_normal((30, d)) * 3e19 + 2e20,
                            np.full((5, d), 3e38)]).astype(np.float32)
        out[f"overflow_{d}"] = (big[None], q[None], 0)
        # NaN coordinates in references and queries
        r = rng.standard_normal((500, d)).astype(np.float32)
        r[rng.random(r.shape) < 0.05] = np.nan
        r[:3] = np.nan
        q = rng.standard_normal((200, d)).astype(np.float32)
        q[rng.random(q.shape) < 0.05] = np.nan
        out[f"nan_{d}"] = (r[None], q[None], 0)
    return out


def large_nn_case(seed, b, pn1, pn2, dim):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((b, pn1, dim)) * 0.1).astype(np.float32), \
        (rng.standard_normal((b, pn2, dim)) * 0.1).astype(np.float32)


def model_points(kind, n):
    """A closed surface at LINEMOD scale (metres), float32 [n,3]: an ellipsoid (diameter 0.12) or a torus
    (diameter 0.2), sampled on a Fibonacci lattice so the points are spread evenly."""
    i = np.arange(n) + 0.5
    u = np.arccos(1 - 2 * i / n)
    v = np.pi * (1 + 5 ** 0.5) * i
    if kind == "ellipsoid":
        p = np.stack([0.06 * np.sin(u) * np.cos(v), 0.04 * np.sin(u) * np.sin(v), 0.03 * np.cos(u)], 1)
        return p.astype(np.float32), 0.12
    a, r = 0.07, 0.03
    th, ph = 2 * np.pi * i / n * 37, 2 * np.pi * i / n
    p = np.stack([(a + r * np.cos(th)) * np.cos(ph), (a + r * np.cos(th)) * np.sin(ph), r * np.sin(th)], 1)
    return p.astype(np.float32), 2 * (a + r)


def rotation(axis, angle):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    k = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * k + (1 - np.cos(angle)) * k @ k


def random_gt_pose(rng):
    R = rotation(rng.standard_normal(3), rng.uniform(0, np.pi))
    t = np.array([rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1), rng.uniform(0.7, 1.2)])
    return np.concatenate([R, t[:, None]], 1).astype(np.float32)
