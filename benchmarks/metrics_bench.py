"""Timing of the pose-accuracy metrics at b = 16 images per batch and pn model points (one JSON line per
measurement, each with the card's name and power limit read in the same run).

    python benchmarks/metrics_bench.py [--pn 2048 8192 16384] [--b 16] [--out FILE]

arms, per pn:
  nn_kernel          pvnet_find_nearest_point_idx alone, [b,pn,3] against [b,pn,3]: time and pairs/s
  metrics_plain      pose_metrics without symmetric forms (one launch)
  metrics_adds       pose_metrics with ADD-S (cloud launch + nearest-neighbour launch + metric launch)
  ref_nn_per_image   the reference's findNearestPointIdxLauncher (oracle/_ref/libpvnet_refnn.so) called once per
                     image on host arrays, as Evaluator.add_metric_sym does: its cudaMalloc, copies, launch,
                     blocking copy back and cudaFree included (host clock; the call ends synchronised)
  host_numpy_plain   the reference's numpy add_metric + projection_2d + cm_degree_5_metric, per image
  host_numpy_adds    the same with add_metric_sym, its search on the reference launcher, per image
Device arms: CUDA events around `iters` back-to-back calls after `warmup` calls of the same shape.  The inputs
(at most 3 MB) stay in L2 between calls.  Host arms: time.perf_counter over the b images of one batch.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import metrics_oracle as mo  # noqa: E402
from oracle import ref_nn  # noqa: E402
from pvnet_b200 import evaluation as ev  # noqa: E402
from pvnet_b200 import extend_utils as eu  # noqa: E402

K = np.array([[572.4114, 0., 325.2611], [0., 573.57043, 242.04899], [0., 0., 1.]])


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in q.split(","))
    return {"gpu": name, "power_limit": power}


def device_ms(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def inputs(b, pn, seed=0):
    rng = np.random.default_rng(seed)
    i = np.arange(pn) + 0.5
    u, v = np.arccos(1 - 2 * i / pn), np.pi * (1 + 5 ** 0.5) * i
    X = np.stack([0.06 * np.sin(u) * np.cos(v), 0.04 * np.sin(u) * np.sin(v), 0.03 * np.cos(u)], 1).astype(np.float32)
    gt, pred = [], []
    for _ in range(b):
        a = rng.standard_normal(3)
        a *= rng.uniform(0, np.pi) / np.linalg.norm(a)
        R = _rodrigues(a)
        t = np.array([rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1), rng.uniform(0.7, 1.2)])
        gt.append(np.concatenate([R, t[:, None]], 1).astype(np.float32))
        d = rng.standard_normal(3) * 0.05
        pred.append(np.concatenate([_rodrigues(d) @ R, (t + rng.standard_normal(3) * 0.01)[:, None]], 1))
    return X, np.stack(pred), np.stack(gt)


def _rodrigues(r):
    th = np.linalg.norm(r)
    k = r / th
    kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * kx + (1 - np.cos(th)) * kx @ kx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pn", type=int, nargs="+", default=[2048, 8192, 16384])
    ap.add_argument("--b", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_bench needs a CUDA device")
    info = card()
    dev = "cuda:0"
    lines = []

    def emit(d):
        d = {**info, "b": a.b, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    for pn in a.pn:
        X, pred, gt = inputs(a.b, pn)
        Xd, pd, gd = (torch.from_numpy(v).to(dev) for v in (X, pred, gt))
        cloud = torch.from_numpy(np.einsum("nk,bjk->bnj", X, gt[:, :, :3]) + gt[:, None, :, 3]).float().to(dev)
        cloud_p = torch.from_numpy(np.einsum("nk,bjk->bnj", X, pred[:, :, :3]) + pred[:, None, :, 3]).float().to(dev)
        ms = device_ms(lambda: eu.find_nearest_point_idx_batched(cloud_p, cloud), a.warmup, a.iters)
        emit({"arm": "nn_kernel", "pn": pn, "ms": ms, "pairs_per_s": a.b * pn * pn / (ms * 1e-3)})
        for sym in (False, True):
            ms = device_ms(lambda: ev.pose_metrics(pd, gd, Xd, K, 0.12, sym_add=sym), a.warmup, a.iters)
            emit({"arm": "metrics_adds" if sym else "metrics_plain", "pn": pn, "ms": ms})
        if ref_nn.available():
            cp, cg = cloud_p.cpu().numpy(), cloud.cpu().numpy()
            ref_nn.find_nearest_point_idx(cp[0], cg[0])
            t0 = time.perf_counter()
            for i in range(a.b):
                ref_nn.find_nearest_point_idx(cp[i], cg[i])
            emit({"arm": "ref_nn_per_image", "pn": pn, "ms": (time.perf_counter() - t0) * 1e3})
        t0 = time.perf_counter()
        for i in range(a.b):
            mo.add_metric(pred[i], gt[i], X, 0.12)
            mo.projection_2d(pred[i], gt[i], X, K)
            mo.cm_degree_5_metric(pred[i], gt[i])
        emit({"arm": "host_numpy_plain", "pn": pn, "ms": (time.perf_counter() - t0) * 1e3})
        if ref_nn.available():
            t0 = time.perf_counter()
            for i in range(a.b):
                mp = np.dot(X, pred[i][:, :3].T) + pred[i][:, 3]
                mt = np.dot(X, gt[i][:, :3].T) + gt[i][:, 3]
                idx = ref_nn.find_nearest_point_idx(mp, mt)
                np.mean(np.linalg.norm(mp[idx] - mt, 2, 1))
                mo.projection_2d(pred[i], gt[i], X, K)
                mo.cm_degree_5_metric(pred[i], gt[i])
            emit({"arm": "host_numpy_adds", "pn": pn, "ms": (time.perf_counter() - t0) * 1e3})
        # the device result equals the reference launcher's on the timed inputs
        if ref_nn.available():
            got = eu.find_nearest_point_idx_batched(cloud_p, cloud).cpu().numpy()
            want = ref_nn.find_nearest_point_idx_batched(cloud_p.cpu().numpy(), cloud.cpu().numpy())
            emit({"arm": "check_nn_equals_reference", "pn": pn, "equal": bool(np.array_equal(got, want))})
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
