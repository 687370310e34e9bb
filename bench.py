#!/usr/bin/env python
"""bench.py -- PVNet per-image inference hot path on B200: images/sec (480x640, K=9),
backbone (Resnet18_8s) + RANSAC vote (ransac_voting_layer_v3).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (rank 0)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --config 4 | --config 5                  # another BASELINE config as the headline
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs to DIR/*.npy

One "step" = one batch of 16 synthetic 480x640 images per GPU (BASELINE config 2, the headline at
every N so that the per-GPU work is fixed -- "weak" scaling):
Resnet18_8s(ver_dim=18, seg_dim=2).eval() forward -> per-pixel argmax (fused into the head)
-> ransac_voting_layer_v3(mask, vertex, 256, inlier_thresh=0.99).  Weights are random-init
(reference init scheme, seeded) with the segmentation bias calibrated so that about 20000
pixels per image come out as foreground (config 2's mask size); inputs are N(0,1) images.

The same JSON line also carries `config4`: BASELINE config 4's per-GPU workload (config 2 +
estimate_voting_distribution_with_mean(256, 4096), the 8-GPU config) measured the same two ways in
the same process at the same N, so a 1/2/4/8 run yields config 4's scaling as well.
`--config 5`: K=17, ~92160 foreground px, v3(1024, max_num=30000) + with_mean(1024, 1024), batch 4/GPU.

Prints ONE JSON line (rank 0).  `value` = device-resident inputs; `e2e` = the same step
through the public API (PoseKeypointPipeline) from pinned HOST buffers -- raw uint8 HWC images,
normalised on the device -- with the H2D of the image batch and the D2H of the keypoints (and
covariances) inside the timed region.  Also: `roofline` of the dominant kernel (the tcgen05
convolutions, timed per layer with CUDA events inside this process), `roofline_vote` (the voting
layer timed in place: tests/s, FP32-issue fraction, algorithmic HBM GB/s), `cpu_baseline` (the same
workload on the host cores: the reference graph under torch CPU + the oracle port of the voting
kernels, bounded sample), `clocks`, `gpu_launches`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W, K_KP, HYP, BATCH = 480, 640, 9, 256, 16
THRESH = 0.99
VOTE_ISSUE_SLOTS_PER_TEST = 5.0   # k_vote3's sweep in SASS: 160 instructions per 32 tests = 2 FFMA2 + FADD + LEA.HI + 1/2 FMNMX3
#                                   per test + 12 LDS.128 + 4 loop instructions; also its FMA-pipe cycles (FFMA2 = 2)
VOTE_MICRO_CYCLES_PER_TEST = 7.17  # that mix alone, in registers, at the kernel's 4 resident warps per sub-partition
#                                    (profiles/r02_micro_vote_mix.txt row 16; 6.32 at 6 warps): what the SM sustains

# BASELINE.json configs that bench.py can run as the headline (per-GPU batch: weak scaling)
CONFIGS = {
    2: dict(k=9, hyp=256, batch=16, fg=20000, cov=None, max_num=30000,
            name="BASELINE config 2: Resnet18_8s(18,2) forward + argmax + ransac_voting_layer_v3(256 hyp, thresh 0.99), "
                 "batch 16 per GPU, 480x640, K=9"),
    4: dict(k=9, hyp=256, batch=16, fg=20000, cov=(256, 4096), max_num=30000,
            name="BASELINE config 4 (per-GPU part): config 2 + estimate_voting_distribution_with_mean(256, 4096), "
                 "batch 16 per GPU"),
    5: dict(k=17, hyp=1024, batch=4, fg=92160, cov=(1024, 1024), max_num=30000,
            name="BASELINE config 5 (per-GPU part): Resnet18_8s(34,2) + v3(1024 hyp, max_num 30000) + "
                 "with_mean(1024, 1024), K=17, ~30 % foreground, batch 4 per GPU (32 on 8 GPUs)"),
}
GFLOP_PER_IMAGE = 144.87          # SURVEY.md App. B (26 convs, 72.44 GMAC)
TARGET_FG = 20000


def _host_cores():
    """Host threads this process may really use: CPU affinity capped by the cgroup CPU quota
    (os.cpu_count() counts the box, not the container; oversubscribing made the CPU arm 4-40x slower)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, min(n, 64))


def _rank_world():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._reader, daemon=True).start()
        except Exception:
            self.proc = None

    def _reader(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- model
def build_model(torch, dev, k=K_KP):
    from pvnet_b200.model_repository import Resnet18_8s
    torch.manual_seed(0)
    net = Resnet18_8s(ver_dim=2 * k, seg_dim=2)
    g = torch.Generator().manual_seed(0)
    for m in net.modules():                  # exercise BN folding (SURVEY.md §8d)
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
    return net.to(dev).eval()


def calibrate_foreground(torch, net, x, target_fg=TARGET_FG):
    """Shift the class-1 logit bias so that ~target_fg pixels per image are foreground."""
    with torch.no_grad():
        out = net.forward_native(x[:4])
        margin = (out[:, 1] - out[:, 0]).flatten()
        kth = margin.numel() - target_fg * x[:4].shape[0]
        cut = torch.kthvalue(margin.float().cpu(), max(1, kth)).values.item()
        net.convraw[3].bias[1] -= cut
        _, mask = net.forward_native(x, with_mask=True)
        return float(mask.float().sum().item() / x.shape[0])


def make_pipe(net, cfg):
    """The public end-to-end object (pvnet_b200/pipeline.py); its .step is the device-resident step."""
    from pvnet_b200.pipeline import PoseKeypointPipeline
    cov = cfg["cov"]
    return PoseKeypointPipeline(net, round_hyp_num=cfg["hyp"], inlier_thresh=THRESH, rng="device",
                                with_covariance=cov is not None, cov_round_hyp_num=cov[0] if cov else 256,
                                cov_min_hyp_num=cov[1] if cov else 4096, max_num=cfg["max_num"])


def make_step(torch, net, with_cov=False):
    """Device-resident step of config 2 (or 4 with with_cov); used by benchmarks/*.py too."""
    pipe = make_pipe(net, CONFIGS[4 if with_cov else 2])

    def step(x):
        r = pipe.step(x)
        return r[0] if isinstance(r, tuple) else r
    return step


# ----------------------------------------------------------------------------- roofline
def _ncu_traffic():
    """DRAM bytes (read+write) of the conv launches of one step from the committed ncu --set full
    capture; NOT measured in this run (the profiler cannot run inside the timed process)."""
    for name in ("r02_conv_dram_traffic.json", "r01_conv_dram_traffic.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            return {"dram_bytes_per_step": d["bytes_per_step"], "source": d["source"], "measured": False,
                    "note": f"constant read from profiles/{name} (one ncu --set full capture of the same step), "
                            "not re-measured by this run"}
        except Exception:
            continue
    return None


def conv_roofline(torch, net, x, peaks, k=K_KP):
    """Per-stage device time of one forward pass, CUDA events recorded on the launch stream
    between the single-kernel stages; aggregates the tcgen05 convolution launches."""
    import ctypes

    from pvnet_b200 import _native
    L = _native.lib()
    dev = x.device
    b = x.shape[0]
    handle = net._prepare_native(dev)
    n = ctypes.c_size_t()
    L.pvnet_backbone_workspace_bytes(handle, b, H, W, ctypes.byref(n))
    ws = net._workspace(n.value, dev)
    out = torch.empty([b, 2 + 2 * k, H, W], dtype=torch.float32, device=dev)
    mask = torch.empty([b, H, W], dtype=torch.uint8, device=dev)
    ns = L.pvnet_backbone_num_stages()
    names = [L.pvnet_backbone_stage_name(i).decode() for i in range(ns)]
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    # 5 untimed forwards, then 20 timed ones enqueued back to back (one synchronize at the end, so the
    # GPU stays as busy -- and as power-capped -- as in the timed loop); per-stage median over the reps
    warm, reps = 5, 20
    evs = []
    for rep in range(warm + reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(ns + 1)] if rep >= warm else None
        if ev:
            ev[0].record()
        for i in range(ns):
            _native.check(L.pvnet_backbone_run_stage(handle, i, x.data_ptr(), b, H, W, out.data_ptr(), mask.data_ptr(),
                                                     1, ws.data_ptr(), ws.numel(), stream), "run_stage")
            if ev:
                ev[i + 1].record()
        if ev:
            evs.append(ev)
    torch.cuda.synchronize()
    ms = np.median(np.array([[ev[i].elapsed_time(ev[i + 1]) for i in range(ns)] for ev in evs]), axis=0)
    is_conv = np.array([("layer" in nm or nm.startswith("fc") or nm.startswith("conv") or nm.startswith("stem"))
                        and "head" not in nm for nm in names])
    conv_ms = float(ms[is_conv].sum())
    backbone_ms = float(ms.sum())
    gflop_img = GFLOP_PER_IMAGE + 0.039 * (k - K_KP)               # SURVEY App. B: +0.039 GFLOP per extra keypoint
    flops = gflop_img * 1e9 * b
    achieved = flops / (conv_ms * 1e-3) / 1e12
    bf16 = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1590.0
    peak = bf16 / 2.0
    stages = [{"stage": nm, "ms": round(float(t), 4)} for nm, t in zip(names, ms)]
    return {
        "bound": "tensor", "kernel": "k_conv_tap_p + k_conv_col (tcgen05.mma kind::tf32; every conv of the network incl. "
                                     "stem and fused 1x1 head)",
        "achieved": round(achieved, 2), "peak": round(peak, 1), "unit": "TFLOP/s", "frac": round(achieved / peak, 4),
        "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained / 2 (tcgen05 tf32 = half the bf16 rate)"
                        if "bf16_tflops_sustained" in peaks else "fallback 1590/2"),
        "algorithmic_gflop_per_launch_set": round(flops / 1e9, 1), "conv_ms_per_step": round(conv_ms, 3),
        "backbone_ms_per_step": round(backbone_ms, 3),
        "frac_whole_backbone": round(flops / (backbone_ms * 1e-3) / 1e12 / peak, 4),
        "traffic": _ncu_traffic(),
    }, stages


def vote_roofline(torch, pipe, x, peaks, clocks, cfg):
    """The voting layer timed in place (CUDA events around the public call on the launch stream, 20
    back-to-back repetitions after 5 warm ones, median): inlier tests per second, the fraction of the
    FP32-issue roof (tests x instructions per test / (SMs x 128 lanes x clock)) and the algorithmic
    HBM rate B_alg / t against the measured copy bandwidth (SURVEY.md section 8d)."""
    from pvnet_b200 import ransac_voting_gpu as rv
    net = pipe.net
    out, mask = net.forward_native(x, with_mask=True, mask_dtype=torch.uint8, pixel_major=True)     # as pipe.step does
    b, h, w, c = out.shape
    k = (c - 2) // 2
    vertex = out[..., 2:].unflatten(3, (k, 2))
    cov = cfg["cov"]
    hn = cfg["hyp"]
    hnt = 0 if cov is None else cov[0] * -(-cov[1] // cov[0])

    def call():
        return rv.ransac_voting_pipeline(mask, vertex, hn, THRESH, cov is not None, cov[0] if cov else 256,
                                         cov[1] if cov else 4096, THRESH, max_num=cfg["max_num"], rng="device")
    _, dbg = rv.ransac_voting_pipeline(mask, vertex, hn, THRESH, False, max_num=cfg["max_num"], rng="device",
                                       return_debug=True)
    tn = dbg["tn"].cpu().numpy().astype(np.int64)
    for _ in range(5):
        call()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
    for e0, e1 in evs:
        e0.record()
        call()
        e1.record()
    torch.cuda.synchronize()
    ms = float(np.median([e0.elapsed_time(e1) for e0, e1 in evs]))
    tests = float(tn.sum()) * k * (hn + hnt + 1)                    # +1: the winner's vote of the refit
    clk = ((clocks or {}).get("sm_mhz") or 1900.0) * 1e6
    sms = torch.cuda.get_device_properties(x.device).multi_processor_count
    issue_roof = sms * 128 * clk / VOTE_ISSUE_SLOTS_PER_TEST
    micro_roof = sms * 128 * clk / VOTE_MICRO_CYCLES_PER_TEST
    b_alg = b * (h * w * 1 + k * 24 + (hn + hnt) * k * 8) + float(tn.sum()) * k * 8
    hbm = peaks.get("hbm_gbs") or 6575.0
    return {
        "kernel": "k_vote3 inside pvnet_ransac_voting_pipeline (whole layer timed: compaction, gather, hypotheses, "
                  "vote, refit" + (", covariance)" if cov else ")"),
        "layer_ms": round(ms, 4), "tests": int(tests), "tests_per_s": round(tests / (ms * 1e-3), 1),
        "issue_slots_per_test": VOTE_ISSUE_SLOTS_PER_TEST, "micro_cycles_per_32_tests": VOTE_MICRO_CYCLES_PER_TEST,
        "sm_clock_mhz": round(clk / 1e6, 1),
        "issue_frac": round(tests / (ms * 1e-3) / issue_roof, 4),
        "micro_frac": round(tests / (ms * 1e-3) / micro_roof, 4), "bound": "fp32 issue",
        "alg_bytes": int(b_alg), "alg_hbm_gbs": round(b_alg / (ms * 1e-3) / 1e9, 2),
        "alg_hbm_frac": round(b_alg / (ms * 1e-3) / 1e9 / hbm, 5), "hbm_peak_gbs": hbm,
        "fg_px_per_image": round(float(tn.mean()), 1),
        "note": "whole layer timed (10 launches); FP32-issue bound by construction (SURVEY 8d): the [hn,K,tn] inlier tensor the "
                "reference streams through HBM never exists here; issue_frac = tests/s over SMs x 128 lanes x clock / 5.0 slots, "
                "micro_frac = over what the instruction mix alone sustains in a register-only microbenchmark at the same "
                "occupancy; the kernel's own ncu DRAM bytes (1.00x its algorithmic bytes) are in profiles/r02_ncu_vote.md",
    }


# ----------------------------------------------------------------------------- cpu side
def _cpu_path():
    """The whole path on the HOST cores, one image per call: the reference network graph (our
    nn.Module is the reference graph on the CPU, tests/test_backbone_cpu.py) in eval mode under
    torch CPU + the oracle port of the voting kernels (the reference has no CPU voting code: its
    extension is CUDA only).  Returns (step function, threads used)."""
    import torch

    from oracle import pvnet_oracle as po
    from pvnet_b200 import synthetic as syn
    from pvnet_b200.model_repository import Resnet18_8s
    ncpu = _host_cores()
    torch.set_num_threads(ncpu)          # torchrun exports OMP_NUM_THREADS=1; this leg may use every host core
    po.set_num_threads(ncpu)
    torch.manual_seed(0)
    net = Resnet18_8s(2 * K_KP, 2).eval()
    x = torch.from_numpy(syn.backbone_input(1, 0))
    mask = syn.disc_mask(TARGET_FG)
    idxs = [syn.draw_idxs(TARGET_FG, HYP, K_KP, seed=0)]

    def step():
        with torch.no_grad():
            seg, ver = net._forward_torch(x)
        vertex = ver.permute(0, 2, 3, 1).reshape(1, H, W, K_KP, 2).numpy()
        # vote on a 20000-px disc (random-init logits have no object), same sizes as the GPU arm
        return po.ransac_voting_layer_v3(mask[None], vertex, HYP, inlier_thresh=THRESH, idxs=idxs)
    return step, po.num_threads()


def cpu_path_baseline(seconds_budget=20.0, max_images=16):
    """`cpu_baseline` of the GPU arm: bounded sample of the same workload on the host cores."""
    step, cores = _cpu_path()
    step()                                                                   # warm
    n, t0 = 0, time.perf_counter()
    while n < 2 or (time.perf_counter() - t0 < seconds_budget and n < max_images):
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": round(n / dt, 3), "unit": "images/sec", "cores": cores, "kind": "port",
            "sample": f"{n} images x (Resnet18_8s(18,2) eval forward under torch CPU + ransac_voting_layer_v3 of "
                      f"20000 fg px, K=9, 256 hyp by oracle/pvnet_oracle.c with OpenMP)"}


def run_reference_arm(args):
    """--impl reference: the reference's path on the HOST cores.  The reference has no CPU
    voting code of its own (its extension is CUDA only), so this arm is: the reference
    network graph (our nn.Module is bit-identical to the reference classes on the CPU, see
    tests/test_backbone_cpu.py) in eval mode under torch CPU + the oracle port of the voting
    kernels, all host threads.  Bounded sample: 1 image per step."""
    rank, world, _ = _rank_world()
    if rank != 0:
        return
    step, cores = _cpu_path()
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        kp = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"keypoints": kp})
    val = steps / dt
    line = {
        "impl": "reference", "metric": "images/sec (480x640, K=9) backbone+vote", "value": round(val, 4),
        "unit": "images/sec", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": round(dt / steps * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE config 2 shape, 1 image/step on the host: Resnet18_8s(18,2) eval forward "
                               "(torch CPU, reference graph) + ransac_voting_layer_v3(256 hyp, thresh 0.99, 20000 fg px)"},
        "cpu_baseline": {"value": round(val, 4), "unit": "images/sec", "cores": cores, "kind": "port",
                         "sample": f"{steps} steps x 1 image"},
        "e2e": {"value": round(val, 4), "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- main
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dst, arrays):
    """Writes each array as dst/<name>.npy in float32 (float64 stays float64), so that two builds run with
    the same arguments -- hence the same inputs -- can be compared output for output."""
    os.makedirs(dst, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        out[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    for name, a in out.items():
        np.save(os.path.join(dst, name + ".npy"), a)


def measure(torch, dist, pd, pipe, xs, hosts, batch, k, steps, warmup, world, sampler=None, rank=0):
    """One configuration, two ways: K steps on device-resident inputs, and the same K steps through
    PoseKeypointPipeline.run from pinned host buffers.  Returns per-rank (ms_device, ms_e2e, launches,
    clocks or None, outputs): outputs = what the last step of each timed loop returned, by name."""
    from pvnet_b200 import _native
    with_cov = pipe.with_cov

    def gather(r):
        if world > 1:                                   # pose inputs to every rank (SURVEY.md section 8e)
            if isinstance(r, tuple):
                pd.gather_results(r[0], batch * world)
                pd.gather_results(r[1], batch * world)
            else:
                pd.gather_results(r, batch * world)

    def full_step(x):
        r = pipe.step(x)
        gather(r)
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for i in range(warmup):
            full_step(xs[i % 3])
        barrier()
        if sampler is not None and rank == 0:
            sampler.start()
        for i in range(30 if sampler is not None else 5):   # ~0.3 s of the same load on every rank so that
            full_step(xs[i % 3])                             # nvidia-smi's 100 ms sampling sees clocks under load
        barrier()
        _native.launch_count_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            r = full_step(xs[i % 3])
        e1.record()
        barrier()
        launches = _native.launch_count()
        ms_dev = e0.elapsed_time(e1)
        outputs = {"keypoints": r[0].cpu(), "covariance": r[1].cpu()} if with_cov else {"keypoints": r.cpu()}

        kp_hosts = [torch.empty([batch, k, 2]).pin_memory() for _ in range(steps)]
        cov_hosts = [torch.empty([batch, k, 2, 2]).pin_memory() for _ in range(steps)] if with_cov else None

        def hook(i, r):
            gather(r)
        pipe.run([hosts[i % 3] for i in range(3)], out_host=kp_hosts[:3], cov_host=cov_hosts[:3] if with_cov else None,
                 on_result=hook)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        pipe.run([hosts[i % 3] for i in range(steps)], out_host=kp_hosts, cov_host=cov_hosts, on_result=hook)
        f1.record()
        barrier()
        ms_e2e = f0.elapsed_time(f1)
        clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    outputs["e2e_keypoints"] = kp_hosts[-1]
    if with_cov:
        outputs["e2e_covariance"] = cov_hosts[-1]
    return ms_dev, ms_e2e, launches, clocks, outputs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                    help="BASELINE config run as the headline (default 2; the line always carries config 4 too)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--with-cov", action="store_true", help="same as --config 4")
    ap.add_argument("--e2e-input", default="u8", choices=["u8", "f32"],
                    help="host buffers of the e2e arm: raw uint8 HWC images normalised on the device, or float32 NCHW")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step returned as DIR/<name>.npy (rank 0): "
                         "keypoints (and covariance) of the device-resident arm, e2e_* of the end-to-end arm, "
                         "config4_* for config 4's measurement in the same line")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.with_cov:
        args.config = 4
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    from pvnet_b200 import _native
    from pvnet_b200 import distributed as pd
    from pvnet_b200 import synthetic as syn
    from pvnet_b200.pipeline import IMAGENET_MEAN, IMAGENET_STD

    rank, world, local = _rank_world()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: pvnet_b200 has no CPU path")
    _native.lib()                                    # fail loudly if the extension is missing
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = CONFIGS[args.config]
    k, batch = cfg["k"], cfg["batch"]
    net = build_model(torch, dev, k)
    # 3 rotating input batches (3 x 59 MB of activations-in > 126 MB L2); different per rank.  Raw uint8 HWC
    # images on the host (what a decoder yields); the device-resident arm gets the same images already
    # normalised to float32 NCHW (ToTensor + Normalize, tools/demo.py:89-95).
    rng = np.random.default_rng(1000 * args.config + 17 * rank)
    hosts_u8 = [torch.from_numpy(rng.integers(0, 256, (batch, H, W, 3), dtype=np.uint8)).pin_memory() for _ in range(3)]
    mean = torch.tensor(IMAGENET_MEAN, device=dev).view(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD, device=dev).view(1, 3, 1, 1)
    xs = [((h8.to(dev).permute(0, 3, 1, 2).float() / 255.0 - mean) / std).contiguous() for h8 in hosts_u8]
    hosts = hosts_u8 if args.e2e_input == "u8" else [x.cpu().pin_memory() for x in xs]
    torch.cuda.synchronize()
    fg = calibrate_foreground(torch, net, xs[0], cfg["fg"])

    pipe = make_pipe(net, cfg)
    ms_total, ms_e2e, launches, clocks, outputs = measure(torch, dist, pd, pipe, xs, hosts, batch, k, args.steps,
                                                          args.warmup, world, ClockSampler(local), rank)
    extra = None
    if args.config == 2:                             # config 4's per-GPU workload in the same process, same N
        pipe4 = make_pipe(net, CONFIGS[4])
        extra = measure(torch, dist, pd, pipe4, xs, hosts, batch, k, args.steps, args.warmup, world)
        outputs.update({"config4_" + name: a for name, a in extra[4].items()})
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)

    vals = [ms_total, ms_e2e] + ([extra[0], extra[1]] if extra else [0.0, 0.0])
    t = torch.tensor(vals, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms4, ms4_e2e = t.tolist()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        with torch.no_grad():
            roofline, stages = conv_roofline(torch, net, xs[0], peaks, k)
            vote_rf = vote_roofline(torch, pipe, xs[0], peaks, clocks, cfg)
        images = batch * world * args.steps
        in_bytes = int(hosts[0].numel() * hosts[0].element_size())

        def d2h(with_cov):
            return int(batch * k * 2 * 4 * (3 if with_cov else 1))
        line = {
            "metric": "images/sec (480x640, K=%d) backbone+vote%s" % (k, "+covariance" if cfg["cov"] else ""),
            "value": round(images / (ms_total * 1e-3), 2), "unit": "images/sec",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_total / args.steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "tf32 (fp32 storage, fp32 accumulate; vote fp32/fp64)", "data": "synthetic",
            "config": {"workload": cfg["name"],
                       "global_batch": batch * world, "parallelism": f"batch-sharded dp{world}",
                       "fg_px_per_image": round(fg, 1), "rng": "device (in-kernel Philox)",
                       "weights": "random-init, BN stats randomised",
                       "e2e_input": ("uint8 HWC images, normalised on the device" if args.e2e_input == "u8"
                                     else "float32 NCHW"),
                       "l2": "3 rotating input batches and a ~3.7 GB activation working set per step, both > 126 MB L2"},
            "e2e": {"value": round(images / (ms_e2e * 1e-3), 2), "unit": "images/sec",
                    "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": d2h(cfg["cov"] is not None)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "roofline_vote": vote_rf,
            "stages_ms": stages,
        }
        if extra:
            with torch.no_grad():
                vote4 = vote_roofline(torch, pipe4, xs[0], peaks, clocks, CONFIGS[4])
            line["config4"] = {
                "workload": CONFIGS[4]["name"], "value": round(images / (ms4 * 1e-3), 2), "unit": "images/sec",
                "ms_per_step": round(ms4 / args.steps, 4), "per_gpu": round(images / (ms4 * 1e-3) / world, 2),
                "e2e": {"value": round(images / (ms4_e2e * 1e-3), 2), "unit": "images/sec",
                        "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": d2h(True)},
                "gpu_launches": int(extra[2]), "roofline_vote": vote4,
            }
        if not args.no_cpu_baseline and world == 1:        # the host-core baseline is an N=1 figure
            try:
                line["cpu_baseline"] = cpu_path_baseline()
            except Exception as e:          # the checker being unavailable must not hide the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "images/sec", "cores": 0, "kind": "port",
                                        "sample": f"unavailable: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
