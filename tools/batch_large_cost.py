"""Cost of the cluster update of the batched filters (ekf_batch_create_large, capacity 100: n = 614, a cluster of 3 CTAs).

A single filter with capacity 128 runs through a cfg3-like scene (bench.make_scene's camera and motion, 640 x 480) holding 100
features; before every step a batch of B filters (1024 and 4096) is seeded from it (one kernel) and given the same perturbed
camera states, so every step does the same work.  Per step: predict, match and update milliseconds from the step's CUDA events
(ekf_batch_last_step_ms), and filter-steps/s from a host clock around the step call (which ends in a device synchronise).

The update class's FP64 rate is computed from shapes: every stacked update of a filter (Li, then Hi, as the step's counters
report them) runs as blocks of at most 32 features (k = 2 m rows); per block 2 n^2 k for the downdate Sigma -= V V^T plus
2 n k nd (nd = 13 for inverse-depth features) for the gather W = Sigma H^T.  The DGEMM rate of tools/dgemm_probe.py (torch's
cuBLAS, n = 8192) is measured in the same call, with the card's name and power limit.

    python tools/batch_large_cost.py [--filters 1024 4096] [--steps 10] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402  (camera, motion and configuration of the cfg3 workload)
import ekfb200  # noqa: E402
from batch_xyz_cost import card  # noqa: E402

NFEAT, CAP = 100, 100


def update_flops(n, k_li, k_hi, nd=13):
    """FP64 operations of one filter's updates from shapes: blocks of <= 32 features."""
    tot = 0.0
    for m_all in (k_li, k_hi):
        for a0 in range(0, m_all, 32):
            k = 2 * min(32, m_all - a0)
            tot += 2.0 * n * n * k + 2.0 * n * k * nd
    return tot


def dgemm_tflops(n=8192):
    import torch
    a = torch.randn(n, n, dtype=torch.float64, device="cuda"); b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); a @ b; e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2 * n ** 3 / best / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, nargs="+", default=[1024, 4096])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = ekfb200.load_package()
    pkg.lib()
    name, limit = card()
    lines = [json.dumps({"card": name, "power.limit, clocks.max.sm": limit})]
    print(lines[0], flush=True)

    def emit(d):
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)

    emit({"probe": "cublas_dgemm", "n": 8192, "tflops": round(dgemm_tflops(), 2)})
    nfr = args.warmup + args.steps + 1
    scene = pkg.synth.Scene(n_features=NFEAT, width=640, height=480, n_frames=nfr, seed=1235, speed=0.1, omega=0.02,
                            accel_sigma=0.002, border=44, depth_range=bench.BENCH_DEPTH_RANGE)
    cfg = bench.bench_config(pkg, scene)
    g = pkg.VSlamFilter(cfg, feature_capacity=128)
    g.captureNewFrame(scene.frame(0), scene.stamps[0])
    for p in scene.feature_pixels:
        g.addFeature(*p)
    for B in args.filters:
        batch = pkg.FilterBatch(cfg, B, feature_capacity=CAP, large=True)
        ctas, resident = batch.update_clusters()
        rng = np.random.default_rng(B)
        ms, wall, flops, lis, his = [], [], [], [], []
        src = pkg.VSlamFilter(cfg, feature_capacity=128)
        src.captureNewFrame(scene.frame(0), scene.stamps[0])
        for p in scene.feature_pixels:
            src.addFeature(*p)
        for t in range(1, nfr):
            img, picks = scene.frame(t), scene.picks(t, NFEAT)
            batch.seed_from(src)
            mu0 = src.get_full()[0]
            cams = np.tile(mu0[:14], (B, 1))
            cams[:, 0:3] += rng.normal(scale=1e-3, size=(B, 3))
            batch.set_camera_states(cams)
            batch.captureNewFrame(img, scene.stamps[t])
            t0 = time.perf_counter()
            batch.step(picks)
            t1 = time.perf_counter()
            src.captureNewFrame(img, scene.stamps[t]); src.predict(); src.update(picks)
            if t <= args.warmup:
                continue
            _, st = batch.camera_states()
            n = batch.state_dim(0)
            f = sum(update_flops(batch.state_dim(b) if b == 0 else n, int(st[b, 2]), int(st[b, 3])) for b in range(B))
            d = batch.last_step_ms()
            ms.append(d); wall.append(t1 - t0); flops.append(f)
            lis.append(float(st[:, 2].mean())); his.append(float(st[:, 3].mean()))
        upd = np.array([d["update"] for d in ms])
        rate = np.array(flops) / (upd * 1e-3) / 1e12
        emit({"filters": B, "features": NFEAT, "n": 14 + 6 * NFEAT, "capacity": CAP, "ctas_per_filter": ctas,
              "clusters_resident": resident,
              "predict_ms": round(float(np.median([d["predict"] for d in ms])), 3),
              "match_ms": round(float(np.median([d["match"] for d in ms])), 3),
              "update_ms": round(float(np.median(upd)), 3),
              "step_wall_ms": round(float(np.median(wall)) * 1e3, 3),
              "filter_steps_per_s": round(B / float(np.median(wall)), 1),
              "update_fp64_tflops": round(float(np.median(rate)), 3),
              "mean_li": round(float(np.mean(lis)), 1), "mean_hi": round(float(np.mean(his)), 2), "steps": len(ms)})
        batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
