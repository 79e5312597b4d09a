"""Cost of XYZ conversion in the batched filters (cfg3: 4096 filters x 30 features, 640 x 480).

1. Steady state: two batches on the cfg3 scene, xyz_conversion 0 and 1, stepped alternately through the same frames.  In this
   scene no feature passes the linearity test, so the difference is what deciding costs inside k_batch_update.
2. Conversion-heavy step: both batches reseeded from a filter in which `--convert` features have their rho variance cut by
   1e-4, so that every filter converts them in its next step; one step of each is timed, alternately, `--reps` times.  Also
   FilterBatch.convert2XYZ_ifLinearAll alone on such a batch (decide kernel + fused removal / conversion pass).

Times are host clock around calls that end in a device synchronise (FilterBatch.step returns after the per-filter counters
have reached the host).  Prints the card name and power limit, then one JSON line per measurement.

    python tools/batch_xyz_cost.py [--filters 4096] [--steps 20] [--warmup 3] [--convert 8] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (scene and configuration of the cfg3 workload)
import ekfb200  # noqa: E402


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the measurement stands without it, but say so
        limit = f"unavailable ({e})"
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=bench.BATCH_FILTERS)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--convert", type=int, default=8, help="features per filter made to convert in the conversion-heavy step")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    pkg = ekfb200.load_package()
    pkg.lib()
    name, limit = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {limit}", flush=True)
    workload = "cfg3_batch4096"
    nfeat = bench.WORKLOADS[workload][0]
    B, K, W = args.filters, args.steps, args.warmup
    scene = bench.make_scene(pkg, workload, 2 + W + K, seed=1235)
    picks = [scene.picks(t, nfeat) for t in range(scene.n_frames)]
    cfgs = {}
    for xyz in (0, 1):
        c = bench.bench_config(pkg, scene)
        c.xyz_conversion = xyz
        cfgs[xyz] = c

    def seed_filter(xyz, shrink=0):
        f = pkg.VSlamFilter(cfgs[xyz], feature_capacity=nfeat + 2)
        assert bench.seed_filter(f, scene) == nfeat
        if shrink:
            mu, S = f.get_full()
            for i in range(0, 2 * shrink, 2):
                p = f.feature(i).position_in_state
                S[p + 5, :] *= 1e-2; S[:, p + 5] *= 1e-2   # variance x 1e-4
            f.set_full(mu, S)
        return f

    def reseed(b, f):
        b.seed_from(f)
        b.set_camera_states(pkg.dist.ensemble_camera_states(f.getState(), range(B)))
        return b

    def seeded(xyz):
        return reseed(pkg.FilterBatch(cfgs[xyz], B, feature_capacity=nfeat + 2), seed_filter(xyz))

    def step(b, t):
        b.captureNewFrame(scene.frame(t), scene.stamps[t])
        t0 = time.perf_counter()
        b.step(picks[t])
        return (time.perf_counter() - t0) * 1e3

    def xyz_count(b):
        return sum(sum(b.feature(f, i).coding for i in range(b.numOfFeatures(f))) for f in (0, B // 2, B - 1))

    # 1. steady state, alternating
    batches = {xyz: seeded(xyz) for xyz in (0, 1)}
    ms = {0: [], 1: []}
    for t in range(1, 1 + W + K):
        order = (0, 1) if t % 2 else (1, 0)
        for xyz in order:
            v = step(batches[xyz], t)
            if t > W:
                ms[xyz].append(v)
    launches = {xyz: batches[xyz].kernel_launches() for xyz in (0, 1)}
    print(f"XYZ features in filters 0, B/2, B-1 after the steady-state steps: {xyz_count(batches[1])}", flush=True)
    for xyz in (0, 1):
        a = np.array(ms[xyz])
        print(json.dumps({"measure": "steady_step_ms", "xyz_conversion": xyz, "filters": B, "features": nfeat, "steps": K,
                          "median": round(float(np.median(a)), 3), "min": round(float(a.min()), 3), "max": round(float(a.max()), 3),
                          "kernel_launches_total": launches[xyz]}), flush=True)

    # 2. one step in which every filter converts `--convert` features, against the same step without conversion; the batches
    # are reseeded (no allocation) before every timed step
    shrunk = {xyz: seed_filter(xyz, shrink=args.convert) for xyz in (0, 1)}
    heavy = {0: [], 1: []}
    conv_ms, counts = [], []
    for r in range(args.reps):
        for xyz in ((0, 1) if r % 2 else (1, 0)):
            heavy[xyz].append(step(reseed(batches[xyz], shrunk[xyz]), 1))
            if xyz:
                counts.append(xyz_count(batches[1]))
        reseed(batches[1], shrunk[1])
        t0 = time.perf_counter()
        batches[1].convert2XYZ_ifLinearAll()
        conv_ms.append((time.perf_counter() - t0) * 1e3)
        counts.append(xyz_count(batches[1]))
    print(f"XYZ features in filters 0, B/2, B-1 after each converting call: {counts} (expected {3 * args.convert} each)", flush=True)
    for xyz in (0, 1):
        a = np.array(heavy[xyz])
        print(json.dumps({"measure": "converting_step_ms", "xyz_conversion": xyz, "filters": B, "converted_per_filter": args.convert * xyz,
                          "reps": args.reps, "median": round(float(np.median(a)), 3), "min": round(float(a.min()), 3),
                          "max": round(float(a.max()), 3)}), flush=True)
    a = np.array(conv_ms)
    print(json.dumps({"measure": "convert2XYZ_ifLinearAll_ms", "filters": B, "converted_per_filter": args.convert, "reps": args.reps,
                      "median": round(float(np.median(a)), 3), "min": round(float(a.min()), 3), "max": round(float(a.max()), 3)}),
          flush=True)


if __name__ == "__main__":
    main()
