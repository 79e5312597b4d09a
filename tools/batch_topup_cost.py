"""Cost of the top-up (findNewFeatures, vslamRansac.cpp:1312-1315) in the batched filters (cfg3: 4096 filters, 640 x 480).

1. Steady state: two batches on the cfg3 scene, top-up off and on, stepped alternately through the same frames.  Nobody asks
   for features there (min_features = 0), so the two should cost the same.
2. Top-up step: batches reseeded from a filter holding 30 - k of the scene's features, with min_features = 30 and capacity 32,
   so that every filter asks for k features in its next step; one step with top-up on is timed against the same step with
   top-up off, alternately, `--reps` times, for k in 1, 4, 16.  Detection alone (FilterBatch.detect_corners(k)) and
   detection + adds (FilterBatch.findNewFeatures(k)) on such a batch are timed as well.

Times are host clock around calls that end in a device synchronise.  Prints one JSON line with the card name and power limit, then
one per measurement; --out also writes them to a file.

    python tools/batch_topup_cost.py [--filters 4096] [--steps 20] [--warmup 3] [--reps 5] [--out FILE]
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
import bench  # noqa: E402  (scene and configuration of the cfg3 workload)
import ekfb200  # noqa: E402
from batch_xyz_cost import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=bench.BATCH_FILTERS)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
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

    workload = "cfg3_batch4096"
    nfeat = bench.WORKLOADS[workload][0]
    B, K, W = args.filters, args.steps, args.warmup
    scene = bench.make_scene(pkg, workload, 2 + W + K, seed=1235)
    picks = [scene.picks(t, nfeat) for t in range(scene.n_frames)]
    cfg = bench.bench_config(pkg, scene)

    def seed_filter(c, n):
        f = pkg.VSlamFilter(c, feature_capacity=32)
        f.captureNewFrame(scene.frame(0), scene.stamps[0])
        assert sum(f.addFeature(*p) for p in scene.feature_pixels[:n]) == n
        return f

    def reseed(b, f):
        b.seed_from(f)
        b.set_camera_states(pkg.dist.ensemble_camera_states(f.getState(), range(B)))
        return b

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return (time.perf_counter() - t0) * 1e3, r

    def step(b, t):
        b.captureNewFrame(scene.frame(t), scene.stamps[t])
        return timed(lambda: b.step(picks[t]))[0]

    # 1. steady state, nobody asks
    batches = {}
    for on in (0, 1):
        b = reseed(pkg.FilterBatch(cfg, B, feature_capacity=nfeat + 2), seed_filter(cfg, nfeat))
        b.set_topup(on)
        batches[on] = b
    ms = {0: [], 1: []}
    for t in range(1, 1 + W + K):
        for on in ((0, 1) if t % 2 else (1, 0)):
            v = step(batches[on], t)
            if t > W:
                ms[on].append(v)
    for on in (0, 1):
        a = np.array(ms[on])
        emit({"measure": "steady_step_ms", "topup": on, "filters": B, "features": nfeat, "steps": K, "median": round(float(np.median(a)), 3),
              "min": round(float(a.min()), 3), "max": round(float(a.max()), 3), "kernel_launches_total": batches[on].kernel_launches()})
    del batches

    # 2. every filter asks for k features
    ctop = bench.bench_config(pkg, scene)
    ctop.min_features = nfeat
    tb = {on: pkg.FilterBatch(ctop, B, feature_capacity=32) for on in (0, 1)}
    tb[1].set_topup(1)
    for k in (1, 4, 16):
        src = seed_filter(ctop, nfeat - k)
        heavy = {0: [], 1: []}
        det, add, added = [], [], []
        for r in range(args.reps):
            for on in ((0, 1) if r % 2 else (1, 0)):
                heavy[on].append(step(reseed(tb[on], src), 1))
                if on:
                    added.append(int(tb[1].last_added().sum()))
            b = reseed(tb[0], src)
            b.captureNewFrame(scene.frame(1), scene.stamps[1])
            det.append(timed(lambda: b.detect_corners(k))[0])
            v, a = timed(lambda: b.findNewFeatures(k))
            add.append(v)
            added.append(int(a.sum()))
        for on in (0, 1):
            a = np.array(heavy[on])
            emit({"measure": "topup_step_ms", "topup": on, "asked_per_filter": k, "filters": B, "reps": args.reps,
                  "median": round(float(np.median(a)), 3), "min": round(float(a.min()), 3), "max": round(float(a.max()), 3)})
        for what, vals in (("detect_corners_ms", det), ("find_new_features_ms", add)):
            a = np.array(vals)
            emit({"measure": what, "asked_per_filter": k, "filters": B, "reps": args.reps, "median": round(float(np.median(a)), 3),
                  "min": round(float(a.min()), 3), "max": round(float(a.max()), 3)})
        emit({"measure": "features_added_per_call", "asked_per_filter": k, "filters": B, "values": sorted(set(added))})
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
