"""Cost of motion-blur template prediction (Patch::blur, Patch.cpp:50-57; libblur.cpp:17-81) in the batched filters (cfg3:
4096 filters x 30 features, 640 x 480).

Batches seeded from the same filter step alternately through the same frames of the cfg3 scene:
  * blur off (the default);
  * blur on with a threshold nothing exceeds (set_motion_blur(99999)): one launch more, nothing blurred;
  * blur on with threshold 0, so that every gated template is blurred, at T_camera = 1, 4, 16, 64 (the blur displacement is
    the predicted motion over T_camera frames, so the line kernels grow with it; the mean displacement is estimated from
    filter 0's predicted measurements of consecutive steps).
For each, the step time (host clock around a call that ends in a device synchronise) and the predict time of the step's CUDA
events (k_batch_predict + k_batch_predict_blur) are recorded.  Prints one JSON line with the card name and power limit, then
one per measurement; --out also writes them to a file.

    python tools/batch_blur_cost.py [--filters 4096] [--steps 20] [--warmup 3] [--out FILE]
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

T_CAMERAS = (1.0, 4.0, 16.0, 64.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=bench.BATCH_FILTERS)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
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

    runs = [("off", 0.0, None), ("on_nothing_blurred", 0.0, 99999)] + [(f"on_all_blurred_T{t:g}", t, 0) for t in T_CAMERAS]
    batches = {}
    for key, tcam, ks in runs:
        cfg = bench.bench_config(pkg, scene)
        cfg.T_camera = tcam
        f = pkg.VSlamFilter(cfg, feature_capacity=32)
        assert bench.seed_filter(f, scene) == nfeat
        b = pkg.FilterBatch(cfg, B, feature_capacity=nfeat + 2)
        b.seed_from(f)
        b.set_camera_states(pkg.dist.ensemble_camera_states(f.getState(), range(B)))
        if ks is not None:
            b.set_motion_blur(ks)
        batches[key] = b
    ms = {k: [] for k, _, _ in runs}
    pred = {k: [] for k, _, _ in runs}
    launches = {k: [] for k, _, _ in runs}
    blurred = {k: [] for k, _, _ in runs}
    motion = []
    h_prev = None
    for t in range(1, 1 + W + K):
        order = runs if t % 2 else runs[::-1]
        for key, _, _ in order:
            b = batches[key]
            b.captureNewFrame(scene.frame(t), scene.stamps[t])
            k0 = b.kernel_launches()
            t0 = time.perf_counter()
            b.step(picks[t])
            dt = (time.perf_counter() - t0) * 1e3
            if t > W:
                ms[key].append(dt)
                pred[key].append(b.last_step_ms()["predict"])
                launches[key].append(b.kernel_launches() - k0)
                blurred[key].append(int(b.last_blur_counts().sum()))
        h = np.array([list(batches["off"].feature(0, i).h) for i in range(batches["off"].numOfFeatures(0))])
        if h_prev is not None and h.shape == h_prev.shape and t > W:
            motion.append(float(np.mean(np.linalg.norm(h - h_prev, axis=1))))
        h_prev = h
    px_per_frame = float(np.mean(motion)) if motion else float("nan")
    emit({"measure": "predicted_motion_px_per_frame", "filter": 0, "mean": round(px_per_frame, 3)})
    for key, tcam, ks in runs:
        a, p = np.array(ms[key]), np.array(pred[key])
        d = {"measure": "step_ms", "run": key, "filters": B, "features": nfeat, "steps": K, "median": round(float(np.median(a)), 3),
             "min": round(float(a.min()), 3), "max": round(float(a.max()), 3), "predict_event_ms_median": round(float(np.median(p)), 3),
             "launches_per_step": sorted(set(launches[key])), "templates_blurred_per_step": int(np.median(blurred[key]))}
        if ks == 0:
            d["T_camera"] = tcam
            d["approx_displacement_px"] = round(tcam * px_per_frame, 1)
        emit(d)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
