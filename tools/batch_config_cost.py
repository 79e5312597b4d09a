"""Cost of forsePlane (vslamRansac.cpp:1245-1272) and of resized / BGR capture (vslamRansac.cpp:226-245) in the batched filters.

forsePlane: a single filter runs through the cfg3 scene (640 x 480, 30 features); before every step two batches of 4096
filters are seeded from it (one kernel) and given the same perturbed camera states, then step alternately on the same frame,
one with the plane off (the default), one with set_force_plane(1).  Both steps start from the same state, so they match the
same features and differ only by the plane block (the scene's camera is not held in the plane: run free, a plane-on ensemble
would drift to other states and other work).  For each, the step time (host clock around a call that ends in a device
synchronise), the update class of the step's CUDA events (k_batch_update) and the launches per step are recorded, with the
number of filter-steps that had high-innovation rows (with the plane on, every filter runs a second update; without Hi rows
it holds the plane block alone).

Capture: host frames of a user's camera sizes, each through a batch whose scale resizes them to the filter's frame: a
2560 x 1920 BGR frame at scale 10 and a 1280 x 960 gray frame at scale 2, against the scale-1 copies of a 640 x 480 and a
1280 x 960 gray frame.  Host clock around captureNewFrame and a device synchronise, alternating the cases.

Prints one JSON line with the card name and power limit, then one per measurement; --out also writes them to a file.

    python tools/batch_config_cost.py [--filters 4096] [--steps 20] [--warmup 3] [--captures 50] [--out FILE]
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

CAPTURES = (("gray_640x480_scale1", 640, 480, 1, 1), ("gray_1280x960_scale1", 1280, 960, 1, 1),
            ("gray_1280x960_scale2", 1280, 960, 1, 2), ("bgr_2560x1920_scale10", 2560, 1920, 3, 10))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=bench.BATCH_FILTERS)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--captures", type=int, default=50)
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

    def summary(a):
        a = np.asarray(a, dtype=np.float64)
        return {"median": round(float(np.median(a)), 3), "min": round(float(a.min()), 3), "max": round(float(a.max()), 3)}

    # ---- forsePlane on the cfg3 scene
    workload = "cfg3_batch4096"
    nfeat = bench.WORKLOADS[workload][0]
    B, K, W = args.filters, args.steps, args.warmup
    scene = bench.make_scene(pkg, workload, 2 + W + K, seed=1235)
    picks = [scene.picks(t, nfeat) for t in range(scene.n_frames)]
    runs = ("plane_off", "plane_on")
    cfg = bench.bench_config(pkg, scene)
    f = pkg.VSlamFilter(cfg, feature_capacity=32)
    assert bench.seed_filter(f, scene) == nfeat
    batches = {}
    for key in runs:
        b = pkg.FilterBatch(cfg, B, feature_capacity=nfeat + 2)
        b.set_force_plane(key == "plane_on")
        batches[key] = b
    ms = {k: [] for k in runs}
    upd = {k: [] for k in runs}
    launches = {k: [] for k in runs}
    with_hi = {k: 0 for k in runs}
    for t in range(1, 1 + W + K):
        cams = pkg.dist.ensemble_camera_states(f.getState(), range(B))
        for key in runs:
            batches[key].seed_from(f)
            batches[key].set_camera_states(cams)
        for key in (runs if t % 2 else runs[::-1]):
            b = batches[key]
            b.captureNewFrame(scene.frame(t), scene.stamps[t])
            k0 = b.kernel_launches()
            t0 = time.perf_counter()
            b.step(picks[t])
            dt = (time.perf_counter() - t0) * 1e3
            if t > W:
                ms[key].append(dt)
                upd[key].append(b.last_step_ms()["update"])
                launches[key].append(b.kernel_launches() - k0)
                _, st = b.camera_states()
                with_hi[key] += int((st[:, pkg._abi.BSTAT["hi"]] > 0).sum())
        f.captureNewFrame(scene.frame(t), scene.stamps[t]); f.predict(); f.update(picks[t])
    for key in runs:
        emit(dict({"measure": "step_ms", "run": key, "filters": B, "features": nfeat, "steps": K}, **summary(ms[key]),
                  update_event_ms=summary(upd[key]), launches_per_step=sorted(set(launches[key])),
                  filter_steps_with_hi_rows=with_hi[key]))
    del batches

    # ---- capture
    rng = np.random.default_rng(5)
    cases = []
    for key, w, h, ch, scale in CAPTURES:
        b = pkg.FilterBatch(cfg, 2, feature_capacity=nfeat + 2)
        b.set_scale(scale)
        img = rng.integers(0, 256, (h, w, ch) if ch == 3 else (h, w), dtype=np.uint8)
        b.captureNewFrame(img, 1.0)   # sizes the device buffers
        b.sync()
        cases.append((key, b, img, w // scale, h // scale, []))
    for r in range(args.captures + 3):
        for key, b, img, _, _, times in (cases if r % 2 else cases[::-1]):
            t0 = time.perf_counter()
            b.captureNewFrame(img)
            b.sync()
            if r >= 3:
                times.append((time.perf_counter() - t0) * 1e3)
    for key, b, img, dw, dh, times in cases:
        assert b.returnGrayImg().shape == (dh, dw)
        emit(dict({"measure": "capture_ms", "run": key, "source_bytes": int(img.size), "frame": [dw, dh],
                   "captures": args.captures}, **summary(times)))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
