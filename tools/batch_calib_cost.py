"""Cost of intrinsics per filter in the batched filters (ekf_batch_set_intrinsics), on the cfg3 scene (bench.py's camera,
motion and 640 x 480 frames, 30 features, 4096 filters).

Per-class CUDA-event times of a step (predict, match, update; FilterBatch.last_step_ms), the host clock around capture + step
(which ends in a device synchronise) and the host clock around the capture alone, for three layouts of the same 4096 filters:
  1 camera                  every filter with the configuration's intrinsics (today's batch);
  1 camera, 4096 rows       every filter with intrinsics of its own (fx, fy, u0, v0, k1, k2 scaled by 1 + N(0, 1e-3));
  64 x 64, 64 rows          64 cameras of 64 hypotheses, one row per camera (params[camera_of]), controls per filter;
  64 x 64, mixed sizes      the same at four frame sizes (640 x 480, 600 x 440, 560 x 420 and 500 x 380, the top left of the
                            scene's frame) in one padded stack (set_frame_sizes): the capture zeroes the pads.
Last, set_intrinsics itself: host clock of one call with 4096 rows (it ends in a device synchronise).

    python tools/batch_calib_cost.py [--filters 4096] [--steps 10] [--warmup 2] [--out FILE]
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

NFEAT = 30
KEYS = ("fx", "fy", "u0", "v0", "k1", "k2", "k3", "p1", "p2")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096)
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

    B = args.filters
    nfr = 1 + args.warmup + args.steps
    sc = bench.make_scene(pkg, "cfg3_batch4096", nfr)
    cfg = bench.bench_config(pkg, sc)
    src = pkg.VSlamFilter(cfg, feature_capacity=32)
    bench.seed_filter(src, sc)
    rng = np.random.default_rng(B)
    cams = np.tile(src.get_full()[0][:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=1e-3, size=(B, 3))
    row = np.array([getattr(cfg, k) for k in KEYS])
    rows = np.tile(row, (B, 1))
    rows[:, :6] *= 1.0 + rng.normal(scale=1e-3, size=(B, 6))
    dv = np.zeros((B, 3)); dw = np.zeros((B, 3))

    for label, K, table in (("1 camera, configuration intrinsics", 1, None), ("1 camera, 4096 intrinsics rows", 1, rows),
                            ("64 cameras x 64 hypotheses, a row per camera", 64, "per camera"),
                            ("64 cameras x 64 hypotheses, a row per camera, four frame sizes", 64, "sizes")):
        batch = pkg.FilterBatch(cfg, B, feature_capacity=32)
        batch.seed_from(src)
        if K > 1:
            cam_of = np.arange(B) // (B // K)
            batch.set_cameras(K, cam_of)
            if table == "sizes":
                batch.set_frame_sizes([[(640, 480), (600, 440), (560, 420), (500, 380)][c % 4] for c in range(K)])
            table = rows[:K][cam_of]
        if table is not None:
            batch.set_intrinsics(table)
        wall, cap, ev, matched = [], [], [], 0
        for t in range(1, nfr):
            img = sc.frame(t)
            stack = np.ascontiguousarray(np.broadcast_to(img, (K,) + img.shape))
            batch.set_camera_states(cams)
            t0 = time.perf_counter()
            if K == 1:
                batch.captureNewFrame(img, sc.stamps[t])
            else:
                batch.captureNewFrames(stack, np.full(K, sc.stamps[t]))
            batch.sync()
            t1 = time.perf_counter()
            if K == 1:
                batch.step(sc.picks(t, NFEAT))
            else:
                batch.step(sc.picks(t, NFEAT), dv=dv, dw=dw, vcontrol=np.zeros(B, np.int32))
            t2 = time.perf_counter()
            if t <= args.warmup:
                continue
            wall.append((t2 - t0) * 1e3); cap.append((t1 - t0) * 1e3)
            ev.append(batch.last_step_ms())
            matched += int(batch.camera_states()[1][:, 1].sum())
        emit({"layout": label, "filters": B, "cameras": K, "features": NFEAT,
              "predict_ms_median": round(float(np.median([e["predict"] for e in ev])), 3),
              "match_ms_median": round(float(np.median([e["match"] for e in ev])), 3),
              "update_ms_median": round(float(np.median([e["update"] for e in ev])), 3),
              "capture_ms_median": round(float(np.median(cap)), 3),
              "capture_plus_step_wall_ms_median": round(float(np.median(wall)), 3),
              "matched_per_filter": round(matched / len(wall) / B, 2), "steps": len(wall)})
        if table is rows:
            ts = []
            for _ in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                batch.set_intrinsics(rows)
                ts.append((time.perf_counter() - t0) * 1e3)
            emit({"set_intrinsics": f"{B} rows ({72 * B} bytes)", "ms_median": round(float(np.median(ts[args.warmup:])), 3),
                  "repeats": args.steps})
        batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
