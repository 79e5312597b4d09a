"""Cost of stepping and capturing a subset of a batch (ekf_batch_step_filters, ekf_batch_capture_camera_frames), on the cfg3
scene (bench.py's camera, motion and 640 x 480 frames, 30 features): 4096 filters as 64 cameras x 64 hypotheses, controls
per filter.

Per-class CUDA-event times of a step (predict, match, update; FilterBatch.last_step_ms) and the host clock around the step
(which ends in a device synchronise), for the full step (ekf_batch_step_controls) and for step_filters on the filters of all,
1/2, 1/8 and 1/64 of the cameras.  Each timed step follows a capture of the cameras whose filters step.  Then the host clock
around a capture (ended by a device synchronise) of all 64 cameras against a capture of 8 of them, gray host frames at scale 1.

    python tools/batch_subset_cost.py [--steps 10] [--warmup 2] [--out FILE]
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
K, M = 64, 64


def main():
    ap = argparse.ArgumentParser()
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

    B = K * M
    nfr = 1 + args.warmup + args.steps
    sc = bench.make_scene(pkg, "cfg3_batch4096", nfr)
    cfg = bench.bench_config(pkg, sc)
    src = pkg.VSlamFilter(cfg, feature_capacity=32)
    bench.seed_filter(src, sc)
    rng = np.random.default_rng(B)
    cams = np.tile(src.get_full()[0][:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=1e-3, size=(B, 3))
    cam_of = np.repeat(np.arange(K), M)
    dv = np.zeros((B, 3)); dw = np.zeros((B, 3))

    def make():
        batch = pkg.FilterBatch(cfg, B, feature_capacity=32)
        batch.seed_from(src)
        batch.set_cameras(K, cam_of)
        batch.set_camera_states(cams)
        return batch

    full_ms = None
    for label, nk in (("full step (step_controls)", None), ("step_filters, all cameras", K), ("step_filters, 1/2 of the cameras", K // 2),
                      ("step_filters, 1/8 of the cameras", K // 8), ("step_filters, 1/64 of the cameras", K // 64)):
        batch = make()
        img = sc.frame(0)
        batch.captureNewFrames(np.ascontiguousarray(np.broadcast_to(img, (K,) + img.shape)), np.full(K, sc.stamps[0]))
        ncam = K if nk is None else nk
        sel = np.arange(ncam, dtype=np.int32)
        filt = np.arange(ncam * M, dtype=np.int32)
        wall, ev, matched = [], [], 0
        for t in range(1, nfr):
            img = sc.frame(t)
            stack = np.ascontiguousarray(np.broadcast_to(img, (ncam,) + img.shape))
            batch.captureNewFrames(stack, np.full(ncam, sc.stamps[t]), cameras=None if nk is None else sel)
            batch.sync()
            t0 = time.perf_counter()
            if nk is None:
                batch.step(sc.picks(t, NFEAT), dv=dv, dw=dw, vcontrol=np.zeros(B, np.int32))
            else:
                batch.step(sc.picks(t, NFEAT), dv=dv[filt], dw=dw[filt], vcontrol=np.zeros(filt.size, np.int32), filters=filt)
            t1 = time.perf_counter()
            if t <= args.warmup:
                continue
            wall.append((t1 - t0) * 1e3)
            ev.append(batch.last_step_ms())
            matched += int(batch.camera_states()[1][filt, 1].sum())
        med = {k: float(np.median([e[k] for e in ev])) for k in ("predict", "match", "update")}
        total = sum(med.values())
        if nk is None:
            full_ms = total
        row = {"layout": label, "filters_stepped": int(filt.size), "cameras_stepped": ncam,
               "predict_ms_median": round(med["predict"], 3), "match_ms_median": round(med["match"], 3),
               "update_ms_median": round(med["update"], 3), "predict_match_update_ms": round(total, 3),
               "of_full_step": round(total / full_ms, 4), "step_wall_ms_median": round(float(np.median(wall)), 3),
               "matched_per_filter": round(matched / len(wall) / filt.size, 2), "steps": len(wall)}
        if nk == K // 8:
            row["bar"] = "predict + match + update at most 1/4 of the full step's"
            row["meets_bar"] = bool(total <= full_ms / 4)
        emit(row)
        batch.close()

    batch = make()
    img = sc.frame(1)
    for label, nk in (("capture of all 64 cameras", None), ("capture of 8 of 64 cameras", 8)):
        ncam = K if nk is None else nk
        stack = np.ascontiguousarray(np.broadcast_to(img, (ncam,) + img.shape))
        sel = np.arange(0, K, K // 8, dtype=np.int32)[:ncam] if nk else None
        ts = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            batch.captureNewFrames(stack, np.full(ncam, 1.0 + i), cameras=sel)
            batch.sync()
            ts.append((time.perf_counter() - t0) * 1e3)
        emit({"capture": label, "frames": ncam, "frame": f"{img.shape[1]} x {img.shape[0]} gray, host, scale 1",
              "wall_ms_median": round(float(np.median(ts[args.warmup:])), 3), "repeats": args.steps})
    batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
