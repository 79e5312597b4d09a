"""Cost of the feature archive and the map export of the batched filters (ekf_batch_set_archive, ekf_batch_get_points_features).

Step time, archive off against archive on, on the cfg3 scene (bench.py's camera, motion and 640 x 480 frames, 30 features, 4096
filters) with removals occurring: a single filter first tracks every feature for seven frames (n_find 7), its rho variances are
cut and its features converted to XYZ; then, before every timed step, both batches are seeded from it (one kernel) and given the
same perturbed camera states, and the step sees a frame in which only every second feature is drawn.  quality_ratio is 0.1, so
each filter deletes its ~15 hidden XYZ features for quality in every step, and with the archive on archives them all.  The two
batches alternate step by step.  Per step: the host clock around ekf_batch_step (which ends in a device synchronise) and the
step's predict / match / update events.

Then the points_features export of every filter (one ekf_batch_get_points_features launch with out, plus the row-count query
FilterBatch.points_features makes first), at capacity 32 and at capacity 128 (a cluster batch), each filter holding its live map
after such a step and that step's archived records.  Host clock around the calls, which end in a device synchronise; the 12-double rows are copied to pageable
host memory.

    python tools/batch_archive_cost.py [--filters 4096] [--steps 10] [--warmup 2] [--out FILE]
"""
import argparse
import ctypes as C
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

NFEAT, TRACK = 30, 7


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--archive", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = ekfb200.load_package()
    L = pkg.lib()
    name, limit = card()
    lines = [json.dumps({"card": name, "power.limit, clocks.max.sm": limit})]
    print(lines[0], flush=True)

    def emit(d):
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)

    B = args.filters
    nfr = TRACK + 1 + args.warmup + args.steps
    full = bench.make_scene(pkg, "cfg3_batch4096", nfr)
    half = bench.make_scene(pkg, "cfg3_batch4096", nfr, visible_every=2)
    over = {f: getattr(bench.bench_config(pkg, full), f) for f, _ in pkg._abi.EkfConfig._fields_}
    over.update(quality_ratio=0.1, xyz_conversion=1, min_features=0, max_features=1000000)
    cfg = pkg.default_config(**over)
    src = pkg.VSlamFilter(cfg, feature_capacity=32)
    bench.seed_filter(src, full)
    for t in range(1, TRACK + 1):
        src.captureNewFrame(full.frame(t), full.stamps[t]); src.predict(); src.update(full.picks(t, NFEAT))
    mu, S = src.get_full()
    for i in range(src.numOfFeatures()):
        p = src.feature(i).position_in_state
        S[p + 5, :] *= 1e-4; S[:, p + 5] *= 1e-4
    src.set_full(mu, S)
    src.convert2XYZ_ifLinearAll()
    xyz = sum(src.feature(i).coding for i in range(src.numOfFeatures()))
    off = pkg.FilterBatch(cfg, B, feature_capacity=32)
    on = pkg.FilterBatch(cfg, B, feature_capacity=32)
    on.set_archive(args.archive)
    rng = np.random.default_rng(B)
    res = {"off": [], "on": []}
    removed = archived = 0
    for t in range(TRACK + 1, nfr):
        img, picks = half.frame(t), half.picks(t, NFEAT)
        mu0 = src.get_full()[0]
        cams = np.tile(mu0[:14], (B, 1))
        cams[:, 0:3] += rng.normal(scale=1e-3, size=(B, 3))
        for key, batch in (("off", off), ("on", on)) if t % 2 else (("on", on), ("off", off)):
            batch.seed_from(src)
            batch.set_camera_states(cams)
            batch.captureNewFrame(img, half.stamps[t])
            t0 = time.perf_counter()
            batch.step(picks)
            t1 = time.perf_counter()
            if t < TRACK + 1 + args.warmup:
                continue
            res[key].append((t1 - t0, batch.last_step_ms()))
            if key == "on":
                _, st = batch.camera_states()
                removed += int(st[:, 6].sum()); archived += int(batch.num_deleted().sum())
    for key in ("off", "on"):
        wall = np.array([w for w, _ in res[key]]) * 1e3
        emit({"step": f"archive {key}", "filters": B, "features": NFEAT, "xyz_features": int(xyz),
              "archive_capacity": args.archive if key == "on" else 0,
              "step_wall_ms_median": round(float(np.median(wall)), 3), "step_wall_ms_min": round(float(wall.min()), 3),
              "step_wall_ms_max": round(float(wall.max()), 3),
              "update_ms_median": round(float(np.median([d["update"] for _, d in res[key]])), 3), "steps": len(wall)})
    emit({"removed_per_step_and_filter": round(removed / max(1, len(res["on"])) / B, 2),
          "archived_per_step_and_filter": round(archived / max(1, len(res["on"])) / B, 2)})
    off.close()
    # the export: every filter holds its live map after a step above and that step's records
    for cap, large in ((32, False), (128, True)):
        batch = on if cap == 32 else pkg.FilterBatch(cfg, B, feature_capacity=cap, large=True)
        if large:
            batch.set_archive(args.archive)
            batch.seed_from(src); batch.set_camera_states(cams)
            batch.captureNewFrame(half.frame(nfr - 1), half.stamps[nfr - 1]); batch.step(half.picks(nfr - 1, NFEAT))
        held = batch.num_deleted()
        rows = np.zeros(B, dtype=np.int32)
        L.ekf_batch_get_points_features(batch.h, 0, B, None, 0, rows.ctypes.data_as(C.c_void_p))
        rc = int(rows.max())
        out = np.zeros((B, rc, 12))
        one, both = [], []
        for _ in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            assert L.ekf_batch_get_points_features(batch.h, 0, B, out.ctypes.data_as(C.c_void_p), rc, rows.ctypes.data_as(C.c_void_p)) == 0
            t1 = time.perf_counter()
            batch.points_features()
            t2 = time.perf_counter()
            one.append(t1 - t0); both.append(t2 - t1)
        one, both = np.array(one[args.warmup:]) * 1e3, np.array(both[args.warmup:]) * 1e3
        emit({"export": "points_features, all filters", "capacity": cap, "filters": B, "rows": rc, "archived_per_filter": float(held.mean()),
              "bytes_out": int(out.nbytes), "call_ms_median": round(float(np.median(one)), 3), "call_ms_min": round(float(one.min()), 3),
              "python_points_features_ms_median": round(float(np.median(both)), 3), "repeats": len(one)})
        batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
