"""Cost of tuning per filter in the batched filters (ekf_batch_set_filter_params), on the cfg3 scene (bench.py's camera,
motion and 640 x 480 frames, 30 features, 4096 filters).

Per-class CUDA-event times of a step (predict, match, update; FilterBatch.last_step_ms), the host clock around capture +
step (which ends in a device synchronise) and the mean Li / Hi rows per filter (the update's work), for these layouts of the
same 4096 filters:
  no table                  today's batch;
  configuration rows        every filter's row equal to the configuration (the table instantiations, the default bits);
  4096 rows, same work      every row distinct in its bits, with the decisions of the configuration: the six process-noise
                            sigmas scaled by 1 + U(-1e-9, 1e-9), the thresholds by 1 + U(-1e-6, 1e-6), ransac_nhyp0 and
                            max_features above anything reached;
  4096 rows                 every filter with a tuning of its own: the six process-noise sigmas, sigma_rho_0, the NCC, quality,
                            linearity, Li and Hi thresholds scaled by 1 + U(-0.1, 0.1), sigma_pixel 1 to 3 (this changes the
                            work: the Li threshold moves with sigma_pixel);
  64 x 64, no table         64 cameras of 64 hypotheses, controls per filter, the baseline of
  64 x 64, 64 rows          the same with one row per camera (rows[camera_of]).
Last, set_filter_params itself: host clock of one call with 4096 rows (it ends in a device synchronise).

    python tools/batch_params_cost.py [--filters 4096] [--steps 10] [--warmup 2] [--out FILE]
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
PERTURBED = ("sigma_vx", "sigma_vy", "sigma_vz", "sigma_wx", "sigma_wy", "sigma_wz", "sigma_rho_0", "ncc_threshold", "quality_ratio",
             "linearity_threshold", "li_threshold_factor", "hi_chi2_threshold")


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
    _, same = pkg._abi.batch_rows(cfg, [cfg] * B)
    _, quiet = pkg._abi.batch_rows(cfg, [cfg] * B)
    for f in range(B):
        for k in PERTURBED[:6]:
            setattr(quiet[f], k, getattr(cfg, k) * (1.0 + rng.uniform(-1e-9, 1e-9)))
        for k in PERTURBED[7:]:
            setattr(quiet[f], k, getattr(cfg, k) * (1.0 + rng.uniform(-1e-6, 1e-6)))
        quiet[f].ransac_nhyp0 = cfg.ransac_nhyp0 + f
        quiet[f].max_features = cfg.max_features + f
    _, rows = pkg._abi.batch_rows(cfg, [cfg] * B)
    for f in range(B):
        for k in PERTURBED:
            setattr(rows[f], k, getattr(cfg, k) * (1.0 + rng.uniform(-0.1, 0.1)))
        rows[f].sigma_pixel = 1 + f % 3
    dv = np.zeros((B, 3)); dw = np.zeros((B, 3))

    for label, K, table in (("1 camera, no table", 1, None), ("1 camera, every row the configuration's", 1, same),
                            ("1 camera, 4096 distinct rows, the configuration's decisions", 1, quiet),
                            ("1 camera, 4096 distinct rows", 1, rows),
                            ("64 cameras x 64 hypotheses, no table", 64, None),
                            ("64 cameras x 64 hypotheses, a row per camera", 64, "per camera")):
        batch = pkg.FilterBatch(cfg, B, feature_capacity=32)
        batch.seed_from(src)
        if K > 1:
            cam_of = np.arange(B) // (B // K)
            batch.set_cameras(K, cam_of)
            if table is not None:
                table = [rows[int(c)] for c in cam_of]
        if table is not None:
            batch.set_filter_params(table)
        wall, ev, matched, li, hi = [], [], 0, 0, 0
        for t in range(1, nfr):
            img = sc.frame(t)
            stack = np.ascontiguousarray(np.broadcast_to(img, (K,) + img.shape))
            batch.set_camera_states(cams)
            t0 = time.perf_counter()
            if K == 1:
                batch.captureNewFrame(img, sc.stamps[t])
                batch.step(sc.picks(t, NFEAT))
            else:
                batch.captureNewFrames(stack, np.full(K, sc.stamps[t]))
                batch.step(sc.picks(t, NFEAT), dv=dv, dw=dw, vcontrol=np.zeros(B, np.int32))
            t2 = time.perf_counter()
            if t <= args.warmup:
                continue
            wall.append((t2 - t0) * 1e3)
            ev.append(batch.last_step_ms())
            st = batch.camera_states()[1]
            matched += int(st[:, 1].sum()); li += int(st[:, 2].sum()); hi += int(st[:, 3].sum())
        emit({"layout": label, "filters": B, "cameras": K, "features": NFEAT,
              "predict_ms_median": round(float(np.median([e["predict"] for e in ev])), 3),
              "match_ms_median": round(float(np.median([e["match"] for e in ev])), 3),
              "update_ms_median": round(float(np.median([e["update"] for e in ev])), 3),
              "capture_plus_step_wall_ms_median": round(float(np.median(wall)), 3),
              "matched_per_filter": round(matched / len(wall) / B, 2), "li_per_filter": round(li / len(wall) / B, 2),
              "hi_per_filter": round(hi / len(wall) / B, 2), "steps": len(wall)})
        if table is rows:
            ts = []
            for _ in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                batch.set_filter_params(rows)
                ts.append((time.perf_counter() - t0) * 1e3)
            emit({"set_filter_params": f"{B} rows", "ms_median": round(float(np.median(ts[args.warmup:])), 3), "repeats": args.steps})
        batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
