"""Cost of batched filters on cameras of their own (ekf_batch_set_cameras), on the cfg3 scene (bench.py's camera, motion and
640 x 480 frames, 30 features, 4096 filters).

Per-class CUDA-event times of a step (predict, match, update; FilterBatch.last_step_ms) and the host clock around the step
(which ends in a device synchronise) for three layouts of the same 4096 filters:
  1 camera         every filter on one frame (today's batch, ekf_batch_step);
  64 x 64          64 cameras of 64 hypotheses each, controls per filter (ekf_batch_step_controls);
  4096 cameras     one camera per filter, controls per filter.
Every camera's frame is the scene's frame with its own brightness offset (the NCC matcher is invariant to it), so every layout
matches the same features while the matcher reads its windows from the camera's own frame.
Then the capture of the 4096-frame gray stack (1.26 GB) from pinned host memory and from device memory, and one
find_new_features call over all 4096 cameras (every filter asks for 5 corners).  Host clock around calls that end in a device
synchronise.  Last, in a pass of its own, one more such call under torch.profiler: device time per kernel, summed by kernel
(eig maps, keys, segmented sorts, threshold, selection, adds).

    python tools/batch_cameras_cost.py [--filters 4096] [--steps 10] [--warmup 2] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
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
    H, W = sc.frame(0).shape
    offs = (np.arange(B) % 17).astype(np.int16)   # per-camera brightness offset
    dv = np.zeros((B, 3)); dw = np.zeros((B, 3))

    for label, K in (("1 camera", 1), ("64 cameras x 64 hypotheses", 64), ("4096 cameras", B)):
        batch = pkg.FilterBatch(cfg, B, feature_capacity=32)
        batch.seed_from(src)
        if K > 1:
            batch.set_cameras(K, np.arange(B) // (B // K))
        stack = np.empty((K, H, W), np.uint8)
        wall, ev, matched = [], [], 0
        for t in range(1, nfr):
            f = sc.frame(t).astype(np.int16)
            for c in range(K):
                stack[c] = np.clip(f + offs[c], 0, 255)
            batch.set_camera_states(cams)
            t0 = time.perf_counter()
            if K == 1:
                batch.captureNewFrame(stack[0], sc.stamps[t]); batch.step(sc.picks(t, NFEAT))
            else:
                batch.captureNewFrames(stack, np.full(K, sc.stamps[t])); batch.step(sc.picks(t, NFEAT), dv=dv, dw=dw, vcontrol=np.zeros(B, np.int32))
            t1 = time.perf_counter()
            if t <= args.warmup:
                continue
            wall.append((t1 - t0) * 1e3)
            ev.append(batch.last_step_ms())
            matched += int(batch.camera_states()[1][:, 1].sum())
        emit({"layout": label, "filters": B, "cameras": K, "features": NFEAT,
              "predict_ms_median": round(float(np.median([e["predict"] for e in ev])), 3),
              "match_ms_median": round(float(np.median([e["match"] for e in ev])), 3),
              "update_ms_median": round(float(np.median([e["update"] for e in ev])), 3),
              "capture_plus_step_wall_ms_median": round(float(np.median(wall)), 3),
              "matched_per_filter": round(matched / len(wall) / B, 2), "steps": len(wall)})
        if K == B:
            pinned = torch.from_numpy(stack).pin_memory()
            dev = torch.from_numpy(stack).cuda()
            torch.cuda.synchronize()
            hp, dp = [], []
            for _ in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                batch.captureNewFrames(pinned.numpy())   # a view of the pinned buffer
                batch.sync()
                t1 = time.perf_counter()
                batch.captureNewFrames_device(dev.data_ptr(), W, H, W)
                batch.sync()
                t2 = time.perf_counter()
                hp.append((t1 - t0) * 1e3); dp.append((t2 - t1) * 1e3)
            hp, dp = np.array(hp[args.warmup:]), np.array(dp[args.warmup:])
            gb = stack.nbytes / 1e9
            emit({"capture": "4096-frame gray stack", "bytes": int(stack.nbytes),
                  "pinned_host_ms_median": round(float(np.median(hp)), 3), "pinned_host_GBps": round(gb / (np.median(hp) / 1e3), 1),
                  "device_ms_median": round(float(np.median(dp)), 3), "device_GBps": round(gb / (np.median(dp) / 1e3), 1),
                  "repeats": len(hp)})
            fn = []
            for r in range(2):
                batch.seed_from(src); batch.set_camera_states(cams)
                batch.captureNewFrames_device(dev.data_ptr(), W, H, W)
                batch.sync()
                t0 = time.perf_counter()
                added = batch.findNewFeatures(5)
                t1 = time.perf_counter()
                fn.append((t1 - t0) * 1e3)
            emit({"find_new_features": "all cameras, 5 corners a filter", "cameras": K, "ms_first": round(fn[0], 3),
                  "ms_second": round(fn[1], 3), "added_per_filter": round(float(added.mean()), 2)})
            batch.seed_from(src); batch.set_camera_states(cams)
            batch.captureNewFrames_device(dev.data_ptr(), W, H, W)
            batch.sync()
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                batch.findNewFeatures(5)
                batch.sync()
            groups = {"k_det_eig": "eig maps", "k_bdet_keys": "keys", "SegmentedRadixSort": "segmented sorts",
                      "k_bdet_threshold": "threshold", "k_bdet_select": "selection", "k_batch_add": "adds"}
            per, calls, total = {}, {}, 0.0
            for ev in prof.key_averages():
                t = getattr(ev, "device_time_total", None)
                t = ev.cuda_time_total if t is None else t
                if t <= 0:
                    continue
                total += t
                g = next((v for k, v in groups.items() if k in ev.key), "other")
                per[g] = per.get(g, 0.0) + t / 1e3
                calls[g] = calls.get(g, 0) + ev.count
            emit({"find_new_features_kernels": "device ms per kernel group, one call over all cameras (profiled pass)",
                  "device_ms_total": round(total / 1e3, 3),
                  "ms": {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}, "launches": calls})
        batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
