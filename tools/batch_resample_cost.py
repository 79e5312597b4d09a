"""Cost of resampling the batched filters (ekf_batch_resample) against a device-to-device copy of the same bytes.

Workloads: the cfg3 scene (bench.py's camera and 640 x 480 frames, 30 features) with 4096 filters as 64 cameras x 64 hypotheses,
resampling 1/2 and 1/8 of the filters; and 512 filters of capacity 128 (the cluster-update batch) holding about 100 features,
resampling 1/2.  Each takes a vector from systematic_ancestors (every source keeps its slot: one launch) and one that moves the
same destinations from each other (a cycle over them, so every source is overwritten and staged first).

The bytes a resample must move are computed from shapes: per moved filter its live Sigma rows (n x ld doubles), mu (n), the
feature table (N entries of every field), the pending XYZ decisions (N), both templates (N x tstride bytes each) and its
archive's held records, each read once and written once.  The time is CUDA events on the batch's stream around the call (the
pair upload included; the call ends in a synchronise), median over repeats; beside it a torch copy_ (cudaMemcpyAsync, device
to device) of the same byte count, timed in the same run.  Every filter of a seeded batch has the same n, so repeats of a
vector move the same bytes.

    python tools/batch_resample_cost.py [--repeats 20] [--warmup 3] [--out FILE]
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

PTS_COLS = 12
BAR = 0.6   # the non-aliased half resample reaches at least this share of the copy's byte rate


def filter_bytes(d, n, N, tstride, held=0):
    """Bytes of one filter a resample reads (and writes): live Sigma rows, mu, table, XYZ decisions, templates, archive."""
    table = N * (11 * 4 + 4 * 4 + 34 * 8)     # 11 int fields, center / quality / last_ncc floats, z / h / Hc / S2 doubles
    xyz = N * (4 + 21 * 8)                    # flag, 3 x 6 Jacobian and point
    return 8 * n * d.ld + 8 * n + table + xyz + 2 * N * tstride + held * (PTS_COLS * 8 + 4)


def vectors(pkg, cam_of, M, frac):
    """(systematic, aliased) ancestors moving `frac` of every camera's M filters."""
    B = cam_of.size
    keep = M - int(round(M * frac))
    w = np.tile((np.arange(M) < keep).astype(np.float64), B // M)
    sysv = pkg.systematic_ancestors(w, 0.5, camera_of=cam_of)
    moved = np.flatnonzero(sysv != np.arange(B))
    alias = np.arange(B, dtype=np.int32)
    for c in np.unique(cam_of):   # destinations of camera c copy each other in a cycle
        dc = moved[cam_of[moved] == c]
        alias[dc] = np.roll(dc, 1)
    return sysv, alias


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
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

    stream = torch.cuda.Stream()

    def timed(fn):
        ts, wall = [], []
        for i in range(args.warmup + args.repeats):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            if i >= args.warmup:
                ts.append(a.elapsed_time(b))
                wall.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ts)), float(np.median(wall))

    def copy_ms(nbytes):
        src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        dst = torch.empty_like(src)
        with torch.cuda.stream(stream):
            ms, _ = timed(lambda: dst.copy_(src))
        del src, dst
        return ms

    cases = []
    sc = bench.make_scene(pkg, "cfg3_batch4096", 2)
    cases.append(("cfg3: 4096 filters x 30 features, 64 cameras x 64", sc, 32, False, 64, 64, (0.5, 0.125)))
    big = pkg.synth.Scene(n_features=100, width=640, height=480, n_frames=2, seed=1236, speed=0.1, omega=0.02)
    cases.append(("512 filters of capacity 128, 8 cameras x 64", big, 128, True, 8, 64, (0.5,)))
    for label, scene, cap, large, K, M, fracs in cases:
        cfg = bench.bench_config(pkg, scene)
        src = pkg.VSlamFilter(cfg, feature_capacity=cap)
        bench.seed_filter(src, scene)
        B = K * M
        cam_of = np.repeat(np.arange(K), M)
        batch = pkg.FilterBatch(cfg, B, feature_capacity=cap, large=large)
        batch.seed_from(src)
        batch.set_cameras(K, cam_of)
        batch.set_stream(stream.cuda_stream)
        d = batch.describe()
        n, N = batch.state_dim(0), batch.numOfFeatures(0)
        tstride = (cfg.window_size * cfg.window_size + 15) & ~15
        per = filter_bytes(d, n, N, tstride)
        for frac in fracs:
            sysv, alias = vectors(pkg, cam_of, M, frac)
            moved = int((sysv != np.arange(B)).sum())
            one_way = moved * per
            cms = copy_ms(one_way)
            for kind, anc in (("systematic_ancestors (no staging)", sysv), ("a cycle over the same destinations (all staged)", alias)):
                l0 = batch.kernel_launches()
                batch.resample(anc)
                launches = batch.kernel_launches() - l0
                ms, wall = timed(lambda: batch.resample(anc))
                row = {"workload": label, "n": n, "N": N, "ld": d.ld, "filters_moved": moved, "of_filters": round(moved / B, 4),
                       "vector": kind, "launches": launches, "bytes_each_way": one_way,
                       "resample_ms_median": round(ms, 4), "resample_wall_ms_median": round(wall, 4),
                       "resample_GBps": round(one_way / ms / 1e6, 1), "copy_same_bytes_ms_median": round(cms, 4),
                       "copy_GBps": round(one_way / cms / 1e6, 1), "of_copy_rate": round(cms / ms, 3), "repeats": args.repeats}
                if frac == 0.5 and not kind.startswith("a cycle"):
                    row["bar"] = f"at least {BAR} of the copy's byte rate"
                    row["meets_bar"] = bool(cms / ms >= BAR)
                emit(row)
        batch.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
