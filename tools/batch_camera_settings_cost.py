"""Cost of camera settings in the batched filters (ekf_batch_set_camera_settings, FilterBatch.from_configs).

Per-class CUDA-event times of a step (predict, match, update; FilterBatch.last_step_ms) and the host clock around capture +
step (which ends in a device synchronise), medians over the timed steps, for:
  cfg3, no table              bench.py's cfg3 batch (4096 filters x 30 features, window 11, 640 x 480 frames);
  cfg3, tuning rows           the same with every tuning row the configuration's (ekf_batch_set_filter_params): the per-filter
                              row instantiations without a camera table;
  cfg3, camera table          the same with a camera table equal to the configuration (window 11, scale 1, blur off);
  rigs, one batch             the four shipped rigs' window, scale and blur threshold (conf 21 / 2 / 1000, firewire 21 / 1 / off,
                              kinect 15 / 2 / 1000, sim 30 / 10 / 3) x `--hyp` hypotheses in one batch built by from_configs, every
                              camera delivering 2560 x 1920 frames;
  rigs, four batches          the same filters as four one-camera batches built by from_config, captured and stepped one after
                              another (times summed over the four).
The rigs' scenes are rendered at each camera's resized size and every pixel replicated scale x scale; each filter starts from
the scene's features added on frame 0 and a perturbed camera state, and both layouts step the same frames with the same picks
(the stack of the one batch is built before the clock starts).
--cases selects layouts by key (cfg3_none, cfg3_rows, cfg3_table, rigs): a build without camera settings can run the first two.

    python tools/batch_camera_settings_cost.py [--cases ...] [--steps 10] [--warmup 2] [--hyp 1024] [--out FILE]
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
RIGS = (("conf", 21, 2, 1000), ("firewire", 21, 1, 1000000000), ("kinect", 15, 2, 1000), ("sim", 30, 10, 3))
IN_W, IN_H = 2560, 1920


def _ms(batch):
    d = batch.last_step_ms()
    return [d["predict"], d["match"], d["update"]]


def _medians(ev, wall):
    return {"predict_ms_median": round(float(np.median([e[0] for e in ev])), 3),
            "match_ms_median": round(float(np.median([e[1] for e in ev])), 3),
            "update_ms_median": round(float(np.median([e[2] for e in ev])), 3),
            "capture_plus_step_wall_ms_median": round(float(np.median(wall)), 3), "steps": len(wall)}


def cfg3(pkg, args, cases, emit):
    B = 4096
    nfr = 1 + args.warmup + args.steps
    sc = bench.make_scene(pkg, "cfg3_batch4096", nfr)
    cfg = bench.bench_config(pkg, sc)
    src = pkg.VSlamFilter(cfg, feature_capacity=32)
    bench.seed_filter(src, sc)
    rng = np.random.default_rng(B)
    cams = np.tile(src.get_full()[0][:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=1e-3, size=(B, 3))
    for key, label in (("cfg3_none", "cfg3, no table"), ("cfg3_rows", "cfg3, tuning rows (the configuration's)"),
                       ("cfg3_table", "cfg3, camera table (the configuration's)")):
        if key not in cases:
            continue
        batch = pkg.FilterBatch(cfg, B, feature_capacity=32)
        if key == "cfg3_rows":
            batch.set_filter_params(pkg._abi.batch_rows(cfg, [cfg] * B)[1])
        if key == "cfg3_table":
            batch.set_camera_settings([[cfg.window_size, cfg.scale, cfg.kernel_size]])
        batch.seed_from(src)
        wall, ev, matched = [], [], 0
        for t in range(1, nfr):
            batch.set_camera_states(cams)
            t0 = time.perf_counter()
            batch.captureNewFrame(sc.frame(t), sc.stamps[t])
            batch.step(sc.picks(t, NFEAT))
            t1 = time.perf_counter()
            if t <= args.warmup:
                continue
            wall.append((t1 - t0) * 1e3)
            ev.append(_ms(batch))
            matched += int(batch.camera_states()[1][:, 1].sum())
        emit(dict({"layout": label, "filters": B, "features": NFEAT, "matched_per_filter": round(matched / len(wall) / B, 2)},
                  **_medians(ev, wall)))
        batch.close()


def rigs(pkg, args, emit):
    M = args.hyp
    K = len(RIGS)
    nfr = 1 + args.warmup + args.steps
    scenes, cfgs = [], []
    for c, (name, w, s, k) in enumerate(RIGS):
        sc = pkg.synth.Scene(n_features=24, n_frames=nfr, seed=1400 + c, width=IN_W // s, height=IN_H // s, window=w, template_smooth=2.0)
        scenes.append(sc)
        cfgs.append(pkg.default_config(**dict(sc.config_overrides(), window_size=w, scale=s, kernel_size=k, xyz_conversion=1)))
    frames = [[np.ascontiguousarray(np.repeat(np.repeat(sc.frame(t), s, axis=0), s, axis=1)) for sc, (_, _, s, _) in zip(scenes, RIGS)]
              for t in range(nfr)]
    stacks = [np.stack(fr) for fr in frames]
    stamps = [[sc.stamps[t] for sc in scenes] for t in range(nfr)]
    camera_of = np.repeat(np.arange(K), M)
    rng = np.random.default_rng(7)

    one = pkg.FilterBatch.from_configs([cfgs[c] for c in camera_of], camera_of, feature_capacity=32)
    one.seed_from(pkg.VSlamFilter(cfgs[0], feature_capacity=32))   # empty: seeds any table
    parts = []
    for c in cfgs:
        p = pkg.FilterBatch.from_config(c, M, feature_capacity=32)
        p.seed_from(pkg.VSlamFilter(c, feature_capacity=32))
        parts.append(p)
    one.captureNewFrames(stacks[0], stamps[0])
    for c, p in enumerate(parts):
        p.captureNewFrame(frames[0][c], stamps[0][c])
        for m in range(M):
            for u, v in scenes[c].feature_pixels:
                one.addFeature(c * M + m, u, v)
                p.addFeature(m, u, v)
    cams = np.concatenate([np.tile(one.get_full(c * M)[0][:14], (M, 1)) for c in range(K)])
    cams[:, 0:3] += rng.normal(scale=1e-3, size=(K * M, 3))
    one.set_camera_states(cams)
    for c, p in enumerate(parts):
        p.set_camera_states(cams[c * M:(c + 1) * M])
    w1, e1, w4, e4, m1, m4 = [], [], [], [], 0, 0
    for t in range(1, nfr):
        picks = scenes[0].picks(t, NFEAT)
        t0 = time.perf_counter()
        one.captureNewFrames(stacks[t], stamps[t])
        one.step(picks)
        t1 = time.perf_counter()
        for c, p in enumerate(parts):
            p.captureNewFrame(frames[t][c], stamps[t][c])
            p.step(picks)
        t2 = time.perf_counter()
        if t <= args.warmup:
            continue
        ev, mt = np.zeros(3), 0
        for p in parts:
            ev += np.asarray(_ms(p))
            mt += int(p.camera_states()[1][:, 1].sum())
        w1.append((t1 - t0) * 1e3); e1.append(_ms(one)); m1 += int(one.camera_states()[1][:, 1].sum())
        w4.append((t2 - t1) * 1e3); e4.append(list(ev)); m4 += mt
    rig = ", ".join(f"{n} {w}/{s}/{'off' if k >= 100000 else k}" for n, w, s, k in RIGS)
    emit(dict({"layout": "rigs, one batch", "rigs (window/scale/blur)": rig, "hypotheses_per_rig": M, "input": f"{IN_W} x {IN_H}",
               "matched_per_filter": round(m1 / len(w1) / (K * M), 2)}, **_medians(e1, w1)))
    emit(dict({"layout": "rigs, four batches stepped in turn (sums)", "hypotheses_per_rig": M,
               "matched_per_filter": round(m4 / len(w4) / (K * M), 2)}, **_medians(e4, w4)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="cfg3_none,cfg3_rows,cfg3_table,rigs")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--hyp", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    cases = set(args.cases.split(","))
    pkg = ekfb200.load_package()
    pkg.lib()
    name, limit = card()
    lines = [json.dumps({"card": name, "power.limit, clocks.max.sm": limit})]
    print(lines[0], flush=True)

    def emit(d):
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)
    cfg3(pkg, args, cases, emit)
    if "rigs" in cases:
        rigs(pkg, args, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
