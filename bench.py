import os as _os_env
_os_env.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # one hardware queue per stream (see _lib.py); before CUDA starts
#!/usr/bin/env python
"""bench.py — MonoSLAM EKF hot path on B200: frames/s of predict + active-search match + update.

Headline workload (BASELINE.json configs[1]): single filter, 500 inverse-depth features (state dim 3014),
synthetic 640x480 sequence, fp64.  One "step" = one camera frame through captureNewFrame -> predict
-> update (match + RANSAC + both EKF corrections + book-keeping), exactly the call sequence of
ImageConverter::imageCb (monoslam_ransac.cpp:404-557).

  value    : frames/s with the frames already resident in HBM (ekf_capture_frame_device)
  e2e      : frames/s through the public API with HOST frames (H2D inside the timed step) and the
             state / covariance / feature flags read back to the host every step
  parity   : one frame of THIS configuration, from identical inputs, against the CPU oracle (cfg1 / cfg2 / cfg3) or
             an independent fp64 numpy / LAPACK evaluation (cfg4), taken before the timing
  sharded  : (default workload only) short passes of the two paths that shard across GPUs, in the same run —
             cfg3 (batch of filters, sharded by filter, weak scaling) and cfg4 (large map, covariance row blocks
             partitioned across the ranks, strong scaling) — with their own value / ms_per_step / per-class times /
             exchanged bytes / parity, so that `--gpus N` measures them at every N
  N > 1    : the single-filter cfg2 path does not shard ("replicas only", DESIGN.md): every rank runs an
             independent replica, value = total frames / max-over-ranks time, scaling "weak"
  --impl reference : the CPU oracle (dense reference algebra, all host threads) on the same workload, rank 0 only;
             it does not load the CUDA library

Timing: W warm-up steps, then K steps each bracketed by CUDA events on the launching stream; L2 is
flushed (256 MiB write) between timed steps, outside the event pairs; max over ranks.

--dump-outputs DIR: after the timed steps, rank 0 writes what the headline path computed in its last step as
DIR/<name>.npy (float32 / float64, at most 64 MB in all), so that two builds can be compared output for output
on the same seeded inputs.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

sys.dont_write_bytecode = True   # the tree may be read-only: nothing is cached in it
ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

UNIT = "frames/s"
WORKLOADS = {
    # name: (features, width, height)
    "cfg1_n50": (50, 640, 480),
    "cfg2_n500": (500, 640, 480),
    # BASELINE configs[2]: 4096 independent filters x 30 features per GPU, sharded by filter
    "cfg3_batch4096": (30, 640, 480),
    # BASELINE configs[3]: large map, 2000 features (n = 12014, Sigma = 1.15 GB)
    "cfg4_n2000": (2000, 1920, 1080),
    # BASELINE configs[4]: stateless active-search NCC matching, 256 frames x 200 features, 11x11 patches
    "cfg5_match": (200, 1920, 1080),
}
MATCH_FRAMES = 256
METRIC_MATCH = "active-search NCC matches/s (Patch::findMatch, 11x11 templates, 200 features per 1920x1080 frame, 256 frames)"
UNIT_MATCH = "matches/s"
BATCH_FILTERS = 4096
METRIC_BATCH = "batched EKF filter-steps/s (predict+match+update), 4096 independent filters x N=30 features per GPU"
UNIT_BATCH = "filter-steps/s"
PARITY_TOL = 1e-9
DUMP_LIMIT = 64 << 20
BENCH_DEPTH_RANGE = (1.5, 3.0)
BENCH_RHO_0 = 0.5


def metric_for(workload):
    n = WORKLOADS[workload][0]
    return f"EKF frames/s (predict+match+update), single filter, N={n} features"


def workload_string(workload, match_every=1):
    """The same text in both arms (ours / --impl reference): nothing measured goes in here."""
    nfeat, width, height = WORKLOADS[workload]
    return (f"{workload}: single filter, {nfeat} inverse-depth features (n={14 + 6 * nfeat}), {width}x{height} u8 frames, "
            f"predict+match+update per frame, "
            + ("all features matched" if match_every <= 1 else f"every {match_every}th feature visible")
            + ", map held at N features for the whole run (depths 1.5-3 m, rho_0 = 0.5, quality_ratio = 1e9: no deletions)")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed passes run (one sampler, rank 0's GPU)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index, enabled=True):
        self.rows = []
        self.gpu = gpu_index
        self.proc = None
        self.enabled = enabled

    def start(self):
        if not self.enabled:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.enabled:
            return None
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_scene(pkg, workload, n_frames, seed=1235, visible_every=1):
    nfeat, W, H = WORKLOADS[workload]
    # slow motion so that all seeded features stay inside the image for the whole run (fixed N)
    # depths of 1.5 - 3 m around the prior rho_0 = 0.5 (bench_config): with the reference's default prior (rho_0 = 0.1 at a
    # variance of 0.25) the first updates drive a few inverse depths through zero and the reference deletes those features
    # (vslamRansac.cpp:1296-1299), which would shrink the state below the size the metric names
    return pkg.synth.Scene(n_features=nfeat, width=W, height=H, n_frames=n_frames, seed=seed, speed=0.1, omega=0.02,
                           accel_sigma=0.002, border=44, visible_every=visible_every, depth_range=BENCH_DEPTH_RANGE)


def bench_config(pkg, scene):
    """ekf_config of every bench workload: the scene's camera, and the map held at N features for the whole run
    (a feature that misses a few early matches would otherwise be deleted mid-run and shrink the state below the
    size the metric names)."""
    over = scene.config_overrides()
    over["quality_ratio"] = 1.0e9
    over["rho_0"] = BENCH_RHO_0
    return pkg.default_config(**over)


def seed_filter(filt, scene):
    filt.captureNewFrame(scene.frame(0), scene.stamps[0])
    if hasattr(filt, "addFeatures"):       # the oracle's bulk form (bit-identical to per-feature calls)
        return filt.addFeatures(scene.feature_pixels)
    return sum(filt.addFeature(*p) for p in scene.feature_pixels)


def dgemm_peak_tflops(torch, n=4096):
    a = torch.randn(n, n, dtype=torch.float64, device="cuda"); b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(4):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); a @ b; e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / best / 1e9


def hbm_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(path)) if os.path.exists(path) else {}
    return float(peaks.get("hbm_gbs", 6456.5)), ("MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else
                                                 "fallback 6456.5 GB/s (MEASURED_PEAKS.json absent)")


# ------------------------------------------------------------------------------------------------
# process context: one process per GPU, torch.distributed (NCCL) only for barriers / reductions of timings
# ------------------------------------------------------------------------------------------------
def make_ctx():
    import torch
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return types.SimpleNamespace(torch=torch, rank=rank, world=world, local=local, dist=dist,
                                 device=torch.device("cuda", local))


def ctx_barrier(ctx):
    if ctx.dist is not None:
        ctx.dist.barrier()
    ctx.torch.cuda.synchronize()


def ctx_max(ctx, v):
    if ctx.dist is None:
        return float(v)
    t = ctx.torch.tensor([float(v)], dtype=ctx.torch.float64, device="cuda")
    ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
    return float(t.item())


def dump_outputs(directory, arrays):
    """Writes every array as DIR/<name>.npy in float64 (float32 arrays stay float32)."""
    arrays = {k: np.asarray(v) if np.asarray(v).dtype == np.float32 else np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"outputs of {total} bytes exceed the {DUMP_LIMIT} byte limit"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"dumped {len(arrays)} outputs ({total / 2**20:.1f} MiB) to {directory}")


def filter_outputs(filt):
    """What a caller of one filter step receives: the state, the covariance (whole when it fits half the dump limit,
    else a fixed seeded sample of its rows, all columns) and the feature table."""
    from helpers import INT_FIELDS
    mu, S = filt.get_full()
    n = S.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(n, min(n, (DUMP_LIMIT // 2) // (8 * n)), replace=False))
    feats = [filt.feature(i) for i in range(filt.numOfFeatures())]
    st = filt.stats()
    return {"mu": mu, "sigma_rows": S[rows], "sigma_row_index": rows,
            "feature_center": np.array([tuple(a.center) for a in feats], dtype=np.float32).reshape(-1, 2),
            "feature_z": np.array([tuple(a.z) for a in feats]).reshape(-1, 2),
            "feature_h": np.array([tuple(a.h) for a in feats]).reshape(-1, 2),
            "feature_table": np.array([[getattr(a, k) for k in INT_FIELDS] for a in feats]).reshape(-1, len(INT_FIELDS)),
            "step_stats": np.array([getattr(st, k) for k, _ in type(st)._fields_ if k != "kernel_launches"])}


def state_digest(mu, S):
    hsh = hashlib.sha256()
    hsh.update(np.ascontiguousarray(mu).tobytes()); hsh.update(np.ascontiguousarray(S).tobytes())
    return hsh.digest()


# ------------------------------------------------------------------------------------------------
# parity probes (one frame of the benchmarked configuration, before the timing)
# ------------------------------------------------------------------------------------------------
def tables_equal(g, o):
    from helpers import INT_FIELDS
    if g.numOfFeatures() != o.numOfFeatures():
        return False
    for i in range(g.numOfFeatures()):
        a, b = g.feature(i), o.feature(i)
        for f in INT_FIELDS:
            if getattr(a, f) != getattr(b, f):
                return False
        if tuple(a.center) != tuple(b.center):
            return False
    return True


def parity_vs_oracle(pkg, scene, cfg, new_filter, nfeat):
    """Frame 1 on the CUDA path and on the CPU oracle (dense reference algebra, OpenMP) from identical inputs."""
    import orc
    from helpers import relerr
    orc.build()
    L = orc.lib(omp=True)
    L.orc_set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    g = new_filter(attach=False)
    o = orc.OracleFilter(cfg, kind=0, omp=True)
    o.captureNewFrame(scene.frame(0), scene.stamps[0])
    o.import_from(g)
    mu, S = o.get_full(); g.set_full(mu, S)
    img = scene.frame(1)
    for f in (g, o):
        f.captureNewFrame(img, scene.stamps[1]); f.predict(); f.update(scene.picks(1, nfeat))
    mg, Sg = g.get_full(); mo, So = o.get_full()
    sg, so = g.stats(), o.stats()
    counters = all(getattr(sg, k) == getattr(so, k) for k in ("n_matched", "n_li", "n_hi", "ransac_hypotheses", "n_removed"))
    res = {"against": f"CPU oracle, dense reference algebra, fp64 state / float matcher, {L.orc_num_threads()} threads",
           "frames": 1, "n": int(mg.size), "n_li": int(sg.n_li),
           "mu_rel": float(relerr(mg, mo)), "sigma_rel": float(relerr(Sg, So)),
           "tables_equal": bool(tables_equal(g, o) and counters), "tol": PARITY_TOL,
           "seconds": round(time.perf_counter() - t0, 1)}
    res["ok"] = bool(res["tables_equal"] and res["mu_rel"] <= PARITY_TOL and res["sigma_rel"] <= PARITY_TOL)
    del g, o
    return res


def parity_vs_numpy(pkg, scene, cfg, filt, nfeat):
    """Frame 1 on `filt` (collective when it is row-block partitioned: every rank calls this); rank-local result
    against the independent numpy / LAPACK evaluation of the covariance correction (tests/helpers.py)."""
    from helpers import numpy_stacked_update, relerr
    t0 = time.perf_counter()
    filt.captureNewFrame(scene.frame(1), scene.stamps[1]); filt.predict()
    filt.match()
    mu0, S0 = filt.get_full()
    feats = [filt.feature(i) for i in range(filt.numOfFeatures())]
    filt.update_after_match(scene.picks(1, nfeat))
    st = filt.stats()
    mu1, S1 = filt.get_full()
    return dict(mu0=mu0, S0=S0, feats=feats, st=st, mu1=mu1, S1=S1, t0=t0,
                finish=lambda: _numpy_finish(filt, cfg, mu0, S0, feats, st, mu1, S1, t0, numpy_stacked_update, relerr))


def _numpy_finish(filt, cfg, mu0, S0, feats, st, mu1, S1, t0, numpy_stacked_update, relerr):
    sel = [i for i in range(filt.numOfFeatures()) if filt.feature(i).is_in_li]
    if st.n_hi != 0 or st.n_removed != 0:
        return {"against": "numpy", "ok": False, "note": f"scene not all-inlier (n_hi={st.n_hi}, removed={st.n_removed})"}
    mu_ref, S_ref = numpy_stacked_update(mu0, S0, feats, sel, float(cfg.sigma_pixel) ** 2)
    res = {"against": "independent fp64 numpy / LAPACK evaluation of Sigma - Sigma H^T (H Sigma H^T + R)^-1 H Sigma + "
                      "normalizeQuaternion from the same H rows (tests/helpers.numpy_stacked_update); decisions are the CUDA path's own",
           "frames": 1, "n": int(mu1.size), "n_li": int(st.n_li),
           "mu_rel": float(relerr(mu1, mu_ref)), "sigma_rel": float(relerr(S1, S_ref)),
           "dsigma_rel": float(relerr(S1 - S0, S_ref - S0)), "tables_equal": None, "tol": PARITY_TOL,
           "seconds": round(time.perf_counter() - t0, 1)}
    res["ok"] = bool(res["mu_rel"] <= PARITY_TOL and res["sigma_rel"] <= PARITY_TOL)
    return res


# ------------------------------------------------------------------------------------------------
# single-filter workloads (cfg1 / cfg2: replicas at N > 1; cfg4: row-block partitioned at N > 1)
# ------------------------------------------------------------------------------------------------
def bench_single(args, ctx, workload, K, Wm, with_cpu=True, with_clocks=True, with_parity=True, dump_dir=None):
    torch, dist, rank, world, local = ctx.torch, ctx.dist, ctx.rank, ctx.world, ctx.local
    import ekfb200
    pkg = ekfb200.load_package()
    pkg.lib()  # fails loudly if the CUDA library is missing
    nfeat, width, height = WORKLOADS[workload]
    # cfg4 (large map) at N > 1: ONE filter whose stacked update is partitioned by covariance row blocks
    # (every rank holds a replica and runs the same calls); other single-filter workloads: replicas only
    partitioned = world > 1 and workload.startswith("cfg4")
    scene = make_scene(pkg, workload, 1 + Wm + K, seed=1235 + (0 if (partitioned or world == 1) else rank),
                       visible_every=max(1, args.match_every))
    frames = [scene.frame(t) for t in range(scene.n_frames)]
    cfg = bench_config(pkg, scene)
    stream = torch.cuda.current_stream()
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def new_filter(attach=True):
        f = pkg.VSlamFilter(cfg, feature_capacity=nfeat + 4, device=local)
        f.set_stream(stream.cuda_stream)
        f.set_symmetric_downdate(not args.full_square)
        added = seed_filter(f, scene)
        assert added == nfeat, f"seeded {added} of {nfeat}"
        if partitioned and attach:
            pkg.dist.attach_row_partition(f, dist, torch.device("cuda", local))
        return f

    # ---- parity probe at this configuration ------------------------------------------------------
    parity = None
    if with_parity:
        if nfeat <= 600:
            if rank == 0:
                parity = parity_vs_oracle(pkg, scene, cfg, new_filter, nfeat)
                log(f"[{workload}] parity probe: {parity}")
        else:
            filt = new_filter()
            pr = parity_vs_numpy(pkg, scene, cfg, filt, nfeat)     # collective when partitioned
            del filt
            if partitioned:
                dig = torch.tensor(list(state_digest(pr["mu1"], pr["S1"])), dtype=torch.uint8, device="cuda")
                parts = [torch.empty_like(dig) for _ in range(world)]
                dist.all_gather(parts, dig)
                identical = all(bool(torch.equal(parts[0], p)) for p in parts)
            if rank == 0:
                parity = pr["finish"]()
                if partitioned:
                    from helpers import relerr
                    g1 = new_filter(attach=False)                  # the same frame on ONE GPU, un-partitioned
                    g1.captureNewFrame(scene.frame(1), scene.stamps[1]); g1.predict(); g1.update(scene.picks(1, nfeat))
                    m1, S1 = g1.get_full()
                    del g1
                    parity["replicas_bit_identical"] = bool(identical)
                    parity["vs_single_gpu_mu_rel"] = float(relerr(pr["mu1"], m1))
                    parity["vs_single_gpu_sigma_rel"] = float(relerr(pr["S1"], S1))
                    parity["ok"] = bool(parity["ok"] and identical and parity["vs_single_gpu_sigma_rel"] <= 1e-10
                                        and parity["vs_single_gpu_mu_rel"] <= 1e-10)
                log(f"[{workload}] parity probe: {parity}")
            del pr
        ctx_barrier(ctx)

    def timed_pass(step_fn, filt, profile=False):
        times = []
        for t in range(1, 1 + Wm):
            step_fn(filt, t)
        torch.cuda.synchronize()
        if profile:
            filt.set_profiling(True); filt.profile(reset=True)
        l0 = filt.stats().kernel_launches
        ctx_barrier(ctx)
        for t in range(1 + Wm, 1 + Wm + K):
            flush_buf.fill_(t & 255)  # L2 flush, outside the event pair
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            step_fn(filt, t)
            e1.record(stream)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        ctx_barrier(ctx)
        launches = filt.stats().kernel_launches - l0
        prof = filt.profile(reset=True) if profile else None
        if profile:
            filt.set_profiling(False)
        return np.array(times), launches, prof

    dev_frames = [torch.from_numpy(f).cuda() for f in frames]
    picks = [scene.picks(t, nfeat) for t in range(scene.n_frames)]

    def step_resident(f, t):
        f.captureNewFrame_device(dev_frames[t].data_ptr(), width, height, width, scene.stamps[t])
        f.predict()
        f.update(picks[t])

    pinned = [torch.from_numpy(f).pin_memory() for f in frames]
    last = {}

    def step_e2e(f, t):
        f.captureNewFrame(pinned[t].numpy(), scene.stamps[t])   # H2D inside the step
        f.predict()
        f.update(picks[t])                                       # D2H of the packed step record inside
        last["state"] = f.getState(); last["sigma"] = f.getSigma()  # accessors the ROS node reads

    # one sampler (rank 0's GPU) running through BOTH timed passes, so that neither is penalised against the other
    sampler = ClockSampler(local, enabled=(with_clocks and rank == 0))
    sampler.start()
    # ---- pass A: frames resident in HBM ---------------------------------------------------------
    filt = new_filter()
    tA, launches, _ = timed_pass(step_resident, filt)          # the reported value: no per-kernel events in the stream
    stA = filt.stats()
    n_end = filt.state_dim()
    dist_bytes_A = filt.dist_info()["allgather_bytes"] if partitioned else 0
    if dump_dir:
        outputs = filter_outputs(filt)          # every rank: reading a row-partitioned filter is collective
        if rank == 0:
            dump_outputs(dump_dir, outputs)
        del outputs
    del filt
    # ---- pass B: end to end through the public API with host buffers -----------------------------
    filt = new_filter()
    tB, _, _ = timed_pass(step_e2e, filt)
    peer_memory = bool(filt.dist_info()["peer_memory"]) if partitioned else False
    del filt
    clocks = sampler.stop()
    # ---- profiled pass: the same sequence with CUDA-event brackets per kernel class ---------------
    filt = new_filter()
    tP, _, prof = timed_pass(step_resident, filt, profile=True)
    n_state = filt.state_dim()
    assert n_state == n_end == 14 + 6 * nfeat, f"map changed size during the run: {n_end} / {n_state}"
    # the same downdate launch timed ALONE (CUDA events, this run, not under a profiler): what the kernel does when V, Gx and the
    # correction GEMM are not sharing the fp64 pipe with it — reported beside the in-step figure, never instead of it
    alone_ms = None
    if not partitioned:
        try:
            alone_ms = filt.debug_time_downdate(20)
        except Exception as ex:   # diagnostic only
            sys.stderr.write(f"debug_time_downdate: {ex}\n")
    del filt
    h2d = width * height + 4 * nfeat
    d2h = 210 * 8 + (16 + 3 * nfeat) * 4 + 2 * 88 + 14 * 8 + 196 * 8

    totA, totB = ctx_max(ctx, tA.sum()), ctx_max(ctx, tB.sum())
    nfil = 1 if partitioned else world   # partitioned: all ranks step the same filter
    value = nfil * K / (totA / 1e3)
    e2e_value = nfil * K / (totB / 1e3)
    if rank != 0:
        return None
    gemm_ms, gemm_launches = prof["downdate_gemm"]
    ub = int(pkg.lib().ekf_update_block_rows()) if hasattr(pkg.lib(), "ekf_update_block_rows") else 128
    # algorithmic flops of one rank-`ub` downdate launch: 2 n^2 k for the full square, n (n + tile) k when only tiles
    # touching the lower triangle are computed (SURVEY.md 8(d) K4d, SYRK form)
    flops_per_launch = 2.0 * n_state * n_state * ub if args.full_square else 1.0 * n_state * (n_state + 128) * ub
    if partitioned:   # a rank downdates its row block over all columns
        r0, r1, _ = pkg.dist.row_block(rank, world, n_state)
        flops_per_launch = 2.0 * (r1 - r0) * n_state * ub
    peak = dgemm_peak_tflops(torch)
    achieved = flops_per_launch * gemm_launches / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tfile = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tfile) and workload.startswith("cfg2"):
        try:
            tj = json.load(open(tfile))
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = "static: " + tj.get("source", "ncu --set full capture committed under profiles/ (not measured in this run)")
        except Exception:
            traffic = None
    ms_per_step = totA / K
    out = {
        "metric": metric_for(workload), "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong" if partitioned else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(workload, args.match_every),
                   "l2": "flushed between timed steps (256 MiB write outside the event pairs)",
                   "multi_gpu": ("one filter, stacked update partitioned by covariance row blocks, look-ahead pipeline; partial S blocks "
                                 "and V panels exchanged " + ("by peer-memory stores from inside the producing kernels (NVLink)"
                                                              if peer_memory else "by NCCL all-reduce / all-gather")
                                 + ", row blocks of Sigma all-gathered by NCCL once per update (strong scaling)") if partitioned else
                                ("replicas only (one independent filter per rank)" if world > 1 else "n/a")},
        "run": {"n_state": int(n_state), "n_li_last_step": int(stA.n_li), "downdate": "full square" if args.full_square else "lower triangle + mirror"},
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": {"kernel": f"k_gemm_nt_sub (Sigma -= V V^T, DMMA.8x8x4, K={ub} per launch, "
                               + ("rank 0's row block x all columns" if partitioned else
                                  ("full square" if args.full_square else "lower-triangle tiles + mirror")) + ")", "bound": "tensor",
                     "achieved": round(achieved, 3), "peak": round(peak, 2), "unit": "TFLOP/s",
                     "frac": round(achieved / peak, 4) if peak > 0 else None, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": "cuBLAS DGEMM 4096^3 measured in this run (MEASURED_PEAKS.json has no fp64 entry; "
                                    "DMMA issue peak measured by tools/fp64_probe: 37.05 TFLOP/s)",
                     "flops_per_launch": flops_per_launch, "launches": int(gemm_launches),
                     "avg_launch_ms": round(gemm_ms / max(gemm_launches, 1), 5),
                     "kernel_alone": ({"avg_launch_ms": round(alone_ms, 5), "achieved": round(flops_per_launch / (alone_ms / 1e3) / 1e12, 3),
                                       "frac": round(flops_per_launch / (alone_ms / 1e3) / 1e12 / peak, 4),
                                       "note": "same launch, 20 back-to-back repetitions alone on the stream (L2-warm), CUDA events; "
                                               "inside the step V_b, Gx and the correction GEMM share the fp64 pipe with it"}
                                      if alone_ms and peak > 0 else None),
                     "share_of_step": round(gemm_ms / K / ms_per_step, 4),
                     "step_flops_frac_of_peak": round(flops_per_launch * gemm_launches / K / (ms_per_step / 1e3) / 1e12 / peak, 4)},
        "kernel_ms_per_step": {k: round(v[0] / K, 5) for k, v in prof.items() if v[1] > 0 or v[0] > 0},
        "profiled_pass_ms_per_step": round(float(tP.mean()), 4),
    }
    if clocks is not None:
        out["clocks"] = clocks
    if parity is not None:
        out["parity"] = parity
    if partitioned:
        out["exchange_bytes_per_step"] = int(dist_bytes_A / max(K + Wm, 1))
    if world == 1 and with_cpu and not args.no_cpu_baseline:
        if nfeat > 600:
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                   "sample": "not run: one dense reference frame at n = 12014 is ~2.8e13 flops (minutes per frame); "
                                             "see the cfg2 line for the measured CPU baseline"}
        else:
            out["cpu_baseline"] = cpu_baseline(pkg, workload, budget_s=args.cpu_budget)
            out["cpu_baseline"]["single_thread"] = cpu_baseline_single_thread(pkg, workload, budget_s=args.cpu_budget / 2)
    return out


# ------------------------------------------------------------------------------------------------
# cfg5: the stateless batched matcher
# ------------------------------------------------------------------------------------------------
def _dp4a_pipe(delta, n_features, ms, clocks):
    """DP4A warp-instructions the tile matcher issues per launch over the pipe's measured rate (tools/idp_rate_probe: 2 per cycle per SM,
    shared with IMAD): 864 per 4x4-candidate tile (528 for the dot products + 336 for the window sums), tiles round-robin over 32 lanes."""
    side = 2 * delta + 1
    tiles = ((side + 3) // 4) ** 2
    rounds = (tiles + 31) // 32
    per_feature = 864 * rounds
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 2.0 * 148 * mhz * 1e6
    ach = per_feature * n_features / (ms / 1e3)
    return {"warp_instr_per_feature": per_feature, "achieved_per_s": round(ach, 1), "peak_per_s": peak, "frac": round(ach / peak, 4)}


def bench_match(args, ctx, workload, K, Wm, dump_dir=None):
    """BASELINE configs[4]: the stateless batched matcher (ekf_match_batch), frames sharded across ranks."""
    torch, dist, rank, world, local = ctx.torch, ctx.dist, ctx.rank, ctx.world, ctx.local
    import ekfb200
    pkg = ekfb200.load_package()
    pkg.lib()
    M, width, height = WORKLOADS[workload]
    F = args.frames
    w = 11
    d = pkg.synth.match_batch_inputs(n_frames=F, features_per_frame=M, width=width, height=height, window=w, seed=1239 + rank)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream()
    host = {k: torch.from_numpy(np.ascontiguousarray(d[k])).pin_memory() for k in ("frames", "templates", "h", "S")}
    res = {k: host[k].to(dev) for k in host}
    uv = torch.zeros((F * M, 2), dtype=torch.int32, device=dev); sc = torch.zeros(F * M, dtype=torch.float32, device=dev)
    uv_h = torch.zeros((F * M, 2), dtype=torch.int32).pin_memory(); sc_h = torch.zeros(F * M, dtype=torch.float32).pin_memory()

    def launch(t):
        pkg.match_batch(t["frames"].data_ptr(), F, width, height, width, t["templates"].data_ptr(), M, w, t["h"].data_ptr(),
                        t["S"].data_ptr(), uv.data_ptr(), sc.data_ptr(), sigma_size=3.0, stream=stream.cuda_stream)

    def step_resident():
        launch(res)

    stage = {k: torch.empty_like(res[k]) for k in res}

    def step_e2e():
        for k in stage:
            stage[k].copy_(host[k], non_blocking=True)          # H2D inside the step
        launch(stage)
        uv_h.copy_(uv, non_blocking=True); sc_h.copy_(sc, non_blocking=True)   # D2H inside the step

    def timed(fn):
        for _ in range(Wm):
            fn()
        ctx_barrier(ctx)
        ts = []
        for _ in range(K):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream); fn(); e1.record(stream)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ctx_barrier(ctx)
        return np.array(ts)

    sampler = ClockSampler(local, enabled=(rank == 0))
    sampler.start()
    tA = timed(step_resident)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"uv": uv.cpu().numpy(), "score": sc.cpu().numpy()})
    tB = timed(step_e2e)
    clocks = sampler.stop()
    found = int((uv_h[:, 0] >= 0).sum())
    assert np.array_equal(uv_h.numpy()[uv_h.numpy()[:, 0] >= 0], d["truth"][uv_h.numpy()[:, 0] >= 0]), "matches differ from the planted truth"
    totA, totB = ctx_max(ctx, tA.sum()), ctx_max(ctx, tB.sum())
    if rank != 0:
        return None
    hbm_peak, peak_src = hbm_peak_gbs()
    delta = 12  # 3 sigma of S = diag(16,16)
    win_bytes = (2 * delta + w) * (2 * delta + w) + w * w + 16 + 32 + 12
    bytes_per_launch = float(win_bytes) * F * M
    ms = float(tA.mean())
    cand = 3.14159 * delta * delta            # in-ellipse candidates per feature
    out = {"metric": METRIC_MATCH, "value": round(world * F * M * K / (totA / 1e3), 1), "unit": UNIT_MATCH, "n_gpus": world,
           "steps": K, "warmup": Wm, "ms_per_step": round(totA / K, 4), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": f"{workload}: {F} frames {width}x{height} u8 per GPU x {M} features, 11x11 templates, "
                                  f"S = diag(16,16) +- 10 % => ~{cand:.0f} in-ellipse candidates per feature; {found} of {F * M} accepted",
                      "l2": f"inputs larger than L2 ({F * width * height / 1e6:.0f} MB of frames)",
                      "multi_gpu": "sharded by frame, no collective" if world > 1 else "n/a"},
           "e2e": {"value": round(world * F * M * K / (totB / 1e3), 1), "unit": UNIT_MATCH,
                   "h2d_bytes_per_step": int(sum(host[k].numel() * host[k].element_size() for k in host)),
                   "d2h_bytes_per_step": int(uv_h.numel() * 4 + sc_h.numel() * 4)},
           "gpu_launches": 2 * K, "clocks": clocks,   # k_match_batch_warp2 + k_match_batch_marked per call
           "parity": {"against": "planted ground-truth coordinates of the synthetic frames (every accepted match must equal them); "
                                 "bit-exact oracle comparison in tests/test_gpu_match_batch.py", "ok": True},
           "roofline": {"kernel": "k_match_batch_warp2 (one warp per feature, 4x4-candidate tiles scored in registers by DP4A, float "
                                  "pre-selection, exact fp64 re-score of the band; near-ties marked for k_match_batch_marked = the CTA "
                                  "matcher with TMA staging); bound by the DP4A / IMAD pipe, not HBM: see issue", "bound": "hbm",
                        "achieved": round(bytes_per_launch / (ms / 1e3) / 1e9, 2), "peak": hbm_peak, "unit": "GB/s",
                        "frac": round(bytes_per_launch / (ms / 1e3) / 1e9 / hbm_peak, 5), "traffic": None,
                        "peak_source": peak_src, "bytes_per_launch": bytes_per_launch,
                        "avg_launch_ms": round(ms, 4), "share_of_step": 1.0,
                        "issue": {"candidates_per_launch": cand * F * M,
                                  "ns_per_candidate": round(ms * 1e6 / (cand * F * M), 4),
                                  "dp4a_pipe": _dp4a_pipe(delta, F * M, ms, clocks),
                                  "note": "every candidate costs an 11x11 u8 dot product (33 DP4A) + 21 DP4A of window sums per 4x4 "
                                          "tile row; only the band candidates are re-scored in fp64"}}}
    if world == 1 and not args.no_cpu_baseline:
        import orc
        orc.build()
        nf = 2
        t0 = time.perf_counter()
        orc.lib(omp=True).orc_set_num_threads(os.cpu_count() or 1)
        orc.match_batch(d["frames"][:nf], d["templates"][:nf * M], d["h"][:nf * M], d["S"][:nf * M], sigma_size=3.0, omp=True)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": round(nf * M / dt, 1), "unit": UNIT_MATCH, "cores": orc.lib(omp=True).orc_num_threads(), "kind": "port",
                               "sample": f"{nf} frames x {M} features through the oracle's Patch::findMatch (OpenMP over features), {dt:.2f} s"}
    return out


# ------------------------------------------------------------------------------------------------
# cfg3: batch of independent filters, sharded by filter
# ------------------------------------------------------------------------------------------------
def bench_batch(args, ctx, workload, K, Wm, with_cpu=True, with_clocks=True, with_parity=True, dump_dir=None):
    """BASELINE configs[2]: a Monte-Carlo ensemble of independent filters, sharded by filter across
    ranks with no data-path collective (weak scaling: BATCH_FILTERS filters per GPU)."""
    torch, dist, rank, world, local = ctx.torch, ctx.dist, ctx.rank, ctx.world, ctx.local
    import ekfb200
    pkg = ekfb200.load_package()
    pkg.lib()
    B = args.filters
    nfeat, width, height = WORKLOADS[workload]
    scene = make_scene(pkg, workload, 1 + Wm + K, seed=1235)
    frames = [scene.frame(t) for t in range(scene.n_frames)]
    cfg = bench_config(pkg, scene)
    stream = torch.cuda.current_stream()

    def new_batch(keep_seed=False):
        f = pkg.VSlamFilter(cfg, feature_capacity=nfeat + 2, device=local)
        added = seed_filter(f, scene)
        assert added == nfeat
        b = pkg.FilterBatch(cfg, B, feature_capacity=nfeat + 2, device=local)
        b.set_stream(stream.cuda_stream)
        b.seed_from(f)
        # per-hypothesis perturbation of the camera state: filters [rank*B, (rank+1)*B) of the ensemble
        b.set_camera_states(pkg.dist.ensemble_camera_states(f.getState(), pkg.dist.ensemble_slice(rank, world, B)))
        if keep_seed:
            return b, f
        del f
        return b

    picks = [scene.picks(t, nfeat) for t in range(scene.n_frames)]

    parity = None
    if with_parity and rank == 0:
        import orc
        from helpers import relerr
        orc.build()
        t0 = time.perf_counter()
        batch, seedf = new_batch(keep_seed=True)
        probe = sorted({0, B // 2, B - 1})
        oracles = []
        for fidx in probe:
            o = orc.OracleFilter(cfg, kind=0, omp=False)
            o.captureNewFrame(scene.frame(0), scene.stamps[0])
            o.import_from(seedf)
            mu, S = batch.get_full(fidx)
            o.set_full(mu, S)
            oracles.append(o)
        batch.captureNewFrame(frames[1], scene.stamps[1]); batch.step(picks[1])
        em = es = 0.0
        teq = True
        for fidx, o in zip(probe, oracles):
            o.captureNewFrame(frames[1], scene.stamps[1]); o.predict(); o.update(picks[1])
            mg, Sg = batch.get_full(fidx); mo, So = o.get_full()
            if mg.shape != mo.shape:
                teq = False
                continue
            em = max(em, float(relerr(mg, mo))); es = max(es, float(relerr(Sg, So)))
            for i in range(o.numOfFeatures()):
                a, b_ = batch.feature(fidx, i), o.feature(i)
                teq = teq and all(getattr(a, k) == getattr(b_, k) for k in ("is_in_innovation", "is_in_li", "is_in_hi", "n_tot", "n_find"))
                teq = teq and tuple(a.center) == tuple(b_.center)
        parity = {"against": f"CPU oracle on filters {probe} of the ensemble (dense reference algebra)", "frames": 1,
                  "n": int(batch.state_dim(0)), "mu_rel": em, "sigma_rel": es, "tables_equal": bool(teq), "tol": PARITY_TOL,
                  "ok": bool(teq and em <= PARITY_TOL and es <= PARITY_TOL), "seconds": round(time.perf_counter() - t0, 1)}
        log(f"[{workload}] parity probe: {parity}")
        del batch, seedf, oracles
    ctx_barrier(ctx)

    def timed(step_fn, batch):
        times, cls = [], {"predict": 0.0, "match": 0.0, "update": 0.0}
        for t in range(1, 1 + Wm):
            step_fn(batch, t)
        torch.cuda.synchronize()
        l0 = batch.kernel_launches()
        ctx_barrier(ctx)
        for t in range(1 + Wm, 1 + Wm + K):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            step_fn(batch, t)
            e1.record(stream)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
            for k, v in batch.last_step_ms().items():
                cls[k] += v
        ctx_barrier(ctx)
        return np.array(times), batch.kernel_launches() - l0, {k: v / K for k, v in cls.items()}

    dev_frames = [torch.from_numpy(f).cuda() for f in frames]

    def step_resident(b, t):
        b.captureNewFrame_device(dev_frames[t].data_ptr(), width, height, width, scene.stamps[t])
        b.step(picks[t])

    pinned = [torch.from_numpy(f).pin_memory() for f in frames]
    last = {}

    def step_e2e(b, t):
        b.captureNewFrame(pinned[t].numpy(), scene.stamps[t])   # H2D inside the step
        b.step(picks[t])                                        # D2H of camera states + counters inside
        last["mu"], last["st"] = b.camera_states()

    sampler = ClockSampler(local, enabled=(with_clocks and rank == 0))
    sampler.start()
    batch = new_batch()
    tA, launches, cls = timed(step_resident, batch)
    mu14, st = batch.camera_states()
    if dump_dir and rank == 0:
        _, sigma14, _ = batch.camera_states(want_sigma=True)
        dump_outputs(dump_dir, {"camera_states": mu14, "camera_sigma": sigma14, "step_counters": st})
    n_state = batch.state_dim(0)
    n_min = min(batch.state_dim(i) for i in (0, B // 2, B - 1))
    li_mean = float(st[:, 2].mean())
    del batch
    batch = new_batch()
    tB, _, _ = timed(step_e2e, batch)
    del batch
    clocks = sampler.stop()
    h2d = width * height + 4 * nfeat
    d2h = B * 14 * 8 + B * 8 * 4
    totA, totB = ctx_max(ctx, tA.sum()), ctx_max(ctx, tB.sum())
    all_cams = pkg.dist.gather_camera_states(last["mu"], dist, "cuda")   # reporting only (SURVEY.md 8(e))
    assert all_cams.shape == (world * B, 14) and np.isfinite(all_cams).all()
    if rank != 0:
        return None
    hbm_peak, peak_src = hbm_peak_gbs()
    # k_batch_update: algorithmic bytes = read + write of every filter's covariance (SURVEY.md 8(d): 16 n^2)
    bytes_per_launch = 16.0 * n_state * n_state * B
    upd_ms = cls["update"]
    achieved = bytes_per_launch / (upd_ms / 1e3) / 1e9 if upd_ms > 0 else 0.0
    out = {
        "metric": METRIC_BATCH, "value": round(world * B * K / (totA / 1e3), 1), "unit": UNIT_BATCH, "n_gpus": world, "steps": K,
        "warmup": Wm, "ms_per_step": round(totA / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{workload}: {B} independent filters per GPU x {nfeat} inverse-depth features (n={14 + 6 * nfeat}), "
                               f"one shared {width}x{height} u8 frame per step, predict+match+update per filter, maps held at N features",
                   "l2": f"inputs larger than L2 ({B * n_state * n_state * 8 / 1e6:.0f} MB of covariance per step vs 126 MB)",
                   "multi_gpu": "sharded by filter, no data-path collective" if world > 1 else "n/a",
                   "filters_per_gpu": B},
        "run": {"n_state": int(n_state), "n_state_min_probe": int(n_min), "mean_n_li": round(li_mean, 2)},
        "e2e": {"value": round(world * B * K / (totB / 1e3), 1), "unit": UNIT_BATCH, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "k_batch_update (one CTA per filter: RANSAC, W = Sigma H^T, Cholesky gain, DMMA downdate from smem)",
                     "bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(achieved / hbm_peak, 4), "traffic": None,
                     "peak_source": peak_src, "bytes_per_launch": bytes_per_launch,
                     "avg_launch_ms": round(upd_ms, 4), "share_of_step": round(upd_ms / (totA / K), 4)},
        "kernel_ms_per_step": {k: round(v, 4) for k, v in cls.items()},
    }
    if clocks is not None:
        out["clocks"] = clocks
    if parity is not None:
        out["parity"] = parity
    tfile = os.path.join(ROOT, "profiles", "batch_update_traffic.json")
    if os.path.exists(tfile):
        try:
            tj = json.load(open(tfile))
            out["roofline"]["traffic"] = tj.get("dram_bytes_per_launch")
            out["roofline"]["traffic_source"] = "static: ncu --set full capture committed under profiles/ (not measured in this run)"
        except Exception:
            pass
    if world == 1 and with_cpu and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_batch(pkg, workload, budget_s=args.cpu_budget)
    return out


# ------------------------------------------------------------------------------------------------
# CPU baselines (the oracle = restatement of the reference's dense algebra; never the product path)
# ------------------------------------------------------------------------------------------------
def cpu_baseline_batch(pkg, workload, budget_s=20.0):
    """The oracle (dense reference algebra) on a bounded sample of the ensemble: filters are
    independent, so they are spread over the host cores with one oracle filter per thread."""
    import concurrent.futures as cf
    import orc
    orc.build()
    nfeat = WORKLOADS[workload][0]
    scene = make_scene(pkg, workload, 3)
    cfg = bench_config(pkg, scene)
    cores = os.cpu_count() or 1

    def one(_):
        o = orc.OracleFilter(cfg, kind=0, omp=False)
        seed_filter(o, scene)
        t0 = time.perf_counter()
        n = 0
        for t in (1, 2):
            o.captureNewFrame(scene.frame(t), scene.stamps[t]); o.predict(); o.update(scene.picks(t, nfeat))
            n += 1
        return n, time.perf_counter() - t0

    nfil = max(cores, 8)
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(max_workers=cores) as ex:   # ctypes releases the GIL inside the oracle calls
        res = list(ex.map(one, range(nfil)))
    wall = time.perf_counter() - t0
    steps = sum(r[0] for r in res)
    busy = sum(r[1] for r in res)
    return {"value": round(steps / (busy / cores), 3), "unit": UNIT_BATCH, "cores": cores, "kind": "port",
            "sample": f"{nfil} filters x 2 steps of {workload} on {cores} threads (one oracle filter per thread, dense reference "
                      f"algebra, fp64), {busy / steps * 1e3:.1f} ms per filter-step per core, wall {wall:.1f} s incl. seeding"}


def _oracle_seeded(pkg, orc, workload, n_frames, omp=True, kind=0, nfeat=None):
    """An oracle filter holding the workload's seeded map, seeded by the oracle's OWN addFeature (the sparsity-exploiting
    bulk form, bit-identical to the reference's dense per-feature calls): the CUDA library is not involved."""
    scene = make_scene(pkg, workload, n_frames)
    if nfeat is not None and nfeat != scene.n_features:
        W, H = WORKLOADS[workload][1:]
        scene = pkg.synth.Scene(n_features=nfeat, width=W, height=H, n_frames=n_frames, seed=1235, speed=0.1, omega=0.02,
                                accel_sigma=0.002, border=44, depth_range=BENCH_DEPTH_RANGE)
    cfg = bench_config(pkg, scene)
    o = orc.OracleFilter(cfg, kind=kind, omp=omp)
    added = seed_filter(o, scene)
    assert added == scene.n_features
    return o, scene


def cpu_baseline(pkg, workload, budget_s=30.0):
    """The oracle (dense reference algebra, vslamRansac.cpp as written) on this host's cores, on a
    bounded sample of the same workload."""
    import orc
    orc.build()
    L = orc.lib(omp=True)
    L.orc_set_num_threads(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1; the baseline uses every host core
    cores = L.orc_num_threads()
    nfeat = WORKLOADS[workload][0]
    o, scene = _oracle_seeded(pkg, orc, workload, 4)
    times = []
    t_start = time.perf_counter()
    for t in range(1, 4):
        img = scene.frame(t)
        t0 = time.perf_counter()
        o.captureNewFrame(img, scene.stamps[t]); o.predict(); o.update(scene.picks(t, nfeat))
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    per = float(np.mean(times))
    return {"value": round(1.0 / per, 5), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} frame(s) of {workload} (dense n x n algebra as the reference executes it, "
                      f"fp64, -O3 -march=x86-64-v3, OpenMP over GEMM rows), {per:.2f} s/frame"}


def cpu_baseline_single_thread(pkg, workload, budget_s=15.0):
    """BASELINE.md section 3.1 `cpu-ref-dense`: the same code built the way the reference is built (-O2 -msse4, ONE thread,
    mono-slam/CMakeLists.txt:3), Scalar = float (what the reference computes) and Scalar = double.  A dense frame at
    N = 500 costs about a minute on one thread, so the frames are MEASURED on a smaller map of the same scene family and
    scaled by the (n / n_sample)^3 law of the dense products (labelled as extrapolated)."""
    import orc
    orc.build()
    nfeat = WORKLOADS[workload][0]
    ns = min(nfeat, 150)
    n_full, n_s = 14 + 6 * nfeat, 14 + 6 * ns
    out = {"cores": 1, "kind": "port", "flags": "-O2 -msse4 -ffp-contract=off -DNDEBUG, no OpenMP (liborc.so)", "measured_at_features": ns}
    for name, kind in (("double", 2), ("float", 1)):
        o, scene = _oracle_seeded(pkg, orc, workload, 3, omp=False, kind=kind, nfeat=ns)
        ts = []
        t_begin = time.perf_counter()
        for t in (1, 2):
            img = scene.frame(t)
            t0 = time.perf_counter()
            o.captureNewFrame(img, scene.stamps[t]); o.predict(); o.update(scene.picks(t, ns))
            ts.append(time.perf_counter() - t0)
            if time.perf_counter() - t_begin > budget_s / 2:
                break
        per = float(np.min(ts))
        scale = (n_full / n_s) ** 3
        out[name] = {"s_per_frame_measured": round(per, 3), "frames": len(ts),
                     "value": round(1.0 / (per * scale), 6), "unit": UNIT,
                     "note": "measured" if ns == nfeat else f"extrapolated to N={nfeat} by (n/n_sample)^3 = {scale:.1f}"}
    return out


def run_reference(args):
    """The reference's CPU implementation of the path (the oracle port: the reference itself needs Eigen / OpenCV / ROS,
    absent here), all host threads, on the same workload.  Does not import or load the CUDA library."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import ekfb200
    pkg = ekfb200.load_package()     # pure-Python parts only (synthetic scene, config struct); lib() is never called here
    import orc
    orc.build()
    L = orc.lib(omp=True)
    L.orc_set_num_threads(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core
    cores = L.orc_num_threads()
    workload = args.workload if not args.workload.startswith(("cfg3", "cfg5")) else "cfg2_n500"
    nfeat = WORKLOADS[workload][0]
    K, Wm = args.steps, args.warmup
    budget = args.ref_budget
    o, scene = _oracle_seeded(pkg, orc, workload, 1 + Wm + K)
    t_begin = time.perf_counter()
    times = []
    done_w = 0
    for t in range(1, 1 + Wm + K):
        img = scene.frame(t)
        t0 = time.perf_counter()
        o.captureNewFrame(img, scene.stamps[t]); o.predict(); o.update(scene.picks(t, nfeat))
        dt = time.perf_counter() - t0
        if done_w < Wm:
            done_w += 1
        else:
            times.append(dt)
        if time.perf_counter() - t_begin > budget and len(times) >= 1:
            break
    per = float(np.mean(times))
    val = 1.0 / per
    out = {"impl": "reference", "metric": metric_for(workload), "value": round(val, 5), "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
           "steps": len(times), "warmup": done_w, "ms_per_step": round(per * 1e3, 2), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_string(workload, 1)},
           "run": {"n_state": int(o.state_dim()), "n_li_last_step": int(o.stats().n_li),
                   "arm": "CPU oracle of the reference's dense algebra (the reference itself needs Eigen/OpenCV/ROS, absent here), "
                          "seeded by its own addFeature; libekf_b200.so is not loaded",
                   "bounded": f"stopped after {len(times)} timed frame(s) (time budget {budget:.0f} s)"},
           "cpu_baseline": {"value": round(val, 5), "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": f"{len(times)} timed frame(s), {per:.2f} s/frame"},
           "e2e": {"value": round(val, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def sharded_summary(o):
    if o is None:
        return None
    keep = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "e2e", "kernel_ms_per_step", "parity",
            "exchange_bytes_per_step", "gpu_launches", "run")
    s = {k: o[k] for k in keep if k in o}
    s["workload"] = o["config"]["workload"]
    s["multi_gpu"] = o["config"].get("multi_gpu")
    s["roofline"] = {k: o["roofline"][k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "share_of_step") if k in o["roofline"]}
    return s


def main():
    # keep stdout to the single JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_n500", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="default workload only: skip the short cfg3 / cfg4 passes")
    ap.add_argument("--no-parity", action="store_true", help="skip the one-frame parity probe taken before the timing")
    ap.add_argument("--sharded-steps", type=int, default=6, help="timed steps of the cfg3 / cfg4 passes of the default run")
    ap.add_argument("--match-every", type=int, default=1,
                    help="single-filter workloads: only every k-th feature is visible after frame 0 (m = N / k matches per frame; "
                         "the headline uses k = 1, all features matched, the stated worst case)")
    ap.add_argument("--full-square", action="store_true", help="downdate all n x n tiles instead of lower triangle + mirror")
    ap.add_argument("--frames", type=int, default=MATCH_FRAMES, help="frames per GPU of the matcher workload")
    ap.add_argument("--filters", type=int, default=BATCH_FILTERS, help="filters per GPU of the batched workload")
    ap.add_argument("--cpu-budget", type=float, default=30.0)
    ap.add_argument("--ref-budget", type=float, default=150.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline path computed in its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    ctx = make_ctx()
    K, Wm = args.steps, max(args.warmup, 3)
    parity = not args.no_parity
    if args.workload.startswith("cfg3"):
        out = bench_batch(args, ctx, args.workload, K, Wm, with_parity=parity, dump_dir=args.dump_outputs)
    elif args.workload.startswith("cfg5"):
        out = bench_match(args, ctx, args.workload, K, Wm, dump_dir=args.dump_outputs)
    else:
        out = bench_single(args, ctx, args.workload, K, Wm, with_parity=parity, dump_dir=args.dump_outputs)
        if args.workload == "cfg2_n500" and not args.no_sharded and args.match_every <= 1:
            # the paths that shard, measured in the same run at this N (VERDICT r1 item 2)
            Ks = max(2, min(args.sharded_steps, K))
            sh = {}
            for name, fn in (("cfg3_batch4096", bench_batch), ("cfg4_n2000", bench_single)):
                t0 = time.perf_counter()
                try:
                    o = fn(args, ctx, name, Ks, 3, with_cpu=False, with_clocks=False, with_parity=parity)
                    if ctx.rank == 0:
                        sh[name] = sharded_summary(o)
                        sh[name]["wall_s"] = round(time.perf_counter() - t0, 1)
                except Exception as e:  # the headline line must still be printed
                    log(f"sharded pass {name} failed: {e!r}")
                    if ctx.rank == 0:
                        sh[name] = {"error": repr(e)}
                    if ctx.world > 1:
                        raise
            if out is not None:
                out["sharded"] = sh
    if ctx.dist is not None:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
