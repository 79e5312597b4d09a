"""-m gpu: resampling the batched filters (ekf_batch_resample, FilterBatch.resample, systematic_ancestors).

Two batches x and y run the same calls; then only x resamples.  Every filter f of x must equal filter ancestors[f] of y, bit for
bit, in everything an accessor reports, and keep equalling it when later steps give f its ancestor's controls."""
import ctypes as C

import numpy as np
import pytest

import bench
from test_gpu_batch_archive import _run_pair, _same_records
from test_gpu_batch_subset import _batches_equal, _perturbed, _row, _seed

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -1, -5


def _compare(x, y, anc, ctx, filters=None, points=True):
    """x against y[anc]: camera rows, counters, added and blur counts, archive sizes, dT; then whole filters (all, or `filters`)."""
    mx, Sx, stx = x.camera_states(want_sigma=True)
    my, Sy, sty = y.camera_states(want_sigma=True)
    assert np.array_equal(stx, sty[anc]), f"{ctx}: counters"
    assert np.array_equal(mx, my[anc]) and np.array_equal(Sx, Sy[anc]), f"{ctx}: camera rows"
    assert np.array_equal(x.last_added(), y.last_added()[anc]), f"{ctx}: added"
    assert np.array_equal(x.last_blur_counts(), y.last_blur_counts()[anc]), f"{ctx}: blur counts"
    assert np.array_equal(x.num_deleted(), y.num_deleted()[anc]), f"{ctx}: archive sizes"
    assert np.array_equal(x.getDt(), y.getDt()), f"{ctx}: dT"
    for f in (range(x.B) if filters is None else filters):
        a = int(anc[f])
        assert x.state_dim(f) == y.state_dim(a), f"{ctx} filter {f}: state dimension"
        _batches_equal(x, f, y, a, f"{ctx} filter {f} (ancestor {a})")
        if points:
            assert np.array_equal(x.getPointsFeatures(f), y.getPointsFeatures(a)), f"{ctx} filter {f}: points"


def _frames(sc, t, K):
    base = sc.frame(t).astype(np.int16)
    fr = np.stack([np.clip(base + (c % 5) * 4 - 8, 0, 255).astype(np.uint8) for c in range(K)])
    return fr, sc.stamps[t] * (1.0 + 0.01 * np.arange(K))


def _ensemble(gpu_pkg, cap, large, K=4, M=6, seed=960):
    """Twin batches of K cameras x M hypotheses: intrinsics per filter, blur, top-up, XYZ conversion and archive on, controls per
    filter.  Three steps, then removals and additions that differ per filter, then a fourth step: the filters differ in N and
    in real indices."""
    B = K * M
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=12, seed=seed, speed=0.9, omega=0.5, template_smooth=2.5)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=20, xyz_conversion=1, T_camera=0.5))
    src = _seed(gpu_pkg, cfg, sc, cap)
    cams = _perturbed(src.get_full()[0], B, 61)
    rows = np.stack([_row(cfg) * (1.0 + 2e-4 * f) for f in range(B)])
    rng = np.random.default_rng(seed)
    dv = rng.normal(scale=1e-3, size=(B, 3)); dw = rng.normal(scale=1e-3, size=(B, 3))
    vc = (np.arange(B) % 3 == 0).astype(np.int32)
    x, y = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap, large=large) for _ in range(2))
    for z in (x, y):
        z.seed_from(src); z.set_cameras(K, np.repeat(np.arange(K), M)); z.set_intrinsics(rows); z.set_camera_states(cams)
        z.set_topup(True); z.set_archive(64); z.set_motion_blur(3)
    ctl = dict(dv=dv, dw=dw, vcontrol=vc)
    for t in range(1, 5):
        fr, stamps = _frames(sc, t, K)
        for z in (x, y):
            z.captureNewFrames(fr, stamps)
            z.step(sc.picks(t, 24), **ctl)
        if t == 3:
            for f in range(B):
                for z in (x, y):
                    if f % 3 == 1:
                        z.removeFeature(f, f % z.numOfFeatures(f))
                    for k in range(f % 3 if z.numOfFeatures(f) + 2 <= cap else 0):
                        z.addFeature(f, 120.0 + 37.0 * k + 11.0 * (f % 5), 90.0 + 23.0 * k + 7.0 * (f % 4))
    N = [x.numOfFeatures(f) for f in range(B)]
    ri = [max(x.feature(f, i).real_index for i in range(N[f])) for f in range(B)]
    assert len(set(N)) > 1 and len(set(ri)) > 1, "the filters did not diverge"
    return sc, x, y, ctl


@pytest.mark.parametrize("cap,large", [(32, False), (128, True)])
def test_copies_equal_their_sources(gpu_pkg, cap, large):
    """Identities, duplicates, a swap, a 3-cycle and a filter that is both source and destination.  Right after the call and after
    findNewFeatures(None) and three more steps (x's filters given their ancestors' controls), x[f] equals y[ancestors[f]]."""
    K, M = 4, 6
    sc, x, y, ctl = _ensemble(gpu_pkg, cap, large, K, M)
    B = K * M
    anc = np.arange(B)
    anc[2] = anc[3] = 0                        # camera 0: two copies of a filter that stays
    anc[4], anc[5] = 5, 4                      # a swap
    anc[6], anc[7], anc[8] = 7, 8, 6           # camera 1: a 3-cycle
    anc[12], anc[13], anc[15] = 13, 14, 13     # camera 2: 13 is copied from and overwritten
    n0 = x.kernel_launches()
    x.resample(anc)
    assert x.kernel_launches() - n0 == 3, "stage, direct and staged launches"
    ident = np.arange(B)
    _compare(x, y, anc, "after resample")
    ax, ay = x.findNewFeatures(None), y.findNewFeatures(None)
    assert np.array_equal(ax, ay[anc]), "findNewFeatures(None)"
    _compare(x, y, anc, "after findNewFeatures(None)")
    for t in range(5, 8):
        fr, stamps = _frames(sc, t, K)
        for z in (x, y):
            z.captureNewFrames(fr, stamps)
        x.step(sc.picks(t, 24), **{k: v[anc] for k, v in ctl.items()})
        y.step(sc.picks(t, 24), **ctl)
        _compare(x, y, anc, f"step {t}")
    _, st = y.camera_states()
    assert st[:, 1].sum() > 0 and not np.array_equal(anc, ident)


def test_identity_and_untouched_filters(gpu_pkg):
    """The identity launches nothing and changes nothing.  With a partial vector every filter with ancestors[f] == f stays
    bit-identical, also when it is someone's source."""
    K, M = 3, 4
    sc, x, y, _ = _ensemble(gpu_pkg, 32, False, K, M, seed=970)
    B = K * M
    n0 = x.kernel_launches()
    x.resample(np.arange(B))
    assert x.kernel_launches() == n0
    _compare(x, y, np.arange(B), "identity")
    anc = np.arange(B)
    anc[1] = 0                 # 0 is a source and stays
    anc[5], anc[6] = 6, 7      # 6 is a source and a destination, 7 a source that stays
    anc[9], anc[10] = 10, 9    # a swap
    n0 = x.kernel_launches()
    x.resample(anc)
    assert x.kernel_launches() - n0 == 3
    fixed = np.flatnonzero(anc == np.arange(B))
    assert {0, 7} <= set(fixed.tolist())
    _compare(x, y, anc, "partial")   # fixed filters against y's own


def test_archive_overflow_travels_without_a_false_alarm(gpu_pkg):
    """Capacity-1 archives beside capacity-64 twins.  Once a filter's archive has dropped records, a filter whose archive has not
    copies it.  The next steps return EKF_OK unless a record is newly dropped, and then name the first filter that dropped one."""
    ERR_CAP = gpu_pkg._abi.EKF_ERR_CAPACITY
    anc, prev, checked = None, None, 0
    for t, rcs, errs, (small, big) in _run_pair(gpu_pkg, [1, 64]):
        assert rcs[1] == 0, f"frame {t}: {errs[1]}"
        counts = big.num_deleted().astype(np.int64)
        if anc is None:
            over = [b for b in range(4) if counts[b] > 1]
            if not over:
                continue
            s = over[0]
            rest = [b for b in range(4) if b != s]
            d = min(rest, key=lambda b: (counts[b] > 1, b))   # preferably a filter that has dropped nothing
            anc = np.arange(4)
            anc[d] = s
            for z in (small, big):
                z.resample(anc)
            _same_records(small.deleted(d), small.deleted(s), 0.0, f"frame {t}: copied archive")
            assert small.num_deleted()[d] == 1
            prev = big.num_deleted().astype(np.int64)
            continue
        new = [b for b in range(4) if counts[b] > 1 and counts[b] > prev[b]]
        if new:
            assert rcs[0] == ERR_CAP and errs[0].startswith(f"filter {new[0]}:"), (t, rcs[0], errs[0], new)
        else:
            assert rcs[0] == 0, (t, errs[0])
        prev = counts
        checked += 1
    assert anc is not None and checked > 0, "no step after an archive overflowed"


def test_large_ensemble(gpu_pkg):
    """4096 filters as 64 cameras x 64 hypotheses on the cfg3 scene; half the filters step once more on their own.  Ancestors from
    systematic_ancestors on random weights: they never alias (one launch), every camera row and a sample of whole filters equal
    y[ancestors], and so does a further step with the ancestors' controls."""
    K, M = 64, 64
    B = K * M
    sc = bench.make_scene(gpu_pkg, "cfg3_batch4096", 5)
    cfg = bench.bench_config(gpu_pkg, sc)
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    bench.seed_filter(src, sc)
    cam_of = np.repeat(np.arange(K), M)
    cams = _perturbed(src.get_full()[0], B, 81, perturb=1e-3)
    rng = np.random.default_rng(82)
    dv = rng.normal(scale=1e-3, size=(B, 3)); dw = rng.normal(scale=1e-3, size=(B, 3))
    x, y = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=32) for _ in range(2))
    for z in (x, y):
        z.seed_from(src); z.set_cameras(K, cam_of); z.set_camera_states(cams)
    half = np.flatnonzero(np.arange(B) % M < M // 2).astype(np.int32)
    for t in range(1, 4):
        fr, stamps = _frames(sc, t, K)
        for z in (x, y):
            z.captureNewFrames(fr, stamps)
            if t < 3:
                z.step(sc.picks(t, 30), dv=dv, dw=dw)
            else:
                z.step(sc.picks(t, 30), dv=dv[half], dw=dw[half], filters=half)
    w = rng.random(B) ** 4
    anc = gpu_pkg.systematic_ancestors(w, float(rng.random()), camera_of=cam_of)
    moved = np.flatnonzero(anc != np.arange(B))
    assert moved.size > B // 8
    assert not np.isin(anc[moved], moved).any(), "a source is also overwritten"
    assert np.array_equal(cam_of[anc], cam_of)
    n0 = x.kernel_launches()
    x.resample(anc)
    assert x.kernel_launches() - n0 == 1
    sample = np.concatenate([rng.choice(moved, 24, replace=False), rng.choice(np.setdiff1d(np.arange(B), moved), 8, replace=False)])
    _compare(x, y, anc, "after resample", filters=sample, points=False)
    fr, stamps = _frames(sc, 4, K)
    for z in (x, y):
        z.captureNewFrames(fr, stamps)
    x.step(sc.picks(4, 30), dv=dv[anc], dw=dw[anc])
    y.step(sc.picks(4, 30), dv=dv, dw=dw)
    _compare(x, y, anc, "step 4", filters=sample, points=False)


def test_errors_leave_the_batch_unchanged(gpu_pkg):
    sc = gpu_pkg.synth.Scene(n_features=12, n_frames=3, seed=990)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    K, M = 3, 2
    B = K * M
    fresh = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
    L = fresh.L
    ip = lambda v: (C.c_int32 * len(v))(*v)   # noqa: E731
    assert L.ekf_batch_resample(fresh.h, ip(list(range(B)))) == ERR_STATE
    assert b"seed" in L.ekf_batch_last_error(fresh.h)
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
    batch.seed_from(_seed(gpu_pkg, cfg, sc, 16))
    batch.set_cameras(K, np.repeat(np.arange(K), M))
    batch.set_archive(8)
    batch.captureNewFrames(np.stack([sc.frame(1)] * K), [sc.stamps[1]] * K)
    batch.step(sc.picks(1, 12))
    h = batch.h
    state = [(batch.get_full(f), batch.numOfFeatures(f)) for f in range(B)]
    rows = batch.camera_states(want_sigma=True)
    n0 = batch.kernel_launches()
    for bad, first in (([1, 0, 2, 3, 4, B], 5), ([0, 0, -1, 3, 4, 5], 2), ([1, 0, 2, 3, 0, 5], 4), ([0, 1, 0, 3, 4, 5], 2)):
        assert L.ekf_batch_resample(h, ip(bad)) == ERR_ARG, bad
        assert f"ancestors[{first}]".encode() in L.ekf_batch_last_error(h), (bad, L.ekf_batch_last_error(h))
    assert L.ekf_batch_resample(h, None) == ERR_ARG
    with pytest.raises(ValueError):
        batch.resample(np.arange(B - 1))
    assert batch.kernel_launches() == n0
    for f in range(B):
        (m, S), N = batch.get_full(f), batch.numOfFeatures(f)
        assert np.array_equal(m, state[f][0][0]) and np.array_equal(S, state[f][0][1]) and N == state[f][1], f"filter {f}"
    after = batch.camera_states(want_sigma=True)
    assert all(np.array_equal(a, b) for a, b in zip(rows, after))
