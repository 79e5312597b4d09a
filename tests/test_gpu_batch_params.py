"""-m gpu: batched filters with tuning of their own (ekf_batch_set_filter_params, FilterBatch.set_configs).

Filter f predicts, matches, updates, deletes, asks for features and adds them with row f of the batch's tuning table.  Every
filter still runs the single filter's algorithm, so a filter with tuning T must follow a single CUDA filter whose ekf_config
carries T: tables, NCC scores and templates bit for bit, state within 1e-8; a batch of four rigs must equal four batches
configured with those rigs bit for bit; and a table equal to the configuration is today's batch: same bits, same launches."""

import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, assert_scaled_close, relerr, seed_features
from test_gpu_batch_calib import BLUR_SCENE, RIGS, _batches_equal, _perturbed, _tables_equal

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

# The tuning of the reference's shipped configurations (mono-slam/conf/conf.cfg, conf_firewire.cfg, conf_kinect.cfg and
# conf_sim.cfg; ConfigVSLAM's defaults where a file sets nothing).  Window, scale and blur are the batch's, shared.
TUNING = {
    "conf": dict(sigma_vx=0.01, sigma_vy=0.01, sigma_vz=0.01, sigma_wx=0.005, sigma_wy=0.005, sigma_wz=0.005, rho_0=0.1,
                 sigma_rho_0=0.25, sigma_pixel=2, T_camera=0.1, min_features=30, max_features=100, sigma_size=2),
    "firewire": dict(sigma_vx=0.01, sigma_vy=0.01, sigma_vz=0.01, sigma_wx=0.005, sigma_wy=0.005, sigma_wz=0.005, rho_0=0.1,
                     sigma_rho_0=0.25, sigma_pixel=2, T_camera=0.5, min_features=20, max_features=60, sigma_size=2),
    "kinect": dict(sigma_vx=0.03, sigma_vy=0.03, sigma_vz=0.03, sigma_wx=0.015, sigma_wy=0.015, sigma_wz=0.015, rho_0=0.2,
                   sigma_rho_0=0.25, sigma_pixel=2, T_camera=0.0, min_features=100, max_features=1000, sigma_size=2),
    "sim": dict(sigma_vx=8e-7, sigma_vy=8e-7, sigma_vz=8e-11, sigma_wx=4e-9, sigma_wy=4e-7, sigma_wz=4e-11, rho_0=0.1,
                sigma_rho_0=0.25, sigma_pixel=2, T_camera=0.2, min_features=20, max_features=35, sigma_size=4),
}
CAM_KEYS = ("fx", "fy", "u0", "v0", "k1", "k2", "k3", "p1", "p2")
SIGMAS = ("sigma_vx", "sigma_vy", "sigma_vz", "sigma_wx", "sigma_wy", "sigma_wz")


def _tunings(over, M, seed, minf):
    """M tunings around `over`: every row changes several fields at once."""
    rng = np.random.default_rng(seed)
    out = []
    for m in range(M):
        t = dict(over)
        scale = float(rng.uniform(0.3, 3.0))
        for k in SIGMAS:
            t[k] = 0.01 * scale
        t.update(rho_0=(0.1, 0.2)[m % 2], sigma_rho_0=(0.25, 0.1, 0.5)[m % 3], sigma_pixel=(1, 2, 3)[m % 3],
                 sigma_size=(2, 3)[(m // 2) % 2], ncc_threshold=(0.8, 0.75, 0.85)[m % 3], quality_ratio=(0.2, 0.3)[(m // 3) % 2],
                 linearity_threshold=(0.01, 0.03, 0.005)[(m + 1) % 3], min_features=minf + (m % 3) - 1, max_features=(1000, minf + 2)[m % 2],
                 ransac_p=(0.99, 0.9)[(m // 2) % 2], ransac_nhyp0=(10000, 40)[m % 2], li_threshold_factor=(2.0, 1.5, 3.0)[m % 3],
                 hi_chi2_threshold=(1.0, 2.0)[(m // 4) % 2])
        out.append(t)
    return out


def _step_compare(gpu_pkg, batch, singles, sc, frames):
    """Steps the batch and the single filters; returns the matches over all and the templates each filter blurred."""
    matched = 0
    blurred = np.zeros(len(singles), int)
    for t in frames:
        picks = sc.picks(t, 64)
        batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(picks)
        matched += int(batch.camera_states()[1][:, 1].sum())
        counts = batch.last_blur_counts()
        for b, s in enumerate(singles):
            s.captureNewFrame(sc.frame(t), sc.stamps[t]); s.predict(); s.update(picks)
            ctx = f"frame {t} filter {b}"
            assert counts[b] == s.stats().blur_requests, f"{ctx}: blurred templates {counts[b]} vs {s.stats().blur_requests}"
            blurred[b] += int(counts[b])
            _tables_equal(batch, b, s, ctx)
            mb, Sb = batch.get_full(b); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"{ctx}: mu {relerr(mb, ms):.2e} Sigma {relerr(Sb, Ss):.2e}"
    return matched, blurred


@pytest.mark.parametrize("cap,large,nfeat,minf,blur", [(32, False, 24, 20, False), (100, True, 60, 55, False),
                                                        (32, False, 20, 16, True)])
def test_tuning_ensemble_follows_single_filters(gpu_pkg, cap, large, nfeat, minf, blur):
    """M = 8 tunings about one camera, each changing the process noise (x 0.3 to 3), the inverse-depth prior, sigma_pixel,
    sigma_size, the NCC, quality and linearity thresholds, min / max_features, the RANSAC and Hi thresholds.  From an empty
    seed, the scene's features added on frame 0 (with each filter's prior), then steps with top-up and XYZ conversion on;
    the blur case varies T_camera too.  Each filter against a single CUDA filter whose ekf_config carries its row: tables,
    NCC scores and templates bit-exact, state within 1e-8, every step."""
    sc = gpu_pkg.synth.Scene(n_features=nfeat, n_frames=11 if not blur else 7, seed=900, **(BLUR_SCENE if blur else {}))
    over = dict(sc.config_overrides(), min_features=minf, max_features=1000, xyz_conversion=1)
    if blur:
        over["kernel_size"] = 3
    M = 8
    tun = _tunings(over, M, 31, minf)
    if blur:
        for m, t in enumerate(tun):
            t["T_camera"] = (0.5, 0.2, 0.8, 0.0)[m % 4]
    cfg = gpu_pkg.default_config(**over)
    cfgs = [gpu_pkg.default_config(**t) for t in tun]
    batch = gpu_pkg.FilterBatch.from_config(cfg, M, feature_capacity=cap, large=large)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=cap))
    batch.set_configs(cfgs)
    batch.set_topup(True)
    singles = [gpu_pkg.VSlamFilter(c, feature_capacity=cap) for c in cfgs]
    batch.captureNewFrame(sc.frame(0), sc.stamps[0])
    for b, s in enumerate(singles):
        s.captureNewFrame(sc.frame(0), sc.stamps[0])
        for u, v in sc.feature_pixels:
            assert batch.addFeature(b, u, v) == 1 and s.addFeature(u, v) == 1
        _tables_equal(batch, b, s, f"frame 0 filter {b}")
        assert np.array_equal(batch.get_full(b)[1], s.get_full()[1]), f"frame 0 filter {b}: prior"
    matched, blurred = _step_compare(gpu_pkg, batch, singles, sc, range(1, sc.n_frames))
    assert matched > 0
    if blur:   # templates were blurred, and how many follows each filter's T_camera (0 blurs none)
        assert blurred.sum() > 0, f"blurred {blurred}"
        assert len(set(blurred.tolist())) > 1, f"blurred {blurred}"
        assert all(blurred[m] == 0 for m in range(M) if tun[m]["T_camera"] == 0.0), f"blurred {blurred}"
    # the rows took effect: filters that started from one state now disagree
    assert not np.array_equal(batch.get_full(0)[1], batch.get_full(1)[1])


@pytest.mark.parametrize("blur,plane", [(False, False), (True, False), (False, True)])
def test_shipped_configurations_are_separate_batches(gpu_pkg, blur, plane):
    """K = 4 rigs with the shipped tunings and calibrations (one shared window), each scene rendered with its camera model,
    M = 4 perturbed hypotheses each, in one batch of 4 cameras given the rigs' configurations by set_configs, against four
    one-camera batches built from those configurations.  mu, Sigma, tables, templates and counters bit-identical every step."""
    names = list(RIGS)
    K, M = len(names), 4
    extra = BLUR_SCENE if blur else {}
    scenes = [gpu_pkg.synth.Scene(n_features=20, n_frames=7, seed=920 + c, window=11,
                                  camera=gpu_pkg.synth.Camera(*RIGS[n]), **extra) for c, n in enumerate(names)]
    shared = dict(kernel_size=3 if blur else 1000000000, forsePlane=int(plane), xyz_conversion=1)
    cfgs = [gpu_pkg.default_config(**dict(sc.config_overrides(), **TUNING[n], **shared)) for sc, n in zip(scenes, names)]

    def make(cfg, n):
        b = gpu_pkg.FilterBatch.from_config(cfg, n, feature_capacity=32)
        b.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=32))
        return b
    grouped = make(cfgs[0], K * M)
    camera_of = np.repeat(np.arange(K), M)
    grouped.set_cameras(K, camera_of)
    grouped.set_configs([cfgs[c] for c in camera_of])
    parts = [make(c, M) for c in cfgs]
    grouped.captureNewFrames(np.stack([sc.frame(0) for sc in scenes]), [sc.stamps[0] for sc in scenes])
    for c, (p, sc) in enumerate(zip(parts, scenes)):
        p.captureNewFrame(sc.frame(0), sc.stamps[0])
        for m in range(M):
            for u, v in sc.feature_pixels:
                assert grouped.addFeature(c * M + m, u, v) == 1 and p.addFeature(m, u, v) == 1
    cams = _perturbed(grouped.get_full(0)[0], K * M, 9)
    grouped.set_camera_states(cams)
    for c, p in enumerate(parts):
        p.set_camera_states(cams[c * M:(c + 1) * M])
    matched = np.zeros(K, int)
    topup = np.zeros(K, int)
    blurred = np.zeros(K, int)
    for t in range(1, 7):
        picks = scenes[0].picks(t, 24)
        grouped.captureNewFrames(np.stack([sc.frame(t) for sc in scenes]), [sc.stamps[t] for sc in scenes])
        grouped.step(picks)
        _, stg = grouped.camera_states()
        for c, (p, sc) in enumerate(zip(parts, scenes)):
            p.captureNewFrame(sc.frame(t), sc.stamps[t]); p.step(picks)
            _, stp = p.camera_states()
            assert np.array_equal(stg[c * M:(c + 1) * M], stp), f"frame {t} rig {names[c]}: counters"
            if blur:
                assert np.array_equal(grouped.last_blur_counts()[c * M:(c + 1) * M], p.last_blur_counts())
                blurred[c] += int(p.last_blur_counts().sum())
            for m in range(M):
                _batches_equal(grouped, c * M + m, p, m, f"frame {t} rig {names[c]} hypothesis {m}")
            matched[c] += int(stp[:, 1].sum())
            topup[c] = int(stp[0, 7])
    assert (matched > 0).all(), f"matches per rig {matched}"
    if blur:   # kinect's T_camera is 0: it blurs nothing, the others blur some templates
        assert blurred[names.index("kinect")] == 0 and blurred.sum() > 0, f"blurred per rig {blurred}"
    # the rigs visibly diverge: different top-up requests (min_features) and different covariances from one perturbed start
    assert len(set(topup.tolist())) > 1, f"top-up requests {topup}"
    S = [grouped.get_full(c * M)[1][:13, :13] for c in range(K)]
    assert all(not np.array_equal(S[0], S[c]) for c in range(1, K))


def test_tunings_against_oracle(gpu_pkg, orc):
    """Three filters with three tunings on one camera.  Each step from identical inputs (batch state <- oracle state) against an
    oracle built with that filter's configuration: counters and tables bit-exact, state within TOL and the scaled bars."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=940)
    over = dict(sc.config_overrides(), xyz_conversion=0)
    tun = [dict(over), dict(over, sigma_vx=0.03, sigma_vy=0.03, sigma_vz=0.03, sigma_wx=0.015, sigma_wy=0.015, sigma_wz=0.015,
                            sigma_pixel=3, li_threshold_factor=1.5, sigma_size=3, ncc_threshold=0.75),
           dict(over, sigma_vx=0.004, sigma_vy=0.004, sigma_vz=0.004, sigma_wx=0.004, sigma_wy=0.004, sigma_wz=0.004, sigma_pixel=1,
                hi_chi2_threshold=3.0, ransac_p=0.9, quality_ratio=0.5)]
    cfgs = [gpu_pkg.default_config(**t) for t in tun]
    B = 3
    batch = gpu_pkg.FilterBatch(cfgs[0], B, feature_capacity=32)
    batch.seed_from(gpu_pkg.VSlamFilter(cfgs[0], feature_capacity=32))
    batch.set_configs(cfgs)
    batch.captureNewFrame(sc.frame(0), sc.stamps[0])
    oracles = []
    for b, cfg in enumerate(cfgs):
        for p in sc.feature_pixels:
            assert batch.addFeature(b, *p) == 1
        o = orc.OracleFilter(cfg, kind=0, omp=False)
        seed_features(o, sc)
        oracles.append(o)
    for t in range(1, sc.n_frames):
        picks = sc.picks(t, 20)
        for b, o in enumerate(oracles):
            assert batch.numOfFeatures(b) == o.numOfFeatures(), f"frame {t} filter {b}: feature count"
            batch.set_full(b, *o.get_full())
        batch.captureNewFrame(sc.frame(t), sc.stamps[t])
        batch.step(picks)
        _, _, st = batch.camera_states(want_sigma=True)
        for b, o in enumerate(oracles):
            ctx = f"frame {t} tuning {b}"
            o.captureNewFrame(sc.frame(t), sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert (st[b, 1], st[b, 2], st[b, 3], st[b, 4], st[b, 6]) == \
                (so.n_matched, so.n_li, so.n_hi, so.ransac_hypotheses, so.n_removed), f"{ctx}: counters {st[b]}"
            assert so.n_matched > 0, f"{ctx}: nothing matched"
            assert batch.numOfFeatures(b) == o.numOfFeatures(), f"{ctx}: feature count"
            mg, Sg = batch.get_full(b); mo, So = o.get_full()
            assert relerr(mg, mo) <= TOL and relerr(Sg, So) <= TOL, f"{ctx}: mu {relerr(mg, mo):.2e} Sigma {relerr(Sg, So):.2e}"
            assert_scaled_close(mg, Sg, mo, So, ctx)
            for i in range(o.numOfFeatures()):
                a, c = batch.feature(b, i), o.feature(i)
                for f in INT_FIELDS:
                    assert getattr(a, f) == getattr(c, f), f"{ctx} feature {i} {f}: {getattr(a, f)} vs {getattr(c, f)}"
                assert tuple(a.center) == tuple(c.center) and a.last_ncc == c.last_ncc, f"{ctx} feature {i} match"


def _seeded(gpu_pkg, sc, cfg, B, cap=32, seed=11):
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    cams = _perturbed(src.get_full()[0], B, seed)
    return src, cams


def test_configuration_rows_are_todays_batch(gpu_pkg):
    """No table, every row the configuration's, and a table set then cleared with None: bit-identical states and the same kernel
    launches around every capture and step, with top-up and XYZ conversion on."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=960)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=16, xyz_conversion=1))
    B = 4
    src, cams = _seeded(gpu_pkg, sc, cfg, B)
    x, y, z = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=32) for _ in range(3))
    for w in (x, y, z):
        w.seed_from(src); w.set_camera_states(cams); w.set_topup(True)
    _, rows = gpu_pkg._abi.batch_rows(cfg, [cfg] * B)
    y.set_filter_params(rows)
    z.set_configs([gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=16, xyz_conversion=1, sigma_vx=0.05, sigma_pixel=3))] * B)
    z.set_configs(None)
    for t in range(1, sc.n_frames):
        picks = sc.picks(t, 20)
        counts = []
        for w in (x, y, z):
            l0 = w.kernel_launches()
            w.captureNewFrame(sc.frame(t), sc.stamps[t])
            l1 = w.kernel_launches()
            w.step(picks)
            counts.append((l1 - l0, w.kernel_launches() - l1))
        assert counts[0] == counts[1] == counts[2], f"frame {t}: launches {counts}"
        for w in (y, z):
            assert np.array_equal(x.camera_states()[1], w.camera_states()[1])
            for b in range(B):
                _batches_equal(x, b, w, b, f"frame {t} filter {b}")


def test_interactions(gpu_pkg):
    """The tuning table against the batch's other calls, each against a reference batch: resample moves rows with filters (a
    copy given its ancestor's controls reproduces the ancestor's bits); seed_from and set_cameras keep the table;
    set_intrinsics(None) keeps the tuning and set_filter_params(None) the intrinsics; step_filters uses each listed filter's row
    and leaves the others bit-identical; find_new_features(None) serves each filter's own min_features request."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=9, seed=980)
    over = dict(sc.config_overrides(), min_features=14, max_features=1000, xyz_conversion=1)
    cfg = gpu_pkg.default_config(**over)
    B = 4
    src, cams = _seeded(gpu_pkg, sc, cfg, B)
    tun = _tunings(over, B, 41, 14)
    for m, t in enumerate(tun):
        t["min_features"] = (14, 30, 10, 22)[m]
        t["fx"] = cfg.fx * (1.0 + 0.01 * m)
    cfgs = [gpu_pkg.default_config(**t) for t in tun]
    _, rows = gpu_pkg._abi.batch_rows(cfg, cfgs)

    def make():
        w = gpu_pkg.FilterBatch(cfg, B, feature_capacity=32)
        w.seed_from(src); w.set_camera_states(cams)
        return w
    ref = make()
    ref.set_configs(cfgs)
    x = make()
    x.set_configs(cfgs)
    x.seed_from(src); x.set_camera_states(cams)          # seed_from keeps the table
    x.set_cameras(1, np.zeros(B, np.int32))              # and so does set_cameras
    ref.set_cameras(1, np.zeros(B, np.int32))
    x.set_intrinsics(None); x.set_intrinsics(np.array([[getattr(c, k) for k in CAM_KEYS] for c in cfgs]))
    x.set_filter_params(None); x.set_filter_params(rows)
    y = make()                                           # intrinsics only, then tuning cleared: the intrinsics stay
    y.set_configs(cfgs); y.set_filter_params(None)
    yref = make()
    yref.set_intrinsics(np.array([[getattr(c, k) for k in CAM_KEYS] for c in cfgs]))
    for t in (1, 2):
        picks = sc.picks(t, 24)
        for w in (ref, x, y, yref):
            w.captureNewFrame(sc.frame(t), sc.stamps[t]); w.step(picks)
        for b in range(B):
            _batches_equal(ref, b, x, b, f"frame {t} filter {b} (seed_from / set_cameras / tables re-set)")
            _batches_equal(yref, b, y, b, f"frame {t} filter {b} (tuning cleared)")
    # find_new_features(None) serves each filter's own request
    st = ref.camera_states()[1]
    req = st[:, 7]
    assert len(set(req.tolist())) > 1, f"requests {req}"
    n0 = [ref.numOfFeatures(b) for b in range(B)]
    corners = x.detect_corners(np.maximum(req, 0))   # x holds ref's state: the corners ref's request finds
    added = ref.findNewFeatures(None)
    for b in range(B):
        want = 0 if req[b] <= 0 else min(len(corners[b]), 32 - n0[b])
        assert len(corners[b]) <= max(req[b], 0), f"filter {b}: {len(corners[b])} corners for a request of {req[b]}"
        assert ref.numOfFeatures(b) - n0[b] == added[b] == want, f"filter {b}: added {added[b]}, want {want}, request {req[b]}"
    assert (np.asarray(added)[req > 0] > 0).any()
    assert np.array_equal(x.findNewFeatures(None), added)
    # resample: filter 1 becomes a copy of filter 3 and filter 0 of filter 2; given the ancestors' controls they reproduce them
    anc = np.array([2, 3, 2, 3], np.int32)
    ref.resample(anc)
    t = 3
    picks = sc.picks(t, 24)
    ref.captureNewFrame(sc.frame(t), sc.stamps[t]); ref.step(picks)
    for f in range(B):
        _batches_equal(ref, f, ref, int(anc[f]), f"after resample: filter {f} vs ancestor {anc[f]}")
    # step_filters with a table: the listed filters as a full step, the others untouched
    x2 = make(); x2.set_configs(cfgs); full = make(); full.set_configs(cfgs)
    for w in (x2, full):
        w.set_topup(True)
    lst = [0, 2]
    t = 4
    picks = sc.picks(t, 24)
    before = [x2.get_full(b) for b in range(B)]
    for w in (x2, full):
        w.captureNewFrame(sc.frame(t), sc.stamps[t])
    x2.step(picks, filters=lst)
    full.step(picks)
    for b in range(B):
        if b in lst:
            _batches_equal(x2, b, full, b, f"frame {t} listed filter {b}")
        else:
            m, S = x2.get_full(b)
            assert np.array_equal(m, before[b][0]) and np.array_equal(S, before[b][1]), f"frame {t} unlisted filter {b}"


@pytest.mark.parametrize("field,value", [("sigma_vx", np.nan), ("T_camera", np.inf), ("sigma_wz", -0.01), ("sigma_rho_0", -1.0),
                                         ("sigma_pixel", 0), ("sigma_size", 0), ("ransac_p", 1.0), ("ransac_p", 0.0),
                                         ("ransac_nhyp0", 0), ("min_features", -1), ("max_features", -5)])
def test_errors(gpu_pkg, field, value):
    """EKF_ERR_ARG for each invalid field, naming the filter and the field, and the table stays as it was: the next step is
    bit-identical to a batch that never saw the call.  A NULL batch is refused."""
    sc = gpu_pkg.synth.Scene(n_features=10, n_frames=3, seed=990)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    B = 3
    src, cams = _seeded(gpu_pkg, sc, cfg, B, cap=16)
    tun = [dict(sc.config_overrides(), sigma_vx=0.02 * (m + 1), sigma_pixel=m + 1) for m in range(B)]
    _, rows = gpu_pkg._abi.batch_rows(cfg, [gpu_pkg.default_config(**t) for t in tun])

    def make():
        w = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
        w.seed_from(src); w.set_camera_states(cams); w.set_filter_params(rows)
        return w
    x, ref = make(), make()
    bad = (gpu_pkg._abi.EkfFilterParams * B).from_buffer_copy(rows)
    setattr(bad[2], field, value)
    L, h = x.L, x.h
    assert L.ekf_batch_set_filter_params(h, bad) == -1
    msg = L.ekf_batch_last_error(h)
    assert b"filter 2" in msg and field.encode() in msg, msg
    assert L.ekf_batch_set_filter_params(None, None) == -1
    for t in (1, 2):
        for w in (x, ref):
            w.captureNewFrame(sc.frame(t), sc.stamps[t]); w.step(sc.picks(t, 10))
        for b in range(B):
            _batches_equal(x, b, ref, b, f"frame {t} filter {b}")


def test_set_configs_checks_everything_first_and_follows_the_batch(gpu_pkg):
    """A configuration set that set_configs refuses (one invalid row) changes neither table: the next steps are bit-identical
    to a batch that never saw the call.  The shared fields are checked against what the batch runs: after set_motion_blur and
    set_force_plane, configurations with that kernel_size and forsePlane are accepted, and the caller's EkfConfig is untouched."""
    sc = gpu_pkg.synth.Scene(n_features=10, n_frames=3, seed=995)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    B = 3
    src, cams = _seeded(gpu_pkg, sc, cfg, B, cap=16)
    good = [gpu_pkg.default_config(**dict(sc.config_overrides(), sigma_vx=0.02 * (m + 1), fx=cfg.fx * (1 + 0.01 * m))) for m in range(B)]
    bad = [gpu_pkg._abi.EkfConfig.from_buffer_copy(c) for c in good]
    for c in bad:
        c.fx *= 1.05
    bad[2].sigma_pixel = 0

    def make():
        w = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
        w.seed_from(src); w.set_camera_states(cams); w.set_configs(good)
        return w
    x, ref = make(), make()
    with pytest.raises(ValueError, match="filter 2: sigma_pixel"):
        x.set_configs(bad)
    for t in (1, 2):
        for w in (x, ref):
            w.captureNewFrame(sc.frame(t), sc.stamps[t]); w.step(sc.picks(t, 10))
        for b in range(B):
            _batches_equal(x, b, ref, b, f"frame {t} filter {b}")
    before = bytes(cfg)
    y = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
    y.set_motion_blur(3)
    y.set_force_plane(True)
    y.set_configs([gpu_pkg.default_config(**dict(sc.config_overrides(), kernel_size=3, forsePlane=1))] * B)
    with pytest.raises(ValueError, match="kernel_size"):
        y.set_configs([cfg] * B)
    assert bytes(cfg) == before
