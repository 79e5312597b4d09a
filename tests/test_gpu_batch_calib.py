"""-m gpu: batched filters with intrinsics of their own (ekf_batch_set_intrinsics) and frame sizes of their own
(ekf_batch_set_frame_sizes).

Camera c's frame is the top-left w_c x h_c of slot c of one padded stack; a filter on it must follow a single filter fed the
own-size frame, and nothing may depend on the bytes of the pads.

Filter f projects, linearises and unprojects with row f of the batch's intrinsics table.  Every filter still runs the single
filter's algorithm, so a filter with intrinsics K must follow a single CUDA filter whose ekf_config carries K: tables, NCC scores
and templates bit for bit, state within 1e-8; a batch of four rigs must equal four batches configured with those rigs bit for
bit; and every row equal to the configuration's is today's batch: same bits, same launches."""
import ctypes as C

import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, assert_scaled_close, relerr, seed_features

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

KEYS = ("fx", "fy", "u0", "v0", "k1", "k2", "k3", "p1", "p2")
# The reference's shipped calibrations (mono-slam/conf/conf.cfg, conf_firewire.cfg, conf_kinect.cfg and conf_sim.cfg), for a
# 640 x 480 frame.  conf_sim.cfg's camera is 2560 x 1920: fx, fy, u0 and v0 are divided by 4, as ConfigVSLAM divides them by
# scale.
RIGS = {
    "conf": (718.4109, 706.0125, 315.47895, 216.44625, -0.0182844, 0.04502865, 0.0, 0.0, 0.0),
    "firewire": (563.21765, 558.45293, 347.75115, 246.19144, -0.45720, 0.30980, -0.13950, -0.00265, 0.00078),
    "kinect": (537.673722507338, 534.380205679756, 321.226061527052, 249.773992466202, 0.0395956005042652,
               -0.111310452999064, 0.0, 0.00211988964071199, 0.00070924348636878),
    "sim": (2217.0187 / 4, 2217.0187 / 4, 1280.5 / 4, 960.5 / 4, 0.0, 0.0, 0.0, 0.0, 0.0),
}
BLUR_SCENE = dict(speed=0.9, omega=0.5, template_smooth=2.5)


def _row(cfg):
    return np.array([getattr(cfg, k) for k in KEYS])


def _with(cfg_over, row):
    return dict(cfg_over, **dict(zip(KEYS, (float(x) for x in row))))


def _tables_equal(batch, b, s, ctx):
    N = s.numOfFeatures()
    assert batch.numOfFeatures(b) == N, f"{ctx}: feature count {batch.numOfFeatures(b)} vs {N}"
    for i in range(N):
        a, c = batch.feature(b, i), s.feature(i)
        for f in INT_FIELDS:
            assert getattr(a, f) == getattr(c, f), f"{ctx}: feature {i} {f}"
        assert tuple(a.center) == tuple(c.center), f"{ctx}: feature {i} centre"
        assert a.last_ncc == c.last_ncc, f"{ctx}: feature {i} NCC score"
        assert np.array_equal(batch.template(b, i), s.template(i)), f"{ctx}: feature {i} template"


def _batches_equal(x, bx, y, by, ctx):
    """Filter bx of batch x against filter by of batch y: mu, Sigma, tables, both templates, bit for bit."""
    mx, Sx = x.get_full(bx); my, Sy = y.get_full(by)
    assert np.array_equal(mx, my) and np.array_equal(Sx, Sy), f"{ctx}: state"
    N = y.numOfFeatures(by)
    assert x.numOfFeatures(bx) == N, f"{ctx}: feature count"
    for i in range(N):
        a, c = x.feature(bx, i), y.feature(by, i)
        for f in INT_FIELDS:
            assert getattr(a, f) == getattr(c, f), f"{ctx}: feature {i} {f}"
        assert tuple(a.center) == tuple(c.center) and a.last_ncc == c.last_ncc, f"{ctx}: feature {i} match"
        for w in (0, 1):
            assert np.array_equal(x.template(bx, i, w), y.template(by, i, w)), f"{ctx}: feature {i} template {w}"


def _perturbed(mu0, B, seed, perturb=2e-3):
    rng = np.random.default_rng(seed)
    cams = np.tile(mu0[:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=perturb, size=(B, 3))
    cams[:, 3:7] += rng.normal(scale=perturb, size=(B, 4))
    cams[:, 3:7] /= np.linalg.norm(cams[:, 3:7], axis=1, keepdims=True)
    cams[:, 7:13] += rng.normal(scale=perturb, size=(B, 6))
    return cams


@pytest.mark.parametrize("cap,large,nfeat,minf", [(32, False, 24, 20), (100, True, 60, 55)])
def test_calibration_ensemble_follows_single_filters(gpu_pkg, cap, large, nfeat, minf):
    """M = 8 hypotheses about one camera's calibration: fx, fy, u0, v0, k1 and k2 each perturbed by about 1 %.  From an empty
    seed, the scene's features added on frame 0 (each filter unprojects with its own row), then steps with top-up (which adds
    detector corners) and XYZ conversion on.
    Each filter against a single CUDA filter whose ekf_config carries its row: tables, NCC scores and templates bit-exact,
    state within 1e-8, every step."""
    sc = gpu_pkg.synth.Scene(n_features=nfeat, n_frames=11, seed=800)
    over = dict(sc.config_overrides(), min_features=minf, max_features=1000, xyz_conversion=1)
    cfg = gpu_pkg.default_config(**over)
    M = 8
    rng = np.random.default_rng(21)
    rows = np.tile(_row(cfg), (M, 1))
    rows[:, :6] *= 1.0 + rng.normal(scale=0.01, size=(M, 6))
    batch = gpu_pkg.FilterBatch(cfg, M, feature_capacity=cap, large=large)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=cap))
    batch.set_intrinsics(rows)
    batch.set_topup(True)
    singles = [gpu_pkg.VSlamFilter(gpu_pkg.default_config(**_with(over, r)), feature_capacity=cap) for r in rows]
    batch.captureNewFrame(sc.frame(0), sc.stamps[0])
    for b, s in enumerate(singles):
        s.captureNewFrame(sc.frame(0), sc.stamps[0])
        for u, v in sc.feature_pixels:
            assert batch.addFeature(b, u, v) == 1 and s.addFeature(u, v) == 1
        _tables_equal(batch, b, s, f"frame 0 filter {b}")
    matched = 0
    for t in range(1, sc.n_frames):
        picks = sc.picks(t, 64)
        batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(picks)
        matched += int(batch.camera_states()[1][:, 1].sum())
        for b, s in enumerate(singles):
            s.captureNewFrame(sc.frame(t), sc.stamps[t]); s.predict(); s.update(picks)
            ctx = f"frame {t} filter {b}"
            _tables_equal(batch, b, s, ctx)
            mb, Sb = batch.get_full(b); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"{ctx}: mu {relerr(mb, ms):.2e} Sigma {relerr(Sb, Ss):.2e}"
    assert matched > 0
    # the rows took effect: hypotheses that started from the same frame now disagree
    assert not np.array_equal(batch.get_full(0)[0][:14], batch.get_full(1)[0][:14])


@pytest.mark.parametrize("window,blur,plane", [(11, True, False), (11, False, True), (21, False, False)])
def test_shipped_calibrations_are_separate_batches(gpu_pkg, window, blur, plane):
    """K = 4 rigs with the shipped calibrations, each scene rendered with its own camera model, M = 4 perturbed hypotheses
    each, in one batch of 4 cameras with intrinsics per filter, against four one-camera batches whose ekf_config carries that
    rig's calibration.  Features are added per filter (addFeature unprojects with the filter's row).  mu, Sigma, tables,
    templates and counters bit-identical every step."""
    names = list(RIGS)
    K, M = len(names), 4
    extra = BLUR_SCENE if blur else {}
    scenes = [gpu_pkg.synth.Scene(n_features=20, n_frames=7, seed=820 + c, window=window,
                                  camera=gpu_pkg.synth.Camera(*RIGS[n]), **extra) for c, n in enumerate(names)]
    overs = [dict(sc.config_overrides(), T_camera=0.5 if blur else 0.0) for sc in scenes]
    cfgs = [gpu_pkg.default_config(**o) for o in overs]

    def make(cfg, n):
        b = gpu_pkg.FilterBatch(cfg, n, feature_capacity=32)
        b.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=32))
        if blur:
            b.set_motion_blur(3)
        b.set_force_plane(plane)
        return b
    grouped = make(cfgs[0], K * M)
    grouped.set_cameras(K, np.repeat(np.arange(K), M))
    grouped.set_intrinsics(np.repeat(np.stack([_row(c) for c in cfgs]), M, axis=0))
    parts = [make(c, M) for c in cfgs]
    grouped.captureNewFrames(np.stack([sc.frame(0) for sc in scenes]), [sc.stamps[0] for sc in scenes])
    for c, (p, sc) in enumerate(zip(parts, scenes)):
        p.captureNewFrame(sc.frame(0), sc.stamps[0])
        for m in range(M):
            for u, v in sc.feature_pixels:
                assert grouped.addFeature(c * M + m, u, v) == 1 and p.addFeature(m, u, v) == 1
    mu0 = grouped.get_full(0)[0]
    cams = _perturbed(mu0, K * M, 9)
    grouped.set_camera_states(cams)
    for c, p in enumerate(parts):
        p.set_camera_states(cams[c * M:(c + 1) * M])
    for c in range(K):
        for m in range(M):
            _batches_equal(grouped, c * M + m, parts[c], m, f"frame 0 camera {c} hypothesis {m}")
    blurred = 0
    matched = np.zeros(K, int)
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
                blurred += int(p.last_blur_counts().sum())
            for m in range(M):
                _batches_equal(grouped, c * M + m, p, m, f"frame {t} rig {names[c]} hypothesis {m}")
            matched[c] += int(stp[:, 1].sum())
    assert (matched > 0).all(), f"matches per rig {matched}"
    if blur:
        assert blurred > 0


def test_calibrations_against_oracle(gpu_pkg, orc):
    """Three filters on three cameras with three shipped calibrations and three frame sizes in one padded stack, each scene
    rendered with its camera model at its size.  Each step
    from identical inputs (batch state <- oracle state) against an oracle built with that filter's configuration and fed its
    camera's frame: counters and tables bit-exact (matches, NCC scores), state within TOL and the scaled bars."""
    names = ("conf", "firewire", "kinect")
    sizes = [(640, 480), (501, 377), (752, 480)]
    scenes = [gpu_pkg.synth.Scene(n_features=20, n_frames=7, seed=840 + c, width=sizes[c][0], height=sizes[c][1],
                                  camera=gpu_pkg.synth.Camera(*RIGS[n])) for c, n in enumerate(names)]
    cfgs = [gpu_pkg.default_config(**sc.config_overrides()) for sc in scenes]
    B = 3
    batch = gpu_pkg.FilterBatch(cfgs[0], B, feature_capacity=32)
    batch.seed_from(gpu_pkg.VSlamFilter(cfgs[0], feature_capacity=32))
    batch.set_cameras(B)
    batch.set_intrinsics(np.stack([_row(c) for c in cfgs]))
    batch.set_frame_sizes(sizes)
    batch.captureNewFrames([sc.frame(0) for sc in scenes], [sc.stamps[0] for sc in scenes])
    oracles = []
    for b, (sc, cfg) in enumerate(zip(scenes, cfgs)):
        for p in sc.feature_pixels:
            assert batch.addFeature(b, *p) == 1
        o = orc.OracleFilter(cfg, kind=0, omp=False)
        seed_features(o, sc)
        oracles.append(o)
    for t in range(1, 7):
        picks = scenes[0].picks(t, 20)
        for b, o in enumerate(oracles):
            assert batch.numOfFeatures(b) == o.numOfFeatures(), f"frame {t} filter {b}: feature count"
            batch.set_full(b, *o.get_full())
        batch.captureNewFrames([sc.frame(t) for sc in scenes], [sc.stamps[t] for sc in scenes])
        batch.step(picks)
        _, _, st = batch.camera_states(want_sigma=True)
        for b, (o, sc) in enumerate(zip(oracles, scenes)):
            ctx = f"frame {t} rig {names[b]}"
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
                assert tuple(a.center) == tuple(c.center), f"{ctx} feature {i} match"
                assert a.last_ncc == c.last_ncc, f"{ctx} feature {i} NCC score"


def test_configuration_rows_are_todays_batch(gpu_pkg):
    """set_intrinsics with every row the configuration's, set_frame_sizes with the camera at the slot size, and a table and sizes
    set then reset with None, against a batch that never calls them: bit-identical states and the same kernel launches around every capture and step, with top-up
    and XYZ conversion on."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=860)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=16, xyz_conversion=1))
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    B = 4
    cams = _perturbed(src.get_full()[0], B, 11)
    x, y, z, u = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=32) for _ in range(4))
    for w in (x, y, z, u):
        w.seed_from(src); w.set_camera_states(cams); w.set_topup(True)
    y.set_intrinsics(_row(cfg))
    y.set_frame_sizes([[sc.width, sc.height]])
    z.set_intrinsics(np.tile(_row(cfg), (B, 1)) * 1.01)
    z.set_intrinsics(None)
    z.set_frame_sizes([[320, 240]])
    z.set_frame_sizes(None)
    u.set_frame_sizes([[sc.width, sc.height]])
    for t in range(1, sc.n_frames):
        picks = sc.picks(t, 20)
        counts = []
        for w in (x, y, z, u):
            l0 = w.kernel_launches()
            w.captureNewFrame(sc.frame(t), sc.stamps[t])
            l1 = w.kernel_launches()
            w.step(picks)
            counts.append((l1 - l0, w.kernel_launches() - l1))
        assert counts[0] == counts[1] == counts[2] == counts[3], f"frame {t}: launches {counts}"
        for w in (y, z, u):
            assert np.array_equal(x.camera_states()[1], w.camera_states()[1])
            for b in range(B):
                _batches_equal(x, b, w, b, f"frame {t} filter {b}")


def test_errors(gpu_pkg):
    """EKF_ERR_ARG for a non-finite entry and for fx <= 0 or fy <= 0, and the table stays as it was; wrong shapes are refused
    in Python.  The table survives set_cameras."""
    sc = gpu_pkg.synth.Scene(n_features=10, n_frames=3, seed=880)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=16)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    B = 3
    ERR_ARG = -1
    rows = np.tile(_row(cfg), (B, 1))
    rows[:, 0] *= 1.01

    def make():
        b = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
        b.seed_from(src)
        return b
    x, ref = make(), make()
    ref.set_intrinsics(rows)
    x.set_intrinsics(rows)
    L, h = x.L, x.h
    for col, val in ((0, np.nan), (3, np.inf), (6, -np.inf), (0, 0.0), (1, -5.0)):
        bad = rows.copy()
        bad[2, col] = val
        bad = np.ascontiguousarray(bad)
        assert L.ekf_batch_set_intrinsics(h, bad.ctypes.data_as(C.c_void_p)) == ERR_ARG, f"column {col} = {val}"
        assert b"filter 2" in L.ekf_batch_last_error(h)
    assert L.ekf_batch_set_intrinsics(None, None) == ERR_ARG
    with pytest.raises(ValueError):
        x.set_intrinsics(np.zeros((B + 1, 9)))
    with pytest.raises(ValueError):
        x.set_intrinsics(np.zeros(8))
    for w in (x, ref):
        w.set_cameras(1, np.zeros(B, np.int32))
    for t in (1, 2):
        for w in (x, ref):
            w.captureNewFrame(sc.frame(t), sc.stamps[t]); w.step(sc.picks(t, 10))
        for b in range(B):
            _batches_equal(x, b, ref, b, f"frame {t} filter {b}")


SIZES4 = [(640, 480), (320, 240), (752, 480), (501, 377)]


def _padded(frames, W, H, rng=None):
    """A (K, H, W) stack with frame c at the top left of slot c; the pads zero, or random bytes from rng."""
    out = rng.integers(0, 256, (len(frames), H, W), dtype=np.uint8) if rng is not None else np.zeros((len(frames), H, W), np.uint8)
    for c, f in enumerate(frames):
        out[c, :f.shape[0], :f.shape[1]] = f
    return out


def test_mixed_frame_sizes_follow_single_filters(gpu_pkg):
    """Cameras of 640 x 480, 320 x 240, 752 x 480 and 501 x 377 in one padded stack, two filters each, the scenes seeded close
    to every camera's right and bottom edges.  Each filter against a single filter fed its own-size frame: tables, NCC scores
    and templates bit-exact, state within 1e-8, every step; returnGrayImg(c) has the camera's own shape."""
    K, M = len(SIZES4), 2
    B = K * M
    scenes = [gpu_pkg.synth.Scene(n_features=24, n_frames=8, seed=900 + c, width=w, height=h, border=12)
              for c, (w, h) in enumerate(SIZES4)]
    cfgs = [gpu_pkg.default_config(**sc.config_overrides()) for sc in scenes]
    batch = gpu_pkg.FilterBatch(cfgs[0], B, feature_capacity=32)
    batch.seed_from(gpu_pkg.VSlamFilter(cfgs[0], feature_capacity=32))
    batch.set_cameras(K, np.arange(B) // M)
    batch.set_intrinsics(np.repeat(np.stack([_row(c) for c in cfgs]), M, axis=0))
    batch.set_frame_sizes(SIZES4)
    batch.captureNewFrames([sc.frame(0) for sc in scenes], [sc.stamps[0] for sc in scenes])
    singles = []
    for b in range(B):
        sc = scenes[b // M]
        s = gpu_pkg.VSlamFilter(cfgs[b // M], feature_capacity=32)
        s.captureNewFrame(sc.frame(0), sc.stamps[0])
        for u, v in sc.feature_pixels:
            assert batch.addFeature(b, u, v) == s.addFeature(u, v)
        singles.append(s)
    near = [max(float(np.max(sc.feature_pixels[:, 0])) - sc.width, float(np.max(sc.feature_pixels[:, 1])) - sc.height) for sc in scenes]
    assert max(near) > -12 - 11, f"no feature near an edge: {near}"
    for c, (w, h) in enumerate(SIZES4):
        assert batch.returnGrayImg(c).shape == (h, w)
        assert np.array_equal(batch.returnGrayImg(c), scenes[c].frame(0))
    matched = 0
    for t in range(1, 8):
        picks = scenes[0].picks(t, 24)
        batch.captureNewFrames([sc.frame(t) for sc in scenes], [sc.stamps[t] for sc in scenes]); batch.step(picks)
        matched += int(batch.camera_states()[1][:, 1].sum())
        for b, s in enumerate(singles):
            sc = scenes[b // M]
            s.captureNewFrame(sc.frame(t), sc.stamps[t]); s.predict(); s.update(picks)
            _tables_equal(batch, b, s, f"frame {t} filter {b}")
            mb, Sb = batch.get_full(b); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"frame {t} filter {b}"
    assert matched > 0


def _near_tie(W, H):
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:H, 0:W]
    smooth = (127 + 60 * np.sin(xx / 23.0) + 50 * np.cos(yy / 17.0) + rng.normal(scale=1.5, size=(H, W))).clip(0, 255)
    periodic = (((xx % 8) * 16 + (yy % 8) * 12) % 256).astype(np.float64)
    coarse = ((rng.integers(0, 4, size=(H // 4 + 1, W // 4 + 1)).repeat(4, 0).repeat(4, 1)[:H, :W]) * 64).astype(np.float64)
    return [smooth.astype(np.uint8), periodic.astype(np.uint8), coarse.astype(np.uint8)]


def _tie_frames(t):
    """Window-11 near-tie images (the CTA matcher takes some of their features), one per camera of SIZES4, cropped to size."""
    base = _near_tie(752, 480)
    return [np.roll(base[c % 3], t, axis=1)[:h, :w].copy() for c, (w, h) in enumerate(SIZES4)]


def test_small_cameras_defer_to_the_cta_matcher(gpu_pkg):
    """Window 11 on near-tie images at the four sizes, corners found by findNewFeatures up to each small camera's edges: features
    defer to the CTA matcher, whose TMA box reaches past a small camera's edge into the zeroed pad, and every filter still
    follows a single filter fed its own-size frame bit for bit."""
    K = len(SIZES4)
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    batch = gpu_pkg.FilterBatch(cfg, K, feature_capacity=32)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=32))
    batch.set_cameras(K)
    batch.set_frame_sizes(SIZES4)
    batch.captureNewFrames(_tie_frames(0), [0.0] * K)
    added = batch.findNewFeatures(np.full(K, 30, np.int32))
    singles = []
    for c in range(K):
        s = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
        s.captureNewFrame(_tie_frames(0)[c], 0.0)
        assert s.findNewFeatures(30) == added[c] > 0
        _tables_equal(batch, c, s, f"frame 0 camera {c}")
        singles.append(s)
    deferred = 0
    for t in range(1, 4):
        fr = _tie_frames(t)
        picks = np.arange(1, 41, dtype=np.uint32) * 7919
        batch.captureNewFrames(fr, [t / 30.0] * K); batch.step(picks)
        deferred += batch.last_match_deferred()
        for c, s in enumerate(singles):
            s.captureNewFrame(fr[c], t / 30.0); s.predict(); s.update(picks)
            _tables_equal(batch, c, s, f"frame {t} camera {c}")
            mb, Sb = batch.get_full(c); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"frame {t} camera {c}"
    assert deferred > 0, "no feature reached the CTA matcher"


def test_pad_contents_do_not_matter(gpu_pkg):
    """The same near-tie sequence at the four sizes with the pads zero and with the pads random: states, tables, templates, the
    corners detect_corners returns and what findNewFeatures adds are bit-identical."""
    K = len(SIZES4)
    W, H = max(w for w, _ in SIZES4), max(h for _, h in SIZES4)
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    rng = np.random.default_rng(77)

    def make():
        b = gpu_pkg.FilterBatch(cfg, K, feature_capacity=32)
        b.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=32))
        b.set_cameras(K)
        b.set_frame_sizes(SIZES4)
        return b
    x, y = make(), make()
    x.captureNewFrames(_padded(_tie_frames(0), W, H), [0.0] * K)
    y.captureNewFrames(_padded(_tie_frames(0), W, H, rng), [0.0] * K)
    num = np.full(K, 25, np.int32)
    cx, cy = x.detect_corners(num), y.detect_corners(num)
    for c in range(K):
        assert np.array_equal(cx[c], cy[c]), f"camera {c}: corners"
    assert np.array_equal(x.findNewFeatures(num), y.findNewFeatures(num))
    for t in range(1, 4):
        picks = np.arange(1, 41, dtype=np.uint32) * 7919
        x.captureNewFrames(_padded(_tie_frames(t), W, H), [t / 30.0] * K); x.step(picks)
        y.captureNewFrames(_padded(_tie_frames(t), W, H, rng), [t / 30.0] * K); y.step(picks)
        assert np.array_equal(x.camera_states()[1], y.camera_states()[1])
        for c in range(K):
            _batches_equal(x, c, y, c, f"frame {t} camera {c}")


@pytest.mark.parametrize("cap,large", [(12, False), (100, True)])
def test_detector_with_frame_sizes(gpu_pkg, cap, large):
    """12 cameras of three sizes in a 320 x 240 slot, 2 filters each, camera 5 asked nothing; a budget of 5 slots' scratch
    makes one call span three chunks.  Each filter's corners, in order, are a single filter's detect_corners on its camera's
    frame cropped to size; findNewFeatures adds exactly those."""
    W, H = 320, 240
    K, M = 12, 2
    B = K * M
    sizes = [[(320, 240), (257, 199), (301, 181)][c % 3] for c in range(K)]
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    imgs = []
    for c, (w, h) in enumerate(sizes):
        r = np.random.default_rng(700 + c)
        im = cv2.GaussianBlur(r.integers(0, 256, (h, w)).astype(np.float32), (0, 0), 2.5)
        imgs.append(np.clip((im - im.min()) / (im.max() - im.min()) * 200 + 20, 0, 255).astype(np.uint8))
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap, large=large)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=cap))
    batch.set_cameras(K, np.arange(B) // M)
    batch.set_frame_sizes(sizes)
    batch.set_detect_budget(5 * 36 * W * H)
    batch.captureNewFrames(_padded(imgs, W, H, np.random.default_rng(1)), None)
    rng = np.random.default_rng(5)
    for b in range(B):
        w, h = sizes[b // M]
        for u, v in rng.uniform(20, min(w, h) - 20, (b % 4, 2)):
            assert batch.addFeature(b, u, v) == 1
    num = np.array([(7 + 3 * b) % 33 for b in range(B)], dtype=np.int32)
    num[[5 * M, 5 * M + 1]] = 0
    got = batch.detect_corners(num)

    def single(b):
        s = gpu_pkg.VSlamFilter(cfg, feature_capacity=128)
        s.captureNewFrame(imgs[b // M], 1.0)
        for i in range(batch.numOfFeatures(b)):
            s.addFeature(*batch.feature(b, i).center)
        return s
    for b in range(B):
        want = single(b).detect_corners(int(num[b])) if num[b] > 0 else np.zeros((0, 2), np.float32)
        assert np.array_equal(got[b], want), f"filter {b} (camera {b // M}): batch vs single filter"
    assert sum(len(g) for g in got) > 0
    N0 = [batch.numOfFeatures(b) for b in range(B)]
    wants = [(single(b).detect_corners(int(num[b])) if num[b] > 0 else np.zeros((0, 2), np.float32))[:cap - N0[b]] for b in range(B)]
    added = batch.findNewFeatures(num)
    for b in range(B):
        assert added[b] == len(wants[b]), f"filter {b}: added {added[b]} vs {len(wants[b])}"
        new = np.array([batch.feature(b, i).center for i in range(N0[b], batch.numOfFeatures(b))], np.float32).reshape(-1, 2)
        assert np.array_equal(new, wants[b]), f"filter {b}: added corners"


@pytest.mark.parametrize("scale", [2, 3])
def test_resized_and_bgr_frame_sizes(gpu_pkg, scale):
    """50 BGR cameras of odd sizes (so that w_c / scale truncates) in 1600 x 1200 slots: the host stack (288 MB) is staged 46
    cameras at a time, and the cameras checked include both sides of that boundary.  Each camera equals cv2.resize + cvtColor
    of its crop, and returnGrayImg(c) has its own shape; a gray stack of the same crops as well."""
    W, H, K = 1600, 1200, 50
    sizes = [(W - 2 * c - 1, H - 3 * c - 1) if c % 2 else (W - 7 * c, H - 5 * c) for c in range(K)]
    cfg = gpu_pkg.default_config(window_size=11)
    rng = np.random.default_rng(scale)
    base = rng.integers(0, 256, (2, H, W, 3), dtype=np.uint8)
    bgr = np.stack([np.roll(base[c % 2], 7 * c, axis=1) for c in range(K)])
    batch = gpu_pkg.FilterBatch(cfg, K, feature_capacity=8)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=8))
    batch.set_scale(scale)
    batch.set_cameras(K)
    batch.set_frame_sizes(sizes)
    batch.captureNewFrames(bgr)
    for c in (0, 1, 44, 45, 46, 47, 49):
        w, h = sizes[c]
        want = cv2.cvtColor(cv2.resize(bgr[c, :h, :w], (w // scale, h // scale)), cv2.COLOR_BGR2GRAY)
        got = batch.returnGrayImg(c)
        assert got.shape == (h // scale, w // scale), f"camera {c}: shape {got.shape}"
        assert np.array_equal(got, want), f"bgr camera {c}: differs from cv2"
    gray = np.stack([cv2.cvtColor(bgr[c], cv2.COLOR_BGR2GRAY) for c in range(K)])
    batch.captureNewFrames(gray)
    for c in (0, 3, 46, 49):
        w, h = sizes[c]
        assert np.array_equal(batch.returnGrayImg(c), cv2.resize(gray[c, :h, :w], (w // scale, h // scale))), f"gray camera {c}"


def test_frame_size_errors(gpu_pkg):
    """EKF_ERR_ARG: non-positive sizes, a camera larger than the capture's slot, a resized side below 8.  set_cameras returns
    to uniform sizes."""
    cfg = gpu_pkg.default_config(window_size=11)
    B = 2
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=8)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=8))
    batch.set_cameras(B)
    L, h = batch.L, batch.h
    ERR_ARG = -1
    for bad in ([[0, 10], [20, 20]], [[20, 20], [20, -1]]):
        a = np.ascontiguousarray(bad, dtype=np.int32)
        assert L.ekf_batch_set_frame_sizes(h, a.ctypes.data_as(C.c_void_p)) == ERR_ARG
    stack = np.zeros((B, 120, 160), np.uint8)
    batch.set_frame_sizes([[160, 120], [161, 100]])
    assert L.ekf_batch_capture_frames(h, stack.ctypes.data_as(C.c_void_p), 160, 120, 160, None) == ERR_ARG
    assert b"larger" in L.ekf_batch_last_error(h)
    batch.set_frame_sizes([[160, 120], [100, 15]])
    batch.set_scale(2)
    assert L.ekf_batch_capture_frames(h, stack.ctypes.data_as(C.c_void_p), 160, 120, 160, None) == ERR_ARG
    batch.set_scale(1)
    batch.captureNewFrames(stack)
    assert batch.returnGrayImg(1).shape == (15, 100)
    batch.set_cameras(B)
    batch.captureNewFrames(stack)
    assert batch.returnGrayImg(1).shape == (120, 160)
