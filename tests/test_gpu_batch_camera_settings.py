"""-m gpu: batched filters on cameras with settings of their own (ekf_batch_set_camera_settings, FilterBatch.from_configs).

Filter f runs with the window, scale and blur threshold of its camera exactly as a batch created with them would, so a filter
must follow a single CUDA filter whose ekf_config carries its camera's settings and its tuning (tables, NCC scores, templates
and blur counts bit for bit, state within 1e-8), and the four shipped configurations in one batch must equal four batches built
from them, bit for bit.  Frames at the input resolution are rendered at the resized size and each pixel replicated s x s: both
sides resize the same way whatever the frames are, this only keeps the features trackable."""

import ctypes as C

import numpy as np
import pytest

from helpers import relerr
from test_gpu_batch_calib import BLUR_SCENE, RIGS, _batches_equal, _perturbed, _tables_equal

pytestmark = pytest.mark.gpu
OFF = 1000000000
# The tuning of the shipped configurations (conf.cfg, conf_firewire.cfg, conf_kinect.cfg, conf_sim.cfg), as in the tuning tests.
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


def _up(img, s):
    return np.ascontiguousarray(np.repeat(np.repeat(img, s, axis=0), s, axis=1))


def _rig_camera(gpu_pkg, name, width):
    """The shipped calibration, its focal lengths and principal point scaled from 640 px to `width`."""
    k = width / 640.0
    fx, fy, u0, v0, *dist = RIGS[name]
    return gpu_pkg.synth.Camera(fx * k, fy * k, u0 * k, v0 * k, *dist)


@pytest.mark.parametrize("cap,large,nfeat,minf", [(32, False, 16, 20), (100, True, 30, 34)])
def test_each_filter_follows_a_single_filter(gpu_pkg, cap, large, nfeat, minf):
    """K = 4 cameras with windows 7, 11, 15, 21, scales 1, 2, 3, 1 and blur thresholds 3, 2, off, 3, M = 2 tunings each, top-up
    (min_features above the seeded count, so every step detects with the camera's window) and XYZ conversion on, in fast motion
    that blurs templates.  Each filter against a VSlamFilter whose ekf_config carries its camera's window, scale and kernel_size
    and its tuning: tables, NCC scores, templates and blur counts bit-exact, state within 1e-8, every step; templates were
    blurred on the blur-on cameras and none on the other, and top-up added features."""
    W, H = 960, 720
    wins, scales, kers = (7, 11, 15, 21), (1, 2, 3, 1), (3, 2, OFF, 3)
    K, M = 4, 2
    scenes = [gpu_pkg.synth.Scene(n_features=nfeat, n_frames=7, seed=1100 + c, width=W // s, height=H // s, window=w, **BLUR_SCENE)
              for c, (w, s) in enumerate(zip(wins, scales))]
    cfgs = []
    for c, sc in enumerate(scenes):
        for m in range(M):
            cfgs.append(gpu_pkg.default_config(**dict(sc.config_overrides(), window_size=wins[c], scale=scales[c], kernel_size=kers[c],
                                                      T_camera=(0.5, 0.8)[m], sigma_pixel=(2, 3)[m], min_features=minf,
                                                      max_features=1000, xyz_conversion=1)))
    camera_of = np.repeat(np.arange(K), M)
    batch = gpu_pkg.FilterBatch.from_configs(cfgs, camera_of, feature_capacity=cap, large=large)
    assert batch.camera_settings.tolist() == [[w, s, k] for w, s, k in zip(wins, scales, kers)]
    batch.seed_from(gpu_pkg.VSlamFilter(cfgs[0], feature_capacity=cap))   # an empty source seeds any table
    batch.set_topup(True)
    singles = [gpu_pkg.VSlamFilter(c, feature_capacity=cap) for c in cfgs]

    def frames(t):
        return [_up(sc.frame(t), s) for sc, s in zip(scenes, scales)]
    fr = frames(0)
    batch.captureNewFrames(np.stack(fr), [sc.stamps[0] for sc in scenes])
    for c in range(K):
        assert batch.returnGrayImg(c).shape == (H // scales[c], W // scales[c])
    for f, s in enumerate(singles):
        c = camera_of[f]
        s.captureNewFrame(fr[c], scenes[c].stamps[0])
        assert np.array_equal(batch.returnGrayImg(c), s.returnGrayImg()), f"camera {c}: resized frame"
        for u, v in scenes[c].feature_pixels:
            assert batch.addFeature(f, u, v) == s.addFeature(u, v)
        _tables_equal(batch, f, s, f"frame 0 filter {f}")
    matched, blurred, added = np.zeros(K, int), np.zeros(K, int), np.zeros(K, int)
    for t in range(1, 7):
        picks = scenes[0].picks(t, 64)
        fr = frames(t)
        batch.captureNewFrames(np.stack(fr), [sc.stamps[t] for sc in scenes])
        batch.step(picks)
        st = batch.camera_states()[1]
        counts = batch.last_blur_counts()
        np.add.at(blurred, camera_of, counts)
        np.add.at(added, camera_of, batch.last_added())
        for f, s in enumerate(singles):
            c = camera_of[f]
            s.captureNewFrame(fr[c], scenes[c].stamps[t]); s.predict(); s.update(picks)
            ctx = f"frame {t} filter {f} (window {wins[c]}, scale {scales[c]})"
            assert counts[f] == s.stats().blur_requests, f"{ctx}: blurred {counts[f]} vs {s.stats().blur_requests}"
            _tables_equal(batch, f, s, ctx)
            mb, Sb = batch.get_full(f); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"{ctx}: mu {relerr(mb, ms):.2e} Sigma {relerr(Sb, Ss):.2e}"
            matched[c] += int(st[f, 1])
    assert (matched > 0).all(), f"matches per camera {matched}"
    assert blurred[2] == 0 and blurred[[0, 1, 3]].sum() > 0, f"blurred templates per camera {blurred}"
    assert added.sum() > 0, f"features added by top-up per camera {added}"


SHIPPED = {"conf": (21, 2, 1000), "firewire": (21, 1, OFF), "kinect": (15, 2, 1000), "sim": (30, 10, 3)}


@pytest.mark.parametrize("mode", ["plain", "sizes", "subset"])
def test_shipped_configurations_in_one_batch(gpu_pkg, mode):
    """The four shipped rigs as shipped (window, scale, blur, tuning, calibration) x M = 2 in one batch by from_configs, against
    four one-camera batches by from_config: mu, Sigma, tables, templates, counters and blur counts bit-identical every step.
    sizes: a frame size per camera; subset: cameras 0 and 2 deliver only every other frame (cameras= / filters=)."""
    names = list(SHIPPED)
    K, M = 4, 2
    # input sizes: 2560 x 1920 for every camera (plain, subset), or each camera's own (sizes); the scenes render at input / scale
    ins = {n: (1280 * (2 if n == "sim" else 1), 960 * (2 if n == "sim" else 1)) for n in names} if mode == "sizes" else \
          {n: (2560, 1920) for n in names}
    scenes, cfgs = [], []
    for c, n in enumerate(names):
        w, s, k = SHIPPED[n]
        rw, rh = ins[n][0] // s, ins[n][1] // s
        sc = gpu_pkg.synth.Scene(n_features=16, n_frames=7, seed=1200 + c, width=rw, height=rh, window=w, template_smooth=2.0,
                                 camera=_rig_camera(gpu_pkg, n, rw))
        scenes.append(sc)
        cfgs.append(gpu_pkg.default_config(**dict(sc.config_overrides(), **TUNING[n], window_size=w, scale=s, kernel_size=k,
                                                  xyz_conversion=1)))
    camera_of = np.repeat(np.arange(K), M)
    grouped = gpu_pkg.FilterBatch.from_configs([cfgs[c] for c in camera_of], camera_of, feature_capacity=32)
    grouped.seed_from(gpu_pkg.VSlamFilter(cfgs[0], feature_capacity=32))
    if mode == "sizes":
        grouped.set_frame_sizes(np.array([ins[n] for n in names]))
    parts = []
    for c in cfgs:
        p = gpu_pkg.FilterBatch.from_config(c, M, feature_capacity=32)
        p.seed_from(gpu_pkg.VSlamFilter(c, feature_capacity=32))
        parts.append(p)

    def frame(c, t):
        return _up(scenes[c].frame(t), SHIPPED[names[c]][1])

    def capture(t, cams):
        fr = [frame(c, t) for c in cams]
        st = [scenes[c].stamps[t] for c in cams]
        every = len(cams) == K
        if mode == "sizes":
            grouped.captureNewFrames(fr, st, cameras=None if every else cams)
        else:
            grouped.captureNewFrames(np.stack(fr), st, cameras=None if every else cams)
        for c, x in zip(cams, fr):
            parts[c].captureNewFrame(x, scenes[c].stamps[t])
    capture(0, list(range(K)))
    for c, p in enumerate(parts):
        for m in range(M):
            for u, v in scenes[c].feature_pixels:
                assert grouped.addFeature(c * M + m, u, v) == p.addFeature(m, u, v)
    cams = _perturbed(grouped.get_full(0)[0], K * M, 9)
    grouped.set_camera_states(cams)
    for c, p in enumerate(parts):
        p.set_camera_states(cams[c * M:(c + 1) * M])
    matched = np.zeros(K, int)
    for t in range(1, 7):
        picks = scenes[0].picks(t, 24)
        live = [0, 1, 2, 3] if (mode != "subset" or t % 2 == 0) else [1, 3]
        capture(t, live)
        if len(live) == K:
            grouped.step(picks)
        else:
            grouped.step(picks, filters=[f for f in range(K * M) if camera_of[f] in live])
        _, stg = grouped.camera_states()
        blur_g = grouped.last_blur_counts()
        for c in live:
            p = parts[c]
            p.step(picks)
            _, stp = p.camera_states()
            ctx = f"frame {t} rig {names[c]}"
            assert np.array_equal(stg[c * M:(c + 1) * M], stp), f"{ctx}: counters"
            assert np.array_equal(blur_g[c * M:(c + 1) * M], p.last_blur_counts()), f"{ctx}: blur counts"
            for m in range(M):
                _batches_equal(grouped, c * M + m, p, m, f"{ctx} hypothesis {m}")
            matched[c] += int(stp[:, 1].sum())
    assert (matched > 0).all(), f"matches per rig {matched}"
    for c, n in enumerate(names):
        w, s, _ = SHIPPED[n]
        assert grouped.returnGrayImg(c).shape == (ins[n][1] // s, ins[n][0] // s)
        if grouped.numOfFeatures(c * M):
            assert grouped.template(c * M, 0).shape == (w, w)


def _seeded_pair(gpu_pkg, sc, cfg, B, seed=11):
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    return src, _perturbed(src.get_full()[0], B, seed)


def test_table_of_the_batch_values_is_todays_batch(gpu_pkg):
    """A table equal to the batch's own window, scale and blur threshold: the same bits and the same kernel launches as no table."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=1300)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=16, xyz_conversion=1))
    B = 4
    src, cams = _seeded_pair(gpu_pkg, sc, cfg, B)
    x, y = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=32) for _ in range(2))
    y.set_camera_settings([[cfg.window_size, 1, cfg.kernel_size]])
    for w in (x, y):
        w.seed_from(src); w.set_camera_states(cams); w.set_topup(True)
    for t in range(1, sc.n_frames):
        picks = sc.picks(t, 20)
        launches = []
        for w in (x, y):
            l0 = w.kernel_launches()
            w.captureNewFrame(sc.frame(t), sc.stamps[t]); w.step(picks)
            launches.append(w.kernel_launches() - l0)
        assert launches[0] == launches[1], f"frame {t}: launches {launches}"
        for b in range(B):
            _batches_equal(y, b, x, b, f"frame {t} filter {b}")
        assert np.array_equal(x.camera_states()[1], y.camera_states()[1])


def test_window_11_beside_window_21(gpu_pkg):
    """A batch created at window 21 whose camera 0 runs window 11 and camera 1 window 21: camera 0's filters have the bits of a
    window-11 batch, camera 1's those of a window-21 batch (full-window and CTA matchers in one step)."""
    s11 = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=1310, window=11)
    s21 = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=1311, window=21)
    c11 = gpu_pkg.default_config(**dict(s11.config_overrides(), xyz_conversion=1))
    c21 = gpu_pkg.default_config(**dict(s21.config_overrides(), xyz_conversion=1))
    M = 3
    mixed = gpu_pkg.FilterBatch.from_configs([c11] * M + [c21] * M, [0] * M + [1] * M)
    mixed.seed_from(gpu_pkg.VSlamFilter(c11, feature_capacity=32))
    ref = [gpu_pkg.FilterBatch.from_config(c, M) for c in (c11, c21)]
    for r, c in zip(ref, (c11, c21)):
        r.seed_from(gpu_pkg.VSlamFilter(c, feature_capacity=32))
    scenes = (s11, s21)
    mixed.captureNewFrames(np.stack([s11.frame(0), s21.frame(0)]), [s11.stamps[0], s21.stamps[0]])
    for c, (r, sc) in enumerate(zip(ref, scenes)):
        r.captureNewFrame(sc.frame(0), sc.stamps[0])
        for m in range(M):
            for u, v in sc.feature_pixels:
                assert mixed.addFeature(c * M + m, u, v) == r.addFeature(m, u, v)
    cams = _perturbed(mixed.get_full(0)[0], 2 * M, 5)
    cams[M:] = _perturbed(mixed.get_full(M)[0], M, 6)
    mixed.set_camera_states(cams)
    ref[0].set_camera_states(cams[:M]); ref[1].set_camera_states(cams[M:])
    for t in range(1, 6):
        picks = s11.picks(t, 20)
        mixed.captureNewFrames(np.stack([s11.frame(t), s21.frame(t)]), [s11.stamps[t], s21.stamps[t]])
        mixed.step(picks)
        for c, (r, sc) in enumerate(zip(ref, scenes)):
            r.captureNewFrame(sc.frame(t), sc.stamps[t]); r.step(picks)
            for m in range(M):
                _batches_equal(mixed, c * M + m, r, m, f"frame {t} window {(11, 21)[c]} hypothesis {m}")
    assert mixed.camera_states()[1][:, 1].sum() > 0


def test_resample_inside_a_window_15_camera(gpu_pkg):
    """Copies made by resample inside a camera of window 15 (batch window 21) equal their ancestors over three more steps."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=1320, window=15)
    c15 = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=1))
    c21 = gpu_pkg.default_config(**dict(sc.config_overrides(), window_size=21, xyz_conversion=1))
    M = 4
    batch = gpu_pkg.FilterBatch.from_configs([c15] * M + [c21] * M, [0] * M + [1] * M)
    batch.seed_from(gpu_pkg.VSlamFilter(c15, feature_capacity=32))
    batch.captureNewFrames(np.stack([sc.frame(0)] * 2), [sc.stamps[0]] * 2)
    for f in range(2 * M):
        for u, v in sc.feature_pixels:
            batch.addFeature(f, u, v)
    batch.set_camera_states(_perturbed(batch.get_full(0)[0], 2 * M, 3))
    for t in (1, 2):
        batch.captureNewFrames(np.stack([sc.frame(t)] * 2), [sc.stamps[t]] * 2); batch.step(sc.picks(t, 20))
    anc = np.arange(2 * M)
    anc[2], anc[3] = 0, 1
    batch.resample(anc)
    for t in (3, 4, 5):
        batch.captureNewFrames(np.stack([sc.frame(t)] * 2), [sc.stamps[t]] * 2); batch.step(sc.picks(t, 20))
        for f in (2, 3):
            _batches_equal(batch, f, batch, anc[f], f"frame {t} copy {f}")
            assert batch.template(f, 0).shape == (15, 15)


def test_refusals_leave_the_batch_as_it_was(gpu_pkg):
    """Every refusal of set_camera_settings and the calls it constrains, with the table and the state unchanged afterwards."""
    EkfError = gpu_pkg.EkfError
    sc = gpu_pkg.synth.Scene(n_features=12, n_frames=3, seed=1330, window=15)
    c21 = gpu_pkg.default_config(**dict(sc.config_overrides(), window_size=21))
    c15 = gpu_pkg.default_config(**dict(sc.config_overrides(), window_size=15))
    b = gpu_pkg.FilterBatch(c21, 4, feature_capacity=32)
    b.set_cameras(2, [0, 0, 1, 1])
    for bad, what in (([[2, 1, OFF], [21, 1, OFF]], "camera 0: window_size = 2"),
                      ([[21, 1, OFF], [23, 1, OFF]], "camera 1: window_size = 23"),
                      ([[21, 0, OFF], [21, 1, OFF]], "camera 0: scale = 0"),
                      ([[21, 1, OFF], [21, 65, OFF]], "camera 1: scale = 65")):
        with pytest.raises(EkfError, match=what):
            b.set_camera_settings(bad)
    assert b.camera_settings is None
    b.set_camera_settings([[15, 1, OFF], [21, 2, 3]])
    with pytest.raises(EkfError, match="camera settings"):
        b.set_scale(2)
    with pytest.raises(EkfError, match="camera settings"):
        b.set_motion_blur(5)
    # a seed with features of window 15 needs every camera at 15
    src = gpu_pkg.VSlamFilter(c15, feature_capacity=32)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    with pytest.raises(EkfError, match="camera 1 runs window_size 21"):
        b.seed_from(src)
    b.set_camera_settings([[15, 1, OFF], [15, 2, 3]])
    b.seed_from(src)
    assert b.numOfFeatures(0) == src.numOfFeatures() > 0
    for i in range(src.numOfFeatures()):
        assert np.array_equal(b.template(3, i), src.template(i)) and b.template(3, i).shape == (15, 15)
    # a window change under features: EKF_ERR_STATE naming the filter, nothing changes
    before = b.get_full(2)
    with pytest.raises(EkfError, match="filter 0 holds features of window_size 15"):
        b.set_camera_settings([[11, 1, OFF], [15, 2, 3]])
    with pytest.raises(EkfError, match="filter 0 holds features of window_size 15"):
        b.set_camera_settings(None)
    with pytest.raises(EkfError, match="filter 0 holds features of window_size 15"):
        b.set_cameras(4)
    assert b.n_cameras == 2 and b.camera_settings.tolist() == [[15, 1, OFF], [15, 2, 3]]
    b.set_camera_settings([[15, 3, 7], [15, 1, OFF]])   # scale and blur may change under features
    assert all(np.array_equal(x, y) for x, y in zip(before, b.get_full(2)))
    out = np.zeros(15 * 15 + 1, np.uint8)
    assert b.L.ekf_batch_get_template(b.h, 0, 0, 0, out.ctypes.data_as(C.c_void_p)) == 0
    assert out[-1] == 0 and np.array_equal(out[:-1].reshape(15, 15), src.template(0))
