"""-m gpu: batched filters on cameras with their own frame times (ekf_batch_capture_camera_frames*, ekf_batch_step_filters).

A capture may list some cameras and a step some filters.  A listed filter runs exactly what a full step runs for it, so a
filter fed only its camera's frames must equal, bit for bit, a one-camera batch fed the same frames; an unlisted filter
and an unlisted camera stay exactly as they were."""
import ctypes as C

import numpy as np
import pytest

from helpers import INT_FIELDS

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

ERR_ARG, ERR_STATE = -1, -5


def _batches_equal(x, bx, y, by, ctx, every_mpatch=False):
    """Filter bx of batch x against filter by of batch y: mu, Sigma, tables, both templates, archive, bit for bit.  The
    matching template is compared for the features in the innovation set (a predict wrote it), or with every_mpatch for all
    (a feature added since the last predict has none yet)."""
    mx, Sx = x.get_full(bx); my, Sy = y.get_full(by)
    assert np.array_equal(mx, my) and np.array_equal(Sx, Sy), f"{ctx}: state"
    N = y.numOfFeatures(by)
    assert x.numOfFeatures(bx) == N, f"{ctx}: feature count {x.numOfFeatures(bx)} vs {N}"
    for i in range(N):
        a, c = x.feature(bx, i), y.feature(by, i)
        for f in INT_FIELDS:
            assert getattr(a, f) == getattr(c, f), f"{ctx}: feature {i} {f}"
        assert tuple(a.center) == tuple(c.center) and a.last_ncc == c.last_ncc, f"{ctx}: feature {i} match"
        for w in (0, 1) if (every_mpatch or a.is_in_innovation) else (0,):
            assert np.array_equal(x.template(bx, i, w), y.template(by, i, w)), f"{ctx}: feature {i} template {w}"
    dx, dy = x.deleted(bx), y.deleted(by)
    assert len(dx) == len(dy), f"{ctx}: archive size {len(dx)} vs {len(dy)}"
    for (ra, pa, ca), (rb, pb, cb) in zip(dx, dy):
        assert ra == rb and np.array_equal(pa, pb) and np.array_equal(ca, cb), f"{ctx}: archive record {ra}"


def _perturbed(mu0, B, seed, perturb=2e-3):
    rng = np.random.default_rng(seed)
    cams = np.tile(mu0[:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=perturb, size=(B, 3))
    cams[:, 3:7] += rng.normal(scale=perturb, size=(B, 4))
    cams[:, 3:7] /= np.linalg.norm(cams[:, 3:7], axis=1, keepdims=True)
    cams[:, 7:13] += rng.normal(scale=perturb, size=(B, 6))
    return cams


def _row(cfg):
    return np.array([cfg.fx, cfg.fy, cfg.u0, cfg.v0, cfg.k1, cfg.k2, cfg.k3, cfg.p1, cfg.p2])


def _seed(gpu_pkg, cfg, sc, cap):
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    return src


def test_full_list_is_todays_step(gpu_pkg):
    """64 cameras x 64 hypotheses, controls per filter, top-up and XYZ conversion on: step_filters over every filter gives
    step_controls' bits (mu and Sigma of every filter, tables and both templates of one filter per camera, counters,
    added features)."""
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=4, seed=900)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=20, xyz_conversion=1))
    K, M = 64, 64
    B = K * M
    src = _seed(gpu_pkg, cfg, sc, 32)
    cams = _perturbed(src.get_full()[0], B, 21)
    rng = np.random.default_rng(4)
    dv = rng.normal(scale=1e-3, size=(B, 3)); dw = rng.normal(scale=1e-3, size=(B, 3))
    vc = (np.arange(B) % 3 == 0).astype(np.int32)
    x, y = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=32) for _ in range(2))
    for z in (x, y):
        z.seed_from(src); z.set_cameras(K, np.repeat(np.arange(K), M)); z.set_camera_states(cams); z.set_topup(True)
    every = np.arange(B, dtype=np.int32)
    for t in range(1, sc.n_frames):
        base = sc.frame(t).astype(np.int16)
        fr = np.stack([np.clip(base + (c % 9) * 5 - 20, 0, 255).astype(np.uint8) for c in range(K)])
        stamps = sc.stamps[t] * (1.0 + 0.01 * np.arange(K))
        picks = sc.picks(t, 24)
        for z in (x, y):
            z.captureNewFrames(fr, stamps)
        x.step(picks, dv=dv, dw=dw, vcontrol=vc)
        y.step(picks, dv=dv, dw=dw, vcontrol=vc, filters=every)
        mx, Sx, stx = x.camera_states(want_sigma=True); my, Sy, sty = y.camera_states(want_sigma=True)
        assert np.array_equal(stx, sty) and np.array_equal(mx, my) and np.array_equal(Sx, Sy), f"frame {t}: camera states"
        assert np.array_equal(x.last_added(), y.last_added()), f"frame {t}: added"
        assert int(stx[:, 1].sum()) > 0
        for b in range(B):
            mxb, Sxb = x.get_full(b); myb, Syb = y.get_full(b)
            assert np.array_equal(mxb, myb) and np.array_equal(Sxb, Syb), f"frame {t} filter {b}: state"
        for c in range(K):
            _batches_equal(x, c * M + (c * 7) % M, y, c * M + (c * 7) % M, f"frame {t} camera {c}")


@pytest.mark.parametrize("cap,large", [(32, False), (48, True)])
@pytest.mark.parametrize("mode", ["blur", "plane"])
def test_rates_per_camera_are_separate_batches(gpu_pkg, cap, large, mode):
    """K = 4 cameras of three hypotheses each at four frame sizes, camera c delivering a frame every 1 + c % 3 ticks with its
    stamps; camera 2 once more at tick 5, between steps of its filters.  Each tick captures the cameras that delivered and steps the
    filters that follow them (controls per filter, intrinsics per filter, top-up, archive and XYZ conversion on).  Every filter
    equals, bit for bit, a one-camera batch fed only its camera's frames and stamps: state, tables, templates, archive,
    counters, blur counts and dT."""
    K, M = 4, 3
    B = K * M
    sizes = [(640, 480), (600, 450), (560, 420), (640, 400)]
    blur = mode == "blur"
    extra = dict(speed=0.9, omega=0.5, template_smooth=2.5) if blur else {}
    scenes = [gpu_pkg.synth.Scene(n_features=26, n_frames=11, seed=910 + c, width=sizes[c][0], height=sizes[c][1],
                                  planar=(mode == "plane"), **extra) for c in range(K)]
    cfgs = [gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=18, xyz_conversion=1, T_camera=0.5 if blur else 0.0))
            for sc in scenes]
    cfg = cfgs[0]
    rows = np.stack([_row(cfgs[c]) * (1.0 + 2e-4 * m) for c in range(K) for m in range(M)])
    src = _seed(gpu_pkg, cfg, scenes[0], cap)
    cams = _perturbed(src.get_full()[0], B, 23)
    rng = np.random.default_rng(8)
    dv = rng.normal(scale=1e-3, size=(B, 3)); dw = rng.normal(scale=1e-3, size=(B, 3))
    vc = (np.arange(B) % 2).astype(np.int32)

    empty = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)

    def make(n):
        z = gpu_pkg.FilterBatch(cfg, n, feature_capacity=cap, large=large)
        z.seed_from(empty)
        z.set_topup(True); z.set_archive(64); z.set_force_plane(mode == "plane")
        if blur:
            z.set_motion_blur(3)
        return z
    grouped = make(B)
    grouped.set_cameras(K, np.repeat(np.arange(K), M))
    grouped.set_intrinsics(rows); grouped.set_camera_states(cams); grouped.set_frame_sizes(sizes)
    parts = [make(M) for _ in range(K)]
    for c, p in enumerate(parts):
        p.set_intrinsics(rows[c * M:(c + 1) * M]); p.set_camera_states(cams[c * M:(c + 1) * M])
    grouped.captureNewFrames([sc.frame(0) for sc in scenes], [sc.stamps[0] for sc in scenes])
    for c, p in enumerate(parts):   # every filter starts from its own camera's scene
        p.captureNewFrame(scenes[c].frame(0), scenes[c].stamps[0])
        for m in range(M):
            for px in scenes[c].feature_pixels:
                assert grouped.addFeature(c * M + m, *px) == 1 and p.addFeature(m, *px) == 1
    steps, matched = np.zeros(K, int), np.zeros(K, int)
    blurred = 0
    for t in range(1, 11):
        cams_t = [c for c in range(K) if t % (1 + c % 3) == 0]
        if not cams_t:
            continue
        if t == 5:   # camera 2 (every third tick) delivers an extra frame between steps of its filters
            grouped.captureNewFrames([scenes[2].frame(5)], [scenes[2].stamps[5]], cameras=[2])
            parts[2].captureNewFrame(scenes[2].frame(5), scenes[2].stamps[5])
        order = cams_t[::-1]   # any order
        grouped.captureNewFrames([scenes[c].frame(t) for c in order], [scenes[c].stamps[t] for c in order], cameras=order)
        filt = np.concatenate([np.arange(c * M, (c + 1) * M) for c in cams_t]).astype(np.int32)
        picks = scenes[0].picks(t, 26)
        grouped.step(picks, dv=dv[filt], dw=dw[filt], vcontrol=vc[filt], filters=filt)
        _, stg = grouped.camera_states()
        rest = np.setdiff1d(np.arange(B), filt)
        assert not stg[rest].any(), f"tick {t}: counters of filters that did not step"
        for c in cams_t:
            p, s = parts[c], slice(c * M, (c + 1) * M)
            p.captureNewFrame(scenes[c].frame(t), scenes[c].stamps[t])
            p.step(picks, dv=dv[s], dw=dw[s], vcontrol=vc[s])
            _, stp = p.camera_states()
            ctx = f"tick {t} camera {c}"
            assert np.array_equal(stg[s], stp), f"{ctx}: counters"
            assert np.array_equal(grouped.last_added()[s], p.last_added()), f"{ctx}: added"
            assert np.array_equal(grouped.getDt()[s], p.getDt()), f"{ctx}: dT"
            if blur:
                assert np.array_equal(grouped.last_blur_counts()[s], p.last_blur_counts()), f"{ctx}: blur counts"
                blurred += int(p.last_blur_counts().sum())
            for m in range(M):
                _batches_equal(grouped, c * M + m, p, m, f"{ctx} hypothesis {m}")
            steps[c] += 1
            if t == 6 and c == 2:   # the last interval, as captureNewFrame twice on the single filter
                assert grouped.getDt()[2 * M] == scenes[2].stamps[6] - scenes[2].stamps[5]
            matched[c] += int(stp[:, 1].sum())
    assert (steps > 0).all() and len(set(steps.tolist())) > 1
    assert (matched > 0).all(), f"matches per camera {matched}"
    if blur:
        assert blurred > 0


def test_frozen_filters_are_untouched(gpu_pkg):
    """Three cameras of four filters, blur, top-up and archive on; cameras 0 and 2 step four times, camera 1's filters never.
    Against a twin batch that never steps, each of camera 1's filters keeps state, table, templates and archive, and its next
    added feature takes the same real_index; its counters, added and blur counts read zero.  camera_states equals the head of
    get_full for every filter, also after set_camera_states and set_full.  findNewFeatures(None) adds nothing to it."""
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=6, seed=930, speed=0.9, omega=0.5, template_smooth=2.5)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=22, xyz_conversion=1, T_camera=0.5))
    K, M = 3, 4
    B = K * M
    src = _seed(gpu_pkg, cfg, sc, 32)
    cams = _perturbed(src.get_full()[0], B, 31)
    x, y = (gpu_pkg.FilterBatch(cfg, B, feature_capacity=32) for _ in range(2))
    for z in (x, y):
        z.seed_from(src); z.set_cameras(K, np.repeat(np.arange(K), M)); z.set_camera_states(cams)
        z.set_topup(True); z.set_archive(32); z.set_motion_blur(3)
    frozen = np.arange(M, 2 * M)
    moving = np.array([f for f in range(B) if f not in frozen], np.int32)

    blurred = 0

    def heads_equal(ctx):
        mu, S, _ = x.camera_states(want_sigma=True)
        for f in range(B):
            m, Sf = x.get_full(f)
            assert np.array_equal(mu[f], m[:14]) and np.array_equal(S[f], Sf[:14, :14]), f"{ctx}: camera rows of filter {f}"
    first = np.stack([sc.frame(0)] * K)
    for z in (x, y):
        z.captureNewFrames(first, [sc.stamps[0]] * K)
    for t in range(1, 5):
        fr = np.stack([sc.frame(t)] * 2)
        x.captureNewFrames(fr, [sc.stamps[t]] * 2, cameras=[0, 2])
        y.captureNewFrames(fr, [sc.stamps[t]] * 2, cameras=[0, 2])
        x.step(sc.picks(t, 24), filters=moving)
        _, st = x.camera_states()
        assert not st[frozen].any() and not x.last_added()[frozen].any() and not x.last_blur_counts()[frozen].any()
        assert st[moving, 1].sum() > 0
        blurred += int(x.last_blur_counts()[moving].sum())
        heads_equal(f"step {t}")
    assert blurred > 0
    for f in frozen:
        _batches_equal(x, f, y, f, f"frozen filter {f}", every_mpatch=True)
    assert np.array_equal(x.num_deleted()[frozen], y.num_deleted()[frozen])
    # camera rows after set_camera_states / set_full, then a step of the others
    new = _perturbed(cams[0], B, 41)
    x.set_camera_states(new); y.set_camera_states(new)
    f0 = int(frozen[1])
    m, S = x.get_full(f0)
    m[0] += 1e-3
    x.set_full(f0, m, S); y.set_full(f0, m, S)
    x.captureNewFrames(np.stack([sc.frame(5)] * 2), [sc.stamps[5]] * 2, cameras=[0, 2])
    y.captureNewFrames(np.stack([sc.frame(5)] * 2), [sc.stamps[5]] * 2, cameras=[0, 2])
    x.step(sc.picks(5, 24), filters=moving)
    heads_equal("after set_camera_states / set_full")
    added = x.findNewFeatures(None)
    assert not added[frozen].any()
    for f in frozen:
        _batches_equal(x, f, y, f, f"frozen filter {f} after findNewFeatures(None)", every_mpatch=True)
    for f in frozen:   # the next feature's real_index
        assert x.addFeature(f, 300.0, 200.0) == 1 and y.addFeature(f, 300.0, 200.0) == 1
        n = x.numOfFeatures(f)
        assert x.feature(f, n - 1).real_index == y.feature(f, n - 1).real_index
        _batches_equal(x, f, y, f, f"frozen filter {f} after addFeature")


@pytest.mark.parametrize("scale", [1, 2, 10])
def test_subset_capture_is_the_full_capture(gpu_pkg, scale):
    """Five cameras at five frame sizes.  A capture of cameras (3, 1) after a full capture: the listed cameras' frames equal a
    full capture of the same images, bit for bit, gray from the host, gray from the device and BGR; the others keep their
    frame bytes and dT."""
    torch = pytest.importorskip("torch")
    K = 5
    W, H = 160 * scale, 120 * scale
    sizes = [(W, H), (W - 2 * scale - 1, H - 3 * scale), (W // 2 + 7, H - 1), (W - 9, H // 2 + 5), (W // 2 + 1, H // 2 + 1)]
    cfg = gpu_pkg.default_config(window_size=11)
    rng = np.random.default_rng(scale)
    first = rng.integers(0, 256, (K, H, W, 3), dtype=np.uint8)
    second = rng.integers(0, 256, (K, H, W, 3), dtype=np.uint8)
    lst = [3, 1]

    def make():
        z = gpu_pkg.FilterBatch(cfg, K, feature_capacity=8)
        z.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=8))
        z.set_scale(scale); z.set_cameras(K); z.set_frame_sizes(sizes)
        return z
    for kind in ("gray", "gray_device", "bgr"):
        x, ref = make(), make()
        conv = (lambda a: a) if kind == "bgr" else (lambda a: np.ascontiguousarray(np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in a])))
        a, b = conv(first), conv(second)
        x.captureNewFrames(a, np.arange(K) + 1.0)
        before = [x.returnGrayImg(c) for c in range(K)]
        dt0 = x.getDt()
        if kind == "gray_device":
            t = torch.from_numpy(np.ascontiguousarray(b[lst])).cuda()
            torch.cuda.synchronize()
            x.captureNewFrames_device(t.data_ptr(), W, H, W, [10.0, 20.0], cameras=lst)
        else:
            x.captureNewFrames(b[lst], [10.0, 20.0], cameras=lst)
        full = a.copy()
        full[lst] = b[lst]
        ref.captureNewFrames(full)
        for c in range(K):
            got = x.returnGrayImg(c)
            if c in lst:
                assert np.array_equal(got, ref.returnGrayImg(c)), f"{kind} camera {c}: differs from the full capture"
                assert got.shape == (sizes[c][1] // scale, sizes[c][0] // scale)
            else:
                assert np.array_equal(got, before[c]), f"{kind} camera {c}: changed by a capture that did not list it"
        dt = x.getDt()
        assert dt[3] == 10.0 - 4.0 and dt[1] == 20.0 - 2.0
        assert np.array_equal(dt[[0, 2, 4]], dt0[[0, 2, 4]])


def test_errors_leave_the_batch_unchanged(gpu_pkg):
    sc = gpu_pkg.synth.Scene(n_features=12, n_frames=4, seed=950)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    K, M = 3, 2
    B = K * M
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
    batch.seed_from(_seed(gpu_pkg, cfg, sc, 16))
    batch.set_cameras(K, np.repeat(np.arange(K), M))
    L, h = batch.L, batch.h
    ip = lambda *v: (C.c_int32 * len(v))(*v)   # noqa: E731
    img = np.ascontiguousarray(sc.frame(1))
    W, H = img.shape[1], img.shape[0]
    one = img.ctypes.data_as(C.c_void_p)
    # no camera holds a frame: the first subset capture defines the slot; the other cameras stay without a frame
    batch.captureNewFrames(img[None], [sc.stamps[1]], cameras=[0])
    w, hh = C.c_int(0), C.c_int(0)
    assert L.ekf_batch_get_camera_frame(h, 1, None, C.byref(w), C.byref(hh)) == ERR_STATE
    assert L.ekf_batch_step_filters(h, 1, ip(2), None, None, None, None, 0) == ERR_STATE        # filter 2 follows camera 1
    assert L.ekf_batch_step(h, None, None, 0, None, 0) == ERR_STATE
    assert b"captureNewFrame" in L.ekf_batch_last_error(h)
    assert L.ekf_batch_add_feature(h, 3, 100.0, 100.0) == ERR_STATE
    num = np.zeros(B, np.int32); num[2] = 5
    xy = np.zeros((B, 32, 2), np.float32); n = np.zeros(B, np.int32)
    assert L.ekf_batch_detect_corners(h, num.ctypes.data_as(C.c_void_p), xy.ctypes.data_as(C.c_void_p),
                                      n.ctypes.data_as(C.c_void_p)) == ERR_STATE
    assert L.ekf_batch_find_new_features(h, num.ctypes.data_as(C.c_void_p), None) == ERR_STATE
    num[:] = 0; num[1] = 5                                                                      # camera 0's filter: fine
    assert L.ekf_batch_detect_corners(h, num.ctypes.data_as(C.c_void_p), xy.ctypes.data_as(C.c_void_p),
                                      n.ctypes.data_as(C.c_void_p)) == 0
    batch.step(sc.picks(1, 12), filters=[0, 1])
    # argument errors change nothing
    state = [batch.get_full(f) for f in range(B)]
    frame0, dt = batch.returnGrayImg(0), batch.getDt()
    for lst in ((1, 0), (0, 0), (-1,), (B,), (0, 1, 1)):
        assert L.ekf_batch_step_filters(h, len(lst), ip(*lst), None, None, None, None, 0) == ERR_ARG, lst
    assert L.ekf_batch_step_filters(h, 0, ip(0), None, None, None, None, 0) == ERR_ARG
    assert L.ekf_batch_step_filters(h, 1, None, None, None, None, None, 0) == ERR_ARG
    stamps = (C.c_double * 3)(5.0, 6.0, 7.0)
    two = np.ascontiguousarray(np.stack([img, img]))
    tp = two.ctypes.data_as(C.c_void_p)
    for lst in ((0, 0), (-1, 0), (K, 0), (0, 1, 0)):
        assert L.ekf_batch_capture_camera_frames(h, len(lst), ip(*lst), tp, W, H, W, stamps) == ERR_ARG, lst
    assert L.ekf_batch_capture_camera_frames(h, 0, ip(0), one, W, H, W, stamps) == ERR_ARG
    assert L.ekf_batch_capture_camera_frames(h, K + 1, ip(0, 1, 2, 0), tp, W, H, W, stamps) == ERR_ARG
    assert L.ekf_batch_capture_camera_frames(h, 1, None, one, W, H, W, stamps) == ERR_ARG
    small = np.ascontiguousarray(img[:H - 16, :W - 16])                                         # another slot while camera 0 holds a frame
    assert L.ekf_batch_capture_camera_frames(h, 1, ip(1), small.ctypes.data_as(C.c_void_p), W - 16, H - 16, W - 16, stamps) == ERR_ARG
    assert b"slot" in L.ekf_batch_last_error(h)
    bgr = np.ascontiguousarray(np.stack([cv2.cvtColor(img, cv2.COLOR_GRAY2BGR)] * 2))
    assert L.ekf_batch_capture_camera_frames_bgr(h, 2, ip(2, 2), bgr.ctypes.data_as(C.c_void_p), W, H, 3 * W, stamps) == ERR_ARG
    for f in range(B):
        m, S = batch.get_full(f)
        assert np.array_equal(m, state[f][0]) and np.array_equal(S, state[f][1]), f"filter {f}"
    assert np.array_equal(batch.returnGrayImg(0), frame0) and np.array_equal(batch.getDt(), dt)
    assert L.ekf_batch_get_camera_frame(h, 1, None, C.byref(w), C.byref(hh)) == ERR_STATE
    # a full capture of another slot is allowed; set_frame_sizes forgets every frame
    batch.captureNewFrames(np.stack([small] * K))
    assert batch.returnGrayImg(2).shape == small.shape
    batch.set_frame_sizes([[W - 16, H - 16]] * K)
    assert L.ekf_batch_get_camera_frame(h, 0, None, C.byref(w), C.byref(hh)) == ERR_STATE
    with pytest.raises(ValueError):
        batch.step(sc.picks(2, 12), filters=[])
