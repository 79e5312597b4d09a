"""-m gpu: batched filters on cameras of their own (ekf_batch_set_cameras).

Filter b follows camera camera_of[b]: its frame and time stamp are its camera's, its controls its own (ekf_batch_step_controls).
Every filter still runs the single filter's algorithm, so a filter on camera c must follow a single CUDA filter fed camera c's
frames bit for bit in its feature table and templates, and a batch of grouped cameras must equal separate one-camera batches
bit for bit.  One camera is today's batch: same bits, same launches."""
import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, assert_scaled_close, relerr, seed_features

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

BLUR_SCENE = dict(speed=0.9, omega=0.5, template_smooth=2.5)


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
        assert tuple(a.center) == tuple(c.center)
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


def _textured(seed, W=320, H=240):
    rng = np.random.default_rng(seed)
    img = cv2.GaussianBlur(rng.integers(0, 256, (H, W)).astype(np.float32), (0, 0), 2.5)
    img = (img - img.min()) / (img.max() - img.min()) * 160 + 40
    for _ in range(30):
        x, y = int(rng.integers(10, W - 50)), int(rng.integers(10, H - 50))
        img[y:y + int(rng.integers(8, 30)), x:x + int(rng.integers(8, 30))] += rng.uniform(-40, 40)
    return np.clip(img, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("cap,large,nfind,minf", [(32, False, 20, 15), (100, True, 60, 45)])
def test_independent_sequences_follow_single_filters(gpu_pkg, cap, large, nfind, minf):
    """Six scenes (one hard, one planar) on six cameras with stamps at 30, 25 and 15 fps and controls per filter, from an empty
    seed and findNewFeatures on every camera's frame 0; top-up and XYZ conversion on.  Each filter against a single CUDA filter
    fed its scene: tables and templates bit-exact, state within 1e-8, getDt equal, every step."""
    fps = [30.0, 25.0, 15.0, 30.0, 25.0, 15.0]
    scenes = [gpu_pkg.synth.Scene(n_features=40, n_frames=13, seed=600 + c, fps=fps[c], hard=(c == 1), planar=(c == 2))
              for c in range(6)]
    cfg = gpu_pkg.default_config(**dict(scenes[0].config_overrides(), min_features=minf, max_features=1000, xyz_conversion=1))
    B = 6
    rng = np.random.default_rng(7)
    dv = rng.normal(scale=1e-3, size=(B, 3)); dw = rng.normal(scale=1e-3, size=(B, 3))
    vc = np.array([0, 1, 0, 1, 1, 0], dtype=np.int32)
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap, large=large)
    batch.seed_from(src)
    batch.set_cameras(B)
    batch.set_topup(True)
    singles = [gpu_pkg.VSlamFilter(cfg, feature_capacity=cap) for _ in range(B)]
    batch.captureNewFrames(np.stack([sc.frame(0) for sc in scenes]), [sc.stamps[0] for sc in scenes])
    added = batch.findNewFeatures(nfind)
    for b, (s, sc) in enumerate(zip(singles, scenes)):
        s.captureNewFrame(sc.frame(0), sc.stamps[0])
        assert s.findNewFeatures(nfind) == added[b]
        _tables_equal(batch, b, s, f"frame 0 filter {b}")
    assert (added > 0).all()
    for t in range(1, 13):
        picks = scenes[0].picks(t, 64)
        batch.captureNewFrames(np.stack([sc.frame(t) for sc in scenes]), [sc.stamps[t] for sc in scenes])
        batch.step(picks, dv=dv, dw=dw, vcontrol=vc)
        dts = batch.getDt()
        for b, (s, sc) in enumerate(zip(singles, scenes)):
            s.captureNewFrame(sc.frame(t), sc.stamps[t]); s.predict(dv[b], dw[b], bool(vc[b])); s.update(picks)
            ctx = f"frame {t} filter {b}"
            assert dts[b] == s.getDt() and batch.view(b).getDt() == s.getDt(), f"{ctx}: dT"
            _tables_equal(batch, b, s, ctx)
            mb, Sb = batch.get_full(b); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"{ctx}: mu {relerr(mb, ms):.2e} Sigma {relerr(Sb, Ss):.2e}"
    assert len({round(d, 6) for d in batch.getDt()}) == 3


@pytest.mark.parametrize("window,blur,plane", [(11, True, False), (11, False, True), (21, False, False)])
def test_grouped_cameras_are_separate_batches(gpu_pkg, window, blur, plane):
    """3 cameras x 5 perturbed hypotheses against three one-camera batches of 5 on the same frames: each camera's frames are the
    scene's with its own brightness offset and noise (same predicted positions, different pixels and templates) and its own
    clock.  mu, Sigma, tables, templates and counters bit-identical every step."""
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=8, seed=640, window=window, **(BLUR_SCENE if blur else {}))
    over = dict(sc.config_overrides(), T_camera=0.5 if blur else 0.0)
    cfg = gpu_pkg.default_config(**over)
    K, M = 3, 5
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    cams = _perturbed(src.get_full()[0], K * M, 9)
    rng = np.random.default_rng(3)

    def frames(t):
        out = []
        for c in range(K):
            f = sc.frame(t).astype(np.int16) + 12 * c + rng.integers(-2, 3, sc.frame(t).shape) * (c > 0)
            out.append(np.clip(f, 0, 255).astype(np.uint8))
        return np.stack(out)

    def make(n):
        b = gpu_pkg.FilterBatch(cfg, n, feature_capacity=32)
        b.seed_from(src)
        if blur:
            b.set_motion_blur(3)
        b.set_force_plane(plane)
        return b
    grouped = make(K * M)
    grouped.set_cameras(K, np.repeat(np.arange(K), M))
    grouped.set_camera_states(cams)
    parts = [make(M) for _ in range(K)]
    for c, p in enumerate(parts):
        p.set_camera_states(cams[c * M:(c + 1) * M])
    blurred = matched = 0
    for t in range(1, sc.n_frames):
        fr = frames(t)
        stamps = np.array([sc.stamps[t] * (1.0 + 0.25 * c) for c in range(K)])
        picks = sc.picks(t, 24)
        grouped.captureNewFrames(fr, stamps); grouped.step(picks)
        _, stg = grouped.camera_states()
        for c, p in enumerate(parts):
            p.captureNewFrame(fr[c], stamps[c]); p.step(picks)
            _, stp = p.camera_states()
            assert np.array_equal(stg[c * M:(c + 1) * M], stp), f"frame {t} camera {c}: counters"
            if blur:
                assert np.array_equal(grouped.last_blur_counts()[c * M:(c + 1) * M], p.last_blur_counts())
                blurred += int(p.last_blur_counts().sum())
            assert np.array_equal(grouped.getDt()[c * M:(c + 1) * M], p.getDt())
            for m in range(M):
                _batches_equal(grouped, c * M + m, p, m, f"frame {t} camera {c} hypothesis {m}")
        matched += int(stg[:, 1].sum())
    assert matched > 0
    if blur:
        assert blurred > 0


def test_one_camera_is_todays_batch(gpu_pkg):
    """set_cameras(1) + captureNewFrames of a stack of one + controls per filter (equal rows) against captureNewFrame + step:
    bit-identical states and the same kernel launches."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=650)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=16, xyz_conversion=1))
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    B = 4
    cams = _perturbed(src.get_full()[0], B, 11)
    x, y = gpu_pkg.FilterBatch(cfg, B, feature_capacity=32), gpu_pkg.FilterBatch(cfg, B, feature_capacity=32)
    for z in (x, y):
        z.seed_from(src); z.set_camera_states(cams); z.set_topup(True)
    y.set_cameras(1, np.zeros(B, np.int32))
    dv, dw = np.array([1e-3, -2e-3, 5e-4]), np.array([-1e-3, 1e-3, 2e-4])
    for t in range(1, sc.n_frames):
        picks = sc.picks(t, 20)
        lx, ly = x.kernel_launches(), y.kernel_launches()
        x.captureNewFrame(sc.frame(t), sc.stamps[t]); x.step(picks, dv=dv, dw=dw, vcontrol=True)
        y.captureNewFrames(sc.frame(t)[None], [sc.stamps[t]]); y.step(picks, dv=np.tile(dv, (B, 1)), dw=np.tile(dw, (B, 1)),
                                                                     vcontrol=np.ones(B, np.int32))
        assert x.kernel_launches() - lx == y.kernel_launches() - ly, f"frame {t}: launches"
        assert np.array_equal(x.camera_states()[1], y.camera_states()[1])
        for b in range(B):
            _batches_equal(x, b, y, b, f"frame {t} filter {b}")
        assert np.array_equal(x.returnGrayImg(), y.returnGrayImg(0))


@pytest.mark.parametrize("cap,large", [(12, False), (100, True)])
def test_detector_per_camera(gpu_pkg, cap, large):
    """12 cameras of 2 filters each with different patches; cameras 3 and 8 asked nothing.  A budget of 5 cameras' scratch
    makes one call span three chunks.  Each filter's corners, in order, are a single filter's detect_corners on its camera's
    frame with the same patch centres; findNewFeatures adds exactly those."""
    W, H = 320, 240
    K, M = 12, 2
    B = K * M
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    imgs = np.stack([_textured(700 + c, W, H) for c in range(K)])
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    src.captureNewFrame(imgs[0], 1.0)
    for p in [(60.0, 60.0), (160.0, 120.0)]:
        assert src.addFeature(*p) == 1
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap, large=large)
    batch.seed_from(src)
    batch.set_cameras(K, np.arange(B) // M)
    batch.set_detect_budget(5 * 36 * W * H)
    batch.captureNewFrames(imgs, None)
    rng = np.random.default_rng(5)
    for b in range(B):
        for u, v in rng.uniform(20, 220, (b % 5, 2)):
            assert batch.addFeature(b, u, v) == 1
    num = np.array([(7 + 3 * b) % 33 for b in range(B)], dtype=np.int32)
    num[[3 * M, 3 * M + 1, 8 * M, 8 * M + 1]] = 0
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
    ask = num * (2 if large else 1)
    wants = [(single(b).detect_corners(int(ask[b])) if ask[b] > 0 else np.zeros((0, 2), np.float32))[:cap - N0[b]] for b in range(B)]
    added = batch.findNewFeatures(ask)
    for b in range(B):
        want = wants[b]
        assert added[b] == len(want), f"filter {b}: added {added[b]} vs {len(want)}"
        new = np.array([batch.feature(b, i).center for i in range(N0[b], batch.numOfFeatures(b))], np.float32).reshape(-1, 2)
        assert np.array_equal(new, want), f"filter {b}: added corners"


@pytest.mark.parametrize("scale", [2, 10])
def test_stacks_of_resized_and_bgr_frames(gpu_pkg, scale):
    """Each camera's returnGrayImg(c) equals cv2 resize + cvtColor and a single filter's frame, bit for bit, for a host BGR
    stack, a host gray stack with padded rows and a device gray stack.  At scale 10 the BGR stack (72 frames of 1600 x 1200,
    5.76 MB each, 415 MB) is staged 46 cameras at a time (256 MB); the cameras checked include both sides of that boundary."""
    torch = pytest.importorskip("torch")
    W, H = 160 * scale, 120 * scale
    K = 72 if scale == 10 else 5
    cfg = gpu_pkg.default_config(window_size=11)
    rng = np.random.default_rng(scale)
    base = rng.integers(0, 256, (4, H, W, 3), dtype=np.uint8)
    bgr = np.stack([np.roll(base[c % 4], 7 * c, axis=1) for c in range(K)])
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=8)
    batch = gpu_pkg.FilterBatch(cfg, K, feature_capacity=8)
    batch.seed_from(src)
    batch.set_scale(scale)
    batch.set_cameras(K)
    single = gpu_pkg.VSlamFilter(gpu_pkg.default_config(window_size=11, scale=scale), feature_capacity=8)
    gray = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr[:5]])
    padded = np.zeros((5, H, W + 24), np.uint8); padded[:, :, :W] = gray
    for kind in ("bgr", "gray_padded", "gray_device"):
        if kind == "bgr":
            batch.captureNewFrames(bgr)
            frames = bgr
        elif kind == "gray_padded":
            batch.set_cameras(5, np.arange(K) % 5)
            batch.captureNewFrames(padded[:, :, :W])
            frames = gray
        else:
            t = torch.from_numpy(gray).cuda()
            torch.cuda.synchronize()
            batch.captureNewFrames_device(t.data_ptr(), W, H, W)
            frames = gray
        for c in range(len(frames)) if kind != "bgr" or K == 5 else (0, 1, 45, 46, 71):
            want = cv2.resize(frames[c], (W // scale, H // scale))
            if frames[c].ndim == 3:
                want = cv2.cvtColor(want, cv2.COLOR_BGR2GRAY)
            got = batch.returnGrayImg(c)
            assert np.array_equal(got, want), f"{kind} camera {c}: differs from cv2"
            single.captureNewFrame(frames[c], 1.0)
            assert np.array_equal(got, single.returnGrayImg()), f"{kind} camera {c}: differs from the single filter"


def test_errors(gpu_pkg):
    sc = gpu_pkg.synth.Scene(n_features=10, n_frames=3, seed=660)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=16)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        src.addFeature(*p)
    B = 4
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=16)
    batch.seed_from(src)
    L, h = batch.L, batch.h
    ERR_ARG, ERR_STATE = -1, -5
    import ctypes as C
    good = (C.c_int32 * B)(0, 1, 1, 0)
    assert L.ekf_batch_set_cameras(h, 0, good) == ERR_ARG
    assert L.ekf_batch_set_cameras(h, B + 1, None) == ERR_ARG
    assert L.ekf_batch_set_cameras(h, 2, None) == ERR_ARG                      # NULL = identity needs n == B
    assert L.ekf_batch_set_cameras(h, 2, (C.c_int32 * B)(0, 1, 2, 0)) == ERR_ARG
    assert L.ekf_batch_set_cameras(h, 2, (C.c_int32 * B)(0, -1, 1, 0)) == ERR_ARG
    batch.captureNewFrame(sc.frame(1), sc.stamps[1])                            # still one camera: accepted
    assert L.ekf_batch_set_cameras(h, 2, good) == 0
    batch.n_cameras = 2
    assert L.ekf_batch_step(h, None, None, 0, None, 0) == ERR_STATE             # a step after set_cameras before a capture
    assert b"captureNewFrame" in L.ekf_batch_last_error(h)
    img = np.ascontiguousarray(sc.frame(1))
    ptr = img.ctypes.data_as(C.c_void_p)
    assert L.ekf_batch_capture_frame(h, ptr, 640, 480, 640, 1.0) == ERR_STATE
    assert b"ekf_batch_capture_frames" in L.ekf_batch_last_error(h)
    assert L.ekf_batch_capture_frame_device(h, ptr, 640, 480, 640, 1.0) == ERR_STATE
    assert L.ekf_batch_capture_frame_bgr(h, ptr, 640, 160, 1920, 1.0) == ERR_STATE
    stack = np.ascontiguousarray(np.stack([sc.frame(1), sc.frame(2)]))
    assert L.ekf_batch_capture_frames(h, stack.ctypes.data_as(C.c_void_p), 640, 480, 639, None) == ERR_ARG   # stride < width
    batch.captureNewFrames(stack, [sc.stamps[1], sc.stamps[2]])
    w, hh = C.c_int(0), C.c_int(0)
    assert L.ekf_batch_get_frame(h, None, C.byref(w), C.byref(hh)) == ERR_STATE
    assert b"ekf_batch_get_camera_frame" in L.ekf_batch_last_error(h)
    assert L.ekf_batch_get_camera_frame(h, 2, None, C.byref(w), C.byref(hh)) == ERR_ARG
    assert np.array_equal(batch.returnGrayImg(1), sc.frame(2))
    batch.step(sc.picks(1, 10))
    assert L.ekf_batch_set_detect_budget(h, 0) == ERR_ARG


def test_distinct_cameras_against_oracle(gpu_pkg, orc):
    """Three filters on three cameras: three scenes (one hard) with stamps at 30, 25 and 15 fps and controls per filter.  Each
    step from identical inputs (batch state <- oracle state) against an oracle fed its own camera's frame, stamp and controls:
    counters and tables bit-exact (matches, NCC scores), state within TOL and the scaled bars."""
    fps = [30.0, 25.0, 15.0]
    scenes = [gpu_pkg.synth.Scene(n_features=20, n_frames=7, seed=680 + c, fps=fps[c], hard=(c == 1)) for c in range(3)]
    cfg = gpu_pkg.default_config(**scenes[0].config_overrides())
    B = 3
    rng = np.random.default_rng(13)
    dv = rng.normal(scale=1e-3, size=(B, 3)); dw = rng.normal(scale=1e-3, size=(B, 3))
    vc = np.array([1, 0, 1], dtype=np.int32)
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=32)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=32))
    batch.set_cameras(B)
    batch.captureNewFrames(np.stack([sc.frame(0) for sc in scenes]), [sc.stamps[0] for sc in scenes])
    oracles = []
    for b, sc in enumerate(scenes):
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
        batch.captureNewFrames(np.stack([sc.frame(t) for sc in scenes]), [sc.stamps[t] for sc in scenes])
        batch.step(picks, dv=dv, dw=dw, vcontrol=vc)
        mu14, S14, st = batch.camera_states(want_sigma=True)
        for b, (o, sc) in enumerate(zip(oracles, scenes)):
            ctx = f"frame {t} filter {b}"
            o.captureNewFrame(sc.frame(t), sc.stamps[t]); o.predict(dv[b], dw[b], bool(vc[b])); o.update(picks)
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


def _near_tie_frames(W=640, H=480):
    """Images that make the tile matcher hand near-ties to the CTA matcher (as helpers.near_tie_scene, full size): a smooth
    gradient, an exactly periodic texture and a coarse four-level block image."""
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:H, 0:W]
    smooth = (127 + 60 * np.sin(xx / 23.0) + 50 * np.cos(yy / 17.0) + rng.normal(scale=1.5, size=(H, W))).clip(0, 255)
    periodic = (((xx % 8) * 16 + (yy % 8) * 12) % 256).astype(np.float64)
    coarse = ((rng.integers(0, 4, size=(H // 4 + 1, W // 4 + 1)).repeat(4, 0).repeat(4, 1)[:H, :W]) * 64).astype(np.float64)
    return np.stack([smooth, periodic, coarse]).astype(np.uint8)


def test_deferred_matcher_reads_the_cameras_frame(gpu_pkg):
    """Window 11 on frames with near-ties: the tile matcher defers some features to the CTA matcher, which stages its windows
    through the 3-D tensor map of the stack (z = camera).  Three cameras with different images, two filters each; every filter
    against a single CUDA filter on its camera's frames: tables, NCC scores and templates bit-exact."""
    base = _near_tie_frames()
    K, M = 3, 2
    B = K * M
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=32)
    batch.seed_from(gpu_pkg.VSlamFilter(cfg, feature_capacity=32))
    batch.set_cameras(K, np.arange(B) // M)
    stamps = lambda t: [t / 30.0] * K   # noqa: E731
    batch.captureNewFrames(base, stamps(0))
    nfind = np.array([20, 12, 20, 12, 20, 12], dtype=np.int32)
    added = batch.findNewFeatures(nfind)
    singles = []
    for b in range(B):
        s = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
        s.captureNewFrame(base[b // M], 0.0)
        assert s.findNewFeatures(int(nfind[b])) == added[b] > 0
        singles.append(s)
    deferred = 0
    for t in range(1, 4):
        fr = np.stack([np.roll(base[c], t, axis=1) for c in range(K)])
        picks = np.arange(1, 41, dtype=np.uint32) * 7919
        batch.captureNewFrames(fr, stamps(t)); batch.step(picks)
        deferred += batch.last_match_deferred()
        for b, s in enumerate(singles):
            s.captureNewFrame(fr[b // M], t / 30.0); s.predict(); s.update(picks)
            _tables_equal(batch, b, s, f"frame {t} filter {b}")
            mb, Sb = batch.get_full(b); ms, Ss = s.get_full()
            assert relerr(mb, ms) <= 1e-8 and relerr(Sb, Ss) <= 1e-8, f"frame {t} filter {b}"
    assert deferred > 0, "no feature reached the CTA matcher"
