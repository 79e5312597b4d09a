"""-m gpu: resized and BGR frames (captureNewFrame's scale / BGR path, vslamRansac.cpp:226-245) and the forsePlane
pseudo-measurement (vslamRansac.cpp:1245-1272) in the batched filters.

ekf_batch_create refuses scale != 1 and forsePlane; both are switched on after creation (FilterBatch.set_scale /
set_force_plane, or FilterBatch.from_config with a single filter's configuration).  A batch's frame must be the single
filter's and cv2's bit for bit; a step with forsePlane the oracle's (tables bit-exact, the state within the per-step bars);
filter 0 must follow a single CUDA filter; the simulation setup (conf_sim.cfg's switches) must run end to end; and with the
switches off a batch must run exactly as one that never had them."""
import ctypes as C

import numpy as np
import pytest

from helpers import relerr, seed_features
from test_gpu_batch_blur import BLUR_SCENE, _moving
from test_gpu_batch_topup import _centers, _check, _perturbed, _single_with

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _blow_up(gray, s):
    """A BGR frame s times larger whose resize by 1 / s and BGR2GRAY give `gray` back exactly: constant s x s blocks of three
    equal channels (INTER_LINEAR / INTER_AREA of a constant block is the constant; BGR2GRAY's weights sum to 1 << 15)."""
    return np.kron(gray[:, :, None], np.ones((s, s, 3), dtype=np.uint8))


def _padded(img, pad):
    """img inside rows of stride row_bytes + pad, and that stride."""
    row = img.shape[1] * (img.shape[2] if img.ndim == 3 else 1)
    buf = np.full((img.shape[0], row + pad), 77, dtype=np.uint8)
    buf[:, :row] = img.reshape(img.shape[0], row)
    return buf, row + pad


def _raw_capture(batch, name, img, stride, stamp=-1.0, width=None):
    """The C entry `name` on a host buffer with an explicit stride (width: pixels a row, default img.shape[1]); returns its
    code."""
    w = img.shape[1] if width is None else width
    return getattr(batch.L, name)(batch.h, img.ctypes.data_as(C.c_void_p), w, img.shape[0], stride, float(stamp))


@pytest.mark.parametrize("scale", [2, 3, 10])
def test_frames_equal_single_filter_and_cv2(gpu_pkg, scale):
    """Gray and BGR from the host (contiguous and with padded rows) and gray from the device: batch.returnGrayImg() equals a
    single filter's returnGrayImg() on the same input and cv2 resize + cvtColor, bit for bit."""
    torch = pytest.importorskip("torch")
    H, W = (1080, 1920) if scale == 10 else (481, 643)
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    batch = gpu_pkg.FilterBatch(cfg, 2, feature_capacity=8)
    batch.set_scale(scale)
    single = gpu_pkg.VSlamFilter(gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0, scale=scale),
                                 feature_capacity=8)
    rng = np.random.default_rng(scale)
    for kind in ("gray", "bgr", "gray_padded", "bgr_padded", "device"):
        img = rng.integers(0, 256, (H, W, 3) if kind.startswith("bgr") else (H, W), dtype=np.uint8)
        want = cv2.resize(img, (W // scale, H // scale))
        if img.ndim == 3:
            want = cv2.cvtColor(want, cv2.COLOR_BGR2GRAY)
        if kind == "device":
            t = torch.from_numpy(img).cuda()
            torch.cuda.synchronize()
            batch.captureNewFrame_device(t.data_ptr(), W, H, t.stride(0))
            single.captureNewFrame_device(t.data_ptr(), W, H, t.stride(0))
        elif kind.endswith("padded"):
            buf, stride = _padded(img, 13)
            fn = "ekf_batch_capture_frame_bgr" if img.ndim == 3 else "ekf_batch_capture_frame"
            assert _raw_capture(batch, fn, buf, stride, width=W) == 0
            single.captureNewFrame(img)
        else:
            batch.captureNewFrame(img)
            single.captureNewFrame(img)
        got = batch.returnGrayImg()
        assert got.shape == (H // scale, W // scale), kind
        assert np.array_equal(got, want), f"{kind}: {(got != want).sum()} of {want.size} pixels differ from cv2"
        assert np.array_equal(got, single.returnGrayImg()), f"{kind}: differs from the single filter"


def test_capture_arguments(gpu_pkg):
    """EKF_ERR_STATE before a frame; EKF_ERR_ARG for a scale < 1, a resized side below 8 px and a stride shorter than a row
    (BGR: 3 bytes a pixel).  A refused capture leaves the frame as it was."""
    abi = gpu_pkg._abi
    batch = gpu_pkg.FilterBatch(gpu_pkg.default_config(window_size=11, xyz_conversion=0), 2, feature_capacity=8)
    w, h = C.c_int(0), C.c_int(0)
    assert batch.L.ekf_batch_get_frame(batch.h, None, C.byref(w), C.byref(h)) == abi.EKF_ERR_STATE
    for bad in (0, -3, 65):
        assert batch.L.ekf_batch_set_scale(batch.h, bad) == abi.EKF_ERR_ARG
    batch.set_scale(10)
    ok = np.full((80, 80, 3), 9, dtype=np.uint8)
    batch.captureNewFrame(ok, 1.0)
    assert batch.returnGrayImg().shape == (8, 8)
    for shape in ((80, 79), (79, 80)):   # 7 px after the resize
        for ch in (1, 3):
            img = np.zeros(shape + ((3,) if ch == 3 else ()), dtype=np.uint8)
            fn = "ekf_batch_capture_frame_bgr" if ch == 3 else "ekf_batch_capture_frame"
            assert _raw_capture(batch, fn, img, shape[1] * ch, 2.0) == abi.EKF_ERR_ARG, (shape, ch)
    big = np.zeros((160, 160, 3), dtype=np.uint8)
    assert _raw_capture(batch, "ekf_batch_capture_frame_bgr", big, 160 * 3 - 1) == abi.EKF_ERR_ARG
    assert _raw_capture(batch, "ekf_batch_capture_frame", big[:, :, 0].copy(), 159) == abi.EKF_ERR_ARG
    assert batch.returnGrayImg().shape == (8, 8) and (batch.returnGrayImg() == 9).all()
    batch.set_scale(1)
    assert _raw_capture(batch, "ekf_batch_capture_frame_bgr", np.zeros((7, 40, 3), dtype=np.uint8), 120) == abi.EKF_ERR_ARG


def test_dt_follows_stamps_through_resize(gpu_pkg):
    """BGR frames blown up 2x at scale 2: filter 0 of a batch from from_config and a single filter with the same configuration
    step through the same frames and stamps.  The batch works on the scene's frame, and its filter 0 stays with the single
    filter to the free-running bar; a dT that did not follow the stamps would move the prediction by orders more."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=41)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), scale=2))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    g.captureNewFrame(_blow_up(sc.frame(0), 2), sc.stamps[0])
    for p in sc.feature_pixels:
        assert g.addFeature(*p) == 1
    batch = gpu_pkg.FilterBatch.from_config(cfg, 2)
    batch.seed_from(g)
    for t in range(1, sc.n_frames):
        big, picks = _blow_up(sc.frame(t), 2), sc.picks(t, 20)
        batch.captureNewFrame(big, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(big, sc.stamps[t]); g.predict(); g.update(picks)
        assert np.array_equal(batch.returnGrayImg(), sc.frame(t)), f"frame {t}"
        assert abs(g.getDt() - (sc.stamps[t] - sc.stamps[t - 1])) < 1e-12
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert mb.shape == mg.shape and relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}"
        assert g.stats().n_matched > 0


def _oracles(orc, cfg_o, g, img0, stamp0, cams):
    mu0, S0 = g.get_full()
    out = []
    for cam in cams:
        o = orc.OracleFilter(cfg_o, kind=0, omp=False)
        o.captureNewFrame(img0, stamp0); o.import_from(g)
        m = mu0.copy(); m[:14] = cam
        o.set_full(m, S0)
        out.append(o)
    return out


def test_force_plane_step_against_oracle(gpu_pkg, orc):
    """Filters 0-2 of a perturbed ensemble with set_force_plane(1), per step from identical inputs (batch state <- oracle
    state), on the single filter's forsePlane scenes (hard False / True): tables bit-exact, n_li / n_hi equal, the state within
    TOL and the scaled bars.  Both kinds of second update must occur: the plane rows alone (n_hi = 0) and beside Hi rows.  A
    batch with the plane off, fed the same state, must end elsewhere: the plane rows do act."""
    plane_only = with_hi = 0
    moved = 0.0
    for hard in (False, True):
        sc = gpu_pkg.synth.Scene(n_features=30, n_frames=5, seed=61, hard=hard)
        cfg_b = gpu_pkg.default_config(**sc.config_overrides())
        cfg_o = gpu_pkg.default_config(**dict(sc.config_overrides(), forsePlane=1))
        g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
        seed_features(g, sc)
        B = 3
        batch = gpu_pkg.FilterBatch(cfg_b, B, feature_capacity=32)
        batch.seed_from(g)
        batch.set_force_plane(1)
        off = gpu_pkg.FilterBatch(cfg_b, B, feature_capacity=32)
        off.seed_from(g)
        cams = _perturbed(g.get_full()[0], B, 7)
        batch.set_camera_states(cams); off.set_camera_states(cams)
        oracles = _oracles(orc, cfg_o, g, sc.frame(0), sc.stamps[0], cams)
        for t in range(1, sc.n_frames):
            img, picks = sc.frame(t), sc.picks(t, 30)
            for b, o in enumerate(oracles):
                batch.set_full(b, *o.get_full()); off.set_full(b, *o.get_full())
            for x in (batch, off):
                x.captureNewFrame(img, sc.stamps[t]); x.step(picks)
            _, st = batch.camera_states()
            mo, _ = off.camera_states()
            mb, _ = batch.camera_states()
            for b, o in enumerate(oracles):
                o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
                so = o.stats()
                assert (st[b, 2], st[b, 3]) == (so.n_li, so.n_hi), f"hard {hard} frame {t} filter {b}: n_li / n_hi"
                plane_only += int(so.n_hi == 0); with_hi += int(so.n_hi > 0)
                moved = max(moved, relerr(mo[b], mb[b]))
            _check(batch, oracles, f"hard {hard} frame {t}")
        mu, _ = batch.get_full(0)
        assert abs(mu[1]) < 1e-2 and abs(mu[4]) < 1e-2   # the pseudo-measurement holds y and q_x near zero
    print(f"second updates: {plane_only} plane only, {with_hi} with Hi rows; plane off vs on: camera rel {moved:.2e}")
    assert plane_only > 0 and with_hi > 0, (plane_only, with_hi)
    assert moved > 1e-6


def test_force_plane_filter0_follows_single_filter(gpu_pkg):
    """Filter 0 (unperturbed) of a batch from from_config runs free beside a single CUDA filter with forsePlane = 1 (and top-up
    and XYZ conversion): both run the Hi block, then the plane block, then one normalisation."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=10, seed=93, hard=True, outlier_frac=0.15)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), forsePlane=1, min_features=22, max_features=26, xyz_conversion=1))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(src, sc)
    batch = gpu_pkg.FilterBatch.from_config(cfg, 3)
    batch.seed_from(src)
    batch.set_topup(True)
    batch.set_camera_states(_perturbed(g.get_full()[0], 3, 6))
    n_hi = []
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        _, st = batch.camera_states()
        assert (st[0, 2], st[0, 3]) == (g.stats().n_li, g.stats().n_hi), f"frame {t}: n_li / n_hi"
        n_hi.append(int(st[0, 3]))
        N = g.numOfFeatures()
        assert batch.numOfFeatures(0) == N, f"frame {t}: feature count {batch.numOfFeatures(0)} vs {N}"
        fb = [batch.feature(0, i) for i in range(N)]
        fg = [g.feature(i) for i in range(N)]
        for f in ("real_index", "coding"):
            assert [getattr(a, f) for a in fb] == [getattr(c, f) for c in fg], f"frame {t}: {f}"
        assert [tuple(f.center) for f in fb] == [tuple(f.center) for f in fg], f"frame {t}: centres"
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}: mu {relerr(mb, mg):.2e} Sigma {relerr(Sb, Sg):.2e}"
    print(f"n_hi per step: {n_hi}")


SIM = dict(window_size=30, kernel_size=3, scale=10, sigma_size=4, T_camera=0.2, min_features=20, max_features=35, xyz_conversion=1)


@pytest.mark.parametrize("plane", [0, 1])
def test_simulation_setup_end_to_end(gpu_pkg, orc, plane):
    """conf_sim.cfg's switches (window 30, blur kernel_size 3 at T_camera 0.2, scale 10, sigma_size 4, min / max 20 / 35, top-up
    and XYZ conversion; forsePlane in the second parametrisation) through FilterBatch.from_config, on BGR frames ten times the
    scene's.  Filters 0-2, per step from identical inputs, against the oracle fed the resized frame in the reference order
    (predict with blur, update, addFeatures on the batch's new centres, convert2XYZ_ifLinearAll).  The scene is a ground
    robot's (planar: the plane pseudo-measurements hold) turning fast enough for blur at T_camera 0.2, with 16 features for a
    minimum of 20.  Blur, top-up and the forsePlane switch must all have acted, and no filter may have reached its 32-feature
    capacity (a full batch filter would stop adding where the reference would not)."""
    sc = gpu_pkg.synth.Scene(n_features=16, n_frames=5, seed=502, window=30, planar=True, **dict(BLUR_SCENE, omega=1.5))
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), forsePlane=plane, **SIM))
    cfg_o = gpu_pkg.default_config(**dict(sc.config_overrides(), **dict(SIM, scale=1, xyz_conversion=0), forsePlane=plane))
    big0 = _blow_up(sc.frame(0), 10)
    assert np.array_equal(cv2.cvtColor(cv2.resize(big0, (sc.width, sc.height)), cv2.COLOR_BGR2GRAY), sc.frame(0))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    g.captureNewFrame(big0, sc.stamps[0])
    assert np.array_equal(g.returnGrayImg(), sc.frame(0))
    mu, S = g.get_full()
    mu[0:3], mu[3:7] = sc.r[0], sc.q[0]
    g.set_full(mu, S)
    for p in sc.feature_pixels:
        assert g.addFeature(*p) == 1
    B = 3
    batch = gpu_pkg.FilterBatch.from_config(cfg, B)
    # the same batch with forsePlane the other way, for the first step only: its camera states must differ
    twin = gpu_pkg.FilterBatch.from_config(gpu_pkg.default_config(**dict(sc.config_overrides(), forsePlane=1 - plane, **SIM)), B)
    cams = _moving(_perturbed(g.get_full()[0], B, 5), sc)
    for x in (batch, twin):
        x.seed_from(g); x.set_topup(True); x.set_camera_states(cams)
    oracles = _oracles(orc, cfg_o, g, sc.frame(0), sc.stamps[0], cams)
    blurred = added_total = 0
    most = 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        big = _blow_up(img, 10)
        for b, o in enumerate(oracles):
            batch.set_full(b, *o.get_full())
        batch.captureNewFrame(big, sc.stamps[t]); batch.step(picks)
        assert np.array_equal(batch.returnGrayImg(), img), f"frame {t}: resized frame"
        mb, st = batch.camera_states()
        if t == 1:
            twin.captureNewFrame(big, sc.stamps[t]); twin.step(picks)
            mt, _ = twin.camera_states()
            switch = max(relerr(mt[b], mb[b]) for b in range(B))
        added, counts = batch.last_added(), batch.last_blur_counts()
        for b, o in enumerate(oracles):
            nb0 = o.stats().blur_requests
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert counts[b] == so.blur_requests - nb0, f"frame {t} filter {b}: blurred"
            assert (st[b, 2], st[b, 3]) == (so.n_li, so.n_hi), f"frame {t} filter {b}: n_li / n_hi"
            assert (st[b, 6], st[b, 7]) == (so.n_removed, so.topup_request), f"frame {t} filter {b}: removed / top-up"
            want = 0
            if so.topup_request > 0:
                survivors = _centers(o)
                corners = _single_with(gpu_pkg, cfg_o, img, survivors).detect_corners(int(so.topup_request))
                want = min(len(corners), int(so.topup_request), 32 - len(survivors))
            assert added[b] == want, f"frame {t} filter {b}: added {added[b]}, single filter {want}"
            nb = batch.numOfFeatures(b)
            if added[b]:
                new = [tuple(batch.feature(b, i).center) for i in range(nb - added[b], nb)]
                assert o.addFeatures(np.array(new, dtype=np.float32)) == added[b]
            o.convert2XYZ_ifLinearAll()
            blurred += int(counts[b]); added_total += int(added[b])
            most = max(most, nb)
        print(f"frame {t}: blurred {list(counts)} n_hi {list(st[:, 3])} added {list(added)} features {[batch.numOfFeatures(b) for b in range(B)]}")
        _check(batch, oracles, f"plane {plane} frame {t}")
    print(f"blurred {blurred}, added {added_total}, most features {most}, forsePlane {1 - plane} vs {plane}: camera rel {switch:.2e}")
    assert blurred > 0 and added_total > 0, (blurred, added_total)
    assert switch > 1e-6, "forsePlane made no difference"
    assert most < 32, f"a filter reached the 32-feature capacity ({most})"


def test_switches_off_change_nothing(gpu_pkg):
    """A batch that never had the switches and one where set_force_plane(1), set_scale(3), then set_force_plane(0), set_scale(1)
    were called, on the same ensemble and frames: the same launches per step and every filter's mu and Sigma bit-identical."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=7, seed=93, hard=True)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=1))
    runs = []
    for touched in (False, True):
        g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
        seed_features(g, sc)
        batch = gpu_pkg.FilterBatch(cfg, 4, feature_capacity=32)
        batch.seed_from(g)
        batch.set_camera_states(_perturbed(g.get_full()[0], 4, 4))
        if touched:
            batch.set_force_plane(1); batch.set_scale(3)
            batch.set_force_plane(0); batch.set_scale(1)
        launches, states = [], []
        for t in range(1, sc.n_frames):
            k0 = batch.kernel_launches()
            batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(sc.picks(t, 20))
            launches.append(batch.kernel_launches() - k0)
            states.append([batch.get_full(b) for b in range(4)])
        runs.append((launches, states))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1, f"launches per step: never switched {l0}, switched off {l1}"
    for t, (a, c) in enumerate(zip(s0, s1)):
        for b, ((ma, Sa), (mc, Sc)) in enumerate(zip(a, c)):
            assert np.array_equal(ma, mc) and np.array_equal(Sa, Sc), f"step {t + 1} filter {b}"
