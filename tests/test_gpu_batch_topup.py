"""-m gpu: findNewFeatures / addFeature in the batched filters (vslamRansac.cpp:309-371, :783-839, :1312-1315).

Every filter of a batch must detect exactly the corners a single filter holding the same patch centres detects (and cv2's
goodFeaturesToTrack with the reference's mask), add them bit for bit as consecutive single-filter addFeature calls do, and,
with top-up switched on, end a step in the reference order: removals, findNewFeatures, convert2XYZ_ifLinearAll."""
import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, assert_scaled_close, relerr, seed_features

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _reference_mask(shape, centers, w):
    """vslamRansac.cpp:788-818."""
    H, W = shape
    mask = np.zeros((H, W), np.uint8)
    mask[w:H - w, w:W - w] = 255
    win = 2 * w + 1
    for cx, cy in centers:
        if cx > w and cy > w and cx < W - w and cy < H - w:
            x = int(cx - win // 2) if cx - win // 2 > 0 else 0
            y = int(cy - win // 2) if cy - win // 2 > 0 else 0
            mask[y:y + win, x:x + win] = 0
    return mask


def _textured(seed, W=640, H=480):
    """Smooth random texture with a few hundred distinct corners (blurred noise + rectangles)."""
    rng = np.random.default_rng(seed)
    img = cv2.GaussianBlur(rng.integers(0, 256, (H, W)).astype(np.float32), (0, 0), 2.5)
    img = (img - img.min()) / (img.max() - img.min()) * 160 + 40
    for _ in range(60):
        x, y = int(rng.integers(20, W - 60)), int(rng.integers(20, H - 60))
        img[y:y + int(rng.integers(8, 40)), x:x + int(rng.integers(8, 40))] += rng.uniform(-40, 40)
    return np.clip(img, 0, 255).astype(np.uint8)


def _blocks(seed, W=640, H=480):
    """8 x 8 blocks of four grey levels: many corners with exactly equal scores, flat plateaus between them."""
    rng = np.random.default_rng(seed)
    return np.kron(rng.integers(0, 4, (H // 8, W // 8)) * 60 + 20, np.ones((8, 8))).astype(np.uint8)


def _centers(f, b=None):
    if b is None:
        return [tuple(f.feature(i).center) for i in range(f.numOfFeatures())]
    return [tuple(f.feature(b, i).center) for i in range(f.numOfFeatures(b))]


def _single_with(pkg, cfg, img, centers, cap=64):
    """A single CUDA filter on `img` holding patches at `centers` (rejected ones leave no box either: isInsideImage rejects
    only centres the mask skips)."""
    s = pkg.VSlamFilter(cfg, feature_capacity=cap)
    s.captureNewFrame(img, 1.0)
    for c in centers:
        s.addFeature(*c)
    return s


@pytest.mark.parametrize("image,num", [(1, 30), (2, 100), (3, 12), (4, 200), (5, 60), (6, 150), (8, 300), ("blocks", 32)])
def test_detection_is_exact_per_filter(gpu_pkg, image, num):
    """Different extra patches per filter (none, a few, up to capacity, some rejected at the border); each filter's corners, in
    order, are the single filter's and cv2's on that filter's mask.  On the block image (exact ties) the bar is the single
    filter alone: cv2's float pipeline differs from the restated one in the last bits, which ties expose (csrc/ekf_detect.cu)."""
    img = _textured(image) if image != "blocks" else _blocks(9)
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0, min_features=0)
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=64)
    g.captureNewFrame(img, 1.0)
    for p in [(100.0, 100.0), (320.0, 240.0), (500.0, 400.0)]:
        assert g.addFeature(*p) == 1
    B, cap = 5, 12
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap)
    batch.seed_from(g)
    batch.captureNewFrame(img, 1.0)
    rng = np.random.default_rng(17)
    extra = {0: [], 1: [(200.0, 150.0), (420.5, 300.25)], 2: [tuple(p) for p in rng.uniform(30, 440, (5, 2))],
             3: [tuple(p) for p in rng.uniform(30, 440, (cap - 3, 2))], 4: [(3.0, 200.0), (636.0, 100.0), (50.0, 50.0)]}
    for b, pts in extra.items():
        for u, v in pts:
            inside = 5 < u < 640 - 5 and 5 < v < 480 - 5
            assert batch.addFeature(b, u, v) == int(inside)
    assert batch.numOfFeatures(3) == cap
    with pytest.raises(gpu_pkg.EkfError):
        batch.addFeature(3, 300.0, 300.0)   # at capacity
    k = min(num, 32)
    got = batch.detect_corners(k)
    for b in range(B):
        cen = _centers(batch, b)
        want = _single_with(gpu_pkg, cfg, img, cen).detect_corners(k)
        assert np.array_equal(got[b], want), f"image {image} filter {b}: batch vs single filter"
        if image != "blocks":
            ref = cv2.goodFeaturesToTrack(img, k, 0.01, 12, mask=_reference_mask(img.shape, cen, 11)).reshape(-1, 2)
            assert np.array_equal(got[b], ref), f"image {image} filter {b}: batch vs cv2"
        assert len(got[b]) == k
    assert batch.detect_corners([0, 5, 0, 1, 40])[0].shape == (0, 2)


def _perturbed(mu0, B, seed, perturb=2e-3):
    rng = np.random.default_rng(seed)
    cams = np.tile(mu0[:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=perturb, size=(B, 3))
    cams[:, 3:7] += rng.normal(scale=perturb, size=(B, 4))
    cams[:, 3:7] /= np.linalg.norm(cams[:, 3:7], axis=1, keepdims=True)
    cams[:, 7:13] += rng.normal(scale=perturb, size=(B, 6))
    cams[0] = mu0[:14]
    return cams


def test_adds_equal_single_filter_bit_for_bit(gpu_pkg, orc):
    """Several corners per filter in one findNewFeatures call (counts 0 to capacity-bound); each filter against a single filter
    from the same state calling addFeature on the same pixels (array_equal), and against the oracle's addFeature."""
    sc = gpu_pkg.synth.Scene(n_features=8, n_frames=4, seed=71)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    B, cap = 5, 20
    num = np.array([3, 0, 7, 20, 1], dtype=np.int32)

    def single():
        s = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
        seed_features(s, sc)
        for t in (1, 2):
            s.captureNewFrame(sc.frame(t), sc.stamps[t]); s.predict(); s.update(sc.picks(t, 8))
        return s
    g = single()
    mu0, S0 = g.get_full()
    cams = _perturbed(mu0, B, 4)
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap)
    batch.seed_from(g)
    img = sc.frame(3)
    singles, oracles = [], []
    for b in range(B):
        s = single()
        m = mu0.copy(); m[:14] = cams[b]
        s.set_full(m, S0); batch.set_full(b, m, S0)
        o = orc.OracleFilter(cfg, kind=0, omp=False)
        o.captureNewFrame(img, sc.stamps[3]); o.import_from(s)
        s.captureNewFrame(img, sc.stamps[3])
        singles.append(s); oracles.append(o)
    batch.captureNewFrame(img, sc.stamps[3])
    found = [len(c) for c in batch.detect_corners(np.minimum(num, 32))]
    N0 = [batch.numOfFeatures(b) for b in range(B)]
    added = batch.findNewFeatures(num)
    assert list(added) == [min(int(num[b]), cap - N0[b], found[b]) for b in range(B)]
    assert added[1] == 0 and added[3] == cap - N0[3] and added.sum() > 0
    for b, (s, o) in enumerate(zip(singles, oracles)):
        new = _centers(batch, b)[N0[b]:]
        assert len(new) == added[b]
        for c in new:
            assert s.addFeature(*c) == 1
        o.addFeatures(np.array(new, dtype=np.float32).reshape(-1, 2))
        mb, Sb = batch.get_full(b); ms, Ss = s.get_full()
        assert np.array_equal(mb, ms) and np.array_equal(Sb, Ss), f"filter {b}: state differs from the single filter"
        assert s.numOfFeatures() == batch.numOfFeatures(b)
        for i in range(s.numOfFeatures()):
            a, c = batch.feature(b, i), s.feature(i)
            for f in INT_FIELDS:
                assert getattr(a, f) == getattr(c, f), f"filter {b} feature {i} {f}"
            assert tuple(a.center) == tuple(c.center)
            assert np.array_equal(batch.template(b, i), s.template(i)), f"filter {b} feature {i} template"
        mo, So = o.get_full()
        assert relerr(mb, mo) <= TOL and relerr(Sb, So) <= TOL, f"filter {b}: vs oracle"
        assert_scaled_close(mb, Sb, mo, So, f"filter {b} vs oracle addFeature")
        assert [batch.feature(b, i).real_index for i in range(batch.numOfFeatures(b))] == \
            [o.feature(i).real_index for i in range(o.numOfFeatures())]


def test_counts_requests_and_errors(gpu_pkg):
    sc = gpu_pkg.synth.Scene(n_features=10, n_frames=3, seed=72, hard=True)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=14))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    batch = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=16)
    with pytest.raises(gpu_pkg.EkfError):
        batch.addFeature(0, 100.0, 100.0)          # before seeding
    with pytest.raises(gpu_pkg.EkfError):
        batch.findNewFeatures(3)                    # before seeding
    batch.seed_from(g)
    with pytest.raises(gpu_pkg.EkfError):
        batch.detect_corners(3)                     # before a frame
    with pytest.raises(gpu_pkg.EkfError):
        batch.addFeature(0, 100.0, 100.0)           # before a frame
    batch.captureNewFrame(sc.frame(1), sc.stamps[1])
    with pytest.raises(gpu_pkg.EkfError):
        batch.findNewFeatures()                     # num=None without a completed step
    for bad in (-1, 3):
        with pytest.raises(gpu_pkg.EkfError):
            batch.addFeature(bad, 100.0, 100.0)
    assert batch.addFeature(0, 2.0, 100.0) == 0     # isInsideImage
    batch.step(sc.picks(1, 10))                     # top-up off: the request is reported, nothing added
    _, st = batch.camera_states()
    topup = st[:, 7]
    assert (topup > 0).all() and not batch.last_added().any()
    N = [batch.numOfFeatures(b) for b in range(3)]
    found = [len(c) for c in batch.detect_corners(np.minimum(topup, 32))]
    added = batch.findNewFeatures()                 # num=None: EKF_BSTAT_TOPUP of the last step
    assert list(added) == [min(int(topup[b]), 16 - N[b], found[b]) for b in range(3)]
    assert [batch.numOfFeatures(b) for b in range(3)] == [N[b] + added[b] for b in range(3)]
    N = [batch.numOfFeatures(b) for b in range(3)]
    found = [len(c) for c in batch.detect_corners(32)]
    added = batch.findNewFeatures(40)               # capacity-bound
    assert list(added) == [min(40, 16 - N[b], found[b]) for b in range(3)]
    assert all(batch.numOfFeatures(b) == 16 for b in range(3))


def _shrink(o, features, factor):
    mu, S = o.get_full()
    for i in features:
        p = o.feature(i).position_in_state
        S[p + 5, :] *= factor; S[:, p + 5] *= factor
    return mu, S


def _plan(b, o):
    """Inverse-depth features of filter b whose rho variance is cut before a step: none for filter 0."""
    if b == 0:
        return [], 1.0
    inv = [i for i in range(o.numOfFeatures()) if not o.feature(i).coding]
    return inv[b % 3::4][:1 + b % 2], 10.0 ** -(3 + b % 3)


def _check(batch, oracles, ctx, tol=TOL):
    for b, o in enumerate(oracles):
        assert batch.numOfFeatures(b) == o.numOfFeatures(), f"{ctx} filter {b}: feature count"
        assert batch.state_dim(b) == o.state_dim(), f"{ctx} filter {b}: state dim"
        mg, Sg = batch.get_full(b); mo, So = o.get_full()
        em, es = relerr(mg, mo), relerr(Sg, So)
        assert em <= tol and es <= tol, f"{ctx} filter {b}: mu {em:.2e} Sigma {es:.2e}"
        assert_scaled_close(mg, Sg, mo, So, f"{ctx} filter {b}")
        for i in range(o.numOfFeatures()):
            a, c = batch.feature(b, i), o.feature(i)
            for f in INT_FIELDS:
                assert getattr(a, f) == getattr(c, f), f"{ctx} filter {b} feature {i} {f}: {getattr(a, f)} vs {getattr(c, f)}"
            assert tuple(a.center) == tuple(c.center), f"{ctx} filter {b} feature {i} centre"


@pytest.mark.parametrize("xyz", [0, 1])
def test_step_tops_up_in_reference_order(gpu_pkg, orc, xyz):
    """Identical inputs per step (batch state <- oracle state).  Oracle side: update without conversion, addFeatures on the
    batch's new centres, then convert2XYZ_ifLinearAll.  The filters track 20 of the scene's points and filter 2 the other
    four as well, so it starts above min_features while the others ask for features; max_features = 16 makes their top-ups
    take the removeFeature(0) branch first."""
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=6, seed=502, hard=True)
    over = dict(sc.config_overrides(), min_features=21, max_features=16)
    cfg_b = gpu_pkg.default_config(**dict(over, xyz_conversion=xyz))
    cfg_o = gpu_pkg.default_config(**dict(over, xyz_conversion=0))
    g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
    g.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels[:20]:
        assert g.addFeature(*p) == 1
    B = 4
    batch = gpu_pkg.FilterBatch(cfg_b, B, feature_capacity=32)
    batch.seed_from(g)
    batch.set_topup(True)
    mu0, S0 = g.get_full()
    cams = _perturbed(mu0, B, 5)
    batch.set_camera_states(cams)
    img0 = sc.frame(0)
    batch.captureNewFrame(img0, sc.stamps[0])
    oracles = []
    for b in range(B):
        o = orc.OracleFilter(cfg_o, kind=0, omp=False)
        o.captureNewFrame(img0, sc.stamps[0]); o.import_from(g)
        m = mu0.copy(); m[:14] = cams[b]
        o.set_full(m, S0)
        oracles.append(o)
    for u, v in sc.feature_pixels[20:]:   # filter 2: the other four points, on both sides
        assert batch.addFeature(2, u, v) == 1 and oracles[2].addFeature(u, v) == 1
    full = mixed = dropped = False
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        for b, o in enumerate(oracles):
            mu, S = _shrink(o, *_plan(b, o)) if xyz else o.get_full()
            o.set_full(mu, S); batch.set_full(b, mu, S)
        batch.captureNewFrame(img, sc.stamps[t])
        batch.step(picks)
        _, st = batch.camera_states()
        added = batch.last_added()
        for b, o in enumerate(oracles):
            before = {o.feature(i).real_index: o.feature(i).coding for i in range(o.numOfFeatures())}
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert (st[b, 6], st[b, 7]) == (so.n_removed, so.topup_request), f"frame {t} filter {b}: removed / top-up"
            survivors = _centers(o)
            want = 0
            if so.topup_request > 0:
                corners = _single_with(gpu_pkg, cfg_o, img, survivors).detect_corners(int(so.topup_request))
                want = min(len(corners), int(so.topup_request), 32 - len(survivors))
            assert added[b] == want, f"frame {t} filter {b}: added {added[b]}, single filter {want}"
            nb = batch.numOfFeatures(b)
            new = [tuple(batch.feature(b, i).center) for i in range(nb - added[b], nb)]
            if added[b]:
                assert np.array_equal(np.array(new, dtype=np.float32), corners[:want]), f"frame {t} filter {b}: new centres"
                assert o.addFeatures(np.array(new, dtype=np.float32)) == added[b]
                dropped |= len(survivors) > 16
            if xyz:
                o.convert2XYZ_ifLinearAll()
            conv = sum(1 for i in range(o.numOfFeatures()) if o.feature(i).coding and not before.get(o.feature(i).real_index, 0))
            full |= so.n_removed > 0 and added[b] > 0 and conv > 0
        mixed |= (added > 0).any() and (added == 0).any()
        print(f"frame {t}: removed {list(st[:, 6])} top-up {list(st[:, 7])} added {list(added)}")
        _check(batch, oracles, f"frame {t}")
    assert mixed, "no step in which one filter topped up and another did not"
    assert dropped, "no top-up through the removeFeature(0) branch"
    if xyz:
        assert full, "no filter removed, topped up and converted in the same step"


def test_filter0_follows_single_filter(gpu_pkg):
    """Filter 0 (unperturbed) runs free against a single CUDA filter of the same capacity, which tops up by itself in
    ekf_update_after_match."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=12, seed=93, hard=True, outlier_frac=0.15)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=22, max_features=26, xyz_conversion=1))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    batch = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=32)
    batch.seed_from(g)
    batch.set_topup(True)
    mu0, _ = g.get_full()
    batch.set_camera_states(_perturbed(mu0, 3, 6))
    N_start, removals = g.numOfFeatures(), 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        removals += g.stats().n_removed
        N = g.numOfFeatures()
        assert batch.numOfFeatures(0) == N, f"frame {t}: feature count {batch.numOfFeatures(0)} vs {N}"
        fb = [batch.feature(0, i) for i in range(N)]
        fg = [g.feature(i) for i in range(N)]
        assert [f.real_index for f in fb] == [f.real_index for f in fg], f"frame {t}: real_index"
        assert [f.coding for f in fb] == [f.coding for f in fg], f"frame {t}: codings"
        assert [tuple(f.center) for f in fb] == [tuple(f.center) for f in fg], f"frame {t}: centres"
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}: mu {relerr(mb, mg):.2e} Sigma {relerr(Sb, Sg):.2e}"
    assert removals > 0
    assert g.numOfFeatures() >= N_start


def test_no_cost_when_nothing_tops_up(gpu_pkg):
    """min_features = 0: no filter asks.  Top-up on and off give the same launches per step and bit-identical states."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=93, hard=True)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=1))
    runs = []
    for on in (False, True):
        g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
        seed_features(g, sc)
        batch = gpu_pkg.FilterBatch(cfg, 4, feature_capacity=32)
        batch.seed_from(g)
        batch.set_camera_states(_perturbed(g.get_full()[0], 4, 4))
        batch.set_topup(on)
        launches, states = [], []
        for t in range(1, sc.n_frames):
            k0 = batch.kernel_launches()
            batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(sc.picks(t, 20))
            launches.append(batch.kernel_launches() - k0)
            assert not batch.last_added().any() and not batch.camera_states()[1][:, 7].any()
            states.append([batch.get_full(b) for b in range(4)])
        runs.append((launches, states))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1, f"launches per step: off {l0}, on {l1}"
    for t, (a, c) in enumerate(zip(s0, s1)):
        for b, ((ma, Sa), (mc, Sc)) in enumerate(zip(a, c)):
            assert np.array_equal(ma, mc) and np.array_equal(Sa, Sc), f"step {t + 1} filter {b}"
