"""-m gpu: batched filters of up to 128 features (ekf_batch_create_large, FilterBatch(..., large=True)).

Above 32 features a filter's update runs on a thread-block cluster of 2 to 4 CTAs as blocks of at most 32 features.  A large
batch must describe itself right, be exactly an ordinary batch at capacity <= 32, match the oracle per step at cluster sizes 2,
3 and 4 (with forsePlane and XYZ conversion), top up past 32 features as the reference does, let filter 0 follow a single
CUDA filter of capacity 128, and agree with the one-CTA update where both apply."""
import ctypes as C

import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, TOL_SCALED_MU, TOL_SCALED_SIGMA, relerr, scaled_errors, seed_features
from test_gpu_batch_config import _oracles
from test_gpu_batch_topup import _centers, _perturbed, _plan, _shrink, _single_with

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


# With forsePlane the plane rows (R = 1e-5) shrink the variances of y, q_x and q_z by orders, and the scaled mean bar divides by
# those: the rounding differences between the blocked Li update (3 or 4 blocks at these sizes) and the oracle's one stacked
# solve reach 2e-10 sigma there (without the plane they stay below 8e-12).  The covariance bar is unchanged.
PLANE_SCALED_MU = 5e-10


def _check_large(batch, oracles, ctx, mu_bar):
    for b, o in enumerate(oracles):
        assert batch.numOfFeatures(b) == o.numOfFeatures() and batch.state_dim(b) == o.state_dim(), f"{ctx} filter {b}: size"
        mg, Sg = batch.get_full(b); mo, So = o.get_full()
        em, es = relerr(mg, mo), relerr(Sg, So)
        assert em <= TOL and es <= TOL, f"{ctx} filter {b}: mu {em:.2e} Sigma {es:.2e}"
        sS, sm = scaled_errors(mg, Sg, mo, So)
        print(f"{ctx} filter {b}: scaled err Sigma {sS:.2e} mu {sm:.2e} sigma")
        assert sS <= TOL_SCALED_SIGMA and sm <= mu_bar, f"{ctx} filter {b}: scaled Sigma {sS:.2e} mu {sm:.2e}"
        for i in range(o.numOfFeatures()):
            a, c = batch.feature(b, i), o.feature(i)
            for f in INT_FIELDS:
                assert getattr(a, f) == getattr(c, f), f"{ctx} filter {b} feature {i} {f}: {getattr(a, f)} vs {getattr(c, f)}"
            assert tuple(a.center) == tuple(c.center), f"{ctx} filter {b} feature {i} centre"


def _dims(cap):
    ncap = 14 + 6 * cap
    return ncap, (ncap + 7) & ~7


def test_create_large_descriptors_and_errors(gpu_pkg):
    """Capacities on both sides of each cluster-size boundary; 129 is refused, and ekf_batch_create still refuses 33."""
    cfg = gpu_pkg.default_config(window_size=11, xyz_conversion=0)
    for cap, ctas in ((33, 2), (67, 2), (68, 3), (101, 3), (102, 4), (128, 4)):
        batch = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=cap, large=True)
        d = batch.describe()
        ncap, ld = _dims(cap)
        assert (d.n_filters, d.feature_capacity, d.state_capacity, d.ld) == (3, cap, ncap, ld), cap
        c, resident = batch.update_clusters()
        print(f"capacity {cap}: ld {ld}, {c} CTAs per filter, {resident} clusters resident")
        assert c == ctas and resident >= 1, (cap, c, resident)
        batch.close()
    assert gpu_pkg.FilterBatch(cfg, 3, feature_capacity=32, large=True).update_clusters() == (1, 0)
    h = C.c_void_p()
    L = gpu_pkg.lib()
    assert L.ekf_batch_create_large(C.byref(cfg), 3, 129, 0, C.byref(h)) == gpu_pkg._abi.EKF_ERR_CAPACITY
    assert L.ekf_batch_create_large(C.byref(cfg), 3, 0, 0, C.byref(h)) == gpu_pkg._abi.EKF_ERR_ARG
    with pytest.raises(gpu_pkg.EkfError):
        gpu_pkg.FilterBatch(cfg, 3, feature_capacity=33)


def test_large_at_32_is_the_ordinary_batch(gpu_pkg):
    """create_large at capacity <= 32 builds what ekf_batch_create builds: the same launches per step and bit-identical states
    (top-up and XYZ conversion on)."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=93, hard=True)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=22, max_features=26, xyz_conversion=1))
    runs = []
    for large in (False, True):
        g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
        seed_features(g, sc)
        batch = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=32, large=large)
        batch.seed_from(g); batch.set_topup(True)
        batch.set_camera_states(_perturbed(g.get_full()[0], 3, 4))
        launches, states = [], []
        for t in range(1, sc.n_frames):
            k0 = batch.kernel_launches()
            batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(sc.picks(t, 20))
            launches.append(batch.kernel_launches() - k0)
            states.append([batch.get_full(b) for b in range(3)])
        runs.append((launches, states))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1, f"launches per step: create {l0}, create_large {l1}"
    for t, (a, c) in enumerate(zip(s0, s1)):
        for b, ((ma, Sa), (mc, Sc)) in enumerate(zip(a, c)):
            assert np.array_equal(ma, mc) and np.array_equal(Sa, Sc), f"step {t + 1} filter {b}"


@pytest.mark.parametrize("xyz", [0, 1])
@pytest.mark.parametrize("plane", [0, 1])
@pytest.mark.parametrize("cap,nfeat", [(48, 40), (100, 90), (128, 120)])
def test_step_against_oracle(gpu_pkg, orc, cap, nfeat, plane, xyz):
    """Filters 0-2 of a perturbed ensemble, per step from identical inputs (batch state <- oracle state), on a clean and a
    noisy scene with displaced outliers: n_li / n_hi equal, tables bit-exact, the state within TOL and the scaled bars (the
    mean's bar PLANE_SCALED_MU with the plane).  Li updates of more than 32 features (several blocks) must occur, and with the
    plane Hi updates of more than 32 features (several Hi blocks): pulled towards the plane, the scene's off-plane camera
    leaves features for the rescue (without the plane this scene rescues none; n_hi equals the oracle's either way).  With
    xyz, some features' rho variance is cut before a step so that conversions happen."""
    max_li = n_hi = 0
    clusters = None
    for hard in (False, True):
        sc = gpu_pkg.synth.Scene(n_features=nfeat, n_frames=4, seed=300 + nfeat + int(hard), hard=hard,
                                 **(dict(outlier_frac=0.15) if hard else {}))
        cfg_b = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=xyz))
        cfg_o = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=xyz, forsePlane=plane))
        g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=cap)
        seed_features(g, sc)
        B = 3
        batch = gpu_pkg.FilterBatch(cfg_b, B, feature_capacity=cap, large=True)
        clusters = batch.update_clusters()[0]
        batch.seed_from(g)
        batch.set_force_plane(plane)
        cams = _perturbed(g.get_full()[0], B, 7)
        batch.set_camera_states(cams)
        oracles = _oracles(orc, cfg_o, g, sc.frame(0), sc.stamps[0], cams)
        for t in range(1, sc.n_frames):
            img, picks = sc.frame(t), sc.picks(t, nfeat)
            for b, o in enumerate(oracles):
                mu, S = _shrink(o, *_plan(b, o)) if xyz else o.get_full()
                o.set_full(mu, S); batch.set_full(b, mu, S)
            batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
            _, st = batch.camera_states()
            for b, o in enumerate(oracles):
                o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
                so = o.stats()
                assert (st[b, 2], st[b, 3]) == (so.n_li, so.n_hi), f"hard {hard} frame {t} filter {b}: n_li / n_hi"
                assert st[b, 6] == so.n_removed, f"hard {hard} frame {t} filter {b}: removed"
                max_li = max(max_li, int(so.n_li)); n_hi += int(so.n_hi)
            _check_large(batch, oracles, f"cap {cap} plane {plane} xyz {xyz} hard {hard} frame {t}",
                         PLANE_SCALED_MU if plane else TOL_SCALED_MU)
    print(f"cap {cap} ({clusters} CTAs): largest Li update {max_li} features, Hi features in all {n_hi}")
    assert max_li > 32, f"no Li update of more than 32 features ({max_li})"
    if plane:
        assert n_hi > 32, f"no Hi update of several blocks ({n_hi})"


@pytest.mark.parametrize("minf,maxf", [(30, 100), (20, 35)])
def test_topup_past_32(gpu_pkg, orc, minf, maxf):
    """min_features / max_features of conf.cfg (30 / 100) and conf_sim.cfg (20 / 35), top-up on, capacity 128, per step from
    identical inputs against the oracle in the reference order (update, addFeatures on the batch's new centres).  Each filter
    adds min(corners, request, capacity - survivors) features, as a single filter's detector finds them.  After frame 0 only
    every third scene point is drawn, and quality_ratio is 1e9 (no quality deletions, as in bench.py), so the unseen features
    stay and the filters ask for features every step.  With 30 / 100 the filters start from 20 features and the maps must
    grow past 32; with 20 / 35 they start from 40 and must take the removeFeature(0) branch of the max_features rule."""
    sc = gpu_pkg.synth.Scene(n_features=40, n_frames=6, seed=502, visible_every=3)
    cap = 128
    over = dict(sc.config_overrides(), min_features=minf, max_features=maxf, quality_ratio=1e9)
    cfg = gpu_pkg.default_config(**over)
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    g.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels[:20 if maxf >= 100 else 40]:
        assert g.addFeature(*p) == 1
    B = 3
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=cap, large=True)
    batch.seed_from(g)
    batch.set_topup(True)
    cams = _perturbed(g.get_full()[0], B, 5)
    batch.set_camera_states(cams)
    batch.captureNewFrame(sc.frame(0), sc.stamps[0])
    oracles = _oracles(orc, cfg, g, sc.frame(0), sc.stamps[0], cams)
    most, dropped = 0, 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 40)
        for b, o in enumerate(oracles):
            batch.set_full(b, *o.get_full())
        N0 = [batch.numOfFeatures(b) for b in range(B)]
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        _, st = batch.camera_states()
        added = batch.last_added()
        for b, o in enumerate(oracles):
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert (st[b, 2], st[b, 3]) == (so.n_li, so.n_hi), f"frame {t} filter {b}: n_li / n_hi"
            assert (st[b, 6], st[b, 7]) == (so.n_removed, so.topup_request), f"frame {t} filter {b}: removed / top-up"
            survivors = _centers(o)
            want = 0
            if so.topup_request > 0:
                corners = _single_with(gpu_pkg, cfg, img, survivors, cap=cap).detect_corners(int(so.topup_request))
                want = min(len(corners), int(so.topup_request), cap - len(survivors))
                # removeFeature(0) ran: without quality deletions it is the step's only removal
                dropped += int(so.n_removed == 1 and N0[b] > maxf)
            assert added[b] == want, f"frame {t} filter {b}: added {added[b]}, single filter {want}"
            nb = batch.numOfFeatures(b)
            if added[b]:
                new = [tuple(batch.feature(b, i).center) for i in range(nb - added[b], nb)]
                assert np.array_equal(np.array(new, dtype=np.float32), corners[:want]), f"frame {t} filter {b}: new centres"
                assert o.addFeatures(np.array(new, dtype=np.float32)) == added[b]
            most = max(most, nb)
        print(f"frame {t}: removed {list(st[:, 6])} top-up {list(st[:, 7])} added {list(added)} "
              f"features {[batch.numOfFeatures(b) for b in range(B)]}")
        _check_large(batch, oracles, f"min {minf} max {maxf} frame {t}", TOL_SCALED_MU)
    print(f"most features {most}, steps through the removeFeature(0) branch {dropped}")
    assert most > 32, f"no map grew past 32 features ({most})"
    if maxf < 40:
        assert dropped > 0, "no removal by the max_features rule"


def test_filter0_follows_single_filter(gpu_pkg):
    """Filter 0 (unperturbed) of a capacity-128 batch runs free beside a single CUDA filter of capacity 128 with the
    reference's default min_features / max_features (30 / 100), top-up and XYZ conversion, while the map grows from 24 past 32
    features: after frame 0 only every second scene point is drawn and quality_ratio is 1e9, so unseen features stay and the
    filter keeps asking."""
    sc = gpu_pkg.synth.Scene(n_features=48, n_frames=12, seed=93, visible_every=2)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), min_features=30, max_features=100, xyz_conversion=1,
                                        quality_ratio=1e9))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=128)
    g.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels[:24]:
        assert g.addFeature(*p) == 1
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=128)
    src.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels[:24]:
        assert src.addFeature(*p) == 1
    batch = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=128, large=True)
    batch.seed_from(src)
    batch.set_topup(True)
    batch.set_camera_states(_perturbed(g.get_full()[0], 3, 6))
    most, added = 0, 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 48)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        _, st = batch.camera_states()
        assert (st[0, 2], st[0, 3]) == (g.stats().n_li, g.stats().n_hi), f"frame {t}: n_li / n_hi"
        N = g.numOfFeatures()
        assert batch.numOfFeatures(0) == N, f"frame {t}: feature count {batch.numOfFeatures(0)} vs {N}"
        fb = [batch.feature(0, i) for i in range(N)]
        fg = [g.feature(i) for i in range(N)]
        for f in ("real_index", "coding"):
            assert [getattr(a, f) for a in fb] == [getattr(c, f) for c in fg], f"frame {t}: {f}"
        assert [tuple(f.center) for f in fb] == [tuple(f.center) for f in fg], f"frame {t}: centres"
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}: mu {relerr(mb, mg):.2e} Sigma {relerr(Sb, Sg):.2e}"
        most = max(most, N)
        added += int(batch.last_added()[0])
    print(f"features: most {most}, filter 0 added {added}")
    assert most > 32, f"the map never grew past 32 features ({most})"


def test_cluster_update_against_one_cta_update(gpu_pkg):
    """A capacity-33 batch (cluster of 2) and a capacity-32 batch (k_batch_update), seeded from the same 30-feature filter,
    step the same frames: the same decisions, and states within 1e-9 in the covariance's units."""
    sc = gpu_pkg.synth.Scene(n_features=30, n_frames=8, seed=61, hard=True)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=1))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    cams = _perturbed(g.get_full()[0], 4, 9)
    small = gpu_pkg.FilterBatch(cfg, 4, feature_capacity=32)
    big = gpu_pkg.FilterBatch(cfg, 4, feature_capacity=33, large=True)
    assert big.update_clusters()[0] == 2
    for x in (small, big):
        x.seed_from(g); x.set_camera_states(cams)
    worst_S = worst_mu = 0.0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 30)
        for x in (small, big):
            x.captureNewFrame(img, sc.stamps[t]); x.step(picks)
        _, s0 = small.camera_states()
        _, s1 = big.camera_states()
        assert np.array_equal(s0, s1), f"frame {t}: counters {s0.tolist()} vs {s1.tolist()}"
        for b in range(4):
            assert small.numOfFeatures(b) == big.numOfFeatures(b)
            for i in range(small.numOfFeatures(b)):
                a, c = small.feature(b, i), big.feature(b, i)
                assert (a.coding, a.real_index, a.is_in_li, a.is_in_hi) == (c.coding, c.real_index, c.is_in_li, c.is_in_hi)
            m0, S0 = small.get_full(b); m1, S1 = big.get_full(b)
            eS, em = scaled_errors(m1, S1, m0, S0)
            worst_S, worst_mu = max(worst_S, eS), max(worst_mu, em)
            assert relerr(m1, m0) <= TOL and relerr(S1, S0) <= TOL, f"frame {t} filter {b}"
    print(f"cluster vs one-CTA update: largest scaled difference Sigma {worst_S:.2e}, mu {worst_mu:.2e} sigma")
    assert worst_S <= 1e-9 and worst_mu <= 1e-9, (worst_S, worst_mu)
