"""-m gpu: the batched-filter path (BASELINE config 3) against the CPU oracle, filter by filter.
Every filter of a batch must reproduce the single-filter algorithm: integer tables / matches
bit-exact, state and covariance within 1e-9 relative per step from identical inputs."""
import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, assert_scaled_close, make_pair, relerr, seed_features

pytestmark = pytest.mark.gpu


def _ensemble(pkg, orc, sc, B, seed, perturb=2e-3, **cfg_over):
    """A seeded single GPU filter, a batch cloned from it, and B oracle filters holding the same
    per-hypothesis perturbed camera states."""
    g, o0 = make_pair(pkg, orc, sc, **cfg_over)
    seed_features(g, sc); seed_features(o0, sc)
    cfg = g.cfg
    batch = pkg.FilterBatch(cfg, B, feature_capacity=min(32, sc.n_features + 2))
    batch.seed_from(g)
    rng = np.random.default_rng(seed)
    mu0, S0 = g.get_full()
    cams = np.tile(mu0[:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=perturb, size=(B, 3))
    dq = rng.normal(scale=perturb, size=(B, 4)); cams[:, 3:7] += dq
    cams[:, 3:7] /= np.linalg.norm(cams[:, 3:7], axis=1, keepdims=True)
    cams[:, 7:13] += rng.normal(scale=perturb, size=(B, 6))
    cams[0] = mu0[:14]
    batch.set_camera_states(cams)
    oracles = []
    for b in range(B):
        o = orc.OracleFilter(cfg, kind=0, omp=False)
        o.captureNewFrame(sc.frame(0), sc.stamps[0])
        o.import_from(g)
        m = mu0.copy(); m[:14] = cams[b]
        o.set_full(m, S0)
        oracles.append(o)
    return g, batch, oracles


def _check(batch, oracles, ctx, tol=TOL):
    worst = 0.0
    for b, o in enumerate(oracles):
        assert batch.numOfFeatures(b) == o.numOfFeatures(), f"{ctx} filter {b}: feature count"
        mg, Sg = batch.get_full(b); mo, So = o.get_full()
        assert mg.shape == mo.shape, f"{ctx} filter {b}"
        em, es = relerr(mg, mo), relerr(Sg, So)
        assert em <= tol and es <= tol, f"{ctx} filter {b}: mu {em:.2e} Sigma {es:.2e}"
        assert_scaled_close(mg, Sg, mo, So, f"{ctx} filter {b}", free_running=tol > TOL)
        worst = max(worst, em, es)
        for i in range(o.numOfFeatures()):
            a, c = batch.feature(b, i), o.feature(i)
            for f in INT_FIELDS:
                assert getattr(a, f) == getattr(c, f), f"{ctx} filter {b} feature {i} {f}: {getattr(a, f)} vs {getattr(c, f)}"
            assert tuple(a.center) == tuple(c.center), f"{ctx} filter {b} feature {i} match"
            assert a.last_ncc == c.last_ncc
    return worst


@pytest.mark.parametrize("n_features,hard,B", [(12, False, 5), (30, False, 4), (30, True, 6)])
def test_batch_matches_oracle_per_filter(gpu_pkg, orc, n_features, hard, B):
    sc = gpu_pkg.synth.Scene(n_features=n_features, n_frames=6, seed=300 + n_features + B, hard=hard)
    g, batch, oracles = _ensemble(gpu_pkg, orc, sc, B, seed=5)
    worst = 0.0
    for t in range(1, sc.n_frames):
        img = sc.frame(t); picks = sc.picks(t, n_features)
        # identical inputs per step: batch state <- oracle state
        for b, o in enumerate(oracles):
            if batch.numOfFeatures(b) == o.numOfFeatures():
                batch.set_full(b, *o.get_full())
        batch.captureNewFrame(img, sc.stamps[t])
        batch.step(picks)
        mu14, S14, st = batch.camera_states(want_sigma=True)
        for b, o in enumerate(oracles):
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert st[b, 1] == so.n_matched and st[b, 2] == so.n_li and st[b, 3] == so.n_hi and st[b, 4] == so.ransac_hypotheses, \
                f"frame {t} filter {b}: stats {st[b]} vs oracle ({so.n_matched}, {so.n_li}, {so.n_hi}, {so.ransac_hypotheses})"
            assert st[b, 6] == so.n_removed
            mo, So = o.get_full()
            assert relerr(mu14[b], mo[:14]) <= TOL and relerr(S14[b], So[:14, :14]) <= TOL
        worst = max(worst, _check(batch, oracles, f"frame {t}"))
    print(f"batch N={n_features} hard={hard}: worst per-step rel err {worst:.2e}")


def test_batch_free_running_and_single_filter_agree(gpu_pkg, orc):
    """Filter 0 of the batch (unperturbed) follows the single-filter CUDA path step for step."""
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=8, seed=91)
    g, batch, oracles = _ensemble(gpu_pkg, orc, sc, 3, seed=7)
    for t in range(1, sc.n_frames):
        img = sc.frame(t); picks = sc.picks(t, 24)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}"
        for b, o in enumerate(oracles):
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
        _check(batch, oracles, f"free-running frame {t}", tol=1e-8)


def test_batch_capacity_and_errors(gpu_pkg):
    cfg = gpu_pkg.default_config(xyz_conversion=0)
    with pytest.raises(gpu_pkg.EkfError):
        gpu_pkg.FilterBatch(cfg, 4, feature_capacity=33)
    b = gpu_pkg.FilterBatch(cfg, 4, feature_capacity=8)
    d = b.describe()
    assert (d.n_filters, d.feature_capacity, d.state_capacity) == (4, 8, 14 + 48)
    with pytest.raises(gpu_pkg.EkfError):
        b.step()   # not seeded


def test_small_windows_take_the_warp_matcher(gpu_pkg, orc):
    """Tight process noise and a sharp depth prior shrink the 3-sigma search ellipses to a few pixels: every feature fits the
    warp-per-feature matchers and none is deferred to the CTA matcher; results stay bit-exact against the oracle."""
    small = dict(sigma_vx=1e-4, sigma_vy=1e-4, sigma_vz=1e-4, sigma_wx=1e-4, sigma_wy=1e-4, sigma_wz=1e-4, sigma_rho_0=1e-5, sigma_size=2)
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=5, seed=411, speed=0.05, omega=0.01, accel_sigma=1e-4)
    g, batch, oracles = _ensemble(gpu_pkg, orc, sc, 4, seed=9, perturb=1e-5, **small)
    for t in range(1, sc.n_frames):
        img = sc.frame(t); picks = sc.picks(t, 24)
        for b, o in enumerate(oracles):
            if batch.numOfFeatures(b) == o.numOfFeatures():
                batch.set_full(b, *o.get_full())
        batch.captureNewFrame(img, sc.stamps[t])
        batch.step(picks)
        assert batch.last_match_deferred() == 0, f"frame {t}: {batch.last_match_deferred()} features left the warp path"
        for o in oracles:
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
        _check(batch, oracles, f"small windows frame {t}")
    mu, st = batch.camera_states()
    assert (st[:, 1] > 0).all(), "features must actually match in this scene"
    # the default noise model opens the windows to the 20 px clamp (41 x 41 candidates): the full-window tile matcher
    # (k_match_filter_batch_warp2) decides those as well; only near-ties would go to the CTA matcher, and noise frames have none
    g2, batch2, oracles2 = _ensemble(gpu_pkg, orc, sc, 2, seed=9, perturb=1e-5)
    img = sc.frame(1); picks = sc.picks(1, 24)
    batch2.captureNewFrame(img, sc.stamps[1]); batch2.step(picks)
    assert batch2.last_match_deferred() == 0
    for o in oracles2:
        o.captureNewFrame(img, sc.stamps[1]); o.predict(); o.update(picks)
    _check(batch2, oracles2, "full windows, tile matcher")
