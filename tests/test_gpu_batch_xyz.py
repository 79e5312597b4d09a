"""-m gpu: XYZ conversion in the batched filters (convert2XYZ_ifLinearAll, vslamRansac.cpp:776-780 and :1317).  Every filter
of a batch created with xyz_conversion = 1 must convert exactly the features its own oracle converts, alone
(FilterBatch.convert2XYZ_ifLinearAll) and at the end of every step, together with the removals of that step.  Features are made
to convert by cutting their rho variances, by different factors and for different features per filter."""
import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, assert_scaled_close, make_pair, relerr, seed_features

pytestmark = pytest.mark.gpu


def _ensemble(pkg, orc, sc, B, seed, perturb=2e-3, **cfg_over):
    """A seeded single GPU filter, a batch cloned from it, and B oracle filters holding the same per-hypothesis perturbed camera
    states (filter 0 unperturbed).  XYZ conversion is on unless cfg_over says otherwise."""
    cfg_over.setdefault("xyz_conversion", 1)
    g, _ = make_pair(pkg, orc, sc, **cfg_over)
    seed_features(g, sc)
    cfg = g.cfg
    batch = pkg.FilterBatch(cfg, B, feature_capacity=min(32, sc.n_features + 2))
    batch.seed_from(g)
    rng = np.random.default_rng(seed)
    mu0, S0 = g.get_full()
    cams = np.tile(mu0[:14], (B, 1))
    cams[:, 0:3] += rng.normal(scale=perturb, size=(B, 3))
    cams[:, 3:7] += rng.normal(scale=perturb, size=(B, 4))
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


def _shrink(o, features, factor):
    """mu, Sigma of `o` with the rho variance (row and column pos + 5) of the given features scaled by `factor`."""
    mu, S = o.get_full()
    for i in features:
        p = o.feature(i).position_in_state
        assert not o.feature(i).coding
        S[p + 5, :] *= factor; S[:, p + 5] *= factor
    return mu, S


def _plan(b, t, o):
    """Inverse-depth features of filter b whose rho variance is cut before frame t, and the factor: none for filter 0, one to
    three features for the others."""
    if b == 0:
        return [], 1.0
    inv = [i for i in range(o.numOfFeatures()) if not o.feature(i).coding]
    return inv[(b + t) % 3::3 * (1 + b % 3)][:1 + b % 3], 10.0 ** -(3 + b % 3)


def _codings(f, B=None):
    if B is None:
        return {f.feature(i).real_index: f.feature(i).coding for i in range(f.numOfFeatures())}
    return [[f.feature(b, i).coding for i in range(f.numOfFeatures(b))] for b in range(B)]


def _converted(o, before):
    """Features of `o` that are XYZ now and were inverse depth in `before` (real_index -> coding)."""
    return sum(1 for i in range(o.numOfFeatures()) if o.feature(i).coding and not before[o.feature(i).real_index])


def _check(batch, oracles, ctx, tol=TOL):
    """Per filter: feature count, state dimension, every integer field and the match bit-exact; mu and Sigma within `tol`
    relative and (from identical inputs) within the scaled bars."""
    for b, o in enumerate(oracles):
        assert batch.numOfFeatures(b) == o.numOfFeatures(), f"{ctx} filter {b}: feature count"
        assert batch.state_dim(b) == o.state_dim(), f"{ctx} filter {b}: state dim {batch.state_dim(b)} vs {o.state_dim()}"
        mg, Sg = batch.get_full(b); mo, So = o.get_full()
        em, es = relerr(mg, mo), relerr(Sg, So)
        assert em <= tol and es <= tol, f"{ctx} filter {b}: mu {em:.2e} Sigma {es:.2e}"
        assert_scaled_close(mg, Sg, mo, So, f"{ctx} filter {b}", free_running=tol > TOL)
        for i in range(o.numOfFeatures()):
            a, c = batch.feature(b, i), o.feature(i)
            for f in INT_FIELDS:
                assert getattr(a, f) == getattr(c, f), f"{ctx} filter {b} feature {i} {f}: {getattr(a, f)} vs {getattr(c, f)}"
            assert tuple(a.center) == tuple(c.center), f"{ctx} filter {b} feature {i} match"


def test_explicit_conversion_matches_oracle_per_filter(gpu_pkg, orc):
    sc = gpu_pkg.synth.Scene(n_features=16, n_frames=4, seed=611)
    g, batch, oracles = _ensemble(gpu_pkg, orc, sc, 4, seed=3)
    for t in range(1, sc.n_frames):   # a few frames first: correlated covariance, XYZ-free so far
        img, picks = sc.frame(t), sc.picks(t, 16)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        for o in oracles:
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
    plans = {0: ([], 1.0), 1: ([1, 4, 7], 1e-4), 2: ([0, 15], 1e-3), 3: (list(range(0, 16, 2)), 1e-5)}
    for b, o in enumerate(oracles):
        mu, S = _shrink(o, *plans[b])
        o.set_full(mu, S); batch.set_full(b, mu, S)
    before = [_codings(o) for o in oracles]
    mu_keep, S_keep = batch.get_full(0)
    batch.convert2XYZ_ifLinearAll()
    for o in oracles:
        o.convert2XYZ_ifLinearAll()
    conv = [_converted(o, before[b]) for b, o in enumerate(oracles)]
    assert conv == [0, 3, 2, 8], conv
    _check(batch, oracles, "explicit conversion")
    mu0, S0 = batch.get_full(0)
    assert np.array_equal(mu0, mu_keep) and np.array_equal(S0, S_keep), "a filter with nothing to convert must keep its state"
    # a second call converts nothing more
    batch.convert2XYZ_ifLinearAll()
    for o in oracles:
        o.convert2XYZ_ifLinearAll()
    _check(batch, oracles, "second explicit conversion")


@pytest.mark.parametrize("n_features,hard,B,seed", [(12, False, 4, 501), (30, True, 5, 502)])
def test_step_converts_like_oracle_per_filter(gpu_pkg, orc, n_features, hard, B, seed):
    """Identical inputs per step (batch state <- oracle state, after the variance cut); the step's conversions, removals,
    codings and states must be the oracle's.  Later steps run the mixed-coding RANSAC, updates and rescue."""
    sc = gpu_pkg.synth.Scene(n_features=n_features, n_frames=6, seed=seed, hard=hard)
    g, batch, oracles = _ensemble(gpu_pkg, orc, sc, B, seed=5)
    multi = none_beside_multi = remove_and_convert = False
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, n_features)
        before = []
        for b, o in enumerate(oracles):
            mu, S = _shrink(o, *_plan(b, t, o))
            o.set_full(mu, S); batch.set_full(b, mu, S)
            before.append(_codings(o))
        batch.captureNewFrame(img, sc.stamps[t])
        batch.step(picks)
        mu14, S14, st = batch.camera_states(want_sigma=True)
        conv = []
        for b, o in enumerate(oracles):
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            got = (st[b, 1], st[b, 2], st[b, 3], st[b, 4], st[b, 6], st[b, 7])
            want = (so.n_matched, so.n_li, so.n_hi, so.ransac_hypotheses, so.n_removed, so.topup_request)
            assert got == want, f"frame {t} filter {b}: stats {got} vs oracle {want}"
            mo, So = o.get_full()
            assert relerr(mu14[b], mo[:14]) <= TOL and relerr(S14[b], So[:14, :14]) <= TOL
            conv.append(_converted(o, before[b]))
            remove_and_convert |= so.n_removed > 0 and conv[b] > 0
        multi_now = [b for b in range(B) if conv[b] >= 2]
        multi |= bool(multi_now)
        none_beside_multi |= bool(multi_now) and 0 in conv
        print(f"frame {t}: conversions per filter {conv}, removals {list(st[:, 6])}")
        _check(batch, oracles, f"frame {t}")
    assert multi, "no filter converted two or more features in one step"
    assert none_beside_multi, "no step in which one filter converted several features and another none"
    if hard:
        assert remove_and_convert, "no step in which a filter both removed and converted features"


def test_free_running_filter0_follows_single_filter(gpu_pkg, orc):
    """Filter 0 (unperturbed) against the single-filter CUDA path with xyz_conversion = 1, both starting from the same state with
    four rho variances cut: the first step converts them, the later ones run with mixed codings."""
    sc = gpu_pkg.synth.Scene(n_features=24, n_frames=9, seed=92)
    g, batch, oracles = _ensemble(gpu_pkg, orc, sc, 3, seed=8)
    mu, S = g.get_full()
    for i in (2, 9, 13, 20):
        p = g.feature(i).position_in_state
        S[p + 5, :] *= 1e-4; S[:, p + 5] *= 1e-4
    g.set_full(mu, S)
    batch.set_full(0, mu, S)
    n_xyz = 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert mb.shape == mg.shape, f"frame {t}: state dim {mb.size} vs {mg.size}"
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}: mu {relerr(mb, mg):.2e} Sigma {relerr(Sb, Sg):.2e}"
        cb = [batch.feature(0, i).coding for i in range(batch.numOfFeatures(0))]
        cg = [g.feature(i).coding for i in range(g.numOfFeatures())]
        assert cb == cg, f"frame {t}: codings"
        n_xyz = sum(cg)
    assert n_xyz >= 4


def test_no_cost_when_nothing_converts(gpu_pkg, orc):
    """Untouched variances: no feature passes the linearity test.  Conversion on and off then give bit-identical states and the
    same kernel launches per step."""
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=6, seed=93, hard=True)
    runs = []
    for xyz in (0, 1):
        g, batch, _ = _ensemble(gpu_pkg, orc, sc, 4, seed=4, xyz_conversion=xyz)
        launches, states = [], []
        for t in range(1, sc.n_frames):
            k0 = batch.kernel_launches()
            batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(sc.picks(t, 20))
            launches.append(batch.kernel_launches() - k0)
            states.append([batch.get_full(b) for b in range(4)])
        assert not any(any(c) for c in _codings(batch, 4))
        runs.append((launches, states))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1, f"launches per step: off {l0}, on {l1}"
    for t, (a, c) in enumerate(zip(s0, s1)):
        for b, ((ma, Sa), (mc, Sc)) in enumerate(zip(a, c)):
            assert np.array_equal(ma, mc) and np.array_equal(Sa, Sc), f"step {t + 1} filter {b}"


def test_create_accepts_xyz_conversion(gpu_pkg):
    cfg = gpu_pkg.default_config()
    assert cfg.xyz_conversion == 1
    b = gpu_pkg.FilterBatch(cfg, 2, feature_capacity=8)
    assert b.describe().n_filters == 2
    with pytest.raises(gpu_pkg.EkfError):
        b.convert2XYZ_ifLinearAll()   # not seeded
    for over in (dict(kernel_size=1000), dict(scale=2), dict(forsePlane=1)):
        with pytest.raises(gpu_pkg.EkfError):
            gpu_pkg.FilterBatch(gpu_pkg.default_config(**over), 2, feature_capacity=8)
