"""CPU: the oracle (oracle/ekf_oracle.hpp) against independent checks — finite-difference Jacobians,
dense-vs-structured identities and a numpy restatement of the reference algebra.  The reference
ships no tests for this path (SURVEY.md §4); these, tests/test_oracle_vs_ref.py (the reference's
own sources compiled against API shims) and tests/golden/ are what pin the oracle."""
import numpy as np
import pytest

from helpers import make_oracle, relerr, seed_features


def _scene(pkg, **kw):
    return pkg.synth.Scene(**kw)


def _dense_H(o):
    """Stack the compact 2x13 Jacobians of the in-innovation features into the dense k x n Ht."""
    n = o.state_dim()
    rows, hs, zs, idx = [], [], [], []
    for i in range(o.numOfFeatures()):
        f = o.feature(i)
        if not f.is_in_innovation:
            continue
        Hc = np.array(list(f.H)).reshape(2, 13)
        H = np.zeros((2, n))
        H[:, 0:7] = Hc[:, 0:7]
        fs = 3 if f.coding else 6
        H[:, f.position_in_state:f.position_in_state + fs] = Hc[:, 7:7 + fs]
        rows.append(H); hs.append(list(f.h)); zs.append(list(f.z)); idx.append(i)
    return np.vstack(rows), np.array(hs).reshape(-1), np.array(zs).reshape(-1), idx


def test_init_state_matches_reference_constructor(pkg, orc):
    """vslamRansac.cpp:163-216."""
    sc = _scene(pkg, n_features=4, n_frames=2)
    o = make_oracle(pkg, orc, sc)
    mu, S = o.get_full()
    assert mu.shape == (14,)
    assert np.array_equal(mu, np.array([0, 0, 0, 0, 0, -0.707106781, 0.707106781, 0, 0, 0, 0, 0, 0, 1.0]))
    d = np.full(14, 4e-10); d[7:10] = 0.0004 ** 2; d[10:13] = 0.0004 ** 2; d[13] = 0.09
    assert np.allclose(S, np.diag(d), rtol=1e-15, atol=0)


def test_predict_covariance_is_F_Sigma_Ft_plus_Q(pkg, orc):
    """Sigma <- Fc Sigma Fc^T + Q (vslamRansac.cpp:451-480): F recovered by finite differences of
    the oracle's own Predict_State, Q from the reference formula."""
    sc = _scene(pkg, n_features=6, n_frames=3, seed=3)
    o = make_oracle(pkg, orc, sc)
    seed_features(o, sc)
    mu0, S0 = o.get_full()
    rng = np.random.default_rng(0)
    mu0[7:13] = rng.normal(scale=0.05, size=6)     # non-zero v, w so the quaternion Jacobians matter
    A = rng.normal(size=S0.shape) * 1e-3
    S0 = S0 + A @ A.T * 1e-3
    n = mu0.size
    dT = sc.stamps[1] - sc.stamps[0]

    def predicted_mu(m):
        o.set_full(m, S0)
        o.captureNewFrame(sc.frame(1), o._stamp + dT)
        o._stamp += dT
        o.predict()
        return o.get_full()[0]

    o._stamp = sc.stamps[0]
    base = predicted_mu(mu0)
    S1 = o.get_full()[1]
    F = np.eye(n)
    eps = 1e-6
    for j in range(13):
        mp = mu0.copy(); mp[j] += eps
        mm = mu0.copy(); mm[j] -= eps
        F[:13, j] = (predicted_mu(mp)[:13] - predicted_mu(mm)[:13]) / (2 * eps)
    assert np.allclose(base[13:], mu0[13:])        # features and map_scale untouched
    # Q = F[:,7:13] (2 Vmax / dT^2) F[:,7:13]^T (vslamRansac.cpp:463-473, Vcontrol = false)
    V = np.diag([2 * 0.01 ** 2] * 6) / dT / dT
    Q = np.zeros((n, n)); Q[:13, :13] = F[:13, 7:13] @ V @ F[:13, 7:13].T
    want = F @ S0 @ F.T + Q
    assert relerr(S1, want) < 5e-8                 # limited by the finite-difference F


def test_measurement_jacobian_finite_difference(pkg, orc):
    """Compact H (2 x 13) of every gated-in feature vs central differences of the oracle's h(mu)
    (vslamRansac.cpp:508-551, camModel.cpp:68-111)."""
    sc = _scene(pkg, n_features=10, n_frames=3, seed=8)
    o = make_oracle(pkg, orc, sc)
    seed_features(o, sc)
    mu0, S0 = o.get_full()
    mu0[7:13] = 0.0                                # v = w = 0: predict leaves the pose where it is
    rng = np.random.default_rng(1)
    mu0[0:3] += rng.normal(scale=0.02, size=3)
    q = mu0[3:7] + rng.normal(scale=0.01, size=4); mu0[3:7] = q / np.linalg.norm(q)
    stamp = [sc.stamps[0]]

    def h_all(m):
        o.set_full(m, S0)
        stamp[0] += 1.0 / 30
        o.captureNewFrame(sc.frame(1), stamp[0])
        o.predict()
        return [(f.is_in_innovation, np.array(list(f.h)), np.array(list(f.H)).reshape(2, 13), f.position_in_state)
                for f in (o.feature(i) for i in range(o.numOfFeatures()))]

    base = h_all(mu0)
    assert sum(b[0] for b in base) >= 8
    eps = 1e-6
    for i, (inn, h, Hc, pos) in enumerate(base):
        if not inn:
            continue
        cols = list(range(7)) + list(range(pos, pos + 6))
        for c, j in enumerate(cols):
            mp = mu0.copy(); mp[j] += eps
            mm = mu0.copy(); mm[j] -= eps
            hp, hm = h_all(mp)[i][1], h_all(mm)[i][1]
            fd = (hp - hm) / (2 * eps)
            assert np.allclose(fd, Hc[:, c], rtol=2e-6, atol=2e-5), f"feature {i} column {c}: fd {fd} analytic {Hc[:, c]}"


def test_S_blocks_equal_dense_H_Sigma_Ht(pkg, orc):
    """The 2x2 blocks the matcher consumes are the diagonal blocks of St = Ht Sigma Ht^T + sigma^2 I
    (vslamRansac.cpp:598, 875)."""
    sc = _scene(pkg, n_features=14, n_frames=3, seed=5)
    o = make_oracle(pkg, orc, sc)
    seed_features(o, sc)
    o.captureNewFrame(sc.frame(1), sc.stamps[1]); o.predict()
    mu, S = o.get_full()
    H, h, z, idx = _dense_H(o)
    St = H @ S @ H.T + 4.0 * np.eye(H.shape[0])
    assert relerr(o.St(), St) < 1e-12
    blocks = o.S_blocks()
    for j, i in enumerate(idx):
        assert relerr(blocks[i], St[2 * j:2 * j + 2, 2 * j:2 * j + 2]) < 1e-12


def test_update_matches_numpy_restatement(pkg, orc):
    """One low-innovation update against plain numpy: K = Sigma H^T St^-1, mu += K (z - h),
    Sigma <- (I - K H) Sigma, then normalizeQuaternion (vslamRansac.cpp:1053-1064, 1625-1642)."""
    sc = _scene(pkg, n_features=18, n_frames=3, seed=21)
    o = make_oracle(pkg, orc, sc)
    seed_features(o, sc)
    o.captureNewFrame(sc.frame(1), sc.stamps[1]); o.predict()
    assert o.match() == 18
    mu, S = o.get_full()
    H, h, z, idx = _dense_H(o)
    o.update_after_match(sc.picks(1, 18))
    st = o.stats()
    assert st.n_li == 18 and st.n_hi == 0
    St = H @ S @ H.T + 4.0 * np.eye(H.shape[0])
    K = S @ H.T @ np.linalg.inv(St)
    mu1 = mu + K @ (z - h)
    S1 = (np.eye(mu.size) - K @ H) @ S
    q = mu1[3:7].copy(); nq = np.linalg.norm(q)
    J = (nq * nq * np.eye(4) - np.outer(q, q)) / nq ** 3
    Qc = np.eye(mu.size); Qc[3:7, 3:7] = J
    mu1[3:7] = q / nq
    S1 = Qc @ S1 @ Qc.T
    mu_o, S_o = o.get_full()
    assert relerr(mu_o, mu1) < 1e-11
    assert relerr(S_o, S1) < 1e-9   # LU-inverse vs numpy inverse on cond(St) ~ 1e5


def test_add_feature_structure(pkg, orc):
    """addFeature (vslamRansac.cpp:309-371): new block = [I3 | J] Sigma[0:7, :] with pixel and rho
    variances on the new diagonal; sigma_rho_0 enters UNSQUARED (quirk, :365)."""
    sc = _scene(pkg, n_features=3, n_frames=2, seed=2)
    o = make_oracle(pkg, orc, sc)
    o.captureNewFrame(sc.frame(0), sc.stamps[0])
    assert o.addFeature(*sc.feature_pixels[0]) == 1
    mu, S = o.get_full()
    assert mu.size == 20
    assert np.array_equal(mu[14:17], mu[0:3])
    assert mu[19] == 0.1
    assert abs(S[19, 19] - 0.25) < 1e-15
    assert np.allclose(S[14:17, 14:17], S[0:3, 0:3])
    assert np.allclose(S[14:17, 0:14], S[0:3, 0:14])
    assert np.allclose(S, S.T, atol=1e-18)
    # bearing: the new feature re-projects onto the pixel it was initialised from
    th, ph = mu[17], mu[18]
    m = np.array([np.sin(th) * np.cos(ph), -np.sin(ph), np.cos(th) * np.cos(ph)])
    Rcw = pkg.synth.quat2rot(mu[3:7] * np.array([1, -1, -1, -1.0]))
    uv = sc.cam.project(Rcw @ m)
    assert np.allclose(uv, sc.feature_pixels[0], atol=1e-6)


def _ncc_numpy(t, p):
    """computeCorrelation (Patch.cpp:293-329) in numpy: two passes, double accumulation row-major,
    result rounded to float."""
    n = t.size
    m1 = float(t.astype(np.int64).sum()) / n
    m2 = float(p.astype(np.int64).sum()) / n
    n1 = n2 = c = 0.0
    for a, b in zip(t.reshape(-1).astype(np.float64), p.reshape(-1).astype(np.float64)):
        n1 += (a - m1) * (a - m1)
        n2 += (b - m2) * (b - m2)
        c += (a - m1) * (b - m2)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.float32(c / np.sqrt(n2 * n1))


def _find_match_numpy(frame, t, h, S, sigma_size=3.0, thr=0.8, clamp=20.0):
    """Patch::findMatch (Patch.cpp:215-291) restated with numpy scalars (float32 where the reference
    types float)."""
    f32 = np.float32
    Hh, Ww = frame.shape
    w = t.shape[0]
    uc, vc = int(h[0]), int(h[1])
    inv = np.linalg.inv(S.reshape(2, 2))
    x2, y2, yx = f32(inv[0, 0]), f32(inv[1, 1]), f32(2 * inv[1, 0])
    s2 = f32(sigma_size) * f32(sigma_size)
    du = min(f32(sigma_size * np.sqrt(S[0])), f32(clamp))
    dv = min(f32(sigma_size * np.sqrt(S[3])), f32(clamp))
    best, arg = f32(-1), None
    i = int(f32(uc) - du)
    while f32(i) <= f32(uc) + du:
        j = int(f32(vc) - dv)
        while f32(j) <= f32(vc) + dv:
            if i > w // 2 and j > w // 2 and i < Ww - w // 2 and j < Hh - w // 2:
                di, dj = f32(i - uc), f32(j - vc)
                e = f32(f32(f32(x2 * di) * di) + f32(f32(y2 * dj) * dj)) + f32(f32(yx * di) * dj)
                if f32(e) <= s2:
                    sc = _ncc_numpy(t, frame[j - w // 2:j - w // 2 + w, i - w // 2:i - w // 2 + w])
                    if sc > best:
                        best, arg = sc, (i, j)
            j += 1
        i += 1
    if best < f32(thr) or arg is None:
        return (-1, -1), best
    return arg, best


def test_matcher_matches_numpy_restatement(pkg, orc):
    d = pkg.synth.match_batch_inputs(n_frames=1, features_per_frame=6, width=160, height=120, window=11, seed=4,
                                     s_diag=6.0, pred_sigma=1.5)
    uv, sc = orc.match_batch(d["frames"], d["templates"], d["h"], d["S"], sigma_size=3.0)
    for k in range(6):
        (i, j), best = _find_match_numpy(d["frames"][0], d["templates"][k], d["h"][k], d["S"][k])
        assert (uv[k, 0], uv[k, 1]) == (i, j)
        assert np.float32(sc[k]) == best
    assert (uv[:, 0] >= 0).sum() >= 4


def test_float_oracle_stays_near_double_oracle(pkg, orc):
    """kind=1 (all float, what the reference really runs) vs kind=0 (fp64 parity target): decisions
    agree on an easy scene and the state differs at fp32 level — documents the precision gap."""
    sc = _scene(pkg, n_features=12, n_frames=3, seed=6)
    od = make_oracle(pkg, orc, sc, kind=0)
    of = make_oracle(pkg, orc, sc, kind=1)
    for o in (od, of):
        seed_features(o, sc)
        o.captureNewFrame(sc.frame(1), sc.stamps[1]); o.predict(); o.update(sc.picks(1, 12))
    for i in range(12):
        a, b = od.feature(i), of.feature(i)
        assert tuple(a.center) == tuple(b.center) and a.is_in_li == b.is_in_li
    e = relerr(of.get_full()[0], od.get_full()[0])
    assert 1e-12 < e < 1e-3


def test_sparse_numpy_update_matches_oracle(pkg, orc):
    """tests/helpers.numpy_stacked_update (the independent fp64 evaluation the N = 2000 GPU test is checked
    against) reproduces the oracle's low-innovation update on a map small enough for the dense oracle."""
    from helpers import numpy_stacked_update
    sc = _scene(pkg, n_features=40, n_frames=3, seed=21)
    o = make_oracle(pkg, orc, sc, omp=True)
    seed_features(o, sc)
    o.captureNewFrame(sc.frame(1), sc.stamps[1]); o.predict()
    assert o.match() == 40
    mu, S = o.get_full()
    feats = [o.feature(i) for i in range(o.numOfFeatures())]
    o.update_after_match(sc.picks(1, 40))
    st = o.stats()
    assert st.n_hi == 0 and st.n_li > 30
    sel = [i for i in range(o.numOfFeatures()) if o.feature(i).is_in_li]
    mu1, S1 = numpy_stacked_update(mu, S, feats, sel, 4.0, chunk=16)
    mo, So = o.get_full()
    assert relerr(mo, mu1) < 1e-12 and relerr(So, S1) < 1e-12
    assert relerr(So - S, S1 - S) < 1e-10


def test_scaled_bar_catches_what_the_norm_bar_misses(pkg, orc):
    """tests/helpers.scaled_errors: errors in the small-variance parts of Sigma that the norm-wise bar (1e-9 of |Sigma|_F) lets
    through — every anchor-xyz block off by 10 %, the quaternion block off by 5e-4 — fail the bar in the covariance's own
    units, while two fp64 evaluations of the same update (the oracle and numpy / LAPACK) pass it."""
    from helpers import TOL, TOL_SCALED_MU, TOL_SCALED_SIGMA, numpy_stacked_update, scaled_errors
    N = 150
    sc = _scene(pkg, n_features=N, n_frames=3, seed=6)
    o = make_oracle(pkg, orc, sc, omp=True)
    seed_features(o, sc)
    o.captureNewFrame(sc.frame(1), sc.stamps[1]); o.predict(); o.update(sc.picks(1, N))
    o.captureNewFrame(sc.frame(2), sc.stamps[2]); o.predict()
    assert o.match() > 0
    mu0, S0 = o.get_full()
    feats = [o.feature(i) for i in range(o.numOfFeatures())]
    o.update_after_match(sc.picks(2, N))
    st = o.stats()
    assert st.n_hi == 0 and st.n_removed == 0 and st.n_li > 100
    sel = [i for i in range(o.numOfFeatures()) if o.feature(i).is_in_li]
    mu_np, S_np = numpy_stacked_update(mu0, S0, feats, sel, 4.0)
    mu, S = o.get_full()
    sS, sm = scaled_errors(mu_np, S_np, mu, S)
    assert sS <= TOL_SCALED_SIGMA / 10 and sm <= TOL_SCALED_MU / 10, (sS, sm)

    anchors = S.copy()
    for i in range(o.numOfFeatures()):
        p = o.feature(i).position_in_state
        anchors[p:p + 3, p:p + 3] *= 1.1
    quat = S.copy()
    quat[3:7, 3:7] *= 1 + 5e-4
    for name, P, expect in (("anchor-xyz blocks x 1.1", anchors, 0.1), ("quaternion block x (1 + 5e-4)", quat, 5e-4)):
        assert relerr(P, S) <= TOL, f"{name}: the norm-wise bar no longer passes it"
        sS, sm = scaled_errors(mu, P, mu, S)
        assert sm == 0.0
        assert sS > TOL_SCALED_SIGMA, f"{name}: scaled error {sS:.2e} passes the bar"
        assert abs(sS - expect) <= 0.01 * expect, f"{name}: scaled error {sS:.3e}, expected {expect}"


def test_scaled_errors_zero_variance():
    """Entries with Sigma_ii = 0 must agree exactly; any difference there is an infinite scaled error."""
    from helpers import scaled_errors
    S = np.diag([4.0, 0.0, 1.0]); mu = np.array([1.0, 2.0, 3.0])
    assert scaled_errors(mu, S, mu, S) == (0.0, 0.0)
    T = S.copy(); T[0, 2] = T[2, 0] = 1e-3
    assert scaled_errors(mu, T, mu, S)[0] == 1e-3 / 2.0
    T = S.copy(); T[1, 0] = T[0, 1] = 1e-300
    assert scaled_errors(mu, T, mu, S)[0] == np.inf
    m2 = mu.copy(); m2[1] = np.nextafter(m2[1], 3.0)
    assert scaled_errors(m2, S, mu, S)[1] == np.inf
    m2 = mu.copy(); m2[2] += 2.0 ** -40
    assert scaled_errors(m2, S, mu, S)[1] == 2.0 ** -40
