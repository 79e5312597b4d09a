"""Shared helpers for the parity tests (oracle vs CUDA path on the same seeded inputs)."""
import numpy as np

# BASELINE.json tolerance: state and covariance within 1e-9 relative in fp64 (norm-wise, per step from
# identical inputs — SURVEY.md §7 "Hard parts").
TOL = 1e-9
# The same comparisons in the covariance's own units (scaled_errors): a norm-wise ratio over the whole of Sigma lets through
# errors of 10 % in the anchor blocks, whose variances (~4e-10) are far below |Sigma|_F * 1e-9.  Two fp64 evaluations of the
# same update (the oracle's LU and a LAPACK Cholesky) differ by <= 1.1e-11 in correlation units and <= 2.5e-13 sigma in the mean.
TOL_SCALED_SIGMA = 1e-9   # max |dSigma_ij| / sqrt(Sigma_ii Sigma_jj)
TOL_SCALED_MU = 1e-10     # max |dmu_i| / sqrt(Sigma_ii)

INT_FIELDS = ("position_in_state", "position_in_z", "coding", "n_tot", "n_find", "real_index",
              "is_in_innovation", "is_in_li", "is_in_hi", "remove_flag")


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    d = np.linalg.norm(a - b)
    s = np.linalg.norm(b)
    return d / s if s > 0 else d


def make_pair(pkg, orc, scene, capacity=None, **cfg_over):
    over = scene.config_overrides()
    over.update(cfg_over)
    cfg = pkg.default_config(**over)
    g = pkg.VSlamFilter(cfg, feature_capacity=capacity or max(8, scene.n_features + 8))
    o = orc.OracleFilter(cfg, kind=0, omp=True)
    return g, o


def make_oracle(pkg, orc, scene, kind=0, omp=False, **cfg_over):
    """A CPU oracle filter configured for `scene` (no GPU needed)."""
    over = scene.config_overrides()
    over.update(cfg_over)
    return orc.OracleFilter(pkg.default_config(**over), kind=kind, omp=omp)


def seed_features(filt, scene):
    filt.captureNewFrame(scene.frame(0), scene.stamps[0])
    return [filt.addFeature(*p) for p in scene.feature_pixels]


def assert_tables_equal(g, o, fields=INT_FIELDS, ctx=""):
    """Integer / flag state of every feature must be bit-identical."""
    assert g.numOfFeatures() == o.numOfFeatures(), f"{ctx}: feature count {g.numOfFeatures()} vs {o.numOfFeatures()}"
    for i in range(g.numOfFeatures()):
        a, b = g.feature(i), o.feature(i)
        for f in fields:
            assert getattr(a, f) == getattr(b, f), f"{ctx}: feature {i} field {f}: gpu {getattr(a, f)} oracle {getattr(b, f)}"


def scaled_errors(g_mu, g_S, o_mu, o_S):
    """max |dSigma_ij| / sqrt(Sigma_ii Sigma_jj) and max |dmu_i| / sqrt(Sigma_ii), both with the diagonal of the reference
    (o_S).  Where Sigma_ii = 0 exactly (no uncertainty), row and column i and mu_i must agree exactly: any difference there
    is an infinite error."""
    g_mu = np.asarray(g_mu, dtype=np.float64); o_mu = np.asarray(o_mu, dtype=np.float64)
    g_S = np.asarray(g_S, dtype=np.float64); o_S = np.asarray(o_S, dtype=np.float64)
    d = np.diag(o_S).copy()
    assert (d >= 0).all(), "reference covariance with a negative variance"
    s = np.sqrt(d)
    dS = np.abs(g_S - o_S)
    dm = np.abs(g_mu - o_mu)
    with np.errstate(divide="ignore", invalid="ignore"):   # Sigma_ii = 0: x / 0 = inf unless x = 0; NaN counts as inf
        rS = np.where(dS == 0, 0.0, dS / np.outer(s, s))
        rm = np.where(dm == 0, 0.0, dm / s)
    return float(np.where(np.isnan(rS), np.inf, rS).max()), float(np.where(np.isnan(rm), np.inf, rm).max())


def assert_scaled_close(g_mu, g_S, o_mu, o_S, ctx="", free_running=False):
    """The bars in the covariance's own units, for comparisons from identical inputs; a free-running comparison only reports
    the figure (its states drift apart by design).  Returns (Sigma, mu) scaled errors."""
    sS, sm = scaled_errors(g_mu, g_S, o_mu, o_S)
    print(f"{ctx}: scaled err Sigma {sS:.2e} mu {sm:.2e} sigma{' (free running, not a bar)' if free_running else ''}")
    if not free_running:
        assert sS <= TOL_SCALED_SIGMA, f"{ctx}: max |dSigma_ij| / sqrt(Sigma_ii Sigma_jj) = {sS:.3e}"
        assert sm <= TOL_SCALED_MU, f"{ctx}: max |dmu_i| / sigma_i = {sm:.3e}"
    return sS, sm


def assert_state_close(g, o, tol=TOL, ctx="", free_running=False):
    """mu and Sigma of the filter g against the reference o: the norm-wise bar (tol), and for comparisons from identical inputs
    the scaled bars of assert_scaled_close."""
    mg, Sg = g.get_full()
    mo, So = o.get_full()
    assert mg.shape == mo.shape, ctx
    em, es = relerr(mg, mo), relerr(Sg, So)
    assert em <= tol, f"{ctx}: mu rel err {em:.3e}"
    assert es <= tol, f"{ctx}: Sigma rel err {es:.3e}"
    assert_scaled_close(mg, Sg, mo, So, ctx, free_running)
    return em, es


# ---- independent fp64 evaluation of the stacked EKF correction (numpy / LAPACK) -----------------------------
def _feature_rows(feats, sel):
    """idx (m, 13) state indices, Hc (m, 2, 13), innovation z - h (2m) for the selected features, in patch order.
    XYZ features use 10 entries: the last three columns are zero and point at index 0."""
    m = len(sel)
    idx = np.zeros((m, 13), dtype=np.int64)
    Hc = np.zeros((m, 2, 13))
    nu = np.zeros(2 * m)
    for j, i in enumerate(sel):
        f = feats[i]
        nd = 7 + (3 if f.coding else 6)
        idx[j, :7] = np.arange(7)
        idx[j, 7:nd] = f.position_in_state + np.arange(nd - 7)
        H = np.array(list(f.H), dtype=np.float64).reshape(2, 13)
        Hc[j, :, :nd] = H[:, :nd]
        nu[2 * j] = f.z[0] - f.h[0]
        nu[2 * j + 1] = f.z[1] - f.h[1]
    return idx, Hc, nu


def numpy_stacked_update(mu, S, feats, sel, sigma_pixel_2, chunk=256):
    """mu + K nu and Sigma - Sigma H^T (H Sigma H^T + R)^-1 H Sigma (vslamRansac.cpp:1053-1060) followed by
    normalizeQuaternion (vslamRansac.cpp:1625-1642), evaluated with numpy / LAPACK in fp64 from the sparse rows
    of H (13 non-zeros per row).  Independent of both the oracle and the CUDA path: used where a dense oracle
    frame is too slow (n = 12014)."""
    import scipy.linalg as sla
    n = mu.size
    idx, Hc, nu = _feature_rows(feats, sel)
    m = len(sel)
    W = np.empty((n, 2 * m))
    for a in range(0, m, chunk):                       # W = Sigma H^T, a block of features at a time
        b = min(m, a + chunk)
        G = S[:, idx[a:b].reshape(-1)].reshape(n, b - a, 13)
        W[:, 2 * a:2 * b] = np.einsum("nfc,frc->nfr", G, Hc[a:b]).reshape(n, 2 * (b - a))
    St = np.empty((2 * m, 2 * m))
    for a in range(0, m, chunk):                       # St = H W + R
        b = min(m, a + chunk)
        G = W[idx[a:b].reshape(-1), :].reshape(b - a, 13, 2 * m)
        St[2 * a:2 * b] = np.einsum("frc,fck->frk", Hc[a:b], G).reshape(2 * (b - a), 2 * m)
    St[np.diag_indices(2 * m)] += sigma_pixel_2
    St = 0.5 * (St + St.T)
    L = sla.cholesky(St, lower=True)
    V = sla.solve_triangular(L, W.T, lower=True)       # k x n
    y = sla.solve_triangular(L, nu, lower=True)
    mu1 = mu + V.T @ y
    S1 = S - V.T @ V
    q = mu1[3:7].copy()
    nq = np.linalg.norm(q)
    J = (nq * nq * np.eye(4) - np.outer(q, q)) / nq ** 3
    mu1[3:7] = q / nq
    S1[3:7, :] = J @ S1[3:7, :]
    S1[:, 3:7] = S1[:, 3:7] @ J.T
    return mu1, S1


def near_tie_scene():
    """Four 320 x 240 frames made to produce near-ties in the NCC search — a smooth gradient, an exactly periodic texture (many
    candidates with identical sums), a coarse 4-level block image and a saturated patch (flat windows) — with 48 templates cut
    from each at random positions.  Returns frames, templates (F*M, 11, 11), h (F*M, 2), S (F*M, 4), F, M."""
    rng = np.random.default_rng(11)
    Wd, Ht, w, M = 320, 240, 11, 48
    yy, xx = np.mgrid[0:Ht, 0:Wd]
    smooth = (127 + 60 * np.sin(xx / 23.0) + 50 * np.cos(yy / 17.0) + rng.normal(scale=1.5, size=(Ht, Wd))).clip(0, 255)
    periodic = (((xx % 8) * 16 + (yy % 8) * 12) % 256).astype(np.float64)
    coarse = ((rng.integers(0, 4, size=(Ht // 4 + 1, Wd // 4 + 1)).repeat(4, 0).repeat(4, 1)[:Ht, :Wd]) * 64).astype(np.float64)
    sat = smooth.copy(); sat[60:140, 80:220] = 255
    frames = np.stack([smooth, periodic, coarse, sat]).astype(np.uint8)
    F = frames.shape[0]
    half = w // 2
    u = rng.integers(40, Wd - 40, size=(F, M)); v = rng.integers(40, Ht - 40, size=(F, M))
    templates = np.zeros((F, M, w, w), dtype=np.uint8)
    for f in range(F):
        for i in range(M):
            templates[f, i] = frames[f, v[f, i] - half:v[f, i] + half + 1, u[f, i] - half:u[f, i] + half + 1]
    h = np.stack([u, v], axis=-1).astype(np.float64) + rng.normal(scale=2.0, size=(F, M, 2))
    S = np.zeros((F, M, 4)); S[..., 0] = 40.0; S[..., 3] = 40.0
    templates = templates.reshape(F * M, w, w); h = h.reshape(F * M, 2); S = S.reshape(F * M, 4)
    return frames, templates, h, S, F, M
