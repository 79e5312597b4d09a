"""CPU: the oracle against the REFERENCE'S OWN sources (oracle/_ref: vslamRansac.cpp, Patch.cpp,
camModel.cpp, utils.cpp compiled unmodified against the API stand-ins of oracle/shim).  Each scenario runs
one filter and records what is compared; the reference's records are stored under tests/golden/vs_ref/
(oracle/gen_golden_vs_ref.py), so the comparison runs wherever the repository is checked out.

fp64 variant (the reference with `float` re-typed to double) vs the oracle's all-double kind, and
the fp32 variant (as written) vs the all-float kind: integer tables must be identical and the state
must agree to rounding (observed: bit-identical — same operation order).  To keep the stored records small,
Sigma is recorded as P^T Sigma P for a fixed seeded n x 4 Gaussian P (every entry of Sigma enters it), each
Jacobian row H_i as its product with a fixed seeded vector, and templates as SHA-256 digests."""
import hashlib
import os

import numpy as np
import pytest

from helpers import INT_FIELDS, relerr

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vs_ref")
VARIANTS = [pytest.param(True, 2, 1e-12, id="fp64"), pytest.param(False, 1, 1e-5, id="fp32")]
SEQUENCES = [(12, False, 3), (30, False, 41), (40, True, 9)]
RTS_CASES = [(1, False), (2, False), (3, True)]
EXACT = ("_center", "_dt", "_uv")     # float records that must agree bit for bit
H_PROBE = np.random.default_rng(26).standard_normal(26)


def case_id(scenario, fp64, *params):
    return "_".join([scenario, "fp64" if fp64 else "fp32"] + [str(p) for p in params])


def _cfg(pkg, sc, **over):
    o = sc.config_overrides()
    o["xyz_conversion"] = 1  # VSlamFilter::update always ends with convert2XYZ_ifLinearAll (vslamRansac.cpp:1317)
    o.update(over)
    return pkg.default_config(**o)


def _sketch(S):
    P = np.random.default_rng(S.shape[0]).standard_normal((S.shape[0], 4))
    return P.T @ S @ P


def _digest(arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def _state(rec, key, f):
    mu, S = f.get_full()
    rec[key + "_mu"] = mu
    rec[key + "_Ssketch"] = _sketch(S)


def _tables(rec, key, f, skip=()):
    n = f.numOfFeatures()
    feats = [f.feature(i) for i in range(n)]
    rec[key + "_tab"] = np.array([[0 if fld in skip else getattr(a, fld) for fld in INT_FIELDS] for a in feats],
                                 dtype=np.int32).reshape(n, len(INT_FIELDS))
    rec[key + "_center"] = np.array([tuple(a.center) for a in feats], dtype=np.float32).reshape(n, 2)
    rec[key + "_tmpl"] = _digest(f.template(i, 0) for i in range(n))


def _hypotheses(f):
    return f.last_hypotheses() if hasattr(f, "last_hypotheses") else f.stats().ransac_hypotheses


def save_record(path, rec):
    """A record as one flat int64 and one flat float64 array plus a key / shape index (a few hundred small arrays
    would cost more in per-array headers than in data)."""
    keys = sorted(rec)
    arrs = [np.asarray(rec[k]) for k in keys]
    is_int = np.array([a.dtype.kind in "iub" for a in arrs])
    np.savez_compressed(path, keys=np.array(keys), is_int=is_int, ndim=np.array([a.ndim for a in arrs]),
                        shape=np.array([d for a in arrs for d in a.shape], dtype=np.int64),
                        ints=np.concatenate([np.zeros(0, np.int64)] + [a.ravel().astype(np.int64) for a, i in zip(arrs, is_int) if i]),
                        floats=np.concatenate([np.zeros(0)] + [a.ravel().astype(np.float64) for a, i in zip(arrs, is_int) if not i]))


def load_record(path):
    z = np.load(path)
    flat = {True: z["ints"], False: z["floats"]}
    pos = {True: 0, False: 0}
    shapes = iter(z["shape"].tolist())
    rec = {}
    for k, nd, i in zip(z["keys"].tolist(), z["ndim"].tolist(), z["is_int"].tolist()):
        shape = tuple(next(shapes) for _ in range(nd))
        size = int(np.prod(shape))
        rec[k] = flat[i][pos[i]:pos[i] + size].reshape(shape)
        pos[i] += size
    return rec


def compare(rec, case, tol):
    """Every record of the stored reference run against the oracle's: integers and EXACT keys bit for bit,
    other floats norm-wise relative (row by row for keys ending in _rows)."""
    gold = load_record(os.path.join(GOLD, case + ".npz"))
    assert sorted(rec) == sorted(gold), f"{case}: recorded keys differ from the reference's"
    for k in sorted(gold):
        r, g = np.asarray(rec[k]), gold[k]
        assert r.shape == g.shape, f"{case}: {k} shape {r.shape}, reference {g.shape}"
        if g.dtype.kind in "iub" or k.endswith(EXACT):
            assert np.array_equal(r, g), f"{case}: {k} differs from the reference"
        elif k.endswith("_rows"):
            for i, (a, b) in enumerate(zip(r, g)):
                assert relerr(a, b) <= tol, f"{case}: {k} row {i} rel err {relerr(a, b):.2e} vs the reference"
        else:
            assert relerr(r, g) <= tol, f"{case}: {k} rel err {relerr(r, g):.2e} vs the reference"


def run_sequence(pkg, make, n_features, hard, seed):
    sc = pkg.synth.Scene(n_features=n_features, n_frames=7, seed=seed, hard=hard)
    f = make(_cfg(pkg, sc))
    rec = {}
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    assert sum(f.addFeature(*p) for p in sc.feature_pixels) == n_features
    _state(rec, "init", f)
    for t in range(1, sc.n_frames):
        f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict()
        rec[f"t{t}_dt"] = f.getDt()
        _state(rec, f"t{t}_pred", f)
        rec[f"t{t}_Sblocks"] = f.S_blocks()
        rec[f"t{t}_innov"] = np.array([f.feature(i).is_in_innovation for i in range(f.numOfFeatures())], dtype=np.int32)
        inn = [f.feature(i) for i in range(f.numOfFeatures()) if f.feature(i).is_in_innovation]
        rec[f"t{t}_h_rows"] = np.array([list(a.h) for a in inn]).reshape(-1, 2)
        rec[f"t{t}_H_rows"] = np.array([[np.dot(list(a.H), H_PROBE)] for a in inn]).reshape(-1, 1)
        f.update(sc.picks(t, n_features))
        rec[f"t{t}_hypotheses"] = _hypotheses(f)
        _tables(rec, f"t{t}", f)
        _state(rec, f"t{t}", f)
    if hard:
        assert any(not f.feature(i).is_in_li for i in range(f.numOfFeatures())) or f.numOfFeatures() < n_features
    return rec, f


def run_controls_remove_and_accessors(pkg, make):
    sc = pkg.synth.Scene(n_features=14, n_frames=4, seed=17)
    f = make(_cfg(pkg, sc))
    rec = {}
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        f.addFeature(*p)
    assert f.addFeature(2.0, 3.0) == 0           # outside the gate (vslamRansac.cpp:314)
    f.removeFeature(3); f.removeFeature(0); f.removeFeature(f.numOfFeatures() - 1)
    # Patch::position_in_z is not initialised by the reference's constructor (Patch.cpp:78-103): it is
    # garbage until the first predict assigns it (vslamRansac.cpp:589)
    _tables(rec, "removed", f, skip=("position_in_z",)); _state(rec, "removed", f)
    f.captureNewFrame(sc.frame(1), sc.stamps[1])
    f.predict(dv=(0.01, -0.02, 0.005), dw=(0.002, 0.001, -0.003), vcontrol=True)
    _state(rec, "predict_controls", f)
    f.update(sc.picks(1, 14))
    _tables(rec, "update", f); _state(rec, "update", f)
    rec["state14"] = f.getState(); rec["sigma14"] = f.getSigma()
    rec["covariance_parameter"] = f.Covariance_Parameter()
    return rec, f


def run_xyz_conversion(pkg, make):
    sc = pkg.synth.Scene(n_features=10, n_frames=4, seed=23)
    f = make(_cfg(pkg, sc))
    rec = {}
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        f.addFeature(*p)
    mu, S = f.get_full()
    for i in (1, 4, 9):
        pos = 14 + 6 * i
        S[pos + 5, :] *= 1e-3; S[:, pos + 5] *= 1e-3
    f.set_full(mu, S)
    f.convert2XYZ_ifLinearAll()
    assert f.state_dim() == 14 + 6 * 10 - 3 * 3
    assert [f.feature(i).coding for i in range(10)] == [0, 1, 0, 0, 1, 0, 0, 0, 0, 1]
    _tables(rec, "converted", f, skip=("position_in_z",)); _state(rec, "converted", f)
    for t in (1, 2):
        f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, 10))
        _tables(rec, f"t{t}", f); _state(rec, f"t{t}", f)
    return rec, f


def find_match_inputs(pkg):
    d = pkg.synth.match_batch_inputs(n_frames=1, features_per_frame=24, width=320, height=240, window=11, seed=5, s_diag=20.0)
    h = d["h"].copy(); S = d["S"].copy(); tm = d["templates"].copy()
    h[0] = (3.2, 4.9); h[1] = (317.5, 238.5); tm[2] = 128; S[3] = (400.0, 390.0, 390.0, 400.0)
    return d["frames"], tm, h, S


def run_motion_blur_templates(pkg, make):
    sc = pkg.synth.Scene(n_features=16, n_frames=6, seed=29, speed=0.9, omega=0.5, template_smooth=2.5)
    f = make(_cfg(pkg, sc, kernel_size=3, T_camera=0.5))
    rec = {}
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        f.addFeature(*p)
    blurred = 0
    for t in range(1, sc.n_frames):
        f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict()
        inn = [i for i in range(f.numOfFeatures()) if f.feature(i).is_in_innovation]
        patches = [f.template(i, 1) for i in inn]           # matching_patch after Patch::blur
        rec[f"t{t}_blurred_features"] = np.array(inn, dtype=np.int32)
        rec[f"t{t}_blurred_tmpl"] = _digest(patches)
        blurred += sum(int(not np.array_equal(b, f.template(i, 0))) for i, b in zip(inn, patches))
        f.update(sc.picks(t, 16))
        _tables(rec, f"t{t}", f); _state(rec, f"t{t}", f)
    assert blurred >= 10, f"only {blurred} templates were blurred: the scene does not exercise the path"
    return rec, f


def run_forse_plane(pkg, make):
    sc = pkg.synth.Scene(n_features=14, n_frames=5, seed=61, hard=True)
    f = make(_cfg(pkg, sc, forsePlane=1))
    rec = {}
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        f.addFeature(*p)
    for t in range(1, sc.n_frames):
        f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, 14))
        _tables(rec, f"t{t}", f); _state(rec, f"t{t}", f)
    return rec, f


def rts_inputs(seed, zero_w):
    rng = np.random.default_rng(seed)
    def state():
        mu = np.zeros(13)
        mu[:3] = rng.normal(0, 0.5, 3)
        q = rng.normal(0, 1, 4); mu[3:7] = q / np.linalg.norm(q)
        mu[7:10] = rng.normal(0, 0.2, 3); mu[10:13] = rng.normal(0, 0.1, 3)
        A = rng.normal(0, 1, (13, 13))
        return mu, A @ A.T * 1e-3 + np.eye(13) * 1e-4
    (mu, sg), (mus, sgs), dts, drs = state(), state(), rng.normal(0, 0.01, 3), rng.normal(0, 0.01, 3)
    if zero_w:
        mu[10:13] = 0; drs[:] = 0   # |w| = 0 branch of Jacobian_qt_w (Sinc = 1, n_w = 0)
    return mu, sg, mus, sgs, dts, drs


def run_rts_epoch(pkg, make, seed, zero_w):
    f = make(pkg.default_config())
    mu, sg, mus, sgs, dts, drs = rts_inputs(seed, zero_w)
    m, S = f.rts_epoch(mu, sg, mus, sgs, dts, drs, 1 / 30)
    assert relerr(m, mu) > 1e-6   # the epoch did something
    return {"mu": m, "sigma": S}, f


def run_deleted_archive(pkg, make):
    sc = pkg.synth.Scene(n_features=10, n_frames=9, seed=77)
    f = make(_cfg(pkg, sc))
    rec = {}
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        f.addFeature(*p)
    for t in range(1, 9):
        f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, 10))
    mu, S = f.get_full()     # shrink rho's variance until the linearity index passes (as run_xyz_conversion)
    for i in (1, 4, 9):
        pos = 14 + 6 * i
        S[pos + 5, :] *= 1e-4; S[:, pos + 5] *= 1e-4
    f.set_full(mu, S)
    f.convert2XYZ_ifLinearAll()
    xyz = [i for i in range(f.numOfFeatures()) if f.feature(i).coding]
    assert len(xyz) >= 2
    rec["xyz"] = np.array(xyz, dtype=np.int32)
    # RosVSLAM::getPointsFeatures, from the reference's own RosVSLAMRansac.cpp (oracle/_ref), before and after removals
    P = f.getPointsFeatures()
    assert np.count_nonzero(np.abs(P).sum(axis=1)) == len(xyz)
    rec["points"] = P
    # feature 0 is inverse-depth: removed, not archived.  The LAST feature stays: once it is gone the reference's
    # getPointsFeatures writes the archived rows with a larger real_index past its matrix (RosVSLAMRansac.cpp:349 sizes
    # it by the last live patch) — undefined behaviour that the oracle and the CUDA path replace by dropping those rows.
    victims = [i for i in xyz if i != f.numOfFeatures() - 1][:3]
    for i in sorted(victims + [0], reverse=True):
        f.removeFeature(i)
    deleted = f.deleted()
    assert len(deleted) == len(victims) >= 2
    for k, (ri, xyz_pos, cov) in enumerate(deleted):
        rec[f"deleted{k}_index"] = np.int32(ri); rec[f"deleted{k}_xyz"] = xyz_pos; rec[f"deleted{k}_cov"] = cov
    P = f.getPointsFeatures()
    assert np.count_nonzero(np.abs(P).sum(axis=1)) == len(xyz)
    rec["points_archived"] = P
    return rec, f


def _oracle(orc, kind):
    return lambda cfg: orc.OracleFilter(cfg, kind=kind)


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
@pytest.mark.parametrize("n_features,hard,seed", SEQUENCES)
def test_sequence(pkg, orc, fp64, kind, tol, n_features, hard, seed):
    rec, _ = run_sequence(pkg, _oracle(orc, kind), n_features, hard, seed)
    compare(rec, case_id("sequence", fp64, n_features, hard, seed), tol)


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
def test_controls_remove_and_accessors(pkg, orc, fp64, kind, tol):
    rec, _ = run_controls_remove_and_accessors(pkg, _oracle(orc, kind))
    compare(rec, case_id("controls", fp64), tol)


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
def test_xyz_conversion(pkg, orc, fp64, kind, tol):
    """convert2XYZ_ifLinear (vslamRansac.cpp:741-780): shrink rho's variance until the linearity index
    passes, convert, then run a step with mixed inverse-depth / XYZ features."""
    rec, _ = run_xyz_conversion(pkg, _oracle(orc, kind))
    compare(rec, case_id("xyz", fp64), tol)


def test_find_match_standalone(pkg, orc):
    """Patch::findMatch of the reference (fp32, as written) vs the oracle's batched matcher."""
    frames, tm, h, S = find_match_inputs(pkg)
    uv, _ = orc.match_batch(frames, tm, h, S, sigma_size=3.0, kind_mf=0)
    compare({"uv": uv}, case_id("find_match", False), 0.0)


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
def test_motion_blur_templates(pkg, orc, fp64, kind, tol):
    """Patch::blur / blurPatch / evaluateKernel (Patch.cpp:50-57, libblur.cpp:17-81) with the reference's own
    libblur.cpp compiled in: kernel_size = 3 as conf_sim.cfg, T_camera = 0.5, a fast camera so that the
    predicted displacement over the exposure exceeds the threshold for most features."""
    rec, o = run_motion_blur_templates(pkg, _oracle(orc, kind))
    compare(rec, case_id("blur", fp64), tol)
    assert o.stats().blur_requests > 0


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
def test_forse_plane(pkg, orc, fp64, kind, tol):
    """forsePlane pseudo-measurement (vslamRansac.cpp:1245-1263, 1272)."""
    rec, _ = run_forse_plane(pkg, _oracle(orc, kind))
    compare(rec, case_id("forse_plane", fp64), tol)


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
@pytest.mark.parametrize("seed,zero_w", RTS_CASES)
def test_rts_epoch(pkg, orc, fp64, kind, tol, seed, zero_w):
    """VSlamFilter::rts_epoch (vslamRansac.cpp:423-449) on 13-dimensional camera states."""
    rec, _ = run_rts_epoch(pkg, _oracle(orc, kind), seed, zero_w)
    compare(rec, case_id("rts", fp64, seed, zero_w), tol)


@pytest.mark.parametrize("fp64,kind,tol", VARIANTS)
def test_deleted_archive(pkg, orc, fp64, kind, tol):
    """removeFeature archives XYZ features seen more than five times (vslamRansac.cpp:394-404)."""
    rec, o = run_deleted_archive(pkg, _oracle(orc, kind))
    compare(rec, case_id("deleted", fp64), tol)
    # oracle only: removing the last (XYZ, archived) feature drops its row instead of overflowing
    last = o.numOfFeatures() - 1
    if o.feature(last).coding:
        o.removeFeature(last)
        P2 = o.getPointsFeatures()
        assert P2.shape[0] == o.feature(o.numOfFeatures() - 1).real_index + 1 and np.isfinite(P2).all()
