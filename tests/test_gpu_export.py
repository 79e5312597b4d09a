"""-m gpu: the caller-side rows of SURVEY.md section 8(f) item 4 on the CUDA path against the oracle:
the feature archive and RosVSLAM::getPointsFeatures (RosVSLAMRansac.cpp:340-418), VSlamFilter::rts_epoch
(vslamRansac.cpp:423-449), and the key-frame recorder driven by the GPU filter and by the oracle."""
import numpy as np
import pytest

from helpers import TOL, assert_scaled_close, assert_state_close, assert_tables_equal, make_pair, relerr, seed_features

pytestmark = pytest.mark.gpu


def _converted_pair(gpu_pkg, orc, n=12, frames=9, seed=31):
    sc = gpu_pkg.synth.Scene(n_features=n, n_frames=frames, seed=seed)
    g, o = make_pair(gpu_pkg, orc, sc, xyz_conversion=1)
    seed_features(g, sc); seed_features(o, sc)
    for t in range(1, frames):
        for f in (g, o):
            f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, n))
    for f in (g, o):   # shrink rho's variance until the linearity index passes, then convert
        mu, S = f.get_full()
        for i in (1, 4, 7, 9):
            pos = f.feature(i).position_in_state
            S[pos + 5, :] *= 1e-4; S[:, pos + 5] *= 1e-4
        f.set_full(mu, S)
        f.convert2XYZ_ifLinearAll()
    return sc, g, o


def test_points_features_and_archive(gpu_pkg, orc):
    sc, g, o = _converted_pair(gpu_pkg, orc)
    assert_tables_equal(g, o, ctx="after conversion")
    xyz = [i for i in range(g.numOfFeatures()) if g.feature(i).coding]
    assert len(xyz) >= 3
    Pg, Po = g.getPointsFeatures(), o.getPointsFeatures()
    assert Pg.shape == Po.shape == (g.feature(g.numOfFeatures() - 1).real_index + 1, 12)
    assert relerr(Pg, Po) <= TOL
    assert np.count_nonzero(np.abs(Pg).sum(axis=1)) == len(xyz)          # inverse-depth rows stay zero
    # remove two XYZ features (seen more than five times -> archived) and an inverse-depth one (not archived)
    inv = [i for i in range(g.numOfFeatures()) if not g.feature(i).coding][0]
    for i in sorted(xyz[:2] + [inv], reverse=True):
        g.removeFeature(i); o.removeFeature(i)
    dg, do = g.deleted(), o.deleted()
    assert len(dg) == len(do) == 2
    for (ia, xa, ca), (ib, xb, cb) in zip(dg, do):
        assert ia == ib and relerr(xa, xb) <= TOL and relerr(ca, cb) <= TOL
    Pg, Po = g.getPointsFeatures(), o.getPointsFeatures()
    assert Pg.shape == Po.shape and relerr(Pg, Po) <= TOL
    assert np.count_nonzero(np.abs(Pg).sum(axis=1)) == len(xyz)          # archived rows are filled from the archive
    assert_state_close(g, o, ctx="after removal")
    # remove features from the END of the map until an archived XYZ one has gone: the reference would write its row past
    # the matrix (sized by the last live patch); oracle and CUDA path drop it
    while g.numOfFeatures() > 2:
        last = g.numOfFeatures() - 1
        was_xyz = bool(g.feature(last).coding)
        g.removeFeature(last); o.removeFeature(last)
        if was_xyz:
            break
    Pg, Po = g.getPointsFeatures(), o.getPointsFeatures()
    assert Pg.shape == Po.shape == (g.feature(g.numOfFeatures() - 1).real_index + 1, 12) and relerr(Pg, Po) <= TOL
    assert len(g.deleted()) == len(o.deleted()) == 3


@pytest.mark.parametrize("seed,zero_w", [(1, False), (2, False), (3, True)])
def test_rts_epoch(gpu_pkg, orc, seed, zero_w):
    rng = np.random.default_rng(seed)

    def state():
        mu = np.zeros(13)
        mu[:3] = rng.normal(0, 0.5, 3)
        q = rng.normal(0, 1, 4); mu[3:7] = q / np.linalg.norm(q)
        mu[7:10] = rng.normal(0, 0.2, 3); mu[10:13] = rng.normal(0, 0.1, 3)
        A = rng.normal(0, 1, (13, 13))
        return mu, A @ A.T * 1e-3 + np.eye(13) * 1e-4

    (mu, sg), (mus, sgs) = state(), state()
    dts, drs = rng.normal(0, 0.01, 3), rng.normal(0, 0.01, 3)
    if zero_w:
        mu[10:13] = 0; drs[:] = 0
    cfg = gpu_pkg.default_config()
    g, o = gpu_pkg.VSlamFilter(cfg, feature_capacity=8), orc.OracleFilter(cfg, kind=0)
    mg, Sg = g.rts_epoch(mu, sg, mus, sgs, dts, drs, 1 / 30)
    mo, So = o.rts_epoch(mu, sg, mus, sgs, dts, drs, 1 / 30)
    assert relerr(mg, mo) <= TOL and relerr(Sg, So) <= TOL, f"mu {relerr(mg, mo):.2e} Sigma {relerr(Sg, So):.2e}"
    assert_scaled_close(mg, Sg, mo, So, "rts_epoch")
    assert relerr(mg, mu) > 1e-6
    with pytest.raises(Exception):
        g.rts_epoch(mu, sg, mus, sgs, dts, drs, 0.0)


def test_keyframe_recorder_on_gpu_filter_matches_oracle(gpu_pkg, orc, tmp_path):
    """The recorder reads only accessors; driven by the CUDA filter and by the oracle over the same sequence it must
    pick the same key frames and write files that agree to the printed precision."""
    kf = gpu_pkg.keyframes
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=24, seed=13)
    g, o = make_pair(gpu_pkg, orc, sc, xyz_conversion=1)
    seed_features(g, sc); seed_features(o, sc)
    recs = []
    for name, f in (("gpu", g), ("cpu", o)):
        d = tmp_path / name
        rec = kf.KeyframeRecorder(str(d))
        rec.MoveThresh = 0.6          # the synthetic camera moves centimetres per frame; the reference's 18 suits a robot
        recs.append((rec, d, f))
    for t in range(1, 24):
        for rec, d, f in recs:
            f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, 20))
            rec.on_frame(f, t, sc.frame(t))
    for rec, d, f in recs:
        rec.finish(f)
    (rg, dg, _), (ro, do_, _) = recs
    assert rg.key_frames == ro.key_frames and len(rg.key_frames) >= 2
    Pg, Cg, Ng = kf.read_sba_inputs(str(dg))
    Po, Co, No = kf.read_sba_inputs(str(do_))
    assert Pg.shape == Po.shape and Cg.shape == Co.shape and len(Ng) == len(No)
    assert np.allclose(Pg, Po, rtol=1e-5, atol=1e-12) and np.allclose(Cg, Co, rtol=1e-5, atol=1e-15)
    for (ca, pa, ja), (cb, pb, jb) in zip(Ng, No):
        assert ca == cb and ja == jb and np.allclose(pa, pb, rtol=1e-5, atol=1e-9)


def test_points_features_empty_and_inverse_depth_only(gpu_pkg, orc):
    """No feature: one zero row (psize = 0, RosVSLAMRansac.cpp:349 guarded); inverse-depth features only: all rows zero."""
    sc = gpu_pkg.synth.Scene(n_features=6, n_frames=2, seed=3)
    g, o = make_pair(gpu_pkg, orc, sc)
    for f in (g, o):
        f.captureNewFrame(sc.frame(0), sc.stamps[0])
    Pg, Po = g.getPointsFeatures(), o.getPointsFeatures()
    assert Pg.shape == Po.shape == (1, 12) and not Pg.any() and not Po.any()
    assert g.deleted() == [] and o.deleted() == []
    for f in (g, o):
        for p in sc.feature_pixels:
            f.addFeature(*p)
    Pg, Po = g.getPointsFeatures(), o.getPointsFeatures()
    assert Pg.shape == Po.shape == (g.feature(5).real_index + 1, 12) and not Pg.any() and not Po.any()
    assert g.L.ekf_get_points_features(g.h, None, 0, None) < 0      # rows pointer is mandatory


def test_cuda_path_reproduces_reference_export_fixture(gpu_pkg):
    """rts_epoch, getPointsFeatures and the feature archive against vectors produced by the reference's own sources
    (tests/golden/export_rts_points.npz, oracle/gen_golden_export.py)."""
    import gen_golden_export as gg
    from test_golden_export import GOLD, compare_export
    gold = np.load(GOLD)
    rec = gg.run_export_case(gpu_pkg, lambda over: gpu_pkg.VSlamFilter(gpu_pkg.default_config(**over), feature_capacity=16))
    worst = compare_export(rec, gold, 1e-8, "CUDA path")   # eight free-running frames precede the export (helpers.py: 1e-8 over sequences)
    print(f"CUDA path vs reference export fixture: worst rel err {worst:.2e}")
