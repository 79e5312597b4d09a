"""-m gpu: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): integer match coordinates and accept/reject decisions
bit-exact; state and covariance within 1e-9 relative (Frobenius / 2-norm, per step from identical
inputs).
"""
import numpy as np
import pytest

from helpers import TOL, assert_state_close, assert_tables_equal, make_pair, relerr, seed_features

pytestmark = pytest.mark.gpu


def _scene(pkg, **kw):
    return pkg.synth.Scene(**kw)


def test_init_and_add_feature(gpu_pkg, orc):
    sc = _scene(gpu_pkg, n_features=20, n_frames=2, seed=11)
    g, o = make_pair(gpu_pkg, orc, sc)
    assert relerr(g.getState(), o.getState()) == 0.0
    assert relerr(g.getSigma(), o.getSigma()) == 0.0
    rg, ro = seed_features(g, sc), seed_features(o, sc)
    assert rg == ro and sum(rg) == 20
    # a point outside the gate is rejected by both (vslamRansac.cpp:314)
    assert g.addFeature(2.0, 3.0) == 0 and o.addFeature(2.0, 3.0) == 0
    assert g.state_dim() == o.state_dim() == 14 + 6 * 20
    assert_state_close(g, o, ctx="after addFeature")
    assert_tables_equal(g, o, ctx="after addFeature")
    for i in range(20):
        assert np.array_equal(g.template(i), o.template(i))
        assert np.array_equal(g.returnCentrPatchIndx(i), np.array(o.feature(i).center))


@pytest.mark.parametrize("n_features,hard", [(12, False), (50, False), (70, True)])
def test_step_by_step_parity(gpu_pkg, orc, n_features, hard):
    """predict / match / update, each stage compared, GPU state re-seeded from the oracle each frame."""
    sc = _scene(gpu_pkg, n_features=n_features, n_frames=7, seed=100 + n_features, hard=hard)
    g, o = make_pair(gpu_pkg, orc, sc)
    seed_features(g, sc); seed_features(o, sc)
    worst = [0.0, 0.0]
    for t in range(1, sc.n_frames):
        mu, S = o.get_full()
        g.set_full(mu, S)  # identical inputs
        img = sc.frame(t)
        g.captureNewFrame(img, sc.stamps[t]); o.captureNewFrame(img, sc.stamps[t])
        assert g.getDt() == o.getDt()
        g.predict(); o.predict()
        assert_state_close(g, o, ctx=f"frame {t} predict")
        assert_tables_equal(g, o, fields=("is_in_innovation", "position_in_z", "remove_flag"), ctx=f"frame {t} predict")
        Sg, So = g.S_blocks(), o.S_blocks()
        assert relerr(Sg, So) <= TOL
        for i in range(g.numOfFeatures()):
            a, b = g.feature(i), o.feature(i)
            if b.is_in_innovation:
                assert relerr(list(a.h), list(b.h)) <= TOL
                assert relerr(list(a.H), list(b.H)) <= TOL, f"H of feature {i}"
        ng = g.match(); no = o.match()
        assert ng == no
        for i in range(g.numOfFeatures()):
            a, b = g.feature(i), o.feature(i)
            assert a.is_in_innovation == b.is_in_innovation and a.n_tot == b.n_tot
            assert tuple(a.center) == tuple(b.center), f"frame {t} feature {i} match {tuple(a.center)} vs {tuple(b.center)}"
            assert tuple(a.z) == tuple(b.z)
            assert a.last_ncc == b.last_ncc, "NCC score must be bit-identical"
            if b.is_in_innovation:
                assert np.array_equal(g.template(i, 1), o.template(i, 1))
        picks = sc.picks(t, n_features)
        g.update_after_match(picks); o.update_after_match(picks)
        sg, so = g.stats(), o.stats()
        for f in ("n_matched", "n_li", "n_hi", "ransac_hypotheses", "n_removed", "topup_request"):
            assert getattr(sg, f) == getattr(so, f), f"frame {t} stat {f}: {getattr(sg, f)} vs {getattr(so, f)}"
        assert_tables_equal(g, o, ctx=f"frame {t} update")
        em, es = assert_state_close(g, o, ctx=f"frame {t} update")
        worst = [max(worst[0], em), max(worst[1], es)]
    print(f"N={n_features} hard={hard}: worst per-step rel err mu {worst[0]:.2e} Sigma {worst[1]:.2e}; "
          f"oracle min decision margin {o.min_margin():.3g}")


def test_free_running_trajectory(gpu_pkg, orc):
    """No re-seeding: both filters run 12 frames on their own state; drift must stay inside tolerance."""
    sc = _scene(gpu_pkg, n_features=40, n_frames=13, seed=77)
    g, o = make_pair(gpu_pkg, orc, sc)
    seed_features(g, sc); seed_features(o, sc)
    for t in range(1, sc.n_frames):
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t])
            f.predict()
            f.update(sc.picks(t, 40))
        assert_tables_equal(g, o, ctx=f"frame {t}")
        assert_state_close(g, o, tol=1e-8, ctx=f"frame {t} free-running", free_running=True)
    assert abs(g.Covariance_Parameter() - o.Covariance_Parameter()) <= 1e-9 * abs(o.Covariance_Parameter())


@pytest.mark.parametrize("symmetric", [False, True])
def test_multi_block_update(gpu_pkg, orc, symmetric):
    """More than 64 matched features: the stacked update spans several 128-row blocks.  Both
    downdate modes (full square / lower triangle + mirror) must stay inside the tolerance."""
    sc = _scene(gpu_pkg, n_features=150, n_frames=3, seed=5)
    g, o = make_pair(gpu_pkg, orc, sc)
    g.set_symmetric_downdate(symmetric)
    seed_features(g, sc); seed_features(o, sc)
    for t in range(1, 3):
        mu, S = o.get_full(); g.set_full(mu, S)
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t]); f.predict(); f.update(sc.picks(t, 150))
        assert g.stats().n_li == o.stats().n_li and g.stats().n_li > 64
        assert_tables_equal(g, o, ctx=f"frame {t}")
        assert_state_close(g, o, ctx=f"frame {t} multi-block")


@pytest.mark.parametrize("env,n_features,sched", [("EKF_LOOKAHEAD_MIN_N", 150, 1), ("EKF_PIPE_MIN_N", 150, 0), ("EKF_PIPE_MIN_N", 210, 0),
                                                  ("EKF_PIPE_MIN_N", 150, 1), ("EKF_PIPE_MIN_N", 210, 1), ("EKF_PIPE_MIN_N", 290, 1),
                                                  ("EKF_PIPE_MIN_N", 290, 2), ("EKF_PIPE_MIN_N", 150, 3), ("EKF_PIPE_MIN_N", 290, 3),
                                                  ("EKF_PIPE_MIN_N", 290, 4), ("EKF_PIPE_MIN_N", 290, 5)])
def test_lookahead_pipeline_parity(gpu_pkg, orc, monkeypatch, env, n_features, sched):
    """The pipelined stacked updates forced on at n = 914 (three update blocks), 1274 (four) and 1754 (five, the last one
    partial): the look-ahead schedule (second stream, W correction GEMM; default for n >= 6000) and the two schedules for
    1000 <= n < 6000 — factor-beside-downdate (EKF_SCHED=0: S_b from the raw gather minus G G^T, correction on a third stream)
    and chain-short (EKF_SCHED=1, default: G_b by a 128-row solve on rows of W_{b-1}, the n-row solve V_b off the chain on a
    fourth stream, delta ping-pong).  Same tolerance as the plain path."""
    monkeypatch.setenv("EKF_LOOKAHEAD_MIN_N", "1000000")
    monkeypatch.setenv(env, "1")
    # 3: resident-chain schedule (k_chain_factor); 5: chain-short with the pre-positioned factor kernel (k_blk_factor_wait)
    monkeypatch.setenv("EKF_SCHED", "2" if sched == 3 else "3" if sched == 5 else str(min(sched, 1)))
    if sched == 4:   # chain-short with the S look-ahead (hot rows of W'' gathered a block earlier, second correction term -G2 G2^T)
        monkeypatch.setenv("EKF_S_LOOKAHEAD", "1")
    if sched == 2:   # chain-short with the downdate walking the hot-first tile list and the next gather gated on its hot tiles
        monkeypatch.setenv("EKF_SPLIT_DD", "1")
    sc = _scene(gpu_pkg, n_features=n_features, n_frames=4, seed=6)
    g, o = make_pair(gpu_pkg, orc, sc)
    if sched == 2:
        g.set_symmetric_downdate(1)   # the tile list enumerates the lower triangle
    seed_features(g, sc); seed_features(o, sc)
    for t in range(1, 4):
        mu, S = o.get_full(); g.set_full(mu, S)
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t]); f.predict(); f.update(sc.picks(t, n_features))
        assert g.stats().n_li == o.stats().n_li and g.stats().n_li > 128
        assert_tables_equal(g, o, ctx=f"frame {t}")
        assert_state_close(g, o, ctx=f"frame {t} {env}")


def test_remove_feature_and_controls(gpu_pkg, orc):
    sc = _scene(gpu_pkg, n_features=16, n_frames=3, seed=9)
    g, o = make_pair(gpu_pkg, orc, sc)
    seed_features(g, sc); seed_features(o, sc)
    for f in (g, o):
        f.removeFeature(3); f.removeFeature(0); f.removeFeature(f.numOfFeatures() - 1)
    assert_tables_equal(g, o, ctx="after remove"); assert_state_close(g, o, ctx="after remove")
    img = sc.frame(1)
    for f in (g, o):
        f.captureNewFrame(img, sc.stamps[1])
        f.predict(dv=(0.01, -0.02, 0.005), dw=(0.002, 0.001, -0.003), vcontrol=True)
    assert_state_close(g, o, ctx="predict with controls")
    for f in (g, o):
        f.update(sc.picks(1, 16))
    assert_tables_equal(g, o, ctx="update after remove"); assert_state_close(g, o, ctx="update after remove")


def test_xyz_conversion_and_mixed_update(gpu_pkg, orc):
    """convert2XYZ_ifLinear(All) (vslamRansac.cpp:741-780) and steps with mixed inverse-depth / XYZ
    features (XYZ measurement branch :552-578, RANSAC quirk :1016, removal archive :394-404)."""
    sc = _scene(gpu_pkg, n_features=20, n_frames=6, seed=23)
    g, o = make_pair(gpu_pkg, orc, sc, xyz_conversion=1)
    seed_features(g, sc); seed_features(o, sc)
    mu, S = o.get_full()
    for i in (1, 4, 9, 10, 19):
        pos = 14 + 6 * i
        S[pos + 5, :] *= 1e-3; S[:, pos + 5] *= 1e-3
    for f in (g, o):
        f.set_full(mu, S)
    g.convert2XYZ_ifLinear(4); o.convert2XYZ_ifLinear(4)          # one feature
    g.convert2XYZ_ifLinear(0); o.convert2XYZ_ifLinear(0)          # not linear enough: no-op
    assert g.state_dim() == o.state_dim() == 14 + 6 * 20 - 3
    assert_tables_equal(g, o, ctx="single conversion"); assert_state_close(g, o, ctx="single conversion")
    g.convert2XYZ_ifLinearAll(); o.convert2XYZ_ifLinearAll()      # the remaining four at once
    assert g.state_dim() == o.state_dim() == 14 + 6 * 20 - 3 * 5
    assert [g.feature(i).coding for i in range(20)] == [o.feature(i).coding for i in range(20)]
    assert_tables_equal(g, o, ctx="convert all"); assert_state_close(g, o, ctx="convert all")
    for t in range(1, sc.n_frames):
        m, Sg = o.get_full(); g.set_full(m, Sg)
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t]); f.predict(); f.update(sc.picks(t, 20))
        assert_tables_equal(g, o, ctx=f"mixed frame {t}"); assert_state_close(g, o, ctx=f"mixed frame {t}")
    g.removeFeature(4); o.removeFeature(4)                        # an XYZ feature
    assert_tables_equal(g, o, ctx="remove xyz"); assert_state_close(g, o, ctx="remove xyz")


def test_motion_blur_templates(gpu_pkg, orc):
    """Patch::blur (Patch.cpp:50-57) + blurPatch / evaluateKernel (libblur.cpp:17-81), kernel_size = 3 and
    T_camera = 0.5 as conf_sim.cfg, fast camera: blurred templates, matches and the step bit-exact / 1e-9."""
    sc = _scene(gpu_pkg, n_features=24, n_frames=6, seed=29, speed=0.9, omega=0.5, template_smooth=2.5)
    g, o = make_pair(gpu_pkg, orc, sc, kernel_size=3, T_camera=0.5)
    seed_features(g, sc); seed_features(o, sc)
    blurred = 0
    for t in range(1, sc.n_frames):
        mu, S = o.get_full(); g.set_full(mu, S)
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t]); f.predict()
        for i in range(g.numOfFeatures()):
            if o.feature(i).is_in_innovation:
                a, b = g.template(i, 1), o.template(i, 1)
                assert np.array_equal(a, b), f"frame {t} feature {i}: blurred template differs in {(a != b).sum()} pixels"
                blurred += int(not np.array_equal(b, o.template(i, 0)))
        picks = sc.picks(t, 24)
        g.update(picks); o.update(picks)
        assert g.stats().n_matched == o.stats().n_matched
        assert_tables_equal(g, o, ctx=f"blur frame {t}")
        for i in range(g.numOfFeatures()):
            assert g.feature(i).last_ncc == o.feature(i).last_ncc
        assert_state_close(g, o, ctx=f"blur frame {t}")
    assert blurred >= 10 and g.stats().blur_requests > 0


@pytest.mark.parametrize("hard", [False, True])
def test_forse_plane_pseudo_measurement(gpu_pkg, orc, hard):
    """forsePlane (vslamRansac.cpp:1245-1263): mu[1] = mu[4] = mu[6] = 0 with R = 1e-5 I appended to the second
    update — with and without high-innovation rows beside it."""
    sc = _scene(gpu_pkg, n_features=30, n_frames=5, seed=61, hard=hard)
    g, o = make_pair(gpu_pkg, orc, sc, forsePlane=1)
    seed_features(g, sc); seed_features(o, sc)
    for t in range(1, sc.n_frames):
        mu, S = o.get_full(); g.set_full(mu, S)
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t]); f.predict(); f.update(sc.picks(t, 30))
        assert (g.stats().n_li, g.stats().n_hi) == (o.stats().n_li, o.stats().n_hi)
        assert_tables_equal(g, o, ctx=f"plane frame {t}")
        assert_state_close(g, o, ctx=f"plane frame {t}")
    mu, _ = g.get_full()
    assert abs(mu[1]) < 1e-2 and abs(mu[4]) < 1e-2     # the pseudo-measurement holds y and q_x near zero


def test_unsupported_configs_fail_loudly(gpu_pkg):
    for over in (dict(window_size=33), dict(search_clamp=25.0), dict(scale=0)):
        cfg = gpu_pkg.default_config(xyz_conversion=0, **over)
        with pytest.raises(gpu_pkg.EkfError):
            gpu_pkg.VSlamFilter(cfg)
