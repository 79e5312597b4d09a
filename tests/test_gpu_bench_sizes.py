"""-m gpu: parity at the sizes bench.py reports (VERDICT r1 item 1).

* cfg2 (N = 500, n = 3014, 8 update blocks): the DEFAULT path of the library — no environment overrides, i.e. the
  factor-beside-downdate schedule, cluster RANSAC — in both downdate modes, two frames from identical inputs against the
  CPU oracle (dense reference algebra, OpenMP): decisions and tables bit-exact, state / covariance <= 1e-9 relative.
* cfg4 (N = 2000, n = 12014, 32 update blocks, look-ahead pipeline): one dense oracle frame is ~3e13 flops, so the
  covariance correction is compared with an independent fp64 numpy / LAPACK evaluation of
  Sigma - Sigma H^T (H Sigma H^T + R)^-1 H Sigma built from the same H rows (tests/helpers.py), <= 1e-9 relative.
* the cluster RANSAC with more than 8 * 512 candidates (ADVICE r1: the erase used to stop after 4096 entries).
"""
import numpy as np
import pytest

import bench
from helpers import TOL, assert_scaled_close, assert_state_close, assert_tables_equal, numpy_stacked_update, relerr

pytestmark = pytest.mark.gpu


def _seed(filt, scene):
    filt.captureNewFrame(scene.frame(0), scene.stamps[0])
    return sum(filt.addFeature(*p) for p in scene.feature_pixels)


@pytest.mark.parametrize("symmetric", [True, False])
def test_cfg2_n500_default_path(gpu_pkg, orc, symmetric, monkeypatch):
    for v in ("EKF_LOOKAHEAD_MIN_N", "EKF_PIPE_MIN_N", "EKF_RANSAC_CLUSTER", "EKF_GEMM_TM", "EKF_BLOCK_ROWS"):
        monkeypatch.delenv(v, raising=False)
    nfeat = bench.WORKLOADS["cfg2_n500"][0]
    sc = bench.make_scene(gpu_pkg, "cfg2_n500", 3)
    cfg = bench.bench_config(gpu_pkg, sc)
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=nfeat + 4)
    g.set_symmetric_downdate(symmetric)
    assert _seed(g, sc) == nfeat
    o = orc.OracleFilter(cfg, kind=0, omp=True)
    orc.lib(omp=True).orc_set_num_threads(__import__("os").cpu_count() or 1)
    o.captureNewFrame(sc.frame(0), sc.stamps[0])
    o.import_from(g)
    assert g.state_dim() == o.state_dim() == 14 + 6 * nfeat
    worst = [0.0, 0.0]
    for t in (1, 2):
        mu, S = o.get_full(); g.set_full(mu, S)          # identical inputs
        img = sc.frame(t)
        for f in (g, o):
            f.captureNewFrame(img, sc.stamps[t]); f.predict(); f.update(sc.picks(t, nfeat))
        sg, so = g.stats(), o.stats()
        for k in ("n_matched", "n_li", "n_hi", "ransac_hypotheses", "n_removed"):
            assert getattr(sg, k) == getattr(so, k), f"frame {t} stat {k}: {getattr(sg, k)} vs {getattr(so, k)}"
        assert sg.n_li > 450, f"benchmark regime needs n_li > 450, got {sg.n_li}"
        assert_tables_equal(g, o, ctx=f"cfg2 frame {t}")
        em, es = assert_state_close(g, o, ctx=f"cfg2 frame {t} symmetric={symmetric}")
        worst = [max(worst[0], em), max(worst[1], es)]
    print(f"cfg2 N=500 symmetric={symmetric}: n={g.state_dim()} n_li={g.stats().n_li} worst rel err mu {worst[0]:.2e} "
          f"Sigma {worst[1]:.2e}")


def _numpy_check(gpu_pkg, workload, n_frames_checked=1, symmetric=True):
    nfeat = bench.WORKLOADS[workload][0]
    sc = bench.make_scene(gpu_pkg, workload, 1 + n_frames_checked)
    cfg = bench.bench_config(gpu_pkg, sc)
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=nfeat + 4)
    g.set_symmetric_downdate(symmetric)
    assert _seed(g, sc) == nfeat
    out = []
    for t in range(1, 1 + n_frames_checked):
        g.captureNewFrame(sc.frame(t), sc.stamps[t]); g.predict()
        assert g.match() > 0.9 * nfeat
        mu0, S0 = g.get_full()
        feats = [g.feature(i) for i in range(g.numOfFeatures())]
        g.update_after_match(sc.picks(t, nfeat))
        st = g.stats()
        assert st.n_removed == 0 and st.n_hi == 0, "the synthetic scene is all-inlier: one stacked update per frame"
        post = [g.feature(i) for i in range(g.numOfFeatures())]
        sel = [i for i, f in enumerate(post) if f.is_in_li]
        assert len(sel) == st.n_li
        mu_ref, S_ref = numpy_stacked_update(mu0, S0, feats, sel, float(cfg.sigma_pixel) ** 2)
        mu1, S1 = g.get_full()
        em, es = relerr(mu1, mu_ref), relerr(S1, S_ref)
        # the change itself must be resolved, not just the unchanged bulk of Sigma
        ed = relerr(S1 - S0, S_ref - S0)
        out.append((st.n_li, em, es, ed))
        assert em <= TOL and es <= TOL, f"{workload} frame {t}: mu {em:.3e} Sigma {es:.3e}"
        assert_scaled_close(mu1, S1, mu_ref, S_ref, f"{workload} frame {t} vs numpy")
        assert ed <= 1e-7, f"{workload} frame {t}: relative error of the covariance correction {ed:.3e}"
    return g.state_dim(), out


def test_cfg2_n500_against_numpy(gpu_pkg):
    n, out = _numpy_check(gpu_pkg, "cfg2_n500", 2)
    print(f"cfg2 vs numpy: n={n} (n_li, mu, Sigma, dSigma) = {out}")


def test_cfg4_n2000_against_numpy(gpu_pkg, monkeypatch):
    """32 update blocks through the look-ahead pipeline (default for n >= 6000) on one GPU."""
    for v in ("EKF_LOOKAHEAD_MIN_N", "EKF_PIPE_MIN_N"):
        monkeypatch.delenv(v, raising=False)
    n, out = _numpy_check(gpu_pkg, "cfg4_n2000", 1)
    assert n == 14 + 6 * 2000 and out[0][0] > 1900
    print(f"cfg4 vs numpy: n={n} (n_li, mu, Sigma, dSigma) = {out}")


def test_cluster_ransac_long_candidate_list(gpu_pkg, monkeypatch):
    """More than 8 * 512 matched features: the pick-without-replacement erase of the cluster kernel must shift
    the whole tail (vslamRansac.cpp:991).  The one-CTA kernel (1024 threads x 8) restates the same loop; both
    must leave identical hypothesis counts, Li flags and therefore bit-identical states."""
    N = 4500
    sc = gpu_pkg.synth.Scene(n_features=N, width=1920, height=1080, n_frames=2, seed=77, speed=0.1, omega=0.02,
                             accel_sigma=0.002, border=44)
    cfg = gpu_pkg.default_config(**sc.config_overrides())
    res = []
    for cluster in ("1", "0"):
        monkeypatch.setenv("EKF_RANSAC_CLUSTER", cluster)
        g = gpu_pkg.VSlamFilter(cfg, feature_capacity=N + 4)
        added = _seed(g, sc)
        g.captureNewFrame(sc.frame(1), sc.stamps[1]); g.predict()
        nm = g.match()
        # picks of 0 draw the FIRST candidate every time, so each erase moves the whole list; every third measurement
        # is displaced so that bad hypotheses keep the adaptive loop running for several iterations
        rng = np.random.default_rng(5)
        for i in range(2, added, 3):
            f = g.feature(i)
            if f.is_in_innovation:
                g.inject_match(i, f.z[0] + 40.0 * rng.standard_normal(), f.z[1] + 40.0 * rng.standard_normal(), True)
        g.update_after_match(np.zeros(64, dtype=np.uint32))
        st = g.stats()
        flags = np.array([g.feature(i).is_in_li for i in range(g.numOfFeatures())])
        res.append((nm, st.ransac_hypotheses, st.n_li, st.n_hi, flags, g.getState()))
        del g
    assert res[0][0] > 4200, "need more than 4096 candidates"
    assert res[0][1] >= 2, "the test needs more than one hypothesis to exercise the erase"
    assert res[0][1:4] == res[1][1:4], f"cluster {res[0][1:4]} vs one CTA {res[1][1:4]}"
    assert np.array_equal(res[0][4], res[1][4])
    assert np.array_equal(res[0][5], res[1][5])
