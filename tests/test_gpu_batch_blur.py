"""-m gpu: motion-blur template prediction in the batched filters (Patch::blur, Patch.cpp:50-57; evaluateKernel / blurPatch,
libblur.cpp:17-81).

A batch is created with blur off (ekf_batch_create refuses it) and switched on with FilterBatch.set_motion_blur(3); the single
filter and the oracle are built with kernel_size = 3.  The scene is the single filter's blur scene (a fast camera, smooth
templates, T_camera = 0.5 as conf_sim.cfg).  Every filter's predicted templates must be the single CUDA filter's bit for bit,
and a step the oracle's: tables and NCC scores bit-exact, the state within the per-step bars."""
import numpy as np
import pytest

from helpers import relerr, seed_features
from test_gpu_batch_topup import _centers, _check, _perturbed, _single_with

pytestmark = pytest.mark.gpu

BLUR_SCENE = dict(speed=0.9, omega=0.5, template_smooth=2.5)
OFF = 1000000000


def _scene(pkg, **kw):
    return pkg.synth.Scene(**dict(BLUR_SCENE, **kw))


def _cfgs(pkg, sc, **over):
    """(batch configuration: blur off, single-filter / oracle configuration: kernel_size = 3), both with T_camera = 0.5."""
    base = dict(sc.config_overrides(), T_camera=0.5, **over)
    return pkg.default_config(**dict(base, kernel_size=OFF)), pkg.default_config(**dict(base, kernel_size=3))


def _moving(cams, sc):
    """Camera states moving with the scene's camera (world-frame v, body-frame w): without matches the filters' own velocity
    estimates stay at the prior's zero, and nothing would blur."""
    cams = cams.copy()
    cams[:, 7:10] += sc.v[1]
    cams[:, 10:13] += sc.w[1]
    return cams


def _blur_batch(pkg, cfg_b, src, B, cap=32):
    batch = pkg.FilterBatch(cfg_b, B, feature_capacity=cap)
    batch.seed_from(src)
    batch.set_motion_blur(3)
    return batch


def test_predicted_templates_equal_single_filter(gpu_pkg):
    """ncc_threshold > 1: no match is accepted, so after a step every filter's matching templates are its predict's.  Each
    filter, moving at the scene's velocities, against a single CUDA filter from the same state after predict, bit for bit;
    blur counts against its stats."""
    sc = _scene(gpu_pkg, n_features=24, n_frames=4, seed=29)
    cfg_b, cfg_s = _cfgs(gpu_pkg, sc, ncc_threshold=2.0, quality_ratio=1e30)
    g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
    seed_features(g, sc)
    B = 5
    batch = _blur_batch(gpu_pkg, cfg_b, g, B)
    mu0, S0 = g.get_full()
    cams = _moving(_perturbed(mu0, B, 11, perturb=5e-3), sc)
    batch.set_camera_states(cams)
    blurred = compared = 0
    for t in (1, 2, 3):
        img, picks = sc.frame(t), sc.picks(t, 24)
        states = [batch.get_full(b) for b in range(B)]
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        counts = batch.last_blur_counts()
        assert counts.dtype == np.int32 and counts.shape == (B,)
        for b in range(B):
            s = gpu_pkg.VSlamFilter(cfg_s, feature_capacity=32)
            seed_features(s, sc)
            if t > 1:
                s.captureNewFrame(sc.frame(t - 1), sc.stamps[t - 1])   # the batch's dT
            s.set_full(*states[b])
            s.captureNewFrame(img, sc.stamps[t]); s.predict()
            assert s.numOfFeatures() == batch.numOfFeatures(b)
            for i in range(s.numOfFeatures()):
                if not s.feature(i).is_in_innovation:
                    continue
                a, c = batch.template(b, i, 1), s.template(i, 1)
                assert np.array_equal(a, c), f"frame {t} filter {b} feature {i}: blurred template differs in {(a != c).sum()} pixels"
                compared += 1
                blurred += int(not np.array_equal(c, s.template(i, 0)))
            s.update(picks)
            assert counts[b] == s.stats().blur_requests, f"frame {t} filter {b}: {counts[b]} blurred, single filter {s.stats().blur_requests}"
        print(f"frame {t}: blurred per filter {list(counts)}")
    assert blurred >= 10, f"only {blurred} of {compared} templates were blurred: the scene does not exercise the path"


def _bits(x):
    return int(np.float32(x).view(np.uint32))


def _ensemble(pkg, orc, sc, cfg_b, cfg_o, B, seed):
    g = pkg.VSlamFilter(cfg_b, feature_capacity=32)
    seed_features(g, sc)
    batch = _blur_batch(pkg, cfg_b, g, B)
    mu0, S0 = g.get_full()
    cams = _perturbed(mu0, B, seed)
    batch.set_camera_states(cams)
    oracles = []
    for b in range(B):
        o = orc.OracleFilter(cfg_o, kind=0, omp=False)
        o.captureNewFrame(sc.frame(0), sc.stamps[0]); o.import_from(g)
        m = mu0.copy(); m[:14] = cams[b]
        o.set_full(m, S0)
        oracles.append(o)
    return batch, oracles


@pytest.mark.parametrize("window", [11, 21, 30])
def test_step_against_oracle(gpu_pkg, orc, window):
    """Filters 0-2 of a perturbed ensemble, per step from identical inputs (batch state <- oracle state): tables and last_ncc
    bit-exact, the state within TOL and the scaled bars, blur counts equal to the oracle's.  Window 11 runs the tile matcher,
    21 and 30 the CTA matcher; 30 is conf_sim's."""
    sc = _scene(gpu_pkg, n_features=24, n_frames=6, seed=29, window=window)
    cfg_b, cfg_o = _cfgs(gpu_pkg, sc)
    B = 3
    batch, oracles = _ensemble(gpu_pkg, orc, sc, cfg_b, cfg_o, B, 7)
    blurred = matched = 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        for b, o in enumerate(oracles):
            batch.set_full(b, *o.get_full())
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        _, st = batch.camera_states()
        counts = batch.last_blur_counts()
        for b, o in enumerate(oracles):
            before = o.stats().blur_requests
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert counts[b] == so.blur_requests - before, f"frame {t} filter {b}: blurred {counts[b]} vs {so.blur_requests - before}"
            assert st[b, 1] == so.n_matched, f"frame {t} filter {b}: matched {st[b, 1]} vs {so.n_matched}"
            for i in range(o.numOfFeatures()):
                assert _bits(batch.feature(b, i).last_ncc) == _bits(o.feature(i).last_ncc), f"frame {t} filter {b} feature {i}: NCC"
            blurred += int(counts[b]); matched += int(st[b, 1])
        _check(batch, oracles, f"window {window} frame {t}")
    print(f"window {window}: {blurred} templates blurred, {matched} matches")
    assert blurred >= 10 and matched > 0


def test_blur_topup_and_xyz_in_reference_order(gpu_pkg, orc):
    """Blur, top-up and XYZ conversion all on; per step from identical inputs against the oracle run in the reference order:
    predict with blur, update without conversion, addFeatures on the batch's new centres, convert2XYZ_ifLinearAll."""
    sc = _scene(gpu_pkg, n_features=24, n_frames=6, seed=502, hard=True)
    over = dict(min_features=21, max_features=16)
    cfg_b, _ = _cfgs(gpu_pkg, sc, xyz_conversion=1, **over)
    _, cfg_o = _cfgs(gpu_pkg, sc, xyz_conversion=0, **over)
    g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
    g.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels[:20]:
        assert g.addFeature(*p) == 1
    B = 4
    batch = _blur_batch(gpu_pkg, cfg_b, g, B)
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
    for u, v in sc.feature_pixels[20:]:
        assert batch.addFeature(2, u, v) == 1 and oracles[2].addFeature(u, v) == 1
    blurred = added_total = converted = 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        for b, o in enumerate(oracles):
            mu, S = o.get_full()
            if b:   # cut one inverse-depth feature's rho variance so that conversions happen
                inv = [i for i in range(o.numOfFeatures()) if not o.feature(i).coding]
                if inv:
                    p = o.feature(inv[(b + t) % len(inv)]).position_in_state
                    S[p + 5, :] *= 10.0 ** -(3 + b % 3); S[:, p + 5] *= 10.0 ** -(3 + b % 3)
            o.set_full(mu, S); batch.set_full(b, mu, S)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        _, st = batch.camera_states()
        added, counts = batch.last_added(), batch.last_blur_counts()
        for b, o in enumerate(oracles):
            before = {o.feature(i).real_index: o.feature(i).coding for i in range(o.numOfFeatures())}
            nb0 = o.stats().blur_requests
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            so = o.stats()
            assert counts[b] == so.blur_requests - nb0, f"frame {t} filter {b}: blurred"
            assert (st[b, 6], st[b, 7]) == (so.n_removed, so.topup_request), f"frame {t} filter {b}: removed / top-up"
            want = 0
            if so.topup_request > 0:
                survivors = _centers(o)
                corners = _single_with(gpu_pkg, cfg_o, img, survivors).detect_corners(int(so.topup_request))
                want = min(len(corners), int(so.topup_request), 32 - len(survivors))
            assert added[b] == want, f"frame {t} filter {b}: added {added[b]}, single filter {want}"
            nb = batch.numOfFeatures(b)
            if added[b]:
                new = [tuple(batch.feature(b, i).center) for i in range(nb - added[b], nb)]
                assert o.addFeatures(np.array(new, dtype=np.float32)) == added[b]
            o.convert2XYZ_ifLinearAll()
            converted += sum(1 for i in range(o.numOfFeatures()) if o.feature(i).coding and not before.get(o.feature(i).real_index, 0))
            blurred += int(counts[b]); added_total += int(added[b])
        print(f"frame {t}: blurred {list(counts)} removed {list(st[:, 6])} added {list(added)}")
        _check(batch, oracles, f"frame {t}")
    assert blurred > 0 and added_total > 0 and converted > 0, (blurred, added_total, converted)


def test_filter0_follows_single_filter(gpu_pkg):
    """Filter 0 (unperturbed) runs free against a single CUDA filter with blur (and top-up and XYZ conversion)."""
    sc = _scene(gpu_pkg, n_features=20, n_frames=10, seed=93, hard=True, outlier_frac=0.15)
    cfg_b, cfg_s = _cfgs(gpu_pkg, sc, min_features=22, max_features=26, xyz_conversion=1)
    g = gpu_pkg.VSlamFilter(cfg_s, feature_capacity=32)
    seed_features(g, sc)
    src = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
    seed_features(src, sc)
    batch = _blur_batch(gpu_pkg, cfg_b, src, 3)
    batch.set_topup(True)
    mu0, _ = g.get_full()
    batch.set_camera_states(_perturbed(mu0, 3, 6))
    blurred = 0
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 24)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        assert batch.last_blur_counts()[0] == g.stats().blur_requests, f"frame {t}: blurred"
        blurred += g.stats().blur_requests
        N = g.numOfFeatures()
        assert batch.numOfFeatures(0) == N, f"frame {t}: feature count {batch.numOfFeatures(0)} vs {N}"
        fb = [batch.feature(0, i) for i in range(N)]
        fg = [g.feature(i) for i in range(N)]
        for f in ("real_index", "coding"):
            assert [getattr(a, f) for a in fb] == [getattr(c, f) for c in fg], f"frame {t}: {f}"
        assert [tuple(f.center) for f in fb] == [tuple(f.center) for f in fg], f"frame {t}: centres"
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}: mu {relerr(mb, mg):.2e} Sigma {relerr(Sb, Sg):.2e}"
    assert blurred >= 10


def test_no_change_when_off(gpu_pkg):
    """Blur on with a threshold no displacement exceeds gives the states of blur off bit for bit, with exactly one launch more
    per step; switching it off again restores the launch count; the counts are zeros throughout."""
    sc = _scene(gpu_pkg, n_features=20, n_frames=7, seed=93, hard=True)
    cfg_b, _ = _cfgs(gpu_pkg, sc, xyz_conversion=1)
    runs = []
    for ks in (OFF, 99999):
        g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
        seed_features(g, sc)
        batch = gpu_pkg.FilterBatch(cfg_b, 4, feature_capacity=32)
        batch.seed_from(g)
        batch.set_camera_states(_perturbed(g.get_full()[0], 4, 4))
        batch.set_motion_blur(ks)
        launches, states = [], []
        for t in range(1, sc.n_frames):
            if ks != OFF and t == sc.n_frames - 2:
                batch.set_motion_blur(OFF)
            k0 = batch.kernel_launches()
            batch.captureNewFrame(sc.frame(t), sc.stamps[t]); batch.step(sc.picks(t, 20))
            launches.append(batch.kernel_launches() - k0)
            assert not batch.last_blur_counts().any()
            states.append([batch.get_full(b) for b in range(4)])
        runs.append((launches, states))
    (l0, s0), (l1, s1) = runs
    cut = sc.n_frames - 3
    assert [b - a for a, b in zip(l0, l1)] == [1] * cut + [0] * (len(l0) - cut), f"launches per step: off {l0}, on {l1}"
    for t, (a, c) in enumerate(zip(s0, s1)):
        for b, ((ma, Sa), (mc, Sc)) in enumerate(zip(a, c)):
            assert np.array_equal(ma, mc) and np.array_equal(Sa, Sc), f"step {t + 1} filter {b}"


def test_kernel_above_cap_is_reported(gpu_pkg):
    """Displacements beyond 256 px (T_camera = 60 at the scene's velocities): the step runs to its end, then raises
    EKF_ERR_UNSUPPORTED naming the first such filter, as the single filter's update does."""
    sc = _scene(gpu_pkg, n_features=16, n_frames=3, seed=29)
    base = dict(sc.config_overrides(), T_camera=60.0)
    cfg_b = gpu_pkg.default_config(**dict(base, kernel_size=OFF))
    cfg_s = gpu_pkg.default_config(**dict(base, kernel_size=3))
    g = gpu_pkg.VSlamFilter(cfg_b, feature_capacity=32)
    seed_features(g, sc)
    batch = _blur_batch(gpu_pkg, cfg_b, g, 2)
    mu, S = g.get_full()
    mu[:14] = _moving(mu[None, :14], sc)[0]
    for b in range(2):
        batch.set_full(b, mu, S)
    batch.captureNewFrame(sc.frame(1), sc.stamps[1])
    with pytest.raises(gpu_pkg.EkfError, match=r"filter 0: a motion-blur kernel exceeded 256 x 256"):
        batch.step(sc.picks(1, 16))
    cams, st = batch.camera_states()   # the step completed
    assert np.array_equal(cams[0], cams[1]) and np.array_equal(st[0], st[1])
    s = gpu_pkg.VSlamFilter(cfg_s, feature_capacity=32)
    seed_features(s, sc)
    s.set_full(mu, S)
    s.captureNewFrame(sc.frame(1), sc.stamps[1])
    s.predict()
    with pytest.raises(gpu_pkg.EkfError, match="256 x 256"):
        s.update(sc.picks(1, 16))
