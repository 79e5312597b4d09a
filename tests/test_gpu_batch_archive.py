"""-m gpu: the feature archive and the map export of the batched filters (ekf_batch_set_archive, ekf_batch_remove_feature,
ekf_batch_get_deleted, ekf_batch_get_points_features, FilterBatch.view).

The scene of most tests: frames 1-7 show every feature, the rho variances are cut before frame 6 so that features convert to
XYZ, and from frame 8 on only the even features are drawn.  With min_features = the seeded count and max_features two below it,
frame 8 takes the max_features removeFeature(0) branch on a well-observed XYZ feature, and later frames delete the hidden
features for quality.  _Routes counts the steps in which each route archived, from the step counters alone: a step that
removed one feature while the max_features rule had to fire archived its victim; a step that archived two records, or one
without the rule, archived a quality deletion."""
import ctypes as C

import numpy as np
import pytest

from helpers import INT_FIELDS, TOL, relerr, seed_features
from test_gpu_batch_config import _oracles
from test_gpu_batch_topup import _perturbed

pytestmark = pytest.mark.gpu

N0 = 16
SWITCH = 8      # first frame with the odd features hidden
SHRINK = 6      # rho variances cut before this frame's step


def _scenes(pkg, seed=71, n_frames=14):
    full = pkg.synth.Scene(n_features=N0, n_frames=n_frames, seed=seed)
    half = pkg.synth.Scene(n_features=N0, n_frames=n_frames, seed=seed, visible_every=2)
    return full, lambda t: (full if t < SWITCH else half).frame(t)


def _cfg(pkg, sc, **over):
    return pkg.default_config(**dict(sc.config_overrides(), min_features=N0, max_features=N0 - 2, xyz_conversion=1, **over))


def _shrunk(f, factor=1e-4):
    mu, S = f.get_full()
    for i in range(f.numOfFeatures()):
        ft = f.feature(i)
        if not ft.coding:
            p = ft.position_in_state
            S[p + 5, :] *= factor; S[:, p + 5] *= factor
    return mu, S


class _Routes:
    def __init__(self, max_features):
        self.maxf, self.quality, self.victim = max_features, 0, 0

    def step(self, N_before, n_removed, topup_request, archived):
        if n_removed == 1 and topup_request > 0 and N_before - 1 > self.maxf:
            self.victim += int(archived == 1)
        elif archived >= 2 or (archived >= 1 and topup_request == 0):
            self.quality += 1


def _same_records(a, b, tol, ctx):
    assert len(a) == len(b), f"{ctx}: {len(a)} records vs {len(b)}"
    for k, ((ia, xa, ca), (ib, xb, cb)) in enumerate(zip(a, b)):
        assert ia == ib, f"{ctx} record {k}: real_index {ia} vs {ib}"
        assert relerr(xa, xb) <= tol and relerr(ca, cb) <= tol, f"{ctx} record {k}: {relerr(xa, xb):.2e} {relerr(ca, cb):.2e}"


@pytest.mark.parametrize("cap,large", [(32, False), (128, True)])
def test_filter0_follows_single_filter(gpu_pkg, cap, large):
    """Filter 0 (unperturbed) runs free beside a single CUDA filter with top-up and XYZ conversion: its archive has the single
    filter's length, order and real_indices with values within 1e-8, and so does its points matrix; both routes archive."""
    sc, frame = _scenes(gpu_pkg)
    cfg = _cfg(gpu_pkg, sc)
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=cap)
    seed_features(g, sc); seed_features(src, sc)
    batch = gpu_pkg.FilterBatch.from_config(cfg, 3, feature_capacity=cap, large=large, archive=64)
    batch.seed_from(src)
    batch.set_topup(True)
    batch.set_camera_states(_perturbed(g.get_full()[0], 3, 6))
    routes = _Routes(cfg.max_features)
    for t in range(1, sc.n_frames):
        if t == SHRINK:
            mu, S = _shrunk(g)
            g.set_full(mu, S); batch.set_full(0, mu, S)
        img, picks = frame(t), sc.picks(t, N0)
        N_before, held = g.numOfFeatures(), len(g.deleted())
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        routes.step(N_before, g.stats().n_removed, g.stats().topup_request, len(g.deleted()) - held)
        N = g.numOfFeatures()
        assert batch.numOfFeatures(0) == N, f"frame {t}: feature count"
        assert [batch.feature(0, i).real_index for i in range(N)] == [g.feature(i).real_index for i in range(N)], f"frame {t}"
        mb, Sb = batch.get_full(0); mg, Sg = g.get_full()
        assert relerr(mb, mg) <= 1e-8 and relerr(Sb, Sg) <= 1e-8, f"frame {t}: mu {relerr(mb, mg):.2e} Sigma {relerr(Sb, Sg):.2e}"
        _same_records(batch.deleted(0), g.deleted(), 1e-8, f"frame {t}")
        Pb, Pg = batch.getPointsFeatures(0), g.getPointsFeatures()
        assert Pb.shape == Pg.shape and relerr(Pb, Pg) <= 1e-8, f"frame {t}: points {Pb.shape} {Pg.shape}"
    print(f"cap {cap}: archived {len(g.deleted())}, steps archiving quality deletions {routes.quality}, max_features victims "
          f"{routes.victim}, counts {list(batch.num_deleted())}")
    assert routes.quality > 0 and routes.victim > 0


def test_step_against_oracle(gpu_pkg, orc):
    """Every filter of a perturbed batch, per step from identical inputs (batch state <- oracle state): archive records and
    points matrices against OracleFilter at TOL.  The reference archives one step's quality deletions in descending index
    (vslamRansac.cpp:1296-1299), the single CUDA filter and the batch in ascending index; the records are compared by
    real_index."""
    sc, frame = _scenes(gpu_pkg, seed=72)
    cfg = _cfg(gpu_pkg, sc)
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    B = 3
    batch = gpu_pkg.FilterBatch(cfg, B, feature_capacity=32)
    batch.set_archive(32)
    batch.seed_from(g)
    cams = _perturbed(g.get_full()[0], B, 8)
    batch.set_camera_states(cams)
    oracles = _oracles(orc, cfg, g, sc.frame(0), sc.stamps[0], cams)
    routes = [_Routes(cfg.max_features) for _ in oracles]
    for t in range(1, sc.n_frames):
        img, picks = frame(t), sc.picks(t, N0)
        for b, o in enumerate(oracles):
            mu, S = _shrunk(o) if t == SHRINK else o.get_full()
            o.set_full(mu, S); batch.set_full(b, mu, S)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        _, st = batch.camera_states()
        for b, o in enumerate(oracles):
            N_before, held = o.numOfFeatures(), len(o.deleted())
            o.captureNewFrame(img, sc.stamps[t]); o.predict(); o.update(picks)
            routes[b].step(N_before, o.stats().n_removed, o.stats().topup_request, len(o.deleted()) - held)
            assert st[b, 6] == o.stats().n_removed, f"frame {t} filter {b}: removed"
            assert batch.numOfFeatures(b) == o.numOfFeatures()
            for i in range(o.numOfFeatures()):
                a, c = batch.feature(b, i), o.feature(i)
                assert all(getattr(a, f) == getattr(c, f) for f in INT_FIELDS), f"frame {t} filter {b} feature {i}"
            _same_records(sorted(batch.deleted(b), key=lambda r: r[0]), sorted(o.deleted(), key=lambda r: r[0]), TOL,
                          f"frame {t} filter {b}")
        for b, (Pb, o) in enumerate(zip(batch.points_features(), oracles)):
            Po = o.getPointsFeatures()
            assert Pb.shape == Po.shape and relerr(Pb, Po) <= TOL, f"frame {t} filter {b}: points"
    for b, (o, r) in enumerate(zip(oracles, routes)):
        print(f"filter {b}: archived {len(o.deleted())}, steps archiving quality deletions {r.quality}, max_features victims {r.victim}")
    assert sum(r.victim for r in routes) > 0 and sum(r.quality for r in routes) > 0


def _source(pkg, archive_removals=0):
    """A single filter after seven frames in which only the even features were drawn (quality_ratio 1e9 keeps the others), then
    the rho variances of all but the last four features cut and converted: XYZ features with n_find 7 (even) and 0 (odd), and
    inverse-depth ones.  archive_removals: that many well-observed XYZ features are removed from it afterwards."""
    sc = pkg.synth.Scene(n_features=16, n_frames=8, seed=74, visible_every=2)
    cfg = pkg.default_config(**dict(sc.config_overrides(), quality_ratio=1e9, xyz_conversion=0))
    g = pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    for t in range(1, sc.n_frames):
        g.captureNewFrame(sc.frame(t), sc.stamps[t]); g.predict(); g.update(sc.picks(t, 16))
    mu, S = g.get_full()
    for i in range(g.numOfFeatures() - 4):
        p = g.feature(i).position_in_state
        S[p + 5, :] *= 1e-4; S[:, p + 5] *= 1e-4
    g.set_full(mu, S)
    g.convert2XYZ_ifLinearAll()
    for _ in range(archive_removals):
        i = next(i for i in range(g.numOfFeatures()) if g.feature(i).coding and g.feature(i).n_find > 5)
        g.removeFeature(i)
    return cfg, g


def test_remove_feature(gpu_pkg):
    """removeFeature(f, i) on an XYZ feature with n_find > 5, an XYZ feature seen less often and an inverse-depth feature
    matches VSlamFilter.removeFeature on the same source: state within TOL, table exact, archive; the other filters keep
    every bit.  Error codes for bad arguments and before seeding."""
    cfg, src = _source(gpu_pkg)
    E = gpu_pkg._abi
    L = gpu_pkg.lib()
    fresh = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=32)
    assert L.ekf_batch_remove_feature(fresh.h, 0, 0) == E.EKF_ERR_STATE
    batch = gpu_pkg.FilterBatch(cfg, 3, feature_capacity=32)
    batch.set_archive(8)
    batch.seed_from(src)
    batch.set_camera_states(_perturbed(src.get_full()[0], 3, 3))
    cases = {
        "xyz seen > 5": lambda f: f.coding and f.n_find > 5,
        "xyz seen <= 5": lambda f: f.coding and f.n_find <= 5,
        "inverse depth": lambda f: not f.coding,
    }
    L0 = batch.kernel_launches()
    for name, pick in cases.items():
        i = next(i for i in range(src.numOfFeatures()) if pick(src.feature(i)))
        before = [(batch.get_full(b), [batch.feature(b, k).real_index for k in range(batch.numOfFeatures(b))]) for b in (1, 2)]
        batch.removeFeature(0, i); src.removeFeature(i)
        assert batch.numOfFeatures(0) == src.numOfFeatures() and batch.state_dim(0) == src.state_dim(), name
        mb, Sb = batch.get_full(0); ms, Ss = src.get_full()
        assert relerr(mb, ms) <= TOL and relerr(Sb, Ss) <= TOL, name
        for k in range(src.numOfFeatures()):
            a, c = batch.feature(0, k), src.feature(k)
            assert all(getattr(a, f) == getattr(c, f) for f in INT_FIELDS), f"{name}: feature {k}"
        _same_records(batch.deleted(0), src.deleted(), 0.0, name)
        for (b, ((m0, S0), ri0)) in zip((1, 2), before):
            m1, S1 = batch.get_full(b)
            assert np.array_equal(m0, m1) and np.array_equal(S0, S1), f"{name}: filter {b} changed"
            assert ri0 == [batch.feature(b, k).real_index for k in range(batch.numOfFeatures(b))]
    assert batch.kernel_launches() - L0 == 3, "one launch per removal"
    assert list(batch.num_deleted()) == [1, 0, 0] and len(src.deleted()) == 1
    for f, i in ((3, 0), (-1, 0), (1, -1), (1, batch.numOfFeatures(1))):
        assert L.ekf_batch_remove_feature(batch.h, f, i) == E.EKF_ERR_ARG, (f, i)
    assert L.ekf_batch_set_archive(batch.h, -1) == E.EKF_ERR_ARG


def test_seeding_copies_the_archive(gpu_pkg):
    cfg, src = _source(gpu_pkg, archive_removals=3)
    want = src.deleted()
    assert len(want) == 3
    batch = gpu_pkg.FilterBatch(cfg, 4, feature_capacity=32)
    batch.set_archive(3)
    batch.seed_from(src)
    assert list(batch.num_deleted()) == [3] * 4
    for b in range(4):
        _same_records(batch.deleted(b), want, 0.0, f"filter {b}")
        assert np.array_equal(batch.getPointsFeatures(b), src.getPointsFeatures())
    small = gpu_pkg.FilterBatch(cfg, 2, feature_capacity=32)
    small.set_archive(2)
    assert gpu_pkg.lib().ekf_batch_seed_from(small.h, src.h) == gpu_pkg._abi.EKF_ERR_CAPACITY
    off = gpu_pkg.FilterBatch(cfg, 2, feature_capacity=32)
    off.seed_from(src)
    assert list(off.num_deleted()) == [0, 0] and off.deleted(1) == []


def _run_pair(pkg, caps, topup=True, steps=None):
    """Batches with the given archive capacities (None: set_archive never called) stepped over the scene; yields per step the
    return codes, last errors and the batches."""
    sc, frame = _scenes(pkg, seed=75)
    cfg = _cfg(pkg, sc)
    g = pkg.VSlamFilter(cfg, feature_capacity=32)
    seed_features(g, sc)
    cams = _perturbed(g.get_full()[0], 4, 11)
    batches = []
    for cap in caps:
        x = pkg.FilterBatch(cfg, 4, feature_capacity=32)
        if cap is not None:
            x.set_archive(cap)
        x.seed_from(g); x.set_topup(topup); x.set_camera_states(cams)
        x.setup_launches = x.kernel_launches()
        batches.append(x)
    L = pkg.lib()
    for t in range(1, steps or sc.n_frames):
        if t == SHRINK:
            for x in batches:
                for b in range(4):
                    x.set_full(b, *_shrunk(_BatchMember(x, b)))
        img, picks = frame(t), np.ascontiguousarray(sc.picks(t, N0), dtype=np.uint32)
        rcs, errs = [], []
        for x in batches:
            x.captureNewFrame(img, sc.stamps[t])
            z = np.zeros(3)
            rcs.append(L.ekf_batch_step(x.h, z.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p), 0,
                                        picks.ctypes.data_as(C.c_void_p), picks.size))
            errs.append(L.ekf_batch_last_error(x.h).decode())
        yield t, rcs, errs, batches


class _BatchMember:
    """get_full / feature / numOfFeatures of one filter of a batch, for _shrunk."""

    def __init__(self, batch, b):
        self.x, self.b = batch, b

    def get_full(self):
        return self.x.get_full(self.b)

    def feature(self, i):
        return self.x.feature(self.b, i)

    def numOfFeatures(self):
        return self.x.numOfFeatures(self.b)


def _states(x):
    out = []
    for b in range(x.B):
        tab = [tuple(getattr(x.feature(b, i), f) for f in INT_FIELDS) for i in range(x.numOfFeatures(b))]
        out.append((x.get_full(b), tab))
    return out


def test_overflow(gpu_pkg):
    """A capacity-1 archive drops records: the step runs to its end (states equal a capacity-64 batch bit for bit), then
    returns EKF_ERR_CAPACITY naming the first filter that dropped one in that step."""
    cap = 1
    errors = 0
    prev = np.zeros(4, dtype=np.int64)
    for t, rcs, errs, (small, big) in _run_pair(gpu_pkg, [cap, 64]):
        assert rcs[1] == 0, f"frame {t}: {errs[1]}"
        counts = big.num_deleted().astype(np.int64)
        over = [b for b in range(4) if counts[b] > cap and counts[b] > prev[b]]
        if over:
            errors += 1
            assert rcs[0] == gpu_pkg._abi.EKF_ERR_CAPACITY and errs[0].startswith(f"filter {over[0]}:"), (t, rcs[0], errs[0], over)
        else:
            assert rcs[0] == 0, (t, errs[0])
        prev = counts
        assert list(small.num_deleted()) == [min(int(c), cap) for c in counts]
        for b in range(4):
            _same_records(small.deleted(b), big.deleted(b)[:cap], 0.0, f"frame {t} filter {b}")
        _, s0 = small.camera_states(); _, s1 = big.camera_states()
        assert np.array_equal(s0, s1)
        for (a, ta), (c, tc) in zip(_states(small), _states(big)):
            assert np.array_equal(a[0], c[0]) and np.array_equal(a[1], c[1]) and ta == tc, f"frame {t}"
    print(f"steps that overflowed: {errors}, records {list(prev)}")
    assert errors > 0


def test_points_features_range_and_errors(gpu_pkg):
    for t, rcs, errs, (x,) in _run_pair(gpu_pkg, [16], steps=SWITCH + 3):
        pass
    assert x.num_deleted().sum() > 0
    each = [x.getPointsFeatures(b) for b in range(4)]
    assert all(np.array_equal(a, b) for a, b in zip(x.points_features(), each))
    assert all(np.array_equal(a, b) for a, b in zip(x.points_features(1, 2), each[1:3]))
    L, E = gpu_pkg.lib(), gpu_pkg._abi
    rows = np.zeros(4, dtype=np.int32)
    rp = rows.ctypes.data_as(C.c_void_p)
    assert L.ekf_batch_get_points_features(x.h, 0, 4, None, 0, rp) == 0
    assert list(rows) == [len(a) for a in each]
    big = int(rows.max())
    out = np.full((4, big + 3, 12), 7.0)
    assert L.ekf_batch_get_points_features(x.h, 0, 4, out.ctypes.data_as(C.c_void_p), big + 3, rp) == 0
    for k in range(4):
        assert np.array_equal(out[k, :rows[k]], each[k]) and not out[k, rows[k]:].any()
    assert L.ekf_batch_get_points_features(x.h, 0, 4, out.ctypes.data_as(C.c_void_p), big - 1, rp) == E.EKF_ERR_ARG
    for first, count in ((-1, 1), (0, 0), (3, 2), (4, 1)):
        assert L.ekf_batch_get_points_features(x.h, first, count, None, 0, rp) == E.EKF_ERR_ARG, (first, count)
    assert L.ekf_batch_get_points_features(x.h, 0, 1, None, 0, None) == E.EKF_ERR_ARG


def test_archive_off_changes_nothing(gpu_pkg):
    """A batch that never called set_archive, one whose archive was switched on and off again, and one with it on take the same
    launches per step and end every step with bit-identical states, tables and counters (removals occur)."""
    removed = 0
    launches = None
    for t, rcs, errs, xs in _run_pair(gpu_pkg, [None, 0, 64]):
        assert rcs == [0, 0, 0], errs
        if launches is None:   # seeding launched one more kernel with the archive on: the copy of the source's archive
            assert [x.setup_launches for x in xs][2] == xs[0].setup_launches + 1 == xs[1].setup_launches + 1
            launches = [x.setup_launches for x in xs]
        ks = [x.kernel_launches() for x in xs]
        assert ks[0] - launches[0] == ks[1] - launches[1] == ks[2] - launches[2], f"frame {t}: launches {ks} {launches}"
        launches = ks
        st = [x.camera_states()[1] for x in xs]
        assert np.array_equal(st[0], st[1]) and np.array_equal(st[0], st[2]), f"frame {t}: counters"
        removed += int(st[0][:, 6].sum())
        s = [_states(x) for x in xs]
        for other in s[1:]:
            for (a, ta), (c, tc) in zip(s[0], other):
                assert np.array_equal(a[0], c[0]) and np.array_equal(a[1], c[1]) and ta == tc, f"frame {t}"
    assert removed > 0 and xs[2].num_deleted().sum() > 0 and xs[0].num_deleted().sum() == 0


def test_keyframe_recorder_on_batch_view(gpu_pkg, tmp_path):
    """KeyframeRecorder driven by batch.view(0) and by a free-running single filter picks the same key frames and writes files
    that agree to the printed precision; recorders on three views share one camera-state read per frame."""
    kf = gpu_pkg.keyframes
    sc = gpu_pkg.synth.Scene(n_features=20, n_frames=24, seed=13)
    cfg = gpu_pkg.default_config(**dict(sc.config_overrides(), xyz_conversion=1))
    g = gpu_pkg.VSlamFilter(cfg, feature_capacity=28)
    src = gpu_pkg.VSlamFilter(cfg, feature_capacity=28)
    seed_features(g, sc); seed_features(src, sc)
    batch = gpu_pkg.FilterBatch.from_config(cfg, 3, feature_capacity=28, archive=32)
    batch.seed_from(src)
    batch.set_camera_states(_perturbed(g.get_full()[0], 3, 2))
    reads = [0]
    real = batch.camera_states

    def counted(*a, **k):
        reads[0] += 1
        return real(*a, **k)
    batch.camera_states = counted

    def rec(name):
        r = kf.KeyframeRecorder(str(tmp_path / name))
        r.MoveThresh = 0.6
        return r
    rg = rec("single")
    rv = [rec(f"view{b}") for b in range(3)]
    views = [batch.view(b) for b in range(3)]
    for t in range(1, sc.n_frames):
        img, picks = sc.frame(t), sc.picks(t, 20)
        g.captureNewFrame(img, sc.stamps[t]); g.predict(); g.update(picks)
        batch.captureNewFrame(img, sc.stamps[t]); batch.step(picks)
        rg.on_frame(g, t, img)
        for r, v in zip(rv, views):
            r.on_frame(v, t, img)
        assert reads[0] == t, f"frame {t}: {reads[0]} camera-state reads"
        cg, cv = g.Covariance_Parameter(), views[0].Covariance_Parameter()
        assert abs(cg - cv) <= 1e-8 * abs(cg), (t, cg, cv)
    rg.finish(g)
    for r, v in zip(rv, views):
        r.finish(v)
    assert rv[0].key_frames == rg.key_frames and len(rg.key_frames) >= 2
    Pg, Cg, Ng = kf.read_sba_inputs(str(tmp_path / "single"))
    Pb, Cb, Nb = kf.read_sba_inputs(str(tmp_path / "view0"))
    assert Pg.shape == Pb.shape and Cg.shape == Cb.shape and len(Ng) == len(Nb)
    assert np.allclose(Pb, Pg, rtol=1e-5, atol=1e-12) and np.allclose(Cb, Cg, rtol=1e-5, atol=1e-15)
    for (ca, pa, ja), (cb, pb, jb) in zip(Ng, Nb):
        assert ca == cb and ja == jb and np.allclose(pa, pb, rtol=1e-5, atol=1e-9)
    print(f"key frames: single {rg.key_frames}, views {[r.key_frames for r in rv]}")
