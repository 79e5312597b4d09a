"""CPU: the fused removal + XYZ-conversion pass of the batched filters.  k_batch_compact rebuilds a filter's state once,
through a row map that both drops the removed features and converts the features k_batch_update decided on the
pre-removal state.  tests/xyz_fused_emu.cu runs that pass on the host with the same __host__ __device__ functions the
kernels call (xyz_linear_decide, xyz_apply_entry in csrc/ekf_math.cuh).  Its result must equal, bit for bit, the oracle's
removeFeature calls followed by convert2XYZ_ifLinearAll on the same state."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import make_oracle, seed_features

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "ekf-monoslam_for_3d-reconstruction_b200", "csrc")


@pytest.fixture(scope="module")
def emu():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = os.path.join(HERE, "_build", "libxyz_fused_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(HERE, "xyz_fused_emu.cu")
    deps = [src, os.path.join(CSRC, "ekf_math.cuh"), os.path.join(CSRC, "ekf_common.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        # host code only: -ffp-contract=off as the oracle, so no FMA contraction changes the arithmetic
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "--fmad=false", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-Xcompiler", "-ffp-contract=off", "-diag-suppress", "550", "-shared", "-I", CSRC, "-I", os.path.join(ROOT, "include"),
                        src, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    lib.emu_remove_convert.restype = ctypes.c_int
    return lib


@pytest.fixture(scope="module")
def base(pkg, orc):
    """An oracle filter with 12 inverse-depth features after three frames (correlated covariance)."""
    sc = pkg.synth.Scene(n_features=12, n_frames=4, seed=77)
    o = make_oracle(pkg, orc, sc)
    seed_features(o, sc)
    for t in range(1, sc.n_frames):
        o.captureNewFrame(sc.frame(t), sc.stamps[t]); o.predict(); o.update(sc.picks(t, 12))
    assert o.numOfFeatures() == 12
    return pkg, orc, sc, o


def _clone(pkg, orc, sc, src, shrink=()):
    """A copy of `src` in which the rho variance of the features in `shrink` is cut by 1e-4 (they then pass the linearity
    test); every other feature keeps its state."""
    o = make_oracle(pkg, orc, sc)
    o.captureNewFrame(sc.frame(0), sc.stamps[0])
    o.import_from(src)
    mu, S = o.get_full()
    for i in shrink:
        p = o.feature(i).position_in_state
        assert not o.feature(i).coding
        S[p + 5, :] *= 1e-4; S[:, p + 5] *= 1e-4
    o.set_full(mu, S)
    return o


def _emu(lib, o, removed, cfg):
    mu, S = o.get_full()
    n, N = mu.size, o.numOfFeatures()
    pos = np.array([o.feature(i).position_in_state for i in range(N)], dtype=np.int32)
    cod = np.array([o.feature(i).coding for i in range(N)], dtype=np.int32)
    rem = np.zeros(N, dtype=np.int32); rem[list(removed)] = 1
    mu2 = np.zeros(n); S2 = np.zeros(n * n); pos2 = np.zeros(N, dtype=np.int32); cod2 = np.zeros(N, dtype=np.int32)
    N2 = ctypes.c_int(0)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    mu = np.ascontiguousarray(mu); S = np.ascontiguousarray(S)
    n2 = lib.emu_remove_convert(n, N, p(mu), p(S), p(pos), p(cod), p(rem), ctypes.c_double(cfg.linearity_threshold),
                                int(cfg.abs_int_quirk), p(mu2), p(S2), p(pos2), p(cod2), ctypes.byref(N2))
    return mu2[:n2], S2[:n2 * n2].reshape(n2, n2), pos2[:N2.value], cod2[:N2.value]


def _reference(o, removed):
    for i in sorted(removed, reverse=True):   # book-keeping order (V:1296-1299), then removeFeature(0) would be the first survivor
        o.removeFeature(i)
    o.convert2XYZ_ifLinearAll()
    mu, S = o.get_full()
    N = o.numOfFeatures()
    return (mu, S, np.array([o.feature(i).position_in_state for i in range(N)]), np.array([o.feature(i).coding for i in range(N)]))


def _compare(emu, pkg, orc, sc, src, shrink, removed):
    before = _clone(pkg, orc, sc, src, shrink)
    was = [before.feature(i).coding for i in range(before.numOfFeatures())]
    mu_e, S_e, pos_e, cod_e = _emu(emu, before, removed, before.cfg)
    mu_o, S_o, pos_o, cod_o = _reference(before, removed)
    assert mu_e.shape == mu_o.shape and S_e.shape == S_o.shape
    assert np.array_equal(pos_e, pos_o) and np.array_equal(cod_e, cod_o)
    assert np.array_equal(mu_e.view(np.uint64), mu_o.view(np.uint64)), "mu differs bitwise"
    assert np.array_equal(S_e.view(np.uint64), S_o.view(np.uint64)), "Sigma differs bitwise"
    survivors = [c for i, c in enumerate(was) if i not in set(removed)]
    return [i for i, (a, c) in enumerate(zip(survivors, cod_o)) if c and not a]   # new indices of the converted features


def test_removals_interleaved_with_conversions(emu, base):
    pkg, orc, sc, o = base
    # converts 1, 3, 7, 10 (4 is shrunk too but removed); removes 2, 4, 5, 8 between them
    conv = _compare(emu, pkg, orc, sc, o, shrink=(1, 3, 4, 7, 10), removed=(2, 4, 5, 8))
    assert conv == [1, 2, 4, 6]


def test_removal_of_a_converted_feature(emu, base):
    pkg, orc, sc, o = base
    first = _clone(pkg, orc, sc, o, shrink=(0, 6, 9))
    first.convert2XYZ_ifLinearAll()
    assert [first.feature(i).coding for i in (0, 6, 9)] == [1, 1, 1]
    # removes XYZ features 6 and 0 and inverse-depth feature 3; converts 2, 5 and 11
    conv = _compare(emu, pkg, orc, sc, first, shrink=(2, 5, 11), removed=(0, 3, 6))
    assert conv == [1, 3, 8]


def test_converted_feature_is_the_last(emu, base):
    pkg, orc, sc, o = base
    conv = _compare(emu, pkg, orc, sc, o, shrink=(0, 11), removed=(5,))
    assert conv == [0, 10]
    conv = _compare(emu, pkg, orc, sc, o, shrink=(11,), removed=(10,))   # the feature before it is removed
    assert conv == [10]


def test_only_removals_and_only_conversions(emu, base):
    pkg, orc, sc, o = base
    assert _compare(emu, pkg, orc, sc, o, shrink=(), removed=(0, 4, 11)) == []
    assert _compare(emu, pkg, orc, sc, o, shrink=tuple(range(12)), removed=()) == list(range(12))
