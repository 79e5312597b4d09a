"""CPU: the batched map export (k_batch_points_features) and archive record (k_batch_compact) assemble exactly the oracle's rows.

tests/batch_points_emu.cu runs the export flow of one filter on the host with the same __host__ __device__ functions the kernels
call (csrc/ekf_points.cuh).  Here it is fed synthetic feature tables and archives and compared bit for bit with a numpy
restatement of oracle/ekf_oracle.hpp's getPointsFeatures and removeFeature: empty maps, inverse-depth-only maps, archived
real_indices above the live maximum (dropped), archived rows over live rows, and the clear rule at 7000 and 7001 records,
which a GPU test cannot practically reach."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "ekf-monoslam_for_3d-reconstruction_b200", "csrc")


@pytest.fixture(scope="module")
def emu():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = os.path.join(HERE, "_build", "libbatch_points_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(HERE, "batch_points_emu.cu")
    deps = [src, os.path.join(CSRC, "ekf_points.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "--fmad=false", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-Xcompiler", "-ffp-contract=off", "-shared", "-I", CSRC, src, "-o", out], check=True)
    return ctypes.CDLL(out)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def oracle_points(coding, pos, real_index, mu, S, archive):
    """ekf_oracle.hpp::getPointsFeatures restated: returns (matrix, cleared)."""
    psize = int(real_index[-1]) if len(real_index) else 0
    P = np.zeros((psize + 1, 12))
    map_scale = mu[13]
    for c, p, r in zip(coding, pos, real_index):
        if not c:
            continue
        row = np.zeros(12)
        for i2 in range(9):
            row[3 + i2] = S[p + i2 // 3, p + i2 % 3]
        for k in range(3):
            row[k] = mu[p + k] * map_scale
        P[r] = row
    for r, rec in archive:
        if r > psize:
            continue
        P[r, 3:] = rec[3:]
        for k in range(3):
            P[r, k] = rec[k] * map_scale
    return P, len(archive) > 7000


def oracle_record(mu, S, p):
    """ekf_oracle.hpp::removeFeature's XYZ_pos and cov_4_delete, as one 12-double record."""
    rec = np.zeros(12)
    rec[:3] = mu[p:p + 3]
    for c in range(3):
        for r in range(3):
            rec[3 + c * 3 + r] = S[p + c, p + r]
    return rec


def _table(rng, N, xyz_frac, gap=3):
    coding = (rng.random(N) < xyz_frac).astype(np.int32)
    pos, n = [], 14
    for c in coding:
        pos.append(n); n += 3 if c else 6
    real = np.cumsum(rng.integers(1, gap + 1, size=N)).astype(np.int32) - 1 if N else np.zeros(0, np.int32)
    mu = rng.normal(size=n); mu[13] = rng.uniform(0.5, 3.0)
    A = rng.normal(size=(n, n))
    S = np.ascontiguousarray(A @ A.T)
    return coding, np.array(pos, dtype=np.int32), real, mu, S


def _run(emu, coding, pos, real, mu, S, archive, rows_cap=None):
    N = len(coding)
    ari = np.array([r for r, _ in archive] or [0], dtype=np.int32)
    arec = np.ascontiguousarray(np.array([rec for _, rec in archive] or [np.zeros(12)], dtype=np.float64))
    rows_cap = rows_cap or (int(real[-1]) + 1 if N else 1)
    out = np.full((rows_cap, 12), np.nan)
    clears = ctypes.c_int(-1)
    coding = np.ascontiguousarray(coding, np.int32); pos = np.ascontiguousarray(pos, np.int32)
    real = np.ascontiguousarray(real, np.int32); mu = np.ascontiguousarray(mu); S = np.ascontiguousarray(S)
    rows = emu.emu_points(N, _p(coding), _p(pos), _p(real), _p(mu), _p(S), S.shape[1], len(archive), _p(ari), _p(arec), _p(out),
                          rows_cap, ctypes.byref(clears))
    return rows, out, clears.value


def _archive(rng, ris):
    return [(int(r), rng.normal(size=12)) for r in ris]


@pytest.mark.parametrize("case", ["empty", "empty_with_archive", "inverse_depth_only", "mixed", "above_live_max", "over_live",
                                  "duplicates"])
def test_rows_equal_oracle(emu, case):
    rng = np.random.default_rng(sum(map(ord, case)))
    N = {"empty": 0, "empty_with_archive": 0}.get(case, 24)
    frac = 0.0 if case == "inverse_depth_only" else 0.5
    coding, pos, real, mu, S = _table(rng, N, frac)
    if N == 0:
        mu = rng.normal(size=14); S = np.eye(14)
    top = int(real[-1]) if N else 0
    if case in ("empty", "inverse_depth_only"):
        archive = []
    elif case == "empty_with_archive":
        archive = _archive(rng, [0, 3, 1])            # psize 0: only real_index 0 has a row
    elif case == "above_live_max":
        archive = _archive(rng, [top + 1, 2, top + 5, top, 0])
    elif case == "over_live":                         # records on rows of live XYZ features and on inverse-depth rows
        archive = _archive(rng, list(real[:: 3]))
    elif case == "duplicates":                        # the later record wins
        archive = _archive(rng, [4, 7, 4, 9, 7, 4])
    else:
        gaps = sorted(set(range(top)) - set(real.tolist()))
        archive = _archive(rng, rng.choice(gaps, size=min(8, len(gaps)), replace=False))
    want, cleared = oracle_points(coding, pos, real, mu, S, archive)
    rows, got, clears = _run(emu, coding, pos, real, mu, S, archive)
    assert rows == want.shape[0] and clears == int(cleared)
    assert np.array_equal(got[:rows], want), case
    if case == "inverse_depth_only":
        assert not got.any()
    if case == "above_live_max":
        assert rows == top + 1


def test_rows_past_the_count_are_zero_and_small_cap_writes_nothing(emu):
    rng = np.random.default_rng(5)
    coding, pos, real, mu, S = _table(rng, 10, 0.6)
    rows, got, _ = _run(emu, coding, pos, real, mu, S, _archive(rng, [1]), rows_cap=int(real[-1]) + 9)
    assert rows == real[-1] + 1 and not got[rows:].any()
    rows, got, _ = _run(emu, coding, pos, real, mu, S, [], rows_cap=int(real[-1]))
    assert rows == real[-1] + 1 and np.isnan(got).all()


@pytest.mark.parametrize("held,clears", [(0, 0), (7000, 0), (7001, 1)])
def test_clear_rule(emu, held, clears):
    rng = np.random.default_rng(held)
    coding, pos, real, mu, S = _table(rng, 30, 0.5, gap=400)
    archive = _archive(rng, rng.integers(0, int(real[-1]) + 60, size=held))
    want, cleared = oracle_points(coding, pos, real, mu, S, archive)
    rows, got, c = _run(emu, coding, pos, real, mu, S, archive)
    assert c == clears == int(cleared)
    assert np.array_equal(got[:rows], want)


def test_record_and_rule_equal_remove_feature(emu):
    rng = np.random.default_rng(9)
    coding, pos, real, mu, S = _table(rng, 12, 0.5)
    for p in pos:
        rec = np.zeros(12)
        emu.emu_record(_p(mu), _p(S), S.shape[1], int(p), _p(rec))
        assert np.array_equal(rec, oracle_record(mu, S, int(p)))
    for c in (0, 1):
        for nf in range(0, 9):
            assert emu.emu_archived(c, nf) == int(c == 1 and nf > 5)
