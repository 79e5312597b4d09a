"""The dense kernels of the stacked EKF update, one at a time, against scipy / numpy in fp64 (tests/update_kernels.cu runs each
launch wrapper on host arrays).

End to end, a kernel only meets the shapes the scenes happen to produce and well-conditioned innovation blocks; here each one
meets the partial blocks, row offsets, odd sizes, K values and conditioning where blocked kernels go wrong:

* the block factor — cta_chol128 (default), cta_chol_panel<128> (EKF_CHOL_SMEM=1), the flag-waiting launch, and the batched
  filter's cta_chol_panel<64> — on random SPD matrices of condition 1 .. 1e12 and on innovation blocks of a synthetic scene;
* the blocked triangular solve k_blk_V, in place and out of place;
* the downdate GEMM k_gemm_nt_sub in both tile variants: square (both triangle modes), correction and row-block shapes, K
  through kconst and kdev, and the tile-list grid;
* k_blk_Sg and k_delta_rows.

Integer-valued operands, where every partial sum is exact, must give the exact result; real operands must meet an error bound.
Every buffer region a kernel must not write is filled with a NaN canary and checked bit for bit afterwards."""
import ctypes
import glob
import importlib
import os
import shutil
import subprocess

import numpy as np
import pytest
import scipy.linalg as sla

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "ekf-monoslam_for_3d-reconstruction_b200", "csrc")
SRC = os.path.join(HERE, "update_kernels.cu")
OUT = os.path.join(HERE, "_build", "libupdate_kernels.so")
EPS = np.finfo(np.float64).eps
CANARY = np.uint64(0x7FF4DEADBEEFCAFE)   # a NaN: a kernel that reads it spreads NaN, one that writes over it is seen bit for bit
UB = 128                                  # rows of one update block (EKF_UB)

dp = ctypes.POINTER(ctypes.c_double)


def build_harness():
    """nvcc with the product's flags: the harness (which compiles csrc/ekf_gemm.cu into itself) and csrc/ekf_update.cu, into
    tests/_build/.  Rebuilt when a source or header is newer than the library."""
    pkg_build = importlib.import_module("ekf_b200.build")
    nvcc = pkg_build._nvcc()
    deps = [SRC] + glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h"))
    if os.path.exists(OUT) and all(os.path.getmtime(d) <= os.path.getmtime(OUT) for d in deps):
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    tmp = OUT + f".{os.getpid()}.tmp"
    subprocess.run([nvcc] + pkg_build.NVCC_FLAGS + ["-shared", "-I", CSRC, "-I", os.path.join(ROOT, "include"), SRC,
                                                   os.path.join(CSRC, "ekf_update.cu"), "-o", tmp], check=True)
    os.replace(tmp, OUT)
    return OUT


def test_harness_builds_for_sm100a(pkg):
    """CPU: the harness and the update kernels compile for sm_100a and export every entry point."""
    path = build_harness()
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(importlib.import_module("ekf_b200.build")._nvcc()), "cuobjdump")
    elf = subprocess.run([cuobjdump, "--list-elf", path], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in elf, elf
    lib = ctypes.CDLL(path)
    for name in ("uk_init", "uk_factor128", "uk_factor64", "uk_blk_V", "uk_gemm", "uk_blk_Sg", "uk_delta_rows"):
        assert hasattr(lib, name), name


@pytest.fixture(scope="module")
def uk(pkg):
    lib = ctypes.CDLL(build_harness())
    i, ll = ctypes.c_int, ctypes.c_longlong
    lib.uk_factor128.argtypes = [i, dp, dp, dp, dp, dp, ctypes.POINTER(i)]
    lib.uk_factor64.argtypes = [dp, i, dp, dp, i, i, dp, i, dp, ctypes.POINTER(i)]
    lib.uk_blk_V.argtypes = [dp, i, i, i, dp, dp, dp, dp, dp, dp]
    lib.uk_gemm.argtypes = [i, dp, ll, i, ll, dp, ll, i, ll, dp, ll, i, i, i, i, i, i, ctypes.POINTER(ctypes.c_ushort), i, i,
                            ctypes.POINTER(ctypes.c_uint)]
    lib.uk_blk_Sg.argtypes = [dp, dp]
    lib.uk_delta_rows.argtypes = [dp, i, dp, dp, i]
    assert lib.uk_init() == 0
    return lib


# ---- helpers -----------------------------------------------------------------------------------------------------------------
def _p(a):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags.c_contiguous
    return a.ctypes.data_as(dp)


def canary(shape):
    return np.full(shape, CANARY, dtype=np.uint64).view(np.float64)


def is_canary(a):
    return np.asarray(a).view(np.uint64) == CANARY


def bits(a):
    a = np.asarray(a, dtype=np.float64)
    return np.where(a == 0, 0.0, a).view(np.uint64)   # -0 and +0 compare equal; NaN payloads are kept


def assert_exact(got, ref, what):
    bad = bits(got) != bits(ref)
    assert not bad.any(), f"{what}: {int(bad.sum())} entries differ, first at {np.argwhere(bad)[0]}: {got[bad][0]!r} vs {ref[bad][0]!r}"


def spd(rng, k, cond):
    """k x k symmetric positive definite, eigenvalues log-spaced from 1 down to 1 / cond, random eigenvectors."""
    Q, _ = np.linalg.qr(rng.standard_normal((k, k)))
    lam = np.logspace(0.0, -np.log10(cond), k) if k > 1 else np.ones(1)
    S = (Q * lam) @ Q.T
    return 0.5 * (S + S.T)


def padded_block(Sk, nuk, nb=UB):
    """The block as k_blk_S pads a partial one: live rows first, identity (and nu = 0) after them."""
    k = Sk.shape[0]
    S = np.eye(nb); S[:k, :k] = Sk
    nu = np.zeros(nb); nu[:k] = nuk
    return S, nu


# ---- factor ------------------------------------------------------------------------------------------------------------------
FACTORS = ["chol128", "chol128_wait", "panel128", "panel64"]


@pytest.fixture
def factor(uk, monkeypatch):
    """factor(impl, S, nu) -> (rc, L, D, y, chol_fail, S buffer after the call).  The strict upper triangle of S holds the canary:
    only the lower triangle may be read."""
    def run(impl, S, nu):
        nb = S.shape[0]
        fail = ctypes.c_int(-1)
        if impl == "panel64":
            assert nb == 64
            lds, ldd = 64 + 4, 36                      # the batched filter's strides (BLDW, BLDD)
            Sbuf = canary((64, lds)); Sbuf[:, :64] = np.where(np.tril(np.ones((64, 64), bool)), S, canary((64, 64)))
            D = canary((2, 32, ldd)); y = canary(64)
            rc = uk.uk_factor64(_p(Sbuf), lds, _p(np.ascontiguousarray(nu)), None, 0, 1, _p(D), ldd, _p(y), ctypes.byref(fail))
            assert is_canary(Sbuf[:, 64:]).all() and is_canary(D[:, :, 32:]).all(), "row padding of L or D written"
            return rc, Sbuf[:, :64].copy(), D[:, :, :32].copy(), y, fail.value, Sbuf
        assert nb == UB
        monkeypatch.setenv("EKF_CHOL_SMEM", "1" if impl == "panel128" else "0")
        assert uk.uk_init() == 0
        Sbuf = np.where(np.tril(np.ones((nb, nb), bool)), S, canary((nb, nb)))
        L = canary((nb, nb)); D = canary((4, 32, 32)); y = canary(nb)
        rc = uk.uk_factor128(1 if impl == "chol128_wait" else 0, _p(Sbuf), _p(np.ascontiguousarray(nu)), _p(L), _p(D), _p(y),
                             ctypes.byref(fail))
        return rc, L, D, y, fail.value, Sbuf
    yield run
    monkeypatch.delenv("EKF_CHOL_SMEM", raising=False)
    assert uk.uk_init() == 0


def check_factor(impl, S, nu, k, out, ctx):
    """The factor of a block whose first k rows are live (identity after them) against LAPACK."""
    rc, L, D, y, fail, _ = out
    nb = S.shape[0]
    assert rc == 0, f"{ctx}: CUDA error {rc}"
    assert fail == 0, f"{ctx}: chol_fail {fail}"
    # what the factor writes above the diagonal: zeros (cta_chol_panel), or zeros inside the 8 x 8 diagonal tiles and nothing
    # outside them (cta_chol128)
    iu = np.triu_indices(nb, 1)
    if impl.startswith("chol128"):
        same_tile = (iu[0] // 8) == (iu[1] // 8)
        assert (L[iu][same_tile] == 0).all(), f"{ctx}: L above the diagonal inside a diagonal tile"
        assert is_canary(L[iu][~same_tile]).all(), f"{ctx}: L written above the diagonal tiles"
    else:
        assert (L[iu] == 0).all(), f"{ctx}: L above the diagonal"
    # the padded rows: exactly identity, y = nu = 0 there
    assert_exact(L[k:, :k], np.zeros((nb - k, k)), f"{ctx}: L of the padding rows")
    assert (np.abs(np.tril(L)[k:, k:] - np.eye(nb - k)) <= 4 * EPS).all(), f"{ctx}: L of the padding block"

    assert_exact(y[k:], nu[k:], f"{ctx}: y of the padding rows")
    Lk = np.tril(L[:k, :k]); Sk = S[:k, :k]
    kappa = np.linalg.cond(Sk)
    back = np.linalg.norm(Lk @ Lk.T - Sk) / np.linalg.norm(Sk)
    assert back <= 2 * nb * EPS, f"{ctx}: backward error {back:.2e} (cond {kappa:.1e})"
    Lref = sla.cholesky(Sk, lower=True)
    fwd = np.linalg.norm(Lk - Lref) / np.linalg.norm(Lref)
    assert fwd <= 2 * nb * EPS * kappa, f"{ctx}: |L - L_lapack| / |L| = {fwd:.2e} (cond {kappa:.1e})"
    Lfull = np.tril(L)
    for J in range(nb // 32):
        LJ = Lfull[32 * J:32 * J + 32, 32 * J:32 * J + 32]
        DJ = D[J]
        assert_exact(np.triu(DJ, 1), np.zeros((32, 32)), f"{ctx}: D_{J} above the diagonal")
        res = np.abs(DJ @ LJ - np.eye(32)).max()
        assert res <= 2 * 32 * EPS * np.linalg.cond(LJ), f"{ctx}: |D_{J} L_{J}{J} - I| = {res:.2e}"
    yref = sla.solve_triangular(Lfull, nu, lower=True)
    ey = np.linalg.norm(y - yref) / max(np.linalg.norm(yref), 1e-300)
    assert ey <= 2 * nb * EPS * np.linalg.cond(Lfull), f"{ctx}: y = L^-1 nu off by {ey:.2e}"
    return back, fwd


KS = [2, 4, 6, 8, 10, 30, 32, 34, 62, 64, 66, 96, 126, 128]


@pytest.mark.gpu
@pytest.mark.parametrize("impl", FACTORS)
@pytest.mark.parametrize("cond", [1e0, 1e6, 1e12])
def test_factor_random_spd(factor, impl, cond):
    nb = 64 if impl == "panel64" else UB
    rng = np.random.default_rng(int(np.log10(cond)) * 131 + len(impl))
    worst = 0.0
    for k in [k for k in KS if k <= nb]:
        S, nu = padded_block(spd(rng, k, cond), rng.standard_normal(k), nb)
        back, fwd = check_factor(impl, S, nu, k, factor(impl, S, nu), f"{impl} cond {cond:.0e} k {k}")
        worst = max(worst, back)
    print(f"factor {impl} cond {cond:.0e}: worst backward error {worst:.2e} ({worst / EPS:.1f} eps)")


@pytest.fixture(scope="module")
def innovation_blocks(pkg, orc):
    """Innovation blocks of a 200-feature scene (n = 1214) after predict and match of frame 1 on the oracle: block 0 of
    S = H Sigma H^T + sigma^2 I, and the Schur complement that the last block (3, partial) sees after blocks 0 .. 2, with
    the nu it sees.  Returns [(name, S_k, nu_k)].  (The oracle seeds a 500-feature map in minutes; 200 is enough for four
    blocks.)"""
    from helpers import _feature_rows, make_oracle, seed_features
    sc = pkg.synth.Scene(n_features=200, n_frames=3, seed=6)
    o = make_oracle(pkg, orc, sc, omp=True)
    seed_features(o, sc)
    o.captureNewFrame(sc.frame(1), sc.stamps[1]); o.predict()
    assert o.match() > 3 * UB // 2
    mu, Sig = o.get_full()
    feats = [o.feature(i) for i in range(o.numOfFeatures())]
    sel = [i for i, f in enumerate(feats) if f.is_in_innovation]
    idx, Hc, nu = _feature_rows(feats, sel)
    H = np.zeros((2 * len(sel), mu.size))
    for j in range(len(sel)):
        np.add.at(H[2 * j:2 * j + 2].T, idx[j], Hc[j].T)   # unused columns of an XYZ feature are zero and point at index 0
    St = H @ Sig @ H.T + 4.0 * np.eye(H.shape[0])
    St = 0.5 * (St + St.T)
    out = [("block 0", St[:UB, :UB], nu[:UB])]
    b0, b1 = 3 * UB, min(4 * UB, St.shape[0])
    A, Bm = St[:b0, :b0], St[:b0, b0:b1]
    X = sla.cho_solve(sla.cho_factor(A, lower=True), np.column_stack([Bm, nu[:b0]]))
    Sc = St[b0:b1, b0:b1] - Bm.T @ X[:, :-1]
    out.append(("block 3 Schur complement", 0.5 * (Sc + Sc.T), nu[b0:b1] - Bm.T @ X[:, -1]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("impl", FACTORS)
def test_factor_innovation_blocks(factor, innovation_blocks, impl):
    nb = 64 if impl == "panel64" else UB
    for name, Sk, nuk in innovation_blocks:
        k = min(nb, Sk.shape[0])
        S, nu = padded_block(Sk[:k, :k], nuk[:k], nb)
        back, fwd = check_factor(impl, S, nu, k, factor(impl, S, nu), f"{impl} {name}")
        print(f"factor {impl} {name} (k {k}, cond {np.linalg.cond(Sk[:k, :k]):.1e}): backward {back:.2e}, |L - L_lapack| {fwd:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("impl", FACTORS)
def test_factor_indefinite_sets_flag(factor, impl):
    """One negative pivot: chol_fail is raised and the kernel returns normally."""
    nb = 64 if impl == "panel64" else UB
    row = 77 if nb == UB else 37
    rng = np.random.default_rng(77)
    L0 = np.eye(nb) + np.tril(rng.uniform(-0.2, 0.2, (nb, nb)), -1) / np.sqrt(nb)
    d = np.ones(nb); d[row] = -1.0
    S = (L0 * d) @ L0.T
    S = 0.5 * (S + S.T)
    assert (np.linalg.eigvalsh(S) < 0).sum() == 1
    rc, L, D, y, fail, _ = factor(impl, S, rng.standard_normal(nb))
    assert rc == 0
    assert fail != 0
    Lk = np.tril(L[:row, :row])                         # the rows before the bad pivot are still right
    assert np.abs(Lk @ Lk.T - S[:row, :row]).max() < 1e-12


# ---- blocked triangular solve (k_blk_V) ---------------------------------------------------------------------------------------
def _solve_operands(rng, cond=1e4):
    L = np.linalg.cholesky(spd(rng, UB, cond))
    D = np.stack([np.tril(sla.solve_triangular(L[32 * J:32 * J + 32, 32 * J:32 * J + 32], np.eye(32), lower=True))
                  for J in range(UB // 32)])
    L_in = np.where(np.tril(np.ones((UB, UB), bool)), L, canary((UB, UB)))   # above the diagonal: not read
    return L, L_in, np.ascontiguousarray(D), rng.standard_normal(UB)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["inplace", "inplace_delta_in", "vout", "vout_delta_in", "no_delta"])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 914, 3014])
@pytest.mark.parametrize("rbase", [0, 7, 457])
def test_blk_V(uk, n, rbase, mode):
    if rbase >= n:
        pytest.skip("empty row range")
    rng = np.random.default_rng(n * 7 + rbase)
    L, L_in, D, y = _solve_operands(rng)
    rows = n + 5
    W = canary((rows, UB)); W[:n] = rng.standard_normal((n, UB))
    W0 = W.copy()
    delta = None if mode == "no_delta" else canary(rows)
    if delta is not None:
        delta[:n] = rng.standard_normal(n)
    delta0 = None if delta is None else delta.copy()
    din = None
    if mode.endswith("delta_in"):
        din = canary(rows); din[:n] = rng.standard_normal(n)
    Vout = canary((rows, UB)) if mode.startswith("vout") else None
    rc = uk.uk_blk_V(_p(W), rows, rbase, n, _p(L_in), _p(D), _p(y), _p(delta), _p(Vout), _p(din))
    assert rc == 0
    V = Vout if Vout is not None else W
    r = slice(rbase, n)
    Vref = sla.solve_triangular(L, W0[r].T, lower=True).T
    kappa = np.linalg.cond(L)
    err = np.linalg.norm(V[r] - Vref, axis=1) / np.linalg.norm(Vref, axis=1)
    assert err.max() <= 2 * UB * EPS * kappa, f"row {rbase + err.argmax()}: {err.max():.2e}"
    # rows outside [rbase, n) of every output untouched; W untouched when V goes to Vout
    assert_exact(W[:rbase], W0[:rbase], "W rows before rbase")
    assert is_canary(W[n:]).all()
    if Vout is not None:
        assert_exact(W, W0, "W with Vout")
        assert is_canary(Vout[:rbase]).all() and is_canary(Vout[n:]).all()
    if delta is not None:
        base = (din if din is not None else delta0)[r]
        dref = base + Vref @ y
        bound = 2 * UB * EPS * kappa * (np.abs(Vref) @ np.abs(y)) + 2 * EPS * np.abs(base)
        assert (np.abs(delta[r] - dref) <= bound).all()
        assert_exact(delta[:rbase], delta0[:rbase], "delta before rbase")
        assert is_canary(delta[n:]).all()


# ---- downdate GEMM (k_gemm_nt_sub) -------------------------------------------------------------------------------------------
def gemm(uk, tm, C, ldc, c_off, A, B, M, N, K, kdev, lower_only, tlist=None, n_hot=0):
    """C (flat, ldc) at row offset c_off -= A[c_off ..] B^T.  A, B: rows x 128 (K contiguous)."""
    hc = ctypes.c_uint(0xFFFFFFFF)
    tl = None
    if tlist is not None:
        tlist = np.ascontiguousarray(tlist, dtype=np.uint16)
        tl = tlist.ctypes.data_as(ctypes.POINTER(ctypes.c_ushort))
    rc = uk.uk_gemm(tm, _p(C), C.size, ldc, c_off * ldc, _p(A), A.size, UB, c_off * UB, _p(B), B.size, UB, M, N, K, int(kdev),
                    int(lower_only), tl, 0 if tlist is None else len(tlist), n_hot, ctypes.byref(hc))
    return rc, hc.value


def gemm_operands(rng, rows_a, rows_b, K, integer, same=False):
    """A (rows_a x 128) and B (rows_b x 128) with the canary past column K and in three extra rows."""
    def one(rows):
        X = canary((rows + 3, UB))
        X[:rows, :K] = rng.integers(-8, 9, (rows, K)) if integer else rng.standard_normal((rows, K))
        return X
    A = one(rows_a)
    return A, (A if same else one(rows_b))


def gemm_bound(A, B, C, K):
    return 2 * K * EPS * (np.abs(A) @ np.abs(B).T + np.abs(C)) + np.finfo(np.float64).tiny


@pytest.mark.gpu
@pytest.mark.parametrize("tm", [64, 128])
@pytest.mark.parametrize("K,kdev", [(128, False), (128, True), (126, False), (126, True), (2, False), (2, True)])
@pytest.mark.parametrize("lower_only", [0, 1])
@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 128, 129, 191, 914, 3014])
def test_gemm_square(uk, n, lower_only, K, kdev, tm):
    """Sigma <- Sigma - V V^T: M = N = n, ldc rounded up to 8 as in the handle."""
    ldc = -(-n // 8) * 8
    kinds = ["int", "real"] if K == 128 and not kdev else ["int"]
    for kind in kinds:
        rng = np.random.default_rng(n * 1000 + K * 10 + lower_only + 5 * (tm == 128))
        integer = kind == "int"
        A, B = gemm_operands(rng, n, n, K, integer, same=bool(lower_only))
        Cm = rng.integers(-2 ** 20, 2 ** 20, (n, n)).astype(np.float64) if integer else rng.standard_normal((n, n))
        if lower_only:
            Cm = np.tril(Cm) + np.tril(Cm, -1).T
        C = canary((n + 3, ldc)); C[:n, :n] = Cm
        rc, _ = gemm(uk, tm, C, ldc, 0, A, B, n, n, K, kdev, lower_only)
        assert rc == 0
        a, b = A[:n, :K], B[:n, :K]
        R = Cm - a @ b.T
        if lower_only:
            R = np.tril(R) + np.tril(R, -1).T
        got = C[:n, :n]
        ctx = f"n {n} K {K} kdev {kdev} lower_only {lower_only} tm {tm} {kind}"
        if integer:
            assert_exact(got, R, ctx)
        else:
            assert (np.abs(got - R) <= gemm_bound(a, b, Cm, K)).all(), ctx
        if lower_only:
            iu = np.triu_indices(n, 1)
            assert_exact(got[iu], got.T[iu], f"{ctx}: upper triangle is not the mirror of the lower")
        assert is_canary(C[:, n:]).all(), f"{ctx}: padding columns written"
        assert is_canary(C[n:]).all(), f"{ctx}: rows past M written"


@pytest.mark.gpu
@pytest.mark.parametrize("tm", [64, 128])
@pytest.mark.parametrize("n", [129, 914, 3014])
def test_gemm_correction_shape(uk, n, tm):
    """cor -= V G^T: M = n, N = 128 (the correction of the next block's panel)."""
    rng = np.random.default_rng(n + tm)
    for integer in (True, False):
        A, B = gemm_operands(rng, n, UB, UB, integer)
        Cm = rng.integers(-2 ** 20, 2 ** 20, (n, UB)).astype(np.float64) if integer else rng.standard_normal((n, UB))
        C = canary((n + 3, UB)); C[:n] = Cm
        rc, _ = gemm(uk, tm, C, UB, 0, A, B, n, UB, UB, False, 0)
        assert rc == 0
        R = Cm - A[:n] @ B[:UB].T
        if integer:
            assert_exact(C[:n], R, f"n {n} tm {tm}")
        else:
            assert (np.abs(C[:n] - R) <= gemm_bound(A[:n], B[:UB], Cm, UB)).all()
        assert is_canary(C[n:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("tm", [64, 128])
@pytest.mark.parametrize("kdev", [False, True])
@pytest.mark.parametrize("n,r0,M", [(914, 0, 457), (914, 457, 457), (3014, 457, 1005), (3014, 2950, 64)])
def test_gemm_row_block(uk, n, r0, M, kdev, tm):
    """The row-block downdate of the row-partitioned update: rows [r0, r0 + M) of Sigma, C and A offset by r0, all n columns,
    both triangles (lower_only 0).  Rows outside the block stay as they were."""
    ldc = -(-n // 8) * 8
    rng = np.random.default_rng(n + r0 + M + tm)
    for integer in (True, False):
        A, _ = gemm_operands(rng, n, n, UB, integer)
        Cm = rng.integers(-2 ** 20, 2 ** 20, (n, n)).astype(np.float64) if integer else rng.standard_normal((n, n))
        C = canary((n + 3, ldc)); C[:n, :n] = Cm
        C0 = C.copy()
        rc, _ = gemm(uk, tm, C, ldc, r0, A, A, M, n, UB, kdev, 0)
        assert rc == 0
        rb = slice(r0, r0 + M)
        R = Cm[rb] - A[rb] @ A[:n].T
        if integer:
            assert_exact(C[rb, :n], R, f"n {n} r0 {r0} M {M}")
        else:
            assert (np.abs(C[rb, :n] - R) <= gemm_bound(A[rb], A[:n], Cm[rb], UB)).all()
        assert_exact(C[:r0], C0[:r0], "rows before the block")
        assert_exact(C[r0 + M:], C0[r0 + M:], "rows after the block")
        assert is_canary(C[:, n:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [129, 914, 3014])
def test_gemm_tile_list(uk, n):
    """The 1-D grid over a shuffled list of all lower 64 x 64 tiles gives bitwise the 2-D grid's result, and the CTAs of the first
    n_hot list entries bump hot_counter exactly n_hot times.  The product wrapper rejects a list for a non-square shape."""
    rng = np.random.default_rng(n)
    T = -(-n // 64)
    tiles = np.array([(i, j) for i in range(T) for j in range(i + 1)], dtype=np.uint16)
    tiles = tiles[rng.permutation(len(tiles))]
    n_hot = max(1, len(tiles) // 3)
    ldc = -(-n // 8) * 8
    A, _ = gemm_operands(rng, n, n, UB, False)
    Cm = rng.standard_normal((n, n)); Cm = np.tril(Cm) + np.tril(Cm, -1).T
    C1 = canary((n + 3, ldc)); C1[:n, :n] = Cm
    C2 = C1.copy()
    rc, _ = gemm(uk, 64, C1, ldc, 0, A, A, n, n, UB, False, 1)
    assert rc == 0
    rc, hot = gemm(uk, 0, C2, ldc, 0, A, A, n, n, UB, True, 1, tlist=tiles, n_hot=n_hot)
    assert rc == 0
    assert_exact(C2, C1, "tile list vs 2-D grid")
    assert hot == n_hot
    rc, _ = gemm(uk, 0, C1.copy(), ldc, 0, A, A, n - 1, n, UB, False, 1, tlist=tiles, n_hot=n_hot)
    assert rc == 1   # cudaErrorInvalidValue


# ---- k_blk_Sg and k_delta_rows ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("integer", [True, False])
def test_blk_Sg(uk, integer):
    """Sg = -G G^T on the lower 32 x 32 blocks; the blocks above the diagonal are not written."""
    rng = np.random.default_rng(3)
    G = rng.integers(-64, 65, (UB, UB)).astype(np.float64) if integer else rng.standard_normal((UB, UB))
    Sg = canary((UB, UB))
    assert uk.uk_blk_Sg(_p(G), _p(Sg)) == 0
    R = -G @ G.T
    blk = np.arange(UB) // 32
    low = blk[:, None] >= blk[None, :]
    if integer:
        assert_exact(Sg[low], R[low], "Sg")
    else:
        assert (np.abs(Sg[low] - R[low]) <= (2 * UB * EPS * (np.abs(G) @ np.abs(G).T))[low]).all()
    assert is_canary(Sg[~low]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("integer", [True, False])
@pytest.mark.parametrize("n", [1, 7, 8, 9, 914, 3014])
def test_delta_rows(uk, n, integer):
    """delta[i] += V[i, :] y for every row i < n; rows past n untouched."""
    rng = np.random.default_rng(n)
    rows = n + 3
    V = canary((rows, UB))
    V[:n] = rng.integers(-1000, 1001, (n, UB)) if integer else rng.standard_normal((n, UB))
    y = rng.integers(-1000, 1001, UB).astype(np.float64) if integer else rng.standard_normal(UB)
    d = canary(rows); d[:n] = rng.integers(-2 ** 30, 2 ** 30, n) if integer else rng.standard_normal(n)
    d0 = d[:n].copy()
    assert uk.uk_delta_rows(_p(V), rows, _p(y), _p(d), n) == 0
    R = d0 + V[:n] @ y
    if integer:
        assert_exact(d[:n], R, "delta")
    else:
        assert (np.abs(d[:n] - R) <= 2 * UB * EPS * (np.abs(V[:n]) @ np.abs(y) + np.abs(d0))).all()
    assert is_canary(d[n:]).all()
