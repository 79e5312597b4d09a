"""CPU: the batched motion-blur kernel's form gives exactly the single filter's blurred templates.

k_predict_blur (single filter) rasterises evaluateKernel's line into a bit mask and has every output pixel walk all
krows x kcols bits; k_batch_predict_blur keeps each distinct line point once, orders the points by (row, column) with
blur_rank and has every pixel walk that list.  tests/batch_blur_emu.cu runs both on the host from the same __host__
__device__ functions the kernels call (csrc/ekf_blur.cuh).  Here both are compared, bit for bit, with each other and with
a numpy restatement of evaluateKernel + filter2D in its direct form (libblur.cpp:17-81: a line of ones, normalised by its
sum, correlated with the template around the kernel centre, BORDER_REFLECT_101, round half to even, saturate to u8), over
random templates, every window the batch runs, displacements in all four quadrants, along the axes, near the diagonal,
below a pixel and up to the 256 x 256 cap.  Host trigonometry may differ from the device's in the last ulp, so the line
parameters the numpy side uses come from the shared code; the GPU tests pin the device against the single filter."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "ekf-monoslam_for_3d-reconstruction_b200", "csrc")
MAXPTS = 384
WINDOWS = (3, 11, 21, 30, 31)


@pytest.fixture(scope="module")
def emu():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = os.path.join(HERE, "_build", "libbatch_blur_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(HERE, "batch_blur_emu.cu")
    deps = [src] + [os.path.join(CSRC, f) for f in ("ekf_blur.cuh", "ekf_math.cuh", "ekf_common.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "--fmad=false", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-Xcompiler", "-ffp-contract=off", "-shared", "-I", CSRC, src, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    D, I, P = ctypes.c_double, ctypes.c_int, ctypes.c_void_p
    lib.emu_blur_decide.argtypes = [D, D, I, P, P]
    lib.emu_blur_line.argtypes = [D, D, P, P]
    lib.emu_blur_bits.argtypes = [P, I, D, D, I, I, P]
    lib.emu_blur_list.argtypes = [P, I, D, D, I, I, P, P, P]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def decide(emu, dx, dy, kmin=0):
    r, c = np.zeros(1, np.int32), np.zeros(1, np.int32)
    d = emu.emu_blur_decide(dx, dy, kmin, _p(r), _p(c))
    return d, int(r[0]), int(c[0])


def _reflect101(i, n):
    while i < 0 or i >= n:
        i = -i if i < 0 else 2 * n - 2 - i
    return i


def numpy_blur(emu, src, dx, dy, krows, kcols):
    """evaluateKernel (libblur.cpp:17-43) + blurPatch's filter2D (libblur.cpp:57-81) in direct form."""
    par, xy0 = np.zeros(3), np.zeros(2, np.int32)
    emu.emu_blur_line(dx, dy, _p(par), _p(xy0))
    s, c, length = (float(v) for v in par)
    x0, y0 = int(xy0[0]), int(xy0[1])
    kernel = np.zeros((krows, kcols))
    i = 0
    while i < length:
        x, y = int(i * s + x0), int(i * c + y0)
        if 0 <= x < krows and 0 <= y < kcols:
            kernel[x, y] = 1.0
        i += 1
    kernel = kernel / kernel.sum()
    w = src.shape[0]
    ay, ax = krows // 2, kcols // 2
    acc = np.zeros((w, w))
    for ky, kx in zip(*np.nonzero(kernel)):          # row-major: OpenCV's direct-form order
        rows = [_reflect101(y + ky - ay, w) for y in range(w)]
        cols = [_reflect101(x + kx - ax, w) for x in range(w)]
        acc = acc + kernel[ky, kx] * src[np.ix_(rows, cols)].astype(np.float64)
    return np.clip(np.rint(acc), 0, 255).astype(np.uint8), int(np.count_nonzero(kernel))


def _displacements(rng):
    fixed = [(0.3, 0.4), (-0.45, 0.2), (0.0, -0.7),                          # below a pixel
             (5.0, 0.0), (-17.0, 0.0), (0.0, 9.0), (0.0, -40.0),             # along the axes
             (12.0, 12.0), (-12.0, 12.000000001), (30.5, -30.5), (-64.0, -63.999999),  # on and near the diagonal
             (3.7, 2.2), (-3.7, 2.2), (3.7, -2.2), (-3.7, -2.2),             # the four quadrants
             (41.3, 7.9), (-7.9, 41.3), (120.2, -77.7), (-200.5, -3.25),
             (255.9, 0.5), (0.25, -255.99), (255.5, 255.5), (-255.99, 255.99)]   # up to the 256 cap
    rand = [tuple(rng.uniform(-1, 1, 2) * 10.0 ** rng.uniform(-0.5, 2.4)) for _ in range(40)]
    return fixed + rand


@pytest.mark.parametrize("w", WINDOWS)
def test_list_walk_equals_bitmask_walk_and_filter2d(emu, w):
    rng = np.random.default_rng(100 + w)
    repeats = 0
    for k, (dx, dy) in enumerate(_displacements(rng)):
        d, krows, kcols = decide(emu, dx, dy)
        assert d == 1, (dx, dy)
        src = np.ascontiguousarray(rng.integers(0, 256, (w, w)), dtype=np.uint8)
        if k % 3 == 0:   # smooth templates too: sums near x.5 after rounding
            src = np.ascontiguousarray(np.repeat(np.repeat(src[: (w + 1) // 2, : (w + 1) // 2], 2, 0), 2, 1)[:w, :w])
        a, b = np.zeros((w, w), np.uint8), np.zeros((w, w), np.uint8)
        coef, npts = np.zeros(MAXPTS, np.int32), np.zeros(1, np.int32)
        count = emu.emu_blur_bits(_p(src), w, dx, dy, krows, kcols, _p(a))
        m = emu.emu_blur_list(_p(src), w, dx, dy, krows, kcols, _p(b), _p(coef), _p(npts))
        ctx = f"w {w} displacement ({dx}, {dy}) kernel {krows} x {kcols}"
        assert m == count, f"{ctx}: {m} listed coefficients, {count} set bits"
        keys = [(int(p) >> 16, int(p) & 0xffff) for p in coef[:m]]
        assert keys == sorted(set(keys)), f"{ctx}: list not in ascending (row, column) order or not distinct"
        assert np.array_equal(a, b), f"{ctx}: list walk differs from the bit mask walk in {(a != b).sum()} pixels"
        ref, nref = numpy_blur(emu, src, dx, dy, krows, kcols)
        assert nref == count and np.array_equal(a, ref), f"{ctx}: differs from filter2D in {(a != ref).sum()} pixels"
        repeats += int(npts[0] > m)
    assert repeats >= 10, "too few lines with repeated points: de-duplication not exercised"


def test_cap_decision(emu):
    """Patch::blur's threshold and the 256 x 256 cap: kernel side = int(|d| + 1)."""
    assert decide(emu, 255.5, 0.0) == (1, 1, 256)
    assert decide(emu, 255.999, -255.999) == (1, 256, 256)
    assert decide(emu, 256.0, 0.0) == (-1, 1, 257)
    assert decide(emu, 0.0, -256.0) == (-1, 257, 1)
    assert decide(emu, -256.5, 100.0)[0] == -1
    assert decide(emu, 3.0, 4.0, kmin=5)[0] == 0      # dn = 5 is not > 5
    assert decide(emu, 3.0, 4.0001, kmin=5) == (1, 5, 4)
    assert decide(emu, 0.0, 0.0, kmin=0)[0] == 0
