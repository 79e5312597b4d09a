"""CPU: the batched corner detection finds, for every filter, exactly the corners of the single filter's pipeline.

The batched detector (csrc/ekf_batch_detect.cu) builds ONE candidate list per frame (every 3x3 local maximum of eig inside
the base mask, sorted once) and lets each filter walk it with its own mask and threshold.  tests/batch_topup_emu.cu runs
that flow on the host with the same __host__ __device__ functions the kernels call (csrc/ekf_detect.cuh).  Here it is fed
planted eigenvalue maps — equal scores, plateaus, negative values, masks that hide the global maximum — and compared with a
numpy restatement of the single filter's pipeline (csrc/ekf_detect.cu): the mask, its maximum, THRESH_TOZERO, 3x3 maxima
of the thresholded map, the (score bits << 32 | pixel) sort, the greedy 12 px selection."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "ekf-monoslam_for_3d-reconstruction_b200", "csrc")
MAXC = 32


@pytest.fixture(scope="module")
def emu():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = os.path.join(HERE, "_build", "libbatch_topup_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(HERE, "batch_topup_emu.cu")
    deps = [src, os.path.join(CSRC, "ekf_detect.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "--fmad=false", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-Xcompiler", "-ffp-contract=off", "-shared", "-I", CSRC, src, "-o", out], check=True)
    return ctypes.CDLL(out)


def _mask(H, W, centers, w):
    """vslamRansac.cpp:788-818 (as tests/test_gpu_detect.py states it)."""
    mask = np.zeros((H, W), np.uint8)
    mask[w:H - w, w:W - w] = 255
    win = 2 * w + 1
    for cx, cy in centers:
        if cx > w and cy > w and cx < W - w and cy < H - w:
            x = int(cx - win // 2) if cx - win // 2 > 0 else 0
            y = int(cy - win // 2) if cy - win // 2 > 0 else 0
            mask[y:y + win, x:x + win] = 0
    return mask


def single_filter_corners(eig, mask, num):
    """The single filter's detector after the eig map: k_det_max, k_det_candidates, k_det_select."""
    H, W = eig.shape
    m = eig[mask != 0]
    mx = np.float32(max(0.0, float(m.max()))) if m.size else np.float32(0)
    thr = np.float32(np.float64(mx) * 0.01)
    T = np.where(eig > thr, eig, np.float32(0)).astype(np.float32)
    P = np.pad(T, 1)
    nb = np.max(np.stack([P[1 + dy:1 + dy + H, 1 + dx:1 + dx + W] for dy in (-1, 0, 1) for dx in (-1, 0, 1)]), axis=0)
    cand = (T != 0) & (mask != 0) & (T == nb)
    cand[0, :] = cand[-1, :] = False
    cand[:, 0] = cand[:, -1] = False
    idx = np.flatnonzero(cand).astype(np.uint64)
    keys = (T.reshape(-1)[idx].view(np.uint32).astype(np.uint64) << np.uint64(32)) | idx
    keys = np.sort(keys)[::-1]
    acc = []
    for k in keys:
        if len(acc) >= num:
            break
        i = int(k & np.uint64(0xffffffff))
        x, y = np.float32(i % W), np.float32(i // W)
        if all((x - ax) * (x - ax) + (y - ay) * (y - ay) >= np.float32(144.0) for ax, ay in acc):
            acc.append((x, y))
    return np.array(acc, dtype=np.float32).reshape(-1, 2)


def _eig_map(rng, H, W, kind):
    if kind == "smooth":
        e = rng.normal(size=(H, W)).astype(np.float32)
        for _ in range(3):
            e = (e + np.roll(e, 1, 0) + np.roll(e, 1, 1) + np.roll(e, -1, 0) + np.roll(e, -1, 1)) / np.float32(5)
    elif kind == "quantised":   # few levels: many equal scores and plateaus
        e = rng.integers(-1, 6, size=(H, W)).astype(np.float32) * np.float32(0.125)
        e = np.repeat(np.repeat(e[: H // 2 + 1, : W // 2 + 1], 2, 0), 2, 1)[:H, :W].copy()
    else:                       # "spike": a few huge corners the masks hide, on a low quantised floor
        e = rng.integers(0, 3, size=(H, W)).astype(np.float32) * np.float32(1e-3)
        ys, xs = rng.integers(12, H - 12, 6), rng.integers(12, W - 12, 6)
        e[ys, xs] = np.float32(1.0)
    return np.ascontiguousarray(e, dtype=np.float32)


@pytest.mark.parametrize("kind,seed", [("smooth", 1), ("smooth", 2), ("quantised", 3), ("quantised", 4), ("spike", 5), ("spike", 6)])
def test_batch_detection_equals_single_filter_pipeline(emu, kind, seed):
    rng = np.random.default_rng(seed)
    H, W, w, B = 96, 128, 7, 12
    eig = _eig_map(rng, H, W, kind)
    centers = np.zeros((B, MAXC, 2), dtype=np.float32)
    N = np.zeros(B, dtype=np.int32)
    num = rng.integers(1, MAXC + 1, size=B).astype(np.int32)
    num[1] = 0
    for b in range(B):
        N[b] = 0 if b == 0 else int(rng.integers(1, 10 if b < B - 1 else MAXC + 1))
        c = np.stack([rng.uniform(0, W, N[b]), rng.uniform(0, H, N[b])], axis=1)
        if kind == "spike" and b % 2:   # boxes over the global maxima: the masked maximum is then far below them
            top = np.argwhere(eig == eig.max())[: N[b]]
            c[: len(top)] = top[:, ::-1] + rng.uniform(-3, 3, size=(len(top), 2))
        centers[b, :N[b]] = c
    out = np.zeros((B, MAXC, 2), dtype=np.float32)
    n = np.zeros(B, dtype=np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    emu.emu_batch_detect(p(eig), W, H, w, B, MAXC, p(centers), p(N), p(num), p(out), p(n))
    total = 0
    for b in range(B):
        want = single_filter_corners(eig, _mask(H, W, centers[b, :N[b]], w), max(0, int(num[b])))
        got = out[b, :n[b]]
        assert np.array_equal(got, want), f"{kind} seed {seed} filter {b} (N {N[b]}, num {num[b]}): {got[:4]} vs {want[:4]}"
        total += len(want)
    assert total > 0 and n[1] == 0
