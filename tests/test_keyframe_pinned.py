"""CPU: the key-frame recorder (host/keyframe_recorder.hpp and keyframes.py) against the REFERENCE'S OWN selector —
the live part of ImageConverter::imageCb (monoslam_ransac.cpp:585, 609-687, helpers :40-60) compiled from the
unmodified source into oracle/_ref/libref_selector_f64.so (oracle/build_ref_selector.py, `float` -> double).  Same
trajectory into both: nodes_and_prjcts.txt, cams_cov.txt and cams_cov2.txt must be BYTE-IDENTICAL and the images
written must carry the same names in the same order.  Trajectories are built so that every branch of the selector is
taken (candidate in the half-threshold band, key frame = current frame, key frame = earlier candidate, the
"frameId < 5" start-up rule, the reset of min_cov_for_pose).  The reference selector's files for these trajectories are
stored under tests/golden/keyframes/ (oracle/gen_golden_keyframes.py), and every test here compares against them, so the
comparison runs without the reference.  What stays unpinned: Eigen's number formatting itself (the absent dependency; the shim follows its documented
default IOFormat)."""
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from test_keyframes import Stub, _run_python, _trajectory

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "keyframes")
FILES = ("nodes_and_prjcts.txt", "cams_cov.txt", "cams_cov2.txt")


def trajectories():
    """name -> (states, sigmas, covs, points).  Shapes: a steady walk with a wiggling covariance (both key-frame
    sub-branches), a fast start (start-up rule: key frames at frame ids < 5 with no candidate), and a slow drift with long
    stays inside the half-threshold band and a monotonically growing covariance (candidate = first frame of the band)."""
    out = {"walk5": _trajectory(60, seed=5), "walk11": _trajectory(80, seed=11)}
    rng = np.random.default_rng(3)
    states, sigmas, covs = [], [], []
    for t in range(50):
        s = np.zeros(14)
        s[:3] = [6.0 * t if t < 4 else 24.0 + 0.35 * (t - 4), 0.0, 0.1 * t]
        ang = np.pi + 0.05 * t
        ax = np.array([0.0, -1.0, 1.0]) / np.sqrt(2)
        s[3] = np.cos(ang / 2); s[4:7] = np.sin(ang / 2) * ax; s[13] = 1.0
        A = rng.normal(0, 1e-2, (14, 14))
        states.append(s); sigmas.append(A @ A.T + np.eye(14) * 1e-6)
        covs.append(2e-4 * t + (5e-4 if t % 7 == 3 else 0.0))
    out["fast_start_then_drift"] = (states, sigmas, covs, np.zeros((1, 12)))
    st, sg, _, pts = _trajectory(70, seed=21)
    out["steady_cov"] = (st, sg, [1e-3 + 1e-6 * t for t in range(70)], pts)   # cov(now) - min_cov < 0.000085: the CURRENT frame is written
    return out


def reference_run(directory, name):
    """The reference selector's output for trajectory `name`: its three files copied into `directory`; returns the
    image names it wrote, in order."""
    gold = os.path.join(GOLD, name)
    for f in FILES:
        shutil.copyfile(os.path.join(gold, f), os.path.join(directory, f))
    return open(os.path.join(gold, "images.txt")).read().split()


@pytest.mark.parametrize("name", sorted(trajectories()))
def test_python_recorder_equals_reference_selector(pkg, tmp_path, name):
    traj = trajectories()[name]
    refdir = tmp_path / "ref"; pydir = tmp_path / "py"
    refdir.mkdir(); pydir.mkdir()
    ref_images = reference_run(refdir, name)
    rec, saved = _run_python(pkg, pydir, traj)
    assert [os.path.basename(p) for p in saved] == ref_images
    assert len(ref_images) >= 3
    for f in FILES:
        assert (pydir / f).read_bytes() == (refdir / f).read_bytes(), f"{name}: {f} differs from the reference selector's"


def test_every_branch_is_exercised(tmp_path):
    """The three trajectories together take both sub-branches of the key-frame case and the start-up rule."""
    seen_current, seen_candidate, seen_startup, seen_cov2 = False, False, False, False
    for name in trajectories():
        d = tmp_path / name; d.mkdir()
        imgs = reference_run(d, name)
        text = (d / "nodes_and_prjcts.txt").read_text()
        seen_current |= "0  0  0" in text          # literal written with the CURRENT frame (:640, :672)
        seen_candidate |= "\n0 0 0\n" in text      # min_projs (MatrixX3i::Zero(1,3)) written with an EARLIER candidate (:650)
        n2 = len((d / "cams_cov2.txt").read_text().strip().splitlines()) // 7
        n1 = len((d / "cams_cov.txt").read_text().strip().splitlines()) // 7
        seen_startup |= n1 > n2 and imgs[0] in ("1.png", "2.png", "3.png", "4.png")
        seen_cov2 |= n2 > 0                        # cams_cov2.txt is only written by the "current frame is as good" branch (:637-645)
    assert seen_current and seen_candidate and seen_startup and seen_cov2


def test_cpp_recorder_equals_reference_selector(tmp_path):
    name = "walk11"
    traj = trajectories()[name]
    refdir = tmp_path / "ref"; cdir = tmp_path / "cpp"
    refdir.mkdir(); cdir.mkdir()
    ref_images = reference_run(refdir, name)
    states, sigmas, covs, pts = traj
    blob = struct.pack("i", len(states))
    for s, S, c in zip(states, sigmas, covs):
        blob += np.asarray(s, dtype=np.float64).tobytes() + np.asarray(S, dtype=np.float64).tobytes() + struct.pack("d", c)
    blob += struct.pack("i", pts.shape[0]) + np.asarray(pts, dtype=np.float64).tobytes()
    (tmp_path / "traj.bin").write_bytes(blob)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "keyframe_stub"
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-o", str(exe), os.path.join(root, "tests", "keyframe_stub.cpp")])
    out = subprocess.check_output([str(exe), str(tmp_path / "traj.bin"), str(cdir)], text=True)
    assert [os.path.basename(p) for p in out.split()] == ref_images
    for f in FILES:
        assert (cdir / f).read_bytes() == (refdir / f).read_bytes(), f


@pytest.mark.parametrize("name", sorted(trajectories()))
def test_python_recorder_equals_committed_reference_files(pkg, tmp_path, name):
    """Same comparison against the committed outputs of the reference selector (runs without /root/reference)."""
    traj = trajectories()[name]
    _, saved = _run_python(pkg, tmp_path, traj)
    gold = os.path.join(GOLD, name)
    assert os.path.isdir(gold), "run oracle/gen_golden_keyframes.py"
    assert [os.path.basename(p) for p in saved] == open(os.path.join(gold, "images.txt")).read().split()
    for f in FILES:
        assert (tmp_path / f).read_bytes() == open(os.path.join(gold, f), "rb").read(), f
