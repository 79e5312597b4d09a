"""synth.Scene's camera field: scenes rendered with a given calibration, today's camera by default."""
import numpy as np


def test_scene_camera_field(pkg):
    synth = pkg.synth
    base = synth.Scene(n_features=12, n_frames=2, seed=5)
    assert base.cam == synth.Camera(u0=320.0, v0=240.0)
    cam = synth.Camera(fx=563.2, fy=558.5, u0=347.8, v0=246.2, k1=-0.457, k2=0.31, k3=-0.14, p1=-0.00265, p2=0.00078)
    sc = synth.Scene(n_features=12, n_frames=2, seed=5, camera=cam)
    assert sc.cam is cam
    over = sc.config_overrides()
    assert tuple(over[k] for k in ("fx", "fy", "u0", "v0", "k1", "k2", "k3", "p1", "p2")) == \
        (cam.fx, cam.fy, cam.u0, cam.v0, cam.k1, cam.k2, cam.k3, cam.p1, cam.p2)
    # the frame-0 seeds project back onto themselves through the scene's own camera
    uv, z = sc.projections(0)
    assert (z > 0).all() and np.abs(uv - sc.feature_pixels).max() < 1e-6
    assert not np.array_equal(sc.frame(1), base.frame(1))
