"""CPU: the layout of ekf_camera_settings against its ctypes mirror, and the checks FilterBatch.from_configs and set_configs
apply to configurations of cameras with their own window, scale and blur threshold, without a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ekf_b200.h")


def test_camera_settings_match_c_layout(pkg, tmp_path):
    """sizeof / offsetof of ekf_camera_settings from the C compiler."""
    ct = pkg._abi.EkfCameraSettings
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
             'printf("size %zu\\n", sizeof(ekf_camera_settings));']
    lines += [f'printf("{f} %zu\\n", offsetof(ekf_camera_settings, {f}));' for f, _ in ct._fields_]
    lines.append("return 0;}")
    src = tmp_path / "lay.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "lay"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == C.sizeof(ct) == 16
    for f, _ in ct._fields_:
        assert int(got[f]) == getattr(ct, f).offset, f


def test_camera_fields_split_the_shared_fields(pkg):
    abi = pkg._abi
    assert set(abi.CAMERA_FIELDS) | set(abi.BATCH_WIDE_FIELDS) == set(abi.BATCH_SHARED_FIELDS)
    assert not set(abi.CAMERA_FIELDS) & set(abi.BATCH_WIDE_FIELDS)
    assert [f for f, _ in abi.EkfCameraSettings._fields_][:3] == list(abi.CAMERA_FIELDS)


def _shipped(abi):
    """Window, scale and blur threshold of the reference's four shipped configuration files."""
    return [abi.default_config(window_size=w, scale=s, kernel_size=k) for w, s, k in
            ((21, 2, 1000), (21, 1, 1000000000), (15, 2, 1000), (30, 10, 3))]


def test_camera_settings_of_shipped_rigs(pkg):
    abi = pkg._abi
    cfgs = _shipped(abi)
    camera_of = np.repeat(np.arange(4), 3)
    table = abi.camera_settings_of([cfgs[c] for c in camera_of], camera_of)
    assert table.tolist() == [[21, 2, 1000], [21, 1, 1000000000], [15, 2, 1000], [30, 10, 3]]


@pytest.mark.parametrize("field,value", [("window_size", 15), ("scale", 3), ("kernel_size", 7)])
def test_filters_of_one_camera_must_agree(pkg, field, value):
    abi = pkg._abi
    cfgs = [abi.default_config() for _ in range(4)]
    setattr(cfgs[3], field, value)
    with pytest.raises(ValueError, match=f"filter 3: {field} = {value} differs .* filter 2, which follows the same camera 1"):
        abi.camera_settings_of(cfgs, [0, 0, 1, 1])
    abi.camera_settings_of(cfgs, [0, 0, 1, 2])   # on a camera of its own it may differ


@pytest.mark.parametrize("field,value", [("search_clamp", 15.0), ("forsePlane", 1), ("xyz_conversion", 0), ("abs_int_quirk", 1)])
def test_batch_wide_fields_must_agree(pkg, field, value):
    abi = pkg._abi
    cfgs = [abi.default_config() for _ in range(3)]
    setattr(cfgs[2], field, value)
    with pytest.raises(ValueError, match=f"filter 2: {field} = .* differs from filter 0's"):
        abi.camera_settings_of(cfgs, [0, 1, 2])


def test_camera_without_filter_and_bad_map(pkg):
    abi = pkg._abi
    cfgs = [abi.default_config() for _ in range(3)]
    with pytest.raises(ValueError, match="camera 1 has no filter"):
        abi.camera_settings_of(cfgs, [0, 2, 2])
    with pytest.raises(ValueError, match="one camera"):
        abi.camera_settings_of(cfgs, [0, 1])


def test_per_camera_rows_check_against_the_filters_camera(pkg):
    """batch_rows_per_camera: the camera fields against the filter's camera row, the batch-wide ones against the batch."""
    abi = pkg._abi
    base = abi.default_config(window_size=21)
    settings = np.array([[11, 1, 1000000000], [21, 2, 3]])
    camera_of = [0, 1, 1]
    cfgs = [abi.default_config(window_size=11), abi.default_config(window_size=21, scale=2, kernel_size=3, sigma_pixel=3),
            abi.default_config(window_size=21, scale=2, kernel_size=3)]
    cam, rows = abi.batch_rows_per_camera(base, cfgs, settings, camera_of)
    assert cam.shape == (3, 9) and rows[1].sigma_pixel == 3
    bad = list(cfgs)
    bad[2] = abi.default_config(window_size=21, scale=1, kernel_size=3)
    with pytest.raises(ValueError, match="filter 2: scale = 1 differs from camera 1's 2; it is shared by every filter of a camera"):
        abi.batch_rows_per_camera(base, bad, settings, camera_of)
    bad[2] = abi.default_config(window_size=21, scale=2, kernel_size=3, search_clamp=10.0)
    with pytest.raises(ValueError, match="filter 2: search_clamp = 10.0 differs from the batch's 20.0"):
        abi.batch_rows_per_camera(base, bad, settings, camera_of)
    bad[2] = abi.default_config(window_size=21, scale=2, kernel_size=3, sigma_pixel=0)
    with pytest.raises(ValueError, match="filter 2: sigma_pixel < 1"):
        abi.batch_rows_per_camera(base, bad, settings, camera_of)
    # without a table the batch's values still apply to every filter, as before
    with pytest.raises(ValueError, match="filter 0: window_size = 11 differs from the batch's 21"):
        abi.batch_rows(base, cfgs)


def test_from_configs_refuses_before_creating(pkg):
    """from_configs raises on disagreeing filters before it touches a device."""
    abi = pkg._abi
    cfgs = _shipped(abi)
    cfgs[1] = abi.default_config(window_size=21, scale=1, kernel_size=1000000000, forsePlane=1)
    with pytest.raises(ValueError, match="filter 1: forsePlane = 1 differs from filter 0's 0"):
        pkg.FilterBatch.from_configs(cfgs, [0, 1, 2, 3])
    with pytest.raises(ValueError, match="filter 1: window_size = 21 differs from 15 of filter 0"):
        pkg.FilterBatch.from_configs([abi.default_config(window_size=15), abi.default_config(window_size=21)], [0, 0])
