"""CPU: the layout of ekf_filter_params against its ctypes mirror, and the conversion of per-filter configurations into the
batch's tables (FilterBatch.set_configs) without a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ekf_b200.h")


def test_filter_params_match_c_layout(pkg, tmp_path):
    """sizeof / offsetof of ekf_filter_params from the C compiler."""
    ct = pkg._abi.EkfFilterParams
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
             'printf("size %zu\\n", sizeof(ekf_filter_params));']
    lines += [f'printf("{f} %zu\\n", offsetof(ekf_filter_params, {f}));' for f, _ in ct._fields_]
    lines.append("return 0;}")
    src = tmp_path / "lay.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "lay"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == C.sizeof(ct) == 15 * 8 + 6 * 4
    for f, _ in ct._fields_:
        assert int(got[f]) == getattr(ct, f).offset, f


def test_filter_params_fields_are_config_fields(pkg):
    """Every field but the padding names an ekf_config field of the same type; none is shared by the batch."""
    abi = pkg._abi
    cfg_types = dict(abi.EkfConfig._fields_)
    for f, t in abi.EkfFilterParams._fields_:
        if f == "_pad":
            continue
        assert cfg_types[f] is t, f
        assert f not in abi.BATCH_SHARED_FIELDS and f not in abi.INTRINSICS, f


def _cfgs(pkg):
    base = pkg.default_config(window_size=11, min_features=20, max_features=60)
    a = pkg.default_config(window_size=11, sigma_vx=0.03, rho_0=0.2, sigma_pixel=3, sigma_size=4, min_features=100,
                           max_features=1000, ransac_nhyp0=500, fx=600.0, k2=0.1)
    b = pkg.default_config(window_size=11, T_camera=0.1, ncc_threshold=0.7, quality_ratio=0.3, linearity_threshold=0.02,
                           li_threshold_factor=1.5, hi_chi2_threshold=2.0, ransac_p=0.95, min_features=30, max_features=35)
    return base, [a, b, pkg._abi.EkfConfig.from_buffer_copy(base)]


def test_rows_in_field_order(pkg):
    base, cfgs = _cfgs(pkg)
    cam, rows = pkg._abi.batch_rows(base, cfgs)
    assert cam.shape == (3, 9) and cam.dtype == np.float64
    for f, c in enumerate(cfgs):
        assert list(cam[f]) == [getattr(c, k) for k in pkg._abi.INTRINSICS]
        for name, _ in pkg._abi.EkfFilterParams._fields_:
            if name != "_pad":
                assert getattr(rows[f], name) == getattr(c, name), (f, name)
        assert rows[f]._pad == 0
    assert (rows[0].sigma_vx, rows[0].sigma_vy, rows[0].sigma_pixel, rows[0].min_features) == (0.03, 0.01, 3, 100)
    assert (rows[1].T_camera, rows[1].ransac_p, rows[1].max_features) == (0.1, 0.95, 35)
    # the memory the C call reads: doubles first, then the int32s
    raw = bytes(rows)[C.sizeof(pkg._abi.EkfFilterParams):2 * C.sizeof(pkg._abi.EkfFilterParams)]
    d = np.frombuffer(raw[:120], dtype=np.float64)
    i = np.frombuffer(raw[120:], dtype=np.int32)
    assert d[8] == 0.1 and d[10] == 0.95 and list(i) == [2, 2, 30, 35, 10000, 0]


def test_init_features_is_not_read(pkg):
    base, cfgs = _cfgs(pkg)
    cfgs[1].nInitFeatures = 77
    cam, rows = pkg._abi.batch_rows(base, cfgs)
    cam2, rows2 = pkg._abi.batch_rows(base, _cfgs(pkg)[1])
    assert np.array_equal(cam, cam2) and bytes(rows) == bytes(rows2)


@pytest.mark.parametrize("field,value", [("window_size", 21), ("search_clamp", 10.0), ("scale", 2), ("kernel_size", 3),
                                         ("forsePlane", 1), ("xyz_conversion", 0), ("abs_int_quirk", 1)])
def test_shared_field_differing_is_refused(pkg, field, value):
    base, cfgs = _cfgs(pkg)
    setattr(cfgs[2], field, value)
    with pytest.raises(ValueError, match=rf"filter 2: {field}"):
        pkg._abi.batch_rows(base, cfgs)


@pytest.mark.parametrize("field,value,says", [("sigma_pixel", 0, "sigma_pixel < 1"), ("sigma_size", 0, "sigma_size < 1"),
                                              ("ransac_p", 1.0, "ransac_p"), ("ransac_nhyp0", 0, "ransac_nhyp0"),
                                              ("sigma_wy", -0.1, "sigma_wy is negative"), ("rho_0", float("nan"), "rho_0"),
                                              ("min_features", -1, "min_features"), ("fx", 0.0, "fx / fy"),
                                              ("k1", float("inf"), "k1 is not finite")])
def test_invalid_rows_are_refused_before_any_table(pkg, field, value, says):
    """batch_rows refuses what the C calls refuse, naming filter and field, so set_configs changes neither table."""
    base, cfgs = _cfgs(pkg)
    setattr(cfgs[1], field, value)
    with pytest.raises(ValueError, match=rf"filter 1: {says}"):
        pkg._abi.batch_rows(base, cfgs)
