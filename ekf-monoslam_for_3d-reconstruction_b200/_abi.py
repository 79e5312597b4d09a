"""ctypes mirrors of the structs in include/ekf_b200.h (kept field-for-field in sync)."""
import ctypes as C

import numpy as np

STATE_DIM = 14  # vslamRansac.cpp:22

EKF_OK, EKF_ERR_ARG, EKF_ERR_CUDA, EKF_ERR_CAPACITY, EKF_ERR_UNSUPPORTED, EKF_ERR_STATE = 0, -1, -2, -3, -4, -5


class EkfConfig(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "sigma_vx", "sigma_vy", "sigma_vz", "sigma_wx", "sigma_wy", "sigma_wz",
        "rho_0", "sigma_rho_0", "T_camera",
        "fx", "fy", "u0", "v0", "k1", "k2", "k3", "p1", "p2",
        "ncc_threshold", "search_clamp", "ransac_p", "li_threshold_factor", "hi_chi2_threshold",
        "quality_ratio", "linearity_threshold")] + [(n, C.c_int32) for n in (
        "window_size", "sigma_pixel", "kernel_size", "sigma_size", "scale",
        "nInitFeatures", "min_features", "max_features", "forsePlane",
        "ransac_nhyp0", "xyz_conversion", "abs_int_quirk")]


class EkfFilterParams(C.Structure):
    """ekf_filter_params: the ekf_config fields a filter of a batch may take on its own (ekf_batch_set_filter_params)."""
    _fields_ = [(n, C.c_double) for n in (
        "sigma_vx", "sigma_vy", "sigma_vz", "sigma_wx", "sigma_wy", "sigma_wz",
        "rho_0", "sigma_rho_0", "T_camera", "ncc_threshold", "ransac_p", "li_threshold_factor", "hi_chi2_threshold",
        "quality_ratio", "linearity_threshold")] + [(n, C.c_int32) for n in (
        "sigma_pixel", "sigma_size", "min_features", "max_features", "ransac_nhyp0", "_pad")]


class EkfCameraSettings(C.Structure):
    """ekf_camera_settings: the ekf_config fields a camera of a batch may take on its own (ekf_batch_set_camera_settings)."""
    _fields_ = [(n, C.c_int32) for n in ("window_size", "scale", "kernel_size", "_pad")]


# ekf_config fields every filter of a batch shares (buffer sizes, launch structure, emulation mode); intrinsics have their own
# table (ekf_batch_set_intrinsics), nInitFeatures is never read by a batch.  With a camera table (ekf_batch_set_camera_settings)
# the CAMERA_FIELDS among them are shared by the filters of a camera only, and BATCH_WIDE_FIELDS stay shared by the batch.
BATCH_SHARED_FIELDS = ("window_size", "search_clamp", "scale", "kernel_size", "forsePlane", "xyz_conversion", "abs_int_quirk")
CAMERA_FIELDS = ("window_size", "scale", "kernel_size")
BATCH_WIDE_FIELDS = ("search_clamp", "forsePlane", "xyz_conversion", "abs_int_quirk")
INTRINSICS = ("fx", "fy", "u0", "v0", "k1", "k2", "k3", "p1", "p2")


def batch_rows(base, cfgs):
    """The per-filter tables of a batch built from `base` whose filter f runs configuration cfgs[f]: an (n, 9) float64 array
    of intrinsics (INTRINSICS order) and an array of n EkfFilterParams.  ValueError, naming the field and the filter, when a
    field of BATCH_SHARED_FIELDS differs from base's or a row is one the C calls refuse."""
    def want(f, name):
        return getattr(base, name), "the batch's", "every filter of a batch"
    return _rows(cfgs, want)


def batch_rows_per_camera(base, cfgs, settings, camera_of):
    """batch_rows for a batch with a camera table: filter f's CAMERA_FIELDS are checked against row camera_of[f] of settings
    (an (n_cameras, 3) array of window_size, scale, kernel_size), its BATCH_WIDE_FIELDS against base's."""
    settings = np.asarray(settings).reshape(-1, 3)
    camera_of = np.asarray(camera_of).reshape(-1)

    def want(f, name):
        if name in CAMERA_FIELDS:
            k = int(camera_of[f])
            return int(settings[k, CAMERA_FIELDS.index(name)]), f"camera {k}'s", "every filter of a camera"
        return getattr(base, name), "the batch's", "every filter of a batch"
    return _rows(cfgs, want)


def camera_settings_of(cfgs, camera_of):
    """The camera table of a batch whose filter f runs cfgs[f] and follows camera camera_of[f]: an (n_cameras, 3) int array of
    (window_size, scale, kernel_size), n_cameras = max(camera_of) + 1.  ValueError, naming the filter and field, when filters
    of one camera disagree on a CAMERA_FIELDS entry or any filters on a BATCH_WIDE_FIELDS entry, or a camera has no filter."""
    cfgs = list(cfgs)
    cam = np.asarray(camera_of, dtype=np.int64).reshape(-1)
    if cam.shape != (len(cfgs),) or len(cfgs) < 1 or cam.min() < 0:
        raise ValueError("camera_of needs one camera >= 0 per configuration")
    n_cam = int(cam.max()) + 1
    first = np.full(n_cam, -1)
    for f in range(len(cfgs)):
        if first[cam[f]] < 0:
            first[cam[f]] = f
    if (first < 0).any():
        raise ValueError(f"camera {int(np.argmax(first < 0))} has no filter")
    for f, c in enumerate(cfgs):
        for name in CAMERA_FIELDS:
            g = cfgs[first[cam[f]]]
            if getattr(c, name) != getattr(g, name):
                raise ValueError(f"filter {f}: {name} = {getattr(c, name)} differs from {getattr(g, name)} of filter "
                                 f"{first[cam[f]]}, which follows the same camera {cam[f]}; it is shared by every filter of a camera")
        for name in BATCH_WIDE_FIELDS:
            if getattr(c, name) != getattr(cfgs[0], name):
                raise ValueError(f"filter {f}: {name} = {getattr(c, name)} differs from filter 0's {getattr(cfgs[0], name)}; "
                                 f"it is shared by every filter of a batch")
    return np.array([[getattr(cfgs[first[k]], n) for n in CAMERA_FIELDS] for k in range(n_cam)], dtype=np.int64)


def _rows(cfgs, want):
    cfgs = list(cfgs)
    cam = np.zeros((len(cfgs), 9), dtype=np.float64)
    rows = (EkfFilterParams * len(cfgs))()
    for f, c in enumerate(cfgs):
        for name in BATCH_SHARED_FIELDS:
            v, whose, shared = want(f, name)
            if getattr(c, name) != v:
                raise ValueError(f"filter {f}: {name} = {getattr(c, name)} differs from {whose} {v}; it is shared by {shared}")
        cam[f] = [getattr(c, n) for n in INTRINSICS]
        for name, _ in EkfFilterParams._fields_:
            if name != "_pad":
                setattr(rows[f], name, getattr(c, name))
        bad = _row_error(cam[f], rows[f])
        if bad:
            raise ValueError(f"filter {f}: {bad}")
    return cam, rows


def _row_error(cam, p):
    """What ekf_batch_set_intrinsics / ekf_batch_set_filter_params refuse in one filter's rows (None when both are valid), so
    that FilterBatch.set_configs can check every row before it changes either table."""
    for n, v in zip(INTRINSICS, cam):
        if not np.isfinite(v):
            return f"{n} is not finite"
    if not (cam[0] > 0 and cam[1] > 0):
        return "fx / fy <= 0"
    for name, t in EkfFilterParams._fields_:
        if t is C.c_double and not np.isfinite(getattr(p, name)):
            return f"{name} is not finite"
    for name in ("sigma_vx", "sigma_vy", "sigma_vz", "sigma_wx", "sigma_wy", "sigma_wz", "sigma_rho_0"):
        if getattr(p, name) < 0:
            return f"{name} is negative"
    if p.sigma_pixel < 1:
        return "sigma_pixel < 1"
    if p.sigma_size < 1:
        return "sigma_size < 1"
    if not 0 < p.ransac_p < 1:
        return "ransac_p outside (0, 1)"
    if p.ransac_nhyp0 < 1:
        return "ransac_nhyp0 < 1"
    if p.min_features < 0 or p.max_features < 0:
        return "min_features / max_features negative"
    return None


def default_config(**over) -> EkfConfig:
    """ConfigVSLAM.cpp:27-47 + camModel.hpp:25-33 + hard-coded constants (same as ekf_config_default)."""
    c = EkfConfig(
        sigma_vx=0.01, sigma_vy=0.01, sigma_vz=0.01, sigma_wx=0.01, sigma_wy=0.01, sigma_wz=0.01,
        rho_0=0.1, sigma_rho_0=0.25, T_camera=0.5,
        fx=592.2860, fy=584.9968, u0=362.1059, v0=275.9642, k1=-0.3954, k2=0.5521, k3=0.0,
        p1=-0.0075, p2=0.0140,
        ncc_threshold=0.8, search_clamp=20.0, ransac_p=0.99, li_threshold_factor=2.0,
        hi_chi2_threshold=1.0, quality_ratio=0.2, linearity_threshold=0.01,
        window_size=21, sigma_pixel=2, kernel_size=1000000000, sigma_size=2, scale=1,
        nInitFeatures=5, min_features=30, max_features=100, forsePlane=0,
        ransac_nhyp0=10000, xyz_conversion=1, abs_int_quirk=0)
    for k, v in over.items():
        if not hasattr(c, k):
            raise AttributeError(f"ekf_config has no field {k!r}")
        setattr(c, k, v)
    return c


class EkfFeatureInfo(C.Structure):
    _fields_ = [
        ("position_in_state", C.c_int32), ("position_in_z", C.c_int32), ("coding", C.c_int32),
        ("n_tot", C.c_int32), ("n_find", C.c_int32), ("real_index", C.c_int32),
        ("is_in_innovation", C.c_int32), ("is_in_li", C.c_int32), ("is_in_hi", C.c_int32),
        ("remove_flag", C.c_int32),
        ("center", C.c_float * 2), ("quality_index", C.c_float), ("last_ncc", C.c_float),
        ("z", C.c_double * 2), ("h", C.c_double * 2), ("H", C.c_double * 26),
        ("state", C.c_double * 6), ("cov", C.c_double * 36)]


class EkfDeletedInfo(C.Structure):
    _fields_ = [("real_index", C.c_int32), ("_pad", C.c_int32), ("xyz_pos", C.c_double * 3), ("cov_4_delete", C.c_double * 9)]


class EkfStepStats(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_in_innovation_predict", "n_matched", "n_li", "n_hi", "ransac_hypotheses", "n_removed",
        "topup_request", "blur_requests")] + [("kernel_launches", C.c_int64)]


PROF_CLASSES = ("predict", "match", "ransac", "gather_W", "factor_S", "V_trsm", "downdate_gemm", "quat_normalise",
                "hi_rescue", "bookkeeping", "add_remove", "nccl_allgather")


class EkfProfile(C.Structure):
    _fields_ = [("ms", C.c_double * 12), ("launches", C.c_int64 * 12)]


class EkfBatchDesc(C.Structure):
    _fields_ = [("n_filters", C.c_int32), ("feature_capacity", C.c_int32), ("state_capacity", C.c_int32), ("ld", C.c_int32),
                ("device", C.c_int32), ("reserved", C.c_int32 * 3)]


BATCH_STAT_FIELDS = 8
BATCH_MAX_CORNERS = 32   # EKF_BATCH_MAX_CORNERS
BSTAT = dict(innov=0, matched=1, li=2, hi=3, hyps=4, chol_fail=5, removed=6, topup=7)
