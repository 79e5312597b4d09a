"""ctypes mirrors of the structs in include/ekf_b200.h (kept field-for-field in sync)."""
import ctypes as C

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
