"""Loads libekf_b200.so (the C ABI of include/ekf_b200.h) through ctypes.

There is no CPU fallback: if the shared library is missing or has no usable CUDA device the calls
raise.  build.build() compiles it with nvcc (works without a GPU).
"""
import os as _os
# One hardware work queue per stream as far as the device allows (the default is 8; a filter handle owns 8 streams): streams that share a
# queue serialise against each other.  Only effective when set before the CUDA context exists; an explicit setting wins.
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import ctypes as C
import os

from . import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libekf_b200.so")

# name -> (restype, argtypes); one entry per declaration in include/ekf_b200.h
_vp, _i, _d, _f = C.c_void_p, C.c_int, C.c_double, C.c_float
_P = C.POINTER
SIGNATURES = {
    "ekf_config_default": (None, [_P(_abi.EkfConfig)]),
    "ekf_create": (_i, [_P(_abi.EkfConfig), _i, _i, _P(_vp)]),
    "ekf_destroy": (_i, [_vp]),
    "ekf_set_stream": (_i, [_vp, _vp]),
    "ekf_sync": (_i, [_vp]),
    "ekf_last_error": (C.c_char_p, [_vp]),
    "ekf_capture_frame": (_i, [_vp, _vp, _i, _i, _i, _d]),
    "ekf_capture_frame_bgr": (_i, [_vp, _vp, _i, _i, _i, _d]),
    "ekf_get_frame": (_i, [_vp, _vp, _P(_i), _P(_i)]),
    "ekf_capture_frame_device": (_i, [_vp, _vp, _i, _i, _i, _d]),
    "ekf_predict": (_i, [_vp, _vp, _vp, _i]),
    "ekf_match": (_i, [_vp, _P(_i)]),
    "ekf_update_after_match": (_i, [_vp, _vp, _i]),
    "ekf_update": (_i, [_vp, _vp, _i]),
    "ekf_inject_match": (_i, [_vp, _i, _d, _d, _i]),
    "ekf_add_feature": (_i, [_vp, _f, _f]),
    "ekf_remove_feature": (_i, [_vp, _i]),
    "ekf_find_new_features": (_i, [_vp, _i]),
    "ekf_detect_corners": (_i, [_vp, _i, _vp, _P(_i)]),
    "ekf_convert2xyz_if_linear": (_i, [_vp, _i]),
    "ekf_convert2xyz_if_linear_all": (_i, [_vp]),
    "ekf_num_features": (_i, [_vp]),
    "ekf_state_dim": (_i, [_vp]),
    "ekf_get_state": (_i, [_vp, _vp]),
    "ekf_get_sigma": (_i, [_vp, _vp]),
    "ekf_covariance_parameter": (_i, [_vp, _P(_d)]),
    "ekf_get_dt": (_d, [_vp]),
    "ekf_get_center": (_i, [_vp, _i, _vp]),
    "ekf_num_deleted": (_i, [_vp]),
    "ekf_get_deleted": (_i, [_vp, _i, _vp]),
    "ekf_get_points_features": (_i, [_vp, _vp, _i, _vp]),
    "ekf_rts_epoch": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d]),
    "ekf_get_feature": (_i, [_vp, _i, _P(_abi.EkfFeatureInfo)]),
    "ekf_get_template": (_i, [_vp, _i, _i, _vp]),
    "ekf_get_step_stats": (_i, [_vp, _P(_abi.EkfStepStats)]),
    "ekf_get_full": (_i, [_vp, _vp, _vp, _i]),
    "ekf_set_full": (_i, [_vp, _vp, _vp, _i]),
    "ekf_get_S_blocks": (_i, [_vp, _vp]),
    "ekf_match_batch": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _f, _f, _f, _vp, _vp, _vp]),
    "ekf_batch_create": (_i, [_P(_abi.EkfConfig), _i, _i, _i, _P(_vp)]),
    "ekf_batch_create_large": (_i, [_P(_abi.EkfConfig), _i, _i, _i, _P(_vp)]),
    "ekf_batch_update_clusters": (_i, [_vp, _P(_i), _P(_i)]),
    "ekf_batch_destroy": (_i, [_vp]),
    "ekf_batch_describe": (_i, [_vp, _P(_abi.EkfBatchDesc)]),
    "ekf_batch_set_stream": (_i, [_vp, _vp]),
    "ekf_batch_sync": (_i, [_vp]),
    "ekf_batch_last_error": (C.c_char_p, [_vp]),
    "ekf_batch_seed_from": (_i, [_vp, _vp]),
    "ekf_batch_set_camera_states": (_i, [_vp, _vp]),
    "ekf_batch_capture_frame": (_i, [_vp, _vp, _i, _i, _i, _d]),
    "ekf_batch_capture_frame_device": (_i, [_vp, _vp, _i, _i, _i, _d]),
    "ekf_batch_capture_frame_bgr": (_i, [_vp, _vp, _i, _i, _i, _d]),
    "ekf_batch_get_frame": (_i, [_vp, _vp, _P(_i), _P(_i)]),
    "ekf_batch_set_scale": (_i, [_vp, _i]),
    "ekf_batch_set_force_plane": (_i, [_vp, _i]),
    "ekf_batch_step": (_i, [_vp, _vp, _vp, _i, _vp, _i]),
    "ekf_batch_convert2xyz_if_linear_all": (_i, [_vp]),
    "ekf_batch_get_camera_states": (_i, [_vp, _vp, _vp, _vp]),
    "ekf_batch_num_features": (_i, [_vp, _i]),
    "ekf_batch_state_dim": (_i, [_vp, _i]),
    "ekf_batch_get_full": (_i, [_vp, _i, _vp, _vp, _i]),
    "ekf_batch_set_full": (_i, [_vp, _i, _vp, _vp, _i]),
    "ekf_batch_get_feature": (_i, [_vp, _i, _i, _P(_abi.EkfFeatureInfo)]),
    "ekf_batch_add_feature": (_i, [_vp, _i, _f, _f]),
    "ekf_batch_detect_corners": (_i, [_vp, _vp, _vp, _vp]),
    "ekf_batch_find_new_features": (_i, [_vp, _vp, _vp]),
    "ekf_batch_set_topup": (_i, [_vp, _i]),
    "ekf_batch_last_added": (_i, [_vp, _vp]),
    "ekf_batch_set_motion_blur": (_i, [_vp, _i]),
    "ekf_batch_last_blur_counts": (_i, [_vp, _vp]),
    "ekf_batch_set_archive": (_i, [_vp, _i]),
    "ekf_batch_remove_feature": (_i, [_vp, _i, _i]),
    "ekf_batch_num_deleted": (_i, [_vp, _vp]),
    "ekf_batch_get_deleted": (_i, [_vp, _i, _vp, _i, _P(_i)]),
    "ekf_batch_get_points_features": (_i, [_vp, _i, _i, _vp, _i, _vp]),
    "ekf_batch_get_template": (_i, [_vp, _i, _i, _i, _vp]),
    "ekf_batch_kernel_launches": (C.c_int64, [_vp]),
    "ekf_batch_last_step_ms": (_i, [_vp, _vp]),
    "ekf_batch_last_match_deferred": (_i, [_vp]),
    "ekf_batch_set_cameras": (_i, [_vp, _i, _vp]),
    "ekf_batch_capture_frames": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "ekf_batch_capture_frames_device": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "ekf_batch_capture_frames_bgr": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "ekf_batch_get_camera_frame": (_i, [_vp, _i, _vp, _P(_i), _P(_i)]),
    "ekf_batch_get_dt": (_i, [_vp, _vp]),
    "ekf_batch_set_detect_budget": (_i, [_vp, C.c_int64]),
    "ekf_batch_set_intrinsics": (_i, [_vp, _vp]),
    "ekf_batch_set_frame_sizes": (_i, [_vp, _vp]),
    "ekf_batch_step_controls": (_i, [_vp, _vp, _vp, _vp, _vp, _i]),
    "ekf_batch_capture_camera_frames": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _vp]),
    "ekf_batch_capture_camera_frames_device": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _vp]),
    "ekf_batch_capture_camera_frames_bgr": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _vp]),
    "ekf_batch_step_filters": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i]),
    "ekf_batch_resample": (_i, [_vp, _vp]),
    "ekf_dist_load_nccl": (_i, [C.c_char_p]),
    "ekf_dist_unique_id": (_i, [_vp]),
    "ekf_dist_attach": (_i, [_vp, _vp, _i, _i]),
    "ekf_dist_detach": (_i, [_vp]),
    "ekf_dist_info": (_i, [_vp, _P(_i), _P(_i), _P(C.c_int64)]),
    "ekf_dist_peer_memory": (_i, [_vp]),
    "ekf_set_profiling": (_i, [_vp, _i]),
    "ekf_get_profile": (_i, [_vp, _P(_abi.EkfProfile), _i]),
    "ekf_set_symmetric_downdate": (_i, [_vp, _i]),
    "ekf_debug_time_downdate": (_i, [_vp, _i, _P(C.c_float)]),
    "ekf_build_info": (C.c_char_p, []),
}

_lib = None


def lib():
    """The loaded library.  Raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with __graft_entry__.build(); "
                               "this package has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
