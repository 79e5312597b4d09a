"""ctypes binding of oracle/_ref/libref_selector_f64.so — the reference's own key-frame selector (monoslam_ransac.cpp:585,
609-687) compiled from the unmodified source by oracle/build_ref_selector.py.  TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_ref", "libref_selector_f64.so")
        if os.path.isdir(os.environ.get("EKF_REFERENCE_ROOT", "/root/reference")):
            import build_ref_selector
            path = build_ref_selector.build()
        L = C.CDLL(path)
        L.refsel_create.restype = C.c_void_p; L.refsel_create.argtypes = [C.c_char_p]
        L.refsel_destroy.restype = None; L.refsel_destroy.argtypes = [C.c_void_p]
        L.refsel_frame.restype = None; L.refsel_frame.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_void_p]
        L.refsel_num_written.restype = C.c_int
        L.refsel_written.restype = C.c_char_p; L.refsel_written.argtypes = [C.c_int]
        L.refsel_scalar_bytes.restype = C.c_int
        assert L.refsel_scalar_bytes() == 8
        _LIB = L
    return _LIB


def run(directory, states, sigmas, covs, first_frame_id=1):
    """Feeds a trajectory (per frame: 14 camera states, 14 x 14 covariance, Covariance_Parameter) to the reference selector;
    the three text files land in `directory`.  Returns the image names the node would have written, in order."""
    L = lib()
    h = L.refsel_create(str(directory).encode())
    try:
        for t, (s, S, c) in enumerate(zip(states, sigmas, covs)):
            s = np.ascontiguousarray(s, dtype=np.float64); S = np.ascontiguousarray(S, dtype=np.float64)
            L.refsel_frame(h, first_frame_id + t, s.ctypes.data_as(C.c_void_p), float(c), S.ctypes.data_as(C.c_void_p))
        names = [L.refsel_written(i).decode() for i in range(L.refsel_num_written())]
    finally:
        L.refsel_destroy(h)
    return names
