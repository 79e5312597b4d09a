"""ctypes binding of oracle/_ref/libref_f{32,64}.so — the REFERENCE'S OWN sources compiled against
the API stand-ins of oracle/shim (see oracle/ref_capi.cpp).  TEST INFRASTRUCTURE ONLY; exists only
where /root/reference is present (this container), never on the GPU box."""
import ctypes as C
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)
import ekfb200  # noqa: E402

abi = ekfb200.load_package()._abi


def build(force=False):
    sys.path.insert(0, _HERE)
    import build_ref
    return build_ref.build(force=force)


_libs = {}


def lib(fp64=True):
    key = "f64" if fp64 else "f32"
    if key in _libs:
        return _libs[key]
    path = os.path.join(_HERE, "_ref", f"libref_{key}.so")
    if not os.path.exists(path):
        build()
    L = C.CDLL(path)
    vp, i32, f64, f32 = C.c_void_p, C.c_int, C.c_double, C.c_float
    sig = {
        "ref_scalar_bytes": (i32, []), "ref_set_log_level": (None, [i32]),
        "ref_create": (vp, [C.POINTER(abi.EkfConfig)]), "ref_destroy": (None, [vp]),
        "ref_capture": (None, [vp, vp, i32, i32, i32, f64]),
        "ref_add_feature": (i32, [vp, f32, f32]), "ref_remove_feature": (None, [vp, i32]),
        "ref_predict": (None, [vp, vp, vp, i32]), "ref_update": (None, [vp, vp, i32]),
        "ref_last_hypotheses": (i32, [vp]), "ref_convert2xyz": (None, [vp, i32]),
        "ref_state_dim": (i32, [vp]), "ref_num_features": (i32, [vp]), "ref_get_dt": (f64, [vp]),
        "ref_covariance_parameter": (f64, [vp]),
        "ref_get_full": (None, [vp, vp, vp, i32]), "ref_set_full": (None, [vp, vp, vp, i32]),
        "ref_get_state14": (None, [vp, vp, vp]),
        "ref_get_feature": (None, [vp, i32, C.POINTER(abi.EkfFeatureInfo)]),
        "ref_get_template": (None, [vp, i32, i32, vp]), "ref_get_S_blocks": (None, [vp, vp]),
        "ref_find_match": (i32, [vp, i32, i32, i32, vp, i32, vp, vp, f32, vp]),
        "ref_num_deleted": (i32, [vp]), "ref_get_deleted": (None, [vp, i32, vp, vp, vp]),
        "ref_rts_epoch": (None, [vp, vp, vp, vp, vp, vp, vp, f64]),
        "ref_points_features": (i32, [vp, vp, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    assert L.ref_scalar_bytes() == (8 if fp64 else 4)
    _libs[key] = L
    return L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class ReferenceFilter:
    """The reference's VSlamFilter (method names as in vslamRansac.hpp:99-140)."""

    def __init__(self, cfg, fp64=True):
        self.L = lib(fp64)
        self.cfg = cfg
        self.h = self.L.ref_create(C.byref(cfg))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_destroy(self.h)
            self.h = None

    def captureNewFrame(self, img, stamp=-1.0):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        self.L.ref_capture(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0], float(stamp))

    def addFeature(self, u, v):
        return self.L.ref_add_feature(self.h, float(u), float(v))

    def removeFeature(self, i):
        self.L.ref_remove_feature(self.h, int(i))

    def predict(self, dv=(0, 0, 0), dw=(0, 0, 0), vcontrol=False):
        a = np.asarray(dv, dtype=np.float64); b = np.asarray(dw, dtype=np.float64)
        self.L.ref_predict(self.h, _ptr(a), _ptr(b), int(bool(vcontrol)))

    def update(self, picks=None):
        p = np.ascontiguousarray(picks if picks is not None else np.zeros(0), dtype=np.uint32)
        self.L.ref_update(self.h, _ptr(p), int(p.size))

    def last_hypotheses(self):
        return self.L.ref_last_hypotheses(self.h)

    def convert2XYZ_ifLinear(self, i):
        self.L.ref_convert2xyz(self.h, int(i))

    def convert2XYZ_ifLinearAll(self):
        self.L.ref_convert2xyz(self.h, -1)

    def numOfFeatures(self):
        return self.L.ref_num_features(self.h)

    def state_dim(self):
        return self.L.ref_state_dim(self.h)

    def getDt(self):
        return self.L.ref_get_dt(self.h)

    def Covariance_Parameter(self):
        return self.L.ref_covariance_parameter(self.h)

    def get_full(self):
        n = self.state_dim()
        mu = np.zeros(n); S = np.zeros((n, n))
        self.L.ref_get_full(self.h, _ptr(mu), _ptr(S), n)
        return mu, S

    def set_full(self, mu, S):
        mu = np.ascontiguousarray(mu, dtype=np.float64); S = np.ascontiguousarray(S, dtype=np.float64)
        assert mu.size == self.state_dim() and S.shape == (mu.size, mu.size)
        self.L.ref_set_full(self.h, _ptr(mu), _ptr(S), mu.size)

    def getState(self):
        mu = np.zeros(14); S = np.zeros((14, 14))
        self.L.ref_get_state14(self.h, _ptr(mu), _ptr(S))
        return mu

    def getSigma(self):
        mu = np.zeros(14); S = np.zeros((14, 14))
        self.L.ref_get_state14(self.h, _ptr(mu), _ptr(S))
        return S

    def feature(self, i):
        o = abi.EkfFeatureInfo()
        self.L.ref_get_feature(self.h, int(i), C.byref(o))
        return o

    def template(self, i, which=0):
        w = self.cfg.window_size
        out = np.zeros((w, w), dtype=np.uint8)
        self.L.ref_get_template(self.h, int(i), int(which), _ptr(out))
        return out

    def S_blocks(self):
        out = np.zeros((self.numOfFeatures(), 2, 2))
        self.L.ref_get_S_blocks(self.h, _ptr(out))
        return out

    def deleted(self):
        out = []
        for i in range(self.L.ref_num_deleted(self.h)):
            ri = np.zeros(1, dtype=np.int32); xyz = np.zeros(3); cov = np.zeros(9)
            self.L.ref_get_deleted(self.h, i, _ptr(ri), _ptr(xyz), _ptr(cov))
            out.append((int(ri[0]), xyz, cov))
        return out

    def getPointsFeatures(self):
        """RosVSLAM::getPointsFeatures, compiled from RosVSLAMRansac.cpp."""
        rows = self.L.ref_points_features(self.h, None, 0)
        out = np.zeros((rows, 12))
        if rows:
            self.L.ref_points_features(self.h, _ptr(out), rows)
        return out

    def rts_epoch(self, MU, SIGMA, MU_S, SIGMA_S, dTspeed, dRspeed, deltaT):
        mu = np.array(MU, dtype=np.float64).copy(); sg = np.array(SIGMA, dtype=np.float64).reshape(13, 13).copy()
        mus = np.ascontiguousarray(MU_S, dtype=np.float64); sgs = np.ascontiguousarray(SIGMA_S, dtype=np.float64)
        a = np.ascontiguousarray(dTspeed, dtype=np.float64); b = np.ascontiguousarray(dRspeed, dtype=np.float64)
        self.L.ref_rts_epoch(self.h, _ptr(mu), _ptr(sg), _ptr(mus), _ptr(sgs), _ptr(a), _ptr(b), float(deltaT))
        return mu, sg


def find_match(frame, tmpl, h, S, sigma_size=3.0, fp64=False):
    """Patch::findMatch of the reference for one feature -> (u, v) or (-1, -1)."""
    L = lib(fp64)
    frame = np.ascontiguousarray(frame, dtype=np.uint8); tmpl = np.ascontiguousarray(tmpl, dtype=np.uint8)
    h = np.ascontiguousarray(h, dtype=np.float64); S = np.ascontiguousarray(S, dtype=np.float64)
    uv = np.zeros(2, dtype=np.int32)
    L.ref_find_match(_ptr(frame), frame.shape[1], frame.shape[0], frame.strides[0], _ptr(tmpl), tmpl.shape[0], _ptr(h), _ptr(S),
                     float(sigma_size), _ptr(uv))
    return int(uv[0]), int(uv[1])
