"""Python mirror of the reference's `class VSlamFilter` (mono-slam/src/vslamRansac.hpp:27-141) over
the C ABI.  Same method names, argument meaning and call order as the reference class; Eigen / OpenCV
types become numpy arrays.  Used by the tests and bench.py; the C++ twin is host/vslam_filter.hpp.
"""
import ctypes as C

import numpy as np

from . import _abi
from ._lib import lib


class EkfError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class VSlamFilter:
    """VSlamFilter(cfg) — cfg is an EkfConfig (see default_config) instead of a libconfig file name
    (vslamRansac.cpp:142).  feature_capacity bounds the map size of this handle."""

    def __init__(self, cfg=None, feature_capacity=128, device=0):
        self.L = lib()
        self.cfg = cfg if cfg is not None else _abi.default_config()
        h = C.c_void_p()
        rc = self.L.ekf_create(C.byref(self.cfg), int(feature_capacity), int(device), C.byref(h))
        if rc != 0:
            raise EkfError(f"ekf_create failed with {rc} "
                           f"({'unsupported configuration' if rc == _abi.EKF_ERR_UNSUPPORTED else 'see stderr'})")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.ekf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise EkfError(f"ekf error {rc}: {self.L.ekf_last_error(self.h).decode()}")
        return rc

    # ---- the per-frame path ------------------------------------------------------------------
    def captureNewFrame(self, img, stamp=-1.0):
        """vslamRansac.cpp:226-245; img is an HxW (gray) or HxWx3 (BGR) uint8 numpy array (host) — copied,
        resized by 1 / cfg.scale and converted to gray inside the call."""
        img = np.ascontiguousarray(img, dtype=np.uint8)
        if img.ndim == 3:
            self._ck(self.L.ekf_capture_frame_bgr(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0], float(stamp)))
        else:
            self._ck(self.L.ekf_capture_frame(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0], float(stamp)))

    def returnGrayImg(self):
        """vslamRansac.cpp:1364."""
        w, h = C.c_int(0), C.c_int(0)
        self._ck(self.L.ekf_get_frame(self.h, None, C.byref(w), C.byref(h)))
        out = np.zeros((h.value, w.value), dtype=np.uint8)
        self._ck(self.L.ekf_get_frame(self.h, _ptr(out), C.byref(w), C.byref(h)))
        return out

    def captureNewFrame_device(self, dev_ptr, width, height, stride, stamp=-1.0):
        """Same for a frame already in device memory (raw pointer, e.g. tensor.data_ptr())."""
        self._ck(self.L.ekf_capture_frame_device(self.h, C.c_void_p(int(dev_ptr)), width, height, stride, float(stamp)))

    def predict(self, dv=(0.0, 0.0, 0.0), dw=(0.0, 0.0, 0.0), vcontrol=False):
        a = np.asarray(dv, dtype=np.float64); b = np.asarray(dw, dtype=np.float64)
        self._ck(self.L.ekf_predict(self.h, _ptr(a), _ptr(b), int(bool(vcontrol))))

    def match(self, want_count=True):
        n = C.c_int(0)
        self._ck(self.L.ekf_match(self.h, C.byref(n) if want_count else None))
        return n.value

    def update_after_match(self, picks=None):
        p = np.ascontiguousarray(picks if picks is not None else np.zeros(0), dtype=np.uint32)
        self._ck(self.L.ekf_update_after_match(self.h, _ptr(p), int(p.size)))

    def update(self, picks=None):
        """vslamRansac.cpp:868; `picks` replaces rand() (vslamRansac.cpp:989)."""
        p = np.ascontiguousarray(picks if picks is not None else np.zeros(0), dtype=np.uint32)
        self._ck(self.L.ekf_update(self.h, _ptr(p), int(p.size)))

    def inject_match(self, i, zu, zv, accepted=True):
        self._ck(self.L.ekf_inject_match(self.h, int(i), float(zu), float(zv), int(bool(accepted))))

    # ---- map management ----------------------------------------------------------------------
    def addFeature(self, u, v):
        return self._ck(self.L.ekf_add_feature(self.h, float(u), float(v)))

    def removeFeature(self, i):
        self._ck(self.L.ekf_remove_feature(self.h, int(i)))

    def findNewFeatures(self, num=-1):
        """vslamRansac.cpp:783-839; returns the number of features added."""
        return self._ck(self.L.ekf_find_new_features(self.h, int(num)))

    def detect_corners(self, num):
        out = np.zeros((1024, 2), dtype=np.float32); n = C.c_int(0)
        self._ck(self.L.ekf_detect_corners(self.h, int(num), _ptr(out), C.byref(n)))
        return out[:n.value].copy()

    def convert2XYZ_ifLinear(self, i):
        """vslamRansac.cpp:741-772."""
        self._ck(self.L.ekf_convert2xyz_if_linear(self.h, int(i)))

    def convert2XYZ_ifLinearAll(self):
        """vslamRansac.cpp:775-780."""
        self._ck(self.L.ekf_convert2xyz_if_linear_all(self.h))

    # ---- accessors ---------------------------------------------------------------------------
    def numOfFeatures(self):
        return self.L.ekf_num_features(self.h)

    def state_dim(self):
        return self.L.ekf_state_dim(self.h)

    def getState(self):
        out = np.zeros(14)
        self._ck(self.L.ekf_get_state(self.h, _ptr(out)))
        return out

    def getSigma(self):
        out = np.zeros((14, 14))
        self._ck(self.L.ekf_get_sigma(self.h, _ptr(out)))
        return out

    def Covariance_Parameter(self):
        v = C.c_double(0)
        self._ck(self.L.ekf_covariance_parameter(self.h, C.byref(v)))
        return v.value

    def getDt(self):
        return self.L.ekf_get_dt(self.h)

    def returnCentrPatchIndx(self, i):
        out = np.zeros(2, dtype=np.float32)
        self._ck(self.L.ekf_get_center(self.h, int(i), _ptr(out)))
        return out

    def feature(self, i):
        o = _abi.EkfFeatureInfo()
        self._ck(self.L.ekf_get_feature(self.h, int(i), C.byref(o)))
        return o

    def deleted(self):
        """VSlamFilter::deleted_patches (vslamRansac.cpp:394-404): list of (real_index, XYZ_pos[3], cov_4_delete[9])."""
        out = []
        for i in range(self.L.ekf_num_deleted(self.h)):
            o = _abi.EkfDeletedInfo()
            self._ck(self.L.ekf_get_deleted(self.h, i, C.byref(o)))
            out.append((o.real_index, np.array(o.xyz_pos), np.array(o.cov_4_delete)))
        return out

    def getPointsFeatures(self):
        """RosVSLAM::getPointsFeatures (RosVSLAMRansac.cpp:340-418): (last real_index + 1) x 12."""
        rows = C.c_int(0)
        self._ck(self.L.ekf_get_points_features(self.h, None, 0, C.byref(rows)))
        out = np.zeros((rows.value, 12))
        self._ck(self.L.ekf_get_points_features(self.h, _ptr(out), rows.value, C.byref(rows)))
        return out

    def rts_epoch(self, MU, SIGMA, MU_S, SIGMA_S, dTspeed, dRspeed, deltaT):
        """VSlamFilter::rts_epoch (vslamRansac.cpp:423-449) on 13-dimensional camera states; returns (MU, SIGMA)."""
        mu = np.array(MU, dtype=np.float64).copy(); sg = np.array(SIGMA, dtype=np.float64).reshape(13, 13).copy()
        mus = np.ascontiguousarray(MU_S, dtype=np.float64); sgs = np.ascontiguousarray(SIGMA_S, dtype=np.float64)
        a = np.ascontiguousarray(dTspeed, dtype=np.float64); b = np.ascontiguousarray(dRspeed, dtype=np.float64)
        assert mu.size == 13 and mus.size == 13 and sgs.size == 169
        self._ck(self.L.ekf_rts_epoch(self.h, _ptr(mu), _ptr(sg), _ptr(mus), _ptr(sgs), _ptr(a), _ptr(b), float(deltaT)))
        return mu, sg

    def template(self, i, which=0):
        w = self.cfg.window_size
        out = np.zeros((w, w), dtype=np.uint8)
        self._ck(self.L.ekf_get_template(self.h, int(i), int(which), _ptr(out)))
        return out

    def stats(self):
        s = _abi.EkfStepStats()
        self._ck(self.L.ekf_get_step_stats(self.h, C.byref(s)))
        return s

    def get_full(self):
        n = self.state_dim()
        mu = np.zeros(n); S = np.zeros((n, n))
        self._ck(self.L.ekf_get_full(self.h, _ptr(mu), _ptr(S), n))
        return mu, S

    def set_full(self, mu, S):
        mu = np.ascontiguousarray(mu, dtype=np.float64); S = np.ascontiguousarray(S, dtype=np.float64)
        n = self.state_dim()
        if mu.size != n or S.shape != (n, n):
            raise ValueError("set_full: shape mismatch")
        self._ck(self.L.ekf_set_full(self.h, _ptr(mu), _ptr(S), n))

    def S_blocks(self):
        out = np.zeros((self.numOfFeatures(), 2, 2))
        self._ck(self.L.ekf_get_S_blocks(self.h, _ptr(out)))
        return out

    def set_profiling(self, on=True):
        self._ck(self.L.ekf_set_profiling(self.h, int(bool(on))))

    def profile(self, reset=True):
        """dict class -> (ms, launches) accumulated since the last reset."""
        p = _abi.EkfProfile()
        self._ck(self.L.ekf_get_profile(self.h, C.byref(p), int(bool(reset))))
        return {name: (p.ms[i], p.launches[i]) for i, name in enumerate(_abi.PROF_CLASSES)}

    def set_symmetric_downdate(self, on=True):
        self._ck(self.L.ekf_set_symmetric_downdate(self.h, int(bool(on))))

    def debug_time_downdate(self, reps=20):
        """Mean duration (ms) of one covariance-downdate launch timed ALONE (diagnostic; perturbs Sigma by rounding errors)."""
        ms = C.c_float(0)
        self._ck(self.L.ekf_debug_time_downdate(self.h, int(reps), C.byref(ms)))
        return float(ms.value)

    def set_stream(self, cuda_stream_ptr):
        self._ck(self.L.ekf_set_stream(self.h, C.c_void_p(int(cuda_stream_ptr) if cuda_stream_ptr else 0)))

    def sync(self):
        self._ck(self.L.ekf_sync(self.h))

    # ---- large map split across GPUs (row-block partitioned update, ekf_dist_*) -------------------
    def dist_attach(self, nccl_id: bytes, rank: int, world: int):
        buf = (C.c_char * 128).from_buffer_copy(bytes(nccl_id))
        self._ck(self.L.ekf_dist_attach(self.h, C.cast(buf, C.c_void_p), int(rank), int(world)))

    def dist_detach(self):
        self._ck(self.L.ekf_dist_detach(self.h))

    def dist_info(self):
        r, w, b = C.c_int(0), C.c_int(0), C.c_int64(0)
        self._ck(self.L.ekf_dist_info(self.h, C.byref(r), C.byref(w), C.byref(b)))
        return dict(rank=r.value, world=w.value, allgather_bytes=b.value, peer_memory=bool(self.L.ekf_dist_peer_memory(self.h)))


def nccl_unique_id(libnccl_path=None) -> bytes:
    """Loads libnccl (the copy torch uses unless a path is given) and returns a fresh 128-byte id."""
    load_nccl(libnccl_path)
    buf = (C.c_char * 128)()
    rc = lib().ekf_dist_unique_id(C.cast(buf, C.c_void_p))
    if rc != 0:
        raise EkfError(f"ekf_dist_unique_id failed: {rc}")
    return bytes(buf)


def load_nccl(libnccl_path=None):
    if libnccl_path is None:
        try:
            import os
            import nvidia.nccl as _n
            cand = os.path.join(os.path.dirname(_n.__file__), "lib", "libnccl.so.2")
            libnccl_path = cand if os.path.exists(cand) else None
        except Exception:
            libnccl_path = None
    rc = lib().ekf_dist_load_nccl(libnccl_path.encode() if libnccl_path else None)
    if rc != 0:
        raise EkfError(f"ekf_dist_load_nccl failed: {rc}")


def match_batch(frames_dev, n_frames, width, height, stride, templates_dev, features_per_frame, window,
                h_dev, S_dev, out_uv_dev, out_score_dev, sigma_size=3.0, ncc_threshold=0.8, search_clamp=20.0,
                stream=0):
    """ekf_match_batch on raw device pointers (ints)."""
    rc = lib().ekf_match_batch(C.c_void_p(frames_dev), n_frames, width, height, stride, C.c_void_p(templates_dev),
                               features_per_frame, window, C.c_void_p(h_dev), C.c_void_p(S_dev), float(sigma_size),
                               float(ncc_threshold), float(search_clamp), C.c_void_p(out_uv_dev),
                               C.c_void_p(out_score_dev), C.c_void_p(stream))
    if rc != 0:
        raise EkfError(f"ekf_match_batch failed: {rc}")


class FilterBatch:
    """B independent VSlamFilter instances stepped together on one device (BASELINE config 3).
    Seed it from a single VSlamFilter, optionally perturb the camera states, then call
    captureNewFrame / step once per frame.  With set_cameras, filters follow cameras of their own:
    captureNewFrames then takes one frame (and time stamp) per camera."""

    def __init__(self, cfg, n_filters, feature_capacity=32, device=0, large=False):
        """large: up to 128 features per filter (ekf_batch_create_large; the update of a filter above 32 features runs on a
        cluster of CTAs).  Without it the capacity is at most 32."""
        self.L = lib()
        self.cfg = cfg
        h = C.c_void_p()
        create = self.L.ekf_batch_create_large if large else self.L.ekf_batch_create
        rc = create(C.byref(cfg), int(n_filters), int(feature_capacity), int(device), C.byref(h))
        if rc != 0:
            raise EkfError(f"{'ekf_batch_create_large' if large else 'ekf_batch_create'} failed with {rc}")
        self.h = h
        self.B = int(n_filters)
        self.n_cameras = 1
        self.camera_of = np.zeros(self.B, dtype=np.int32)
        self.frame_sizes = None   # (n_cameras, 2) width, height of each camera's frame (set_frame_sizes), None: the whole frame
        self.camera_settings = None   # (n_cameras, 3) window_size, scale, kernel_size (set_camera_settings), None: the batch's
        self._cams = None   # (mu14, Sigma14) of every filter, read once per step for the views

    @classmethod
    def from_config(cls, cfg, n_filters, feature_capacity=32, device=0, large=False, archive=0):
        """A batch from the configuration a VSlamFilter takes: created with motion blur, resize and forsePlane off (which
        ekf_batch_create requires), then set_motion_blur(cfg.kernel_size) when blur is on, set_scale(cfg.scale),
        set_force_plane(cfg.forsePlane) and, when archive > 0, set_archive(archive)."""
        base = _abi.EkfConfig.from_buffer_copy(cfg)
        base.kernel_size, base.scale, base.forsePlane = _abi.default_config().kernel_size, 1, 0
        batch = cls(base, n_filters, feature_capacity=feature_capacity, device=device, large=large)
        batch.cfg = cfg
        if cfg.kernel_size < 100000:
            batch.set_motion_blur(cfg.kernel_size)
        batch.set_scale(cfg.scale)
        batch.set_force_plane(cfg.forsePlane)
        if archive:
            batch.set_archive(archive)
        return batch

    @classmethod
    def from_configs(cls, cfgs, camera_of, feature_capacity=32, large=False, archive=0, device=0):
        """A batch whose filter f runs configuration cfgs[f] (one EkfConfig per filter) and follows camera camera_of[f]: the
        rigs of several configuration files in one batch.  Filters of one camera must agree on window_size, scale and
        kernel_size, and every filter on search_clamp, forsePlane, xyz_conversion and abs_int_quirk (ValueError naming the
        filter and field otherwise).  The batch is created with the largest window, then set_cameras, set_camera_settings,
        set_force_plane, set_configs and, when archive > 0, set_archive."""
        cfgs = list(cfgs)
        cam = np.ascontiguousarray(camera_of, dtype=np.int32).reshape(-1)
        settings = _abi.camera_settings_of(cfgs, cam)
        base = _abi.EkfConfig.from_buffer_copy(cfgs[0])
        base.window_size = int(settings[:, 0].max())
        base.kernel_size, base.scale, base.forsePlane = _abi.default_config().kernel_size, 1, 0
        batch = cls(base, len(cfgs), feature_capacity=feature_capacity, device=device, large=large)
        batch.set_cameras(settings.shape[0], cam)
        batch.set_camera_settings(settings)
        batch.set_force_plane(cfgs[0].forsePlane)
        batch.set_configs(cfgs)
        if archive:
            batch.set_archive(archive)
        return batch

    def close(self):
        if getattr(self, "h", None):
            self.L.ekf_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise EkfError(f"ekf batch error {rc}: {self.L.ekf_batch_last_error(self.h).decode()}")
        return rc

    def _set_cfg(self, **fields):
        """self.cfg follows what the batch runs (set_configs checks the shared fields against it); a copy, so that the
        caller's configuration stays as it was."""
        self.cfg = _abi.EkfConfig.from_buffer_copy(self.cfg)
        for k, v in fields.items():
            setattr(self.cfg, k, v)

    def describe(self):
        d = _abi.EkfBatchDesc()
        self._ck(self.L.ekf_batch_describe(self.h, C.byref(d)))
        return d

    def set_stream(self, cuda_stream_ptr):
        self._ck(self.L.ekf_batch_set_stream(self.h, C.c_void_p(int(cuda_stream_ptr) if cuda_stream_ptr else 0)))

    def sync(self):
        self._ck(self.L.ekf_batch_sync(self.h))

    def seed_from(self, filt):
        self._cams = None
        self._ck(self.L.ekf_batch_seed_from(self.h, filt.h))

    def set_camera_states(self, mu14):
        a = np.ascontiguousarray(mu14, dtype=np.float64)
        if a.shape != (self.B, 14):
            raise ValueError("set_camera_states expects (n_filters, 14)")
        self._cams = None
        self._ck(self.L.ekf_batch_set_camera_states(self.h, _ptr(a)))

    def captureNewFrame(self, img, stamp=-1.0):
        """As VSlamFilter.captureNewFrame: img is an HxW (gray) or HxWx3 (BGR) uint8 host array, resized by 1 / scale
        (set_scale) and converted to gray inside the call."""
        img = np.ascontiguousarray(img, dtype=np.uint8)
        fn = self.L.ekf_batch_capture_frame_bgr if img.ndim == 3 else self.L.ekf_batch_capture_frame
        self._ck(fn(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0], float(stamp)))

    def captureNewFrame_device(self, dev_ptr, width, height, stride, stamp=-1.0):
        self._ck(self.L.ekf_batch_capture_frame_device(self.h, C.c_void_p(int(dev_ptr)), width, height, stride, float(stamp)))

    def set_cameras(self, n, camera_of=None):
        """Filter f follows camera camera_of[f] in [0, n) (None: filter f follows camera f, n == n_filters).  Forgets the
        captured frames; every camera's clock becomes camera 0's."""
        a = None if camera_of is None else np.ascontiguousarray(camera_of, dtype=np.int32)
        if a is not None and a.shape != (self.B,):
            raise ValueError("camera_of expects (n_filters,)")
        self._ck(self.L.ekf_batch_set_cameras(self.h, int(n), _ptr(a) if a is not None else None))
        self.n_cameras = int(n)
        self.camera_of = a.copy() if a is not None else np.arange(self.B, dtype=np.int32)
        self.frame_sizes = None
        self.camera_settings = None   # set_cameras clears the camera table

    def set_camera_settings(self, settings):
        """Window, scale and blur threshold per camera (ekf_batch_set_camera_settings): an (n_cameras, 3) int array of
        (window_size, scale, kernel_size), filter f running with row camera_of[f] as a batch of that window, scale and
        kernel_size would; None returns every camera to the batch's values.  A window above the batch's window_size, a window
        change under features and set_scale / set_motion_blur while a table is set raise EkfError.  A scale change forgets
        the captured frames."""
        if settings is None:
            self._ck(self.L.ekf_batch_set_camera_settings(self.h, None))
            self.camera_settings = None
            return
        a = np.asarray(settings, dtype=np.int64)
        if a.shape != (self.n_cameras, 3):
            raise ValueError(f"set_camera_settings expects ({self.n_cameras}, 3)")
        i32 = np.iinfo(np.int32)
        bad = np.argwhere((a < i32.min) | (a > i32.max))
        if bad.size:   # the C rows are int32: a wider value would wrap (a huge kernel_size could turn blur on)
            c, k = bad[0]
            raise ValueError(f"camera {c}: {_abi.CAMERA_FIELDS[k]} = {a[c, k]} does not fit an int32")
        rows = (_abi.EkfCameraSettings * self.n_cameras)(*[_abi.EkfCameraSettings(int(w), int(s), int(k), 0) for w, s, k in a])
        self._ck(self.L.ekf_batch_set_camera_settings(self.h, rows))
        self.camera_settings = a.copy()

    def window_of(self, f):
        """The template side filter f runs with: its camera's window (set_camera_settings), or the batch's."""
        if self.camera_settings is None:
            return int(self.cfg.window_size)
        return int(self.camera_settings[self.camera_of[int(f)], 0])

    def _stamps(self, stamps, n=None):
        if stamps is None:
            return None
        s = np.ascontiguousarray(np.broadcast_to(np.asarray(stamps, dtype=np.float64), (self.n_cameras if n is None else n,)))
        return s

    @staticmethod
    def _list(ids, what):
        a = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        if a.size < 1:
            raise ValueError(f"{what} must list at least one entry")
        return a

    def set_frame_sizes(self, sizes):
        """A frame size per camera: (n_cameras, 2) width, height in input pixels (before the resize by 1 / scale), or None for the
        whole frame.  Camera c's frame is then the top-left of slot c of the stack captureNewFrames passes.  Forgets the
        captured frames."""
        if sizes is None:
            self._ck(self.L.ekf_batch_set_frame_sizes(self.h, None))
            self.frame_sizes = None
            return
        a = np.ascontiguousarray(sizes, dtype=np.int32)
        if a.shape != (self.n_cameras, 2):
            raise ValueError(f"set_frame_sizes expects ({self.n_cameras}, 2)")
        self._ck(self.L.ekf_batch_set_frame_sizes(self.h, _ptr(a)))
        self.frame_sizes = a.copy()

    def captureNewFrames(self, frames, stamps=None, cameras=None):
        """captureNewFrame for every camera: frames is (n_cameras, H, W) gray or (n_cameras, H, W, 3) BGR uint8 (host),
        stamps one per camera or None.  A strided (n, H, W) view with padded rows is passed as it is.  With set_frame_sizes,
        frames may also be a list of per-camera arrays of the declared sizes; they are packed into a zero-padded stack whose
        slot is the largest width and height.
        cameras: capture these cameras only (ekf_batch_capture_camera_frames): frames is then (len(cameras), H, W[, 3]) or a
        list of per-camera arrays of the declared sizes, in list order, and stamps one per listed camera.  The other cameras
        keep their frames and clocks."""
        cams = None if cameras is None else self._list(cameras, "cameras")
        n = self.n_cameras if cams is None else cams.size
        if isinstance(frames, (list, tuple)):
            if self.frame_sizes is None or len(frames) != n:
                raise ValueError("a list of frames needs set_frame_sizes and one frame per (listed) camera")
            ids = range(n) if cams is None else [int(c) for c in cams]
            fl = [np.asarray(x, dtype=np.uint8) for x in frames]
            for c, x in zip(ids, fl):
                if x.shape[:2] != (int(self.frame_sizes[c, 1]), int(self.frame_sizes[c, 0])) or x.ndim != fl[0].ndim:
                    raise ValueError(f"frame of camera {c} has shape {x.shape}, camera {c} is {tuple(self.frame_sizes[c])} (width, height)")
            H, W = int(self.frame_sizes[:, 1].max()), int(self.frame_sizes[:, 0].max())
            frames = np.zeros((len(fl), H, W) + fl[0].shape[2:], np.uint8)
            for k, x in enumerate(fl):
                frames[k, :x.shape[0], :x.shape[1]] = x
        f = np.asarray(frames, dtype=np.uint8)
        if f.ndim not in (3, 4) or f.shape[0] != n:
            raise ValueError(f"captureNewFrames expects ({n}, H, W) or ({n}, H, W, 3) uint8")
        rowb = f.shape[2] * (3 if f.ndim == 4 else 1)
        if not (f.strides[-1] == 1 and (f.ndim == 3 or f.strides[2] == 3) and f.strides[1] >= rowb
                and f.strides[0] == f.strides[1] * f.shape[1]):
            f = np.ascontiguousarray(f)
        s = self._stamps(stamps, n)
        sp = _ptr(s) if s is not None else None
        if cams is None:
            fn = self.L.ekf_batch_capture_frames_bgr if f.ndim == 4 else self.L.ekf_batch_capture_frames
            self._ck(fn(self.h, _ptr(f), f.shape[2], f.shape[1], f.strides[1], sp))
        else:
            fn = self.L.ekf_batch_capture_camera_frames_bgr if f.ndim == 4 else self.L.ekf_batch_capture_camera_frames
            self._ck(fn(self.h, int(n), _ptr(cams), _ptr(f), f.shape[2], f.shape[1], f.strides[1], sp))

    def captureNewFrames_device(self, dev_ptr, width, height, stride, stamps=None, cameras=None):
        """captureNewFrames from a gray stack in device memory: frame c at dev_ptr + c * height * stride.  cameras: the
        stack holds len(cameras) frames, frame k camera cameras[k]'s (ekf_batch_capture_camera_frames_device)."""
        if cameras is None:
            s = self._stamps(stamps)
            self._ck(self.L.ekf_batch_capture_frames_device(self.h, C.c_void_p(int(dev_ptr)), int(width), int(height), int(stride),
                                                            _ptr(s) if s is not None else None))
            return
        cams = self._list(cameras, "cameras")
        s = self._stamps(stamps, cams.size)
        self._ck(self.L.ekf_batch_capture_camera_frames_device(self.h, int(cams.size), _ptr(cams), C.c_void_p(int(dev_ptr)), int(width),
                                                               int(height), int(stride), _ptr(s) if s is not None else None))

    INTRINSICS = _abi.INTRINSICS

    def set_intrinsics(self, params):
        """Intrinsics per filter, columns in INTRINSICS order (EkfConfig's): a (9,) array for every filter, a (n_filters, 9)
        array with filter f's row f, or None for the configuration's.  For intrinsics per camera, pass params[camera_of]."""
        if params is None:
            self._ck(self.L.ekf_batch_set_intrinsics(self.h, None))
            return
        a = np.asarray(params, dtype=np.float64)
        if a.shape not in ((9,), (self.B, 9)):
            raise ValueError(f"set_intrinsics expects (9,) or ({self.B}, 9)")
        a = np.ascontiguousarray(np.broadcast_to(a, (self.B, 9)))
        self._ck(self.L.ekf_batch_set_intrinsics(self.h, _ptr(a)))

    def set_filter_params(self, rows):
        """Tuning per filter (ekf_batch_set_filter_params): a sequence of n_filters _abi.EkfFilterParams, or None for the
        configuration's values."""
        if rows is None:
            self._ck(self.L.ekf_batch_set_filter_params(self.h, None))
            return
        if len(rows) != self.B:
            raise ValueError(f"set_filter_params expects {self.B} rows")
        arr = rows if isinstance(rows, C.Array) else (_abi.EkfFilterParams * self.B)(*rows)
        self._ck(self.L.ekf_batch_set_filter_params(self.h, arr))

    def set_configs(self, cfgs):
        """Filter f runs configuration cfgs[f], as a VSlamFilter given it would: its intrinsics and its tuning (both tables).
        cfgs holds n_filters EkfConfig (one per camera: [cfgs[c] for c in camera_of]); None returns every filter to the
        batch's configuration.  ValueError, naming the field and the filter, when a field every filter shares
        (_abi.BATCH_SHARED_FIELDS) differs from the batch's configuration as it stands (set_motion_blur, set_scale and
        set_force_plane included), or when a row is invalid; every row is checked before either table changes.  With a camera
        table (set_camera_settings), window_size, scale and kernel_size of cfgs[f] are checked against row camera_of[f] of it
        instead.  nInitFeatures is not read."""
        if cfgs is None:
            self.set_intrinsics(None)
            self.set_filter_params(None)
            return
        cfgs = list(cfgs)
        if len(cfgs) != self.B:
            raise ValueError(f"set_configs expects {self.B} configurations")
        if self.camera_settings is None:
            cam, rows = _abi.batch_rows(self.cfg, cfgs)
        else:
            cam, rows = _abi.batch_rows_per_camera(self.cfg, cfgs, self.camera_settings, self.camera_of)
        self.set_intrinsics(cam)
        self.set_filter_params(rows)

    def set_detect_budget(self, nbytes):
        """Device scratch of one chunk of cameras in the per-camera detector (default 1 GiB)."""
        self._ck(self.L.ekf_batch_set_detect_budget(self.h, int(nbytes)))

    def returnGrayImg(self, camera=0):
        """vslamRansac.cpp:1364: the gray frame the filters of `camera` work on (after resize)."""
        w, h = C.c_int(0), C.c_int(0)
        self._ck(self.L.ekf_batch_get_camera_frame(self.h, int(camera), None, C.byref(w), C.byref(h)))
        out = np.zeros((h.value, w.value), dtype=np.uint8)
        self._ck(self.L.ekf_batch_get_camera_frame(self.h, int(camera), _ptr(out), C.byref(w), C.byref(h)))
        return out

    def getDt(self, f=None):
        """getDt of filter f (its camera's dT), or of every filter when f is None."""
        out = np.zeros(self.B, dtype=np.float64)
        self._ck(self.L.ekf_batch_get_dt(self.h, _ptr(out)))
        return out if f is None else float(out[int(f)])

    def set_scale(self, scale):
        """EkfConfig.scale for the batch's captures (default 1); the configuration's intrinsics are the resized image's."""
        self._ck(self.L.ekf_batch_set_scale(self.h, int(scale)))
        self._set_cfg(scale=int(scale))

    def set_force_plane(self, on=True):
        """EkfConfig.forsePlane for every filter (vslamRansac.cpp:1245-1272; default off)."""
        self._ck(self.L.ekf_batch_set_force_plane(self.h, int(bool(on))))
        self._set_cfg(forsePlane=int(bool(on)))

    def step(self, picks=None, dv=(0.0, 0.0, 0.0), dw=(0.0, 0.0, 0.0), vcontrol=False, filters=None):
        """predict + update of every filter.  dv / dw are 3-vectors for every filter, or (n_filters, 3) arrays with vcontrol
        a bool or an (n_filters,) array: controls per filter (ekf_batch_step_controls).
        filters: step these filters only (strictly ascending; ekf_batch_step_filters), the others stay as they are; dv / dw
        are then (3,) or (len(filters), 3) and vcontrol a bool or a (len(filters),) array."""
        p = np.ascontiguousarray(picks if picks is not None else np.zeros(0), dtype=np.uint32)
        a = np.ascontiguousarray(dv, dtype=np.float64); b = np.ascontiguousarray(dw, dtype=np.float64)
        vc = np.asarray(vcontrol)
        self._cams = None
        if filters is not None:
            fl = self._list(filters, "filters")
            n = fl.size
            a = np.ascontiguousarray(np.broadcast_to(a, (n, 3))); b = np.ascontiguousarray(np.broadcast_to(b, (n, 3)))
            v = np.ascontiguousarray(np.broadcast_to(vc, (n,)), dtype=np.int32)
            self._ck(self.L.ekf_batch_step_filters(self.h, int(n), _ptr(fl), _ptr(a), _ptr(b), _ptr(v), _ptr(p), int(p.size)))
            return
        if a.shape == (3,) and b.shape == (3,) and vc.ndim == 0:
            self._ck(self.L.ekf_batch_step(self.h, _ptr(a), _ptr(b), int(bool(vc)), _ptr(p), int(p.size)))
            return
        a = np.ascontiguousarray(np.broadcast_to(a, (self.B, 3))); b = np.ascontiguousarray(np.broadcast_to(b, (self.B, 3)))
        v = np.ascontiguousarray(np.broadcast_to(vc, (self.B,)), dtype=np.int32)
        self._ck(self.L.ekf_batch_step_controls(self.h, _ptr(a), _ptr(b), _ptr(v), _ptr(p), int(p.size)))

    def convert2XYZ_ifLinearAll(self):
        """vslamRansac.cpp:775-780 on every filter of the batch."""
        self._ck(self.L.ekf_batch_convert2xyz_if_linear_all(self.h))

    def camera_states(self, want_sigma=False):
        mu = np.zeros((self.B, 14)); st = np.zeros((self.B, _abi.BATCH_STAT_FIELDS), dtype=np.int32)
        S = np.zeros((self.B, 14, 14)) if want_sigma else None
        self._ck(self.L.ekf_batch_get_camera_states(self.h, _ptr(mu), _ptr(S) if want_sigma else None, _ptr(st)))
        return (mu, S, st) if want_sigma else (mu, st)

    def numOfFeatures(self, f):
        return self._ck(self.L.ekf_batch_num_features(self.h, int(f)))

    def state_dim(self, f):
        return self._ck(self.L.ekf_batch_state_dim(self.h, int(f)))

    def get_full(self, f):
        n = self.state_dim(f)
        mu = np.zeros(n); S = np.zeros((n, n))
        self._ck(self.L.ekf_batch_get_full(self.h, int(f), _ptr(mu), _ptr(S), n))
        return mu, S

    def set_full(self, f, mu, S):
        mu = np.ascontiguousarray(mu, dtype=np.float64); S = np.ascontiguousarray(S, dtype=np.float64)
        n = self.state_dim(f)
        if mu.size != n or S.shape != (n, n):
            raise ValueError("set_full: shape mismatch")
        self._cams = None
        self._ck(self.L.ekf_batch_set_full(self.h, int(f), _ptr(mu), _ptr(S), n))

    def feature(self, f, i):
        o = _abi.EkfFeatureInfo()
        self._ck(self.L.ekf_batch_get_feature(self.h, int(f), int(i), C.byref(o)))
        return o

    def addFeature(self, f, u, v):
        """vslamRansac.cpp:309-371 on filter f; 1 added, 0 rejected by isInsideImage."""
        return self._ck(self.L.ekf_batch_add_feature(self.h, int(f), float(u), float(v)))

    def removeFeature(self, f, i):
        """vslamRansac.cpp:373-421 on feature i of filter f (archived under the rule of set_archive)."""
        self._ck(self.L.ekf_batch_remove_feature(self.h, int(f), int(i)))

    # ---- the feature archive and the map export ---------------------------------------------------
    def set_archive(self, capacity):
        """Keep every filter's VSlamFilter::deleted_patches (vslamRansac.cpp:394-404), up to `capacity` records per filter
        (0: off, the default).  Empties every archive."""
        self._ck(self.L.ekf_batch_set_archive(self.h, int(capacity)))

    def num_deleted(self):
        """Records in each filter's archive (int32, n_filters)."""
        out = np.zeros(self.B, dtype=np.int32)
        self._ck(self.L.ekf_batch_num_deleted(self.h, _ptr(out)))
        return out

    def deleted(self, f):
        """Filter f's archive as VSlamFilter.deleted(): list of (real_index, XYZ_pos[3], cov_4_delete[9])."""
        n = C.c_int(0)
        self._ck(self.L.ekf_batch_get_deleted(self.h, int(f), None, 0, C.byref(n)))
        recs = (_abi.EkfDeletedInfo * max(n.value, 1))()
        self._ck(self.L.ekf_batch_get_deleted(self.h, int(f), recs, n.value, C.byref(n)))
        return [(o.real_index, np.array(o.xyz_pos), np.array(o.cov_4_delete)) for o in recs[:n.value]]

    def points_features(self, first=0, count=None):
        """RosVSLAM::getPointsFeatures (RosVSLAMRansac.cpp:340-418) for filters [first, first + count) from one export:
        a list of (rows_f, 12) matrices, as VSlamFilter.getPointsFeatures() returns them."""
        count = self.B - int(first) if count is None else int(count)
        rows = np.zeros(max(count, 1), dtype=np.int32)
        self._ck(self.L.ekf_batch_get_points_features(self.h, int(first), count, None, 0, _ptr(rows)))
        cap = int(rows[:count].max())
        out = np.zeros((count, cap, 12))
        self._ck(self.L.ekf_batch_get_points_features(self.h, int(first), count, _ptr(out), cap, _ptr(rows)))
        return [out[k, :rows[k]].copy() for k in range(count)]

    def getPointsFeatures(self, f):
        """Filter f's (rows, 12) matrix, as VSlamFilter.getPointsFeatures()."""
        return self.points_features(f, 1)[0]

    def resample(self, ancestors):
        """Filter f becomes an exact copy of filter ancestors[f] ((n_filters,) ints), both as they stood before the call
        (ekf_batch_resample): state, covariance, feature table, templates, archive, intrinsics row, counters.  Every
        ancestors[f] follows f's camera.  systematic_ancestors builds such a vector from weights."""
        a = np.ascontiguousarray(ancestors, dtype=np.int32)
        if a.shape != (self.B,):
            raise ValueError(f"resample expects ({self.B},) ancestors")
        self._cams = None
        self._ck(self.L.ekf_batch_resample(self.h, _ptr(a)))

    def view(self, f):
        """Filter f as the object keyframes.KeyframeRecorder drives (getState, getSigma, Covariance_Parameter,
        getPointsFeatures, Point4sba).  Every view of the batch reads its camera state from one cached read-back per step."""
        return BatchFilterView(self, int(f))

    def _camera_cache(self):
        if self._cams is None:
            mu, S, _ = self.camera_states(want_sigma=True)
            self._cams = (mu, S)
        return self._cams

    def _num(self, num):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(num, dtype=np.int32), (self.B,)))

    def detect_corners(self, num):
        """findNewFeatures' detection alone (vslamRansac.cpp:783-831) on every filter; num is one count or one per filter
        (capped at 32).  Returns a list of (k_b, 2) float32 arrays."""
        a = self._num(num)
        xy = np.zeros((self.B, _abi.BATCH_MAX_CORNERS, 2), dtype=np.float32); n = np.zeros(self.B, dtype=np.int32)
        self._ck(self.L.ekf_batch_detect_corners(self.h, _ptr(a), _ptr(xy), _ptr(n)))
        return [xy[b, :n[b]].copy() for b in range(self.B)]

    def findNewFeatures(self, num=None):
        """vslamRansac.cpp:783-839 on every filter: num is one count or one per filter (<= 0: none — unlike the single
        filter's nInitFeatures); None takes each filter's EKF_BSTAT_TOPUP of the last step.  Returns the features each
        filter added."""
        added = np.zeros(self.B, dtype=np.int32)
        a = self._num(num) if num is not None else None
        self._ck(self.L.ekf_batch_find_new_features(self.h, _ptr(a) if a is not None else None, _ptr(added)))
        return added

    def set_topup(self, on=True):
        """on: step() ends like ekf_update_after_match — removals, findNewFeatures(EKF_BSTAT_TOPUP), XYZ conversion."""
        self._ck(self.L.ekf_batch_set_topup(self.h, int(bool(on))))

    def last_added(self):
        """Features each filter added in the last step."""
        out = np.zeros(self.B, dtype=np.int32)
        self._ck(self.L.ekf_batch_last_added(self.h, _ptr(out)))
        return out

    def set_motion_blur(self, kernel_size):
        """Patch::blur (Patch.cpp:50-57) in every filter's predict: kernel_size as EkfConfig.kernel_size (>= 100000: off,
        the default); T_camera is the batch configuration's."""
        self._ck(self.L.ekf_batch_set_motion_blur(self.h, int(kernel_size)))
        self._set_cfg(kernel_size=int(kernel_size))

    def last_blur_counts(self):
        """Templates each filter blurred in the last step (int32, zeros with blur off)."""
        out = np.zeros(self.B, dtype=np.int32)
        self._ck(self.L.ekf_batch_last_blur_counts(self.h, _ptr(out)))
        return out

    def template(self, f, i, which=0):
        """Patch::patch (which 0) or Patch::matching_patch (1) of feature i of filter f: window_of(f) x window_of(f)."""
        w = self.window_of(f)
        out = np.zeros((w, w), dtype=np.uint8)
        self._ck(self.L.ekf_batch_get_template(self.h, int(f), int(i), int(which), _ptr(out)))
        return out

    def kernel_launches(self):
        return int(self.L.ekf_batch_kernel_launches(self.h))

    def update_clusters(self):
        """(CTAs per filter in the update, clusters the device holds at once; 0 for a one-CTA update)."""
        c, r = C.c_int(0), C.c_int(0)
        self._ck(self.L.ekf_batch_update_clusters(self.h, C.byref(c), C.byref(r)))
        return c.value, r.value

    def last_match_deferred(self):
        """(filter, feature) pairs of the last step that the warp-per-feature matcher left to the CTA matcher."""
        return self._ck(self.L.ekf_batch_last_match_deferred(self.h))

    def last_step_ms(self):
        out = np.zeros(3, dtype=np.float32)
        self._ck(self.L.ekf_batch_last_step_ms(self.h, _ptr(out)))
        return dict(predict=float(out[0]), match=float(out[1]), update=float(out[2]))


def systematic_ancestors(weights, u, camera_of=None):
    """Ancestors for FilterBatch.resample from one weight per filter: systematic resampling with offset u in [0, 1), separately
    within each camera's filters (camera_of: (n_filters,) ints, None: one group).  A group of M filters draws M times at
    (u + k) / M of its cumulative normalised weight.  Every filter drawn at least once keeps its own slot; the extra copies
    fill the slots of the filters not drawn, in ascending order, so no filter is both read and overwritten.  Equal weights
    give the identity.  ValueError for negative or non-finite weights and for a group whose weights sum to 0."""
    w = np.asarray(weights, dtype=np.float64)
    if w.ndim != 1:
        raise ValueError("weights must be one per filter")
    if not np.all(np.isfinite(w)) or np.any(w < 0):
        raise ValueError("weights must be finite and non-negative")
    if not 0.0 <= float(u) < 1.0:
        raise ValueError("u must lie in [0, 1)")
    B = w.size
    cam = np.zeros(B, dtype=np.int64) if camera_of is None else np.asarray(camera_of, dtype=np.int64)
    if cam.shape != (B,):
        raise ValueError("camera_of must be one camera per filter")
    anc = np.arange(B, dtype=np.int32)
    for c in np.unique(cam):
        idx = np.flatnonzero(cam == c)
        M = idx.size
        top = w[idx].max()
        if top <= 0:
            raise ValueError(f"the weights of camera {int(c)} sum to 0")
        cum = np.cumsum(w[idx] / top)   # scaled so that equal weights give exact integer steps
        pos = (float(u) + np.arange(M)) * (cum[-1] / M)
        draws = np.minimum(np.searchsorted(cum, pos, side="right"), M - 1)
        count = np.bincount(draws, minlength=M)
        extra = np.repeat(np.arange(M), np.maximum(count - 1, 0))
        free = np.flatnonzero(count == 0)
        anc[idx[free]] = idx[extra]
    return anc


class BatchFilterView:
    """One filter of a FilterBatch with the accessors of VSlamFilter that keyframes.KeyframeRecorder reads."""

    Point4sba = np.zeros((1, 3), dtype=np.int32)   # the node's projection list stays empty (monoslam_ransac.cpp:689-752 is dead)

    def __init__(self, batch, f):
        self.batch, self.f = batch, f

    def getState(self):
        return self.batch._camera_cache()[0][self.f].copy()

    def getSigma(self):
        return self.batch._camera_cache()[1][self.f].copy()

    def Covariance_Parameter(self):
        """ekf_covariance_parameter (vslamRansac.cpp:854-855), the same sums in the same order."""
        S = self.batch._camera_cache()[1][self.f]
        P = 0.0
        P += float(S[0, 0]) + float(S[1, 1]) + float(S[2, 2])
        P += float(S[4, 4]) + float(S[5, 5]) + float(S[6, 6]) + float(S[3, 3])
        return P

    def getPointsFeatures(self):
        return self.batch.getPointsFeatures(self.f)

    def getDt(self):
        return self.batch.getDt(self.f)
