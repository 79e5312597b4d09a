"""Seeded synthetic MonoSLAM sequences for the BASELINE.json configs (SURVEY.md §8(d)).

The reference ships no data; its own end-to-end "test" is a Gazebo world (README.md:43-62).  This
generator replaces that harness with deterministic numpy code: a pinhole+distortion camera
(camModel.cpp:68-138 conventions), a constant-velocity trajectory integrated with the filter's own
motion model (vslamRansac.cpp:1575-1589), world points and per-frame 8-bit images in which each
feature's fixed random template is pasted at its rounded ground-truth projection (so NCC == 1.0 at
exactly one pixel).  Pure numpy: no oracle, no CUDA.
"""
from __future__ import annotations

import dataclasses
import numpy as np

Q0 = np.array([0.0, 0.0, -0.707106781, 0.707106781])  # vslamRansac.cpp:180 (w, x, y, z)


@dataclasses.dataclass
class Camera:
    fx: float = 525.0
    fy: float = 525.0
    u0: float = 320.0
    v0: float = 240.0
    k1: float = -0.05
    k2: float = 0.01
    k3: float = 0.0
    p1: float = 1e-3
    p2: float = -5e-4

    def project(self, pc: np.ndarray) -> np.ndarray:
        """camModel.cpp:113-138 for an array of camera-frame points (.., 3) -> pixels (.., 2)."""
        x1 = pc[..., 0] / pc[..., 2]
        y1 = pc[..., 1] / pc[..., 2]
        r2 = x1 * x1 + y1 * y1
        l = 1 + self.k1 * r2 + self.k2 * r2 * r2 + self.k3 * r2 * r2 * r2
        x2 = x1 * l + 2 * self.p1 * x1 * y1 + self.p2 * (r2 + 2 * x1 * x1)
        y2 = y1 * l + 2 * self.p2 * x1 * y1 + self.p1 * (r2 + 2 * y1 * y1)
        return np.stack([self.fx * x2 + self.u0, self.fy * y2 + self.v0], axis=-1)

    def unproject(self, px: np.ndarray) -> np.ndarray:
        """camModel.cpp:140-176 (50 fixed-point iterations) -> rays (.., 3) with z = 1."""
        x2 = (px[..., 0] - self.u0) / self.fx
        y2 = (px[..., 1] - self.v0) / self.fy
        x1, y1 = x2.copy(), y2.copy()
        for _ in range(50):
            r2 = x1 * x1 + y1 * y1
            l = 1 + self.k1 * r2 + self.k2 * r2 * r2 + self.k3 * r2 * r2 * r2
            dx = 2 * self.p1 * x1 * y1 + self.p2 * (r2 + 2 * x1 * x1)
            dy = 2 * self.p2 * x1 * y1 + self.p1 * (r2 + 2 * y1 * y1)
            x1 = (x2 - dx) / l
            y1 = (y2 - dy) / l
        return np.stack([x1, y1, np.ones_like(x1)], axis=-1)


def quat2rot(q: np.ndarray) -> np.ndarray:
    """vslamRansac.cpp:1408-1421 (w first, un-normalised form)."""
    qr, qi, qj, qk = q
    return np.array([
        [qr * qr + qi * qi - qj * qj - qk * qk, -2 * qr * qk + 2 * qi * qj, 2 * qr * qj + 2 * qi * qk],
        [2 * qr * qk + 2 * qi * qj, qr * qr - qi * qi + qj * qj - qk * qk, -2 * qr * qi + 2 * qj * qk],
        [-2 * qr * qj + 2 * qi * qk, 2 * qr * qi + 2 * qj * qk, qr * qr - qi * qi - qj * qj + qk * qk]])


def quat_mul(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """vslamRansac.cpp:1423-1460 (Yupsilon(a) @ b)."""
    r1, x1, y1, z1 = a
    Y = np.array([[r1, -x1, -y1, -z1], [x1, r1, -z1, y1], [y1, z1, r1, -x1], [z1, -y1, x1, r1]])
    return Y @ b


def vec2quat(v: np.ndarray) -> np.ndarray:
    a = np.linalg.norm(v)
    if a == 0:
        return np.array([1.0, 0.0, 0.0, 0.0])
    return np.concatenate([[np.cos(a / 2)], v * np.sin(a / 2) / a])


@dataclasses.dataclass
class Scene:
    """A synthetic sequence: call frame(t) for images, feature_pixels for the frame-0 seeds."""
    n_features: int = 50
    width: int = 640
    height: int = 480
    n_frames: int = 16
    seed: int = 1234
    window: int = 11
    fps: float = 30.0
    speed: float = 0.2        # |v| m/s
    omega: float = 0.1        # |w| rad/s
    accel_sigma: float = 0.01  # per-frame velocity perturbation (matches sigma_v, sigma_w)
    depth_range: tuple = (2.0, 12.0)
    border: int = 36          # frame-0 seeds stay this far from the image border
    hard: bool = False        # N(0,20^2) pixel noise + 2 % displaced outliers
    outlier_frac: float = 0.02
    outlier_shift: int = 8
    noise_sigma: float = 20.0
    visible_every: int = 1    # > 1: after frame 0 only every visible_every-th feature's template is in the image (m = N / visible_every matches)
    template_smooth: float = 0.0  # > 0: low-pass templates (Gaussian sigma in px) that survive motion-blur prediction
    planar: bool = False      # a ground robot's camera: y = 0, q = (w, 0, q_y, 0) (identity at frame 0), moving in the x-z plane and
                              # turning about y only, so that forsePlane's pseudo-measurements (vslamRansac.cpp:1245-1272) hold;
                              # the filter's prior orientation is Q0, so set its camera state to (r[0], q[0]) before adding features
    camera: Camera | None = None  # the calibration frames are rendered with (config_overrides reports it); None: Camera(u0=W/2, v0=H/2)

    def __post_init__(self):
        rng = np.random.default_rng(self.seed)
        self.cam = self.camera if self.camera is not None else Camera(u0=self.width / 2.0, v0=self.height / 2.0)
        T = self.n_frames
        dT = 1.0 / self.fps
        # trajectory (world-frame v, body-frame w), integrated like Predict_State
        v = np.zeros((T, 3)); w = np.zeros((T, 3))
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        e = rng.normal(size=3); e /= np.linalg.norm(e)
        in_plane = np.array([1.0, 0.0, 1.0]) if self.planar else np.ones(3)      # v components kept
        about_y = np.array([0.0, 1.0, 0.0]) if self.planar else np.ones(3)       # w components kept
        if self.planar:
            d = d * in_plane / np.linalg.norm(d * in_plane); e = np.array([0.0, np.sign(e[1]) or 1.0, 0.0])
        v[0] = self.speed * d; w[0] = self.omega * e
        for t in range(1, T):
            v[t] = v[t - 1] + rng.normal(scale=self.accel_sigma, size=3) * in_plane
            w[t] = w[t - 1] + rng.normal(scale=self.accel_sigma, size=3) * about_y
        r = np.zeros((T, 3)); q = np.zeros((T, 4)); q[0] = np.array([1.0, 0.0, 0.0, 0.0]) if self.planar else Q0
        for t in range(1, T):
            r[t] = r[t - 1] + dT * v[t]
            q[t] = quat_mul(q[t - 1], vec2quat(dT * w[t]))
        self.r, self.q, self.v, self.w = r, q, v, w
        self.stamps = 1.0 + np.arange(T) * dT
        # frame-0 seeds on a jittered grid (min separation > window)
        N = self.n_features
        W, H, b = self.width, self.height, self.border
        aspect = (W - 2 * b) / (H - 2 * b)
        ny = max(1, int(np.floor(np.sqrt(N / aspect))))
        nx = int(np.ceil(N / ny))
        while nx * ny < N:
            nx += 1
        cw = (W - 2 * b) / nx; ch = (H - 2 * b) / ny
        jx = max(0.0, (cw - self.window - 2) / 2); jy = max(0.0, (ch - self.window - 2) / 2)
        cells = rng.permutation(nx * ny)[:N]
        gx = cells % nx; gy = cells // nx
        px = b + (gx + 0.5) * cw + rng.uniform(-jx, jx, size=N)
        py = b + (gy + 0.5) * ch + rng.uniform(-jy, jy, size=N)
        self.feature_pixels = np.stack([np.round(px), np.round(py)], axis=1).astype(np.float32)
        depth = rng.uniform(*self.depth_range, size=N)
        rays = self.cam.unproject(self.feature_pixels.astype(np.float64))
        pc = rays * depth[:, None]
        self.points = r[0][None, :] + pc @ quat2rot(q[0]).T
        self.templates = rng.integers(0, 256, size=(N, self.window, self.window), dtype=np.uint8)
        if self.template_smooth > 0:
            k = int(3 * self.template_smooth) + 1
            g = np.exp(-0.5 * (np.arange(-k, k + 1) / self.template_smooth) ** 2); g /= g.sum()
            big = rng.normal(size=(N, self.window + 2 * k, self.window + 2 * k))
            sm = np.apply_along_axis(lambda v: np.convolve(v, g, mode="valid"), 1, big)
            sm = np.apply_along_axis(lambda v: np.convolve(v, g, mode="valid"), 2, sm)
            lo = sm.min(axis=(1, 2), keepdims=True); hi = sm.max(axis=(1, 2), keepdims=True)
            self.templates = np.round((sm - lo) / (hi - lo) * 255).astype(np.uint8)
        self.outliers = np.zeros(N, dtype=bool)
        if self.hard:
            k = max(1, int(round(self.outlier_frac * N)))
            self.outliers[rng.choice(N, size=k, replace=False)] = True

    # ------------------------------------------------------------------------------------------
    def projections(self, t: int):
        """Ground-truth pixel positions (N,2) and camera-frame depth (N,) at frame t."""
        Rcw = quat2rot(self.q[t] * np.array([1.0, -1.0, -1.0, -1.0]))
        pc = (self.points - self.r[t][None, :]) @ Rcw.T
        with np.errstate(divide="ignore", invalid="ignore"):
            uv = self.cam.project(pc)
        return uv, pc[:, 2]

    def frame(self, t: int) -> np.ndarray:
        """H x W uint8 image of frame t."""
        rng = np.random.default_rng([self.seed, 7919, t])
        img = rng.integers(0, 256, size=(self.height, self.width), dtype=np.uint8)
        uv, z = self.projections(t)
        half = self.window // 2
        for i in range(self.n_features):
            if not (z[i] > 0 and np.isfinite(uv[i]).all()):
                continue
            u = int(np.round(uv[i, 0])); v = int(np.round(uv[i, 1]))
            if t > 0 and self.visible_every > 1 and i % self.visible_every:
                continue
            if self.outliers[i] and t > 0:
                u += self.outlier_shift
            x0, y0 = u - half, v - half
            if x0 < 0 or y0 < 0 or x0 + self.window > self.width or y0 + self.window > self.height:
                continue
            img[y0:y0 + self.window, x0:x0 + self.window] = self.templates[i]
        if self.hard and t > 0:
            noise = rng.normal(scale=self.noise_sigma, size=img.shape)
            img = np.clip(np.round(img.astype(np.float64) + noise), 0, 255).astype(np.uint8)
        return img

    def picks(self, t: int, n: int) -> np.ndarray:
        """Pre-drawn stand-ins for rand() (vslamRansac.cpp:989) for frame t."""
        rng = np.random.default_rng([self.seed, 104729, t])
        return rng.integers(0, 2 ** 31 - 1, size=max(1, n), dtype=np.uint32)

    def config_overrides(self) -> dict:
        """ekf_config fields for this scene (SURVEY.md §8(d))."""
        c = self.cam
        return dict(fx=c.fx, fy=c.fy, u0=c.u0, v0=c.v0, k1=c.k1, k2=c.k2, k3=c.k3, p1=c.p1, p2=c.p2,
                    window_size=self.window, sigma_pixel=2, sigma_size=3, kernel_size=1000000000,
                    T_camera=0.0, rho_0=0.1, sigma_rho_0=0.25, scale=1, forsePlane=0,
                    sigma_vx=0.01, sigma_vy=0.01, sigma_vz=0.01, sigma_wx=0.01, sigma_wy=0.01,
                    sigma_wz=0.01, min_features=0, max_features=1000000, xyz_conversion=0)


def match_batch_inputs(n_frames=256, features_per_frame=200, width=1920, height=1080, window=11,
                       seed=1239, s_diag=16.0, pred_sigma=3.0):
    """BASELINE config 5: frames, templates, predicted h and 2x2 S blocks for the stateless
    batched matcher.  Returns dict of numpy arrays (host)."""
    rng = np.random.default_rng(seed)
    F, M, w = n_frames, features_per_frame, window
    frames = rng.integers(0, 256, size=(F, height, width), dtype=np.uint8)
    templates = rng.integers(0, 256, size=(F, M, w, w), dtype=np.uint8)
    half = w // 2
    truth = np.zeros((F, M, 2), dtype=np.int32)
    # grid placement so templates never overlap within a frame
    nx = int(np.ceil(np.sqrt(M * width / height))); ny = int(np.ceil(M / nx))
    cw = (width - 80) / nx; ch = (height - 80) / ny
    for f in range(F):
        cells = rng.permutation(nx * ny)[:M]
        u = (40 + (cells % nx + 0.5) * cw + rng.uniform(-(cw - w - 2) / 2, (cw - w - 2) / 2, size=M)).round().astype(np.int32)
        v = (40 + (cells // nx + 0.5) * ch + rng.uniform(-(ch - w - 2) / 2, (ch - w - 2) / 2, size=M)).round().astype(np.int32)
        truth[f, :, 0] = u; truth[f, :, 1] = v
        for i in range(M):
            frames[f, v[i] - half:v[i] - half + w, u[i] - half:u[i] - half + w] = templates[f, i]
    h = truth.astype(np.float64) + rng.normal(scale=pred_sigma, size=(F, M, 2))
    S = np.zeros((F, M, 2, 2))
    off = rng.uniform(-0.2, 0.2, size=(F, M)) * s_diag
    S[..., 0, 0] = s_diag * rng.uniform(0.9, 1.1, size=(F, M))
    S[..., 1, 1] = s_diag * rng.uniform(0.9, 1.1, size=(F, M))
    S[..., 0, 1] = off; S[..., 1, 0] = off
    return dict(frames=frames, templates=templates.reshape(F * M, w, w), h=h.reshape(F * M, 2),
                S=S.reshape(F * M, 4), truth=truth.reshape(F * M, 2))
