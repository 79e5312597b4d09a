// csrc/ekf_predict.cu — K1 (motion model + block covariance propagation), K2 (batched h(x), compact H,
// gating, 2x2 innovation blocks), K4e (quaternion renormalisation), K6 (add / remove feature edits).
// SURVEY.md §8(a) rows a3-a10, a16, a21, a22.  Citations V: = mono-slam/src/vslamRansac.cpp.
#include "ekf_kernels.h"
#include "ekf_blur.cuh"
#include "ekf_math.cuh"

// ------------------------------------------------------------------------------------------------
// K1: Sigma <- Fc Sigma Fc^T + Qtot, Fc = I with a 13x13 corner (V:451-480).  Only the 13 camera
// rows and 13 camera columns change: algorithmic traffic 4*13*n*8 B instead of the dense 4 n^3 flops.
//   block 0            : 13x13 corner  (F C F^T + Q) and Predict_State -> ctl->mu_cam_new
//   blocks 1..         : thread j (>= 13): column j of rows 0:13  <- F * Sigma[0:13, j]
//                                          row j of cols 0:13     <- Sigma[j, 0:13] * F^T
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void predict_cov_body(int bid, double* __restrict__ Sigma, int ld, int n, const double* __restrict__ mu,
                                                 DevCtl* ctl, const DevCfg& cfg, double dT, double3 dv, double3 dw, int vcontrol) {
  __shared__ double F[169];
  __shared__ double C[169], T[169], Q[169];
  if (threadIdx.x == 0) {
    const double ctrl[3] = {dw.x, dw.y, dw.z};
    double mu13[13];
    for (int i = 0; i < 13; ++i) mu13[i] = mu[i];
    d_system_jacobian(mu13, dT, ctrl, F);
  }
  __syncthreads();
  if (bid == 0) {
    for (int e = threadIdx.x; e < 169; e += blockDim.x) C[e] = Sigma[(size_t)(e / 13) * ld + (e % 13)];
    __syncthreads();
    // Q = (F6 * Vs) * F6^T, Vs = (V/dT)/dT diagonal, F6 = F[:, 7:13] (V:463-473)
    for (int e = threadIdx.x; e < 169; e += blockDim.x) {
      const int a = e / 13, b = e % 13;
      double s = 0;
      for (int k = 0; k < 6; ++k) {
        const double vmax = vcontrol ? cfg.Vmax[k] : cfg.Vmax[k] * 2.0;
        const double vs = (vmax / dT) / dT;
        // (F6*Vs)[a,k] = sum_c F6[a,c]*Vs[c,k]: only c == k is non-zero (exact zeros elsewhere)
        s += (F[a * 13 + 7 + k] * vs) * F[b * 13 + 7 + k];
      }
      Q[e] = s;
      double t = 0;
      for (int k = 0; k < 13; ++k) t += F[a * 13 + k] * C[k * 13 + b];
      T[e] = t;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 169; e += blockDim.x) {
      const int a = e / 13, b = e % 13;
      double s = 0;
      for (int k = 0; k < 13; ++k) s += T[a * 13 + k] * F[b * 13 + k];
      Sigma[(size_t)a * ld + b] = s + Q[e];
    }
    if (threadIdx.x == 0) {
      double X[13];
      for (int i = 0; i < 13; ++i) X[i] = mu[i];
      const double a[3] = {dv.x, dv.y, dv.z}, b[3] = {dw.x, dw.y, dw.z};
      d_predict_state(X, a, b, dT);
      for (int i = 0; i < 13; ++i) ctl->mu_cam_new[i] = X[i];
    }
    return;
  }
  const int j = 13 + (bid - 1) * blockDim.x + threadIdx.x;
  if (j >= n) return;
  double x[13], y[13];
  // column j of the camera rows (coalesced across threads)
  for (int c = 0; c < 13; ++c) x[c] = Sigma[(size_t)c * ld + j];
  for (int a = 0; a < 13; ++a) {
    double s = 0;
    for (int c = 0; c < 13; ++c) s += F[a * 13 + c] * x[c];
    y[a] = s;
  }
  for (int a = 0; a < 13; ++a) Sigma[(size_t)a * ld + j] = y[a];
  // row j of the camera columns
  double* row = Sigma + (size_t)j * ld;
  for (int c = 0; c < 13; ++c) x[c] = row[c];
  for (int a = 0; a < 13; ++a) {
    double s = 0;
    for (int c = 0; c < 13; ++c) s += x[c] * F[a * 13 + c];
    y[a] = s;
  }
  for (int a = 0; a < 13; ++a) row[a] = y[a];
}

// ------------------------------------------------------------------------------------------------
// K2: per-feature prediction (V:482-602): rho <= 0 guard, h, compact H, in-image / in-front gate,
// template reset (Patch::blur with blur disabled, Patch.cpp:50-57), 2x2 diagonal block of
// St = H Sigma H^T + sigma_px^2 I (the only part of St the reference consumes, V:875), and — by the
// last block to finish — the ordered compaction that assigns position_in_z (V:584-592).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int predict_features_body(int i, const double* cam, const double* __restrict__ mu, FeatTab ft, int N, FrameView fr,
                                                     const DevCfg& cfg) {
  int ok = 0;
  if (i < N) {
    const int pos = ft.pos[i], coding = ft.coding[i];
    const int fsz = coding ? 3 : 6;
    double fs[6];
    for (int c = 0; c < fsz; ++c) fs[c] = mu[pos + c];
    bool skip = false;
    if (!coding && fs[5] <= 0) {  // V:517-522
      ft.removef[i] = 1;
      skip = true;
    }
    if (!skip) {
      double qc[4] = {cam[3], -cam[4], -cam[5], -cam[6]}, Rcw[9], hi[2], Hc[26], hcz;
      d_quat2rot(qc, Rcw);
      d_feature_hH(cfg.cam, fs, coding, cam, qc, Rcw, hi, Hc, &hcz);
      const int half = cfg.window / 2;
      ok = (hi[0] > half && hi[1] > half && hi[0] < fr.w - half && hi[1] < fr.h - half) && (hcz >= 0);  // V:529,1644-1652
      if (ok) {
        ft.h[2 * i] = hi[0]; ft.h[2 * i + 1] = hi[1];
        for (int c = 0; c < 26; ++c) ft.Hc[26 * i + c] = Hc[c];
      }
    }
    ft.innov[i] = ok; ft.li[i] = 0; ft.hi[i] = 0;  // Patch::setIsInInnovation (Patch.cpp:123-132)
  }
  // matching_patch <- patch for gated-in features (Patch.cpp:54-56): 16-byte chunks of the record
  if (ok) {
    const int chunks = cfg.tstride >> 4;
    const uint4* src = reinterpret_cast<const uint4*>(ft.patch + (size_t)i * cfg.tstride);
    uint4* dst = reinterpret_cast<uint4*>(ft.mpatch + (size_t)i * cfg.tstride);
    for (int c = 0; c < chunks; ++c) dst[c] = src[c];
  }
  return ok;
}

// K1 and K2 in ONE launch: CTAs [0, nb_cov) propagate the covariance, CTAs [nb_cov, ..) predict the features.  The two
// are independent once every feature CTA forms the predicted camera state itself (Predict_State on the thirteen old camera
// entries: the bits CTA 0 writes to ctl->mu_cam_new); mu is committed — and the in-innovation list compacted — by the last
// CTA of the grid to finish, after every CTA has read the old mu (one launch and one dependent-launch gap less than the
// two kernels this replaces).
__global__ void __launch_bounds__(256) k_predict_fused(double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu, FeatTab ft,
                                                       int N, FrameView fr, DevCtl* ctl, DevCfg cfg, double dT, double3 dv, double3 dw,
                                                       int vcontrol, int nb_cov) {
  __shared__ int is_last;
  __shared__ double camS[13];
  if ((int)blockIdx.x < nb_cov) {
    predict_cov_body((int)blockIdx.x, Sigma, ld, n, mu, ctl, cfg, dT, dv, dw, vcontrol);
  } else {
    if (threadIdx.x == 0) {
      double X[13];
      for (int i = 0; i < 13; ++i) X[i] = mu[i];
      const double a[3] = {dv.x, dv.y, dv.z}, b[3] = {dw.x, dw.y, dw.z};
      d_predict_state(X, a, b, dT);
      for (int i = 0; i < 13; ++i) camS[i] = X[i];
    }
    __syncthreads();
    double cam[13];
    for (int c = 0; c < 13; ++c) cam[c] = camS[c];
    predict_features_body(((int)blockIdx.x - nb_cov) * blockDim.x + threadIdx.x, cam, mu, ft, N, fr, cfg);
  }
  // last CTA of the grid: commit the predicted camera state and compact
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&ctl->ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x < 13) mu[threadIdx.x] = ctl->mu_cam_new[threadIdx.x];
  const int m = block_compact(ft.innov, N, ft.sel, ft.pos_in_z);
  if (threadIdx.x == 0) {
    ctl->m_innov = m;
    ctl->ticket = 0;
    ctl->blur_count = 0;
    ctl->blur_too_large = 0;
  }
}

// Motion-blur template prediction (V:498-500, 546-548, 575-576; Patch::blur Patch.cpp:50-57; evaluateKernel /
// blurPatch libblur.cpp:17-81).  One CTA per gated-in feature: project the feature from the pose the camera
// will have T_camera * dT later; if that moves the prediction by more than kernel_min_size pixels the
// template is correlated with a normalised line kernel of that displacement (double arithmetic,
// BORDER_REFLECT_101, round-half-even to u8) into matching_patch.  The kernel lives as a bit mask
// (<= 256 x 256); its set coefficients are visited in row-major order like OpenCV's direct filter engine.
// The arithmetic is ekf_blur.cuh, shared with the batched k_batch_predict_blur.
__global__ void __launch_bounds__(128) k_predict_blur(const double* __restrict__ mu, FeatTab ft, int N, DevCtl* ctl, DevCfg cfg,
                                                      double dT) {
  __shared__ unsigned kbits[BLUR_MAXK * BLUR_MAXK / 32];
  __shared__ int s_rows, s_cols, s_do;
  __shared__ double s_kf, s_dx, s_dy;
  const int f = blockIdx.x, tid = threadIdx.x;
  if (f >= N || !ft.innov[f]) return;
  const int w = cfg.window;
  if (tid == 0) {
    s_do = 0;
    double cam[13], rb[3], Rb[9];
    for (int c = 0; c < 13; ++c) cam[c] = mu[c];   // predicted camera state, committed by k_predict_features
    blur_pose(cam, cfg.T_camera, dT, rb, Rb);
    const int pos = ft.pos[f], coding = ft.coding[f];
    double fs[6], ddx, ddy;
    for (int c = 0; c < (coding ? 3 : 6); ++c) fs[c] = mu[pos + c];
    blur_displacement(cfg.cam, fs, coding, rb, Rb, ft.h[2 * f], ft.h[2 * f + 1], &ddx, &ddy);
    int krows = 0, kcols = 0;
    const int d = blur_decide(ddx, ddy, cfg.kernel_min_size, &krows, &kcols);
    if (d < 0) { ctl->blur_too_large = 1; }
    else if (d > 0) { s_do = 1; s_rows = krows; s_cols = kcols; s_dx = ddx; s_dy = ddy; }
  }
  __syncthreads();
  if (!s_do) return;   // matching_patch already holds the unblurred template (k_predict_features)
  const int krows = s_rows, kcols = s_cols;
  for (int e = tid; e < (krows * kcols + 31) / 32; e += 128) kbits[e] = 0u;
  __syncthreads();
  if (tid == 0) {
    // rasterise the line, libblur.cpp:25-43
    const BlurLine L = blur_line(s_dx, s_dy);
    int count = 0;
    for (int i = 0; i < L.length; ++i) {
      int x, y;
      if (blur_line_point(L, i, krows, kcols, &x, &y)) {
        const int bit = x * kcols + y;
        if (!(kbits[bit >> 5] & (1u << (bit & 31)))) { kbits[bit >> 5] |= 1u << (bit & 31); ++count; }
      }
    }
    s_kf = 1.0 / (double)count;   // kernel / sum(kernel): every set coefficient is 1 / count
    atomicAdd(&ctl->blur_count, 1);
  }
  __syncthreads();
  const double kf = s_kf;
  const uint8_t* src = ft.patch + (size_t)f * cfg.tstride;
  uint8_t* dst = ft.mpatch + (size_t)f * cfg.tstride;
  for (int e = tid; e < w * w; e += 128) dst[e] = blur_pixel_bits(src, w, e, kbits, krows, kcols, kf);
}

// 2x2 diagonal block of St = H Sigma H^T + sigma_px^2 I for every gated-in feature (V:598 restricted
// to what V:875 consumes).  One warp per feature: lane b < nd forms column b of Hc * Sigma_sub
// (13 coalesced loads), the 2x2 sums are reduced over lanes with shuffles.
__global__ void __launch_bounds__(128) k_predict_S2(const double* __restrict__ Sigma, int ld, FeatTab ft, int N, DevCfg cfg) {
  const int f = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (f >= N || !ft.innov[f]) return;
  const int pos = ft.pos[f], nd = 7 + (ft.coding[f] ? 3 : 6);
  const double* hc = ft.Hc + 26 * f;
  double t0 = 0, t1 = 0, h0 = 0, h1 = 0;
  if (lane < nd) {
    const int jb = ekf_idx13(lane, pos);
    // all 13 loads of Sigma and of H in flight before the first use (the rolled loop paid the L2 latency per term: 11 us for this
    // kernel); same terms, same order
    double sg[13], ha[13], hb[13];
#pragma unroll
    for (int c = 0; c < 13; ++c) {
      const bool in = c < nd;
      sg[c] = in ? Sigma[(size_t)ekf_idx13(c, pos) * ld + jb] : 0.0;
      ha[c] = in ? hc[c] : 0.0; hb[c] = in ? hc[13 + c] : 0.0;
    }
#pragma unroll
    for (int c = 0; c < 13; ++c)
      if (c < nd) { t0 += ha[c] * sg[c]; t1 += hb[c] * sg[c]; }
    h0 = hc[lane]; h1 = hc[13 + lane];
  }
  double s00 = t0 * h0, s01 = t0 * h1, s10 = t1 * h0, s11 = t1 * h1;
  for (int o = 8; o > 0; o >>= 1) {
    s00 += __shfl_down_sync(0xffffffffu, s00, o, 16); s01 += __shfl_down_sync(0xffffffffu, s01, o, 16);
    s10 += __shfl_down_sync(0xffffffffu, s10, o, 16); s11 += __shfl_down_sync(0xffffffffu, s11, o, 16);
  }
  if (lane == 0) {
    ft.S2[4 * f + 0] = s00 + cfg.sigma_pixel_2; ft.S2[4 * f + 1] = s01;
    ft.S2[4 * f + 2] = s10; ft.S2[4 * f + 3] = s11 + cfg.sigma_pixel_2;
  }
}

// ------------------------------------------------------------------------------------------------
// K4e: normalizeQuaternion (V:1625-1642): q <- q/|q|, Sigma <- Qc Sigma Qc^T with Qc = I except the
// 4x4 block J = (|q|^2 I - q q^T)/|q|^3 on rows/cols 3:7.  Structured: 4 rows + 4 columns.
// Runs only when the preceding stacked update had rows (ctl->k_rows > 0), as in the reference.
// ------------------------------------------------------------------------------------------------
// mu += delta fused in: every CTA forms the updated, not yet normalised quaternion q = mu[3:7] + delta[3:7] itself; thread j
// of the row / column CTAs also commits mu[j] += delta[j] for the entries outside the quaternion; the last CTA of the grid
// (device ticket) writes the quaternion — normalised if the update had rows — after every CTA has read the old one.
// One launch instead of three (apply_delta, normalise, commit).
__global__ void __launch_bounds__(256) k_finish_update(double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu,
                                                       const double* __restrict__ delta, DevCtl* ctl) {
  __shared__ double J[16];
  __shared__ double C[16], T[16];
  __shared__ double qs[4], qn[4];
  __shared__ int is_last;
  const bool rows = ctl->k_rows > 0;
  if (threadIdx.x == 0) {
    double q[4];
    for (int i = 0; i < 4; ++i) q[i] = mu[3 + i] + delta[3 + i];
    const double norma = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    for (int i = 0; i < 4; ++i) { qs[i] = q[i]; qn[i] = q[i] / norma; }
    const double sc = 1 / (norma * norma * norma);
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) J[i * 4 + j] = ((norma * norma) * (i == j ? 1.0 : 0.0) - q[i] * q[j]) * sc;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    if (rows) {
      if (threadIdx.x < 16) C[threadIdx.x] = Sigma[(size_t)(3 + threadIdx.x / 4) * ld + 3 + (threadIdx.x % 4)];
      __syncthreads();
      if (threadIdx.x < 16) {
        const int a = threadIdx.x / 4, b = threadIdx.x % 4;
        double t = 0;
        for (int k = 0; k < 4; ++k) t += J[a * 4 + k] * C[k * 4 + b];
        T[threadIdx.x] = t;
      }
      __syncthreads();
      if (threadIdx.x < 16) {
        const int a = threadIdx.x / 4, b = threadIdx.x % 4;
        double s = 0;
        for (int k = 0; k < 4; ++k) s += T[a * 4 + k] * J[b * 4 + k];
        Sigma[(size_t)(3 + a) * ld + 3 + b] = s;
      }
    }
  } else {
    int j = (blockIdx.x - 1) * blockDim.x + threadIdx.x;  // index over states outside 3..6
    if (j >= 3) j += 4;
    if (j < n) {
      mu[j] += delta[j];
      if (rows) {
        double x[4], y[4];
        for (int c = 0; c < 4; ++c) x[c] = Sigma[(size_t)(3 + c) * ld + j];
        for (int a = 0; a < 4; ++a) {
          double s = 0;
          for (int c = 0; c < 4; ++c) s += J[a * 4 + c] * x[c];
          y[a] = s;
        }
        for (int a = 0; a < 4; ++a) Sigma[(size_t)(3 + a) * ld + j] = y[a];
        double* row = Sigma + (size_t)j * ld + 3;
        for (int c = 0; c < 4; ++c) x[c] = row[c];
        for (int a = 0; a < 4; ++a) {
          double s = 0;
          for (int c = 0; c < 4; ++c) s += x[c] * J[a * 4 + c];
          y[a] = s;
        }
        for (int a = 0; a < 4; ++a) row[a] = y[a];
      }
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&ctl->ticket, 1u);
    is_last = (t == gridDim.x - 1);
    if (is_last) ctl->ticket = 0;
  }
  __syncthreads();
  if (is_last && threadIdx.x < 4) mu[3 + threadIdx.x] = rows ? qn[threadIdx.x] : qs[threadIdx.x];
}

// ------------------------------------------------------------------------------------------------
// K6a: addFeature (V:309-371); the arithmetic is add_feature_* in ekf_math.cuh (shared with k_batch_add).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_add_feature(double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu,
                                                     FeatTab ft, int fidx, FrameView fr, DevCfg cfg, float pfx, float pfy,
                                                     int real_index) {
  __shared__ double A[6 * 7], Ap[6 * 3], fnew[6];
  if (threadIdx.x == 0) add_feature_jacobians(cfg.cam, mu, pfx, pfy, cfg.rho_0, A, Ap, fnew);
  __syncthreads();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) add_feature_cross(Sigma, ld, n, t, A);   // new rows, column t; new columns, row t
  if (blockIdx.x == 0) {
    __shared__ double Tc[6 * 7];
    __syncthreads();
    for (int e = threadIdx.x; e < 42; e += blockDim.x) Tc[e] = add_feature_corner_T(Sigma, ld, A, e);
    __syncthreads();
    for (int e = threadIdx.x; e < 36; e += blockDim.x)
      Sigma[(size_t)(n + e / 6) * ld + n + e % 6] = add_feature_corner(Tc, A, Ap, e, cfg.sigma_pixel_2, cfg.sigma_rho_0);
    if (threadIdx.x < 6) mu[n + threadIdx.x] = fnew[threadIdx.x];
    const int w = cfg.window, w2 = w * w;
    for (int e = threadIdx.x; e < w2; e += blockDim.x) ft.patch[(size_t)fidx * cfg.tstride + e] = add_feature_template_px(fr, w, pfx, pfy, e);
    if (threadIdx.x == 0) add_feature_record(ft, fidx, n, pfx, pfy, real_index);
  }
}

// K6b: removeFeature (V:373-421) for a set of features at once: Sigma'[i,j] = Sigma[map[i], map[j]].
__global__ void k_gather_sigma(const double* __restrict__ src, double* __restrict__ dst, int ld, int n2,
                               const int* __restrict__ map) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j < n2) dst[(size_t)i * ld + j] = src[(size_t)map[i] * ld + map[j]];
}
__global__ void k_gather_vec(const double* __restrict__ src, double* __restrict__ dst, int n2, const int* __restrict__ map) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n2) dst[j] = src[map[j]];
}
// Compacts the feature table in place order-preserving: keep[] lists surviving old indices
// (ascending), newpos[] their new position_in_state.  src/dst are distinct tables.
__global__ void k_gather_features(FeatTab src, FeatTab dst, int N2, const int* __restrict__ keep,
                                  const int* __restrict__ newpos, int w2) {
  const int f = blockIdx.x;
  if (f >= N2) return;
  const int o = keep[f];
  for (int e = threadIdx.x; e < (w2 >> 4); e += blockDim.x) {  // w2 = record stride in bytes
    reinterpret_cast<uint4*>(dst.patch + (size_t)f * w2)[e] = reinterpret_cast<const uint4*>(src.patch + (size_t)o * w2)[e];
    reinterpret_cast<uint4*>(dst.mpatch + (size_t)f * w2)[e] = reinterpret_cast<const uint4*>(src.mpatch + (size_t)o * w2)[e];
  }
  for (int e = threadIdx.x; e < 26; e += blockDim.x) dst.Hc[26 * f + e] = src.Hc[26 * o + e];
  if (threadIdx.x == 0) {
    dst.pos[f] = newpos[f]; dst.coding[f] = src.coding[o]; dst.innov[f] = src.innov[o];
    dst.li[f] = src.li[o]; dst.hi[f] = src.hi[o]; dst.removef[f] = src.removef[o];
    dst.n_tot[f] = src.n_tot[o]; dst.n_find[f] = src.n_find[o]; dst.real_index[f] = src.real_index[o];
    dst.pos_in_z[f] = src.pos_in_z[o]; dst.quality[f] = src.quality[o]; dst.last_ncc[f] = src.last_ncc[o];
    for (int c = 0; c < 2; ++c) {
      dst.center[2 * f + c] = src.center[2 * o + c]; dst.z[2 * f + c] = src.z[2 * o + c];
      dst.h[2 * f + c] = src.h[2 * o + c];
    }
    for (int c = 0; c < 4; ++c) dst.S2[4 * f + c] = src.S2[4 * o + c];
  }
}

// ------------------------------------------------------------------------------------------------
// K6c: convert2XYZ_ifLinear(All) (V:741-780) and inverseDepth2XyzWorld (V:690-738).
// Decisions for all inverse-depth features are taken at once from the pre-conversion state: a
// conversion only touches its own 6 rows / columns (J is the identity elsewhere), so the linearity
// index of a later feature (its own state, mu[0:3] and Sigma[pos+5,pos+5]) is unaffected by earlier
// conversions of the same call.  The arithmetic (quirks included) is xyz_linear_decide / xyz_apply_entry
// in ekf_math.cuh.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_xyz_decide(const double* __restrict__ Sigma, int ld, const double* __restrict__ mu,
                                                    FeatTab ft, int N, DevCfg cfg, int only, int* __restrict__ flag,
                                                    double* __restrict__ yout, double* __restrict__ Jout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int conv = 0;
  if (!ft.coding[i] && (only < 0 || only == i)) {
    const int pos = ft.pos[i];
    double f[6], r[3];
    for (int c = 0; c < 6; ++c) f[c] = mu[pos + c];
    for (int c = 0; c < 3; ++c) r[c] = mu[c];
    conv = xyz_linear_decide(f, r, Sigma[(size_t)(pos + 5) * ld + pos + 5], cfg.linearity_threshold, cfg.abs_int_quirk,
                             yout + 3 * i, Jout + 18 * i);
  }
  flag[i] = conv;
}
// Sigma' = J Sigma J^T for all converted features at once (xyz_apply_entry); rmap[i'] = (src, code).
__global__ void k_xyz_apply(const double* __restrict__ src, double* __restrict__ dst, int ld, int n2, const int2* __restrict__ rmap,
                            const double* __restrict__ Jall) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j >= n2) return;
  dst[(size_t)i * ld + j] = xyz_apply_entry(src, ld, rmap[i], rmap[j], Jall);
}
__global__ void k_xyz_mu(const double* __restrict__ musrc, double* __restrict__ mudst, int n2, const int2* __restrict__ rmap,
                         const double* __restrict__ yall) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n2) return;
  const int2 r = rmap[j];
  mudst[j] = (r.y < 0) ? musrc[r.x] : yall[3 * (r.y >> 2) + (r.y & 3)];
}
__global__ void k_set_pos_coding(FeatTab ft, int N, const int* __restrict__ pos, const int* __restrict__ coding) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) { ft.pos[i] = pos[i]; ft.coding[i] = coding[i]; }
}

// ---- launch wrappers ---------------------------------------------------------------------------
void launch_predict(cudaStream_t st, double* Sigma, int ld, int n, double* mu, FeatTab ft, int N, FrameView fr,
                    DevCtl* ctl, const DevCfg& cfg, double dT, const double dv[3], const double dw[3], int vcontrol,
                    long long* launches) {
  const int nb = 1 + (n - 13 + 255) / 256;
  const int fb = N > 0 ? (N + 255) / 256 : 1;
  k_predict_fused<<<nb + fb, 256, 0, st>>>(Sigma, ld, n, mu, ft, N, fr, ctl, cfg, dT, make_double3(dv[0], dv[1], dv[2]),
                                          make_double3(dw[0], dw[1], dw[2]), vcontrol, nb);
  *launches += 1;
  if (N > 0 && cfg.kernel_min_size < 100000) {   // motion-blur templates enabled
    k_predict_blur<<<N, 128, 0, st>>>(mu, ft, N, ctl, cfg, dT);
    *launches += 1;
  }
  if (N > 0) {
    k_predict_S2<<<(N + 3) / 4, 128, 0, st>>>(Sigma, ld, ft, N, cfg);
    *launches += 1;
  }
}
// mu += delta and, when the update had rows, the quaternion renormalisation with its Jacobian on Sigma (V:1625-1642)
void launch_finish_update(cudaStream_t st, double* Sigma, int ld, int n, double* mu, const double* delta, DevCtl* ctl,
                          long long* launches) {
  const int nb = 1 + (n - 4 + 255) / 256;
  k_finish_update<<<nb, 256, 0, st>>>(Sigma, ld, n, mu, delta, ctl);
  *launches += 1;
}
void launch_add_feature(cudaStream_t st, double* Sigma, int ld, int n, double* mu, FeatTab ft, int fidx, FrameView fr,
                        const DevCfg& cfg, float pfx, float pfy, int real_index, long long* launches) {
  const int nb = (n + 255) / 256;
  k_add_feature<<<nb, 256, 0, st>>>(Sigma, ld, n, mu, ft, fidx, fr, cfg, pfx, pfy, real_index);
  *launches += 1;
}
void launch_gather_state(cudaStream_t st, const double* Ssrc, double* Sdst, int ld, const double* musrc, double* mudst,
                         int n2, const int* map, long long* launches) {
  if (n2 <= 0) return;
  dim3 g((n2 + 255) / 256, n2);
  k_gather_sigma<<<g, 256, 0, st>>>(Ssrc, Sdst, ld, n2, map);
  k_gather_vec<<<(n2 + 255) / 256, 256, 0, st>>>(musrc, mudst, n2, map);
  *launches += 2;
}
void launch_gather_features(cudaStream_t st, FeatTab src, FeatTab dst, int N2, const int* keep, const int* newpos, int w2,
                            long long* launches) {
  if (N2 <= 0) return;
  k_gather_features<<<N2, 64, 0, st>>>(src, dst, N2, keep, newpos, w2);
  *launches += 1;
}
void launch_xyz_decide(cudaStream_t st, const double* Sigma, int ld, const double* mu, FeatTab ft, int N, const DevCfg& cfg, int only,
                       int* flag, double* y, double* J, long long* launches) {
  if (N <= 0) return;
  k_xyz_decide<<<(N + 127) / 128, 128, 0, st>>>(Sigma, ld, mu, ft, N, cfg, only, flag, y, J);
  *launches += 1;
}
void launch_xyz_apply(cudaStream_t st, const double* Ssrc, double* Sdst, int ld, const double* musrc, double* mudst, int n2,
                      const int* rmap, const double* J, const double* y, FeatTab ft, int N, const int* pos, const int* coding,
                      long long* launches) {
  dim3 g((n2 + 255) / 256, n2);
  k_xyz_apply<<<g, 256, 0, st>>>(Ssrc, Sdst, ld, n2, reinterpret_cast<const int2*>(rmap), J);
  k_xyz_mu<<<(n2 + 255) / 256, 256, 0, st>>>(musrc, mudst, n2, reinterpret_cast<const int2*>(rmap), y);
  k_set_pos_coding<<<(N + 255) / 256, 256, 0, st>>>(ft, N, pos, coding);
  *launches += 3;
}
