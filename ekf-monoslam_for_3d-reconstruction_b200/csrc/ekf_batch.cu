// csrc/ekf_batch.cu — batch of independent filters (BASELINE config 3; SURVEY.md §8(e)).
//
// B filters x N <= 32 features (n <= 206).  One filter's covariance is n x ld fp64 (~310 KB at N = 30):
// it does not fit one SM's shared memory, but one CTA per filter keeps it L2-resident for the whole
// step (148 concurrent filters x 310 KB = 46 MB of the 126 MB L2), so HBM sees each Sigma once in and
// once out.  Three launches per step:
//   k_batch_predict  (B CTAs)       motion model, block covariance propagation, h / H / gate, S blocks
//   (k_batch_predict_blur (B CTAs)  motion-blur templates, only once ekf_batch_set_motion_blur switched them on)
//   k_match_filter_batch (N x B)    active search, each filter on its camera's frame (ekf_match.cu)
//   k_batch_update   (B CTAs)       1-point RANSAC, Li update, Hi rescue, Hi update, book-keeping:
//                                   W = Sigma H^T (n x k <= 64) and its Cholesky gain live in shared
//                                   memory, the rank-k downdate Sigma -= V V^T runs on the fp64 tensor
//                                   pipe (DMMA.8x8x4) straight from shared-memory V.  With forsePlane
//                                   (ekf_batch_set_force_plane) the second update adds the plane block.
// plus k_batch_compact when a filter flagged features for deletion or, with cfg.xyz_conversion, has
// inverse-depth features to convert to XYZ (convert2XYZ_ifLinearAll, V:1317): k_batch_update decides the
// conversions, k_batch_compact applies removals and conversions in one pass over Sigma.  With top-up on and a
// filter asking for features (V:1312-1315), that filter's pass removes only; the batched detector
// (ekf_batch_detect.cu) and k_batch_add then add its new features, and a second k_batch_compact converts.
// Frames are captured once per camera (ekf_batch_set_cameras; one camera by default), resized and converted to gray when
// ekf_batch_set_scale / a BGR source ask, into one contiguous stack of n_cameras frames; filter b reads frame cam_of[b] of it,
// and its predict the camera's dT and, from ekf_batch_step_controls, its own controls (BatchStepIn).
// ekf_batch_create_large: up to BNCAP_L = 128 features (n <= 782); the update then runs on a cluster of 2 to 4 CTAs per filter
// (k_batch_update_cluster) and the other kernels take their BNCAP_L instantiations.  Sigma and the compaction scratch are
// B x ncap x ld doubles each: 4.9 MB per filter each at capacity 128, 40 GB in total for 4096 filters.
// Every stage evaluates the same expressions as the single-filter kernels (same device functions).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <string>
#include <type_traits>
#include <vector>

#include <cooperative_groups.h>

#include "../../include/ekf_b200.h"
#include "ekf_blur.cuh"
#include "ekf_cta.cuh"
#include "ekf_factor.cuh"
#include "ekf_handle.h"
#include "ekf_kernels.h"
#include "ekf_math.cuh"
#include "ekf_points.cuh"

namespace cg = cooperative_groups;

#define BK 64                 // measurement rows of one stacked update (<= 32 features)
#define BNCAP 32              // feature capacity of a batched filter created by ekf_batch_create
#define BNCAP_L EKF_BATCH_MAX_FEATURES   // 128: feature capacity of one from ekf_batch_create_large
#define BNMAX (EKF_CAM + 6 * BNCAP + 2)  // 208: state rows rounded up to a multiple of 8
#define BLDW (BK + 4)         // row stride of W / V / Linv in shared memory (conflict-free fragment reads)
#define BUPD_THREADS FACT_THREADS

struct BatchView {
  double* Sigma;        // [B][ncap * ld]
  double* mu;           // [B][ld]
  FeatTab ft;           // every field [B][Ncap]
  DevCtl* ctl;          // [B]
  int* n;               // [B] state dimension
  int* N;               // [B] feature count
  long long sstride;    // doubles between consecutive filters' Sigma
  int ld, Ncap, tstride;
  // XYZ conversions decided for the next k_batch_compact, kept out of FeatTab (single filters have their own arrays)
  int* xyz_flag;        // [B][Ncap] feature converts
  double* xyz_J;        // [B][Ncap][18] its 3 x 6 Jacobian
  double* xyz_y;        // [B][Ncap][3] its XYZ point
  int* xyz_count;       // [B] conversions pending (k_batch_compact resets it)
  int* patchnumbre;     // [B] real_index of the filter's next new feature (VSlamFilter::patchnumbre)
  const CamParams* cam; // [B] intrinsics of each filter (ekf_batch_set_intrinsics); null: every filter uses cfg.cam
};

// The intrinsics filter b projects, linearises and unprojects with.  INTR: the batch has a table (kernels that project take it
// as a template parameter, so that a batch without one runs the code it ran before).  A reference, so that the fields load
// where they are used.
template <bool INTR>
__device__ __forceinline__ const CamParams& filter_cam(const BatchView& bv, const DevCfg& cfg, int b) {
  if constexpr (INTR) return bv.cam[b];
  else return cfg.cam;
}

// convert2XYZ_ifLinear's decision (V:741-772, xyz_linear_decide) for feature i = lane of filter b, if `eligible` and still
// in inverse depth.  Called by the whole of warp 0 (N <= BNCAP = 32); lane 0 stores the filter's count.
__device__ void warp_xyz_decide(const BatchView& bv, int b, const double* Sigma, const double* mu, const FeatTab& ft, int N,
                                bool eligible, const DevCfg& cfg) {
  const int i = threadIdx.x;
  const size_t k = (size_t)b * bv.Ncap + i;
  int conv = 0;
  if (eligible && i < N && !ft.coding[i]) {
    const int pos = ft.pos[i];
    conv = xyz_linear_decide(mu + pos, mu, Sigma[(size_t)(pos + 5) * bv.ld + pos + 5], cfg.linearity_threshold,
                             cfg.abs_int_quirk, bv.xyz_y + 3 * k, bv.xyz_J + 18 * k);
  }
  if (i < N) bv.xyz_flag[k] = conv;
  const int cnt = __popc(__ballot_sync(0xffffffffu, conv));
  if (i == 0) bv.xyz_count[b] = cnt;
}

// The same decisions for up to blockDim.x features, one thread per feature (large batches).  use_alive: only features not
// flagged for removal and other than `victim` are eligible (in a step); otherwise every one (convert2XYZ_ifLinearAll).
// Called by the whole CTA; thread 0 stores the filter's count.
__device__ void cta_xyz_decide(const BatchView& bv, int b, const double* Sigma, const double* mu, const FeatTab& ft, int N,
                               bool use_alive, int victim, const DevCfg& cfg) {
  const int i = threadIdx.x;
  const size_t k = (size_t)b * bv.Ncap + i;
  int conv = 0;
  if (i < N && !ft.coding[i] && (!use_alive || (!ft.removef[i] && i != victim))) {
    const int pos = ft.pos[i];
    conv = xyz_linear_decide(mu + pos, mu, Sigma[(size_t)(pos + 5) * bv.ld + pos + 5], cfg.linearity_threshold,
                             cfg.abs_int_quirk, bv.xyz_y + 3 * k, bv.xyz_J + 18 * k);
  }
  if (i < N) bv.xyz_flag[k] = conv;
  const int cnt = __syncthreads_count(conv);
  if (i == 0) bv.xyz_count[b] = cnt;
}

// Per-filter inputs of a step, uploaded in one copy with the picks; a null field leaves the kernel's scalar argument in place
// (one camera and ekf_batch_step: every field null).  ctl / vcontrol are indexed by CTA: by filter without a list, in list
// order with one.
struct BatchStepIn {
  const int* cam_of;       // [B] camera of each filter (null: camera 0)
  const double* dT;        // [n_cameras] each camera's dT
  const double* ctl;       // [B][6] dv, dw of each filter (ekf_batch_step_controls)
  const int* vcontrol;     // [B]
  const int* fsize;        // [n_cameras][4] frame sizes (ekf_batch_set_frame_sizes): the gate uses [2], [3] of the filter's camera
  const int* act;          // [n] the filters ekf_batch_step_filters steps, ascending; read by the ACT instantiations only
};
// The filter CTA i of a per-filter launch works on: i itself, or with a list (ACT, ekf_batch_step_filters) the list's entry i.
// A template parameter, so that a step without a list runs the code it ran before.
template <bool ACT>
__device__ __forceinline__ int act_filter(const int* __restrict__ act, int i) {
  if constexpr (ACT) return act[i];
  else return i;
}
__device__ __forceinline__ double step_dT(const BatchStepIn& in, int b, double dT) {
  return in.dT ? in.dT[in.cam_of ? in.cam_of[b] : 0] : dT;
}

// ------------------------------------------------------------------------------------------------
// predict for one filter per CTA: same arithmetic as k_predict_cov / k_predict_features / k_predict_S2
// ------------------------------------------------------------------------------------------------
#define BPRED_THREADS 128
template <bool INTR, bool ACT>
__global__ void __launch_bounds__(BPRED_THREADS, 4) k_batch_predict(BatchView bv, FrameView fr, DevCfg cfg, double dT, double3 dv,
                                                                 double3 dw, int vcontrol, BatchStepIn in) {
  __shared__ double F[169], C[169], T[169], Q[169], cam[13];
  const int i0 = blockIdx.x, b = act_filter<ACT>(in.act, i0), tid = threadIdx.x;
  dT = step_dT(in, b, dT);
  if (in.ctl) {
    const double* c = in.ctl + 6 * (size_t)i0;
    dv = make_double3(c[0], c[1], c[2]); dw = make_double3(c[3], c[4], c[5]);
  }
  if (in.vcontrol) vcontrol = in.vcontrol[i0];
  const int n = bv.n[b], N = bv.N[b], ld = bv.ld;
  double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  double* mu = bv.mu + (size_t)b * ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  DevCtl* ctl = bv.ctl + b;
  if (tid == 0) {
    const double ctrl[3] = {dw.x, dw.y, dw.z};
    double mu13[13];
    for (int i = 0; i < 13; ++i) mu13[i] = mu[i];
    d_system_jacobian(mu13, dT, ctrl, F);
    const double a3[3] = {dv.x, dv.y, dv.z};
    d_predict_state(mu13, a3, ctrl, dT);
    for (int i = 0; i < 13; ++i) cam[i] = mu13[i];
  }
  for (int e = tid; e < 169; e += BPRED_THREADS) C[e] = Sigma[(size_t)(e / 13) * ld + (e % 13)];
  __syncthreads();
  for (int e = tid; e < 169; e += BPRED_THREADS) {
    const int a = e / 13, c = e % 13;
    double s = 0;
    for (int k = 0; k < 6; ++k) {
      const double vmax = vcontrol ? cfg.Vmax[k] : cfg.Vmax[k] * 2.0;
      const double vs = (vmax / dT) / dT;
      s += (F[a * 13 + 7 + k] * vs) * F[c * 13 + 7 + k];
    }
    Q[e] = s;
    double t = 0;
    for (int k = 0; k < 13; ++k) t += F[a * 13 + k] * C[k * 13 + c];
    T[e] = t;
  }
  __syncthreads();
  for (int e = tid; e < 169; e += BPRED_THREADS) {
    const int a = e / 13, c = e % 13;
    double s = 0;
    for (int k = 0; k < 13; ++k) s += T[a * 13 + k] * F[c * 13 + k];
    Sigma[(size_t)a * ld + c] = s + Q[e];
  }
  for (int j = 13 + tid; j < n; j += BPRED_THREADS) {
    double x[13], y[13];
    for (int c = 0; c < 13; ++c) x[c] = Sigma[(size_t)c * ld + j];
    for (int a = 0; a < 13; ++a) {
      double s = 0;
      for (int c = 0; c < 13; ++c) s += F[a * 13 + c] * x[c];
      y[a] = s;
    }
    for (int a = 0; a < 13; ++a) Sigma[(size_t)a * ld + j] = y[a];
    double* row = Sigma + (size_t)j * ld;
    for (int c = 0; c < 13; ++c) x[c] = row[c];
    for (int a = 0; a < 13; ++a) {
      double s = 0;
      for (int c = 0; c < 13; ++c) s += x[c] * F[a * 13 + c];
      y[a] = s;
    }
    for (int a = 0; a < 13; ++a) row[a] = y[a];
  }
  __syncthreads();  // Sigma of this filter is final for the rest of the kernel
  // per-feature prediction (k_predict_features)
  for (int i = tid; i < N; i += BPRED_THREADS) {
    int ok = 0;
    const int pos = ft.pos[i], coding = ft.coding[i];
    const int fsz = coding ? 3 : 6;
    double fs[6];
    for (int c = 0; c < fsz; ++c) fs[c] = mu[pos + c];
    bool skip = false;
    if (!coding && fs[5] <= 0) { ft.removef[i] = 1; skip = true; }
    if (!skip) {
      double cm[13];
      for (int c = 0; c < 13; ++c) cm[c] = cam[c];
      double qc[4] = {cm[3], -cm[4], -cm[5], -cm[6]}, Rcw[9], hi[2], Hc[26], hcz;
      d_quat2rot(qc, Rcw);
      d_feature_hH(filter_cam<INTR>(bv, cfg, b), fs, coding, cm, qc, Rcw, hi, Hc, &hcz);
      const int half = cfg.window / 2;
      int fw = fr.w, fh = fr.h;
      if (in.fsize) {
        const int c = in.cam_of ? in.cam_of[b] : 0;
        fw = in.fsize[4 * c + 2]; fh = in.fsize[4 * c + 3];
      }
      ok = (hi[0] > half && hi[1] > half && hi[0] < fw - half && hi[1] < fh - half) && (hcz >= 0);
      if (ok) {
        ft.h[2 * i] = hi[0]; ft.h[2 * i + 1] = hi[1];
        for (int c = 0; c < 26; ++c) ft.Hc[26 * i + c] = Hc[c];
      }
    }
    ft.innov[i] = ok; ft.li[i] = 0; ft.hi[i] = 0;
    if (ok) {
      const int chunks = cfg.tstride >> 4;
      const uint4* src = reinterpret_cast<const uint4*>(ft.patch + (size_t)i * cfg.tstride);
      uint4* dst = reinterpret_cast<uint4*>(ft.mpatch + (size_t)i * cfg.tstride);
      for (int c = 0; c < chunks; ++c) dst[c] = src[c];
    }
  }
  __syncthreads();
  if (tid < 13) mu[tid] = cam[tid];
  const int m = block_compact(ft.innov, N, ft.sel, ft.pos_in_z);
  if (tid == 0) ctl->m_innov = m;
  __syncthreads();
  // 2x2 innovation blocks (k_predict_S2): one warp per feature
  const int lane = tid & 31;
  for (int f = tid >> 5; f < N; f += BPRED_THREADS / 32) {
    if (!ft.innov[f]) continue;
    const int pos = ft.pos[f], nd = 7 + (ft.coding[f] ? 3 : 6);
    const double* hc = ft.Hc + 26 * f;
    double t0 = 0, t1 = 0, h0 = 0, h1 = 0;
    if (lane < nd) {
      const int jb = ekf_idx13(lane, pos);
      double sg[13];
#pragma unroll
      for (int c = 0; c < 13; ++c) sg[c] = (c < nd) ? Sigma[(size_t)ekf_idx13(c, pos) * ld + jb] : 0.0;  // independent loads in flight
#pragma unroll
      for (int c = 0; c < 13; ++c)
        if (c < nd) { t0 += hc[c] * sg[c]; t1 += hc[13 + c] * sg[c]; }
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
}

// ------------------------------------------------------------------------------------------------
// motion-blur template prediction (Patch::blur, Patch.cpp:50-57; libblur.cpp:17-81) for one filter per CTA, after
// k_batch_predict: same arithmetic as k_predict_blur (ekf_blur.cuh), another shape.  Warp 0 takes the blur decision with
// lane = feature; then every blurred template goes to one warp, which stages it in shared memory, rasterises the line
// with lane = point, keeps each distinct coefficient once, orders them by (row, column) and has every output pixel walk
// that list: the terms and their order are the bit mask walk's, without the zeros.  out[i] = templates blurred,
// out[gridDim.x + i] = 1 when a kernel exceeded BLUR_MAXK (that template stays unblurred, as in k_predict_blur), i the CTA:
// the filter, or its position in the list.
// ------------------------------------------------------------------------------------------------
#define BBLUR_WARPS 4
// NC: feature capacity (BNCAP or BNCAP_L); warp 0 takes the decisions 32 features at a time, in ascending order.
template <int NC, bool INTR, bool ACT>
__global__ void __launch_bounds__(BBLUR_WARPS * 32) k_batch_predict_blur(BatchView bv, DevCfg cfg, double dT, int* __restrict__ out,
                                                                     BatchStepIn in) {
  __shared__ int s_feat[NC], s_rows[NC], s_cols[NC], s_nblur;
  __shared__ double s_dx[NC], s_dy[NC];
  __shared__ __align__(16) uint8_t s_tmpl[BBLUR_WARPS][1024];
  __shared__ int s_seq[BBLUR_WARPS][BLUR_MAXPTS], s_coef[BBLUR_WARPS][BLUR_MAXPTS];
  const int b = act_filter<ACT>(in.act, blockIdx.x), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  dT = step_dT(in, b, dT);
  const int N = bv.N[b], ld = bv.ld;
  const double* mu = bv.mu + (size_t)b * ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  if (warp == 0) {   // one feature per lane, NC / 32 rounds
    int nblur = 0;
    unsigned anybig = 0u;
#pragma unroll
    for (int f0 = 0; f0 < NC; f0 += 32) {
      const int f = f0 + lane;
      int d = 0, krows = 0, kcols = 0;
      double ddx = 0.0, ddy = 0.0;
      if (f < N && ft.innov[f]) {
        double cam[13], rb[3], Rb[9];
        for (int c = 0; c < 13; ++c) cam[c] = mu[c];   // predicted camera state, committed by k_batch_predict
        blur_pose(cam, cfg.T_camera, dT, rb, Rb);
        const int pos = ft.pos[f], coding = ft.coding[f];
        double fs[6];
        for (int c = 0; c < (coding ? 3 : 6); ++c) fs[c] = mu[pos + c];
        blur_displacement(filter_cam<INTR>(bv, cfg, b), fs, coding, rb, Rb, ft.h[2 * f], ft.h[2 * f + 1], &ddx, &ddy);
        d = blur_decide(ddx, ddy, cfg.kernel_min_size, &krows, &kcols);
      }
      const unsigned blur = __ballot_sync(0xffffffffu, d > 0), big = __ballot_sync(0xffffffffu, d < 0);
      if (d > 0) {
        const int k = nblur + __popc(blur & ((1u << lane) - 1u));
        s_feat[k] = f; s_rows[k] = krows; s_cols[k] = kcols; s_dx[k] = ddx; s_dy[k] = ddy;
      }
      nblur += __popc(blur);
      anybig |= big;
    }
    if (lane == 0) {
      s_nblur = nblur;
      out[blockIdx.x] = nblur;
      out[gridDim.x + blockIdx.x] = anybig != 0u;
    }
  }
  __syncthreads();
  const int w = cfg.window, w2 = w * w;
  uint8_t* tm = s_tmpl[warp];
  int* seq = s_seq[warp];
  int* coef = s_coef[warp];
  for (int k = warp; k < s_nblur; k += BBLUR_WARPS) {
    const int f = s_feat[k], krows = s_rows[k], kcols = s_cols[k];
    const uint4* src = reinterpret_cast<const uint4*>(ft.patch + (size_t)f * bv.tstride);
    for (int c = lane; c < (bv.tstride >> 4); c += 32) reinterpret_cast<uint4*>(tm)[c] = src[c];
    // the distinct coefficients in line order: lane = point i of evaluateKernel's loop (libblur.cpp:25-43)
    const BlurLine L = blur_line(s_dx[k], s_dy[k]);
    int m = 0;
    for (int base = 0; base < L.length; base += 32) {
      const int i = base + lane;
      int x = 0, y = 0;
      const bool nw = i < L.length && blur_line_point_new(L, i, krows, kcols, &x, &y);
      const unsigned bal = __ballot_sync(0xffffffffu, nw);
      if (nw) seq[m + __popc(bal & ((1u << lane) - 1u))] = blur_pack(x, y);
      m += __popc(bal);
    }
    __syncwarp();
    for (int j = lane; j < m; j += 32) coef[blur_rank(seq, m, j)] = seq[j];
    __syncwarp();
    const double kf = 1.0 / (double)m;   // kernel / sum(kernel): every set coefficient is 1 / count
    uint8_t* dst = ft.mpatch + (size_t)f * bv.tstride;
    for (int e = lane; e < w2; e += 32) dst[e] = blur_pixel_list(tm, w, e, coef, m, krows, kcols, kf);
    __syncwarp();   // tm, seq and coef are reused by the warp's next template
  }
}

// ------------------------------------------------------------------------------------------------
// update for one filter per CTA
// ------------------------------------------------------------------------------------------------
struct UpdSmem {
  double* W;      // [BNMAX][BLDW]   W = Sigma H^T, then V = W L^-T
  double* fact;   // Cholesky workspace / row staging of the W gather (kFactDoubles)
  double* Dv;     // [BK / 32][32][BLDD] inverses of the diagonal blocks of L
  double* Sb;     // [BK][BLDW]      S, then L
  double* nu;     // [BK]
  double* y;      // [BK]
  double* mu_i;   // [BNMAX]
  double* Hs;     // [BNCAP][27]
  double* qj;     // [48] quaternion-normalisation scratch: J[16], C[16], T[16]
  int* ibuf;      // cand[BNCAP], fids[BNCAP], poss[BNCAP], nds[BNCAP]
};
#define BLDD 36
static constexpr size_t kFactDoubles = 2 * 16 * BNMAX > cta_chol_panel_smem_doubles<BK>() ? 2 * 16 * BNMAX : cta_chol_panel_smem_doubles<BK>();
static constexpr size_t kUpdSmemDoubles =
    (size_t)BNMAX * BLDW + kFactDoubles + (BK / 32) * 32 * BLDD + (size_t)BK * BLDW + BK + BK + BNMAX + BNCAP * 27 + 48 + (4 * BNCAP) / 2;
static constexpr size_t kUpdSmemBytes = kUpdSmemDoubles * sizeof(double);

// One stacked update block is a gather (W, S, nu in shared memory), then cta_block_gain_downdate, and the update ends with one
// cta_normalize_quaternion.  cta_stacked_update is the usual single block; with forsePlane the second update is the Hi block, the
// plane block (cta_gather_plane), then the normalisation, as the single filter's stacked_update / launch_finish_update.
//
// Gather of the Hi / Li block over the `cnt` features listed in ft.sel (V:1036-1064 / V:1245-1284): W = Sigma H^T, S = H W + R
// padded with identity to BK, nu = z - h.
__device__ void cta_gather_features(const UpdSmem& sm, const double* __restrict__ Sigma, int ld, int n, const FeatTab& ft, int cnt,
                                    const DevCfg& cfg) {
  const int tid = threadIdx.x;
  const int k = 2 * cnt;
  int* fids = sm.ibuf + BNCAP; int* poss = fids + BNCAP; int* nds = poss + BNCAP;
  for (int a = tid; a < BNCAP; a += BUPD_THREADS) {
    if (a < cnt) {
      const int f = ft.sel[a];
      fids[a] = f; poss[a] = ft.pos[f]; nds[a] = 7 + (ft.coding[f] ? 3 : 6);
    } else { fids[a] = -1; poss[a] = 0; nds[a] = 0; }
  }
  __syncthreads();
  for (int e = tid; e < BNCAP * 26; e += BUPD_THREADS) {
    const int a = e / 26, c = e % 26;
    sm.Hs[a * 27 + c] = (a < cnt) ? ft.Hc[26 * fids[a] + c] : 0.0;
  }
  if (tid < BK) {
    double v = 0.0;
    if (tid < k) { const int f = fids[tid >> 1]; v = ft.z[2 * f + (tid & 1)] - ft.h[2 * f + (tid & 1)]; }
    sm.nu[tid] = v;
  }
  __syncthreads();
  // W = Sigma H^T (n x k), zero-padded to BNMAX x BK.  Sigma rows are staged through shared memory
  // (the Cholesky workspace is idle here) in chunks of 16 rows with cp.async, double buffered, so the
  // 13-column gathers hit shared memory instead of 13 dependent L2 round trips; thread = (row, feature).
  {
    constexpr int CH = 16;
    double* stage = sm.fact;                      // 2 x CH x ld doubles (ld <= 208)
    const int nchunk = (n + CH - 1) / CH;
    const int vec_per_row = ld >> 1;              // 16-byte pieces per row (ld is a multiple of 8)
    auto issue = [&](int ck) {
      const int r0 = ck * CH;
      double* dst = stage + (size_t)(ck & 1) * CH * ld;
      for (int e = tid; e < CH * vec_per_row; e += BUPD_THREADS) {
        const int r = e / vec_per_row, v = e - r * vec_per_row;
        if (r0 + r < n) {
          const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + (size_t)r * ld + 2 * v);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(Sigma + (size_t)(r0 + r) * ld + 2 * v));
        }
      }
      asm volatile("cp.async.commit_group;\n" ::);
    };
    issue(0);
    const int rl = tid >> 5, a = tid & 31;       // 16 rows x 32 features per chunk
    const int pos = poss[a], nd = nds[a];
    const double* hs = sm.Hs + a * 27;
    for (int ck = 0; ck < nchunk; ++ck) {
      if (ck + 1 < nchunk) { issue(ck + 1); asm volatile("cp.async.wait_group 1;\n" ::); }
      else asm volatile("cp.async.wait_group 0;\n" ::);
      __syncthreads();
      const int i = ck * CH + rl;
      double w0 = 0, w1 = 0;
      if (i < n && a < cnt) {
        const double* row = stage + (size_t)(ck & 1) * CH * ld + (size_t)rl * ld;
        for (int c = 0; c < nd; ++c) {
          const double s = row[ekf_idx13(c, pos)];
          w0 += s * hs[c]; w1 += s * hs[13 + c];
        }
      }
      if (i < BNMAX) *reinterpret_cast<double2*>(sm.W + (size_t)i * BLDW + 2 * a) = make_double2(w0, w1);
      __syncthreads();
    }
    for (int e = tid; e < (BNMAX - nchunk * CH) * (BK / 2); e += BUPD_THREADS) {   // zero rows past the last chunk
      const int i = nchunk * CH + e / (BK / 2), aa = e % (BK / 2);
      *reinterpret_cast<double2*>(sm.W + (size_t)i * BLDW + 2 * aa) = make_double2(0.0, 0.0);
    }
  }
  __syncthreads();
  // S = H W + sigma_px^2 I; rows / columns past k are identity
  for (int e = tid; e < BK * BK; e += BUPD_THREADS) {
    const int r = e / BK, s = e % BK;
    double v = (r == s) ? 1.0 : 0.0;
    if (r < k && s < k) {
      const int a = r >> 1;
      const int pos = poss[a], nd = nds[a];
      const double* hc = sm.Hs + a * 27 + 13 * (r & 1);
      double acc = 0;
      for (int c = 0; c < nd; ++c) acc += hc[c] * sm.W[(size_t)ekf_idx13(c, pos) * BLDW + s];
      v = acc + ((r == s) ? cfg.sigma_pixel_2 : 0.0);
    }
    sm.Sb[r * BLDW + s] = v;
  }
  __syncthreads();
}

// forsePlane (V:1245-1263): the pseudo-measurements mu[1] = mu[4] = mu[6] = 0 with R = 1e-5 I3 as one more block of k = 3 rows, the
// unit rows e1, e4, e6 (k_plane_gather / k_plane_S): W[:, j] = Sigma[:, k_j], nu_j = 0 - mu[k_j] with mu already corrected by the
// Hi block (the single filter's (0 - mu[k_j]) - delta[k_j] over the same sequential blocks), S = W[{1, 4, 6}, :] + 1e-5 I.
__device__ void cta_gather_plane(const UpdSmem& sm, const double* __restrict__ Sigma, int ld, int n, const double* __restrict__ mu,
                                 DevCtl* ctl) {
  const int tid = threadIdx.x;
  for (int e = tid; e < BNMAX * (BK / 2); e += BUPD_THREADS) {
    const int i = e / (BK / 2), c = 2 * (e % (BK / 2));
    double2 v = make_double2(0.0, 0.0);
    if (i < n && c == 0) v = make_double2(Sigma[(size_t)i * ld + 1], Sigma[(size_t)i * ld + 4]);
    if (i < n && c == 2) v.x = Sigma[(size_t)i * ld + 6];
    *reinterpret_cast<double2*>(sm.W + (size_t)i * BLDW + c) = v;
  }
  if (tid < BK) sm.nu[tid] = (tid < 3) ? 0.0 - mu[tid == 0 ? 1 : (tid == 1 ? 4 : 6)] : 0.0;
  if (tid == 0) ctl->k_rows += 3;
  __syncthreads();
  for (int e = tid; e < BK * BK; e += BUPD_THREADS) {
    const int r = e / BK, s = e % BK;
    double v = (r == s) ? 1.0 : 0.0;
    if (r < 3 && s < 3) v = sm.W[(size_t)(r == 0 ? 1 : (r == 1 ? 4 : 6)) * BLDW + s] + ((r == s) ? 0.00001 : 0.0);
    sm.Sb[r * BLDW + s] = v;
  }
  __syncthreads();
}

// Gain and downdate of the gathered block of k rows: L = chol(S), V = W L^-T, mu += V L^-1 nu, Sigma -= V V^T.
__device__ void cta_block_gain_downdate(const UpdSmem& sm, double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu, int k,
                                        DevCtl* ctl) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t4 = lane & 3;
  cta_chol_panel<BK>(sm.fact, sm.Sb, BLDW, sm.nu, sm.Sb, BLDW, sm.Dv, BLDD, sm.y, &ctl->chol_fail);
  // V = W L^-T in place: every warp owns 8-row tiles for the whole blocked triangular solve
  for (int rt = warp; rt < BNMAX / 8; rt += BUPD_THREADS / 32) {
    double part = warp_trsm_tile<BK>(sm.W + (size_t)rt * 8 * BLDW, BLDW, sm.Sb, BLDW, sm.Dv, BLDD, sm.y);
    // mu += V y: the four lanes of a row hold its partial sums
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    const int i = rt * 8 + g;
    if (t4 == 0 && i < n) mu[i] += part;
  }
  __syncthreads();
  // Sigma -= V V^T on the fp64 tensor pipe: 16 x 16 warp tiles (2 x 2 DMMA tiles), K = ceil(k / 4) * 4.
  // The C tile of a warp's next tile is loaded before the DMMAs of the current one (L2 latency hidden).
  {
    const int nt = (n + 15) >> 4, ksteps = (k + 3) >> 2, ntile = nt * nt;
    auto load_c = [&](int t, double (&c)[2][2][2]) {
      const int ti = t / nt, tj = t - ti * nt;
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int r = ti * 16 + a * 8 + g, col = tj * 16 + cc * 8 + 2 * t4;
          double2 v = make_double2(0.0, 0.0);
          if (t < ntile) {
            if (r < n && col + 1 < n) v = *reinterpret_cast<const double2*>(Sigma + (size_t)r * ld + col);
            else if (r < n && col < n) v.x = Sigma[(size_t)r * ld + col];
          }
          c[a][cc][0] = v.x; c[a][cc][1] = v.y;
        }
    };
    double nxt[2][2][2];
    load_c(warp, nxt);
    for (int t = warp; t < ntile; t += BUPD_THREADS / 32) {
      const int ti = t / nt, tj = t - ti * nt;
      double acc[2][2][2];
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) { acc[a][cc][0] = nxt[a][cc][0]; acc[a][cc][1] = nxt[a][cc][1]; }
      load_c(t + BUPD_THREADS / 32, nxt);
      const double* va = sm.W + (size_t)(ti * 16 + g) * BLDW + t4;
      const double* vb = sm.W + (size_t)(tj * 16 + g) * BLDW + t4;
      for (int q = 0; q < ksteps; ++q) {
        const double a0 = va[4 * q], a1 = va[8 * BLDW + 4 * q];
        const double b0 = -vb[4 * q], b1 = -vb[8 * BLDW + 4 * q];
        dmma884f(acc[0][0][0], acc[0][0][1], a0, b0);
        dmma884f(acc[0][1][0], acc[0][1][1], a0, b1);
        dmma884f(acc[1][0][0], acc[1][0][1], a1, b0);
        dmma884f(acc[1][1][0], acc[1][1][1], a1, b1);
      }
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int r = ti * 16 + a * 8 + g, col = tj * 16 + cc * 8 + 2 * t4;
          if (r < n && col + 1 < n) *reinterpret_cast<double2*>(Sigma + (size_t)r * ld + col) = make_double2(acc[a][cc][0], acc[a][cc][1]);
          else if (r < n && col < n) Sigma[(size_t)r * ld + col] = acc[a][cc][0];
        }
    }
  }
  __syncthreads();
}

// normalizeQuaternion (V:1625-1642): 4 rows + 4 columns
__device__ void cta_normalize_quaternion(const UpdSmem& sm, double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu) {
  const int tid = threadIdx.x;
  double* J = sm.qj; double* Cq = J + 16; double* Tq = Cq + 16;
  if (tid == 0) {
    double q[4];
    for (int i = 0; i < 4; ++i) q[i] = mu[3 + i];
    const double norma = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    const double sc = 1 / (norma * norma * norma);
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) J[i * 4 + j] = ((norma * norma) * (i == j ? 1.0 : 0.0) - q[i] * q[j]) * sc;
    for (int i = 0; i < 4; ++i) mu[3 + i] = q[i] / norma;
  }
  if (tid >= 32 && tid < 48) Cq[tid - 32] = Sigma[(size_t)(3 + (tid - 32) / 4) * ld + 3 + ((tid - 32) % 4)];
  __syncthreads();
  if (tid < 16) {
    const int a = tid / 4, c = tid % 4;
    double t = 0;
    for (int kk = 0; kk < 4; ++kk) t += J[a * 4 + kk] * Cq[kk * 4 + c];
    Tq[tid] = t;
  }
  __syncthreads();
  if (tid < 16) {
    const int a = tid / 4, c = tid % 4;
    double s = 0;
    for (int kk = 0; kk < 4; ++kk) s += Tq[a * 4 + kk] * J[c * 4 + kk];
    Sigma[(size_t)(3 + a) * ld + 3 + c] = s;
  }
  for (int jj = tid; jj < n - 4; jj += BUPD_THREADS) {
    const int j = jj >= 3 ? jj + 4 : jj;
    double x[4], yv[4];
    for (int c = 0; c < 4; ++c) x[c] = Sigma[(size_t)(3 + c) * ld + j];
    for (int a = 0; a < 4; ++a) {
      double s = 0;
      for (int c = 0; c < 4; ++c) s += J[a * 4 + c] * x[c];
      yv[a] = s;
    }
    for (int a = 0; a < 4; ++a) Sigma[(size_t)(3 + a) * ld + j] = yv[a];
    double* row = Sigma + (size_t)j * ld + 3;
    for (int c = 0; c < 4; ++c) x[c] = row[c];
    for (int a = 0; a < 4; ++a) {
      double s = 0;
      for (int c = 0; c < 4; ++c) s += x[c] * J[a * 4 + c];
      yv[a] = s;
    }
    for (int a = 0; a < 4; ++a) row[a] = yv[a];
  }
  __syncthreads();
}

// One stacked update over the `cnt` features listed in ft.sel (V:1036-1064 / V:1245-1284).
__device__ void cta_stacked_update(const UpdSmem& sm, double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu,
                                   const FeatTab& ft, int cnt, const DevCfg& cfg, DevCtl* ctl) {
  cta_gather_features(sm, Sigma, ld, n, ft, cnt, cfg);
  cta_block_gain_downdate(sm, Sigma, ld, n, mu, 2 * cnt, ctl);
  cta_normalize_quaternion(sm, Sigma, ld, n, mu);
}

// PLANE: forsePlane (ekf_batch_set_force_plane), a separate instantiation so that the plane-off kernel is the same code as without it.
// ACT: CTA i updates filter act[i] (ekf_batch_step_filters).
template <bool PLANE, bool INTR, bool ACT>
__global__ void __launch_bounds__(BUPD_THREADS, 1) k_batch_update(BatchView bv, DevCfg cfg, const uint32_t* __restrict__ picks,
                                                                  int n_picks, double* __restrict__ out_mu14,
                                                                  double* __restrict__ out_S14, int* __restrict__ out_stats,
                                                                  int min_features, int max_features, int xyz_conversion,
                                                                  const int* __restrict__ act) {
  extern __shared__ __align__(16) double usm[];
  UpdSmem sm;
  sm.W = usm;
  sm.fact = sm.W + (size_t)BNMAX * BLDW;
  sm.Dv = sm.fact + kFactDoubles;
  sm.Sb = sm.Dv + (BK / 32) * 32 * BLDD;
  sm.nu = sm.Sb + (size_t)BK * BLDW;
  sm.y = sm.nu + BK;
  sm.mu_i = sm.y + BK;
  sm.Hs = sm.mu_i + BNMAX;
  sm.qj = sm.Hs + BNCAP * 27;
  sm.ibuf = reinterpret_cast<int*>(sm.qj + 48);
  const int b = act_filter<ACT>(act, blockIdx.x), tid = threadIdx.x;
  const int n = bv.n[b], N = bv.N[b], ld = bv.ld;
  double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  double* mu = bv.mu + (size_t)b * ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  DevCtl* ctl = bv.ctl + b;
  if (tid == 0) ctl->chol_fail = 0;
  // 1-point RANSAC, low-innovation update
  if constexpr (INTR) {   // a configuration with the filter's intrinsics for cta_ransac; the Hi rescue below reads the row itself
    DevCfg rcfg = cfg;
    rcfg.cam = bv.cam[b];
    cta_ransac(Sigma, ld, n, mu, ft, N, ctl, rcfg, picks, n_picks, sm.mu_i, sm.ibuf);
  } else {
    cta_ransac(Sigma, ld, n, mu, ft, N, ctl, cfg, picks, n_picks, sm.mu_i, sm.ibuf);
  }
  __syncthreads();
  const int n_li = ctl->n_li;
  if (n_li > 0) cta_stacked_update(sm, Sigma, ld, n, mu, ft, n_li, cfg, ctl);
  // high-innovation rescue (k_hi_rescue): pose from the old mu, feature parameters from mu_tmp
  for (int i = tid; i < N; i += BUPD_THREADS) {
    int flag = 0;
    if (!ft.li[i] && ft.innov[i]) {
      const int pos = ft.pos[i], coding = ft.coding[i];
      const int fsz = coding ? 3 : 6, nd = 7 + fsz;
      double fs[6], r[3], qc[4], Rcw[9], hi[2], Hc[26], hcz;
      for (int c = 0; c < fsz; ++c) fs[c] = mu[pos + c];
      for (int c = 0; c < 3; ++c) r[c] = ctl->cam_old[c];
      qc[0] = ctl->cam_old[3]; qc[1] = -ctl->cam_old[4]; qc[2] = -ctl->cam_old[5]; qc[3] = -ctl->cam_old[6];
      d_quat2rot(qc, Rcw);
      d_feature_hH(filter_cam<INTR>(bv, cfg, b), fs, coding, r, qc, Rcw, hi, Hc, &hcz);
      ft.h[2 * i] = hi[0]; ft.h[2 * i + 1] = hi[1];
      for (int c = 0; c < 26; ++c) ft.Hc[26 * i + c] = Hc[c];
      double Tm[26];
      for (int bb = 0; bb < nd; ++bb) {
        const int jb = ekf_idx13(bb, pos);
        double sg[13];
#pragma unroll
        for (int c = 0; c < 13; ++c) sg[c] = (c < nd) ? Sigma[(size_t)ekf_idx13(c, pos) * ld + jb] : 0.0;
        double t0 = 0, t1 = 0;
#pragma unroll
        for (int c = 0; c < 13; ++c)
          if (c < nd) { t0 += Hc[c] * sg[c]; t1 += Hc[13 + c] * sg[c]; }
        Tm[bb] = t0; Tm[13 + bb] = t1;
      }
      double S[4] = {0, 0, 0, 0};
      for (int bb = 0; bb < nd; ++bb) {
        S[0] += Tm[bb] * Hc[bb]; S[1] += Tm[bb] * Hc[13 + bb];
        S[2] += Tm[13 + bb] * Hc[bb]; S[3] += Tm[13 + bb] * Hc[13 + bb];
      }
      const double det = S[0] * S[3] - S[2] * S[1];
      const double invdet = 1.0 / det;
      const double i00 = S[3] * invdet, i10 = -S[2] * invdet, i01 = -S[1] * invdet, i11 = S[0] * invdet;
      const double e0 = hi[0] - ft.z[2 * i], e1 = hi[1] - ft.z[2 * i + 1];
      const double t0 = e0 * i00 + e1 * i10;
      const double t1 = e0 * i01 + e1 * i11;
      const double chi = t0 * e0 + t1 * e1;
      flag = (chi <= cfg.th_hi) ? 1 : 0;
    }
    ft.hi[i] = flag;
  }
  __syncthreads();
  const int n_hi = block_compact(ft.hi, N, ft.sel, ft.pos_in_z);
  if (tid == 0) { ctl->n_hi = n_hi; ctl->k_rows = 2 * n_hi; }
  __syncthreads();
  if constexpr (PLANE) {   // the second update runs with or without Hi rows (z_hi.rows() > 0 with the plane rows, V:1245-1272)
    if (n_hi > 0) {
      cta_gather_features(sm, Sigma, ld, n, ft, n_hi, cfg);
      cta_block_gain_downdate(sm, Sigma, ld, n, mu, 2 * n_hi, ctl);
    }
    cta_gather_plane(sm, Sigma, ld, n, mu, ctl);
    cta_block_gain_downdate(sm, Sigma, ld, n, mu, 3, ctl);
    cta_normalize_quaternion(sm, Sigma, ld, n, mu);
  } else {
    if (n_hi > 0) cta_stacked_update(sm, Sigma, ld, n, mu, ft, n_hi, cfg, ctl);
  }
  // book-keeping (k_bookkeeping) + visibility count (V:1296-1315)
  int my_remove = 0, my_vis = 0;
  for (int i = tid; i < N; i += BUPD_THREADS) {
    int nfind = ft.n_find[i];
    const int ntot = ft.n_tot[i];
    if (ft.hi[i] || ft.li[i]) nfind++;
    ft.n_find[i] = nfind;
    const float qi = (float)(ntot - nfind) / ((float)nfind);
    ft.quality[i] = qi;
    if (qi > cfg.quality_ratio) ft.removef[i] = 1;
    if (ft.removef[i]) my_remove++;
    else if (ft.innov[i]) my_vis++;
  }
  const int n_rem = __syncthreads_count(my_remove);   // N <= 32 <= blockDim: one feature per thread
  const int n_vis = __syncthreads_count(my_vis);
  for (int e = tid; e < 14; e += BUPD_THREADS) out_mu14[(size_t)b * 14 + e] = mu[e];
  if (out_S14)
    for (int e = tid; e < 196; e += BUPD_THREADS) out_S14[(size_t)b * 196 + e] = Sigma[(size_t)(e / 14) * ld + (e % 14)];
  if (tid == 0) {
    int* st = out_stats + (size_t)b * EKF_BATCH_STAT_FIELDS;
    int removed = n_rem, topup = 0;
    if (n_vis < min_features) {
      if (N - n_rem > max_features) removed += 1;   // removeFeature(0) (V:1313), applied by k_batch_compact
      topup = min_features - n_vis;
    }
    ctl->n_remove = removed;
    ctl->n_visible = n_vis;
    st[EKF_BSTAT_INNOV] = ctl->m_innov; st[EKF_BSTAT_MATCHED] = ctl->n_matched; st[EKF_BSTAT_LI] = n_li;
    st[EKF_BSTAT_HI] = n_hi; st[EKF_BSTAT_HYPS] = ctl->ransac_hyps; st[EKF_BSTAT_CHOL_FAIL] = ctl->chol_fail;
    st[EKF_BSTAT_REMOVED] = removed; st[EKF_BSTAT_TOPUP] = topup;
  }
  // convert2XYZ_ifLinearAll (V:1317) of the features that survive this step: not flagged, and not the removeFeature(0)
  // victim, the first unflagged feature (V:1312-1313).  The reference removes, then converts; deciding here, on the
  // pre-removal state, gives the same decisions: removal moves entries without changing a value, and the linearity index
  // reads only the feature's own mu entries, the camera position mu[0:3] and the feature's own rho variance.
  // k_batch_compact then applies removals and conversions together.
  if (xyz_conversion && tid < 32) {
    const bool alive = tid < N && !ft.removef[tid];
    const unsigned alive_mask = __ballot_sync(0xffffffffu, alive);
    const bool drop_first = (n_vis < min_features) && (N - n_rem > max_features);
    const int victim = drop_first ? __ffs(alive_mask) - 1 : -1;
    warp_xyz_decide(bv, b, Sigma, mu, ft, N, alive && tid != victim, cfg);
  }
}

// ------------------------------------------------------------------------------------------------
// update for one filter per CLUSTER of C = ceil(ld / BSTRIP) CTAs (2 to 4; ekf_batch_create_large, capacity 33 to 128).
// Every CTA has k_batch_update's 512 threads and UpdSmem layout; CTA r owns rows [BSTRIP r, BSTRIP r + BSTRIP) of W / V, of
// Sigma and of the correction delta (sm.mu_i), and reads the other CTAs' W / V panels and delta strips through distributed
// shared memory.  BSTRIP = 208 = 13 x 16, so the downdate's 16 x 16 tiles never straddle two CTAs.
//   * rank 0 runs 1-point RANSAC (mu_i in its idle Cholesky workspace), the Hi rescue and the book-keeping; the others wait at
//     the cluster barrier.
//   * an update over cnt features runs as ceil(cnt / 32) blocks of at most BK rows, block b with the innovation
//     (z_b - h_b) - H_b delta, delta the correction of the earlier blocks (the single filter's blocked schedules,
//     ekf_update.cu); mu += delta and one quaternion normalisation follow the last block.
//   * per block: each CTA gathers its rows of W = Sigma H^T; barrier; every CTA forms the same S = H W + R and nu from the
//     owners' W rows and delta entries; barrier; every CTA factors S (same inputs, same code: the same L bits everywhere), solves
//     V = W L^-T and accumulates delta += V y on its rows; barrier; each CTA downdates its row strip over all columns, the
//     b-fragments of a column tile from its owner's V; barrier.
// ------------------------------------------------------------------------------------------------
#define BSTRIP BNMAX
#define BCL_MAX 4

static __device__ __forceinline__ void cl_sync() { cg::this_cluster().sync(); }
// row `row` of the panel `p` (W or the delta strip, row stride ldp) of the CTA owning it
static __device__ __forceinline__ double* cl_row(double* p, int row, int ldp) {
  return cg::this_cluster().map_shared_rank(p + (size_t)(row % BSTRIP) * ldp, row / BSTRIP);
}

// One block of the features ft.sel[a0 .. a0 + m) (m <= BK / 2): W own rows, S, nu; ends with the S / nu cluster barrier.
__device__ void cl_gather_features(const UpdSmem& sm, int rank, double* Sigma, int ld, int n, const FeatTab& ft, int a0, int m,
                                   const DevCfg& cfg) {
  const int tid = threadIdx.x, k = 2 * m, row0 = rank * BSTRIP;
  int* fids = sm.ibuf + BNCAP; int* poss = fids + BNCAP; int* nds = poss + BNCAP;
  for (int a = tid; a < BNCAP; a += BUPD_THREADS) {
    if (a < m) {
      const int f = ft.sel[a0 + a];
      fids[a] = f; poss[a] = ft.pos[f]; nds[a] = 7 + (ft.coding[f] ? 3 : 6);
    } else { fids[a] = -1; poss[a] = 0; nds[a] = 0; }
  }
  __syncthreads();
  for (int e = tid; e < BNCAP * 26; e += BUPD_THREADS) {
    const int a = e / 26, c = e % 26;
    sm.Hs[a * 27 + c] = (a < m) ? ft.Hc[26 * fids[a] + c] : 0.0;
  }
  __syncthreads();
  // W = Sigma H^T on the CTA's rows: thread = (row, feature), 16 rows x 32 features a pass, the 13 loads of a row in flight
  {
    const int rl = tid >> 5, a = tid & 31;
    const int pos = poss[a], nd = nds[a];
    const double* hs = sm.Hs + a * 27;
    for (int r0 = 0; r0 < BSTRIP; r0 += 16) {
      const int il = r0 + rl, i = row0 + il;
      double w0 = 0, w1 = 0;
      if (i < n && a < m) {
        const double* row = Sigma + (size_t)i * ld;
        double sg[13];
#pragma unroll
        for (int c = 0; c < 13; ++c) sg[c] = (c < nd) ? row[ekf_idx13(c, pos)] : 0.0;
#pragma unroll
        for (int c = 0; c < 13; ++c)
          if (c < nd) { w0 += sg[c] * hs[c]; w1 += sg[c] * hs[13 + c]; }
      }
      *reinterpret_cast<double2*>(sm.W + (size_t)il * BLDW + 2 * a) = make_double2(w0, w1);
    }
  }
  __syncthreads();
  cl_sync();   // every CTA's W rows and delta strip are final
  if (tid < BK) {   // nu = (z - h) - H delta
    double v = 0.0;
    if (tid < k) {
      const int a = tid >> 1, f = fids[a];
      v = ft.z[2 * f + (tid & 1)] - ft.h[2 * f + (tid & 1)];
      if (a0 > 0) {
        const int pos = poss[a], nd = nds[a];
        const double* hc = sm.Hs + a * 27 + 13 * (tid & 1);
        double acc = 0;
        for (int c = 0; c < nd; ++c) acc += hc[c] * *cl_row(sm.mu_i, ekf_idx13(c, pos), 1);
        v = v - acc;
      }
    }
    sm.nu[tid] = v;
  }
  // S = H W + sigma_px^2 I from the owners' W rows; rows / columns past k are identity
  for (int e = tid; e < BK * BK; e += BUPD_THREADS) {
    const int r = e / BK, s = e % BK;
    double v = (r == s) ? 1.0 : 0.0;
    if (r < k && s < k) {
      const int a = r >> 1;
      const int pos = poss[a], nd = nds[a];
      const double* hc = sm.Hs + a * 27 + 13 * (r & 1);
      double acc = 0;
      for (int c = 0; c < nd; ++c) acc += hc[c] * cl_row(sm.W, ekf_idx13(c, pos), BLDW)[s];
      v = acc + ((r == s) ? cfg.sigma_pixel_2 : 0.0);
    }
    sm.Sb[r * BLDW + s] = v;
  }
  __syncthreads();
  cl_sync();   // no CTA reads another's W or delta any more: V may overwrite W
}

// The plane block (cta_gather_plane) in a cluster: W[:, j] = Sigma[:, k_j] on the CTA's rows, nu_j = (0 - mu[k_j]) - delta[k_j],
// S = W[{1, 4, 6}, :] + 1e-5 I from rank 0's rows.
__device__ void cl_gather_plane(const UpdSmem& sm, int rank, double* Sigma, int ld, int n, const double* mu, DevCtl* ctl) {
  const int tid = threadIdx.x, row0 = rank * BSTRIP;
  for (int e = tid; e < BSTRIP * (BK / 2); e += BUPD_THREADS) {
    const int il = e / (BK / 2), c = 2 * (e % (BK / 2)), i = row0 + il;
    double2 v = make_double2(0.0, 0.0);
    if (i < n && c == 0) v = make_double2(Sigma[(size_t)i * ld + 1], Sigma[(size_t)i * ld + 4]);
    if (i < n && c == 2) v.x = Sigma[(size_t)i * ld + 6];
    *reinterpret_cast<double2*>(sm.W + (size_t)il * BLDW + c) = v;
  }
  if (rank == 0 && tid == 0) ctl->k_rows += 3;
  __syncthreads();
  cl_sync();
  if (tid < BK) {
    double v = 0.0;
    if (tid < 3) {
      const int kj = tid == 0 ? 1 : (tid == 1 ? 4 : 6);
      v = (0.0 - mu[kj]) - *cl_row(sm.mu_i, kj, 1);
    }
    sm.nu[tid] = v;
  }
  for (int e = tid; e < BK * BK; e += BUPD_THREADS) {
    const int r = e / BK, s = e % BK;
    double v = (r == s) ? 1.0 : 0.0;
    if (r < 3 && s < 3) v = cl_row(sm.W, r == 0 ? 1 : (r == 1 ? 4 : 6), BLDW)[s] + ((r == s) ? 0.00001 : 0.0);
    sm.Sb[r * BLDW + s] = v;
  }
  __syncthreads();
  cl_sync();
}

// Gain and downdate of the gathered block of k rows: L = chol(S) in every CTA, V = W L^-T and delta += V y on the CTA's rows,
// Sigma -= V V^T on its row strip over all columns (b-fragments from the column tile's owner).  Ends with a cluster barrier.
__device__ void cl_block_gain_downdate(const UpdSmem& sm, int rank, double* __restrict__ Sigma, int ld, int n, int k, DevCtl* ctl) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t4 = lane & 3;
  const int row0 = rank * BSTRIP;
  cta_chol_panel<BK>(sm.fact, sm.Sb, BLDW, sm.nu, sm.Sb, BLDW, sm.Dv, BLDD, sm.y, &ctl->chol_fail);
  for (int rt = warp; rt < BSTRIP / 8; rt += BUPD_THREADS / 32) {
    double part = warp_trsm_tile<BK>(sm.W + (size_t)rt * 8 * BLDW, BLDW, sm.Sb, BLDW, sm.Dv, BLDD, sm.y);
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    const int il = rt * 8 + g;
    if (t4 == 0 && row0 + il < n) sm.mu_i[il] += part;
  }
  __syncthreads();
  cl_sync();   // every CTA's V is final
  {
    const int rows = min(max(n - row0, 0), BSTRIP);
    const int nt = (n + 15) >> 4, rtl = (rows + 15) >> 4, ksteps = (k + 3) >> 2, ntile = rtl * nt;
    auto load_c = [&](int t, double (&c)[2][2][2]) {
      const int ti = t / nt, tj = t - ti * nt;
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int r = row0 + ti * 16 + a * 8 + g, col = tj * 16 + cc * 8 + 2 * t4;
          double2 v = make_double2(0.0, 0.0);
          if (t < ntile) {
            if (r < n && col + 1 < n) v = *reinterpret_cast<const double2*>(Sigma + (size_t)r * ld + col);
            else if (r < n && col < n) v.x = Sigma[(size_t)r * ld + col];
          }
          c[a][cc][0] = v.x; c[a][cc][1] = v.y;
        }
    };
    double nxt[2][2][2];
    load_c(warp, nxt);
    for (int t = warp; t < ntile; t += BUPD_THREADS / 32) {
      const int ti = t / nt, tj = t - ti * nt;
      double acc[2][2][2];
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) { acc[a][cc][0] = nxt[a][cc][0]; acc[a][cc][1] = nxt[a][cc][1]; }
      load_c(t + BUPD_THREADS / 32, nxt);
      const double* va = sm.W + (size_t)(ti * 16 + g) * BLDW + t4;
      const double* vb = cl_row(sm.W, tj * 16 + g, BLDW) + t4;   // the owner's V (tiles never straddle two CTAs)
      for (int q = 0; q < ksteps; ++q) {
        const double a0 = va[4 * q], a1 = va[8 * BLDW + 4 * q];
        const double b0 = -vb[4 * q], b1 = -vb[8 * BLDW + 4 * q];
        dmma884f(acc[0][0][0], acc[0][0][1], a0, b0);
        dmma884f(acc[0][1][0], acc[0][1][1], a0, b1);
        dmma884f(acc[1][0][0], acc[1][0][1], a1, b0);
        dmma884f(acc[1][1][0], acc[1][1][1], a1, b1);
      }
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int r = row0 + ti * 16 + a * 8 + g, col = tj * 16 + cc * 8 + 2 * t4;
          if (r < n && col + 1 < n) *reinterpret_cast<double2*>(Sigma + (size_t)r * ld + col) = make_double2(acc[a][cc][0], acc[a][cc][1]);
          else if (r < n && col < n) Sigma[(size_t)r * ld + col] = acc[a][cc][0];
        }
    }
  }
  __syncthreads();
  cl_sync();   // no CTA reads another's V any more: the next block may overwrite W
}

// End of an update: mu += delta on every CTA's rows, then normalizeQuaternion (V:1625-1642): every CTA takes J from mu[3..6]
// and applies it to columns 3..6 of its rows; rank 0, the owner of rows 3..6, also to those rows and the 4 x 4 corner.  Ends
// with a cluster barrier: Sigma and mu are final for every CTA.
__device__ void cl_finish_update(const UpdSmem& sm, int rank, double* __restrict__ Sigma, int ld, int n, double* __restrict__ mu) {
  const int tid = threadIdx.x, row0 = rank * BSTRIP, rows = min(max(n - row0, 0), BSTRIP);
  for (int il = tid; il < rows; il += BUPD_THREADS) { mu[row0 + il] += sm.mu_i[il]; sm.mu_i[il] = 0.0; }
  __syncthreads();
  cl_sync();   // mu[3..6] final
  double* J = sm.qj; double* Cq = J + 16; double* Tq = Cq + 16;
  double q[4] = {0.0, 0.0, 0.0, 0.0}, norma = 0.0;
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) q[i] = mu[3 + i];
    norma = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    const double sc = 1 / (norma * norma * norma);
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) J[i * 4 + j] = ((norma * norma) * (i == j ? 1.0 : 0.0) - q[i] * q[j]) * sc;
  }
  if (rank == 0 && tid >= 32 && tid < 48) Cq[tid - 32] = Sigma[(size_t)(3 + (tid - 32) / 4) * ld + 3 + ((tid - 32) % 4)];
  __syncthreads();
  cl_sync();   // every CTA has read mu[3..6]
  if (rank == 0) {
    if (tid == 0)
      for (int i = 0; i < 4; ++i) mu[3 + i] = q[i] / norma;
    if (tid < 16) {
      const int a = tid / 4, c = tid % 4;
      double t = 0;
      for (int kk = 0; kk < 4; ++kk) t += J[a * 4 + kk] * Cq[kk * 4 + c];
      Tq[tid] = t;
    }
    __syncthreads();
    if (tid < 16) {
      const int a = tid / 4, c = tid % 4;
      double s = 0;
      for (int kk = 0; kk < 4; ++kk) s += Tq[a * 4 + kk] * J[c * 4 + kk];
      Sigma[(size_t)(3 + a) * ld + 3 + c] = s;
    }
    for (int jj = tid; jj < n - 4; jj += BUPD_THREADS) {   // rows 3..6, every column but 3..6
      const int j = jj >= 3 ? jj + 4 : jj;
      double x[4], yv[4];
      for (int c = 0; c < 4; ++c) x[c] = Sigma[(size_t)(3 + c) * ld + j];
      for (int a = 0; a < 4; ++a) {
        double s = 0;
        for (int c = 0; c < 4; ++c) s += J[a * 4 + c] * x[c];
        yv[a] = s;
      }
      for (int a = 0; a < 4; ++a) Sigma[(size_t)(3 + a) * ld + j] = yv[a];
    }
  }
  for (int il = tid; il < rows; il += BUPD_THREADS) {   // columns 3..6 of the CTA's rows but 3..6
    const int j = row0 + il;
    if (j >= 3 && j < 7) continue;
    double x[4], yv[4];
    double* row = Sigma + (size_t)j * ld + 3;
    for (int c = 0; c < 4; ++c) x[c] = row[c];
    for (int a = 0; a < 4; ++a) {
      double s = 0;
      for (int c = 0; c < 4; ++c) s += x[c] * J[a * 4 + c];
      yv[a] = s;
    }
    for (int a = 0; a < 4; ++a) row[a] = yv[a];
  }
  __syncthreads();
  cl_sync();
}

// A stacked update over the `cnt` features listed in ft.sel, in blocks of at most BK / 2 features.
__device__ void cl_feature_blocks(const UpdSmem& sm, int rank, double* Sigma, int ld, int n, const FeatTab& ft, int cnt,
                                  const DevCfg& cfg, DevCtl* ctl) {
  for (int a0 = 0; a0 < cnt; a0 += BK / 2) {
    const int m = min(BK / 2, cnt - a0);
    cl_gather_features(sm, rank, Sigma, ld, n, ft, a0, m, cfg);
    cl_block_gain_downdate(sm, rank, Sigma, ld, n, 2 * m, ctl);
  }
}

// high-innovation rescue (k_hi_rescue) by rank 0: pose from the old mu, feature parameters from mu_tmp; sets ft.hi, ft.sel, n_hi
static __device__ __noinline__ void cl_hi_rescue(double* Sigma, int ld, const double* mu, FeatTab ft, int N, DevCtl* ctl,
                                                 const DevCfg& cfg) {
  const int tid = threadIdx.x;
  for (int i = tid; i < N; i += BUPD_THREADS) {
    int flag = 0;
    if (!ft.li[i] && ft.innov[i]) {
      const int pos = ft.pos[i], coding = ft.coding[i];
      const int fsz = coding ? 3 : 6, nd = 7 + fsz;
      double fs[6], r[3], qc[4], Rcw[9], hi[2], Hc[26], hcz;
      for (int c = 0; c < fsz; ++c) fs[c] = mu[pos + c];
      for (int c = 0; c < 3; ++c) r[c] = ctl->cam_old[c];
      qc[0] = ctl->cam_old[3]; qc[1] = -ctl->cam_old[4]; qc[2] = -ctl->cam_old[5]; qc[3] = -ctl->cam_old[6];
      d_quat2rot(qc, Rcw);
      d_feature_hH(cfg.cam, fs, coding, r, qc, Rcw, hi, Hc, &hcz);
      ft.h[2 * i] = hi[0]; ft.h[2 * i + 1] = hi[1];
      for (int c = 0; c < 26; ++c) ft.Hc[26 * i + c] = Hc[c];
      double Tm[26];
      for (int bb = 0; bb < nd; ++bb) {
        const int jb = ekf_idx13(bb, pos);
        double sg[13];
#pragma unroll
        for (int c = 0; c < 13; ++c) sg[c] = (c < nd) ? Sigma[(size_t)ekf_idx13(c, pos) * ld + jb] : 0.0;
        double t0 = 0, t1 = 0;
#pragma unroll
        for (int c = 0; c < 13; ++c)
          if (c < nd) { t0 += Hc[c] * sg[c]; t1 += Hc[13 + c] * sg[c]; }
        Tm[bb] = t0; Tm[13 + bb] = t1;
      }
      double S[4] = {0, 0, 0, 0};
      for (int bb = 0; bb < nd; ++bb) {
        S[0] += Tm[bb] * Hc[bb]; S[1] += Tm[bb] * Hc[13 + bb];
        S[2] += Tm[13 + bb] * Hc[bb]; S[3] += Tm[13 + bb] * Hc[13 + bb];
      }
      const double det = S[0] * S[3] - S[2] * S[1];
      const double invdet = 1.0 / det;
      const double i00 = S[3] * invdet, i10 = -S[2] * invdet, i01 = -S[1] * invdet, i11 = S[0] * invdet;
      const double e0 = hi[0] - ft.z[2 * i], e1 = hi[1] - ft.z[2 * i + 1];
      const double t0 = e0 * i00 + e1 * i10;
      const double t1 = e0 * i01 + e1 * i11;
      const double chi = t0 * e0 + t1 * e1;
      flag = (chi <= cfg.th_hi) ? 1 : 0;
    }
    ft.hi[i] = flag;
  }
  __syncthreads();
  const int nh = block_compact(ft.hi, N, ft.sel, ft.pos_in_z);
  if (tid == 0) { ctl->n_hi = nh; ctl->k_rows = 2 * nh; }
}

template <bool PLANE, bool INTR, bool ACT>
__global__ void __launch_bounds__(BUPD_THREADS, 1) k_batch_update_cluster(BatchView bv, DevCfg cfg, const uint32_t* __restrict__ picks,
                                                                          int n_picks, double* __restrict__ out_mu14,
                                                                          double* __restrict__ out_S14, int* __restrict__ out_stats,
                                                                          int min_features, int max_features, int xyz_conversion,
                                                                          const int* __restrict__ act) {
  extern __shared__ __align__(16) double usm[];
  UpdSmem sm;
  sm.W = usm;
  sm.fact = sm.W + (size_t)BNMAX * BLDW;
  sm.Dv = sm.fact + kFactDoubles;
  sm.Sb = sm.Dv + (BK / 32) * 32 * BLDD;
  sm.nu = sm.Sb + (size_t)BK * BLDW;
  sm.y = sm.nu + BK;
  sm.mu_i = sm.y + BK;   // here: the correction delta of the CTA's rows
  sm.Hs = sm.mu_i + BNMAX;
  sm.qj = sm.Hs + BNCAP * 27;
  sm.ibuf = reinterpret_cast<int*>(sm.qj + 48);
  const int C = (int)cg::this_cluster().num_blocks(), rank = (int)cg::this_cluster().block_rank();
  const int b = act_filter<ACT>(act, blockIdx.x / C), tid = threadIdx.x;
  const int n = bv.n[b], N = bv.N[b], ld = bv.ld;
  double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  double* mu = bv.mu + (size_t)b * ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  DevCtl* ctl = bv.ctl + b;
  if constexpr (INTR) cfg.cam = bv.cam[b];   // every device function below projects with the filter's intrinsics
  for (int i = tid; i < BSTRIP; i += BUPD_THREADS) sm.mu_i[i] = 0.0;
  if (rank == 0) {   // 1-point RANSAC: mu_i (n <= 782) in the Cholesky workspace, the candidates (N <= 128) in ibuf
    if (tid == 0) ctl->chol_fail = 0;
    cta_ransac(Sigma, ld, n, mu, ft, N, ctl, cfg, picks, n_picks, sm.fact, sm.ibuf);
  }
  __syncthreads();
  cl_sync();
  const int n_li = *(volatile int*)&ctl->n_li;
  if (n_li > 0) {
    cl_feature_blocks(sm, rank, Sigma, ld, n, ft, n_li, cfg, ctl);
    cl_finish_update(sm, rank, Sigma, ld, n, mu);
  }
  if (rank == 0) cl_hi_rescue(Sigma, ld, mu, ft, N, ctl, cfg);
  __syncthreads();
  cl_sync();
  const int n_hi = *(volatile int*)&ctl->n_hi;
  if constexpr (PLANE) {   // the Hi blocks, the plane block, one normalisation
    if (n_hi > 0) cl_feature_blocks(sm, rank, Sigma, ld, n, ft, n_hi, cfg, ctl);
    cl_gather_plane(sm, rank, Sigma, ld, n, mu, ctl);
    cl_block_gain_downdate(sm, rank, Sigma, ld, n, 3, ctl);
    cl_finish_update(sm, rank, Sigma, ld, n, mu);
  } else {
    if (n_hi > 0) {
      cl_feature_blocks(sm, rank, Sigma, ld, n, ft, n_hi, cfg, ctl);
      cl_finish_update(sm, rank, Sigma, ld, n, mu);
    }
  }
  if (rank != 0) return;   // the last cluster barrier is behind every CTA: nobody reads this CTA's shared memory any more
  // book-keeping (k_bookkeeping) + visibility count (V:1296-1315), as k_batch_update
  int my_remove = 0, my_vis = 0;
  for (int i = tid; i < N; i += BUPD_THREADS) {
    int nfind = ft.n_find[i];
    const int ntot = ft.n_tot[i];
    if (ft.hi[i] || ft.li[i]) nfind++;
    ft.n_find[i] = nfind;
    const float qi = (float)(ntot - nfind) / ((float)nfind);
    ft.quality[i] = qi;
    if (qi > cfg.quality_ratio) ft.removef[i] = 1;
    if (ft.removef[i]) my_remove++;
    else if (ft.innov[i]) my_vis++;
  }
  const int n_rem = __syncthreads_count(my_remove);   // N <= 128 <= blockDim: one feature per thread
  const int n_vis = __syncthreads_count(my_vis);
  for (int e = tid; e < 14; e += BUPD_THREADS) out_mu14[(size_t)b * 14 + e] = mu[e];
  if (out_S14)
    for (int e = tid; e < 196; e += BUPD_THREADS) out_S14[(size_t)b * 196 + e] = Sigma[(size_t)(e / 14) * ld + (e % 14)];
  const bool drop_first = (n_vis < min_features) && (N - n_rem > max_features);
  if (tid == 0) {
    int* st = out_stats + (size_t)b * EKF_BATCH_STAT_FIELDS;
    int removed = n_rem, topup = 0;
    if (n_vis < min_features) {
      if (N - n_rem > max_features) removed += 1;   // removeFeature(0) (V:1313), applied by k_batch_compact
      topup = min_features - n_vis;
    }
    ctl->n_remove = removed;
    ctl->n_visible = n_vis;
    st[EKF_BSTAT_INNOV] = ctl->m_innov; st[EKF_BSTAT_MATCHED] = ctl->n_matched; st[EKF_BSTAT_LI] = n_li;
    st[EKF_BSTAT_HI] = n_hi; st[EKF_BSTAT_HYPS] = ctl->ransac_hyps; st[EKF_BSTAT_CHOL_FAIL] = ctl->chol_fail;
    st[EKF_BSTAT_REMOVED] = removed; st[EKF_BSTAT_TOPUP] = topup;
    int victim = -1;   // removeFeature(0)'s victim: the first feature not flagged (k_batch_update's decision)
    if (drop_first)
      for (int f = 0; f < N && victim < 0; ++f)
        if (!ft.removef[f]) victim = f;
    sm.ibuf[0] = victim;
  }
  __syncthreads();
  if (xyz_conversion) cta_xyz_decide(bv, b, Sigma, mu, ft, N, true, sm.ibuf[0], cfg);
}

// ------------------------------------------------------------------------------------------------
// removeFeature (V:373-421) for every flagged feature (remove != 0) and convert2XYZ_ifLinear (V:741-772) for every
// feature decided in bv.xyz_flag, of every filter that has either, in one pass: Sigma / mu are rebuilt through the
// filter's slice of the scratch buffer, the feature table through registers.  The row map carries (src, code) as in
// k_xyz_apply: code < 0 copies old entry src, code = 4 f + x is row x of converted feature f (old index).  Removal keeps
// the order of the survivors, so J Sigma J^T over the survivors' rows (xyz_apply_entry) is bit for bit the reference's
// removals followed by its one-at-a-time conversions.  A filter with nothing to do returns at once.
// ------------------------------------------------------------------------------------------------
#define BCMP_THREADS 256
// The feature archive of a batch (VSlamFilter::deleted_patches, ekf_batch_set_archive): cap records per filter, each a
// real_index and PTS_COLS doubles (ekf_points.cuh).  cap = 0: off, and nothing is archived.
struct BatchArchive {
  double* rec;       // [B][cap][PTS_COLS]
  int* real_index;   // [B][cap]
  int* count;        // [B] records held
  int* overflow;     // [B] records dropped for want of room, ever (ekf_batch_step compares it with its last read-back)
  int cap;
};

// hold (stats of the step, or NULL): a filter whose EKF_BSTAT_TOPUP is set only removes here, and its pending decisions move
// with the surviving records; the conversions follow its new features (ekf_batch_step).  NC: feature capacity (BNCAP or
// BNCAP_L); one CTA covers every entry of n2 x n2 either way, and every record (N2 <= 128 <= BCMP_THREADS).
// one >= 0 (grid of one CTA): removeFeature(one_idx) on filter `one` alone (ekf_batch_remove_feature): no other removal, no
// max_features rule, no conversion; pending decisions move with the records as under hold.  ACT: CTA i works on filter act[i].
// With the archive on, every removed feature that removeFeature archives (XYZ, n_find > 5) is appended to the filter's archive
// in the single filter's order: the flagged features in ascending index (ekf_update_after_match's victims), then the
// removeFeature(0) victim.  The records are read from Sigma and mu before the pass overwrites them.  A conversion fused into
// the same pass never touches a removed feature's block: the reference removes before it converts, the decisions exclude the
// removed features, and J is the identity on every row but the converted feature's.
template <int NC, bool ACT>
__global__ void __launch_bounds__(BCMP_THREADS, 1) k_batch_compact(BatchView bv, double* __restrict__ scratch, int min_features,
                                                                int max_features, int remove, const int* __restrict__ hold_stats,
                                                                BatchArchive ar, int one, int one_idx, const int* __restrict__ act) {
  constexpr int MV = (EKF_CAM + 6 * NC + BCMP_THREADS - 1) / BCMP_THREADS;   // state entries a thread moves: 1 at NC = 32
  __shared__ int keep[NC], newpos[NC], conv[NC], arch[NC];
  __shared__ int2 rmap[EKF_CAM + 6 * NC + 2];
  __shared__ int s_N2, s_n2, s_narch, s_abase;
  const bool single = one >= 0;
  const int b = single ? one : act_filter<ACT>(act, blockIdx.x), tid = threadIdx.x;
  DevCtl* ctl = bv.ctl + b;
  const bool rem = single || (remove && ctl->n_remove > 0);
  const bool hold = single || (hold_stats && hold_stats[(size_t)b * EKF_BATCH_STAT_FIELDS + EKF_BSTAT_TOPUP] > 0);
  const int nconv = hold ? 0 : bv.xyz_count[b];
  if (!rem && nconv <= 0) return;
  const int N = bv.N[b], ld = bv.ld;
  double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  double* tmp = scratch + (size_t)b * bv.sstride;
  double* mu = bv.mu + (size_t)b * ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  int* cflag = bv.xyz_flag + (size_t)b * bv.Ncap;
  double* Jall = bv.xyz_J + (size_t)b * bv.Ncap * 18;
  double* yall = bv.xyz_y + (size_t)b * bv.Ncap * 3;
  if (tid == 0) {
#define DEAD(f) (single ? (f) == one_idx : (rem && ft.removef[f] != 0))
    int flagged = 0;
    for (int f = 0; f < N; ++f) flagged += DEAD(f) ? 1 : 0;
    // removeFeature(0) after the flagged ones are gone (V:1312-1313): first survivor
    const bool drop_first = !single && rem && (ctl->n_visible < min_features) && (N - flagged > max_features);
    int victim = -1;
    for (int f = 0; drop_first && f < N && victim < 0; ++f)
      if (!DEAD(f)) victim = f;
    if (ar.cap > 0) {   // archive order: the flagged features ascending, then the victim
      int na = 0;
      for (int f = 0; f < N; ++f)
        if (DEAD(f) && pts_archived(ft.coding[f], ft.n_find[f])) arch[na++] = f;
      if (victim >= 0 && pts_archived(ft.coding[victim], ft.n_find[victim])) arch[na++] = victim;
      const int base = ar.count[b], room = base < ar.cap ? ar.cap - base : 0, kept = na < room ? na : room;
      ar.count[b] = base + kept;
      if (na > kept) ar.overflow[b] += na - kept;
      s_narch = kept; s_abase = base;
    }
    int N2 = 0, n2 = EKF_CAM;
    for (int i = 0; i < EKF_CAM; ++i) rmap[i] = make_int2(i, -1);
    for (int f = 0; f < N; ++f) {
      if (DEAD(f) || f == victim) continue;
      const int cv = nconv > 0 && cflag[f];
      keep[N2] = f; newpos[N2] = n2; conv[N2] = cv; ++N2;
      if (cv) {
        for (int x = 0; x < 3; ++x) rmap[n2++] = make_int2(ft.pos[f], 4 * f + x);
      } else {
        const int fs = ft.coding[f] ? 3 : 6;
        for (int c = 0; c < fs; ++c) rmap[n2++] = make_int2(ft.pos[f] + c, -1);
      }
    }
    s_N2 = N2; s_n2 = n2;
#undef DEAD
  }
  __syncthreads();
  const int N2 = s_N2, n2 = s_n2;
  if (ar.cap > 0)   // before Sigma, mu and the table are rewritten (barriers below)
    for (int k = tid; k < s_narch; k += BCMP_THREADS) {
      const int f = arch[k];
      const size_t slot = (size_t)b * ar.cap + s_abase + k;
      pts_record(mu, Sigma, ld, ft.pos[f], ar.rec + slot * PTS_COLS);
      ar.real_index[slot] = ft.real_index[f];
    }
  for (int e = tid; e < n2 * n2; e += BCMP_THREADS) {
    const int i = e / n2, j = e - i * n2;
    tmp[(size_t)i * ld + j] = xyz_apply_entry(Sigma, ld, rmap[i], rmap[j], Jall);
  }
  double mv[MV];
#pragma unroll
  for (int q = 0; q < MV; ++q) {
    const int i = tid + q * BCMP_THREADS;
    mv[q] = 0.0;
    if (i < n2) {
      const int2 r = rmap[i];
      mv[q] = (r.y < 0) ? mu[r.x] : yall[3 * (r.y >> 2) + (r.y & 3)];
    }
  }
  __syncthreads();
  for (int e = tid; e < n2 * n2; e += BCMP_THREADS) {
    const int i = e / n2, j = e - i * n2;
    Sigma[(size_t)i * ld + j] = tmp[(size_t)i * ld + j];
  }
#pragma unroll
  for (int q = 0; q < MV; ++q)
    if (tid + q * BCMP_THREADS < n2) mu[tid + q * BCMP_THREADS] = mv[q];
  // feature table: thread f < N2 moves record keep[f] -> f through registers
  const int w16 = bv.tstride >> 4;
  int o = -1;
  int iv[10]; float fv[4]; double dv[8 + 26];
  int hflag = 0; double hJ[18], hy[3];   // held decision of the record (hold only)
  if (tid < N2) {
    o = keep[tid];
    iv[0] = ft.coding[o]; iv[1] = ft.innov[o]; iv[2] = ft.li[o]; iv[3] = ft.hi[o]; iv[4] = ft.removef[o];
    iv[5] = ft.n_tot[o]; iv[6] = ft.n_find[o]; iv[7] = ft.real_index[o]; iv[8] = ft.pos_in_z[o]; iv[9] = 0;
    fv[0] = ft.center[2 * o]; fv[1] = ft.center[2 * o + 1]; fv[2] = ft.quality[o]; fv[3] = ft.last_ncc[o];
    for (int c = 0; c < 2; ++c) { dv[c] = ft.z[2 * o + c]; dv[2 + c] = ft.h[2 * o + c]; }
    for (int c = 0; c < 4; ++c) dv[4 + c] = ft.S2[4 * o + c];
    for (int c = 0; c < 26; ++c) dv[8 + c] = ft.Hc[26 * o + c];
    if (hold) {
      hflag = cflag[o];
      for (int c = 0; c < 18; ++c) hJ[c] = Jall[18 * o + c];
      for (int c = 0; c < 3; ++c) hy[c] = yall[3 * o + c];
    }
  }
  __syncthreads();
  if (tid < N2) {
    ft.pos[tid] = newpos[tid]; ft.coding[tid] = conv[tid] ? 1 : iv[0]; ft.innov[tid] = iv[1]; ft.li[tid] = iv[2]; ft.hi[tid] = iv[3];
    ft.removef[tid] = iv[4]; ft.n_tot[tid] = iv[5]; ft.n_find[tid] = iv[6]; ft.real_index[tid] = iv[7]; ft.pos_in_z[tid] = iv[8];
    ft.center[2 * tid] = fv[0]; ft.center[2 * tid + 1] = fv[1]; ft.quality[tid] = fv[2]; ft.last_ncc[tid] = fv[3];
    for (int c = 0; c < 2; ++c) { ft.z[2 * tid + c] = dv[c]; ft.h[2 * tid + c] = dv[2 + c]; }
    for (int c = 0; c < 4; ++c) ft.S2[4 * tid + c] = dv[4 + c];
    for (int c = 0; c < 26; ++c) ft.Hc[26 * tid + c] = dv[8 + c];
    if (hold) {
      cflag[tid] = hflag;
      for (int c = 0; c < 18; ++c) Jall[18 * tid + c] = hJ[c];
      for (int c = 0; c < 3; ++c) yall[3 * tid + c] = hy[c];
    }
  }
  // templates: records only move towards lower indices, in ascending order
  for (int f = 0; f < N2; ++f) {
    const int src = keep[f];
    if (src == f) continue;
    uint4 a = make_uint4(0, 0, 0, 0), c = make_uint4(0, 0, 0, 0);
    if (tid < w16) {
      a = reinterpret_cast<const uint4*>(ft.patch + (size_t)src * bv.tstride)[tid];
      c = reinterpret_cast<const uint4*>(ft.mpatch + (size_t)src * bv.tstride)[tid];
    }
    __syncthreads();
    if (tid < w16) {
      reinterpret_cast<uint4*>(ft.patch + (size_t)f * bv.tstride)[tid] = a;
      reinterpret_cast<uint4*>(ft.mpatch + (size_t)f * bv.tstride)[tid] = c;
    }
    __syncthreads();
  }
  if (tid == 0) {
    bv.n[b] = n2; bv.N[b] = N2;
    if (!hold) bv.xyz_count[b] = 0;
    if (remove) ctl->n_remove = 0;
  }
}

// convert2XYZ_ifLinearAll (V:776-780) outside a step: the decisions of every filter, one CTA per filter, one thread per
// feature; k_batch_compact (remove = 0) applies them.
__global__ void __launch_bounds__(BNCAP) k_batch_xyz_decide(BatchView bv, DevCfg cfg) {
  const int b = blockIdx.x;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  warp_xyz_decide(bv, b, bv.Sigma + (size_t)b * bv.sstride, bv.mu + (size_t)b * bv.ld, ft, bv.N[b], true, cfg);
}
// The same for a large batch (capacity up to BNCAP_L): one thread per feature, BNCAP_L threads.
__global__ void __launch_bounds__(BNCAP_L) k_batch_xyz_decide_large(BatchView bv, DevCfg cfg) {
  const int b = blockIdx.x;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  cta_xyz_decide(bv, b, bv.Sigma + (size_t)b * bv.sstride, bv.mu + (size_t)b * bv.ld, ft, bv.N[b], false, -1, cfg);
}

// addFeature (V:309-371) for the corners of every filter that has some (cnt[b] of them at xy + 2 * EKF_BATCH_MAX_CORNERS * b),
// one CTA per filter, one add after the other in corner order with a barrier between adds: add j reads the rows add j - 1
// wrote, exactly as consecutive ekf_add_feature calls do, and through the same device functions (ekf_math.cuh), so the
// result is the single filter's bit for bit.  n <= 200 before an add, so one CTA covers every row.  one >= 0: filter `one`
// adds the pixel (u, v) instead.  decide: the new features' convert2XYZ_ifLinear decisions join the ones k_batch_update
// took for the filter's older features (adds change no entry their linearity test reads), for k_batch_compact to apply.
// LARGE (capacity up to BNCAP_L): the corners sit at xy + 2 * BNCAP_L * b, the rows (n <= 776 before an add) are taken
// BADD_THREADS at a time and the decisions one thread per feature.  Templates come from frame cam_of[b] of the stack fr
// (cam_of null: frame 0).  ACT: CTA i works on filter act[i] (ekf_batch_step_filters).
#define BADD_THREADS 256
template <bool LARGE, bool INTR, bool ACT>
__global__ void __launch_bounds__(BADD_THREADS) k_batch_add(BatchView bv, FrameView fr, DevCfg cfg, const float* __restrict__ xy,
                                                            const int* __restrict__ cnt, int one, float u, float v, int decide,
                                                            const int* __restrict__ cam_of, const int* __restrict__ act) {
  constexpr int CS = LARGE ? BNCAP_L : EKF_BATCH_MAX_CORNERS;   // corner stride of xy
  __shared__ double A[6 * 7], Ap[6 * 3], fnew[6], Tc[6 * 7];
  const int b = one >= 0 ? one : (ACT ? act[blockIdx.x] : blockIdx.x), tid = threadIdx.x;
  const int k = one >= 0 ? 1 : cnt[b];
  if (k <= 0) return;
  if (cam_of) fr.px += (size_t)cam_of[b] * fr.h * fr.stride;
  const int ld = bv.ld, w = cfg.window, w2 = w * w;
  double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  double* mu = bv.mu + (size_t)b * ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  int n = bv.n[b], N = bv.N[b], real = bv.patchnumbre[b];
  const int N0 = N;
  for (int j = 0; j < k; ++j) {
    const float px = one >= 0 ? u : xy[(size_t)b * 2 * CS + 2 * j];
    const float py = one >= 0 ? v : xy[(size_t)b * 2 * CS + 2 * j + 1];
    if (tid == 0) add_feature_jacobians(filter_cam<INTR>(bv, cfg, b), mu, px, py, cfg.rho_0, A, Ap, fnew);
    __syncthreads();
    if constexpr (LARGE) {
      for (int r = tid; r < n; r += BADD_THREADS) add_feature_cross(Sigma, ld, n, r, A);
    } else {
      if (tid < n) add_feature_cross(Sigma, ld, n, tid, A);
    }
    for (int e = tid; e < 42; e += BADD_THREADS) Tc[e] = add_feature_corner_T(Sigma, ld, A, e);   // rows / columns < 7: not written above
    __syncthreads();
    for (int e = tid; e < 36; e += BADD_THREADS)
      Sigma[(size_t)(n + e / 6) * ld + n + e % 6] = add_feature_corner(Tc, A, Ap, e, cfg.sigma_pixel_2, cfg.sigma_rho_0);
    if (tid < 6) mu[n + tid] = fnew[tid];
    for (int e = tid; e < w2; e += BADD_THREADS) ft.patch[(size_t)N * cfg.tstride + e] = add_feature_template_px(fr, w, px, py, e);
    if (tid == 0) add_feature_record(ft, N, n, px, py, real);
    __syncthreads();
    n += 6; N += 1; real += 1;
  }
  if (tid == 0) { bv.n[b] = n; bv.N[b] = N; bv.patchnumbre[b] = real; }
  if constexpr (LARGE) {
    if (decide) {   // one thread per feature (N <= BNCAP_L <= BADD_THREADS)
      const int i = tid;
      const size_t kk = (size_t)b * bv.Ncap + i;
      int conv = 0;
      if (i >= N0 && i < N) {
        const int pos = ft.pos[i];
        conv = xyz_linear_decide(mu + pos, mu, Sigma[(size_t)(pos + 5) * ld + pos + 5], cfg.linearity_threshold, cfg.abs_int_quirk,
                                 bv.xyz_y + 3 * kk, bv.xyz_J + 18 * kk);
        bv.xyz_flag[kk] = conv;
      }
      const int c = __syncthreads_count(conv);
      if (i == 0) bv.xyz_count[b] += c;
    }
    return;
  }
  if (decide && tid < 32) {   // N <= BNCAP = 32
    const int i = tid;
    const size_t kk = (size_t)b * bv.Ncap + i;
    int conv = 0;
    if (i >= N0 && i < N) {
      const int pos = ft.pos[i];
      conv = xyz_linear_decide(mu + pos, mu, Sigma[(size_t)(pos + 5) * ld + pos + 5], cfg.linearity_threshold, cfg.abs_int_quirk,
                               bv.xyz_y + 3 * kk, bv.xyz_J + 18 * kk);
      bv.xyz_flag[kk] = conv;
    }
    const int c = __popc(__ballot_sync(0xffffffffu, conv));
    if (i == 0) bv.xyz_count[b] += c;
  }
}

// seed: every filter <- the single filter `src`
__global__ void __launch_bounds__(256) k_batch_seed(BatchView bv, const double* __restrict__ Ssrc, int ld_src,
                                                    const double* __restrict__ musrc, FeatTab src, int n, int N, int patchnumbre) {
  const int b = blockIdx.x, tid = threadIdx.x;
  double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  double* mu = bv.mu + (size_t)b * bv.ld;
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  for (int e = tid; e < n * n; e += 256) {
    const int i = e / n, j = e - i * n;
    Sigma[(size_t)i * bv.ld + j] = Ssrc[(size_t)i * ld_src + j];
  }
  for (int e = tid; e < n; e += 256) mu[e] = musrc[e];
  for (int f = tid; f < N; f += 256) {
    ft.pos[f] = src.pos[f]; ft.coding[f] = src.coding[f]; ft.innov[f] = src.innov[f]; ft.li[f] = src.li[f]; ft.hi[f] = src.hi[f];
    ft.removef[f] = src.removef[f]; ft.n_tot[f] = src.n_tot[f]; ft.n_find[f] = src.n_find[f]; ft.real_index[f] = src.real_index[f];
    ft.pos_in_z[f] = src.pos_in_z[f]; ft.quality[f] = src.quality[f]; ft.last_ncc[f] = src.last_ncc[f];
    for (int c = 0; c < 2; ++c) { ft.center[2 * f + c] = src.center[2 * f + c]; ft.z[2 * f + c] = src.z[2 * f + c]; ft.h[2 * f + c] = src.h[2 * f + c]; }
    for (int c = 0; c < 4; ++c) ft.S2[4 * f + c] = src.S2[4 * f + c];
    for (int c = 0; c < 26; ++c) ft.Hc[26 * f + c] = src.Hc[26 * f + c];
  }
  for (int e = tid; e < N * bv.tstride; e += 256) { ft.patch[e] = src.patch[e]; ft.mpatch[e] = src.mpatch[e]; }
  if (tid == 0) { bv.n[b] = n; bv.N[b] = N; bv.ctl[b] = DevCtl{}; bv.patchnumbre[b] = patchnumbre; }
}
// deleted_patches of the seed filter into every filter's archive (ekf_batch_seed_from with the archive on): n records staged at
// rec / ri.
__global__ void __launch_bounds__(256) k_batch_seed_archive(BatchArchive ar, const double* __restrict__ rec, const int* __restrict__ ri,
                                                            int n) {
  const int b = blockIdx.x, tid = threadIdx.x;
  double* dst = ar.rec + (size_t)b * ar.cap * PTS_COLS;
  for (int e = tid; e < n * PTS_COLS; e += 256) dst[e] = rec[e];
  for (int e = tid; e < n; e += 256) ar.real_index[(size_t)b * ar.cap + e] = ri[e];
  if (tid == 0) ar.count[b] = n;
}

// RosVSLAM::getPointsFeatures (RosVSLAMRansac.cpp:340-418) for filters [first, first + gridDim.x), one CTA per filter, with the
// row assembly of ekf_points.cuh: rows_out / held_out receive each filter's row count and archive size.  With out (a
// rows_cap x PTS_COLS slice per filter, zeroed here) and the filter's rows within rows_cap: the live XYZ rows, one thread per
// feature, then the archived records in archive order, warp 0 taking 32 at a time (of records with the same real_index the
// later one writes, as sequential overwrites would leave it).  map_scale is the filter's mu[13].  The clear rule
// (pts_clears) is the caller's, once every requested filter is known to fit.
#define BPTS_THREADS 256
__global__ void __launch_bounds__(BPTS_THREADS) k_batch_points_features(BatchView bv, BatchArchive ar, int first, int rows_cap,
                                                                        double* __restrict__ out, int* __restrict__ rows_out,
                                                                        int* __restrict__ held_out) {
  const int k = blockIdx.x, b = first + k, tid = threadIdx.x;
  const int N = bv.N[b];
  const FeatTab ft = feattab_slice(bv.ft, b, bv.Ncap, bv.tstride);
  const int rows = pts_row_count(N, ft.real_index);
  const int held = ar.cap > 0 ? ar.count[b] : 0;
  if (tid == 0) { rows_out[k] = rows; held_out[k] = held; }
  if (!out || rows > rows_cap) return;
  double* o = out + (size_t)k * rows_cap * PTS_COLS;
  for (size_t e = tid; e < (size_t)rows * PTS_COLS; e += BPTS_THREADS) o[e] = 0.0;
  for (size_t e = (size_t)rows * PTS_COLS + tid; e < (size_t)rows_cap * PTS_COLS; e += BPTS_THREADS) o[e] = 0.0;
  __syncthreads();
  const double* mu = bv.mu + (size_t)b * bv.ld;
  const double* Sigma = bv.Sigma + (size_t)b * bv.sstride;
  const double map_scale = mu[13];
  for (int i = tid; i < N; i += BPTS_THREADS) {
    const int ri = ft.real_index[i];
    if (pts_archive_in_range(ri, rows)) pts_live_row(ft.coding[i], ft.pos[i], mu, Sigma, bv.ld, map_scale, o + (size_t)ri * PTS_COLS);
  }
  __syncthreads();
  if (tid < 32) {
    for (int k0 = 0; k0 < held; k0 += 32) {
      const int kk = k0 + tid;
      const size_t slot = (size_t)b * ar.cap + kk;
      const int ri = kk < held ? ar.real_index[slot] : -1;
      const bool in = kk < held && pts_archive_in_range(ri, rows);
      const unsigned same = __match_any_sync(0xffffffffu, in ? ri : -1);
      if (in && (same & ~((2u << tid) - 1u)) == 0u) pts_archive_row(ar.rec + slot * PTS_COLS, map_scale, o + (size_t)ri * PTS_COLS);
      __syncwarp();
    }
  }
}

__global__ void k_batch_set_cam(BatchView bv, const double* __restrict__ mu14, int B) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < B * 14) bv.mu[(size_t)(e / 14) * bv.ld + (e % 14)] = mu14[e];
}

// The rows ekf_batch_get_camera_states reports, mu[0:14] and Sigma[0:14, 0:14], of every filter from its state as it stands: a
// step with a list writes only its filters' rows, so the others' are gathered here after a call that changed them.
__global__ void k_batch_camera_rows(BatchView bv, double* __restrict__ out_mu14, double* __restrict__ out_S14, int B) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * 210) return;
  const int b = e / 210, r = e - b * 210;
  if (r < 14) out_mu14[(size_t)b * 14 + r] = bv.mu[(size_t)b * bv.ld + r];
  else out_S14[(size_t)b * 196 + r - 14] = bv.Sigma[(size_t)b * bv.sstride + (size_t)((r - 14) / 14) * bv.ld + (r - 14) % 14];
}

// Everything of a filter that a later call reads (ekf_batch_resample), in a set of slots: the batch's own, or the staging slots of
// filters that are both copied from and overwritten (Sigma in the compaction scratch, the rest in a temporary buffer).  All sets
// share the batch's ld, sstride, Ncap, tstride and archive capacity.
struct BatchSlots {
  BatchView v;        // Sigma, mu, ft, ctl, n, N, patchnumbre, xyz_*; v.cam is not used (cam below)
  BatchArchive ar;    // records, count, overflow; cap 0: no archive
  CamParams* cam;     // intrinsics row; null: the batch has no table
  double* mu14;       // [14] the camera rows ekf_batch_get_camera_states reports
  double* S14;        // [196]
  int* stats;         // [EKF_BATCH_STAT_FIELDS] the last step's counters (findNewFeatures(NULL) reads EKF_BSTAT_TOPUP)
};

// dst slot pairs[p].x <- src slot pairs[p].y, for p = blockIdx.x.  Sigma rows [0, n) are n * ld contiguous doubles: gridDim.y CTAs
// share them in 16-byte vectors (sstride and ld are multiples of 8 doubles), four loads in flight a thread.  CTA y = 0 also copies
// the rest: mu[0, n), the N table entries and templates, the pending XYZ decisions, the archive's held records, the rows.
#define BRS_THREADS 256
__global__ void __launch_bounds__(BRS_THREADS, 4) k_batch_resample(BatchSlots dst, BatchSlots src, const int2* __restrict__ pairs) {
  const int2 pr = pairs[blockIdx.x];
  const int d = pr.x, s = pr.y, tid = threadIdx.x;
  const int n = src.v.n[s], N = src.v.N[s];
  const double2* __restrict__ S = reinterpret_cast<const double2*>(src.v.Sigma + (size_t)s * src.v.sstride);
  double2* __restrict__ D = reinterpret_cast<double2*>(dst.v.Sigma + (size_t)d * dst.v.sstride);
  const size_t nv = (size_t)n * src.v.ld / 2, stride = (size_t)gridDim.y * BRS_THREADS;
  size_t i = (size_t)blockIdx.y * BRS_THREADS + tid;
  for (; i + 3 * stride < nv; i += 4 * stride) {
    const double2 a = S[i], b = S[i + stride], c = S[i + 2 * stride], e = S[i + 3 * stride];
    D[i] = a; D[i + stride] = b; D[i + 2 * stride] = c; D[i + 3 * stride] = e;
  }
  for (; i < nv; i += stride) D[i] = S[i];
  if (blockIdx.y != 0) return;

  const double* smu = src.v.mu + (size_t)s * src.v.ld;
  double* dmu = dst.v.mu + (size_t)d * dst.v.ld;
  for (int e = tid; e < n; e += BRS_THREADS) dmu[e] = smu[e];
  const int Ncap = src.v.Ncap, ts = src.v.tstride;
  const FeatTab a = feattab_slice(src.v.ft, s, Ncap, ts), o = feattab_slice(dst.v.ft, d, Ncap, ts);
  const size_t ks = (size_t)s * Ncap, kd = (size_t)d * Ncap;
  for (int f = tid; f < N; f += BRS_THREADS) {
    o.pos[f] = a.pos[f]; o.coding[f] = a.coding[f]; o.innov[f] = a.innov[f]; o.li[f] = a.li[f]; o.hi[f] = a.hi[f];
    o.removef[f] = a.removef[f]; o.n_tot[f] = a.n_tot[f]; o.n_find[f] = a.n_find[f]; o.real_index[f] = a.real_index[f];
    o.pos_in_z[f] = a.pos_in_z[f]; o.sel[f] = a.sel[f]; o.quality[f] = a.quality[f]; o.last_ncc[f] = a.last_ncc[f];
    dst.v.xyz_flag[kd + f] = src.v.xyz_flag[ks + f];
  }
  for (int e = tid; e < 2 * N; e += BRS_THREADS) { o.center[e] = a.center[e]; o.z[e] = a.z[e]; o.h[e] = a.h[e]; }
  for (int e = tid; e < 4 * N; e += BRS_THREADS) o.S2[e] = a.S2[e];
  for (int e = tid; e < 26 * N; e += BRS_THREADS) o.Hc[e] = a.Hc[e];
  for (int e = tid; e < 18 * N; e += BRS_THREADS) dst.v.xyz_J[18 * kd + e] = src.v.xyz_J[18 * ks + e];
  for (int e = tid; e < 3 * N; e += BRS_THREADS) dst.v.xyz_y[3 * kd + e] = src.v.xyz_y[3 * ks + e];
  {   // both templates, tstride a multiple of 16 bytes
    const uint4* __restrict__ p = reinterpret_cast<const uint4*>(a.patch);
    const uint4* __restrict__ m = reinterpret_cast<const uint4*>(a.mpatch);
    uint4* __restrict__ po = reinterpret_cast<uint4*>(o.patch);
    uint4* __restrict__ mo = reinterpret_cast<uint4*>(o.mpatch);
    for (int e = tid; e < N * ts / 16; e += BRS_THREADS) { po[e] = p[e]; mo[e] = m[e]; }
  }
  if (src.ar.cap > 0) {
    const int held = src.ar.count[s];
    const double* r = src.ar.rec + (size_t)s * src.ar.cap * PTS_COLS;
    double* ro = dst.ar.rec + (size_t)d * dst.ar.cap * PTS_COLS;
    for (int e = tid; e < held * PTS_COLS; e += BRS_THREADS) ro[e] = r[e];
    for (int e = tid; e < held; e += BRS_THREADS) dst.ar.real_index[(size_t)d * dst.ar.cap + e] = src.ar.real_index[(size_t)s * src.ar.cap + e];
    if (tid == 0) { dst.ar.count[d] = held; dst.ar.overflow[d] = src.ar.overflow[s]; }
  }
  if (tid < 14) dst.mu14[(size_t)d * 14 + tid] = src.mu14[(size_t)s * 14 + tid];
  if (tid < 196) dst.S14[(size_t)d * 196 + tid] = src.S14[(size_t)s * 196 + tid];
  if (tid < EKF_BATCH_STAT_FIELDS)
    dst.stats[(size_t)d * EKF_BATCH_STAT_FIELDS + tid] = src.stats[(size_t)s * EKF_BATCH_STAT_FIELDS + tid];
  if (tid == 0) {
    dst.v.n[d] = n; dst.v.N[d] = N; dst.v.patchnumbre[d] = src.v.patchnumbre[s]; dst.v.xyz_count[d] = src.v.xyz_count[s];
    dst.v.ctl[d] = src.v.ctl[s];
    if (src.cam) dst.cam[d] = src.cam[s];
  }
}

// frame z of a stack of dw x dh slots: every pixel outside the camera's fsize[4z + 2] x fsize[4z + 3] becomes 0.  SLOTS: frame z is
// slot slot[z].
template <bool SLOTS>
__global__ void k_batch_zero_pads(uint8_t* __restrict__ frame, int dw, int dstride, int dh, const int* __restrict__ fsize,
                                  const int* __restrict__ slot) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= dw) return;
  const int z = SLOTS ? slot[blockIdx.z] : blockIdx.z;
  const int* q = fsize + 4 * z;
  if (x >= q[2] || y >= q[3]) frame[((size_t)z * dh + y) * dstride + x] = 0;
}

// ================================================================================================
// host side
// ================================================================================================
struct ekf_batch {
  ekf_config cfg;
  DevCfg dcfg;
  int device = 0, B = 0, Ncap = 0, ncap = 0, ld = 0;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  BatchView bv{};
  double* scratch = nullptr;
  uint8_t* frame = nullptr;                     // n_cam frames of fv.stride x fv.h, contiguous
  size_t frame_cap = 0;
  uint8_t* raw = nullptr;                       // device staging of host frames that are resized or converted (cfg.scale > 1 or BGR)
  size_t raw_cap = 0;
  int n_cam = 1;                                // cameras (ekf_batch_set_cameras)
  int* cam_dev = nullptr;                       // [B] camera of each filter; null with one camera
  std::vector<int> cam_host;                    // [B] the same on the host
  std::vector<double> cam_dT, cam_ts;           // [n_cam] each camera's dT / old_ts (captureNewFrame's clock)
  std::vector<int> size_in;                     // [n_cam][2] input frame sizes (ekf_batch_set_frame_sizes); empty: the whole slot
  std::vector<int> fsize_host;                  // [n_cam][4] in w, in h, resized w, h of the last capture with sizes (fsize_dev)
  int* fsize_dev = nullptr;
  bool fsize_on = false;                        // the captured stack has per-camera sizes
  CamParams* intr_dev = nullptr;                // [B] intrinsics of each filter (ekf_batch_set_intrinsics); bv.cam, null without
  int* det_slot = nullptr;                      // [n_cam] position of each camera among those a detection asks from, or -1
  int* h_det_slot = nullptr;                    // pinned
  size_t det_budget = (size_t)1 << 30;          // scratch of one chunk of cameras of the per-camera detector
  void* step_dev = nullptr;                     // a step's per-camera dT, per-filter controls and picks, uploaded in one copy
  void* step_host = nullptr;                    // pinned
  size_t step_cap = 0;
  FrameView fv{nullptr, 0, 0, 0};
  EkfTensorMap frame_map{};
  int* match_defer = nullptr;   // [B * Ncap] (filter, feature) pairs the warp matcher left to the CTA matcher, then the count
  uint32_t* picks_dev = nullptr;
  int picks_cap = 0;
  double *out_mu14 = nullptr, *out_S14 = nullptr;
  int* out_stats = nullptr;
  double *h_mu14 = nullptr, *h_S14 = nullptr;   // pinned
  int* h_stats = nullptr;                       // pinned
  int* h_xyz_count = nullptr;                   // pinned mirror of bv.xyz_count
  int *h_n = nullptr, *h_N = nullptr;           // pinned mirrors of bv.n / bv.N
  double* stage_mu14 = nullptr;                 // device staging for set_camera_states
  BatchDetectBufs det;                          // batched corner detection (ekf_batch_detect.cu)
  float* det_xy = nullptr;                      // [B][cstride][2] corners of the last detection
  int *det_n = nullptr, *det_num = nullptr;     // [B] their count; [B] corners asked for (host num staged)
  float* h_det_xy = nullptr;                    // pinned
  int *h_det_n = nullptr, *h_num = nullptr;     // pinned
  int* h_added = nullptr;                       // pinned: features each filter added in the last step / top-up call
  int* blur_out = nullptr;                      // [2][B] k_batch_predict_blur: templates blurred, kernel too large
  int* h_blur = nullptr;                        // pinned mirror of blur_out
  std::vector<char> cam_frame;                  // [n_cam] the camera holds a frame (a capture that listed it since the frames were forgotten)
  int* slot_dev = nullptr;                      // [n_cam] destination slots of a capture of listed cameras
  bool rows_stale = true;                       // out_mu14 / out_S14 may differ from some filter's state (seed, set_camera_states, set_full)
  bool seeded = false, results_valid = false, topup = false, blur = false;
  bool large = false;                           // ekf_batch_create_large with capacity > 32: the cluster update, BNCAP_L kernels
  int cl_ctas = 1, cl_resident = 0;             // CTAs per filter in the update; clusters resident at once (large only)
  int cstride = EKF_BATCH_MAX_CORNERS;          // corners per filter in det_xy (BNCAP_L when large)
  long long launches = 0;
  BatchArchive ar{};                            // feature archive (ekf_batch_set_archive; cap 0: off)
  int* h_over = nullptr;                        // pinned mirror of ar.overflow, read back with the step's n / N
  std::vector<int> over_seen;                   // ar.overflow at the last check
  int *pts_dev = nullptr, *h_pts = nullptr;     // [2][B] row counts and archive sizes of ekf_batch_get_points_features; pinned mirror
  int2* rs_pairs = nullptr;                     // [2 * B] (destination, source) slot pairs of ekf_batch_resample's launches
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::string err;
};

static int bfail(ekf_batch* b, int code, const std::string& msg) {
  if (b) b->err = msg;
  return code;
}
#define BCHECK(expr)                                                                                    \
  do {                                                                                                  \
    cudaError_t _e = (expr);                                                                            \
    if (_e != cudaSuccess) {                                                                            \
      char _buf[400];                                                                                   \
      snprintf(_buf, sizeof _buf, "CUDA error %d (%s) at %s:%d: %s", (int)_e, cudaGetErrorString(_e), __FILE__, __LINE__, #expr); \
      return bfail(b, EKF_ERR_CUDA, _buf);                                                              \
    }                                                                                                   \
  } while (0)

template <class T>
static cudaError_t balloc(T** p, size_t count) { return cudaMalloc((void**)p, sizeof(T) * std::max<size_t>(count, 1)); }

extern "C" {

const char* ekf_batch_last_error(const ekf_batch* b) { return b ? b->err.c_str() : "null batch"; }

int ekf_batch_destroy(ekf_batch* b) {
  if (!b) return EKF_OK;
  cudaSetDevice(b->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  FeatTab& t = b->bv.ft;
  cudaFree(t.pos); cudaFree(t.coding); cudaFree(t.innov); cudaFree(t.li); cudaFree(t.hi); cudaFree(t.removef);
  cudaFree(t.n_tot); cudaFree(t.n_find); cudaFree(t.real_index); cudaFree(t.pos_in_z); cudaFree(t.sel);
  cudaFree(t.center); cudaFree(t.quality); cudaFree(t.last_ncc); cudaFree(t.z); cudaFree(t.h); cudaFree(t.Hc);
  cudaFree(t.S2); cudaFree(t.patch); cudaFree(t.mpatch);
  cudaFree(b->bv.xyz_flag); cudaFree(b->bv.xyz_J); cudaFree(b->bv.xyz_y); cudaFree(b->bv.xyz_count);
  cudaFree(b->bv.Sigma); cudaFree(b->bv.mu); cudaFree(b->bv.ctl); cudaFree(b->bv.n); cudaFree(b->bv.N);
  cudaFree(b->match_defer);
  cudaFree(b->scratch); cudaFree(b->frame); cudaFree(b->raw); cudaFree(b->picks_dev); cudaFree(b->out_mu14); cudaFree(b->out_S14);
  cudaFree(b->out_stats); cudaFree(b->stage_mu14); cudaFree(b->bv.patchnumbre);
  cudaFree(b->cam_dev); cudaFree(b->det_slot); cudaFree(b->step_dev); cudaFree(b->intr_dev); cudaFree(b->fsize_dev); cudaFree(b->slot_dev);
  if (b->h_det_slot) cudaFreeHost(b->h_det_slot);
  if (b->step_host) cudaFreeHost(b->step_host);
  batch_detect_free(b->det);
  cudaFree(b->det_xy); cudaFree(b->det_n); cudaFree(b->det_num);
  if (b->h_det_xy) cudaFreeHost(b->h_det_xy);
  if (b->h_det_n) cudaFreeHost(b->h_det_n);
  if (b->h_num) cudaFreeHost(b->h_num);
  if (b->h_added) cudaFreeHost(b->h_added);
  cudaFree(b->blur_out);
  if (b->h_blur) cudaFreeHost(b->h_blur);
  if (b->h_mu14) cudaFreeHost(b->h_mu14);
  if (b->h_S14) cudaFreeHost(b->h_S14);
  if (b->h_stats) cudaFreeHost(b->h_stats);
  if (b->h_xyz_count) cudaFreeHost(b->h_xyz_count);
  if (b->h_n) cudaFreeHost(b->h_n);
  if (b->h_N) cudaFreeHost(b->h_N);
  cudaFree(b->ar.rec); cudaFree(b->ar.real_index); cudaFree(b->ar.count); cudaFree(b->ar.overflow); cudaFree(b->pts_dev);
  cudaFree(b->rs_pairs);
  if (b->h_over) cudaFreeHost(b->h_over);
  if (b->h_pts) cudaFreeHost(b->h_pts);
  for (auto& e : b->ev) if (e) cudaEventDestroy(e);
  if (b->own_stream) cudaStreamDestroy(b->own_stream);
  delete b;
  return EKF_OK;
}

// launch configuration of k_batch_update_cluster for B filters of C CTAs each
static cudaLaunchConfig_t cluster_config(int B, int C, cudaStream_t st, cudaLaunchAttribute* attr) {
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3((unsigned)(B * C), 1, 1);
  lc.blockDim = dim3(BUPD_THREADS, 1, 1);
  lc.dynamicSmemBytes = kUpdSmemBytes;
  lc.stream = st;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  lc.attrs = attr;
  lc.numAttrs = 1;
  return lc;
}

static int batch_create(const ekf_config* cfg, int n_filters, int feature_capacity, int device, bool large, ekf_batch** out) {
  if (cfg->kernel_size < 100000 || cfg->scale != 1 || cfg->forsePlane != 0) return EKF_ERR_UNSUPPORTED;
  if (cfg->window_size < 3 || cfg->window_size > 31 || cfg->search_clamp > 20 || cfg->search_clamp < 0) return EKF_ERR_UNSUPPORTED;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return EKF_ERR_CUDA;
  ekf_batch* b = new ekf_batch;
  b->cfg = *cfg; b->device = device; b->B = n_filters; b->Ncap = feature_capacity;
  b->ncap = EKF_CAM + 6 * feature_capacity;
  b->ld = (b->ncap + 7) & ~7;
  b->large = large;
  if (large) {
    b->cl_ctas = (b->ld + BSTRIP - 1) / BSTRIP;
    b->cstride = BNCAP_L;
  }
  const int w2 = (cfg->window_size * cfg->window_size + 15) & ~15;
  auto fail = [&](cudaError_t e, const char* what) {
    fprintf(stderr, "ekf_batch_create: %s: %s\n", what, cudaGetErrorString(e));
    ekf_batch_destroy(b);
    return EKF_ERR_CUDA;
  };
  cudaError_t e;
#define TRY(x) if ((e = (x)) != cudaSuccess) return fail(e, #x);
  TRY(cudaSetDevice(device))
  TRY(cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking))
  b->stream = b->own_stream;
  for (void* k : {(void*)k_batch_update<false, false, false>, (void*)k_batch_update<true, false, false>,
                  (void*)k_batch_update<false, true, false>, (void*)k_batch_update<true, true, false>,
                  (void*)k_batch_update<false, false, true>, (void*)k_batch_update<true, false, true>,
                  (void*)k_batch_update<false, true, true>, (void*)k_batch_update<true, true, true>})
    TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUpdSmemBytes))
  if (large) {
    void* const cl[8] = {(void*)k_batch_update_cluster<false, false, false>, (void*)k_batch_update_cluster<true, false, false>,
                         (void*)k_batch_update_cluster<false, true, false>, (void*)k_batch_update_cluster<true, true, false>,
                         (void*)k_batch_update_cluster<false, false, true>, (void*)k_batch_update_cluster<true, false, true>,
                         (void*)k_batch_update_cluster<false, true, true>, (void*)k_batch_update_cluster<true, true, true>};
    for (void* k : cl) TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUpdSmemBytes))
    cudaLaunchAttribute attr[1];
    for (int i = 0; i < 8; ++i) {   // forsePlane x intrinsics table x filter list
      const cudaLaunchConfig_t lc = cluster_config(1, b->cl_ctas, nullptr, attr);
      int ncl = 0;
      TRY(cudaOccupancyMaxActiveClusters(&ncl, cl[i], &lc))
      if (ncl < 1) {
        fprintf(stderr, "ekf_batch_create_large: the device cannot hold one cluster of %d CTAs with %zu bytes of shared memory each\n",
                b->cl_ctas, kUpdSmemBytes);
        ekf_batch_destroy(b);
        return EKF_ERR_UNSUPPORTED;
      }
      b->cl_resident = i ? std::min(b->cl_resident, ncl) : ncl;
    }
  }  const size_t Bn = (size_t)n_filters, cap = Bn * feature_capacity;
  BatchView& v = b->bv;
  v.ld = b->ld; v.Ncap = feature_capacity; v.tstride = w2;
  v.sstride = (long long)b->ncap * b->ld;
  TRY(balloc(&v.Sigma, Bn * v.sstride)) TRY(balloc(&b->scratch, Bn * v.sstride)) TRY(balloc(&v.mu, Bn * b->ld))
  TRY(balloc(&v.ctl, Bn)) TRY(balloc(&v.n, Bn)) TRY(balloc(&v.N, Bn))
  TRY(balloc(&b->match_defer, cap + 1))
  FeatTab& t = v.ft;
  TRY(balloc(&t.pos, cap)) TRY(balloc(&t.coding, cap)) TRY(balloc(&t.innov, cap)) TRY(balloc(&t.li, cap)) TRY(balloc(&t.hi, cap))
  TRY(balloc(&t.removef, cap)) TRY(balloc(&t.n_tot, cap)) TRY(balloc(&t.n_find, cap)) TRY(balloc(&t.real_index, cap))
  TRY(balloc(&t.pos_in_z, cap)) TRY(balloc(&t.sel, cap)) TRY(balloc(&t.center, 2 * cap)) TRY(balloc(&t.quality, cap))
  TRY(balloc(&t.last_ncc, cap)) TRY(balloc(&t.z, 2 * cap)) TRY(balloc(&t.h, 2 * cap)) TRY(balloc(&t.Hc, 26 * cap))
  TRY(balloc(&t.S2, 4 * cap)) TRY(balloc(&t.patch, cap * w2)) TRY(balloc(&t.mpatch, cap * w2))
  TRY(balloc(&v.xyz_flag, cap)) TRY(balloc(&v.xyz_J, 18 * cap)) TRY(balloc(&v.xyz_y, 3 * cap)) TRY(balloc(&v.xyz_count, Bn))
  TRY(balloc(&b->out_mu14, Bn * 14)) TRY(balloc(&b->out_S14, Bn * 196)) TRY(balloc(&b->out_stats, Bn * EKF_BATCH_STAT_FIELDS))
  TRY(balloc(&b->stage_mu14, Bn * 14)) TRY(balloc(&v.patchnumbre, Bn))
  TRY(balloc(&b->det_xy, Bn * 2 * b->cstride)) TRY(balloc(&b->det_n, Bn)) TRY(balloc(&b->det_num, Bn))
  TRY(cudaMallocHost((void**)&b->h_det_xy, sizeof(float) * Bn * 2 * EKF_BATCH_MAX_CORNERS))
  TRY(cudaMallocHost((void**)&b->h_det_n, sizeof(int) * Bn)) TRY(cudaMallocHost((void**)&b->h_num, sizeof(int) * Bn))
  TRY(cudaMallocHost((void**)&b->h_added, sizeof(int) * Bn))
  TRY(balloc(&b->blur_out, 2 * Bn)) TRY(cudaMallocHost((void**)&b->h_blur, sizeof(int) * 2 * Bn))
  TRY(cudaMallocHost((void**)&b->h_mu14, sizeof(double) * Bn * 14)) TRY(cudaMallocHost((void**)&b->h_S14, sizeof(double) * Bn * 196))
  TRY(cudaMallocHost((void**)&b->h_stats, sizeof(int) * Bn * EKF_BATCH_STAT_FIELDS))
  TRY(cudaMallocHost((void**)&b->h_n, sizeof(int) * Bn)) TRY(cudaMallocHost((void**)&b->h_N, sizeof(int) * Bn))
  TRY(cudaMallocHost((void**)&b->h_xyz_count, sizeof(int) * Bn))
  TRY(balloc(&b->det_slot, 2)) TRY(cudaMallocHost((void**)&b->h_det_slot, sizeof(int) * 2))
  TRY(cudaMemsetAsync(v.Sigma, 0, sizeof(double) * Bn * v.sstride, b->stream))
  TRY(cudaMemsetAsync(v.mu, 0, sizeof(double) * Bn * b->ld, b->stream))
  TRY(cudaMemsetAsync(v.ctl, 0, sizeof(DevCtl) * Bn, b->stream))
  TRY(cudaMemsetAsync(v.n, 0, sizeof(int) * Bn, b->stream)) TRY(cudaMemsetAsync(v.N, 0, sizeof(int) * Bn, b->stream))
  TRY(cudaMemsetAsync(v.xyz_count, 0, sizeof(int) * Bn, b->stream))
  for (auto& evn : b->ev) TRY(cudaEventCreate(&evn))
  TRY(cudaStreamSynchronize(b->stream))
#undef TRY
  for (size_t i = 0; i < Bn; ++i) { b->h_n[i] = 0; b->h_N[i] = 0; b->h_added[i] = 0; }
  b->cam_host.assign(Bn, 0);
  b->cam_dT.assign(1, 1.0); b->cam_ts.assign(1, -1.0);
  b->cam_frame.assign(1, 0);
  std::fill(b->h_blur, b->h_blur + 2 * Bn, 0);
  DevCfg& d = b->dcfg;
  d.cam = CamParams{cfg->fx, cfg->fy, cfg->u0, cfg->v0, cfg->k1, cfg->k2, cfg->k3, cfg->p1, cfg->p2};
  d.Vmax[0] = cfg->sigma_vx * cfg->sigma_vx; d.Vmax[1] = cfg->sigma_vy * cfg->sigma_vy; d.Vmax[2] = cfg->sigma_vz * cfg->sigma_vz;
  d.Vmax[3] = cfg->sigma_wx * cfg->sigma_wx; d.Vmax[4] = cfg->sigma_wy * cfg->sigma_wy; d.Vmax[5] = cfg->sigma_wz * cfg->sigma_wz;
  d.sigma_pixel_2 = (double)(cfg->sigma_pixel * cfg->sigma_pixel);
  d.th_low = cfg->li_threshold_factor * cfg->sigma_pixel;
  d.th_hi = cfg->hi_chi2_threshold;
  d.ransac_p = cfg->ransac_p;
  d.linearity_threshold = cfg->linearity_threshold;
  d.rho_0 = cfg->rho_0; d.sigma_rho_0 = cfg->sigma_rho_0;
  d.T_camera = cfg->T_camera; d.kernel_min_size = cfg->kernel_size;
  d.ncc_threshold = (float)cfg->ncc_threshold; d.search_clamp = (float)cfg->search_clamp;
  d.sigma_size_f = (float)cfg->sigma_size; d.quality_ratio = (float)cfg->quality_ratio;
  d.window = cfg->window_size; d.sigma_pixel = cfg->sigma_pixel; d.nhyp0 = cfg->ransac_nhyp0;
  d.forsePlane = cfg->forsePlane; d.abs_int_quirk = cfg->abs_int_quirk;
  d.tstride = w2;
  *out = b;
  return EKF_OK;
}

int ekf_batch_create(const ekf_config* cfg, int n_filters, int feature_capacity, int device, ekf_batch** out) {
  if (!cfg || !out || n_filters < 1 || feature_capacity < 1) return EKF_ERR_ARG;
  *out = nullptr;
  if (feature_capacity > BNCAP) return EKF_ERR_CAPACITY;
  return batch_create(cfg, n_filters, feature_capacity, device, false, out);
}

int ekf_batch_create_large(const ekf_config* cfg, int n_filters, int feature_capacity, int device, ekf_batch** out) {
  if (!cfg || !out || n_filters < 1 || feature_capacity < 1) return EKF_ERR_ARG;
  *out = nullptr;
  if (feature_capacity > BNCAP_L) return EKF_ERR_CAPACITY;
  return batch_create(cfg, n_filters, feature_capacity, device, feature_capacity > BNCAP, out);
}

int ekf_batch_update_clusters(const ekf_batch* b, int32_t* ctas_per_filter, int32_t* resident) {
  if (!b) return EKF_ERR_ARG;
  if (ctas_per_filter) *ctas_per_filter = b->cl_ctas;
  if (resident) *resident = b->cl_resident;
  return EKF_OK;
}

int ekf_batch_describe(const ekf_batch* b, ekf_batch_desc* out) {
  if (!b || !out) return EKF_ERR_ARG;
  *out = ekf_batch_desc{b->B, b->Ncap, b->ncap, b->ld, b->device, {0, 0, 0}};
  return EKF_OK;
}
int ekf_batch_set_stream(ekf_batch* b, void* s) {
  if (!b) return EKF_ERR_ARG;
  cudaSetDevice(b->device);
  cudaStreamSynchronize(b->stream);
  b->stream = s ? (cudaStream_t)s : b->own_stream;
  return EKF_OK;
}
int ekf_batch_sync(ekf_batch* b) {
  if (!b) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaStreamSynchronize(b->stream));
  return EKF_OK;
}

int ekf_batch_seed_from(ekf_batch* b, ekf_handle* src) {
  if (!b || !src) return EKF_ERR_ARG;
  if (src->device != b->device) return bfail(b, EKF_ERR_ARG, "seed filter lives on another device");
  if (src->N > b->Ncap || src->n > b->ncap) return bfail(b, EKF_ERR_CAPACITY, "seed filter holds more features than the batch capacity");
  if (src->cfg.window_size != b->cfg.window_size) return bfail(b, EKF_ERR_ARG, "window_size differs");
  const int nd = (int)src->deleted.size();
  if (b->ar.cap > 0 && nd > b->ar.cap)
    return bfail(b, EKF_ERR_CAPACITY, "seed filter's feature archive holds more records than the batch's archive capacity");
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaStreamSynchronize(src->stream));
  k_batch_seed<<<b->B, 256, 0, b->stream>>>(b->bv, src->Sigma, src->ld, src->mu, src->ft, src->n, src->N, src->patchnumbre);
  b->launches += 1;
  BCHECK(cudaGetLastError());
  if (b->ar.cap > 0) {   // deleted_patches travels with the filter: every filter starts from the source's archive
    std::vector<double> rec((size_t)std::max(nd, 1) * PTS_COLS);
    std::vector<int> ri((size_t)std::max(nd, 1));
    for (int i = 0; i < nd; ++i) {
      const DeletedPatch& dp = src->deleted[i];
      ri[i] = dp.real_index;
      for (int c = 0; c < 3; ++c) rec[(size_t)i * PTS_COLS + c] = dp.XYZ_pos[c];
      for (int c = 0; c < 9; ++c) rec[(size_t)i * PTS_COLS + 3 + c] = dp.cov_4_delete[c];
    }
    double* d_rec = nullptr;
    int* d_ri = nullptr;
    BCHECK(cudaMallocAsync((void**)&d_rec, sizeof(double) * rec.size(), b->stream));
    BCHECK(cudaMallocAsync((void**)&d_ri, sizeof(int) * ri.size(), b->stream));
    BCHECK(cudaMemcpyAsync(d_rec, rec.data(), sizeof(double) * rec.size(), cudaMemcpyHostToDevice, b->stream));
    BCHECK(cudaMemcpyAsync(d_ri, ri.data(), sizeof(int) * ri.size(), cudaMemcpyHostToDevice, b->stream));
    k_batch_seed_archive<<<b->B, 256, 0, b->stream>>>(b->ar, d_rec, d_ri, nd);
    b->launches += 1;
    BCHECK(cudaGetLastError());
    BCHECK(cudaFreeAsync(d_rec, b->stream));
    BCHECK(cudaFreeAsync(d_ri, b->stream));
  }
  BCHECK(cudaStreamSynchronize(b->stream));
  for (int i = 0; i < b->B; ++i) { b->h_n[i] = src->n; b->h_N[i] = src->N; }
  b->cam_dT.assign(b->n_cam, src->dT); b->cam_ts.assign(b->n_cam, src->old_ts);
  b->seeded = true;
  b->results_valid = false;
  b->rows_stale = true;
  return EKF_OK;
}

int ekf_batch_set_camera_states(ekf_batch* b, const double* mu14) {
  if (!b || !mu14) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaMemcpyAsync(b->stage_mu14, mu14, sizeof(double) * 14 * b->B, cudaMemcpyHostToDevice, b->stream));
  k_batch_set_cam<<<(b->B * 14 + 255) / 256, 256, 0, b->stream>>>(b->bv, b->stage_mu14, b->B);
  b->launches += 1;
  BCHECK(cudaGetLastError());
  BCHECK(cudaStreamSynchronize(b->stream));
  b->rows_stale = true;
  return EKF_OK;
}

// captureNewFrame (vslamRansac.cpp:226-245) for every camera, as the single filter's capture_common: time stamps, then with
// cfg.scale == 1 and gray frames one copy of the whole stack; otherwise a resize to (width / scale) x (height / scale) and
// BGR -> gray in k_capture_resize_gray with the camera in blockIdx.z, from device frames directly and from host frames through
// the staging buffer `raw`, a chunk of cameras at a time so that `raw` stays within kRawBudget (or one frame).  n frames
// (n == b->n_cam), frame c at img + c * height * stride; stamps[c] (stamps may be null: no stamps).
// list (n_list cameras, ekf_batch_capture_camera_frames*): frame k of the stack and stamps[k] are camera list[k]'s, and the
// frames go through k_capture_resize_gray at every scale, which writes frame k to slot list[k] of the existing stack.
static constexpr size_t kRawBudget = (size_t)256 << 20;
static int bcapture(ekf_batch* b, const uint8_t* img, int width, int height, int stride, int channels, const double* stamps, bool dev,
                    int n_list = 0, const int32_t* list = nullptr) {
  if (!b || !img || width < 8 || height < 8 || stride < width * channels) return EKF_ERR_ARG;
  const bool sub = list != nullptr;
  if (sub) {
    if (n_list < 1 || n_list > b->n_cam) return bfail(b, EKF_ERR_ARG, "n must lie in [1, n_cameras]");
    std::vector<char> seen(b->n_cam, 0);
    for (int k = 0; k < n_list; ++k) {
      const int c = list[k];
      if (c < 0 || c >= b->n_cam || seen[c])
        return bfail(b, EKF_ERR_ARG, "cameras[" + std::to_string(k) + "] = " + std::to_string(c) + " is not a camera, or listed twice");
      seen[c] = 1;
    }
  }
  const int scale = b->cfg.scale, n_all = b->n_cam, n = sub ? n_list : n_all;
  const int dw = width / scale, dh = height / scale;   // cv::Size(width / scale, height / scale), integer division
  if (dw < 8 || dh < 8) return bfail(b, EKF_ERR_ARG, "resized frame smaller than 8 x 8 pixels");
  // frame sizes per camera: camera c is the top-left size_in[c] of its slot, resized to size_in[c] / scale
  std::vector<int> fs;
  bool pads = false;
  if (!b->size_in.empty()) {
    fs.resize((size_t)4 * n_all);
    for (int c = 0; c < n_all; ++c) {
      const int wc = b->size_in[2 * c], hc = b->size_in[2 * c + 1];
      if (wc > width || hc > height)
        return bfail(b, EKF_ERR_ARG, "camera " + std::to_string(c) + " is larger than the captured " + std::to_string(width) + " x " +
                                         std::to_string(height) + " slot");
      if (wc / scale < 8 || hc / scale < 8)
        return bfail(b, EKF_ERR_ARG, "camera " + std::to_string(c) + ": resized frame smaller than 8 x 8 pixels");
      fs[4 * c] = wc; fs[4 * c + 1] = hc; fs[4 * c + 2] = wc / scale; fs[4 * c + 3] = hc / scale;
    }
    for (int k = 0; k < n; ++k) {
      const int c = sub ? list[k] : k;
      pads = pads || fs[4 * c + 2] < dw || fs[4 * c + 3] < dh;
    }
  }
  if (sub && std::find(b->cam_frame.begin(), b->cam_frame.end(), 1) != b->cam_frame.end()) {
    // other cameras hold frames in the stack: the slot and every camera's resized size stay as they are
    static const std::vector<int> none;
    if (dw != b->fv.w || dh != b->fv.h || fs != (b->fsize_on ? b->fsize_host : none))
      return bfail(b, EKF_ERR_ARG, "the resized slot " + std::to_string(dw) + " x " + std::to_string(dh) + " differs from the stack's " +
                                       std::to_string(b->fv.w) + " x " + std::to_string(b->fv.h) +
                                       " (or the frame sizes changed): only a capture of every camera may change it");
  }
  BCHECK(cudaSetDevice(b->device));
  for (int k = 0; stamps && k < n; ++k) {
    const int c = sub ? list[k] : k;
    if (stamps[k] >= 0) {
      if (b->cam_ts[c] > 0) b->cam_dT[c] = (stamps[k] - b->cam_ts[c]);
      b->cam_ts[c] = stamps[k];
    }
  }
  const int dstride = (dw + 15) & ~15;
  const size_t fstep = (size_t)dstride * dh, need = fstep * n_all;
  if (!fs.empty() && fs != b->fsize_host) {   // the table goes up when the sizes or the scale change, not per capture
    if (!b->fsize_dev) BCHECK(balloc(&b->fsize_dev, 4 * b->n_cam));
    b->fsize_host = fs;
    BCHECK(cudaMemcpyAsync(b->fsize_dev, b->fsize_host.data(), sizeof(int) * fs.size(), cudaMemcpyHostToDevice, b->stream));
  }
  b->fsize_on = !fs.empty();
  if (need > b->frame_cap) {
    BCHECK(cudaStreamSynchronize(b->stream));
    cudaFree(b->frame);
    b->frame = nullptr;
    b->frame_cap = 0;
    BCHECK(cudaMalloc((void**)&b->frame, need));
    b->frame_cap = need;
  }
  if (sub) {   // the slot of each listed frame, from a pageable copy: the driver has staged it when the call returns
    if (!b->slot_dev) BCHECK(balloc(&b->slot_dev, b->n_cam));
    const std::vector<int> slots(list, list + n);
    BCHECK(cudaMemcpyAsync(b->slot_dev, slots.data(), sizeof(int) * n, cudaMemcpyHostToDevice, b->stream));
  }
  if (scale == 1 && channels == 1 && !sub) {
    BCHECK(cudaMemcpy2DAsync(b->frame, dstride, img, stride, width, (size_t)height * n, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                             b->stream));
  } else {
    const size_t rawframe = (size_t)width * channels * height;
    const int chunk = dev ? 65535 : (int)std::max<size_t>(1, std::min<size_t>(n, kRawBudget / rawframe));   // 65535: gridDim.z
    if (!dev && rawframe * chunk > b->raw_cap) {
      BCHECK(cudaStreamSynchronize(b->stream));
      cudaFree(b->raw);
      b->raw = nullptr;
      b->raw_cap = 0;
      BCHECK(cudaMalloc((void**)&b->raw, rawframe * chunk));
      b->raw_cap = rawframe * chunk;
    }
    for (int c0 = 0; c0 < n; c0 += chunk) {
      const int k = std::min(chunk, n - c0);
      const uint8_t* src = img + (size_t)c0 * height * stride;
      int sstride = stride;
      if (!dev) {   // stream order keeps the next chunk's copy behind this chunk's resize
        BCHECK(cudaMemcpy2DAsync(b->raw, (size_t)width * channels, src, stride, (size_t)width * channels, (size_t)height * k,
                                 cudaMemcpyHostToDevice, b->stream));
        src = b->raw; sstride = width * channels;
      }
      if (sub)
        launch_capture_resize_gray(b->stream, src, width, height, sstride, channels, b->frame, dw, dh, dstride, &b->launches, k,
                                   b->fsize_on ? b->fsize_dev : nullptr, b->slot_dev + c0);
      else
        launch_capture_resize_gray(b->stream, src, width, height, sstride, channels, b->frame + (size_t)c0 * fstep, dw, dh, dstride,
                                   &b->launches, k, b->fsize_on ? b->fsize_dev + 4 * c0 : nullptr);
      BCHECK(cudaGetLastError());
    }
  }
  if (pads) {   // results must not depend on the bytes of a slot outside its camera's frame: zero them, one launch over the stack
    for (int c0 = 0; c0 < n; c0 += 65535) {
      const int k = std::min(65535, n - c0);
      const dim3 grid((dw + 255) / 256, dh, k);
      if (sub) k_batch_zero_pads<true><<<grid, 256, 0, b->stream>>>(b->frame, dw, dstride, dh, b->fsize_dev, b->slot_dev + c0);
      else k_batch_zero_pads<false><<<grid, 256, 0, b->stream>>>(b->frame + (size_t)c0 * fstep, dw, dstride, dh, b->fsize_dev + 4 * c0, nullptr);
      b->launches += 1;
    }
    BCHECK(cudaGetLastError());
  }
  if (b->fv.px != b->frame || b->fv.w != dw || b->fv.h != dh || b->fv.stride != dstride)
    match_make_tensor_map(&b->frame_map, b->frame, dw, dh, dstride, n_all, b->cfg.window_size, (int)b->cfg.search_clamp);
  b->fv = FrameView{b->frame, dw, dh, dstride};
  for (int k = 0; k < n; ++k) b->cam_frame[sub ? list[k] : k] = 1;
  return EKF_OK;
}
static int bcapture1(ekf_batch* b, const uint8_t* img, int width, int height, int stride, int channels, double stamp, bool dev) {
  if (b && b->n_cam > 1)
    return bfail(b, EKF_ERR_STATE, "the batch has " + std::to_string(b->n_cam) + " cameras: capture with ekf_batch_capture_frames" +
                                       (dev ? "_device" : channels == 3 ? "_bgr" : ""));
  return bcapture(b, img, width, height, stride, channels, &stamp, dev);
}
int ekf_batch_capture_frame(ekf_batch* b, const uint8_t* g, int w, int h, int s, double stamp) { return bcapture1(b, g, w, h, s, 1, stamp, false); }
int ekf_batch_capture_frame_device(ekf_batch* b, const uint8_t* g, int w, int h, int s, double stamp) { return bcapture1(b, g, w, h, s, 1, stamp, true); }
int ekf_batch_capture_frame_bgr(ekf_batch* b, const uint8_t* bgr, int w, int h, int s, double stamp) { return bcapture1(b, bgr, w, h, s, 3, stamp, false); }
int ekf_batch_capture_frames(ekf_batch* b, const uint8_t* g, int w, int h, int s, const double* stamps) {
  return bcapture(b, g, w, h, s, 1, stamps, false);
}
int ekf_batch_capture_frames_device(ekf_batch* b, const uint8_t* g, int w, int h, int s, const double* stamps) {
  return bcapture(b, g, w, h, s, 1, stamps, true);
}
int ekf_batch_capture_frames_bgr(ekf_batch* b, const uint8_t* bgr, int w, int h, int s, const double* stamps) {
  return bcapture(b, bgr, w, h, s, 3, stamps, false);
}
int ekf_batch_capture_camera_frames(ekf_batch* b, int n, const int32_t* cameras, const uint8_t* g, int w, int h, int s, const double* stamps) {
  if (b && !cameras) return bfail(b, EKF_ERR_ARG, "cameras is NULL");
  return bcapture(b, g, w, h, s, 1, stamps, false, n, cameras);
}
int ekf_batch_capture_camera_frames_device(ekf_batch* b, int n, const int32_t* cameras, const uint8_t* g, int w, int h, int s,
                                           const double* stamps) {
  if (b && !cameras) return bfail(b, EKF_ERR_ARG, "cameras is NULL");
  return bcapture(b, g, w, h, s, 1, stamps, true, n, cameras);
}
int ekf_batch_capture_camera_frames_bgr(ekf_batch* b, int n, const int32_t* cameras, const uint8_t* bgr, int w, int h, int s,
                                        const double* stamps) {
  if (b && !cameras) return bfail(b, EKF_ERR_ARG, "cameras is NULL");
  return bcapture(b, bgr, w, h, s, 3, stamps, false, n, cameras);
}

int ekf_batch_set_cameras(ekf_batch* b, int n_cameras, const int32_t* camera_of) {
  if (!b) return EKF_ERR_ARG;
  if (n_cameras < 1 || n_cameras > b->B) return bfail(b, EKF_ERR_ARG, "n_cameras must lie in [1, n_filters]");
  if (!camera_of && n_cameras != b->B) return bfail(b, EKF_ERR_ARG, "camera_of = NULL (identity) needs n_cameras == n_filters");
  std::vector<int> cam(b->B);
  for (int f = 0; f < b->B; ++f) {
    cam[f] = camera_of ? camera_of[f] : f;
    if (cam[f] < 0 || cam[f] >= n_cameras)
      return bfail(b, EKF_ERR_ARG, "camera_of[" + std::to_string(f) + "] = " + std::to_string(cam[f]) + " is not a camera");
  }
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaStreamSynchronize(b->stream));
  cudaFree(b->cam_dev); cudaFree(b->det_slot); cudaFreeHost(b->h_det_slot); cudaFree(b->fsize_dev); cudaFree(b->slot_dev);
  b->cam_dev = nullptr; b->det_slot = nullptr; b->h_det_slot = nullptr; b->fsize_dev = nullptr; b->slot_dev = nullptr;
  b->fsize_host.clear();
  if (n_cameras > 1) {
    BCHECK(balloc(&b->cam_dev, b->B));
    BCHECK(cudaMemcpy(b->cam_dev, cam.data(), sizeof(int) * b->B, cudaMemcpyHostToDevice));
  }
  BCHECK(balloc(&b->det_slot, 2 * n_cameras));
  BCHECK(cudaMallocHost((void**)&b->h_det_slot, sizeof(int) * 2 * n_cameras));
  b->size_in.clear();   // sizes are per camera: back to the whole slot
  b->fsize_on = false;
  b->cam_host = cam;
  b->n_cam = n_cameras;
  const double dT = b->cam_dT[0], ts = b->cam_ts[0];
  b->cam_dT.assign(n_cameras, dT); b->cam_ts.assign(n_cameras, ts);
  b->cam_frame.assign(n_cameras, 0);
  b->fv = FrameView{nullptr, 0, 0, 0};   // the next capture encodes the stack's tensor map
  return EKF_OK;
}

static_assert(sizeof(CamParams) == 9 * sizeof(double), "a row of ekf_batch_set_intrinsics is one CamParams");
int ekf_batch_set_intrinsics(ekf_batch* b, const double* cam) {
  if (!b) return EKF_ERR_ARG;
  if (cam) {
    for (int f = 0; f < b->B; ++f) {
      const double* r = cam + 9 * (size_t)f;
      bool ok = r[0] > 0 && r[1] > 0;
      for (int c = 0; c < 9; ++c) ok = ok && std::isfinite(r[c]);
      if (!ok) return bfail(b, EKF_ERR_ARG, "intrinsics of filter " + std::to_string(f) + ": non-finite, or fx / fy <= 0");
    }
  }
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaStreamSynchronize(b->stream));   // work in flight may still read the table
  if (!cam) {
    cudaFree(b->intr_dev);
    b->intr_dev = nullptr;
    b->bv.cam = nullptr;
    return EKF_OK;
  }
  if (!b->intr_dev) BCHECK(balloc(&b->intr_dev, b->B));
  BCHECK(cudaMemcpyAsync(b->intr_dev, cam, sizeof(CamParams) * b->B, cudaMemcpyHostToDevice, b->stream));
  BCHECK(cudaStreamSynchronize(b->stream));   // the caller's array is free once the call returns
  b->bv.cam = b->intr_dev;
  return EKF_OK;
}

int ekf_batch_set_frame_sizes(ekf_batch* b, const int32_t* wh) {
  if (!b) return EKF_ERR_ARG;
  if (wh) {
    for (int c = 0; c < b->n_cam; ++c)
      if (wh[2 * c] < 1 || wh[2 * c + 1] < 1) return bfail(b, EKF_ERR_ARG, "frame size of camera " + std::to_string(c) + " is not positive");
    b->size_in.assign(wh, wh + 2 * (size_t)b->n_cam);
  } else {
    b->size_in.clear();
  }
  b->fsize_on = false;
  std::fill(b->cam_frame.begin(), b->cam_frame.end(), 0);   // the sizes hold from the next capture on
  return EKF_OK;
}

int ekf_batch_set_detect_budget(ekf_batch* b, int64_t bytes) {
  if (!b || bytes < 1) return EKF_ERR_ARG;
  b->det_budget = (size_t)bytes;
  return EKF_OK;
}

int ekf_batch_get_camera_frame(ekf_batch* b, int camera, uint8_t* out, int* width, int* height) {   // returnGrayImg (vslamRansac.cpp:1364)
  if (!b || !width || !height || camera < 0 || camera >= b->n_cam) return EKF_ERR_ARG;
  if (!b->cam_frame[camera]) return bfail(b, EKF_ERR_STATE, "no frame captured for camera " + std::to_string(camera));
  const int w = b->fsize_on ? b->fsize_host[4 * camera + 2] : b->fv.w, h = b->fsize_on ? b->fsize_host[4 * camera + 3] : b->fv.h;
  *width = w; *height = h;
  if (out) {
    BCHECK(cudaSetDevice(b->device));
    BCHECK(cudaMemcpy2DAsync(out, w, b->frame + (size_t)camera * b->fv.h * b->fv.stride, b->fv.stride, w, h,
                             cudaMemcpyDeviceToHost, b->stream));
    BCHECK(cudaStreamSynchronize(b->stream));
  }
  return EKF_OK;
}
int ekf_batch_get_frame(ekf_batch* b, uint8_t* out, int* width, int* height) {
  if (b && b->n_cam > 1)
    return bfail(b, EKF_ERR_STATE, "the batch has " + std::to_string(b->n_cam) + " cameras: read frames with ekf_batch_get_camera_frame");
  return ekf_batch_get_camera_frame(b, 0, out, width, height);
}

int ekf_batch_get_dt(ekf_batch* b, double* out) {   // getDt for every filter
  if (!b || !out) return EKF_ERR_ARG;
  for (int f = 0; f < b->B; ++f) out[f] = b->cam_dT[b->cam_host[f]];
  return EKF_OK;
}

int ekf_batch_set_scale(ekf_batch* b, int32_t scale) {
  if (!b || scale < 1 || scale > 64) return EKF_ERR_ARG;   // the range ekf_create accepts
  b->cfg.scale = scale;
  return EKF_OK;
}

int ekf_batch_set_force_plane(ekf_batch* b, int on) {
  if (!b) return EKF_ERR_ARG;
  b->cfg.forsePlane = on != 0;
  b->dcfg.forsePlane = on != 0;
  return EKF_OK;
}

// The filters a step works on: n_act of them listed at act (device) by ekf_batch_step_filters, or every filter (act null).
struct StepList {
  const int* act = nullptr;
  int n_act = 0;
};
static unsigned step_grid(const ekf_batch* b, const StepList& sl) { return (unsigned)(sl.act ? sl.n_act : b->B); }

// k_batch_compact at the batch's capacity on the step's filters; one >= 0: removeFeature(one_idx) on filter `one` alone (one CTA)
static void launch_compact(ekf_batch* b, int remove, const int* hold_stats, int one = -1, int one_idx = -1, const StepList& sl = {}) {
  const unsigned grid = one >= 0 ? 1u : step_grid(b, sl);
  auto* const compact = b->large ? (sl.act ? k_batch_compact<BNCAP_L, true> : k_batch_compact<BNCAP_L, false>)
                                 : (sl.act ? k_batch_compact<BNCAP, true> : k_batch_compact<BNCAP, false>);
  compact<<<grid, BCMP_THREADS, 0, b->stream>>>(b->bv, b->scratch, b->cfg.min_features, b->cfg.max_features, remove, hold_stats, b->ar,
                                                one, one_idx, sl.act);
  b->launches += 1;
}

// With the archive on: enqueue the overflow counters' read-back beside a read-back of n / N, and after its synchronisation name
// the first filter whose archive dropped records since the last check (EKF_ERR_CAPACITY).
static int archive_readback(ekf_batch* b) {
  if (b->ar.cap > 0)
    BCHECK(cudaMemcpyAsync(b->h_over, b->ar.overflow, sizeof(int) * b->B, cudaMemcpyDeviceToHost, b->stream));
  return EKF_OK;
}
static int archive_check(ekf_batch* b) {
  if (b->ar.cap <= 0) return EKF_OK;
  int first = -1;
  for (int i = 0; i < b->B; ++i) {
    if (b->h_over[i] != b->over_seen[i] && first < 0) first = i;
    b->over_seen[i] = b->h_over[i];
  }
  if (first < 0) return EKF_OK;
  return bfail(b, EKF_ERR_CAPACITY, "filter " + std::to_string(first) + ": feature archive full (capacity " + std::to_string(b->ar.cap) +
                                        "), removed features were not archived");
}

// The batched detector for every filter, filter b asking for num[b * num_stride] corners (<= 0: none; hnum is the same on the
// host).  One camera: the one-frame detector.  Several: the cameras at least one filter asks from, in chunks whose scratch
// (kDetBytesPerPixel a camera) fits det_budget, and whose keys the sorts can still index with an int.  Enqueued only.
// Device bytes a pixel of one camera in a chunk: the eig map (4), pixel and candidate keys before and after sorting (32), and the
// segmented sort's alternate key buffer in its workspace (8).
static constexpr size_t kDetBytesPerPixel = 44;
static int batch_detect(ekf_batch* b, const int* num, const int* hnum, int num_stride, int cap_mode) {
  cudaStream_t st = b->stream;
  const size_t npx = (size_t)b->fv.w * b->fv.h;
  if (b->n_cam == 1 && !b->fsize_on) {
    BCHECK(batch_detect_reserve(b->det, npx, b->B, b->cstride));
    BCHECK(launch_batch_detect(st, b->det, b->fv, b->bv.ft.center, b->bv.N, b->Ncap, b->B, b->cfg.window_size, num, num_stride, cap_mode,
                               b->cstride, b->det_xy, b->det_n, &b->launches));
    return EKF_OK;
  }
  std::vector<int> cams;
  std::fill(b->h_det_slot, b->h_det_slot + b->n_cam, -1);
  for (int f = 0; f < b->B; ++f) {
    const int c = b->cam_host[f];
    if (hnum[(size_t)f * num_stride] > 0 && b->h_det_slot[c] < 0) { b->h_det_slot[c] = (int)cams.size(); cams.push_back(c); }
  }
  const int n_req = (int)cams.size();
  const size_t fit = std::min<size_t>(b->det_budget / (kDetBytesPerPixel * npx), (size_t)INT_MAX / npx);
  const int chunk = (int)std::max<size_t>(1, std::min<size_t>(std::max(n_req, 1), fit));
  std::copy(cams.begin(), cams.end(), b->h_det_slot + b->n_cam);
  BCHECK(cudaMemcpyAsync(b->det_slot, b->h_det_slot, sizeof(int) * (b->n_cam + n_req), cudaMemcpyHostToDevice, st));
  if (n_req > 0) BCHECK(batch_detect_reserve_cams(b->det, npx, chunk, b->B, b->cstride));
  else BCHECK(batch_detect_reserve(b->det, 0, b->B, b->cstride));   // the per-filter buffers only
  BCHECK(launch_batch_detect_cams(st, b->det, b->fv, cams.data(), n_req, chunk, b->cam_dev, b->det_slot, b->bv.ft.center, b->bv.N, b->Ncap,
                                  b->B, b->cfg.window_size, num, num_stride, cap_mode, b->cstride, b->det_xy, b->det_n, &b->launches,
                                  b->fsize_on ? b->fsize_dev : nullptr, b->fsize_on ? b->fsize_host.data() : nullptr,
                                  b->det_slot + b->n_cam));
  return EKF_OK;
}

// k_batch_add at the batch's capacity and intrinsics, with or without a list of filters
static void (*add_kernel(const ekf_batch* b, bool act))(BatchView, FrameView, DevCfg, const float*, const int*, int, float, float, int,
                                                        const int*, const int*) {
  const bool intr = b->bv.cam != nullptr;
  if (b->large) return act ? (intr ? k_batch_add<true, true, true> : k_batch_add<true, false, true>)
                           : (intr ? k_batch_add<true, true, false> : k_batch_add<true, false, false>);
  return act ? (intr ? k_batch_add<false, true, true> : k_batch_add<false, false, true>)
             : (intr ? k_batch_add<false, true, false> : k_batch_add<false, false, false>);
}

// detection + adds for every filter, as batch_detect; decide: also take the new features' XYZ decisions (in-step top-up).
// The detector runs on every filter (one that asks for nothing costs next to nothing), the adds on the step's filters.
// Enqueued only.
static int batch_topup(ekf_batch* b, const int* num, const int* hnum, int num_stride, int decide, const StepList& sl = {}) {
  cudaStream_t st = b->stream;
  const int rc = batch_detect(b, num, hnum, num_stride, 1);
  if (rc) return rc;
  add_kernel(b, sl.act)<<<step_grid(b, sl), BADD_THREADS, 0, st>>>(b->bv, b->fv, b->dcfg, b->det_xy, b->det_n, -1, 0.0f, 0.0f, decide,
                                                                   b->cam_dev, sl.act);
  b->launches += 1;
  BCHECK(cudaGetLastError());
  return EKF_OK;
}
// n / N mirrors (and the per-filter add counts) back to the host: the one synchronisation of a top-up
static int batch_readback(ekf_batch* b, bool added) {
  cudaStream_t st = b->stream;
  const size_t Bn = (size_t)b->B;
  BCHECK(cudaMemcpyAsync(b->h_n, b->bv.n, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(b->h_N, b->bv.N, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  if (added) BCHECK(cudaMemcpyAsync(b->h_added, b->det_n, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  const int rc = archive_readback(b);
  if (rc) return rc;
  BCHECK(cudaStreamSynchronize(st));
  return EKF_OK;
}

// EKF_ERR_STATE unless filter f's camera holds a frame
static int need_frame(ekf_batch* b, int f, const char* what) {
  const int c = b->cam_host[f];
  if (b->cam_frame[c]) return EKF_OK;
  return bfail(b, EKF_ERR_STATE, std::string(what) + " before captureNewFrame: camera " + std::to_string(c) + " of filter " +
                                     std::to_string(f) + " holds no frame");
}

// ekf_batch_step (per_filter false: dv / dw / vcontrol for every filter), ekf_batch_step_controls (per_filter: dv / dw
// n_filters x 3, vcontrol n_filters; null = zeros) and ekf_batch_step_filters (filters: the n_act listed filters, strictly
// ascending, with per_filter controls in list order).  With one camera, shared controls and no list the picks go up alone;
// otherwise the cameras' dT, the filters' controls, the list and the picks are staged together and go up in one copy (BatchStepIn).
// With a list every per-filter kernel runs on the listed filters only; the counters of the others are zeroed on the device and
// their camera rows gathered when they may be stale, so that ekf_batch_get_camera_states reports every filter as it stands.
static int batch_step(ekf_batch* b, const double* dv, const double* dw, int vcontrol, const int32_t* vcontrols, bool per_filter,
                      const uint32_t* picks, int n_picks, const int32_t* filters = nullptr, int n_act = 0) {
  if (!b || n_picks < 0 || (n_picks > 0 && !picks)) return EKF_ERR_ARG;
  if (filters) {
    if (n_act < 1 || n_act > b->B) return bfail(b, EKF_ERR_ARG, "n must lie in [1, n_filters]");
    for (int i = 0; i < n_act; ++i)
      if (filters[i] < 0 || filters[i] >= b->B || (i > 0 && filters[i] <= filters[i - 1]))
        return bfail(b, EKF_ERR_ARG, "filters must be strictly ascending in [0, n_filters): filters[" + std::to_string(i) + "] = " +
                                         std::to_string(filters[i]));
  }
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "batch step before ekf_batch_seed_from");
  const int n_rows = filters ? n_act : b->B;   // filters the step works on
  const bool every_frame = std::find(b->cam_frame.begin(), b->cam_frame.end(), 0) == b->cam_frame.end();
  for (int i = 0; !every_frame && i < n_rows; ++i) {
    const int rc = need_frame(b, filters ? filters[i] : i, "batch step");
    if (rc) return rc;
  }
  BCHECK(cudaSetDevice(b->device));
  cudaStream_t st = b->stream;
  const size_t Bn = (size_t)b->B;
  BatchStepIn in{b->cam_dev, nullptr, nullptr, nullptr, b->fsize_on ? b->fsize_dev : nullptr, nullptr};
  StepList sl;
  const uint32_t* picks_dev = b->picks_dev;
  const double z3[3] = {0, 0, 0};
  const double* a = (dv && !per_filter) ? dv : z3; const double* w = (dw && !per_filter) ? dw : z3;
  if (b->n_cam == 1 && !per_filter && !filters) {
    if (n_picks > b->picks_cap) {
      BCHECK(cudaStreamSynchronize(st));
      cudaFree(b->picks_dev);
      b->picks_dev = nullptr;
      BCHECK(cudaMalloc((void**)&b->picks_dev, sizeof(uint32_t) * n_picks));
      b->picks_cap = n_picks;
    }
    if (n_picks > 0) BCHECK(cudaMemcpyAsync(b->picks_dev, picks, sizeof(uint32_t) * n_picks, cudaMemcpyHostToDevice, st));
    picks_dev = b->picks_dev;
  } else {
    // [dT: n_cam doubles, n_cam > 1][ctl: rows x 6 doubles, vcontrol: rows int32, per_filter][act: n_act int32, a list][picks]
    const size_t rows = (size_t)n_rows;
    const size_t n_dT = b->n_cam > 1 ? (size_t)b->n_cam : 0, n_ctl = per_filter ? 6 * rows : 0, n_vc = per_filter ? rows : 0;
    const size_t n_al = filters ? rows : 0;
    const size_t bytes = sizeof(double) * (n_dT + n_ctl) + sizeof(int) * (n_vc + n_al) + sizeof(uint32_t) * (size_t)n_picks;
    if (bytes > b->step_cap) {
      BCHECK(cudaStreamSynchronize(st));
      cudaFree(b->step_dev); cudaFreeHost(b->step_host);
      b->step_dev = nullptr; b->step_host = nullptr; b->step_cap = 0;
      BCHECK(cudaMalloc(&b->step_dev, bytes));
      BCHECK(cudaMallocHost(&b->step_host, bytes));
      b->step_cap = bytes;
    }
    double* hd = static_cast<double*>(b->step_host);
    std::copy(b->cam_dT.begin(), b->cam_dT.begin() + n_dT, hd);
    for (size_t f = 0; f < n_ctl / 6; ++f)
      for (int c = 0; c < 3; ++c) {
        hd[n_dT + 6 * f + c] = dv ? dv[3 * f + c] : 0.0;
        hd[n_dT + 6 * f + 3 + c] = dw ? dw[3 * f + c] : 0.0;
      }
    int* hi = reinterpret_cast<int*>(hd + n_dT + n_ctl);
    for (size_t f = 0; f < n_vc; ++f) hi[f] = vcontrols ? (vcontrols[f] != 0) : 0;
    if (n_al) std::copy(filters, filters + n_al, hi + n_vc);
    uint32_t* hp = reinterpret_cast<uint32_t*>(hi + n_vc + n_al);
    if (n_picks > 0) std::copy(picks, picks + n_picks, hp);
    BCHECK(cudaMemcpyAsync(b->step_dev, b->step_host, bytes, cudaMemcpyHostToDevice, st));
    const double* dd = static_cast<const double*>(b->step_dev);
    const int* di = reinterpret_cast<const int*>(dd + n_dT + n_ctl);
    if (n_dT) in.dT = dd;
    if (per_filter) { in.ctl = dd + n_dT; in.vcontrol = di; }
    if (filters) { in.act = di + n_vc; sl.act = in.act; sl.n_act = n_act; }
    picks_dev = reinterpret_cast<const uint32_t*>(di + n_vc + n_al);
  }
  const bool act = sl.act != nullptr, intr = b->bv.cam != nullptr;
  const unsigned grid = step_grid(b, sl);
  if (act) {   // the others' counters read zero; their camera rows are gathered once a call changed some filter's
    BCHECK(cudaMemsetAsync(b->out_stats, 0, sizeof(int) * Bn * EKF_BATCH_STAT_FIELDS, st));
    if (b->rows_stale) {
      k_batch_camera_rows<<<(unsigned)((Bn * 210 + 255) / 256), 256, 0, st>>>(b->bv, b->out_mu14, b->out_S14, b->B);
      b->launches += 1;
    }
  }
  BCHECK(cudaEventRecord(b->ev[0], st));
  auto* const predict = act ? (intr ? k_batch_predict<true, true> : k_batch_predict<false, true>)
                            : (intr ? k_batch_predict<true, false> : k_batch_predict<false, false>);
  predict<<<grid, BPRED_THREADS, 0, st>>>(b->bv, b->fv, b->dcfg, b->cam_dT[0], make_double3(a[0], a[1], a[2]),
                                          make_double3(w[0], w[1], w[2]), vcontrol, in);
  b->launches += 1;
  if (b->blur) {   // matching_patch <- blurred patch where the prediction moves far enough (k_batch_predict copied patch)
    void (*blur)(BatchView, DevCfg, double, int*, BatchStepIn);
    if (b->large) blur = act ? (intr ? k_batch_predict_blur<BNCAP_L, true, true> : k_batch_predict_blur<BNCAP_L, false, true>)
                             : (intr ? k_batch_predict_blur<BNCAP_L, true, false> : k_batch_predict_blur<BNCAP_L, false, false>);
    else blur = act ? (intr ? k_batch_predict_blur<BNCAP, true, true> : k_batch_predict_blur<BNCAP, false, true>)
                    : (intr ? k_batch_predict_blur<BNCAP, true, false> : k_batch_predict_blur<BNCAP, false, false>);
    blur<<<grid, BBLUR_WARPS * 32, 0, st>>>(b->bv, b->dcfg, b->cam_dT[0], b->blur_out, in);
    b->launches += 1;
  }
  BCHECK(cudaEventRecord(b->ev[1], st));
  launch_match_filter_batch(st, b->bv.ft, b->Ncap, b->bv.N, (int)grid, b->fv, b->dcfg, &b->frame_map, b->match_defer,
                            b->match_defer + (size_t)b->B * b->Ncap, &b->launches, b->cam_dev, b->fsize_on ? b->fsize_dev : nullptr, sl.act);
  BCHECK(cudaEventRecord(b->ev[2], st));
  const bool plane = b->cfg.forsePlane != 0;
  if (b->large) {   // one cluster of cl_ctas CTAs per filter
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t lc = cluster_config((int)grid, b->cl_ctas, st, attr);
    void (*update)(BatchView, DevCfg, const uint32_t*, int, double*, double*, int*, int, int, int, const int*);
    if (act) update = plane ? (intr ? k_batch_update_cluster<true, true, true> : k_batch_update_cluster<true, false, true>)
                            : (intr ? k_batch_update_cluster<false, true, true> : k_batch_update_cluster<false, false, true>);
    else update = plane ? (intr ? k_batch_update_cluster<true, true, false> : k_batch_update_cluster<true, false, false>)
                        : (intr ? k_batch_update_cluster<false, true, false> : k_batch_update_cluster<false, false, false>);
    BCHECK(cudaLaunchKernelEx(&lc, update, b->bv, b->dcfg, picks_dev, n_picks, b->out_mu14, b->out_S14,
                              b->out_stats, (int)b->cfg.min_features, (int)b->cfg.max_features, (int)b->cfg.xyz_conversion, sl.act));
  } else {
    void (*update)(BatchView, DevCfg, const uint32_t*, int, double*, double*, int*, int, int, int, const int*);
    if (act) update = plane ? (intr ? k_batch_update<true, true, true> : k_batch_update<true, false, true>)
                            : (intr ? k_batch_update<false, true, true> : k_batch_update<false, false, true>);
    else update = plane ? (intr ? k_batch_update<true, true, false> : k_batch_update<true, false, false>)
                        : (intr ? k_batch_update<false, true, false> : k_batch_update<false, false, false>);
    update<<<grid, BUPD_THREADS, kUpdSmemBytes, st>>>(b->bv, b->dcfg, picks_dev, n_picks, b->out_mu14, b->out_S14,
                                                      b->out_stats, b->cfg.min_features, b->cfg.max_features,
                                                      b->cfg.xyz_conversion, sl.act);
  }
  b->launches += 1;
  BCHECK(cudaEventRecord(b->ev[3], st));
  BCHECK(cudaGetLastError());
  BCHECK(cudaMemcpyAsync(b->h_stats, b->out_stats, sizeof(int) * Bn * EKF_BATCH_STAT_FIELDS, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(b->h_mu14, b->out_mu14, sizeof(double) * Bn * 14, cudaMemcpyDeviceToHost, st));
  if (b->cfg.xyz_conversion) BCHECK(cudaMemcpyAsync(b->h_xyz_count, b->bv.xyz_count, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  if (b->blur) BCHECK(cudaMemcpyAsync(b->h_blur, b->blur_out, sizeof(int) * 2 * grid, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  b->results_valid = true;
  b->rows_stale = false;
  if (b->blur && act) {   // the kernel wrote list positions: scatter them to filters, zeros for the others
    const std::vector<int> got(b->h_blur, b->h_blur + 2 * (size_t)n_act);
    std::fill(b->h_blur, b->h_blur + 2 * Bn, 0);
    for (int i = 0; i < n_act; ++i) { b->h_blur[filters[i]] = got[i]; b->h_blur[Bn + filters[i]] = got[n_act + i]; }
  }
  long long removed = 0, converted = 0, fails = 0, topups = 0;
  for (int k = 0; k < n_rows; ++k) {   // the step's filters: the others have zero counters and nothing pending
    const size_t i = filters ? (size_t)filters[k] : (size_t)k;
    removed += b->h_stats[i * EKF_BATCH_STAT_FIELDS + EKF_BSTAT_REMOVED];
    fails += b->h_stats[i * EKF_BATCH_STAT_FIELDS + EKF_BSTAT_CHOL_FAIL];
    topups += b->h_stats[i * EKF_BATCH_STAT_FIELDS + EKF_BSTAT_TOPUP] > 0;
    if (b->cfg.xyz_conversion) converted += b->h_xyz_count[i];
  }
  std::fill(b->h_added, b->h_added + Bn, 0);
  if (!b->topup || topups == 0) {
    if (removed > 0 || converted > 0) {   // removals, then convert2XYZ_ifLinearAll (V:1312-1317), in one pass
      launch_compact(b, 1, nullptr, -1, -1, sl);
      BCHECK(cudaGetLastError());
      const int rc = batch_readback(b, false);
      if (rc) return rc;
    }
  } else {
    // The reference order (V:1312-1317): removals, findNewFeatures, convert2XYZ_ifLinearAll.  A filter that tops up must
    // convert after its adds: the new feature's cross-covariance with a converted feature f is J (A Sigma[cam, f]) there,
    // and converting first would give A (J Sigma[cam, f]), equal only up to rounding.  So its compaction removes only;
    // every other filter keeps the fused pass.
    if (removed > 0 || converted > 0) {
      launch_compact(b, 1, b->out_stats, -1, -1, sl);
    }
    int rc = batch_topup(b, b->out_stats + EKF_BSTAT_TOPUP, b->h_stats + EKF_BSTAT_TOPUP, EKF_BATCH_STAT_FIELDS, b->cfg.xyz_conversion, sl);
    if (rc) return rc;
    if (b->cfg.xyz_conversion) {   // the held conversions and the new features' (filters with none return at once)
      launch_compact(b, 0, nullptr, -1, -1, sl);
    }
    BCHECK(cudaGetLastError());
    rc = batch_readback(b, true);
    if (rc) return rc;
  }
  if (fails > 0) return bfail(b, EKF_ERR_STATE, "innovation covariance not positive definite in at least one filter");
  for (size_t i = 0; b->blur && i < Bn; ++i)
    if (b->h_blur[Bn + i])
      return bfail(b, EKF_ERR_UNSUPPORTED, "filter " + std::to_string(i) + ": a motion-blur kernel exceeded 256 x 256 pixels");
  return archive_check(b);
}
int ekf_batch_step(ekf_batch* b, const double dv[3], const double dw[3], int vcontrol, const uint32_t* picks, int n_picks) {
  return batch_step(b, dv, dw, vcontrol, nullptr, false, picks, n_picks);
}
int ekf_batch_step_controls(ekf_batch* b, const double* dv, const double* dw, const int32_t* vcontrol, const uint32_t* picks, int n_picks) {
  return batch_step(b, dv, dw, 0, vcontrol, true, picks, n_picks);
}
int ekf_batch_step_filters(ekf_batch* b, int n, const int32_t* filters, const double* dv, const double* dw, const int32_t* vcontrol,
                           const uint32_t* picks, int n_picks) {
  if (b && !filters) return bfail(b, EKF_ERR_ARG, "filters is NULL");
  return batch_step(b, dv, dw, 0, vcontrol, true, picks, n_picks, filters, n);
}

int ekf_batch_convert2xyz_if_linear_all(ekf_batch* b) {
  if (!b) return EKF_ERR_ARG;
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "convert2XYZ_ifLinearAll before ekf_batch_seed_from");
  BCHECK(cudaSetDevice(b->device));
  cudaStream_t st = b->stream;
  const size_t Bn = (size_t)b->B;
  if (b->large) k_batch_xyz_decide_large<<<b->B, BNCAP_L, 0, st>>>(b->bv, b->dcfg);
  else k_batch_xyz_decide<<<b->B, BNCAP, 0, st>>>(b->bv, b->dcfg);
  b->launches += 1;
  BCHECK(cudaGetLastError());
  BCHECK(cudaMemcpyAsync(b->h_xyz_count, b->bv.xyz_count, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  long long converted = 0;
  for (size_t i = 0; i < Bn; ++i) converted += b->h_xyz_count[i];
  if (converted == 0) return EKF_OK;
  launch_compact(b, 0, nullptr);
  BCHECK(cudaGetLastError());
  BCHECK(cudaMemcpyAsync(b->h_n, b->bv.n, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(b->h_N, b->bv.N, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  return EKF_OK;
}

int ekf_batch_get_camera_states(ekf_batch* b, double* mu14, double* sigma14, int32_t* stats) {
  if (!b) return EKF_ERR_ARG;
  if (!b->results_valid) return bfail(b, EKF_ERR_STATE, "no completed step");
  BCHECK(cudaSetDevice(b->device));
  const size_t Bn = (size_t)b->B;
  if (sigma14) {
    BCHECK(cudaMemcpyAsync(b->h_S14, b->out_S14, sizeof(double) * Bn * 196, cudaMemcpyDeviceToHost, b->stream));
    BCHECK(cudaStreamSynchronize(b->stream));
    std::copy(b->h_S14, b->h_S14 + Bn * 196, sigma14);
  }
  if (mu14) std::copy(b->h_mu14, b->h_mu14 + Bn * 14, mu14);
  if (stats) std::copy(b->h_stats, b->h_stats + Bn * EKF_BATCH_STAT_FIELDS, stats);
  return EKF_OK;
}

int ekf_batch_num_features(ekf_batch* b, int f) { return (!b || f < 0 || f >= b->B) ? EKF_ERR_ARG : b->h_N[f]; }
int ekf_batch_state_dim(ekf_batch* b, int f) { return (!b || f < 0 || f >= b->B) ? EKF_ERR_ARG : b->h_n[f]; }

int ekf_batch_get_full(ekf_batch* b, int f, double* mu, double* sigma, int ld) {
  if (!b || f < 0 || f >= b->B || !mu) return EKF_ERR_ARG;
  const int n = b->h_n[f];
  if (sigma && ld < n) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaMemcpyAsync(mu, b->bv.mu + (size_t)f * b->ld, sizeof(double) * n, cudaMemcpyDeviceToHost, b->stream));
  if (sigma)
    BCHECK(cudaMemcpy2DAsync(sigma, sizeof(double) * ld, b->bv.Sigma + (size_t)f * b->bv.sstride, sizeof(double) * b->ld,
                             sizeof(double) * n, n, cudaMemcpyDeviceToHost, b->stream));
  BCHECK(cudaStreamSynchronize(b->stream));
  return EKF_OK;
}
int ekf_batch_set_full(ekf_batch* b, int f, const double* mu, const double* sigma, int ld) {
  if (!b || f < 0 || f >= b->B || !mu || !sigma) return EKF_ERR_ARG;
  const int n = b->h_n[f];
  if (ld < n) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaMemcpyAsync(b->bv.mu + (size_t)f * b->ld, mu, sizeof(double) * n, cudaMemcpyHostToDevice, b->stream));
  BCHECK(cudaMemcpy2DAsync(b->bv.Sigma + (size_t)f * b->bv.sstride, sizeof(double) * b->ld, sigma, sizeof(double) * ld,
                           sizeof(double) * n, n, cudaMemcpyHostToDevice, b->stream));
  BCHECK(cudaStreamSynchronize(b->stream));
  b->rows_stale = true;
  return EKF_OK;
}

int ekf_batch_get_feature(ekf_batch* b, int f, int idx, ekf_feature_info* o) {
  if (!b || f < 0 || f >= b->B || !o || idx < 0 || idx >= b->h_N[f]) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  const FeatTab t = feattab_slice(b->bv.ft, f, b->Ncap, b->bv.tstride);
  memset(o, 0, sizeof *o);
  cudaStream_t st = b->stream;
  int iv[10];
  const int* isrc[10] = {t.pos, t.pos_in_z, t.coding, t.n_tot, t.n_find, t.real_index, t.innov, t.li, t.hi, t.removef};
  for (int c = 0; c < 10; ++c) BCHECK(cudaMemcpyAsync(&iv[c], isrc[c] + idx, sizeof(int), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(o->center, t.center + 2 * idx, 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(&o->quality_index, t.quality + idx, sizeof(float), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(&o->last_ncc, t.last_ncc + idx, sizeof(float), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(o->z, t.z + 2 * idx, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(o->h, t.h + 2 * idx, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(o->H, t.Hc + 26 * idx, 26 * sizeof(double), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  o->position_in_state = iv[0]; o->position_in_z = iv[1]; o->coding = iv[2]; o->n_tot = iv[3]; o->n_find = iv[4];
  o->real_index = iv[5]; o->is_in_innovation = iv[6]; o->is_in_li = iv[7]; o->is_in_hi = iv[8]; o->remove_flag = iv[9];
  const int pos = iv[0], fs = iv[2] ? 3 : 6;
  const double* mu = b->bv.mu + (size_t)f * b->ld;
  const double* Sg = b->bv.Sigma + (size_t)f * b->bv.sstride;
  BCHECK(cudaMemcpyAsync(o->state, mu + pos, sizeof(double) * fs, cudaMemcpyDeviceToHost, st));
  double blk[36];
  BCHECK(cudaMemcpy2DAsync(blk, sizeof(double) * fs, Sg + (size_t)pos * b->ld + pos, sizeof(double) * b->ld, sizeof(double) * fs, fs,
                           cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  for (int a = 0; a < fs; ++a)
    for (int c = 0; c < fs; ++c) o->cov[a * 6 + c] = blk[a * fs + c];
  return EKF_OK;
}

int ekf_batch_add_feature(ekf_batch* b, int f, float u, float v) {
  if (!b || f < 0 || f >= b->B) return EKF_ERR_ARG;
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "addFeature before ekf_batch_seed_from");
  const int rc = need_frame(b, f, "addFeature");
  if (rc) return rc;
  BCHECK(cudaSetDevice(b->device));
  const int half = b->cfg.window_size / 2;
  // isInsideImage (vslamRansac.cpp:314,1644-1652), as ekf_add_feature
  const double x = (double)u, y = (double)v;
  const int c = b->cam_host[f], fw = b->fsize_on ? b->fsize_host[4 * c + 2] : b->fv.w, fh = b->fsize_on ? b->fsize_host[4 * c + 3] : b->fv.h;
  if (!(x > half && y > half && x < fw - half && y < fh - half)) return 0;
  if (b->h_N[f] >= b->Ncap || b->h_n[f] + 6 > b->ncap) return bfail(b, EKF_ERR_CAPACITY, "feature capacity exceeded");
  add_kernel(b, false)<<<1, BADD_THREADS, 0, b->stream>>>(b->bv, b->fv, b->dcfg, nullptr, nullptr, f, u, v, 0, b->cam_dev, nullptr);
  b->launches += 1;
  BCHECK(cudaGetLastError());
  b->h_N[f] += 1;
  b->h_n[f] += 6;
  return 1;
}

// EKF_ERR_STATE unless the camera of every filter that asks for corners (num[f * stride] > 0) holds a frame
static int need_frames_asked(ekf_batch* b, const int* num, int stride) {
  for (int f = 0; f < b->B; ++f) {
    if (num[(size_t)f * stride] <= 0) continue;
    const int rc = need_frame(b, f, "findNewFeatures");
    if (rc) return rc;
  }
  return EKF_OK;
}

static int batch_stage_num(ekf_batch* b, const int32_t* num) {
  std::copy(num, num + b->B, b->h_num);
  BCHECK(cudaMemcpyAsync(b->det_num, b->h_num, sizeof(int) * b->B, cudaMemcpyHostToDevice, b->stream));
  return EKF_OK;
}

int ekf_batch_detect_corners(ekf_batch* b, const int32_t* num, float* out_xy, int32_t* out_n) {
  if (!b || !num || !out_xy || !out_n) return EKF_ERR_ARG;
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "findNewFeatures before ekf_batch_seed_from");
  int rc = need_frames_asked(b, num, 1);
  if (rc) return rc;
  BCHECK(cudaSetDevice(b->device));
  cudaStream_t st = b->stream;
  const size_t Bn = (size_t)b->B;
  rc = batch_stage_num(b, num);
  if (rc) return rc;
  rc = batch_detect(b, b->det_num, b->h_num, 1, 0);
  if (rc) return rc;
  if (b->cstride == EKF_BATCH_MAX_CORNERS)
    BCHECK(cudaMemcpyAsync(b->h_det_xy, b->det_xy, sizeof(float) * Bn * 2 * EKF_BATCH_MAX_CORNERS, cudaMemcpyDeviceToHost, st));
  else   // the public layout: EKF_BATCH_MAX_CORNERS corners a filter (cap_mode 0 detects no more)
    BCHECK(cudaMemcpy2DAsync(b->h_det_xy, sizeof(float) * 2 * EKF_BATCH_MAX_CORNERS, b->det_xy, sizeof(float) * 2 * b->cstride,
                             sizeof(float) * 2 * EKF_BATCH_MAX_CORNERS, Bn, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(b->h_det_n, b->det_n, sizeof(int) * Bn, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  std::copy(b->h_det_xy, b->h_det_xy + Bn * 2 * EKF_BATCH_MAX_CORNERS, out_xy);
  std::copy(b->h_det_n, b->h_det_n + Bn, out_n);
  return EKF_OK;
}

int ekf_batch_find_new_features(ekf_batch* b, const int32_t* num, int32_t* added) {
  if (!b) return EKF_ERR_ARG;
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "findNewFeatures before ekf_batch_seed_from");
  if (!num && !b->results_valid) return bfail(b, EKF_ERR_STATE, "findNewFeatures(EKF_BSTAT_TOPUP) without a completed step");
  int rc = num ? need_frames_asked(b, num, 1) : need_frames_asked(b, b->h_stats + EKF_BSTAT_TOPUP, EKF_BATCH_STAT_FIELDS);
  if (rc) return rc;
  BCHECK(cudaSetDevice(b->device));
  rc = num ? batch_stage_num(b, num) : EKF_OK;
  if (rc) return rc;
  rc = num ? batch_topup(b, b->det_num, b->h_num, 1, 0)
           : batch_topup(b, b->out_stats + EKF_BSTAT_TOPUP, b->h_stats + EKF_BSTAT_TOPUP, EKF_BATCH_STAT_FIELDS, 0);
  if (rc) return rc;
  rc = batch_readback(b, true);
  if (rc) return rc;
  long long total = 0;
  for (int i = 0; i < b->B; ++i) total += b->h_added[i];
  if (added) std::copy(b->h_added, b->h_added + b->B, added);
  return (int)total;
}

int ekf_batch_set_topup(ekf_batch* b, int on) {
  if (!b) return EKF_ERR_ARG;
  b->topup = on != 0;
  return EKF_OK;
}

int ekf_batch_set_motion_blur(ekf_batch* b, int32_t kernel_size) {
  if (!b) return EKF_ERR_ARG;
  b->dcfg.kernel_min_size = kernel_size;
  b->blur = kernel_size < 100000;
  if (!b->blur) std::fill(b->h_blur, b->h_blur + 2 * (size_t)b->B, 0);   // steps without blur leave the counts at zero
  return EKF_OK;
}

int ekf_batch_last_blur_counts(ekf_batch* b, int32_t* out) {
  if (!b || !out) return EKF_ERR_ARG;
  std::copy(b->h_blur, b->h_blur + b->B, out);
  return EKF_OK;
}

int ekf_batch_last_added(ekf_batch* b, int32_t* added) {
  if (!b || !added) return EKF_ERR_ARG;
  std::copy(b->h_added, b->h_added + b->B, added);
  return EKF_OK;
}

int ekf_batch_get_template(ekf_batch* b, int f, int idx, int which, uint8_t* out) {
  if (!b || f < 0 || f >= b->B || !out || idx < 0 || idx >= b->h_N[f]) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  const FeatTab t = feattab_slice(b->bv.ft, f, b->Ncap, b->bv.tstride);
  const uint8_t* src = (which ? t.mpatch : t.patch) + (size_t)idx * b->bv.tstride;
  BCHECK(cudaMemcpyAsync(out, src, (size_t)b->cfg.window_size * b->cfg.window_size, cudaMemcpyDeviceToHost, b->stream));
  BCHECK(cudaStreamSynchronize(b->stream));
  return EKF_OK;
}

int ekf_batch_set_archive(ekf_batch* b, int32_t capacity) {
  if (!b || capacity < 0) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaStreamSynchronize(b->stream));
  cudaFree(b->ar.rec); cudaFree(b->ar.real_index); cudaFree(b->ar.count); cudaFree(b->ar.overflow);
  b->ar = BatchArchive{};
  if (capacity == 0) return EKF_OK;
  const size_t Bn = (size_t)b->B, slots = Bn * (size_t)capacity;
  BatchArchive a{};
  cudaError_t e = balloc(&a.rec, slots * PTS_COLS);
  if (e == cudaSuccess) e = balloc(&a.real_index, slots);
  if (e == cudaSuccess) e = balloc(&a.count, Bn);
  if (e == cudaSuccess) e = balloc(&a.overflow, Bn);
  if (e == cudaSuccess && !b->h_over) e = cudaMallocHost((void**)&b->h_over, sizeof(int) * Bn);
  if (e != cudaSuccess) {
    cudaFree(a.rec); cudaFree(a.real_index); cudaFree(a.count); cudaFree(a.overflow);
    return bfail(b, EKF_ERR_CUDA, std::string("feature archive allocation: ") + cudaGetErrorString(e));
  }
  a.cap = capacity;
  BCHECK(cudaMemsetAsync(a.count, 0, sizeof(int) * Bn, b->stream));
  BCHECK(cudaMemsetAsync(a.overflow, 0, sizeof(int) * Bn, b->stream));
  BCHECK(cudaStreamSynchronize(b->stream));
  std::fill(b->h_over, b->h_over + Bn, 0);
  b->over_seen.assign(Bn, 0);
  b->ar = a;
  return EKF_OK;
}

int ekf_batch_remove_feature(ekf_batch* b, int f, int index) {
  if (!b || f < 0 || f >= b->B) return EKF_ERR_ARG;
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "removeFeature before ekf_batch_seed_from");
  if (index < 0 || index >= b->h_N[f]) return bfail(b, EKF_ERR_ARG, "feature index out of range");
  BCHECK(cudaSetDevice(b->device));
  launch_compact(b, 0, nullptr, f, index);
  BCHECK(cudaGetLastError());
  const int rc = batch_readback(b, false);
  if (rc) return rc;
  return archive_check(b);
}

int ekf_batch_num_deleted(ekf_batch* b, int32_t* counts) {
  if (!b || !counts) return EKF_ERR_ARG;
  if (b->ar.cap <= 0) {
    std::fill(counts, counts + b->B, 0);
    return EKF_OK;
  }
  BCHECK(cudaSetDevice(b->device));
  BCHECK(cudaMemcpyAsync(counts, b->ar.count, sizeof(int) * b->B, cudaMemcpyDeviceToHost, b->stream));
  BCHECK(cudaStreamSynchronize(b->stream));
  return EKF_OK;
}

int ekf_batch_get_deleted(ekf_batch* b, int f, ekf_deleted_info* out, int cap, int* n) {
  if (!b || f < 0 || f >= b->B || !n || cap < 0 || (cap > 0 && !out)) return EKF_ERR_ARG;
  *n = 0;
  if (b->ar.cap <= 0) return EKF_OK;
  BCHECK(cudaSetDevice(b->device));
  cudaStream_t st = b->stream;
  int held = 0;
  BCHECK(cudaMemcpyAsync(&held, b->ar.count + f, sizeof(int), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  *n = held;
  const int k = std::min(held, cap);
  if (k <= 0) return EKF_OK;
  std::vector<double> rec((size_t)k * PTS_COLS);
  std::vector<int> ri(k);
  const size_t slot = (size_t)f * b->ar.cap;
  BCHECK(cudaMemcpyAsync(rec.data(), b->ar.rec + slot * PTS_COLS, sizeof(double) * rec.size(), cudaMemcpyDeviceToHost, st));
  BCHECK(cudaMemcpyAsync(ri.data(), b->ar.real_index + slot, sizeof(int) * k, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  for (int i = 0; i < k; ++i) {
    ekf_deleted_info& o = out[i];
    o.real_index = ri[i]; o._pad = 0;
    for (int c = 0; c < 3; ++c) o.xyz_pos[c] = rec[(size_t)i * PTS_COLS + c];
    for (int c = 0; c < 9; ++c) o.cov_4_delete[c] = rec[(size_t)i * PTS_COLS + 3 + c];
  }
  return EKF_OK;
}

int ekf_batch_get_points_features(ekf_batch* b, int first, int count, double* out, int rows_cap, int32_t* rows) {
  if (!b || !rows || first < 0 || count < 1 || first > b->B - count || (out && rows_cap < 1)) return EKF_ERR_ARG;
  BCHECK(cudaSetDevice(b->device));
  cudaStream_t st = b->stream;
  const size_t Bn = (size_t)b->B;
  if (!b->pts_dev) {
    BCHECK(balloc(&b->pts_dev, 2 * Bn));
    BCHECK(cudaMallocHost((void**)&b->h_pts, sizeof(int) * 2 * Bn));
  }
  const size_t bytes = out ? sizeof(double) * PTS_COLS * (size_t)rows_cap * count : 0;
  double* dev = nullptr;
  if (out) BCHECK(cudaMallocAsync((void**)&dev, bytes, st));
  k_batch_points_features<<<count, BPTS_THREADS, 0, st>>>(b->bv, b->ar, first, rows_cap, dev, b->pts_dev, b->pts_dev + count);
  b->launches += 1;
  BCHECK(cudaGetLastError());
  BCHECK(cudaMemcpyAsync(b->h_pts, b->pts_dev, sizeof(int) * 2 * count, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaStreamSynchronize(st));
  int most = 0;
  for (int k = 0; k < count; ++k) most = std::max(most, b->h_pts[k]);
  std::copy(b->h_pts, b->h_pts + count, rows);
  if (!out) return EKF_OK;
  if (most > rows_cap) {
    BCHECK(cudaFreeAsync(dev, st));
    BCHECK(cudaStreamSynchronize(st));
    return bfail(b, EKF_ERR_ARG, "rows_cap " + std::to_string(rows_cap) + " below the largest row count " + std::to_string(most));
  }
  BCHECK(cudaMemcpyAsync(out, dev, bytes, cudaMemcpyDeviceToHost, st));
  BCHECK(cudaFreeAsync(dev, st));
  for (int k = 0; k < count; ++k)   // the clear rule (R:395-403), on the device's archive of every exported filter
    if (pts_clears(b->h_pts[count + k])) BCHECK(cudaMemsetAsync(b->ar.count + first + k, 0, sizeof(int), st));
  BCHECK(cudaStreamSynchronize(st));
  return EKF_OK;
}

// Filter f <- filter ancestors[f], both as they stood before the call.  Pairs with ancestors[f] != f move; a source that is itself
// overwritten (ancestors[s] != s) is first staged, once however many destinations read it: its Sigma rows into its scratch slot
// (the compaction scratch is idle between calls), everything else into a temporary buffer of one slot per staged filter.  Then
// one launch copies the pairs whose source is not overwritten, and one the pairs whose source was staged.  The moved filters'
// host mirrors (n, N, counters, camera rows, added and blur counts, archive overflow) follow on the host.
static constexpr size_t kResampleBytesPerCta = (size_t)64 << 10;   // Sigma bytes one CTA of k_batch_resample copies, about
int ekf_batch_resample(ekf_batch* b, const int32_t* ancestors) {
  if (!b) return EKF_ERR_ARG;
  if (!ancestors) return bfail(b, EKF_ERR_ARG, "ancestors is NULL");
  for (int f = 0; f < b->B; ++f) {
    const int a = ancestors[f];
    if (a < 0 || a >= b->B)
      return bfail(b, EKF_ERR_ARG, "ancestors[" + std::to_string(f) + "] = " + std::to_string(a) + " lies outside [0, n_filters)");
    if (b->cam_host[a] != b->cam_host[f])
      return bfail(b, EKF_ERR_ARG, "ancestors[" + std::to_string(f) + "] = " + std::to_string(a) + " follows camera " +
                                       std::to_string(b->cam_host[a]) + ", filter " + std::to_string(f) + " camera " +
                                       std::to_string(b->cam_host[f]));
  }
  if (!b->seeded) return bfail(b, EKF_ERR_STATE, "resample before ekf_batch_seed_from");
  const int B = b->B;
  std::vector<int> slot(B, -1);
  std::vector<int2> stage, direct, staged;   // (staging slot, filter), (filter, filter), (filter, staging slot)
  int most = 0;
  for (int f = 0; f < B; ++f) {
    const int a = ancestors[f];
    if (a == f) continue;
    most = std::max(most, b->h_n[a]);
    if (ancestors[a] == a) { direct.push_back(make_int2(f, a)); continue; }
    if (slot[a] < 0) { slot[a] = (int)stage.size(); stage.push_back(make_int2(slot[a], a)); }
    staged.push_back(make_int2(f, slot[a]));
  }
  if (direct.empty() && staged.empty()) return EKF_OK;
  BCHECK(cudaSetDevice(b->device));
  cudaStream_t st = b->stream;
  if (!b->rs_pairs) BCHECK(balloc(&b->rs_pairs, 2 * (size_t)B));
  std::vector<int2> pairs(stage);
  pairs.insert(pairs.end(), direct.begin(), direct.end());
  pairs.insert(pairs.end(), staged.begin(), staged.end());
  BCHECK(cudaMemcpyAsync(b->rs_pairs, pairs.data(), sizeof(int2) * pairs.size(), cudaMemcpyHostToDevice, st));
  const BatchSlots live{b->bv, b->ar, b->intr_dev, b->out_mu14, b->out_S14, b->out_stats};
  const unsigned ctas = (unsigned)std::max<size_t>(1, (sizeof(double) * most * b->ld + kResampleBytesPerCta - 1) / kResampleBytesPerCta);
  const int2* pd = b->rs_pairs;
  void* tmp = nullptr;
  if (!stage.empty()) {
    // the staging slots: Sigma in the scratch, the rest carved from one allocation (256-byte aligned arrays)
    const size_t ns = stage.size(), nf = ns * b->Ncap, tsb = (size_t)b->bv.tstride;
    BatchSlots sg = live;
    sg.v.Sigma = b->scratch;
    auto layout = [&](char* base) {
      size_t off = 0;
      auto take = [&](auto*& p, size_t count) {
        using T = std::remove_reference_t<decltype(*p)>;
        off = (off + 255) & ~(size_t)255;
        p = reinterpret_cast<T*>(base + off);
        off += sizeof(T) * count;
      };
      FeatTab& t = sg.v.ft;
      take(sg.v.mu, ns * b->ld);
      for (int** p : {&t.pos, &t.coding, &t.innov, &t.li, &t.hi, &t.removef, &t.n_tot, &t.n_find, &t.real_index, &t.pos_in_z, &t.sel})
        take(*p, nf);
      take(t.center, 2 * nf); take(t.quality, nf); take(t.last_ncc, nf);
      take(t.z, 2 * nf); take(t.h, 2 * nf); take(t.Hc, 26 * nf); take(t.S2, 4 * nf);
      take(t.patch, nf * tsb); take(t.mpatch, nf * tsb);
      take(sg.v.ctl, ns); take(sg.v.n, ns); take(sg.v.N, ns); take(sg.v.patchnumbre, ns);
      take(sg.v.xyz_flag, nf); take(sg.v.xyz_J, 18 * nf); take(sg.v.xyz_y, 3 * nf); take(sg.v.xyz_count, ns);
      if (live.cam) take(sg.cam, ns);
      if (b->ar.cap > 0) {
        take(sg.ar.rec, ns * b->ar.cap * PTS_COLS); take(sg.ar.real_index, ns * b->ar.cap);
        take(sg.ar.count, ns); take(sg.ar.overflow, ns);
      }
      take(sg.mu14, 14 * ns); take(sg.S14, 196 * ns); take(sg.stats, EKF_BATCH_STAT_FIELDS * ns);
      return off;
    };
    const size_t bytes = layout(nullptr);
    BCHECK(cudaMallocAsync(&tmp, bytes, st));
    layout(static_cast<char*>(tmp));
    k_batch_resample<<<dim3((unsigned)ns, ctas), BRS_THREADS, 0, st>>>(sg, live, pd);
    b->launches += 1;
    BCHECK(cudaGetLastError());
    if (!direct.empty()) {
      k_batch_resample<<<dim3((unsigned)direct.size(), ctas), BRS_THREADS, 0, st>>>(live, live, pd + ns);
      b->launches += 1;
    }
    k_batch_resample<<<dim3((unsigned)staged.size(), ctas), BRS_THREADS, 0, st>>>(live, sg, pd + ns + direct.size());
    b->launches += 1;
    BCHECK(cudaGetLastError());
    BCHECK(cudaFreeAsync(tmp, st));
  } else {
    k_batch_resample<<<dim3((unsigned)direct.size(), ctas), BRS_THREADS, 0, st>>>(live, live, pd);
    b->launches += 1;
    BCHECK(cudaGetLastError());
  }
  BCHECK(cudaStreamSynchronize(st));
  auto follow = [&](auto* p, size_t width) {   // row f of a host mirror <- row ancestors[f]
    using T = std::remove_reference_t<decltype(*p)>;
    const std::vector<T> old(p, p + (size_t)B * width);
    for (int f = 0; f < B; ++f) std::copy_n(old.begin() + (size_t)ancestors[f] * width, width, p + (size_t)f * width);
  };
  follow(b->h_n, 1); follow(b->h_N, 1); follow(b->h_added, 1); follow(b->h_xyz_count, 1);
  follow(b->h_mu14, 14); follow(b->h_stats, EKF_BATCH_STAT_FIELDS);
  follow(b->h_blur, 1); follow(b->h_blur + B, 1);   // [2][B]: blurred templates, then kernel too large
  if (b->ar.cap > 0) { follow(b->h_over, 1); follow(b->over_seen.data(), 1); }
  return EKF_OK;
}

int64_t ekf_batch_kernel_launches(const ekf_batch* b) { return b ? b->launches : 0; }

int ekf_batch_last_step_ms(ekf_batch* b, float out[3]) {
  if (!b || !out) return EKF_ERR_ARG;
  if (!b->results_valid) return bfail(b, EKF_ERR_STATE, "no completed step");
  for (int i = 0; i < 3; ++i)
    if (cudaEventElapsedTime(&out[i], b->ev[i], b->ev[i + 1]) != cudaSuccess) out[i] = -1.0f;
  return EKF_OK;
}

int ekf_batch_last_match_deferred(ekf_batch* b) {
  if (!b) return EKF_ERR_ARG;
  if (cudaSetDevice(b->device) != cudaSuccess) return EKF_ERR_CUDA;
  int v = 0;
  if (cudaMemcpyAsync(&v, b->match_defer + (size_t)b->B * b->Ncap, sizeof(int), cudaMemcpyDeviceToHost, b->stream) != cudaSuccess ||
      cudaStreamSynchronize(b->stream) != cudaSuccess)
    return EKF_ERR_CUDA;
  return v;
}

}  // extern "C"
