/* include/ekf_b200.h — C ABI of the B200-native MonoSLAM EKF hot path.
 *
 * Drop-in boundary for ONE path of engyasin/EKF-MonoSLAM_for_3D-reconstruction: the per-frame EKF
 * of `class VSlamFilter` (mono-slam/src/vslamRansac.hpp:27-141, vslamRansac.cpp) together with the
 * active-search matcher `Patch::findMatch` (mono-slam/src/Patch.cpp:215-329) and the camera model
 * (mono-slam/src/camModel.cpp).  The reference has no FFI of its own; its seam is the C++ class.
 * Each entry point below names the reference member it replaces.  A C++ class with the reference's
 * method names over this ABI lives in ekf-monoslam_for_3d-reconstruction_b200/host/vslam_filter.hpp;
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *  - plain C types only; every function returns an int status (EKF_OK or a negative error) unless
 *    it mirrors a reference function with its own return value (documented per function);
 *  - all arithmetic is fp64 on the GPU (the reference is fp32 Eigen; BASELINE.json asks for fp64);
 *  - matrices cross the boundary row-major; the state layout is the reference's:
 *    mu = [ r(3) q(4, w first) v(3) w(3) map_scale | features... ], STATE_DIM 14
 *    (vslamRansac.cpp:22,163-164), inverse-depth feature = (x y z theta phi rho), XYZ = (x y z);
 *  - a handle owns all device state, is bound to one CUDA device and one stream, and is not
 *    thread-safe (the reference is a single-threaded ros::spin loop, monoslam_ransac.cpp:865);
 *  - there is NO CPU fallback: every call fails with EKF_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef EKF_B200_H_
#define EKF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EKF_STATE_DIM 14 /* vslamRansac.cpp:22 */

enum {
  EKF_OK = 0,
  EKF_ERR_ARG = -1,         /* bad argument */
  EKF_ERR_CUDA = -2,        /* CUDA runtime error, see ekf_last_error() */
  EKF_ERR_CAPACITY = -3,    /* feature / state capacity of the handle exceeded */
  EKF_ERR_UNSUPPORTED = -4, /* configuration asks for a reference feature outside this path */
  EKF_ERR_STATE = -5        /* call order violated (e.g. update before predict) */
};

/* ConfigVSLAM (mono-slam/src/ConfigVSLAM.h:23-48, defaults ConfigVSLAM.cpp:27-47) + camConfig
 * (camModel.hpp:9-11, defaults camModel.hpp:25-33) + the constants the reference hard-codes,
 * each named with its source line.  ekf_config_default() fills the reference values. */
typedef struct ekf_config {
  double sigma_vx, sigma_vy, sigma_vz; /* ConfigVSLAM.cpp:28 */
  double sigma_wx, sigma_wy, sigma_wz; /* ConfigVSLAM.cpp:29 */
  double rho_0, sigma_rho_0;           /* ConfigVSLAM.cpp:34-35 */
  double T_camera;                     /* ConfigVSLAM.cpp:39 */
  double fx, fy, u0, v0, k1, k2, k3, p1, p2; /* camModel.hpp:25-33 */
  double ncc_threshold;        /* Patch.cpp:14          0.8   */
  double search_clamp;         /* Patch.cpp:240-241     20 px */
  double ransac_p;             /* vslamRansac.cpp:967   0.99  */
  double li_threshold_factor;  /* vslamRansac.cpp:968   2 (x sigma_pixel) */
  double hi_chi2_threshold;    /* vslamRansac.cpp:1066  1     */
  double quality_ratio;        /* Patch.hpp:39          0.2   */
  double linearity_threshold;  /* vslamRansac.cpp:701   0.01  */
  int32_t window_size;         /* ConfigVSLAM.cpp:31    21    */
  int32_t sigma_pixel;         /* ConfigVSLAM.cpp:32    2     */
  int32_t kernel_size;         /* Patch::blur threshold in px; no default in the reference (ConfigVSLAM.cpp:76); here 1e9 = blur off */
  int32_t sigma_size;          /* ConfigVSLAM.cpp:41    2     */
  int32_t scale;               /* ConfigVSLAM.cpp:37    1     */
  int32_t nInitFeatures, min_features, max_features, forsePlane; /* ConfigVSLAM.cpp:43-48 */
  int32_t ransac_nhyp0;        /* vslamRansac.cpp:966   10000 */
  int32_t xyz_conversion;      /* vslamRansac.cpp:1317  1 = convert2XYZ_ifLinearAll() every update */
  int32_t abs_int_quirk;       /* vslamRansac.cpp:719   0 = abs(float) is fabs (modern libstdc++) */
} ekf_config;

/* One feature as RosVSLAM / the ROS node read it (Patch.hpp:18-106; RosVSLAMRansac.cpp:177-183). */
typedef struct ekf_feature_info {
  int32_t position_in_state, position_in_z, coding /* 0 = inverse depth, 1 = XYZ */;
  int32_t n_tot, n_find, real_index;
  int32_t is_in_innovation, is_in_li, is_in_hi, remove_flag;
  float center[2];     /* Patch::center (cv::Point2f) */
  float quality_index; /* Patch::quality_index */
  float last_ncc;      /* best NCC of the last findMatch (diagnostic) */
  double z[2], h[2];   /* Patch::z, Patch::h */
  double H[26];        /* Patch::H, compact 2 x 13: columns [0,7) = d/d(r,q), [7,13) = d/d(feature) */
  double state[6];     /* mu[pos .. pos+6) (3 used when XYZ) */
  double cov[36];      /* Sigma[pos.., pos..] row-major 6 x 6 (3 x 3 top-left when XYZ) */
} ekf_feature_info;

/* Counters of the last completed step (diagnostics; not in the reference). */
typedef struct ekf_step_stats {
  int32_t n_in_innovation_predict; /* features that passed the gate in predict (vslamRansac.cpp:529) */
  int32_t n_matched;               /* vslamRansac.cpp:984 */
  int32_t n_li, n_hi;              /* rows/2 of the two updates */
  int32_t ransac_hypotheses;       /* loop trips of vslamRansac.cpp:986 */
  int32_t n_removed;               /* features dropped by vslamRansac.cpp:1296-1299 */
  int32_t topup_request;           /* argument passed to findNewFeatures at vslamRansac.cpp:1314 (0 = no top-up this step) */
  int32_t blur_requests;           /* templates blurred by the last predict (Patch::blur, Patch.cpp:52) */
  int64_t kernel_launches;         /* kernels of this library launched on the handle so far */
} ekf_step_stats;

typedef struct ekf_handle ekf_handle;

/* ---- life cycle ------------------------------------------------------------------------------ */
/* Fills *cfg with the reference defaults (ConfigVSLAM.cpp:27-47, camModel.hpp:25-33). */
void ekf_config_default(ekf_config* cfg);
/* VSlamFilter::VSlamFilter (vslamRansac.cpp:142-223).  `feature_capacity` bounds the number of
 * simultaneously tracked features (device buffers are sized for n = 14 + 6*capacity). `device` is
 * a CUDA ordinal.  A window_size outside [3, 31] or a search_clamp above 20 px return
 * EKF_ERR_UNSUPPORTED. */
int ekf_create(const ekf_config* cfg, int feature_capacity, int device, ekf_handle** out);
int ekf_destroy(ekf_handle* h);
/* Use `cuda_stream` (a cudaStream_t) for all work of this handle; NULL = the handle's own stream. */
int ekf_set_stream(ekf_handle* h, void* cuda_stream);
/* Blocks until all work queued on the handle is done. */
int ekf_sync(ekf_handle* h);
const char* ekf_last_error(const ekf_handle* h);

/* ---- the per-frame path ---------------------------------------------------------------------- */
/* VSlamFilter::captureNewFrame(cv::Mat, double) (vslamRansac.cpp:226-245): 8-bit gray, HOST
 * memory, copied to the device inside the call.  stamp < 0 = the no-stamp overload. */
int ekf_capture_frame(ekf_handle* h, const uint8_t* gray, int width, int height, int stride, double stamp);
/* The 3-channel case of captureNewFrame (vslamRansac.cpp:238-241): 8-bit BGR, HOST memory.  With
 * cfg.scale > 1 every capture call first resizes to (width / scale) x (height / scale) like cv::resize
 * (INTER_LINEAR) and then converts BGR to gray, on the GPU; the intrinsics of ekf_config are those of the
 * resized image, as ConfigVSLAM.cpp:89-120 produces them. */
int ekf_capture_frame_bgr(ekf_handle* h, const uint8_t* bgr, int width, int height, int stride, double stamp);
/* VSlamFilter::returnGrayImg (vslamRansac.cpp:1364): the gray frame the filter works on (after resize);
 * out may be NULL to query the size only. */
int ekf_get_frame(ekf_handle* h, uint8_t* out, int* width, int* height);
/* Same, for a frame already resident in DEVICE memory (copied device-to-device). */
int ekf_capture_frame_device(ekf_handle* h, const uint8_t* gray_dev, int width, int height, int stride, double stamp);
/* VSlamFilter::predict (vslamRansac.cpp:451-603). */
int ekf_predict(ekf_handle* h, const double dv[3], const double dw[3], int vcontrol);
/* The active-search loop at the top of VSlamFilter::update (vslamRansac.cpp:870-880), split out so
 * it can be timed and so matches can be injected.  Returns the matched count in *n_matched if not
 * NULL (forces a device sync). */
int ekf_match(ekf_handle* h, int* n_matched);
/* The rest of VSlamFilter::update (vslamRansac.cpp:964-1341).  `picks` replaces rand()
 * (vslamRansac.cpp:970,989): hypothesis k draws picks[k % n_picks] % candidates (0 if n_picks==0).
 * n_picks <= EKF_PICKS_CAP (the device copy is sized at ekf_create; more returns EKF_ERR_CAPACITY). */
#define EKF_PICKS_CAP 65536
int ekf_update_after_match(ekf_handle* h, const uint32_t* picks, int n_picks);
/* VSlamFilter::update = ekf_match + ekf_update_after_match. */
int ekf_update(ekf_handle* h, const uint32_t* picks, int n_picks);
/* Overrides Patch::z / center of feature idx and marks it matched (test hook for injected matches). */
int ekf_inject_match(ekf_handle* h, int idx, double zu, double zv, int accepted);

/* ---- map management -------------------------------------------------------------------------- */
/* VSlamFilter::addFeature (vslamRansac.cpp:309-371): returns 1 added, 0 rejected, <0 error. */
int ekf_add_feature(ekf_handle* h, float u, float v);
/* VSlamFilter::removeFeature (vslamRansac.cpp:373-421). */
int ekf_remove_feature(ekf_handle* h, int index);
/* VSlamFilter::findNewFeatures(num) (vslamRansac.cpp:783-839): builds the reference's mask around the
 * existing patches, detects up to `num` (<= 0: nInitFeatures; capped at 1024) Shi-Tomasi corners with
 * the parameters the reference passes to OpenCV goodFeaturesToTrack (quality 0.01, min distance 12,
 * 3x3 block) and calls addFeature on each.  Returns the number added (>= 0) or an error.  The
 * detector restates OpenCV's published algorithm; see csrc/ekf_detect.cu for the parity statement. */
int ekf_find_new_features(ekf_handle* h, int num);
/* The detection alone: up to `num` corners as (x, y) pairs into out_xy (capacity 2 * 1024 floats). */
int ekf_detect_corners(ekf_handle* h, int num, float* out_xy, int* out_n);
/* VSlamFilter::convert2XYZ_ifLinear / convert2XYZ_ifLinearAll (vslamRansac.cpp:741-780). */
int ekf_convert2xyz_if_linear(ekf_handle* h, int index);
int ekf_convert2xyz_if_linear_all(ekf_handle* h);

/* ---- accessors the ROS node / RosVSLAM read ---------------------------------------------------- */
int ekf_num_features(const ekf_handle* h);                     /* numOfFeatures, vslamRansac.cpp:127 */
int ekf_state_dim(const ekf_handle* h);                        /* mu.rows() */
int ekf_get_state(ekf_handle* h, double out[EKF_STATE_DIM]);   /* getState, vslamRansac.cpp:135-140 */
int ekf_get_sigma(ekf_handle* h, double out[EKF_STATE_DIM * EKF_STATE_DIM]); /* getSigma, :131-133 */
int ekf_covariance_parameter(ekf_handle* h, double* out);      /* Covariance_Parameter, :841-866 */
double ekf_get_dt(const ekf_handle* h);                        /* getDt, :247 */
int ekf_get_center(ekf_handle* h, int idx, float out[2]);      /* returnCentrPatchIndx, vslamRansac.hpp:136 */
int ekf_get_feature(ekf_handle* h, int idx, ekf_feature_info* out);
/* which: 0 = Patch::patch, 1 = Patch::matching_patch; out holds window_size^2 bytes */
int ekf_get_template(ekf_handle* h, int idx, int which, uint8_t* out);
int ekf_get_step_stats(ekf_handle* h, ekf_step_stats* out);

/* ---- caller-side rows (SURVEY.md section 8(f) item 4) ------------------------------------------ */
/* Patch archived by removeFeature (Patch::XYZ_pos / cov_4_delete, vslamRansac.cpp:394-404): XYZ features seen
 * more than five times keep their last position and 3x3 covariance (column-major copy of block^T = the block
 * row by row) in VSlamFilter::deleted_patches, which RosVSLAM reads (RosVSLAMRansac.cpp:312-332, 397-416). */
typedef struct ekf_deleted_info {
  int32_t real_index;
  int32_t _pad;
  double xyz_pos[3];
  double cov_4_delete[9];
} ekf_deleted_info;
int ekf_num_deleted(const ekf_handle* h);                      /* deleted_patches.size() */
int ekf_get_deleted(ekf_handle* h, int i, ekf_deleted_info* out);
/* RosVSLAM::getPointsFeatures (RosVSLAMRansac.cpp:340-418), the matrix points.txt is written from
 * (monoslam_ransac.cpp:273-275): (real_index of the last patch + 1) rows x 12, row r = feature with
 * real_index r: XYZ position * map_scale and its 3x3 covariance; rows of inverse-depth or unknown features
 * stay zero; archived features fill theirs.  *rows receives the row count; out may be NULL to query it.
 * As in the reference, more than 7000 archived patches are cleared by the call. */
int ekf_get_points_features(ekf_handle* h, double* out, int rows_cap, int* rows);
/* VSlamFilter::rts_epoch (vslamRansac.cpp:423-449): one backward Rauch-Tung-Striebel step on the 13 camera
 * states (System_model_jacobian is 13 x 13).  mu / sigma (13, 13 x 13 row-major) are updated in place from the
 * smoothed successor (mu_s, sigma_s) and the controls that were applied between the two epochs. */
int ekf_rts_epoch(ekf_handle* h, double mu[13], double sigma[169], const double mu_s[13], const double sigma_s[169],
                  const double dTspeed[3], const double dRspeed[3], double deltaT);

/* ---- whole-state get / set (checkpoint-resume and per-step parity with identical inputs) ------- */
/* mu: n doubles; sigma: n x n row-major with leading dimension ld >= n. */
int ekf_get_full(ekf_handle* h, double* mu, double* sigma, int ld);
int ekf_set_full(ekf_handle* h, const double* mu, const double* sigma, int ld);
/* Innovation covariance after predict (St of vslamRansac.cpp:598): the 2x2 diagonal block of every
 * feature (4 doubles each, row-major, zeros if not in innovation).  Only these blocks are consumed
 * by the reference (vslamRansac.cpp:875). */
int ekf_get_S_blocks(ekf_handle* h, double* out /* 4 * num_features */);

/* ---- stateless batched matcher (BASELINE config 5) --------------------------------------------- */
/* Patch::findMatch (Patch.cpp:215-291) for F frames x M features, everything in DEVICE memory:
 *   frames    F x height x stride u8
 *   templates F*M x w x w u8        (Patch::matching_patch)
 *   h         F*M x 2 doubles       (Patch::h)
 *   S         F*M x 4 doubles       (2x2 block of St, row-major)
 *   out_uv    F*M x 2 int32         (Patch::center / z; -1,-1 when rejected)
 *   out_score F*M floats            (best NCC; -1 when no candidate)
 * `stream` is a cudaStream_t (NULL = default stream). */
int ekf_match_batch(const uint8_t* frames, int n_frames, int width, int height, int stride,
                    const uint8_t* templates, int features_per_frame, int window_size,
                    const double* h, const double* S, float sigma_size, float ncc_threshold,
                    float search_clamp, int32_t* out_uv, float* out_score, void* stream);

/* ---- batch of independent filters (BASELINE config 3: multi-hypothesis / Monte-Carlo) ----------- */
/* B filters built from one configuration, stepped together on one device: one fused CTA per filter
 * for predict (vslamRansac.cpp:451-603) and for update (:964-1341), one CTA per (filter, feature)
 * for the active search (:870-880).  Filter b follows camera camera_of[b] (ekf_batch_set_cameras): each camera has its
 * own frame and time stamp, and every filter of a camera searches that camera's frame.  By default one camera is followed
 * by every filter (many hypotheses around one camera); B cameras of one filter each run B independent sequences.
 * Every filter runs exactly the single-filter algorithm; there is no exchange between filters, so a
 * batch shards across GPUs by filter index with no collective (one ekf_batch per device / rank).
 * A step ends like the single filter's update: feature deletion, then, once ekf_batch_set_topup has
 * switched it on, findNewFeatures (vslamRansac.cpp:1312-1315) on every filter that sees fewer than
 * min_features features, then, when cfg.xyz_conversion is set, convert2XYZ_ifLinearAll (:1317) on every
 * filter.  Top-up is off by default: the step then only reports in EKF_BSTAT_TOPUP how many features
 * each filter asks for, and ekf_batch_find_new_features serves those requests when the caller wants.
 * ekf_batch_create takes feature_capacity <= 32 (the stacked update of one filter is kept in one CTA's shared memory);
 * ekf_batch_create_large takes up to 128 (the update of one filter on a cluster of CTAs).  ekf_batch_create
 * refuses motion blur (kernel_size < 100000), scale != 1 and forsePlane (EKF_ERR_UNSUPPORTED); each of them is
 * switched on after creation instead, with ekf_batch_set_motion_blur, ekf_batch_set_scale and
 * ekf_batch_set_force_plane, so that a batch honours every ConfigVSLAM switch a single filter honours.
 * The configuration is every filter's by default; ekf_batch_set_intrinsics and ekf_batch_set_filter_params give each filter
 * intrinsics and tuning of its own, ekf_batch_set_camera_settings each camera a window_size, scale and kernel_size of its own,
 * while search_clamp, forsePlane, xyz_conversion and abs_int_quirk stay shared by the batch. */
typedef struct ekf_batch ekf_batch;
typedef struct ekf_batch_desc {
  int32_t n_filters, feature_capacity, state_capacity /* 14 + 6 * feature_capacity */, ld /* Sigma row stride */;
  int32_t device;
  int32_t reserved[3];
} ekf_batch_desc;
/* per-filter counters of the last step, EKF_BATCH_STAT_FIELDS int32 each */
#define EKF_BATCH_STAT_FIELDS 8
enum { EKF_BSTAT_INNOV = 0, EKF_BSTAT_MATCHED = 1, EKF_BSTAT_LI = 2, EKF_BSTAT_HI = 3, EKF_BSTAT_HYPS = 4,
       EKF_BSTAT_CHOL_FAIL = 5, EKF_BSTAT_REMOVED = 6, EKF_BSTAT_TOPUP = 7 };

int ekf_batch_create(const ekf_config* cfg, int n_filters, int feature_capacity, int device, ekf_batch** out);
/* A batch of up to EKF_BATCH_MAX_FEATURES features per filter (1 <= feature_capacity <= 128; EKF_ERR_CAPACITY above).
 * With feature_capacity <= 32 it is exactly what ekf_batch_create builds.  Above 32, each filter's update runs on a
 * thread-block cluster of ceil(ld / 208) CTAs (2 to 4) that share the stacked update through distributed shared memory;
 * EKF_ERR_UNSUPPORTED when the device cannot hold one such cluster.  Every other ekf_batch_* entry works on it unchanged.
 * Memory: Sigma and the compaction scratch are n_filters x state_capacity x ld doubles each, 4.9 MB per filter each at
 * capacity 128 (40 GB in total for 4096 filters). */
#define EKF_BATCH_MAX_FEATURES 128
int ekf_batch_create_large(const ekf_config* cfg, int n_filters, int feature_capacity, int device, ekf_batch** out);
/* CTAs per filter in the batch's update (1 for capacity <= 32) and, for a cluster update, how many clusters the device holds
 * at once (0 otherwise); either pointer may be NULL. */
int ekf_batch_update_clusters(const ekf_batch* b, int32_t* ctas_per_filter, int32_t* resident);
int ekf_batch_destroy(ekf_batch* b);
int ekf_batch_describe(const ekf_batch* b, ekf_batch_desc* out);
int ekf_batch_set_stream(ekf_batch* b, void* cuda_stream);
int ekf_batch_sync(ekf_batch* b);
const char* ekf_batch_last_error(const ekf_batch* b);
/* Every filter of the batch becomes a copy of `src` (state, covariance, feature table, templates,
 * time stamps); src must live on the same device and hold <= feature_capacity features. */
int ekf_batch_seed_from(ekf_batch* b, ekf_handle* src);
/* Overwrites the 14 camera entries of every filter's state (HOST array, n_filters x 14, row-major):
 * the per-hypothesis perturbation of a Monte-Carlo ensemble. */
int ekf_batch_set_camera_states(ekf_batch* b, const double* mu14);
/* captureNewFrame for the whole batch (vslamRansac.cpp:226-245): 8-bit gray from HOST / DEVICE memory, 8-bit BGR from
 * HOST memory.  With a scale > 1 (ekf_batch_set_scale) every capture resizes and converts as ekf_capture_frame_bgr does;
 * a resized side below 8 px returns EKF_ERR_ARG. */
int ekf_batch_capture_frame(ekf_batch* b, const uint8_t* gray, int width, int height, int stride, double stamp);
int ekf_batch_capture_frame_device(ekf_batch* b, const uint8_t* gray_dev, int width, int height, int stride, double stamp);
int ekf_batch_capture_frame_bgr(ekf_batch* b, const uint8_t* bgr, int width, int height, int stride, double stamp);
/* returnGrayImg (vslamRansac.cpp:1364) for the batch: the gray frame every filter works on (after resize); out may be
 * NULL to query the size only.  EKF_ERR_STATE before a frame.  With more than one camera ekf_batch_capture_frame* and
 * ekf_batch_get_frame return EKF_ERR_STATE: use the plural entries below. */
int ekf_batch_get_frame(ekf_batch* b, uint8_t* out, int* width, int* height);
/* Cameras: filter f follows camera camera_of[f] in [0, n_cameras) (HOST array of n_filters entries; NULL = identity, which
 * needs n_cameras == n_filters), 1 <= n_cameras <= n_filters, else EKF_ERR_ARG.  Cameras share the configuration (window,
 * scale); intrinsics may differ per filter (ekf_batch_set_intrinsics) and frame sizes per camera (ekf_batch_set_frame_sizes).  The default is one camera
 * followed by every filter.  The call forgets the captured frames (a step then needs a capture first) and sets every camera's clock (dT, time stamp) to camera 0's;
 * ekf_batch_seed_from sets every camera's clock from the source filter.  Memory: the gray frames, n_cameras x stride x
 * height bytes after resize (stride = width rounded up to 16), e.g. 1.26 GB for 4096 cameras of 640 x 480. */
int ekf_batch_set_cameras(ekf_batch* b, int n_cameras, const int32_t* camera_of);
/* Intrinsics per filter: cam is a HOST array of n_filters x 9 doubles in ekf_config order (fx fy u0 v0 k1 k2 k3 p1 p2), and
 * filter f projects, linearises and unprojects with row f in predict, the blur prediction, RANSAC, the Hi rescue and
 * addFeature.  NULL returns every filter to the configuration's intrinsics, which is the default.  A non-finite entry or
 * fx <= 0 or fy <= 0 returns EKF_ERR_ARG and leaves the table as it was.  As for ekf_batch_set_scale, the intrinsics are
 * those of the resized image.  The table goes to the device inside this call (no per-step copy); ekf_batch_seed_from and
 * ekf_batch_set_cameras leave it alone.  For intrinsics per camera, pass row camera_of[f] for filter f.  Memory: one device
 * row of 240 B per filter (intrinsics and tuning together) while this table or the tuning table is set.  The tuning (ekf_batch_set_filter_params) is a table of its own: setting or
 * clearing one leaves the other alone.  Window, search clamp and scale stay shared by the batch. */
int ekf_batch_set_intrinsics(ekf_batch* b, const double* cam);
/* The ekf_config fields a filter of a batch may take on its own (its tuning), under their ekf_config names and types. */
typedef struct ekf_filter_params {
  double sigma_vx, sigma_vy, sigma_vz; /* process noise: Vmax of predict (vslamRansac.cpp:194-200) */
  double sigma_wx, sigma_wy, sigma_wz;
  double rho_0, sigma_rho_0;           /* addFeature's inverse-depth prior */
  double T_camera;                     /* blur pose (with ekf_batch_set_motion_blur) */
  double ncc_threshold;                /* matcher acceptance */
  double ransac_p;                     /* 1-point RANSAC */
  double li_threshold_factor;          /* Li threshold = li_threshold_factor * sigma_pixel */
  double hi_chi2_threshold;            /* Hi rescue */
  double quality_ratio;                /* quality deletion */
  double linearity_threshold;          /* XYZ conversion decisions */
  int32_t sigma_pixel;                 /* R, the S blocks and addFeature's covariance */
  int32_t sigma_size;                  /* matcher search box */
  int32_t min_features, max_features;  /* top-up request (EKF_BSTAT_TOPUP) and the removeFeature(0) rule */
  int32_t ransac_nhyp0;
  int32_t _pad;
} ekf_filter_params;
/* Tuning per filter: rows is a HOST array of n_filters ekf_filter_params, and filter f predicts, matches, updates, deletes,
 * asks for features and adds them with row f (predict and its blur pose, the three matcher kernels, RANSAC, the Hi rescue,
 * both updates, the book-keeping, the XYZ decisions and addFeature), exactly as a single filter whose ekf_config carries
 * row f.  NULL returns every filter to the configuration's values, which is the default.  A non-finite entry, a negative
 * standard deviation (sigma_v*, sigma_w*, sigma_rho_0), sigma_pixel < 1, sigma_size < 1, ransac_p outside (0, 1),
 * ransac_nhyp0 < 1 or a negative min_features / max_features returns EKF_ERR_ARG, ekf_batch_last_error names the first bad
 * filter and field, and the table stays as it was; EKF_ERR_ARG for a NULL batch.  The table goes to the device inside this
 * call (no per-step copy).  It is independent of ekf_batch_set_intrinsics (setting or clearing one leaves the other alone);
 * ekf_batch_seed_from and ekf_batch_set_cameras leave it alone, ekf_batch_resample moves the row with the filter,
 * ekf_batch_step_filters steps each listed filter with its row, and ekf_batch_find_new_features(NULL) serves each filter's
 * request from its own min_features.  For a tuning per camera, pass row camera_of[f] for filter f.  Memory: one row of
 * 240 B per filter on the device (the row it shares with the intrinsics) while either table is set. */
int ekf_batch_set_filter_params(ekf_batch* b, const ekf_filter_params* rows);
/* Settings per camera: the three ekf_config fields a camera's filters may take on their own (ekf_batch_set_camera_settings). */
typedef struct ekf_camera_settings {
  int32_t window_size;   /* template side, 3 .. the window_size the batch was created with */
  int32_t scale;         /* capture resizes by 1 / scale, 1 .. 64 */
  int32_t kernel_size;   /* Patch::blur threshold; >= 100000: no motion blur on this camera */
  int32_t _pad;
} ekf_camera_settings;
/* Window, scale and blur threshold per camera: rows is a HOST array of n_cameras ekf_camera_settings, and filter f runs with
 * row camera_of[f] exactly as it would in a batch created with that row's window, scale and blur threshold: the same matches,
 * NCC scores, templates, feature tables, counters, state and covariance, bit for bit.  NULL returns every camera to the
 * batch's values (window_size of the configuration, ekf_batch_set_scale, ekf_batch_set_motion_blur), which is the default.
 *  - Templates stay stored at the create-time stride, so the configuration's window_size is the largest window a camera may take.
 *  - A window outside [3, create-time window_size] or a scale outside [1, 64] returns EKF_ERR_ARG, ekf_batch_last_error names the
 *    camera and the field, and the table stays as it was.  kernel_size takes any value, as in ekf_batch_set_motion_blur.
 *  - A call that changes the window of a camera whose filters hold features returns EKF_ERR_STATE and names the filter (its
 *    templates have the old size); the table stays as it was.
 *  - Frames: camera c's frame is resized to w_c / s_c x h_c / s_c, w_c x h_c its ekf_batch_set_frame_sizes size or the whole slot.
 *    The stack's slot is sized by the smallest scale s_min: n_cameras x (width / s_min rounded up to 16) x height / s_min bytes,
 *    however large the other cameras' scales are.  A call that changes some camera's scale forgets the captured frames, as
 *    ekf_batch_set_frame_sizes does.  Gray frames at scale 1 on every camera, captured for every camera, still go up in one copy.
 *  - While a table is set, ekf_batch_set_scale and ekf_batch_set_motion_blur return EKF_ERR_STATE; ekf_batch_set_cameras clears
 *    the table (EKF_ERR_STATE, changing nothing, when that would change the window of a filter that holds features);
 *    ekf_batch_seed_from with a source that holds features returns EKF_ERR_ARG unless the source's window equals every camera's
 *    (an empty source seeds any table); ekf_batch_resample moves filters within a camera, so their settings stay.
 *  - Motion blur runs in a step when some camera's kernel_size is below 100000; each filter uses its camera's threshold and its
 *    own T_camera, and the filters of a camera with blur off blur nothing.
 *  - ekf_batch_get_template writes window_c^2 bytes for a filter of camera c; findNewFeatures' mask border and patch boxes,
 *    addFeature's isInsideImage, the prediction gate and the matcher use the camera's window.
 * Memory: one device row of 240 B per filter (the row of ekf_batch_set_filter_params) and 4 B per camera while the table is set. */
int ekf_batch_set_camera_settings(ekf_batch* b, const ekf_camera_settings* rows);
/* A frame size per camera: wh is a HOST array of n_cameras x 2 int32 (width, height) in INPUT pixels, before the resize by
 * 1 / scale; NULL (the default) means every camera uses the whole frame the capture calls pass.  The stack keeps one slot per
 * camera: the capture calls' width / height / stride describe the slot, and camera c's frame is the top-left w_c x h_c of slot
 * c, resized to w_c / scale x h_c / scale (integer division, like cv::Size) inside a slot of width / scale x height / scale.
 * Prediction gate, matching and its window clipping, detection, addFeature's isInsideImage and ekf_batch_get_camera_frame use
 * the camera's own size.  The bytes of a slot outside its camera's frame do not change any result: a capture zeroes them (one
 * launch over the stack, none when every camera fills its slot).  Non-positive sizes return EKF_ERR_ARG; a capture with a
 * camera larger than its slot or a resized side below 8 returns EKF_ERR_ARG.  The sizes hold from the next capture on (the
 * call forgets the captured frames); ekf_batch_set_cameras returns to NULL.  Memory: 16 B per camera on the device; the stack
 * stays n_cameras x slot. */
int ekf_batch_set_frame_sizes(ekf_batch* b, const int32_t* wh);
/* captureNewFrame for every camera: a stack of n_cameras frames, frame c at img + c * height * stride (the layout of
 * ekf_match_batch), gray from HOST / DEVICE memory or BGR from HOST memory.  stamps: n_cameras doubles or NULL; camera c
 * applies the single filter's rule to stamps[c] (>= 0: dT = stamp - old_ts once old_ts > 0).  Resize and colour conversion
 * are ekf_batch_capture_frame*'s, frame by frame; host frames that need them are staged a chunk of cameras at a time. */
int ekf_batch_capture_frames(ekf_batch* b, const uint8_t* gray, int width, int height, int stride, const double* stamps);
int ekf_batch_capture_frames_device(ekf_batch* b, const uint8_t* gray_dev, int width, int height, int stride, const double* stamps);
int ekf_batch_capture_frames_bgr(ekf_batch* b, const uint8_t* bgr, int width, int height, int stride, const double* stamps);
/* captureNewFrame for the listed cameras only: frame k of the stack (img + k * height * stride) is camera cameras[k]'s, and
 * stamps (n entries or NULL) follow the same order.  Cameras that are not listed keep their frame, time stamp and dT.
 * cameras holds 1 <= n distinct cameras in [0, n_cameras), in any order; else EKF_ERR_ARG and nothing changes.
 * Each camera has a frame from the capture that last listed it (a capture of every camera lists all); ekf_batch_set_cameras
 * and ekf_batch_set_frame_sizes forget every frame.  The frames go into the stack's slots: the first capture after the
 * frames were forgotten defines the slot (width / scale x height / scale), and the other cameras stay without a frame; while
 * some camera holds a frame, a call whose resized slot (or frame sizes) differs returns EKF_ERR_ARG, and only a capture of
 * every camera may change it.  Scale, BGR input and frame sizes act camera by camera as in a capture of every camera, and
 * a listed camera's frame is bit-identical to the one such a capture of the same image produces (its pads zeroed).  Each
 * listed camera applies the single filter's stamp rule, so a camera captured twice between steps of its filters has the
 * last interval.  Host frames go up in one copy per staging chunk, device frames are read in place, and one launch places
 * (and resizes) the listed frames. */
int ekf_batch_capture_camera_frames(ekf_batch* b, int n, const int32_t* cameras, const uint8_t* gray, int width, int height,
                                    int stride, const double* stamps);
int ekf_batch_capture_camera_frames_device(ekf_batch* b, int n, const int32_t* cameras, const uint8_t* gray_dev, int width,
                                           int height, int stride, const double* stamps);
int ekf_batch_capture_camera_frames_bgr(ekf_batch* b, int n, const int32_t* cameras, const uint8_t* bgr, int width, int height,
                                        int stride, const double* stamps);
/* returnGrayImg for one camera (out may be NULL to query the size); EKF_ERR_ARG for a bad camera, EKF_ERR_STATE while the
 * camera holds no frame. */
int ekf_batch_get_camera_frame(ekf_batch* b, int camera, uint8_t* out, int* width, int* height);
/* getDt for every filter (HOST array of n_filters): its camera's dT. */
int ekf_batch_get_dt(ekf_batch* b, double* out);
/* Device scratch of one chunk of cameras in the batched detector with several cameras (about 44 bytes a pixel a camera;
 * default 1 GiB, at least one camera a chunk).  Cameras no filter asks corners from cost nothing.  EKF_ERR_ARG below 1. */
int ekf_batch_set_detect_budget(ekf_batch* b, int64_t bytes);
/* ekf_config.scale for the batch's captures (1 to 64, the range ekf_create accepts; default 1).  As for a single filter,
 * the intrinsics of the batch's configuration must be those of the resized image (ConfigVSLAM.cpp:89-120). */
int ekf_batch_set_scale(ekf_batch* b, int32_t scale);
/* ekf_config.forsePlane for every filter (default 0): the second update of each step carries the pseudo-measurements
 * mu[1] = mu[4] = mu[6] = 0 with R = 1e-5 I3 (vslamRansac.cpp:1245-1272) and runs even without high-innovation rows.
 * EKF_BSTAT_HI still counts the rescued features only. */
int ekf_batch_set_force_plane(ekf_batch* b, int on);
/* predict + update (match, 1-point RANSAC, both corrections, book-keeping, feature deletion, top-up if
 * switched on, XYZ conversion if cfg.xyz_conversion) for every filter.  dv / dw / vcontrol as ekf_predict; picks as ekf_update (every filter draws from the
 * same sequence).  Returns after the per-filter counters have reached the host. */
int ekf_batch_step(ekf_batch* b, const double dv[3], const double dw[3], int vcontrol, const uint32_t* picks, int n_picks);
/* ekf_batch_step with controls per filter: dv and dw n_filters x 3 doubles, vcontrol n_filters int32 (HOST arrays; any may be
 * NULL, meaning zeros).  picks stay shared. */
int ekf_batch_step_controls(ekf_batch* b, const double* dv, const double* dw, const int32_t* vcontrol, const uint32_t* picks,
                            int n_picks);
/* ekf_batch_step_controls for the listed filters only.  filters: 1 <= n filters, strictly ascending in [0, n_filters), else
 * EKF_ERR_ARG and nothing changes.  dv / dw are n x 3 and vcontrol is n, in list order (any may be NULL, meaning zeros).  The
 * picks are shared, as in ekf_batch_step.  Each listed filter runs exactly what ekf_batch_step_controls runs for it: predict
 * (with blur if on), match, both updates, removals and archive, top-up if on, and XYZ conversion.  Every other filter stays
 * bit-identical: state, covariance, feature table, both templates, archive and its overflow count, real_index counter.
 * After the call ekf_batch_get_camera_states reports every filter's camera state and block as it stands; the counters
 * (EKF_BSTAT_*), ekf_batch_last_added and ekf_batch_last_blur_counts are zero for the filters not listed, so
 * ekf_batch_find_new_features(NULL) adds nothing to them.  EKF_ERR_STATE when a listed filter's camera holds no frame (as
 * ekf_batch_step / ekf_batch_step_controls for any filter's).  The per-filter kernels run on the listed filters only, so the
 * step's cost follows the list. */
int ekf_batch_step_filters(ekf_batch* b, int n, const int32_t* filters, const double* dv, const double* dw,
                           const int32_t* vcontrol, const uint32_t* picks, int n_picks);
/* convert2XYZ_ifLinearAll (vslamRansac.cpp:776-780) on every filter of the batch. */
int ekf_batch_convert2xyz_if_linear_all(ekf_batch* b);
/* Results of the last step, HOST output arrays: camera state (n_filters x 14), 14 x 14 covariance
 * block (n_filters x 196, may be NULL), counters (n_filters x EKF_BATCH_STAT_FIELDS, may be NULL). */
int ekf_batch_get_camera_states(ekf_batch* b, double* mu14, double* sigma14, int32_t* stats);
/* Single-filter views for parity tests and checkpointing. */
int ekf_batch_num_features(ekf_batch* b, int filter);
int ekf_batch_state_dim(ekf_batch* b, int filter);
int ekf_batch_get_full(ekf_batch* b, int filter, double* mu, double* sigma, int ld);
int ekf_batch_set_full(ekf_batch* b, int filter, const double* mu, const double* sigma, int ld);
int ekf_batch_get_feature(ekf_batch* b, int filter, int idx, ekf_feature_info* out);
/* VSlamFilter::addFeature (vslamRansac.cpp:309-371) on one filter of the batch: returns 1 added, 0 rejected by
 * isInsideImage, EKF_ERR_CAPACITY when the filter is full, EKF_ERR_STATE while the filter's camera holds no frame or before
 * seeding.  The new
 * feature's real_index comes from the filter's own counter (seeded from the source filter's), as in ekf_add_feature. */
int ekf_batch_add_feature(ekf_batch* b, int filter, float u, float v);
/* findNewFeatures' detection alone (vslamRansac.cpp:783-831) for every filter: its own mask around its own patches, its
 * camera's frame.  num: HOST array of n_filters entries; filter b gets up to min(num[b], EKF_BATCH_MAX_CORNERS) corners
 * (none when num[b] <= 0), as (x, y) pairs in out_xy (n_filters x EKF_BATCH_MAX_CORNERS x 2 floats), their count in
 * out_n (n_filters).  Each filter's list equals ekf_detect_corners on a single filter holding the same patch centres.
 * EKF_ERR_STATE when a filter that asks for corners follows a camera that holds no frame (here and in
 * ekf_batch_find_new_features). */
#define EKF_BATCH_MAX_CORNERS 32
int ekf_batch_detect_corners(ekf_batch* b, const int32_t* num, float* out_xy, int32_t* out_n);
/* VSlamFilter::findNewFeatures(num[b]) (vslamRansac.cpp:783-839) on every filter in one call: detection as above, then
 * addFeature on each corner in order until the filter is full.  Unlike the single filter, where num <= 0 means
 * nInitFeatures, num[b] <= 0 means filter b adds nothing.  num == NULL takes each filter's EKF_BSTAT_TOPUP of the last
 * step (EKF_ERR_STATE without a completed step).  added (n_filters, may be NULL) receives the features each filter added.
 * Returns the total added over the batch, or an error. */
int ekf_batch_find_new_features(ekf_batch* b, const int32_t* num, int32_t* added);
/* on != 0: ekf_batch_step ends like ekf_update_after_match, with removals, then findNewFeatures(EKF_BSTAT_TOPUP) on
 * every filter that asks, then the XYZ conversions.  Default 0 (the step reports the request and adds nothing). */
int ekf_batch_set_topup(ekf_batch* b, int on);
/* Features each filter added in the last step (n_filters entries; zeros with top-up off). */
int ekf_batch_last_added(ekf_batch* b, int32_t* added);
/* Patch::blur (Patch.cpp:50-57, libblur.cpp:17-81) in every filter's predict: kernel_size has the meaning of
 * ekf_config.kernel_size for a single filter (a template is blurred when the prediction moves by more than kernel_size px
 * over T_camera * dT; >= 100000 = off, the default).  ekf_batch_create still refuses a configuration with blur on.
 * T_camera is the filter's (ekf_batch_set_filter_params; the configuration's by default).  A kernel above 256 x 256 px leaves that template unblurred; the step then runs
 * to its end and returns EKF_ERR_UNSUPPORTED, and ekf_batch_last_error names the first such filter. */
int ekf_batch_set_motion_blur(ekf_batch* b, int32_t kernel_size);
/* Templates each filter blurred in the last step (n_filters entries; zeros with blur off). */
int ekf_batch_last_blur_counts(ekf_batch* b, int32_t* out);
/* The feature archive of every filter (VSlamFilter::deleted_patches, vslamRansac.cpp:394-404), off by default.
 * capacity > 0 turns it on with room for `capacity` records per filter and empties every filter's archive; 0 turns it off.
 * Device memory: n_filters x capacity x 100 bytes (real_index + 12 doubles), e.g. 4096 filters x 7001 records = 2.9 GB.  The
 * reference keeps its archive bounded only through the export's clear rule (more than 7000 records are cleared), so a capacity of
 * at least 7001 lets an exporting caller never run out.  With the archive on, every removal (the step's quality deletions in
 * ascending index, then its max_features removeFeature(0), and ekf_batch_remove_feature) archives each XYZ feature with
 * n_find > 5, as ekf_get_deleted reports them for a single filter.  When a filter's archive is full its record is dropped: the
 * step (or removal) still runs to its end, then returns EKF_ERR_CAPACITY and ekf_batch_last_error names the first filter that
 * dropped one.  ekf_batch_seed_from copies the source's archive into every filter (EKF_ERR_CAPACITY if it holds more than
 * capacity records).  EKF_ERR_ARG for a negative capacity. */
int ekf_batch_set_archive(ekf_batch* b, int32_t capacity);
/* VSlamFilter::removeFeature (vslamRansac.cpp:373-421) on feature `index` of one filter, on the device: exactly that feature
 * goes (archived under the rule above), without the step's max_features rule.  EKF_ERR_ARG for a bad filter or index,
 * EKF_ERR_STATE before seeding. */
int ekf_batch_remove_feature(ekf_batch* b, int filter, int index);
/* Records in each filter's archive (counts: n_filters entries; zeros with the archive off). */
int ekf_batch_num_deleted(ekf_batch* b, int32_t* counts);
/* One filter's archive in archive order, in ekf_get_deleted's layout: *n receives the record count, and the first
 * min(*n, cap) records go to out (which may be NULL with cap = 0 to query the count). */
int ekf_batch_get_deleted(ekf_batch* b, int filter, ekf_deleted_info* out, int cap, int* n);
/* ekf_get_points_features (RosVSLAM::getPointsFeatures, RosVSLAMRansac.cpp:340-418) for filters [first, first + count) in one
 * launch.  rows[k] receives filter first + k's row count (real_index of its last live feature + 1, or 1 without features).
 * out holds count x rows_cap x 12 doubles: filter first + k's matrix starts at out + k * rows_cap * 12, and its rows past rows[k]
 * are zero.  out == NULL only queries rows; EKF_ERR_ARG when rows_cap is below the largest row count.  Rows as for a single
 * filter: live XYZ features write position * map_scale and their 3 x 3 block, inverse-depth rows stay zero, then archived
 * records overwrite theirs in archive order (position * the filter's current map_scale = mu[13]; records past the last live
 * real_index are dropped).  After the export every exported filter whose archive holds more than 7000 records has it cleared. */
int ekf_batch_get_points_features(ekf_batch* b, int first, int count, double* out, int rows_cap, int32_t* rows);
/* Resampling of a multi-hypothesis ensemble: filter f becomes an exact copy of filter ancestors[f] (HOST array of n_filters
 * entries), both as they stood before the call, so duplicates, swaps and cycles are all fine; ancestors[f] == f leaves f
 * untouched, and the identity launches nothing.  What moves is everything of the filter that a later call reads: state and
 * covariance, feature table, both templates, real_index counter, pending XYZ decisions, archive (with its overflow count,
 * so the next step reports only new drops), intrinsics row (ekf_batch_set_intrinsics), tuning row
 * (ekf_batch_set_filter_params), counters, added and blur counts.
 * Afterwards every per-filter accessor reports for f what it reported for ancestors[f] before the call: ekf_batch_get_full,
 * _get_feature, _get_template, _num_features, _state_dim, _get_camera_states (camera rows and counters), _last_added,
 * _last_blur_counts, _num_deleted, _get_deleted and _get_points_features; and every later call treats f as it treats its
 * ancestor (a step that gives f its ancestor's controls produces its ancestor's bits).  ancestors[f] must lie in
 * [0, n_filters) and follow f's camera (a hypothesis maps one camera's scene); otherwise EKF_ERR_ARG, ekf_batch_last_error
 * names the first bad entry and nothing changes.  EKF_ERR_ARG for NULL, EKF_ERR_STATE before seeding; no frame is needed.
 * A source that is itself overwritten is staged first (its covariance in the compaction scratch, the rest in a temporary
 * buffer), which costs one more read and write of it; a vector from systematic resampling that keeps every drawn filter in
 * its own slot never needs that.  Returns once the copy is done. */
int ekf_batch_resample(ekf_batch* b, const int32_t* ancestors);
/* which: 0 = Patch::patch, 1 = Patch::matching_patch of feature idx of one filter; out holds window_size^2 bytes (the window of
 * the filter's camera, ekf_batch_set_camera_settings) */
int ekf_batch_get_template(ekf_batch* b, int filter, int idx, int which, uint8_t* out);
/* Kernels of this library launched on the batch so far. */
int64_t ekf_batch_kernel_launches(const ekf_batch* b);
/* CUDA-event time (ms) of the three kernel classes of the last step: predict, match, update. */
int ekf_batch_last_step_ms(ekf_batch* b, float out[3]);
/* Matcher of the last step: number of (filter, feature) pairs whose search window did not fit the warp-per-feature path
 * (candidate grid > 16 x 16 or template side > 15) and were matched by the CTA-per-feature kernel instead.  Diagnostic. */
int ekf_batch_last_match_deferred(ekf_batch* b);

/* ---- large map split across GPUs (BASELINE config 4) ------------------------------------------- */
/* One process per GPU, each with its own ekf_handle holding a replica of the same filter (same calls
 * in the same order on every rank).  Once attached, the stacked EKF update — W = Sigma H^T, gain,
 * Sigma -= V V^T, > 95 % of a large-map step — is partitioned by covariance ROW BLOCKS: rank r updates
 * rows [r * rpr, (r + 1) * rpr) only, and NCCL (all-gather over NVLink / NVSwitch) carries the W_b /
 * V_b panels (n x 128 fp64 per 64 features), the state correction and, once per update, the row
 * blocks of Sigma.  Everything else (predict, match, RANSAC, book-keeping) is O(n) or O(N) work that
 * every rank repeats on its replica.  libnccl is opened at run time: pass the path of the library the
 * host already uses (NULL = "libnccl.so.2").  The 128-byte id comes from ekf_dist_unique_id on one
 * rank and is distributed by the host (the Python host broadcasts it with torch.distributed). */
int ekf_dist_load_nccl(const char* libnccl_path);
int ekf_dist_unique_id(char out[128]);
int ekf_dist_attach(ekf_handle* h, const char id[128], int rank, int world);
int ekf_dist_detach(ekf_handle* h);
int ekf_dist_info(const ekf_handle* h, int* rank, int* world, int64_t* allgather_bytes);
/* 1 when the panels of the partitioned look-ahead update travel by peer-memory stores from inside the producing kernels
 * (CUDA IPC mappings set up by ekf_dist_attach; EKF_DIST_P2P=0 or a failed mapping keeps the NCCL collectives), else 0. */
int ekf_dist_peer_memory(const ekf_handle* h);

/* ---- per-kernel timing (CUDA events on the handle's stream; off by default) ---------------------- */
#define EKF_PROF_CLASSES 12
typedef struct ekf_profile {
  /* classes: 0 predict_cov+features, 1 match, 2 ransac, 3 gather W, 4 factor S, 5 V=W L^-T,
   * 6 downdate GEMM (DMMA), 7 quat normalise, 8 hi rescue, 9 bookkeeping, 10 add/remove, 11 NCCL all-gathers */
  double ms[EKF_PROF_CLASSES];
  int64_t launches[EKF_PROF_CLASSES];
} ekf_profile;
/* on != 0: bracket every kernel class with CUDA events; totals accumulate until read. */
int ekf_set_profiling(ekf_handle* h, int on);
/* Copies the accumulated totals and, if reset != 0, clears them. */
int ekf_get_profile(ekf_handle* h, ekf_profile* out, int reset);
/* 0 = full-square downdate; 1 = lower-triangle tiles + mirrored store (Sigma is symmetrised). */
int ekf_set_symmetric_downdate(ekf_handle* h, int on);
/* Diagnostic (bench.py's roofline object): launches the covariance downdate of one 128-row block `reps` times ALONE on the
 * filter's stream — Sigma -= V V^T with the panel of the last update as V, negated on alternate launches so that Sigma ends where it
 * started up to rounding — and returns the mean launch duration measured with CUDA events.  Changes Sigma by rounding errors: call
 * it on a filter that is not used afterwards. */
int ekf_debug_time_downdate(ekf_handle* h, int reps, float* ms_per_launch);

/* Library version / build info: returns a static string naming the compiled arch. */
const char* ekf_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* EKF_B200_H_ */
