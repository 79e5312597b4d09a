// csrc/ekf_kernels.h — host-side launch wrappers of the kernels in ekf_*.cu (internal to libekf_b200).
#pragma once
#include "ekf_common.cuh"
#include "ekf_detect.cuh"

#define EKF_UB 128  // rows per update block (64 features): K of the rank-b downdate GEMM

// ekf_predict.cu
void launch_predict(cudaStream_t st, double* Sigma, int ld, int n, double* mu, FeatTab ft, int N, FrameView fr,
                    DevCtl* ctl, const DevCfg& cfg, double dT, const double dv[3], const double dw[3], int vcontrol,
                    long long* launches);
void launch_finish_update(cudaStream_t st, double* Sigma, int ld, int n, double* mu, const double* delta, DevCtl* ctl,
                          long long* launches);
void launch_add_feature(cudaStream_t st, double* Sigma, int ld, int n, double* mu, FeatTab ft, int fidx, FrameView fr,
                        const DevCfg& cfg, float pfx, float pfy, int real_index, long long* launches);
void launch_gather_state(cudaStream_t st, const double* Ssrc, double* Sdst, int ld, const double* musrc, double* mudst,
                         int n2, const int* map, long long* launches);
void launch_gather_features(cudaStream_t st, FeatTab src, FeatTab dst, int N2, const int* keep, const int* newpos, int w2,
                            long long* launches);
void launch_xyz_decide(cudaStream_t st, const double* Sigma, int ld, const double* mu, FeatTab ft, int N, const DevCfg& cfg, int only,
                       int* flag, double* y, double* J, long long* launches);
void launch_xyz_apply(cudaStream_t st, const double* Ssrc, double* Sdst, int ld, const double* musrc, double* mudst, int n2,
                      const int* rmap, const double* J, const double* y, FeatTab ft, int N, const int* pos, const int* coding,
                      long long* launches);
// ekf_match.cu
// A TMA tensor map (CUtensorMap, 128 bytes) of a stack of u8 frames for the matcher's window staging, kept opaque here so that
// only ekf_match.cu needs the driver header.  ok == 0: the frames cannot be described (base or row stride not 16-byte aligned,
// driver entry point unavailable): the kernels then stage the window with ordinary loads.
struct alignas(64) EkfTensorMap {
  unsigned long long opaque[16];
  int ok;
};
void match_make_tensor_map(EkfTensorMap* out, const uint8_t* frames, int width, int height, int stride, int n_frames, int w, int clamp);
void launch_match_filter(cudaStream_t st, FeatTab ft, int N, FrameView fr, const DevCfg& cfg, const EkfTensorMap* tmap, long long* launches);
void launch_match_filter_batch(cudaStream_t st, FeatTab base, int Ncap, const int* Nper, int B, FrameView fr, const DevCfg& cfg,
                               const EkfTensorMap* tmap, int* defer_list, int* defer_cnt, long long* launches,
                               const int* cam_of = nullptr,    // cam_of [B]: filter b searches frame cam_of[b] of the stack fr
                               const int* fsize = nullptr,     // [n_cameras][4] (in w, in h, w, h): camera c is the top-left w x h of its slot
                               const int* act = nullptr);      // [B]: the pairs' filter i is filter act[i] (a list of B filters)
int launch_match_batch(cudaStream_t st, const uint8_t* frames, int n_frames, int width, int height, int stride,
                       const uint8_t* templates, int fpf, int w, const double* h, const double* S, float sigma_size,
                       float thr, float clampv, int32_t* out_uv, float* out_score);
// ekf_update.cu
int update_kernels_init();
void launch_ransac(cudaStream_t st, const double* Sigma, int ld, int n, const double* mu, FeatTab ft, int N, DevCtl* ctl,
                   const DevCfg& cfg, const uint32_t* picks, int n_picks, double* mu_i, int* cand, long long* launches);
void launch_hi_rescue(cudaStream_t st, const double* Sigma, int ld, const double* mu, FeatTab ft, int N, DevCtl* ctl,
                      const DevCfg& cfg, long long* launches, double* outd = nullptr, int* outi = nullptr);
void launch_blk_gather(cudaStream_t st, const double* Sigma, int ld, int row0, int row1, FeatTab ft, int f0, int cnt,
                       const double* delta, double* W, double* nu, long long* launches);
void launch_blk_factor(cudaStream_t st, const double* W, FeatTab ft, int f0, int cnt, const double* nu, const DevCfg& cfg,
                       double* Sb, double* Lb, double* Dblk, double* yb, DevCtl* ctl, long long* launches);
void launch_blk_S_nu(cudaStream_t st, const double* W, FeatTab ft, int f0, int cnt, const DevCfg& cfg, const double* delta,
                     double* Sb, double* nu, long long* launches);
void launch_blk_S_nu_G(cudaStream_t st, const double* Wraw, FeatTab ft, int f0, int cnt, const DevCfg& cfg, const double* delta,
                       const double* G, double* Sb, double* nu, long long* launches, const double* gy = nullptr,
                       BlkTab bt = BlkTab{nullptr, nullptr, nullptr, nullptr}, const double* Sg = nullptr, unsigned int* pub_ticket = nullptr,
                       unsigned int* pub_flag = nullptr, unsigned int pub_token = 0, const double* Sg2 = nullptr);
void launch_blk_gather_hot(cudaStream_t st, const double* Sigma, int ld, int n, FeatTab ft, int f0, int cnt, double* W, long long* launches, BlkTab bt,
                           const int* cnt_dev = nullptr);
void launch_blk_Sg(cudaStream_t st, const double* G, double* Sg, long long* launches, unsigned int* pub_ticket = nullptr,
                   unsigned int* pub_flag = nullptr, unsigned int pub_token = 0);
void launch_blk_prep(cudaStream_t st, FeatTab ft, int cnt, double* H, double* zmh, int* pos, int* nd, long long* launches,
                     const int* cnt_dev = nullptr);
// per update block g: the 64 x 64 tiles of the lower triangle (T x T tiles) ordered with the tiles gather g reads first; n_hot[g] of them
void launch_blk_tile_order(cudaStream_t st, FeatTab ft, int cnt, int T, ushort2* order, int* n_hot, unsigned int* hot_counters, long long* launches);
// the gather of block f0 / 64 started BESIDE the downdate that produces its columns: waits until hot_counter reaches *n_hot
void launch_blk_gather2_after_tiles(cudaStream_t st, const double* Sigma, int ld, int n, FeatTab ft, int f0, int cnt, double* W, double* W2,
                                    const unsigned int* hot_counter, const int* n_hot, DevCtl* ctl, long long* launches,
                                    BlkTab bt = BlkTab{nullptr, nullptr, nullptr, nullptr});
void launch_blk_Gx(cudaStream_t st, const double* Wc, FeatTab ft, int f0, int cnt, const double* Lb, const double* Dblk, const double* yb,
                   double* G, double* gy, long long* launches, BlkTab bt = BlkTab{nullptr, nullptr, nullptr, nullptr}, const unsigned int* wait_flag = nullptr,
                   unsigned int wait_token = 0, DevCtl* ctl = nullptr);
// arguments of k_chain_factor (ekf_update.cu), filled by stacked_update_resident_chain
struct ChainFactorArgs {
  const double* S;          // S_b (lower 32 x 32 blocks), written by k_blk_S_tiled
  const double* nu;
  double* L[2];             // factor outputs, block b -> set b & 1
  double* D[2];
  double* y[2];
  ChainFlags fl;
  int nblk;
};
void launch_chain_factor(cudaStream_t st, const ChainFactorArgs& a, DevCtl* ctl, long long* launches);
void launch_wait_flag(cudaStream_t st, const unsigned int* flag, unsigned int token, DevCtl* ctl, long long* launches);
void launch_blk_gather2(cudaStream_t st, const double* Sigma, int ld, int n, FeatTab ft, int f0, int cnt, double* W, double* W2,
                        long long* launches, BlkTab bt = BlkTab{nullptr, nullptr, nullptr, nullptr}, const int* cnt_dev = nullptr, unsigned int* pub_ticket = nullptr,
                        unsigned int* pub_flag = nullptr, unsigned int pub_token = 0);
void launch_blk_G(cudaStream_t st, const double* Vprev, FeatTab ft, int f0, int cnt, double* G, long long* launches);
void launch_blk_factor_only(cudaStream_t st, const double* Sb, const double* nu, double* Lb, double* Dblk, double* yb, DevCtl* ctl,
                            long long* launches);
void launch_blk_factor_wait(cudaStream_t st, const double* Sb, const double* nu, double* Lb, double* Dblk, double* yb, DevCtl* ctl,
                            const unsigned int* flag, unsigned int token, long long* launches);
void launch_plane_gather(cudaStream_t st, const double* Sigma, int ld, int row0, int row1, const double* mu, const double* delta,
                         double* W, double* nu, DevCtl* ctl, long long* launches);
void launch_plane_S(cudaStream_t st, const double* W, double* Sb, long long* launches);
void launch_blk_V(cudaStream_t st, double* W, int row0, int row1, const double* Lb, const double* Dblk, const double* yb,
                  double* delta, long long* launches, double* Vout = nullptr, const double* delta_in = nullptr);
void launch_blk_S_part(cudaStream_t st, const double* W, FeatTab ft, int f0, int cnt, const DevCfg& cfg, int row0, int row1, int add_diag,
                       const double* delta, double* nu, double* Sb, long long* launches);
void launch_blk_S_part_p2p(cudaStream_t st, const double* W, FeatTab ft, int f0, int cnt, const DevCfg& cfg, int row0, int row1, int add_diag,
                           const double* delta, double* nu, double* Sb, const P2PView& pv, unsigned int* ticket, long long* launches);
void launch_blk_factor_p2p(cudaStream_t st, const double* spart, const unsigned long long* flags, int world, unsigned long long epoch,
                           double* Ssum, const double* nu, double* Lb, double* Dblk, double* yb, DevCtl* ctl, long long* launches);
void launch_blk_V_p2p(cudaStream_t st, double* W, int row0, int row1, const double* Lb, const double* Dblk, const double* yb,
                      const P2PView& pv, unsigned int* ticket, const unsigned long long* flags, int world, unsigned long long epoch,
                      DevCtl* ctl, long long* launches);
void launch_delta_rows(cudaStream_t st, const double* V, const double* y, double* delta, int n, long long* launches);
void launch_bookkeeping(cudaStream_t st, const double* Sigma, int ld, const double* mu, FeatTab ft, int N, DevCtl* ctl,
                        const DevCfg& cfg, double* outd, int* outi, long long* launches);
// ekf_export.cu
void launch_points_features(cudaStream_t st, const double* Sigma, int ld, const double* mu, FeatTab ft, int N, double* out, int rows,
                            long long* launches);
void launch_rts_epoch(cudaStream_t st, double* io, const DevCfg& cfg, double dT, int* singular, long long* launches);
// ekf_gemm.cu
int launch_gemm_nt_sub(cudaStream_t st, double* C, int ldc, const double* A, int lda, const double* B, int ldb, int M, int N,
                       int kconst, const int* kdev, int lower_only, int* counters, long long* launches,
                       const ushort2* tlist = nullptr, int n_tiles = 0, const int* n_hot = nullptr, unsigned int* hot_counter = nullptr);
bool gemm_uses_square_tiles();
int gemm_kernels_preload();
// ekf_detect.cu
int launch_detect_corners(cudaStream_t st, FrameView fr, FeatTab ft, int N, int window, uint8_t* mask, float* eig,
                          unsigned long long* keys, int key_cap, int* counters, int max_corners, float* out_xy, long long* launches);
// the min-eigenvalue map of goodFeaturesToTrack for a whole frame (k_det_eig)
void launch_det_eig(cudaStream_t st, FrameView fr, float* eig, long long* launches);
void launch_capture_resize_gray(cudaStream_t st, const uint8_t* src, int sw, int sh, int sstride, int cn, uint8_t* dst, int dw, int dh,
                                int dstride, long long* launches, int n_frames = 1,    // n_frames: a contiguous stack, frame z in blockIdx.z
                                const int* fsize = nullptr,    // [n_frames][4]: frame z resizes its top-left fsize[0..1] to fsize[2..3]
                                const int* slot = nullptr);    // [n_frames]: frame z goes to slot slot[z] of dst (and reads fsize row slot[z])
// ekf_batch_detect.cu: findNewFeatures' detection for every filter of a batch (one frame, per-filter masks)
struct BatchDetectBufs {
  float* eig = nullptr;                 // [cap] min-eigenvalue map
  unsigned long long* keys = nullptr;   // [4][cap] pixel keys, candidate keys, both sorted
  void* tmp = nullptr;                  // CUB radix-sort workspace
  size_t tmp_bytes = 0, cap = 0;        // cap: pixels the buffers hold
  DetBox* boxes = nullptr;              // [B][cstride] mask boxes per filter
  unsigned* thr_bits = nullptr;         // [B] per-filter threshold (float bits)
  int* limit = nullptr;                 // [B] corners each filter may take
  int* offs = nullptr;                  // [offs_chunk + 1] segment offsets s * offs_npx of the per-camera sorts
  int offs_chunk = 0;
  size_t offs_npx = 0;
};
cudaError_t batch_detect_reserve(BatchDetectBufs& d, size_t px, int B, int cstride);
void batch_detect_free(BatchDetectBufs& d);
// num[b * num_stride] corners for filter b, capped at EKF_BATCH_MAX_CORNERS (cap_mode 0) or at Ncap - N[b] (cap_mode 1), and at
// cstride, the boxes and corners a filter has room for: EKF_BATCH_MAX_CORNERS, or EKF_BATCH_MAX_FEATURES for a large batch;
// out_xy [B][cstride][2], out_n [B]
cudaError_t launch_batch_detect(cudaStream_t st, BatchDetectBufs& d, FrameView fr, const float* centers, const int* N, int Ncap, int B,
                                int window, const int* num, int num_stride, int cap_mode, int cstride, float* out_xy, int* out_n,
                                long long* launches);
// Per camera (ekf_batch_set_cameras): the frames of the n_req cameras listed in HOST cams, frame c at fr.px + c * fr.h * fr.stride,
// in chunks of `chunk` cameras (scratch from batch_detect_reserve_cams); filter b walks the segment of camera cam_of[b], whose
// position in cams is slot_of_cam[cam_of[b]] (-1: nobody asks from it; the filter finds nothing).  Same outputs as above.
cudaError_t batch_detect_reserve_cams(BatchDetectBufs& d, size_t npx, int chunk, int B, int cstride);
cudaError_t launch_batch_detect_cams(cudaStream_t st, BatchDetectBufs& d, FrameView fr, const int* cams, int n_req, int chunk,
                                     const int* cam_of, const int* slot_of_cam, const float* centers, const int* N, int Ncap, int B,
                                     int window, const int* num, int num_stride, int cap_mode, int cstride, float* out_xy, int* out_n,
                                     long long* launches, const int* fsize = nullptr, const int* fsize_host = nullptr,
                                     const int* seg_cam = nullptr);   // per-camera sizes (device / host [n_cameras][4]); seg_cam: cams on the device
