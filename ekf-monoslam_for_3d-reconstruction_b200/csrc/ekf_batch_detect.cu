// csrc/ekf_batch_detect.cu — findNewFeatures' detection (vslamRansac.cpp:783-831) for every filter of a batch at once.
//
// All filters see one frame, so the min-eigenvalue map (k_det_eig) is computed once per call.  What differs per filter is
// the mask (the base border minus a box around each of the filter's patches) and with it the threshold
// thr_b = 0.01 * max(eig over mask_b).  The single filter's candidates are the pixels p that
//   (1) lie in rows / columns 1 .. size-2 and are 3x3 local maxima of THRESH_TOZERO(eig, thr_b),
//   (2) have eig[p] > thr_b, and (3) are set in mask_b.
// Given (2), (1) is the same as "no raw neighbour exceeds eig[p]": a neighbour above eig[p] is above thr_b and survives the
// threshold, one at or below eig[p] cannot beat it whether zeroed or not.  So (1) does not depend on the filter, and one
// list of every local maximum with eig > 0 inside the base mask, sorted once by the single filter's key (score bits << 32 |
// pixel index), holds every filter's candidates as a subsequence in the same order.  Each filter then walks that list
// (det_select_walk), skipping its boxes and stopping at its threshold or its corner limit.  The list is dense (one slot per
// pixel, zero where there is no candidate), so it can never be truncated and its length is known on the host.
//
// The masked maximum must be exact: the frame's pixel keys (base mask, eig > 0) are sorted once, and one warp per filter
// walks down that order until the first pixel outside the filter's boxes.  The walk is long only as far as the top pixels
// sit inside the filter's own boxes (at most N (2 w + 1)^2 pixels, N <= 32, or <= 128 in a large batch).
//
// Early stop: every pixel inside the mask is at least window_size from the border, more than the window_size / 2 of
// isInsideImage, so addFeature accepts every detected corner and the single filter's loop over them (V:832-835) stops only
// on its capacity: taking min(num_b, Ncap - N_b) corners is exactly what it adds.
//
// Cameras (ekf_batch_set_cameras): the argument holds per frame, so each camera that at least one filter asks corners from
// gets its own eig map, keys and sorted lists (one segment of npx slots), and each filter walks its camera's segment.  The
// cameras asked from are processed in chunks whose scratch (44 bytes a pixel a camera, the sort's workspace included) fits a fixed
// budget and whose C * npx keys stay within int range; a segmented radix
// sort orders every segment of a chunk by the same key, so each camera's order is exactly the single filter's.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include <vector>

#include "../../include/ekf_b200.h"
#include "ekf_detect.cuh"
#include "ekf_kernels.h"

// pixel keys (base mask, eig > 0) and candidate keys (those that are also raw 3x3 local maxima), one slot per pixel
// (blockIdx.z: the camera's segment of a chunk)
// fsize (ekf_batch_set_frame_sizes): segment z holds camera seg_cam[z] of fsize[4c + 2] x fsize[4c + 3] pixels, packed at the
// segment's start with that width; the segment's other slots get no key.
__global__ void k_bdet_keys(const float* __restrict__ eig, int W, int H, int estrem, unsigned long long* __restrict__ kp,
                            unsigned long long* __restrict__ kc, const int* __restrict__ fsize, const int* __restrict__ seg_cam) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= W) return;
  const size_t seg = (size_t)blockIdx.z * W * H;
  eig += seg; kp += seg; kc += seg;
  if (fsize) {
    const int j = y * W + x, c = seg_cam[blockIdx.z], wc = fsize[4 * c + 2], hc = fsize[4 * c + 3];
    if (j >= wc * hc) { kp[j] = 0ull; kc[j] = 0ull; return; }
    W = wc; H = hc; x = j % wc; y = j / wc;
  }
  const size_t i = (size_t)y * W + x;
  const float v = eig[i];
  unsigned long long p = 0ull, c = 0ull;
  if (v > 0.0f && det_in_base(x, y, W, H, estrem)) {
    p = det_key(__float_as_uint(v), (unsigned)i);
    if (x >= 1 && x < W - 1 && y >= 1 && y < H - 1) {
      bool mx = true;
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) mx = mx && !(eig[(size_t)(y + dy) * W + x + dx] > v);
      if (mx) c = p;
    }
  }
  kp[i] = p;
  kc[i] = c;
}

// Segment of filter b in a chunk of cameras: cam_of == nullptr (one camera) gives segment 0 for every filter; otherwise filter b
// belongs to the chunk when its camera's slot among the cameras asked from lies in [lo, hi), and -1 is returned when it does not.
__device__ __forceinline__ int bdet_segment(const int* __restrict__ cam_of, const int* __restrict__ slot_of_cam, int lo, int hi, int b) {
  if (!cam_of) return 0;
  const int s = slot_of_cam[cam_of[b]];
  return (s >= lo && s < hi) ? s - lo : -1;
}

// One warp per filter: its boxes, its corner limit and thr_b from the first sorted pixel outside its boxes.  CS: boxes and
// corners a filter has room for (EKF_BATCH_MAX_CORNERS, or EKF_BATCH_MAX_FEATURES in a large batch).
#define BDET_WARPS 8
template <int CS>
__global__ void __launch_bounds__(32 * BDET_WARPS) k_bdet_threshold(const unsigned long long* __restrict__ kp, int npx, int W, int H,
                                                                     int window, const float* __restrict__ centers,
                                                                     const int* __restrict__ N, int Ncap, int B,
                                                                     const int* __restrict__ num, int num_stride, int cap_mode,
                                                                     DetBox* __restrict__ boxes, unsigned* __restrict__ thr_bits,
                                                                     int* __restrict__ limit, const int* __restrict__ cam_of,
                                                                     const int* __restrict__ slot_of_cam, int lo, int hi,
                                                                     const int* __restrict__ fsize) {
  __shared__ DetBox sb[BDET_WARPS][CS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * BDET_WARPS + warp;
  if (b >= B) return;   // the whole warp
  const int seg = bdet_segment(cam_of, slot_of_cam, lo, hi, b);
  if (seg < 0) return;
  kp += (size_t)seg * npx;
  if (fsize) {   // the camera's own size: its boxes clip and its keys decode with it
    const int c = cam_of ? cam_of[b] : 0;
    W = fsize[4 * c + 2]; H = fsize[4 * c + 3];
  }
  const int nb = N[b];
  int lim = min(num[(size_t)b * num_stride], cap_mode ? Ncap - nb : EKF_BATCH_MAX_CORNERS);
  lim = max(0, min(lim, CS));
#pragma unroll
  for (int i = lane; i < CS; i += 32) {
    DetBox bx{0, 0, 0, 0};
    if (i < nb) bx = det_patch_box(centers[2 * ((size_t)b * Ncap + i)], centers[2 * ((size_t)b * Ncap + i) + 1], W, H, window);
    sb[warp][i] = bx;
    boxes[(size_t)b * CS + i] = bx;
  }
  __syncwarp();
  if (lane == 0) limit[b] = lim;
  if (lim == 0) return;
  unsigned maxbits = 0;   // no pixel of the mask above 0: threshold 0, as k_det_max leaves it
  for (int i0 = 0; i0 < npx; i0 += 32) {
    const int i = i0 + lane;
    const unsigned long long k = i < npx ? kp[i] : 0ull;
    bool stop = (k == 0ull);
    if (!stop) {
      const unsigned idx = (unsigned)(k & 0xffffffffull);
      stop = !det_in_boxes((int)(idx % (unsigned)W), (int)(idx / (unsigned)W), sb[warp], nb);
    }
    const unsigned m = __ballot_sync(0xffffffffu, stop);
    if (m) {
      maxbits = (unsigned)(__shfl_sync(0xffffffffu, k, __ffs(m) - 1) >> 32);
      break;
    }
  }
  if (lane == 0) thr_bits[b] = __float_as_uint((float)((double)__uint_as_float(maxbits) * 0.01));
}

// One thread per filter: goodFeaturesToTrack's greedy selection over the shared candidate list.
template <int CS>
__global__ void k_bdet_select(const unsigned long long* __restrict__ kc, int nkeys, int W, const DetBox* __restrict__ boxes,
                              const int* __restrict__ N, const unsigned* __restrict__ thr_bits, const int* __restrict__ limit, int B,
                              float* __restrict__ out_xy, int* __restrict__ out_n, const int* __restrict__ cam_of,
                              const int* __restrict__ slot_of_cam, int lo, int hi, const int* __restrict__ fsize) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int seg = bdet_segment(cam_of, slot_of_cam, lo, hi, b);
  if (seg < 0) return;
  kc += (size_t)seg * nkeys;
  if (fsize) W = fsize[4 * (cam_of ? cam_of[b] : 0) + 2];
  const int lim = limit[b];
  out_n[b] = lim > 0 ? det_select_walk(kc, nkeys, W, thr_bits[b], boxes + (size_t)b * CS, N[b], 144.0f, lim,
                                       out_xy + (size_t)b * 2 * CS)
                     : 0;
}

cudaError_t batch_detect_reserve(BatchDetectBufs& d, size_t px, int B, int cstride) {
  cudaError_t e;
  if (!d.boxes) {
    if ((e = cudaMalloc((void**)&d.boxes, sizeof(DetBox) * cstride * (size_t)B)) != cudaSuccess) return e;
    if ((e = cudaMalloc((void**)&d.thr_bits, sizeof(unsigned) * (size_t)B)) != cudaSuccess) return e;
    if ((e = cudaMalloc((void**)&d.limit, sizeof(int) * (size_t)B)) != cudaSuccess) return e;
  }
  if (px <= d.cap) return cudaSuccess;
  cudaFree(d.eig); cudaFree(d.keys); cudaFree(d.tmp);
  d.eig = nullptr; d.keys = nullptr; d.tmp = nullptr; d.cap = 0;
  size_t tmp = 0;
  if ((e = cub::DeviceRadixSort::SortKeysDescending(nullptr, tmp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                    (int)px)) != cudaSuccess)
    return e;
  if ((e = cudaMalloc((void**)&d.eig, sizeof(float) * px)) != cudaSuccess) return e;
  if ((e = cudaMalloc((void**)&d.keys, sizeof(unsigned long long) * 4 * px)) != cudaSuccess) return e;
  if ((e = cudaMalloc(&d.tmp, tmp)) != cudaSuccess) return e;
  d.tmp_bytes = tmp;
  d.cap = px;
  return cudaSuccess;
}

// scratch for chunks of up to `chunk` cameras of npx pixels each: the per-camera buffers, the segment offsets and the larger of
// the two sorts' workspaces
cudaError_t batch_detect_reserve_cams(BatchDetectBufs& d, size_t npx, int chunk, int B, int cstride) {
  cudaError_t e = batch_detect_reserve(d, npx * (size_t)chunk, B, cstride);
  if (e != cudaSuccess) return e;
  size_t tmp = 0;
  if ((e = cub::DeviceSegmentedRadixSort::SortKeysDescending(nullptr, tmp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                             (int)(npx * chunk), chunk, (const int*)nullptr, (const int*)nullptr)) != cudaSuccess)
    return e;
  if (tmp > d.tmp_bytes) {
    cudaFree(d.tmp);
    d.tmp = nullptr; d.tmp_bytes = 0;
    if ((e = cudaMalloc(&d.tmp, tmp)) != cudaSuccess) return e;
    d.tmp_bytes = tmp;
  }
  if (d.offs_chunk == chunk && d.offs_npx == npx) return cudaSuccess;
  std::vector<int> offs((size_t)chunk + 1);
  for (int s = 0; s <= chunk; ++s) offs[s] = (int)(s * npx);
  cudaFree(d.offs);
  d.offs = nullptr; d.offs_chunk = 0;
  if ((e = cudaMalloc((void**)&d.offs, sizeof(int) * offs.size())) != cudaSuccess) return e;
  if ((e = cudaMemcpy(d.offs, offs.data(), sizeof(int) * offs.size(), cudaMemcpyHostToDevice)) != cudaSuccess) return e;
  d.offs_chunk = chunk; d.offs_npx = npx;
  return cudaSuccess;
}

void batch_detect_free(BatchDetectBufs& d) {
  cudaFree(d.eig); cudaFree(d.keys); cudaFree(d.tmp); cudaFree(d.boxes); cudaFree(d.thr_bits); cudaFree(d.limit); cudaFree(d.offs);
  d = BatchDetectBufs{};
}

cudaError_t launch_batch_detect(cudaStream_t st, BatchDetectBufs& d, FrameView fr, const float* centers, const int* N, int Ncap, int B,
                                int window, const int* num, int num_stride, int cap_mode, int cstride, float* out_xy, int* out_n,
                                long long* launches) {
  const int W = fr.w, H = fr.h, npx = W * H;
  unsigned long long *kp = d.keys, *kc = d.keys + d.cap, *kp_s = d.keys + 2 * d.cap, *kc_s = d.keys + 3 * d.cap;
  launch_det_eig(st, fr, d.eig, launches);
  k_bdet_keys<<<dim3((W + 255) / 256, H), 256, 0, st>>>(d.eig, W, H, window, kp, kc, nullptr, nullptr);
  size_t tmp = d.tmp_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortKeysDescending(d.tmp, tmp, kp, kp_s, npx, 0, 64, st);
  if (e != cudaSuccess) return e;
  tmp = d.tmp_bytes;
  e = cub::DeviceRadixSort::SortKeysDescending(d.tmp, tmp, kc, kc_s, npx, 0, 64, st);
  if (e != cudaSuccess) return e;
  const unsigned gt = (B + BDET_WARPS - 1) / BDET_WARPS, gs = (B + 127) / 128;
  if (cstride == EKF_BATCH_MAX_CORNERS) {
    k_bdet_threshold<EKF_BATCH_MAX_CORNERS><<<gt, 32 * BDET_WARPS, 0, st>>>(kp_s, npx, W, H, window, centers, N, Ncap, B, num,
                                                                           num_stride, cap_mode, d.boxes, d.thr_bits, d.limit,
                                                                           nullptr, nullptr, 0, 0, nullptr);
    k_bdet_select<EKF_BATCH_MAX_CORNERS><<<gs, 128, 0, st>>>(kc_s, npx, W, d.boxes, N, d.thr_bits, d.limit, B, out_xy, out_n,
                                                             nullptr, nullptr, 0, 0, nullptr);
  } else {
    k_bdet_threshold<EKF_BATCH_MAX_FEATURES><<<gt, 32 * BDET_WARPS, 0, st>>>(kp_s, npx, W, H, window, centers, N, Ncap, B, num,
                                                                            num_stride, cap_mode, d.boxes, d.thr_bits, d.limit,
                                                                            nullptr, nullptr, 0, 0, nullptr);
    k_bdet_select<EKF_BATCH_MAX_FEATURES><<<gs, 128, 0, st>>>(kc_s, npx, W, d.boxes, N, d.thr_bits, d.limit, B, out_xy, out_n,
                                                              nullptr, nullptr, 0, 0, nullptr);
  }
  *launches += 5;   // keys, the two sorts (counted once each), threshold, select; the eig map counts itself
  return cudaGetLastError();
}

cudaError_t launch_batch_detect_cams(cudaStream_t st, BatchDetectBufs& d, FrameView fr, const int* cams, int n_req, int chunk,
                                     const int* cam_of, const int* slot_of_cam, const float* centers, const int* N, int Ncap, int B,
                                     int window, const int* num, int num_stride, int cap_mode, int cstride, float* out_xy, int* out_n,
                                     long long* launches, const int* fsize, const int* fsize_host, const int* seg_cam) {
  const int W = fr.w, H = fr.h, npx = W * H;
  const size_t fstep = (size_t)fr.h * fr.stride;
  cudaError_t e = cudaMemsetAsync(out_n, 0, sizeof(int) * (size_t)B, st);   // filters of cameras nobody asks from find nothing
  if (e != cudaSuccess) return e;
  unsigned long long *kp = d.keys, *kc = d.keys + d.cap, *kp_s = d.keys + 2 * d.cap, *kc_s = d.keys + 3 * d.cap;
  const unsigned gt = (B + BDET_WARPS - 1) / BDET_WARPS, gs = (B + 127) / 128;
  for (int lo = 0; lo < n_req; lo += chunk) {
    const int C = std::min(chunk, n_req - lo), hi = lo + C;
    for (int s = 0; s < C; ++s) {   // with sizes, the eig map of the camera's own w x h (Sobel border at its own edge)
      const int c = cams[lo + s], wc = fsize_host ? fsize_host[4 * c + 2] : W, hc = fsize_host ? fsize_host[4 * c + 3] : H;
      launch_det_eig(st, FrameView{fr.px + (size_t)c * fstep, wc, hc, fr.stride}, d.eig + (size_t)s * npx, launches);
    }
    k_bdet_keys<<<dim3((W + 255) / 256, H, C), 256, 0, st>>>(d.eig, W, H, window, kp, kc, fsize, fsize ? seg_cam + lo : nullptr);
    size_t tmp = d.tmp_bytes;
    e = cub::DeviceSegmentedRadixSort::SortKeysDescending(d.tmp, tmp, kp, kp_s, C * npx, C, d.offs, d.offs + 1, 0, 64, st);
    if (e != cudaSuccess) return e;
    tmp = d.tmp_bytes;
    e = cub::DeviceSegmentedRadixSort::SortKeysDescending(d.tmp, tmp, kc, kc_s, C * npx, C, d.offs, d.offs + 1, 0, 64, st);
    if (e != cudaSuccess) return e;
    if (cstride == EKF_BATCH_MAX_CORNERS) {
      k_bdet_threshold<EKF_BATCH_MAX_CORNERS><<<gt, 32 * BDET_WARPS, 0, st>>>(kp_s, npx, W, H, window, centers, N, Ncap, B, num,
                                                                             num_stride, cap_mode, d.boxes, d.thr_bits, d.limit,
                                                                             cam_of, slot_of_cam, lo, hi, fsize);
      k_bdet_select<EKF_BATCH_MAX_CORNERS><<<gs, 128, 0, st>>>(kc_s, npx, W, d.boxes, N, d.thr_bits, d.limit, B, out_xy, out_n,
                                                               cam_of, slot_of_cam, lo, hi, fsize);
    } else {
      k_bdet_threshold<EKF_BATCH_MAX_FEATURES><<<gt, 32 * BDET_WARPS, 0, st>>>(kp_s, npx, W, H, window, centers, N, Ncap, B, num,
                                                                              num_stride, cap_mode, d.boxes, d.thr_bits, d.limit,
                                                                              cam_of, slot_of_cam, lo, hi, fsize);
      k_bdet_select<EKF_BATCH_MAX_FEATURES><<<gs, 128, 0, st>>>(kc_s, npx, W, d.boxes, N, d.thr_bits, d.limit, B, out_xy, out_n,
                                                                cam_of, slot_of_cam, lo, hi, fsize);
    }
    *launches += 5;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return cudaSuccess;
}
