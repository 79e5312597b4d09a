// csrc/ekf_detect.cu — VSlamFilter::findNewFeatures (vslamRansac.cpp:783-839; SURVEY.md §8(f) row 2):
// the visibility mask the reference builds around the existing patches, and a Shi-Tomasi corner
// detector standing in for OpenCV's goodFeaturesToTrack(frame, corners, num, 0.01, 12, mask) with its
// default blockSize = 3 / Sobel aperture 3:
//   eig = min eigenvalue of the 3x3 box sum of [dx^2 dxdy; dxdy dy^2], dx / dy = Sobel * 1/(4*3*255),
//   BORDER_REFLECT_101; threshold at 0.01 * max(eig over the mask) (THRESH_TOZERO); 3x3 local maxima
//   (rows / columns 1 .. size-2); sorted by score (ties: higher address first); greedy selection with
//   a minimum Euclidean distance of 12 px; at most `num` corners.
// PARITY: unpinned.  The arithmetic lives in an un-vendored dependency of the reference (OpenCV, version
// unpinned); this restates the published algorithm and is checked against the cv2 4.13 wheel of this
// image (tests/test_gpu_detect.py), whose float pipeline (SIMD FMA, sliding box sums) differs from
// these direct sums in the last bits, so scores agree to ~1e-6 relative and the selected corners agree
// except on exact ties.
#include <cfloat>

#include "ekf_detect.cuh"
#include "ekf_kernels.h"

#define DET_TX 32
#define DET_TY 8

__device__ __forceinline__ int reflect101(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// mask (vslamRansac.cpp:788-818): 255 inside the `estrem` border, 0 in a (2w+1)^2 box around every patch (ekf_detect.cuh)
__global__ void k_det_mask_base(uint8_t* __restrict__ mask, int W, int H, int estrem) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x < W) mask[(size_t)y * W + x] = det_in_base(x, y, W, H, estrem) ? 255 : 0;
}
__global__ void k_det_mask_patches(uint8_t* __restrict__ mask, int W, int H, FeatTab ft, int N, int w) {
  const int f = blockIdx.x;
  if (f >= N) return;
  const DetBox b = det_patch_box(ft.center[2 * f], ft.center[2 * f + 1], W, H, w);
  for (int e = threadIdx.x; e < b.w * b.h; e += blockDim.x) {
    const int xx = b.x0 + e % b.w, yy = b.y0 + e / b.w;
    if (xx < W && yy < H) mask[(size_t)yy * W + xx] = 0;
  }
}

// eig map (float), one thread per pixel, u8 tile with a halo of 2 in shared memory
__global__ void __launch_bounds__(DET_TX * DET_TY) k_det_eig(const uint8_t* __restrict__ img, int W, int H, int stride,
                                                           float* __restrict__ eig) {
  __shared__ float px[DET_TY + 4][DET_TX + 4];
  __shared__ float gx[DET_TY + 2][DET_TX + 2], gy[DET_TY + 2][DET_TX + 2];
  const int bx = blockIdx.x * DET_TX, by = blockIdx.y * DET_TY;
  const int tid = threadIdx.y * DET_TX + threadIdx.x;
  for (int e = tid; e < (DET_TY + 4) * (DET_TX + 4); e += DET_TX * DET_TY) {
    const int ly = e / (DET_TX + 4), lx = e % (DET_TX + 4);
    // Sobel taps use REFLECT_101 around the true image border; the box filter reflects the derivative maps
    const int yy = reflect101(reflect101(by + ly - 2, H), H), xx = reflect101(reflect101(bx + lx - 2, W), W);
    px[ly][lx] = (float)img[(size_t)yy * stride + xx];
  }
  __syncthreads();
  const float s = (float)(1.0 / (4.0 * 3.0 * 255.0)), s2 = 2.0f * s;
  for (int e = tid; e < (DET_TY + 2) * (DET_TX + 2); e += DET_TX * DET_TY) {
    const int ly = e / (DET_TX + 2), lx = e % (DET_TX + 2);   // derivative at image (by + ly - 1, bx + lx - 1)
    const int iy = by + ly - 1, ix = bx + lx - 1;
    float dxv = 0.0f, dyv = 0.0f;
    if (iy <= H && ix <= W) {   // positions one past the border are needed by the last row / column only
      // the box filter reflects the derivative maps (REFLECT_101): evaluate at the reflected pixel ...
      const int ry = reflect101(iy, H), rx = reflect101(ix, W);
      // ... whose own Sobel taps are reflected at the image border; all of them lie inside the halo-2 tile
      auto P = [&](int y, int x) { return px[reflect101(y, H) - by + 2][reflect101(x, W) - bx + 2]; };
      const float r0 = __fsub_rn(P(ry - 1, rx + 1), P(ry - 1, rx - 1)), r1 = __fsub_rn(P(ry, rx + 1), P(ry, rx - 1)),
                  r2 = __fsub_rn(P(ry + 1, rx + 1), P(ry + 1, rx - 1));
      dxv = __fadd_rn(__fmul_rn(r1, s2), __fmul_rn(__fadd_rn(r0, r2), s));
      const float h0 = __fadd_rn(__fmul_rn(P(ry - 1, rx), s2), __fmul_rn(__fadd_rn(P(ry - 1, rx - 1), P(ry - 1, rx + 1)), s));
      const float h2 = __fadd_rn(__fmul_rn(P(ry + 1, rx), s2), __fmul_rn(__fadd_rn(P(ry + 1, rx - 1), P(ry + 1, rx + 1)), s));
      dyv = __fsub_rn(h2, h0);
    }
    gx[ly][lx] = dxv; gy[ly][lx] = dyv;
  }
  __syncthreads();
  const int x = bx + threadIdx.x, y = by + threadIdx.y;
  if (x >= W || y >= H) return;
  float a = 0, b = 0, c = 0;
#pragma unroll
  for (int dy = 0; dy < 3; ++dy) {
    float ra = 0, rb = 0, rc = 0;
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
      const float u = gx[threadIdx.y + dy][threadIdx.x + dx], v = gy[threadIdx.y + dy][threadIdx.x + dx];
      ra = __fadd_rn(ra, __fmul_rn(u, u)); rb = __fadd_rn(rb, __fmul_rn(u, v)); rc = __fadd_rn(rc, __fmul_rn(v, v));
    }
    a = __fadd_rn(a, ra); b = __fadd_rn(b, rb); c = __fadd_rn(c, rc);
  }
  const float ha = __fmul_rn(a, 0.5f), hc = __fmul_rn(c, 0.5f);
  const float d = __fsub_rn(ha, hc);
  eig[(size_t)y * W + x] = __fsub_rn(__fadd_rn(ha, hc), sqrtf(__fadd_rn(__fmul_rn(d, d), __fmul_rn(b, b))));
}

__global__ void k_det_max(const float* __restrict__ eig, const uint8_t* __restrict__ mask, int n, unsigned* __restrict__ maxbits) {
  float m = 0.0f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    if (mask[i]) m = fmaxf(m, eig[i]);
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(maxbits, __float_as_uint(m));   // non-negative floats order like their bits
}

// thresholded 3x3 local maxima inside the mask -> (score bits << 32 | pixel index) keys
__global__ void k_det_candidates(const float* __restrict__ eig, const uint8_t* __restrict__ mask, int W, int H,
                                 const unsigned* __restrict__ maxbits, unsigned long long* __restrict__ keys, int cap,
                                 int* __restrict__ count) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y + 1;
  if (x < 1 || x >= W - 1 || y >= H - 1) return;
  const float thr = (float)((double)__uint_as_float(*maxbits) * 0.01);
  auto T = [&](int yy, int xx) { const float v = eig[(size_t)yy * W + xx]; return v > thr ? v : 0.0f; };   // THRESH_TOZERO
  const float val = T(y, x);
  if (val == 0.0f || !mask[(size_t)y * W + x]) return;
  float mx = val;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) mx = fmaxf(mx, T(y + dy, x + dx));
  if (val != mx) return;
  const int slot = atomicAdd(count, 1);
  if (slot < cap) keys[slot] = ((unsigned long long)__float_as_uint(val) << 32) | (unsigned)(y * W + x);
}

// descending bitonic sort of `n2` keys (power of two, padded with zeros) by one CTA, then the greedy
// minimum-distance selection in score order
__global__ void __launch_bounds__(1024) k_det_select(unsigned long long* __restrict__ keys, int n2, const int* __restrict__ count,
                                                     int cap, int W, float min_dist2, int max_corners, float* __restrict__ out_xy,
                                                     int* __restrict__ out_n) {
  const int tid = threadIdx.x;
  const int total = min(*count, cap);
  n2 = 2;
  while (n2 < total) n2 <<= 1;   // sort only what exists (the buffer holds `cap` = a power of two >= n2 keys)
  for (int i = total + tid; i < n2; i += 1024) keys[i] = 0ull;
  __syncthreads();
  for (int k = 2; k <= n2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n2; i += 1024) {
        const int l = i ^ j;
        if (l > i) {
          const unsigned long long a = keys[i], b = keys[l];
          const bool desc = (i & k) == 0;
          if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[l] = a; }
        }
      }
      __syncthreads();
    }
  __shared__ float ax[1024], ay[1024];
  __shared__ int nacc;
  if (tid == 0) nacc = 0;
  __syncthreads();
  const int limit = min(max_corners, 1024);
  for (int i = 0; i < total; ++i) {
    const unsigned idx = (unsigned)(keys[i] & 0xffffffffull);
    const float x = (float)(idx % W), y = (float)(idx / W);
    int bad = 0;
    for (int m = tid; m < nacc; m += 1024) {
      const float dx = x - ax[m], dy = y - ay[m];
      if (dx * dx + dy * dy < min_dist2) bad = 1;
    }
    const int anybad = __syncthreads_or(bad);
    if (!anybad && tid == 0) { ax[nacc] = x; ay[nacc] = y; out_xy[2 * nacc] = x; out_xy[2 * nacc + 1] = y; nacc = nacc + 1; }
    __syncthreads();
    if (nacc >= limit) break;
  }
  if (tid == 0) *out_n = nacc;
}

int launch_detect_corners(cudaStream_t st, FrameView fr, FeatTab ft, int N, int window, uint8_t* mask, float* eig,
                          unsigned long long* keys, int key_cap, int* counters /* [0] count, [1] max bits, [2] out n */,
                          int max_corners, float* out_xy, long long* launches) {
  const int W = fr.w, H = fr.h;
  cudaMemsetAsync(counters, 0, 4 * sizeof(int), st);
  k_det_mask_base<<<dim3((W + 255) / 256, H), 256, 0, st>>>(mask, W, H, window);
  if (N > 0) k_det_mask_patches<<<N, 128, 0, st>>>(mask, W, H, ft, N, window);
  k_det_eig<<<dim3((W + DET_TX - 1) / DET_TX, (H + DET_TY - 1) / DET_TY), dim3(DET_TX, DET_TY), 0, st>>>(fr.px, W, H, fr.stride, eig);
  k_det_max<<<296, 256, 0, st>>>(eig, mask, W * H, reinterpret_cast<unsigned*>(counters + 1));
  k_det_candidates<<<dim3((W + 255) / 256, H - 2), 256, 0, st>>>(eig, mask, W, H, reinterpret_cast<unsigned*>(counters + 1), keys, key_cap,
                                                                 counters);
  k_det_select<<<1, 1024, 0, st>>>(keys, key_cap, counters, key_cap, W, 144.0f, max_corners, out_xy, counters + 2);
  *launches += N > 0 ? 6 : 5;
  return 0;
}

void launch_det_eig(cudaStream_t st, FrameView fr, float* eig, long long* launches) {
  k_det_eig<<<dim3((fr.w + DET_TX - 1) / DET_TX, (fr.h + DET_TY - 1) / DET_TY), dim3(DET_TX, DET_TY), 0, st>>>(fr.px, fr.w, fr.h, fr.stride, eig);
  *launches += 1;
}

// ------------------------------------------------------------------------------------------------
// captureNewFrame (vslamRansac.cpp:234-245): cv::resize(frame, Size(w / scale, h / scale)) followed by
// cvtColor(BGR2GRAY) when the frame has three channels.  Restates OpenCV's 8-bit paths:
//   INTER_LINEAR: 11-bit fixed-point coefficients, horizontal pass in int, vertical pass
//                 ((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2 >> 2;
//   exact 2x decimation: OpenCV switches to INTER_AREA, (s00 + s01 + s10 + s11 + 2) >> 2;
//   BGR2GRAY: (3735 B + 19235 G + 9798 R + 16384) >> 15 (OpenCV 4 coefficients).
// PARITY: unpinned (OpenCV is an un-vendored, unpinned dependency of the reference); bit-exact against
// the cv2 4.13 wheel of this image (tests/test_gpu_detect.py).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void resize_coeff(int d, double scale, int ssize, int* s0, short* a0, short* a1) {
  float f = (float)((d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= s;
  if (s < 0) { f = 0; s = 0; }
  if (s >= ssize - 1) { f = 0; s = ssize - 1; }
  *s0 = s;
  // saturate_cast<short>(float): round to nearest even
  *a0 = (short)__float2int_rn((1.f - f) * 2048.f);
  *a1 = (short)__float2int_rn(f * 2048.f);
}
// SLOTS: frame z of the source stack goes to slot slot[z] of the destination stack (a capture of some cameras of a batch).
template <bool SLOTS>
__global__ void k_capture_resize_gray(const uint8_t* __restrict__ src, int sw, int sh, int sstride, int cn, uint8_t* __restrict__ dst,
                                      int dw, int dh, int dstride, const int* __restrict__ fsize, const int* __restrict__ slot) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= dw || y >= dh) return;
  int z = blockIdx.z;
  src += (size_t)z * sh * sstride;   // frame z of a stack (batched cameras)
  if constexpr (SLOTS) z = slot[z];
  dst += (size_t)z * dh * dstride;
  if (fsize) {   // frame z is the top-left fsize[0] x fsize[1] of its slot, resized to fsize[2] x fsize[3] (cv::resize of the crop)
    const int* q = fsize + 4 * z;
    sw = q[0]; sh = q[1]; dw = q[2]; dh = q[3];
    if (x >= dw || y >= dh) return;
  }
  int ch[3] = {0, 0, 0};
  if (sw == dw && sh == dh) {
    for (int c = 0; c < cn; ++c) ch[c] = src[(size_t)y * sstride + x * cn + c];
  } else {
    const double scale_x = (double)sw / dw, scale_y = (double)sh / dh;
    const bool area2 = (sw == 2 * dw) && (sh == 2 * dh);
    if (area2) {
      for (int c = 0; c < cn; ++c) {
        const uint8_t* p = src + (size_t)(2 * y) * sstride + (2 * x) * cn + c;
        ch[c] = (p[0] + p[cn] + p[sstride] + p[sstride + cn] + 2) >> 2;
      }
    } else {
      int sx, sy; short ax0, ax1, by0, by1;
      resize_coeff(x, scale_x, sw, &sx, &ax0, &ax1);
      resize_coeff(y, scale_y, sh, &sy, &by0, &by1);
      const int sx1 = min(sx + 1, sw - 1), sy1 = min(sy + 1, sh - 1);
      for (int c = 0; c < cn; ++c) {
        const int r0 = src[(size_t)sy * sstride + sx * cn + c] * ax0 + src[(size_t)sy * sstride + sx1 * cn + c] * ax1;
        const int r1 = src[(size_t)sy1 * sstride + sx * cn + c] * ax0 + src[(size_t)sy1 * sstride + sx1 * cn + c] * ax1;
        ch[c] = (((by0 * (r0 >> 4)) >> 16) + ((by1 * (r1 >> 4)) >> 16) + 2) >> 2;
      }
    }
  }
  int g = ch[0];
  if (cn == 3) g = (ch[0] * 3735 + ch[1] * 19235 + ch[2] * 9798 + 16384) >> 15;
  dst[(size_t)y * dstride + x] = (uint8_t)min(max(g, 0), 255);
}
void launch_capture_resize_gray(cudaStream_t st, const uint8_t* src, int sw, int sh, int sstride, int cn, uint8_t* dst, int dw, int dh,
                                int dstride, long long* launches, int n_frames, const int* fsize, const int* slot) {
  const dim3 grid((dw + 255) / 256, dh, n_frames);
  if (slot) k_capture_resize_gray<true><<<grid, 256, 0, st>>>(src, sw, sh, sstride, cn, dst, dw, dh, dstride, fsize, slot);
  else k_capture_resize_gray<false><<<grid, 256, 0, st>>>(src, sw, sh, sstride, cn, dst, dw, dh, dstride, fsize, slot);
  *launches += 1;
}
