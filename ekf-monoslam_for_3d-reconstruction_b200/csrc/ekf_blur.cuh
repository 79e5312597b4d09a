// csrc/ekf_blur.cuh — motion-blur template prediction (V:498-500, 546-548, 575-576; Patch::blur Patch.cpp:50-57;
// evaluateKernel / blurPatch libblur.cpp:17-81), the per-feature arithmetic shared by the single filter's k_predict_blur
// and the batched k_batch_predict_blur, so that both give the same bits.  Everything but the pose and the projection is
// __host__ __device__: tests/batch_blur_emu.cu runs it on the CPU.  Compiled with --fmad=false like the rest.
#pragma once
#include "ekf_math.cuh"

#define BLUR_MAXK 256     // largest kernel side supported (rows and columns)
#define BLUR_MAXPTS 384   // > points of the longest line: length < 256 * sqrt(2), so at most 363

// The pose the camera will have T_camera * dT later (V:498-499): position rb, world-to-camera rotation Rb.
__device__ inline void blur_pose(const double* cam, double T_camera, double dT, double rb[3], double Rb[9]) {
  const double q[4] = {cam[3], cam[4], cam[5], cam[6]};
  double wb[3], hb[4], qb[4];
  for (int c = 0; c < 3; ++c) wb[c] = (cam[10 + c] * T_camera) * dT;
  d_vec2quat(wb, hb);
  d_quat_mul(q, hb, qb);
  const double qbc[4] = {qb[0], -qb[1], -qb[2], -qb[3]};
  d_quat2rot(qbc, Rb);
  for (int c = 0; c < 3; ++c) rb[c] = cam[c] + (cam[7 + c] * T_camera) * dT;
}

// The feature's displacement between its prediction (hx, hy) and its projection from the blur pose (V:546-548 / 575-576).
__device__ inline void blur_displacement(const CamParams& cm, const double* fs, int coding, const double rb[3], const double Rb[9],
                                         double hx, double hy, double* ddx, double* ddy) {
  double hib[2];
  d_feature_h(cm, fs, coding, rb, Rb, hib);
  *ddx = hx - hib[0];
  *ddy = hy - hib[1];
}

// Patch::blur's test (Patch.cpp:52) and the kernel size of evaluateKernel (cv::Mat::zeros(width, height), libblur.cpp:20-23):
// 0 = the template stays as it is, 1 = blurred with a krows x kcols kernel, -1 = the kernel exceeds BLUR_MAXK.
__host__ __device__ inline int blur_decide(double ddx, double ddy, int kernel_min_size, int* krows, int* kcols) {
  const double dn = sqrt(ddx * ddx + ddy * ddy);
  if (!(dn > kernel_min_size)) return 0;
  *kcols = (int)(fabs(ddx) + 1);
  *krows = (int)(fabs(ddy) + 1);
  return (*krows > BLUR_MAXK || *kcols > BLUR_MAXK) ? -1 : 1;
}

// The rasterised line of evaluateKernel (libblur.cpp:25-43): points i = 0, 1, ... while i < length.
struct BlurLine {
  double s, c, length;
  int x0, y0;
};
__host__ __device__ inline BlurLine blur_line(double dx, double dy) {
  BlurLine L;
  const double theta = atan2(dy, dx);
  L.length = sqrt(dx * dx + dy * dy);
  L.c = cos(theta);
  L.s = sin(theta);
  L.x0 = (int)(L.s < 0 ? -L.s * L.length : 0.0);
  L.y0 = (int)(L.c < 0 ? -L.c * L.length : 0.0);
  return L;
}
// Point i of the line: kernel row x, column y; true when it lies inside the krows x kcols kernel (one past the kernel is
// undefined behaviour in the reference, and skipped).
__host__ __device__ inline bool blur_line_point(const BlurLine& L, int i, int krows, int kcols, int* x, int* y) {
  *x = (int)(i * L.s + L.x0);
  *y = (int)(i * L.c + L.y0);
  return *x >= 0 && *y >= 0 && *x < krows && *y < kcols;
}
// Point i inside the kernel and not a repeat of point i - 1.  Row and column are each monotone in i (a fixed-sign step,
// rounded and truncated), so the points inside the kernel are a contiguous run of i and repeats are consecutive: the
// points this accepts are the distinct coefficients, each once.
__host__ __device__ inline bool blur_line_point_new(const BlurLine& L, int i, int krows, int kcols, int* x, int* y) {
  if (!blur_line_point(L, i, krows, kcols, x, y)) return false;
  int px, py;
  return i == 0 || !blur_line_point(L, i - 1, krows, kcols, &px, &py) || px != *x || py != *y;
}

__host__ __device__ __forceinline__ int blur_pack(int x, int y) { return (x << 16) | y; }
__host__ __device__ __forceinline__ int blur_row(int p) { return p >> 16; }
__host__ __device__ __forceinline__ int blur_col(int p) { return p & 0xffff; }

// seq[0..m): the distinct coefficients in line order (blur_line_point_new).  Returns the place of seq[j] in ascending
// (row, column) order, OpenCV's direct-form order.  Rows and columns are monotone along seq: the coefficients of a row are
// one run [a, b] of seq, the runs come in ascending or descending row order, and inside a run the columns ascend or
// descend together with the whole line.
__host__ __device__ inline int blur_rank(const int* seq, int m, int j) {
  const bool rows_up = blur_row(seq[0]) <= blur_row(seq[m - 1]);
  const bool cols_up = blur_col(seq[0]) <= blur_col(seq[m - 1]);
  const int r = blur_row(seq[j]);
  int lo = 0, hi = m;   // a = first index of row r
  while (lo < hi) {
    const int mid = (lo + hi) >> 1, v = blur_row(seq[mid]);
    if (rows_up ? v < r : v > r) lo = mid + 1; else hi = mid;
  }
  const int a = lo;
  hi = m;               // b + 1 = first index past row r
  while (lo < hi) {
    const int mid = (lo + hi) >> 1, v = blur_row(seq[mid]);
    if (v == r) lo = mid + 1; else hi = mid;
  }
  const int b = lo - 1;
  return (rows_up ? a : m - 1 - b) + (cols_up ? j - a : b - j);
}

// BORDER_REFLECT_101 (w >= 2): ... 2 1 | 0 1 2 ... w-1 | w-2 ...
__host__ __device__ __forceinline__ int blur_reflect101(int i, int w) {
  const int p = 2 * w - 2;
  i %= p;
  if (i < 0) i += p;
  return i < w ? i : p - i;
}
// acc + kf * v rounded step by step; saturate_cast<uchar>(cvRound(acc)): round half to even, clamp to [0, 255]
__host__ __device__ __forceinline__ double blur_fma_free(double acc, double kf, double v) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(acc, __dmul_rn(kf, v));
#else
  return acc + kf * v;
#endif
}
__host__ __device__ __forceinline__ uint8_t blur_round_u8(double acc) {
#ifdef __CUDA_ARCH__
  const int iv = __double2int_rn(acc);
#else
  const int iv = (int)nearbyint(acc);
#endif
  return (uint8_t)(iv < 0 ? 0 : (iv > 255 ? 255 : iv));
}

// Output pixel e of the w x w template src correlated with the kernel whose set coefficients (every one 1 / count = kf)
// are the bits of kbits (krows x kcols, row-major), visited row by row: the single filter's form.
__host__ __device__ inline uint8_t blur_pixel_bits(const uint8_t* src, int w, int e, const unsigned* kbits, int krows, int kcols,
                                                   double kf) {
  const int y = e / w, x = e - y * w;
  const int ax = kcols / 2, ay = krows / 2;
  double acc = 0.0;
  for (int ky = 0; ky < krows; ++ky) {
    const int yy = blur_reflect101(y + ky - ay, w);
    for (int kx = 0; kx < kcols; ++kx) {
      const int bit = ky * kcols + kx;
      if (!(kbits[bit >> 5] & (1u << (bit & 31)))) continue;
      acc = blur_fma_free(acc, kf, (double)src[yy * w + blur_reflect101(x + kx - ax, w)]);
    }
  }
  return blur_round_u8(acc);
}
// The same pixel from the list of the m set coefficients (blur_pack(row, column)) in ascending (row, column) order: the
// same terms in the same order, without visiting the zeros.
__host__ __device__ inline uint8_t blur_pixel_list(const uint8_t* src, int w, int e, const int* coef, int m, int krows, int kcols,
                                                   double kf) {
  const int y = e / w, x = e - y * w;
  const int ax = kcols / 2, ay = krows / 2;
  double acc = 0.0;
  for (int k = 0; k < m; ++k) {
    const int p = coef[k];
    acc = blur_fma_free(acc, kf, (double)src[blur_reflect101(y + blur_row(p) - ay, w) * w + blur_reflect101(x + blur_col(p) - ax, w)]);
  }
  return blur_round_u8(acc);
}
