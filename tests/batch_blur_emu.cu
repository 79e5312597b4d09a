// tests/batch_blur_emu.cu — TEST INFRASTRUCTURE.  The motion-blur template arithmetic of csrc/ekf_blur.cuh on the CPU, built
// from the same __host__ __device__ functions the kernels call, so that tests/test_batch_blur_emu.py can check without a GPU
// that the batched kernel's form (k_batch_predict_blur: distinct line points, ordered by blur_rank, one list walk per pixel)
// gives exactly the single filter's form (k_predict_blur: bit mask, row-major walk), and that both equal a restatement of
// evaluateKernel + filter2D.  The warp's ballot compaction is a plain loop here; everything else is the shipped code.
// Compiled as HOST code by nvcc (tests build it on the fly); nothing here is shipped.
#include <cstring>
#include <vector>

#include "ekf_blur.cuh"

extern "C" {

// blur_decide: 0 unchanged, 1 blurred (krows x kcols), -1 kernel above BLUR_MAXK
int emu_blur_decide(double ddx, double ddy, int kernel_min_size, int* krows, int* kcols) {
  *krows = 0; *kcols = 0;
  return blur_decide(ddx, ddy, kernel_min_size, krows, kcols);
}

// the line of evaluateKernel: out[0..3) = s, c, length; xy0 = x0, y0
void emu_blur_line(double dx, double dy, double* out, int* xy0) {
  const BlurLine L = blur_line(dx, dy);
  out[0] = L.s; out[1] = L.c; out[2] = L.length;
  xy0[0] = L.x0; xy0[1] = L.y0;
}

// The single filter's form: the bit mask of k_predict_blur, then blur_pixel_bits.  Returns the coefficient count.
int emu_blur_bits(const uint8_t* src, int w, double dx, double dy, int krows, int kcols, uint8_t* out) {
  std::vector<unsigned> kbits((krows * kcols + 31) / 32, 0u);
  const BlurLine L = blur_line(dx, dy);
  int count = 0;
  for (int i = 0; i < L.length; ++i) {
    int x, y;
    if (blur_line_point(L, i, krows, kcols, &x, &y)) {
      const int bit = x * kcols + y;
      if (!(kbits[bit >> 5] & (1u << (bit & 31)))) { kbits[bit >> 5] |= 1u << (bit & 31); ++count; }
    }
  }
  const double kf = 1.0 / (double)count;
  for (int e = 0; e < w * w; ++e) out[e] = blur_pixel_bits(src, w, e, kbits.data(), krows, kcols, kf);
  return count;
}

// The batched form: distinct points in line order (blur_line_point_new), placed by blur_rank, walked by blur_pixel_list.
// coef (BLUR_MAXPTS) receives the ordered list as (row << 16 | column); *npts the number of line points.  Returns its length.
int emu_blur_list(const uint8_t* src, int w, double dx, double dy, int krows, int kcols, uint8_t* out, int* coef, int* npts) {
  const BlurLine L = blur_line(dx, dy);
  std::vector<int> seq;
  int n = 0;
  for (int i = 0; i < L.length; ++i, ++n) {
    int x, y;
    if (blur_line_point_new(L, i, krows, kcols, &x, &y)) seq.push_back(blur_pack(x, y));
  }
  *npts = n;
  const int m = (int)seq.size();
  if (m > BLUR_MAXPTS) return -1;
  for (int j = 0; j < m; ++j) coef[blur_rank(seq.data(), m, j)] = seq[j];
  const double kf = 1.0 / (double)m;
  for (int e = 0; e < w * w; ++e) out[e] = blur_pixel_list(src, w, e, coef, m, krows, kcols, kf);
  return m;
}

}  // extern "C"
