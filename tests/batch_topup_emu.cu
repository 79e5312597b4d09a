// tests/batch_topup_emu.cu — TEST INFRASTRUCTURE.  The batched corner detection of csrc/ekf_batch_detect.cu on the CPU, built
// from the same __host__ __device__ code the kernels run (csrc/ekf_detect.cuh: det_patch_box, det_in_base, det_in_boxes,
// det_key, det_select_walk), so that tests/test_batch_topup_emu.py can compare it with a restatement of the single filter's
// pipeline (mask, masked maximum, THRESH_TOZERO, 3x3 maxima, key sort, greedy 12 px) on planted eigenvalue maps, without a
// GPU.  The flow mirrors the kernels: one list of pixel keys and one of candidate keys for the whole frame, each sorted once;
// per filter the first pixel outside its boxes gives the threshold, then the walk over the candidate list.
// Compiled as HOST code by nvcc (tests build it on the fly); nothing here is shipped.
#include <algorithm>
#include <cstring>
#include <functional>
#include <vector>

#include "ekf_detect.cuh"

static unsigned fbits(float v) { unsigned u; std::memcpy(&u, &v, 4); return u; }
static float bitsf(unsigned u) { float v; std::memcpy(&v, &u, 4); return v; }

extern "C" {

// eig: H x W floats.  centers: B x maxc x 2, N: B patch counts, num: B corner limits.  out_xy: B x maxc x 2, out_n: B.
void emu_batch_detect(const float* eig, int W, int H, int window, int B, int maxc, const float* centers, const int* N, const int* num,
                      float* out_xy, int* out_n) {
  const size_t npx = (size_t)W * H;
  std::vector<unsigned long long> kp(npx, 0ull), kc(npx, 0ull);
  for (int y = 0; y < H; ++y)
    for (int x = 0; x < W; ++x) {
      const size_t i = (size_t)y * W + x;
      const float v = eig[i];
      if (!(v > 0.0f) || !det_in_base(x, y, W, H, window)) continue;
      kp[i] = det_key(fbits(v), (unsigned)i);
      if (x < 1 || x >= W - 1 || y < 1 || y >= H - 1) continue;
      bool mx = true;
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) mx = mx && !(eig[(size_t)(y + dy) * W + x + dx] > v);
      if (mx) kc[i] = kp[i];
    }
  std::sort(kp.begin(), kp.end(), std::greater<unsigned long long>());
  std::sort(kc.begin(), kc.end(), std::greater<unsigned long long>());
  std::vector<DetBox> boxes(maxc);
  for (int b = 0; b < B; ++b) {
    const int nb = N[b], lim = std::max(0, std::min(num[b], maxc));
    for (int f = 0; f < nb; ++f) boxes[f] = det_patch_box(centers[2 * (b * maxc + f)], centers[2 * (b * maxc + f) + 1], W, H, window);
    unsigned maxbits = 0;
    for (size_t i = 0; i < npx; ++i) {
      if (kp[i] == 0ull) break;
      const unsigned idx = (unsigned)kp[i];
      if (!det_in_boxes((int)(idx % (unsigned)W), (int)(idx / (unsigned)W), boxes.data(), nb)) { maxbits = (unsigned)(kp[i] >> 32); break; }
    }
    const unsigned thr = fbits((float)((double)bitsf(maxbits) * 0.01));
    out_n[b] = det_select_walk(kc.data(), (int)npx, W, thr, boxes.data(), nb, 144.0f, lim, out_xy + (size_t)b * 2 * maxc);
  }
}

}  // extern "C"
