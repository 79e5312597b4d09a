// csrc/ekf_detect.cuh — findNewFeatures' mask (vslamRansac.cpp:788-831) and the greedy corner selection of
// goodFeaturesToTrack, as __host__ __device__ code shared by the single filter's detector (ekf_detect.cu), the batched
// detector (ekf_batch_detect.cu) and a host test harness (tests/batch_topup_emu.cu), so that the box geometry and the
// selection order cannot drift apart.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// The box cleared around one patch centre: columns [x0, x0 + w), rows [y0, y0 + h); w = h = 0 when the reference skips the
// centre (V:806).  Float -> int conversions as cv::Rect_<int> makes them.
struct DetBox {
  int x0, y0, w, h;
};
__host__ __device__ inline DetBox det_patch_box(float cx, float cy, int W, int H, int w) {
  if (!(cx > w && cy > w && cx < W - w && cy < H - w)) return DetBox{0, 0, 0, 0};
  const int winSize = 2 * w + 1;
  DetBox b;
  b.x0 = (int)((cx - winSize / 2 > 0) ? cx - winSize / 2 : 0.0f);
  b.y0 = (int)((cy - winSize / 2 > 0) ? cy - winSize / 2 : 0.0f);
  b.w = winSize - ((cx + winSize / 2 <= W) ? 0 : (int)(W - cx - winSize / 2));
  b.h = winSize - ((cy + winSize / 2 <= H) ? 0 : (int)(H - cy - winSize / 2));
  return b;
}
// 255 of the base mask: inside the `estrem` (= window_size) border
__host__ __device__ __forceinline__ bool det_in_base(int x, int y, int W, int H, int estrem) {
  return x >= estrem && x < W - estrem && y >= estrem && y < H - estrem;
}
__host__ __device__ __forceinline__ bool det_in_boxes(int x, int y, const DetBox* boxes, int n) {
  for (int i = 0; i < n; ++i) {
    const DetBox& b = boxes[i];
    if (x >= b.x0 && x < b.x0 + b.w && y >= b.y0 && y < b.y0 + b.h) return true;
  }
  return false;
}
// Sort key of a pixel: score bits above the row-major index.  Non-negative floats order like their bits, and equal scores
// put the higher address first (OpenCV's greaterThanPtr).
__host__ __device__ __forceinline__ unsigned long long det_key(unsigned score_bits, unsigned idx) {
  return ((unsigned long long)score_bits << 32) | idx;
}

// goodFeaturesToTrack's selection for one filter: walk `keys` (sorted descending, zero-padded) in order, skip pixels inside
// one of the filter's boxes, stop at the first score <= thr (all later ones are lower) or once `limit` corners are accepted;
// a corner closer than sqrt(min_dist2) to an accepted one is rejected.  Writes (x, y) pairs to xy, returns their count.
// The keys must hold every candidate of the filter: every 3x3 local maximum of eig inside the base mask with a score above
// thr (see ekf_batch_detect.cu for why that one list serves every filter).
__host__ __device__ inline int det_select_walk(const unsigned long long* keys, int nkeys, int W, unsigned thr_bits,
                                               const DetBox* boxes, int nbox, float min_dist2, int limit, float* xy) {
  int nacc = 0;
  if (limit <= 0) return 0;
  for (int i = 0; i < nkeys; ++i) {
    const unsigned long long k = keys[i];
    if ((unsigned)(k >> 32) <= thr_bits) break;
    const unsigned idx = (unsigned)(k & 0xffffffffull);
    const int px = (int)(idx % (unsigned)W), py = (int)(idx / (unsigned)W);
    if (det_in_boxes(px, py, boxes, nbox)) continue;
    const float x = (float)px, y = (float)py;
    bool bad = false;
    for (int m = 0; m < nacc && !bad; ++m) {
      const float dx = x - xy[2 * m], dy = y - xy[2 * m + 1];
      if (dx * dx + dy * dy < min_dist2) bad = true;
    }
    if (bad) continue;
    xy[2 * nacc] = x; xy[2 * nacc + 1] = y;
    if (++nacc >= limit) break;
  }
  return nacc;
}
