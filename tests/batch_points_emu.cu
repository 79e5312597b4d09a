// tests/batch_points_emu.cu — TEST INFRASTRUCTURE.  The batched map export of csrc/ekf_batch.cu (k_batch_points_features) and
// the archive record of k_batch_compact on the CPU, built from the same __host__ __device__ code the kernels run
// (csrc/ekf_points.cuh), so that tests/test_batch_points_emu.py can compare them with a restatement of the oracle's
// getPointsFeatures and removeFeature without a GPU.  The flow mirrors the kernel for one filter: the row count, the zeroed
// matrix, the live rows, then the archived records in archive order, and the clear decision.
// Compiled as HOST code by nvcc (tests build it on the fly); nothing here is shipped.
#include <cstring>

#include "ekf_points.cuh"

extern "C" {

// One filter: N live features (coding, pos, real_index), mu / Sigma (row stride ld) with map_scale = mu[13]; `held` archived
// records (ari, arec: held x PTS_COLS).  out: rows_cap x PTS_COLS.  Returns the row count (and writes nothing when it exceeds
// rows_cap); *clears receives the clear decision.
int emu_points(int N, const int* coding, const int* pos, const int* real_index, const double* mu, const double* Sigma, int ld, int held,
               const int* ari, const double* arec, double* out, int rows_cap, int* clears) {
  const int rows = pts_row_count(N, real_index);
  *clears = pts_clears(held) ? 1 : 0;
  if (rows > rows_cap) return rows;
  std::memset(out, 0, sizeof(double) * PTS_COLS * (size_t)rows_cap);
  const double map_scale = mu[13];
  for (int i = 0; i < N; ++i)
    if (pts_archive_in_range(real_index[i], rows))
      pts_live_row(coding[i], pos[i], mu, Sigma, ld, map_scale, out + (size_t)real_index[i] * PTS_COLS);
  for (int k = 0; k < held; ++k)
    if (pts_archive_in_range(ari[k], rows)) pts_archive_row(arec + (size_t)k * PTS_COLS, map_scale, out + (size_t)ari[k] * PTS_COLS);
  return rows;
}

// The archive record of the feature at state position pos (k_batch_compact), and the archiving rule.
void emu_record(const double* mu, const double* Sigma, int ld, int pos, double* rec) { pts_record(mu, Sigma, ld, pos, rec); }
int emu_archived(int coding, int n_find) { return pts_archived(coding, n_find) ? 1 : 0; }

}  // extern "C"
