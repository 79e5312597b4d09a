// csrc/ekf_points.cuh — the row assembly of RosVSLAM::getPointsFeatures (RosVSLAMRansac.cpp:340-418) and the archive record of
// removeFeature (vslamRansac.cpp:394-404) for the batched filters, as __host__ __device__ functions: k_batch_points_features and
// k_batch_compact (ekf_batch.cu) call them, and tests/batch_points_emu.cu runs the same code on the host.
//
// A record is 12 doubles, XYZ_pos[3] then cov_4_delete[9], beside its real_index.  cov_4_delete is
// Sigma.block<3,3>(pos, pos).transpose() copied in Eigen's column-major linear order, which is the block row by row, as
// remove_features (ekf_api.cu) and the oracle's removeFeature build it.  A points row is the same 12 doubles with the position
// scaled by map_scale = mu[13].
#pragma once

#define PTS_COLS 12
#define PTS_CLEAR_ABOVE 7000   // RosVSLAMRansac.cpp:395-403: more archived patches than this are cleared after an export

// Rows of the matrix: real_index of the last live feature + 1, or 1 without features (R:349 reads patches[size - 1] unguarded).
__host__ __device__ inline int pts_row_count(int N, const int* real_index) { return (N > 0 ? real_index[N - 1] : 0) + 1; }

// removeFeature archives a feature when it is XYZ and was found more than five times (V:394-404).
__host__ __device__ inline bool pts_archived(int coding, int n_find) { return coding == 1 && n_find > 5; }

// The archive record of the XYZ feature at state position pos, read from mu and Sigma (row stride ld) before the removal.
__host__ __device__ inline void pts_record(const double* mu, const double* Sigma, int ld, int pos, double* rec) {
  for (int c = 0; c < 3; ++c) rec[c] = mu[pos + c];
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) rec[3 + c * 3 + r] = Sigma[(size_t)(pos + c) * ld + pos + r];
}

// The row of a live feature: XYZ features write position * map_scale and the 3 x 3 block row by row; inverse-depth features
// leave their row as it is (zero, R:357-367).  Returns whether it wrote.
__host__ __device__ inline bool pts_live_row(int coding, int pos, const double* mu, const double* Sigma, int ld, double map_scale,
                                             double* row) {
  if (!coding) return false;
  for (int c = 0; c < 3; ++c) row[c] = mu[pos + c] * map_scale;
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) row[3 + a * 3 + b] = Sigma[(size_t)(pos + a) * ld + pos + b];
  return true;
}

// An archived record's row, written after every live row and in archive order.  A record whose real_index lies past the
// matrix (its feature was newer than the last live one) is dropped, as the single filter and the oracle drop it.
__host__ __device__ inline bool pts_archive_in_range(int real_index, int rows) { return real_index >= 0 && real_index < rows; }
__host__ __device__ inline void pts_archive_row(const double* rec, double map_scale, double* row) {
  for (int c = 0; c < 9; ++c) row[3 + c] = rec[3 + c];
  for (int c = 0; c < 3; ++c) row[c] = rec[c] * map_scale;
}

// The reference clears deleted_patches after an export when it holds more than 7000 records.
__host__ __device__ inline bool pts_clears(int archived) { return archived > PTS_CLEAR_ABOVE; }
