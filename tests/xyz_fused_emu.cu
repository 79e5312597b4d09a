// tests/xyz_fused_emu.cu — TEST INFRASTRUCTURE.  Runs the two functions the fused removal + XYZ-conversion pass of the
// batched filters is built from (csrc/ekf_math.cuh: xyz_linear_decide, xyz_apply_entry — the same __host__ __device__ code
// k_batch_update / k_batch_xyz_decide and k_batch_compact execute) on the CPU, so that tests/test_xyz_fused_emu.py can
// compare one fused pass with the oracle's removeFeature calls followed by convert2XYZ_ifLinearAll, bit for bit, without a
// GPU.  The flow mirrors the kernels: decisions on the pre-removal state for every surviving inverse-depth feature, then one
// (src, code) row map over the survivors in order, then Sigma' = J Sigma J^T and mu' entry by entry.
// Compiled as HOST code by nvcc (tests build it on the fly); nothing here is shipped.
#include <cstdlib>
#include <vector>

#include "ekf_math.cuh"

extern "C" {

// n x n state (mu, Sigma row-major, ld = n) with N features (pos, coding); removed[f] != 0 drops feature f.
// Writes the new state (mu_out, Sigma_out with ld = n2) and table (pos_out, coding_out, N2 entries); returns n2.
int emu_remove_convert(int n, int N, const double* mu, const double* Sigma, const int* pos, const int* coding, const int* removed,
                       double threshold, int abs_int_quirk, double* mu_out, double* Sigma_out, int* pos_out, int* coding_out,
                       int* N_out) {
  std::vector<double> Jall(18 * (size_t)(N > 0 ? N : 1)), yall(3 * (size_t)(N > 0 ? N : 1));
  std::vector<int> conv(N, 0);
  for (int f = 0; f < N; ++f)
    if (!removed[f] && !coding[f])
      conv[f] = xyz_linear_decide(mu + pos[f], mu, Sigma[(size_t)(pos[f] + 5) * n + pos[f] + 5], threshold, abs_int_quirk,
                                  yall.data() + 3 * f, Jall.data() + 18 * f);
  std::vector<int2> rmap;
  for (int i = 0; i < EKF_CAM; ++i) rmap.push_back(make_int2(i, -1));
  int N2 = 0;
  for (int f = 0; f < N; ++f) {
    if (removed[f]) continue;
    pos_out[N2] = (int)rmap.size();
    coding_out[N2] = conv[f] ? 1 : coding[f];
    ++N2;
    if (conv[f]) {
      for (int x = 0; x < 3; ++x) rmap.push_back(make_int2(pos[f], 4 * f + x));
    } else {
      for (int c = 0; c < (coding[f] ? 3 : 6); ++c) rmap.push_back(make_int2(pos[f] + c, -1));
    }
  }
  const int n2 = (int)rmap.size();
  for (int i = 0; i < n2; ++i) {
    for (int j = 0; j < n2; ++j) Sigma_out[(size_t)i * n2 + j] = xyz_apply_entry(Sigma, n, rmap[i], rmap[j], Jall.data());
    const int2 r = rmap[i];
    mu_out[i] = (r.y < 0) ? mu[r.x] : yall[3 * (r.y >> 2) + (r.y & 3)];
  }
  *N_out = N2;
  return n2;
}

}  // extern "C"
