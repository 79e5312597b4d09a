// tests/update_kernels.cu — host entry points that run the dense kernels of the stacked EKF update one at a time on host arrays,
// for tests/test_gpu_update_kernels.py.  Linked with csrc/ekf_update.cu; csrc/ekf_gemm.cu is compiled INTO this file so that both
// tile variants of the downdate GEMM (launch_variant, file-static there) can be called directly, whatever EKF_GEMM_TM the product
// wrapper cached.
//
// Every entry point copies ALL of the caller's buffers to the device (so the regions the kernel must not touch keep the caller's
// canary pattern), runs the existing launch wrapper, synchronises and copies every buffer back.  Returns 0 or a cudaError_t.
#include <cstdint>
#include <cstring>
#include <vector>

#include "ekf_kernels.h"
#include "ekf_factor.cuh"
#include "ekf_gemm.cu"

namespace {

// device buffers of one call, freed on every return path
struct DevBufs {
  std::vector<void*> p;
  ~DevBufs() { for (void* q : p) cudaFree(q); }
  template <class T>
  cudaError_t in(T** d, const T* h, size_t n) {   // allocate and copy in (h may be null: zero-filled)
    *d = nullptr;
    if (n == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(d), n * sizeof(T));
    if (e != cudaSuccess) return e;
    p.push_back(*d);
    return h ? cudaMemcpy(*d, h, n * sizeof(T), cudaMemcpyHostToDevice) : cudaMemset(*d, 0, n * sizeof(T));
  }
};

template <class T>
cudaError_t out(T* h, const T* d, size_t n) { return (h && d && n) ? cudaMemcpy(h, d, n * sizeof(T), cudaMemcpyDeviceToHost) : cudaSuccess; }

cudaError_t finish() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return cudaDeviceSynchronize();
}

#define UK_CHECK(x) do { const cudaError_t _e = (x); if (_e != cudaSuccess) return (int)_e; } while (0)

// the batched filter's factor (ekf_batch.cu runs cta_chol_panel<64> on shared-memory operands; here they are in global memory)
__global__ void __launch_bounds__(FACT_THREADS) k_uk_chol_panel64(const double* Sb, int lds, const double* nu, double* Lout, int ldl,
                                                                   double* Dout, int ldd, double* yout, int* chol_fail) {
  extern __shared__ __align__(16) double uk_sm[];
  cta_chol_panel<64>(uk_sm, Sb, lds, nu, Lout, ldl, Dout, ldd, yout, chol_fail);
}

}  // namespace

extern "C" {

// update_kernels_init(): re-reads EKF_CHOL_SMEM (0: cta_chol128 in registers, 1: cta_chol_panel<128> in shared memory)
int uk_init() { return update_kernels_init(); }

// One 128-row block factor through the product's wrappers.  which 0: launch_blk_factor_only, 1: launch_blk_factor_wait with its
// flag raised before the launch.  S, L: 128 x 128 (ld 128); D: 4 x 32 x 32; nu, y: 128.  L, D, y are copied in and out.
int uk_factor128(int which, const double* S, const double* nu, double* L, double* D, double* y, int* chol_fail) {
  DevBufs b;
  double *dS, *dnu, *dL, *dD, *dy;
  DevCtl* ctl;
  unsigned int* flag;
  const unsigned int token = 0x5a5a0001u;
  UK_CHECK(b.in(&dS, S, 128 * 128));
  UK_CHECK(b.in(&dnu, nu, 128));
  UK_CHECK(b.in(&dL, L, 128 * 128));
  UK_CHECK(b.in(&dD, D, 128 * 32));
  UK_CHECK(b.in(&dy, y, 128));
  UK_CHECK(b.in(&ctl, (const DevCtl*)nullptr, 1));
  UK_CHECK(b.in(&flag, &token, 1));
  long long launches = 0;
  if (which == 0) launch_blk_factor_only(nullptr, dS, dnu, dL, dD, dy, ctl, &launches);
  else if (which == 1) launch_blk_factor_wait(nullptr, dS, dnu, dL, dD, dy, ctl, flag, token, &launches);
  else return (int)cudaErrorInvalidValue;
  UK_CHECK(finish());
  UK_CHECK(out(L, dL, 128 * 128));
  UK_CHECK(out(D, dD, 128 * 32));
  UK_CHECK(out(y, dy, 128));
  DevCtl h;
  UK_CHECK(out(&h, ctl, 1));
  *chol_fail = h.chol_fail;
  return 0;
}

// cta_chol_panel<64>, the batched filter's factor.  S: 64 x lds, L: 64 x ldl, D: 2 x 32 x ldd; alias != 0: L is written over S
// (as in ekf_batch.cu), and the L argument is ignored.
int uk_factor64(double* S, int lds, const double* nu, double* L, int ldl, int alias, double* D, int ldd, double* y, int* chol_fail) {
  DevBufs b;
  double *dS, *dnu, *dL = nullptr, *dD, *dy;
  int* dfail;
  UK_CHECK(b.in(&dS, S, (size_t)64 * lds));
  UK_CHECK(b.in(&dnu, nu, 64));
  if (!alias) UK_CHECK(b.in(&dL, L, (size_t)64 * ldl));
  UK_CHECK(b.in(&dD, D, (size_t)64 * ldd));
  UK_CHECK(b.in(&dy, y, 64));
  UK_CHECK(b.in(&dfail, (const int*)nullptr, 1));
  const size_t smem = (size_t)cta_chol_panel_smem_doubles<64>() * sizeof(double);
  UK_CHECK(cudaFuncSetAttribute(k_uk_chol_panel64, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_uk_chol_panel64<<<1, FACT_THREADS, smem>>>(dS, lds, dnu, alias ? dS : dL, alias ? lds : ldl, dD, ldd, dy, dfail);
  UK_CHECK(finish());
  UK_CHECK(out(alias ? S : L, alias ? dS : dL, (size_t)64 * (alias ? lds : ldl)));
  UK_CHECK(out(D, dD, (size_t)64 * ldd));
  UK_CHECK(out(y, dy, 64));
  UK_CHECK(out(chol_fail, dfail, 1));
  return 0;
}

// launch_blk_V on rows [rbase, n) of W (rows x 128).  delta (rows) may be null; vout != 0: V goes to Vout (rows x 128) and W stays;
// delta_in (rows) may be null.  Every buffer that is passed is copied in and out.
int uk_blk_V(double* W, int rows, int rbase, int n, const double* L, const double* D, const double* y, double* delta, double* Vout,
             const double* delta_in) {
  DevBufs b;
  double *dW, *dL, *dD, *dy, *dd = nullptr, *dV = nullptr, *ddi = nullptr;
  UK_CHECK(b.in(&dW, W, (size_t)rows * 128));
  UK_CHECK(b.in(&dL, L, 128 * 128));
  UK_CHECK(b.in(&dD, D, 128 * 32));
  UK_CHECK(b.in(&dy, y, 128));
  if (delta) UK_CHECK(b.in(&dd, delta, rows));
  if (Vout) UK_CHECK(b.in(&dV, Vout, (size_t)rows * 128));
  if (delta_in) UK_CHECK(b.in(&ddi, delta_in, rows));
  long long launches = 0;
  launch_blk_V(nullptr, dW, rbase, n, dL, dD, dy, dd, &launches, dV, ddi);
  UK_CHECK(finish());
  UK_CHECK(out(W, dW, (size_t)rows * 128));
  UK_CHECK(out(delta, dd, rows));
  UK_CHECK(out(Vout, dV, (size_t)rows * 128));
  return 0;
}

// C[c_off ..] -= A[a_off ..] B^T through the downdate GEMM.  tm 0: the product wrapper launch_gemm_nt_sub (tile shape from
// EKF_GEMM_TM, 64 x 64 by default); tm 64 / 128: that tile variant directly.  use_kdev: K is read from device memory (kconst is
// then passed as 0, so a kernel that ignored kdev would do nothing).  tlist (2 x n_tiles: tile row, tile column) with n_hot: the
// tile-list grid; *hot_counter returns the counter the kernel bumps.
int uk_gemm(int tm, double* C, long long c_len, int ldc, long long c_off, const double* A, long long a_len, int lda, long long a_off,
            const double* B, long long b_len, int ldb, int M, int N, int K, int use_kdev, int lower_only, const unsigned short* tlist,
            int n_tiles, int n_hot, unsigned int* hot_counter) {
  DevBufs b;
  double *dC, *dA, *dB;
  int *dk = nullptr, *dnh = nullptr;
  ushort2* dt = nullptr;
  unsigned int* dhc = nullptr;
  UK_CHECK(b.in(&dC, C, (size_t)c_len));
  UK_CHECK(b.in(&dA, A, (size_t)a_len));
  UK_CHECK(b.in(&dB, B, (size_t)b_len));
  if (use_kdev) UK_CHECK(b.in(&dk, &K, 1));
  if (tlist) {
    static_assert(sizeof(ushort2) == 2 * sizeof(unsigned short), "ushort2");
    UK_CHECK(b.in(&dt, reinterpret_cast<const ushort2*>(tlist), (size_t)n_tiles));
    UK_CHECK(b.in(&dnh, &n_hot, 1));
    UK_CHECK(b.in(&dhc, (const unsigned int*)nullptr, 1));
  }
  const int kc = use_kdev ? 0 : K;
  long long launches = 0;
  int rc;
  if (tm == 0)
    rc = launch_gemm_nt_sub(nullptr, dC + c_off, ldc, dA + a_off, lda, dB, ldb, M, N, kc, dk, lower_only, nullptr, &launches, dt, n_tiles, dnh, dhc);
  else if (tm == 64)
    rc = launch_variant<64, 2, 4>(nullptr, dC + c_off, ldc, dA + a_off, lda, dB, ldb, M, N, kc, dk, lower_only, 0u, dt, n_tiles, dnh, dhc);
  else if (tm == 128 && !tlist)
    rc = launch_variant<128, 3, 2>(nullptr, dC + c_off, ldc, dA + a_off, lda, dB, ldb, M, N, kc, dk, lower_only, 0u);
  else
    return (int)cudaErrorInvalidValue;
  if (rc) return rc;
  UK_CHECK(finish());
  UK_CHECK(out(C, dC, (size_t)c_len));
  UK_CHECK(out(hot_counter, dhc, 1));
  return 0;
}

// launch_blk_Sg: Sg (128 x 128, copied in and out) gets -G G^T on its lower 32 x 32 blocks.  G: 128 x 128.
int uk_blk_Sg(const double* G, double* Sg) {
  DevBufs b;
  double *dG, *dS;
  UK_CHECK(b.in(&dG, G, 128 * 128));
  UK_CHECK(b.in(&dS, Sg, 128 * 128));
  long long launches = 0;
  launch_blk_Sg(nullptr, dG, dS, &launches);
  UK_CHECK(finish());
  UK_CHECK(out(Sg, dS, 128 * 128));
  return 0;
}

// launch_delta_rows: delta[i] += V[i, :] y for i < n.  V: rows x 128, delta: rows (copied in and out), y: 128.
int uk_delta_rows(const double* V, int rows, const double* y, double* delta, int n) {
  DevBufs b;
  double *dV, *dy, *dd;
  UK_CHECK(b.in(&dV, V, (size_t)rows * 128));
  UK_CHECK(b.in(&dy, y, 128));
  UK_CHECK(b.in(&dd, delta, rows));
  long long launches = 0;
  launch_delta_rows(nullptr, dV, dy, dd, n, &launches);
  UK_CHECK(finish());
  UK_CHECK(out(delta, dd, rows));
  return 0;
}

}  // extern "C"
