// Band-limited resampling (see resample_kernels.h).  Semantics: resampy.resample(filter='kaiser_best'), restated in
// oracle/resample_oracle.py.  One thread per output sample; a block keeps the interpolation table `win` in shared memory
// for its whole life and walks tiles of consecutive outputs (grid = resident blocks), so the 128 KB table is staged once
// per block instead of once per tile.  `delta` is read through the read-only cache: the two tables together (256 KB) do
// not fit in shared memory.
#include "resample_kernels.h"

#include <cmath>

namespace asep {

namespace {

constexpr int kThreads = 512;
constexpr double kNumTable = 512.0;      // 2^precision of kaiser_best (precision = 9): table entries per zero crossing

__global__ void __launch_bounds__(kThreads) k_resample(const float* __restrict__ x, const double* __restrict__ time,
                                                       const float* __restrict__ win, const float* __restrict__ delta,
                                                       float* __restrict__ y, long long L_in, long long L_out,
                                                       long long tiles_per_row, long long n_tiles, int nwin, double scale,
                                                       int step) {
  extern __shared__ float s_win[];
  for (int i = threadIdx.x; i < nwin; i += blockDim.x) s_win[i] = win[i];
  __syncthreads();
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long row = tile / tiles_per_row;
    const long long t = (tile - row * tiles_per_row) * kThreads + threadIdx.x;
    if (t >= L_out) continue;
    const float* xr = x + row * L_in;
    const double T = time[t];
    float out = NAN;
    if (T >= 0.0 && T < (double)L_in) {
      // resampy resample_f, in its operation order; the _rn intrinsics keep the compiler from contracting them
      const long long k = (long long)T;
      double frac = __dmul_rn(scale, __dsub_rn(T, (double)k));
      double idx = __dmul_rn(frac, kNumTable);
      int off = (int)idx;
      double eta = __dsub_rn(idx, (double)off);
      double acc = 0.0;
      const int imax = (int)min(k + 1, (long long)((nwin - off) / step));
      for (int i = 0; i < imax; ++i) {
        const int o = off + i * step;
        acc += ((double)s_win[o] + eta * (double)__ldg(delta + o)) * (double)__ldg(xr + (k - i));
      }
      frac = __dsub_rn(scale, frac);
      idx = __dmul_rn(frac, kNumTable);
      off = (int)idx;
      eta = __dsub_rn(idx, (double)off);
      const int jmax = (int)min(L_in - k - 1, (long long)((nwin - off) / step));
      for (int j = 0; j < jmax; ++j) {
        const int o = off + j * step;
        acc += ((double)s_win[o] + eta * (double)__ldg(delta + o)) * (double)__ldg(xr + (k + 1 + j));
      }
      out = (float)acc;
    }
    y[row * L_out + t] = out;
  }
}

}  // namespace

void launch_resample(const float* audio, const double* time, const float* win, const float* delta, float* out, int N,
                     long long L_in, long long L_out, int nwin, double scale, int step, cudaStream_t s) {
  if (N == 0 || L_out == 0) return;
  const size_t smem = (size_t)nwin * sizeof(float);
  int dev = 0, smem_max = 0, n_sm = 0;
  CUDA_CHECK(cudaGetDevice(&dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  ASEP_CHECK(smem <= (size_t)smem_max, ASEP_ERR_UNSUPPORTED, "resample: a table of %d entries exceeds shared memory (%d bytes)",
             nwin, smem_max);
  CUDA_CHECK(cudaFuncSetAttribute(k_resample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_resample, kThreads, smem));
  ASEP_CHECK(per_sm >= 1, ASEP_ERR_UNSUPPORTED, "resample: kernel does not fit on an SM");
  const long long tiles_per_row = (L_out + kThreads - 1) / kThreads, n_tiles = tiles_per_row * N;
  const int grid = (int)std::min<long long>(n_tiles, (long long)per_sm * n_sm);
  k_resample<<<grid, kThreads, smem, s>>>(audio, time, win, delta, out, L_in, L_out, tiles_per_row, n_tiles, nwin, scale, step);
  ASEP_LAUNCH_CHECK();
}

}  // namespace asep
