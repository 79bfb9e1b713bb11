// Rendering a whole-track separation as multichannel Wiener masks on the original recording (mwf_kernels.cu); restated in
// oracle/mwf_oracle.py.
#pragma once
#include "common.cuh"

namespace asep {

constexpr int kMwfMaxIterations = 10;   // k_mwf streams a row iterations + 1 times and keeps every iteration's R in shared memory

// psd [K, F_out, T_out] <- the K sources' segment magnitudes mag [K, n_seg, F, T] (16 kHz grid, segment hop `hop`,
// neighbours sharing `overlap` frames) as one cross-faded track power per 16 kHz frame, bilinearly mapped onto the output
// STFT grid of out_sr / out_n_fft / out_hop with the 16 kHz bin clamped to [bin_lo, bin_hi].  The caller guarantees
// 2 <= K, 0 <= 2 overlap < T - 1 and 0 <= bin_lo <= bin_hi < F.
void launch_track_psd(const float* mag, float* psd, int K, int n_seg, int F, int T, int hop, int overlap, int bin_lo, int bin_hi,
                      int out_sr, int out_n_fft, int out_hop, int F_out, int T_out, cudaStream_t s);
// out [K, C, F, T] complex64 <- the multichannel Wiener filter with `iterations` EM steps and mixture consistency of the
// mixture stft [C, F, T] complex64 under the source powers psd [K, F, T]; one CTA per frequency row, float64 algebra.
// The caller guarantees 2 <= K <= 8, C in {1, 2}, 0 <= iterations <= kMwfMaxIterations.
void launch_mwf(const float* psd, const float* mix, float* out, int K, int C, int F, int T, int iterations, cudaStream_t s);

}  // namespace asep
