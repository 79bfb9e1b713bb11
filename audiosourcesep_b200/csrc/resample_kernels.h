// Band-limited resampling on the device (resample_kernels.cu): resampy's resample_f with the kaiser_best table, the
// resampler librosa.load(path, sr=16000) runs for the reference (datasets/preprocessing.py:9-26).
#pragma once
#include "common.cuh"

namespace asep {

// audio [N, L_in] fp32 -> out [N, L_out] fp32.  time [L_out] float64: resampy's running time register (shared by every
// row); win / delta [nwin] fp32: the interpolation table and its forward differences; scale = min(1, ratio); step: the
// truncated table stride int(scale * 512).  Per output sample: k = int(time), the left wing reads x[k - i] and the
// right wing x[k + 1 + j] with weights win[off + i step] + eta delta[off + i step] (off / eta from the fractional time,
// double arithmetic in resampy's order); accumulation in double.  A time outside [0, L_in) yields NaN.
void launch_resample(const float* audio, const double* time, const float* win, const float* delta, float* out, int N,
                     long long L_in, long long L_out, int nwin, double scale, int step, cudaStream_t s);

}  // namespace asep
