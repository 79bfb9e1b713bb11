// Mel-spectrogram front end and inversion back end on the device (mel_kernels.cu).  Reference call sites:
// datasets/data_loader.py:144-162 (librosa.stft -> melspectrogram -> power_to_db -> clip) and
// melspec_inversion_basis.py:42-119 (db_to_power -> mel_to_stft -> phase re-use / Wiener filter -> istft).
#pragma once
#include "common.cuh"

namespace asep {

// audio [N, L] fp32 -> stft [N, F = n_fft/2+1, T = 1 + L/hop] complex64 (interleaved re, im); periodic Hann window,
// centred frames with reflect padding, one float64 radix-2 FFT per frame in shared memory.  n_fft: power of two <= 4096.
void launch_stft(const float* audio, float* stft, int N, long long L, int n_fft, int hop, cudaStream_t s);
// mel_db [N, M, T] <- clip(power_to_db(mel_basis |stft|^2), dbmin, dbmax) with librosa's top_db floor taken per segment;
// basis [M, F] fp32 (dense), lo / hi [M]: the non-zero bin range of every filter.
void launch_mel_db(const float* stft, const float* basis, const int* lo, const int* hi, float* mel_db, int N, int M, int F, int T,
                   float amin, float top_db, float dbmin, float dbmax, cudaStream_t s);
// mag [N, F, T] <- (argmin_{X >= 0} ||basis X - 10^(mel_db/10)||^2)^(1/2): X0 = clip(pinv . B), `iters` FISTA projected
// gradient steps of size `step`; pinv [F, M]; flo / fhi [F]: the filters that contain each bin.
void launch_mel_to_stft(const float* mel_db, const float* basis, const float* pinv, const int* flo, const int* fhi, float* mag, int N,
                        int M, int F, int T, float step, int iters, cudaStream_t s);
// out [S, N, F, T] complex64: wiener = 1: mag^2 / (sum_s mag^2 + 1e-10) * mix; wiener = 0: mag * mix / |mix| (phase re-use)
void launch_stft_filter(const float* mag, const float* mix, float* out, int S, long long NFT, int wiener, cudaStream_t s);
// one Griffin-Lim iteration's phase update (librosa.griffinlim with momentum): next = mag * unit(rebuilt - m/(1+m) tprev),
// tprev <- rebuilt; all complex64 [n] (interleaved), mag fp32 [n]
void launch_griffinlim_update(const float* mag, const float* rebuilt, float* tprev, float* next, float momentum, long long n,
                              cudaStream_t s);
// stft [N, F, T] complex64 -> audio [N, hop * (T - 1)]: windowed overlap-add of the inverse FFT frames divided by the
// window sum of squares, n_fft/2 samples trimmed at both ends (librosa.istft, center = True); frames: scratch [N, T, n_fft]
void launch_istft(const float* stft, float* frames, float* audio, int N, int n_fft, int hop, int T, cudaStream_t s);
// stft [S, n_seg, F, T] complex64 of overlapping segments of one track (segment g starts at sample g P, P = hop (T-1) -
// overlap) -> audio [S, length]: each segment's iSTFT value as launch_istft computes it, cross-faded linearly over the
// `overlap` samples two neighbours share (hard cut when overlap = 0) and written straight into the track; the caller
// guarantees 0 <= 2 overlap < hop (T-1) and length <= (n_seg-1) P + hop (T-1).  frames: scratch [S, n_seg, T, n_fft]
void launch_istft_track(const float* stft, float* frames, float* audio, int S, int n_seg, int n_fft, int hop, int T, int overlap,
                        long long length, cudaStream_t s);

}  // namespace asep
