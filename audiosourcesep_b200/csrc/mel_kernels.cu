// Mel-spectrogram front end / back end kernels (see mel_kernels.h).  Semantics follow librosa as the reference calls it
// (restated in oracle/mel_oracle.py): the FFTs run in float64 like numpy's, results are stored as float32 / complex64.
#include "mel_kernels.h"

#include <cmath>
#include <map>
#include <vector>

namespace asep {

namespace {

constexpr double kPi = 3.14159265358979323846;

// twiddle table exp(-2 pi i k / n), k < n/2, per FFT size (device, float64)
std::map<int, double2*> g_twiddles;
const double2* twiddles(int n) {
  auto it = g_twiddles.find(n);
  if (it != g_twiddles.end()) return it->second;
  std::vector<double2> h((size_t)n / 2);
  for (int k = 0; k < n / 2; ++k) h[k] = make_double2(std::cos(-2.0 * kPi * k / n), std::sin(-2.0 * kPi * k / n));
  double2* d = nullptr;
  CUDA_CHECK(cudaMalloc(&d, h.size() * sizeof(double2)));
  CUDA_CHECK(cudaMemcpy(d, h.data(), h.size() * sizeof(double2), cudaMemcpyHostToDevice));
  g_twiddles[n] = d;
  return d;
}

__device__ __forceinline__ unsigned bitrev(unsigned v, int bits) { return __brev(v) >> (32 - bits); }

// in-place radix-2 decimation-in-time FFT of buf[n] (already bit-reversed); inverse: conjugated twiddles, no scaling
__device__ void fft_smem(double2* buf, const double2* __restrict__ tw, int n, int logn, bool inverse) {
  for (int s = 1; s <= logn; ++s) {
    const int half = 1 << (s - 1), stride = n >> s;
    __syncthreads();
    for (int b = threadIdx.x; b < n / 2; b += blockDim.x) {
      const int j = b & (half - 1), k = ((b >> (s - 1)) << s) + j;
      double2 w = tw[j * stride];
      if (inverse) w.y = -w.y;
      const double2 u = buf[k], v = buf[k + half];
      const double2 t = make_double2(w.x * v.x - w.y * v.y, w.x * v.y + w.y * v.x);
      buf[k] = make_double2(u.x + t.x, u.y + t.y);
      buf[k + half] = make_double2(u.x - t.x, u.y - t.y);
    }
  }
  __syncthreads();
}

// grid (T, N): frame t of segment n
__global__ void __launch_bounds__(256) k_stft(const float* __restrict__ audio, float2* __restrict__ out,
                                              const double2* __restrict__ tw, long long L, int n_fft, int logn, int hop, int T) {
  extern __shared__ double2 fbuf[];
  const int t = blockIdx.x, n = blockIdx.y;
  const float* y = audio + (size_t)n * L;
  for (int i = threadIdx.x; i < n_fft; i += blockDim.x) {
    long long g = (long long)t * hop + i - n_fft / 2;
    if (g < 0) g = -g;                                  // np.pad(mode='reflect')
    if (g >= L) g = 2 * (L - 1) - g;
    const double w = 0.5 - 0.5 * cospi(2.0 * (double)i / (double)n_fft);   // periodic Hann
    fbuf[bitrev((unsigned)i, logn)] = make_double2(w * (double)y[g], 0.0);
  }
  fft_smem(fbuf, tw, n_fft, logn, false);
  const int F = n_fft / 2 + 1;
  for (int f = threadIdx.x; f < F; f += blockDim.x)
    out[((size_t)n * F + f) * T + t] = make_float2((float)fbuf[f].x, (float)fbuf[f].y);
}

__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  // monotone mapping of IEEE floats onto signed ints (v is never NaN here)
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// pass 1: log_spec = 10 log10(max(amin, basis . |S|^2)); per-segment maximum.  thread = (n, m, t), t fastest
__global__ void __launch_bounds__(256) k_mel_logspec(const float2* __restrict__ stft, const float* __restrict__ basis,
                                                     const int* __restrict__ lo, const int* __restrict__ hi, float* __restrict__ out,
                                                     float* __restrict__ segmax, int M, int F, int T, float amin, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int t = (int)(i % T), m = (int)((i / T) % M);
  const long long n = i / ((long long)T * M);
  const float2* S = stft + (size_t)n * F * T + t;
  const float* b = basis + (size_t)m * F;
  float acc = 0.f;
  for (int f = lo[m]; f < hi[m]; ++f) {
    const float2 v = S[(size_t)f * T];
    const float a = hypotf(v.x, v.y);                   // np.abs(complex64) ** 2
    acc = fmaf(b[f], a * a, acc);
  }
  const float db = 10.f * log10f(fmaxf(amin, acc));
  out[i] = db;
  atomic_max_float(segmax + n, db);
}

__global__ void __launch_bounds__(256) k_mel_floor_clip(float* __restrict__ out, const float* __restrict__ segmax, long long per_seg,
                                                        float top_db, float dbmin, float dbmax, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float v = fmaxf(out[i], segmax[i / per_seg] - top_db);
  out[i] = fminf(fmaxf(v, dbmin), dbmax);
}

// one block per (frame t, segment n): non-negative least squares of one spectrogram column
__global__ void __launch_bounds__(1024) k_nnls(const float* __restrict__ mel_db, const float* __restrict__ basis,
                                               const float* __restrict__ pinv, const int* __restrict__ flo, const int* __restrict__ fhi,
                                               float* __restrict__ mag, int M, int F, int T, float step, int iters) {
  extern __shared__ float sm[];
  float* b = sm;               // [M]   target power
  float* r = b + M;            // [M]   residual A y - b
  float* y = r + M;            // [F]   extrapolated point
  const int t = blockIdx.x, n = blockIdx.y;
  for (int m = threadIdx.x; m < M; m += blockDim.x) b[m] = exp10f(0.1f * mel_db[((size_t)n * M + m) * T + t]);   // db_to_power
  __syncthreads();
  // per-thread state for the bins it owns (F <= 2 * blockDim.x)
  float x[2] = {0.f, 0.f}, xp[2] = {0.f, 0.f};
  for (int q = 0; q < 2; ++q) {
    const int f = threadIdx.x + q * blockDim.x;
    if (f < F) {
      float a = 0.f;
      for (int m = 0; m < M; ++m) a = fmaf(pinv[(size_t)f * M + m], b[m], a);
      x[q] = xp[q] = fmaxf(a, 0.f);
      y[f] = x[q];
    }
  }
  for (int k = 1; k <= iters; ++k) {
    __syncthreads();
    // residual: every filter m sums its bins (warp per filter, lanes over the bin range)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int m = warp; m < M; m += nw) {
      float a = 0.f;
      // bins of filter m: where basis[m][f] > 0 -- scanned through the per-bin lists' inverse: contiguous range
      const float* row = basis + (size_t)m * F;
      for (int f = lane; f < F; f += 32) {
        const float w = row[f];
        if (w != 0.f) a = fmaf(w, y[f], a);
      }
      a = warp_sum(a);
      if (lane == 0) r[m] = a - b[m];
    }
    __syncthreads();
    const float mom = (float)(k - 1) / (float)(k + 2);
    for (int q = 0; q < 2; ++q) {
      const int f = threadIdx.x + q * blockDim.x;
      if (f < F) {
        float g = 0.f;
        for (int m = flo[f]; m < fhi[f]; ++m) g = fmaf(basis[(size_t)m * F + f], r[m], g);
        const float xn = fmaxf(0.f, y[f] - step * g);
        y[f] = xn + mom * (xn - xp[q]);
        xp[q] = xn;
        x[q] = xn;
      }
    }
  }
  for (int q = 0; q < 2; ++q) {
    const int f = threadIdx.x + q * blockDim.x;
    if (f < F) mag[((size_t)n * F + f) * T + t] = sqrtf(x[q]);          // ^(1 / power), power = 2
  }
}

__global__ void __launch_bounds__(256) k_stft_filter(const float* __restrict__ mag, const float2* __restrict__ mix,
                                                     float2* __restrict__ out, int S, long long NFT, int wiener) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NFT) return;
  const float2 x = mix[i];
  if (wiener) {                                         // melspec_inversion_basis.py:93-119 on psd = mag^2
    float tot = 1e-10f;
    for (int s = 0; s < S; ++s) { const float m = mag[(size_t)s * NFT + i]; tot += m * m; }
    for (int s = 0; s < S; ++s) {
      const float m = mag[(size_t)s * NFT + i];
      const float g = m * m / tot;
      out[(size_t)s * NFT + i] = make_float2(g * x.x, g * x.y);
    }
  } else {                                              // complex_array(amplitudes, np.angle(stft_mixture)), :17-18, :84
    const float a = hypotf(x.x, x.y);
    const float cx = a > 0.f ? x.x / a : 1.f, cy = a > 0.f ? x.y / a : 0.f;     // angle(0) = 0
    for (int s = 0; s < S; ++s) {
      const float m = mag[(size_t)s * NFT + i];
      out[(size_t)s * NFT + i] = make_float2(m * cx, m * cy);
    }
  }
}

// One Griffin-Lim phase update (librosa.griffinlim, the "fast" variant with momentum): angles = rebuilt - m/(1+m) * tprev,
// normalised to unit modulus; next = mag * angles; tprev <- rebuilt.  Element-wise on complex64 arrays.
__global__ void __launch_bounds__(256) k_griffinlim_update(const float* __restrict__ mag, const float2* __restrict__ rebuilt,
                                                           float2* __restrict__ tprev, float2* __restrict__ next, float coef,
                                                           long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float2 r = rebuilt[i], t = tprev[i];
  float ax = r.x - coef * t.x, ay = r.y - coef * t.y;
  const float inv = 1.f / (hypotf(ax, ay) + 1e-16f);
  ax *= inv; ay *= inv;
  const float m = mag[i];
  next[i] = make_float2(m * ax, m * ay);
  tprev[i] = r;
}

// grid (T, N): inverse real FFT of frame t, windowed, to frames [N, T, n_fft]
__global__ void __launch_bounds__(256) k_istft_frames(const float2* __restrict__ stft, float* __restrict__ frames,
                                                      const double2* __restrict__ tw, int n_fft, int logn, int T) {
  extern __shared__ double2 fbuf[];
  const int t = blockIdx.x, n = blockIdx.y;
  const int F = n_fft / 2 + 1;
  for (int i = threadIdx.x; i < n_fft; i += blockDim.x) {
    const int f = i < F ? i : n_fft - i;                // Hermitian extension (irfft ignores the imaginary part of DC / Nyquist)
    const float2 v = stft[((size_t)n * F + f) * T + t];
    double im = i < F ? (double)v.y : -(double)v.y;
    if (i == 0 || i == n_fft / 2) im = 0.0;
    fbuf[bitrev((unsigned)i, logn)] = make_double2((double)v.x, im);
  }
  fft_smem(fbuf, tw, n_fft, logn, true);
  for (int i = threadIdx.x; i < n_fft; i += blockDim.x) {
    const double w = 0.5 - 0.5 * cospi(2.0 * (double)i / (double)n_fft);
    frames[((size_t)n * T + t) * n_fft + i] = (float)(w * fbuf[i].x / (double)n_fft);
  }
}

// sample o of one segment's trimmed iSTFT: windowed frames [T, n_fft] of the segment summed over the (at most n_fft / hop)
// frames covering it, divided by the window sum of squares, in double
__device__ __forceinline__ double ola_sample(const float* __restrict__ seg_frames, long long o, int n_fft, int hop, int T) {
  const long long p = o + n_fft / 2;                    // position in the untrimmed signal
  const int t1 = (int)min((long long)T - 1, p / hop);
  const int t0 = p >= n_fft ? (int)((p - n_fft) / hop + 1) : 0;
  double acc = 0.0, wss = 0.0;
  for (int t = t0; t <= t1; ++t) {
    const int k = (int)(p - (long long)t * hop);
    if (k < 0 || k >= n_fft) continue;
    const double w = 0.5 - 0.5 * cospi(2.0 * (double)k / (double)n_fft);
    acc += (double)seg_frames[(size_t)t * n_fft + k];
    wss += w * w;
  }
  return wss > 1.1754943508222875e-38 ? acc / wss : acc;
}

__global__ void __launch_bounds__(256) k_overlap_add(const float* __restrict__ frames, float* __restrict__ audio, int n_fft, int hop,
                                                     int T, long long out_len, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / out_len, o = i % out_len;
  audio[i] = (float)ola_sample(frames + (size_t)n * T * n_fft, o, n_fft, hop, T);
}

// Whole-track overlap-add: frames [S, n_seg, T, n_fft] -> audio [S, length].  Segment g spans track samples
// [g P, g P + V), V = hop (T - 1), P = V - overlap; 2 overlap < V, so one or two segments cover a sample.  Each covering
// segment contributes its trimmed iSTFT value u_g (ola_sample) with a cross-fade weight c_g: 1 inside the segment, a linear
// ramp over the `overlap` samples it shares with a neighbour (none at either end of the track).  out = sum c_g u_g / sum c_g.
__global__ void __launch_bounds__(256) k_overlap_add_track(const float* __restrict__ frames, float* __restrict__ audio, int n_seg,
                                                           int n_fft, int hop, int T, int overlap, long long length, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long s = i / length, n = i % length;
  const long long V = (long long)hop * (T - 1), P = V - overlap;
  const int last = (int)min((long long)n_seg - 1, n / P);
  double num = 0.0, den = 0.0;
  for (int g = max(0, last - 1); g <= last; ++g) {
    const long long j = n - (long long)g * P;            // position inside segment g
    if (j < 0 || j >= V) continue;
    double c = 1.0;
    if (g > 0 && j < overlap) c = ((double)j + 0.5) / (double)overlap;                 // fade in after segment g - 1
    if (g < n_seg - 1 && j >= P) c = ((double)(V - j) - 0.5) / (double)overlap;       // fade out into segment g + 1
    num += c * ola_sample(frames + ((size_t)s * n_seg + g) * T * n_fft, j, n_fft, hop, T);
    den += c;
  }
  audio[i] = (float)(num / den);
}

int ilog2(int n) { int l = 0; while ((1 << l) < n) ++l; return l; }

}  // namespace

void launch_stft(const float* audio, float* stft, int N, long long L, int n_fft, int hop, cudaStream_t s) {
  ASEP_CHECK(n_fft >= 64 && n_fft <= 4096 && (n_fft & (n_fft - 1)) == 0, ASEP_ERR_UNSUPPORTED, "stft: n_fft = %d (power of two, 64..4096)", n_fft);
  ASEP_CHECK(L > n_fft / 2 && hop >= 1, ASEP_ERR_BAD_ARG, "stft: %lld samples are too few for reflect padding by %d", L, n_fft / 2);
  const int T = 1 + (int)(L / hop);
  static bool attr = false;
  if (!attr) {
    CUDA_CHECK(cudaFuncSetAttribute(k_stft, cudaFuncAttributeMaxDynamicSharedMemorySize, 4096 * (int)sizeof(double2)));
    CUDA_CHECK(cudaFuncSetAttribute(k_istft_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, 4096 * (int)sizeof(double2)));
    attr = true;
  }
  k_stft<<<dim3(T, N), 256, (size_t)n_fft * sizeof(double2), s>>>(audio, reinterpret_cast<float2*>(stft), twiddles(n_fft), L, n_fft,
                                                                  ilog2(n_fft), hop, T);
  ASEP_LAUNCH_CHECK();
}

void launch_mel_db(const float* stft, const float* basis, const int* lo, const int* hi, float* mel_db, int N, int M, int F, int T,
                   float amin, float top_db, float dbmin, float dbmax, cudaStream_t s) {
  float* segmax = nullptr;
  CUDA_CHECK(cudaMallocAsync(&segmax, (size_t)N * sizeof(float), s));
  std::vector<float> init((size_t)N, -INFINITY);
  CUDA_CHECK(cudaMemcpyAsync(segmax, init.data(), (size_t)N * sizeof(float), cudaMemcpyHostToDevice, s));
  CUDA_CHECK(cudaStreamSynchronize(s));                // `init` is a pageable stack-lifetime buffer
  const long long total = (long long)N * M * T;
  k_mel_logspec<<<cdiv(total, 256), 256, 0, s>>>(reinterpret_cast<const float2*>(stft), basis, lo, hi, mel_db, segmax, M, F, T, amin, total);
  ASEP_LAUNCH_CHECK();
  k_mel_floor_clip<<<cdiv(total, 256), 256, 0, s>>>(mel_db, segmax, (long long)M * T, top_db, dbmin, dbmax, total);
  ASEP_LAUNCH_CHECK();
  CUDA_CHECK(cudaFreeAsync(segmax, s));
}

void launch_mel_to_stft(const float* mel_db, const float* basis, const float* pinv, const int* flo, const int* fhi, float* mag, int N,
                        int M, int F, int T, float step, int iters, cudaStream_t s) {
  ASEP_CHECK(F <= 2048 && M <= 512, ASEP_ERR_UNSUPPORTED, "mel_to_stft: F = %d, M = %d", F, M);
  k_nnls<<<dim3(T, N), 1024, (size_t)(2 * M + F) * sizeof(float), s>>>(mel_db, basis, pinv, flo, fhi, mag, M, F, T, step, iters);
  ASEP_LAUNCH_CHECK();
}

void launch_stft_filter(const float* mag, const float* mix, float* out, int S, long long NFT, int wiener, cudaStream_t s) {
  k_stft_filter<<<cdiv(NFT, 256), 256, 0, s>>>(mag, reinterpret_cast<const float2*>(mix), reinterpret_cast<float2*>(out), S, NFT, wiener);
  ASEP_LAUNCH_CHECK();
}

void launch_griffinlim_update(const float* mag, const float* rebuilt, float* tprev, float* next, float momentum, long long n,
                              cudaStream_t s) {
  if (n == 0) return;
  k_griffinlim_update<<<cdiv(n, 256), 256, 0, s>>>(mag, reinterpret_cast<const float2*>(rebuilt), reinterpret_cast<float2*>(tprev),
                                                  reinterpret_cast<float2*>(next), momentum / (1.f + momentum), n);
  ASEP_LAUNCH_CHECK();
}

void launch_istft(const float* stft, float* frames, float* audio, int N, int n_fft, int hop, int T, cudaStream_t s) {
  ASEP_CHECK(n_fft >= 64 && n_fft <= 4096 && (n_fft & (n_fft - 1)) == 0, ASEP_ERR_UNSUPPORTED, "istft: n_fft = %d", n_fft);
  static bool attr = false;
  if (!attr) {
    CUDA_CHECK(cudaFuncSetAttribute(k_istft_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, 4096 * (int)sizeof(double2)));
    attr = true;
  }
  k_istft_frames<<<dim3(T, N), 256, (size_t)n_fft * sizeof(double2), s>>>(reinterpret_cast<const float2*>(stft), frames,
                                                                          twiddles(n_fft), n_fft, ilog2(n_fft), T);
  ASEP_LAUNCH_CHECK();
  const long long out_len = (long long)hop * (T - 1), total = out_len * N;
  k_overlap_add<<<cdiv(total, 256), 256, 0, s>>>(frames, audio, n_fft, hop, T, out_len, total);
  ASEP_LAUNCH_CHECK();
}

void launch_istft_track(const float* stft, float* frames, float* audio, int S, int n_seg, int n_fft, int hop, int T, int overlap,
                        long long length, cudaStream_t s) {
  ASEP_CHECK(n_fft >= 64 && n_fft <= 4096 && (n_fft & (n_fft - 1)) == 0, ASEP_ERR_UNSUPPORTED, "istft_track: n_fft = %d", n_fft);
  static bool attr = false;
  if (!attr) {
    CUDA_CHECK(cudaFuncSetAttribute(k_istft_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, 4096 * (int)sizeof(double2)));
    attr = true;
  }
  k_istft_frames<<<dim3(T, S * n_seg), 256, (size_t)n_fft * sizeof(double2), s>>>(reinterpret_cast<const float2*>(stft), frames,
                                                                                  twiddles(n_fft), n_fft, ilog2(n_fft), T);
  ASEP_LAUNCH_CHECK();
  const long long total = (long long)S * length;
  k_overlap_add_track<<<cdiv(total, 256), 256, 0, s>>>(frames, audio, n_seg, n_fft, hop, T, overlap, length, total);
  ASEP_LAUNCH_CHECK();
}

}  // namespace asep
