// Multichannel Wiener-mask rendering of a whole-track separation (see mwf_kernels.h; oracle/mwf_oracle.py).
//
// This file is compiled with -fmad=false (Makefile): k_mwf relies on products being rounded before they are added, so that
// bitwise-equal channels (dual-mono input) give bitwise-equal entries R00 = R11 = Re R01, Im R01 = 0, an exactly zero
// det(M) and an exactly zero adj(M) x.  A fused multiply-add would expose the rounding error of one product and let the
// eps I regulariser's inverse leak into the gains.
#include "mwf_kernels.h"

namespace asep {

namespace {

constexpr double kEps = 1e-10;          // the regulariser of the single-channel Wiener filter (k_stft_filter)
constexpr long long kModelSr = 16000;   // the rate of the mel grid the separated magnitudes live on
constexpr int kMwfThreads = 128;

struct PsdGrid {
  int K, n_seg, F, T, hop, overlap, bin_lo, bin_hi, out_sr, out_n_fft, out_hop, F_out, T_out, T16;
};

// The one or two segment frames holding 16 kHz track frame tau, with their cross-fade weights (the weight of the frame's
// centre sample, as k_overlap_add_track's ramps give it) normalised to sum to one.  The same for every source and bin.
struct FrameMix {
  int s0, j0, s1, j1;  // s1 < 0: one segment holds the frame
  double w0, w1;
};

__device__ FrameMix frame_mix(const PsdGrid& g, int tau) {
  const int Q = g.T - 1 - g.overlap;                    // frames between segment starts
  const int last = min(g.n_seg - 1, tau / Q);
  const double V = (double)g.hop * (g.T - 1), O = (double)g.hop * g.overlap, P = V - O;
  FrameMix m{-1, 0, -1, 0, 0.0, 0.0};
  double den = 0.0;
  for (int s = max(0, last - 1); s <= last; ++s) {
    const int j = tau - s * Q;
    if (j < 0 || j >= g.T) continue;
    const double p = (double)g.hop * j;                 // the frame's centre, in samples from the segment start
    double w = 1.0;
    if (s > 0 && g.overlap > 0 && p < O) w = (p + 0.5) / O;
    if (s < g.n_seg - 1 && p >= P) w = g.overlap > 0 ? fmax(0.0, (V - p - 0.5) / O) : 0.0;
    if (m.s0 < 0) { m.s0 = s; m.j0 = j; m.w0 = w; }
    else { m.s1 = s; m.j1 = j; m.w1 = w; }
    den += w;
  }
  m.w0 /= den;                                          // den > 0: the segment starting last before tau weighs > 0
  m.w1 /= den;
  return m;
}

// cross-faded power of one source (mag_k [n_seg, F, T]) at one track frame and 16 kHz bin
__device__ __forceinline__ double frame_power(const float* __restrict__ mag_k, const PsdGrid& g, const FrameMix& m, int bin) {
  const double a = (double)mag_k[((size_t)m.s0 * g.F + bin) * g.T + m.j0];
  double pw = m.w0 * (a * a);
  if (m.s1 >= 0) {
    const double b = (double)mag_k[((size_t)m.s1 * g.F + bin) * g.T + m.j1];
    pw += m.w1 * (b * b);
  }
  return pw;
}

// one thread per output bin and frame (b', u), u fastest; the grid position and the frame weights serve every source
__global__ void __launch_bounds__(256) k_track_psd(const float* __restrict__ mag, float* __restrict__ psd, PsdGrid g,
                                                   long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int u = (int)(i % g.T_out), b = (int)(i / g.T_out);
  const int n16 = 2 * (g.F - 1);
  double q = (double)((long long)u * g.out_hop * kModelSr) / (double)((long long)g.out_sr * g.hop);
  q = fmin(fmax(q, 0.0), (double)(g.T16 - 1));
  const int q0 = (int)floor(q), q1 = min(q0 + 1, g.T16 - 1);
  const double a = q - q0;
  double p = (double)((long long)b * g.out_sr * n16) / (double)((long long)g.out_n_fft * kModelSr);
  p = fmin(fmax(p, (double)g.bin_lo), (double)g.bin_hi);
  const int p0 = (int)floor(p), p1 = min(p0 + 1, g.bin_hi);
  const double beta = p - p0;
  const FrameMix m0 = frame_mix(g, q0), m1 = frame_mix(g, q1);
  for (int k = 0; k < g.K; ++k) {
    const float* mk = mag + (size_t)k * g.n_seg * g.F * g.T;
    const double r0 = frame_power(mk, g, m0, p0) * (1.0 - beta) + frame_power(mk, g, m0, p1) * beta;
    const double r1 = frame_power(mk, g, m1, p0) * (1.0 - beta) + frame_power(mk, g, m1, p1) * beta;
    psd[(size_t)k * total + i] = (float)(r0 * (1.0 - a) + r1 * a);
  }
}

// out = R w for one source: C = 1: R [R0]; C = 2: R = [[R0, R2 + i R3], [R2 - i R3, R1]] (Hermitian)
template <int C>
__device__ __forceinline__ void apply_r(const double* R, const double* wr, const double* wi, double* outr, double* outi) {
  if (C == 1) {
    outr[0] = R[0] * wr[0];
    outi[0] = R[0] * wi[0];
  } else {
    outr[0] = R[0] * wr[0] + (R[2] * wr[1] - R[3] * wi[1]);
    outi[0] = R[0] * wi[0] + (R[2] * wi[1] + R[3] * wr[1]);
    outr[1] = (R[2] * wr[0] + R[3] * wi[0]) + R[1] * wr[1];
    outi[1] = (R[2] * wi[0] - R[3] * wr[0]) + R[1] * wi[1];
  }
}

// One bin's EM chain.  After `steps` steps source k's estimate is y_k = a_k (B_k w) + r with B_k = I at step 0 and the
// row's R_k of that iteration afterwards, w = x at step 0 and C_xx^-1 x afterwards, r the residual share (x - sum_k
// a_k B_k w) / K.  Everything but the row's R's is per-bin, so the chain is recomputed instead of stored.
template <int K, int C>
struct Chain {
  double xr[C], xi[C], a[K], wr[C], wi[C], rr[C], ri[C];
  int step;

  __device__ __forceinline__ void source(const double (*R)[K][4], int k, double* yr, double* yi) const {
    double br[C], bi[C];
    if (step == 0) {
#pragma unroll
      for (int c = 0; c < C; ++c) { br[c] = wr[c]; bi[c] = wi[c]; }
    } else {
      apply_r<C>(R[step][k], wr, wi, br, bi);
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      yr[c] = a[k] * br[c] + rr[c];
      yi[c] = a[k] * bi[c] + ri[c];
    }
  }

  // residual share of the pre-consistency estimates a_k B_k w
  __device__ __forceinline__ void consistency(const double (*R)[K][4]) {
#pragma unroll
    for (int c = 0; c < C; ++c) { rr[c] = 0.0; ri[c] = 0.0; }
    double sr[C], si[C];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double yr[C], yi[C];
      source(R, k, yr, yi);                             // rr = ri = 0 here: the pre-consistency estimate
#pragma unroll
      for (int c = 0; c < C; ++c) {
        sr[c] = k == 0 ? yr[c] : sr[c] + yr[c];
        si[c] = k == 0 ? yi[c] : si[c] + yi[c];
      }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      rr[c] = (xr[c] - sr[c]) / (double)K;
      ri[c] = (xi[c] - si[c]) / (double)K;
    }
  }

  __device__ void init(const double* v) {
    double s = v[0];
#pragma unroll
    for (int k = 1; k < K; ++k) s += v[k];
    s += kEps;
#pragma unroll
    for (int k = 0; k < K; ++k) a[k] = v[k] / s;
#pragma unroll
    for (int c = 0; c < C; ++c) { wr[c] = xr[c]; wi[c] = xi[c]; }
    step = 0;
    consistency(nullptr);
  }

  // one EM step with the row's R_k of iteration p = step + 1
  __device__ void advance(const double (*R)[K][4]) {
    double v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double yr[C], yi[C];
      source(R, k, yr, yi);
      double e = yr[0] * yr[0] + yi[0] * yi[0];
      if (C == 2) e += yr[1] * yr[1] + yi[1] * yi[1];
      v[k] = e / (double)C;
    }
    const int p = step + 1;
    double m[4] = {0.0, 0.0, 0.0, 0.0};                 // M = sum_k v_k R_k
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int e = 0; e < (C == 2 ? 4 : 1); ++e) m[e] += v[k] * R[p][k][e];
    // z = (M + eps I)^-1 x = (adj(M) x + eps x) / (max(det M, 0) + eps tr M + eps^2)
    if (C == 1) {
      const double d = m[0] + kEps;
      wr[0] = xr[0] / d;
      wi[0] = xi[0] / d;
    } else {
      const int c1 = C - 1;                             // == 1; keeps the indices in range for the C = 1 instantiation
      const double det = fmax(m[0] * m[1] - (m[2] * m[2] + m[3] * m[3]), 0.0) + kEps * (m[0] + m[1]) + kEps * kEps;
      const double z0r = m[1] * xr[0] - (m[2] * xr[c1] - m[3] * xi[c1]) + kEps * xr[0];
      const double z0i = m[1] * xi[0] - (m[2] * xi[c1] + m[3] * xr[c1]) + kEps * xi[0];
      const double z1r = (-m[2] * xr[0] - m[3] * xi[0]) + m[0] * xr[c1] + kEps * xr[c1];
      const double z1i = (-m[2] * xi[0] + m[3] * xr[0]) + m[0] * xi[c1] + kEps * xi[c1];
      wr[0] = z0r / det;
      wi[0] = z0i / det;
      wr[c1] = z1r / det;
      wi[c1] = z1i / det;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) a[k] = v[k];
    step = p;
    consistency(R);
  }
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
  return v;
}

// One CTA per frequency row f.  Pass p = 0..iterations streams the row, recomputes every bin's chain up to step p and
// either reduces the statistics of R_k for iteration p + 1 (fixed-order block reduction: warp shuffles, then warps in
// order) or, in the last pass, writes y.  No intermediate y in HBM, no atomics: bitwise reproducible.
template <int K, int C>
__global__ void __launch_bounds__(kMwfThreads, 1) k_mwf(const float* __restrict__ psd, const float2* __restrict__ mix,
                                                     float2* __restrict__ out, int F, int T, int iterations) {
  constexpr int NS = C == 2 ? 5 : 2;                    // per source: sum |y_0|^2 (, sum |y_1|^2, Re, Im sum y_0 y_1^*), sum v
  constexpr int NW = kMwfThreads / 32;
  __shared__ double R[kMwfMaxIterations + 1][K][4];
  __shared__ double red[NW][K * NS];
  const int f = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int pass = 0; pass <= iterations; ++pass) {
    const bool last = pass == iterations;
    double acc[K * NS];
#pragma unroll
    for (int i = 0; i < K * NS; ++i) acc[i] = 0.0;
    for (int t = threadIdx.x; t < T; t += kMwfThreads) {
      Chain<K, C> ch;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float2 x = mix[((size_t)c * F + f) * T + t];
        ch.xr[c] = (double)x.x;
        ch.xi[c] = (double)x.y;
      }
      double v[K];
#pragma unroll
      for (int k = 0; k < K; ++k) v[k] = (double)psd[((size_t)k * F + f) * T + t];
      ch.init(v);
      for (int p = 1; p <= pass; ++p) ch.advance(R);
#pragma unroll
      for (int k = 0; k < K; ++k) {
        double yr[C], yi[C];
        ch.source(R, k, yr, yi);
        if (last) {
#pragma unroll
          for (int c = 0; c < C; ++c) out[(((size_t)k * C + c) * F + f) * T + t] = make_float2((float)yr[c], (float)yi[c]);
        } else {
          const double e0 = yr[0] * yr[0] + yi[0] * yi[0];
          acc[k * NS] += e0;
          if (C == 2) {
            const int c1 = C - 1;
            const double e1 = yr[c1] * yr[c1] + yi[c1] * yi[c1];
            acc[k * NS + 1] += e1;
            acc[k * NS + 2] += yr[0] * yr[c1] + yi[0] * yi[c1];
            acc[k * NS + 3] += yi[0] * yr[c1] - yr[0] * yi[c1];
            acc[k * NS + NS - 1] += (e0 + e1) / (double)C;
          } else {
            acc[k * NS + NS - 1] += e0 / (double)C;
          }
        }
      }
    }
    if (last) break;
#pragma unroll
    for (int i = 0; i < K * NS; ++i) {
      const double s = warp_sum_d(acc[i]);
      if (lane == 0) red[warp][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < K) {
      const int k = threadIdx.x;
      double s[NS];
#pragma unroll
      for (int e = 0; e < NS; ++e) {
        s[e] = red[0][k * NS + e];
#pragma unroll
        for (int w = 1; w < NW; ++w) s[e] += red[w][k * NS + e];
      }
      const double den = kEps + s[NS - 1];
      R[pass + 1][k][0] = s[0] / den;
      R[pass + 1][k][1] = C == 2 ? s[1] / den : 0.0;
      R[pass + 1][k][2] = C == 2 ? s[2 % NS] / den : 0.0;
      R[pass + 1][k][3] = C == 2 ? s[3 % NS] / den : 0.0;
    }
    __syncthreads();
  }
}

template <int K, int C>
void launch_mwf_kc(const float* psd, const float* mix, float* out, int F, int T, int iterations, cudaStream_t s) {
  k_mwf<K, C><<<F, kMwfThreads, 0, s>>>(psd, reinterpret_cast<const float2*>(mix), reinterpret_cast<float2*>(out), F, T,
                                       iterations);
  ASEP_LAUNCH_CHECK();
}

template <int K>
void launch_mwf_k(const float* psd, const float* mix, float* out, int C, int F, int T, int iterations, cudaStream_t s) {
  if (C == 1) launch_mwf_kc<K, 1>(psd, mix, out, F, T, iterations, s);
  else launch_mwf_kc<K, 2>(psd, mix, out, F, T, iterations, s);
}

}  // namespace

void launch_track_psd(const float* mag, float* psd, int K, int n_seg, int F, int T, int hop, int overlap, int bin_lo, int bin_hi,
                      int out_sr, int out_n_fft, int out_hop, int F_out, int T_out, cudaStream_t s) {
  const PsdGrid g{K, n_seg, F, T, hop, overlap, bin_lo, bin_hi, out_sr, out_n_fft, out_hop, F_out, T_out,
                  (n_seg - 1) * (T - 1 - overlap) + T};
  const long long total = (long long)F_out * T_out;
  if (total == 0) return;
  k_track_psd<<<cdiv(total, 256), 256, 0, s>>>(mag, psd, g, total);
  ASEP_LAUNCH_CHECK();
}

void launch_mwf(const float* psd, const float* mix, float* out, int K, int C, int F, int T, int iterations, cudaStream_t s) {
  if (F == 0 || T == 0) return;
  switch (K) {
    case 2: launch_mwf_k<2>(psd, mix, out, C, F, T, iterations, s); break;
    case 3: launch_mwf_k<3>(psd, mix, out, C, F, T, iterations, s); break;
    case 4: launch_mwf_k<4>(psd, mix, out, C, F, T, iterations, s); break;
    case 5: launch_mwf_k<5>(psd, mix, out, C, F, T, iterations, s); break;
    case 6: launch_mwf_k<6>(psd, mix, out, C, F, T, iterations, s); break;
    case 7: launch_mwf_k<7>(psd, mix, out, C, F, T, iterations, s); break;
    case 8: launch_mwf_k<8>(psd, mix, out, C, F, T, iterations, s); break;
    default: ASEP_CHECK(false, ASEP_ERR_BAD_ARG, "mwf: K = %d outside 2..8", K);
  }
}

}  // namespace asep
