// Fused BASIS Langevin update (run_basis_sep.py:163-181, dB mixing :131-147) for K = 2..8 sources: every source, the
// mixture-consistency gradient, noise injection and the step-size scaling in ONE HBM-bound pass:
// (2K+1) reads + K writes of 4 B per element with in-kernel Philox noise ((3K+1) reads with injected noise).
#include <cmath>
#include <type_traits>

#include "kernels.h"

namespace asep {
namespace {

// Philox4x32-10 (Salmon et al. 2011), counter = (elem_lo, elem_hi, step, stream), key = seed.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}

__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  // u1 in (0,1], u2 in [0,1)
  float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);
  float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);
  float rad = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif(2.0f * u2, &s, &c);
  return make_float2(rad * c, rad * s);
}

// Four standard normals for the group of 4 consecutive elements starting at global index 4*g.
__device__ __forceinline__ float4 normal4(uint64_t seed, uint64_t step, uint32_t stream_id, uint64_t group) {
  uint4 ctr = make_uint4((uint32_t)group, (uint32_t)(group >> 32), (uint32_t)step,
                         (uint32_t)(step >> 32) ^ (stream_id * 0x9E3779B9u));
  uint4 r = philox4x32_10(ctr, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  float2 a = box_muller(r.x, r.y), b = box_muller(r.z, r.w);
  return make_float4(a.x, a.y, b.x, b.y);
}

// g = (10/ln10)(logsumexp_k(x_k ln10/10) - ln K) and w_k = softmax_k: the max, the exponentials and the sum are taken
// in source order, so K = 2 is the two-source arithmetic op for op.  lnK = (float)log(K), computed on the host.
template <int K>
__device__ __forceinline__ void mix_db(const float (&x)[K], float lnK, float& g, float (&w)[K]) {
  const float k = 0.23025850929940458f;      // ln(10)/10
  float a[K];
#pragma unroll
  for (int i = 0; i < K; ++i) a[i] = x[i] * k;
  float m = a[0];
#pragma unroll
  for (int i = 1; i < K; ++i) m = fmaxf(m, a[i]);
  float e[K];
#pragma unroll
  for (int i = 0; i < K; ++i) e[i] = expf(a[i] - m);
  float sum = e[0];
#pragma unroll
  for (int i = 1; i < K; ++i) sum += e[i];
  g = (1.0f / k) * (m + logf(sum) - lnK);
#pragma unroll
  for (int i = 0; i < K; ++i) w[i] = e[i] / sum;
}

__device__ __forceinline__ float get4(const float4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }

// kDev: the scalars that change from one Langevin step to the next (step size, Philox step number, position in the injected
// noise / per-step dump tensors) are read from device memory, so that ONE captured CUDA graph of a whole BASIS step can
// be replayed for every step of every noise level (api.cu: basis graphs).  In that mode p.n[k] is the base of source k's
// injected noise and noise_stride the element distance between two of its steps.
template <int K, bool kInjected, bool kDev>
__global__ void __launch_bounds__(256) k_langevin(LangevinSources p, const float* __restrict__ mixed, float eta, float lambda,
                                                  float noise_scale, float lnK, uint64_t seed, uint64_t step,
                                                  uint64_t elem_offset, int* __restrict__ nan_count, long long n4,
                                                  long long noise_stride, const LangevinDev* __restrict__ dev,
                                                  float* __restrict__ dump) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  long long noise_off = 0;
  if constexpr (kDev) {
    eta = dev->eta; lambda = dev->lambda; noise_scale = dev->noise_scale; step = dev->step;
    const long long t = (long long)dev->t;
    if constexpr (kInjected) noise_off = t * noise_stride;
    if (dump != nullptr) dump += K * t * n4 * 4;
  }
  float4 a[K], sc[K], z[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    a[k] = reinterpret_cast<const float4*>(p.x[k])[i];
    sc[k] = reinterpret_cast<const float4*>(p.s[k])[i];
  }
  const float4 mx = reinterpret_cast<const float4*>(mixed)[i];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    if constexpr (kInjected) z[k] = reinterpret_cast<const float4*>(p.n[k] + noise_off)[i];
    else z[k] = normal4(seed, step, (uint32_t)(k + 1), (elem_offset >> 2) + (uint64_t)i);   // source k: stream k + 1
  }
  float o[K][4];
  bool bad = false;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float v[K], w[K], g;
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = get4(a[k], j);
    mix_db<K>(v, lnK, g, w);
    float resid = get4(mx, j) - g;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      // evaluation order of run_basis_sep.py:180-181
      o[k][j] = v[k] + eta * (get4(sc[k], j) + lambda * w[k] * resid) + noise_scale * get4(z[k], j);
      bad |= o[k][j] != o[k][j];
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) reinterpret_cast<float4*>(p.x[k])[i] = make_float4(o[k][0], o[k][1], o[k][2], o[k][3]);
  if constexpr (kDev) {
    if (dump != nullptr) {                       // per-step state dump [T, K, ...]
#pragma unroll
      for (int k = 0; k < K; ++k) reinterpret_cast<float4*>(dump)[k * n4 + i] = make_float4(o[k][0], o[k][1], o[k][2], o[k][3]);
    }
  }
  if (nan_count != nullptr && bad) atomicAdd(nan_count, 1);
}

__global__ void k_langevin_advance(LangevinDev* dev) {
  dev->step += 1;
  dev->t += 1;
}

template <int K>
__global__ void k_mixing_db(MixingSources p, float lnK, float* __restrict__ g, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v[K], w[K], gg;
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = p.x[k][i];
  mix_db<K>(v, lnK, gg, w);
  g[i] = gg;
#pragma unroll
  for (int k = 0; k < K; ++k) p.w[k][i] = w[k];
}

__global__ void k_philox_normal(float* __restrict__ out, uint64_t seed, uint64_t step, uint32_t stream_id,
                                uint64_t elem_offset, long long n4) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  reinterpret_cast<float4*>(out)[i] = normal4(seed, step, stream_id, (elem_offset >> 2) + (uint64_t)i);
}

// Runs f(std::integral_constant<int, K>{}) for the runtime source count K (2..kMaxSources, checked by the callers).
template <class F>
void with_sources(int K, F&& f) {
  switch (K) {
    case 2: f(std::integral_constant<int, 2>{}); break;
    case 3: f(std::integral_constant<int, 3>{}); break;
    case 4: f(std::integral_constant<int, 4>{}); break;
    case 5: f(std::integral_constant<int, 5>{}); break;
    case 6: f(std::integral_constant<int, 6>{}); break;
    case 7: f(std::integral_constant<int, 7>{}); break;
    case 8: f(std::integral_constant<int, 8>{}); break;
    default: throw Error(ASEP_ERR_BAD_ARG, strfmt("the number of sources must be in [2, %d] (got %d)", kMaxSources, K));
  }
}

float ln_sources(int K) { return (float)std::log((double)K); }

}  // namespace

void launch_langevin(int K, const LangevinSources& p, const float* mixed, float eta, float lambda, float noise_scale,
                     uint64_t seed, uint64_t step, uint64_t elem_offset, int* nan_count, long long n, cudaStream_t s) {
  if (n == 0) return;
  ASEP_CHECK(n % 4 == 0 && elem_offset % 4 == 0, ASEP_ERR_BAD_SHAPE,
             "langevin: element count %lld and offset must be multiples of 4", n);
  const bool injected = p.n[0] != nullptr;
  // (2K+1) reads + K writes of 4 bytes per element with in-kernel noise, K more reads with injected noise (SURVEY 8(d))
  HbmScope prof(kHbmLangevin, (injected ? 4.0 * K + 1.0 : 3.0 * K + 1.0) * 4.0 * (double)n, s);
  const long long n4 = n / 4;
  const float lnK = ln_sources(K);
  with_sources(K, [&](auto kc) {
    constexpr int KK = decltype(kc)::value;
    if (injected)
      k_langevin<KK, true, false><<<cdiv(n4, 256), 256, 0, s>>>(p, mixed, eta, lambda, noise_scale, lnK, seed, step,
                                                                elem_offset, nan_count, n4, 0, nullptr, nullptr);
    else
      k_langevin<KK, false, false><<<cdiv(n4, 256), 256, 0, s>>>(p, mixed, eta, lambda, noise_scale, lnK, seed, step,
                                                                 elem_offset, nan_count, n4, 0, nullptr, nullptr);
  });
  ASEP_LAUNCH_CHECK();
}

void launch_langevin_dev(int K, const LangevinSources& p, const float* mixed, long long noise_stride, float* dump,
                         LangevinDev* dev, uint64_t seed, uint64_t elem_offset, int* nan_count, long long n, cudaStream_t s) {
  if (n == 0) return;
  ASEP_CHECK(n % 4 == 0 && elem_offset % 4 == 0, ASEP_ERR_BAD_SHAPE,
             "langevin: element count %lld and offset must be multiples of 4", n);
  const long long n4 = n / 4;
  const float lnK = ln_sources(K);
  with_sources(K, [&](auto kc) {
    constexpr int KK = decltype(kc)::value;
    if (p.n[0] != nullptr)
      k_langevin<KK, true, true><<<cdiv(n4, 256), 256, 0, s>>>(p, mixed, 0.f, 0.f, 0.f, lnK, seed, 0, elem_offset, nan_count,
                                                               n4, noise_stride, dev, dump);
    else
      k_langevin<KK, false, true><<<cdiv(n4, 256), 256, 0, s>>>(p, mixed, 0.f, 0.f, 0.f, lnK, seed, 0, elem_offset,
                                                                nan_count, n4, noise_stride, dev, dump);
  });
  ASEP_LAUNCH_CHECK();
  k_langevin_advance<<<1, 1, 0, s>>>(dev);
  ASEP_LAUNCH_CHECK();
}

void launch_mixing_db(int K, const MixingSources& p, float* g, long long n, cudaStream_t s) {
  if (n == 0) return;
  const float lnK = ln_sources(K);
  with_sources(K, [&](auto kc) {
    k_mixing_db<decltype(kc)::value><<<cdiv(n, 256), 256, 0, s>>>(p, lnK, g, n);
  });
  ASEP_LAUNCH_CHECK();
}

void launch_philox_normal(float* out, uint64_t seed, uint64_t step, uint64_t stream_id, uint64_t elem_offset,
                          long long n, cudaStream_t s) {
  if (n == 0) return;
  ASEP_CHECK(n % 4 == 0 && elem_offset % 4 == 0, ASEP_ERR_BAD_SHAPE, "philox: counts must be multiples of 4");
  k_philox_normal<<<cdiv(n / 4, 256), 256, 0, s>>>(out, seed, step, (uint32_t)stream_id, elem_offset, n / 4);
  ASEP_LAUNCH_CHECK();
}

}  // namespace asep
