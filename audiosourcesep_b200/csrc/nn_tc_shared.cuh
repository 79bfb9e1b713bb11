// Pieces shared by the tcgen05 coupling-network kernels (nn_tc.cu: K-pipelined bf16 / fp16 kernel; nn_tcx.cu:
// two-pass split-precision kernel): operand layout, stage-1 im2col builders, col2im gather kernels, weight tile images.
#pragma once
#include "nn_tc.h"
#include "tc_ptx.cuh"

#include <cmath>
#include <cstring>

namespace asep {
namespace {

constexpr int kF = kTcF;
constexpr int kTileM = 128;
constexpr int kPanelBytes = kTileM * 128;        // one 64-wide bf16 K panel of the A operand
constexpr int kNumPanels = kF / 64;              // 8
constexpr int kARegionBytes = kNumPanels * kPanelBytes;   // 128 KB
constexpr int kStageRows = 256;
constexpr int kStageBytes = kStageRows * 128;    // 32 KB weight tile image
constexpr int kStages = 3;
constexpr int kBiasBytes = kF * 4;                // one fp32 bias vector staged in shared memory
constexpr int kTmemCols = 512;

struct TCParams {
  const float* src;      // fwd: state [M, C]; bwd: gr [M, C]
  int src_stride;        // floats per pixel row
  int src_off;           // first channel used
  int src_ch;            // channels used (fwd C/2, bwd C)
  int tap_sign;          // +1: A row p reads pixel p+off(tap) (fwd); -1: p-off(tap) (bwd)
  const __nv_bfloat16* wimg;
  const __nv_bfloat16* wimg_lo;   // nn_tcx.cu, three-product mode: residual weight images (same layout), else NULL
  int f16_s1;                     // nn_tcx.cu: stage-1 operand and weights as fp16 pairs (forward of ASEP_PREC_FP16X3)
  float acc_scale;                // nn_tcx.cu: every accumulator is multiplied by this (1 / weight scale of the tile images)
  int k1_steps, k1_panels, n3p;
  const float* bias1;    // fwd only
  const float* bias2;
  uint32_t* mask1;       // fwd: optional output; bwd: input
  uint32_t* mask2;
  float* out;            // [M, n3p]
  int H, W;
  long long M;
  __nv_bfloat16* dump1;      // optional [M, 512] bf16 copies of the stage-1 / stage-2 epilogue outputs (training:
  __nv_bfloat16* dump2;      //   forward a1 = relu(p1), a2 = relu(p2); backward gp2 = dL/dp2, gp1 = dL/dp1)
  long long* dbg_out;        // debug: per-tile phase timestamps of CTA 0 (clock64), 8 per round
  int f16;                   // forward: fp16 hidden activations / stage-2,3 weights
  long long part_stride;     // nn_tcx.cu: floats between the two K-split partial outputs in `out`
  int tiles_per_cta_round;   // grid size (all CTAs advance together)
  int num_rounds;
};

// source widths the stage-1 operand builders are instantiated for: the register path takes <= 8 channels (1, 2, 4, 8;
// any other width would be built as 4), the rebuild path 16 (data gradient of C = 16 only)
inline bool stage1_width_supported(int src_ch, bool bwd) {
  return src_ch == 1 || src_ch == 2 || src_ch == 4 || src_ch == 8 || (bwd && src_ch == 16);
}

// byte offset of element (row, k) inside the 128-row A region made of 64-wide SWIZZLE_128B panels
__device__ __forceinline__ uint32_t a_offset(int row, int k) {
  return (uint32_t)((k >> 6) * kPanelBytes + row * 128 + ((((k & 63) >> 3) ^ (row & 7)) << 4) + ((k & 7) << 1));
}


constexpr int kThreadsTC2 = 64 + 256;
constexpr int kWorkers2 = 256;

// (hi, lo) pair words of two values: bf16 pairs (16 significant bits, fp32 range) or fp16 pairs (22 bits, |v| < 65504)
template <bool kHalf>
__device__ __forceinline__ void split_pair(float a, float b, uint32_t& hi, uint32_t& lo) {
  if constexpr (kHalf) {
    __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<uint32_t*>(&h);
    lo = *reinterpret_cast<uint32_t*>(&l);
  } else {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    hi = *reinterpret_cast<uint32_t*>(&h);
    __nv_bfloat162 l = __floats2bfloat162_rn(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xffff0000u));
    lo = *reinterpret_cast<uint32_t*>(&l);
  }
}

// im2col of taps [t_begin, t_end) of one operand row as split-bf16 [hi | lo]
template <int SC>
__device__ __forceinline__ void build_a1_taps(uint8_t* sA, int row, const float* __restrict__ src, long long p, bool valid,
                                              int h, int w, int H, int W, int stride, int off, int sign, int t_begin,
                                              int t_end) {
  constexpr int K1h = 9 * SC;
  constexpr int TG = SC >= 16 ? 3 : 5;
  for (int t0 = t_begin; t0 < t_end; t0 += TG) {
    float v[TG][SC];
#pragma unroll
    for (int tt = 0; tt < TG; ++tt) {
      const int tap = t0 + tt;
      const int dy = (tap / 3 - 1) * sign, dx = (tap % 3 - 1) * sign;
      const int hh = h + dy, ww = w + dx;
      const bool ok = valid && tap < t_end && hh >= 0 && hh < H && ww >= 0 && ww < W;
      const float* s = src + (p + (long long)dy * W + dx) * stride + off;
      if constexpr (SC % 4 == 0) {
#pragma unroll
        for (int q = 0; q < SC / 4; ++q) {
          float4 t = ok ? __ldg(reinterpret_cast<const float4*>(s) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
          v[tt][4 * q] = t.x; v[tt][4 * q + 1] = t.y; v[tt][4 * q + 2] = t.z; v[tt][4 * q + 3] = t.w;
        }
      } else if constexpr (SC == 2) {
        float2 t = ok ? __ldg(reinterpret_cast<const float2*>(s)) : make_float2(0.f, 0.f);
        v[tt][0] = t.x; v[tt][1] = t.y;
      } else {
#pragma unroll
        for (int ci = 0; ci < SC; ++ci) v[tt][ci] = ok ? __ldg(s + ci) : 0.f;
      }
    }
#pragma unroll
    for (int tt = 0; tt < TG; ++tt) {
      if (t0 + tt >= t_end) break;
      const int k0 = (t0 + tt) * SC;
      float lo[SC];
      uint32_t hp[(SC + 1) / 2], lp[(SC + 1) / 2];
#pragma unroll
      for (int ci = 0; ci < SC; ++ci) lo[ci] = v[tt][ci] - __bfloat162float(__float2bfloat16_rn(v[tt][ci]));
      if constexpr (SC == 1) {
        *reinterpret_cast<__nv_bfloat16*>(sA + a_offset(row, k0)) = __float2bfloat16_rn(v[tt][0]);
        *reinterpret_cast<__nv_bfloat16*>(sA + a_offset(row, K1h + k0)) = __float2bfloat16_rn(lo[0]);
      } else {
#pragma unroll
        for (int q = 0; q < SC / 2; ++q) {
          hp[q] = pack_bf16(v[tt][2 * q], v[tt][2 * q + 1]);
          lp[q] = pack_bf16(lo[2 * q], lo[2 * q + 1]);
        }
        if constexpr (SC == 2) {
          *reinterpret_cast<uint32_t*>(sA + a_offset(row, k0)) = hp[0];
          *reinterpret_cast<uint32_t*>(sA + a_offset(row, K1h + k0)) = lp[0];
        } else if constexpr (SC == 4) {
          *reinterpret_cast<uint2*>(sA + a_offset(row, k0)) = make_uint2(hp[0], hp[1]);
          *reinterpret_cast<uint2*>(sA + a_offset(row, K1h + k0)) = make_uint2(lp[0], lp[1]);
        } else {
#pragma unroll
          for (int q = 0; q < SC / 8; ++q) {
            *reinterpret_cast<uint4*>(sA + a_offset(row, k0 + 8 * q)) =
                make_uint4(hp[4 * q], hp[4 * q + 1], hp[4 * q + 2], hp[4 * q + 3]);
            *reinterpret_cast<uint4*>(sA + a_offset(row, K1h + k0 + 8 * q)) =
                make_uint4(lp[4 * q], lp[4 * q + 1], lp[4 * q + 2], lp[4 * q + 3]);
          }
        }
      }
    }
  }
}

// im2col of up to five taps [t_begin, t_end) of one operand row, split in a LOAD half (global -> registers, issued
// while the worker is idle) and a STORE half (split-bf16 [hi | lo] -> swizzled shared memory, once the panels are free)
template <int SC>
__device__ __forceinline__ void a1_load(float (&v)[40], const float* __restrict__ src, long long p, bool valid, int h, int w,
                                        int H, int W, int stride, int off, int sign, int t_begin, int t_end) {
  static_assert(SC <= 8, "register prefetch is sized for <= 8 source channels");
#pragma unroll
  for (int tt = 0; tt < 5; ++tt) {
    const int tap = t_begin + tt;
    const int dy = (tap / 3 - 1) * sign, dx = (tap % 3 - 1) * sign;
    const int hh = h + dy, ww = w + dx;
    const bool ok = valid && tap < t_end && hh >= 0 && hh < H && ww >= 0 && ww < W;
    const float* s = src + (p + (long long)dy * W + dx) * stride + off;
    if constexpr (SC == 8) {
      const float4 t = ok ? __ldg(reinterpret_cast<const float4*>(s)) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 u = ok ? __ldg(reinterpret_cast<const float4*>(s) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
      v[8 * tt] = t.x; v[8 * tt + 1] = t.y; v[8 * tt + 2] = t.z; v[8 * tt + 3] = t.w;
      v[8 * tt + 4] = u.x; v[8 * tt + 5] = u.y; v[8 * tt + 6] = u.z; v[8 * tt + 7] = u.w;
    } else if constexpr (SC == 4) {
      const float4 t = ok ? __ldg(reinterpret_cast<const float4*>(s)) : make_float4(0.f, 0.f, 0.f, 0.f);
      v[4 * tt] = t.x; v[4 * tt + 1] = t.y; v[4 * tt + 2] = t.z; v[4 * tt + 3] = t.w;
    } else if constexpr (SC == 2) {
      const float2 t = ok ? __ldg(reinterpret_cast<const float2*>(s)) : make_float2(0.f, 0.f);
      v[2 * tt] = t.x; v[2 * tt + 1] = t.y;
    } else {
      v[tt] = ok ? __ldg(s) : 0.f;
    }
  }
}
template <int SC, bool kHalf = false>
__device__ __forceinline__ void a1_store(uint8_t* sA, int row, const float (&v)[40], int t_begin, int t_end) {
  constexpr int K1h = 9 * SC;
#pragma unroll
  for (int tt = 0; tt < 5; ++tt) {
    if (t_begin + tt >= t_end) break;
    const int k0 = (t_begin + tt) * SC;
    if constexpr (SC == 1) {
      uint32_t hi, lo;
      split_pair<kHalf>(v[tt], 0.f, hi, lo);
      *reinterpret_cast<uint16_t*>(sA + a_offset(row, k0)) = (uint16_t)(hi & 0xffffu);
      *reinterpret_cast<uint16_t*>(sA + a_offset(row, K1h + k0)) = (uint16_t)(lo & 0xffffu);
    } else {
      uint32_t hi[SC / 2], lo[SC / 2];
#pragma unroll
      for (int q = 0; q < SC / 2; ++q) split_pair<kHalf>(v[tt * SC + 2 * q], v[tt * SC + 2 * q + 1], hi[q], lo[q]);
      if constexpr (SC == 2) {
        *reinterpret_cast<uint32_t*>(sA + a_offset(row, k0)) = hi[0];
        *reinterpret_cast<uint32_t*>(sA + a_offset(row, K1h + k0)) = lo[0];
      } else if constexpr (SC == 4) {
        *reinterpret_cast<uint2*>(sA + a_offset(row, k0)) = make_uint2(hi[0], hi[1]);
        *reinterpret_cast<uint2*>(sA + a_offset(row, K1h + k0)) = make_uint2(lo[0], lo[1]);
      } else {
        *reinterpret_cast<uint4*>(sA + a_offset(row, k0)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(sA + a_offset(row, K1h + k0)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
    }
  }
}

// [n3p/4 float4 columns][128 rows][4 floats] (k_nn_tc4)
template <bool kTiled>
__device__ __forceinline__ long long g_index(long long pp, int col, int n3p) {
  if constexpr (!kTiled) return pp * n3p + col;
  else return (pp >> 7) * (128ll * n3p) + (long long)(col >> 2) * 512 + (pp & 127) * 4 + (col & 3);
}

template <bool kTiled>
__global__ void __launch_bounds__(256) k_gather_fwd(const float* __restrict__ G, const float* __restrict__ const3,
                                                    const float* __restrict__ c3, float* __restrict__ r, int H, int W,
                                                    int C, int n3p, long long total, int nparts,
                                                    long long part_stride) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = idx % C;
  const long long p = idx / C;
  const int w = p % W, h = (p / W) % H;
  float acc = c3[c];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int dy = tap / 3 - 1, dx = tap % 3 - 1;
    const int hh = h + dy, ww = w + dx;
    if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
    const long long gi = g_index<kTiled>(p + (long long)dy * W + dx, tap * C + c, n3p);
    float t = G[gi];
    for (int q = 1; q < nparts; ++q) t += G[gi + q * part_stride];      // K-split partial sums (nn_tcx.cu)
    acc += t + const3[tap * C + c];
  }
  r[idx] = acc;
}

// gxb[p][ci] = sum_{tap: p-off in bounds} G'[p-off(tap)][tap*Ch+ci]
template <bool kTiled>
__global__ void __launch_bounds__(256) k_gather_bwd(const float* __restrict__ G, float* __restrict__ gxb, int H, int W,
                                                    int Ch, int n3p, long long total, int nparts,
                                                    long long part_stride) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = idx % Ch;
  const long long p = idx / Ch;
  const int w = p % W, h = (p / W) % H;
  float acc = 0.f;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int dy = tap / 3 - 1, dx = tap % 3 - 1;
    const int hh = h - dy, ww = w - dx;
    if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
    const long long gi = g_index<kTiled>(p - (long long)dy * W - dx, tap * Ch + c, n3p);
    for (int q = 0; q < nparts; ++q) acc += G[gi + q * part_stride];
  }
  gxb[idx] = acc;
}

// Vector forms for the tiled G layout: one thread per (pixel, group of V = 4 or 2 consecutive channels); every tap is
// one 16- or 8-byte load (the channels of a tap are contiguous inside a float4 column because C % V == 0).
template <int V, bool kFwd>
__global__ void __launch_bounds__(256) k_gather_vec(const float* __restrict__ G, const float* __restrict__ const3,
                                                    const float* __restrict__ c3, float* __restrict__ out, int H, int W,
                                                    int C, int n3p, long long total, int nparts,
                                                    long long part_stride) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int CV = C / V;
  const int cv = (int)(idx % CV);
  const long long p = idx / CV;
  const int w = (int)(p % W), h = (int)((p / W) % H);
  float acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = kFwd ? c3[cv * V + v] : 0.f;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int dy = (tap / 3 - 1) * (kFwd ? 1 : -1), dx = (tap % 3 - 1) * (kFwd ? 1 : -1);
    const int hh = h + dy, ww = w + dx;
    if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
    const long long pp = p + (long long)dy * W + dx;
    const int col = tap * C + cv * V;
    const float* g = G + (pp >> 7) * (128ll * n3p) + (long long)(col >> 2) * 512 + (pp & 127) * 4 + (col & 3);
    if constexpr (V == 4) {
      float4 t = __ldg(reinterpret_cast<const float4*>(g));
      for (int q = 1; q < nparts; ++q) {      // K-split partial sums (nn_tcx.cu)
        const float4 u = __ldg(reinterpret_cast<const float4*>(g + q * part_stride));
        t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
      }
      if constexpr (kFwd) {      // same association as the scalar kernel: acc += (G + const3)
        const float4 k = __ldg(reinterpret_cast<const float4*>(const3 + col));
        t.x += k.x; t.y += k.y; t.z += k.z; t.w += k.w;
      }
      acc[0] += t.x; acc[1] += t.y; acc[2] += t.z; acc[3] += t.w;
    } else {
      float2 t = __ldg(reinterpret_cast<const float2*>(g));
      for (int q = 1; q < nparts; ++q) {
        const float2 u = __ldg(reinterpret_cast<const float2*>(g + q * part_stride));
        t.x += u.x; t.y += u.y;
      }
      if constexpr (kFwd) {
        const float2 k = __ldg(reinterpret_cast<const float2*>(const3 + col));
        t.x += k.x; t.y += k.y;
      }
      acc[0] += t.x; acc[1] += t.y;
    }
  }
  if constexpr (V == 4) reinterpret_cast<float4*>(out)[idx] = make_float4(acc[0], acc[1], acc[2], acc[3]);
  else reinterpret_cast<float2*>(out)[idx] = make_float2(acc[0], acc[1]);
}

inline int pad16(int n) { return (n + 15) / 16 * 16; }

// col2im of the tiled G (nparts K-split partial sums, part_stride floats apart): r = c3 + sum_taps (G + const3)
inline void launch_gather_fwd(const float* G, const float* const3, const float* c3, float* r, long long M, int H, int W, int C,
                              int n3p, int nparts, long long part_stride, cudaStream_t s) {
  const long long total = M * C;
  HbmScope prof(kHbmGather, 4.0 * (9.0 * C * nparts + C) * (double)M, s);      // 9 per-tap partials in, r out
  if (C % 4 == 0) k_gather_vec<4, true><<<cdiv(total / 4, 256), 256, 0, s>>>(G, const3, c3, r, H, W, C, n3p, total / 4, nparts, part_stride);
  else k_gather_fwd<true><<<cdiv(total, 256), 256, 0, s>>>(G, const3, c3, r, H, W, C, n3p, total, nparts, part_stride);
  ASEP_LAUNCH_CHECK();
}
// gxb[p][ci] = sum_taps G'[p - off(tap)][tap*Ch + ci]
inline void launch_gather_bwd(const float* G, float* gxb, long long M, int H, int W, int Ch, int n3p, int nparts,
                              long long part_stride, cudaStream_t s) {
  const long long total = M * Ch;
  HbmScope prof(kHbmGather, 4.0 * (9.0 * Ch * nparts + Ch) * (double)M, s);
  if (Ch % 4 == 0) k_gather_vec<4, false><<<cdiv(total / 4, 256), 256, 0, s>>>(G, nullptr, nullptr, gxb, H, W, Ch, n3p, total / 4, nparts, part_stride);
  else if (Ch % 2 == 0) k_gather_vec<2, false><<<cdiv(total / 2, 256), 256, 0, s>>>(G, nullptr, nullptr, gxb, H, W, Ch, n3p, total / 2, nparts, part_stride);
  else k_gather_bwd<true><<<cdiv(total, 256), 256, 0, s>>>(G, gxb, H, W, Ch, n3p, total, nparts, part_stride);
  ASEP_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ host: weight tile images
// Writes one image of `rows` rows x 64 k (16-bit words, SWIZZLE_128B K-major) for rows n0.., k0..
// f16: IEEE half instead of bfloat16 in the same 16-bit slots.  lo_part: the residual word lo = rn(v - hi) of the
// split-precision weights (nn_tcx.cu, three-product mode) instead of hi = rn(v).
template <typename Fn>
void write_image(std::vector<__nv_bfloat16>& dst, int rows, int n0, int n_valid, int k0, int k_valid, Fn&& get, bool f16 = false,
                 bool lo_part = false, float wscale = 1.f) {
  const size_t base = dst.size();
  dst.resize(base + (size_t)rows * 64, __float2bfloat16(0.f));
  for (int r = 0; r < rows; ++r) {
    for (int k = 0; k < 64; ++k) {
      float v = 0.f;
      if (r < n_valid && k < k_valid) v = get(n0 + r, k0 + k) * wscale;
      const size_t off = (size_t)r * 64 + (size_t)((((k >> 3) ^ (r & 7)) << 3) + (k & 7));
      uint16_t bits;
      if (f16) {
        ASEP_CHECK(std::fabs(v) < 60000.f, ASEP_ERR_UNSUPPORTED, "coupling-network weight %g outside the fp16 range of this precision mode", v);
        __half hv = __float2half(v);
        if (lo_part) hv = __float2half(v - __half2float(hv));
        std::memcpy(&bits, &hv, sizeof(bits));
      } else {
        __nv_bfloat16 bv = __float2bfloat16(v);
        if (lo_part) bv = __float2bfloat16(v - __bfloat162float(bv));
        std::memcpy(&bits, &bv, sizeof(bits));
      }
      std::memcpy(reinterpret_cast<uint16_t*>(dst.data()) + base + off, &bits, sizeof(bits));
    }
  }
}

// f16_1 / f16_23: stage-1 / stage-2,3 weights as IEEE half.  lo_part: the residual images of the three-product mode;
// the stage-1 operand is [x_hi | x_lo] against [W1 ; W1], so the residual image is [W1_lo ; 0] (x_hi . W1_lo only).
// wscale: power of two the weights are multiplied by before rounding (the kernel multiplies the accumulators by
// 1 / wscale): keeps the fp16 residuals of O(0.04) weights out of the subnormal range.
template <typename F1, typename F2, typename F3>
void build_stage_set(TCStageSet& set, int K1, int N3, F1&& b1, F2&& b2, F3&& b3, bool f16_23, bool f16_1 = false,
                     bool lo_part = false, float wscale = 1.f) {
  set.k1_steps = (K1 + 15) / 16;
  set.k1_panels = (K1 + 63) / 64;
  set.n3p = pad16(N3);
  ASEP_CHECK(set.k1_panels <= kNumPanels && set.n3p <= 256, ASEP_ERR_UNSUPPORTED,
             "coupling network shape outside the tcgen05 kernel (K1=%d, N3=%d)", K1, N3);
  std::vector<__nv_bfloat16> img;
  const int K1h = K1 / 2;
  auto b1p = [&](int n, int k) { return (lo_part && k >= K1h) ? 0.f : b1(n, k); };
  for (int half = 0; half < 2; ++half)
    for (int kp = 0; kp < set.k1_panels; ++kp)
      write_image(img, kStageRows, half * 256, 256, kp * 64, std::min(64, K1 - kp * 64), b1p, f16_1, lo_part, wscale);
  for (int half = 0; half < 2; ++half)
    for (int kp = 0; kp < kNumPanels; ++kp) write_image(img, kStageRows, half * 256, 256, kp * 64, 64, b2, f16_23, lo_part, wscale);
  for (int kp = 0; kp < kNumPanels; ++kp) write_image(img, set.n3p, 0, N3, kp * 64, 64, b3, f16_23, lo_part, wscale);
  set.bytes = img.size() * sizeof(__nv_bfloat16);
  CUDA_CHECK(cudaMalloc(&set.img, set.bytes));
  CUDA_CHECK(cudaMemcpy(set.img, img.data(), set.bytes, cudaMemcpyHostToDevice));
}

inline float* upload(const std::vector<float>& v) {
  float* d = nullptr;
  CUDA_CHECK(cudaMalloc(&d, v.size() * sizeof(float)));
  CUDA_CHECK(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return d;
}

}  // namespace
}  // namespace asep
