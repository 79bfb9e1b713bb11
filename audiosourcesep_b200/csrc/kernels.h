// Host-side launchers of every kernel in libasep.so.  All tensors are fp32 NHWC on the device.
#pragma once
#include "common.cuh"

namespace asep {

// Per-step element-wise constants, laid out as floats:
//   [0,C) exp(log_scale)  [C,2C) shift  [2C,2C+C*C) W[i][o]  [2C+C*C, 2C+2C*C) W^-1[i][o]
inline int step_const_floats(int C) { return 2 * C + 2 * C * C; }

// Per-tap partial outputs of the tensor-core coupling network (nn_tc.cu / nn_tcx.cu) still in the tiled layout
// [tile][n3p/4 float4 columns][128 rows][4 floats]; `nparts` K-split partial sums `part_stride` floats apart.  The
// flow-step kernels below can consume it directly (col2im fused into the element-wise pass: no r round trip, one
// launch less per flow step).
struct GatherSrc {
  const float* G = nullptr;
  const float* const3 = nullptr;   // forward only: [9][C] border-aware BatchNorm offset of conv3
  const float* c3 = nullptr;       // forward only: conv3 bias [C]
  int n3p = 0, nparts = 1, H = 0, W = 0;
  long long part_stride = 0;
};

// ---- flow_kernels.cu
// u = (x*scale+shift) . W                      (flow_tfp_bijectors.py:243, :304-305)
void launch_pre(const float* x, float* u, const float* sc, long long M, int C, cudaStream_t s);
// y = [ua*exp(tanh(raw))+t, ub]; acc[n] += sum tanh(raw); then (optional) out = pre_next(y)
void launch_post_pre(const float* u, const float* r, float* out, const float* sc_next, double* acc, long long M,
                     int HW, int C, cudaStream_t s);
// as launch_post_pre / launch_inv_step / launch_bwd_pre with the network output gathered from the tiled G on the fly:
// r = c3 + sum_{tap in bounds} (G[p + off(tap)][tap] + const3[tap]); r_out (may be NULL) receives r when the backward
// pass needs it.  bwd: gxb = sum_{tap} G'[p - off(tap)][tap].
void launch_post_pre_g(const float* u, const GatherSrc& g, float* r_out, float* out, const float* sc_next, double* acc,
                       long long M, int HW, int C, cudaStream_t s);
void launch_inv_step_g(const float* y, const GatherSrc& g, float* x, const float* sc, double* acc, long long M, int HW,
                       int C, cudaStream_t s);
void launch_bwd_pre_g(const float* gu, const GatherSrc& g, float* gx, const float* sc, long long M, int C, cudaStream_t s);
bool fused_gather_supported(int C);   // channel counts the fused-gather kernels are built for (4, 8, 16)
// x = (( [ (ya-t)/exp(tanh raw), yb ] . W^-1 ) - shift) / scale ; acc[n] -= sum tanh(raw) when acc != NULL
void launch_inv_step(const float* y, const float* r, float* x, const float* sc, double* acc, long long M, int HW,
                     int C, cudaStream_t s);
// backward of the coupling: gr = [graw, gt], gu = [gya*exp(sl), gyb]
void launch_bwd_coupling(const float* gy, const float* u, const float* r, float* gr, float* gu, long long M, int C,
                         cudaStream_t s);
// gx = (([gua, gyb + gxb]) . W^T) * scale
void launch_bwd_pre(const float* gu, const float* gxb, float* gx, const float* sc, long long M, int C, cudaStream_t s);
// Squeeze (space-to-depth; H, W, C describe the UNSQUEEZED side) fused with an affine map:
// mode 0 none, 1 SpecPreprocessing forward (p0=minval, p1=maxval), 2 its inverse, 3 multiply by p0.
// inverse=0: x unsqueezed -> y squeezed;  inverse=1: x squeezed -> y unsqueezed.
void launch_squeeze(const float* x, float* y, int N, int H, int W, int C, int mode, float p0, float p1, int inverse,
                    cudaStream_t s);
// Factor-out plumbing of GlowBijector_*blocks (flow_glow.py:176-196).  o [N,H,W,C]: channels [0,Cz) map to the
// latent (plain row-major reshape to [Hl*Wl, nb], channel offset coff of CL, Dl = latent dims per sample), the
// remaining channels map to the squeezed next-level state.  merge=0: o -> (z, next); merge=1: (z, next) -> o.
void launch_split_merge(float* o, float* z, float* next, int N, int H, int W, int C, int Cz, int nb, int CL,
                        int coff, long long Dl, int merge, cudaStream_t s);
// acc[n] += sum_d -0.5 q^2 - ls - 0.5 log 2pi ; gz = -(z-loc)/exp(2 ls) when gz != NULL
void launch_prior(const float* z, const float* loc, const float* log_scale, double* acc, float* gz, int N, int D,
                  cudaStream_t s);
// z = loc + exp(ls) * eps
void launch_prior_sample(const float* eps, const float* loc, const float* log_scale, float* z, int N, int D,
                         cudaStream_t s);
// out[n] = (acc[n] + add + *dev_add) * scale   (dev_add: optional device-resident constant, e.g. the sum of the per-step
// log-det constants that the training path keeps on the device)
void launch_finish(const double* acc, float* out, double add, double scale, int N, cudaStream_t s,
                   const double* dev_add = nullptr);
void launch_channel_stats(const float* x, double* mean_std, long long M, int C, cudaStream_t s);
void launch_scale(float* x, float a, long long n, cudaStream_t s);
void launch_actnorm(const float* x, const float* log_scale, const float* shift, float* y, long long M, int C,
                    int inverse, cudaStream_t s);
void launch_chanmix(const float* x, const float* w, float* y, long long M, int C, cudaStream_t s);

// ---- langevin.cu
// BASIS separates K = 2..kMaxSources sources: the bound keeps the per-element state of the fused update in registers
// and bounds the side streams of the step graph.
constexpr int kMaxSources = 8;
// Per-source pointers of one update, passed by value: states x[k] (updated in place), scores s[k] and injected standard
// normals n[k] (all NULL for in-kernel Philox noise, source k drawing from stream k + 1).
struct LangevinSources {
  float* x[kMaxSources];
  const float* s[kMaxSources];
  const float* n[kMaxSources];
};
void launch_langevin(int K, const LangevinSources& p, const float* mixed, float eta, float lambda, float noise_scale,
                     uint64_t seed, uint64_t step, uint64_t elem_offset, int* nan_count, long long n, cudaStream_t s);
// Device-resident scalars of one Langevin step (see k_langevin<.., kDev>): written by the host before a run of graph
// replays, advanced (step, t) by the kernel pair itself after every step.
struct LangevinDev {
  float eta, lambda, noise_scale, pad;
  unsigned long long step;     // Philox step number of the next update
  unsigned long long t;        // index of the next update inside the injected-noise / dump tensors
};
// as launch_langevin with the per-step scalars in *dev; p.n[k] is the base of source k's injected noise (step t at
// p.n[k] + t * noise_stride), dump the base of the [T, K, ...] per-step dump (or NULL)
void launch_langevin_dev(int K, const LangevinSources& p, const float* mixed, long long noise_stride, float* dump,
                         LangevinDev* dev, uint64_t seed, uint64_t elem_offset, int* nan_count, long long n, cudaStream_t s);
// g = (10/ln10)(logsumexp_k(x_k ln10/10) - ln K) and w_k = softmax_k of the K inputs x[k]
struct MixingSources {
  const float* x[kMaxSources];
  float* w[kMaxSources];
};
void launch_mixing_db(int K, const MixingSources& p, float* g, long long n, cudaStream_t s);
void launch_philox_normal(float* out, uint64_t seed, uint64_t step, uint64_t stream_id, uint64_t elem_offset,
                          long long n, cudaStream_t s);

// ---- nn_fp32.cu  (CUDA-core "exact" coupling network)
struct NNWeightsF32 {
  const float *k1, *c1, *g1, *b1;  // conv1 kernel [3,3,Ch,F], bias, folded BN scale/offset [F]
  const float *k2, *k2t, *c2, *g2, *b2;  // conv2 kernel [F,F] (in,out), its transpose
  const float *k3, *c3;            // conv3 kernel [3,3,F,C], bias [C]
};
// state [N,H,W,C] (input = channels C/2..C) -> r [M,C]; a1,a2 [M,F] scratch hold relu(p1), relu(p2)
void nn_fp32_forward(const NNWeightsF32& w, const float* state, float* a1, float* a2, float* r, int N, int H, int W,
                     int C, int F, cudaStream_t s);
// gr [M,C] -> gxb [M,C/2]; a1,a2 from a forward on the same input; g1,g2 [M,F] scratch
void nn_fp32_backward(const NNWeightsF32& w, const float* a1, const float* a2, const float* gr, float* t1, float* t2,
                      float* gxb, int N, int H, int W, int C, int F, cudaStream_t s);

}  // namespace asep
