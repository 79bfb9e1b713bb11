// tcgen05 / TMEM / TMA implementation of ShiftAndLogScaleConvNet and of its data gradient
// (ASEP_PREC_BF16).  See nn_tc.cu for the kernel design.
#pragma once
#include <vector>
#include "common.cuh"
#include "kernels.h"

namespace asep {

constexpr int kTcF = 512;   // hidden width the tcgen05 kernel is built for (configs/melspec_glow.yml:10)

// Level widths C the tcgen05 coupling kernels are built for: their stage-1 operand builders handle C/2 (forward) and
// C (data gradient) source channels in {2, 4, 8, 16} only, and the stage-3 outputs of C = 32 do not fit the staging area.
inline bool nn_tc_supported(int C) { return C == 4 || C == 8 || C == 16; }

struct TCStageSet {
  __nv_bfloat16* img = nullptr;  // weight tile images in consumption order (device)
  int k1_steps = 0;              // K=16 MMA steps of stage 1
  int k1_panels = 0;             // 64-wide K panels of stage 1
  int n3p = 0;                   // padded N of stage 3 (multiple of 16)
  size_t bytes = 0;
};

struct NNWeightsTC {
  TCStageSet fwd, bwd;
  TCStageSet fwd_lo, bwd_lo;  // residual images w - rn(w) of the three-product mode (ASEP_PREC_FP16X3), else empty
  bool x3 = false;
  float wscale_fwd = 1.f;     // power of two folded into the forward tile images (fp16 residuals stay normal numbers)
  float* bias1 = nullptr;   // c1                                   [F]
  float* bias2 = nullptr;   // c2 + b1' . K2                        [F]
  float* const3 = nullptr;  // [9][C]  sum_k b2'[k] K3[tap][k][c]   (border-aware BN offset of conv3)
  float* c3 = nullptr;      // [C]
  bool f16 = false;         // forward stage-2/3 tile images and hidden activations in fp16 (ASEP_PREC_FP16)
};

struct NNScratchTC {
  float* G = nullptr;        // [M, n3p] fp32 per-tap partial outputs of the small-N stage
  uint32_t* mask1 = nullptr; // [M, F/32] relu masks of p1 (scratch for one step)
  uint32_t* mask2 = nullptr;
};

// Host-side preparation: builds the bf16 SWIZZLE_128B tile images for both directions.
// k1 [3,3,Ch,F], k2 [F,F] (in,out), k3 [3,3,F,C]; g*/b* folded BatchNorm scale/offset.
void nn_tc_prepare(NNWeightsTC& w, const float* k1, const float* c1, const float* g1, const float* b1,
                   const float* k2, const float* c2, const float* g2, const float* b2, const float* k3,
                   const float* c3, int C, int F, bool f16 = false, bool x3 = false);
void nn_tc_release(NNWeightsTC& w);

// state [N,H,W,C] (network input = channels C/2..C) -> r [M,C] (conv3 output incl. bias).
// mask1/mask2 (may be NULL) receive the ReLU masks needed by the backward pass.
// dump1/dump2 (may be NULL; 8-warp kernels only): bf16 [M,512] copies of relu(p1), relu(p2) for the weight gradients.
void nn_tc_forward(const NNWeightsTC& w, const NNScratchTC& sc, const float* state, float* r, uint32_t* mask1,
                   uint32_t* mask2, int N, int H, int W, int C, cudaStream_t s, __nv_bfloat16* dump1 = nullptr,
                   __nv_bfloat16* dump2 = nullptr);
// gr [M,C] -> gxb [M,C/2] using the masks written by nn_tc_forward on the same input.
// dump_gp2/dump_gp1 (may be NULL): bf16 [M,512] copies of dL/dp2 and dL/dp1.
void nn_tc_backward(const NNWeightsTC& w, const NNScratchTC& sc, const float* gr, const uint32_t* mask1,
                    const uint32_t* mask2, float* gxb, int N, int H, int W, int C, cudaStream_t s,
                    __nv_bfloat16* dump_gp2 = nullptr, __nv_bfloat16* dump_gp1 = nullptr);

size_t nn_tc_g_floats(long long M, int C);   // capacity needed for NNScratchTC::G
// r == NULL (forward) / gxb == NULL (backward) skips the col2im gather kernel: the caller consumes the tiled G through
// the fused flow-step kernels (launch_post_pre_g / launch_inv_step_g / launch_bwd_pre_g) with this descriptor.
// split = the two-part G of nn_tcx_forward / nn_tcx_backward.
GatherSrc nn_tc_gather_src(const NNWeightsTC& w, const NNScratchTC& sc, bool backward, long long M, int H, int W, bool split);

// ---- split-precision ("exact") tensor-core form (nn_tcx.cu; ASEP_PREC_BF16X2 / ASEP_PREC_FP16X2): the same tile images,
// hidden activations carried as (hi + lo) 16-bit pairs -> two tcgen05 products per hidden GEMM, 16 (bf16 pairs) or 22
// (fp16 pairs) significant bits instead of 8 / 11.  Same contracts as nn_tc_forward / nn_tc_backward (no dumps).
void nn_tcx_forward(const NNWeightsTC& w, const NNScratchTC& sc, const float* state, float* r, uint32_t* mask1,
                    uint32_t* mask2, int N, int H, int W, int C, cudaStream_t s);
void nn_tcx_backward(const NNWeightsTC& w, const NNScratchTC& sc, const float* gr, const uint32_t* mask1,
                     const uint32_t* mask2, float* gxb, int N, int H, int W, int C, cudaStream_t s);
size_t nn_tcx_g_floats(long long M, int C);  // two K-split partial outputs
// CUDA-event timing of every tensor-core kernel launch (on its own stream) while switched on.
void nn_tc_profile(int on);
struct TcProfToken { cudaEvent_t a = nullptr, b = nullptr; bool on = false; };
TcProfToken nn_tc_prof_begin(cudaStream_t s);                                  // shared by nn_tc.cu and nn_tcx.cu
void nn_tc_prof_end(const TcProfToken& tok, cudaStream_t s, double flops);
bool nn_tc_profile_enabled();
void nn_tc_profile_read(double* total_ms, long long* launches, double* flops);

}  // namespace asep
