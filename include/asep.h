/*
 * asep.h -- C ABI of libasep.so, the B200 (sm_100a) implementation of the
 * SamArgt/AudioSourceSep separation hot path.
 *
 * This is the drop-in boundary: plain C, no torch / CUDA types in the signatures
 * (a stream crosses as `void*` holding a cudaStream_t; NULL = the legacy default stream).
 * Tensors cross as DLPack `DLTensor*` (asep_dlpack.h): float32, row-major contiguous NHWC
 * unless stated, resident on the CUDA device the handle was created on; `set_param`
 * additionally accepts host (kDLCPU) tensors.  The caller owns every tensor it passes;
 * the library never retains a pointer beyond the call (parameters are copied).
 *
 * Every function returns 0 on success or a negative asep_status; asep_last_error() holds
 * the message (thread-local).  Handles are not thread-safe.
 *
 * Each entry point cites the reference interface it replaces (path:line under the
 * reference repository SamArgt/AudioSourceSep).
 */
#ifndef ASEP_H_
#define ASEP_H_

#include <stdint.h>
#include "asep_dlpack.h"

#ifdef __cplusplus
extern "C" {
#endif

#define ASEP_ABI_VERSION 1

typedef enum {
  ASEP_OK = 0,
  ASEP_ERR_BAD_ARG = -1,     /* NULL pointer, unknown name, bad enum            */
  ASEP_ERR_BAD_SHAPE = -2,   /* shape contract violated (reference asserts)     */
  ASEP_ERR_BAD_DTYPE = -3,   /* not float32 (or the int32 / bf16 / float64 stated) */
  ASEP_ERR_BAD_LAYOUT = -4,  /* non-contiguous / misaligned                     */
  ASEP_ERR_BAD_DEVICE = -5,  /* tensor not on the handle's CUDA device          */
  ASEP_ERR_CUDA = -6,        /* CUDA runtime / driver error                     */
  ASEP_ERR_NAN = -7,         /* NaN detected by a --debug style check           */
  ASEP_ERR_STATE = -8,       /* call order violated (e.g. prepare() missing)    */
  ASEP_ERR_UNSUPPORTED = -9  /* configuration outside the built kernels         */
} asep_status;

/* Arithmetic the coupling / score network contractions run in. */
typedef enum {
  ASEP_PREC_FP32 = 0, /* CUDA-core fp32 kernels: bit-level "exact" mode used as the on-device checker   */
  ASEP_PREC_BF16 = 1, /* tcgen05 (UMMA) bf16 x bf16 -> fp32 TMEM accumulation: the production path      */
  ASEP_PREC_FP16 = 3,  /* Glow only: as ASEP_PREC_BF16 but the hidden activations / stage-2,3 weights of the forward
                        * coupling network are fp16 (10 mantissa bits): ~8x closer to fp32, ~8 % slower under the
                        * power cap.  The data-gradient pass stays bf16 (gradients have unbounded range).        */
  ASEP_PREC_BF16X3 = 2, /* score networks only: activations and weights as (hi + lo) bf16 pairs, three tcgen05
                         * products per convolution (hi.hi + lo.hi + hi.lo), fp32 accumulation: ~2^-16 relative */
  ASEP_PREC_BF16X2 = 4, /* Glow only: the tensor-core "exact" mode.  Hidden activations of the coupling network as
                         * (hi + lo) bf16 pairs (16 significant bits, fp32 range), two tcgen05 products per hidden GEMM
                         * against the bf16 weight images: meets inverse(forward(x)) <= 1e-4 on tensor cores      */
  ASEP_PREC_FP16X2 = 5, /* as ASEP_PREC_BF16X2 with (hi + lo) fp16 pairs (22 bits) and fp16 stage-2/3 weights in the
                         * forward network; hidden activations must stay below 65504 (else NaN); gradients use bf16 pairs */
  ASEP_PREC_FP16X3 = 6  /* Glow only: the score-exact tensor-core mode.  Weights as (hi + lo) pairs as well, three tcgen05
                         * products per GEMM (hi.hi + lo.hi + hi.lo); fp16 pairs end to end in the forward network
                         * (fp32-level pre-activations and ReLU masks), bf16 pairs in the data-gradient pass: meets the
                         * per-Langevin-step gate at every noise level like ASEP_PREC_FP32, on tensor cores           */
} asep_precision;

const char* asep_last_error(void);
int asep_abi_version(void);
/* Selects the device, checks it is sm_100, creates the library context. */
int asep_init(int device);
/* Number of kernels this library has launched since asep_init (all handles). */
int64_t asep_launch_count(void);

/* ------------------------------------------------------------------ Glow prior
 * Replaces flow_models/flow_builder.py:60-146 (build_glow) and the TFP distribution it
 * returns (log_prob / sample), plus run_basis_sep.py:73-79 (compute_grad_logprob). */
typedef struct {
  int32_t H, W, C;      /* data_shape, flow_builder.py:60                                  */
  int32_t L, K;         /* blocks, steps per block (configs/melspec_glow.yml:8-9)          */
  int32_t n_filters;    /* hidden width of ShiftAndLogScaleConvNet (flow_tfk_layers.py:46) */
  int32_t learntop;     /* learnable diagonal-Gaussian prior, flow_builder.py:130-141      */
  float minval, maxval; /* SpecPreprocessing(minval, maxval, use_logit=False)              */
} asep_glow_cfg;

typedef struct asep_glow_s* asep_glow_t;

int asep_glow_create(const asep_glow_cfg* cfg, asep_glow_t* out);
int asep_glow_destroy(asep_glow_t h);
/* Parameter names: see audiosourcesep_b200/weights.py ("b{b}/s{k}/actnorm/log_scale", ...).
 * Mirrors tf.Variable assignment / checkpoint restore (train_utils.py:62-75). */
int asep_glow_set_param(asep_glow_t h, const char* name, const DLTensor* value);
int asep_glow_get_param(asep_glow_t h, const char* name, DLTensor* out);
/* Derives the per-step constants (W, W^-1 in double, folded bf16 GEMM operands, constant
 * log-det terms).  Must be called after parameters change and before any compute call. */
int asep_glow_prepare(asep_glow_t h, int precision);
/* ActNorm data-dependent init incl. the raw-minibatch quirk of the 3/4-block classes
 * (flow_tfp_bijectors.py:222-240, flow_glow.py:44-49,156-174).  minibatch: [N,H,W,C] raw data. */
int asep_glow_init_actnorm(asep_glow_t h, const DLTensor* minibatch, void* stream);
/* Chain([glow, SpecPreprocessing]).forward + forward_log_det_jacobian (flow_builder.py:127,
 * flow_glow.py:176-209).  x [N,H,W,C] -> z [N,H/2^L,W/2^L,C*4^L], fldj [N]. */
int asep_glow_forward(asep_glow_t h, const DLTensor* x, DLTensor* z, DLTensor* fldj, void* stream);
/* Chain.inverse (flow_glow.py:187-196): z -> x. */
int asep_glow_inverse(asep_glow_t h, const DLTensor* z, DLTensor* x, void* stream);
/* TransformedDistribution.log_prob (flow_builder.py:140-141): x -> logp [N]. */
int asep_glow_log_prob(asep_glow_t h, const DLTensor* x, DLTensor* logp, void* stream);
/* compute_grad_logprob (run_basis_sep.py:73-79): grad [N,H,W,C]; logp may be NULL. */
int asep_glow_grad_log_prob(asep_glow_t h, const DLTensor* x, DLTensor* grad, DLTensor* logp, void* stream);
/* prior.sample -> Chain.inverse with the standard-normal draw injected: eps [N,latent]. */
int asep_glow_sample(asep_glow_t h, const DLTensor* eps, DLTensor* x, void* stream);

/* ------------------------------------------------------------------ Glow training step
 * Replaces train_glow.py:29-44 (loss = sum_i -log_prob(x_i) / global_batch, tape.gradient over all trainable
 * variables, optimizer.apply_gradients with Keras Adamax, train_utils.py:29-30) and the noise-perturbed loss of
 * train_noisy_glow.py:30-33.  Data parallelism = one process per GPU: every rank calls train_grads on its shard
 * with the GLOBAL batch size, the host all-reduces (SUM, NCCL) `grads` and `loss`, every rank calls adamax_step. */
/* Moves the trainables into one flat device vector (order: weights.py glow_param_shapes filtered by is_trainable),
 * allocates optimiser state.  Works in ASEP_PREC_FP32 (CUDA cores) and ASEP_PREC_BF16 / ASEP_PREC_FP16 (tcgen05, the
 * default); the split-precision modes have no weight-gradient path. */
int asep_glow_enable_training(asep_glow_t h);
int asep_glow_num_trainable(asep_glow_t h, int64_t* out);
/* x [N,H,W,C] raw data; noise NULL or [N,H,W,C] standard normals scaled by sigma and added to x in raw units
 * (train_noisy_glow.py:31-32); grads [num_trainable] and loss [1] are device float32 outputs. */
int asep_glow_train_grads(asep_glow_t h, const DLTensor* x, const DLTensor* noise, float sigma, int global_batch,
                          DLTensor* grads, DLTensor* loss, void* stream);
/* theta <- Adamax(theta, grads) with the Keras update m=b1 m+(1-b1) g; u=max(b2 u,|g|); theta -= lr/(1-b1^t) m/(u+eps);
 * then every derived per-step constant is refreshed on the device. */
int asep_glow_adamax_step(asep_glow_t h, const DLTensor* grads, float lr, float beta1, float beta2, float eps,
                          void* stream);
/* theta <- Adam(theta, grads), the Keras update of `optimizer: adam` (train_utils.py:27-28): m = b1 m + (1-b1) g;
 * v = b2 v + (1-b2) g^2; theta -= lr sqrt(1-b2^t)/(1-b1^t) m / (sqrt(v) + eps).  One optimizer per handle. */
int asep_glow_adam_step(asep_glow_t h, const DLTensor* grads, float lr, float beta1, float beta2, float eps,
                        void* stream);
/* Flat trainable vector out / in (device float32 [num_trainable]); set_flat refreshes the derived constants. */
int asep_glow_get_flat(asep_glow_t h, DLTensor* theta, void* stream);
int asep_glow_set_flat(asep_glow_t h, const DLTensor* theta, void* stream);
/* Copies the trained values back into the named-parameter store (get_param / prepare see them). */
int asep_glow_sync_host(asep_glow_t h);

/* ------------------------------------------------------------------ single bijectors
 * Stateless kernels behind the reference's Bijector classes, so each can be unit-tested the
 * way unittest_flow_models.py:25-51 does.  `inverse` != 0 selects _inverse. */
/* ActNorm (flow_tfp_bijectors.py:242-253): log_scale, shift [C] device tensors. */
int asep_actnorm(const DLTensor* x, const DLTensor* log_scale, const DLTensor* shift, DLTensor* y,
                 int inverse, void* stream);
/* Invertible1x1Conv (flow_tfp_bijectors.py:299-317): w [C,C] is W (forward) or W^-1 (inverse). */
int asep_inv1x1(const DLTensor* x, const DLTensor* w, DLTensor* y, void* stream);
/* AffineCouplingLayerSplit given the raw NN output r=[raw_log_s | t] (flow_tfp_bijectors.py:134-153);
 * logdet [N] (float32) is overwritten with sum tanh(raw) (forward) / its negative (inverse). */
int asep_coupling(const DLTensor* x, const DLTensor* r, DLTensor* y, DLTensor* logdet, int inverse, void* stream);
/* Squeeze (flow_tfp_bijectors.py:170-180). */
int asep_squeeze(const DLTensor* x, DLTensor* y, int inverse, void* stream);
/* ShiftAndLogScaleConvNet of step (block,step) of a prepared model (flow_tfk_layers.py:73-84):
 * state [N,Hb,Wb,Cb] (the second half of the channels is the network input) -> r [N,Hb,Wb,Cb]
 * = conv3 output before tanh/split. */
int asep_glow_coupling_nn(asep_glow_t h, int block, int step, const DLTensor* state, DLTensor* r, void* stream);
/* Data gradient of the same network: gr [N,Hb,Wb,Cb] -> gxb [N,Hb,Wb,Cb/2]. */
int asep_glow_coupling_nn_backward(asep_glow_t h, int block, int step, const DLTensor* state, const DLTensor* gr,
                                   DLTensor* gxb, void* stream);

/* ------------------------------------------------------------------ BASIS Langevin
 * One fused update of run_basis_sep.py:163-181 for both sources (dB mixing, :131-147):
 *   x_k <- x_k + eta*(s_k + lambda*softmax_k*(mixed - g(x1,x2))) + noise_scale*n_k
 * x1,x2 are updated in place from the OLD states.  n1/n2: injected standard normals, or NULL
 * for in-kernel Philox4x32-10 + Box-Muller keyed by (seed, step, global element index).
 * elem_offset = global index of element 0 (segment sharding keeps draws identical for any
 * number of GPUs).  nan_count: optional int32[1] device counter incremented per NaN. */
int asep_langevin_step(DLTensor* x1, DLTensor* x2, const DLTensor* s1, const DLTensor* s2, const DLTensor* mixed,
                       const DLTensor* n1, const DLTensor* n2, float eta, float lambda, float noise_scale,
                       uint64_t seed, uint64_t step, uint64_t elem_offset, DLTensor* nan_count, void* stream);
/* Mixing function g and its gradient (run_basis_sep.py:131-147), for tests. */
int asep_mixing_db(const DLTensor* x1, const DLTensor* x2, DLTensor* g, DLTensor* w1, DLTensor* w2, void* stream);
/* Standard normal draws of the in-kernel generator (for tests / reproducibility audits). */
int asep_philox_normal(DLTensor* out, uint64_t seed, uint64_t step, uint64_t stream_id, uint64_t elem_offset,
                       void* stream);
/* T inner steps at one noise level with two Glow priors (run_basis_sep.py:152-181, model_type
 * 'glow').  noise1/noise2: NULL or [T,N,H,W,C] injected draws; per_step: NULL or
 * [T,2,N,H,W,C] state dump for parity tests. */
int asep_basis_glow_inner(asep_glow_t m1, asep_glow_t m2, const DLTensor* mixed, DLTensor* x1, DLTensor* x2,
                          int T, float eta, float lambda, float noise_scale, const DLTensor* noise1,
                          const DLTensor* noise2, uint64_t seed, uint64_t step0, uint64_t elem_offset,
                          DLTensor* per_step, DLTensor* nan_count, void* stream);

/* ---- BASIS with K sources, 2 <= K <= 8 (any other K fails with ASEP_ERR_BAD_ARG before a launch).  Stacked layout: the
 * states, scores, injected noise, per-step dumps and snapshots of all K sources are ONE contiguous tensor with the source
 * axis after the step / level axis: x [K, ...], noise [T, K, ...], per_step [T, K, ...], snapshots [L, K, ...], where
 * ... is the shape of `mixed`.  The update is the two-source one with g = (10/ln10)(logsumexp_k(x_k ln10/10) - ln K) and
 * grad g = softmax_k; in-kernel noise of source k (0-based) is Philox stream k + 1, so K = 2 equals the two-source entry
 * points bit for bit.  The same handle may serve several sources. */
int asep_mixing_db_k(int K, const DLTensor* x, DLTensor* g, DLTensor* w, void* stream);
int asep_langevin_step_k(int K, DLTensor* x, const DLTensor* score, const DLTensor* mixed, const DLTensor* noise, float eta,
                         float lambda, float noise_scale, uint64_t seed, uint64_t step, uint64_t elem_offset,
                         DLTensor* nan_count, void* stream);
/* m: K Glow priors, one per source. */
int asep_basis_glow_inner_k(int K, const asep_glow_t* m, const DLTensor* mixed, DLTensor* x, int T, float eta, float lambda,
                            float noise_scale, const DLTensor* noise, uint64_t seed, uint64_t step0, uint64_t elem_offset,
                            DLTensor* per_step, DLTensor* nan_count, void* stream);
/* m: n_models * K handles, level i using m[(n_models == 1 ? 0 : i) * K + k] for source k. */
int asep_basis_glow_run_k(int K, const asep_glow_t* m, int n_models, const DLTensor* mixed, DLTensor* x, int L, int T,
                          const float* eta, const float* lambda, const float* noise_scale, uint64_t seed, uint64_t elem_offset,
                          DLTensor* snapshots, DLTensor* nan_count, void* stream);

/* ------------------------------------------------------------------ NCSN score networks
 * Replaces ncsn/utils.py:41-64 (get_uncompiled_model / get_uncompiled_model_v2) and the Keras call
 * `model([perturbed_X, sigma_idx], training=True)` on CondRefineNetDilated (ncsn/score_network.py:224-296,
 * version 1) / RefineNetDilated (ncsn/score_network_v2.py:202-278, version 2). */
typedef struct {
  int32_t version;      /* 1 = CondRefineNetDilated, 2 = RefineNetDilated                          */
  int32_t H, W, C;      /* data_shape (configs/melspec_ncsnv*.yml: 96, 64, 1)                       */
  int32_t ngf;          /* n_filters (192 for v1, 128 for v2)                                       */
  int32_t num_classes;  /* noise levels (rows of the v1 conditional-norm Embedding; length of sigmas) */
} asep_ncsn_cfg;

typedef struct asep_ncsn_s* asep_ncsn_t;

int asep_ncsn_create(const asep_ncsn_cfg* cfg, asep_ncsn_t* out);
int asep_ncsn_destroy(asep_ncsn_t h);
/* Parameter names: audiosourcesep_b200/weights.py:ncsn_param_shapes ("Res1_1/conv1/kernel", ...). */
int asep_ncsn_set_param(asep_ncsn_t h, const char* name, const DLTensor* value);
/* Noise levels sigma_1..sigma_L (host or device float32 [L]); v2 divides its output by sigma[idx]
 * (score_network_v2.py:275-276). */
int asep_ncsn_set_sigmas(asep_ncsn_t h, const DLTensor* sigmas);
/* ASEP_PREC_BF16 (default) or ASEP_PREC_BF16X3; takes effect at the next asep_ncsn_prepare(). */
int asep_ncsn_set_precision(asep_ncsn_t h, int precision);
/* Builds the bf16 tcgen05 weight tile images; call after parameters change. */
int asep_ncsn_prepare(asep_ncsn_t h);
/* score = model([x, sigma_idx], training=True): x [N,H,W,1] float32, sigma_idx [N] int32 -> score [N,H,W,1]. */
int asep_ncsn_forward(asep_ncsn_t h, const DLTensor* x, const DLTensor* sigma_idx, DLTensor* score, void* stream);
/* ---- NCSN denoising-score-matching training (replaces train_ncsn.py:26-57 train_step: get_noise_conditionned_data,
 * compute_train_loss, tape.gradient, optimizer.apply_gradients; optimizer of train_utils.py:23-41).
 * enable_training moves every parameter into one flat fp32 device vector (name order, each tensor 16-byte aligned) and
 * builds the data-gradient weight images; param_span gives a parameter's offset / element count in that vector.
 * train_grads: x [N,H,W,1] data, noise [N,H,W,1] standard-normal draws, sigma_idx [N] int32; perturbed_X = x +
 * sigma[idx] * noise; grads [num_trainable] <- d loss / d theta with loss [1] = sum_n 1/2 ||score + noise/sigma_n||^2 *
 * sigma_n^2 / global_batch (the SUM over data-parallel ranks is the reference's compute_average_loss).  The three GEMMs of
 * every convolution (forward, data gradient, weight gradient) run on tcgen05 in the handle's precision mode.
 * adam_step: Keras Adam on the flat vector, then the tile images are rebuilt on the device.  enable_training fails with
 * ASEP_ERR_UNSUPPORTED for patches wider than 64 (the weight gradient tiles 64 pixels; W = 128 runs inference only). */
int asep_ncsn_enable_training(asep_ncsn_t h);
int asep_ncsn_num_trainable(asep_ncsn_t h, int64_t* out);
int asep_ncsn_param_span(asep_ncsn_t h, const char* name, int64_t* offset, int64_t* numel);
int asep_ncsn_train_grads(asep_ncsn_t h, const DLTensor* x, const DLTensor* noise, const DLTensor* sigma_idx,
                          int global_batch, DLTensor* grads, DLTensor* loss, void* stream);
int asep_ncsn_adam_step(asep_ncsn_t h, const DLTensor* grads, float lr, float beta1, float beta2, float eps,
                        void* stream);
int asep_ncsn_get_flat(asep_ncsn_t h, DLTensor* theta, void* stream);
int asep_ncsn_set_flat(asep_ncsn_t h, const DLTensor* theta, void* stream);
/* T inner Langevin steps at noise level sigma_idx with two score networks (run_basis_sep.py:152-181, model_type
 * 'ncsn'); arguments as asep_basis_glow_inner. */
int asep_basis_ncsn_inner(asep_ncsn_t m1, asep_ncsn_t m2, const DLTensor* mixed, DLTensor* x1, DLTensor* x2,
                          int sigma_idx, int T, float eta, float lambda, float noise_scale, const DLTensor* noise1,
                          const DLTensor* noise2, uint64_t seed, uint64_t step0, uint64_t elem_offset,
                          DLTensor* per_step, DLTensor* nan_count, void* stream);
/* basis_outer_loop + basis_inner_loop (run_basis_sep.py:217-260, :152-181) entirely inside the library: L noise levels x T
 * Langevin steps with in-kernel Philox noise (step number = level * T + t, as the Python host numbers them), no host
 * synchronisation between levels.  eta / lambda / noise_scale: HOST arrays [L] of the float32 constants of :158-164.
 * snapshots: NULL or device [L, 2, N, H, W, C], the raw states after every level (x_arr, :243-244), copied on the
 * stream.  Glow: m1 / m2 are arrays of n_models handles, n_models = L (the per-sigma fine-tuned priors the reference
 * restores at :228-234, all resident) or 1 (one pair for every level). */
int asep_basis_glow_run(const asep_glow_t* m1, const asep_glow_t* m2, int n_models, const DLTensor* mixed, DLTensor* x1,
                        DLTensor* x2, int L, int T, const float* eta, const float* lambda, const float* noise_scale,
                        uint64_t seed, uint64_t elem_offset, DLTensor* snapshots, DLTensor* nan_count, void* stream);
int asep_basis_ncsn_run(asep_ncsn_t m1, asep_ncsn_t m2, const DLTensor* mixed, DLTensor* x1, DLTensor* x2, int L, int T,
                        const float* eta, const float* lambda, const float* noise_scale, uint64_t seed, uint64_t elem_offset,
                        DLTensor* snapshots, DLTensor* nan_count, void* stream);
/* K score networks m[K]; stacked layout and limits of asep_basis_glow_inner_k. */
int asep_basis_ncsn_inner_k(int K, const asep_ncsn_t* m, const DLTensor* mixed, DLTensor* x, int sigma_idx, int T, float eta,
                            float lambda, float noise_scale, const DLTensor* noise, uint64_t seed, uint64_t step0,
                            uint64_t elem_offset, DLTensor* per_step, DLTensor* nan_count, void* stream);
int asep_basis_ncsn_run_k(int K, const asep_ncsn_t* m, const DLTensor* mixed, DLTensor* x, int L, int T, const float* eta,
                          const float* lambda, const float* noise_scale, uint64_t seed, uint64_t elem_offset,
                          DLTensor* snapshots, DLTensor* nan_count, void* stream);
/* Event timing of the tcgen05 convolution launches of the score networks (same contract as asep_tc_profile). */
int asep_conv_profile(int on);
int asep_conv_profile_read(double* total_ms, int64_t* launches, double* flops);
/* ---- the tcgen05 convolutions of the score networks one launch at a time, so each can be tested against a float64
 * reference.  Shapes are checked before anything is launched (ASEP_ERR_BAD_SHAPE / _BAD_DTYPE / _UNSUPPORTED).
 * asep_conv_tc_image: kernel fp32 HWIO [k,k,Cin,Cout] (k = 1 or 3) -> img bf16 with k*k*Cin*Cout elements, the
 *   SWIZZLE_128B tile images the convolution streams: per (tap, 64-channel panel) one [rows x 64] block, element (r, c)
 *   at r*64 + (((c>>3) ^ (r&7))<<3) + (c&7).  transposed = 1: the image of the data gradient, K'[tap][co][ci] =
 *   K[k*k-1-tap][ci][co]; lo = 1: the low word bf16(v - bf16(v)) of the split-bf16 mode.  on_device = 1 builds it with
 *   the kernel the training step uses after every optimizer step (kernel on the device), on_device = 0 with the host
 *   builder of asep_ncsn_prepare (kernel on the host or the device; transposed = lo = 0 only).
 * asep_conv_tc_forward: out [N,H,W,Cout] fp32 = 'same' stride-1 convolution of x bf16 [N,H,W,Cin] with the image
 *   + bias [Cout] + add + add2 ([N,H,W,Cout] fp32).  bias, add, add2, stats and out_bf16 may be NULL; add may alias out.
 *   stats: float64 [N,Cout,2], per-(image, channel) sum and sum of squares of out (zeroed first); out_bf16: bf16 copy of
 *   out [N,H,W,Cout].  Cout in {128, 192, 256, 384}, Cin a multiple of 64, W dividing 128 and H a multiple of 128/W.
 * asep_conv_wgrad_tc: dk fp32 [k,k,Cin,Cout] += the weight gradient sum_p x[p + offset(tap)] g[p] of the same
 *   convolution (it accumulates); x bf16 [N,H,W,Cin], g bf16 [N,H,W,Cout], W dividing 64. */
int asep_conv_tc_image(const DLTensor* kernel, int transposed, int lo, int on_device, DLTensor* img, void* stream);
int asep_conv_tc_forward(const DLTensor* img, const DLTensor* bias, int ksize, int Cin, int Cout, int dil, const DLTensor* x,
                         const DLTensor* add, const DLTensor* add2, DLTensor* out, DLTensor* stats, DLTensor* out_bf16,
                         void* stream);
int asep_conv_wgrad_tc(const DLTensor* x, const DLTensor* g, DLTensor* dk, int ksize, int dil, void* stream);

/* CRC-32C (Castagnoli) of a HOST buffer, continuing from `crc` (0 to start): the checksum of the TensorFlow checkpoint
 * (TensorBundle) files tf.train.Checkpoint writes (train_utils.py:62-75), used by audiosourcesep_b200/tf_checkpoint.py. */
uint32_t asep_crc32c(const void* data, uint64_t n, uint32_t crc);

/* Measurement aid for the HBM-bound kernels (bench.py `roofline_hbm`): while on, every launch of a profiled category is
 * bracketed by a CUDA event pair on its own stream.  Categories: 0 fused flow step (ActNorm + 1x1 + coupling + log-det,
 * flow_tfp_bijectors.py:134-153,242-253,299-322), 1 fused Langevin update (run_basis_sep.py:163-181), 2 score-network
 * normalise + ELU + cast (score_network.py:203-221), 3 score-network pooling / resize (score_network.py:18,74,142),
 * 4 stand-alone col2im gather.  _read synchronises the events and returns the summed kernel time, the launch count and
 * the ALGORITHMIC bytes (what the op must read and write once) of the recorded launches. */
int asep_hbm_profile(int on);
int asep_hbm_profile_read(int category, double* total_ms, int64_t* launches, double* bytes);

/* ------------------------------------------------------------------ evaluation on the device
 * BSS Eval v4 (replaces bsseval_v4.py:79-300 bss_eval; helpers :449-617) for mono images.  reference_sources /
 * estimated_sources: device float64 [nsrc, nsampl].  The distortion filters (filters_len taps) are estimated on samples
 * [filt_start, filt_stop) (the whole signal for framewise_filters = False, the window itself otherwise); every window
 * [win_start[t], win_stop[t]) (HOST arrays) is decomposed into true source / spatial / interference / artifact parts
 * and out [4, nsrc, nsrc, nwin] float64 receives (SDR, ISR, SIR, SAR)[jtrue][jest][t] (s_r of :214; NaN where a source is
 * silent, :258-279).  sources_version = 1: the bss_eval_sources criteria (:575-585).  Framing, permutation search and
 * the result selection (:202-213, :281-300) stay on the host (audiosourcesep_b200/bsseval_v4.py). */
int asep_bss_eval(const DLTensor* reference_sources, const DLTensor* estimated_sources, int filters_len, int64_t filt_start,
                  int64_t filt_stop, const int64_t* win_start, const int64_t* win_stop, int nwin, int sources_version,
                  DLTensor* out, void* stream);
/* IRM_melspec (binary = 0) / IBM_melspec (binary = 1, majority vote theta) of oracle_systems.py:264-350: mixture
 * [...] and sources [nsrc, ...] fp32 mel spectrograms -> estimates [nsrc, ...]. */
int asep_ideal_mask(const DLTensor* mixture, const DLTensor* sources, DLTensor* estimates, int binary, float theta, void* stream);

/* ------------------------------------------------------------------ mel front end / back end
 * Replace the librosa calls of datasets/data_loader.py:144-162 (stft -> melspectrogram -> power_to_db -> clip) and of
 * melspec_inversion_basis.py:42-119 (db_to_power -> mel_to_stft -> phase re-use / single_channel_wiener_filter -> istft).
 * All tensors device fp32; complex64 arrays carry a trailing [2] (re, im).  The mel basis, its pseudo-inverse and the
 * index ranges are built on the host (audiosourcesep_b200/melspec.py, librosa.filters.mel restated).
 * asep_stft: audio [N, L] -> stft [N, n_fft/2+1, 1 + L/hop, 2]; periodic Hann, centred frames, reflect padding.
 * asep_mel_db: mel_db [N, M, T] = clip(power_to_db(basis |stft|^2, amin, top_db per segment), dbmin, dbmax).
 * asep_mel_to_stft: mag [N, F, T] = sqrt(argmin_{X>=0} ||basis X - 10^(mel_db/10)||): clipped least-squares start + `iters`
 *   FISTA steps (librosa uses L-BFGS-B from the same start; the minimiser is not unique -- see INTEGRATION.md).
 * asep_stft_filter: out [S, N, F, T, 2] = Wiener mask mag^2 / (sum_s mag^2 + 1e-10) * mixture (wiener = 1) or mag *
 *   exp(i angle(mixture)) (wiener = 0).
 * asep_istft: stft [N, F, T, 2] -> audio [N, hop (T-1)] (window sum-of-squares normalised overlap-add, centre trimmed). */
int asep_stft(const DLTensor* audio, int n_fft, int hop, DLTensor* stft, void* stream);
int asep_mel_db(const DLTensor* stft, const DLTensor* basis, const DLTensor* lo, const DLTensor* hi, DLTensor* mel_db, float amin,
                float top_db, float dbmin, float dbmax, void* stream);
int asep_mel_to_stft(const DLTensor* mel_db, const DLTensor* basis, const DLTensor* pinv, const DLTensor* flo, const DLTensor* fhi,
                     DLTensor* mag, float step, int iters, void* stream);
int asep_stft_filter(const DLTensor* mag, const DLTensor* stft_mixture, DLTensor* out, int wiener, void* stream);
int asep_istft(const DLTensor* stft, int hop, DLTensor* audio, void* stream);
/* Whole-track iSTFT of overlapping segments: stft [S, n_seg, F, T, 2] -> audio [S, length].  Segment g starts at sample g P,
 * P = V - O, V = hop (T-1) (the span one segment's iSTFT reconstructs), O = hop * overlap_frames.  Every sample is the
 * per-segment value asep_istft computes, cross-faded linearly over the O samples two neighbours share (hard cut when
 * overlap_frames = 0, no ramp at either end of the track) and written straight into the track; no per-segment waveform is
 * stored.  Requires 0 <= 2 overlap_frames < T - 1 (0..31 for T = 64) and length <= (n_seg-1) P + V (ASEP_ERR_BAD_ARG). */
int asep_istft_track(const DLTensor* stft, int hop, int overlap_frames, DLTensor* audio, void* stream);
/* One phase update of librosa.griffinlim (momentum variant; melspec_inversion_basis.py:21-39 through
 * librosa.feature.inverse.mel_to_audio): next = mag * unit(rebuilt - momentum/(1+momentum) * tprev); tprev <- rebuilt.
 * mag [...] fp32; rebuilt / tprev / next [..., 2] complex64.  The iteration (istft -> stft -> update) is driven from
 * audiosourcesep_b200/melspec.py:griffinlim. */
int asep_griffinlim_update(const DLTensor* mag, const DLTensor* rebuilt, DLTensor* tprev, DLTensor* next, float momentum,
                           void* stream);

/* ------------------------------------------------------------------ resampling
 * Replaces the resampler of librosa.load(path, sr=16000) (datasets/preprocessing.py:9-26; librosa's default
 * res_type='kaiser_best' = resampy.resample): audio [N, L_in] fp32 -> out [N, L_out] fp32.  time [L_out] float64 is
 * resampy's running time register (0, 1/ratio, 2/ratio, ... accumulated by repeated addition), shared by every row;
 * win / delta [nwin] fp32 the interpolation table and its forward differences (built on the host,
 * audiosourcesep_b200/resample.py); scale = min(1, ratio); step >= 1 the truncated table stride int(scale * 512).
 * librosa's length fix (ceil(L_in * ratio) samples) and the equal-rate short-cut stay on the host. */
int asep_resample(const DLTensor* audio, const DLTensor* time, const DLTensor* win, const DLTensor* delta, double scale, int step,
                  DLTensor* out, void* stream);

/* CUDA-graph replay of whole Langevin steps inside asep_basis_{glow,ncsn}_inner (on by default; steps 2..T of a call
 * with T >= 3 are replays of one captured step whose per-step scalars live in device memory).  0 = launch every step
 * eagerly (parity tests compare the two), and drop the cached graphs. */
int asep_basis_graphs(int on);

/* Measurement aid (bench.py roofline leg): while on, every launch of the tcgen05 coupling kernel is bracketed
 * by a CUDA event pair on its own stream.  _read synchronises those events and returns the summed kernel time,
 * the launch count and the algorithmic FLOPs (2 x conv MACs, unpadded) of the recorded launches. */
int asep_tc_profile(int on);
int asep_tc_profile_read(double* total_ms, int64_t* launches, double* flops);

#ifdef __cplusplus
}
#endif
#endif /* ASEP_H_ */
