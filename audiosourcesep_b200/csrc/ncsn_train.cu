// NCSN denoising-score-matching train step (reference: train_ncsn.py:26-57 -- get_noise_conditionned_data,
// compute_train_loss, train_step -- and train_utils.py:23-41 for the optimizer): loss, gradients of every parameter of
// CondRefineNetDilated / RefineNetDilated, Keras Adam on fp32 master weights, device-side rebuild of the tcgen05 weight
// images.  The forward walker of ncsn_model.cu records one tape entry per layer; the reverse sweep below replays it
// backwards.  Every convolution costs three tensor-core GEMMs: forward (k_conv_tc), data gradient (k_conv_tc on the
// transposed / flipped kernel image) and weight gradient (k_conv_wgrad_tc).
#include <cmath>
#include <cstring>

#include "ncsn_model.h"
#include "ncsn_train_kernels.h"
#include "train_kernels.h"

namespace asep {

void NcsnModel::enable_training() {
  if (training_) return;
  ASEP_CHECK(prepared_, ASEP_ERR_STATE, "asep_ncsn_prepare() must be called before asep_ncsn_enable_training()");
  ASEP_CHECK(sigmas_dev_ != nullptr, ASEP_ERR_STATE, "training needs the noise levels (asep_ncsn_set_sigmas)");
  // the weight gradient tiles 64 pixels where the forward convolution tiles 128 (W = 128 runs inference only): refuse
  // such a patch here instead of inside the first train_grads
  ASEP_CHECK(conv_wgrad_tc_supported(cfg_.ngf, cfg_.ngf, cfg_.H, cfg_.W) &&
                 conv_wgrad_tc_supported(2 * cfg_.ngf, 2 * cfg_.ngf, cfg_.H / 2, cfg_.W / 2),
             ASEP_ERR_UNSUPPORTED, "patch %dx%d with %d filters is outside the tcgen05 weight-gradient tiling (W <= 64)",
             cfg_.H, cfg_.W, cfg_.ngf);
  CUDA_CHECK(cudaSetDevice(device_));
  CUDA_CHECK(cudaDeviceSynchronize());
  ++generation_;
  long long off = 0;
  for (auto& kv : params_) {                       // std::map: name order
    kv.second.flat_off = off;
    off += ((long long)kv.second.host.size() + 3) & ~3LL;      // every tensor starts on a 16-byte boundary
  }
  n_flat_ = off;
  CUDA_CHECK(cudaMalloc(&theta_, (size_t)n_flat_ * sizeof(float)));
  CUDA_CHECK(cudaMemset(theta_, 0, (size_t)n_flat_ * sizeof(float)));
  CUDA_CHECK(cudaMalloc(&adam_m_, (size_t)n_flat_ * sizeof(float)));
  CUDA_CHECK(cudaMalloc(&adam_v_, (size_t)n_flat_ * sizeof(float)));
  CUDA_CHECK(cudaMemset(adam_m_, 0, (size_t)n_flat_ * sizeof(float)));
  CUDA_CHECK(cudaMemset(adam_v_, 0, (size_t)n_flat_ * sizeof(float)));
  CUDA_CHECK(cudaMalloc(&loss_acc_, sizeof(double)));
  for (auto& kv : params_) {
    NcsnParam& p = kv.second;
    float* dst = theta_ + p.flat_off;
    CUDA_CHECK(cudaMemcpy(dst, p.host.data(), p.host.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (p.dev) cudaFree(p.dev);
    p.dev = dst;
  }
  // convolution biases now live in the flat vector; data-gradient images next to the forward ones
  for (auto& kv : convs_) {
    ConvWeightsTC& w = kv.second;
    if (w.bias && w.bias_owned) cudaFree(w.bias);
    w.bias = has(kv.first + "/bias") ? params_.at(kv.first + "/bias").dev : nullptr;
    w.bias_owned = false;
    conv_tc_alloc(convs_t_[kv.first], w.ksize, w.Cout, w.Cin, w.dil);
    if (x3_) conv_tc_alloc(convs_t_lo_[kv.first], w.ksize, w.Cout, w.Cin, w.dil);
  }
  training_ = true;
  adam_t_ = 0;
  refresh_images(nullptr);
  CUDA_CHECK(cudaDeviceSynchronize());
}

void NcsnModel::param_span(const std::string& name, long long* offset, long long* numel) const {
  ASEP_CHECK(training_, ASEP_ERR_STATE, "asep_ncsn_enable_training() has not been called");
  const NcsnParam& p = param(name);
  if (offset) *offset = p.flat_off;
  if (numel) *numel = (long long)p.host.size();
}

// tile images (forward + data gradient, hi + lo) of every tensor-core convolution from the fp32 master kernels
void NcsnModel::refresh_images(cudaStream_t s) {
  for (auto& kv : convs_) {
    const ConvWeightsTC& w = kv.second;
    const float* k = params_.at(kv.first + "/kernel").dev;
    const int taps = w.ksize * w.ksize;
    launch_build_conv_image(k, w.img, taps, w.Cin, w.Cout, 0, 0, s);
    launch_build_conv_image(k, convs_t_.at(kv.first).img, taps, w.Cin, w.Cout, 1, 0, s);
    if (x3_) {
      launch_build_conv_image(k, convs_lo_.at(kv.first).img, taps, w.Cin, w.Cout, 0, 1, s);
      launch_build_conv_image(k, convs_t_lo_.at(kv.first).img, taps, w.Cin, w.Cout, 1, 1, s);
    }
  }
  images_dirty_ = false;
}

float* NcsnModel::grad_of(const float* p) const {
  auto it = grad_of_.find(p);
  ASEP_CHECK(it != grad_of_.end(), ASEP_ERR_STATE, "backward: tensor without a gradient buffer");
  return it->second;
}

float* NcsnModel::G(const std::string& name) const { return grads_cur_ + param(name).flat_off; }

void NcsnModel::train_grads(const float* x, const float* noise, const int* idx, int N, int global_batch, float* grads,
                            float* loss, cudaStream_t s) {
  ASEP_CHECK(training_, ASEP_ERR_STATE, "asep_ncsn_enable_training() has not been called");
  ASEP_CHECK(N >= 1 && global_batch >= N, ASEP_ERR_BAD_ARG, "bad batch sizes (local %d, global %d)", N, global_batch);
  CUDA_CHECK(cudaSetDevice(device_));
  s_ = s;
  N_ = N;
  const int HW = cfg_.H * cfg_.W;
  if (images_dirty_) refresh_images(s);
  // size both arenas with a dry run of the training graph
  train_ = true;
  dry_ = true; arena_off_ = 0; garena_off_ = 0;
  run(nullptr, nullptr, nullptr);
  // scratch of the reverse sweep: bf16 copies (hi, lo) of the largest output gradient, pooling temp, norm reductions
  const size_t big = (size_t)N * HW * (2 * cfg_.ngf);           // >= every activation (channels double where H, W halve)
  __nv_bfloat16* gob_hi = static_cast<__nv_bfloat16*>(take_g(big * sizeof(__nv_bfloat16)));
  __nv_bfloat16* gob_lo = static_cast<__nv_bfloat16*>(take_g(big * sizeof(__nv_bfloat16)));
  float* ptmp = static_cast<float*>(take_g(big * sizeof(float)));
  double* red = static_cast<double*>(take_g((size_t)N * 2 * cfg_.ngf * 2 * sizeof(double)));
  float2* qr = static_cast<float2*>(take_g((size_t)N * 2 * cfg_.ngf * sizeof(float2)));
  (void)gob_hi; (void)gob_lo; (void)ptmp; (void)red; (void)qr;
  const size_t need = arena_off_, gneed = garena_off_;
  dry_ = false;
  if (need > arena_cap_ || gneed > garena_cap_ || N > train_cap_) {
    CUDA_CHECK(cudaDeviceSynchronize());
    ++generation_;
    if (need > arena_cap_) {
      if (arena_) cudaFree(arena_);
      arena_ = nullptr;
      CUDA_CHECK(cudaMalloc(&arena_, need));
      arena_cap_ = need;
    }
    if (gneed > garena_cap_) {
      if (garena_) cudaFree(garena_);
      garena_ = nullptr;
      CUDA_CHECK(cudaMalloc(&garena_, gneed));
      garena_cap_ = gneed;
    }
    if (N > train_cap_) {
      for (float** p : {&xt_, &tscore_, &gscore_})
        if (*p) { cudaFree(*p); *p = nullptr; }
      for (float** p : {&xt_, &tscore_, &gscore_}) CUDA_CHECK(cudaMalloc(p, (size_t)N * HW * sizeof(float)));
      train_cap_ = N;
    }
  }
  arena_off_ = 0; garena_off_ = 0;
  tape_.clear();
  grad_of_.clear();
  grads_cur_ = grads;
  CUDA_CHECK(cudaMemsetAsync(garena_, 0, gneed, s));
  CUDA_CHECK(cudaMemsetAsync(grads, 0, (size_t)n_flat_ * sizeof(float), s));
  CUDA_CHECK(cudaMemsetAsync(loss_acc_, 0, sizeof(double), s));
  launch_dsm_perturb(x, noise, sigmas_dev_, idx, xt_, N, HW, s);              // train_ncsn.py:36-41
  try {
    run(xt_, idx, tscore_);                                                   // records the tape
    gob_hi = static_cast<__nv_bfloat16*>(take_g(big * sizeof(__nv_bfloat16)));
    gob_lo = static_cast<__nv_bfloat16*>(take_g(big * sizeof(__nv_bfloat16)));
    ptmp = static_cast<float*>(take_g(big * sizeof(float)));
    red = static_cast<double*>(take_g((size_t)N * 2 * cfg_.ngf * 2 * sizeof(double)));
    qr = static_cast<float2*>(take_g((size_t)N * 2 * cfg_.ngf * sizeof(float2)));
    launch_dsm_loss(tscore_, noise, sigmas_dev_, idx, gscore_, loss_acc_, N, HW, 1.0 / (double)global_batch, s);
    if (loss) launch_double_to_float(loss_acc_, loss, s);

    // ---- reverse sweep
    const int* sidx = v1_ ? idx : nullptr;       // Embedding rows are per-sample only in v1
    for (auto it = tape_.rbegin(); it != tape_.rend(); ++it) {
      const Op& o = *it;
      switch (o.kind) {
        case Op::kEnd: {
          const NcsnParam& ek = param("end_conv/kernel");
          const float* sg = v1_ ? nullptr : sigmas_dev_;
          launch_end_conv_bwd_data(gscore_, ek.dev, sg, sg ? idx : nullptr, o.bf.gy, N, cfg_.H, cfg_.W, cfg_.ngf, s);
          launch_end_conv_bwd_w(gscore_, o.bf.hi, o.bf.lo, sg, sg ? idx : nullptr, G("end_conv/kernel"), G("end_conv/bias"), N,
                                cfg_.H, cfg_.W, cfg_.ngf, s);
          break;
        }
        case Op::kPrep: {
          const T& xv = o.a;
          const T& xs = o.b;
          const int hw = xv.H * xv.W;
          if (o.norm.coef) {
            const std::string& nm = o.norm.name;
            launch_prep_bwd_reduce(xv.p, o.bf.gy, o.norm.coef, o.elu ? 1 : 0, red, N, hw, xv.C, s);
            const float *gamma, *alpha, *beta;
            float *dg, *da, *db;
            int stride = 0;
            if (v1_) {
              const float* e = param(nm + "/embed").dev;
              float* de = G(nm + "/embed");
              gamma = e; alpha = e + xv.C; beta = e + 2 * xv.C;
              dg = de; da = de + xv.C; db = de + 2 * xv.C;
              stride = 3 * xv.C;
            } else {
              gamma = param(nm + "/gamma").dev; alpha = param(nm + "/alpha").dev; beta = param(nm + "/beta").dev;
              dg = G(nm + "/gamma"); da = G(nm + "/alpha"); db = G(nm + "/beta");
            }
            launch_norm_bwd_coef(red, o.norm.sums, gamma, alpha, beta, stride, sidx, param(nm + "/in_gamma").dev,
                                 param(nm + "/in_beta").dev, dg, da, db, G(nm + "/in_gamma"), G(nm + "/in_beta"), qr, N, hw,
                                 xv.C, s);
            if (xs.p == xv.p) {
              launch_prep_bwd_apply(xv.p, o.bf.gy, o.norm.coef, o.elu ? 1 : 0, qr, xv.g, N, hw, xv.C, s);
            } else {                              // CRP: statistics of the un-pooled tensor, values of the pooled one
              launch_prep_bwd_apply(xv.p, o.bf.gy, o.norm.coef, o.elu ? 1 : 0, nullptr, xv.g, N, hw, xv.C, s);
              launch_prep_bwd_apply(xs.p, nullptr, nullptr, 0, qr, xs.g, N, hw, xs.C, s);
            }
          } else {
            launch_prep_bwd_apply(xv.p, o.bf.gy, nullptr, o.elu ? 1 : 0, nullptr, xv.g, N, hw, xv.C, s);
          }
          break;
        }
        case Op::kConv: {
          const ConvWeightsTC& w = convs_.at(o.name);
          const int H = o.a.H, W = o.a.W;
          const long long P = (long long)N * H * W;
          const float* gout = o.out.g;
          if (o.add) launch_axpy(gout, grad_of(o.add), P * w.Cout, s);
          if (o.add2) launch_axpy(gout, grad_of(o.add2), P * w.Cout, s);
          launch_prep(gout, nullptr, gob_hi, x3_ ? gob_lo : nullptr, N, H * W, w.Cout, 0, s);
          // data gradient: 'same' convolution of gout with the transposed, flipped kernel
          const ConvWeightsTC& wt = convs_t_.at(o.name);
          if (!x3_) {
            conv_tc_forward(wt, gob_hi, nullptr, o.bf.gy, N, H, W, s);
          } else {
            conv_tc_forward(convs_t_lo_.at(o.name), gob_hi, nullptr, o.bf.gy, N, H, W, s);
            conv_tc_forward(wt, gob_lo, o.bf.gy, o.bf.gy, N, H, W, s);
            conv_tc_forward(wt, gob_hi, o.bf.gy, o.bf.gy, N, H, W, s);
          }
          // weight gradient
          float* dk = G(o.name + "/kernel");
          if (x3_) {
            conv_wgrad_tc(o.bf.lo, gob_hi, dk, N, H, W, w.Cin, w.Cout, w.ksize, w.dil, s);
            conv_wgrad_tc(o.bf.hi, gob_lo, dk, N, H, W, w.Cin, w.Cout, w.ksize, w.dil, s);
          }
          conv_wgrad_tc(o.bf.hi, gob_hi, dk, N, H, W, w.Cin, w.Cout, w.ksize, w.dil, s);
          if (w.bias) launch_colsum_f32(gout, G(o.name + "/bias"), P, w.Cout, s);
          break;
        }
        case Op::kAvgPool2:
          launch_avgpool2_bwd(o.out.g, o.a.g, N, o.out.H, o.out.W, o.out.C, s);
          break;
        case Op::kPool5:
          if (v1_) launch_pool5_avg_bwd(o.out.g, ptmp, o.a.g, N, o.a.H, o.a.W, o.a.C, s);
          else launch_pool5_max_bwd(o.a.p, o.out.g, o.a.g, N, o.a.H, o.a.W, o.a.C, s);
          break;
        case Op::kResizeAdd:
          launch_resize2x_bwd(o.out.g, o.a.g, N, o.a.H, o.a.W, o.a.C, s);
          if (o.b.p) launch_axpy(o.out.g, o.b.g, (long long)N * o.out.H * o.out.W * o.out.C, s);
          break;
        case Op::kElu:
          launch_elu_bwd(o.a.p, o.out.g, o.a.g, (long long)N * o.a.H * o.a.W * o.a.C, s);
          break;
        case Op::kAdd: {
          const long long n = (long long)N * o.out.H * o.out.W * o.out.C;
          launch_axpy(o.out.g, o.a.g, n, s);
          launch_axpy(o.out.g, o.b.g, n, s);
          break;
        }
        case Op::kBegin:
          launch_begin_conv_bwd_w(xt_, o.out.g, G("begin_conv/kernel"), G("begin_conv/bias"), N, cfg_.H, cfg_.W, cfg_.ngf,
                                  v1_ ? 1 : 0, s);
          break;
      }
    }
  } catch (...) {
    train_ = false;
    throw;
  }
  train_ = false;
}

void NcsnModel::adam_step(const float* grads, float lr, float beta1, float beta2, float eps, cudaStream_t s) {
  ASEP_CHECK(training_, ASEP_ERR_STATE, "asep_ncsn_enable_training() has not been called");
  CUDA_CHECK(cudaSetDevice(device_));
  ++adam_t_;
  const double t = (double)adam_t_;
  const float lr_t = (float)((double)lr * std::sqrt(1.0 - std::pow((double)beta2, t)) / (1.0 - std::pow((double)beta1, t)));
  launch_adam(theta_, grads, adam_m_, adam_v_, n_flat_, lr_t, beta1, beta2, eps, s);
  refresh_images(s);
}

void NcsnModel::copy_flat(float* dst, cudaStream_t s) const {
  ASEP_CHECK(training_, ASEP_ERR_STATE, "asep_ncsn_enable_training() has not been called");
  CUDA_CHECK(cudaMemcpyAsync(dst, theta_, (size_t)n_flat_ * sizeof(float), cudaMemcpyDeviceToDevice, s));
}

void NcsnModel::set_flat(const float* src, cudaStream_t s) {
  ASEP_CHECK(training_, ASEP_ERR_STATE, "asep_ncsn_enable_training() has not been called");
  CUDA_CHECK(cudaMemcpyAsync(theta_, src, (size_t)n_flat_ * sizeof(float), cudaMemcpyDeviceToDevice, s));
  refresh_images(s);
}

void NcsnModel::sync_host() {
  if (!training_) return;
  CUDA_CHECK(cudaDeviceSynchronize());
  for (auto& kv : params_)
    CUDA_CHECK(cudaMemcpy(kv.second.host.data(), kv.second.dev, kv.second.host.size() * sizeof(float), cudaMemcpyDeviceToHost));
}

}  // namespace asep
