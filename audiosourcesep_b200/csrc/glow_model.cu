#include "glow_model.h"

#include <cmath>
#include <cstring>

namespace asep {

// ------------------------------------------------------------------ arena
void DeviceArena::reserve(size_t bytes) {
  if (bytes <= cap_) { off_ = 0; return; }
  release();
  CUDA_CHECK(cudaMalloc(&base_, bytes));
  cap_ = bytes;
  off_ = 0;
}
void* DeviceArena::take(size_t bytes) {
  size_t al = (bytes + 255) & ~(size_t)255;
  ASEP_CHECK(off_ + al <= cap_, ASEP_ERR_STATE, "arena overflow (%zu + %zu > %zu)", off_, al, cap_);
  void* p = base_ + off_;
  off_ += al;
  return p;
}
void DeviceArena::release() {
  if (base_) cudaFree(base_);
  base_ = nullptr;
  cap_ = off_ = 0;
}

// ------------------------------------------------------------------ small dense helpers (host, double)
namespace {
using Mat = std::vector<double>;
Mat matmul(const Mat& a, const Mat& b, int n) {
  Mat c((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < n; ++k)
      for (int j = 0; j < n; ++j) c[(size_t)i * n + j] += a[(size_t)i * n + k] * b[(size_t)k * n + j];
  return c;
}
Mat mat_inverse(Mat a, int n) {  // Gauss-Jordan with partial pivoting
  Mat inv((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i) inv[(size_t)i * n + i] = 1.0;
  for (int col = 0; col < n; ++col) {
    int piv = col;
    for (int r = col + 1; r < n; ++r)
      if (std::fabs(a[(size_t)r * n + col]) > std::fabs(a[(size_t)piv * n + col])) piv = r;
    ASEP_CHECK(std::fabs(a[(size_t)piv * n + col]) > 1e-300, ASEP_ERR_BAD_ARG, "singular 1x1-convolution factor");
    if (piv != col)
      for (int j = 0; j < n; ++j) {
        std::swap(a[(size_t)piv * n + j], a[(size_t)col * n + j]);
        std::swap(inv[(size_t)piv * n + j], inv[(size_t)col * n + j]);
      }
    double d = a[(size_t)col * n + col];
    for (int j = 0; j < n; ++j) { a[(size_t)col * n + j] /= d; inv[(size_t)col * n + j] /= d; }
    for (int r = 0; r < n; ++r) {
      if (r == col) continue;
      double f = a[(size_t)r * n + col];
      if (f == 0.0) continue;
      for (int j = 0; j < n; ++j) {
        a[(size_t)r * n + j] -= f * a[(size_t)col * n + j];
        inv[(size_t)r * n + j] -= f * inv[(size_t)col * n + j];
      }
    }
  }
  return inv;
}
float* dev_upload(const std::vector<float>& v) {
  float* d = nullptr;
  CUDA_CHECK(cudaMalloc(&d, std::max<size_t>(v.size(), 1) * sizeof(float)));
  CUDA_CHECK(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return d;
}
constexpr double kBnEps = 1e-3;  // Keras BatchNormalization epsilon
}  // namespace

// ------------------------------------------------------------------ construction
namespace { std::atomic<long long> g_next_uid{1}; }

GlowModel::GlowModel(const asep_glow_cfg& cfg, int device) : cfg_(cfg), device_(device) {
  uid_ = g_next_uid.fetch_add(1);
  ASEP_CHECK(cfg.L >= 2 && cfg.L <= 4, ASEP_ERR_BAD_ARG, "L should be 2, 3 or 4");   // flow_builder.py:77-78
  ASEP_CHECK(cfg.K >= 1 && cfg.n_filters >= 1 && cfg.C >= 1, ASEP_ERR_BAD_ARG, "bad K / n_filters / C");
  const int s = 1 << cfg.L;
  ASEP_CHECK(cfg.H % s == 0 && cfg.W % s == 0, ASEP_ERR_BAD_SHAPE, "H and W must be divisible by 2^L");
  ASEP_CHECK(cfg.maxval > cfg.minval, ASEP_ERR_BAD_ARG, "maxval must exceed minval");
  int c = cfg.C;
  for (int b = 0; b < cfg.L; ++b) {
    levels_.push_back(Level{cfg.H >> (b + 1), cfg.W >> (b + 1), c * 4});
    c = c * 4 / 2;
  }
  Hl_ = cfg.H / s; Wl_ = cfg.W / s; CL_ = cfg.C * s * s;
  Dl_ = Hl_ * Wl_ * CL_;
  const int F = cfg.n_filters;
  auto add = [&](const std::string& name, std::vector<int64_t> shape, float fill) {
    Param p;
    p.shape = std::move(shape);
    p.host.assign((size_t)p.numel(), fill);
    CUDA_CHECK(cudaMalloc(&p.dev, std::max<int64_t>(p.numel(), 1) * sizeof(float)));
    CUDA_CHECK(cudaMemcpy(p.dev, p.host.data(), p.host.size() * sizeof(float), cudaMemcpyHostToDevice));
    params_[name] = std::move(p);
    order_.push_back(name);
  };
  for (int b = 0; b < cfg.L; ++b) {
    const int C = levels_[b].C, Ch = C / 2;
    for (int k = 0; k < cfg.K; ++k) {
      const std::string pre = "b" + std::to_string(b) + "/s" + std::to_string(k) + "/";
      add(pre + "actnorm/log_scale", {C}, 0.f);
      add(pre + "actnorm/shift", {C}, 0.f);
      add(pre + "inv1x1/P", {C, C}, 0.f);
      add(pre + "inv1x1/L", {C, C}, 0.f);
      add(pre + "inv1x1/U", {C, C}, 0.f);
      add(pre + "inv1x1/log_S", {C}, 0.f);
      add(pre + "inv1x1/sign_S", {C}, 1.f);
      // identity permutation so that an un-parameterised model is still a bijection
      for (int i = 0; i < C; ++i) params_[pre + "inv1x1/P"].host[(size_t)i * C + i] = 1.f;
      CUDA_CHECK(cudaMemcpy(params_[pre + "inv1x1/P"].dev, params_[pre + "inv1x1/P"].host.data(),
                            (size_t)C * C * sizeof(float), cudaMemcpyHostToDevice));
      add(pre + "nn/conv1/kernel", {3, 3, Ch, F}, 0.f);
      add(pre + "nn/conv1/bias", {F}, 0.f);
      add(pre + "nn/bn1/gamma", {F}, 1.f);
      add(pre + "nn/bn1/beta", {F}, 0.f);
      add(pre + "nn/bn1/moving_mean", {F}, 0.f);
      add(pre + "nn/bn1/moving_variance", {F}, 1.f);
      add(pre + "nn/conv2/kernel", {F, F}, 0.f);
      add(pre + "nn/conv2/bias", {F}, 0.f);
      add(pre + "nn/bn2/gamma", {F}, 1.f);
      add(pre + "nn/bn2/beta", {F}, 0.f);
      add(pre + "nn/bn2/moving_mean", {F}, 0.f);
      add(pre + "nn/bn2/moving_variance", {F}, 1.f);
      add(pre + "nn/conv3/kernel", {3, 3, F, C}, 0.f);
      add(pre + "nn/conv3/bias", {C}, 0.f);
    }
  }
  if (cfg.learntop) {
    add("prior/loc", {Hl_, Wl_, CL_}, 0.f);
    add("prior/log_scale", {Hl_, Wl_, CL_}, 0.f);
  }
  steps_.resize((size_t)cfg.L * cfg.K);
}

GlowModel::~GlowModel() {
  for (auto& kv : params_)
    if (kv.second.dev && !kv.second.in_flat) cudaFree(kv.second.dev);
  if (score_buf_) cudaFree(score_buf_);
  if (refresh_table_) cudaFree(refresh_table_);
  if (tgraph_.exec) cudaGraphExecDestroy(tgraph_.exec);
  for (auto& kv : igraphs_)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  if (ig_stream_) cudaStreamDestroy(ig_stream_);
  for (void* p : {(void*)ig_in_, (void*)ig_out_, (void*)ig_lp_})
    if (p) cudaFree(p);
  if (tg_stream_) cudaStreamDestroy(tg_stream_);
  if (tg_ev_in_) cudaEventDestroy(tg_ev_in_);
  if (tg_ev_out_) cudaEventDestroy(tg_ev_out_);
  for (void* p : {(void*)tg_x_, (void*)tg_noise_, (void*)tg_grads_, (void*)tg_loss_})
    if (p) cudaFree(p);
  for (void* p : {(void*)theta_, (void*)adam_m_, (void*)adam_u_, (void*)tscratch_, (void*)ldc_, (void*)ld_total_,
                  (void*)da1_, (void*)da2_, (void*)dgp2_, (void*)dgp1_, (void*)dcol_})
    if (p) cudaFree(p);
  for (TrainSlot& t : tslots_) {
    for (void* p : {(void*)t.gp2, (void*)t.gp1, (void*)t.col, (void*)t.gr, (void*)t.gu, (void*)t.gxb, (void*)t.scratch})
      if (p) cudaFree(p);
    for (cudaEvent_t e : {t.ev_fork, t.ev_a, t.ev_join})
      if (e) cudaEventDestroy(e);
  }
  for (cudaStream_t q : tside_)
    if (q) cudaStreamDestroy(q);
  for (auto& s : steps_) {
    for (float* p : {s.sc, s.g1, s.b1, s.g2, s.b2, s.k2t})
      if (p) cudaFree(p);
    nn_tc_release(s.wtc);
  }
}

void GlowModel::set_param(const std::string& name, const float* src, const std::vector<int64_t>& shape,
                          bool src_on_device) {
  auto it = params_.find(name);
  ASEP_CHECK(it != params_.end(), ASEP_ERR_BAD_ARG, "unknown parameter '%s'", name.c_str());
  Param& p = it->second;
  int64_t n = 1;
  for (auto s : shape) n *= s;
  bool same = shape == p.shape;
  // conv2 kernel may arrive as Keras [1,1,F,F]
  if (!same && n == p.numel() && name.find("conv2/kernel") != std::string::npos) same = true;
  ASEP_CHECK(same, ASEP_ERR_BAD_SHAPE, "parameter '%s': shape mismatch (%lld elements given, %lld expected)",
             name.c_str(), (long long)n, (long long)p.numel());
  if (src_on_device) {
    CUDA_CHECK(cudaMemcpy(p.host.data(), src, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  } else {
    std::memcpy(p.host.data(), src, (size_t)n * sizeof(float));
  }
  CUDA_CHECK(cudaMemcpy(p.dev, p.host.data(), (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
  prepared_ = false;
}

const Param& GlowModel::get_param(const std::string& name) const {
  auto it = params_.find(name);
  ASEP_CHECK(it != params_.end(), ASEP_ERR_BAD_ARG, "unknown parameter '%s'", name.c_str());
  return it->second;
}

void GlowModel::require_prepared() const {
  ASEP_CHECK(prepared_, ASEP_ERR_STATE, "asep_glow_prepare() must be called after setting parameters");
}

// W = P (L*tril(-1)+I) (U*triu(+1)+diag(sign*exp(log_s)))   flow_tfp_bijectors.py:300-303
void GlowModel::build_step_consts(int b, int k) {
  const int C = levels_[b].C;
  const std::string pre = "b" + std::to_string(b) + "/s" + std::to_string(k) + "/";
  const auto& P = params_.at(pre + "inv1x1/P").host;
  const auto& Lp = params_.at(pre + "inv1x1/L").host;
  const auto& Up = params_.at(pre + "inv1x1/U").host;
  const auto& ls = params_.at(pre + "inv1x1/log_S").host;
  const auto& sg = params_.at(pre + "inv1x1/sign_S").host;
  const auto& an_ls = params_.at(pre + "actnorm/log_scale").host;
  const auto& an_sh = params_.at(pre + "actnorm/shift").host;
  Mat Pm((size_t)C * C), Lm((size_t)C * C, 0.0), Um((size_t)C * C, 0.0);
  for (int i = 0; i < C; ++i)
    for (int j = 0; j < C; ++j) {
      Pm[(size_t)i * C + j] = P[(size_t)i * C + j];
      if (j < i) Lm[(size_t)i * C + j] = Lp[(size_t)i * C + j];
      if (j > i) Um[(size_t)i * C + j] = Up[(size_t)i * C + j];
    }
  for (int i = 0; i < C; ++i) {
    Lm[(size_t)i * C + i] = 1.0;
    Um[(size_t)i * C + i] = (double)sg[i] * std::exp((double)ls[i]);
  }
  Mat Wm = matmul(Pm, matmul(Lm, Um, C), C);
  Mat Wi = matmul(mat_inverse(Um, C), matmul(mat_inverse(Lm, C), mat_inverse(Pm, C), C), C);   // :312-315
  std::vector<float> sc((size_t)step_const_floats(C));
  double sum_ls = 0.0, sum_lw = 0.0;
  for (int i = 0; i < C; ++i) {
    sc[i] = std::exp(an_ls[i]);
    sc[C + i] = an_sh[i];
    sum_ls += an_ls[i];
    sum_lw += ls[i];
  }
  for (int i = 0; i < C * C; ++i) {
    sc[2 * C + i] = (float)Wm[i];
    sc[2 * C + C * C + i] = (float)Wi[i];
  }
  StepDerived& sd = step(b, k);
  if (!sd.sc) CUDA_CHECK(cudaMalloc(&sd.sc, sc.size() * sizeof(float)));
  CUDA_CHECK(cudaMemcpy(sd.sc, sc.data(), sc.size() * sizeof(float), cudaMemcpyHostToDevice));
  sd.logdet_const = (double)levels_[b].H * levels_[b].W * (sum_ls + sum_lw);   // :250-253, :319-322
}

void GlowModel::invalidate_graphs() {
  ++generation_;                             // graphs captured elsewhere (api.cu: BASIS step graphs) are keyed by this
  if (tgraph_.exec) {
    cudaDeviceSynchronize();                 // a replay may still be in flight on the private stream
    cudaGraphExecDestroy(tgraph_.exec);
    tgraph_.exec = nullptr;
  }
  tg_calls_ = 0;                             // the next train_grads runs eagerly and re-sizes its scratch
  if (!igraphs_.empty()) {
    cudaDeviceSynchronize();
    for (auto& kv : igraphs_)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    igraphs_.clear();
  }
}

// ------------------------------------------------------------------ small-batch inference graphs
namespace { constexpr int kInferGraphMaxN = 128; }

bool GlowModel::infer_graph_ok(int N, cudaStream_t s) const {
  static const bool no_graph = getenv("ASEP_NO_GRAPH") != nullptr;
  if (no_graph || !is_tc() || N > kInferGraphMaxN || nn_tc_profile_enabled() || hbm_profile_enabled()) return false;
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess) { cudaGetLastError(); return false; }
  return st == cudaStreamCaptureStatusNone;      // (a BASIS step graph is being captured: launch directly)
}

template <class Body>
void GlowModel::run_infer_graph(int kind, int N, const float* in, size_t n_in, float* out, size_t n_out, float* lp,
                                cudaStream_t s, Body&& body) {
  InferGraph& g = igraphs_[{kind, N}];
  if (g.seen == 0) {                              // eager: allocates / re-carves whatever this direction needs
    const long long gen = generation_;
    body(in, out, lp, s);
    if (generation_ == gen) igraphs_[{kind, N}].seen = 1;   // (a re-carve cleared the map: the entry is new again)
    return;
  }
  if (N > ig_cap_) {
    CUDA_CHECK(cudaDeviceSynchronize());
    for (float** p : {&ig_in_, &ig_out_, &ig_lp_})
      if (*p) { cudaFree(*p); *p = nullptr; }
    const size_t d = (size_t)kInferGraphMaxN * std::max<size_t>((size_t)cfg_.H * cfg_.W * cfg_.C, (size_t)Dl_);
    CUDA_CHECK(cudaMalloc(&ig_in_, d * sizeof(float)));
    CUDA_CHECK(cudaMalloc(&ig_out_, d * sizeof(float)));
    CUDA_CHECK(cudaMalloc(&ig_lp_, (size_t)kInferGraphMaxN * sizeof(float)));
    ig_cap_ = kInferGraphMaxN;
  }
  if (!g.exec) {
    if (!ig_stream_) CUDA_CHECK(cudaStreamCreateWithFlags(&ig_stream_, cudaStreamNonBlocking));
    CUDA_CHECK(cudaStreamSynchronize(s));         // the eager pass of this key may still be using the workspace
    cudaGraph_t graph = nullptr;
    const long long c0 = g_launch_count.load();
    CUDA_CHECK(cudaStreamBeginCapture(ig_stream_, cudaStreamCaptureModeRelaxed));
    try {
      body(ig_in_, ig_out_, ig_lp_, ig_stream_);
    } catch (...) {
      cudaStreamEndCapture(ig_stream_, &graph);
      if (graph) cudaGraphDestroy(graph);
      throw;
    }
    CUDA_CHECK(cudaStreamEndCapture(ig_stream_, &graph));
    g.launches = g_launch_count.load() - c0;
    g_launch_count.fetch_sub(g.launches);         // a capture launches nothing
    CUDA_CHECK(cudaGraphInstantiate(&g.exec, graph, 0));
    CUDA_CHECK(cudaGraphDestroy(graph));
  }
  CUDA_CHECK(cudaMemcpyAsync(ig_in_, in, n_in * sizeof(float), cudaMemcpyDeviceToDevice, s));
  CUDA_CHECK(cudaGraphLaunch(g.exec, s));
  g_launch_count.fetch_add(g.launches);
  if (out) CUDA_CHECK(cudaMemcpyAsync(out, ig_out_, n_out * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (lp) CUDA_CHECK(cudaMemcpyAsync(lp, ig_lp_, (size_t)N * sizeof(float), cudaMemcpyDeviceToDevice, s));
}

void GlowModel::prepare(int precision) {
  const bool tcx_mode = precision == ASEP_PREC_BF16X2 || precision == ASEP_PREC_FP16X2 || precision == ASEP_PREC_FP16X3;
  const bool tc_mode = precision == ASEP_PREC_BF16 || precision == ASEP_PREC_FP16 || tcx_mode;
  const bool f16_mode = precision == ASEP_PREC_FP16 || precision == ASEP_PREC_FP16X2 || precision == ASEP_PREC_FP16X3;
  ASEP_CHECK(precision == ASEP_PREC_FP32 || tc_mode, ASEP_ERR_BAD_ARG, "unknown precision %d", precision);
  ASEP_CHECK(!(training_ && tcx_mode), ASEP_ERR_UNSUPPORTED,
             "the split-precision modes have no weight-gradient path: train in ASEP_PREC_BF16 / FP16 / FP32");
  const int F = cfg_.n_filters;
  if (tc_mode) {
    ASEP_CHECK(F == kTcF, ASEP_ERR_UNSUPPORTED, "the tcgen05 modes need n_filters = %d (got %d)", kTcF, F);
    for (int b = 0; b < cfg_.L; ++b)
      ASEP_CHECK(nn_tc_supported(levels_[b].C), ASEP_ERR_UNSUPPORTED,
                 "the tcgen05 coupling kernels are built for level widths 4, 8 and 16 (block %d has %d channels)", b,
                 levels_[b].C);
  }
  CUDA_CHECK(cudaSetDevice(device_));
  invalidate_graphs();                       // the per-step constants and tile images below are re-allocated
  refresh_dirty_ = true;                     // ... and so are the pointers in the device-side refresh table
  for (int b = 0; b < cfg_.L; ++b) {
    const int C = levels_[b].C;
    for (int k = 0; k < cfg_.K; ++k) {
      build_step_consts(b, k);
      const std::string pre = "b" + std::to_string(b) + "/s" + std::to_string(k) + "/nn/";
      StepDerived& sd = step(b, k);
      // inference-mode BatchNorm folded to y = g'*x + b'   (SURVEY.md 8(a) row 6)
      std::vector<float> g1(F), b1(F), g2(F), b2(F);
      auto fold = [&](const std::string& bn, std::vector<float>& g, std::vector<float>& bo) {
        const auto& ga = params_.at(pre + bn + "/gamma").host;
        const auto& be = params_.at(pre + bn + "/beta").host;
        const auto& mu = params_.at(pre + bn + "/moving_mean").host;
        const auto& va = params_.at(pre + bn + "/moving_variance").host;
        for (int i = 0; i < F; ++i) {
          double gg = (double)ga[i] / std::sqrt((double)va[i] + kBnEps);
          g[i] = (float)gg;
          bo[i] = (float)((double)be[i] - gg * (double)mu[i]);
        }
      };
      fold("bn1", g1, b1);
      fold("bn2", g2, b2);
      const auto& k2 = params_.at(pre + "conv2/kernel").host;
      std::vector<float> k2t((size_t)F * F);
      for (int i = 0; i < F; ++i)
        for (int j = 0; j < F; ++j) k2t[(size_t)j * F + i] = k2[(size_t)i * F + j];
      for (float** p : {&sd.g1, &sd.b1, &sd.g2, &sd.b2, &sd.k2t})
        if (*p) { cudaFree(*p); *p = nullptr; }
      sd.g1 = dev_upload(g1); sd.b1 = dev_upload(b1); sd.g2 = dev_upload(g2); sd.b2 = dev_upload(b2);
      sd.k2t = dev_upload(k2t);
      sd.w32.k1 = params_.at(pre + "conv1/kernel").dev; sd.w32.c1 = params_.at(pre + "conv1/bias").dev;
      sd.w32.g1 = sd.g1; sd.w32.b1 = sd.b1;
      sd.w32.k2 = params_.at(pre + "conv2/kernel").dev; sd.w32.k2t = sd.k2t;
      sd.w32.c2 = params_.at(pre + "conv2/bias").dev;
      sd.w32.g2 = sd.g2; sd.w32.b2 = sd.b2;
      sd.w32.k3 = params_.at(pre + "conv3/kernel").dev; sd.w32.c3 = params_.at(pre + "conv3/bias").dev;
      if (tc_mode) {
        nn_tc_prepare(sd.wtc, params_.at(pre + "conv1/kernel").host.data(), params_.at(pre + "conv1/bias").host.data(),
                      g1.data(), b1.data(), k2.data(), params_.at(pre + "conv2/bias").host.data(), g2.data(),
                      b2.data(), params_.at(pre + "conv3/kernel").host.data(),
                      params_.at(pre + "conv3/bias").host.data(), C, F, f16_mode, precision == ASEP_PREC_FP16X3);
      } else {
        nn_tc_release(sd.wtc);
      }
    }
  }
  if (precision != precision_) {   // the workspace composition depends on the precision
    CUDA_CHECK(cudaDeviceSynchronize());
    work_ = Work{};
  }
  precision_ = precision;
  prepared_ = true;
}

// Constant part of the log-det.  While training is enabled the per-step constants live on the device (ld_total_ is
// refreshed by derive_on_device after every optimizer step / set_flat): the host sum would be stale, so only the
// SpecPreprocessing term is returned here and launch_finish adds *const_logdet_dev().
double GlowModel::const_logdet() const {
  double s = 0.0;
  if (!training_)
    for (const auto& sd : steps_) s += sd.logdet_const;
  // SpecPreprocessing fldj: D * log(1/(max-min))      flow_tfp_bijectors.py:390-396
  s += (double)cfg_.H * cfg_.W * cfg_.C * std::log(1.0 / ((double)cfg_.maxval - (double)cfg_.minval));
  return s;
}

// latent slice of block b: Cz channels leave, reshaped row-major to [Hl*Wl, nb] at channel offset coff
void GlowModel::latent_slice(int b, int& Cz, int& nb, int& coff) const {
  coff = 0;
  for (int i = 0; i <= b; ++i) {
    const Level& lv = levels_[i];
    const bool last = i == cfg_.L - 1;
    const int cz = last ? lv.C : lv.C / 2;
    const int n = (int)((long long)lv.H * lv.W * cz / (Hl_ * Wl_));
    if (i == b) { Cz = cz; nb = n; return; }
    coff += n;
  }
}

// ------------------------------------------------------------------ workspace
void GlowModel::ensure_work(int N, bool save, bool dumps) {
  if (work_.N >= N && (work_.save || !save) && (work_.dumps || !dumps) && work_.N > 0) return;
  const int L = cfg_.L, K = cfg_.K, F = cfg_.n_filters;
  const bool fp32 = precision_ == ASEP_PREC_FP32;
  const long long M0 = (long long)N * levels_[0].H * levels_[0].W;
  // per-step mask storage: 128 B per pixel per step; kept while it stays below 48 GB
  double mask_bytes = 0.0;
  for (int b = 0; b < L; ++b) mask_bytes += 2.0 * N * levels_[b].H * levels_[b].W * (F / 8.0) * K;
  const bool keep_masks = mask_bytes <= 48e9;
  double dump_bytes = 0.0;
  for (int b = 0; b < L; ++b) dump_bytes += 2.0 * N * levels_[b].H * levels_[b].W * (double)F * 2.0 * K;
  dumps = dumps && save && !fp32 && keep_masks && dump_bytes <= 40e9;
  size_t bytes = 0;
  auto need = [&](size_t n) { bytes += (n + 255) & ~(size_t)255; };
  for (int pass = 0; pass < 2; ++pass) {
    if (pass == 1) {
      CUDA_CHECK(cudaDeviceSynchronize());
      invalidate_graphs();                   // the arena is re-carved (and possibly re-allocated)
      arena_.reserve(bytes);
      work_ = Work{};
      work_.N = N;
      work_.save = save;
      work_.X.resize(L); work_.O.resize(L); work_.U.resize(L); work_.R.resize(L);
      work_.M1.assign(L, {}); work_.M2.assign(L, {});
      work_.D1.assign(L, {}); work_.D2.assign(L, {});
      work_.dumps = dumps;
    }
    auto get = [&](size_t n_floats) -> float* {
      if (pass == 0) { need(n_floats * sizeof(float)); return nullptr; }
      return arena_.take_n<float>(n_floats);
    };
    for (int b = 0; b < L; ++b) {
      const size_t st = (size_t)N * levels_[b].H * levels_[b].W * levels_[b].C;
      float* x = get(st);
      float* o = get(st);
      if (pass == 1) { work_.X[b] = x; work_.O[b] = o; }
      const int nu = save ? std::max(K, 2) : 2, nr = save ? K : 1;
      for (int i = 0; i < nu; ++i) { float* u = get(st); if (pass == 1) work_.U[b].push_back(u); }
      for (int i = 0; i < nr; ++i) { float* r = get(st); if (pass == 1) work_.R[b].push_back(r); }
      if (save && !fp32 && keep_masks) {
        // 2 x 512 mask bits per pixel and step: the backward pass then needs no forward recompute
        const size_t mw = (size_t)N * levels_[b].H * levels_[b].W * (F / 32);
        for (int i = 0; i < K; ++i) {
          uint32_t* m1 = reinterpret_cast<uint32_t*>(get(mw));
          uint32_t* m2 = reinterpret_cast<uint32_t*>(get(mw));
          if (pass == 1) { work_.M1[b].push_back(m1); work_.M2[b].push_back(m2); }
        }
      }
      if (dumps) {
        const size_t dn = (size_t)N * levels_[b].H * levels_[b].W * F / 2;          // bf16 elements, counted in floats
        for (int i = 0; i < K; ++i) {
          __nv_bfloat16* d1 = reinterpret_cast<__nv_bfloat16*>(get(dn));
          __nv_bfloat16* d2 = reinterpret_cast<__nv_bfloat16*>(get(dn));
          if (pass == 1) { work_.D1[b].push_back(d1); work_.D2[b].push_back(d2); }
        }
      }
    }
    const size_t st0 = (size_t)M0 * levels_[0].C;
    float* z = get((size_t)N * Dl_);
    float* gz = get((size_t)N * Dl_);
    float *gA = get(st0), *gB = get(st0), *gr = get(st0), *gu = get(st0), *gxb = get(st0);
    double* acc = nullptr;
    if (pass == 0) need(2 * (size_t)N * sizeof(double)); else acc = arena_.take_n<double>(2 * (size_t)N);
    float *a1 = nullptr, *a2 = nullptr, *t1 = nullptr, *t2 = nullptr;
    NNScratchTC tc{};
    if (fp32) {
      a1 = get((size_t)M0 * F); a2 = get((size_t)M0 * F);
      if (save) { t1 = get((size_t)M0 * F); t2 = get((size_t)M0 * F); }
    } else {
      size_t gfl = 0;
      for (int b = 0; b < L; ++b)
        gfl = std::max(gfl, is_tcx() ? nn_tcx_g_floats((long long)N * levels_[b].H * levels_[b].W, levels_[b].C)
                                     : nn_tc_g_floats((long long)N * levels_[b].H * levels_[b].W, levels_[b].C));
      tc.G = get(gfl);
      if (save) {
        tc.mask1 = reinterpret_cast<uint32_t*>(get((size_t)M0 * (F / 32)));
        tc.mask2 = reinterpret_cast<uint32_t*>(get((size_t)M0 * (F / 32)));
      }
    }
    if (pass == 1) {
      work_.z = z; work_.gz = gz; work_.gA = gA; work_.gB = gB; work_.gr = gr; work_.gu = gu; work_.gxb = gxb;
      work_.acc_ld = acc; work_.acc_prior = acc + N;
      work_.a1 = a1; work_.a2 = a2; work_.t1 = t1; work_.t2 = t2; work_.tc = tc;
    }
  }
}

// ------------------------------------------------------------------ coupling network dispatch
// r == nullptr (tensor-core modes only): the col2im gather is left to the consuming flow-step kernel (fused_gather()).
void GlowModel::nn_forward(int b, int k, const float* state, float* r, int N, bool save, cudaStream_t s) {
  const Level& lv = levels_[b];
  StepDerived& sd = step(b, k);
  if (precision_ == ASEP_PREC_FP32) {
    nn_fp32_forward(sd.w32, state, work_.a1, work_.a2, r, N, lv.H, lv.W, lv.C, cfg_.n_filters, s);
  } else {
    uint32_t *m1 = nullptr, *m2 = nullptr;
    if (save && !work_.M1.empty() && !work_.M1[b].empty()) { m1 = work_.M1[b][k]; m2 = work_.M2[b][k]; }
    if (is_tcx()) {
      nn_tcx_forward(sd.wtc, work_.tc, state, r, m1, m2, N, lv.H, lv.W, lv.C, s);
    } else {
      __nv_bfloat16 *d1 = nullptr, *d2 = nullptr;
      if (save && dumping_ && !work_.D1[b].empty()) { d1 = work_.D1[b][k]; d2 = work_.D2[b][k]; }
      nn_tc_forward(sd.wtc, work_.tc, state, r, m1, m2, N, lv.H, lv.W, lv.C, s, d1, d2);
    }
  }
}

bool GlowModel::fused_gather(int b) const { return is_tc() && fused_gather_supported(levels_[b].C); }

GatherSrc GlowModel::gather_src(int b, int k, int N, bool backward) {
  const Level& lv = levels_[b];
  return nn_tc_gather_src(step(b, k).wtc, work_.tc, backward, (long long)N * lv.H * lv.W, lv.H, lv.W, is_tcx());
}

void GlowModel::nn_backward(int b, int k, const float* state, const float* gr, float* gxb, int N, cudaStream_t s) {
  const Level& lv = levels_[b];
  StepDerived& sd = step(b, k);
  // Activations are recomputed from the saved step input instead of being stored for all 120 steps
  // (flows are cheap to checkpoint: the step input is only C floats per pixel).
  if (precision_ == ASEP_PREC_FP32) {
    nn_fp32_forward(sd.w32, state, work_.a1, work_.a2, work_.gxb /*scratch r*/, N, lv.H, lv.W, lv.C,
                    cfg_.n_filters, s);
    nn_fp32_backward(sd.w32, work_.a1, work_.a2, gr, work_.t1, work_.t2, gxb, N, lv.H, lv.W, lv.C, cfg_.n_filters, s);
  } else if (is_tcx()) {
    nn_tcx_forward(sd.wtc, work_.tc, state, work_.gxb /*scratch r*/, work_.tc.mask1, work_.tc.mask2, N, lv.H, lv.W,
                   lv.C, s);
    nn_tcx_backward(sd.wtc, work_.tc, gr, work_.tc.mask1, work_.tc.mask2, gxb, N, lv.H, lv.W, lv.C, s);
  } else {
    nn_tc_forward(sd.wtc, work_.tc, state, work_.gxb /*scratch r*/, work_.tc.mask1, work_.tc.mask2, N, lv.H, lv.W,
                  lv.C, s);
    nn_tc_backward(sd.wtc, work_.tc, gr, work_.tc.mask1, work_.tc.mask2, gxb, N, lv.H, lv.W, lv.C, s);
  }
}

// ------------------------------------------------------------------ forward pass
// Leaves: work_.z (latent), work_.acc_ld (sum of data-dependent log-dets).  save=true keeps every
// step's coupling input u and network output r for the backward pass.
void GlowModel::run_forward(const float* x, int N, bool save, cudaStream_t s, bool dumps) {
  require_prepared();
  ensure_work(N, save, dumps);
  dumping_ = dumps && work_.dumps;            // only the training forward writes the activation copies
  const int L = cfg_.L, K = cfg_.K;
  CUDA_CHECK(cudaMemsetAsync(work_.acc_ld, 0, 2 * (size_t)work_.N * sizeof(double), s));
  // SpecPreprocessing + first squeeze
  launch_squeeze(x, work_.X[0], N, cfg_.H, cfg_.W, cfg_.C, 1, cfg_.minval, cfg_.maxval, 0, s);
  for (int b = 0; b < L; ++b) {
    const Level& lv = levels_[b];
    const long long M = (long long)N * lv.H * lv.W;
    const int HW = lv.H * lv.W;
    auto ubuf = [&](int k) { return work_.save ? work_.U[b][k] : work_.U[b][k & 1]; };
    auto rbuf = [&](int k) { return work_.save ? work_.R[b][k] : work_.R[b][0]; };
    // GlowBlock applies glowStep_{K-1} first (flow_glow.py:51-52)
    launch_pre(work_.X[b], ubuf(K - 1), step(b, K - 1).sc, M, lv.C, s);
    const bool fuse = fused_gather(b);
    for (int k = K - 1; k >= 0; --k) {
      float* out = k > 0 ? ubuf(k - 1) : work_.O[b];
      const float* sc_next = k > 0 ? step(b, k - 1).sc : nullptr;
      if (fuse) {
        // tensor-core modes: the flow-step kernel gathers the per-tap outputs itself; r is only written when the
        // backward pass will need it
        nn_forward(b, k, ubuf(k), nullptr, N, save, s);
        launch_post_pre_g(ubuf(k), gather_src(b, k, N, false), work_.save ? rbuf(k) : nullptr, out, sc_next, work_.acc_ld, M,
                          HW, lv.C, s);
      } else {
        nn_forward(b, k, ubuf(k), rbuf(k), N, save, s);
        launch_post_pre(ubuf(k), rbuf(k), out, sc_next, work_.acc_ld, M, HW, lv.C, s);
      }
    }
    int Cz, nb, coff;
    latent_slice(b, Cz, nb, coff);
    float* next = b + 1 < L ? work_.X[b + 1] : nullptr;
    launch_split_merge(work_.O[b], work_.z, next, N, lv.H, lv.W, lv.C, Cz, nb, CL_, coff, Dl_, 0, s);
  }
  dumping_ = false;
}

float* GlowModel::score_scratch(int N, int slots) {
  const size_t need = (size_t)slots * N * cfg_.H * cfg_.W * cfg_.C * sizeof(float);
  if (need > score_cap_) {
    CUDA_CHECK(cudaDeviceSynchronize());
    if (score_buf_) cudaFree(score_buf_);
    score_buf_ = nullptr;
    CUDA_CHECK(cudaMalloc(&score_buf_, need));
    score_cap_ = need;
  }
  return score_buf_;
}

void GlowModel::forward(const float* x, float* z, float* fldj, int N, cudaStream_t s) {
  if (N == 0) return;
  run_forward(x, N, false, s);
  CUDA_CHECK(cudaMemcpyAsync(z, work_.z, (size_t)N * Dl_ * sizeof(float), cudaMemcpyDeviceToDevice, s));
  launch_finish(work_.acc_ld, fldj, const_logdet(), 1.0, N, s, const_logdet_dev());
}

void GlowModel::log_prob(const float* x, float* logp, int N, cudaStream_t s) {
  if (N == 0) return;
  if (!infer_graph_ok(N, s)) return log_prob_body(x, logp, N, s);
  run_infer_graph(0, N, x, (size_t)N * cfg_.H * cfg_.W * cfg_.C, nullptr, 0, logp, s,
                  [&](const float* in, float*, float* lp, cudaStream_t st) { log_prob_body(in, lp, N, st); });
}

void GlowModel::log_prob_body(const float* x, float* logp, int N, cudaStream_t s) {
  run_forward(x, N, false, s);
  const float* loc = cfg_.learntop ? params_.at("prior/loc").dev : nullptr;
  const float* ls = cfg_.learntop ? params_.at("prior/log_scale").dev : nullptr;
  launch_prior(work_.z, loc, ls, work_.acc_ld, nullptr, N, Dl_, s);
  launch_finish(work_.acc_ld, logp, const_logdet(), 1.0, N, s, const_logdet_dev());
}

void GlowModel::grad_log_prob(const float* x, float* grad, float* logp, int N, cudaStream_t s) {
  if (N == 0) return;
  if (!infer_graph_ok(N, s)) return grad_log_prob_body(x, grad, logp, N, s);
  const size_t n = (size_t)N * cfg_.H * cfg_.W * cfg_.C;
  run_infer_graph(logp ? 2 : 1, N, x, n, grad, n, logp, s,
                  [&](const float* in, float* out, float* lp, cudaStream_t st) { grad_log_prob_body(in, out, lp, N, st); });
}

void GlowModel::grad_log_prob_body(const float* x, float* grad, float* logp, int N, cudaStream_t s) {
  run_forward(x, N, true, s);
  const int L = cfg_.L, K = cfg_.K;
  const float* loc = cfg_.learntop ? params_.at("prior/loc").dev : nullptr;
  const float* ls = cfg_.learntop ? params_.at("prior/log_scale").dev : nullptr;
  launch_prior(work_.z, loc, ls, work_.acc_ld, work_.gz, N, Dl_, s);
  if (logp) launch_finish(work_.acc_ld, logp, const_logdet(), 1.0, N, s, const_logdet_dev());
  // reverse sweep; gX holds the gradient w.r.t. the (squeezed) input state of the block below
  float* gX_next = nullptr;   // gradient w.r.t. X[b+1]
  for (int b = L - 1; b >= 0; --b) {
    const Level& lv = levels_[b];
    const long long M = (long long)N * lv.H * lv.W;
    int Cz, nb, coff;
    latent_slice(b, Cz, nb, coff);
    // gradient w.r.t. the block output: concat(reshape(gz_b), squeeze^-1 routing of gX[b+1])
    float* gy = work_.gA;
    float* other = work_.gB;
    if (gX_next == gy) std::swap(gy, other);
    launch_split_merge(gy, work_.gz, gX_next, N, lv.H, lv.W, lv.C, Cz, nb, CL_, coff, Dl_, 1, s);
    for (int k = 0; k < K; ++k) {          // steps were applied K-1..0, so unwind 0..K-1
      launch_bwd_coupling(gy, work_.U[b][k], work_.R[b][k], work_.gr, work_.gu, M, lv.C, s);
      const bool saved = is_tc() && !work_.M1.empty() && !work_.M1[b].empty();
      if (saved && fused_gather(b)) {          // masks kept from the forward pass: gradient GEMMs + fused col2im
        if (is_tcx()) nn_tcx_backward(step(b, k).wtc, work_.tc, work_.gr, work_.M1[b][k], work_.M2[b][k], nullptr, N, lv.H, lv.W, lv.C, s);
        else nn_tc_backward(step(b, k).wtc, work_.tc, work_.gr, work_.M1[b][k], work_.M2[b][k], nullptr, N, lv.H, lv.W, lv.C, s);
        launch_bwd_pre_g(work_.gu, gather_src(b, k, N, true), other, step(b, k).sc, M, lv.C, s);
      } else {
        if (saved && is_tcx())
          nn_tcx_backward(step(b, k).wtc, work_.tc, work_.gr, work_.M1[b][k], work_.M2[b][k], work_.gxb, N, lv.H, lv.W, lv.C, s);
        else if (saved)
          nn_tc_backward(step(b, k).wtc, work_.tc, work_.gr, work_.M1[b][k], work_.M2[b][k], work_.gxb, N, lv.H, lv.W, lv.C, s);
        else
          nn_backward(b, k, work_.U[b][k], work_.gr, work_.gxb, N, s);
        launch_bwd_pre(work_.gu, work_.gxb, other, step(b, k).sc, M, lv.C, s);
      }
      std::swap(gy, other);
    }
    gX_next = gy;
  }
  // through the first squeeze and SpecPreprocessing: d x'/d x = 1/(max-min)
  launch_squeeze(gX_next, grad, N, cfg_.H, cfg_.W, cfg_.C, 3, 1.0f / (cfg_.maxval - cfg_.minval), 0.f, 1, s);
}

void GlowModel::inverse(const float* z, float* x, int N, cudaStream_t s) {
  if (N == 0) return;
  if (!infer_graph_ok(N, s)) return inverse_body(z, x, N, s);
  run_infer_graph(3, N, z, (size_t)N * Dl_, x, (size_t)N * cfg_.H * cfg_.W * cfg_.C, nullptr, s,
                  [&](const float* in, float* out, float*, cudaStream_t st) { inverse_body(in, out, N, st); });
}

void GlowModel::inverse_body(const float* z, float* x, int N, cudaStream_t s) {
  require_prepared();
  ensure_work(N, false);
  const int L = cfg_.L, K = cfg_.K;
  // the merge kernel reads the latent through a non-const pointer but never writes it when merge=1
  float* zin = const_cast<float*>(z);
  for (int b = L - 1; b >= 0; --b) {
    const Level& lv = levels_[b];
    const long long M = (long long)N * lv.H * lv.W;
    int Cz, nb, coff;
    latent_slice(b, Cz, nb, coff);
    float* next = b + 1 < L ? work_.X[b + 1] : nullptr;
    float* y = work_.O[b];
    launch_split_merge(y, zin, next, N, lv.H, lv.W, lv.C, Cz, nb, CL_, coff, Dl_, 1, s);
    float* bufs[2] = {work_.U[b][0], work_.U[b][1]};
    for (int k = 0; k < K; ++k) {          // flow_glow.py: Chain.inverse walks steps 0..K-1
      float* out = (k == K - 1) ? work_.X[b] : bufs[k & 1];
      if (fused_gather(b)) {
        nn_forward(b, k, y, nullptr, N, false, s);
        launch_inv_step_g(y, gather_src(b, k, N, false), out, step(b, k).sc, nullptr, M, lv.H * lv.W, lv.C, s);
      } else {
        nn_forward(b, k, y, work_.R[b][0], N, false, s);
        launch_inv_step(y, work_.R[b][0], out, step(b, k).sc, nullptr, M, lv.H * lv.W, lv.C, s);
      }
      y = out;
    }
  }
  launch_squeeze(work_.X[0], x, N, cfg_.H, cfg_.W, cfg_.C, 2, cfg_.minval, cfg_.maxval, 1, s);
}

void GlowModel::sample(const float* eps, float* x, int N, cudaStream_t s) {
  if (N == 0) return;
  require_prepared();
  ensure_work(N, false);
  const float* loc = cfg_.learntop ? params_.at("prior/loc").dev : nullptr;
  const float* ls = cfg_.learntop ? params_.at("prior/log_scale").dev : nullptr;
  launch_prior_sample(eps, loc, ls, work_.gz, N, Dl_, s);
  inverse(work_.gz, x, N, s);
}

void GlowModel::coupling_nn(int block, int stepi, const float* state, float* r, int N, cudaStream_t s) {
  require_prepared();
  ASEP_CHECK(block >= 0 && block < cfg_.L && stepi >= 0 && stepi < cfg_.K, ASEP_ERR_BAD_ARG, "bad block/step");
  ensure_work(N, false);
  nn_forward(block, stepi, state, r, N, false, s);
}

void GlowModel::coupling_nn_backward(int block, int stepi, const float* state, const float* gr, float* gxb, int N,
                                     cudaStream_t s) {
  require_prepared();
  ASEP_CHECK(block >= 0 && block < cfg_.L && stepi >= 0 && stepi < cfg_.K, ASEP_ERR_BAD_ARG, "bad block/step");
  ensure_work(N, true);
  const Level& lv = levels_[block];
  // nn_backward uses work_.gxb as scratch for the recomputed forward output; keep the result separate
  const long long M = (long long)N * lv.H * lv.W;
  nn_backward(block, stepi, state, gr, work_.gu, N, s);
  CUDA_CHECK(cudaMemcpyAsync(gxb, work_.gu, (size_t)M * (lv.C / 2) * sizeof(float), cudaMemcpyDeviceToDevice, s));
}

// ------------------------------------------------------------------ ActNorm data-dependent init
// flow_tfp_bijectors.py:222-240 per step, walked in CONSTRUCTION order 0..K-1 (flow_glow.py:44-49);
// for L >= 3, blocks 2.. are initialised from the raw preprocessed minibatch re-tiled by Squeeze's -1
// reshape (flow_glow.py:162-174) -- quirk Q7.
void GlowModel::init_actnorm(const float* minibatch, int N, cudaStream_t s) {
  ASEP_CHECK(N >= 1, ASEP_ERR_BAD_SHAPE, "empty minibatch");
  CUDA_CHECK(cudaSetDevice(device_));
  // all actnorm parameters to identity first so that prepare() is well defined
  prepare(precision_);
  const int L = cfg_.L, K = cfg_.K;
  const size_t total = (size_t)N * cfg_.H * cfg_.W * cfg_.C;
  float *mb0 = nullptr, *carried = nullptr, *cur = nullptr, *u = nullptr, *r = nullptr, *tmp = nullptr;
  double* stats = nullptr;
  for (float** p : {&mb0, &carried, &cur, &u, &r, &tmp}) CUDA_CHECK(cudaMalloc(p, total * sizeof(float)));
  CUDA_CHECK(cudaMalloc(&stats, 2 * 64 * sizeof(double)));
  // mb0 = SpecPreprocessing.forward(minibatch) (flow_builder.py:96): squeeze mode 1 then undo the squeeze
  launch_squeeze(minibatch, tmp, N, cfg_.H, cfg_.W, cfg_.C, 1, cfg_.minval, cfg_.maxval, 0, s);
  launch_squeeze(tmp, mb0, N, cfg_.H, cfg_.W, cfg_.C, 0, 0.f, 0.f, 1, s);
  CUDA_CHECK(cudaMemcpyAsync(carried, mb0, total * sizeof(float), cudaMemcpyDeviceToDevice, s));
  for (int b = 0; b < L; ++b) {
    const Level& lv = levels_[b];
    const int Hin = lv.H * 2, Win = lv.W * 2, Cin = lv.C / 4;
    const bool quirk = L >= 3 && b >= 1;
    const float* src = quirk ? mb0 : carried;
    // elements available: the carried batch has N*Hin*Win*Cin elements; the raw one N*H*W*C, re-tiled
    const size_t elems = quirk ? total : (size_t)N * Hin * Win * Cin;
    const int Nb = (int)(elems / ((size_t)Hin * Win * Cin));
    const long long M = (long long)Nb * lv.H * lv.W;
    ensure_work(Nb, false);
    launch_squeeze(src, cur, Nb, Hin, Win, Cin, 0, 0.f, 0.f, 0, s);
    for (int k = 0; k < K; ++k) {
      launch_channel_stats(cur, stats, M, lv.C, s);
      std::vector<double> hs(2 * (size_t)lv.C);
      CUDA_CHECK(cudaMemcpyAsync(hs.data(), stats, hs.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
      const std::string pre = "b" + std::to_string(b) + "/s" + std::to_string(k) + "/actnorm/";
      Param& pls = params_.at(pre + "log_scale");
      Param& psh = params_.at(pre + "shift");
      for (int c = 0; c < lv.C; ++c) {
        const float mean = (float)hs[c];
        const float stdv = (float)hs[lv.C + c] + 1e-8f;
        pls.host[c] = std::log(1.0f / stdv);
        psh.host[c] = -mean / stdv;
      }
      CUDA_CHECK(cudaMemcpy(pls.dev, pls.host.data(), pls.host.size() * sizeof(float), cudaMemcpyHostToDevice));
      CUDA_CHECK(cudaMemcpy(psh.dev, psh.host.data(), psh.host.size() * sizeof(float), cudaMemcpyHostToDevice));
      build_step_consts(b, k);
      // minibatch_updated = glow_step.forward(minibatch_updated)
      launch_pre(cur, u, step(b, k).sc, M, lv.C, s);
      nn_forward(b, k, u, r, Nb, false, s);
      launch_post_pre(u, r, cur, nullptr, nullptr, M, lv.H * lv.W, lv.C, s);
    }
    if (b + 1 < L) {
      // the constructors re-run block.forward (steps K-1..0) on the carried batch and keep the second half
      const int Nc = N;
      const long long Mc = (long long)Nc * lv.H * lv.W;
      ensure_work(Nc, false);
      launch_squeeze(carried, cur, Nc, Hin, Win, Cin, 0, 0.f, 0.f, 0, s);
      for (int k = K - 1; k >= 0; --k) {
        launch_pre(cur, u, step(b, k).sc, Mc, lv.C, s);
        nn_forward(b, k, u, r, Nc, false, s);
        launch_post_pre(u, r, cur, nullptr, nullptr, Mc, lv.H * lv.W, lv.C, s);
      }
      // carried <- second half of the channels, kept UNSQUEEZED as [N, H, W, C/2]
      // (launch_split_merge would squeeze it; the next block's squeeze is applied at its own init)
      // reuse k_split_merge with Cz = C/2 writing the z-part to tmp and the squeezed rest to u, then unsqueeze u
      launch_split_merge(cur, tmp, u, Nc, lv.H, lv.W, lv.C, lv.C / 2, lv.H * lv.W * (lv.C / 2), 0, 0,
                         (long long)lv.H * lv.W * (lv.C / 2), 0, s);
      launch_squeeze(u, carried, Nc, lv.H, lv.W, lv.C / 2, 0, 0.f, 0.f, 1, s);
    }
  }
  CUDA_CHECK(cudaStreamSynchronize(s));
  for (float* p : {mb0, carried, cur, u, r, tmp}) cudaFree(p);
  cudaFree(stats);
  work_ = Work{};   // workspace sized for the init batch may be re-carved on the next call
  prepare(precision_);
}

}  // namespace asep
