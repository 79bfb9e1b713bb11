// Glow prior: parameters, derived per-step constants, workspace and the forward / inverse /
// log_prob / grad_log_prob orchestration over the kernels (reference: flow_models/flow_glow.py,
// flow_models/flow_builder.py:60-146, run_basis_sep.py:73-79).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "kernels.h"
#include "nn_tc.h"
#include "train_kernels.h"
#include "wgrad_tc.h"

namespace asep {

struct Param {
  std::vector<int64_t> shape;
  std::vector<float> host;
  float* dev = nullptr;
  bool in_flat = false;        // dev points into the flat trainable vector (training enabled)
  long long flat_off = -1;     // offset of a trainable parameter in the flat vector
  int64_t numel() const { int64_t n = 1; for (auto s : shape) n *= s; return n; }
};

struct Level { int H, W, C; };

struct StepDerived {
  float* sc = nullptr;          // element-wise constants (step_const_floats(C))
  double logdet_const = 0.0;    // H*W*(sum log_scale + sum log_S)
  float *g1 = nullptr, *b1 = nullptr, *g2 = nullptr, *b2 = nullptr, *k2t = nullptr;
  NNWeightsF32 w32{};
  NNWeightsTC wtc{};
};

class DeviceArena {
 public:
  ~DeviceArena() { release(); }
  void reserve(size_t bytes);
  void reset() { off_ = 0; }
  void* take(size_t bytes);
  template <typename T> T* take_n(size_t n) { return reinterpret_cast<T*>(take(n * sizeof(T))); }
  void release();
  size_t capacity() const { return cap_; }
 private:
  char* base_ = nullptr;
  size_t cap_ = 0, off_ = 0;
};

class GlowModel {
 public:
  explicit GlowModel(const asep_glow_cfg& cfg, int device);
  ~GlowModel();

  void set_param(const std::string& name, const float* src, const std::vector<int64_t>& shape, bool src_on_device);
  const Param& get_param(const std::string& name) const;
  void prepare(int precision);
  void init_actnorm(const float* minibatch, int N, cudaStream_t s);

  void forward(const float* x, float* z, float* fldj, int N, cudaStream_t s);
  void inverse(const float* z, float* x, int N, cudaStream_t s);
  void log_prob(const float* x, float* logp, int N, cudaStream_t s);
  void grad_log_prob(const float* x, float* grad, float* logp, int N, cudaStream_t s);
  void sample(const float* eps, float* x, int N, cudaStream_t s);
  void coupling_nn(int block, int step, const float* state, float* r, int N, cudaStream_t s);
  void coupling_nn_backward(int block, int step, const float* state, const float* gr, float* gxb, int N,
                            cudaStream_t s);

  // ---- training (train_glow.py:29-44, train_noisy_glow.py:30-33, train_utils.py:23-41)
  // Moves every trainable parameter into one flat device vector (order of weights.py:glow_param_shapes filtered by
  // is_trainable), allocates the Adamax state and the weight-gradient scratch.  Needs ASEP_PREC_FP32.
  void enable_training();
  long long num_trainable() const { return n_trainable_; }
  // grads [num_trainable] (device) <- d loss / d theta with loss = sum_i -log_prob(x_i + sigma*noise_i) / global_batch
  // over the N local samples (the SUM over data-parallel ranks is then the global-mean gradient); loss [1] likewise.
  void train_grads(const float* x, const float* noise, float sigma, int N, int global_batch, float* grads, float* loss,
                   cudaStream_t s);
  // Keras Adamax update of the flat vector, then every derived constant is refreshed on the device.
  void adamax_step(const float* grads, float lr, float beta1, float beta2, float eps, cudaStream_t s);
  // Keras Adam (train_utils.py:27-28); shares the two moment buffers with Adamax (one optimizer per handle)
  void adam_step(const float* grads, float lr, float beta1, float beta2, float eps, cudaStream_t s);
  // copies the flat vector back into the host-side parameter store (get_param / prepare see the trained values)
  void sync_host();
  void copy_flat(float* dst, cudaStream_t s) const;         // theta -> dst (device)
  void set_flat(const float* src, cudaStream_t s);          // src (device) -> theta, refresh constants

  // persistent scratch for a score tensor [N,H,W,C] (BASIS inner loop), grown on demand
  float* score_scratch(int N, int slots = 1);   // slots = 2: room for both sources when one handle serves as both priors

  const asep_glow_cfg& cfg() const { return cfg_; }
  int device() const { return device_; }
  const Level& level(int b) const { return levels_[b]; }
  int latent_dims() const { return Dl_; }
  int precision() const { return precision_; }
  bool is_tcx() const { return precision_ == ASEP_PREC_BF16X2 || precision_ == ASEP_PREC_FP16X2 || precision_ == ASEP_PREC_FP16X3; }   // split-precision tcgen05
  bool is_tc() const { return precision_ == ASEP_PREC_BF16 || precision_ == ASEP_PREC_FP16 || is_tcx(); }   // tcgen05 modes
  // prepared tile images and constants of the tensor-core coupling network of (block, step) (asep_glow_coupling_tc)
  const NNWeightsTC& tc_weights(int b, int k) const {
    require_prepared();
    return steps_[(size_t)b * cfg_.K + k].wtc;
  }
  // identity of the device allocations a captured graph of this model's kernels would bake in: a process-unique id of
  // the handle and a counter that advances whenever the workspace, the per-step constants or the tile images move
  long long uid() const { return uid_; }
  long long generation() const { return generation_; }

 private:
  struct Work {
    int N = 0;
    bool save = false;
    std::vector<float*> X, O;               // per level: block input / output state
    std::vector<std::vector<float*>> U, R;  // per level, per step (save) or 2 ping-pong / 1 (no save)
    std::vector<std::vector<uint32_t*>> M1, M2;   // tcgen05 path, save: ReLU bit masks of every step (no recompute in backward)
    // training on the tcgen05 path: bf16 copies of relu(p1), relu(p2) of every step, written by the forward pass, so that
    // the weight-gradient GEMMs need no second forward evaluation (kept while they fit in 40 GB)
    std::vector<std::vector<__nv_bfloat16*>> D1, D2;
    bool dumps = false;
    float *z = nullptr, *gz = nullptr, *gA = nullptr, *gB = nullptr, *gr = nullptr, *gu = nullptr, *gxb = nullptr;
    double *acc_ld = nullptr, *acc_prior = nullptr;
    float *a1 = nullptr, *a2 = nullptr, *t1 = nullptr, *t2 = nullptr;   // fp32 NN scratch
    NNScratchTC tc{};
  };
  void ensure_work(int N, bool save, bool dumps = false);
  StepDerived& step(int b, int k) { return steps_[(size_t)b * cfg_.K + k]; }
  void run_forward(const float* x, int N, bool save, cudaStream_t s, bool dumps = false);
  void nn_forward(int b, int k, const float* state, float* r, int N, bool save, cudaStream_t s);
  void nn_backward(int b, int k, const float* state, const float* gr, float* gxb, int N, cudaStream_t s);
  bool fused_gather(int b) const;                           // col2im of the tensor-core network fused into the flow-step kernels
  GatherSrc gather_src(int b, int k, int N, bool backward);
  void build_step_consts(int b, int k);
  void require_prepared() const;
  double const_logdet() const;
  const double* const_logdet_dev() const { return training_ ? ld_total_ : nullptr; }
  void latent_slice(int b, int& Cz, int& nb, int& coff) const;

  void derive_on_device(cudaStream_t s);
  StepRefresh* refresh_table_ = nullptr;     // device rows of the batched refresh (glow_train.cu)
  bool refresh_dirty_ = true;
  long long uid_ = 0, generation_ = 0;
  // ---- small-batch inference graphs: at the reference's batch sizes (N = 30 / 32) a pass is 250-850 launches of
  // 5-30 us each, so log_prob / inverse / grad_log_prob replay ONE captured CUDA graph per (direction, N) between
  // internal staging buffers (the caller's pointers change from call to call).  First call of a key: eager (sizes the
  // workspace); second: capture; then replays on the caller's stream.
  struct InferGraph { cudaGraphExec_t exec = nullptr; long long launches = 0; int seen = 0; };
  std::map<std::pair<int, int>, InferGraph> igraphs_;     // (direction, N)
  float *ig_in_ = nullptr, *ig_out_ = nullptr, *ig_lp_ = nullptr;
  int ig_cap_ = 0;
  cudaStream_t ig_stream_ = nullptr;
  bool infer_graph_ok(int N, cudaStream_t s) const;
  template <class Body> void run_infer_graph(int kind, int N, const float* in, size_t n_in, float* out, size_t n_out,
                                             float* lp, cudaStream_t s, Body&& body);
  void log_prob_body(const float* x, float* logp, int N, cudaStream_t s);
  void grad_log_prob_body(const float* x, float* grad, float* logp, int N, cudaStream_t s);
  void inverse_body(const float* z, float* x, int N, cudaStream_t s);
  bool dumping_ = false;                     // run_forward is writing the training activation copies (Work::D1 / D2)
  StepTrainPtrs step_ptrs(int b, int k);
  std::vector<std::string> order_;          // parameter names in construction order
  float *theta_ = nullptr, *adam_m_ = nullptr, *adam_u_ = nullptr;
  long long n_trainable_ = 0, adam_t_ = 0;
  float *tq2_ = nullptr, *tdc2_ = nullptr, *tr3_ = nullptr, *ts3_ = nullptr, *tdc1_ = nullptr, *td1_ = nullptr;
  __nv_bfloat16 *da1_ = nullptr, *da2_ = nullptr, *dgp2_ = nullptr, *dgp1_ = nullptr, *dcol_ = nullptr;   // bf16 dumps / im2col
  long long dump_rows_ = 0;
  // Ring of per-step backward buffers (tcgen05 training): the weight-gradient work of flow step k (GEMMs, column sums,
  // im2col, statistics, finalize) runs on two side streams while the main stream already computes the data gradient of
  // step k+1; a slot is reused once its side work has finished.  Everything the side work reads or accumulates into
  // that the next step would overwrite lives in the slot.
  static constexpr int kTrainRing = 4;
  struct TrainSlot {
    __nv_bfloat16 *gp2 = nullptr, *gp1 = nullptr, *col = nullptr;   // dL/dp2, dL/dp1 [rows, 512]; im2col scratch [rows, 256]
    float *gr = nullptr, *gu = nullptr, *gxb = nullptr;              // [rows, C] coupling gradients of the step
    char* scratch = nullptr;                                         // accumulators (layout of tscratch_)
    double* stats = nullptr;
    float *q2 = nullptr, *dc2 = nullptr, *dc1 = nullptr, *r3 = nullptr, *s3 = nullptr, *d1 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_a = nullptr, ev_join = nullptr;
    bool busy = false;
  };
  TrainSlot tslots_[kTrainRing];
  cudaStream_t tside_[2] = {nullptr, nullptr};
  long long slot_rows_ = 0;
  void ensure_train_slots(long long rows);
  void carve_scratch(char* base, TrainSlot& t) const;
  void ensure_train_dumps(long long rows);
  // The train step is ~5800 small launches at the reference's batch size (32): after a first eager call (which sizes
  // every scratch buffer) it is captured once per (N, global_batch, sigma, noisy) into a CUDA graph that works on
  // private staging buffers and is replayed on a private stream.
  void train_grads_body(const float* x, const float* noise, float sigma, int N, int global_batch, float* grads,
                        float* loss, cudaStream_t s);
  struct TrainGraph {
    cudaGraphExec_t exec = nullptr;
    int N = 0, global_batch = 0;
    float sigma = 0.f;
    bool noisy = false;
    long long launches = 0;
  } tgraph_;
  // Every captured graph bakes in device pointers of the workspace arena, the training dumps, the per-step constants
  // and the weight tile images: whenever one of those allocations is re-made (ensure_work with a larger batch,
  // ensure_train_dumps, prepare / init_actnorm / sync_host) the graphs are dropped and the next call runs eagerly.
  void invalidate_graphs();
  float *tg_x_ = nullptr, *tg_noise_ = nullptr, *tg_grads_ = nullptr, *tg_loss_ = nullptr;
  size_t tg_x_cap_ = 0;
  cudaStream_t tg_stream_ = nullptr;
  cudaEvent_t tg_ev_in_ = nullptr, tg_ev_out_ = nullptr;
  long long tg_calls_ = 0;      // largest batch size that has run eagerly (its scratch exists)
  double *tstats_ = nullptr, *ldc_ = nullptr, *ld_total_ = nullptr;
  char* tscratch_ = nullptr;                 // one allocation behind tstats_, tq2_, tdc2_, tdc1_, tr3_, ts3_, td1_
  size_t tscratch_bytes_ = 0;
  bool training_ = false;

  asep_glow_cfg cfg_;
  int device_;
  std::vector<Level> levels_;
  int Hl_, Wl_, CL_, Dl_;
  std::map<std::string, Param> params_;
  std::vector<StepDerived> steps_;
  bool prepared_ = false;
  int precision_ = ASEP_PREC_FP32;
  DeviceArena arena_;
  Work work_;
  float* score_buf_ = nullptr;
  size_t score_cap_ = 0;
};

}  // namespace asep
