// extern "C" surface of libasep.so (include/asep.h).  Everything below the ABI is C++/CUDA; errors
// cross as status codes + asep_last_error().
#include <cstdarg>
#include <cstring>
#include <map>
#include <memory>

#include <vector>
#include "bsseval.h"
#include "glow_model.h"
#include "mel_kernels.h"
#include "ncsn_model.h"
#include "ncsn_train_kernels.h"
#include "resample_kernels.h"

namespace asep {

std::atomic<long long> g_launch_count{0};

// ------------------------------------------------------------------ HBM-kernel profiler (common.cuh)
namespace {
struct HbmRec { cudaEvent_t a = nullptr, b = nullptr; int cat = 0; };
bool g_hbm_on = false;
std::vector<HbmRec*> g_hbm_recs, g_hbm_pool;
double g_hbm_bytes[kHbmCatCount] = {0};
}  // namespace

HbmScope::HbmScope(int cat, double bytes, cudaStream_t s) : cat_(cat), s_(s), rec_(nullptr) {
  if (!g_hbm_on) return;
  HbmRec* r;
  if (!g_hbm_pool.empty()) { r = g_hbm_pool.back(); g_hbm_pool.pop_back(); }
  else { r = new HbmRec(); cudaEventCreate(&r->a); cudaEventCreate(&r->b); }
  r->cat = cat;
  cudaEventRecord(r->a, s);
  g_hbm_bytes[cat] += bytes;
  rec_ = r;
}
HbmScope::~HbmScope() {
  if (!rec_) return;
  HbmRec* r = static_cast<HbmRec*>(rec_);
  cudaEventRecord(r->b, s_);
  g_hbm_recs.push_back(r);
}
bool hbm_profile_enabled() { return g_hbm_on; }
void hbm_profile(bool on) {
  g_hbm_on = on;
  if (on) {
    for (auto* r : g_hbm_recs) g_hbm_pool.push_back(r);
    g_hbm_recs.clear();
    for (double& b : g_hbm_bytes) b = 0.0;
  }
}
void hbm_profile_read(int cat, double* ms, long long* launches, double* bytes) {
  double t = 0.0;
  long long n = 0;
  for (auto* r : g_hbm_recs) {
    if (r->cat != cat) continue;
    cudaEventSynchronize(r->b);
    float e = 0.f;
    cudaEventElapsedTime(&e, r->a, r->b);
    t += e;
    ++n;
  }
  if (ms) *ms = t;
  if (launches) *launches = n;
  if (bytes) *bytes = (cat >= 0 && cat < kHbmCatCount) ? g_hbm_bytes[cat] : 0.0;
}
static thread_local std::string g_last_error;
static int g_device = -1;

std::string strfmt(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return std::string(buf);
}
void set_last_error(const std::string& m) { g_last_error = m; }

static int64_t check_contiguous(const DLTensor* t, const char* what) {
  int64_t n = 1;
  for (int i = 0; i < t->ndim; ++i) n *= t->shape[i];
  if (t->strides != nullptr) {
    int64_t expect = 1;
    for (int i = t->ndim - 1; i >= 0; --i) {
      if (t->shape[i] != 1 && t->strides[i] != expect)
        throw Error(ASEP_ERR_BAD_LAYOUT, strfmt("%s: tensor is not row-major contiguous", what));
      expect *= t->shape[i];
    }
  }
  return n;
}

static TView view_any(const DLTensor* t, const char* what, int device, bool allow_host, uint8_t code, uint8_t bits) {
  ASEP_CHECK(t != nullptr, ASEP_ERR_BAD_ARG, "%s: NULL tensor", what);
  ASEP_CHECK(t->ndim >= 0 && t->ndim <= 8, ASEP_ERR_BAD_SHAPE, "%s: unsupported rank %d", what, t->ndim);
  ASEP_CHECK(t->dtype.code == code && t->dtype.bits == bits && t->dtype.lanes == 1, ASEP_ERR_BAD_DTYPE,
             "%s: expected %s%d, got dtype code %d bits %d", what,
             code == kDLFloat ? "float" : (code == kDLBfloat ? "bfloat" : "int"), bits, t->dtype.code, t->dtype.bits);
  TView v;
  v.ndim = t->ndim;
  for (int i = 0; i < t->ndim; ++i) v.shape[i] = t->shape[i];
  v.numel = check_contiguous(t, what);
  const bool dev = t->device.device_type == kDLCUDA || t->device.device_type == kDLCUDAManaged;
  const bool host = t->device.device_type == kDLCPU || t->device.device_type == kDLCUDAHost;
  ASEP_CHECK(dev || (allow_host && host), ASEP_ERR_BAD_DEVICE, "%s: tensor must live on the CUDA device", what);
  if (dev && t->device.device_type == kDLCUDA)
    ASEP_CHECK(device < 0 || t->device.device_id == device, ASEP_ERR_BAD_DEVICE, "%s: tensor on cuda:%d, handle on cuda:%d",
               what, t->device.device_id, device);
  v.on_device = dev;
  v.raw = static_cast<char*>(t->data) + t->byte_offset;
  ASEP_CHECK(v.numel == 0 || v.raw != nullptr, ASEP_ERR_BAD_ARG, "%s: NULL data pointer", what);
  ASEP_CHECK((reinterpret_cast<uintptr_t>(v.raw) & 15) == 0, ASEP_ERR_BAD_LAYOUT, "%s: data must be 16-byte aligned", what);
  v.f32 = static_cast<float*>(v.raw);
  return v;
}
TView view_f32(const DLTensor* t, const char* what, int device, bool allow_host) {
  return view_any(t, what, device, allow_host, kDLFloat, 32);
}
TView view_i32(const DLTensor* t, const char* what, int device) { return view_any(t, what, device, false, kDLInt, 32); }

void expect_shape(const TView& v, const char* what, std::initializer_list<int64_t> shp) {
  bool ok = v.ndim == (int)shp.size();
  int i = 0;
  if (ok)
    for (auto s : shp) {
      ok = ok && (s < 0 || v.shape[i] == s);
      ++i;
    }
  if (!ok) {
    std::string got = "[", want = "[";
    for (int j = 0; j < v.ndim; ++j) got += std::to_string(v.shape[j]) + (j + 1 < v.ndim ? "," : "");
    int j = 0;
    for (auto s : shp) want += (s < 0 ? std::string("N") : std::to_string(s)) + (++j < (int)shp.size() ? "," : "");
    throw Error(ASEP_ERR_BAD_SHAPE, strfmt("%s: shape %s], expected %s]", what, got.c_str(), want.c_str()));
  }
}

}  // namespace asep

using namespace asep;

struct asep_glow_s {
  std::unique_ptr<GlowModel> model;
};
struct asep_ncsn_s {
  std::unique_ptr<NcsnModel> model;
};

#define ASEP_API_BEGIN try {
#define ASEP_API_END                                   \
  return ASEP_OK;                                      \
  }                                                    \
  catch (const ::asep::Error& e) {                     \
    ::asep::set_last_error(e.what());                  \
    return e.code;                                     \
  }                                                    \
  catch (const std::exception& e) {                    \
    ::asep::set_last_error(e.what());                  \
    return ASEP_ERR_CUDA;                              \
  }

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

const char* asep_last_error(void) { return g_last_error.c_str(); }
int asep_abi_version(void) { return ASEP_ABI_VERSION; }
int64_t asep_launch_count(void) { return (int64_t)g_launch_count.load(); }

int asep_init(int device) {
  ASEP_API_BEGIN
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  ASEP_CHECK(e == cudaSuccess && count > 0, ASEP_ERR_CUDA,
             "no CUDA device available (%s); libasep has no CPU fallback", cudaGetErrorString(e));
  ASEP_CHECK(device >= 0 && device < count, ASEP_ERR_BAD_ARG, "device %d out of range (%d devices)", device, count);
  CUDA_CHECK(cudaSetDevice(device));
  int major = 0, minor = 0;
  CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  CUDA_CHECK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
  ASEP_CHECK(major == 10, ASEP_ERR_UNSUPPORTED, "libasep is built for sm_100a only; device is sm_%d%d", major, minor);
  g_device = device;
  ASEP_API_END
}

// ------------------------------------------------------------------ Glow
int asep_glow_create(const asep_glow_cfg* cfg, asep_glow_t* out) {
  ASEP_API_BEGIN
  ASEP_CHECK(cfg != nullptr && out != nullptr, ASEP_ERR_BAD_ARG, "NULL argument");
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  auto h = new asep_glow_s();
  try {
    h->model.reset(new GlowModel(*cfg, g_device));
  } catch (...) {
    delete h;
    throw;
  }
  *out = h;
  ASEP_API_END
}

int asep_glow_destroy(asep_glow_t h) {
  ASEP_API_BEGIN
  if (h) {
    cudaDeviceSynchronize();
    delete h;
  }
  ASEP_API_END
}

int asep_glow_set_param(asep_glow_t h, const char* name, const DLTensor* value) {
  ASEP_API_BEGIN
  ASEP_CHECK(h && name, ASEP_ERR_BAD_ARG, "NULL argument");
  TView v = view_f32(value, name, h->model->device(), /*allow_host=*/true);
  std::vector<int64_t> shape(v.shape, v.shape + v.ndim);
  h->model->set_param(name, v.f32, shape, v.on_device);
  ASEP_API_END
}

int asep_glow_get_param(asep_glow_t h, const char* name, DLTensor* out) {
  ASEP_API_BEGIN
  ASEP_CHECK(h && name, ASEP_ERR_BAD_ARG, "NULL argument");
  const Param& p = h->model->get_param(name);
  TView v = view_f32(out, name, h->model->device(), true);
  ASEP_CHECK(v.numel == p.numel(), ASEP_ERR_BAD_SHAPE, "parameter '%s' has %lld elements, output has %lld", name,
             (long long)p.numel(), (long long)v.numel);
  if (v.on_device) CUDA_CHECK(cudaMemcpy(v.f32, p.dev, (size_t)v.numel * sizeof(float), cudaMemcpyDeviceToDevice));
  else std::memcpy(v.f32, p.host.data(), (size_t)v.numel * sizeof(float));
  ASEP_API_END
}

int asep_glow_prepare(asep_glow_t h, int precision) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  h->model->prepare(precision);
  ASEP_API_END
}

static int batch_of(const TView& x, const GlowModel& m, const char* what) {
  const auto& c = m.cfg();
  expect_shape(x, what, {-1, c.H, c.W, c.C});
  return (int)x.shape[0];
}
static void expect_latent(const TView& z, const GlowModel& m, int N, const char* what) {
  ASEP_CHECK(z.numel == (int64_t)N * m.latent_dims() && z.ndim >= 1 && z.shape[0] == N, ASEP_ERR_BAD_SHAPE,
             "%s: expected [%d, latent = %d] elements", what, N, m.latent_dims());
}

int asep_glow_init_actnorm(asep_glow_t h, const DLTensor* minibatch, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  TView x = view_f32(minibatch, "minibatch", h->model->device());
  int N = batch_of(x, *h->model, "minibatch");   // ActNorm asserts, flow_tfp_bijectors.py:218-220
  h->model->init_actnorm(x.f32, N, as_stream(stream));
  ASEP_API_END
}

int asep_glow_forward(asep_glow_t h, const DLTensor* x, DLTensor* z, DLTensor* fldj, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView xv = view_f32(x, "x", m.device());
  int N = batch_of(xv, m, "x");
  TView zv = view_f32(z, "z", m.device());
  expect_latent(zv, m, N, "z");
  TView lv = view_f32(fldj, "fldj", m.device());
  expect_shape(lv, "fldj", {N});
  m.forward(xv.f32, zv.f32, lv.f32, N, as_stream(stream));
  ASEP_API_END
}

int asep_glow_inverse(asep_glow_t h, const DLTensor* z, DLTensor* x, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView xv = view_f32(x, "x", m.device());
  int N = batch_of(xv, m, "x");
  TView zv = view_f32(z, "z", m.device());
  expect_latent(zv, m, N, "z");
  m.inverse(zv.f32, xv.f32, N, as_stream(stream));
  ASEP_API_END
}

int asep_glow_log_prob(asep_glow_t h, const DLTensor* x, DLTensor* logp, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView xv = view_f32(x, "x", m.device());
  int N = batch_of(xv, m, "x");
  TView lv = view_f32(logp, "logp", m.device());
  expect_shape(lv, "logp", {N});
  m.log_prob(xv.f32, lv.f32, N, as_stream(stream));
  ASEP_API_END
}

int asep_glow_grad_log_prob(asep_glow_t h, const DLTensor* x, DLTensor* grad, DLTensor* logp, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView xv = view_f32(x, "x", m.device());
  int N = batch_of(xv, m, "x");
  TView gv = view_f32(grad, "grad", m.device());
  expect_shape(gv, "grad", {N, m.cfg().H, m.cfg().W, m.cfg().C});
  float* lp = nullptr;
  if (logp != nullptr) {
    TView lv = view_f32(logp, "logp", m.device());
    expect_shape(lv, "logp", {N});
    lp = lv.f32;
  }
  m.grad_log_prob(xv.f32, gv.f32, lp, N, as_stream(stream));
  ASEP_API_END
}

int asep_glow_sample(asep_glow_t h, const DLTensor* eps, DLTensor* x, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView xv = view_f32(x, "x", m.device());
  int N = batch_of(xv, m, "x");
  TView ev = view_f32(eps, "eps", m.device());
  expect_latent(ev, m, N, "eps");
  m.sample(ev.f32, xv.f32, N, as_stream(stream));
  ASEP_API_END
}

int asep_glow_coupling_nn(asep_glow_t h, int block, int step, const DLTensor* state, DLTensor* r, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  ASEP_CHECK(block >= 0 && block < m.cfg().L, ASEP_ERR_BAD_ARG, "block out of range");
  const Level& lv = m.level(block);
  TView sv = view_f32(state, "state", m.device());
  expect_shape(sv, "state", {-1, lv.H, lv.W, lv.C});
  TView rv = view_f32(r, "r", m.device());
  expect_shape(rv, "r", {sv.shape[0], lv.H, lv.W, lv.C});
  m.coupling_nn(block, step, sv.f32, rv.f32, (int)sv.shape[0], as_stream(stream));
  ASEP_API_END
}

int asep_glow_coupling_nn_backward(asep_glow_t h, int block, int step, const DLTensor* state, const DLTensor* gr,
                                   DLTensor* gxb, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  ASEP_CHECK(block >= 0 && block < m.cfg().L, ASEP_ERR_BAD_ARG, "block out of range");
  const Level& lv = m.level(block);
  TView sv = view_f32(state, "state", m.device());
  expect_shape(sv, "state", {-1, lv.H, lv.W, lv.C});
  TView gv = view_f32(gr, "gr", m.device());
  expect_shape(gv, "gr", {sv.shape[0], lv.H, lv.W, lv.C});
  TView ov = view_f32(gxb, "gxb", m.device());
  expect_shape(ov, "gxb", {sv.shape[0], lv.H, lv.W, lv.C / 2});
  m.coupling_nn_backward(block, step, sv.f32, gv.f32, ov.f32, (int)sv.shape[0], as_stream(stream));
  ASEP_API_END
}

// ------------------------------------------------------------------ Glow training
int asep_glow_enable_training(asep_glow_t h) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  h->model->enable_training();
  ASEP_API_END
}

int asep_glow_num_trainable(asep_glow_t h, int64_t* out) {
  ASEP_API_BEGIN
  ASEP_CHECK(h && out, ASEP_ERR_BAD_ARG, "NULL argument");
  *out = (int64_t)h->model->num_trainable();
  ASEP_API_END
}

int asep_glow_train_grads(asep_glow_t h, const DLTensor* x, const DLTensor* noise, float sigma, int global_batch,
                          DLTensor* grads, DLTensor* loss, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView xv = view_f32(x, "x", m.device());
  const int N = batch_of(xv, m, "x");
  const float* nz = nullptr;
  if (noise) {
    TView nv = view_f32(noise, "noise", m.device());
    ASEP_CHECK(nv.numel == xv.numel, ASEP_ERR_BAD_SHAPE, "noise must have the shape of x");
    nz = nv.f32;
  }
  TView gv = view_f32(grads, "grads", m.device());
  ASEP_CHECK(gv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "grads must hold %lld elements", m.num_trainable());
  TView lv = view_f32(loss, "loss", m.device());
  ASEP_CHECK(lv.numel == 1, ASEP_ERR_BAD_SHAPE, "loss must hold one element");
  m.train_grads(xv.f32, nz, sigma, N, global_batch, gv.f32, lv.f32, as_stream(stream));
  ASEP_API_END
}

int asep_glow_adamax_step(asep_glow_t h, const DLTensor* grads, float lr, float beta1, float beta2, float eps,
                          void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView gv = view_f32(grads, "grads", m.device());
  ASEP_CHECK(gv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "grads must hold %lld elements", m.num_trainable());
  m.adamax_step(gv.f32, lr, beta1, beta2, eps, as_stream(stream));
  ASEP_API_END
}

int asep_glow_adam_step(asep_glow_t h, const DLTensor* grads, float lr, float beta1, float beta2, float eps,
                          void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView gv = view_f32(grads, "grads", m.device());
  ASEP_CHECK(gv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "grads must hold %lld elements", m.num_trainable());
  m.adam_step(gv.f32, lr, beta1, beta2, eps, as_stream(stream));
  ASEP_API_END
}

int asep_glow_get_flat(asep_glow_t h, DLTensor* theta, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView tv = view_f32(theta, "theta", m.device());
  ASEP_CHECK(tv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "theta must hold %lld elements", m.num_trainable());
  m.copy_flat(tv.f32, as_stream(stream));
  ASEP_API_END
}

int asep_glow_set_flat(asep_glow_t h, const DLTensor* theta, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel& m = *h->model;
  TView tv = view_f32(theta, "theta", m.device());
  ASEP_CHECK(tv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "theta must hold %lld elements", m.num_trainable());
  m.set_flat(tv.f32, as_stream(stream));
  ASEP_API_END
}

int asep_glow_sync_host(asep_glow_t h) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  h->model->sync_host();
  ASEP_API_END
}

// ------------------------------------------------------------------ single bijectors
static void nhwc(const TView& v, const char* what, int& N, int& H, int& W, int& C) {
  ASEP_CHECK(v.ndim == 4, ASEP_ERR_BAD_SHAPE, "%s: expected a [N,H,W,C] tensor", what);
  N = (int)v.shape[0]; H = (int)v.shape[1]; W = (int)v.shape[2]; C = (int)v.shape[3];
}

int asep_actnorm(const DLTensor* x, const DLTensor* log_scale, const DLTensor* shift, DLTensor* y, int inverse,
                 void* stream) {
  ASEP_API_BEGIN
  TView xv = view_f32(x, "x", g_device), yv = view_f32(y, "y", g_device);
  int N, H, W, C;
  nhwc(xv, "x", N, H, W, C);
  expect_shape(yv, "y", {N, H, W, C});
  TView ls = view_f32(log_scale, "log_scale", g_device), sh = view_f32(shift, "shift", g_device);
  expect_shape(ls, "log_scale", {C});
  expect_shape(sh, "shift", {C});
  launch_actnorm(xv.f32, ls.f32, sh.f32, yv.f32, (long long)N * H * W, C, inverse, as_stream(stream));
  ASEP_API_END
}

int asep_inv1x1(const DLTensor* x, const DLTensor* w, DLTensor* y, void* stream) {
  ASEP_API_BEGIN
  TView xv = view_f32(x, "x", g_device), yv = view_f32(y, "y", g_device), wv = view_f32(w, "w", g_device);
  int N, H, W, C;
  nhwc(xv, "x", N, H, W, C);
  expect_shape(yv, "y", {N, H, W, C});
  expect_shape(wv, "w", {C, C});
  ASEP_CHECK(xv.raw != yv.raw, ASEP_ERR_BAD_ARG, "inv1x1 cannot run in place");
  launch_chanmix(xv.f32, wv.f32, yv.f32, (long long)N * H * W, C, as_stream(stream));
  ASEP_API_END
}

int asep_coupling(const DLTensor* x, const DLTensor* r, DLTensor* y, DLTensor* logdet, int inverse, void* stream) {
  ASEP_API_BEGIN
  TView xv = view_f32(x, "x", g_device), rv = view_f32(r, "r", g_device), yv = view_f32(y, "y", g_device);
  int N, H, W, C;
  nhwc(xv, "x", N, H, W, C);
  ASEP_CHECK(C % 2 == 0, ASEP_ERR_BAD_SHAPE, "coupling needs an even channel count");   // flow_tfp_bijectors.py:130
  expect_shape(rv, "r", {N, H, W, C});
  expect_shape(yv, "y", {N, H, W, C});
  TView lv = view_f32(logdet, "logdet", g_device);
  expect_shape(lv, "logdet", {N});
  cudaStream_t s = as_stream(stream);
  double* acc = nullptr;
  CUDA_CHECK(cudaMalloc(&acc, std::max(N, 1) * sizeof(double)));
  CUDA_CHECK(cudaMemsetAsync(acc, 0, std::max(N, 1) * sizeof(double), s));
  float* sc = nullptr;
  try {
    if (!inverse) {
      launch_post_pre(xv.f32, rv.f32, yv.f32, nullptr, acc, (long long)N * H * W, H * W, C, s);
    } else {
      // identity ActNorm / 1x1 constants: the inverse kernel then reduces to the coupling inverse
      std::vector<float> id((size_t)step_const_floats(C), 0.f);
      for (int i = 0; i < C; ++i) { id[i] = 1.f; id[2 * C + i * C + i] = 1.f; id[2 * C + C * C + i * C + i] = 1.f; }
      CUDA_CHECK(cudaMalloc(&sc, id.size() * sizeof(float)));
      CUDA_CHECK(cudaMemcpyAsync(sc, id.data(), id.size() * sizeof(float), cudaMemcpyHostToDevice, s));
      launch_inv_step(xv.f32, rv.f32, yv.f32, sc, acc, (long long)N * H * W, H * W, C, s);
    }
    launch_finish(acc, lv.f32, 0.0, 1.0, N, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  } catch (...) {
    cudaFree(acc);
    if (sc) cudaFree(sc);
    throw;
  }
  cudaFree(acc);
  if (sc) cudaFree(sc);
  ASEP_API_END
}

int asep_squeeze(const DLTensor* x, DLTensor* y, int inverse, void* stream) {
  ASEP_API_BEGIN
  TView xv = view_f32(x, "x", g_device), yv = view_f32(y, "y", g_device);
  int N, H, W, C;
  nhwc(inverse ? yv : xv, inverse ? "y" : "x", N, H, W, C);      // the unsqueezed side
  ASEP_CHECK(H % 2 == 0 && W % 2 == 0, ASEP_ERR_BAD_SHAPE, "Squeeze needs even H and W");   // :165-166
  expect_shape(inverse ? xv : yv, inverse ? "x" : "y", {N, H / 2, W / 2, 4 * C});
  launch_squeeze(xv.f32, yv.f32, N, H, W, C, 0, 0.f, 0.f, inverse, as_stream(stream));
  ASEP_API_END
}

// ------------------------------------------------------------------ Langevin
static void check_sources(int K) {
  ASEP_CHECK(K >= 2 && K <= kMaxSources, ASEP_ERR_BAD_ARG, "the number of sources K must be in [2, %d] (got %d)", kMaxSources, K);
}

// v = [lead..., *item.shape]: the stacked layout of the K-source entry points (source axis after the step / level axis)
static void expect_stacked(const TView& v, const char* what, std::initializer_list<int64_t> lead, const TView& item) {
  bool ok = v.ndim == (int)lead.size() + item.ndim;
  int i = 0;
  for (auto l : lead) ok = ok && v.shape[i++] == l;
  for (int j = 0; ok && j < item.ndim; ++j) ok = v.shape[i + j] == item.shape[j];
  if (!ok) {
    std::string got = "[", want = "[";
    for (int j = 0; j < v.ndim; ++j) got += std::to_string(v.shape[j]) + (j + 1 < v.ndim ? "," : "");
    for (auto l : lead) want += std::to_string(l) + ",";
    for (int j = 0; j < item.ndim; ++j) want += std::to_string(item.shape[j]) + (j + 1 < item.ndim ? "," : "");
    throw Error(ASEP_ERR_BAD_SHAPE, strfmt("%s: shape %s], expected %s]", what, got.c_str(), want.c_str()));
  }
}

int asep_langevin_step(DLTensor* x1, DLTensor* x2, const DLTensor* s1, const DLTensor* s2, const DLTensor* mixed,
                       const DLTensor* n1, const DLTensor* n2, float eta, float lambda, float noise_scale,
                       uint64_t seed, uint64_t step, uint64_t elem_offset, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  TView a = view_f32(x1, "x1", g_device), b = view_f32(x2, "x2", g_device);
  TView sa = view_f32(s1, "s1", g_device), sb = view_f32(s2, "s2", g_device), mx = view_f32(mixed, "mixed", g_device);
  ASEP_CHECK(a.numel == b.numel && a.numel == sa.numel && a.numel == sb.numel && a.numel == mx.numel,
             ASEP_ERR_BAD_SHAPE, "langevin: all tensors must have the same number of elements");
  ASEP_CHECK((n1 == nullptr) == (n2 == nullptr), ASEP_ERR_BAD_ARG, "inject both noise tensors or neither");
  LangevinSources p{};
  p.x[0] = a.f32; p.x[1] = b.f32;
  p.s[0] = sa.f32; p.s[1] = sb.f32;
  if (n1) {
    TView na = view_f32(n1, "n1", g_device), nb = view_f32(n2, "n2", g_device);
    ASEP_CHECK(na.numel == a.numel && nb.numel == a.numel, ASEP_ERR_BAD_SHAPE, "noise shape mismatch");
    p.n[0] = na.f32; p.n[1] = nb.f32;
  }
  int* nanp = nullptr;
  if (nan_count) nanp = static_cast<int*>(view_i32(nan_count, "nan_count", g_device).raw);
  launch_langevin(2, p, mx.f32, eta, lambda, noise_scale, seed, step, elem_offset, nanp, a.numel, as_stream(stream));
  ASEP_API_END
}

int asep_langevin_step_k(int K, DLTensor* x, const DLTensor* score, const DLTensor* mixed, const DLTensor* noise, float eta,
                         float lambda, float noise_scale, uint64_t seed, uint64_t step, uint64_t elem_offset,
                         DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  check_sources(K);
  TView mx = view_f32(mixed, "mixed", g_device), xv = view_f32(x, "x", g_device), sv = view_f32(score, "score", g_device);
  expect_stacked(xv, "x", {K}, mx);
  expect_stacked(sv, "score", {K}, mx);
  const long long n = mx.numel;
  ASEP_CHECK(n % 4 == 0, ASEP_ERR_BAD_SHAPE, "langevin: the element count of one source (%lld) must be a multiple of 4", n);
  TView nv{};
  if (noise) {
    nv = view_f32(noise, "noise", g_device);
    expect_stacked(nv, "noise", {K}, mx);
  }
  int* nanp = nullptr;
  if (nan_count) nanp = static_cast<int*>(view_i32(nan_count, "nan_count", g_device).raw);
  LangevinSources p{};
  for (int k = 0; k < K; ++k) {
    p.x[k] = xv.f32 + k * n;
    p.s[k] = sv.f32 + k * n;
    p.n[k] = noise ? nv.f32 + k * n : nullptr;
  }
  launch_langevin(K, p, mx.f32, eta, lambda, noise_scale, seed, step, elem_offset, nanp, n, as_stream(stream));
  ASEP_API_END
}

int asep_mixing_db(const DLTensor* x1, const DLTensor* x2, DLTensor* g, DLTensor* w1, DLTensor* w2, void* stream) {
  ASEP_API_BEGIN
  TView a = view_f32(x1, "x1", g_device), b = view_f32(x2, "x2", g_device), gv = view_f32(g, "g", g_device);
  TView wa = view_f32(w1, "w1", g_device), wb = view_f32(w2, "w2", g_device);
  ASEP_CHECK(a.numel == b.numel && a.numel == gv.numel && a.numel == wa.numel && a.numel == wb.numel,
             ASEP_ERR_BAD_SHAPE, "mixing: element counts differ");
  MixingSources p{};
  p.x[0] = a.f32; p.x[1] = b.f32;
  p.w[0] = wa.f32; p.w[1] = wb.f32;
  launch_mixing_db(2, p, gv.f32, a.numel, as_stream(stream));
  ASEP_API_END
}

int asep_mixing_db_k(int K, const DLTensor* x, DLTensor* g, DLTensor* w, void* stream) {
  ASEP_API_BEGIN
  check_sources(K);
  TView xv = view_f32(x, "x", g_device), gv = view_f32(g, "g", g_device), wv = view_f32(w, "w", g_device);
  expect_stacked(xv, "x", {K}, gv);
  expect_stacked(wv, "w", {K}, gv);
  const long long n = gv.numel;
  MixingSources p{};
  for (int k = 0; k < K; ++k) {
    p.x[k] = xv.f32 + k * n;
    p.w[k] = wv.f32 + k * n;
  }
  launch_mixing_db(K, p, gv.f32, n, as_stream(stream));
  ASEP_API_END
}

int asep_philox_normal(DLTensor* out, uint64_t seed, uint64_t step, uint64_t stream_id, uint64_t elem_offset,
                       void* stream) {
  ASEP_API_BEGIN
  TView o = view_f32(out, "out", g_device);
  launch_philox_normal(o.f32, seed, step, stream_id, elem_offset, o.numel, as_stream(stream));
  ASEP_API_END
}

}  // extern "C" (re-opened below)

namespace {
// ---- CUDA graphs of one whole BASIS Langevin step (every score + the fused update), replayed for steps 2..T of a call.
// A graph bakes in the state / noise / dump pointers of the call and the workspaces of the priors, so it is keyed by
// all of them plus each source's prior (uid, generation); per-step scalars are read from `dev` (LangevinDev).  The score
// evaluations of distinct priors are independent until the update: each prior is captured as a branch of its own (the
// first on `stream`, the others on `side[]`), so the small HBM-bound launches of one prior overlap the tensor-core
// launches of the others.  A prior serving several sources evaluates them one after another on its branch.
struct BasisGraphKey {
  const void* p[3 + 3 * kMaxSources];               // mixed, dump, NaN counter, then every source's state, score, noise
  long long uid[kMaxSources], gen[kMaxSources];     // prior of every source
  unsigned long long seed, off;
  long long noise_stride;
  int N, kind, K, pad;                              // kind: 0 Glow priors, 1 NCSN
  bool operator<(const BasisGraphKey& o) const { return std::memcmp(this, &o, sizeof(*this)) < 0; }
};
struct BasisGraph { cudaGraphExec_t exec = nullptr; long long launches = 0; };
struct BasisGraphs {
  std::map<BasisGraphKey, BasisGraph> graphs;
  cudaStream_t stream = nullptr;                    // private: the caller's stream may be the legacy stream (not capturable)
  cudaStream_t side[kMaxSources - 1] = {};
  cudaEvent_t ev_in = nullptr, ev_out = nullptr, ev_fork = nullptr, ev_join[kMaxSources - 1] = {};
  LangevinDev* dev = nullptr;
  bool enabled = true;
  void ensure() {
    if (stream) return;
    CUDA_CHECK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    for (cudaStream_t& st : side) CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    for (cudaEvent_t* e : {&ev_in, &ev_out, &ev_fork}) CUDA_CHECK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    for (cudaEvent_t& e : ev_join) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CUDA_CHECK(cudaMalloc(&dev, sizeof(LangevinDev)));
  }
  void clear() {
    if (stream) cudaStreamSynchronize(stream);
    for (auto& kv : graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    graphs.clear();
  }
};
BasisGraphs& basis_graphs() {
  static BasisGraphs g;
  return g;
}

// One call of T Langevin steps over K sources.  src.n[k] is the base of source k's injected noise (step t at
// src.n[k] + t * noise_stride) or NULL; dump the base of the [T, K, ...] per-step dump or NULL.
struct BasisCall {
  int K;
  LangevinSources src;
  long long noise_stride;
  const float* mixed;
  float* dump;
  int* nanp;
  long long numel;                                  // elements of one source
  int N, T;
  float eta, lambda, noise_scale;
  uint64_t seed, step0, elem_offset;
};

// Sources grouped by prior handle, in order of first use.  The reference treats priors as plain callables
// (run_basis_sep.py:166-175), so one handle may serve several sources: its score scratch then holds one tensor per source.
template <class M>
struct SourceGroups {
  std::vector<M*> models;
  std::vector<std::vector<int>> sources;
};
template <class M>
SourceGroups<M> group_sources(BasisCall& c, M* const* m) {
  SourceGroups<M> g;
  for (int k = 0; k < c.K; ++k) {
    size_t b = 0;
    while (b < g.models.size() && g.models[b] != m[k]) ++b;
    if (b == g.models.size()) {
      g.models.push_back(m[k]);
      g.sources.emplace_back();
    }
    g.sources[b].push_back(k);
  }
  for (size_t b = 0; b < g.models.size(); ++b) {
    float* buf = g.models[b]->score_scratch(c.N, (int)g.sources[b].size());
    for (size_t j = 0; j < g.sources[b].size(); ++j) c.src.s[g.sources[b][j]] = buf + j * c.numel;
  }
  return g;
}

// score(b, stream) launches the score evaluations of branch b (one prior, every source it serves) into c.src.s.
// generations(key) fills key.gen; it is called after the first (eager) step has sized every workspace.
template <class FS, class FG>
void run_basis_steps(const BasisCall& c, BasisGraphKey key, int branches, bool allow_graph, cudaStream_t s, FS&& score,
                     FG&& generations) {
  auto eager_step = [&](int t) {
    for (int b = 0; b < branches; ++b) score(b, s);
    LangevinSources p = c.src;
    for (int k = 0; k < c.K; ++k)
      if (p.n[k]) p.n[k] += (size_t)t * c.noise_stride;
    launch_langevin(c.K, p, c.mixed, c.eta, c.lambda, c.noise_scale, c.seed, c.step0 + t, c.elem_offset, c.nanp, c.numel, s);
    if (c.dump)
      for (int k = 0; k < c.K; ++k)
        CUDA_CHECK(cudaMemcpyAsync(c.dump + (size_t)(c.K * t + k) * c.numel, c.src.x[k], (size_t)c.numel * sizeof(float),
                                   cudaMemcpyDeviceToDevice, s));
  };
  // One Langevin step is 300-1200 small launches per source at the reference's n_mixed = 30: from the second step on the
  // whole step is replayed as ONE CUDA graph whose per-step scalars live in device memory.
  BasisGraphs& bg = basis_graphs();
  static const bool no_graph = getenv("ASEP_NO_GRAPH") != nullptr;
  const bool use_graph = c.T >= 3 && allow_graph && bg.enabled && !no_graph;
  if (!use_graph) {
    for (int t = 0; t < c.T; ++t) eager_step(t);
    return;
  }
  bg.ensure();
  key.p[0] = c.mixed; key.p[1] = c.dump; key.p[2] = c.nanp;
  for (int k = 0; k < c.K; ++k) {
    key.p[3 + 3 * k] = c.src.x[k];
    key.p[4 + 3 * k] = c.src.s[k];
    key.p[5 + 3 * k] = c.src.n[k];
  }
  key.N = c.N; key.K = c.K; key.seed = c.seed; key.off = c.elem_offset; key.noise_stride = c.noise_stride;
  generations(key);
  auto it = bg.graphs.find(key);
  // a cached graph means every workspace already has this size: every step of the call is a replay.  Otherwise the
  // first step runs eagerly (it sizes the workspaces -- a capture may not allocate) and the rest replay the new graph.
  const int t_first = it != bg.graphs.end() ? 0 : 1;
  if (t_first == 1) eager_step(0);
  CUDA_CHECK(cudaEventRecord(bg.ev_in, s));
  CUDA_CHECK(cudaStreamWaitEvent(bg.stream, bg.ev_in, 0));
  LangevinDev h{c.eta, c.lambda, c.noise_scale, 0.f, c.step0 + (uint64_t)t_first, (unsigned long long)t_first};
  CUDA_CHECK(cudaMemcpyAsync(bg.dev, &h, sizeof(h), cudaMemcpyHostToDevice, bg.stream));   // pageable source: staged at once
  if (it == bg.graphs.end()) {
    generations(key);                              // the eager step may have re-carved a workspace
    if (bg.graphs.size() >= 16) bg.clear();
    cudaGraph_t graph = nullptr;
    const long long c0 = g_launch_count.load();
    CUDA_CHECK(cudaStreamBeginCapture(bg.stream, cudaStreamCaptureModeRelaxed));
    try {
      if (branches > 1) {
        CUDA_CHECK(cudaEventRecord(bg.ev_fork, bg.stream));
        for (int b = 1; b < branches; ++b) CUDA_CHECK(cudaStreamWaitEvent(bg.side[b - 1], bg.ev_fork, 0));
        score(0, bg.stream);
        for (int b = 1; b < branches; ++b) {
          score(b, bg.side[b - 1]);
          CUDA_CHECK(cudaEventRecord(bg.ev_join[b - 1], bg.side[b - 1]));
          CUDA_CHECK(cudaStreamWaitEvent(bg.stream, bg.ev_join[b - 1], 0));
        }
      } else {
        score(0, bg.stream);
      }
      launch_langevin_dev(c.K, c.src, c.mixed, c.noise_stride, c.dump, bg.dev, c.seed, c.elem_offset, c.nanp, c.numel,
                          bg.stream);
    } catch (...) {
      cudaStreamEndCapture(bg.stream, &graph);
      if (graph) cudaGraphDestroy(graph);
      throw;
    }
    CUDA_CHECK(cudaStreamEndCapture(bg.stream, &graph));
    BasisGraph g;
    g.launches = g_launch_count.load() - c0;
    g_launch_count.fetch_sub(g.launches);          // a capture launches nothing
    CUDA_CHECK(cudaGraphInstantiate(&g.exec, graph, 0));
    CUDA_CHECK(cudaGraphDestroy(graph));
    it = bg.graphs.emplace(key, g).first;
  }
  for (int t = t_first; t < c.T; ++t) {
    CUDA_CHECK(cudaGraphLaunch(it->second.exec, bg.stream));
    g_launch_count.fetch_add(it->second.launches);
  }
  CUDA_CHECK(cudaEventRecord(bg.ev_out, bg.stream));
  CUDA_CHECK(cudaStreamWaitEvent(s, bg.ev_out, 0));
}

// T steps with K Glow priors m[k] (c.src.x / n, dump and the scalars filled in by the caller)
void basis_glow_steps(BasisCall c, GlowModel* const* m, cudaStream_t s) {
  SourceGroups<GlowModel> g = group_sources(c, m);
  BasisGraphKey key{};
  key.kind = 0;
  for (int k = 0; k < c.K; ++k) key.uid[k] = m[k]->uid();
  const bool allow_graph = !nn_tc_profile_enabled() && !hbm_profile_enabled();
  run_basis_steps(c, key, (int)g.models.size(), allow_graph, s,
                  [&](int b, cudaStream_t st) {
                    for (int k : g.sources[b])                                 // run_basis_sep.py:174-175
                      g.models[b]->grad_log_prob(c.src.x[k], const_cast<float*>(c.src.s[k]), nullptr, c.N, st);
                  },
                  [&](BasisGraphKey& key) {
                    for (int k = 0; k < c.K; ++k) key.gen[k] = m[k]->generation();
                  });
}

// T steps at noise level sigma_idx with K score networks m[k]
void basis_ncsn_steps(BasisCall c, NcsnModel* const* m, int sigma_idx, cudaStream_t s) {
  SourceGroups<NcsnModel> g = group_sources(c, m);
  const int* idx = m[0]->index_scratch(c.N, sigma_idx, s);                     // run_basis_sep.py:167-168
  BasisGraphKey key{};
  key.kind = 1;
  for (int k = 0; k < c.K; ++k) key.uid[k] = m[k]->uid();
  const bool allow_graph = !conv_tc_profile_enabled() && !hbm_profile_enabled();
  run_basis_steps(c, key, (int)g.models.size(), allow_graph, s,
                  [&](int b, cudaStream_t st) {
                    for (int k : g.sources[b])                                 // run_basis_sep.py:169-170
                      g.models[b]->forward(c.src.x[k], idx, const_cast<float*>(c.src.s[k]), c.N, st);
                  },
                  [&](BasisGraphKey& key) {
                    for (int k = 0; k < c.K; ++k) key.gen[k] = m[k]->generation();
                  });
}

// Optional injected noise [T, K, ...] / per-step dump [T, K, ...] of a stacked K-source call whose state is x [K, ...].
const float* stacked_noise(const DLTensor* noise, const TView& x, int T, int dev) {
  if (!noise) return nullptr;
  TView v = view_f32(noise, "noise", dev);
  expect_stacked(v, "noise", {T}, x);
  return v.f32;
}
float* stacked_dump(DLTensor* per_step, const TView& x, int T, int dev) {
  if (!per_step) return nullptr;
  TView v = view_f32(per_step, "per_step", dev);
  expect_stacked(v, "per_step", {T}, x);
  return v.f32;
}
}  // namespace

extern "C" {

int asep_basis_glow_inner(asep_glow_t m1, asep_glow_t m2, const DLTensor* mixed, DLTensor* x1, DLTensor* x2, int T,
                          float eta, float lambda, float noise_scale, const DLTensor* noise1, const DLTensor* noise2,
                          uint64_t seed, uint64_t step0, uint64_t elem_offset, DLTensor* per_step,
                          DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(m1 && m2, ASEP_ERR_BAD_ARG, "NULL handle");
  GlowModel &g1 = *m1->model, &g2 = *m2->model;
  const int dev = g1.device();
  TView a = view_f32(x1, "x1", dev), b = view_f32(x2, "x2", dev), mx = view_f32(mixed, "mixed", dev);
  const int N = batch_of(a, g1, "x1");
  ASEP_CHECK(batch_of(b, g2, "x2") == N && mx.numel == a.numel, ASEP_ERR_BAD_SHAPE, "x1, x2, mixed must match");
  ASEP_CHECK(g2.device() == dev, ASEP_ERR_BAD_DEVICE, "the two priors live on different devices");
  ASEP_CHECK((noise1 == nullptr) == (noise2 == nullptr), ASEP_ERR_BAD_ARG, "inject both noise tensors or neither");
  BasisCall call{2, {}, a.numel, mx.f32, nullptr, nullptr, (long long)a.numel, N, T, eta, lambda, noise_scale, seed, step0,
                 elem_offset};
  call.src.x[0] = a.f32; call.src.x[1] = b.f32;
  if (noise1) {
    TView na = view_f32(noise1, "noise1", dev), nb = view_f32(noise2, "noise2", dev);
    ASEP_CHECK(na.numel == (int64_t)T * a.numel && nb.numel == na.numel, ASEP_ERR_BAD_SHAPE, "noise must be [T, ...]");
    call.src.n[0] = na.f32; call.src.n[1] = nb.f32;
  }
  if (per_step) {
    TView d = view_f32(per_step, "per_step", dev);
    ASEP_CHECK(d.numel == (int64_t)T * 2 * a.numel, ASEP_ERR_BAD_SHAPE, "per_step must be [T, 2, ...]");
    call.dump = d.f32;
  }
  if (nan_count) call.nanp = static_cast<int*>(view_i32(nan_count, "nan_count", dev).raw);
  GlowModel* const ms[2] = {&g1, &g2};
  basis_glow_steps(call, ms, as_stream(stream));
  ASEP_API_END
}

int asep_basis_glow_inner_k(int K, const asep_glow_t* m, const DLTensor* mixed, DLTensor* x, int T, float eta, float lambda,
                            float noise_scale, const DLTensor* noise, uint64_t seed, uint64_t step0, uint64_t elem_offset,
                            DLTensor* per_step, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  check_sources(K);
  ASEP_CHECK(m != nullptr && T >= 0, ASEP_ERR_BAD_ARG, "NULL model array or negative T");
  GlowModel* ms[kMaxSources];
  for (int k = 0; k < K; ++k) {
    ASEP_CHECK(m[k] != nullptr, ASEP_ERR_BAD_ARG, "NULL handle for source %d", k);
    ms[k] = m[k]->model.get();
  }
  const int dev = ms[0]->device();
  TView mx = view_f32(mixed, "mixed", dev), xv = view_f32(x, "x", dev);
  for (int k = 0; k < K; ++k) {
    batch_of(mx, *ms[k], "mixed");                  // every prior models the data shape of the mixture
    ASEP_CHECK(ms[k]->device() == dev, ASEP_ERR_BAD_DEVICE, "the priors live on different devices");
  }
  expect_stacked(xv, "x", {K}, mx);
  ASEP_CHECK(mx.numel % 4 == 0, ASEP_ERR_BAD_SHAPE, "the element count of one source (%lld) must be a multiple of 4",
             (long long)mx.numel);
  BasisCall call{K, {}, (long long)K * mx.numel, mx.f32, stacked_dump(per_step, xv, T, dev), nullptr, (long long)mx.numel,
                 (int)mx.shape[0], T, eta, lambda, noise_scale, seed, step0, elem_offset};
  const float* nz = stacked_noise(noise, xv, T, dev);
  for (int k = 0; k < K; ++k) {
    call.src.x[k] = xv.f32 + k * mx.numel;
    call.src.n[k] = nz ? nz + k * mx.numel : nullptr;
  }
  if (nan_count) call.nanp = static_cast<int*>(view_i32(nan_count, "nan_count", dev).raw);
  basis_glow_steps(call, ms, as_stream(stream));
  ASEP_API_END
}

// ------------------------------------------------------------------ NCSN
int asep_ncsn_create(const asep_ncsn_cfg* cfg, asep_ncsn_t* out) {
  ASEP_API_BEGIN
  ASEP_CHECK(cfg != nullptr && out != nullptr, ASEP_ERR_BAD_ARG, "NULL argument");
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  auto h = new asep_ncsn_s();
  try {
    h->model.reset(new NcsnModel(*cfg, g_device));
  } catch (...) {
    delete h;
    throw;
  }
  *out = h;
  ASEP_API_END
}

int asep_ncsn_destroy(asep_ncsn_t h) {
  ASEP_API_BEGIN
  if (h) {
    cudaDeviceSynchronize();
    delete h;
  }
  ASEP_API_END
}

int asep_ncsn_set_param(asep_ncsn_t h, const char* name, const DLTensor* value) {
  ASEP_API_BEGIN
  ASEP_CHECK(h && name, ASEP_ERR_BAD_ARG, "NULL argument");
  TView v = view_f32(value, name, h->model->device(), /*allow_host=*/true);
  std::vector<int64_t> shape(v.shape, v.shape + v.ndim);
  h->model->set_param(name, v.f32, shape, v.on_device);
  ASEP_API_END
}

int asep_ncsn_set_sigmas(asep_ncsn_t h, const DLTensor* sigmas) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  TView v = view_f32(sigmas, "sigmas", h->model->device(), true);
  std::vector<float> host((size_t)v.numel);
  if (v.on_device) CUDA_CHECK(cudaMemcpy(host.data(), v.f32, host.size() * sizeof(float), cudaMemcpyDeviceToHost));
  else std::memcpy(host.data(), v.f32, host.size() * sizeof(float));
  h->model->set_sigmas(host.data(), (int)host.size());
  ASEP_API_END
}

int asep_ncsn_set_precision(asep_ncsn_t h, int precision) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  ASEP_CHECK(precision == ASEP_PREC_BF16 || precision == ASEP_PREC_BF16X3, ASEP_ERR_BAD_ARG,
             "score networks run in ASEP_PREC_BF16 or ASEP_PREC_BF16X3 (got %d)", precision);
  h->model->set_precision(precision == ASEP_PREC_BF16X3);
  ASEP_API_END
}

int asep_ncsn_prepare(asep_ncsn_t h) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  h->model->prepare();
  ASEP_API_END
}

int asep_ncsn_forward(asep_ncsn_t h, const DLTensor* x, const DLTensor* sigma_idx, DLTensor* score, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  NcsnModel& m = *h->model;
  const auto& c = m.cfg();
  TView xv = view_f32(x, "x", m.device());
  expect_shape(xv, "x", {-1, c.H, c.W, c.C});
  const int N = (int)xv.shape[0];
  TView iv = view_i32(sigma_idx, "sigma_idx", m.device());
  expect_shape(iv, "sigma_idx", {N});
  TView sv = view_f32(score, "score", m.device());
  expect_shape(sv, "score", {N, c.H, c.W, c.C});
  m.forward(xv.f32, static_cast<const int*>(iv.raw), sv.f32, N, as_stream(stream));
  ASEP_API_END
}

// ---- NCSN training (train_ncsn.py:26-57)
int asep_ncsn_enable_training(asep_ncsn_t h) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  h->model->enable_training();
  ASEP_API_END
}

int asep_ncsn_num_trainable(asep_ncsn_t h, int64_t* out) {
  ASEP_API_BEGIN
  ASEP_CHECK(h && out, ASEP_ERR_BAD_ARG, "NULL argument");
  *out = (int64_t)h->model->num_trainable();
  ASEP_API_END
}

int asep_ncsn_param_span(asep_ncsn_t h, const char* name, int64_t* offset, int64_t* numel) {
  ASEP_API_BEGIN
  ASEP_CHECK(h && name, ASEP_ERR_BAD_ARG, "NULL argument");
  long long o = 0, n = 0;
  h->model->param_span(name, &o, &n);
  if (offset) *offset = (int64_t)o;
  if (numel) *numel = (int64_t)n;
  ASEP_API_END
}

int asep_ncsn_train_grads(asep_ncsn_t h, const DLTensor* x, const DLTensor* noise, const DLTensor* sigma_idx,
                          int global_batch, DLTensor* grads, DLTensor* loss, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  NcsnModel& m = *h->model;
  const auto& c = m.cfg();
  TView xv = view_f32(x, "x", m.device());
  expect_shape(xv, "x", {-1, c.H, c.W, c.C});
  const int N = (int)xv.shape[0];
  TView nv = view_f32(noise, "noise", m.device());
  expect_shape(nv, "noise", {N, c.H, c.W, c.C});
  TView iv = view_i32(sigma_idx, "sigma_idx", m.device());
  expect_shape(iv, "sigma_idx", {N});
  TView gv = view_f32(grads, "grads", m.device());
  ASEP_CHECK(gv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "grads must hold %lld elements", m.num_trainable());
  float* lp = nullptr;
  if (loss) {
    TView lv = view_f32(loss, "loss", m.device());
    ASEP_CHECK(lv.numel == 1, ASEP_ERR_BAD_SHAPE, "loss must hold one element");
    lp = lv.f32;
  }
  m.train_grads(xv.f32, nv.f32, static_cast<const int*>(iv.raw), N, global_batch, gv.f32, lp, as_stream(stream));
  ASEP_API_END
}

int asep_ncsn_adam_step(asep_ncsn_t h, const DLTensor* grads, float lr, float beta1, float beta2, float eps,
                        void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  NcsnModel& m = *h->model;
  TView gv = view_f32(grads, "grads", m.device());
  ASEP_CHECK(gv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "grads must hold %lld elements", m.num_trainable());
  m.adam_step(gv.f32, lr, beta1, beta2, eps, as_stream(stream));
  ASEP_API_END
}

int asep_ncsn_get_flat(asep_ncsn_t h, DLTensor* theta, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  NcsnModel& m = *h->model;
  TView tv = view_f32(theta, "theta", m.device());
  ASEP_CHECK(tv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "theta must hold %lld elements", m.num_trainable());
  m.copy_flat(tv.f32, as_stream(stream));
  ASEP_API_END
}

int asep_ncsn_set_flat(asep_ncsn_t h, const DLTensor* theta, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(h, ASEP_ERR_BAD_ARG, "NULL handle");
  NcsnModel& m = *h->model;
  TView tv = view_f32(theta, "theta", m.device());
  ASEP_CHECK(tv.numel == m.num_trainable(), ASEP_ERR_BAD_SHAPE, "theta must hold %lld elements", m.num_trainable());
  m.set_flat(tv.f32, as_stream(stream));
  ASEP_API_END
}

int asep_basis_ncsn_inner(asep_ncsn_t m1, asep_ncsn_t m2, const DLTensor* mixed, DLTensor* x1, DLTensor* x2,
                          int sigma_idx, int T, float eta, float lambda, float noise_scale, const DLTensor* noise1,
                          const DLTensor* noise2, uint64_t seed, uint64_t step0, uint64_t elem_offset,
                          DLTensor* per_step, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(m1 && m2, ASEP_ERR_BAD_ARG, "NULL handle");
  NcsnModel &g1 = *m1->model, &g2 = *m2->model;
  const int dev = g1.device();
  const auto& c = g1.cfg();
  TView a = view_f32(x1, "x1", dev), b = view_f32(x2, "x2", dev), mx = view_f32(mixed, "mixed", dev);
  expect_shape(a, "x1", {-1, c.H, c.W, c.C});
  const int N = (int)a.shape[0];
  expect_shape(b, "x2", {N, c.H, c.W, c.C});
  ASEP_CHECK(mx.numel == a.numel, ASEP_ERR_BAD_SHAPE, "x1, x2, mixed must match");
  const auto& c2 = g2.cfg();
  ASEP_CHECK(c2.H == c.H && c2.W == c.W && c2.C == c.C, ASEP_ERR_BAD_SHAPE,
             "the two score networks must share the data shape (%dx%dx%d vs %dx%dx%d)", c.H, c.W, c.C, c2.H, c2.W, c2.C);
  ASEP_CHECK(g2.device() == dev, ASEP_ERR_BAD_DEVICE, "the two score networks live on different devices");
  ASEP_CHECK(sigma_idx >= 0 && sigma_idx < c.num_classes && sigma_idx < c2.num_classes, ASEP_ERR_BAD_ARG,
             "sigma_idx %d out of range (num_classes %d / %d)", sigma_idx, c.num_classes, c2.num_classes);
  ASEP_CHECK((noise1 == nullptr) == (noise2 == nullptr), ASEP_ERR_BAD_ARG, "inject both noise tensors or neither");
  BasisCall call{2, {}, a.numel, mx.f32, nullptr, nullptr, (long long)a.numel, N, T, eta, lambda, noise_scale, seed, step0,
                 elem_offset};
  call.src.x[0] = a.f32; call.src.x[1] = b.f32;
  if (noise1) {
    TView na = view_f32(noise1, "noise1", dev), nb = view_f32(noise2, "noise2", dev);
    ASEP_CHECK(na.numel == (int64_t)T * a.numel && nb.numel == na.numel, ASEP_ERR_BAD_SHAPE, "noise must be [T, ...]");
    call.src.n[0] = na.f32; call.src.n[1] = nb.f32;
  }
  if (per_step) {
    TView d = view_f32(per_step, "per_step", dev);
    ASEP_CHECK(d.numel == (int64_t)T * 2 * a.numel, ASEP_ERR_BAD_SHAPE, "per_step must be [T, 2, ...]");
    call.dump = d.f32;
  }
  if (nan_count) call.nanp = static_cast<int*>(view_i32(nan_count, "nan_count", dev).raw);
  NcsnModel* const ms[2] = {&g1, &g2};
  basis_ncsn_steps(call, ms, sigma_idx, as_stream(stream));
  ASEP_API_END
}

int asep_basis_ncsn_inner_k(int K, const asep_ncsn_t* m, const DLTensor* mixed, DLTensor* x, int sigma_idx, int T, float eta,
                            float lambda, float noise_scale, const DLTensor* noise, uint64_t seed, uint64_t step0,
                            uint64_t elem_offset, DLTensor* per_step, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  check_sources(K);
  ASEP_CHECK(m != nullptr && T >= 0, ASEP_ERR_BAD_ARG, "NULL model array or negative T");
  NcsnModel* ms[kMaxSources];
  for (int k = 0; k < K; ++k) {
    ASEP_CHECK(m[k] != nullptr, ASEP_ERR_BAD_ARG, "NULL handle for source %d", k);
    ms[k] = m[k]->model.get();
  }
  const int dev = ms[0]->device();
  TView mx = view_f32(mixed, "mixed", dev), xv = view_f32(x, "x", dev);
  for (int k = 0; k < K; ++k) {
    const auto& c = ms[k]->cfg();
    expect_shape(mx, "mixed", {-1, c.H, c.W, c.C});   // every score network models the data shape of the mixture
    ASEP_CHECK(ms[k]->device() == dev, ASEP_ERR_BAD_DEVICE, "the score networks live on different devices");
    ASEP_CHECK(sigma_idx >= 0 && sigma_idx < c.num_classes, ASEP_ERR_BAD_ARG, "sigma_idx %d out of range (num_classes %d)",
               sigma_idx, c.num_classes);
  }
  expect_stacked(xv, "x", {K}, mx);
  ASEP_CHECK(mx.numel % 4 == 0, ASEP_ERR_BAD_SHAPE, "the element count of one source (%lld) must be a multiple of 4",
             (long long)mx.numel);
  BasisCall call{K, {}, (long long)K * mx.numel, mx.f32, stacked_dump(per_step, xv, T, dev), nullptr, (long long)mx.numel,
                 (int)mx.shape[0], T, eta, lambda, noise_scale, seed, step0, elem_offset};
  const float* nz = stacked_noise(noise, xv, T, dev);
  for (int k = 0; k < K; ++k) {
    call.src.x[k] = xv.f32 + k * mx.numel;
    call.src.n[k] = nz ? nz + k * mx.numel : nullptr;
  }
  if (nan_count) call.nanp = static_cast<int*>(view_i32(nan_count, "nan_count", dev).raw);
  basis_ncsn_steps(call, ms, sigma_idx, as_stream(stream));
  ASEP_API_END
}

// ------------------------------------------------------------------ whole sigma x T loops on the device
namespace {
// snapshot of the K states after noise level i into snapshots[i] = [K, N, H, W, C] (x_arr of run_basis_sep.py:243-244)
void snapshot_states(float* snap, int level, int K, float* const* x, long long numel, cudaStream_t s) {
  if (!snap) return;
  float* dst = snap + (size_t)level * K * numel;
  for (int k = 0; k < K; ++k)
    CUDA_CHECK(cudaMemcpyAsync(dst + (size_t)k * numel, x[k], (size_t)numel * sizeof(float), cudaMemcpyDeviceToDevice, s));
}

// the [L, K, ...] snapshots of a K-source run (or NULL); fills x[k] with the state of every source
float* run_snapshots(DLTensor* snapshots, const TView& xv, int K, int L, float** x, int dev) {
  for (int k = 0; k < K; ++k) x[k] = xv.f32 + k * (xv.numel / K);
  if (!snapshots) return nullptr;
  TView sv = view_f32(snapshots, "snapshots", dev);
  ASEP_CHECK(sv.ndim == xv.ndim + 1 && sv.shape[0] == L && sv.numel == (int64_t)L * xv.numel, ASEP_ERR_BAD_SHAPE,
             "snapshots must be [L, K, N, H, W, C]");
  for (int j = 0; j < xv.ndim; ++j)
    ASEP_CHECK(sv.shape[j + 1] == xv.shape[j], ASEP_ERR_BAD_SHAPE, "snapshots must be [L, K, N, H, W, C]");
  return sv.f32;
}
}  // namespace

int asep_basis_glow_run(const asep_glow_t* m1, const asep_glow_t* m2, int n_models, const DLTensor* mixed, DLTensor* x1,
                        DLTensor* x2, int L, int T, const float* eta, const float* lambda, const float* noise_scale,
                        uint64_t seed, uint64_t elem_offset, DLTensor* snapshots, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(m1 && m2 && eta && lambda && noise_scale, ASEP_ERR_BAD_ARG, "NULL argument");
  ASEP_CHECK(L >= 1 && T >= 0 && (n_models == 1 || n_models == L), ASEP_ERR_BAD_ARG,
             "n_models must be 1 (one pair of priors for every level) or L (one pair per level)");
  ASEP_CHECK(m1[0] && m2[0], ASEP_ERR_BAD_ARG, "NULL handle");
  const int dev = m1[0]->model->device();
  TView a = view_f32(x1, "x1", dev), b = view_f32(x2, "x2", dev);
  float* snap = nullptr;
  if (snapshots) {
    TView sv = view_f32(snapshots, "snapshots", dev);
    ASEP_CHECK(sv.numel == (int64_t)L * 2 * a.numel, ASEP_ERR_BAD_SHAPE, "snapshots must be [L, 2, N, H, W, C]");
    snap = sv.f32;
  }
  float* const xs[2] = {a.f32, b.f32};
  for (int i = 0; i < L; ++i) {
    const int k = n_models == 1 ? 0 : i;
    ASEP_CHECK(m1[k] && m2[k], ASEP_ERR_BAD_ARG, "NULL handle at level %d", i);
    const int rc = asep_basis_glow_inner(m1[k], m2[k], mixed, x1, x2, T, eta[i], lambda[i], noise_scale[i], nullptr, nullptr, seed,
                                         (uint64_t)i * (uint64_t)T, elem_offset, nullptr, nan_count, stream);
    if (rc != ASEP_OK) return rc;                      // asep_last_error() holds the inner message
    snapshot_states(snap, i, 2, xs, a.numel, as_stream(stream));
  }
  ASEP_API_END
}

int asep_basis_glow_run_k(int K, const asep_glow_t* m, int n_models, const DLTensor* mixed, DLTensor* x, int L, int T,
                          const float* eta, const float* lambda, const float* noise_scale, uint64_t seed, uint64_t elem_offset,
                          DLTensor* snapshots, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  check_sources(K);
  ASEP_CHECK(m && eta && lambda && noise_scale, ASEP_ERR_BAD_ARG, "NULL argument");
  ASEP_CHECK(L >= 1 && T >= 0 && (n_models == 1 || n_models == L), ASEP_ERR_BAD_ARG,
             "n_models must be 1 (one set of K priors for every level) or L (one set per level)");
  for (int i = 0; i < n_models * K; ++i) ASEP_CHECK(m[i], ASEP_ERR_BAD_ARG, "NULL handle at level %d, source %d", i / K, i % K);
  const int dev = m[0]->model->device();
  TView xv = view_f32(x, "x", dev);
  ASEP_CHECK(xv.ndim >= 1 && xv.shape[0] == K, ASEP_ERR_BAD_SHAPE, "x must be [K = %d, N, H, W, C]", K);
  float* xs[kMaxSources];
  float* snap = run_snapshots(snapshots, xv, K, L, xs, dev);
  for (int i = 0; i < L; ++i) {
    const int rc = asep_basis_glow_inner_k(K, m + (size_t)(n_models == 1 ? 0 : i) * K, mixed, x, T, eta[i], lambda[i],
                                           noise_scale[i], nullptr, seed, (uint64_t)i * (uint64_t)T, elem_offset, nullptr,
                                           nan_count, stream);
    if (rc != ASEP_OK) return rc;
    snapshot_states(snap, i, K, xs, xv.numel / K, as_stream(stream));
  }
  ASEP_API_END
}

int asep_basis_ncsn_run(asep_ncsn_t m1, asep_ncsn_t m2, const DLTensor* mixed, DLTensor* x1, DLTensor* x2, int L, int T,
                        const float* eta, const float* lambda, const float* noise_scale, uint64_t seed, uint64_t elem_offset,
                        DLTensor* snapshots, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(m1 && m2 && eta && lambda && noise_scale, ASEP_ERR_BAD_ARG, "NULL argument");
  ASEP_CHECK(L >= 1 && T >= 0, ASEP_ERR_BAD_ARG, "bad L / T");
  const int dev = m1->model->device();
  TView a = view_f32(x1, "x1", dev), b = view_f32(x2, "x2", dev);
  float* snap = nullptr;
  if (snapshots) {
    TView sv = view_f32(snapshots, "snapshots", dev);
    ASEP_CHECK(sv.numel == (int64_t)L * 2 * a.numel, ASEP_ERR_BAD_SHAPE, "snapshots must be [L, 2, N, H, W, C]");
    snap = sv.f32;
  }
  float* const xs[2] = {a.f32, b.f32};
  for (int i = 0; i < L; ++i) {
    const int rc = asep_basis_ncsn_inner(m1, m2, mixed, x1, x2, i, T, eta[i], lambda[i], noise_scale[i], nullptr, nullptr, seed,
                                         (uint64_t)i * (uint64_t)T, elem_offset, nullptr, nan_count, stream);
    if (rc != ASEP_OK) return rc;
    snapshot_states(snap, i, 2, xs, a.numel, as_stream(stream));
  }
  ASEP_API_END
}

int asep_basis_ncsn_run_k(int K, const asep_ncsn_t* m, const DLTensor* mixed, DLTensor* x, int L, int T, const float* eta,
                          const float* lambda, const float* noise_scale, uint64_t seed, uint64_t elem_offset,
                          DLTensor* snapshots, DLTensor* nan_count, void* stream) {
  ASEP_API_BEGIN
  check_sources(K);
  ASEP_CHECK(m && eta && lambda && noise_scale, ASEP_ERR_BAD_ARG, "NULL argument");
  ASEP_CHECK(L >= 1 && T >= 0, ASEP_ERR_BAD_ARG, "bad L / T");
  for (int k = 0; k < K; ++k) ASEP_CHECK(m[k], ASEP_ERR_BAD_ARG, "NULL handle for source %d", k);
  const int dev = m[0]->model->device();
  TView xv = view_f32(x, "x", dev);
  ASEP_CHECK(xv.ndim >= 1 && xv.shape[0] == K, ASEP_ERR_BAD_SHAPE, "x must be [K = %d, N, H, W, C]", K);
  float* xs[kMaxSources];
  float* snap = run_snapshots(snapshots, xv, K, L, xs, dev);
  for (int i = 0; i < L; ++i) {
    const int rc = asep_basis_ncsn_inner_k(K, m, mixed, x, i, T, eta[i], lambda[i], noise_scale[i], nullptr, seed,
                                           (uint64_t)i * (uint64_t)T, elem_offset, nullptr, nan_count, stream);
    if (rc != ASEP_OK) return rc;
    snapshot_states(snap, i, K, xs, xv.numel / K, as_stream(stream));
  }
  ASEP_API_END
}

int asep_conv_profile(int on) {
  ASEP_API_BEGIN
  conv_tc_profile(on);
  ASEP_API_END
}

int asep_conv_profile_read(double* total_ms, int64_t* launches, double* flops) {
  ASEP_API_BEGIN
  long long n = 0;
  conv_tc_profile_read(total_ms, &n, flops);
  if (launches) *launches = (int64_t)n;
  ASEP_API_END
}

// ---- the tcgen05 convolutions one launch at a time (tests/test_gpu_conv_tc.py): thin wrappers over conv_tc_prepare /
// launch_build_conv_image, conv_tc_forward and conv_wgrad_tc that check every shape before anything is launched
static TView view_bf16(const DLTensor* t, const char* what) { return view_any(t, what, g_device, false, kDLBfloat, 16); }

static void expect_numel(const TView& v, const char* what, int64_t n) {
  ASEP_CHECK(v.numel == n, ASEP_ERR_BAD_SHAPE, "%s: %lld elements, expected %lld", what, (long long)v.numel, (long long)n);
}

int asep_conv_tc_image(const DLTensor* kernel, int transposed, int lo, int on_device, DLTensor* img, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  ASEP_CHECK((transposed == 0 || transposed == 1) && (lo == 0 || lo == 1) && (on_device == 0 || on_device == 1),
             ASEP_ERR_BAD_ARG, "transposed, lo and on_device are 0 or 1");
  ASEP_CHECK(on_device || (!transposed && !lo), ASEP_ERR_BAD_ARG, "the host builder makes the forward hi image only");
  TView kv = view_f32(kernel, "kernel", g_device, /*allow_host=*/!on_device);
  ASEP_CHECK(kv.ndim == 4 && kv.shape[0] == kv.shape[1] && (kv.shape[0] == 1 || kv.shape[0] == 3), ASEP_ERR_BAD_SHAPE,
             "kernel: expected HWIO [k,k,Cin,Cout] with k = 1 or 3");
  const int ksize = (int)kv.shape[0], Cin = (int)kv.shape[2], Cout = (int)kv.shape[3];
  // the contraction extent of the image (Cin, or Cout for the transposed image) is walked in 64-channel panels
  ASEP_CHECK(Cin > 0 && Cout > 0 && (transposed ? Cout : Cin) % 64 == 0, ASEP_ERR_UNSUPPORTED,
             "conv image: Cin=%d Cout=%d, the contraction extent must be a multiple of 64", Cin, Cout);
  TView iv = view_bf16(img, "img");
  expect_numel(iv, "img", kv.numel);
  __nv_bfloat16* dst = static_cast<__nv_bfloat16*>(iv.raw);
  if (on_device) {
    launch_build_conv_image(kv.f32, dst, ksize * ksize, Cin, Cout, transposed, lo, as_stream(stream));
  } else {
    std::vector<float> host((size_t)kv.numel);
    if (kv.on_device) CUDA_CHECK(cudaMemcpy(host.data(), kv.f32, host.size() * sizeof(float), cudaMemcpyDeviceToHost));
    else std::memcpy(host.data(), kv.f32, host.size() * sizeof(float));
    ConvWeightsTC w;
    conv_tc_prepare(w, host.data(), nullptr, ksize, Cin, Cout, 1);
    cudaError_t e = cudaMemcpy(dst, w.img, w.bytes, cudaMemcpyDeviceToDevice);
    conv_tc_release(w);
    CUDA_CHECK(e);
  }
  ASEP_API_END
}

int asep_conv_tc_forward(const DLTensor* img, const DLTensor* bias, int ksize, int Cin, int Cout, int dil, const DLTensor* x,
                         const DLTensor* add, const DLTensor* add2, DLTensor* out, DLTensor* stats, DLTensor* out_bf16,
                         void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  ASEP_CHECK((ksize == 1 || ksize == 3) && dil >= 1, ASEP_ERR_UNSUPPORTED, "conv: kernel size %d (1 or 3), dilation %d",
             ksize, dil);
  TView xv = view_bf16(x, "x");
  ASEP_CHECK(xv.ndim == 4, ASEP_ERR_BAD_SHAPE, "x: expected NHWC [N,H,W,Cin]");
  expect_shape(xv, "x", {-1, -1, -1, Cin});
  const int N = (int)xv.shape[0], H = (int)xv.shape[1], W = (int)xv.shape[2];
  ASEP_CHECK(conv_tc_supported(Cin, Cout, H, W), ASEP_ERR_UNSUPPORTED,
             "tcgen05 conv: unsupported shape Cin=%d Cout=%d H=%d W=%d", Cin, Cout, H, W);
  TView iv = view_bf16(img, "img");
  expect_numel(iv, "img", (int64_t)ksize * ksize * Cin * Cout);
  TView ov = view_f32(out, "out", g_device);
  expect_shape(ov, "out", {N, H, W, Cout});
  const float* addp[2] = {nullptr, nullptr};
  const DLTensor* adds[2] = {add, add2};
  for (int i = 0; i < 2; ++i)
    if (adds[i]) {
      TView av = view_f32(adds[i], i ? "add2" : "add", g_device);
      expect_shape(av, i ? "add2" : "add", {N, H, W, Cout});
      addp[i] = av.f32;
    }
  ConvWeightsTC w;                 // borrows the caller's image and bias: never conv_tc_release'd
  w.img = static_cast<__nv_bfloat16*>(iv.raw);
  w.bias_owned = false;
  if (bias) {
    TView bv = view_f32(bias, "bias", g_device);
    expect_shape(bv, "bias", {Cout});
    w.bias = bv.f32;
  }
  w.Cin = Cin; w.Cout = Cout; w.ksize = ksize; w.dil = dil;
  w.bytes = (size_t)iv.numel * sizeof(__nv_bfloat16);
  double* st = nullptr;
  if (stats) {
    TView sv = view_any(stats, "stats", g_device, false, kDLFloat, 64);
    expect_shape(sv, "stats", {N, Cout, 2});
    st = static_cast<double*>(sv.raw);
  }
  __nv_bfloat16* ob = nullptr;
  if (out_bf16) {
    TView bv = view_bf16(out_bf16, "out_bf16");
    expect_shape(bv, "out_bf16", {N, H, W, Cout});
    ob = static_cast<__nv_bfloat16*>(bv.raw);
  }
  conv_tc_forward(w, static_cast<const __nv_bfloat16*>(xv.raw), addp[0], ov.f32, N, H, W, as_stream(stream), st, ob, addp[1]);
  ASEP_API_END
}

int asep_conv_wgrad_tc(const DLTensor* x, const DLTensor* g, DLTensor* dk, int ksize, int dil, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  ASEP_CHECK((ksize == 1 || ksize == 3) && dil >= 1, ASEP_ERR_UNSUPPORTED, "conv wgrad: kernel size %d (1 or 3), dilation %d",
             ksize, dil);
  TView xv = view_bf16(x, "x");
  ASEP_CHECK(xv.ndim == 4, ASEP_ERR_BAD_SHAPE, "x: expected NHWC [N,H,W,Cin]");
  const int N = (int)xv.shape[0], H = (int)xv.shape[1], W = (int)xv.shape[2], Cin = (int)xv.shape[3];
  TView gv = view_bf16(g, "g");
  ASEP_CHECK(gv.ndim == 4, ASEP_ERR_BAD_SHAPE, "g: expected NHWC [N,H,W,Cout]");
  expect_shape(gv, "g", {N, H, W, -1});
  const int Cout = (int)gv.shape[3];
  TView kv = view_f32(dk, "dk", g_device);
  expect_shape(kv, "dk", {ksize, ksize, Cin, Cout});
  ASEP_CHECK(conv_wgrad_tc_supported(Cin, Cout, H, W), ASEP_ERR_UNSUPPORTED,
             "conv_wgrad_tc: unsupported shape Cin=%d Cout=%d H=%d W=%d", Cin, Cout, H, W);
  conv_wgrad_tc(static_cast<const __nv_bfloat16*>(xv.raw), static_cast<const __nv_bfloat16*>(gv.raw), kv.f32, N, H, W, Cin,
                Cout, ksize, dil, as_stream(stream));
  ASEP_API_END
}

// CRC-32C (Castagnoli), slicing-by-8, host only: checksums of the TensorFlow checkpoint interchange
// (audiosourcesep_b200/tf_checkpoint.py; the TensorBundle format stores a masked crc32c per tensor and per index block).
uint32_t asep_crc32c(const void* data, uint64_t n, uint32_t crc) {
  static uint32_t tab[8][256];
  static bool init = false;
  if (!init) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
      tab[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int t = 1; t < 8; ++t) tab[t][i] = (tab[t - 1][i] >> 8) ^ tab[0][tab[t - 1][i] & 0xFFu];
    init = true;
  }
  const uint8_t* p = static_cast<const uint8_t*>(data);
  uint32_t c = crc ^ 0xFFFFFFFFu;
  while (n >= 8) {
    uint32_t lo, hi;
    std::memcpy(&lo, p, 4);
    std::memcpy(&hi, p + 4, 4);
    lo ^= c;
    c = tab[7][lo & 0xFFu] ^ tab[6][(lo >> 8) & 0xFFu] ^ tab[5][(lo >> 16) & 0xFFu] ^ tab[4][lo >> 24] ^
        tab[3][hi & 0xFFu] ^ tab[2][(hi >> 8) & 0xFFu] ^ tab[1][(hi >> 16) & 0xFFu] ^ tab[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n--) c = tab[0][(c ^ *p++) & 0xFFu] ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}

int asep_basis_graphs(int on) {
  ASEP_API_BEGIN
  basis_graphs().enabled = on != 0;
  if (!on) basis_graphs().clear();
  ASEP_API_END
}

// ------------------------------------------------------------------ evaluation on the device (bsseval.cu)
int asep_bss_eval(const DLTensor* reference_sources, const DLTensor* estimated_sources, int filters_len, int64_t filt_start,
                  int64_t filt_stop, const int64_t* win_start, const int64_t* win_stop, int nwin, int sources_version,
                  DLTensor* out, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  ASEP_CHECK(win_start && win_stop && nwin >= 1, ASEP_ERR_BAD_ARG, "bss_eval: no evaluation window");
  TView r = view_any(reference_sources, "reference_sources", g_device, false, kDLFloat, 64);
  TView e = view_any(estimated_sources, "estimated_sources", g_device, false, kDLFloat, 64);
  ASEP_CHECK(r.ndim == 2 && e.ndim == 2 && r.shape[0] == e.shape[0] && r.shape[1] == e.shape[1], ASEP_ERR_BAD_SHAPE,
             "bss_eval: reference_sources and estimated_sources must both be [nsrc, nsampl] (mono images)");
  const int nsrc = (int)r.shape[0];
  TView o = view_any(out, "out", g_device, false, kDLFloat, 64);
  ASEP_CHECK(o.numel == (int64_t)4 * nsrc * nsrc * nwin, ASEP_ERR_BAD_SHAPE, "bss_eval: out must be [4, nsrc, nsrc, nwin] float64");
  std::vector<long long> w0(win_start, win_start + nwin), w1(win_stop, win_stop + nwin);
  bss_eval_core(static_cast<const double*>(r.raw), static_cast<const double*>(e.raw), nsrc, (long long)r.shape[1], filters_len,
                (long long)filt_start, (long long)filt_stop, w0.data(), w1.data(), nwin, sources_version,
                static_cast<double*>(o.raw), as_stream(stream));
  ASEP_API_END
}

int asep_ideal_mask(const DLTensor* mixture, const DLTensor* sources, DLTensor* estimates, int binary, float theta, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView m = view_f32(mixture, "mixture", g_device), sv = view_f32(sources, "sources", g_device);
  TView ev = view_f32(estimates, "estimates", g_device);
  ASEP_CHECK(sv.ndim == m.ndim + 1 && sv.numel == sv.shape[0] * m.numel && ev.numel == sv.numel, ASEP_ERR_BAD_SHAPE,
             "ideal mask: sources / estimates must be [nsrc, *mixture.shape]");
  launch_ideal_mask(m.f32, sv.f32, ev.f32, (int)sv.shape[0], (long long)m.numel, binary, theta, as_stream(stream));
  ASEP_API_END
}

// ------------------------------------------------------------------ mel front end / back end (mel_kernels.cu)
int asep_stft(const DLTensor* audio, int n_fft, int hop, DLTensor* stft, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView a = view_f32(audio, "audio", g_device), o = view_f32(stft, "stft", g_device);
  ASEP_CHECK(a.ndim == 2, ASEP_ERR_BAD_SHAPE, "audio must be [N, L]");
  const int N = (int)a.shape[0];
  const long long L = a.shape[1];
  ASEP_CHECK(hop >= 1, ASEP_ERR_BAD_ARG, "hop must be positive");
  expect_shape(o, "stft", {N, n_fft / 2 + 1, 1 + L / hop, 2});
  launch_stft(a.f32, o.f32, N, L, n_fft, hop, as_stream(stream));
  ASEP_API_END
}

int asep_mel_db(const DLTensor* stft, const DLTensor* basis, const DLTensor* lo, const DLTensor* hi, DLTensor* mel_db, float amin,
                float top_db, float dbmin, float dbmax, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView sv = view_f32(stft, "stft", g_device), b = view_f32(basis, "basis", g_device), o = view_f32(mel_db, "mel_db", g_device);
  ASEP_CHECK(sv.ndim == 4 && sv.shape[3] == 2 && b.ndim == 2 && b.shape[1] == sv.shape[1], ASEP_ERR_BAD_SHAPE,
             "stft must be [N, F, T, 2] and basis [M, F]");
  const int N = (int)sv.shape[0], F = (int)sv.shape[1], T = (int)sv.shape[2], M = (int)b.shape[0];
  TView l = view_i32(lo, "lo", g_device), h = view_i32(hi, "hi", g_device);
  expect_shape(l, "lo", {M});
  expect_shape(h, "hi", {M});
  expect_shape(o, "mel_db", {N, M, T});
  launch_mel_db(sv.f32, b.f32, static_cast<const int*>(l.raw), static_cast<const int*>(h.raw), o.f32, N, M, F, T, amin, top_db, dbmin,
                dbmax, as_stream(stream));
  ASEP_API_END
}

int asep_mel_to_stft(const DLTensor* mel_db, const DLTensor* basis, const DLTensor* pinv, const DLTensor* flo, const DLTensor* fhi,
                     DLTensor* mag, float step, int iters, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView mv = view_f32(mel_db, "mel_db", g_device), b = view_f32(basis, "basis", g_device), p = view_f32(pinv, "pinv", g_device);
  TView o = view_f32(mag, "mag", g_device);
  ASEP_CHECK(mv.ndim == 3 && b.ndim == 2 && b.shape[0] == mv.shape[1], ASEP_ERR_BAD_SHAPE, "mel_db must be [N, M, T] and basis [M, F]");
  const int N = (int)mv.shape[0], M = (int)mv.shape[1], T = (int)mv.shape[2], F = (int)b.shape[1];
  expect_shape(p, "pinv", {F, M});
  TView l = view_i32(flo, "flo", g_device), h = view_i32(fhi, "fhi", g_device);
  expect_shape(l, "flo", {F});
  expect_shape(h, "fhi", {F});
  expect_shape(o, "mag", {N, F, T});
  ASEP_CHECK(iters >= 0 && step > 0.f, ASEP_ERR_BAD_ARG, "mel_to_stft: iters >= 0 and step > 0");
  launch_mel_to_stft(mv.f32, b.f32, p.f32, static_cast<const int*>(l.raw), static_cast<const int*>(h.raw), o.f32, N, M, F, T, step, iters,
                     as_stream(stream));
  ASEP_API_END
}

int asep_stft_filter(const DLTensor* mag, const DLTensor* stft_mixture, DLTensor* out, int wiener, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView m = view_f32(mag, "mag", g_device), x = view_f32(stft_mixture, "stft_mixture", g_device), o = view_f32(out, "out", g_device);
  ASEP_CHECK(m.ndim == 4 && x.ndim == 4 && x.shape[3] == 2 && m.numel == m.shape[0] * (x.numel / 2) && o.numel == 2 * m.numel,
             ASEP_ERR_BAD_SHAPE, "mag [S, N, F, T], stft_mixture [N, F, T, 2], out [S, N, F, T, 2]");
  launch_stft_filter(m.f32, x.f32, o.f32, (int)m.shape[0], (long long)(x.numel / 2), wiener, as_stream(stream));
  ASEP_API_END
}

int asep_griffinlim_update(const DLTensor* mag, const DLTensor* rebuilt, DLTensor* tprev, DLTensor* next, float momentum,
                           void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView m = view_f32(mag, "mag", g_device), r = view_f32(rebuilt, "rebuilt", g_device), t = view_f32(tprev, "tprev", g_device);
  TView x = view_f32(next, "next", g_device);
  ASEP_CHECK(r.numel == 2 * m.numel && t.numel == r.numel && x.numel == r.numel, ASEP_ERR_BAD_SHAPE,
             "griffinlim: mag [...], rebuilt / tprev / next [..., 2]");
  launch_griffinlim_update(m.f32, r.f32, t.f32, x.f32, momentum, (long long)m.numel, as_stream(stream));
  ASEP_API_END
}

int asep_istft(const DLTensor* stft, int hop, DLTensor* audio, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView sv = view_f32(stft, "stft", g_device), a = view_f32(audio, "audio", g_device);
  ASEP_CHECK(sv.ndim == 4 && sv.shape[3] == 2 && sv.shape[1] >= 2, ASEP_ERR_BAD_SHAPE, "stft must be [N, F, T, 2]");
  const int N = (int)sv.shape[0], F = (int)sv.shape[1], T = (int)sv.shape[2], n_fft = 2 * (F - 1);
  ASEP_CHECK(hop >= 1, ASEP_ERR_BAD_ARG, "hop must be positive");
  expect_shape(a, "audio", {N, (int64_t)hop * (T - 1)});
  cudaStream_t s = as_stream(stream);
  float* frames = nullptr;
  CUDA_CHECK(cudaMallocAsync(&frames, (size_t)N * T * n_fft * sizeof(float), s));
  try {
    launch_istft(sv.f32, frames, a.f32, N, n_fft, hop, T, s);
  } catch (...) {
    cudaFreeAsync(frames, s);
    throw;
  }
  CUDA_CHECK(cudaFreeAsync(frames, s));
  ASEP_API_END
}

int asep_istft_track(const DLTensor* stft, int hop, int overlap_frames, DLTensor* audio, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView sv = view_f32(stft, "stft", g_device), a = view_f32(audio, "audio", g_device);
  ASEP_CHECK(sv.ndim == 5 && sv.shape[4] == 2 && sv.shape[2] >= 2 && sv.shape[3] >= 2, ASEP_ERR_BAD_SHAPE,
             "stft must be [S, n_seg, F, T, 2]");
  ASEP_CHECK(a.ndim == 2 && a.shape[0] == sv.shape[0] && a.shape[1] >= 1, ASEP_ERR_BAD_SHAPE, "audio must be [S, length]");
  const int S = (int)sv.shape[0], n_seg = (int)sv.shape[1], F = (int)sv.shape[2], T = (int)sv.shape[3], n_fft = 2 * (F - 1);
  ASEP_CHECK(n_seg >= 1, ASEP_ERR_BAD_SHAPE, "istft_track: no segments");
  ASEP_CHECK(hop >= 1, ASEP_ERR_BAD_ARG, "hop must be positive");
  // at most two segments may cover a sample: 2 overlap < V = hop (T - 1); for T = 64 frames, 0 <= overlap_frames <= 31
  ASEP_CHECK(overlap_frames >= 0 && 2 * overlap_frames < T - 1, ASEP_ERR_BAD_ARG,
             "istft_track: overlap_frames = %d outside 0..%d for segments of %d frames", overlap_frames, (T - 2) / 2, T);
  const long long V = (long long)hop * (T - 1), O = (long long)hop * overlap_frames, P = V - O;
  const long long length = a.shape[1], span = (long long)(n_seg - 1) * P + V;
  ASEP_CHECK(length <= span, ASEP_ERR_BAD_ARG, "istft_track: %lld samples, but %d segments reconstruct only %lld", length, n_seg,
             span);
  ASEP_CHECK((long long)S * n_seg <= 65535, ASEP_ERR_UNSUPPORTED, "istft_track: %d x %d segments are beyond one launch", S,
             n_seg);
  cudaStream_t s = as_stream(stream);
  float* frames = nullptr;
  CUDA_CHECK(cudaMallocAsync(&frames, (size_t)S * n_seg * T * n_fft * sizeof(float), s));
  try {
    launch_istft_track(sv.f32, frames, a.f32, S, n_seg, n_fft, hop, T, (int)O, length, s);
  } catch (...) {
    cudaFreeAsync(frames, s);
    throw;
  }
  CUDA_CHECK(cudaFreeAsync(frames, s));
  ASEP_API_END
}

// ------------------------------------------------------------------ resampling (resample_kernels.cu)
int asep_resample(const DLTensor* audio, const DLTensor* time, const DLTensor* win, const DLTensor* delta, double scale, int step,
                  DLTensor* out, void* stream) {
  ASEP_API_BEGIN
  ASEP_CHECK(g_device >= 0, ASEP_ERR_STATE, "asep_init() has not been called");
  TView a = view_f32(audio, "audio", g_device), o = view_f32(out, "out", g_device);
  TView tv = view_any(time, "time", g_device, false, kDLFloat, 64);
  TView w = view_f32(win, "win", g_device), d = view_f32(delta, "delta", g_device);
  ASEP_CHECK(a.ndim == 2, ASEP_ERR_BAD_SHAPE, "audio must be [N, L_in]");
  ASEP_CHECK(tv.ndim == 1, ASEP_ERR_BAD_SHAPE, "time must be [L_out]");
  ASEP_CHECK(w.ndim == 1 && w.numel >= 1, ASEP_ERR_BAD_SHAPE, "win must be a non-empty [nwin]");
  expect_shape(d, "delta", {w.numel});
  expect_shape(o, "out", {a.shape[0], tv.numel});
  ASEP_CHECK(step >= 1, ASEP_ERR_BAD_ARG, "step must be >= 1 (got %d)", step);
  ASEP_CHECK(scale > 0.0 && scale <= 1.0, ASEP_ERR_BAD_ARG, "scale must be in (0, 1] (got %g)", scale);
  ASEP_CHECK(w.numel <= INT32_MAX && a.shape[0] <= INT32_MAX, ASEP_ERR_UNSUPPORTED, "resample: table or batch too large");
  launch_resample(a.f32, static_cast<const double*>(tv.raw), w.f32, d.f32, o.f32, (int)a.shape[0], (long long)a.shape[1],
                  (long long)tv.numel, (int)w.numel, scale, step, as_stream(stream));
  ASEP_API_END
}

int asep_hbm_profile(int on) {
  ASEP_API_BEGIN
  hbm_profile(on != 0);
  ASEP_API_END
}

int asep_hbm_profile_read(int category, double* total_ms, int64_t* launches, double* bytes) {
  ASEP_API_BEGIN
  ASEP_CHECK(category >= 0 && category < kHbmCatCount, ASEP_ERR_BAD_ARG, "unknown kernel category %d", category);
  long long n = 0;
  hbm_profile_read(category, total_ms, &n, bytes);
  if (launches) *launches = (int64_t)n;
  ASEP_API_END
}

int asep_tc_profile(int on) {
  ASEP_API_BEGIN
  nn_tc_profile(on);
  ASEP_API_END
}

int asep_tc_profile_read(double* total_ms, int64_t* launches, double* flops) {
  ASEP_API_BEGIN
  long long n = 0;
  nn_tc_profile_read(total_ms, &n, flops);
  if (launches) *launches = (int64_t)n;
  ASEP_API_END
}

}  // extern "C"
