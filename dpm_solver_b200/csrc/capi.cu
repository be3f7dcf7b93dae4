// capi.cu -- the C-ABI of libdpmsolver_b200.so (see include/dpm_solver_b200.h)
#include <atomic>
#include <mutex>
#include <set>
#include <utility>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "launch.cuh"

namespace dpm {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_variant{2}, g_threads{0}, g_ctas{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("DPM_PDL"); return !(e && e[0] == '0'); }();
  return on;
}

int sm_count() {
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cache[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0)
      v = 148;
    cache[dev] = v;
  }
  return cache[dev];
}
int max_smem_optin() {
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 227 * 1024;
  if (cache[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
        v <= 0)
      v = 227 * 1024;
    cache[dev] = v;
  }
  return cache[dev];
}

int ensure_max_smem(const void* kernel, bool nonportable_cluster) {
  static std::mutex mu;
  static std::set<std::pair<int, const void*>> done;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  if (done.count({dev, kernel})) return 0;
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
  const int room = max_smem_optin() - (e == cudaSuccess ? (int)fa.sharedSizeBytes : 0);   // static smem counts too
  if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, room);
  if (e == cudaSuccess && nonportable_cluster)
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e != cudaSuccess) {
    set_error("shared-memory opt-in failed: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return (int)e;
  }
  done.insert({dev, kernel});
  return 0;
}

static inline int esize(int dt) { return dt == DPM_F32 ? 4 : 2; }
static inline bool valid_dtype(int dt) { return dt == DPM_F32 || dt == DPM_BF16 || dt == DPM_F16; }
static inline bool aligned(const void* p, int dt) {
  const uintptr_t a = dt == DPM_F32 ? 32 : 16;
  return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0;
}
static inline const void* off(const void* p, int dt, uint64_t elems) {
  return p ? static_cast<const char*>(p) + elems * esize(dt) : nullptr;
}
static inline void* off(void* p, int dt, uint64_t elems) {
  return p ? static_cast<char*>(p) + elems * esize(dt) : nullptr;
}

struct Needs {
  bool x, m0, m1, m2, ec, eu, xe;
};

// validate a descriptor and translate it into the kernel parameter block
static int build_params(const dpm_step_desc* d, KParams* kp, Needs* nd, bool for_quantile) {
  if (d == nullptr) { set_error("desc is NULL"); return DPM_ERR_ARG; }
  if (!valid_dtype(d->state_dtype) || !valid_dtype(d->model_dtype)) {
    set_error("bad dtype (state %d, model %d)", d->state_dtype, d->model_dtype);
    return DPM_ERR_ARG;
  }
  const int form = for_quantile ? DPM_FORM_NONE : d->form;
  if (form < DPM_FORM_NONE || form > DPM_FORM_SS3T) { set_error("bad form %d", form); return DPM_ERR_ARG; }
  if (d->n_model < 0 || d->n_model > 2) { set_error("n_model must be 0, 1 or 2"); return DPM_ERR_ARG; }
  if (d->param < DPM_PARAM_NOISE || d->param > DPM_PARAM_SCORE) { set_error("bad param %d", d->param); return DPM_ERR_ARG; }
  if (d->raw_round != 0 && ((d->raw_round & ~7) != 0 || ((d->raw_round & 3) != DPM_BF16 && (d->raw_round & 3) != DPM_F16))) {
    set_error("raw_round must be 0 or (DPM_BF16 | DPM_F16) [+ 4]");
    return DPM_ERR_ARG;
  }
  if (d->raw_round != 0 && (d->state_dtype != DPM_F32 || for_quantile)) {
    set_error("raw_round needs an fp32 state and is not available in dpm_dynamic_threshold");
    return DPM_ERR_ARG;
  }
  if ((d->n >> 3) > 0xffffffffull) { set_error("n too large (max 2^35-1 elements per call)"); return DPM_ERR_ARG; }

  nd->x = form != DPM_FORM_NONE;
  nd->m0 = d->n_model == 0;
  nd->m1 = form == DPM_FORM_LIN2 || form == DPM_FORM_LIN3 || form == DPM_FORM_DIFF2 ||
           form == DPM_FORM_MS3 || form == DPM_FORM_SS3T;
  nd->m2 = form == DPM_FORM_LIN3 || form == DPM_FORM_MS3 || form == DPM_FORM_SS3T;
  nd->ec = d->n_model >= 1;
  nd->eu = d->n_model == 2;
  nd->xe = d->n_model >= 1 && (d->param == DPM_PARAM_X_START || d->param == DPM_PARAM_V || d->predict_x0);

  if (for_quantile) {
    if (d->n_model < 1 || !d->predict_x0) { set_error("dynamic threshold needs n_model >= 1 and predict_x0"); return DPM_ERR_ARG; }
  } else {
    if (form == DPM_FORM_NONE && (d->n_model == 0 || d->m_out == nullptr)) {
      set_error("form NONE needs n_model >= 1 and m_out");
      return DPM_ERR_ARG;
    }
    if (form != DPM_FORM_NONE && d->out == nullptr) { set_error("out is NULL"); return DPM_ERR_ARG; }
  }
  const void* xe = d->xe ? d->xe : d->x;
  if ((nd->x && !d->x) || (nd->m0 && !d->m0) || (nd->m1 && !d->m1) || (nd->m2 && !d->m2) ||
      (nd->ec && !d->e_cond) || (nd->eu && !d->e_uncond) || (nd->xe && !xe)) {
    set_error("a tensor required by form %d / n_model %d is NULL", form, d->n_model);
    return DPM_ERR_ARG;
  }
  if (d->thr != nullptr || for_quantile) {
    if (d->per_sample == 0 || d->n % d->per_sample != 0) { set_error("n must be a multiple of per_sample"); return DPM_ERR_ARG; }
    if (!for_quantile && (d->n_model == 0 || !d->predict_x0)) { set_error("thr requires n_model >= 1 and predict_x0"); return DPM_ERR_ARG; }
  }

  memset(kp, 0, sizeof(*kp));
  kp->x = d->x; kp->xe = xe; kp->m0 = d->m0; kp->m1 = d->m1; kp->m2 = d->m2;
  kp->ec = d->e_cond; kp->eu = d->e_uncond;
  kp->m_out = for_quantile ? nullptr : d->m_out;
  kp->out = for_quantile ? nullptr : d->out;
  kp->out2 = (for_quantile || form == DPM_FORM_NONE) ? nullptr : d->out2;
  kp->thr = for_quantile ? nullptr : d->thr;
  kp->n = d->n;
  kp->npk = (uint32_t)(d->n / kPacket);
  kp->per_sample = d->per_sample ? d->per_sample : 1;
  kp->pk_per_sample = (d->per_sample % kPacket == 0) ? (uint32_t)(d->per_sample / kPacket) : 0;
  kp->elem_offset = 0;
  kp->param = d->param; kp->predict_x0 = d->predict_x0 ? 1 : 0; kp->c0_on_old = d->c0_on_old ? 1 : 0;
  kp->use_xe = nd->xe ? 1 : 0;
  kp->xe_is_x = (nd->xe && nd->x && xe == d->x) ? 1 : 0;
  kp->form = form; kp->n_model = d->n_model;
  kp->state_dtype = d->state_dtype; kp->model_dtype = d->model_dtype;
  kp->guidance = d->guidance; kp->alpha_e = d->alpha_e; kp->sigma_e = d->sigma_e;
  kp->a = d->a; kp->c0 = d->c0; kp->c1 = d->c1; kp->c2 = d->c2;
  kp->w0 = d->w0; kp->w1 = d->w1; kp->w2 = d->w2; kp->w3 = d->w3; kp->w4 = d->w4;
  // reciprocal-refinement division (common.cuh: div_const) is used when every divisor the launch
  // can touch qualifies; host IEEE division gives the correctly rounded fp32 reciprocals
  const bool need_alpha = d->n_model >= 1 && d->predict_x0;
  const bool need_w4 = form == DPM_FORM_SS3T;
  bool ok = true;
  if (need_alpha) ok = ok && recip_div_ok(d->alpha_e);
  if (need_w4) ok = ok && recip_div_ok(d->w4);
  kp->r_alpha = need_alpha && ok ? 1.0f / d->alpha_e : 0.f;
  kp->raw_round = d->raw_round;
  kp->r_w4 = need_w4 && ok ? 1.0f / d->w4 : 0.f;
  kp->fast_div = ok ? 1 : 0;
  kp->dev_coef = for_quantile ? nullptr : d->dev_coef;
  return DPM_OK;
}

static bool all_aligned(const KParams& p, const Needs& nd) {
  const int sd = p.state_dtype, md = p.model_dtype;
  bool ok = true;
  if (nd.x) ok &= aligned(p.x, sd);
  if (nd.xe) ok &= aligned(p.xe, sd);
  if (nd.m0) ok &= aligned(p.m0, sd);
  if (nd.m1) ok &= aligned(p.m1, sd);
  if (nd.m2) ok &= aligned(p.m2, sd);
  if (nd.ec) ok &= aligned(p.ec, md);
  if (nd.eu) ok &= aligned(p.eu, md);
  if (p.m_out) ok &= aligned(p.m_out, sd);
  if (p.out) ok &= aligned(p.out, sd);
  if (p.out2) ok &= aligned(p.out2, sd);
  return ok;
}

static KParams shifted(const KParams& p, uint64_t elems) {
  KParams t = p;
  const int sd = p.state_dtype, md = p.model_dtype;
  t.x = off(p.x, sd, elems); t.xe = off(p.xe, sd, elems); t.m0 = off(p.m0, sd, elems);
  t.m1 = off(p.m1, sd, elems); t.m2 = off(p.m2, sd, elems);
  t.ec = off(p.ec, md, elems); t.eu = off(p.eu, md, elems);
  t.m_out = off(p.m_out, sd, elems); t.out = off(p.out, sd, elems); t.out2 = off(p.out2, sd, elems);
  t.n = p.n - elems;
  t.elem_offset = elems;
  return t;
}

static int finish(cudaStream_t) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    set_error("CUDA launch failed: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return (int)e;
  }
  return DPM_OK;
}

static int step_impl(const dpm_step_desc* d, cudaStream_t stream) {
  KParams p;
  Needs nd;
  if (d != nullptr && d->n == 0) return DPM_OK;  // empty tensors: nothing to do (pointers may be NULL)
  int rc = build_params(d, &p, &nd, false);
  if (rc != DPM_OK) return rc;
  if (p.n == 0) return DPM_OK;
  Tuning t{g_variant.load(), g_threads.load(), g_ctas.load()};

  bool body_done = false;
  if (p.npk > 0 && all_aligned(p, nd) && p.dev_coef == nullptr) {   // device-side scalars: generic kernel only
    int r = 1;
    // small launches (a few tiles per SM) gain nothing from the ring; auto keeps them direct
    // fp32 state: direct 256-bit loads sit at the HBM roofline already (fewer instructions per
    // byte); 16-bit state is issue-limited there and gains 10-20% from the ring (profiles/)
    const bool tma = p.raw_round == 0 &&   // reference-rounding mode: the direct variant's <RND> kernels
                     (t.variant == 1 || (t.variant == 2 && p.state_dtype != DPM_F32 &&
                                         p.npk >= (uint32_t)sm_count() * 1024u));
    if (tma) r = launch_step_tma(p, t, stream);
    if (r == 1) r = launch_step_direct(p, t, stream);
    if (r < 0 || r > 1) return r;
    body_done = (r == 0);
  }
  if (!body_done) {
    rc = launch_step_scalar(p, stream);  // whole range on the generic kernel
  } else if (p.n % kPacket) {
    rc = launch_step_scalar(shifted(p, (uint64_t)p.npk * kPacket), stream);  // tail
  }
  if (rc != DPM_OK) return rc;
  return finish(stream);
}

static int sde_step_impl(const dpm_step_desc* d, float cn, const float* noise, uint64_t seed, uint64_t offset,
                         cudaStream_t stream) {
  if (d == nullptr) { set_error("desc is NULL"); return DPM_ERR_ARG; }
  if (d->n == 0) return DPM_OK;
  if (d->form != DPM_FORM_LIN1 && d->form != DPM_FORM_DIFF2) {
    set_error("dpm_sde_step serves DPM_FORM_LIN1 and DPM_FORM_DIFF2 only (form %d)", d->form);
    return d->form < DPM_FORM_NONE || d->form > DPM_FORM_SS3T ? DPM_ERR_ARG : DPM_ERR_UNSUPPORTED;
  }
  if (d->dev_coef != nullptr) { set_error("dpm_sde_step takes its scalars by value (dev_coef must be NULL)"); return DPM_ERR_UNSUPPORTED; }
  if (d->raw_round != 0) { set_error("dpm_sde_step has no reference-rounding mode (raw_round must be 0)"); return DPM_ERR_UNSUPPORTED; }
  if (noise == nullptr && offset % 4 != 0) { set_error("philox offset must be a multiple of 4"); return DPM_ERR_ARG; }
  KParams p;
  Needs nd;
  int rc = build_params(d, &p, &nd, false);
  if (rc != DPM_OK) return rc;
  const bool vec_ok = all_aligned(p, nd) && (noise == nullptr || aligned(noise, DPM_F32));
  rc = launch_sde_step(p, vec_ok, cn, noise, seed, offset, stream);
  if (rc != DPM_OK) return rc;
  return finish(stream);
}

}  // namespace dpm

using namespace dpm;

extern "C" {

int dpm_version(void) { return DPM_B200_VERSION; }
const char* dpm_last_error(void) { return g_err; }
uint64_t dpm_launch_count(void) { return g_launches.load(); }

int dpm_set_tuning(int variant, int threads, int ctas_per_sm) {
  if (variant < 0 || variant > 2) { set_error("variant must be 0 (direct), 1 (TMA ring) or 2 (auto)"); return DPM_ERR_ARG; }
  if (threads != 0 && (threads < 32 || threads > 512 || threads % 32)) { set_error("threads must be a multiple of 32 in [32,512]"); return DPM_ERR_ARG; }
  if (ctas_per_sm < 0 || ctas_per_sm > 32) { set_error("ctas_per_sm must be in [0,32]"); return DPM_ERR_ARG; }
  g_variant = variant; g_threads = threads; g_ctas = ctas_per_sm;
  return DPM_OK;
}
int dpm_get_tuning(int* variant, int* threads, int* ctas_per_sm) {
  if (variant) *variant = g_variant.load();
  if (threads) *threads = g_threads.load();
  if (ctas_per_sm) *ctas_per_sm = g_ctas.load();
  return DPM_OK;
}

int dpm_step(const dpm_step_desc* desc, dpm_stream_t stream) {
  return step_impl(desc, static_cast<cudaStream_t>(stream));
}

int dpm_sde_step(const dpm_step_desc* desc, float noise_scale, const float* noise, uint64_t seed, uint64_t offset,
                 dpm_stream_t stream) {
  return sde_step_impl(desc, noise_scale, noise, seed, offset, static_cast<cudaStream_t>(stream));
}

static dpm_step_desc base_desc(void* out, const void* x, uint64_t n, int dtype, int form) {
  dpm_step_desc d;
  memset(&d, 0, sizeof(d));
  d.out = out; d.x = x; d.n = n; d.state_dtype = dtype; d.model_dtype = dtype; d.form = form;
  return d;
}

int dpm_lincomb(void* out, const void* x, const void* m0, const void* m1, const void* m2, int k,
                float a, float c0, float c1, float c2, uint64_t n, int dtype, dpm_stream_t stream) {
  if (k < 1 || k > 3) { set_error("k must be 1, 2 or 3"); return DPM_ERR_ARG; }
  dpm_step_desc d = base_desc(out, x, n, dtype, k == 1 ? DPM_FORM_LIN1 : k == 2 ? DPM_FORM_LIN2 : DPM_FORM_LIN3);
  d.m0 = m0; d.m1 = m1; d.m2 = m2; d.a = a; d.c0 = c0; d.c1 = c1; d.c2 = c2;
  return dpm_step(&d, stream);
}

int dpm_solver_first_update(void* x_t, const void* x, const void* model_s, float a, float c0,
                            uint64_t n, int dtype, dpm_stream_t stream) {
  dpm_step_desc d = base_desc(x_t, x, n, dtype, DPM_FORM_LIN1);
  d.m0 = model_s; d.a = a; d.c0 = c0;
  return dpm_step(&d, stream);
}

int dpm_multistep_second_update(void* x_t, const void* x, const void* model_prev_0,
                                const void* model_prev_1, float a, float c0, float c1,
                                float inv_r0, uint64_t n, int dtype, dpm_stream_t stream) {
  dpm_step_desc d = base_desc(x_t, x, n, dtype, DPM_FORM_DIFF2);
  d.m0 = model_prev_0; d.m1 = model_prev_1; d.a = a; d.c0 = c0; d.c1 = c1; d.w0 = inv_r0;
  return dpm_step(&d, stream);
}

int dpm_multistep_third_update(void* x_t, const void* x, const void* model_prev_0,
                               const void* model_prev_1, const void* model_prev_2, float a,
                               float c0, float c1, float c2, float inv_r0, float inv_r1, float w,
                               float q, uint64_t n, int dtype, dpm_stream_t stream) {
  dpm_step_desc d = base_desc(x_t, x, n, dtype, DPM_FORM_MS3);
  d.m0 = model_prev_0; d.m1 = model_prev_1; d.m2 = model_prev_2;
  d.a = a; d.c0 = c0; d.c1 = c1; d.c2 = c2; d.w0 = inv_r0; d.w1 = inv_r1; d.w2 = w; d.w3 = q;
  return dpm_step(&d, stream);
}

int dpm_singlestep_diff_update(void* x_t, const void* x, const void* model_s,
                               const void* model_new, float a, float c0, float c1, uint64_t n,
                               int dtype, dpm_stream_t stream) {
  dpm_step_desc d = base_desc(x_t, x, n, dtype, DPM_FORM_DIFF2);
  d.m0 = model_new; d.m1 = model_s; d.a = a; d.c0 = c0; d.c1 = c1; d.w0 = 1.f; d.c0_on_old = 1;
  return dpm_step(&d, stream);
}

int dpm_singlestep_third_taylor_update(void* x_t, const void* x, const void* model_s,
                                       const void* model_s1, const void* model_s2, float a,
                                       float c0, float c1, float c2, float inv_r1, float inv_r2,
                                       float r2, float r1, float r2_minus_r1, uint64_t n,
                                       int dtype, dpm_stream_t stream) {
  dpm_step_desc d = base_desc(x_t, x, n, dtype, DPM_FORM_SS3T);
  d.m0 = model_s2; d.m1 = model_s1; d.m2 = model_s;
  d.a = a; d.c0 = c0; d.c1 = c1; d.c2 = c2;
  d.w0 = inv_r1; d.w1 = inv_r2; d.w2 = r2; d.w3 = r1; d.w4 = r2_minus_r1;
  return dpm_step(&d, stream);
}

int dpm_cfg_combine(void* eps, const void* eps_uncond, const void* eps_cond, float scale,
                    uint64_t n, int dtype, dpm_stream_t stream) {
  dpm_step_desc d = base_desc(nullptr, nullptr, n, dtype, DPM_FORM_NONE);
  d.n_model = 2; d.e_cond = eps_cond; d.e_uncond = eps_uncond; d.guidance = scale;
  d.m_out = eps; d.param = DPM_PARAM_NOISE; d.predict_x0 = 0;
  return dpm_step(&d, stream);
}

int dpm_data_prediction(void* x0, const void* x, const void* eps, float alpha_t, float sigma_t,
                        const float* thr, uint64_t per_sample, uint64_t n, int dtype,
                        dpm_stream_t stream) {
  dpm_step_desc d = base_desc(nullptr, nullptr, n, dtype, DPM_FORM_NONE);
  d.n_model = 1; d.e_cond = eps; d.xe = x; d.m_out = x0; d.predict_x0 = 1;
  d.alpha_e = alpha_t; d.sigma_e = sigma_t; d.thr = thr; d.per_sample = per_sample;
  return dpm_step(&d, stream);
}

int dpm_duplicate(void* out, const void* x, uint64_t n, int dtype, dpm_stream_t stream) {
  if (n == 0) return DPM_OK;
  if (out == nullptr || x == nullptr || !valid_dtype(dtype)) { set_error("duplicate: NULL tensor or bad dtype"); return DPM_ERR_ARG; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint64_t bytes = n * (uint64_t)esize(dtype);
  int r = launch_duplicate(out, x, bytes, st);
  if (r == 1) {   // unaligned views: two plain device-to-device copies
    cudaError_t e = cudaMemcpyAsync(out, x, bytes, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(static_cast<char*>(out) + bytes, x, bytes, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { set_error("duplicate: %s", cudaGetErrorString(e)); cudaGetLastError(); return (int)e; }
    return DPM_OK;
  }
  if (r != 0) return r;
  return finish(st);
}

int dpm_philox_policy(uint64_t numel, uint32_t* grid, uint64_t* counter_offset) {
  if (grid == nullptr || counter_offset == nullptr) { set_error("philox policy: NULL output"); return DPM_ERR_ARG; }
  philox_policy(numel, grid, counter_offset);
  return DPM_OK;
}

int dpm_add_noise_philox(void* xt, const void* x, uint64_t n, int t_count, const float* alpha_t, const float* sigma_t,
                         uint64_t seed, uint64_t offset, int x_dtype, int out_dtype, dpm_stream_t stream) {
  if (n == 0 || t_count == 0) return DPM_OK;
  if (!xt || !x || !alpha_t || !sigma_t || !valid_dtype(x_dtype) || !valid_dtype(out_dtype)) { set_error("add_noise: NULL argument or bad dtype"); return DPM_ERR_ARG; }
  int rc = launch_noise_philox(xt, x, nullptr, nullptr, 0, n, t_count, alpha_t, sigma_t, seed, offset, x_dtype, out_dtype,
                               static_cast<cudaStream_t>(stream));
  return rc != DPM_OK ? rc : finish(static_cast<cudaStream_t>(stream));
}

int dpm_diffedit_corrector(void* out, const void* x, const void* x0, const float* mask, uint64_t mask_n, uint64_t n,
                           float alpha_t, float sigma_t, uint64_t seed, uint64_t offset, int dtype, dpm_stream_t stream) {
  if (n == 0) return DPM_OK;
  if (!out || !x || !x0 || !mask || mask_n == 0 || n % mask_n != 0 || !valid_dtype(dtype)) { set_error("corrector: NULL argument, bad dtype or a mask that does not tile x"); return DPM_ERR_ARG; }
  int rc = launch_noise_philox(out, x0, x, mask, mask_n, n, 1, &alpha_t, &sigma_t, seed, offset, dtype, dtype,
                               static_cast<cudaStream_t>(stream));
  return rc != DPM_OK ? rc : finish(static_cast<cudaStream_t>(stream));
}

size_t dpm_dynamic_threshold_workspace(uint64_t n_samples, uint64_t per_sample) {
  return quantile_workspace_bytes(n_samples, per_sample);
}

int dpm_dynamic_threshold(float* s_out, const dpm_step_desc* desc, float q, float max_val,
                          void* workspace, size_t workspace_bytes, dpm_stream_t stream) {
  if (s_out == nullptr) { set_error("s_out is NULL"); return DPM_ERR_ARG; }
  if (!(q >= 0.f && q <= 1.f)) { set_error("q must be in [0,1]"); return DPM_ERR_ARG; }
  KParams p;
  Needs nd;
  if (desc != nullptr && desc->n == 0) return DPM_OK;
  int rc = build_params(desc, &p, &nd, true);
  if (rc != DPM_OK) return rc;
  if (p.n == 0) return DPM_OK;
  rc = launch_quantile(s_out, p, p.n / p.per_sample, q, max_val, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
  if (rc != DPM_OK) return rc;
  return finish(static_cast<cudaStream_t>(stream));
}

int dpm_adaptive_init(const dpm_adaptive_ctl* ctl, float t_T, float h_init, dpm_stream_t stream) {
  int rc = launch_adaptive_init(ctl, t_T, h_init, static_cast<cudaStream_t>(stream));
  return rc != DPM_OK ? rc : finish(static_cast<cudaStream_t>(stream));
}
int dpm_adaptive_plan(const dpm_adaptive_ctl* ctl, dpm_stream_t stream) {
  int rc = launch_adaptive_plan(ctl, static_cast<cudaStream_t>(stream));
  return rc != DPM_OK ? rc : finish(static_cast<cudaStream_t>(stream));
}
int dpm_adaptive_decide(const dpm_adaptive_ctl* ctl, dpm_stream_t stream) {
  int rc = launch_adaptive_decide(ctl, static_cast<cudaStream_t>(stream));
  return rc != DPM_OK ? rc : finish(static_cast<cudaStream_t>(stream));
}
int dpm_select_copy(void* dst, const void* src, const float* state, uint64_t bytes, dpm_stream_t stream) {
  if (bytes == 0) return DPM_OK;
  if (!dst || !src || !state) { set_error("select copy: NULL argument"); return DPM_ERR_ARG; }
  int rc = launch_select_copy(dst, src, state, bytes, static_cast<cudaStream_t>(stream));
  return rc != DPM_OK ? rc : finish(static_cast<cudaStream_t>(stream));
}

size_t dpm_adaptive_error_workspace(uint64_t n, uint64_t per_sample) {
  return adaptive_workspace_bytes(n, per_sample);
}

int dpm_adaptive_error(float* e_out, const void* x_higher, const void* x_lower, const void* x_prev, float atol,
                       float rtol, uint64_t per_sample, uint64_t n, int dtype, void* workspace,
                       size_t workspace_bytes, dpm_stream_t stream) {
  if (!e_out || !x_higher || !x_lower || !x_prev) { set_error("adaptive error: NULL tensor"); return DPM_ERR_ARG; }
  if (!valid_dtype(dtype) || per_sample == 0 || n == 0 || n % per_sample) { set_error("adaptive error: bad dtype or sizes"); return DPM_ERR_ARG; }
  int rc = launch_adaptive_error(e_out, x_higher, x_lower, x_prev, atol, rtol, per_sample, n, dtype, workspace,
                                 workspace_bytes, static_cast<cudaStream_t>(stream));
  if (rc != DPM_OK) return rc;
  return finish(static_cast<cudaStream_t>(stream));
}

}  // extern "C"
