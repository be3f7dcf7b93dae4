/*
 * dpm_solver_b200.h -- C-ABI of libdpmsolver_b200.so
 *
 * B200 (sm_100a) implementation of DPM-Solver's per-step update path. The reference
 * (LuChengTHU/dpm-solver, dpm_solver_pytorch.py) has no FFI: every function below replaces a
 * run of PyTorch eager elementwise ops in that file; the line ranges are cited per function.
 *
 * Conventions
 *   - all tensor arguments are raw DEVICE pointers to contiguous memory, `n` elements;
 *   - scalars (alpha, sigma, phi, ... ) are fp32 computed on the HOST and passed by value, so
 *     every launch is CUDA-graph capturable and no exp/log runs per element on the device;
 *   - arithmetic is fp32 in registers in the reference's exact operation order with FMA
 *     contraction disabled (results are bit-identical to the reference's fp32 CPU path when the
 *     storage dtype is fp32); bf16/f16 storage is rounded to nearest-even once, on store;
 *   - inputs are read-only and may alias each other; `out` may alias `x` (element-wise
 *     in-place) but no other overlap is allowed;
 *   - every entry point takes the stream explicitly, never synchronises, never allocates;
 *   - return value: 0 on success, negative dpm_status on argument errors, positive cudaError_t
 *     on CUDA errors. dpm_last_error() returns a thread-local description.
 */
#ifndef DPM_SOLVER_B200_H
#define DPM_SOLVER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPM_B200_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define DPM_API __attribute__((visibility("default")))
#else
#define DPM_API
#endif

typedef void* dpm_stream_t; /* cudaStream_t */

typedef enum dpm_status {
  DPM_OK = 0,
  DPM_ERR_ARG = -1,         /* null pointer / bad enum / bad size */
  DPM_ERR_UNSUPPORTED = -2, /* valid request this build cannot serve */
  DPM_ERR_ALIGN = -3        /* reserved: (mis)alignment is handled internally today */
} dpm_status;

typedef enum dpm_dtype { DPM_F32 = 0, DPM_BF16 = 1, DPM_F16 = 2 } dpm_dtype;

/* How the buffered "model value" T0 and the older buffers enter the update.
 * NEW = the most recent model value (computed in-kernel from raw model outputs when
 * n_model > 0, else loaded from m0); M1/M2 = older buffers.
 *
 *   NONE : no state update, only m_out is written (data_prediction_fn :433-442)
 *   LIN1 : out = a*x + c0*NEW                                   (first update :573-588)
 *   LIN2 : out = a*x + c0*NEW + c1*M1                           (generic AXPY chains)
 *   LIN3 : out = a*x + c0*NEW + c1*M1 + c2*M2
 *   DIFF2: D = w0*(NEW - M1); out = a*x + c0*(c0_on_old ? M1 : NEW) + c1*D
 *          multistep-2 :823-851 (c0_on_old=0, w0=1/r0) and the singlestep difference
 *          steps :630-669, :728-739, :767-778 (c0_on_old=1, w0=1, M1 = model_s)
 *   MS3  : D10=w0*(NEW-M1); D11=w1*(M1-M2); dd=D10-D11; D1=D10+w2*dd; D2=w3*dd;
 *          out = a*x + c0*NEW + c1*D1 + c2*D2                   (multistep-3 :880-903)
 *   SS3T : singlestep-3 'taylor' :741-750 / :780-789, M2=model_s, M1=model_s1, NEW=model_s2:
 *          D10=w0*(M1-M2); D11=w1*(NEW-M2); D1=(w2*D10-w3*D11)/w4; D2=(2*(D11-D10))/w4;
 *          out = a*x + c0*M2 + c1*D1 + c2*D2
 * Sums are evaluated left to right, each product and each sum rounded separately.
 */
typedef enum dpm_form {
  DPM_FORM_NONE = 0,
  DPM_FORM_LIN1 = 1,
  DPM_FORM_LIN2 = 2,
  DPM_FORM_LIN3 = 3,
  DPM_FORM_DIFF2 = 4,
  DPM_FORM_MS3 = 5,
  DPM_FORM_SS3T = 6
} dpm_form;

/* Parameterisation of the network output, model_wrapper.noise_pred_fn :288-298 */
typedef enum dpm_param {
  DPM_PARAM_NOISE = 0,   /* eps = out                         :289 */
  DPM_PARAM_X_START = 1, /* eps = (xe - alpha*out)/sigma      :292 */
  DPM_PARAM_V = 2,       /* eps = alpha*out + sigma*xe        :295 */
  DPM_PARAM_SCORE = 3    /* eps = (-sigma)*out                :298 */
} dpm_param;

/* One fused solver step. With n_model == 0 this is a pure update on buffered model values.
 * With n_model >= 1 it is the fused "post-model" step: raw network outputs are converted to
 * the buffered model value (parameterisation -> CFG combine -> eps->x0 -> thresholding
 * clamp), optionally stored to m_out, and consumed by the update in the same pass. */
typedef struct dpm_step_desc {
  /* state dtype tensors */
  const void* x;   /* base state x_s of the update (may be NULL iff form == NONE)          */
  const void* xe;  /* state the model was evaluated at (== x for multistep; x_s1/x_s2 for
                      singlestep); used by x_start/v conversion and eps->x0. NULL => x    */
  const void* m0;  /* NEW buffered model value, read when n_model == 0                      */
  const void* m1;  /* older buffers, as the form requires                                  */
  const void* m2;
  void* m_out;     /* optional: computed model value written here (n_model >= 1)           */
  void* out;       /* x_t; required unless form == NONE                                    */
  void* out2;      /* optional second copy of x_t (e.g. the other half of the network's
                      doubled CFG batch, model_wrapper :326); NULL = none                   */
  /* model dtype tensors */
  const void* e_cond;   /* network output (conditional half under CFG)                     */
  const void* e_uncond; /* unconditional half, n_model == 2; CFG :329-330                  */
  /* per-sample thresholds s_b (already max'ed with thresholding_max_val), fp32 [n/per_sample]
   * or NULL. clamp(x0,-s,s)/s, dynamic_thresholding_fn :423-424 */
  const float* thr;
  uint64_t n;          /* total elements                                                   */
  uint64_t per_sample; /* elements per sample (C*H*W); only read when thr != NULL           */
  int32_t state_dtype; /* dpm_dtype of x, xe, m*, m_out, out                               */
  int32_t model_dtype; /* dpm_dtype of e_cond, e_uncond                                    */
  int32_t form;        /* dpm_form                                                         */
  int32_t n_model;     /* 0, 1 or 2 raw network outputs                                    */
  int32_t param;       /* dpm_param                                                        */
  int32_t predict_x0;  /* 1: buffered value is x0 = (xe - sigma_e*eps)/alpha_e :439         */
  int32_t c0_on_old;   /* DIFF2 only                                                       */
  int32_t raw_round;   /* 0 (default). Reference-rounding mode for networks that return 16-bit NOISE into an
                          fp32 state: bits 0-1 = DPM_BF16 / DPM_F16, the type the raw outputs arrived in --
                          the CFG combine :329-330 then rounds to it after each of its three ops, as the
                          reference's eager 16-bit ops do; bit 2 (+4) = the buffered values are such raw
                          outputs, so their differences (:823, :880-881, :636, :735, :741-742) are rounded
                          to that type before the fp32 coefficients widen them. Generic kernel only.   */
  float guidance;      /* CFG scale s: eps = eps_u + s*(eps_c - eps_u) :330                */
  float alpha_e;       /* alpha, sigma at the model evaluation time                         */
  float sigma_e;
  float a, c0, c1, c2; /* update coefficients (signs folded in)                            */
  float w0, w1, w2, w3, w4;
  /* Optional (NULL = off): the launch reads its scalars from DEVICE memory instead of the by-value fields above --
   * 16 floats {a, c0, c1, c2, w0, w1, w2, w3, w4, alpha_e, sigma_e, 5 reserved}, written earlier on the same stream
   * by dpm_adaptive_plan(): the on-device step-size controller of dpm_solver_adaptive (:956-1010), whose next
   * coefficients depend on an accept/reject decision the host never sees. Served by the generic kernel. */
  const float* dev_coef;
} dpm_step_desc;

/* ---- library ------------------------------------------------------------------------ */
DPM_API int dpm_version(void);
DPM_API const char* dpm_last_error(void);

/* Tuning knobs (process-wide, read at launch): variant 0 = direct 128/256-bit global
 * loads, 1 = TMA (cp.async.bulk) shared-memory ring, 2 = auto (default: the ring for 16-bit state
 * tensors and launches of >= 1024 packets per SM, direct otherwise); threads per CTA; CTAs per SM for the persistent
 * grid; 0 keeps the built-in default. Returns DPM_ERR_ARG on invalid values. */
DPM_API int dpm_set_tuning(int variant, int threads, int ctas_per_sm);
DPM_API int dpm_get_tuning(int* variant, int* threads, int* ctas_per_sm);
/* number of kernels launched by this library since load (all streams) */
DPM_API uint64_t dpm_launch_count(void);

/* ---- the general fused step --------------------------------------------------------- */
DPM_API int dpm_step(const dpm_step_desc* desc, dpm_stream_t stream);

/* ---- named entry points, one per reference function --------------------------------- */

/* out = a*x + c0*m0 [+ c1*m1 [+ c2*m2]], k in 1..3. Generic AXPY chain: add_noise :1026,
 * classifier guidance :321, noise_pred_fn conversions :292-298. */
DPM_API int dpm_lincomb(void* out, const void* x, const void* m0, const void* m1, const void* m2,
                int k, float a, float c0, float c1, float c2, uint64_t n, int dtype,
                dpm_stream_t stream);

/* DPM_Solver.dpm_solver_first_update :547-592.  x_t = a*x + c0*model_s
 * (++: a = sigma_t/sigma_s, c0 = -(alpha_t*expm1(-h)); eps: a = exp(dlog_alpha),
 * c0 = -(sigma_t*expm1(h))). */
DPM_API int dpm_solver_first_update(void* x_t, const void* x, const void* model_s, float a, float c0,
                            uint64_t n, int dtype, dpm_stream_t stream);

/* DPM_Solver.multistep_dpm_solver_second_update :796-852.
 * D1_0 = inv_r0*(model_prev_0 - model_prev_1); x_t = a*x + c0*model_prev_0 + c1*D1_0. */
DPM_API int dpm_multistep_second_update(void* x_t, const void* x, const void* model_prev_0,
                                const void* model_prev_1, float a, float c0, float c1,
                                float inv_r0, uint64_t n, int dtype, dpm_stream_t stream);

/* DPM_Solver.multistep_dpm_solver_third_update :854-904.
 * inv_r0 = 1/r0, inv_r1 = 1/r1, w = r0/(r0+r1), q = 1/(r0+r1). */
DPM_API int dpm_multistep_third_update(void* x_t, const void* x, const void* model_prev_0,
                               const void* model_prev_1, const void* model_prev_2, float a,
                               float c0, float c1, float c2, float inv_r0, float inv_r1,
                               float w, float q, uint64_t n, int dtype, dpm_stream_t stream);

/* The difference step shared by singlestep_dpm_solver_second_update :636-669 and
 * singlestep_dpm_solver_third_update :728-739 / :767-778:
 * x_t = a*x + c0*model_s + c1*(model_new - model_s). */
DPM_API int dpm_singlestep_diff_update(void* x_t, const void* x, const void* model_s,
                               const void* model_new, float a, float c0, float c1, uint64_t n,
                               int dtype, dpm_stream_t stream);

/* singlestep_dpm_solver_third_update, solver_type='taylor' :741-750 / :780-789. */
DPM_API int dpm_singlestep_third_taylor_update(void* x_t, const void* x, const void* model_s,
                                       const void* model_s1, const void* model_s2, float a,
                                       float c0, float c1, float c2, float inv_r1, float inv_r2,
                                       float r2, float r1, float r2_minus_r1, uint64_t n,
                                       int dtype, dpm_stream_t stream);

/* model_wrapper.model_fn classifier-free branch :329-330:
 * eps = eps_uncond + scale*(eps_cond - eps_uncond). */
DPM_API int dpm_cfg_combine(void* eps, const void* eps_uncond, const void* eps_cond, float scale,
                    uint64_t n, int dtype, dpm_stream_t stream);

/* model_wrapper.model_fn classifier-free branch :326: x_in = torch.cat([x] * 2). out holds 2*n elements; x is read
 * once and written to out[0, n) and out[n, 2n). (Inside the sampling loop dpm_step's out2 does this for free; this
 * entry serves the first evaluation of a run.) */
DPM_API int dpm_duplicate(void* out, const void* x, uint64_t n, int dtype, dpm_stream_t stream);

/* DPM_Solver.data_prediction_fn :433-442 (without corrector when thr == NULL):
 * x0 = (x - sigma_t*eps)/alpha_t, then optional clamp(x0,-thr_b,thr_b)/thr_b. */
DPM_API int dpm_data_prediction(void* x0, const void* x, const void* eps, float alpha_t, float sigma_t,
                        const float* thr, uint64_t per_sample, uint64_t n, int dtype,
                        dpm_stream_t stream);

/* ---- noise drawn inside the kernel (torch.randn-compatible Philox) ------------------------------------------
 * ATen's launch policy for a randn of `numel` elements on the current device: the virtual grid the kernels below
 * replay, and the amount the caller must advance the torch CUDA generator's philox offset by afterwards. */
DPM_API int dpm_philox_policy(uint64_t numel, uint32_t* grid, uint64_t* counter_offset);

/* DPM_Solver.add_noise(x, t, noise=None) :1012-1030 with the noise generated in registers:
 *   xt[i] = alpha_t[i]*x + sigma_t[i]*randn[i],  i < t_count <= 16 (alpha_t, sigma_t: HOST arrays),  xt: [t_count, n].
 * (seed, offset) = the torch CUDA generator's state; for that state the result equals
 * torch.randn((t_count, n)) followed by the reference's three eager ops, bit for bit. x_dtype -> out_dtype: the
 * reference's promotion (16-bit x, fp32 result) or 16-bit storage. */
DPM_API int dpm_add_noise_philox(void* xt, const void* x, uint64_t n, int t_count, const float* alpha_t,
                                 const float* sigma_t, uint64_t seed, uint64_t offset, int x_dtype, int out_dtype,
                                 dpm_stream_t stream);

/* One stochastic SDE-DPM-Solver(++) multistep step (orders 1 and 2): the step dpm_step(desc) computes, plus one
 * separately rounded noise term,
 *   out = ((a*x + c0*NEW) + c1*D) + noise_scale*z        (form LIN1: out = (a*x + c0*NEW) + noise_scale*z)
 * with every other field of desc read as dpm_step reads it (n_model 0/1/2, param, CFG, predict_x0, thr, m_out, out2).
 * z is element i, in storage order, of
 *   noise != NULL: the fp32 array noise[n];
 *   noise == NULL: torch.randn(n) drawn from a torch CUDA generator in state (seed, offset), generated in registers
 *                  with the virtual grid of dpm_philox_policy(desc->n); the caller advances the generator's offset
 *                  by that policy's counter_offset. offset must be a multiple of 4.
 * Only DPM_FORM_LIN1 and DPM_FORM_DIFF2 are served, with the scalars by value: another form, dev_coef != NULL or
 * raw_round != 0 returns DPM_ERR_UNSUPPORTED. */
DPM_API int dpm_sde_step(const dpm_step_desc* desc, float noise_scale, const float* noise, uint64_t seed,
                         uint64_t offset, dpm_stream_t stream);

/* DiffEdit corrector (examples/stable-diffusion/scripts/diffedit_inpaint.ipynb corrector_fn + sampler.py:92-96):
 *   out = x*mask + (1 - mask)*(alpha_t*x0 + sigma_t*randn_like(x0)),  one launch, noise in registers.
 * mask: fp32, mask_n elements, broadcast over the leading dimensions of x (n % mask_n == 0). */
DPM_API int dpm_diffedit_corrector(void* out, const void* x, const void* x0, const float* mask, uint64_t mask_n,
                                   uint64_t n, float alpha_t, float sigma_t, uint64_t seed, uint64_t offset,
                                   int dtype, dpm_stream_t stream);

/* DPM_Solver.dynamic_thresholding_fn :416-423, first half: per-sample
 * s_b = max(quantile(|x0_b|, q), max_val) with torch.quantile's linear interpolation between
 * the two adjacent order statistics (rank arithmetic in fp32). x0 is recomputed on the fly from
 * the same inputs dpm_step() takes (desc->x/xe, e_cond, e_uncond, param, guidance, alpha_e,
 * sigma_e; predict_x0 must be 1); desc->thr/form/out/m* are ignored. Always exact.
 * With a workspace of dpm_dynamic_threshold_workspace() bytes (16-byte aligned device memory,
 * contents irrelevant) samples of >= 8192 elements take the streaming pipeline: pivot sampling,
 * one HBM-rate count/compact pass, exact finish on the ~2 % of keys inside the bracket. Without
 * it (workspace == NULL), or for smaller samples, one thread-block cluster per sample runs a
 * radix select with the keys staged in (distributed) shared memory. s_out: fp32 [n/per_sample]. */
DPM_API size_t dpm_dynamic_threshold_workspace(uint64_t n_samples, uint64_t per_sample);
DPM_API int dpm_dynamic_threshold(float* s_out, const dpm_step_desc* desc, float q, float max_val,
                                  void* workspace, size_t workspace_bytes, dpm_stream_t stream);

/* DPM_Solver.dpm_solver_adaptive error estimate :999-1001:
 *   delta = max(atol, rtol*max(|x_lower|, |x_prev|));
 *   E = max over samples of sqrt(mean(((x_higher - x_lower)/delta)^2))  ->  e_out[0] (device fp32).
 * One streaming pass + a one-CTA epilogue, deterministic reduction order. workspace: device memory
 * of dpm_adaptive_error_workspace(n, per_sample) bytes. */
DPM_API size_t dpm_adaptive_error_workspace(uint64_t n, uint64_t per_sample);
DPM_API int dpm_adaptive_error(float* e_out, const void* x_higher, const void* x_lower,
                               const void* x_prev, float atol, float rtol, uint64_t per_sample,
                               uint64_t n, int dtype, void* workspace, size_t workspace_bytes,
                               dpm_stream_t stream);

/* ---- dpm_solver_adaptive with the controller on the device (:956-1010) -------------------------------------
 * Device buffers (caller-allocated, fp32): state[16] (s, lambda_s, lambda_0, h, t, nfe, done, accept, iterations as
 * int bit patterns where integral), coef[4][16] (one dpm_step_desc.dev_coef block per fused launch of an
 * iteration), times[6] (evaluation times s, s1, s2, then the model-input times the network receives), error[1]
 * (written by dpm_adaptive_error). Schedule: discrete (tables as NoiseScheduleVP holds them, plus their flipped
 * copies, all on the device) or the continuous linear VPSDE.
 *   dpm_adaptive_init   : s = t_T, lambda_s, lambda_0, h = h_init                                      :972-977
 *   dpm_adaptive_plan   : t = lambda^-1(lambda_s + h) and every coefficient block / time label of the
 *                         lower- and higher-order updates of this iteration                             :984-992
 *   dpm_adaptive_decide : E <= 1 ? accept (s = t, lambda_s) ; h = min(theta*h*E^(-1/order), lambda_0 - lambda_s);
 *                         nfe += order; done = |s - t_0| <= t_err (2 = NaN error estimate)              :1002-1008
 *   dpm_select_copy     : dst <- src iff the last decide accepted (x <- x_higher, x_prev <- x_lower)     :1003-1005
 * Launch order per iteration for order 2: plan, [net(x,s)] step(coef 0: x_lower), step(coef 1: x_s1, pure),
 * [net(x_s1,s1)] step(coef 2: x_higher), error, decide, select_copy x2; order 3 uses coef 0..3 (see
 * dpm_solver_b200/solver.py). After `done` the plan emits identity coefficients, so a fixed-length chunk of
 * iterations can be enqueued (or graph-captured) and `done` read back once per chunk. */
typedef struct dpm_adaptive_ctl {
  int32_t schedule_kind;       /* 0 discrete, 1 linear */
  int32_t table_len;
  const float* t_array;        /* device, [table_len] */
  const float* log_alpha_array;
  const float* log_alpha_flipped;
  const float* t_flipped;
  float beta_0, beta_1_minus_beta_0, inv_total_N;
  int32_t discrete_time_input; /* 1: the network takes (t - 1/N)*1000 (:278), 0: t */
  int32_t order;               /* 2 or 3 */
  int32_t predict_x0;          /* dpmsolver++ */
  int32_t taylor;              /* solver_type == 'taylor' */
  float t_0, theta, t_err;
  float* state;                /* device [16] */
  float* coef;                 /* device [4][16] */
  float* times;                /* device [6] */
  const float* error;          /* device [1] */
} dpm_adaptive_ctl;

DPM_API int dpm_adaptive_init(const dpm_adaptive_ctl* ctl, float t_T, float h_init, dpm_stream_t stream);
DPM_API int dpm_adaptive_plan(const dpm_adaptive_ctl* ctl, dpm_stream_t stream);
DPM_API int dpm_adaptive_decide(const dpm_adaptive_ctl* ctl, dpm_stream_t stream);
DPM_API int dpm_select_copy(void* dst, const void* src, const float* state, uint64_t bytes, dpm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DPM_SOLVER_B200_H */
