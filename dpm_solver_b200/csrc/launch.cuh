// launch.cuh -- host-side helpers shared by the translation units of libdpmsolver_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace dpm {

struct Tuning {
  int variant;      // 0 direct, 1 TMA ring
  int threads;      // threads per CTA (0 = default)
  int ctas_per_sm;  // persistent-grid CTAs per SM (0 = default)
};

int sm_count();                     // SMs of the current device (cached per device)
int max_smem_optin();               // max opt-in dynamic shared memory per CTA
void count_launch();                // bump the library launch counter
// opt the kernel into the device's maximum dynamic shared memory (and, optionally, non-portable
// cluster sizes) the first time it is used on the current device; later calls are a hash lookup
int ensure_max_smem(const void* kernel, bool nonportable_cluster = false);
void set_error(const char* fmt, ...);

// Programmatic dependent launch (PDL): the step kernels call pdl_wait() after their prologue (barrier init, index
// setup) and before touching global memory, and pdl_trigger() at entry; launched with the programmatic-stream-
// serialization attribute, the CTAs of step i+1 become resident while step i drains and only their first global
// access waits for its completion (and visibility). Without the attribute both are no-ops. Persistent one-wave grids
// only, so an early dependent can never starve its primary.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled();   // DPM_PDL=0 turns the launch attribute off (A/B measurements)

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// each returns 0 on launch, 1 if this variant does not serve the request, <0 / cudaError on error
int launch_step_direct(const KParams& p, const Tuning& t, cudaStream_t stream);
int launch_step_scalar(const KParams& p, cudaStream_t stream);
int launch_step_tma(const KParams& p, const Tuning& t, cudaStream_t stream);
void philox_policy(uint64_t numel, uint32_t* grid, uint64_t* counter_offset);
int launch_sde_step(const KParams& p, bool vec_ok, float cn, const float* noise, uint64_t seed, uint64_t offset,
                    cudaStream_t stream);
int launch_noise_philox(void* out, const void* x, const void* xt, const float* mask, uint64_t mask_n, uint64_t n,
                        int t_count, const float* alpha, const float* sigma, uint64_t seed, uint64_t offset,
                        int x_dtype, int out_dtype, cudaStream_t stream);
int launch_adaptive_init(const dpm_adaptive_ctl* a, float t_T, float h_init, cudaStream_t stream);
int launch_adaptive_plan(const dpm_adaptive_ctl* a, cudaStream_t stream);
int launch_adaptive_decide(const dpm_adaptive_ctl* a, cudaStream_t stream);
int launch_select_copy(void* dst, const void* src, const float* state, uint64_t bytes, cudaStream_t stream);
int launch_duplicate(void* dst, const void* src, uint64_t bytes, cudaStream_t stream);
int launch_quantile(float* s_out, const KParams& p, uint64_t n_samples, float q, float max_val,
                    void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t quantile_workspace_bytes(uint64_t n_samples, uint64_t per_sample);
size_t adaptive_workspace_bytes(uint64_t n, uint64_t per_sample);
int launch_adaptive_error(float* out, const void* xh, const void* xl, const void* xp, float atol, float rtol,
                          uint64_t per_sample, uint64_t n, int dtype, void* ws, size_t ws_bytes, cudaStream_t stream);

}  // namespace dpm
