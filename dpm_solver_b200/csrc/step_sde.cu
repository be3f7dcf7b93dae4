// step_sde.cu -- one stochastic SDE-DPM-Solver(++) step with the Gaussian noise drawn INSIDE the kernel.
//
//   out = ((a*x + c0*NEW) + c1*D) + cn*z          (dpm_sde_step, include/dpm_solver_b200.h)
//
// NEW is the buffered model value (computed in-kernel from the raw network outputs when n_model > 0, exactly as
// dpm_step does: parameterisation -> CFG -> eps->x0 -> thresholding clamp), D = w0*(NEW - M1) for DIFF2, and z is
// element li of torch.randn(numel) for the generator state (seed, offset): curand's Philox4_32_10 through
// curand_normal4, with ATen's launch geometry replayed as a VIRTUAL geometry (csrc/philox.cu). Virtual thread idx,
// iteration k, lane ii own element li = idx + G*(4k + ii), G = 256 * (virtual grid of dpm_philox_policy(n)), and
// read the k-th curand_normal4 of curand_init(seed, idx, offset), i.e. the first one of
// curand_init(seed, idx, offset + 4k).
//
// Work item of the packet kernel: one iteration k and 8 consecutive virtual threads v0..v0+7 (v0 % 8 == 0). Its 8
// Philox calls give 32 normals, which are exactly the elements of four aligned 8-element packets
// v0 + G*(4k + ii), ii = 0..3 (G is a multiple of 256). No Philox output is wasted and every global access is a
// 128-bit (16-bit storage) or 256-bit (fp32) vector access.
//
// This file is compiled WITH fma contraction (build.py, FMAD_DEFAULT): curand's Box-Muller has to round like the
// copy inside torch's randn kernel. Every step of the solver chain is therefore spelled with the never-contracted
// __fmul_rn / __fadd_rn / __fsub_rn / __fdiv_rn intrinsics; of common.cuh only the layout helpers (KParams, packet
// load/store/pack, load_any/store_any, clamp_sym) are used, none of its arithmetic.
#include <curand_kernel.h>

#include "common.cuh"
#include "launch.cuh"

namespace dpm {

constexpr int kSdeThreads = 256;
constexpr int kPhiloxBlockV = 256;   // ATen's block size: G = 256 * virtual grid

struct SdeParams {
  KParams k;
  const float* noise;   // fp32 materialised noise [n] or NULL (Philox)
  uint64_t seed, offset;
  uint64_t G;           // virtual threads of ATen's randn launch for n elements
  uint64_t items;       // work items of the packet kernel: ceil(n / 4G) * G / 8
  float cn;
};

// ---- the element chain, every operation rounded separately ---------------------------------------------------
// x / d for a launch-constant divisor: common.cuh's div_const (same proof, same guard), with the first product
// spelled __fmul_rn so that it cannot be contracted in this translation unit
__device__ __forceinline__ float div_const_rn(float x, float d, float r) {
  float q = __fmul_rn(x, r);
  float e = fmaf(-q, d, x);
  q = fmaf(e, r, q);
  e = fmaf(-q, d, x);
  q = fmaf(e, r, q);
  const float ax = fabsf(x);
  if (!(ax > 1e-25f && ax < 1e30f)) q = __fdiv_rn(x, d);
  return q;
}

// model_wrapper.noise_pred_fn (common.cuh: convert_param)
__device__ __forceinline__ float convert_rn(int param, float out, float xe, float alpha, float sigma) {
  switch (param) {
    case DPM_PARAM_X_START: return __fdiv_rn(__fsub_rn(xe, __fmul_rn(alpha, out)), sigma);
    case DPM_PARAM_V: return __fadd_rn(__fmul_rn(alpha, out), __fmul_rn(sigma, xe));
    case DPM_PARAM_SCORE: return __fmul_rn(-sigma, out);
    default: return out;
  }
}

// raw network output(s) -> buffered model value (common.cuh: model_value without the reference-rounding mode)
__device__ __forceinline__ float model_rn(const KParams& p, int ne, float xe, float ec, float eu, float thr, bool clamp) {
  float eps = convert_rn(p.param, ec, xe, p.alpha_e, p.sigma_e);
  if (ne == 2) {
    const float epu = convert_rn(p.param, eu, xe, p.alpha_e, p.sigma_e);
    eps = __fadd_rn(epu, __fmul_rn(p.guidance, __fsub_rn(eps, epu)));   // CFG combine
  }
  if (p.predict_x0) {
    const float num = __fsub_rn(xe, __fmul_rn(p.sigma_e, eps));
    float x0 = p.fast_div ? div_const_rn(num, p.alpha_e, p.r_alpha) : __fdiv_rn(num, p.alpha_e);
    if (clamp) x0 = __fdiv_rn(clamp_sym(x0, thr), thr);   // dynamic thresholding
    return x0;
  }
  return eps;
}

// LIN1 / DIFF2 (common.cuh: update_value) followed by the separately rounded noise term
__device__ __forceinline__ float update_rn(const KParams& p, int form, float x, float T0, float m1, float cn, float z) {
  float o;
  if (form == DPM_FORM_DIFF2) {
    const float D = __fmul_rn(p.w0, __fsub_rn(T0, m1));
    const float lead = p.c0_on_old ? m1 : T0;
    o = __fadd_rn(__fadd_rn(__fmul_rn(p.a, x), __fmul_rn(p.c0, lead)), __fmul_rn(p.c1, D));
  } else {
    o = __fadd_rn(__fmul_rn(p.a, x), __fmul_rn(p.c0, T0));
  }
  return __fadd_rn(o, __fmul_rn(cn, z));
}

// z of element li (scalar path): one Philox call per element
__device__ __forceinline__ float noise_at(const SdeParams& s, uint64_t li) {
  if (s.noise != nullptr) return s.noise[li];
  const uint64_t r = li / s.G, idx = li - r * s.G;
  curandStatePhilox4_32_10_t st;
  curand_init(s.seed, idx, s.offset + 4 * (r >> 2), &st);
  const float4 v = curand_normal4(&st);
  switch (r & 3) {
    case 0: return v.x;
    case 1: return v.y;
    case 2: return v.z;
    default: return v.w;
  }
}

// one element, any dtype mix / alignment (scalar kernel, and the ragged last packet of the packet kernel)
__device__ __forceinline__ void sde_elem(const SdeParams& s, uint64_t i, float z) {
  const KParams& p = s.k;
  const int sd = p.state_dtype, md = p.model_dtype;
  const float x = load_any(p.x, sd, i);
  const float m1 = p.form == DPM_FORM_DIFF2 ? load_any(p.m1, sd, i) : 0.f;
  float T0;
  if (p.n_model > 0) {
    const float xe = p.use_xe ? (p.xe_is_x ? x : load_any(p.xe, sd, i)) : 0.f;
    const float ec = load_any(p.ec, md, i);
    const float eu = p.n_model == 2 ? load_any(p.eu, md, i) : 0.f;
    const bool clamp = p.thr != nullptr;
    const float thr = clamp ? p.thr[i / p.per_sample] : 1.f;
    const float mv = model_rn(p, p.n_model, xe, ec, eu, thr, clamp);
    T0 = round_any(sd, mv);
    if (p.m_out) store_any(p.m_out, sd, i, mv);
  } else {
    T0 = load_any(p.m0, sd, i);
  }
  const float o = update_rn(p, p.form, x, T0, m1, s.cn, z);
  store_any(p.out, sd, i, o);
  if (p.out2) store_any(p.out2, sd, i, o);
}

static __device__ __noinline__ void ragged_tail(const SdeParams& s, uint64_t e) {
  for (uint64_t i = e; i < s.k.n; ++i) sde_elem(s, i, noise_at(s, i));
}

__global__ void __launch_bounds__(kSdeThreads) k_sde_scalar(const __grid_constant__ SdeParams s) {
  pdl_trigger();
  pdl_wait();
  const uint64_t n = s.k.n;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    sde_elem(s, i, noise_at(s, i));
}

// ---- packet kernel ----------------------------------------------------------------------------------------------
// TE / TS: model / state storage types, NE: raw network outputs (0 = pure update on m0), FORM: LIN1 or DIFF2.
// 16-bit state: the loads of all four packets are issued before the Philox calls, whose ALU work then covers their
// latency; fp32 state (twice the registers per packet) loads packet by packet.
template <typename TE, typename TS, int NE, int FORM>
__global__ void __launch_bounds__(kSdeThreads) k_sde_packet(const __grid_constant__ SdeParams s) {
  constexpr bool kPre = Traits<TS>::kBytes == 2;
  constexpr int kSlots = kPre ? 4 : 1;
  const KParams& p = s.k;
  const TS* __restrict__ gx = static_cast<const TS*>(p.x);
  const TS* __restrict__ gxe = static_cast<const TS*>(p.xe);
  const TS* __restrict__ gm0 = static_cast<const TS*>(p.m0);
  const TS* __restrict__ gm1 = static_cast<const TS*>(p.m1);
  const TE* __restrict__ gec = static_cast<const TE*>(p.ec);
  const TE* __restrict__ geu = static_cast<const TE*>(p.eu);
  TS* __restrict__ gmo = static_cast<TS*>(p.m_out);
  TS* __restrict__ go = static_cast<TS*>(p.out);
  TS* __restrict__ go2 = static_cast<TS*>(p.out2);
  const uint64_t n = p.n, G = s.G, G8 = s.G / 8;
  const bool sep_xe = NE > 0 && p.use_xe && !p.xe_is_x;
  const bool clamp = NE > 0 && p.thr != nullptr;
  pdl_trigger();
  pdl_wait();

  for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < s.items; w += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t k = w / G8, v0 = (w - k * G8) * 8;
    const uint64_t base = v0 + G * 4 * k;   // element of lane ii: base + G*ii

    Raw<TS> rx[kSlots], rxe[kSlots], rm[kSlots], rm1[kSlots];
    Raw<TE> rec[kSlots], reu[kSlots];
    auto load = [&](int slot, uint64_t e) {
      ldg_pk(rx[slot], gx + e);
      if (NE > 0) {
        ldg_pk(rec[slot], gec + e);
        if (NE == 2) ldg_pk(reu[slot], geu + e);
        if (sep_xe) ldg_pk(rxe[slot], gxe + e);
      } else {
        ldg_pk(rm[slot], gm0 + e);
      }
      if (FORM == DPM_FORM_DIFF2) ldg_pk(rm1[slot], gm1 + e);
    };
    if (kPre) {
#pragma unroll
      for (int ii = 0; ii < 4; ++ii) {
        const uint64_t e = base + G * ii;
        if (e + kPacket <= n) load(kPre ? ii : 0, e);
      }
    }

    // z[ii][j]: lane ii of virtual thread v0 + j
    float z[4][8];
    if (s.noise == nullptr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        curandStatePhilox4_32_10_t st;
        curand_init(s.seed, v0 + j, s.offset + 4 * k, &st);
        const float4 r = curand_normal4(&st);
        z[0][j] = r.x; z[1][j] = r.y; z[2][j] = r.z; z[3][j] = r.w;
      }
    }

#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const uint64_t e = base + G * ii;
      if (e + kPacket > n) {
        // the ragged last packet of the tensor (one per launch): element by element, its noise drawn again
        if (e < n) ragged_tail(s, e);
        continue;
      }
      const int slot = kPre ? ii : 0;
      if (!kPre) load(slot, e);
      float fz[8];
      if (s.noise != nullptr) {
        Raw<float> rz;
        ldg_pk(rz, s.noise + e);
        unpack(rz, fz);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) fz[j] = z[ii][j];
      }
      float fx[8], fT[8], fm1[8], fo[8];
      unpack(rx[slot], fx);
      if (FORM == DPM_FORM_DIFF2) unpack(rm1[slot], fm1);
      if (NE > 0) {
        float fec[8], feu[8], fxe[8], thr8[8];
        unpack(rec[slot], fec);
        if (NE == 2) unpack(reu[slot], feu);
        if (sep_xe) unpack(rxe[slot], fxe);
        if (clamp) {
          if (p.pk_per_sample != 0) {
            const float t = __ldg(p.thr + (e / kPacket) / p.pk_per_sample);
#pragma unroll
            for (int j = 0; j < 8; ++j) thr8[j] = t;
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) thr8[j] = __ldg(p.thr + (e + j) / p.per_sample);
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          fT[j] = model_rn(p, NE, sep_xe ? fxe[j] : fx[j], fec[j], NE == 2 ? feu[j] : 0.f, clamp ? thr8[j] : 1.f, clamp);
        Raw<TS> rmo;
        round_pack(rmo, fT);   // NEW as it reads back from storage
        if (gmo != nullptr) stg_pk(gmo + e, rmo);
      } else {
        unpack(rm[slot], fT);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) fo[j] = update_rn(p, FORM, fx[j], fT[j], FORM == DPM_FORM_DIFF2 ? fm1[j] : 0.f, s.cn, fz[j]);
      Raw<TS> ro;
      pack(ro, fo);
      stg_pk(go + e, ro);
      if (go2 != nullptr) stg_pk(go2 + e, ro);
    }
  }
}

typedef void (*SdeKernel)(const SdeParams);

template <typename TE, typename TS, int NE>
static SdeKernel pick_sde_form(int form) {
  return form == DPM_FORM_DIFF2 ? k_sde_packet<TE, TS, NE, DPM_FORM_DIFF2> : k_sde_packet<TE, TS, NE, DPM_FORM_LIN1>;
}
template <typename TE, typename TS>
static SdeKernel pick_sde_ne(int ne, int form) {
  return ne == 2 ? pick_sde_form<TE, TS, 2>(form) : pick_sde_form<TE, TS, 1>(form);
}
static SdeKernel pick_sde(int md, int sd, int ne, int form) {
  if (ne == 0) {
    switch (sd) {
      case DPM_F32: return pick_sde_form<float, float, 0>(form);
      case DPM_BF16: return pick_sde_form<__nv_bfloat16, __nv_bfloat16, 0>(form);
      case DPM_F16: return pick_sde_form<__half, __half, 0>(form);
    }
    return nullptr;
  }
  if (md == DPM_F32 && sd == DPM_F32) return pick_sde_ne<float, float>(ne, form);
  if (md == DPM_BF16 && sd == DPM_BF16) return pick_sde_ne<__nv_bfloat16, __nv_bfloat16>(ne, form);
  if (md == DPM_F16 && sd == DPM_F16) return pick_sde_ne<__half, __half>(ne, form);
  if (md == DPM_BF16 && sd == DPM_F32) return pick_sde_ne<__nv_bfloat16, float>(ne, form);
  if (md == DPM_F16 && sd == DPM_F32) return pick_sde_ne<__half, float>(ne, form);
  return nullptr;   // other mixes: scalar kernel
}

// vec_ok: every tensor the launch touches (noise included) is aligned for packet access
int launch_sde_step(const KParams& p, bool vec_ok, float cn, const float* noise, uint64_t seed, uint64_t offset,
                    cudaStream_t stream) {
  if (p.n == 0) return 0;
  SdeParams s;
  memset(&s, 0, sizeof(s));
  s.k = p;
  s.noise = noise; s.seed = seed; s.offset = offset; s.cn = cn;
  uint32_t vgrid = 0;
  uint64_t unused = 0;
  philox_policy(p.n, &vgrid, &unused);
  s.G = (uint64_t)vgrid * kPhiloxBlockV;
  s.items = (p.n + 4 * s.G - 1) / (4 * s.G) * (s.G / 8);
  SdeKernel k = vec_ok ? pick_sde(p.model_dtype, p.state_dtype, p.n_model, p.form) : nullptr;
  if (k == nullptr) k = k_sde_scalar;
  const uint64_t work = k != k_sde_scalar ? s.items : p.n;
  const uint64_t blocks = (work + kSdeThreads - 1) / kSdeThreads;
  const uint64_t cap = (uint64_t)sm_count() * 8;
  const uint32_t grid = (uint32_t)(blocks < cap ? blocks : cap);
  cudaError_t le = launch_pdl(k, grid, (unsigned)kSdeThreads, 0, stream, s);
  if (le != cudaSuccess) { set_error("sde step launch failed: %s", cudaGetErrorString(le)); cudaGetLastError(); return (int)le; }
  count_launch();
  return 0;
}

}  // namespace dpm
