"""Tensor-level front end of the C-ABI: one call = one fused kernel launch on the current stream.

`StepArgs` mirrors `struct dpm_step_desc` (include/dpm_solver_b200.h) with torch tensors in place
of raw pointers. The only executor shipped is `CudaBackend`, which hands device pointers to
libdpmsolver_b200.so; it refuses CPU tensors (there is no CPU or PyTorch fallback).  Tests may
install another executor with `set_backend()` to exercise the host-side logic without a GPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (DPM_BF16, DPM_F16, DPM_F32, FORM_DIFF2, FORM_LIN1, FORM_LIN2, FORM_LIN3,
                   FORM_MS3, FORM_NONE, FORM_SS3T, PARAM_NOISE, StepDesc)

_DTYPE_CODE = {torch.float32: DPM_F32, torch.bfloat16: DPM_BF16, torch.float16: DPM_F16}
SUPPORTED_DTYPES = tuple(_DTYPE_CODE)


@dataclass
class StepArgs:
    """One fused solver step (see dpm_step_desc for the meaning of every field)."""
    form: int = FORM_NONE
    n_model: int = 0
    x: Optional[torch.Tensor] = None
    xe: Optional[torch.Tensor] = None
    m0: Optional[torch.Tensor] = None
    m1: Optional[torch.Tensor] = None
    m2: Optional[torch.Tensor] = None
    e_cond: Optional[torch.Tensor] = None
    e_uncond: Optional[torch.Tensor] = None
    thr: Optional[torch.Tensor] = None
    per_sample: int = 0
    param: int = PARAM_NOISE
    predict_x0: bool = False
    c0_on_old: bool = False
    guidance: float = 1.0
    alpha_e: float = 1.0
    sigma_e: float = 0.0
    a: float = 0.0
    c0: float = 0.0
    c1: float = 0.0
    c2: float = 0.0
    w0: float = 0.0
    w1: float = 0.0
    w2: float = 0.0
    w3: float = 0.0
    w4: float = 0.0
    want_m_out: bool = False          # materialise the computed model value (n_model >= 1)
    state_dtype: Optional[torch.dtype] = None  # dtype of x/xe/m*/outputs; default: from tensors
    out: Optional[torch.Tensor] = None     # optional preallocated outputs
    out2: Optional[torch.Tensor] = None    # optional second copy of x_t (doubled CFG batch)
    m_out: Optional[torch.Tensor] = None
    raw_round: int = 0                # reference-rounding mode (dpm_step_desc.raw_round); 0 = off
    coef_dev: Optional[torch.Tensor] = None   # 16 fp32 on the device: the launch reads its scalars there (dev_coef)

    def state_tensors(self):
        return [t for t in (self.x, self.xe, self.m0, self.m1, self.m2) if t is not None]

    def model_tensors(self):
        return [t for t in (self.e_cond, self.e_uncond) if t is not None]

    def reference_tensor(self) -> torch.Tensor:
        for t in (self.x, self.xe, self.e_cond, self.m0):
            if t is not None:
                return t
        raise ValueError("StepArgs without tensors")


def check_generator(generator, device) -> None:
    """Raise ValueError unless `generator` (None = the device's default generator) draws on `device`."""
    if generator is None:
        return
    if not isinstance(generator, torch.Generator):
        raise ValueError(f"dpm_solver_b200: `generator` must be a torch.Generator, got {type(generator).__name__}")
    gd, device = generator.device, torch.device(device)
    g_index = gd.index if gd.index is not None or gd.type != "cuda" else torch.cuda.current_device()
    d_index = device.index if device.index is not None or device.type != "cuda" else torch.cuda.current_device()
    if gd.type != device.type or g_index != d_index:
        raise ValueError(f"dpm_solver_b200: the generator is on {gd}, the tensors on {device}")


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
if _raw_stream is None:  # older torch: go through the Stream object
    def _raw_stream(idx):
        return torch.cuda.current_stream(idx).cuda_stream


class CudaBackend:
    """Executes StepArgs through libdpmsolver_b200.so."""

    name = "cuda-sm100a"

    def __init__(self):
        self._lib = _lib.lib()  # fail loudly at construction if the .so is missing

    # -- helpers --------------------------------------------------------------------------
    @staticmethod
    def _layout(t: torch.Tensor) -> Optional[str]:
        """'c' (row-major dense), 'cl' (channels_last dense) or None (needs a copy). Element-wise
        kernels only need every operand to share ONE dense layout: the storage is then a flat array."""
        if t.is_contiguous():
            return "c"
        if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
            return "cl"
        if t.dim() == 5 and t.is_contiguous(memory_format=torch.channels_last_3d):
            return "cl"
        return None

    @staticmethod
    def _check(t: torch.Tensor, what: str, dev, numel: int, dtype=None, layout: str = "c") -> torch.Tensor:
        if not t.is_cuda:
            raise RuntimeError(f"dpm_solver_b200: `{what}` is on {t.device}; this library is CUDA-only "
                               "(no CPU fallback)")
        if t.device != dev:
            raise RuntimeError(f"dpm_solver_b200: `{what}` is on {t.device}, expected {dev}")
        if t.numel() != numel:
            raise ValueError(f"dpm_solver_b200: `{what}` has {t.numel()} elements, expected {numel}")
        if dtype is not None and t.dtype != dtype:
            raise TypeError(f"dpm_solver_b200: `{what}` is {t.dtype}, expected {dtype}")
        if t.dtype not in _DTYPE_CODE:
            raise TypeError(f"dpm_solver_b200: unsupported dtype {t.dtype} for `{what}`")
        if layout == "cl":
            if t.dim() in (4, 5) and t.is_contiguous(memory_format=torch.channels_last if t.dim() == 4 else torch.channels_last_3d):
                return t
            return t.contiguous(memory_format=torch.channels_last if t.dim() == 4 else torch.channels_last_3d) \
                if t.dim() in (4, 5) else t.contiguous()
        return t if t.is_contiguous() else t.contiguous()

    def _fill(self, a: StepArgs):
        ref = a.reference_tensor()
        dev, n = ref.device, ref.numel()
        sdt = a.state_dtype
        if sdt is None:
            st = a.state_tensors()
            sdt = st[0].dtype if st else a.e_cond.dtype
        # channels_last networks hand over channels_last tensors: keep that layout end to end
        layout = self._layout(ref) or "c"
        for t in (a.out, a.m_out, a.out2):
            if t is not None and self._layout(t) != layout:
                layout = "c"   # preallocated row-major outputs: bring the inputs to that layout
        keep = []  # keep converted copies alive until after the launch
        d = StepDesc()

        def ptr(t, what, dtype):
            if t is None:
                return None
            t = self._check(t, what, dev, n, dtype, layout)
            keep.append(t)
            return t.data_ptr()

        d.x = ptr(a.x, "x", sdt)
        d.xe = ptr(a.xe, "xe", sdt)
        d.m0 = ptr(a.m0, "m0", sdt)
        d.m1 = ptr(a.m1, "m1", sdt)
        d.m2 = ptr(a.m2, "m2", sdt)
        mdt = a.e_cond.dtype if a.e_cond is not None else sdt
        d.e_cond = ptr(a.e_cond, "e_cond", mdt)
        d.e_uncond = ptr(a.e_uncond, "e_uncond", mdt)
        if a.thr is not None:
            if not a.thr.is_cuda or a.thr.dtype != torch.float32 or not a.thr.is_contiguous():
                raise TypeError("dpm_solver_b200: `thr` must be a contiguous fp32 CUDA tensor")
            if a.per_sample <= 0 or n % a.per_sample or a.thr.numel() != n // a.per_sample:
                raise ValueError("dpm_solver_b200: `thr` needs one value per sample")
            keep.append(a.thr)
            d.thr = a.thr.data_ptr()
        d.n = n
        d.per_sample = a.per_sample
        d.state_dtype = _DTYPE_CODE[sdt]
        d.model_dtype = _DTYPE_CODE[mdt]
        d.form, d.n_model, d.param = a.form, a.n_model, a.param
        d.predict_x0, d.c0_on_old = int(a.predict_x0), int(a.c0_on_old)
        d.raw_round = int(a.raw_round)
        d.guidance, d.alpha_e, d.sigma_e = a.guidance, a.alpha_e, a.sigma_e
        d.a, d.c0, d.c1, d.c2 = a.a, a.c0, a.c1, a.c2
        d.w0, d.w1, d.w2, d.w3, d.w4 = a.w0, a.w1, a.w2, a.w3, a.w4
        if a.coef_dev is not None:
            cd = a.coef_dev
            if not cd.is_cuda or cd.dtype != torch.float32 or cd.numel() < 16 or not cd.is_contiguous() or cd.device != dev:
                raise TypeError("dpm_solver_b200: `coef_dev` must be 16 contiguous fp32 values on the tensors' device")
            keep.append(cd)
            d.dev_coef = cd.data_ptr()
        return d, keep, ref, sdt, layout

    def _new_like(self, ref, sdt, layout):
        if layout == "cl":
            return torch.empty(ref.shape, dtype=sdt, device=ref.device,
                               memory_format=torch.channels_last if ref.dim() == 4 else torch.channels_last_3d)
        return torch.empty(ref.shape, dtype=sdt, device=ref.device)

    # -- API -----------------------------------------------------------------------------
    def step(self, a: StepArgs) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """Launch one fused step. Returns (m_out, out); either may be None."""
        d, keep, ref, sdt, layout = self._fill(a)
        m_out, out = self._outputs(a, d, ref, sdt, layout)
        self._launch(ref.device, self._lib.dpm_step, C.byref(d))
        return m_out, out

    def _outputs(self, a: StepArgs, d, ref, sdt, layout):
        """Allocate (or check the preallocated) m_out / out / out2 of a step and point the descriptor at them."""
        m_out = out = None
        if a.n_model > 0 and (a.want_m_out or a.form == FORM_NONE):
            m_out = a.m_out if a.m_out is not None else self._new_like(ref, sdt, layout)
            self._check(m_out, "m_out", ref.device, ref.numel(), sdt)
            if self._layout(m_out) != layout:
                raise ValueError("dpm_solver_b200: preallocated m_out must be dense and laid out like the inputs")
            d.m_out = m_out.data_ptr()
        if a.form != FORM_NONE:
            out = a.out if a.out is not None else self._new_like(ref, sdt, layout)
            self._check(out, "out", ref.device, ref.numel(), sdt)
            if self._layout(out) != layout:
                raise ValueError("dpm_solver_b200: preallocated out must be dense and laid out like the inputs")
            d.out = out.data_ptr()
            if a.out2 is not None:
                self._check(a.out2, "out2", ref.device, ref.numel(), sdt)
                if self._layout(a.out2) != layout:      # dense, laid out like `out` (a channels_last half of the
                    raise ValueError("dpm_solver_b200: out2 must be dense and laid out like out")   # doubled CFG batch is)
                d.out2 = a.out2.data_ptr()
        return m_out, out

    def sde_step(self, a: StepArgs, noise_scale: float, generator=None, noise: Optional[torch.Tensor] = None):
        """One stochastic SDE-DPM-Solver step (LIN1 / DIFF2): the step `step(a)` computes plus noise_scale * z, one
        launch (csrc/step_sde.cu). z is `torch.randn_like(x, dtype=torch.float32)` for the state of `generator` (None:
        the default generator of the tensors' device), generated in registers, and the generator is advanced exactly
        as that randn would advance it; or, with `noise=`, that fp32 tensor. Under CUDA-graph capture the noise is
        drawn by torch inside the capture (replays then draw fresh noise) and read from memory; only the default
        generator can be used there. Returns (m_out, out)."""
        if a.form not in (FORM_LIN1, FORM_DIFF2):
            raise ValueError("dpm_solver_b200: the SDE step serves the LIN1 and DIFF2 forms only")
        d, keep, ref, sdt, layout = self._fill(a)
        dev = ref.device
        check_generator(generator, dev)
        m_out, out = self._outputs(a, d, ref, sdt, layout)
        seed = offset = 0
        if noise is None and torch.cuda.is_current_stream_capturing():
            # a (seed, offset) read on the host would be frozen into the graph: let torch draw the noise inside the
            # capture (its default generator is capture-aware) and read it from memory
            if generator is not None and generator is not torch.cuda.default_generators[dev.index]:
                raise RuntimeError("dpm_solver_b200: only the default CUDA generator can draw SDE noise under "
                                   "CUDA-graph capture")
            noise = self._new_like(ref, torch.float32, layout).normal_()
        if noise is not None:
            noise = self._check(noise, "noise", dev, ref.numel(), torch.float32, layout)
            keep.append(noise)
            if self._layout(noise) != layout:
                raise ValueError("dpm_solver_b200: `noise` must be dense and laid out like the inputs")
            nptr = noise.data_ptr()
        else:
            nptr = None
            with torch.cuda.device(dev):
                seed, offset = self._philox_state(dev, ref.numel(), self._lib, generator)
        self._launch(dev, self._lib.dpm_sde_step, C.byref(d), C.c_float(noise_scale), C.c_void_p(nptr),
                     C.c_uint64(seed), C.c_uint64(offset))
        return m_out, out

    def _launch(self, device, fn, *args):
        """Call a C-ABI entry on torch's current stream of `device` (device guard only if needed)."""
        idx = device.index
        if torch.cuda.current_device() == idx:
            rc = fn(*args, C.c_void_p(_raw_stream(idx)))
        else:
            with torch.cuda.device(device):
                rc = fn(*args, C.c_void_p(_raw_stream(idx)))
        if rc != 0:
            _lib.check(rc)

    def dynamic_threshold(self, a: StepArgs, q: float, max_val: float, return_stats: bool = False):
        """Per-sample s_b = max(quantile(|x0_b|, q), max_val) -> fp32 [B].
        return_stats=True also returns the pipeline's per-sample header words (int32 [B, 8]:
        lo key, hi key, #below, #inside, path (1 bracket / 2 exact fallback), ...) for diagnostics."""
        d, keep, ref, _, _ = self._fill(a)
        if a.per_sample <= 0 or ref.numel() % a.per_sample:
            raise ValueError("dpm_solver_b200: per_sample must divide numel")
        nb = ref.numel() // a.per_sample
        s = torch.empty(nb, dtype=torch.float32, device=ref.device)
        ws_bytes = int(self._lib.dpm_dynamic_threshold_workspace(nb, a.per_sample))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=ref.device) if ws_bytes else None
        self._launch(ref.device, self._lib.dpm_dynamic_threshold, C.c_void_p(s.data_ptr()), C.byref(d),
                     C.c_float(q), C.c_float(max_val), C.c_void_p(ws.data_ptr() if ws is not None else None),
                     C.c_size_t(ws_bytes))
        if return_stats:
            hdr = ws[:nb * 32].view(torch.int32).reshape(nb, 8).clone() if ws is not None else None
            return s, hdr
        return s

    def error_norm(self, x_higher, x_lower, x_prev, atol: float, rtol: float, out=None) -> torch.Tensor:
        """E of dpm_solver_adaptive (:999-1001) as a device fp32 tensor of shape (1,)."""
        n, dev = x_higher.numel(), x_higher.device
        ts = [self._check(t, w, dev, n, x_higher.dtype) for t, w in ((x_higher, "x_higher"), (x_lower, "x_lower"), (x_prev, "x_prev"))]
        per_sample = n // x_higher.shape[0]
        if out is None:
            out = torch.empty(1, dtype=torch.float32, device=dev)
        ws_bytes = int(self._lib.dpm_adaptive_error_workspace(n, per_sample))
        ws = torch.empty(max(ws_bytes, 4), dtype=torch.uint8, device=dev)
        self._launch(dev, self._lib.dpm_adaptive_error, C.c_void_p(out.data_ptr()), C.c_void_p(ts[0].data_ptr()),
                     C.c_void_p(ts[1].data_ptr()), C.c_void_p(ts[2].data_ptr()), C.c_float(atol), C.c_float(rtol),
                     C.c_uint64(per_sample), C.c_uint64(n), C.c_int(_DTYPE_CODE[x_higher.dtype]),
                     C.c_void_p(ws.data_ptr()), C.c_size_t(ws_bytes))
        return out

    def duplicate(self, x: torch.Tensor) -> torch.Tensor:
        """torch.cat([x] * 2) (model_wrapper :326) -- one read, two bulk writes; layout of x kept."""
        if x.dtype not in _DTYPE_CODE:
            return torch.cat([x] * 2)
        layout = self._layout(x)
        if layout is None:
            x, layout = x.contiguous(), "c"
        shape = (2 * x.shape[0],) + tuple(x.shape[1:])
        if layout == "cl":
            out = torch.empty(shape, dtype=x.dtype, device=x.device,
                              memory_format=torch.channels_last if x.dim() == 4 else torch.channels_last_3d)
        else:
            out = torch.empty(shape, dtype=x.dtype, device=x.device)
        self._check(x, "x", x.device, x.numel(), layout=layout)
        self._launch(x.device, self._lib.dpm_duplicate, C.c_void_p(out.data_ptr()), C.c_void_p(x.data_ptr()),
                     C.c_uint64(x.numel()), C.c_int(_DTYPE_CODE[x.dtype]))
        return out

    def adaptive_controller(self, ns, device, **kw) -> "AdaptiveController":
        """Device-resident step-size controller of dpm_solver_adaptive (csrc/adaptive_ctl.cu)."""
        return AdaptiveController(self, ns, device, **kw)

    # -- noise drawn inside the kernel (torch.randn-compatible Philox; csrc/philox.cu) ----------------------
    @staticmethod
    def _philox_state(device, numel: int, lib, generator=None):
        """(seed, offset) of the torch CUDA generator for a randn of `numel` elements, advancing it exactly as
        ATen's normal_ kernel would (so later torch RNG calls see the state they would have seen)."""
        gen = generator if generator is not None else torch.cuda.default_generators[device.index]
        grid, inc = C.c_uint32(0), C.c_uint64(0)
        _lib.check(lib.dpm_philox_policy(C.c_uint64(numel), C.byref(grid), C.byref(inc)))
        seed, offset = gen.initial_seed(), gen.get_offset()
        gen.set_offset(offset + inc.value)
        return seed, offset

    def add_noise_philox(self, x: torch.Tensor, alphas, sigmas, out_dtype, generator=None) -> torch.Tensor:
        """[T, *x.shape] = alpha_i * x + sigma_i * randn, the noise generated in registers (reference :1023-1026)."""
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("dpm_solver_b200: in-kernel noise reads the generator state on the host; pass `noise=` under CUDA-graph capture")
        x = self._check(x, "x", x.device, x.numel())
        T = len(alphas)
        out = torch.empty((T,) + tuple(x.shape), dtype=out_dtype, device=x.device)
        with torch.cuda.device(x.device):
            seed, offset = self._philox_state(x.device, T * x.numel(), self._lib, generator)
        fa = (C.c_float * T)(*alphas)
        fs = (C.c_float * T)(*sigmas)
        self._launch(x.device, self._lib.dpm_add_noise_philox, C.c_void_p(out.data_ptr()), C.c_void_p(x.data_ptr()),
                     C.c_uint64(x.numel()), C.c_int(T), fa, fs, C.c_uint64(seed), C.c_uint64(offset),
                     C.c_int(_DTYPE_CODE[x.dtype]), C.c_int(_DTYPE_CODE[out_dtype]))
        return out

    def diffedit_corrector(self, x, x0, mask, alpha: float, sigma: float, generator=None) -> torch.Tensor:
        """x*mask + (1 - mask)*(alpha*x0 + sigma*randn_like(x0)) in one launch (diffedit_inpaint.ipynb corrector_fn)."""
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("dpm_solver_b200: in-kernel noise reads the generator state on the host; not capturable")
        n = x.numel()
        x = self._check(x, "x", x.device, n)
        x0 = self._check(x0, "x0", x.device, n, x.dtype)
        if mask.dtype != torch.float32 or not mask.is_contiguous() or n % max(mask.numel(), 1) \
                or tuple(mask.shape) != tuple(x.shape[x.dim() - mask.dim():]):
            mask = mask.to(torch.float32).expand(x.shape).contiguous()        # any other broadcast: materialise
        if mask.device != x.device:
            raise RuntimeError("dpm_solver_b200: `mask` must live on the device of x")
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            seed, offset = self._philox_state(x.device, n, self._lib, generator)
        self._launch(x.device, self._lib.dpm_diffedit_corrector, C.c_void_p(out.data_ptr()), C.c_void_p(x.data_ptr()),
                     C.c_void_p(x0.data_ptr()), C.c_void_p(mask.data_ptr()), C.c_uint64(mask.numel()), C.c_uint64(n),
                     C.c_float(alpha), C.c_float(sigma), C.c_uint64(seed), C.c_uint64(offset), C.c_int(_DTYPE_CODE[x.dtype]))
        return out

    def prepare(self, a: StepArgs) -> Optional["PreparedStep"]:
        """Freeze the descriptor of a launch whose scalars will not change (one step of a cached coefficient plan):
        later launches of the same step only patch the tensor pointers. None if the launch is not eligible."""
        return PreparedStep.build(self, a)

    def launch_count(self) -> int:
        return int(self._lib.dpm_launch_count())

    def set_tuning(self, variant: int = 2, threads: int = 0, ctas_per_sm: int = 0) -> None:
        _lib.check(self._lib.dpm_set_tuning(variant, threads, ctas_per_sm))


class AdaptiveController:
    """State, coefficient blocks and time labels of dpm_solver_adaptive (:956-1010) in device memory, plus the three
    tiny kernels that advance them (dpm_adaptive_init / _plan / _decide) and the conditional commit
    (dpm_select_copy). `read()` is the only host synchronisation."""

    SUPPORTED = ("discrete", "linear")

    def __init__(self, be: "CudaBackend", ns, device, order: int, predict_x0: bool, taylor: bool, t_0: float,
                 theta: float, t_err: float, discrete_input: bool):
        if ns.schedule not in self.SUPPORTED:
            raise ValueError("the device controller supports the 'discrete' and 'linear' schedules")
        self.be, self.dev = be, torch.device(device)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.state = torch.zeros(16, **f32)
        self.coef = torch.zeros(4, 16, **f32)
        self.times = torch.zeros(6, **f32)
        self.E = torch.zeros(1, **f32)
        c = self.ctl = _lib.AdaptiveCtl()
        self._keep = []
        if ns.schedule == "discrete":
            tabs = ns._table(self.dev)[:4]
            self._keep = [t.to(torch.float32).contiguous() for t in tabs]
            c.schedule_kind, c.table_len = 0, self._keep[0].numel()
            c.t_array, c.log_alpha_array, c.log_alpha_flipped, c.t_flipped = (t.data_ptr() for t in self._keep)
            c.inv_total_N = 1. / ns.total_N
        else:
            c.schedule_kind, c.table_len = 1, 0
            c.beta_0, c.beta_1_minus_beta_0 = ns.beta_0, ns.beta_1 - ns.beta_0
            c.inv_total_N = 1. / ns.total_N
        c.discrete_time_input = int(bool(discrete_input))
        c.order, c.predict_x0, c.taylor = order, int(bool(predict_x0)), int(bool(taylor))
        c.t_0, c.theta, c.t_err = t_0, theta, t_err
        c.state, c.coef, c.times, c.error = (t.data_ptr() for t in (self.state, self.coef, self.times, self.E))
        self._ref = C.byref(c)

    def init(self, t_T: float, h_init: float) -> None:
        self.be._launch(self.dev, self.be._lib.dpm_adaptive_init, self._ref, C.c_float(t_T), C.c_float(h_init))

    def plan(self) -> None:
        self.be._launch(self.dev, self.be._lib.dpm_adaptive_plan, self._ref)

    def decide(self) -> None:
        self.be._launch(self.dev, self.be._lib.dpm_adaptive_decide, self._ref)

    def select_copy(self, dst: torch.Tensor, src: torch.Tensor) -> None:
        """dst <- src iff the last decide() accepted the step."""
        if dst.shape != src.shape or dst.dtype != src.dtype or not dst.is_contiguous() or not src.is_contiguous():
            raise ValueError("select_copy: dense tensors of one shape and dtype")
        self.be._launch(self.dev, self.be._lib.dpm_select_copy, C.c_void_p(dst.data_ptr()), C.c_void_p(src.data_ptr()),
                        C.c_void_p(self.state.data_ptr()), C.c_uint64(dst.numel() * dst.element_size()))

    def block(self, i: int) -> torch.Tensor:
        return self.coef[i]

    def time(self, j: int) -> torch.Tensor:
        return self.times[j:j + 1]

    def input_time(self, j: int) -> torch.Tensor:
        return self.times[3 + j:4 + j]

    def read(self):
        """(done, nfe, iterations): the one device->host read of a chunk."""
        st = self.state.cpu().view(torch.int32)
        return int(st[6]), int(st[5]), int(st[8])


class PreparedStep:
    """One step of a cached coefficient plan, ready to launch: a filled `dpm_step_desc` whose scalar fields are final.
    `launch()` validates the tensors of this call with a handful of attribute reads (dtype, size, density, device),
    patches the pointers, allocates the outputs and calls the C-ABI -- the per-step host path of a steady-state
    sample() loop (tools/host_overhead.py). Anything unusual (other layout, dtype, device, size) returns None and the
    caller takes the general path (`CudaBackend.step`)."""

    __slots__ = ("be", "d", "ref_d", "fn", "n", "dev", "dev_index", "sdt", "mdt", "shape", "shape2", "need_out",
                 "need_m", "fields", "dup", "ptrs", "esize")

    ORDER = ("x", "xe", "m0", "m1", "m2", "e_cond", "e_uncond")     # launch() takes its tensors in this order
    # index of every pointer field inside struct dpm_step_desc (its first 11 members are pointers)
    _PTR = {"x": 0, "xe": 1, "m0": 2, "m1": 3, "m2": 4, "m_out": 5, "out": 6, "out2": 7, "e_cond": 8, "e_uncond": 9}

    @staticmethod
    def build(be: "CudaBackend", a: StepArgs) -> Optional["PreparedStep"]:
        if a.thr is not None or a.raw_round or a.out is not None and a.out2 is None:
            return None
        ref = a.reference_tensor()
        if not ref.is_contiguous():
            return None
        for t in a.state_tensors() + a.model_tensors():
            if not t.is_contiguous() or t.device != ref.device:
                return None
        d, keep, ref, sdt, layout = be._fill(a)
        if layout != "c":
            return None
        self = PreparedStep()
        self.be, self.d, self.ref_d, self.fn = be, d, C.byref(d), be._lib.dpm_step
        self.n, self.dev, self.dev_index = ref.numel(), ref.device, ref.device.index
        self.sdt = sdt
        self.mdt = a.e_cond.dtype if a.e_cond is not None else sdt
        self.shape = tuple(ref.shape)
        self.shape2 = (2 * self.shape[0],) + self.shape[1:]
        self.esize = torch.empty((), dtype=sdt).element_size()
        # the descriptor's pointer members as a uint64 array: patching one is a numpy scalar store, not a ctypes setattr
        import numpy as np
        self.ptrs = np.frombuffer((C.c_char * C.sizeof(d)).from_buffer(d), dtype=np.uint64, count=11)
        self.need_out = a.form != FORM_NONE
        self.need_m = a.n_model > 0 and (a.want_m_out or a.form == FORM_NONE)
        self.dup = a.out2 is not None
        # (descriptor field, StepArgs attribute, expected dtype) of every input tensor this launch reads
        # (pointer slot, position in launch()'s tensor tuple, expected dtype) of every input this launch reads
        self.fields = tuple((self._PTR[name], pos, self.mdt if name in ("e_cond", "e_uncond") else sdt)
                            for pos, name in enumerate(self.ORDER) if getattr(a, name) is not None)
        return self

    def launch(self, tensors: tuple):
        """tensors: (x, xe, m0, m1, m2, e_cond, e_uncond) (`ORDER`; entries the frozen launch does not read are
        ignored). Returns (m_out, out, x_in) -- x_in is the doubled CFG batch when the step was prepared with a second
        output copy -- or None when a tensor does not look like the ones the step was prepared for."""
        n, dev, idx, ptrs = self.n, self.dev, self.dev_index, self.ptrs
        for f, pos, dt in self.fields:
            t = tensors[pos]
            if t is None or t.dtype is not dt or t.numel() != n or not t.is_contiguous() or t.get_device() != idx:
                return None
            ptrs[f] = t.data_ptr()
        m_out = out = x_in = None
        if self.need_m:
            m_out = torch.empty(self.shape, dtype=self.sdt, device=dev)
            ptrs[5] = m_out.data_ptr()
        if self.need_out:
            if self.dup:
                x_in = torch.empty(self.shape2, dtype=self.sdt, device=dev)
                out = x_in[:self.shape[0]]
                base = x_in.data_ptr()
                ptrs[6] = base
                ptrs[7] = base + n * self.esize
            else:
                out = torch.empty(self.shape, dtype=self.sdt, device=dev)
                ptrs[6] = out.data_ptr()
        if torch.cuda.current_device() == idx:
            rc = self.fn(self.ref_d, _raw_stream(idx))
        else:
            with torch.cuda.device(dev):
                rc = self.fn(self.ref_d, _raw_stream(idx))
        if rc != 0:
            _lib.check(rc)
        return m_out, out, x_in


_backend = None


def backend():
    """The active executor (CudaBackend unless a test installed another one)."""
    global _backend
    if _backend is None:
        _backend = CudaBackend()
    return _backend


def set_backend(b) -> None:
    """Install an executor with the CudaBackend interface. Used by tests/ only."""
    global _backend
    _backend = b


# ---- convenience wrappers, named after the reference functions they replace -----------------

def lincomb(x, ms, a, cs, out=None):
    """out = a*x + sum_j cs[j]*ms[j], 1 <= len(ms) <= 3, unfused fp32 chain, left to right."""
    k = len(ms)
    if not 1 <= k <= 3 or len(cs) != k:
        raise ValueError("lincomb takes 1..3 (tensor, coefficient) pairs")
    a_ = StepArgs(form=(FORM_LIN1, FORM_LIN2, FORM_LIN3)[k - 1], x=x, m0=ms[0],
                  m1=ms[1] if k > 1 else None, m2=ms[2] if k > 2 else None, a=a, c0=cs[0],
                  c1=cs[1] if k > 1 else 0.0, c2=cs[2] if k > 2 else 0.0, out=out)
    return backend().step(a_)[1]


def cfg_combine(eps_uncond, eps_cond, scale):
    """model_wrapper.model_fn :329-330."""
    a_ = StepArgs(form=FORM_NONE, n_model=2, e_cond=eps_cond, e_uncond=eps_uncond, guidance=scale,
                  state_dtype=eps_cond.dtype)
    return backend().step(a_)[0]


__all__ = ["StepArgs", "CudaBackend", "backend", "set_backend", "lincomb", "cfg_combine",
           "SUPPORTED_DTYPES", "FORM_NONE", "FORM_LIN1", "FORM_LIN2", "FORM_LIN3", "FORM_DIFF2",
           "FORM_MS3", "FORM_SS3T"]
