"""Drop-in `model_wrapper` and `DPM_Solver` (reference: dpm_solver_pytorch.py:170-334, :337-1245).

Same names, positional order, defaults, return types and error behaviour as the reference; the
per-step arithmetic runs as fused sm_100a kernels behind the C-ABI (ops.py). What changes under
the hood:

* all schedule scalars come from the host-side plan (plan.py) -- no per-step interpolation
  kernels and no `.item()` syncs inside the loop;
* the conversion of the raw network output (x_start/v/score parameterisation :288-298, CFG
  combine :329-330, eps->x0 :439, thresholding clamp :424) is fused with the solver update that
  consumes it: one kernel per model evaluation reads (x, eps[, eps_uncond], older buffers) and
  writes (buffered model value, x_next);
* dynamic thresholding's per-sample quantile (:422) is one exact radix-select launch.

The order of model evaluations, their (x, t) arguments, the hooks (`correcting_x0_fn`,
`correcting_xt_fn`) and `return_intermediate` are those of the reference.
"""
from __future__ import annotations

import dataclasses
import inspect
from dataclasses import dataclass
from typing import List, Optional

import torch
import torch.distributed as dist

from . import ops, plan as P
from ._lib import FORM_LIN1, FORM_NONE, FORM_SS3T, PARAM_BY_NAME, PARAM_NOISE
from .ops import StepArgs

__all__ = ["model_wrapper", "DPM_Solver", "WrappedModel"]

_DEV = object()     # marker: the scalars of this evaluation live in device memory (on-device adaptive controller)


# =================================================================================================
# model_wrapper
# =================================================================================================

@dataclass
class RawOutput:
    """Network output(s) before parameterisation / guidance have been applied."""
    e_cond: torch.Tensor
    e_uncond: Optional[torch.Tensor]
    param: int
    guidance: float


class WrappedModel:
    """Callable returned by `model_wrapper`: `model_fn(x, t_continuous) -> noise` (:309-330).

    Calling it reproduces the reference semantics. `DPM_Solver` additionally uses `raw()` to get
    the un-combined network outputs so that parameterisation + CFG are fused into the solver step.
    """

    def __init__(self, model, noise_schedule, model_type, model_kwargs, guidance_type, condition,
                 unconditional_condition, guidance_scale, classifier_fn, classifier_kwargs):
        self.model = model
        self.noise_schedule = noise_schedule
        self.model_type = model_type
        self.model_kwargs = model_kwargs
        self.guidance_type = guidance_type
        self.condition = condition
        self.unconditional_condition = unconditional_condition
        self.guidance_scale = guidance_scale
        self.classifier_fn = classifier_fn
        self.classifier_kwargs = classifier_kwargs
        self._c_in = None

    # -- pieces of the reference closure ----------------------------------------------------
    def get_model_input_time(self, t_continuous):
        """[1/N, 1] -> [0, 1000*(N-1)/N] for discrete-time models (:271-280)."""
        if self.noise_schedule.schedule == 'discrete':
            return (t_continuous - 1. / self.noise_schedule.total_N) * 1000.
        return t_continuous

    def _call_model(self, x, t_continuous, cond=None, t_input=None):
        if t_input is None:
            t_input = self.get_model_input_time(t_continuous)
        if cond is None:
            return self.model(x, t_input, **self.model_kwargs)
        return self.model(x, t_input, cond, **self.model_kwargs)

    @property
    def uses_cfg(self) -> bool:
        return (self.guidance_type == "classifier-free" and self.guidance_scale != 1.
                and self.unconditional_condition is not None)

    @property
    def fusable(self) -> bool:
        """False only for classifier guidance (needs autograd through the user's classifier)."""
        return self.guidance_type != "classifier"

    def input_rows(self, batch: int) -> int:
        """Length of the time vector the network receives for a batch (doubled under CFG :327)."""
        return 2 * batch if self.uses_cfg else batch

    def _cond_in(self):
        """cat([unconditional_condition, condition]) (:328); constant over a run, so built once."""
        uc, c = self.unconditional_condition, self.condition
        key = (id(uc), getattr(uc, "_version", 0), id(c), getattr(c, "_version", 0))
        if self._c_in is None or self._c_in[0] != key:
            # the pair is kept alive next to the key so that neither id can be recycled
            self._c_in = (key, torch.cat([uc, c]), (uc, c))
        return self._c_in[1]

    def raw(self, x, t_continuous, t_input=None, x_in=None) -> RawOutput:
        """Run the network exactly as the reference does, return its un-combined output(s).

        `t_input`, when given, is the precomputed model-input time vector (`input_rows(B)` long,
        same values as get_model_input_time would produce) so that no per-call arithmetic runs."""
        param = PARAM_BY_NAME[self.model_type]
        if self.guidance_type == "uncond":
            return RawOutput(self._call_model(x, t_continuous, t_input=t_input), None, param, 1.0)
        if self.guidance_type == "classifier-free":
            if not self.uses_cfg:
                return RawOutput(self._call_model(x, t_continuous, cond=self.condition, t_input=t_input), None, param, 1.0)
            if x_in is None:
                x_in = ops.backend().duplicate(x)              # cat([x] * 2) :326 (the solver hands over a prebuilt one)
            t_in = None if t_input is not None else torch.cat([t_continuous] * 2)
            out_u, out_c = self._call_model(x_in, t_in, cond=self._cond_in(), t_input=t_input).chunk(2)  # uncond first
            return RawOutput(out_c, out_u, param, float(self.guidance_scale))
        raise RuntimeError("raw() is not available with classifier guidance")

    def _alpha_sigma(self, t_continuous):
        """Host scalars [(alpha_t, sigma_t)]: one pair when all labels of the batch are equal (the solver's
        case), else one pair per sample (model_fn called directly with a vector of different times)."""
        tc = t_continuous.detach().reshape(-1).cpu()
        ns = self.noise_schedule
        if tc.numel() > 1 and not bool((tc == tc[0]).all()):
            return list(zip(ns.marginal_alpha(tc).tolist(), ns.marginal_std(tc).tolist()))
        t0 = tc[:1]
        return [(float(ns.marginal_alpha(t0)), float(ns.marginal_std(t0)))]

    @staticmethod
    def _per_sample(pairs, batch, launch):
        """Run `launch(rows, alpha, sigma)` once for the whole batch, or once per sample when the time labels
        differ (alpha_t, sigma_t are launch constants of the kernels)."""
        if len(pairs) == 1:
            return launch(slice(None), *pairs[0])
        assert len(pairs) == batch, "one time label per sample expected"
        return torch.cat([launch(slice(i, i + 1), al, sg) for i, (al, sg) in enumerate(pairs)])

    def __call__(self, x, t_continuous):
        be = ops.backend()
        if self.guidance_type == "classifier":
            assert self.classifier_fn is not None
            t_input = self.get_model_input_time(t_continuous)
            with torch.enable_grad():
                x_in = x.detach().requires_grad_(True)
                log_prob = self.classifier_fn(x_in, t_input, self.condition, **self.classifier_kwargs)
                cond_grad = torch.autograd.grad(log_prob.sum(), x_in)[0]
            pairs = self._alpha_sigma(t_continuous)
            out = self._call_model(x, t_continuous)
            param = PARAM_BY_NAME[self.model_type]
            xo, grad = x.to(out.dtype), cond_grad.to(out.dtype)

            def guided(rows, alpha, sigma):
                o = out[rows]
                if param != PARAM_NOISE:
                    o = be.step(StepArgs(form=FORM_NONE, n_model=1, e_cond=o, xe=xo[rows], param=param,
                                         alpha_e=alpha, sigma_e=sigma, state_dtype=out.dtype))[0]
                # noise - guidance_scale * sigma_t * cond_grad (:321); (s*sigma) is formed in fp32 first
                gs = float(torch.tensor(sigma, dtype=torch.float32) * self.guidance_scale)
                return ops.lincomb(o, [grad[rows]], 1.0, [-gs])
            return self._per_sample(pairs, x.shape[0], guided)
        r = self.raw(x, t_continuous)
        if r.e_uncond is None and r.param == PARAM_NOISE:
            return r.e_cond
        pairs = self._alpha_sigma(t_continuous) if r.param != PARAM_NOISE else [(1.0, 0.0)]
        needs_x = r.param in (PARAM_BY_NAME["x_start"], PARAM_BY_NAME["v"])
        xo = x.to(r.e_cond.dtype) if needs_x else None

        def convert(rows, alpha, sigma):
            a = StepArgs(form=FORM_NONE, n_model=2 if r.e_uncond is not None else 1, e_cond=r.e_cond[rows],
                         e_uncond=None if r.e_uncond is None else r.e_uncond[rows], param=r.param,
                         guidance=r.guidance, alpha_e=alpha, sigma_e=sigma, state_dtype=r.e_cond.dtype)
            if needs_x:
                a.xe = xo[rows]
            return be.step(a)[0]
        return self._per_sample(pairs, x.shape[0], convert)


def model_wrapper(model, noise_schedule, model_type="noise", model_kwargs={}, guidance_type="uncond",
                  condition=None, unconditional_condition=None, guidance_scale=1., classifier_fn=None,
                  classifier_kwargs={}):
    """Wrap a network into `model_fn(x, t_continuous) -> noise`; same contract as the reference
    (:170-334): model_type in {noise, x_start, v, score}, guidance_type in {uncond, classifier,
    classifier-free}."""
    assert model_type in ["noise", "x_start", "v", "score"]
    assert guidance_type in ["uncond", "classifier", "classifier-free"]
    return WrappedModel(model, noise_schedule, model_type, model_kwargs, guidance_type, condition,
                        unconditional_condition, guidance_scale, classifier_fn, classifier_kwargs)


# =================================================================================================
# DPM_Solver
# =================================================================================================

class DPM_Solver:
    def __init__(self, model_fn, noise_schedule, algorithm_type="dpmsolver++", correcting_x0_fn=None,
                 correcting_xt_fn=None, thresholding_max_val=1., dynamic_thresholding_ratio=0.995,
                 state_dtype=None, plan_broadcast=False, predict_x0=None, thresholding=None, max_val=None,
                 reference_rounding=False):
        """Same arguments as the reference (:338-347) plus `state_dtype` and `plan_broadcast`:

        state_dtype=None keeps the reference's type promotion (fp32 state and buffers even for
        bf16/fp16 inputs, because its fp32 coefficient tensors promote every update);
        state_dtype=torch.bfloat16 / torch.float16 keeps x and the buffered model values in 16-bit
        storage (fp32 arithmetic in registers, one rounding on store) and halves HBM traffic.

        plan_broadcast=True (batch-sharded multi-GPU runs, torch.distributed initialised): rank 0
        broadcasts the scalar coefficient plan once per sample() so all ranks use bit-identical
        coefficients (distributed.py); the tensors themselves are never communicated.

        reference_rounding=True (opt-in; fp32 state, `model_type="noise"`, network returning bf16/fp16):
        reproduce the two places where the reference computes in the network's 16-bit output type -- the
        CFG combine (:329-330, three rounded ops) and, for the eps-solver, the differences of the
        buffered raw outputs (:823, :880-881, :636, :735, :741-742). Default False: both are evaluated in
        fp32 on the widened values (closer to the exact result, and the fast kernels). Runs on the generic
        kernel for now.

        predict_x0 / thresholding / max_val: keyword spelling of the older constructor that the JAX twin
        still uses (dpm_solver_jax.py:351): predict_x0=True selects "dpmsolver++", thresholding=True
        (valid with predict_x0) selects dynamic thresholding, max_val is `thresholding_max_val`.
        """
        if predict_x0 is not None:
            algorithm_type = "dpmsolver++" if predict_x0 else "dpmsolver"
        if thresholding:
            correcting_x0_fn = "dynamic_thresholding"
        if max_val is not None:
            thresholding_max_val = max_val
        self._wrapped = model_fn
        self.model = lambda x, t: model_fn(x, t.expand((x.shape[0])))
        self.noise_schedule = noise_schedule
        tables = getattr(noise_schedule, "log_alpha_array", None)
        if torch.is_tensor(tables) and tables.dtype != torch.float32:
            # the reference would promote x and every update to that dtype; there are no fp64 kernels
            raise TypeError("dpm_solver_b200 computes in fp32: NoiseScheduleVP(dtype={}) is not supported "
                            "by DPM_Solver".format(tables.dtype))
        assert algorithm_type in ["dpmsolver", "dpmsolver++"] + list(P.SDE_ALGORITHMS)
        self.algorithm_type = algorithm_type
        if reference_rounding and algorithm_type in P.SDE_ALGORITHMS:
            raise ValueError("reference_rounding=True is not available for algorithm_type={!r}".format(algorithm_type))
        if correcting_x0_fn == "dynamic_thresholding":
            self.correcting_x0_fn = self.dynamic_thresholding_fn
            self._dynamic_thresholding = True
        else:
            self.correcting_x0_fn = self._x0_hook(correcting_x0_fn)
            self._dynamic_thresholding = False
        self.correcting_xt_fn = correcting_xt_fn
        self.dynamic_thresholding_ratio = dynamic_thresholding_ratio
        self.thresholding_max_val = thresholding_max_val
        if state_dtype is not None and state_dtype not in ops.SUPPORTED_DTYPES:
            raise TypeError("state_dtype must be one of {}".format(ops.SUPPORTED_DTYPES))
        self.state_dtype = state_dtype
        self.plan_broadcast = bool(plan_broadcast)
        self.reference_rounding = bool(reference_rounding)
        self._rr_run = 0     # raw_round of the buffered values of the run in flight (reference_rounding)
        self._prep_cache = {}   # frozen launch descriptors of cached plan steps (ops.PreparedStep)
        self._prep_on = False

    @staticmethod
    def _x0_hook(fn):
        """`correcting_x0_fn(x0, t)` (:379-380). The older vendored copy calls it with x0 only
        (examples/stable-diffusion/.../dpm_solver.py:447-448); a one-argument callable keeps working."""
        if fn is None or not callable(fn):
            return fn
        try:
            params = [p for p in inspect.signature(fn).parameters.values()
                      if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
            variadic = any(p.kind == p.VAR_POSITIONAL for p in inspect.signature(fn).parameters.values())
        except (TypeError, ValueError):
            return fn
        if len(params) == 1 and not variadic:
            return lambda x0, t: fn(x0)
        return fn

    def _sync_plan(self, coeffs, key=None):
        """Rank 0's coefficients on every rank. One broadcast per sampling configuration: the synced
        plan is cached under the plan key, so steady-state sample() calls issue no collective."""
        if not self.plan_broadcast:
            return coeffs
        from .distributed import broadcast_plan
        if key is None:
            return broadcast_plan(coeffs)
        cache = self.__dict__.setdefault("_synced_cache", {})
        k = (self._schedule_key(), self.algorithm_type) + key
        hit = cache.get(k)
        if hit is None:
            hit = broadcast_plan(coeffs)
            if len(cache) >= self._CACHE_MAX:
                cache.pop(next(iter(cache)))
            cache[k] = hit
        return hit

    # -- small helpers ------------------------------------------------------------------------
    @property
    def _pp(self) -> bool:
        """The buffered model value is x0 (data prediction)."""
        return self.algorithm_type in ("dpmsolver++", "sde-dpmsolver++")

    @property
    def _sde(self) -> bool:
        return self.algorithm_type in P.SDE_ALGORITHMS

    def _no_sde(self, what: str) -> None:
        """The stochastic solvers exist as multistep sample() runs only; never run them silently as the ODE."""
        if self._sde:
            raise ValueError("{} is not available for algorithm_type={!r}: the SDE solvers are served by "
                             "sample(method='multistep', order=1 or 2)".format(what, self.algorithm_type))

    def _sdtype(self, x) -> torch.dtype:
        if self.state_dtype is not None:
            return self.state_dtype
        if x.dtype not in ops.SUPPORTED_DTYPES:
            raise TypeError("dpm_solver_b200 supports float32, bfloat16 and float16 tensors, got {}".format(x.dtype))
        return torch.float32  # reference promotion: fp32 coefficient tensors make every update fp32

    def _state(self, x) -> torch.Tensor:
        """The tensor the kernels read as `x`. In the reference's promotion mode (state_dtype=None) a
        16-bit x is widened to fp32 for the arithmetic -- exactly what its fp32 coefficient tensors do --
        but the NETWORK still receives the caller's 16-bit tensor at that evaluation (only later states
        are fp32), so the pair is remembered for `_evaluate`."""
        sd = self._sdtype(x)
        xs = x.to(sd) if x.dtype != sd else x
        xs = xs if ops.CudaBackend._layout(xs) is not None else xs.contiguous()
        # (re-evaluations at the same state -- a rejected adaptive step -- must see it again: the pair stays
        # until the next _state() call or the end of sample())
        if self.state_dtype is None and x.dtype != sd:
            self._net_input = (xs, x)
        elif self.__dict__.get("_net_input") is not None and self._net_input[0] is not xs:
            self._net_input = None
        return xs

    def _alpha_sigma(self, t_host):
        ns = self.noise_schedule
        return float(ns.marginal_alpha(t_host)), float(ns.marginal_std(t_host))

    # -- model evaluation ---------------------------------------------------------------------
    def _evaluate(self, x, t_dev, t_input=None) -> RawOutput:
        """Call the user's network at (x, t); same call the reference makes through self.model."""
        w = self._wrapped
        orig = self.__dict__.get("_net_input")
        if orig is not None and orig[0] is x:
            x = orig[1]                           # the caller's own (16-bit) tensor, as the reference passes it
        if isinstance(w, WrappedModel) and w.fusable:
            pair = self.__dict__.get("_xin_pair")
            x_in = pair[1] if (pair is not None and pair[0] is x) else None
            # (the continuous label is only read when no precomputed model-input time row is handed over)
            return w.raw(x, t_dev.expand((x.shape[0])) if t_input is None else None, t_input, x_in)
        return RawOutput(self.model(x, t_dev), None, PARAM_NOISE, 1.0)

    def _dup_target(self, x):
        """Under CFG the network consumes cat([x]*2) (:326). When nothing can touch x between the
        update and the next evaluation, the update kernel writes x_t straight into both halves of a
        [2B, ...] buffer: returns (x_in, first half, second half) or None."""
        w = self._wrapped
        if self.correcting_xt_fn is not None or not (isinstance(w, WrappedModel) and w.fusable and w.uses_cfg):
            return None
        shape = (2 * x.shape[0],) + tuple(x.shape[1:])
        if ops.CudaBackend._layout(x) == "cl":      # keep a channels_last network's layout
            x_in = torch.empty(shape, dtype=x.dtype, device=x.device,
                               memory_format=torch.channels_last if x.dim() == 4 else torch.channels_last_3d)
        else:
            x_in = torch.empty(shape, dtype=x.dtype, device=x.device)
        return x_in, x_in[:x.shape[0]], x_in[x.shape[0]:]

    _CACHE_MAX = 16

    def _schedule_key(self):
        """Identity of the schedule the cached plans were computed from. The table tensors are pinned
        in `_schedule_refs` so their ids cannot be recycled; `_version` catches in-place edits."""
        ns = self.noise_schedule
        if getattr(ns, "schedule", None) == "discrete":
            la, ta = ns.log_alpha_array, ns.t_array
            refs = self.__dict__.setdefault("_schedule_refs", {})
            refs[id(la)], refs[id(ta)] = la, ta
            if len(refs) > 64:
                for k in list(refs)[:-8]:
                    refs.pop(k)
                for name in ("_plan_cache", "_table_cache", "_synced_cache"):
                    self.__dict__.pop(name, None)
            return ("discrete", id(la), la._version, id(ta), ta._version, ns.total_N)
        return (getattr(ns, "schedule", None), getattr(ns, "beta_0", None), getattr(ns, "beta_1", None),
                getattr(ns, "T", None))

    def _plan_id(self, key):
        """Hashable identity of a cached plan (schedule + algorithm + sampling arguments): prepared launches are
        keyed by it, so a changed schedule or argument never meets a stale descriptor."""
        return (self._schedule_key(), self.algorithm_type, self.plan_broadcast) + key

    def _host_plan(self, key, build):
        """Coefficient plan of a run, cached per (schedule, algorithm, sampling arguments): repeated
        sample() calls with the same configuration (serving) skip the host scalar work entirely."""
        cache = self.__dict__.setdefault("_plan_cache", {})
        k = (self._schedule_key(), self.algorithm_type) + key
        hit = cache.get(k)
        if hit is None:
            hit = build()
            if len(cache) >= self._CACHE_MAX:
                cache.pop(next(iter(cache)))
            cache[k] = hit
        return hit

    def _device_tables(self, key, t_host, batch, device, n_eval=None):
        """Device copies of the time grid and of the model-input time matrix, cached with the plan
        (they depend on the batch size and the device only)."""
        cache = self.__dict__.setdefault("_table_cache", {})
        k = (self._schedule_key(), self.algorithm_type) + key + (batch, str(device), id(self._wrapped))
        hit = cache.get(k)
        if hit is None:
            t_dev = self._upload(t_host, device)
            tin = self._input_times(t_host if n_eval is None else t_host[:n_eval], batch, device)
            # the per-step views are built once here: indexing a device tensor costs ~1.5 us of host time, three
            # times per solver step
            n = t_dev.shape[0]
            hit = (t_dev, tin, [t_dev[i] for i in range(n)], [t_dev[i:i + 1] for i in range(n)],
                   None if tin is None else [tin[i] for i in range(tin.shape[0])])
            if len(cache) >= self._CACHE_MAX:
                cache.pop(next(iter(cache)))
            cache[k] = hit
        return hit

    def _denoise_tables(self, t_0, batch, device):
        """(device label (1,), model-input time row or None, (alpha, sigma)) of the denoise-to-zero tail."""
        cache = self.__dict__.setdefault("_table_cache", {})
        k = (self._schedule_key(), "d2z", float(t_0), batch, str(device), id(self._wrapped))
        hit = cache.get(k)
        if hit is None:
            th = torch.ones((1,)) * t_0                                   # fp32, as `torch.ones((1,)).to(device) * t_0`
            tin = self._input_times(th, batch, device)
            hit = (self._upload(th, device), None if tin is None else tin[0], self._alpha_sigma(th))
            if len(cache) >= self._CACHE_MAX:
                cache.pop(next(iter(cache)))
            cache[k] = hit
        return hit

    @staticmethod
    def _upload(t_host: torch.Tensor, device):
        """Host vector -> device without draining the stream (pinned staging, async copy)."""
        device = torch.device(device)
        if device.type != "cuda":
            return t_host.to(device)
        return t_host.pin_memory().to(device, non_blocking=True)

    def _input_times(self, t_host: torch.Tensor, batch: int, device):
        """[n_evals, rows] device matrix of model-input times for a whole run (one tiny kernel per
        sample() instead of two per model call); None when the model takes t_continuous itself."""
        w = self._wrapped
        if not (isinstance(w, WrappedModel) and w.fusable and w.noise_schedule.schedule == 'discrete'):
            return None
        t_in = self._upload(w.get_model_input_time(t_host.reshape(-1)), device)   # (t - 1/N) * 1000, fp32, :278
        return t_in[:, None].expand(t_in.shape[0], w.input_rows(batch)).contiguous()

    def _conv_args(self, raw: RawOutput, xe, alsig, sdtype, x0: bool) -> StepArgs:
        """StepArgs fields that turn `raw` into the buffered model value at time t (x0 if `x0`, else
        eps). `alsig` is (alpha_t, sigma_t) from the plan, or the host time tensor to derive them."""
        a = StepArgs(n_model=2 if raw.e_uncond is not None else 1, e_cond=raw.e_cond,
                     e_uncond=raw.e_uncond, param=raw.param, guidance=raw.guidance,
                     predict_x0=x0, state_dtype=sdtype)
        if x0 or raw.param != PARAM_NOISE:
            if alsig is _DEV:
                pass        # (alpha_t, sigma_t) arrive with the launch's device coefficient block (StepArgs.coef_dev)
            else:
                a.alpha_e, a.sigma_e = alsig if isinstance(alsig, tuple) else self._alpha_sigma(alsig)
            a.xe = xe
        return a

    @staticmethod
    def _needs_conversion(raw: RawOutput, sdtype, x0: bool) -> bool:
        return x0 or raw.e_uncond is not None or raw.param != PARAM_NOISE or raw.e_cond.dtype != sdtype

    _RR_CODE = {torch.bfloat16: 1, torch.float16: 2}      # dpm_dtype codes carried by raw_round

    def _rr_code(self, raw: RawOutput) -> int:
        """16-bit dtype code of raw NOISE outputs in reference-rounding mode, else 0."""
        if not self.reference_rounding or self.state_dtype is not None or raw.param != PARAM_NOISE:
            return 0
        return self._RR_CODE.get(raw.e_cond.dtype, 0)

    @staticmethod
    def _rr_coeffs(co: P.Coeffs, code: int) -> P.Coeffs:
        """singlestep-3 'taylor' (:780-783) in reference-rounding mode: r1, r2 that arrive as 0-dim tensors
        (the sample() loop, :1223-1227) are cast to the buffers' 16-bit type where they are the LEFT operand
        of a product (`(1./r1) * (..)`, `r2 * D1_0`, `r1 * D1_1`); python floats (the defaults of the
        directly called method) and right-hand scalars (the divisor `r2 - r1`) enter in fp32 -- torch's CPU
        kernels keep the second operand of mul/div in the op's fp32 math type when it is a scalar."""
        if co.form != FORM_SS3T or not co.r_tensor:
            return co
        T = torch.bfloat16 if code == 1 else torch.float16
        rT = lambda v: float(torch.tensor(v, dtype=torch.float32).to(T))
        r1t, r2t = bool(co.r_tensor & 1), bool(co.r_tensor & 2)
        return dataclasses.replace(co, w0=rT(co.w0) if r1t else co.w0, w1=rT(co.w1) if r2t else co.w1,
                                   w2=rT(co.w2) if r2t else co.w2, w3=rT(co.w3) if r1t else co.w3,
                                   w4=co.w4)

    def _post_model(self, raw: RawOutput, xe, t_dev, alsig, co: Optional[P.Coeffs] = None, x=None,
                    m1=None, m2=None, want_m: bool = True, dup_out: bool = False, x0: Optional[bool] = None,
                    slot=None):
        """The fused post-model step: buffered value from `raw` (+ optional update `co`).

        Returns (m_new, x_next). Falls back to two launches only when a user-supplied
        `correcting_x0_fn` must see the materialised x0 (:440-441).

        `slot` names a step of a CACHED coefficient plan (sample() loops): its launch descriptor is frozen after
        the first run (ops.PreparedStep) and later runs only patch tensor pointers -- the steady-state host path."""
        be = ops.backend()
        pkey = None
        if slot is not None and self._prep_on:
            pkey = (slot, raw.param, raw.guidance, raw.e_uncond is None, raw.e_cond.dtype, xe.dtype, xe.shape,
                    want_m, dup_out)
            prep = self._prep_cache.get(pkey)
            if prep is not None:
                r = prep.launch((x, xe, raw.e_cond, m1, m2, raw.e_cond, raw.e_uncond))
                if r is not None:
                    m_new, x_next, x_in = r
                    if x_in is not None:
                        self._xin_pair = (x_next, x_in)
                    if m_new is None and prep.d.n_model == 0:
                        m_new = raw.e_cond                  # pure update on the raw noise: it IS the buffered value
                    return m_new, x_next
        x0 = self._pp if x0 is None else x0          # buffered value: x0 (dpmsolver++ / data_prediction_fn) or eps
        sd = xe.dtype if xe is not None else (x.dtype if x is not None else raw.e_cond.dtype)
        custom_fix = x0 and self.correcting_x0_fn is not None and not self._dynamic_thresholding
        code = self._rr_code(raw)
        rr = 0
        if code:
            # reference-rounding mode (raw 16-bit NOISE outputs, fp32 state): bits 0-1 make the fused kernel take the
            # CFG combine in the network's type, three rounded ops (:329-330); for the eps-solver the buffered values
            # are those raw outputs, so bit 2 makes their differences round too (:823, :880-881, :636, :735)
            rr = code
            if not x0:
                rr = self._rr_run = code | 4
            if raw.e_uncond is not None and x0 and self._dynamic_thresholding:
                # the quantile kernels take the combine in fp32: give them (and the step) the reference's rounded
                # noise, materialised once (values exactly representable in the network's type, held in fp32)
                e = be.step(StepArgs(form=FORM_NONE, n_model=2, e_cond=raw.e_cond, e_uncond=raw.e_uncond,
                                     param=PARAM_NOISE, guidance=raw.guidance, state_dtype=torch.float32,
                                     raw_round=code))[0]
                raw = RawOutput(e, None, PARAM_NOISE, 1.0)
                rr = 0
        if (rr & 4) and co is not None:
            co = self._rr_coeffs(co, code)
        if not self._needs_conversion(raw, sd, x0):
            m_new = raw.e_cond if ops.CudaBackend._layout(raw.e_cond) is not None else raw.e_cond.contiguous()
            x_next = self._pure_update(co, x, m_new, m1, m2, rr=rr & 4 and rr, pkey=pkey if m_new is raw.e_cond else None) \
                if co is not None else None
            return m_new, x_next
        a = self._conv_args(raw, xe, alsig, sd, x0)
        if alsig is _DEV:
            if co is None or co.dev is None:
                raise RuntimeError("device-side scalars need the coefficient block of the consuming launch")
            a.coef_dev = co.dev
        if x0 and self._dynamic_thresholding:
            a.per_sample = xe.numel() // xe.shape[0]
            a.thr = be.dynamic_threshold(a, float(self.dynamic_thresholding_ratio),
                                         float(self.thresholding_max_val))
        if custom_fix or co is None:
            a.form = FORM_NONE
            a.raw_round = rr & 3
            m_new = be.step(a)[0]
            if custom_fix:
                m_new = self._state_like(self.correcting_x0_fn(m_new, t_dev), sd)
            x_next = self._pure_update(co, x, m_new, m1, m2, rr=rr & 4 and rr) if co is not None else None
            return m_new, x_next
        self._fill_update(a, co, x, m1, m2)
        a.want_m_out = want_m
        a.raw_round = rr
        dup = self._dup_target(x) if dup_out else None
        if dup is not None:
            a.out, a.out2 = dup[1], dup[2]
        m_new, x_next = self._launch(a, co)
        if dup is not None:
            self._xin_pair = (x_next, dup[0])
        if pkey is not None and not a.per_sample:
            self._remember(pkey, a, dup)
        return m_new, x_next

    def _remember(self, pkey, a: StepArgs, dup=None) -> None:
        """Freeze the launch that just ran as the prepared form of its plan step."""
        if dup is not None:
            a.out, a.out2 = dup[1], dup[2]
        prep = ops.backend().prepare(a)
        if prep is not None:
            if len(self._prep_cache) >= 512:
                self._prep_cache.clear()
            self._prep_cache[pkey] = prep

    @staticmethod
    def _state_like(t, sd):
        if t.dtype != sd:
            t = t.to(sd)
        return t if ops.CudaBackend._layout(t) is not None else t.contiguous()   # dense (row-major / channels_last)

    @staticmethod
    def _fill_update(a: StepArgs, co: P.Coeffs, x, m1, m2) -> None:
        a.form, a.x, a.m1, a.m2 = co.form, x, m1, m2
        if co.dev is not None:
            a.coef_dev = co.dev
        a.a, a.c0, a.c1, a.c2 = co.a, co.c0, co.c1, co.c2
        a.w0, a.w1, a.w2, a.w3, a.w4 = co.w0, co.w1, co.w2, co.w3, co.w4
        a.c0_on_old = co.c0_on_old

    def _pure_update(self, co: P.Coeffs, x, m0, m1=None, m2=None, rr: Optional[int] = None, pkey=None):
        if rr is None:
            # directly called update methods: buffers handed over in one 16-bit type are raw outputs
            rr = 0
            dts = {m.dtype for m in (m0, m1, m2) if m is not None}
            if (self.reference_rounding and self.state_dtype is None and x.dtype == torch.float32
                    and len(dts) == 1 and next(iter(dts)) in self._RR_CODE):
                rr = self._RR_CODE[next(iter(dts))] | 4
        a = StepArgs(n_model=0, m0=self._state_like(m0, x.dtype), state_dtype=x.dtype, raw_round=rr)
        self._fill_update(a, co, x, None if m1 is None else self._state_like(m1, x.dtype),
                          None if m2 is None else self._state_like(m2, x.dtype))
        out = self._launch(a, co)[1]
        if pkey is not None and not rr:
            self._remember(pkey, a)
        return out

    def _launch(self, a: StepArgs, co: P.Coeffs):
        """One update launch: the ODE step, or for the SDE algorithms the same step plus co.cn * (fresh noise drawn
        from the generator of the sample() call in flight)."""
        be = ops.backend()
        if self._sde:
            return be.sde_step(a, co.cn, generator=self.__dict__.get("_generator"))
        return be.step(a)

    # -- reference API: model functions ---------------------------------------------------------
    def dynamic_thresholding_fn(self, x0, t):
        """Imagen dynamic thresholding of a materialised x0 (:416-425)."""
        x0c = self._state_like(x0, x0.dtype if x0.dtype in ops.SUPPORTED_DTYPES else torch.float32)
        # x0 = (x0 - 0*0)/1 exactly: reuse the conversion path with eps = 0
        zeros = torch.zeros_like(x0c)
        a = StepArgs(form=FORM_NONE, n_model=1, e_cond=zeros, xe=x0c, predict_x0=True, alpha_e=1.0,
                     sigma_e=0.0, state_dtype=x0c.dtype, per_sample=x0c.numel() // x0c.shape[0])
        be = ops.backend()
        a.thr = be.dynamic_threshold(a, float(self.dynamic_thresholding_ratio), float(self.thresholding_max_val))
        return be.step(a)[0]

    def noise_prediction_fn(self, x, t):
        """Return the noise prediction model (:427-431)."""
        return self.model(x, t)

    def data_prediction_fn(self, x, t):
        """x0 = (x - sigma_t*eps)/alpha_t with corrector (:433-442), one fused launch."""
        xs = self._state(x)
        raw = self._evaluate(xs, t)
        return self._post_model(raw, xs, t, P._cpu(t)[:1], x0=True)[0]   # x0 regardless of algorithm_type

    def model_fn(self, x, t):
        """Noise prediction (dpmsolver) or data prediction (dpmsolver++) (:444-451)."""
        if self._pp:
            return self.data_prediction_fn(x, t)
        xs = self._state(x)
        raw = self._evaluate(xs, t)
        return self._post_model(raw, xs, t, P._cpu(t)[:1])[0]

    # -- reference API: time grids ---------------------------------------------------------------
    def get_time_steps(self, skip_type, t_T, t_0, N, device):
        """Time grid of N+1 points (:453-480). Computed on the host, moved to `device`."""
        if skip_type == 'logSNR':
            lambda_T = self.noise_schedule.marginal_lambda(torch.tensor(t_T))
            lambda_0 = self.noise_schedule.marginal_lambda(torch.tensor(t_0))
            logSNR_steps = torch.linspace(lambda_T.item(), lambda_0.item(), N + 1)
            return self.noise_schedule.inverse_lambda(logSNR_steps).to(device)
        elif skip_type == 'time_uniform':
            return torch.linspace(t_T, t_0, N + 1).to(device)
        elif skip_type == 'time_quadratic':
            t_order = 2
            return torch.linspace(t_T ** (1. / t_order), t_0 ** (1. / t_order), N + 1).pow(t_order).to(device)
        else:
            raise ValueError("Unsupported skip_type {}, need to be 'logSNR' or 'time_uniform' or "
                             "'time_quadratic'".format(skip_type))

    def get_orders_and_timesteps_for_singlestep_solver(self, steps, order, skip_type, t_T, t_0, device):
        """Orders and outer grid of 'DPM-Solver-fast' (:482-539)."""
        orders = P.singlestep_orders(steps, order)
        if skip_type == 'logSNR':
            timesteps_outer = self.get_time_steps(skip_type, t_T, t_0, len(orders), device)
        else:
            idx = torch.cumsum(torch.tensor([0, ] + orders), 0).to(device)
            timesteps_outer = self.get_time_steps(skip_type, t_T, t_0, steps, device)[idx]
        return timesteps_outer, orders

    def denoise_to_zero_fn(self, x, s):
        """Final first-order denoise to t=0 (:541-545)."""
        return self.data_prediction_fn(x, s)

    # -- reference API: single updates (direct-call path; scalars computed per call) -------------
    def dpm_solver_first_update(self, x, s, t, model_s=None, return_intermediate=False):
        """DPM-Solver-1 / DDIM step s -> t (:547-592)."""
        self._no_sde("dpm_solver_first_update")
        x = self._state(x)
        co = P.first_update_coeffs(self.noise_schedule, self.algorithm_type, s, t)
        if model_s is None:
            raw = self._evaluate(x, s)
            model_s, x_t = self._post_model(raw, x, s, P._cpu(s), co, x, want_m=return_intermediate)
        else:
            x_t = self._pure_update(co, x, model_s)
        if return_intermediate:
            return x_t, {'model_s': model_s}
        return x_t

    def _device_time(self, t_host, like):
        return t_host.to(like.device)

    def singlestep_dpm_solver_second_update(self, x, s, t, r1=0.5, model_s=None, return_intermediate=False,
                                            solver_type='dpmsolver'):
        """Singlestep DPM-Solver-2 s -> t (:594-673)."""
        self._no_sde("singlestep_dpm_solver_second_update")
        if solver_type not in ['dpmsolver', 'taylor']:
            raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
        sp = P.singlestep_second(self.noise_schedule, self.algorithm_type, solver_type, s, t, r1)
        x_t, ms = self._run_singlestep(self._state(x), sp, model_s=model_s, keep=return_intermediate)
        if return_intermediate:
            return x_t, {'model_s': ms[0], 'model_s1': ms[1]}
        return x_t

    def singlestep_dpm_solver_third_update(self, x, s, t, r1=1. / 3., r2=2. / 3., model_s=None, model_s1=None,
                                           return_intermediate=False, solver_type='dpmsolver'):
        """Singlestep DPM-Solver-3 s -> t (:675-794)."""
        self._no_sde("singlestep_dpm_solver_third_update")
        if solver_type not in ['dpmsolver', 'taylor']:
            raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
        sp = P.singlestep_third(self.noise_schedule, self.algorithm_type, solver_type, s, t, r1, r2)
        x_t, ms = self._run_singlestep(self._state(x), sp, model_s=model_s, model_s1=model_s1,
                                       keep=return_intermediate)
        if return_intermediate:
            return x_t, {'model_s': ms[0], 'model_s1': ms[1], 'model_s2': ms[2]}
        return x_t

    def _run_singlestep(self, x, sp: P.SinglestepPlan, model_s=None, model_s1=None, keep=False,
                        times_dev: Optional[List[torch.Tensor]] = None, alsig=None, t_inputs=None,
                        dup_last: bool = False, slot=None):
        """Execute one singlestep update: one fused launch per model evaluation.

        Stage j converts the network output evaluated at (x_j, times[j]) and, in the same kernel,
        produces the next intermediate state from the base state x (:630-640, :723-750)."""
        td = times_dev if times_dev is not None else [self._device_time(tt, x) for tt in sp.times]
        als = alsig if alsig is not None else sp.times
        tin = t_inputs if t_inputs is not None else [None] * len(sp.times)
        ms: List[Optional[torch.Tensor]] = [model_s, model_s1, None]
        taylor3 = sp.order == 3 and sp.stages[-1].form == FORM_SS3T
        xe = x
        x_next = None
        for j, co in enumerate(sp.stages):
            last = j == len(sp.stages) - 1
            # buffers the stage reads besides the value it computes itself
            if co.form == FORM_LIN1:
                m1 = m2 = None
            elif co.form == FORM_SS3T:
                m1, m2 = ms[1], ms[0]
            else:
                m1, m2 = ms[0], None
            given = ms[j] if j < 2 else None
            # x_s1 is not needed when the caller already supplies model_s1 (:722)
            skip_update = j == 0 and sp.order == 3 and ms[1] is not None
            if given is not None:
                # caller supplied this model value (the adaptive solver reuses the lower-order ones)
                if not skip_update:
                    x_next = self._pure_update(co, x, given, m1, m2, rr=self._rr_run)
            else:
                raw = self._evaluate(xe, td[j], tin[j])
                want = keep or (not last and (j == 0 or taylor3))
                if skip_update:
                    m_new, _ = self._post_model(raw, xe, td[j], als[j])
                else:
                    m_new, x_next = self._post_model(raw, xe, td[j], als[j], co, x, m1, m2, want_m=want,
                                                     dup_out=(not last) or dup_last,
                                                     slot=None if slot is None else slot + (j,))
                ms[j] = m_new
            xe = x_next
        return x_next, ms

    def multistep_dpm_solver_second_update(self, x, model_prev_list, t_prev_list, t, solver_type="dpmsolver"):
        """Multistep DPM-Solver-2 (:796-852)."""
        self._no_sde("multistep_dpm_solver_second_update")
        if solver_type not in ['dpmsolver', 'taylor']:
            raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
        co = P.multistep_coeffs(self.noise_schedule, self.algorithm_type, solver_type, 2, t_prev_list, t)
        return self._pure_update(co, self._state(x), model_prev_list[-1], model_prev_list[-2])

    def multistep_dpm_solver_third_update(self, x, model_prev_list, t_prev_list, t, solver_type='dpmsolver'):
        """Multistep DPM-Solver-3 (:854-904); needs exactly three buffered values."""
        self._no_sde("multistep_dpm_solver_third_update")
        model_prev_2, model_prev_1, model_prev_0 = model_prev_list
        t_prev_2, t_prev_1, t_prev_0 = t_prev_list
        co = P.multistep_coeffs(self.noise_schedule, self.algorithm_type, solver_type, 3,
                                [t_prev_2, t_prev_1, t_prev_0], t)
        return self._pure_update(co, self._state(x), model_prev_0, model_prev_1, model_prev_2)

    def singlestep_dpm_solver_update(self, x, s, t, order, return_intermediate=False, solver_type='dpmsolver',
                                     r1=None, r2=None):
        """Order dispatch (:906-930)."""
        self._no_sde("singlestep_dpm_solver_update")
        if order == 1:
            return self.dpm_solver_first_update(x, s, t, return_intermediate=return_intermediate)
        elif order == 2:
            return self.singlestep_dpm_solver_second_update(x, s, t, return_intermediate=return_intermediate,
                                                            solver_type=solver_type, r1=r1)
        elif order == 3:
            return self.singlestep_dpm_solver_third_update(x, s, t, return_intermediate=return_intermediate,
                                                           solver_type=solver_type, r1=r1, r2=r2)
        else:
            raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))

    def multistep_dpm_solver_update(self, x, model_prev_list, t_prev_list, t, order, solver_type='dpmsolver'):
        """Order dispatch (:932-954)."""
        self._no_sde("multistep_dpm_solver_update")
        if order == 1:
            return self.dpm_solver_first_update(x, t_prev_list[-1], t, model_s=model_prev_list[-1])
        elif order == 2:
            return self.multistep_dpm_solver_second_update(x, model_prev_list, t_prev_list, t, solver_type=solver_type)
        elif order == 3:
            return self.multistep_dpm_solver_third_update(x, model_prev_list, t_prev_list, t, solver_type=solver_type)
        else:
            raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))

    # -- adaptive solver (:956-1010) ---------------------------------------------------------------
    def dpm_solver_adaptive(self, x, order, t_T, t_0, h_init=0.05, atol=0.0078, rtol=0.05, theta=0.9,
                            t_err=1e-5, solver_type='dpmsolver'):
        """Adaptive step size DPM-Solver-12 / -23 (:956-1010). Updates and the error estimate run on
        the fused kernels; the step-size controller is the reference's host logic."""
        self._no_sde("the adaptive solver")
        ns = self.noise_schedule
        x = self._state(x)
        device = x.device
        if order not in (2, 3):
            raise ValueError("For adaptive step size solver, order must be 2 or 3, got {}".format(order))
        if solver_type not in ['dpmsolver', 'taylor']:
            raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
        if self._device_controller_ok(x):
            return self._adaptive_on_device(x, order, t_T, t_0, h_init, atol, rtol, theta, t_err, solver_type)
        # host controller (schedules / options the device controller does not cover, and the CPU test executor):
        # the controller's scalars live on the host (fp32, reference op order); the network receives
        # device time labels, uploaded once per iteration
        s = t_T * torch.ones((1,))
        lambda_s = ns.marginal_lambda(s)
        lambda_0 = ns.marginal_lambda(t_0 * torch.ones_like(s))
        h = h_init * torch.ones_like(s)
        x_prev = x
        nfe = 0
        if order not in (2, 3):
            raise ValueError("For adaptive step size solver, order must be 2 or 3, got {}".format(order))
        if solver_type not in ['dpmsolver', 'taylor']:
            raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
        while torch.abs((s - t_0)).mean() > t_err:
            t = ns.inverse_lambda(lambda_s + h)
            if order == 2:      # DPM-Solver-12 (:985-988)
                sp_low = P.SinglestepPlan(1, [P._cpu(s)], [P.first_update_coeffs(ns, self.algorithm_type, s, t)])
                sp_high = P.singlestep_second(ns, self.algorithm_type, solver_type, s, t, 0.5)
            else:               # DPM-Solver-23 (:989-992)
                sp_low = P.singlestep_second(ns, self.algorithm_type, solver_type, s, t, 1. / 3.)
                sp_high = P.singlestep_third(ns, self.algorithm_type, solver_type, s, t, 1. / 3., 2. / 3.)
            t_all = self._upload(torch.cat([tt.reshape(-1) for tt in sp_high.times]), device)
            td = [t_all[j:j + 1] for j in range(len(sp_high.times))]
            x_lower, ms = self._run_singlestep(x, sp_low, keep=True, times_dev=td[:len(sp_low.times)])
            x_higher, _ = self._run_singlestep(x, sp_high, model_s=ms[0], model_s1=ms[1] if order == 3 else None,
                                               times_dev=td)
            # E = max_b sqrt(mean(((x_higher - x_lower)/delta)^2)), delta = max(atol, rtol*max(|x_lower|,|x_prev|))
            # (:999-1001): one fused reduction launch; the accept/reject test needs E on the host (:1002)
            E = ops.backend().error_norm(x_higher, x_lower, self._state_like(x_prev, x_higher.dtype), atol, rtol)
            if self.plan_broadcast and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                # batch-sharded run: E is a max over the batch (:1001), so one 4-byte all-reduce(max) per
                # iteration makes every rank take the single-process controller's decisions (SURVEY 8e)
                E = E.reshape(1).float()
                dist.all_reduce(E, op=dist.ReduceOp.MAX)
            E = E.cpu()
            if bool(torch.isnan(E).any()):
                # the reference would reject the step, set h = NaN and spin forever (s never advances, :1002-1008)
                raise FloatingPointError("dpm_solver_adaptive: the error estimate is NaN (the network output diverged)")
            if torch.all(E <= 1.):
                x = x_higher
                s = t
                x_prev = x_lower
                lambda_s = ns.marginal_lambda(s)
            h = torch.min(theta * h * torch.float_power(E, -1. / order).float(), lambda_0 - lambda_s)
            nfe += order
        print('adaptive solver nfe', nfe)
        return x

    adaptive_controller = "device"   # "host": the reference's per-iteration host decision (one sync per iteration)
    adaptive_chunk = 4               # iterations enqueued between two reads of the device-side `done` flag

    def _device_controller_ok(self, x) -> bool:
        be = ops.backend()
        w = self._wrapped
        return (self.adaptive_controller == "device" and hasattr(be, "adaptive_controller") and x.is_cuda
                and getattr(self.noise_schedule, "schedule", None) in ops.AdaptiveController.SUPPORTED
                and not self._dynamic_thresholding        # the quantile call takes alpha_t, sigma_t by value
                and not self.reference_rounding
                and not (isinstance(w, WrappedModel) and not w.fusable)      # classifier guidance: model_fn needs host scalars
                and not torch.cuda.is_current_stream_capturing())

    def _adaptive_on_device(self, x, order, t_T, t_0, h_init, atol, rtol, theta, t_err, solver_type):
        """dpm_solver_adaptive with the controller on the device (csrc/adaptive_ctl.cu): s, lambda_s, h and the
        accept/reject decision never visit the host; every fused launch reads its scalars from the coefficient
        block the plan kernel wrote; `adaptive_chunk` iterations are enqueued per read of the `done` flag."""
        be, ns = ops.backend(), self.noise_schedule
        w = self._wrapped
        discrete_in = isinstance(w, WrappedModel) and w.noise_schedule.schedule == 'discrete'
        ctl = be.adaptive_controller(ns, x.device, order=order, predict_x0=self._pp, taylor=solver_type == 'taylor',
                                     t_0=t_0, theta=theta, t_err=t_err, discrete_input=discrete_in)
        ctl.init(t_T, h_init)
        x = x.clone()                 # the committed state: overwritten in place by accepted steps
        x_prev = x.clone()
        # (a 16-bit x_T reaches the network widened to fp32 here -- same values; the by-identity hand-over of the
        # caller's own tensor at the first evaluation, `_net_input`, cannot follow a buffer that is updated in place)
        self._net_input = None
        rows = w.input_rows(x.shape[0]) if isinstance(w, WrappedModel) else x.shape[0]
        C = P.Coeffs
        if order == 2:     # DPM-Solver-12 (:985-988): coefficient blocks 0 (lower), 1 (x -> x_s1), 2 (higher)
            sp_low = P.SinglestepPlan(1, [None], [C(FORM_LIN1, 0., 0., order=1, dev=ctl.block(0))])
            sp_high = P.SinglestepPlan(2, [None, None], [C(FORM_LIN1, 0., 0., order=2, dev=ctl.block(1)),
                                                         C(ops.FORM_DIFF2, 0., 0., w0=1.0, c0_on_old=True, order=2, dev=ctl.block(2))])
        else:              # DPM-Solver-23 (:989-992): blocks 0 (x -> x_s1), 1 (lower), 2 (x -> x_s2), 3 (higher)
            sp_low = P.SinglestepPlan(2, [None, None], [C(FORM_LIN1, 0., 0., order=2, dev=ctl.block(0)),
                                                        C(ops.FORM_DIFF2, 0., 0., w0=1.0, c0_on_old=True, order=2, dev=ctl.block(1))])
            fin = C(FORM_SS3T, 0., 0., order=3, dev=ctl.block(3)) if solver_type == 'taylor' else \
                C(ops.FORM_DIFF2, 0., 0., w0=1.0, c0_on_old=True, order=3, dev=ctl.block(3))
            sp_high = P.SinglestepPlan(3, [None, None, None], [C(FORM_LIN1, 0., 0., order=3, dev=ctl.block(0)),
                                                               C(ops.FORM_DIFF2, 0., 0., w0=1.0, c0_on_old=True, order=3, dev=ctl.block(2)),
                                                               fin])
        n_high = len(sp_high.times)
        td = [ctl.time(j) for j in range(n_high)]
        tin = [ctl.input_time(j).expand(rows) for j in range(n_high)] if discrete_in else [None] * n_high
        dev_als = [_DEV] * n_high
        sharded = self.plan_broadcast and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        n_low = len(sp_low.times)
        while True:
            for _ in range(max(1, int(self.adaptive_chunk))):
                ctl.plan()
                x_lower, ms = self._run_singlestep(x, sp_low, keep=True, times_dev=td[:n_low], alsig=dev_als[:n_low],
                                                   t_inputs=tin[:n_low])
                x_higher, _ = self._run_singlestep(x, sp_high, model_s=ms[0], model_s1=ms[1] if order == 3 else None,
                                                   times_dev=td, alsig=dev_als, t_inputs=tin)
                be.error_norm(x_higher, x_lower, x_prev, atol, rtol, out=ctl.E)      # :999-1001, one fused reduction
                if sharded:
                    dist.all_reduce(ctl.E, op=dist.ReduceOp.MAX)                    # E is a max over the batch (:1001)
                ctl.decide()                                                          # :1002-1008 on the device
                ctl.select_copy(x, x_higher)
                ctl.select_copy(x_prev, x_lower)
            done, nfe, _ = ctl.read()                                                 # the chunk's only host sync
            if done == 2:
                raise FloatingPointError("dpm_solver_adaptive: the error estimate is NaN (the network output diverged)")
            if done:
                break
        print('adaptive solver nfe', nfe)
        return x

    # -- add_noise / inverse (:1012-1045) --------------------------------------------------------
    def add_noise(self, x, t, noise=None):
        """xt = alpha_t * x + sigma_t * noise for every t in `t` -> (t_size, batch, *shape)."""
        th = P._cpu(t)
        alpha_t, sigma_t = self.noise_schedule.marginal_alpha(th), self.noise_schedule.marginal_std(th)
        be = ops.backend()
        if noise is None and x.is_cuda and hasattr(be, "add_noise_philox") and th.shape[0] <= 16 \
                and x.dtype in ops.SUPPORTED_DTYPES and not torch.cuda.is_current_stream_capturing():
            # the noise never touches HBM: drawn in registers by the generator torch.randn would have used, same
            # (seed, offset) -> same values, the torch generator advanced as randn would have (csrc/philox.cu)
            xs = self._state_like(x, x.dtype)
            outs = be.add_noise_philox(xs, alpha_t.tolist(), sigma_t.tolist(), self._sdtype(x))
            return outs[0] if th.shape[0] == 1 else outs
        if noise is None:
            noise = torch.randn((th.shape[0], *x.shape), device=x.device)
        # result dtype: the reference's fp32 (t_size,1,..) coefficient tensors promote a 16-bit x to fp32 (:1026)
        xs = self._state_like(x, self._sdtype(x))
        noise = noise.reshape((th.shape[0], *x.shape))
        outs = [ops.lincomb(xs, [self._state_like(noise[i], xs.dtype)], float(alpha_t[i]), [float(sigma_t[i])])
                for i in range(th.shape[0])]
        if th.shape[0] == 1:
            return outs[0]
        return torch.stack(outs)

    def inverse(self, x, steps=20, t_start=None, t_end=None, order=2, skip_type='time_uniform',
                method='multistep', lower_order_final=True, denoise_to_zero=False, solver_type='dpmsolver',
                atol=0.0078, rtol=0.05, return_intermediate=False):
        """Invert `x` from t_start (default 1/N) to t_end (default T) (:1032-1045)."""
        self._no_sde("inverse()")
        t_0 = 1. / self.noise_schedule.total_N if t_start is None else t_start
        t_T = self.noise_schedule.T if t_end is None else t_end
        assert t_0 > 0 and t_T > 0, "Time range needs to be greater than 0. For discrete-time DPMs, it needs to be in [1 / N, 1], where N is the length of betas array"
        return self.sample(x, steps=steps, t_start=t_0, t_end=t_T, order=order, skip_type=skip_type,
                           method=method, lower_order_final=lower_order_final, denoise_to_zero=denoise_to_zero,
                           solver_type=solver_type, atol=atol, rtol=rtol, return_intermediate=return_intermediate)

    # -- whole-loop CUDA graph (SURVEY 8f-1; no counterpart in the reference) -----------------------
    def capture(self, x_example, **sample_kwargs):
        """Capture `sample(x, **sample_kwargs)` -- the network calls included -- in ONE CUDA graph.

        Once the coefficient plan and the device tables are cached, the sampling loop performs no
        host<->device copy, no synchronisation and no collective, and every kernel takes its scalars
        by value, so the whole run is capturable whenever the network is. Returns a callable
        `g(x) -> x_0` that copies `x` into the graph's static input and replays; the returned tensor
        is the graph's static output (clone it to keep it across replays). Not available for the
        adaptive method (host-side accept/reject) or with python-side hooks that synchronise."""
        if sample_kwargs.get("method", "multistep") == "adaptive":
            raise ValueError("the adaptive solver decides on the host every iteration; it cannot be captured")
        if sample_kwargs.get("return_intermediate"):
            raise ValueError("capture() returns the final sample only")
        gen = sample_kwargs.get("generator")
        if self._sde and gen is not None and gen is not torch.cuda.default_generators[torch.device(gen.device).index or 0]:
            # the noise of a captured SDE run is drawn inside the graph, which only the default generator follows
            raise ValueError("capture() of algorithm_type={!r} draws its noise from the default CUDA generator; "
                             "pass generator=None".format(self.algorithm_type))
        x_static = self._state(x_example).clone()
        self.sample(x_static, **sample_kwargs)                       # builds and caches plan + tables
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=x_static.device)
        side.wait_stream(torch.cuda.current_stream(x_static.device))
        with torch.cuda.stream(side):
            self.sample(x_static, **sample_kwargs)                   # warm-up on the capture stream
            with torch.cuda.graph(graph, stream=side):
                y_static = self.sample(x_static, **sample_kwargs)
        torch.cuda.current_stream(x_static.device).wait_stream(side)

        def replay(x):
            x_static.copy_(x)
            graph.replay()
            return y_static

        replay.graph, replay.static_input, replay.static_output = graph, x_static, y_static
        return replay

    # -- sample (:1047-1245) ---------------------------------------------------------------------
    def sample(self, x, steps=20, t_start=None, t_end=None, order=2, skip_type='time_uniform',
               method='multistep', lower_order_final=True, denoise_to_zero=False, solver_type='dpmsolver',
               atol=0.0078, rtol=0.05, return_intermediate=False, generator=None):
        """Integrate the diffusion ODE from t_start to t_end; arguments as in the reference.

        For algorithm_type "sde-dpmsolver++" / "sde-dpmsolver" (method='multistep', order 1 or 2) the diffusion SDE is
        integrated instead: every step adds fresh Gaussian noise, drawn in the step kernel from `generator` (a
        torch.Generator on x's device; None = that device's default generator). The ODE algorithms ignore it."""
        t_0 = 1. / self.noise_schedule.total_N if t_end is None else t_end
        t_T = self.noise_schedule.T if t_start is None else t_start
        assert t_0 > 0 and t_T > 0, "Time range needs to be greater than 0. For discrete-time DPMs, it needs to be in [1 / N, 1], where N is the length of betas array"
        if return_intermediate:
            assert method in ['multistep', 'singlestep', 'singlestep_fixed'], "Cannot use adaptive solver when saving intermediate values"
        if self.correcting_xt_fn is not None:
            assert method in ['multistep', 'singlestep', 'singlestep_fixed'], "Cannot use adaptive solver when correcting_xt_fn is not None"
        device = x.device
        if self._sde:
            if method != 'multistep':
                self._no_sde("method={!r}".format(method))
            if order not in (1, 2):
                raise ValueError("algorithm_type={!r} is served by multistep orders 1 and 2, got order {}".format(
                    self.algorithm_type, order))
            ops.check_generator(generator, device)
        self._generator = generator if self._sde else None
        intermediates = []
        ns = self.noise_schedule
        self._xin_pair = None
        self._rr_run = 0
        # prepared launches: the CUDA executor, no python-side x0 hook, no 16-bit reference-rounding mode
        # (not for the SDE algorithms: a frozen descriptor launches dpm_step, which adds no noise)
        self._prep_on = (hasattr(ops.backend(), "prepare") and not self.reference_rounding and not self._sde
                         and (self.correcting_x0_fn is None or self._dynamic_thresholding))
        with torch.no_grad():
            x = self._state(x)
            sd = x.dtype
            if method == 'adaptive':
                x = self.dpm_solver_adaptive(x, order=order, t_T=t_T, t_0=t_0, atol=atol, rtol=rtol,
                                             solver_type=solver_type)
                step = 0
            elif method == 'multistep':
                assert steps >= order
                if solver_type not in ['dpmsolver', 'taylor'] and order >= 2:
                    raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
                if order not in (1, 2, 3):
                    raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))
                key = ("multistep", steps, order, skip_type, t_T, t_0, solver_type, lower_order_final)

                def build():
                    ts = self.get_time_steps(skip_type=skip_type, t_T=t_T, t_0=t_0, N=steps, device='cpu')
                    assert ts.shape[0] - 1 == steps
                    marg = P.Marginals(ns, ts)
                    mk = P.sde_multistep_plan if self._sde else P.multistep_plan
                    plan = mk(ns, self.algorithm_type, solver_type, ts, order, lower_order_final, marginals=marg)
                    # (alpha_t, sigma_t) per grid point: scalars of the eps->x0 / parameterisation step
                    return ts, plan, list(zip(marg.alpha.tolist(), marg.sigma.tolist()))

                ts, plan, alsig = self._host_plan(key, build)
                plan = self._sync_plan(plan, key)
                _, _, ts_dev, _, tin = self._device_tables(key, ts, x.shape[0], device)   # lists of per-step views
                # model evaluation 0, then one fused launch per step:
                #   m_{i} = convert(net(x_i, t_i));  x_{i+1} = update(x_i, m_i, m_{i-1}, m_{i-2})
                step = 0
                pid = self._plan_id(key)
                raw = self._evaluate(x, ts_dev[0], None if tin is None else tin[0])
                xe = x
                if self.correcting_xt_fn is not None:
                    x = self._state_like(self.correcting_xt_fn(x, ts_dev[0], step), sd)
                if return_intermediate:
                    intermediates.append(x)
                older: List[torch.Tensor] = []  # buffered model values, newest last
                for step in range(1, steps + 1):
                    co = plan[step - 1]
                    m1 = older[-1] if co.order >= 2 else None
                    m2 = older[-2] if co.order >= 3 else None
                    want = order >= 2 and step < steps
                    m_new, x_new = self._post_model(raw, xe, ts_dev[step - 1], alsig[step - 1], co, x,
                                                    m1, m2, want_m=want, dup_out=step < steps,
                                                    slot=(pid, step))
                    x = x_new
                    t = ts_dev[step]
                    if self.correcting_xt_fn is not None:
                        x = self._state_like(self.correcting_xt_fn(x, t, step), sd)
                    if return_intermediate:
                        intermediates.append(x)
                    if m_new is not None:
                        older.append(m_new)
                        if len(older) > 2:
                            older.pop(0)
                    # We do not need to evaluate the final model value.
                    if step < steps:
                        raw = self._evaluate(x, t, None if tin is None else tin[step])
                        xe = x
            elif method in ['singlestep', 'singlestep_fixed']:
                key = (method, steps, order, skip_type, t_T, t_0, solver_type)

                def build():
                    if method == 'singlestep':
                        timesteps_outer, orders = self.get_orders_and_timesteps_for_singlestep_solver(
                            steps=steps, order=order, skip_type=skip_type, t_T=t_T, t_0=t_0, device='cpu')
                    else:
                        K = steps // order
                        orders = [order, ] * K
                        timesteps_outer = self.get_time_steps(skip_type=skip_type, t_T=t_T, t_0=t_0, N=K, device='cpu')
                    if solver_type not in ['dpmsolver', 'taylor'] and max(orders) >= 2:
                        raise ValueError("'solver_type' must be either 'dpmsolver' or 'taylor', got {}".format(solver_type))
                    # host plan for the whole run (:1221-1228 evaluated up front, no .item() syncs later)
                    plans = []
                    for i, o in enumerate(orders):
                        s_, t_ = timesteps_outer[i], timesteps_outer[i + 1]
                        timesteps_inner = self.get_time_steps(skip_type=skip_type, t_T=s_.item(), t_0=t_.item(), N=o, device='cpu')
                        lambda_inner = ns.marginal_lambda(timesteps_inner)
                        h = lambda_inner[-1] - lambda_inner[0]
                        r1 = None if o <= 1 else (lambda_inner[1] - lambda_inner[0]) / h
                        r2 = None if o <= 2 else (lambda_inner[2] - lambda_inner[0]) / h
                        plans.append(P.singlestep_plan(ns, self.algorithm_type, solver_type, o, s_, t_, r1, r2))
                    if not plans:
                        # steps < order with 'singlestep_fixed': K = 0, the reference runs no outer step (:1216-1220)
                        return timesteps_outer.reshape(-1), plans, []
                    all_times = torch.cat([tt.reshape(-1) for sp in plans for tt in sp.times])
                    marg = P.Marginals(ns, all_times)
                    return (torch.cat([all_times, timesteps_outer.reshape(-1)]), plans,
                            list(zip(marg.alpha.tolist(), marg.sigma.tolist())))

                packed, plans, alsig = self._host_plan(key, build)
                if self.plan_broadcast and plans:
                    flat = self._sync_plan([co for sp in plans for co in sp.stages], key)
                    plans = [P.SinglestepPlan(sp.order, sp.times, []) for sp in plans]
                    k = 0
                    for sp in plans:
                        n_st = {1: 1, 2: 2, 3: 3}[sp.order]
                        sp.stages = flat[k:k + n_st]
                        k += n_st
                n_eval = len(alsig)
                _, _, _, packed1, tin = self._device_tables(key, packed, x.shape[0], device, n_eval) if plans \
                    else (None, None, None, None, None)
                all_dev, outer_dev = (packed1[:n_eval], packed1[n_eval:]) if plans else (None, None)
                k = 0
                step = 0
                pid = self._plan_id(key)
                for step, sp in enumerate(plans):
                    nt = len(sp.times)
                    td = all_dev[k:k + nt]
                    x, _ = self._run_singlestep(x, sp, times_dev=td, alsig=alsig[k:k + nt],
                                                t_inputs=None if tin is None else tin[k:k + nt],
                                                dup_last=step + 1 < len(plans), slot=(pid, step))
                    k += nt
                    if self.correcting_xt_fn is not None:
                        x = self._state_like(self.correcting_xt_fn(x, outer_dev[step + 1].reshape(()), step), sd)
                    if return_intermediate:
                        intermediates.append(x)
            else:
                raise ValueError("Got wrong method {}".format(method))
            if denoise_to_zero:
                # :1236-1238. The label, its model-input time and (alpha, sigma) at t_0 are cached with the tables:
                # no host<->device traffic in the steady state, so the tail is CUDA-graph capturable too
                t, tin0, als0 = self._denoise_tables(t_0, x.shape[0], device)
                xs = self._state(x)
                x = self._post_model(self._evaluate(xs, t, tin0), xs, t, als0, x0=True)[0]
                if self.correcting_xt_fn is not None:
                    x = self.correcting_xt_fn(x, t, step + 1)
                if return_intermediate:
                    intermediates.append(x)
        self._net_input = None
        self._generator = None
        if return_intermediate:
            return x, intermediates
        else:
            return x
