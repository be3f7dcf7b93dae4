"""Host-side coefficient plan.

Every DPM-Solver update is `x_t = a*x + c0*T0 + c1*T1 + c2*T2` where the T_j are buffered model
values or differences of them (include/dpm_solver_b200.h, `dpm_form`). This module computes the
scalars (a, c_j, w_j) on the HOST, in fp32, in the reference's operation order
(dpm_solver_pytorch.py:563-588, :616-669, :702-789, :815-851, :871-903), vectorised over all
steps of a run, so that the device executes one fused kernel per step and no exp/log/expm1,
no interpolation and no host<->device sync happens inside the sampling loop.

The arithmetic deliberately goes through the same torch CPU scalar ops the reference uses
(`torch.expm1`, `1. / r`, tensor/python-float promotion ...): the resulting fp32 scalars are
bit-identical to the reference evaluated on CPU. All `t` arguments are 1-D fp32 CPU tensors.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Union

import torch

from ._lib import FORM_DIFF2, FORM_LIN1, FORM_MS3, FORM_SS3T

Number = Union[float, torch.Tensor]


@dataclass
class Coeffs:
    """Scalars of one launch (python floats holding exact fp32 values, signs folded in)."""
    form: int
    a: float
    c0: float
    c1: float = 0.0
    c2: float = 0.0
    w0: float = 0.0
    w1: float = 0.0
    w2: float = 0.0
    w3: float = 0.0
    w4: float = 0.0
    c0_on_old: bool = False
    order: int = 1
    r_tensor: int = 0   # SS3T: bit 0 / 1 = r1 / r2 came as tensors (matters to reference_rounding only)
    dev: Optional[torch.Tensor] = None   # scalars live in this device block instead (on-device adaptive controller)
    cn: float = 0.0     # SDE steps: coefficient of the fresh Gaussian noise z (dpm_sde_step's noise_scale)


def _cpu(t: torch.Tensor) -> torch.Tensor:
    """Time label(s) as a 1-D CPU tensor (syncs if `t` lives on a device)."""
    if not torch.is_tensor(t):
        t = torch.tensor(t)
    return t.detach().reshape(-1).cpu()


def _f(v: Number, i: int = 0) -> float:
    """i-th scalar as a python float; c_float conversion then rounds exactly like torch's
    python-scalar -> fp32 cast."""
    if torch.is_tensor(v):
        return float(v.reshape(-1)[i]) if v.numel() > 1 else float(v)
    return float(v)


class Marginals:
    """log(alpha), alpha, sigma, lambda of a vector of times (one vectorised pass; the expressions
    are those of marginal_log_mean_coeff / marginal_std / marginal_lambda / marginal_alpha,
    :127-154, sharing the single evaluation of log(alpha))."""

    def __init__(self, ns, t: Optional[torch.Tensor]):
        if t is None:
            return
        self.t = t
        self.log_alpha = ns.marginal_log_mean_coeff(t)
        e2 = 1. - torch.exp(2. * self.log_alpha)
        self.sigma = torch.sqrt(e2)                           # :146
        self.lam = self.log_alpha - 0.5 * torch.log(e2)       # :153-154
        self.alpha = torch.exp(self.log_alpha)                # :140

    def __getitem__(self, i) -> "Marginals":
        m = Marginals(None, None)
        m.t, m.log_alpha, m.sigma, m.lam, m.alpha = self.t[i], self.log_alpha[i], self.sigma[i], self.lam[i], self.alpha[i]
        return m


# ---- order 1 ----------------------------------------------------------------------------------

def first_update(ns, algorithm_type: str, s: torch.Tensor, t: torch.Tensor):
    """Vectorised dpm_solver_first_update scalars (:563-588) -> tensors (a, c0)."""
    return _first(algorithm_type, Marginals(ns, s), Marginals(ns, t))


def _first(algorithm_type: str, ms: Marginals, mt: Marginals):
    h = mt.lam - ms.lam
    if algorithm_type == "dpmsolver++":
        phi_1 = torch.expm1(-h)
        a = mt.sigma / ms.sigma
        c0 = -(mt.alpha * phi_1)
    else:
        phi_1 = torch.expm1(h)
        a = torch.exp(mt.log_alpha - ms.log_alpha)
        c0 = -(mt.sigma * phi_1)
    return a, c0


def first_update_coeffs(ns, algorithm_type, s, t) -> Coeffs:
    a, c0 = first_update(ns, algorithm_type, _cpu(s), _cpu(t))
    return Coeffs(FORM_LIN1, _f(a), _f(c0), order=1)


# ---- multistep --------------------------------------------------------------------------------

def multistep_second(ns, algorithm_type, solver_type, t_prev_1, t_prev_0, t):
    """multistep_dpm_solver_second_update scalars (:815-851) -> tensors (a, c0, c1, inv_r0)."""
    return _ms2(algorithm_type, solver_type, Marginals(ns, t_prev_1), Marginals(ns, t_prev_0), Marginals(ns, t))


def _ms2(algorithm_type, solver_type, m1: Marginals, m0: Marginals, mt: Marginals):
    h_0 = m0.lam - m1.lam
    h = mt.lam - m0.lam
    r0 = h_0 / h
    inv_r0 = 1. / r0
    if algorithm_type == "dpmsolver++":
        phi_1 = torch.expm1(-h)
        a = mt.sigma / m0.sigma
        b = mt.alpha * phi_1
        c1 = -(0.5 * b) if solver_type == "dpmsolver" else mt.alpha * (phi_1 / h + 1.)
    else:
        phi_1 = torch.expm1(h)
        a = torch.exp(mt.log_alpha - m0.log_alpha)
        b = mt.sigma * phi_1
        c1 = -(0.5 * b) if solver_type == "dpmsolver" else -(mt.sigma * (phi_1 / h - 1.))
    return a, -b, c1, inv_r0


def multistep_third(ns, algorithm_type, t_prev_2, t_prev_1, t_prev_0, t):
    """multistep_dpm_solver_third_update scalars (:871-903); solver_type is ignored there."""
    return _ms3(algorithm_type, *(Marginals(ns, v) for v in (t_prev_2, t_prev_1, t_prev_0, t)))


def _ms3(algorithm_type, m2: Marginals, m1: Marginals, m0: Marginals, mt: Marginals):
    h_1 = m1.lam - m2.lam
    h_0 = m0.lam - m1.lam
    h = mt.lam - m0.lam
    r0, r1 = h_0 / h, h_1 / h
    w0, w1 = 1. / r0, 1. / r1
    w2 = r0 / (r0 + r1)
    w3 = 1. / (r0 + r1)
    if algorithm_type == "dpmsolver++":
        phi_1 = torch.expm1(-h)
        phi_2 = phi_1 / h + 1.
        phi_3 = phi_2 / h - 0.5
        a = mt.sigma / m0.sigma
        c0, c1, c2 = -(mt.alpha * phi_1), mt.alpha * phi_2, -(mt.alpha * phi_3)
    else:
        phi_1 = torch.expm1(h)
        phi_2 = phi_1 / h - 1.
        phi_3 = phi_2 / h - 0.5
        a = torch.exp(mt.log_alpha - m0.log_alpha)
        c0, c1, c2 = -(mt.sigma * phi_1), -(mt.sigma * phi_2), -(mt.sigma * phi_3)
    return a, c0, c1, c2, w0, w1, w2, w3


def multistep_coeffs(ns, algorithm_type, solver_type, order, t_prev_list, t) -> Coeffs:
    """Scalars of one multistep update of the given order (direct-call path)."""
    tp = [_cpu(v) for v in t_prev_list]
    t = _cpu(t)
    if order == 1:
        return first_update_coeffs(ns, algorithm_type, tp[-1], t)
    if order == 2:
        a, c0, c1, w0 = multistep_second(ns, algorithm_type, solver_type, tp[-2], tp[-1], t)
        return Coeffs(FORM_DIFF2, _f(a), _f(c0), _f(c1), w0=_f(w0), order=2)
    if order == 3:
        v = multistep_third(ns, algorithm_type, tp[-3], tp[-2], tp[-1], t)
        return Coeffs(FORM_MS3, *(_f(u) for u in v[:4]), w0=_f(v[4]), w1=_f(v[5]), w2=_f(v[6]),
                      w3=_f(v[7]), order=3)
    raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))


def multistep_orders(steps: int, order: int, lower_order_final: bool) -> List[int]:
    """Order used at update `step` = 1..steps (sample() :1185-1201)."""
    out = []
    for step in range(1, steps + 1):
        if step < order:
            out.append(step)
        elif lower_order_final and steps < 10:
            out.append(min(order, steps + 1 - step))
        else:
            out.append(order)
    return out


def multistep_plan(ns, algorithm_type, solver_type, timesteps: torch.Tensor, order: int,
                   lower_order_final: bool, marginals: Optional[Marginals] = None) -> List[Coeffs]:
    """Coefficients of every update of a multistep run; plan[i] moves timesteps[i] -> [i+1].
    One vectorised evaluation of the schedule over the grid, then one vector op set per order."""
    ts = _cpu(timesteps)
    steps = ts.numel() - 1
    M = marginals if marginals is not None else Marginals(ns, ts)
    orders = multistep_orders(steps, order, lower_order_final)
    plan: List[Optional[Coeffs]] = [None] * steps
    idx = {p: [i for i, o in enumerate(orders) if o == p] for p in (1, 2, 3)}
    if idx[1]:
        i = torch.tensor(idx[1])
        a, c0 = (v.reshape(-1).tolist() for v in _first(algorithm_type, M[i], M[i + 1]))
        for k, j in enumerate(idx[1]):
            plan[j] = Coeffs(FORM_LIN1, a[k], c0[k], order=1)
    if idx[2]:
        i = torch.tensor(idx[2])
        a, c0, c1, w0 = (v.reshape(-1).tolist() for v in _ms2(algorithm_type, solver_type, M[i - 1], M[i], M[i + 1]))
        for k, j in enumerate(idx[2]):
            plan[j] = Coeffs(FORM_DIFF2, a[k], c0[k], c1[k], w0=w0[k], order=2)
    if idx[3]:
        i = torch.tensor(idx[3])
        v = [u.reshape(-1).tolist() for u in _ms3(algorithm_type, M[i - 2], M[i - 1], M[i], M[i + 1])]
        for k, j in enumerate(idx[3]):
            plan[j] = Coeffs(FORM_MS3, v[0][k], v[1][k], v[2][k], v[3][k], w0=v[4][k], w1=v[5][k], w2=v[6][k],
                             w3=v[7][k], order=3)
    return plan  # type: ignore[return-value]


# ---- stochastic multistep (SDE-DPM-Solver / SDE-DPM-Solver++) ---------------------------------
# Step s -> t, h = lambda_t - lambda_s (s = newest buffered time), D0 = m0, D1 = (1/r0)*(m0 - m1), z ~ N(0, I):
#   x_t = a*x + c0*D0 + c1*D1 + cn*z      (order 1: no c1 term)
# sde-dpmsolver++ (data prediction):  a = (sigma_t/sigma_s)*exp(-h), c0 = -(alpha_t*expm1(-2h)),
#     c1 = 0.5*c0 ('dpmsolver') | alpha_t*(expm1(-2h)/(2h) + 1) ('taylor'),  cn = sigma_t*sqrt(-expm1(-2h))
# sde-dpmsolver (noise prediction):   a = exp(log_alpha_t - log_alpha_s), c0 = -2*sigma_t*expm1(h),
#     c1 = -(sigma_t*expm1(h)) ('dpmsolver') | -2*sigma_t*(expm1(h)/h - 1) ('taylor'),  cn = sigma_t*sqrt(expm1(2h))
# (the 'midpoint' and 'heun' second-order terms of the SDE solvers in Hugging Face diffusers, with expm1 in place of
# exp - 1). Every scalar is one fp32 torch CPU op chain in the order written in _sde below.
SDE_ALGORITHMS = ("sde-dpmsolver", "sde-dpmsolver++")


def _sde(algorithm_type: str, solver_type: str, ms: Marginals, mt: Marginals, order: int):
    """(a, c0, c1, cn) tensors of SDE steps ms -> mt (c1 is zero for order 1)."""
    h = mt.lam - ms.lam
    if algorithm_type == "sde-dpmsolver++":
        em = torch.expm1(-2. * h)
        a = (mt.sigma / ms.sigma) * torch.exp(-h)
        c0 = -(mt.alpha * em)
        if order == 1:
            c1 = torch.zeros_like(c0)
        elif solver_type == "dpmsolver":
            c1 = 0.5 * c0
        else:
            c1 = mt.alpha * (em / (2. * h) + 1.)
        cn = mt.sigma * torch.sqrt(-em)
    elif algorithm_type == "sde-dpmsolver":
        ep = torch.expm1(h)
        a = torch.exp(mt.log_alpha - ms.log_alpha)
        c0 = -2. * (mt.sigma * ep)
        if order == 1:
            c1 = torch.zeros_like(c0)
        elif solver_type == "dpmsolver":
            c1 = -(mt.sigma * ep)
        else:
            c1 = -2. * (mt.sigma * (ep / h - 1.))
        cn = mt.sigma * torch.sqrt(torch.expm1(2. * h))
    else:
        raise ValueError("not an SDE algorithm_type: {!r}".format(algorithm_type))
    return a, c0, c1, cn


def sde_multistep_plan(ns, algorithm_type, solver_type, timesteps: torch.Tensor, order: int,
                       lower_order_final: bool, marginals: Optional[Marginals] = None) -> List[Coeffs]:
    """Coefficients of every step of a stochastic multistep run (orders 1 and 2; the order schedule of
    multistep_orders); plan[i] moves timesteps[i] -> [i+1]. Order 1 steps are LIN1, order 2 steps DIFF2 with
    w0 = 1/r0 exactly as in multistep_plan."""
    if order not in (1, 2):
        raise ValueError("{} is served by multistep orders 1 and 2, got order {}".format(algorithm_type, order))
    ts = _cpu(timesteps)
    steps = ts.numel() - 1
    M = marginals if marginals is not None else Marginals(ns, ts)
    orders = multistep_orders(steps, order, lower_order_final)
    plan: List[Optional[Coeffs]] = [None] * steps
    for p in (1, 2):
        idx = [i for i, o in enumerate(orders) if o == p]
        if not idx:
            continue
        i = torch.tensor(idx)
        a, c0, c1, cn = (v.reshape(-1).tolist() for v in _sde(algorithm_type, solver_type, M[i], M[i + 1], p))
        if p == 1:
            for k, j in enumerate(idx):
                plan[j] = Coeffs(FORM_LIN1, a[k], c0[k], order=1, cn=cn[k])
        else:
            h_0 = M[i].lam - M[i - 1].lam
            h = M[i + 1].lam - M[i].lam
            w0 = (1. / (h_0 / h)).reshape(-1).tolist()      # 1/r0, as multistep_plan
            for k, j in enumerate(idx):
                plan[j] = Coeffs(FORM_DIFF2, a[k], c0[k], c1[k], w0=w0[k], order=2, cn=cn[k])
    return plan  # type: ignore[return-value]


# ---- singlestep -------------------------------------------------------------------------------

@dataclass
class SinglestepPlan:
    """One outer singlestep update s -> t of order 1, 2 or 3."""
    order: int
    times: List[torch.Tensor]        # model evaluation times: [s] / [s, s1] / [s, s1, s2] (CPU, (1,))
    stages: List[Coeffs] = field(default_factory=list)  # one launch per model evaluation


def singlestep_second(ns, algorithm_type, solver_type, s, t, r1: Number = 0.5) -> SinglestepPlan:
    """singlestep_dpm_solver_second_update scalars (:613-669)."""
    if r1 is None:
        r1 = 0.5
    s, t = _cpu(s), _cpu(t)
    ms, mt = Marginals(ns, s), Marginals(ns, t)
    h = mt.lam - ms.lam
    s1 = ns.inverse_lambda(ms.lam + r1 * h)
    m1 = Marginals(ns, s1)
    if algorithm_type == "dpmsolver++":
        phi_11 = torch.expm1(-r1 * h)
        phi_1 = torch.expm1(-h)
        st1 = Coeffs(FORM_LIN1, _f(m1.sigma / ms.sigma), _f(-(m1.alpha * phi_11)), order=2)
        b = mt.alpha * phi_1
        if solver_type == "dpmsolver":
            c1 = -((0.5 / r1) * b)
        else:
            c1 = (1. / r1) * (mt.alpha * (phi_1 / h + 1.))
        fin = Coeffs(FORM_DIFF2, _f(mt.sigma / ms.sigma), _f(-b), _f(c1), w0=1.0, c0_on_old=True, order=2)
    else:
        phi_11 = torch.expm1(r1 * h)
        phi_1 = torch.expm1(h)
        st1 = Coeffs(FORM_LIN1, _f(torch.exp(m1.log_alpha - ms.log_alpha)), _f(-(m1.sigma * phi_11)), order=2)
        b = mt.sigma * phi_1
        if solver_type == "dpmsolver":
            c1 = -((0.5 / r1) * b)
        else:
            c1 = -((1. / r1) * (mt.sigma * (phi_1 / h - 1.)))
        fin = Coeffs(FORM_DIFF2, _f(torch.exp(mt.log_alpha - ms.log_alpha)), _f(-b), _f(c1), w0=1.0,
                     c0_on_old=True, order=2)
    return SinglestepPlan(2, [s, s1], [st1, fin])


def singlestep_third(ns, algorithm_type, solver_type, s, t, r1: Number = 1. / 3.,
                     r2: Number = 2. / 3.) -> SinglestepPlan:
    """singlestep_dpm_solver_third_update scalars (:697-789)."""
    if r1 is None:
        r1 = 1. / 3.
    if r2 is None:
        r2 = 2. / 3.
    rt = (1 if torch.is_tensor(r1) else 0) | (2 if torch.is_tensor(r2) else 0)
    s, t = _cpu(s), _cpu(t)
    ms, mt = Marginals(ns, s), Marginals(ns, t)
    h = mt.lam - ms.lam
    s1 = ns.inverse_lambda(ms.lam + r1 * h)
    s2 = ns.inverse_lambda(ms.lam + r2 * h)
    m1, m2 = Marginals(ns, s1), Marginals(ns, s2)
    pp = algorithm_type == "dpmsolver++"
    if pp:
        phi_11 = torch.expm1(-r1 * h)
        phi_12 = torch.expm1(-r2 * h)
        phi_1 = torch.expm1(-h)
        phi_22 = torch.expm1(-r2 * h) / (r2 * h) + 1.
        phi_2 = phi_1 / h + 1.
        phi_3 = phi_2 / h - 0.5
        a1, a2, at = m1.sigma / ms.sigma, m2.sigma / ms.sigma, mt.sigma / ms.sigma
        g1, g2, gt = m1.alpha, m2.alpha, mt.alpha
        st1 = Coeffs(FORM_LIN1, _f(a1), _f(-(g1 * phi_11)), order=3)
        st2 = Coeffs(FORM_DIFF2, _f(a2), _f(-(g2 * phi_12)), _f(r2 / r1 * (g2 * phi_22)), w0=1.0,
                     c0_on_old=True, order=3)
        if solver_type == "dpmsolver":
            fin = Coeffs(FORM_DIFF2, _f(at), _f(-(gt * phi_1)), _f((1. / r2) * (gt * phi_2)), w0=1.0,
                         c0_on_old=True, order=3)
        else:
            fin = Coeffs(FORM_SS3T, _f(at), _f(-(gt * phi_1)), _f(gt * phi_2), _f(-(gt * phi_3)),
                         w0=_f(1. / r1), w1=_f(1. / r2), w2=_f(r2), w3=_f(r1), w4=_f(r2 - r1), order=3, r_tensor=rt)
    else:
        phi_11 = torch.expm1(r1 * h)
        phi_12 = torch.expm1(r2 * h)
        phi_1 = torch.expm1(h)
        phi_22 = torch.expm1(r2 * h) / (r2 * h) - 1.
        phi_2 = phi_1 / h - 1.
        phi_3 = phi_2 / h - 0.5
        a1 = torch.exp(m1.log_alpha - ms.log_alpha)
        a2 = torch.exp(m2.log_alpha - ms.log_alpha)
        at = torch.exp(mt.log_alpha - ms.log_alpha)
        g1, g2, gt = m1.sigma, m2.sigma, mt.sigma
        st1 = Coeffs(FORM_LIN1, _f(a1), _f(-(g1 * phi_11)), order=3)
        st2 = Coeffs(FORM_DIFF2, _f(a2), _f(-(g2 * phi_12)), _f(-(r2 / r1 * (g2 * phi_22))), w0=1.0,
                     c0_on_old=True, order=3)
        if solver_type == "dpmsolver":
            fin = Coeffs(FORM_DIFF2, _f(at), _f(-(gt * phi_1)), _f(-((1. / r2) * (gt * phi_2))), w0=1.0,
                         c0_on_old=True, order=3)
        else:
            fin = Coeffs(FORM_SS3T, _f(at), _f(-(gt * phi_1)), _f(-(gt * phi_2)), _f(-(gt * phi_3)),
                         w0=_f(1. / r1), w1=_f(1. / r2), w2=_f(r2), w3=_f(r1), w4=_f(r2 - r1), order=3, r_tensor=rt)
    return SinglestepPlan(3, [s, s1, s2], [st1, st2, fin])


def singlestep_plan(ns, algorithm_type, solver_type, order, s, t, r1=None, r2=None) -> SinglestepPlan:
    if order == 1:
        s = _cpu(s)
        return SinglestepPlan(1, [s], [first_update_coeffs(ns, algorithm_type, s, t)])
    if order == 2:
        return singlestep_second(ns, algorithm_type, solver_type, s, t, r1)
    if order == 3:
        return singlestep_third(ns, algorithm_type, solver_type, s, t, r1, r2)
    raise ValueError("Solver order must be 1 or 2 or 3, got {}".format(order))


def singlestep_orders(steps: int, order: int) -> List[int]:
    """Orders of 'DPM-Solver-fast' for a budget of `steps` evaluations (:514-533)."""
    if order == 3:
        K = steps // 3 + 1
        if steps % 3 == 0:
            return [3, ] * (K - 2) + [2, 1]
        elif steps % 3 == 1:
            return [3, ] * (K - 1) + [1]
        return [3, ] * (K - 1) + [2]
    if order == 2:
        if steps % 2 == 0:
            return [2, ] * (steps // 2)
        return [2, ] * (steps // 2) + [1]
    if order == 1:
        return [1, ] * steps
    raise ValueError("'order' must be '1' or '2' or '3'.")
