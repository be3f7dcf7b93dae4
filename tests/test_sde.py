"""Stochastic SDE-DPM-Solver(++) multistep sampling (algorithm_type "sde-dpmsolver++" / "sde-dpmsolver").

CPU: the plan scalars against float64, sample() on the numpy executor against a self-contained eager torch SDE
sampler (bit for bit, same CPU generator), the launch budget, every rejected combination, the packed plan and the
C-ABI argument checks. GPU: dpm_sde_step's in-kernel Philox noise against the same launch fed torch.randn_like from
the restored generator state and against the numpy executor, sample() against the eager spec run as torch CUDA ops,
fresh noise per call, the exact N(alpha_t x0*, sigma_t^2) marginals of a point-mass data distribution, and capture().
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from cases import exact_net, seeded
from dpm_solver_b200 import DPM_Solver, model_wrapper, ops
from dpm_solver_b200 import plan as P
from dpm_solver_b200._lib import FORM_DIFF2, FORM_LIN1, FORM_MS3
from dpm_solver_b200.ops import StepArgs
from helpers import product_schedule
from sde_oracle import SdeOracleBackend

SDE = ["sde-dpmsolver++", "sde-dpmsolver"]
EPS32 = float(np.finfo(np.float32).eps)


# ---- the spec: a self-contained eager torch SDE sampler -----------------------------------------------------------
def _orders(steps, order, lower_order_final):
    out = []
    for step in range(1, steps + 1):
        if step < order:
            out.append(step)
        elif lower_order_final and steps < 10:
            out.append(min(order, steps + 1 - step))
        else:
            out.append(order)
    return out


def eager_sde(ns, x, algo, solver_type, order, steps, lower_order_final, generator, guidance=None,
              return_intermediate=False, denoise_to_zero=False):
    """x_t = ((a*x + c0*D0) + c1*D1) + cn*z with z = torch.randn_like(x, dtype=float32) per step, every op a torch
    fp32 op on x's device; time_uniform grid from T to 1/N; network `exact_net` (with CFG: conditions 1 / 0)."""
    dev = x.device
    N = ns.total_N
    ts = torch.linspace(1.0, 1. / N, steps + 1)
    la = ns.marginal_log_mean_coeff(ts)
    sig = torch.sqrt(1. - torch.exp(2. * la))
    lam = la - 0.5 * torch.log(1. - torch.exp(2. * la))
    alp = torch.exp(la)
    pp = algo == "sde-dpmsolver++"

    def net(xx, i, cond):
        t_in = ((ts[i:i + 1] - 1. / N) * 1000.).to(dev).expand(xx.shape[0])
        out = exact_net(xx, t_in)
        return out if cond is None else out + 0.05 * cond

    def model(xx, i):
        if guidance is None:
            eps = net(xx, i, None)
        else:
            e_u, e_c = net(xx, i, 0.), net(xx, i, 1.)
            eps = e_u + guidance * (e_c - e_u)
        if pp:
            return (xx - sig[i].to(dev) * eps) / alp[i].to(dev)
        return eps

    inter = [x]
    ms = [model(x, 0)]
    for step, o in zip(range(1, steps + 1), _orders(steps, order, lower_order_final)):
        s, t = step - 1, step
        h = lam[t] - lam[s]
        if pp:
            em = torch.expm1(-2. * h)
            a = (sig[t] / sig[s]) * torch.exp(-h)
            c0 = -(alp[t] * em)
            c1 = 0.5 * c0 if solver_type == "dpmsolver" else alp[t] * (em / (2. * h) + 1.)
            cn = sig[t] * torch.sqrt(-em)
        else:
            ep = torch.expm1(h)
            a = torch.exp(la[t] - la[s])
            c0 = -2. * (sig[t] * ep)
            c1 = -(sig[t] * ep) if solver_type == "dpmsolver" else -2. * (sig[t] * (ep / h - 1.))
            cn = sig[t] * torch.sqrt(torch.expm1(2. * h))
        a, c0, c1, cn = (v.to(dev) for v in (a, c0, c1, cn))
        z = torch.randn_like(x, dtype=torch.float32, generator=generator)
        if o == 1:
            x = (a * x + c0 * ms[-1]) + cn * z
        else:
            r0 = (lam[s] - lam[s - 1]) / h
            D1 = (1. / r0).to(dev) * (ms[-1] - ms[-2])
            x = ((a * x + c0 * ms[-1]) + c1 * D1) + cn * z
        inter.append(x)
        if step < steps:
            ms = (ms + [model(x, t)])[-2:]
    if denoise_to_zero:
        eps = net(x, steps, None) if guidance is None else None
        x = (x - sig[steps].to(dev) * eps) / alp[steps].to(dev)
        inter.append(x)
    return (x, inter) if return_intermediate else x


@pytest.fixture()
def sde_oracle():
    """Run the product's host logic on the numpy executor with the SDE step."""
    be = SdeOracleBackend()
    old = ops._backend
    ops.set_backend(be)
    yield be
    ops.set_backend(old)


def product_solver(ns, algo, guidance=None, B=2, device="cpu", **kw):
    if guidance is None:
        fn = model_wrapper(exact_net, ns)
    else:
        net = lambda xx, tt, cc: exact_net(xx, tt) + 0.05 * cc.reshape(-1, 1, 1, 1)
        fn = model_wrapper(net, ns, guidance_type="classifier-free", condition=torch.ones(B, 1, device=device),
                           unconditional_condition=torch.zeros(B, 1, device=device), guidance_scale=guidance)
    return DPM_Solver(fn, ns, algorithm_type=algo, **kw)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", SDE)
@pytest.mark.parametrize("solver_type", ["dpmsolver", "taylor"])
@pytest.mark.parametrize("schedule", ["sd", "iddpm_cosine", "vp_linear"])
def test_plan_scalars_match_float64(algo, solver_type, schedule):
    """Every scalar of the SDE plan against a float64 evaluation of the same formulas on the same fp32 marginals.

    Tolerance: a, c0, cn and the 'dpmsolver' c1 are products/quotients of well-conditioned factors (exp, expm1,
    sqrt of an exact fp32 h), each rounded once in fp32 and h itself rounded once: 16 ulp relative covers the
    handful of roundings with room. The 'taylor' c1 is alpha_t*(expm1(-2h)/(2h) + 1) (sigma_t*(expm1(h)/h - 1)):
    the two terms in the bracket cancel for small h, so its fp32 error is bounded relative to the magnitude of the
    terms, not of the result: 16 * eps * |coefficient| * (|phi/h| + 1)."""
    ns = product_schedule(schedule)
    for steps in (5, 20, 50):
        ts = torch.linspace(1.0, 1. / ns.total_N if schedule != "vp_linear" else 1e-3, steps + 1)
        plan = P.sde_multistep_plan(ns, algo, solver_type, ts, 2, False)
        M = P.Marginals(ns, ts)
        lam, la = M.lam.double(), M.log_alpha.double()
        sig, alp = M.sigma.double(), M.alpha.double()
        for i, co in enumerate(plan):
            s, t = i, i + 1
            h = float(lam[t] - lam[s])
            if algo == "sde-dpmsolver++":
                em = math.expm1(-2 * h)
                ref = dict(a=float(sig[t] / sig[s]) * math.exp(-h), c0=-float(alp[t]) * em,
                           cn=float(sig[t]) * math.sqrt(-em))
                phi, scale = em / (2 * h), float(alp[t])
                c1 = 0.5 * ref["c0"] if solver_type == "dpmsolver" else scale * (phi + 1)
            else:
                ep = math.expm1(h)
                ref = dict(a=math.exp(float(la[t] - la[s])), c0=-2 * float(sig[t]) * ep,
                           cn=float(sig[t]) * math.sqrt(math.expm1(2 * h)))
                phi, scale = ep / h, 2 * float(sig[t])
                c1 = -float(sig[t]) * ep if solver_type == "dpmsolver" else -scale * (phi - 1)
            order = co.order
            for f, v in ref.items():
                assert abs(getattr(co, f) - v) <= 16 * EPS32 * abs(v), (i, f, getattr(co, f), v)
                assert float(np.float32(getattr(co, f))) == getattr(co, f)          # exact fp32 values
            if order == 1:
                assert co.c1 == 0.0 and co.form == FORM_LIN1
                continue
            assert co.form == FORM_DIFF2
            tol = 16 * EPS32 * abs(c1) if solver_type == "dpmsolver" else 16 * EPS32 * scale * (abs(phi) + 1)
            assert abs(co.c1 - c1) <= tol, (i, co.c1, c1)


CPU_CASES = [  # (order, steps, lower_order_final, guidance)
    (1, 5, True, None),
    (2, 6, True, 3.0),
    (2, 12, False, None),
    (2, 7, True, None),
]


@pytest.mark.parametrize("algo", SDE)
@pytest.mark.parametrize("solver_type", ["dpmsolver", "taylor"])
@pytest.mark.parametrize("case", CPU_CASES)
def test_sample_matches_eager_spec_on_the_numpy_executor(sde_oracle, algo, solver_type, case):
    order, steps, lof, guidance = case
    ns = product_schedule("sd")
    B = 2
    x = seeded((B, 4, 8, 8), 31)
    s = product_solver(ns, algo, guidance, B)
    y, inter = s.sample(x, steps=steps, order=order, lower_order_final=lof, solver_type=solver_type,
                        generator=torch.Generator().manual_seed(5), return_intermediate=True)
    y_ref, inter_ref = eager_sde(ns, x, algo, solver_type, order, steps, lof, torch.Generator().manual_seed(5),
                                 guidance, return_intermediate=True)
    assert len(inter) == len(inter_ref)
    for u, v in zip(inter, inter_ref):
        assert torch.equal(u, v), float((u - v).abs().max())
    assert torch.equal(y, y_ref)


def test_denoise_to_zero_and_fresh_noise_per_call(sde_oracle):
    """The final denoise is the deterministic x0 prediction; a second call continues the generator's stream."""
    ns = product_schedule("sd")
    x = seeded((2, 4, 8, 8), 7)
    s = product_solver(ns, "sde-dpmsolver++")
    g, g_ref = torch.Generator().manual_seed(9), torch.Generator().manual_seed(9)
    for _ in range(2):
        y = s.sample(x, steps=6, order=2, denoise_to_zero=True, generator=g)
        y_ref = eager_sde(ns, x, "sde-dpmsolver++", "dpmsolver", 2, 6, True, g_ref, denoise_to_zero=True)
        assert torch.equal(y, y_ref)
    y1 = s.sample(x, steps=6, order=2, generator=torch.Generator().manual_seed(1))
    y2 = s.sample(x, steps=6, order=2, generator=torch.Generator().manual_seed(1))
    y3 = s.sample(x, steps=6, order=2, generator=torch.Generator().manual_seed(2))
    assert torch.equal(y1, y2) and not torch.equal(y1, y3)


@pytest.mark.parametrize("algo", SDE)
def test_one_launch_per_model_evaluation(sde_oracle, algo):
    ns = product_schedule("sd")
    x = seeded((2, 4, 8, 8), 3)
    counts = {}
    for a in (algo, algo.replace("sde-", "")):
        s = product_solver(ns, a)
        before = sde_oracle.launches
        s.sample(x, steps=8, order=2)
        counts[a] = sde_oracle.launches - before
    assert counts[algo] == 8 == counts[algo.replace("sde-", "")]


@pytest.mark.parametrize("algo", SDE)
def test_model_functions_stay_deterministic(sde_oracle, algo):
    ns = product_schedule("sd")
    x = seeded((2, 4, 8, 8), 4)
    t = torch.full((1,), 0.5)
    ode = product_solver(ns, algo.replace("sde-", ""))
    sde = product_solver(ns, algo)
    for name in ("model_fn", "data_prediction_fn", "noise_prediction_fn"):
        assert torch.equal(getattr(sde, name)(x, t), getattr(ode, name)(x, t)), name


@pytest.mark.parametrize("algo", SDE)
def test_rejected_combinations_raise(sde_oracle, algo):
    ns = product_schedule("sd")
    x = seeded((2, 4, 8, 8), 2)
    s = product_solver(ns, algo)
    for kw in (dict(order=3), dict(method="singlestep"), dict(method="singlestep_fixed"), dict(method="adaptive"),
               dict(generator="not a generator")):
        with pytest.raises(ValueError, match="sde-dpmsolver|generator"):
            s.sample(x, steps=6, **kw)
    with pytest.raises(ValueError, match=algo.replace("+", r"\+")):
        s.inverse(x, steps=6)
    with pytest.raises(ValueError, match=algo.replace("+", r"\+")):
        product_solver(ns, algo, reference_rounding=True)
    t, s_, m = torch.full((1,), 0.5), torch.full((1,), 0.6), x.clone()
    calls = [
        lambda: s.dpm_solver_first_update(x, s_, t),
        lambda: s.singlestep_dpm_solver_second_update(x, s_, t),
        lambda: s.singlestep_dpm_solver_third_update(x, s_, t),
        lambda: s.multistep_dpm_solver_second_update(x, [m, m], [s_, s_ + 0.1], t),
        lambda: s.multistep_dpm_solver_third_update(x, [m, m, m], [s_, s_ + 0.1, s_ + 0.2], t),
        lambda: s.singlestep_dpm_solver_update(x, s_, t, 2),
        lambda: s.multistep_dpm_solver_update(x, [m], [s_], t, 1),
        lambda: s.dpm_solver_adaptive(x, 2, 1.0, 1e-3),
    ]
    for c in calls:
        with pytest.raises(ValueError, match=algo.replace("+", r"\+")):
            c()
    assert sde_oracle.launches == 0


def test_pack_plan_round_trips_cn():
    from dpm_solver_b200.distributed import pack_plan, unpack_plan
    ns = product_schedule("sd")
    plan = P.sde_multistep_plan(ns, "sde-dpmsolver++", "taylor", torch.linspace(1.0, 1e-3, 9), 2, True)
    back = unpack_plan(pack_plan(plan))
    assert [c.__dict__ for c in back] == [c.__dict__ for c in plan]
    assert all(c.cn > 0 for c in back)


def test_capi_sde_argument_checks_need_no_gpu():
    from dpm_solver_b200 import _lib
    L = _lib.lib()
    assert L.dpm_sde_step(None, 1.0, None, 0, 0, None) == -1
    d = _lib.StepDesc()
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 0, None) == 0          # n == 0: nothing to do
    d.n, d.form = 16, FORM_MS3
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 0, None) == -2         # only LIN1 / DIFF2
    assert b"LIN1" in L.dpm_last_error()
    d.form = 9
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 0, None) == -1         # not a form at all
    d.form = FORM_LIN1
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 6, None) == -1         # offset % 4
    d.raw_round = 1
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 4, None) == -2         # no reference-rounding mode
    d.raw_round = 0
    buf = (C.c_float * 16)()
    d.dev_coef = C.addressof(buf)
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 4, None) == -2         # scalars by value only
    d.dev_coef = None
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 4, None) == -1         # tensors missing
    d.state_dtype = 7
    assert L.dpm_sde_step(C.byref(d), 1.0, None, 0, 4, None) == -1         # bad dtype


# ---- GPU ------------------------------------------------------------------------------------------------------------
DEV = "cuda:0"


def _step_args(shape, sdt, mdt, ne, form, seed, layout="c", thr=False, want_m=True):
    g = torch.Generator().manual_seed(seed)
    mk = lambda dt: (torch.randn(shape, generator=g)).to(dt).to(DEV)
    a = StepArgs(form=form, n_model=ne, predict_x0=ne > 0, guidance=7.5, alpha_e=0.83, sigma_e=0.55, a=0.91,
                 c0=-0.37, c1=0.29, w0=1.7, want_m_out=want_m, state_dtype=sdt)
    a.x = mk(sdt)
    if ne == 0:
        a.m0 = mk(sdt)
    else:
        a.e_cond = mk(mdt)
        if ne == 2:
            a.e_uncond = mk(mdt)
        a.xe = a.x
    if form == FORM_DIFF2:
        a.m1 = mk(sdt)
    if thr:
        a.per_sample = a.x.numel() // shape[0]
        a.thr = (torch.rand(shape[0], generator=g) * 2 + 0.5).to(DEV)
    if layout == "cl":
        for f in ("x", "m0", "m1", "e_cond", "e_uncond"):
            v = getattr(a, f)
            if v is not None:
                setattr(a, f, v.contiguous(memory_format=torch.channels_last))
        a.xe = a.x if ne > 0 else None
    return a


def _cpu_args(a):
    import copy
    b = copy.copy(a)
    for f in ("x", "xe", "m0", "m1", "m2", "e_cond", "e_uncond", "thr", "out", "out2"):
        v = getattr(a, f)
        if v is not None:
            setattr(b, f, v.cpu())
    b.out = b.out2 = None
    if a.xe is not None and a.xe is a.x:
        b.xe = b.x
    return b


KERNEL_CASES = [  # (shape, ne, form, out2, thr, layout[, 16-bit network output into an fp32 state])
    ((4, 4, 32, 32), 2, FORM_DIFF2, True, True, "c"),
    ((4, 4, 32, 32), 1, FORM_LIN1, False, False, "c"),
    ((4, 4, 32, 32), 0, FORM_DIFF2, False, False, "c"),
    ((4, 4, 32, 32), 0, FORM_LIN1, True, False, "c"),
    ((6, 4, 32, 32), 2, FORM_DIFF2, False, False, "cl"),
    ((3, 5, 7, 11), 1, FORM_DIFF2, True, True, "c"),        # n % 8 != 0
    ((2, 3, 7, 9), 2, FORM_LIN1, False, False, "c"),        # n < 1024
    ((700, 4, 64, 64), 1, FORM_DIFF2, False, True, "c"),     # several grid-stride rows of ATen's randn launch
    ((4, 4, 32, 32), 2, FORM_DIFF2, True, False, "c", True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("sdt", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("case", range(len(KERNEL_CASES)))
def test_in_kernel_noise_is_torch_randn(cuda_backend, sdt, case):
    """dpm_sde_step with the noise in registers == the same launch fed torch.randn_like from the restored generator
    state == the numpy executor on that noise, bit for bit; the generator ends at the same offset."""
    shape, ne, form, out2, thr, layout = KERNEL_CASES[case][:6]
    mdt = torch.bfloat16 if KERNEL_CASES[case][6:] and sdt == torch.float32 else sdt
    cn = 0.4375
    a = _step_args(shape, sdt, mdt, ne, form, seed=case, layout=layout, thr=thr)
    gen = torch.Generator(DEV).manual_seed(100 + case)
    torch.randn(5, device=DEV, generator=gen)                         # a non-zero philox offset

    def run(**kw):
        if out2:
            n = a.x.numel()
            buf = torch.empty(2 * n, dtype=sdt, device=DEV)
            a.out, a.out2 = buf[:n].view(shape), buf[n:].view(shape)
        m, o = cuda_backend.sde_step(a, cn, **kw)
        if out2:
            assert o.data_ptr() == a.out.data_ptr() and torch.equal(a.out2, o)
        return m, o.clone()

    state = gen.get_state()
    m1, o1 = run(generator=gen)
    off = gen.get_offset()
    gen.set_state(state)
    z = torch.randn_like(a.x, dtype=torch.float32, generator=gen)
    assert gen.get_offset() == off
    m2, o2 = run(noise=z)
    torch.cuda.synchronize()
    assert torch.equal(o1, o2), float((o1.float() - o2.float()).abs().max())
    if ne > 0:
        assert torch.equal(m1, m2)
    if layout == "cl":
        assert o1.is_contiguous(memory_format=torch.channels_last)
    rm, ro = SdeOracleBackend().sde_step(_cpu_args(a), cn, noise=z.cpu())
    assert torch.equal(o1.cpu(), ro), float((o1.cpu().float() - ro.float()).abs().max())
    if ne > 0:
        assert torch.equal(m1.cpu(), rm)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", SDE)
@pytest.mark.parametrize("solver_type", ["dpmsolver", "taylor"])
def test_sample_matches_eager_spec_on_cuda(cuda_backend, algo, solver_type):
    """fp32 sample() == the eager spec as torch CUDA ops on the same generator state; a second call draws new noise
    and again matches; the same seed gives the same output; generator=None uses the device's default generator."""
    ns = product_schedule("sd")
    x = seeded((4, 4, 32, 32), 11).to(DEV)
    s = product_solver(ns, algo, 2.5, 4, DEV)
    g, g_ref = torch.Generator(DEV).manual_seed(3), torch.Generator(DEV).manual_seed(3)
    outs = []
    for _ in range(2):
        y = s.sample(x, steps=10, order=2, solver_type=solver_type, generator=g)
        y_ref = eager_sde(ns, x, algo, solver_type, 2, 10, True, g_ref, 2.5)
        assert torch.equal(y, y_ref), float((y - y_ref).abs().max())
        outs.append(y)
    assert not torch.equal(outs[0], outs[1])
    assert torch.equal(s.sample(x, steps=10, order=2, solver_type=solver_type,
                                generator=torch.Generator(DEV).manual_seed(3)), outs[0])
    torch.manual_seed(8)
    y = s.sample(x, steps=10, order=2, solver_type=solver_type)
    torch.manual_seed(8)
    assert torch.equal(y, eager_sde(ns, x, algo, solver_type, 2, 10, True, None, 2.5))
    with pytest.raises(ValueError, match="generator"):
        s.sample(x, steps=10, order=2, generator=torch.Generator().manual_seed(0))


class _MaterialisedNoise(ops.CudaBackend):
    """The same solver run with the noise drawn by torch.randn_like and read from memory."""

    def sde_step(self, a, noise_scale, generator=None, noise=None):
        ref = a.reference_tensor()
        z = torch.randn_like(ref, dtype=torch.float32, generator=generator)
        return super().sde_step(a, noise_scale, noise=z)


@pytest.mark.gpu
@pytest.mark.parametrize("sdt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("algo", SDE)
def test_16bit_channels_last_cfg_run_reads_the_same_noise(algo, sdt):
    """state_dtype 16-bit, channels_last network, CFG (out2 into the doubled batch), thresholding for ++: the
    in-kernel noise run equals the run that reads materialised torch.randn_like noise."""
    ns = product_schedule("sd")
    B = 3
    x = seeded((B, 4, 24, 24), 5).to(DEV).contiguous(memory_format=torch.channels_last)
    net = lambda xx, tt, cc: (exact_net(xx, tt) + 0.05 * cc.reshape(-1, 1, 1, 1)).contiguous(
        memory_format=torch.channels_last)
    ys = []
    old = ops._backend
    try:
        for be in (ops.CudaBackend(), _MaterialisedNoise()):
            ops.set_backend(be)
            fn = model_wrapper(net, ns, guidance_type="classifier-free", condition=torch.ones(B, 1, device=DEV),
                               unconditional_condition=torch.zeros(B, 1, device=DEV), guidance_scale=4.0)
            kw = dict(correcting_x0_fn="dynamic_thresholding") if algo == "sde-dpmsolver++" else {}
            s = DPM_Solver(fn, ns, algorithm_type=algo, state_dtype=sdt, **kw)
            ys.append(s.sample(x, steps=8, order=2, generator=torch.Generator(DEV).manual_seed(4)))
    finally:
        ops.set_backend(old)
    assert ys[0].dtype == sdt and ys[0].is_contiguous(memory_format=torch.channels_last)
    assert torch.isfinite(ys[0].float()).all()
    assert torch.equal(ys[0], ys[1])


@pytest.mark.gpu
def test_point_mass_marginals_are_exact(cuda_backend):
    """Data distribution = a point mass x0*, network = the true x0* (x_start parameterisation): SDE-DPM-Solver++
    keeps x_t ~ N(alpha_t x0*, sigma_t^2) exactly. Over >= 10^7 elements the residual r_t = (x_t - alpha_t x0*)/sigma_t
    of every intermediate state has mean 0 and std 1 within 6 standard errors, and the noise each step injects,
    (r_t - exp(-h) r_s)/sqrt(1 - exp(-2h)), is standard normal and uncorrelated with the previous step's."""
    ns = product_schedule("sd")
    shape = (40, 4, 256, 256)
    n = math.prod(shape)
    assert n >= 10 ** 7
    x0 = (torch.rand(shape, device=DEV, generator=torch.Generator(DEV).manual_seed(1)) * 2 - 1)
    steps = 10
    ts = torch.linspace(1.0, 1. / ns.total_N, steps + 1)
    M = P.Marginals(ns, ts)
    al, sg, lam = M.alpha.double().tolist(), M.sigma.double().tolist(), M.lam.double().tolist()
    g = torch.Generator(DEV).manual_seed(2)
    xT = al[0] * x0 + sg[0] * torch.randn(shape, device=DEV, generator=g)
    s = DPM_Solver(model_wrapper(lambda xx, tt: x0, ns, model_type="x_start"), ns, algorithm_type="sde-dpmsolver++")
    _, inter = s.sample(xT, steps=steps, order=2, generator=g, return_intermediate=True)
    six = lambda se: 6 * se
    prev_z = None
    for i, xt in enumerate(inter):
        r = ((xt.double() - al[i] * x0.double()) / sg[i]).reshape(-1)
        assert abs(float(r.mean())) < six(1 / math.sqrt(n)), (i, float(r.mean()))
        assert abs(float(r.std()) - 1) < six(1 / math.sqrt(2 * n)), (i, float(r.std()))
        if i > 0:
            e = math.exp(-(lam[i] - lam[i - 1]))
            z = (r - e * r_prev) / math.sqrt(1 - e * e)
            assert abs(float(z.mean())) < six(1 / math.sqrt(n)) and abs(float(z.std()) - 1) < six(1 / math.sqrt(2 * n))
            assert abs(float((z * r_prev).mean())) < six(1 / math.sqrt(n)), i       # fresh, independent of the state
            if prev_z is not None:
                assert abs(float((z * prev_z).mean())) < six(1 / math.sqrt(n)), i   # not reused / correlated
            prev_z = z
        r_prev = r


@pytest.mark.gpu
@pytest.mark.parametrize("algo", SDE)
def test_captured_sde_run_draws_fresh_noise_per_replay(cuda_backend, algo):
    ns = product_schedule("sd")
    x = seeded((2, 4, 32, 32), 9).to(DEV)
    s = product_solver(ns, algo, 2.0, 2, DEV)
    g = s.capture(x, steps=6, order=2)
    y1 = g(x).clone()
    y2 = g(x).clone()
    torch.cuda.synchronize()
    assert torch.isfinite(y1).all() and torch.isfinite(y2).all()
    assert not torch.equal(y1, y2)
    with pytest.raises(ValueError, match="default CUDA generator"):
        s.capture(x, steps=6, order=2, generator=torch.Generator(DEV).manual_seed(0))
