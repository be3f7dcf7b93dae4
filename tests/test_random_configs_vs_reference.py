"""Randomised end-to-end parity against the UNMODIFIED reference (its results stored in tests/golden/reference/).

Draws sampling configurations at random (schedule, algorithm, method, order, steps, skip type,
solver type, parameterisation, CFG, thresholding, t_end, denoise_to_zero), runs the reference on CPU
and the product's host logic on the numpy executor, and requires bit-identical outputs and an
identical trace of network calls. Complements the fixed golden cases of tests/golden/."""
import random
import warnings

import pytest
import torch

import refstore as S
from cases import exact_net, make_betas, seeded

REF = S.Store(__file__)


def reference_module():
    """The unmodified reference dpm_solver_pytorch.py (only run while recording tests/golden/reference/)."""
    warnings.filterwarnings("ignore")
    return S.original("dpm_solver_pytorch")


def draw(rng):
    method = rng.choice(["multistep", "multistep", "singlestep", "singlestep_fixed"])
    order = rng.choice([1, 2, 3])
    steps = rng.randint(max(order, 3), 24)
    c = dict(schedule=rng.choice(["sd", "ddpm_linear", "iddpm_cosine", "vp_linear"]),
             algo=rng.choice(["dpmsolver++", "dpmsolver"]), method=method, order=order, steps=steps,
             skip_type=rng.choice(["time_uniform", "logSNR", "time_quadratic"]),
             solver_type=rng.choice(["dpmsolver", "taylor"]), model_type=rng.choice(["noise", "noise", "v", "x_start", "score"]),
             cfg=rng.choice([None, None, 1.0, 3.5, 7.5]), lower_order_final=rng.choice([True, False]),
             denoise_to_zero=rng.random() < 0.2, t_end=rng.choice([None, 1e-3, 0.02]), seed=rng.randint(0, 10 ** 6))
    c["thresholding"] = c["algo"] == "dpmsolver++" and rng.random() < 0.25
    if c["schedule"] == "vp_linear" and c["t_end"] is None:
        c["t_end"] = 1e-3
    return c


def run(mod_ns, mod_wrap, mod_solver, c):
    kind, betas = make_betas(c["schedule"])
    ns = mod_ns("linear") if kind == "linear" else mod_ns("discrete", betas=torch.from_numpy(betas))
    B = 2
    x = seeded((B, 3, 8, 8), c["seed"])
    calls = []
    if c["cfg"] is not None:
        def net(xx, tt, cc):
            calls.append((float(tt[0]), tuple(xx.shape)))
            return exact_net(xx, tt) + 0.05 * cc.reshape(-1, 1, 1, 1)
        fn = mod_wrap(net, ns, model_type=c["model_type"], guidance_type="classifier-free", condition=torch.ones(B, 1),
                      unconditional_condition=torch.zeros(B, 1), guidance_scale=c["cfg"])
    else:
        def net(xx, tt):
            calls.append((float(tt[0]), tuple(xx.shape)))
            return exact_net(xx, tt)
        fn = mod_wrap(net, ns, model_type=c["model_type"])
    s = mod_solver(fn, ns, algorithm_type=c["algo"], correcting_x0_fn="dynamic_thresholding" if c["thresholding"] else None)
    y, inter = s.sample(x, steps=c["steps"], order=c["order"], skip_type=c["skip_type"], method=c["method"],
                        lower_order_final=c["lower_order_final"], denoise_to_zero=c["denoise_to_zero"],
                        solver_type=c["solver_type"], t_end=c["t_end"], return_intermediate=True)
    return y, inter, calls


@pytest.mark.parametrize("chunk", range(6))
def test_random_configurations_bit_exact(oracle_backend, chunk):
    import dpm_solver_b200 as new
    rng = random.Random(1000 + chunk)
    done = 0
    i = 0
    while done < 12:
        c = draw(rng)
        i += 1
        try:
            yr, ir, cr = REF(f"bit_exact/{chunk}/{i}", lambda: run_reference(c))
        except Exception as e:   # configurations the reference itself rejects must be rejected the same way
            with pytest.raises(type(e)):
                run(new.NoiseScheduleVP, new.model_wrapper, new.DPM_Solver, c)
            continue
        if not S.all_finite(yr):
            continue
        yn, in_, cn = run(new.NoiseScheduleVP, new.model_wrapper, new.DPM_Solver, c)
        S.assert_same(cn, cr, c)
        S.assert_same(yn, yr, c)
        S.assert_same(in_, ir, c)
        done += 1


def run_reference(c):
    ref = reference_module()
    return run(ref.NoiseScheduleVP, ref.model_wrapper, ref.DPM_Solver, c)


def draw_wide(rng):
    """draw() plus t_start, batch/shape/scale, thresholding ratio / floor and (15 %) the adaptive method."""
    c = draw(rng)
    c.update(t_start=rng.choice([None, None, 0.8, 0.5]), ratio=rng.choice([0.995, 0.995, 0.9, 0.5, 1.0, 0.0]),
             max_val=rng.choice([1.0, 1.0, 0.5, 3.0]), B=rng.choice([1, 2, 3, 5]),
             shape=rng.choice([(3, 8, 8), (4, 4, 4), (1, 7, 5), (2, 16, 16)]), scale=rng.choice([1.0, 0.2, 5.0]))
    if rng.random() < 0.15:
        c.update(method="adaptive", order=rng.choice([2, 3]), atol=rng.choice([0.0078, 0.05]), rtol=rng.choice([0.05, 0.2]))
    if rng.random() < 0.1:
        c["steps"] = rng.randint(25, 60)
    return c


def run_wide(mod, c):
    import contextlib
    import io
    kind, betas = make_betas(c["schedule"])
    ns = mod.NoiseScheduleVP("linear") if kind == "linear" else mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
    B = c["B"]
    x = seeded((B,) + c["shape"], c["seed"]) * c["scale"]
    calls = []
    if c["cfg"] is not None:
        def net(xx, tt, cc):
            calls.append((float(tt[0]), tuple(xx.shape)))
            return exact_net(xx, tt) + 0.05 * cc.reshape(-1, 1, 1, 1)
        fn = mod.model_wrapper(net, ns, model_type=c["model_type"], guidance_type="classifier-free", condition=torch.ones(B, 1),
                               unconditional_condition=torch.zeros(B, 1), guidance_scale=c["cfg"])
    else:
        def net(xx, tt):
            calls.append((float(tt[0]), tuple(xx.shape)))
            return exact_net(xx, tt)
        fn = mod.model_wrapper(net, ns, model_type=c["model_type"])
    s = mod.DPM_Solver(fn, ns, algorithm_type=c["algo"], correcting_x0_fn="dynamic_thresholding" if c["thresholding"] else None,
                       thresholding_max_val=c["max_val"], dynamic_thresholding_ratio=c["ratio"])
    kw = dict(steps=c["steps"], order=c["order"], skip_type=c["skip_type"], method=c["method"],
              lower_order_final=c["lower_order_final"], denoise_to_zero=c["denoise_to_zero"], solver_type=c["solver_type"],
              t_end=c["t_end"], t_start=c["t_start"])
    if c["method"] == "adaptive":
        with contextlib.redirect_stdout(io.StringIO()):
            return s.sample(x, atol=c["atol"], rtol=c["rtol"], **kw), [], calls
    y, inter = s.sample(x, return_intermediate=True, **kw)
    return y, inter, calls


@pytest.mark.parametrize("chunk", range(6))
def test_random_wide_configurations(oracle_backend, chunk):
    """Wider space: t_start, batch sizes / odd shapes / input scale, thresholding ratio and floor, long runs,
    adaptive. Fixed-grid methods must be bit-identical; the adaptive solver must evaluate the network the
    same number of times and agree within the reduction-order tolerance of its error estimate
    (tests/test_adaptive.py; 596 random adaptive runs: 500 bit-identical, worst 1.9e-4 relative)."""
    import dpm_solver_b200 as new

    def reference(c):
        y, inter, calls = run_wide(reference_module(), c)
        if c["method"] == "adaptive":       # compared within a tolerance, by the number of network calls
            return S.sample(y), inter, len(calls)
        return y, inter, calls

    rng = random.Random(5000 + chunk)
    for i in range(20):
        c = draw_wide(rng)
        try:
            yr, ir, cr = REF(f"wide/{chunk}/{i}", lambda: reference(c))
        except Exception as e:
            with pytest.raises(type(e)):
                run_wide(new, c)
            continue
        if not S.all_finite(yr):
            continue
        yn, in_, cn = run_wide(new, c)
        if c["method"] == "adaptive":
            assert len(cn) == cr, c
            assert yr.rel_err(yn) <= 1e-3, c
            continue
        S.assert_same(cn, cr, c)
        S.assert_same(yn, yr, c)
        S.assert_same(in_, ir, c)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_16bit_inputs_follow_the_reference_promotion(oracle_backend, dt):
    """x handed over in bf16/fp16 (state_dtype=None), discrete schedules, no CFG: the network sees the
    caller's 16-bit tensor at the first evaluation and fp32 states afterwards, the arithmetic is fp32 on
    the widened values -- dtype trace and samples bit-identical to the reference. (16-bit CFG outputs and
    the 0-dim coefficients of the 'linear' schedule are documented deviations, DESIGN.md section 2.)"""
    import dpm_solver_b200 as new

    def arm(mod, c):
        _, betas = make_betas(c["schedule"])
        ns = mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
        calls = []

        def net(xx, tt, *cond):
            calls.append((float(tt[0]), tuple(xx.shape), xx.dtype))
            return exact_net(xx.float(), tt).to(xx.dtype)
        if c["cfg"] is not None:
            fn = mod.model_wrapper(net, ns, model_type=c["model_type"], guidance_type="classifier-free",
                                   condition=torch.ones(c["B"], 1), unconditional_condition=torch.zeros(c["B"], 1),
                                   guidance_scale=c["cfg"])
        else:
            fn = mod.model_wrapper(net, ns, model_type=c["model_type"])
        s = mod.DPM_Solver(fn, ns, algorithm_type=c["algo"], correcting_x0_fn="dynamic_thresholding" if c["thresholding"] else None)
        x = (seeded((c["B"],) + c["shape"], c["seed"]) * c["scale"]).to(dt)
        y = s.sample(x, steps=c["steps"], order=c["order"], skip_type=c["skip_type"], method=c["method"],
                     lower_order_final=c["lower_order_final"], denoise_to_zero=c["denoise_to_zero"],
                     solver_type=c["solver_type"], t_end=c["t_end"], t_start=c["t_start"])
        return y, calls

    rng = random.Random(77)
    done = i = 0
    while done < 25:
        c = draw_wide(rng)
        if c["method"] == "adaptive" or c["schedule"] == "vp_linear" or c["cfg"] not in (None, 1.0):
            continue
        i += 1
        yr, cr = REF(f"16bit_inputs/{dt}/{i}", lambda: arm(reference_module(), c))
        if not S.all_finite(yr):
            continue
        yn, cn = arm(new, c)
        S.assert_same(cn, cr, c)
        S.assert_same(yn, yr, c)
        done += 1


@pytest.mark.parametrize("x_16bit", [False, True], ids=["x_fp32", "x_16bit"])
def test_reference_rounding_mode_is_bit_identical(oracle_backend, x_16bit):
    """`DPM_Solver(..., reference_rounding=True)`: a network that returns bf16/fp16 makes the reference
    evaluate the CFG combine (:329-330) and, in the eps-solver, the differences of the buffered raw
    outputs -- for singlestep-3 'taylor' the whole D1/D2 chain (:780-783) -- in that 16-bit type. With
    the option on, samples are bit-identical to the reference for every parameterisation, with and
    without CFG (scales that are not representable in bf16 included), fp32 or 16-bit x_T."""
    import dpm_solver_b200 as new

    def arm(mod, c, dt):
        _, betas = make_betas(c["schedule"])
        ns = mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))

        def net(xx, tt, *cond):
            o = exact_net(xx.float(), tt)
            if cond:
                o = o + 0.05 * cond[0].reshape(-1, 1, 1, 1)
            return o.to(dt)
        if c["cfg"] is not None:
            fn = mod.model_wrapper(net, ns, model_type=c["model_type"], guidance_type="classifier-free",
                                   condition=torch.ones(c["B"], 1), unconditional_condition=torch.zeros(c["B"], 1),
                                   guidance_scale=c["cfg"])
        else:
            fn = mod.model_wrapper(net, ns, model_type=c["model_type"])
        kw = dict(reference_rounding=True) if mod is new else {}
        s = mod.DPM_Solver(fn, ns, algorithm_type=c["algo"],
                           correcting_x0_fn="dynamic_thresholding" if c["thresholding"] else None, **kw)
        x = seeded((c["B"],) + c["shape"], c["seed"]) * c["scale"]
        y = s.sample(x.to(dt) if x_16bit else x, steps=c["steps"], order=c["order"], skip_type=c["skip_type"],
                     method=c["method"], lower_order_final=c["lower_order_final"], denoise_to_zero=c["denoise_to_zero"],
                     solver_type=c["solver_type"], t_end=c["t_end"], t_start=c["t_start"])
        return y

    rng = random.Random(4242 + int(x_16bit))
    done = i = 0
    while done < 30:
        c = draw_wide(rng)
        if c["method"] == "adaptive" or c["schedule"] == "vp_linear":
            continue
        dt = rng.choice([torch.bfloat16, torch.float16])
        if c["cfg"] not in (None, 1.0) and rng.random() < 0.5:
            c["cfg"] = rng.choice([3.7, 2.3, 9.1])
        i += 1
        yr = REF(f"reference_rounding/{x_16bit}/{i}", lambda: arm(reference_module(), c, dt))
        if not S.all_finite(yr):
            continue
        yn = arm(new, c, dt)
        S.assert_same(yn, yr, (c, dt))
        done += 1


@pytest.mark.parametrize("model_type", ["noise", "v", "x_start", "score"])
def test_classifier_guidance_matches_reference(oracle_backend, model_type):
    """guidance_type='classifier' (:315-321): eps - s*sigma_t*grad_x log p(c|x); the guided-diffusion
    example drives the solver this way (runners/diffusion.py:611-628)."""
    import dpm_solver_b200 as new
    kind, betas = make_betas("ddpm_linear")
    W = torch.randn(5, 3 * 8 * 8, generator=torch.Generator().manual_seed(0)) * 0.05

    def classifier_fn(x, t_in, cond, **kw):
        logits = x.reshape(x.shape[0], -1) @ W.t() + 0.001 * t_in.reshape(-1, 1)
        lp = torch.log_softmax(logits, dim=-1)
        return lp[range(x.shape[0]), cond]

    cond = torch.tensor([1, 3])
    x = seeded((2, 3, 8, 8), 11)
    def arm(mod):
        ns = mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
        fn = mod.model_wrapper(exact_net, ns, model_type=model_type, guidance_type="classifier", condition=cond,
                               guidance_scale=2.5, classifier_fn=classifier_fn)
        eps = fn(x, torch.full((2,), 0.6))
        s = mod.DPM_Solver(fn, ns, algorithm_type="dpmsolver++", correcting_x0_fn="dynamic_thresholding")
        y = s.sample(x, steps=8, order=2)
        return eps, y

    want = REF(f"classifier_guidance/{model_type}", lambda: arm(reference_module()))
    for a, b in zip(arm(new), want):
        S.assert_same(a, b)


@pytest.mark.parametrize("method,order,steps", [("multistep", 2, 12), ("multistep", 3, 9), ("singlestep", 3, 10), ("singlestep_fixed", 2, 8)])
@pytest.mark.parametrize("cfg", [None, 4.0])
def test_hooks_match_reference(oracle_backend, method, order, steps, cfg):
    """correcting_xt_fn (DiffEdit-style inpainting mask, :1180-1239) and a user correcting_x0_fn
    (:440-441) see the same arguments in the same order and produce bit-identical samples."""
    import dpm_solver_b200 as new
    kind, betas = make_betas("sd")
    B = 2
    x = seeded((B, 3, 8, 8), 31)
    mask = (seeded((B, 3, 8, 8), 32) > 0).float()
    known = seeded((B, 3, 8, 8), 33)
    def arm(mod):
        ns = mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
        log = []

        def fix_xt(xt, t, step, _ns=ns, _log=log):
            _log.append((round(float(t), 6), int(step)))
            a, s = _ns.marginal_alpha(t.reshape(-1)[:1]), _ns.marginal_std(t.reshape(-1)[:1])
            return xt * mask + (1 - mask) * (a * known + s * 0.5)

        fix_x0 = lambda x0, t: torch.tanh(x0)
        if cfg is not None:
            net = lambda xx, tt, cc: exact_net(xx, tt) + 0.05 * cc.reshape(-1, 1, 1, 1)
            fn = mod.model_wrapper(net, ns, guidance_type="classifier-free", condition=torch.ones(B, 1),
                                   unconditional_condition=torch.zeros(B, 1), guidance_scale=cfg)
        else:
            fn = mod.model_wrapper(exact_net, ns)
        s = mod.DPM_Solver(fn, ns, algorithm_type="dpmsolver++", correcting_x0_fn=fix_x0, correcting_xt_fn=fix_xt)
        y, inter = s.sample(x, steps=steps, order=order, method=method, return_intermediate=True, denoise_to_zero=True)
        return y, inter, log

    yr, ir, lr = REF(f"hooks/{method}/{order}/{steps}/{cfg}", lambda: arm(reference_module()))
    yn, in_, ln = arm(new)
    S.assert_same(ln, lr)
    S.assert_same(yn, yr)
    S.assert_same(in_, ir)


@pytest.mark.parametrize("steps,order", [(2, 3), (1, 2), (1, 3)])
def test_singlestep_fixed_with_fewer_steps_than_order(oracle_backend, steps, order):
    """K = steps // order = 0: the reference runs no outer step and returns x (plus the optional denoise tail)."""
    import dpm_solver_b200 as new
    for d2z in (False, True):
        c = dict(schedule="sd", algo="dpmsolver++", method="singlestep_fixed", order=order, steps=steps, skip_type="time_uniform",
                 solver_type="dpmsolver", model_type="noise", cfg=None, lower_order_final=True, denoise_to_zero=d2z, t_end=None,
                 seed=5, thresholding=False)
        yr, ir, cr = REF(f"fewer_steps/{steps}/{order}/{d2z}", lambda: run_reference(c))
        yn, in_, cn = run(new.NoiseScheduleVP, new.model_wrapper, new.DPM_Solver, c)
        S.assert_same(cn, cr)
        S.assert_same(in_, ir)
        S.assert_same(yn, yr)
