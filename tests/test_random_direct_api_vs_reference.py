"""Randomised parity of the DIRECTLY callable solver methods against the UNMODIFIED reference (its results stored
in tests/golden/reference/): every public update method, the order dispatchers, the model functions, add_noise and
inverse, with random times, r1/r2, solver_type, parameterisation and thresholding. Bit-identical."""
import random

import pytest
import torch

import refstore as S
from cases import exact_net, make_betas, seeded
from test_random_configs_vs_reference import reference_module

REF = S.Store(__file__)


def mk(mod, c):
    kind, betas = make_betas(c["schedule"])
    ns = mod.NoiseScheduleVP("linear") if kind == "linear" else mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
    fn = mod.model_wrapper(exact_net, ns, model_type=c["model_type"])
    return ns, mod.DPM_Solver(fn, ns, algorithm_type=c["algo"], correcting_x0_fn="dynamic_thresholding" if c["thr"] else None)

def flat(o):
    if isinstance(o, tuple):
        x, d = o
        return [x] + [d[k] for k in sorted(d)]
    return [o]

def one(mod, c):
    ns, s = mk(mod, c)
    x = seeded((2, 3, 8, 8), c["seed"])
    ts = sorted(c["ts"], reverse=True)
    t = lambda v: torch.tensor(v)
    k = c["kind"]
    if k == "first":
        return flat(s.dpm_solver_first_update(x, t(ts[0]), t(ts[1]), return_intermediate=c["ri"]))
    if k == "ss2":
        return flat(s.singlestep_dpm_solver_second_update(x, t(ts[0]), t(ts[1]), r1=c["r1"], return_intermediate=c["ri"], solver_type=c["st"]))
    if k == "ss3":
        return flat(s.singlestep_dpm_solver_third_update(x, t(ts[0]), t(ts[1]), r1=c["r1"], r2=c["r2"], return_intermediate=c["ri"], solver_type=c["st"]))
    if k == "ssu":
        return flat(s.singlestep_dpm_solver_update(x, t(ts[0]), t(ts[1]), c["order"], return_intermediate=c["ri"], solver_type=c["st"]))
    ms = [seeded((2, 3, 8, 8), c["seed"] + 1 + i) for i in range(3)]
    tp = [t(ts[0]), t(ts[1]), t(ts[2])]
    if k == "ms2":
        return flat(s.multistep_dpm_solver_second_update(x, ms[1:], tp[1:], t(ts[3]), solver_type=c["st"]))
    if k == "ms3":
        return flat(s.multistep_dpm_solver_third_update(x, ms, tp, t(ts[3]), solver_type=c["st"]))
    if k == "msu":
        o = c["order"]
        return flat(s.multistep_dpm_solver_update(x, ms[3 - o:] if o > 1 else ms[2:], tp[3 - o:] if o > 1 else tp[2:], t(ts[3]), o, solver_type=c["st"]))
    if k == "x0":
        return [s.data_prediction_fn(x, t(ts[0])), s.noise_prediction_fn(x, t(ts[0])), s.model_fn(x, t(ts[0]))]
    if k == "d2z":
        return [s.denoise_to_zero_fn(x, t(ts[1]))]
    if k == "noise":
        return [s.add_noise(x, torch.tensor(ts[:c["order"]]), noise=seeded((c["order"], 2, 3, 8, 8), 9))]
    if k == "inv":
        return [s.inverse(x, steps=c["order"] * 3, order=c["order"], t_start=ts[3], t_end=ts[0], method=c["meth"])]



@pytest.mark.parametrize("chunk", range(4))
def test_direct_api_bit_exact(oracle_backend, chunk):
    import dpm_solver_b200 as new
    for seed in range(75 * chunk, 75 * (chunk + 1)):
        rng = random.Random(31000 + seed)
        c = dict(schedule=rng.choice(["sd", "ddpm_linear", "iddpm_cosine", "vp_linear"]), algo=rng.choice(["dpmsolver++", "dpmsolver"]),
                 model_type=rng.choice(["noise", "v", "x_start", "score"]), thr=False, seed=rng.randint(0, 10**6),
                 ts=[rng.uniform(0.002, 1.0) for _ in range(4)],
                 kind=rng.choice(["first", "ss2", "ss3", "ssu", "ms2", "ms3", "msu", "x0", "d2z", "noise", "inv"]),
                 r1=rng.choice([None, 0.5, 1 / 3, 0.25, 0.7]), r2=rng.choice([None, 2 / 3, 0.8, 0.5]), ri=rng.random() < 0.5,
                 st=rng.choice(["dpmsolver", "taylor"]), order=rng.choice([1, 2, 3]), meth=rng.choice(["multistep", "singlestep"]))
        c["thr"] = c["algo"] == "dpmsolver++" and rng.random() < 0.3
        if c["r1"] is not None and c["r2"] is not None and c["r2"] <= c["r1"]:
            c["r2"] = min(0.95, c["r1"] + 0.2)
        try:
            a = REF(f"direct/{seed}", lambda: one(reference_module(), c))
        except Exception as e:   # what the reference rejects must be rejected the same way
            with pytest.raises(type(e)):
                one(new, c)
            continue
        if not all(S.all_finite(v) for v in a):
            continue
        b = one(new, c)
        assert len(a) == len(b), c
        for u, v in zip(a, b):
            S.assert_same(v, u, c)


@pytest.mark.parametrize("chunk", range(2))
def test_model_fn_with_per_sample_times(oracle_backend, chunk):
    """`model_fn(x, t_continuous)` called directly with a VECTOR of different times (the reference's wrapper
    accepts it for every parameterisation and guidance type, :282-330): bit-identical."""
    import dpm_solver_b200 as new
    for seed in range(40 * chunk, 40 * (chunk + 1)):
        rng = random.Random(seed)
        sched = rng.choice(["sd", "ddpm_linear", "iddpm_cosine", "vp_linear"])
        mt = rng.choice(["noise", "v", "x_start", "score"])
        g = rng.choice(["uncond", "classifier-free", "classifier"])
        scale = rng.choice([1.0, 3.5, 7.5, 2.3])
        B = rng.choice([1, 2, 4])
        tt = (torch.full((B,), rng.uniform(0.01, 1.0)) if rng.random() < 0.3
              else torch.tensor([rng.uniform(0.01, 1.0) for _ in range(B)]))
        x = seeded((B, 3, 8, 8), seed)
        def arm(mod):
            kind, betas = make_betas(sched)
            ns = mod.NoiseScheduleVP("linear") if kind == "linear" else mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
            if g == "uncond":
                fn = mod.model_wrapper(lambda xx, t: exact_net(xx, t), ns, model_type=mt)
            elif g == "classifier-free":
                fn = mod.model_wrapper(lambda xx, t, c: exact_net(xx, t) + 0.05 * c.reshape(-1, 1, 1, 1), ns, model_type=mt,
                                       guidance_type="classifier-free", condition=torch.ones(B, 1),
                                       unconditional_condition=torch.zeros(B, 1), guidance_scale=scale)
            else:
                def cls(xx, t_in, cond, **kw):
                    return -((xx - 0.1 * cond.reshape(-1, 1, 1, 1)) ** 2).flatten(1).sum(1) * 0.01 + 0 * t_in
                fn = mod.model_wrapper(lambda xx, t: exact_net(xx, t), ns, model_type=mt, guidance_type="classifier",
                                       condition=torch.ones(B), guidance_scale=scale, classifier_fn=cls)
            return fn(x, tt)
        a = REF(f"model_fn/{seed}", lambda: arm(reference_module()))
        S.assert_same(arm(new), a, (sched, mt, g, scale))
