"""Paths beside the sampling loop, against the UNMODIFIED reference (its results stored in tests/golden/reference/):
classifier guidance (:315-321),
`add_noise` (:1012-1030), the 'cosine' schedule of the older vendored copies (SD dpm_solver.py:114-175), NaN
propagation of dynamic thresholding (:416-425), and the ADVICE.md round-1 corner cases. Each test runs on the numpy
executor (CPU) and on CudaBackend (`-m gpu`); the reference arm always runs on CPU."""
import numpy as np
import pytest
import torch

import refstore as S
from cases import exact_net, make_betas, seeded
from helpers import rel_err

REF = S.Store(__file__)
EXECUTORS = ["numpy-executor", pytest.param("cuda", marks=pytest.mark.gpu)]


@pytest.fixture(params=EXECUTORS)
def dev(request):
    from dpm_solver_b200 import ops
    old = ops._backend
    if request.param == "cuda":
        ops.set_backend(ops.CudaBackend())
        yield "cuda:0"
    else:
        from oracle_backend import OracleBackend
        ops.set_backend(OracleBackend())
        yield "cpu"
    ops.set_backend(old)


def _sched(mod, name="sd"):
    kind, betas = make_betas(name)
    return mod.NoiseScheduleVP("linear") if kind == "linear" else mod.NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))


# ---- classifier guidance -----------------------------------------------------------------------------
def _classifier_fn(x, t_input, y, **kw):
    """log p(y|x) whose gradient is exact on every device: quadratic in x with power-of-two weights."""
    w = (y.to(x.dtype) * 0.125 + 0.25).reshape(-1, 1, 1, 1)
    return (w * x * x * 0.5 + 0.0625 * x).sum(dim=(1, 2, 3)) + t_input * 0.001


@pytest.mark.parametrize("model_type", ["noise", "x_start", "v", "score"])
@pytest.mark.parametrize("algo,order,method", [("dpmsolver++", 2, "multistep"), ("dpmsolver", 3, "singlestep")])
def test_classifier_guidance_sample(dev, model_type, algo, order, method):
    """model_fn's classifier branch inside sample(): noise - scale * sigma_t * grad (:315-321), bit-identical."""
    import dpm_solver_b200 as new
    B = 3
    x = seeded((B, 3, 8, 8), 77)

    def arm(mod, d):
        ns = _sched(mod, "ddpm_linear")
        y = torch.tensor([1, 4, 7], device=d)
        fn = mod.model_wrapper(exact_net, ns, model_type=model_type, guidance_type="classifier", condition=y,
                               guidance_scale=2.5, classifier_fn=_classifier_fn)
        s = mod.DPM_Solver(fn, ns, algorithm_type=algo)
        return s.sample(x.to(d), steps=9, order=order, method=method).cpu()
    want = REF(f"classifier_sample/{model_type}/{algo}/{order}/{method}", lambda: arm(S.original(), "cpu"))
    assert S.all_finite(want)
    S.assert_same(arm(new, dev), want)


def test_classifier_guidance_direct_call_per_sample_times(dev):
    """model_fn(x, t) called directly with a different time label per sample."""
    import dpm_solver_b200 as new
    x = seeded((4, 3, 8, 8), 5)
    t = torch.tensor([0.9, 0.5, 0.25, 0.05])

    def arm(mod, d):
        ns = _sched(mod, "sd")
        fn = mod.model_wrapper(exact_net, ns, model_type="v", guidance_type="classifier",
                               condition=torch.tensor([0, 1, 2, 3], device=d), guidance_scale=1.5, classifier_fn=_classifier_fn)
        return fn(x.to(d), t.to(d)).cpu()
    S.assert_same(arm(new, dev), REF("classifier_direct_call", lambda: arm(S.original(), "cpu")))


# ---- add_noise -----------------------------------------------------------------------------------------
def test_add_noise_golden_and_reference(dev, golden):
    import dpm_solver_b200 as new
    g = golden["glue"]
    x, noise = torch.from_numpy(g["x"]), torch.from_numpy(g["add_noise_in"])
    ns = _sched(new, "sd")
    got = new.DPM_Solver(None, ns).add_noise(x.to(dev), torch.tensor([0.3, 0.8], device=dev), noise=noise.to(dev))
    np.testing.assert_array_equal(got.cpu().numpy(), g["add_noise"])
    # single time label -> [B, ...] (squeeze rule :1027-1030); 16-bit input promotes like the reference
    for dt in (torch.float32, torch.bfloat16):
        xr = seeded((2, 4, 8, 8), 3).to(dt)
        nz = seeded((1, 2, 4, 8, 8), 4).to(dt)
        want = REF(f"add_noise/{dt}", lambda: (lambda ref: ref.DPM_Solver(None, _sched(ref, "sd")).add_noise(
            xr, torch.tensor([0.45]), noise=nz))(S.original()))
        have = new.DPM_Solver(None, ns).add_noise(xr.to(dev), torch.tensor([0.45], device=dev), noise=nz.to(dev))
        S.assert_same(have.cpu(), want)


# ---- 'cosine' schedule of the older vendored copies -----------------------------------------------------
def test_cosine_schedule_scalars_match_vendored_copy():
    """NoiseScheduleVP('cosine') (examples/stable-diffusion/.../dpm_solver.py:114-175): every marginal and the inverse."""
    from dpm_solver_b200 import NoiseScheduleVP
    names = ("marginal_log_mean_coeff", "marginal_alpha", "marginal_std", "marginal_lambda")
    t = torch.cat([torch.linspace(1e-3, 0.9946, 257), torch.tensor([1e-5, 0.5, 0.9946])])

    def scalars(ns, lam=None):
        out = {name: getattr(ns, name)(t) for name in names}
        out["inverse_lambda"] = ns.inverse_lambda(out["marginal_lambda"] if lam is None else lam)
        return out
    b = REF("cosine_scalars", lambda: (lambda old: dict(T=old.T, total_N=old.total_N, lam=S.keep(old.marginal_lambda(t)),
                                                        **scalars(old)))(S.original("sd_dpm_solver").NoiseScheduleVP("cosine")))
    a = NoiseScheduleVP("cosine")
    assert a.T == b["T"] == 0.9946 and a.total_N == b["total_N"]
    got = scalars(a, b["lam"])
    for name in names + ("inverse_lambda",):
        S.assert_same(got[name], b[name], name)


@pytest.mark.parametrize("kw", [dict(steps=12, order=2, method="multistep", skip_type="time_uniform"),
                                dict(steps=10, order=3, method="singlestep", skip_type="logSNR")])
def test_cosine_schedule_sample_matches_vendored_copy(dev, kw):
    """A whole sample() on the cosine schedule against the vendored copy that defines it."""
    import dpm_solver_b200 as new
    x = seeded((2, 3, 8, 8), 31)
    net = lambda xx, tt: 0.1 * xx + ((tt * 0.05) - 0.02).reshape(-1, 1, 1, 1)

    def arm(mod, d):
        ns = mod.NoiseScheduleVP("cosine")
        s = mod.DPM_Solver(mod.model_wrapper(net, ns), ns, algorithm_type="dpmsolver++")
        return s.sample(x.to(d), t_end=1e-3, **kw).cpu()
    want = REF(f"cosine_sample/{kw['steps']}/{kw['order']}/{kw['method']}", lambda: arm(S.original("sd_dpm_solver"), "cpu"))
    assert S.all_finite(want)
    S.assert_same(arm(new, dev), want)


# ---- NaN propagation (ADVICE r1) ----------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(3, 3, 16, 16), (3, 3, 64, 64)])     # cluster kernel / streaming pipeline
def test_dynamic_thresholding_propagates_nan(dev, shape):
    """A NaN in one sample: torch.quantile returns NaN for that sample, clamp and division propagate it (:422-424);
    the other samples are untouched."""
    import dpm_solver_b200 as new
    x0 = seeded(shape, 9) * 2.0
    x0[1, 0, 2, 3] = float("nan")

    def reference():
        ref = S.original()
        want = ref.DPM_Solver(None, _sched(ref)).dynamic_thresholding_fn(x0, None)
        return want, bool(torch.isnan(want[1]).all()), bool(torch.isfinite(want[0]).all())
    want, nan_1, finite_0 = REF(f"thresholding_nan/{shape[-1]}", reference)
    have = new.DPM_Solver(None, _sched(new)).dynamic_thresholding_fn(x0.to(dev), None).cpu()
    assert nan_1 and finite_0
    S.assert_same(have, want)      # NaNs compare equal positionally


def test_adaptive_raises_on_nan_error_estimate(dev):
    """The reference would spin forever on a NaN error estimate (:1002-1008); the product raises."""
    import dpm_solver_b200 as new
    ns = _sched(new, "vp_linear")
    s = new.DPM_Solver(new.model_wrapper(lambda x, t: x * float("nan"), ns), ns, algorithm_type="dpmsolver")
    with pytest.raises(FloatingPointError):
        s.sample(seeded((2, 3, 8, 8), 1).to(dev), method="adaptive", order=2, t_end=1e-3)


# ---- corner cases from ADVICE.md (round 1) ---------------------------------------------------------------------
def test_cfg_on_channels_last_input(dev):
    """out2 = x_in[B:] of a channels_last doubled batch is dense but not `is_contiguous()`."""
    import dpm_solver_b200 as new
    B = 2
    x = seeded((B, 4, 8, 8), 13)

    def arm(mod, d, cl):
        ns = _sched(mod)
        net = lambda xx, tt, cc: exact_net(xx, tt) + 0.05 * cc.reshape(-1, 1, 1, 1)
        fn = mod.model_wrapper(net, ns, guidance_type="classifier-free", condition=torch.ones(B, 1, device=d),
                               unconditional_condition=torch.zeros(B, 1, device=d), guidance_scale=4.0)
        xi = x.to(d)
        if cl:
            xi = xi.contiguous(memory_format=torch.channels_last)
        return mod.DPM_Solver(fn, ns).sample(xi, steps=8, order=2).cpu()
    want = REF("cfg_channels_last", lambda: arm(S.original(), "cpu", False))
    S.assert_same(arm(new, dev, True).contiguous(), want)


def test_fp32_network_output_with_16bit_state_and_thresholding(dev):
    """model fp32 -> state bf16 with dynamic thresholding: quantile and step take the same dtype mix."""
    import dpm_solver_b200 as new
    ns = _sched(new, "ddpm_linear")
    net = lambda xx, tt: exact_net(xx.float(), tt)
    s = new.DPM_Solver(new.model_wrapper(net, ns), ns, correcting_x0_fn="dynamic_thresholding", state_dtype=torch.bfloat16)
    x = seeded((2, 3, 64, 64), 17).to(dev)
    y = s.sample(x, steps=8, order=2)
    assert y.dtype == torch.bfloat16 and torch.isfinite(y.float()).all()

    def fp32_run(mod):
        nr = _sched(mod, "ddpm_linear")
        return mod.DPM_Solver(mod.model_wrapper(net, nr), nr, correcting_x0_fn="dynamic_thresholding").sample(
            x.cpu().bfloat16().float(), steps=8, order=2)
    want = REF("fp32_net_bf16_state", lambda: fp32_run(S.original()))
    # the reference's values: the product's fp32 path on the numpy executor, bit-identical to the stored digest
    from dpm_solver_b200 import ops
    from oracle_backend import OracleBackend
    old = ops._backend
    ops.set_backend(OracleBackend())
    try:
        yr = fp32_run(new)
    finally:
        ops.set_backend(old)
    S.assert_same(yr, want)
    assert rel_err(y.float().cpu().numpy(), yr.numpy()) < 0.06


@pytest.mark.gpu
def test_capture_with_denoise_to_zero(cuda_backend):
    """The denoise tail (:1236-1238) uses cached device tables: the whole run stays CUDA-graph capturable."""
    import dpm_solver_b200 as new
    ns = _sched(new)
    s = new.DPM_Solver(new.model_wrapper(exact_net, ns), ns)
    x = seeded((2, 4, 16, 16), 1234).cuda()
    kw = dict(steps=10, order=2, denoise_to_zero=True)
    eager = s.sample(x, **kw)
    run = s.capture(x, **kw)
    assert torch.equal(run(x), eager)

    def reference():
        ref = S.original()
        nr = _sched(ref)
        return ref.DPM_Solver(ref.model_wrapper(exact_net, nr), nr).sample(x.cpu(), **kw)
    S.assert_same(eager.cpu(), REF("capture_denoise_to_zero", reference))


# ---- in-kernel noise: add_noise(noise=None) and the DiffEdit corrector (SURVEY 8f-3) ------------------------------
def _notebook_corrector(sampler, init_latent, mask):
    """diffedit_inpaint.ipynb, `corrector_fn`, verbatim."""
    def corrector_fn(x, t, step):
        ratio = sampler.time_to_ratio(t)
        stochastic_intermediate = sampler.stochastic_encode(init_latent, ratio)
        x = x * mask + (1 - mask) * stochastic_intermediate
        return x
    return corrector_fn


def test_diffedit_corrector_matches_the_notebook_on_the_host_executor(oracle_backend):
    """DiffEditCorrector == the notebook's corrector_fn on top of the unmodified SD adapter, same CPU generator state.
    The adapter's time round trip (ratio_to_time(time_to_ratio(t))) is stored with the notebook's results."""
    import adapters as A
    import dpm_solver_b200 as new
    x0, x = seeded((1, 4, 16, 16), 3), seeded((1, 4, 16, 16), 4)
    mask = (seeded((16, 16), 5) > 0).float()
    times = [0.9, 0.5, 0.05]

    def reference():
        mod = A.load_sd_adapter(A.reference_solver("sd"), "diffedit_ref", "cpu")
        sampler = mod.DPMSolverSampler(A.StubLatentDiffusion("cpu"))
        ref_fn = _notebook_corrector(sampler, x0, mask)
        out = []
        for step, tv in enumerate(times):
            t = torch.tensor(tv)
            torch.manual_seed(100 + step)
            want = ref_fn(x, t, step)
            out.append((sampler.ratio_to_time(sampler.time_to_ratio(t)), want))
        return S.keep(torch.stack([te for te, _ in out])), [want for _, want in out]
    tes, want = REF("diffedit_notebook", reference)
    ns = new.NoiseScheduleVP("discrete", alphas_cumprod=A.StubLatentDiffusion("cpu").alphas_cumprod)
    got = []
    for step, (tv, te) in enumerate(zip(times, tes)):
        fused = new.DiffEditCorrector(ns, x0, mask, time_fn=lambda t, te=te: te)
        torch.manual_seed(100 + step)
        got.append(fused(x, torch.tensor(tv), step))
    S.assert_same(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,times", [((2, 4, 64, 64), [0.5]), ((3, 3, 17, 5), [0.3, 0.8, 0.05]), ((700, 4, 64, 64), [0.6])])
def test_add_noise_draws_torch_randn_in_the_kernel(cuda_backend, shape, times):
    """add_noise(noise=None): the noise is generated in registers by curand's Philox exactly as torch.randn would
    have (same seed and offset -> same normals, generator advanced identically), then alpha*x + sigma*noise."""
    import dpm_solver_b200 as new
    s = new.DPM_Solver(None, _sched(new))
    x = seeded(shape, 8).cuda()
    t = torch.tensor(times, device="cuda")
    torch.manual_seed(1234)
    torch.randn(5, device="cuda")                                     # a non-zero philox offset
    state = torch.cuda.get_rng_state()
    before = cuda_backend.launch_count()
    got = s.add_noise(x, t)
    assert cuda_backend.launch_count() == before + 1                  # ONE launch, no randn kernel, no noise tensor
    after_fused = torch.cuda.default_generators[0].get_offset()
    torch.cuda.set_rng_state(state)
    noise = torch.randn((len(times), *x.shape), device="cuda")       # what the reference draws (:1024)
    assert torch.cuda.default_generators[0].get_offset() == after_fused
    want = s.add_noise(x, t, noise=noise)                             # explicit-noise path (bit-exact vs the reference)
    assert got.shape == want.shape
    assert torch.equal(got, want)
    want_cpu = REF(f"add_noise_in_kernel/{shape}/{times}", lambda: (lambda ref: ref.DPM_Solver(None, _sched(ref)).add_noise(
        x.cpu(), t.cpu(), noise=noise.cpu()))(S.original()))
    S.assert_same(got.cpu(), want_cpu)


@pytest.mark.gpu
@pytest.mark.parametrize("sdt", [torch.float32, torch.bfloat16])
def test_diffedit_corrector_fused_kernel(cuda_backend, sdt):
    """One launch == x*mask + (1-mask)*(alpha*x0 + sigma*randn) with torch's own normals for the generator state."""
    import dpm_solver_b200 as new
    ns = _sched(new)
    x0, x = seeded((2, 4, 64, 64), 3).cuda().to(sdt), seeded((2, 4, 64, 64), 4).cuda().to(sdt)
    mask = (seeded((64, 64), 5) > 0).float().cuda()
    fused = new.DiffEditCorrector(ns, x0, mask)
    t = torch.tensor([0.4], device="cuda")
    torch.manual_seed(77)
    state = torch.cuda.get_rng_state()
    before = cuda_backend.launch_count()
    got = fused(x, t, 0)
    assert cuda_backend.launch_count() == before + 1
    torch.cuda.set_rng_state(state)
    noise = torch.randn((1, *x0.shape), device="cuda")
    te = t.cpu().to(sdt).float()            # stochastic_encode rebuilds the label in the latent's dtype (sampler.py:94)
    al, sg = float(ns.marginal_alpha(te)), float(ns.marginal_std(te))
    inter = (torch.tensor(al) * x0.float().cpu() + torch.tensor(sg) * noise[0].cpu())
    want = x.float().cpu() * mask.cpu() + (1 - mask.cpu()) * inter
    np.testing.assert_array_equal(got.float().cpu().numpy(), want.to(sdt).float().numpy())
