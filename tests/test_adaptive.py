"""dpm_solver_adaptive (:956-1010): same NFE and the same sample as the reference. The error estimate
is a reduction (its summation order differs between torch-CPU, numpy and the CUDA kernel), so the
sample is compared with the north-star tolerance instead of bit for bit; the accept/reject decisions
-- hence the NFE the reference prints -- must be identical."""
import numpy as np
import pytest
import torch

import refstore as S
from cases import exact_net, make_betas, seeded
from helpers import product_schedule, rel_err

REF = S.Store(__file__)

CASES = [
    dict(name="ad23_eps_vp", schedule="vp_linear", algo="dpmsolver", order=3, t_end=1e-3, solver_type="dpmsolver"),
    dict(name="ad12_eps_vp", schedule="vp_linear", algo="dpmsolver", order=2, t_end=1e-3, solver_type="dpmsolver"),
    dict(name="ad23_pp_sd", schedule="sd", algo="dpmsolver++", order=3, t_end=None, solver_type="taylor"),
    dict(name="ad12_pp_sd", schedule="sd", algo="dpmsolver++", order=2, t_end=None, solver_type="dpmsolver"),
]


def run(c, device, capsys):
    from dpm_solver_b200 import DPM_Solver, model_wrapper
    ns = product_schedule(c["schedule"])
    x = seeded((2, 3, 8, 8), 77).to(device)
    s = DPM_Solver(model_wrapper(exact_net, ns), ns, algorithm_type=c["algo"])
    y = s.sample(x, method="adaptive", order=c["order"], t_end=c["t_end"], solver_type=c["solver_type"])
    nfe = int(capsys.readouterr().out.split()[-1])
    return y, nfe


@pytest.fixture(scope="module")
def gold():
    import os
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "adaptive.npz"))


@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_adaptive_host_logic(gold, oracle_backend, capsys, c):
    y, nfe = run(c, "cpu", capsys)
    assert nfe == int(gold[c["name"] + "/nfe"])
    assert rel_err(y.numpy(), gold[c["name"] + "/y"]) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_adaptive_gpu(gold, cuda_backend, capsys, monkeypatch, c):
    """Default (device controller): its scalars are correctly rounded fp32 (fp64 evaluation, one rounding), the host's
    SLEEF results differ from that in the last ulp of a few arguments, and an adaptive solve amplifies an ulp through
    h = theta*h*E^(-1/order): same decisions and NFE, the sample within 1e-4 -- on 40 random configurations it is
    bit-identical to the reference's CPU run in 30 and within 5e-5 in the rest, while the reference's own CUDA run
    strays up to 3e-2 and changes NFE once (profiles/r02_adaptive_probe.txt). Host controller: the north-star 1e-5."""
    from dpm_solver_b200 import DPM_Solver
    y, nfe = run(c, "cuda:0", capsys)
    assert nfe == int(gold[c["name"] + "/nfe"])
    assert rel_err(y.cpu().numpy(), gold[c["name"] + "/y"]) <= 1e-4
    monkeypatch.setattr(DPM_Solver, "adaptive_controller", "host")
    y, nfe = run(c, "cuda:0", capsys)
    assert nfe == int(gold[c["name"] + "/nfe"])
    assert rel_err(y.cpu().numpy(), gold[c["name"] + "/y"]) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("shape,dt", [((5, 3, 64, 64), torch.float32), ((3, 1001), torch.float32), ((4, 4, 64, 64), torch.bfloat16)])
def test_error_norm_kernel(cuda_backend, shape, dt):
    g = torch.Generator().manual_seed(5)
    xh, xl, xp = (torch.randn(shape, generator=g).to(dt) for _ in range(3))
    xl = (xh.float() + 0.01 * xl.float()).to(dt)
    got = float(cuda_backend.error_norm(xh.cuda(), xl.cuda(), xp.cuda(), 0.0078, 0.05).cpu())
    h, l, p = (t.double().numpy() for t in (xh, xl, xp))
    delta = np.maximum(0.0078, 0.05 * np.maximum(np.abs(l), np.abs(p)))
    ref = np.sqrt(np.mean(np.square(((h - l) / delta).reshape(shape[0], -1)), axis=-1)).max()
    assert abs(got - ref) <= 2e-6 * ref


# ---- the controller on the device (csrc/adaptive_ctl.cu) ------------------------------------------------------------
def _adaptive_cfgs(n, seed):
    import random
    from test_random_configs_vs_reference import draw_wide
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        c = draw_wide(rng)
        c.update(method="adaptive", order=rng.choice([2, 3]), atol=rng.choice([0.0078, 0.05]), rtol=rng.choice([0.05, 0.2]),
                 thresholding=False, denoise_to_zero=False)
        if c["schedule"] == "iddpm_cosine":
            continue
        out.append(c)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", range(4))
def test_device_controller_matches_reference(cuda_backend, chunk):
    """Random adaptive configurations (schedules, both algorithms and solver types, all parameterisations, CFG,
    t_start / t_end, batch shapes): the device-side controller takes the accept/reject decisions of the UNMODIFIED
    reference (same NFE) and lands on its sample within the reduction-order / device-libm tolerance."""
    import contextlib
    import io
    import dpm_solver_b200 as new
    from test_random_configs_vs_reference import run_wide

    class OnGpu:        # run_wide() builds CPU tensors: move the product arm to the device
        NoiseScheduleVP = new.NoiseScheduleVP

        @staticmethod
        def model_wrapper(net, ns, **kw):
            kw = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in kw.items()}
            return new.model_wrapper(net, ns, **kw)

        class DPM_Solver(new.DPM_Solver):
            def sample(self, x, **kw):
                return super().sample(x.cuda(), **kw).cpu()

    from unittest import mock
    seen_device = 0
    def reference(c):
        with mock.patch("builtins.print") as pr:           # both print 'adaptive solver nfe', N (:1009)
            yr, _, _ = run_wide(S.original(), c)
        return S.sample(yr), pr.call_args[0][-1]

    for i, c in enumerate(_adaptive_cfgs(10, 9000 + chunk)):
        yr, nfe_r = REF(f"device_controller/{chunk}/{i}", lambda: reference(c))
        if not S.all_finite(yr):
            continue
        before = cuda_backend.launch_count()
        with mock.patch("builtins.print") as pn:
            yn, _, _ = run_wide(OnGpu, c)
        seen_device += cuda_backend.launch_count() > before
        assert pn.call_args[0][-1] == nfe_r, ("NFE", c)
        assert yr.rel_err(yn) <= 2e-4, c      # measured: 0 .. 5e-5 (profiles/r02_adaptive_probe.txt)
    assert seen_device


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_device_controller_syncs_once_per_chunk(gold, cuda_backend, capsys, monkeypatch, c):
    """The only device->host read of the adaptive loop is AdaptiveController.read(): once per `adaptive_chunk`
    iterations. Same NFE and sample as the host controller (the reference's per-iteration decision)."""
    from dpm_solver_b200 import DPM_Solver, model_wrapper, ops
    reads = []
    orig = ops.AdaptiveController.read

    def counting(self):
        r = orig(self)
        reads.append(r)
        return r
    monkeypatch.setattr(ops.AdaptiveController, "read", counting)
    y_dev, nfe_dev = run(c, "cuda:0", capsys)
    iters = reads[-1][2]
    assert len(reads) == -(-iters // DPM_Solver.adaptive_chunk) and reads[-1][0] == 1
    assert nfe_dev == int(gold[c["name"] + "/nfe"]) == iters * c["order"]
    monkeypatch.setattr(DPM_Solver, "adaptive_controller", "host")
    y_host, nfe_host = run(c, "cuda:0", capsys)
    assert nfe_host == nfe_dev
    assert rel_err(y_dev.cpu().numpy(), y_host.cpu().numpy()) <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["sd", "vp_linear", "ddpm_linear"])
@pytest.mark.parametrize("algo", ["dpmsolver++", "dpmsolver"])
@pytest.mark.parametrize("solver_type", ["dpmsolver", "taylor"])
@pytest.mark.parametrize("order", [2, 3])
def test_plan_kernel_coefficients_match_host_plan(cuda_backend, schedule, algo, solver_type, order):
    """k_adapt_plan against plan.py (the reference's formulas evaluated with torch-CPU scalars): t, the evaluation
    times, the model-input times and every coefficient block, to a few ulps of the device's expf/logf/expm1f."""
    from dpm_solver_b200 import plan as P
    ns = product_schedule(schedule)
    t_0 = 1e-3 if schedule == "vp_linear" else 1. / ns.total_N
    ctl = cuda_backend.adaptive_controller(ns, torch.device("cuda:0"), order=order, predict_x0=algo == "dpmsolver++",
                                           taylor=solver_type == "taylor", t_0=t_0, theta=0.9, t_err=1e-5,
                                           discrete_input=schedule != "vp_linear")
    for t_T, h0 in [(1.0, 0.05), (0.7, 0.31), (0.2, 0.9)]:
        ctl.init(t_T, h0)
        ctl.plan()
        coef, times, st = ctl.coef.cpu().numpy(), ctl.times.cpu().numpy(), ctl.state.cpu().numpy()
        s = torch.tensor([t_T])
        lam_s = ns.marginal_lambda(s)
        assert abs(st[1] - float(lam_s)) <= 4e-6 * max(1.0, abs(float(lam_s)))
        t = ns.inverse_lambda(lam_s + h0)
        assert abs(st[4] - float(t)) <= 2e-6

        def close(block, co, alsig_time):
            want = [co.a, co.c0, co.c1, co.c2]
            np.testing.assert_allclose(block[:4], want, rtol=3e-5, atol=5e-6)   # phi_3 = phi_2/h - 0.5 cancels: an ulp of expm1f is 3e-4 of it
            if co.form == 6:
                np.testing.assert_allclose(block[4:9], [co.w0, co.w1, co.w2, co.w3, co.w4], rtol=1e-6)
            al, sg = float(ns.marginal_alpha(alsig_time)), float(ns.marginal_std(alsig_time))
            np.testing.assert_allclose(block[9:11], [al, sg], rtol=2e-5, atol=1e-7)

        if order == 2:
            low = P.first_update_coeffs(ns, algo, s, t)
            high = P.singlestep_second(ns, algo, solver_type, s, t, 0.5)
            close(coef[0], low, s)
            close(coef[1], high.stages[0], s)
            close(coef[2], high.stages[1], high.times[1])
            ev = high.times
        else:
            low = P.singlestep_second(ns, algo, solver_type, s, t, 1. / 3.)
            high = P.singlestep_third(ns, algo, solver_type, s, t, 1. / 3., 2. / 3.)
            close(coef[0], low.stages[0], s)
            close(coef[1], low.stages[1], low.times[1])
            close(coef[2], high.stages[1], high.times[1])
            close(coef[3], high.stages[2], high.times[2])
            ev = high.times
        for j, tj in enumerate(ev):
            assert abs(times[j] - float(tj)) <= 2e-6
            want_in = (float(tj) - 1. / ns.total_N) * 1000. if schedule != "vp_linear" else float(tj)
            assert abs(times[3 + j] - want_in) <= 2e-3
