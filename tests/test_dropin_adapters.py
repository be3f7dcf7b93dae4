"""T5 drop-in acceptance: the reference's three example adapters (Stable Diffusion `DPMSolverSampler`, score_sde
`get_dpm_solver_sampler`, guided-diffusion `Diffusion.sample_image`) are executed UNMODIFIED twice -- once on the
reference's own solver on CPU, once on dpm_solver_b200 -- with stub networks. Outputs must be bit-identical
(classifier guidance on the GPU: <= 1e-5, the log_softmax gradient runs through the device's exp()).

Two executors for the product arm: the numpy executor on CPU (host logic, `-m "not gpu"`) and CudaBackend on
cuda:0 (`-m gpu`, the adapters run on the sm_100a kernels through the C-ABI). The reference bytecode comes from
oracle/_ref (tests/adapters.py)."""
import os
import sys

import numpy as np
import pytest
import torch

import adapters as A
from helpers import rel_err

# the adapters are the original project's own example code, which is not part of this repository
needs_adapters = pytest.mark.skipif(not A.available(), reason="the original project's example adapters are not available")

EXECUTORS = ["numpy-executor", pytest.param("cuda", marks=pytest.mark.gpu)]


@pytest.fixture(params=EXECUTORS)
def product_device(request):
    """Installs the executor for the product arm and yields the device its tensors live on."""
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


def _launches():
    from dpm_solver_b200 import ops
    be = ops.backend()
    return be.launch_count() if hasattr(be, "launch_count") else 0


@needs_adapters
@pytest.mark.parametrize("order,steps,method", [(2, 20, "multistep"), (3, 12, "multistep"), (2, 9, "singlestep")])
@pytest.mark.parametrize("tables", ["host", "device"])
def test_stable_diffusion_adapter_runs_unchanged(product_device, order, steps, method, tables):
    """tables="device": the adapter's own behaviour on a GPU -- it moves alphas_cumprod to the device
    (sampler.py:23-27), so NoiseScheduleVP takes its log() THERE and the schedule table differs from a CPU-built
    one in the last ulp of a few entries: the product is then within the north-star tolerance of the CPU reference.
    tables="host": the same adapter with the table kept on the host -> bit-identical."""
    import dpm_solver_b200
    if product_device == "cpu" and tables == "device":
        pytest.skip("same as host on the CPU executor")
    B, shape = 2, (4, 16, 16)
    x_T = torch.randn(B, *shape, generator=torch.Generator().manual_seed(3))
    outs = []
    before = _launches()
    for tag, solver, dev in (("ref", A.reference_solver("sd"), "cpu"), ("b200", dpm_solver_b200, product_device)):
        tdev = dev if tables == "device" else "cpu"
        mod = A.load_sd_adapter(solver, tag + product_device.replace(":", "") + tables, tdev)
        model = A.StubLatentDiffusion(tdev)
        sampler = mod.DPMSolverSampler(model)
        assert sampler.noise_schedule.total_N == 1000
        cond, uncond = torch.ones(B, 1, device=dev), torch.zeros(B, 1, device=dev)
        x, inter = sampler.sample(S=steps, batch_size=B, shape=shape, conditioning=cond, x_T=x_T.clone().to(dev),
                                  unconditional_guidance_scale=7.5, unconditional_conditioning=uncond,
                                  order=order, method=method, verbose=False)
        enc = sampler.stochastic_encode(x_T.to(dev), 0.5, noise=torch.ones_like(x_T).to(dev))
        inv, _ = sampler.encode(S=10, x=x_T.to(dev), encode_ratio=0.6, conditioning=cond,
                                unconditional_guidance_scale=3.0, unconditional_conditioning=uncond)
        outs.append((x.cpu(), [i.cpu() for i in inter], enc.cpu(), inv.cpu(), model.calls))
    (xr, ir, er, vr, cr), (xn, in_, en, vn, cn) = outs
    if product_device != "cpu":
        assert _launches() > before, "the CUDA library did not run"
    assert [c[1] for c in cr] == [c[1] for c in cn]     # same network calls: doubled batch ...
    np.testing.assert_allclose([c[0] for c in cn], [c[0] for c in cr], rtol=1e-6)   # ... same time labels
    assert len(ir) == len(in_)
    if tables == "host":
        np.testing.assert_array_equal(xn.numpy(), xr.numpy())
        for a, b in zip(ir, in_):
            np.testing.assert_array_equal(b.numpy(), a.numpy())
        np.testing.assert_array_equal(en.numpy(), er.numpy())
        np.testing.assert_array_equal(vn.numpy(), vr.numpy())
    else:
        for a, b in [(xr, xn), (er, en), (vr, vn)] + list(zip(ir, in_)):
            assert rel_err(b.numpy(), a.numpy()) <= 1e-5


def _sde_net(x, t):
    return 0.1 * x + ((t * 0.05) - 0.02).reshape(-1, 1, 1, 1)


@needs_adapters
@pytest.mark.parametrize("kw", [dict(), dict(denoise=True, steps=13), dict(algorithm_type="dpmsolver++", thresholding=True, order=2, steps=8),
                                dict(skip_type="time_uniform", method="multistep", order=2, steps=12)])
def test_score_sde_glue_runs_unchanged(product_device, kw):
    """Continuous 'linear' VP schedule, singlestep order 3, logSNR grid, optional denoise / thresholding. The
    example's own vendored (older) solver copy calls `correcting_x0_fn(x0)` with one argument and raises TypeError
    with thresholding (examples/score_sde_pytorch/dpm_solver.py:449), so the current root file is the reference."""
    import dpm_solver_b200
    outs = []
    for tag, solver, dev in (("ref", A.reference_solver("root"), "cpu"), ("b200", dpm_solver_b200, product_device)):
        sampling = A.load_score_sde_sampling(solver, tag)
        fn = sampling.get_dpm_solver_sampler(A.StubVPSDE(), (2, 3, 8, 8), lambda v: v, device=dev, **kw)
        x, nfe = fn(_sde_net)
        outs.append((x.cpu(), nfe))
    assert outs[0][1] == outs[1][1]
    np.testing.assert_array_equal(outs[1][0].numpy(), outs[0][0].numpy())


@needs_adapters
@pytest.mark.parametrize("kw", [dict(),                                                       # classifier guidance + thresholding, ++3M
                                dict(cond_class=False, thresholding=False, sample_type="dpmsolver", order=2, method="singlestep"),
                                dict(denoise=True, timesteps=10, order=2),
                                dict(thresholding=False, scale=0.5, fixed_class=None)])
def test_guided_diffusion_runner_runs_unchanged(product_device, kw):
    """`Diffusion.sample_image` (runners/diffusion.py:524-639): 6-channel network output split to the mean,
    classifier guidance through autograd (:605-608, reference :315-321), dynamic thresholding, DDPM linear betas."""
    import dpm_solver_b200
    from cases import make_betas
    betas = torch.from_numpy(make_betas("ddpm_linear")[1]).float()
    x_T = torch.randn(3, 3, 16, 16, generator=torch.Generator().manual_seed(11))
    use_classifier = kw.get("cond_class", True)
    outs = []
    for tag, solver, dev in (("ref", A.reference_solver("guided"), "cpu"), ("b200", dpm_solver_b200, product_device)):
        _, sample_image = A.load_guided_runner(solver, tag)
        # the schedule is built from `betas` where they live; on the host in both arms, so that the table (a log and
        # a cumsum, :100-104) is the same one -- a device-side cumsum sums in another order
        me = A.guided_self(betas, **kw)
        torch.manual_seed(5)                      # the runner draws the class labels with the global generator (:534-536)
        x, classes = sample_image(me, x_T.to(dev), A.guided_net, last=True,
                                  classifier=A.guided_classifier if use_classifier else None)
        outs.append((x.cpu(), None if classes is None else classes.cpu()))
    (xr, cr), (xn, cn) = outs
    if cr is not None:
        assert torch.equal(cr, cn)
    assert torch.isfinite(xr).all()
    if product_device == "cpu" or not use_classifier:
        np.testing.assert_array_equal(xn.numpy(), xr.numpy())
    else:
        assert rel_err(xn.numpy(), xr.numpy()) <= 1e-5


def test_root_module_name_is_a_drop_in():
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.modules.pop("dpm_solver_pytorch", None)
    import dpm_solver_pytorch as m
    import dpm_solver_b200
    assert m.DPM_Solver is dpm_solver_b200.DPM_Solver and m.NoiseScheduleVP is dpm_solver_b200.NoiseScheduleVP
    assert m.model_wrapper is dpm_solver_b200.model_wrapper
