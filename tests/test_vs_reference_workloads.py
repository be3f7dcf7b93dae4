"""The BENCHMARKED configurations (BASELINE.json configs 2-4 = bench.py workloads c2 / c3 / c4) against the
UNMODIFIED reference (its results stored in tests/golden/reference/), at full per-sample size, on bench.py's own
synthetic inputs.

  * fp32 state: bit-identical to the reference's CPU result (the synthetic network returns stored noise banks, so
    the whole computation is exact IEEE arithmetic in the reference's op order);
  * fp32 state vs the reference executed ON THE GPU (device libm for its schedule scalars): <= 1e-5 relative,
    the north-star tolerance;
  * bf16 / f16 state (`state_dtype=`, the mode bench.py's c2 / c3 run in): storage-precision deviation from the
    fp32 reference, pinned at 1.5x the values measured with the numpy executor -- which the CUDA path reproduces
    bit for bit (tests/test_gpu_sample.py::test_sample_16bit_state):

        max|y - y_ref| / max|y_ref|  (rms(y - y_ref) / rms(y_ref))  measured, seeds 1234 and 7
        c2 ++2M/20  [.,4,64,64]    bf16 2.30e-2 (1.07e-2)   f16 4.09e-3 (1.36e-3)
        c3 eps-3S/15 CFG 7.5       bf16 9.84e-3 (4.07e-3)   f16 1.37e-3 (5.07e-4)
        c4 ++3M/20 + thresholding  bf16 2.34e-2 (5.48e-3)   f16 2.66e-3 (7.11e-4)

The product runs a LARGER batch than the reference slice (TMA ring / persistent-grid paths are the ones exercised);
every op is element-wise or per-sample, so rows [0, n) of its output must equal the reference run on rows [0, n).

Where a bound needs the reference's fp32 values, they are recomputed by the product's fp32 path on the numpy
executor and checked bit for bit against the stored digest of the reference's output first. The reference run as
CUDA ops is stored as a seeded sample of its elements (tests/refstore.py)."""
import numpy as np
import pytest
import torch

import refcheck as R
import refstore as S
from bench import WORKLOADS

REF = S.Store(__file__)

# (max-rel, rms-rel) measured on the numpy executor, see the module docstring
MEASURED_16 = {("c2", torch.bfloat16): (2.30e-2, 1.07e-2), ("c2", torch.float16): (4.09e-3, 1.36e-3),
               ("c3", torch.bfloat16): (9.84e-3, 4.07e-3), ("c3", torch.float16): (1.37e-3, 5.07e-4),
               ("c4", torch.bfloat16): (2.34e-2, 5.48e-3), ("c4", torch.float16): (2.66e-3, 7.11e-4)}
SLACK = 1.5
# product batch on the GPU / reference slice
GPU_B = {"c2": (160, 8), "c3": (160, 8), "c4": (6, 2)}


def reference_values(w, x, banks, key):
    """The reference's fp32 CPU result on (x, banks): the product's fp32 path on the numpy executor, checked bit for
    bit against the stored digest of the reference's own output."""
    from dpm_solver_b200 import ops
    from oracle_backend import OracleBackend
    want = REF(key, lambda: R.reference_sample(w, x, banks))
    old = ops._backend
    ops.set_backend(OracleBackend())
    try:
        y = R.product_sample(w, x.float(), [b.float() for b in banks])
    finally:
        ops.set_backend(old)
    S.assert_same(y, want, key)
    return y


@pytest.mark.parametrize("name", ["c2", "c3", "c4"])
def test_host_logic_bit_exact_vs_reference(oracle_backend, name):
    """CPU: the product's host logic on the numpy executor == the reference, fp32, full per-sample size."""
    w = WORKLOADS[name]
    B = 4 if name != "c4" else 1
    x, banks = R.synthetic(w, B, "cpu", torch.float32)
    yr = REF(f"host_fp32/{name}", lambda: R.reference_sample(w, x, banks))
    yp = R.product_sample(w, x, banks)
    assert S.all_finite(yr)
    S.assert_same(yp, yr)


@pytest.mark.parametrize("name", ["c2", "c3"])
def test_host_logic_bf16_state_bound(oracle_backend, name):
    w = WORKLOADS[name]
    x, banks = R.synthetic(w, 8, "cpu", torch.bfloat16)
    yr = reference_values(w, x, banks, f"host_bf16_inputs/{name}")
    yp = R.product_sample(w, x, banks, state_dtype=torch.bfloat16)
    mx, rms = MEASURED_16[(name, torch.bfloat16)]
    assert R.rel_err(yp.float().numpy(), yr.numpy()) <= SLACK * mx
    assert R.rms_rel_err(yp.float().numpy(), yr.numpy()) <= SLACK * rms


def _gpu_inputs(name, dtype):
    w = WORKLOADS[name]
    Bp, Br = GPU_B[name]
    x, banks = R.synthetic(w, Bp, "cuda:0", dtype)
    xs = x[:Br].cpu()
    bs = [R.slice_rows(b, Bp, Br, w["cfg"]).cpu() for b in banks]
    return w, x, banks, xs, bs, Br


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c2", "c3", "c4"])
def test_gpu_fp32_bit_exact_vs_reference_cpu(cuda_backend, name):
    w, x, banks, xs, bs, Br = _gpu_inputs(name, torch.float32)
    before = cuda_backend.launch_count()
    yp = R.product_sample(w, x, banks)
    assert cuda_backend.launch_count() - before >= w["steps"], "the CUDA library did not run"
    yr = REF(f"gpu_fp32/{name}", lambda: R.reference_sample(w, xs, bs, device="cpu"))   # the reference on the host
    S.assert_same(yp[:Br].cpu(), yr)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c2", "c3", "c4"])
def test_gpu_fp32_vs_reference_on_the_gpu(cuda_backend, name):
    """Reference executed as eager CUDA ops (its schedule scalars come from the device's exp/log/expm1)."""
    w, x, banks, xs, bs, Br = _gpu_inputs(name, torch.float32)
    yp = R.product_sample(w, x, banks)

    yr = REF(f"gpu_on_gpu/{name}", lambda: S.sample(R.reference_sample(w, xs, bs, device="cuda:0")))
    assert yr.rel_err(yp[:Br]) <= 1e-5      # BASELINE.json north_star tolerance


@pytest.mark.gpu
@pytest.mark.parametrize("sdt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("name", ["c2", "c3", "c4"])
def test_gpu_16bit_state_bound_vs_reference(cuda_backend, name, sdt):
    """The mode the headline numbers run in: 16-bit x / buffers / network output, fp32 arithmetic."""
    w, x, banks, xs, bs, Br = _gpu_inputs(name, sdt)
    yp = R.product_sample(w, x, banks, state_dtype=sdt)
    assert yp.dtype == sdt
    yr = reference_values(w, xs, bs, f"gpu_16bit_inputs/{name}/{sdt}")   # fp32 reference on the same (16-bit) inputs
    mx, rms = MEASURED_16[(name, sdt)]
    got = yp[:Br].float().cpu().numpy()
    assert R.rel_err(got, yr.numpy()) <= SLACK * mx
    assert R.rms_rel_err(got, yr.numpy()) <= SLACK * rms
    # and bit-identical to the numpy executor with the same storage semantics (no thresholding: the quantile's
    # tie handling is covered by tests/test_gpu_kernels.py)
    if not w["thresholding"]:
        from dpm_solver_b200 import ops
        from oracle_backend import OracleBackend
        old = ops._backend
        ops.set_backend(OracleBackend())
        try:
            ye = R.product_sample(w, xs, bs, state_dtype=sdt)
        finally:
            ops.set_backend(old)
        assert torch.equal(yp[:Br].cpu(), ye)
