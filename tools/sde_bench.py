"""SDE-DPM-Solver++ 2M against its alternatives on one GPU, in one process, arms alternating.

    python tools/sde_bench.py [--reps 5] [--samples 3] [--out FILE]

Workload: the c2 shape of bench.py -- 20 steps, synthetic eps (network = a bank of three precomputed bf16 outputs),
bf16 state [4096,4,64,64], time_uniform grid, sd schedule. Arms:
  (a) sde-dpmsolver++ 2M, noise generated in registers by the fused step (csrc/step_sde.cu);
  (b) the same kernel reading materialised noise: torch.randn_like(x, dtype=float32) per step, its time included;
  (c) the ODE dpmsolver++ 2M.
Each rep times `--samples` sample() calls of every arm in turn with CUDA events; the medians over reps are reported
as ms per sample() and GElem/s (elements x steps per second). The fused step of each arm is then timed alone
(100 launches between two events) and reported as algorithmic GB/s against the HBM peak, which is measured here as
the rate of a 4 GiB device-to-device copy (read + write bytes). GPU name and power limit are read in the same run.
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from cases import make_betas  # noqa: E402
from dpm_solver_b200 import DPM_Solver, NoiseScheduleVP, model_wrapper, ops  # noqa: E402
from dpm_solver_b200._lib import FORM_DIFF2  # noqa: E402
from dpm_solver_b200.ops import StepArgs  # noqa: E402

SHAPE, STEPS, DT = (4096, 4, 64, 64), 20, torch.bfloat16


class MaterialisedNoise(ops.CudaBackend):
    """Arm (b): torch draws the noise into HBM, the step kernel reads it."""

    def sde_step(self, a, noise_scale, generator=None, noise=None):
        z = torch.randn_like(a.reference_tensor(), dtype=torch.float32, generator=generator)
        return super().sde_step(a, noise_scale, noise=z)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001
        q = f"unavailable ({e})"
    return name, q


def copy_peak_gbs(reps=20):
    src = torch.empty(1 << 31, dtype=torch.int16, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    return 2 * src.numel() * 2 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--samples", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    lines = []
    say = lambda s: (print(s, flush=True), lines.append(s))

    name, power = gpu_info()
    say(f"GPU: {name}; power.limit, clocks.max.sm: {power}")
    say(f"workload: {SHAPE} bf16 state, {STEPS} steps, 2M (order 2), synthetic eps, sd schedule, time_uniform")

    kind, betas = make_betas("sd")
    ns = NoiseScheduleVP("discrete", betas=torch.from_numpy(betas))
    g = torch.Generator(dev).manual_seed(1234)
    x_T = torch.randn(SHAPE, device=dev, generator=g).to(DT)
    banks = [torch.randn(SHAPE, device=dev, generator=g).to(DT) for _ in range(3)]
    cnt = [0]

    def net(xx, tt):
        cnt[0] += 1
        return banks[cnt[0] % 3]

    fn = model_wrapper(net, ns)
    arms = {
        "a_sde_in_kernel_noise": (ops.CudaBackend(), DPM_Solver(fn, ns, algorithm_type="sde-dpmsolver++", state_dtype=DT)),
        "b_sde_materialised_randn": (MaterialisedNoise(), DPM_Solver(fn, ns, algorithm_type="sde-dpmsolver++", state_dtype=DT)),
        "c_ode_dpmsolver++": (ops.CudaBackend(), DPM_Solver(fn, ns, algorithm_type="dpmsolver++", state_dtype=DT)),
    }
    kw = dict(steps=STEPS, order=2, method="multistep", skip_type="time_uniform")
    old = ops._backend
    times = {k: [] for k in arms}
    launches = {}
    try:
        for k, (be, s) in arms.items():          # warm-up: plans, tables, modules
            ops.set_backend(be)
            for _ in range(2):
                s.sample(x_T, **kw)
            torch.cuda.synchronize()
            l0 = be.launch_count()
            s.sample(x_T, **kw)
            launches[k] = be.launch_count() - l0
        for _ in range(args.reps):
            for k, (be, s) in arms.items():
                ops.set_backend(be)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.samples):
                    s.sample(x_T, **kw)
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / args.samples)
    finally:
        ops.set_backend(old)

    E = x_T.numel()
    say("")
    say(f"end to end, median of {args.reps} alternating reps x {args.samples} sample() calls:")
    say(f"{'arm':28s} {'ms/sample':>10s} {'GElem/s':>9s} {'library launches/sample':>24s}  (all reps, ms)")
    for k, v in times.items():
        med = statistics.median(v)
        say(f"{k:28s} {med:10.3f} {E * STEPS / (med * 1e-3) / 1e9:9.1f} {launches[k]:24d}  "
            + " ".join(f"{t:.3f}" for t in v))

    # ---- the fused step alone: sde-dpmsolver++ 2M step (DIFF2, one raw output -> x0, m_out + out) ----
    peak = copy_peak_gbs()
    say("")
    say(f"HBM peak measured here (4 GiB device-to-device copy, read + write): {peak:.0f} GB/s")
    ga = torch.Generator(dev).manual_seed(7)
    mk = lambda: torch.randn(SHAPE, device=dev, generator=ga).to(DT)
    x, ec, m1 = mk(), mk(), mk()
    out, m_out = torch.empty_like(x), torch.empty_like(x)
    a = StepArgs(form=FORM_DIFF2, n_model=1, x=x, xe=x, e_cond=ec, m1=m1, predict_x0=True, alpha_e=0.83, sigma_e=0.55,
                 a=0.9, c0=0.1, c1=0.05, w0=1.3, want_m_out=True, out=out, m_out=m_out, state_dtype=DT)
    be = ops.CudaBackend()
    z = torch.empty(SHAPE, device=dev, dtype=torch.float32)
    step_arms = {
        "a: sde step, in-kernel noise": (lambda: be.sde_step(a, 0.3), 10),
        "b: randn + sde step reading it": (lambda: (z.normal_(), be.sde_step(a, 0.3, noise=z)), 18),
        "b: sde step reading noise only": (lambda: be.sde_step(a, 0.3, noise=z), 14),
        "c: ode step (dpm_step)": (lambda: be.step(a), 10),
    }
    say("fused step alone, 100 launches between two events, median of 5 alternating reps:")
    say(f"{'kernel':32s} {'us/launch':>10s} {'B/elem':>7s} {'GB/s':>8s} {'of peak':>8s} {'GElem/s':>8s}")
    st = {k: [] for k in step_arms}
    for fn_, _ in step_arms.values():
        fn_()
    for _ in range(5):
        for k, (fn_, _) in step_arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(100):
                fn_()
            e1.record()
            torch.cuda.synchronize()
            st[k].append(e0.elapsed_time(e1) * 1e3 / 100)
    for k, (_, bpe) in step_arms.items():
        us = statistics.median(st[k])
        gbs = E * bpe / (us * 1e-6) / 1e9
        say(f"{k:32s} {us:10.1f} {bpe:7d} {gbs:8.0f} {gbs / peak:8.2f} {E / (us * 1e-6) / 1e9:8.1f}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
