#!/usr/bin/env python
"""bench.py -- solver-update throughput of the DPM-Solver hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c3|c4] [--dump-outputs DIR]

One "step" = one full DPM_Solver.sample() over one batch of synthetic input (BASELINE.json
configs[1]: DPM-Solver++ 2M, 20 solver updates, synthetic eps, bf16 latents [4096,4,64,64] per GPU).
metric = solver-update GElem/s = elements(x) * updates / seconds, whole job over all N GPUs.

  value     : inputs resident in HBM, CUDA-event timed over the K steps, max over ranks; no per-launch events in this
              pass (they cost ~7 % of the loop); an instrumented pass of the same K steps follows for the breakdown
  e2e       : same metric through the public API with HOST buffers: x_T comes from pinned host
              memory and the result goes back to host inside the timed region
  roofline  : dominant kernel (fused post-model 2M step): algorithmic bytes / CUDA-event time of
              every launch inside the timed region, against the measured HBM peak
  kernels   : the same for each kernel form seen, plus the north-star kernel (fused 3rd-order
              multistep update at [4096,4,64,64], bf16 and fp32) timed alone
  cpu_baseline : the reference algorithm on the host cores (oracle, torch-CPU namespace: the same
              chain of ATen elementwise ops and sort-based interpolation the reference executes)

  workloads : (default N=1 run) the other single-GPU BASELINE configs, c3 and c4, each with value / roofline / clocks
  parity    : outside the timed region, a batch slice of the run's own output is compared with the UNMODIFIED
              reference (oracle/_ref, CPU fp32) on the same inputs -> config.parity_checked

--dump-outputs DIR writes what the last timed sample() of the headline workload returned (rank 0), as float32:
DIR/x_0.npy holds DUMP_ROWS samples of the batch, rows picked by a fixed seed. The inputs are seeded and the
synthetic network's bank rotation depends only on --steps / --warmup, so two builds of the project run with the same
arguments can be compared output for output.

--impl reference runs the UNMODIFIED reference (oracle/_ref: /root/reference/dpm_solver_pytorch.py byte-compiled by
oracle/build_ref.py, shipped to the box) on the host cores; the oracle port is only the fallback when that
bytecode is missing (cpu_baseline.kind says which).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (shape per GPU, dtype, algorithm, method, order, steps, cfg scale, thresholding, schedule)
    "c2": dict(shape=(4096, 4, 64, 64), dtype="bf16", algo="dpmsolver++", method="multistep", order=2, steps=20,
               cfg=None, thresholding=False, schedule="sd",
               desc="DPM-Solver++2M, 20 steps, synthetic eps, bf16 latents [4096,4,64,64] per GPU"),
    "c3": dict(shape=(2048, 4, 64, 64), dtype="bf16", algo="dpmsolver", method="singlestep", order=3, steps=15,
               cfg=7.5, thresholding=False, schedule="sd",
               desc="DPM-Solver-3 singlestep, 15 steps, CFG 7.5, bf16 [2048,4,64,64] per GPU"),
    "c4": dict(shape=(1024, 3, 256, 256), dtype="f32", algo="dpmsolver++", method="multistep", order=3, steps=20,
               cfg=None, thresholding=True, schedule="ddpm_linear",
               desc="DPM-Solver++3M + dynamic thresholding, fp32 pixel-space [1024,3,256,256] per GPU"),
}
DT = {"bf16": torch.bfloat16, "f32": torch.float32, "f16": torch.float16}
FORM_NAMES = {0: "convert", 1: "first(lin1)", 2: "lin2", 3: "lin3", 4: "diff2(2M/2S)", 5: "ms3(3M)", 6: "ss3-taylor"}


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def usable_cores():
    """Host cores this process may use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except Exception:
        pass
    return n


def n_updates(w):
    return w["steps"]  # NFE == steps; every model evaluation is followed by exactly one state update


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of one GPU DURING a timed region: NVML polled from a thread every
    2 ms (nvidia-smi -lms as a fallback when the NVML bindings are missing)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.rows, self.proc, self.index, self.stop, self.thr, self.h = [], None, index, False, None, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)

    def _poll(self):
        nv, h = self.nv, self.h
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = int(get_reasons(h))
                self.rows.append([str(sm), str(mx), "0"] + [("Active" if r & bit else "Not Active") for bit in (0x8, 0x40, 0x20, 0x4)])
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        try:
            self.nv, self.h = self._nvml_handle()
            self.thr = threading.Thread(target=self._poll, daemon=True)
            self.thr.start()
            return self
        except Exception:
            self.h = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.h is not None and not self.rows:
            # a timed region shorter than the poller's start-up (a few ms): take one sample right at its end
            try:
                nv, h = self.nv, self.h
                get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                r = int(get_reasons(h))
                self.rows.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)), "0"] +
                                 [("Active" if r & bit else "Not Active") for bit in (0x8, 0x40, 0x20, 0x4)])
            except Exception:
                pass
        self.stop = True
        if self.h is not None and self.thr is not None:
            self.thr.join(timeout=1)
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm on host cores
# ------------------------------------------------------------------------------------------------
def host_cores():
    return os.cpu_count() or 1


def _reference_once(w, sample_batch):
    """Closure running one sample() of the UNMODIFIED reference (oracle/_ref) on CPU, or None if unavailable."""
    try:
        import refcheck as R
        from oracle import ref_loader
        if not ref_loader.available():
            return None
        ref = ref_loader.load("dpm_solver_pytorch")
    except Exception:
        return None
    x, banks = R.synthetic(w, sample_batch, "cpu", torch.float32, nbanks=2)
    solver, _ = R._solver(ref, w, banks, "cpu")
    kw = R.sample_kwargs(w)
    return lambda: solver.sample(x, **kw)


def _port_once(w, sample_batch):
    from cases import make_betas
    from oracle import dpm_oracle as O
    TH = O.torch_namespace()
    kind, betas = make_betas(w["schedule"])
    ns = O.VPSchedule.from_betas(betas, xp=TH) if kind == "discrete" else O.VPSchedule("linear", xp=TH)
    shape = (sample_batch,) + tuple(w["shape"][1:])
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(shape, generator=g)
    nb = 2 if w["cfg"] else 1
    banks = [torch.randn((nb * sample_batch,) + shape[1:], generator=g) for _ in range(2)]
    cnt = [0]

    def net(xx, tt):
        cnt[0] += 1
        return banks[cnt[0] % 2]

    smp = O.Sampler(ns, net, algorithm_type=w["algo"], guidance_scale=w["cfg"],
                    thresholding=(0.995, 1.0) if w["thresholding"] else None)
    if w["method"] == "multistep":
        return lambda: smp.multistep(x, w["steps"], w["order"])
    return lambda: smp.singlestep(x, w["steps"], w["order"])


def cpu_arm(w, sample_batch, repeats=1, warmup=0):
    """Time the reference's own CPU implementation on a bounded sample of the workload: the unmodified reference
    from oracle/_ref (kind "reference"), else the oracle port in its torch-CPU namespace (kind "port").
    Returns (GElem/s, seconds per sample() call, threads used, kind)."""
    once, kind = _reference_once(w, sample_batch), "reference"
    if once is None:
        once, kind = _port_once(w, sample_batch), "port"
    cores = usable_cores()
    with torch.no_grad():
        # "all the host threads it can use": on many-core hosts the reference's small scalar ops and
        # MB-sized tensors run slower with every core than with a few, so take the fastest setting
        best = None
        for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
            torch.set_num_threads(nt)
            once()
            t0 = time.perf_counter()
            once()
            dt1 = time.perf_counter() - t0
            if best is None or dt1 < best[0]:
                best = (dt1, nt)
        threads = best[1]
        torch.set_num_threads(threads)
        for _ in range(warmup):
            once()
        t0 = time.perf_counter()
        for _ in range(repeats):
            once()
        dt = (time.perf_counter() - t0) / repeats
    E = sample_batch * int(np.prod(w["shape"][1:]))
    return E * n_updates(w) / dt / 1e9, dt, threads, kind


def cpu_sample_batch(w):
    """Bounded sample of the per-GPU batch for the CPU arms: 8.4 M (latents) / 3.1 M (pixels) elements per tensor --
    33 / 12.6 MB fp32, beyond the per-core caches, about a second per sample() call."""
    return 512 if w["shape"][-1] <= 64 else 16


def eager_cuda_arm(w, dev, repeats=3):
    """The second, fairer baseline: the UNMODIFIED reference (oracle/_ref) run as stock eager PyTorch CUDA ops on the
    same GPU -- per update 3/7/16 full-tensor launches plus ~40 tiny launches per schedule scalar; fp32 state (the
    reference promotes every update to fp32). Full workload shape, or the largest batch torch.quantile accepts
    (16 M elements) when thresholding is on. Falls back to the oracle port's torch namespace when oracle/_ref is
    missing. Returns (GElem/s, ms per sample(), kind)."""
    import refcheck as R
    from oracle import ref_loader
    shape = tuple(w["shape"])
    if w["thresholding"]:
        shape = (min(shape[0], (1 << 24) // int(np.prod(shape[1:])) - 1),) + shape[1:]
    if ref_loader.available():
        kind = "reference"
        x, banks = R.synthetic(w, shape[0], dev, torch.float32, nbanks=2)
        solver, _ = R._solver(ref_loader.load("dpm_solver_pytorch"), w, banks, dev)
        kw = R.sample_kwargs(w)
        once = lambda: solver.sample(x, **kw)
    else:
        kind = "port"
        if w["thresholding"]:
            return None   # the oracle's quantile is a numpy sort: not an eager-CUDA path
        from cases import make_betas
        from oracle import dpm_oracle as O
        TH = O.torch_namespace(dev)
        k2, betas = make_betas(w["schedule"])
        ns = O.VPSchedule.from_betas(betas, xp=TH) if k2 == "discrete" else O.VPSchedule("linear", xp=TH)
        g = torch.Generator(device=dev).manual_seed(1234)
        x = torch.randn(shape, device=dev, generator=g)
        nb = 2 if w["cfg"] else 1
        banks = [torch.randn((nb * shape[0],) + shape[1:], device=dev, generator=g) for _ in range(2)]
        cnt = [0]

        def net(xx, tt):
            cnt[0] += 1
            return banks[cnt[0] % 2]

        smp = O.Sampler(ns, net, algorithm_type=w["algo"], guidance_scale=w["cfg"], thresholding=None)
        smp.log_calls = False
        once = (lambda: smp.multistep(x, w["steps"], w["order"])) if w["method"] == "multistep" else \
            (lambda: smp.singlestep(x, w["steps"], w["order"]))
    with torch.no_grad():
        once()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(repeats):
            once()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / repeats
    return int(np.prod(shape)) * n_updates(w) / (ms * 1e-3) / 1e9, ms, kind


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_batch = cpu_sample_batch(w)
    val, dt, cores, kind = cpu_arm(w, sample_batch, repeats=max(1, args.steps), warmup=max(1, min(args.warmup, 3)))
    out = {
        "impl": "reference", "metric": "solver-update GElem/s", "value": val, "unit": "GElem/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "sample": f"batch {sample_batch} of the per-GPU batch, fp32 on CPU"},
        "cpu_baseline": {"value": val, "unit": "GElem/s", "cores": cores, "threads": cores, "host_cores": host_cores(),
                         "usable_cores": usable_cores(), "kind": kind,
                         "what": "unmodified dpm_solver_pytorch.py (oracle/_ref bytecode) on CPU tensors" if kind == "reference" else "oracle port, torch-CPU namespace",
                         "sample": f"[{sample_batch},{','.join(map(str, w['shape'][1:]))}] fp32, {w['steps']} solver steps per sample() call"},
        "e2e": {"value": val, "unit": "GElem/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def make_timed_backend():
    from dpm_solver_b200 import ops

    class TimedBackend(ops.CudaBackend):
        """CudaBackend that brackets every library launch with CUDA events on the launching stream."""

        def __init__(self):
            super().__init__()
            self.recording = False
            self.records = []  # (key, algorithmic bytes, start event, end event)

        @staticmethod
        def _bytes(a, m_out, out):
            n = a.reference_tensor().numel()
            tot = 0
            seen = set()
            for t in (a.x, a.xe, a.m0, a.m1, a.m2, a.e_cond, a.e_uncond):
                if t is not None and t.data_ptr() not in seen:
                    seen.add(t.data_ptr())
                    tot += n * t.element_size()
            for t in (m_out, out, a.out2):
                if t is not None:
                    tot += n * t.element_size()
            return tot

        def step(self, a):
            if not self.recording:
                return super().step(a)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m_out, out = super().step(a)
            e1.record()
            key = f"{FORM_NAMES[a.form]}|n_model={a.n_model}|m_out={int(m_out is not None)}"
            self.records.append((key, self._bytes(a, m_out, out), e0, e1))
            return m_out, out

        def prepare(self, a):
            """Frozen launches (ops.PreparedStep) bypass step(): wrap them so that they are timed too."""
            prep = super().prepare(a)
            if prep is None:
                return None
            n = a.reference_tensor().numel()
            es = a.reference_tensor().element_size() if a.state_dtype is None else torch.empty((), dtype=a.state_dtype).element_size()
            seen, tot = set(), 0
            for t in (a.x, a.xe, a.m0, a.m1, a.m2, a.e_cond, a.e_uncond):
                if t is not None and t.data_ptr() not in seen:
                    seen.add(t.data_ptr())
                    tot += n * t.element_size()
            tot += n * es * (int(prep.need_m) + int(prep.need_out) * (2 if prep.dup else 1))
            key = f"{FORM_NAMES[a.form]}|n_model={a.n_model}|m_out={int(prep.need_m)}"
            outer = self

            class TimedPrepared:
                d = prep.d

                def launch(self, tensors):   # tensors: tuple in PreparedStep.ORDER
                    if not outer.recording:
                        return prep.launch(tensors)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    r = prep.launch(tensors)
                    e1.record()
                    if r is not None:
                        outer.records.append((key, tot, e0, e1))
                    return r

            return TimedPrepared()

        def duplicate(self, x):
            if not self.recording:
                return super().duplicate(x)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = super().duplicate(x)
            e1.record()
            self.records.append(("cat([x]*2)", 3 * x.numel() * x.element_size(), e0, e1))
            return out

        def dynamic_threshold(self, a, q, max_val):
            if not self.recording:
                return super().dynamic_threshold(a, q, max_val)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            s = super().dynamic_threshold(a, q, max_val)
            e1.record()
            n = a.reference_tensor().numel()
            b = sum(n * t.element_size() for t in (a.xe if a.xe is not None else a.x, a.e_cond, a.e_uncond) if t is not None)
            self.records.append((f"quantile|n_model={a.n_model}", b, e0, e1))
            return s

        def summary(self):
            agg = {}
            for key, b, e0, e1 in self.records:
                d = agg.setdefault(key, {"launches": 0, "ms": 0.0, "bytes": 0})
                d["launches"] += 1
                d["ms"] += e0.elapsed_time(e1)
                d["bytes"] += b
            for d in agg.values():
                d["avg_us"] = d["ms"] * 1e3 / d["launches"]
                d["bytes_per_launch"] = d["bytes"] / d["launches"]
                d["gbs"] = d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else None
            return agg

    return TimedBackend()


def headline_kernels(be, peak, shape=(4096, 4, 64, 64), reps=50):
    """North-star kernel timed alone: fused 3rd-order multistep update, x + 3 buffers -> x_t."""
    from dpm_solver_b200.ops import StepArgs, FORM_MS3
    out = {}
    n = int(np.prod(shape))
    for name, dt in (("bf16", torch.bfloat16), ("f32", torch.float32)):
        sets = []
        for s in range(3):  # rotate through 3 buffer sets: each launch touches > L2 of fresh lines
            sets.append([torch.randn(n, device="cuda", dtype=dt) for _ in range(4)] + [torch.empty(n, device="cuda", dtype=dt)])
        def launch(i):
            x, m0, m1, m2, o = sets[i % 3]
            be.step(StepArgs(form=FORM_MS3, x=x, m0=m0, m1=m1, m2=m2, out=o, a=0.95, c0=-0.1, c1=0.05, c2=-0.01,
                             w0=1.02, w1=0.98, w2=0.51, w3=0.5))
        for i in range(10):
            launch(i)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for i, (a, b) in enumerate(ev):
            a.record(); launch(i); b.record()
        torch.cuda.synchronize()
        us = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
        med = us[len(us) // 2]
        byts = 5 * n * (2 if dt == torch.bfloat16 else 4)
        out[f"ms3_update_{name}_[4096,4,64,64]"] = {
            "bytes_per_launch": byts, "median_us": med, "min_us": us[0], "gbs": byts / (med * 1e-6) / 1e9,
            "frac_of_peak": byts / (med * 1e-6) / 1e9 / peak, "gelem_s": n / (med * 1e-6) / 1e9}
        del sets
        torch.cuda.empty_cache()
    return out


def bind_to_gpu_numa_node(local):
    """Pin this process (and with the default first-touch policy its pinned host buffers) to the CPUs NVML reports
    as local to GPU `local`, BEFORE anything is allocated: with 8 ranks each moving 2 x 134 MB per step through
    pinned memory, buffers on the wrong socket cross the inter-socket link twice. Returns a description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local]) if vis and vis.split(",")[local].strip().isdigit() else local
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, wd in enumerate(mask) for b in range(64) if (int(wd) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus:
            return {"bound": False, "why": "no overlap between the GPU's CPU affinity and this process's cpuset"}
        os.sched_setaffinity(0, cpus)
        node = None
        try:
            for n in sorted(os.listdir("/sys/devices/system/node")):
                if n.startswith("node") and n[4:].isdigit():
                    lst = open(f"/sys/devices/system/node/{n}/cpulist").read().strip()
                    ids = set()
                    for part in lst.split(","):
                        lo, _, hi = part.partition("-")
                        ids.update(range(int(lo), int(hi or lo) + 1))
                    if min(cpus) in ids:
                        node = int(n[4:])
        except Exception:
            pass
        return {"bound": True, "numa_node": node, "cpus": len(cpus)}
    except Exception as e:
        return {"bound": False, "why": repr(e)[:120]}


class Ctx:
    """Per-process state shared by the workloads of one bench run."""

    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback exists)")
        self.numa = bind_to_gpu_numa_node(self.local) if not args.no_numa else {"bound": False, "why": "--no-numa"}
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            # NCCL's own environment (NCCL_DEBUG, ...) is left exactly as the launcher set it
            dist.init_process_group("nccl", device_id=self.dev)
        from dpm_solver_b200 import ops
        self.be = make_timed_backend()
        ops.set_backend(self.be)
        self.be.set_tuning(args.variant, args.threads, args.ctas)

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return v
        t = torch.tensor([v], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def build_solver(ctx, w, B, seed, inputs=None, plan_broadcast=None):
    """Synthetic inputs (or the given (x_T, banks)) + the product solver for a B-sample batch of workload `w` on
    this rank's GPU."""
    from cases import make_betas
    from dpm_solver_b200 import DPM_Solver, NoiseScheduleVP, model_wrapper
    import refcheck as R
    dev, dt = ctx.dev, DT[w["dtype"]]
    kind, betas = make_betas(w["schedule"])
    ns = NoiseScheduleVP("discrete", betas=torch.from_numpy(betas)) if kind == "discrete" else NoiseScheduleVP("linear")
    x_T, banks = inputs if inputs is not None else R.synthetic(w, B, dev, dt, seed=seed)
    cnt = [0]
    if w["cfg"]:
        def net(xx, tt, cc):
            cnt[0] += 1
            return banks[cnt[0] % 3]
        fn = model_wrapper(net, ns, guidance_type="classifier-free", condition=torch.ones(B, 1, device=dev),
                           unconditional_condition=torch.zeros(B, 1, device=dev), guidance_scale=w["cfg"])
    else:
        def net(xx, tt):
            cnt[0] += 1
            return banks[cnt[0] % 3]
        fn = model_wrapper(net, ns)
    solver = DPM_Solver(fn, ns, algorithm_type=w["algo"], state_dtype=dt,
                        correcting_x0_fn="dynamic_thresholding" if w["thresholding"] else None,
                        plan_broadcast=(ctx.world > 1) if plan_broadcast is None else plan_broadcast)
    kw = dict(steps=w["steps"], order=w["order"], method=w["method"], skip_type="time_uniform")
    return solver, kw, x_T, banks, cnt


# measured storage-precision deviation of 16-bit state from the fp32 reference (tests/test_vs_reference_workloads.py)
PARITY_BOUND_16 = {("c2", "bf16"): (2.30e-2, 1.07e-2), ("c3", "bf16"): (9.84e-3, 4.07e-3), ("c4", "bf16"): (2.34e-2, 5.48e-3)}


def parity_check(name, w, solver, kw, x_T, banks, cnt):
    """Outside the timed region: the run's own configuration, one more sample() with the bank rotation reset, a batch
    slice of its output against the UNMODIFIED reference (oracle/_ref, CPU fp32) on the same rows of the inputs."""
    try:
        import refcheck as R
        from oracle import ref_loader
        if not ref_loader.available():
            return {"parity_checked": False, "why": "oracle/_ref not built"}
        B = x_T.shape[0]
        rows = 8 if w["shape"][-1] <= 64 else 2
        cnt[0] = 0
        y = solver.sample(x_T, **kw)
        torch.cuda.synchronize()
        xs = x_T[:rows].cpu()
        bs = [R.slice_rows(b, B, rows, w["cfg"]).cpu() for b in banks]
        yr = R.reference_sample(w, xs, bs, device="cpu")
        got = y[:rows].float().cpu()
        mx, rms = R.rel_err(got.numpy(), yr.numpy()), R.rms_rel_err(got.numpy(), yr.numpy())
        out = {"rows": rows, "max_rel_err": mx, "rms_rel_err": rms, "reference": "unmodified dpm_solver_pytorch.py (oracle/_ref), CPU fp32",
               "reference_absmean": float(yr.abs().mean()), "absmean": float(got.abs().mean())}
        if w["dtype"] == "f32":
            out["bit_exact"] = bool(torch.equal(got, yr))
            out["parity_checked"] = out["bit_exact"]
        else:
            bmx, brms = PARITY_BOUND_16.get((name, w["dtype"]), (5e-2, 2e-2))
            out["bound"] = {"max_rel_err": 1.5 * bmx, "rms_rel_err": 1.5 * brms, "what": "1.5 x the measured bf16-storage deviation"}
            out["parity_checked"] = bool(mx <= 1.5 * bmx and rms <= 1.5 * brms)
        return out
    except Exception as e:
        return {"parity_checked": False, "why": repr(e)[:200]}


def shard_parity(ctx, w):
    """T6 inside the bench: a small global batch (same seed on every rank), split over the ranks, must equal rank 0's
    single-GPU run of the whole batch bit for bit (concatenated shards == unsharded); shards meet by all_gather."""
    import refcheck as R
    dist = ctx.dist
    per = 16 if w["shape"][-1] <= 64 else 2
    Bg = per * ctx.world
    x_g, banks_g = R.synthetic(w, Bg, ctx.dev, DT[w["dtype"]], seed=4321)
    lo, hi = ctx.rank * per, (ctx.rank + 1) * per
    x_s = x_g[lo:hi].contiguous()
    banks_s = [(torch.cat([b[lo:hi], b[Bg + lo:Bg + hi]]) if w["cfg"] else b[lo:hi]).contiguous() for b in banks_g]
    solver_s, kw, _, _, _ = build_solver(ctx, w, per, 0, inputs=(x_s, banks_s))
    y_s = solver_s.sample(x_s, **kw).contiguous()
    gathered = [torch.empty_like(y_s) for _ in range(ctx.world)]
    dist.all_gather(gathered, y_s)
    ok = True
    if ctx.rank == 0:
        # rank 0 alone: no collective may be issued here (its own plan IS the one the shards were synced to)
        solver_g, _, _, _, _ = build_solver(ctx, w, Bg, 0, inputs=(x_g, banks_g), plan_broadcast=False)
        ok = bool(torch.equal(torch.cat(gathered), solver_g.sample(x_g, **kw)))
    flag = torch.tensor([1 if ok else 0], device=ctx.dev)
    dist.broadcast(flag, 0)
    return bool(flag.item())


DUMP_ROWS = 512             # c2 / c3: [512, 4, 64, 64] float32 = 32 MB
DUMP_MAX_ELEMS = 8 << 20    # c4: 42 rows of [3, 256, 256]


def dump_outputs(y, out_dir):
    """A fixed, seeded sample of rows of the output `y` (at most DUMP_MAX_ELEMS elements) -> out_dir/x_0.npy."""
    per = int(np.prod(y.shape[1:]))
    n = max(1, min(y.shape[0], DUMP_ROWS, DUMP_MAX_ELEMS // per))
    rows = torch.randperm(y.shape[0], generator=torch.Generator().manual_seed(0))[:n].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x_0.npy"), y[rows.to(y.device)].float().cpu().numpy())


def measure(ctx, args, name, w, steps, warmup, with_e2e=True, dump_dir=None):
    """Time one workload on this process's GPU; returns the dict of a bench line (rank 0) or None. With `dump_dir`,
    rank 0 writes a sample of the last timed step's output there (dump_outputs)."""
    be, dev, world, rank = ctx.be, ctx.dev, ctx.world, ctx.rank
    dt = DT[w["dtype"]]
    shape = tuple(w["shape"])
    B = shape[0]
    E = int(np.prod(shape))
    solver, kw, x_T, banks, cnt = build_solver(ctx, w, B, seed=1234 + rank)

    # ---- warm-up ----
    for _ in range(max(warmup, 3)):
        y = solver.sample(x_T, **kw)
    ctx.barrier()

    # ---- timed region: inputs resident in HBM. No per-launch events here: bracketing every launch with CUDA events
    # costs ~7 % of the loop (event records between kernels also keep consecutive launches from overlapping
    # programmatically), so the headline pass runs the public API exactly as a user would.
    launches0 = be.launch_count()
    be.recording, be.records = False, []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(ctx.local) as clk:
        ctx.barrier()
        e0.record()
        for _ in range(steps):
            y = solver.sample(x_T, **kw)
        e1.record()
        ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    gpu_launches = be.launch_count() - launches0
    if dump_dir is not None and rank == 0:
        dump_outputs(y, dump_dir)
    # ---- instrumented pass: the same K steps again with CUDA events around every library launch (per-kernel
    # durations for the roofline / kernels breakdown); its whole-pass time is reported as ms_per_step_instrumented
    be.recording, be.records = True, []
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    i0.record()
    for _ in range(steps):
        y = solver.sample(x_T, **kw)
    i1.record()
    ctx.barrier()
    be.recording = False
    ms_instr = ctx.max_over_ranks(i0.elapsed_time(i1))
    ksum = be.summary()
    if os.environ.get("DPM_BENCH_TRACE") and rank == 0:
        recs = be.records
        for key, b, a0, a1 in recs[:2 * w["steps"] + 2]:
            print(f"trace {key:40s} {a0.elapsed_time(a1) * 1e3:8.1f} us", file=sys.stderr)
        for i in range(min(len(recs) - 1, 2 * w["steps"])):
            print(f"gap {i}: {recs[i][3].elapsed_time(recs[i + 1][2]) * 1e3:7.1f} us", file=sys.stderr)
    value = world * E * n_updates(w) * steps / (ms * 1e-3) / 1e9

    e2e = None
    if with_e2e:
        # ---- e2e: host buffers; every step copies its x_T host->device (pinned) and its result device->host inside
        # the timed region. Software-pipelined over three streams (copy-in, compute, copy-out) with double buffers,
        # the way a serving loop would feed the public API.
        n_buf = 2
        x_host = [x_T.cpu().pin_memory() for _ in range(n_buf)]
        y_host = [torch.empty_like(x_host[0]).pin_memory() for _ in range(n_buf)]
        x_dev = [torch.empty_like(x_T) for _ in range(n_buf)]
        s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()

        def e2e_loop(n_steps):
            ev_in = [None] * n_buf      # copy-in of buffer b finished
            ev_cmp = [None] * n_buf     # compute that read x_dev[b] finished
            ev_out = [None] * n_buf     # copy-out into y_host[b] finished
            ys = [None] * n_buf
            for i in range(n_steps):
                b = i % n_buf
                with torch.cuda.stream(s_in):
                    if ev_cmp[b] is not None:
                        s_in.wait_event(ev_cmp[b])               # x_dev[b] no longer read
                    x_dev[b].copy_(x_host[b], non_blocking=True)
                    ev_in[b] = torch.cuda.Event(); ev_in[b].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[b])
                    if ev_out[b] is not None:
                        s_cmp.wait_event(ev_out[b])              # previous result of this slot has left
                    ys[b] = solver.sample(x_dev[b], **kw)
                    ev_cmp[b] = torch.cuda.Event(); ev_cmp[b].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    y_host[b].copy_(ys[b], non_blocking=True)
                    ev_out[b] = torch.cuda.Event(); ev_out[b].record(s_out)
            for st in (s_in, s_cmp, s_out):
                torch.cuda.current_stream().wait_stream(st)

        e2e_loop(2)
        ctx.barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(ctx.local) as clk2:
            e2.record()
            e2e_loop(steps)
            e3.record()
            ctx.barrier()
        clk.rows += clk2.rows
        ms_e2e_rank = e2.elapsed_time(e3)
        ms_e2e = ctx.max_over_ranks(ms_e2e_rank)
        h2d = x_host[0].numel() * x_host[0].element_size()
        d2h = y_host[0].numel() * y_host[0].element_size()
        checksum = float(y_host[(steps - 1) % n_buf].float().abs().mean())
        e2e = {"value": world * E * n_updates(w) * steps / (ms_e2e * 1e-3) / 1e9, "unit": "GElem/s",
               "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world, "ms_per_step": ms_e2e / steps,
               # what bounds it: each rank moves h2d + d2h bytes per step over its PCIe link, concurrently in both directions
               "pcie_gbs_per_rank_each_direction": h2d / (ms_e2e / steps * 1e-3) / 1e9,
               "limiter": "PCIe: one x_T in and one x_0 out per sample() per rank, full duplex; the device-side step takes %.2f ms" % (ms / steps),
               "numa": ctx.numa, "checksum_absmean": checksum}
        del x_host, y_host, x_dev

    par = parity_check(name, w, solver, kw, x_T, banks, cnt) if rank == 0 else None
    if rank != 0:
        return None
    peak, peak_src = hbm_peak()
    dom_key = max(ksum, key=lambda k: ksum[k]["ms"])
    dom = ksum[dom_key]
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get(name, {}).get(dom_key)
            traffic_src = tj.get("_source", "profiles/roofline_traffic.json") + " (static: one ncu --set full capture of this kernel, not measured by this run)"
        except Exception:
            traffic = None
    out = {
        "metric": "solver-update GElem/s", "value": value, "unit": "GElem/s", "n_gpus": world, "steps": steps,
        "warmup": max(warmup, 3), "ms_per_step": ms / steps, "ms_per_step_instrumented": ms_instr / steps,
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
        "config": {"workload": w["desc"], "per_gpu_shape": list(shape), "global_batch": B * world,
                   "parallelism": f"batch-sharded x{world}, one broadcast of the scalar plan, no tensor traffic",
                   "l2": "per-update working set (x, eps bank, buffers: >= 4 x %.0f MB) exceeds the 126 MB L2; eps banks rotate" % (E * x_T.element_size() / 1e6),
                   "variant": args.variant, "parity_checked": bool(par and par.get("parity_checked"))},
        "parity": par,
        # all launches: algorithmic bytes of the K steps / the headline pass's time (gaps included)
        "hbm_gbs_total": sum(d["bytes"] for d in ksum.values()) / (ms * 1e-3) / 1e9,
        "hbm_gbs_kernels": sum(d["bytes"] for d in ksum.values()) / (sum(d["ms"] for d in ksum.values()) * 1e-3) / 1e9,
        "roofline": {"bound": "hbm", "kernel": dom_key, "achieved": dom["gbs"], "peak": peak, "unit": "GB/s",
                     "frac": dom["gbs"] / peak, "peak_source": peak_src, "bytes_per_launch": dom["bytes_per_launch"],
                     "avg_us": dom["avg_us"], "launches": dom["launches"], "traffic": traffic, "traffic_source": traffic_src,
                     "timing": "CUDA events around every launch of this kernel in the instrumented pass (the same K steps, right after the headline pass)"},
        "kernels": ksum,
        "gpu_launches": gpu_launches,
        "clocks": clk.summary(),
    }
    if e2e is not None:
        out["e2e"] = e2e
    del y, banks, x_T, solver
    torch.cuda.empty_cache()
    return out


def run_b200(args, w):
    ctx = Ctx(args)
    out = measure(ctx, args, args.workload, w, args.steps, args.warmup, dump_dir=args.dump_outputs)
    if ctx.world > 1:
        ok = shard_parity(ctx, w)
        if ctx.rank == 0:
            out["config"]["shard_parity"] = ok
    if ctx.rank == 0:
        if not args.no_extras:
            # the other single-GPU BASELINE configs, driver-visible in the same line (value, roofline, clocks each)
            others = {}
            for name in ("c3", "c4"):
                if name == args.workload or ctx.world > 1:
                    continue
                try:
                    o = measure(ctx, args, name, WORKLOADS[name], max(2, min(args.steps, 5)), 3, with_e2e=False)
                    others[name] = {k: o[k] for k in ("value", "unit", "ms_per_step", "ms_per_step_instrumented", "steps", "dtype", "config", "parity", "roofline",
                                                        "hbm_gbs_total", "kernels", "gpu_launches", "clocks")}
                except Exception as e:   # never let an extra leg break the headline
                    others[name] = {"error": repr(e)[:200]}
            if others:
                out["workloads"] = others
        if ctx.world == 1 and not args.no_extras:
            peak, _ = hbm_peak()
            out["kernels_alone"] = headline_kernels(ctx.be, peak)
            sample_batch = cpu_sample_batch(w)
            val, dtc, threads, kind = cpu_arm(w, sample_batch, repeats=1, warmup=0)
            out["cpu_baseline"] = {"value": val, "unit": "GElem/s", "cores": threads, "threads": threads, "host_cores": host_cores(),
                                   "usable_cores": usable_cores(), "kind": kind,
                                   "sample": f"[{sample_batch},{','.join(map(str, w['shape'][1:]))}] fp32, {w['steps']} solver steps, {dtc * 1e3:.0f} ms"}
            try:
                eg = eager_cuda_arm(w, ctx.dev)
                if eg is not None:
                    out["eager_cuda_baseline"] = {"value": eg[0], "unit": "GElem/s", "ms_per_step": eg[1], "dtype": "f32", "kind": eg[2],
                                                  "what": "the reference algorithm as stock eager PyTorch CUDA kernels on the same GPU, full workload shape"}
            except Exception as e:   # never let the extra leg break the bench line
                out["eager_cuda_baseline"] = {"error": repr(e)[:200]}
        print(json.dumps(out), flush=True)
    if ctx.world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", type=int, default=2, help="0 direct, 1 TMA ring, 2 auto")
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--ctas", type=int, default=0)
    ap.add_argument("--no-extras", action="store_true", help="skip the c3/c4, kernel-alone and CPU-baseline legs")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the process to the GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's output to DIR/x_0.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_b200(args, w)


if __name__ == "__main__":
    main()
