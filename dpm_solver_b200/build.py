"""Build libdpmsolver_b200.so in-tree with nvcc for sm_100a.

    python -m dpm_solver_b200.build [--force] [--verbose]

The library has no PyTorch / Python dependency: plain CUDA runtime (static cudart) behind the C-ABI
of include/dpm_solver_b200.h. -fmad=false is REQUIRED: the kernels restate the reference's
unfused chains of fp32 elementwise ops and must not contract a*b+c into an FMA.
"""
from __future__ import annotations

import argparse
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
INCLUDE = ROOT / "include"
OUT_DIR = PKG / "lib"
BUILD_DIR = PKG / "build"
LIB_NAME = "libdpmsolver_b200.so"

SOURCES = ["capi.cu", "step_direct.cu", "step_tma.cu", "quantile.cu", "adaptive.cu", "adaptive_ctl.cu", "philox.cu",
           "step_sde.cu"]
# philox.cu and step_sde.cu embed curand's Box-Muller, which must round exactly like the copy inside torch's randn
# kernel: they are compiled with nvcc's default fma contraction and spell the unfused chains with __fmul_rn/__fadd_rn
FMAD_DEFAULT = {"philox.cu", "step_sde.cu"}
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stamp(extra: list[str]) -> str:
    h = hashlib.sha256()
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(INCLUDE.glob("*.h"))):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    h.update(" ".join(ARCH + NVCC_FLAGS + extra).encode())
    return h.hexdigest()


def lib_path() -> Path:
    return OUT_DIR / LIB_NAME


def build(force: bool = False, verbose: bool = False, extra_flags: list[str] | None = None,
          out_name: str = LIB_NAME) -> Path:
    extra = list(extra_flags or [])
    out = OUT_DIR / out_name
    stamp_file = BUILD_DIR / (out_name + ".stamp")
    stamp = _stamp(extra)
    if not force and out.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return out
    nvcc = _nvcc()
    OUT_DIR.mkdir(exist_ok=True)
    objdir = BUILD_DIR / out_name.replace(".so", "")
    objdir.mkdir(parents=True, exist_ok=True)

    def compile_one(src: str) -> Path:
        obj = objdir / (src.replace(".cu", ".o"))
        flags = [f for f in NVCC_FLAGS if not (src in FMAD_DEFAULT and f == "-fmad=false")]
        cmd = [nvcc, *ARCH, *flags, *extra, "-I", str(INCLUDE), "-I", str(CSRC), "-c",
               str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose and r.stderr:
            print(r.stderr, flush=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    link = [nvcc, *ARCH, "-shared", "-o", str(out), *map(str, objs)]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp_file.write_text(stamp)
    return out


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    p = build(force=a.force, verbose=a.verbose)
    print(p)
    return 0


if __name__ == "__main__":
    sys.exit(main())
