"""Builds libpbn_b200.so (sm_100a) in-tree with nvcc.  `python gym-pbn-stac_b200/build.py [--force]`."""
import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
SRC = [HERE / "csrc" / "pbn_b200.cu", HERE / "csrc" / "pbn_fit.cu"]
DEPS = SRC + [HERE / "csrc" / "pbn_device.cuh", HERE / "csrc" / "pbn_fit.cuh", HERE / "csrc" / "pbn_coop.cuh", HERE / "csrc" / "pbn_smem.cuh", ROOT / "include" / "pbn_b200.h"]
LIB = HERE / "lib" / "libpbn_b200.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",  # the geometric-gap polynomial must round exactly like the CPU oracle; integer code is unaffected
    "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v",
]


def nvcc():
    """nvcc on PATH, else in the CUDA toolkit named by CUDA_HOME (default /usr/local/cuda), as torch's extension builder
    looks for it: a non-login shell often has the toolkit installed but not on PATH."""
    found = shutil.which("nvcc")
    if found:
        return found
    cand = Path(os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda") / "bin" / "nvcc"
    if not cand.exists():
        raise RuntimeError("nvcc not found: put the CUDA toolkit's bin directory on PATH or set CUDA_HOME")
    return str(cand)


def build(force=False, verbose=False, extra=(), out=None):
    """extra/out: experiment builds (e.g. extra=["-DPBN_SSD_MIN_BLOCKS=6"], out=lib/variant.so)."""
    target = Path(out) if out else LIB
    if not force and target.exists() and all(target.stat().st_mtime >= d.stat().st_mtime for d in DEPS):
        return target
    LIB.parent.mkdir(exist_ok=True)
    cmd = [nvcc(), *NVCC_FLAGS, *extra, f"-I{ROOT / 'include'}", f"-I{HERE / 'csrc'}", "-o", str(target), *map(str, SRC)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    (HERE / "lib" / "ptxas.log").write_text(res.stderr)
    if res.returncode != 0:
        sys.stderr.write(res.stderr)
        raise RuntimeError("nvcc failed building libpbn_b200.so")
    if verbose:
        print(res.stderr)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
