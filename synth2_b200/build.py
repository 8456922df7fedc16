"""Builds libs2cuda.so (sm_100a) in-tree with nvcc.  `python -m synth2_b200.build [--force] [-v]`.

The library is plain CUDA C++ behind a C ABI (include/s2_cuda.h); it does not link torch.
nvcc cross-compiles without a GPU, so this runs in the CPU-only build container.
"""
import os
import pathlib
import shutil
import subprocess
import sys

PKG = pathlib.Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libs2cuda.so"
SOURCES = [CSRC / "s2_kernels.cu", CSRC / "s2_kernel_ts.cu", CSRC / "s2_capi.cu",
           CSRC / "s2_patch.cpp", CSRC / "s2_player.cpp", CSRC / "s2_nccl.cpp"]
DEPS = SOURCES + [CSRC / "s2_internal.h", CSRC / "s2_render_body.inc", CSRC / "s2_device.cuh", CSRC / "s2_math.h", CSRC / "s2_cutoff.h",
                  CSRC / "sin_table_bits.inc",
                  PKG.parent / "include" / "s2_cuda.h"]

# -fmad=false / -prec-div / -prec-sqrt / -ftz=false: the render arithmetic is specified as
# individually rounded binary32 operations (SURVEY.md section 8a); fused ops are spelled __fmaf_rn.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared", "-ldl",
]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def stale():
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any(d.stat().st_mtime > t for d in DEPS)


def build_lib(force=False, verbose=False):
    if not force and not stale():
        return LIB
    extra = os.environ.get("S2_NVCC_EXTRA", "").split()          # experiments, e.g. -DS2_TRIP=16
    out = os.environ.get("S2_LIB_OUT", str(LIB))                 # experiments: a variant next to the shipped library
    cmd = [find_nvcc(), *NVCC_FLAGS, *extra, "-o", out, *map(str, SOURCES)]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libs2cuda.so")
    return LIB


if __name__ == "__main__":
    build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
