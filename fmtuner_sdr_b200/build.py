"""Build the engine's shared library in-tree with nvcc (sm_100a only)."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libfmgpu.so")
DROPIN_LIB = os.path.join(HERE, "libfmgpu_dropin.so")
SOURCES = ["kernels.cu", "engine.cu", "decim_tc.cu", "fir_tc.cu", "channelizer.cu", "synth.cu", "probe.cu", "design.cpp",
           "xdr_format.cpp"]
HEADERS = ["engine.h", "kernels.h", "tc_common.cuh", "device_once.h", "cuda_handle.h", "design.h", "fm_math.h", os.path.join("..", "..", "include", "fmgpu.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # only explicit fmaf() may fuse: the CPU oracle evaluates the same operation order
    "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared",
]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def build_lib(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in HEADERS]
    if force or _stale(LIB, deps):
        cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + srcs
        subprocess.run(cmd, check=True, cwd=CSRC)
    return LIB


def build_variant(name: str, defines: list[str]) -> str:
    """Build build/libfmgpu_<name>.so with extra -D macros (measurement variants; load it through
    the FMGPU_LIB environment variable)."""
    out_dir = os.path.join(HERE, "..", "build")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.abspath(os.path.join(out_dir, f"libfmgpu_{name}.so"))
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    cmd = [nvcc_path()] + NVCC_FLAGS + [f"-D{d}" for d in defines] + ["-o", out] + srcs
    subprocess.run(cmd, check=True, cwd=CSRC)
    return out


def build_dropin(force: bool = False) -> str:
    """C++ wrapper classes with the reference's names/signatures over the C ABI."""
    src = os.path.join(HERE, "dropin", "dropin.cpp")
    if not os.path.exists(src):
        return ""
    deps = [src] + [os.path.join(HERE, "dropin", f) for f in os.listdir(os.path.join(HERE, "dropin"))
                    if f.endswith(".h")]
    if force or _stale(DROPIN_LIB, deps + [LIB]):
        cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I", os.path.join(HERE, "dropin"),
               "-I", os.path.join(HERE, "..", "include"), "-o", DROPIN_LIB, src,
               "-L", HERE, "-lfmgpu", "-Wl,-rpath,$ORIGIN"]
        subprocess.run(cmd, check=True)
    return DROPIN_LIB


if __name__ == "__main__":
    print(build_lib(force=True, verbose=True))
    print(build_dropin(force=True))
