"""Build recipes for the native libraries (in-tree, so the .so files travel with a snapshot).

    lib/libsxgpu.so    CUDA kernels + the C ABI of include/sxgpu.h   (nvcc, sm_100a only)
    lib/libsxsoapy.so  host C++: the driver=sx SoapySDR device, SoapySDR/ALSA stand-ins and
                       the sxh_* harness, linked against libsxgpu.so  (g++)

Nothing here touches oracle/: the product never links the CPU oracle.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "lib"

GPU_LIB = LIB / "libsxgpu.so"
SOAPY_LIB = LIB / "libsxsoapy.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # -ffp-contract=off: the host side of sx_time.h must round exactly like the device side's
    # explicit _rn intrinsics on any host (GCC contracts by default on aarch64)
    "-Xcompiler", "-fPIC,-Wall,-ffp-contract=off",
    "-shared",
]

GPU_SOURCES = [CSRC / "sxgpu.cu"]
GPU_DEPS = GPU_SOURCES + [CSRC / "sx_kernels.cuh", CSRC / "sx_bank.cuh", CSRC / "sx_iir.cuh", CSRC / "sx_fir.cuh", CSRC / "sx_nco.cuh", CSRC / "sx_chan.cuh", CSRC / "sx_resident.cuh", CSRC / "sx_synth.h", CSRC / "sx_time.h",
                          CSRC / "host" / "stream_plan.hpp", CSRC / "host" / "par_copy.hpp", ROOT / "include" / "sxgpu.h"]

SOAPY_SOURCES = [
    CSRC / "host" / "SoapySXB200.cpp",
    CSRC / "host" / "SoapySXB200Group.cpp",
    CSRC / "host" / "harness_capi.cpp",
    CSRC / "shim" / "soapy_shim.cpp",
    CSRC / "shim" / "alsa_stub.cpp",
]


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).exists() and Path(d).stat().st_mtime > t for d in deps)


def _find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        raise RuntimeError("nvcc not found: libsxgpu.so cannot be built and there is no CPU fallback")
    return nvcc


def _run(cmd) -> None:
    proc = subprocess.run([str(c) for c in cmd], capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("build failed: %s\n%s\n%s" % (" ".join(map(str, cmd)), proc.stdout, proc.stderr))


def build_gpu_library(force: bool = False) -> Path:
    LIB.mkdir(exist_ok=True)
    if force or _stale(GPU_LIB, GPU_DEPS):
        _run([_find_nvcc(), *NVCC_FLAGS, "-o", GPU_LIB, *GPU_SOURCES])
    return GPU_LIB


def build_soapy_module(force: bool = False) -> Path:
    build_gpu_library()
    deps = SOAPY_SOURCES + list((CSRC / "shim").rglob("*.h*")) + list((CSRC / "host").glob("*.hpp")) + [GPU_LIB]
    if force or _stale(SOAPY_LIB, deps):
        _run([
            os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-ffp-contract=off", "-Wall", "-Wextra", "-fPIC", "-shared",
            "-Wl,-Bsymbolic", "-pthread",
            "-I", CSRC / "shim", "-I", ROOT / "include", "-I", CSRC,
            "-o", SOAPY_LIB, *SOAPY_SOURCES,
            "-L", LIB, "-lsxgpu", "-Wl,-rpath,$ORIGIN",
        ])
    return SOAPY_LIB


EXAMPLE_BIN = LIB / "sx_repeater"
HOOK_EXAMPLE_LIB = LIB / "libsxhook_example.so"


def build_examples(force: bool = False) -> Path:
    """examples/repeater.cpp: a C++ application on the SoapySDR API, linked against the module."""
    build_soapy_module()
    src = ROOT / "examples" / "repeater.cpp"
    if force or _stale(EXAMPLE_BIN, [src, SOAPY_LIB]):
        _run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", "-Wextra",
              "-I", CSRC / "shim", "-o", EXAMPLE_BIN, src,
              "-L", LIB, "-lsxsoapy", "-lsxgpu", "-pthread", "-Wl,-rpath,$ORIGIN"])
    return EXAMPLE_BIN


def build_hook_example(force: bool = False) -> Path:
    """examples/repeater_hook.cu: user DSP compiled into the fused bank iteration (include/sx_hook.cuh)."""
    build_gpu_library()
    src = ROOT / "examples" / "repeater_hook.cu"
    deps = [src, ROOT / "include" / "sx_hook.cuh", CSRC / "sx_bank.cuh", CSRC / "sx_iir.cuh", CSRC / "sx_fir.cuh", CSRC / "sx_nco.cuh", CSRC / "sx_kernels.cuh", GPU_LIB]
    if force or _stale(HOOK_EXAMPLE_LIB, deps):
        _run([_find_nvcc(), *NVCC_FLAGS, "-o", HOOK_EXAMPLE_LIB, src, "-L", LIB, "-lsxgpu",
              "-Xlinker", "-rpath,$ORIGIN"])
    return HOOK_EXAMPLE_LIB


def build_all(force: bool = False) -> None:
    # `force` rebuilds each target once, in link order; the dependencies of each build_* call are
    # only brought up to date.  Forcing them again would relink libsxgpu.so after the libraries
    # linked against it, leaving those older than their dependency, so that the next load finds
    # them stale and relinks them in the tree.
    build_gpu_library(force)
    build_soapy_module(force)
    build_examples(force)
    build_hook_example(force)
