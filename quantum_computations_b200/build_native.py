"""Compile the native libraries in-tree.

``build_cuda()``  -> quantum_computations_b200/csrc/libqsim_b200.so   (nvcc, sm_100a)
``build_emu()``   -> tests/_build/libqsim_emu.so   (g++; host emulator, tests only)
``build_cuda(dev_knobs=True)`` -> tests/_build/libqsim_b200_knobs.so   (the same library with
                   the development A/B switches read from the environment, tests only)

nvcc cross-compiles without a GPU, so both run in the CPU-only build container;
the built ``.so`` files are git-ignored but travel to the GPU box with the tree.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
CUDA_LIB = os.path.join(CSRC, "libqsim_b200.so")
EMU_DIR = os.path.join(ROOT, "tests", "_build")
EMU_LIB = os.path.join(EMU_DIR, "libqsim_emu.so")
CUDA_KNOBS_LIB = os.path.join(EMU_DIR, "libqsim_b200_knobs.so")

_HEADERS = ["plan.h", "planner.h", "tile_exec.h", "elem_ops.h", "backend.h"]
_HOST_SRCS = ["planner.cpp", "capi_host.cpp", "pauli.cpp"]


def _newer_than(target: str, sources) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _run(cmd):
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError("native build failed: " + " ".join(cmd))
    return proc.stdout + proc.stderr


def build_cuda(force: bool = False, verbose: bool = False, dev_knobs: bool = False) -> str:
    """``dev_knobs``: build CUDA_KNOBS_LIB, whose launch variants the tests select per process."""
    target = CUDA_KNOBS_LIB if dev_knobs else CUDA_LIB
    srcs = [os.path.join(CSRC, s) for s in _HOST_SRCS + ["kernels.cu"]]
    deps = srcs + [os.path.join(CSRC, h) for h in _HEADERS] + [os.path.join(ROOT, "include", "qsim_b200.h")]
    if not force and _newer_than(target, deps):
        return target
    os.makedirs(os.path.dirname(target), exist_ok=True)
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, "-O3", "-std=c++17", "-lineinfo",
           "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
           "-o", target] + srcs
    if dev_knobs or os.environ.get("QSIM_DEV_KNOBS"):          # development build: A/B switches read the environment
        cmd.insert(1, "-DQSIM_DEV_KNOBS")
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    out = _run(cmd)
    if verbose:
        print(out)
    return target


def build_emu(force: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in _HOST_SRCS + ["emu.cpp"]]
    deps = srcs + [os.path.join(CSRC, h) for h in _HEADERS] + [os.path.join(ROOT, "include", "qsim_b200.h")]
    if not force and _newer_than(EMU_LIB, deps):
        return EMU_LIB
    os.makedirs(EMU_DIR, exist_ok=True)
    cxx = shutil.which("g++") or "g++"
    _run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-o", EMU_LIB] + srcs)
    return EMU_LIB


if __name__ == "__main__":
    print(build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_emu(force="--force" in sys.argv))
