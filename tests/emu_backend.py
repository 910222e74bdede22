"""Host-emulator backend for the CPU test-suite (TEST INFRASTRUCTURE ONLY).

Duck-types ``engine.CudaBackend`` on top of NumPy arrays and
``tests/_build/libqsim_emu.so`` (built from the product's own planner and
per-thread phase functions, see csrc/emu.cpp).  Lets the not-gpu tests drive the
package's Python layer, the planner and the tile index arithmetic without a
GPU.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from quantum_computations_b200 import _capi  # noqa: E402
from quantum_computations_b200.build_native import build_emu  # noqa: E402


class EmuBackend:
    name = "emu"

    def __init__(self):
        self.lib = C.CDLL(build_emu())
        _capi.declare(self.lib)
        assert self.lib.qsim_has_cuda() == 0

    def empty(self, count):
        return np.empty(int(count), dtype=np.complex128)

    def ptr(self, buf):
        return buf.ctypes.data

    def stream(self):
        return None

    def upload(self, host):
        return np.array(host, copy=True)

    def download(self, buf, out=None):
        if out is None:
            return np.array(buf, copy=True)
        out.reshape(-1)[:] = buf.reshape(-1)
        return out

    def clone(self, buf):
        return np.array(buf, copy=True)

    def divide_(self, buf, value):
        buf /= value

    def zeros(self, count, dtype=np.float64):
        return np.zeros(int(count), dtype=dtype)

    def synchronize(self):
        pass

    def pinned_empty(self, count):
        return np.empty(int(count), dtype=np.complex128)


_EMU = None


def emu() -> EmuBackend:
    global _EMU
    if _EMU is None:
        _EMU = EmuBackend()
    return _EMU
