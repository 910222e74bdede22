"""Device engine: binds ``csrc/libqsim_b200.so`` and keeps states on the GPU.

This is the only execution path of the package.  There is no CPU fallback: if
the CUDA library has not been built, or no CUDA device is visible, every entry
point raises.  PyTorch is used for what it is good at here -- device memory,
streams, pinned host buffers -- and nothing else; all arithmetic happens in the
hand-written kernels behind the C ABI (``include/qsim_b200.h``).

A state is a ``DeviceState``: a 1-D ``torch.complex128`` CUDA tensor of 2^m
amplitudes plus its interpretation (ket of m qubits, or the row-major vec of a
density matrix of m/2 qubits).  Reference qubit q is index bit m-1-q
(DV/numpy_quantum.py:243-247).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import _capi

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libqsim_b200.so")
if os.environ.get("QSIM_LIB"):          # development: try an experimental build of the same library
    _LIB_PATH = os.environ["QSIM_LIB"]

# Planner knobs (0 = library default); bench.py sweeps these.
PLAN_OPTIONS = {"tile_bits": 0, "low_bits": 0, "max_group": 0, "max_dense_ops": 0, "lookahead": 0,
                "merge_1q": 0, "defer_tail": 0, "max_layers": 0, "cta_log2": 0, "reserved0": 0,
                "apply_tail_mask": 0}


def _as_c128(arr) -> np.ndarray:
    return np.ascontiguousarray(arr, dtype=np.complex128)


def _dptr(arr: np.ndarray):
    return arr.ctypes.data_as(_capi.c_double_p)


class CudaBackend:
    """libqsim_b200.so + torch CUDA tensors on one device."""

    name = "cuda"

    def __init__(self, device: int | None = None):
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError(
                f"{_LIB_PATH} is missing: build it with `python -m quantum_computations_b200.build_native` "
                "(or __graft_entry__.build()).  This package has no CPU fallback.")
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device is visible; quantum_computations_b200 has no CPU fallback")
        self.torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.lib = C.CDLL(_LIB_PATH)
        _capi.declare(self.lib)
        if self.lib.qsim_has_cuda() != 1:
            raise RuntimeError("libqsim_b200.so was built without CUDA kernels")
        self._side_streams = []

    def pipeline(self, nstages: int) -> "_StreamPipeline":
        return _StreamPipeline(self, nstages)

    # -- memory ------------------------------------------------------------------
    def empty(self, count: int):
        return self.torch.empty(int(count), dtype=self.torch.complex128, device=self.device)

    def ptr(self, buf) -> int:
        return buf.data_ptr()

    def stream(self) -> int:
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def upload(self, host: np.ndarray):
        """Host array (any dtype) -> device tensor of the same dtype/shape."""
        t = self.torch.from_numpy(np.ascontiguousarray(host))
        return t.to(self.device, non_blocking=False)

    def download(self, buf, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            return buf.cpu().numpy()
        dst = self.torch.from_numpy(out.reshape(-1))
        dst.copy_(buf.reshape(-1))          # synchronous D2H; pinned `out` runs at link speed
        return out

    def download_async(self, buf, out: np.ndarray):
        """Start a device-to-host copy into the (pinned) array ``out`` on a side stream, ordered
        after the work queued so far on the current stream; returns a handle whose ``wait()``
        blocks until the data has landed.  The compute stream is free at once, so the next
        circuit can run while this one's result crosses PCIe."""
        torch = self.torch
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=self.device)
        done = torch.cuda.Event()
        done.record()
        dst = torch.from_numpy(out.reshape(-1))
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(done)
            dst.copy_(buf.reshape(-1), non_blocking=True)
            landed = torch.cuda.Event()
            landed.record()
        return _PendingCopy(buf, dst, landed)

    def clone(self, buf):
        return buf.clone()

    def divide_(self, buf, value: float) -> None:
        buf.div_(value)

    def zeros(self, count: int, dtype=np.float64):
        tdt = {np.float64: self.torch.float64, np.uint8: self.torch.uint8, np.int64: self.torch.int64}[dtype]
        return self.torch.zeros(int(count), dtype=tdt, device=self.device)

    def synchronize(self):
        self.torch.cuda.synchronize(self.device)

    def pinned_empty(self, count: int) -> np.ndarray:
        """Pinned host buffer viewed as a complex128 ndarray (for `out=`)."""
        t = self.torch.empty(int(count), dtype=self.torch.complex128, pin_memory=True)
        return t.numpy()


class _PendingCopy:
    """Handle of ``CudaBackend.download_async``: keeps the device buffer alive until the copy
    has finished."""

    def __init__(self, buf, dst, event):
        self._buf, self._dst, self._event = buf, dst, event

    def done(self) -> bool:
        return self._event is None or self._event.query()

    def wait(self) -> None:
        if self._event is not None:
            self._event.synchronize()
            self._event = self._buf = self._dst = None


class _StreamPipeline:
    """A few side streams with event dependencies between them (used by the sharded
    swap to overlap gather, exchange and scatter)."""

    def __init__(self, backend: "CudaBackend", nstages: int):
        torch = backend.torch
        self.torch = torch
        self.device = backend.device
        if len(backend._side_streams) < nstages:
            backend._side_streams += [torch.cuda.Stream(self.device)
                                      for _ in range(nstages - len(backend._side_streams))]
        self.streams = backend._side_streams[:nstages]
        self.main = torch.cuda.current_stream(self.device)
        start = torch.cuda.Event()
        start.record(self.main)
        for st in self.streams:
            st.wait_event(start)

    def stage(self, i: int):
        return self.torch.cuda.stream(self.streams[i])

    def record(self):
        ev = self.torch.cuda.Event()
        ev.record(self.torch.cuda.current_stream(self.device))
        return ev

    def wait(self, ev) -> None:
        self.torch.cuda.current_stream(self.device).wait_event(ev)

    def join(self) -> None:
        for st in self.streams:
            ev = self.torch.cuda.Event()
            ev.record(st)
            self.main.wait_event(ev)


_backend_lock = threading.Lock()
_backends: dict = {}


def get_backend(device: int | None = None) -> CudaBackend:
    """The CUDA backend for ``device`` (default: torch's current device)."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device is visible; quantum_computations_b200 has no CPU fallback")
    key = torch.cuda.current_device() if device is None else int(device)
    with _backend_lock:
        if key not in _backends:
            _backends[key] = CudaBackend(key)
        return _backends[key]


def launch_count(backend=None) -> int:
    backend = backend or get_backend()
    return int(backend.lib.qsim_launch_count())


# ---- fused plans ---------------------------------------------------------------------
class Plan:
    """A compiled sequence of tile passes for a fixed list of matrix gates."""

    def __init__(self, backend, n_bits: int, ops, options: dict | None = None):
        self.backend = backend
        self.n_bits = int(n_bits)
        lib = backend.lib
        circ = C.c_void_p()
        _capi.check(lib, lib.qsim_circuit_create(self.n_bits, C.byref(circ)))
        try:
            # one call for the whole gate list (a ctypes call per gate costs more than planning)
            ks = np.fromiter((len(t) for t, _m in ops), dtype=np.int32, count=len(ops))
            mats = []
            for (targets, matrix), k in zip(ops, ks):
                m = _as_c128(matrix)
                if m.shape != (1 << k, 1 << k):
                    raise ValueError("Dimensions of given matrix is not compatible with number of indices.")
                mats.append(m.reshape(-1))
            flat_t = np.fromiter((int(q) for t, _m in ops for q in t), dtype=np.int32, count=int(ks.sum()))
            flat_m = np.concatenate(mats) if mats else np.zeros(0, dtype=np.complex128)
            _capi.check(lib, lib.qsim_circuit_add_many(
                circ, len(ops), ks.ctypes.data_as(_capi.c_int_p), flat_t.ctypes.data_as(_capi.c_int_p),
                _dptr(flat_m.view(np.float64))))
            merged = dict(PLAN_OPTIONS)
            if options:
                merged.update(options)
            opt = _capi.PlanOptions(**{k: int(v) for k, v in merged.items()})
            plan = C.c_void_p()
            _capi.check(lib, lib.qsim_plan_compile(circ, C.byref(opt), C.byref(plan)))
            self._plan = plan
        finally:
            lib.qsim_circuit_destroy(circ)
        st = _capi.PlanStats()
        _capi.check(lib, lib.qsim_plan_stats(self._plan, C.byref(st)))
        self.stats = st.as_dict()

    def residual_array(self) -> np.ndarray:
        """With the ``defer_tail`` option: the diagonal / antidiagonal single-qubit gate the
        plan left unapplied on every qubit, shape (n, 2, 2); identities elsewhere."""
        out = np.zeros((self.n_bits, 2, 2), dtype=np.complex128)
        _capi.check(self.backend.lib, self.backend.lib.qsim_plan_residual(self._plan, _dptr(out.view(np.float64))))
        return out

    def residual(self):
        """``residual_array`` as ``[(qubit, 2x2 matrix), ...]`` without the identities."""
        out = self.residual_array()
        eye = np.eye(2)
        return [(q, out[q]) for q in range(self.n_bits) if not np.array_equal(out[q], eye)]

    def execute(self, buf, scratch=None) -> None:
        """Run the plan on ``buf`` in place.  (``scratch`` is accepted for compatibility and
        unused: gates on more than four qubits run in place as well.)"""
        be = self.backend
        _capi.check(be.lib, be.lib.qsim_plan_execute(self._plan, be.ptr(buf), self.n_bits, None, be.stream()))

    def __del__(self):
        plan, self._plan = getattr(self, "_plan", None), None
        if plan is not None:
            try:
                self.backend.lib.qsim_plan_destroy(plan)
            except Exception:
                pass


class PendingState:
    """Result of a non-blocking run: the final state on its way to a pinned host buffer."""

    def __init__(self, copy, array: np.ndarray):
        self._copy, self._array = copy, array

    def done(self) -> bool:
        return self._copy is None or self._copy.done()

    def result(self) -> np.ndarray:
        if self._copy is not None:
            self._copy.wait()
            self._copy = None
        return self._array


# ---- states ------------------------------------------------------------------------------
class DeviceState:
    """A ket (ndim 1) or density matrix (ndim 2, stored as its row-major vec)
    resident in device memory."""

    _qsim_device_state = True

    def __init__(self, backend, buf, n_bits: int, ndim: int, host_dtype=np.complex128):
        self.backend = backend
        self.buf = buf
        self.n_bits = int(n_bits)          # log2(len(buf))
        self.ndim = int(ndim)
        # dtype the reference would have produced so far (NumPy promotion)
        self.host_dtype = np.dtype(host_dtype)
        # measuring the last qubit of a ket leaves a 0-d array in the reference
        # (vector @ vector, DV/gates.py:176); remembered so to_numpy() can mirror it
        self.scalar_shape = False

    # -- construction ------------------------------------------------------------------
    @classmethod
    def from_numpy(cls, arr: np.ndarray, backend=None) -> "DeviceState":
        backend = backend or get_backend()
        arr = np.asarray(arr)
        if arr.ndim not in (1, 2):
            raise ValueError("State has wrong dimensions.")
        size = arr.size
        if size == 0 or size & (size - 1):
            raise ValueError("Given array is not a qubit state nor operator")
        if arr.ndim == 2 and arr.shape[0] != arr.shape[1]:
            raise ValueError("density matrix must be square")
        buf = backend.upload(_as_c128(arr).reshape(-1))
        return cls(backend, buf, size.bit_length() - 1, arr.ndim, arr.dtype)

    @classmethod
    def product(cls, vectors, backend=None) -> "DeviceState":
        """Kronecker product of single-qubit kets (DV/simulator.py:26), built on
        the device without ever forming it on the host."""
        backend = backend or get_backend()
        vecs = [np.asarray(v) for v in vectors]
        n = len(vecs)
        if n == 0:
            raise ValueError("need at least one qubit")
        amps = _as_c128(np.stack([_as_c128(v) for v in vecs]))
        buf = backend.empty(1 << n)
        lib = backend.lib
        _capi.check(lib, lib.qsim_init_product(backend.ptr(buf), n, _dptr(amps.view(np.float64)),
                                               backend.stream()))
        return cls(backend, buf, n, 1, np.result_type(*[v.dtype for v in vecs]))

    # -- views ---------------------------------------------------------------------------
    @property
    def num_qubits(self) -> int:
        return self.n_bits if self.ndim == 1 else self.n_bits // 2

    @property
    def shape(self):
        if self.ndim == 1:
            if self.scalar_shape and self.n_bits == 0:
                return ()
            return (1 << self.n_bits,)
        d = 1 << (self.n_bits // 2)
        return (d, d)

    def copy(self) -> "DeviceState":
        return DeviceState(self.backend, self.backend.clone(self.buf), self.n_bits, self.ndim, self.host_dtype)

    def to_numpy_async(self, out: np.ndarray) -> "PendingState":
        """Start copying the state into the pinned complex128 buffer ``out`` and return at once;
        ``result()`` of the returned object waits for the copy and gives the array."""
        if out.dtype != np.complex128 or out.size != (1 << self.n_bits) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous complex128 array of the state's size")
        start = getattr(self.backend, "download_async", None)
        if start is None:                                   # host emulator: nothing to overlap
            self.backend.download(self.buf, out)
            return PendingState(None, out.reshape(self.shape))
        return PendingState(start(self.buf, out), out.reshape(self.shape))

    def to_numpy(self, out: np.ndarray | None = None, mirror_dtype: bool = True) -> np.ndarray:
        """Copy to the host.  With ``mirror_dtype`` the result is cast to the
        dtype NumPy promotion gives in the reference (real gates on real states
        stay real)."""
        if out is not None:
            if out.dtype != np.complex128 or out.size != (1 << self.n_bits) or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous complex128 array of the state's size")
            self.backend.download(self.buf, out)
            return out.reshape(self.shape)
        host = self.backend.download(self.buf).reshape(self.shape)
        if mirror_dtype and self.host_dtype.kind != "c":
            real = host.real
            if self.host_dtype.kind in "iub":
                return np.rint(real).astype(self.host_dtype)
            return np.ascontiguousarray(real, dtype=self.host_dtype)
        return host

    # -- reductions (DV/numpy_quantum.py:131-166) -------------------------------------------
    def _reduce(self, fn, *args) -> np.ndarray:
        out = np.zeros(2, dtype=np.float64)
        _capi.check(self.backend.lib, fn(*args, _dptr(out), self.backend.stream()))
        return out

    def norm(self) -> float:
        if self.ndim != 1:
            raise TypeError("norm of a density matrix is not defined here; use trace()")
        lib = self.backend.lib
        out = self._reduce(lib.qsim_reduce_norm2, self.backend.ptr(self.buf), C.c_uint64(1 << self.n_bits))
        return float(np.sqrt(out[0]))

    def trace(self) -> complex:
        if self.ndim != 2:
            raise TypeError("trace needs a density matrix")
        lib = self.backend.lib
        out = self._reduce(lib.qsim_reduce_trace, self.backend.ptr(self.buf), self.n_bits // 2)
        return complex(out[0], out[1])

    def purity(self) -> float:
        if self.ndim != 2:
            raise TypeError("purity needs a density matrix")
        lib = self.backend.lib
        out = self._reduce(lib.qsim_reduce_purity, self.backend.ptr(self.buf), self.n_bits // 2)
        return float(out[0])

    def inner(self, other: "DeviceState") -> complex:
        """<self|other> for two kets."""
        if self.ndim != 1 or other.ndim != 1 or self.n_bits != other.n_bits:
            raise TypeError("inner needs two kets of the same size")
        lib = self.backend.lib
        out = self._reduce(lib.qsim_reduce_inner, self.backend.ptr(self.buf), other.backend.ptr(other.buf),
                           C.c_uint64(1 << self.n_bits))
        return complex(out[0], out[1])

    def expect_ket(self, ket: "DeviceState") -> complex:
        """<ket| self |ket> for a density matrix ``self``."""
        if self.ndim != 2 or ket.ndim != 1 or ket.n_bits * 2 != self.n_bits:
            raise TypeError("expect_ket needs a density matrix and a ket of matching size")
        lib = self.backend.lib
        out = self._reduce(lib.qsim_reduce_expect, self.backend.ptr(ket.buf), self.backend.ptr(self.buf),
                           ket.n_bits)
        return complex(out[0], out[1])

    def expect_pauli(self, x_masks, z_masks) -> np.ndarray:
        """Expectation values of the Pauli strings ``(x_masks[t], z_masks[t])`` (bit q =
        reference qubit q, operator i^popc(x & z) X^x Z^z): <P_t> as float64 for a ket,
        tr(rho P_t) as complex128 for a density matrix (``observables`` builds the masks)."""
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        if x.shape != z.shape:
            raise ValueError("x_masks and z_masks must have the same length")
        lib, be = self.backend.lib, self.backend
        if self.ndim == 1:
            out = np.zeros(len(x), dtype=np.float64)
            _capi.check(lib, lib.qsim_expect_pauli(be.ptr(self.buf), self.n_bits, len(x), x.ctypes.data,
                                                   z.ctypes.data, _dptr(out), be.stream()))
            return out
        out = np.zeros(len(x), dtype=np.complex128)
        _capi.check(lib, lib.qsim_expect_pauli_dm(be.ptr(self.buf), self.n_bits // 2, len(x), x.ctypes.data,
                                                  z.ctypes.data, _dptr(out.view(np.float64)), be.stream()))
        return out

    def apply_pauli_rotations(self, x_masks, z_masks, angles) -> "DeviceState":
        """In place: state <- R_{k-1} ... R_0 state with R_t = exp(-i angles[t]/2 P_t) and P_t the
        string ``(x_masks[t], z_masks[t])`` (convention of ``expect_pauli``), in that order; a
        density matrix becomes U rho U^dagger.  Returns ``self``."""
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        a = np.ascontiguousarray(angles, dtype=np.float64).reshape(-1)
        if x.shape != z.shape or x.shape != a.shape:
            raise ValueError("x_masks, z_masks and angles must have the same length")
        lib, be = self.backend.lib, self.backend
        fn, n = (lib.qsim_apply_pauli_rotations, self.n_bits) if self.ndim == 1 else \
            (lib.qsim_apply_pauli_rotations_dm, self.n_bits // 2)
        _capi.check(lib, fn(be.ptr(self.buf), n, len(x), x.ctypes.data, z.ctypes.data, a.ctypes.data, be.stream()))
        self.host_dtype = np.dtype(np.complex128)
        return self

    def apply_pauli_sum(self, x_masks, z_masks, coeffs, out: "DeviceState | None" = None) -> "DeviceState":
        """H|psi> for a ket, H rho for a density matrix, with H = sum_t coeffs[t] P_t (complex
        coefficients, strings as in ``expect_pauli``), into a new state or into ``out`` (a state of
        the same kind and size in another buffer); returns the result.  The state is unchanged."""
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        c = np.ascontiguousarray(coeffs, dtype=np.complex128).reshape(-1)
        if x.shape != z.shape or x.shape != c.shape:
            raise ValueError("x_masks, z_masks and coeffs must have the same length")
        if self.ndim == 2 and len(x) and (int(x.max()) >> self.num_qubits or int(z.max()) >> self.num_qubits):
            raise ValueError("a Pauli mask has a bit at or above n_qubits")
        be = self.backend
        if out is None:
            out = DeviceState(be, be.empty(1 << self.n_bits), self.n_bits, self.ndim)
        elif out.ndim != self.ndim or out.n_bits != self.n_bits:
            raise ValueError("out must be a state of the same kind and size")
        # a density matrix is its vec: a 2N-qubit ket whose qubits 0..N-1 are the row qubits of rho
        _capi.check(be.lib, be.lib.qsim_apply_pauli_sum(be.ptr(self.buf), be.ptr(out.buf), self.n_bits, len(x),
                                                        x.ctypes.data, z.ctypes.data, c.ctypes.data, be.stream()))
        out.host_dtype = np.dtype(np.complex128)
        return out

    def pauli_rotations_adjoint(self, lam: "DeviceState", x_masks, z_masks, angles) -> np.ndarray:
        """The backward sweep of the adjoint method (``qsim_pauli_rotations_adjoint`` / ``_dm``) over
        U = R_{k-1} ... R_0, the rotation list of ``apply_pauli_rotations``, in place on two states:
        ``self`` (psi = U psi0 on entry) returns to psi0 and ``lam`` becomes U^dagger lam.  Returns
        out[t] = Im<lam_t|P_t|psi_t> (kets; d<H>/d theta_t when lam = H psi) or d Re<<lam|rho>>/d theta_t
        (density matrices) as float64, in caller order.  Synchronises."""
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        a = np.ascontiguousarray(angles, dtype=np.float64).reshape(-1)
        if x.shape != z.shape or x.shape != a.shape:
            raise ValueError("x_masks, z_masks and angles must have the same length")
        if lam.ndim != self.ndim or lam.n_bits != self.n_bits:
            raise ValueError("psi and lam must be states of the same kind and size")
        lib, be = self.backend.lib, self.backend
        fn = lib.qsim_pauli_rotations_adjoint if self.ndim == 1 else lib.qsim_pauli_rotations_adjoint_dm
        out = np.zeros(len(x), dtype=np.float64)
        _capi.check(lib, fn(be.ptr(self.buf), be.ptr(lam.buf), self.num_qubits, len(x), x.ctypes.data, z.ctypes.data,
                            a.ctypes.data, out.ctypes.data, be.stream()))
        self.host_dtype = lam.host_dtype = np.dtype(np.complex128)
        return out

    # -- measurement statistics ------------------------------------------------------------------
    def probabilities(self, qubits=None, *, device: bool = False):
        """Marginal distribution over ``qubits`` (default: all qubits): 2^k float64 entries, bit
        k-1-j of the entry number is the value of ``qubits[j]`` (``qubits[0]`` most significant).
        |psi_i|^2 for a ket, Re rho[i, i] for a density matrix, not normalised.  ``device=True``
        returns the device array instead of a NumPy copy."""
        n = self.num_qubits
        q = _qubit_list(qubits, n)
        out = marginal_probs(self.backend, self.buf, n, q, self.ndim == 2)
        return out if device else self.backend.download(out)

    def sample(self, shots: int, qubits=None, *, rng=None) -> np.ndarray:
        """``shots`` measurement outcomes over ``qubits`` (default: all) as int64, ``qubits[0]``
        the most significant bit.  Uniforms come from ``rng.random(shots)`` on the host (``rng``: a
        ``np.random.Generator``, a seed, or None for ``default_rng()``); full basis indices are
        drawn by inverse-CDF sampling on the device (``qsim_sample``) and projected on the qubits.
        The state is left unchanged."""
        n = self.num_qubits
        q = _qubit_list(qubits, n)
        gen = rng if isinstance(rng, np.random.Generator) else np.random.default_rng(rng)
        u = gen.random(int(shots))
        idx, _total = sample_indices(self.backend, self.buf, n, u, self.ndim == 2)
        return project_outcomes(idx, n, q)


def _qubit_list(qubits, n: int) -> list:
    q = list(range(n)) if qubits is None else [int(v) for v in qubits]
    if any(not 0 <= v < n for v in q):
        raise ValueError("qubit out of range")
    if len(set(q)) != len(q):
        raise ValueError("qubits must be distinct")
    return q


def marginal_probs(backend, buf, n: int, qubits, dm: bool = False):
    """``qsim_marginal_probs`` (``_dm``) of the buffer over reference qubits ``qubits`` of an
    n-qubit register: a new device array of 2^len(qubits) doubles."""
    q = np.ascontiguousarray(qubits, dtype=np.int32)
    out = backend.zeros(1 << len(q), np.float64)
    fn = backend.lib.qsim_marginal_probs_dm if dm else backend.lib.qsim_marginal_probs
    _capi.check(backend.lib, fn(backend.ptr(buf), n, len(q), q.ctypes.data_as(_capi.c_int_p), backend.ptr(out),
                                backend.stream()))
    return out


def sample_indices(backend, buf, n: int, uniforms: np.ndarray, dm: bool = False):
    """``qsim_sample`` (``_dm``) with the host uniforms uploaded: (int64 basis indices on the host,
    the total mass sampled from)."""
    u = np.ascontiguousarray(uniforms, dtype=np.float64).reshape(-1)
    shots = len(u)
    if shots == 0:
        return np.zeros(0, dtype=np.int64), 0.0
    lib = backend.lib
    need = C.c_uint64()
    _capi.check(lib, lib.qsim_sample_workspace_bytes(n, shots, C.byref(need)))
    ws = backend.zeros(int(need.value), np.uint8)
    du = backend.upload(u)
    out = backend.zeros(shots, np.int64)                 # uint64 indices < 2^40: the same bits
    total = C.c_double()
    fn = lib.qsim_sample_dm if dm else lib.qsim_sample
    _capi.check(lib, fn(backend.ptr(buf), n, shots, backend.ptr(du), backend.ptr(out), C.byref(total),
                        backend.ptr(ws), need.value, backend.stream()))
    return np.asarray(backend.download(out), dtype=np.int64), float(total.value)


def project_outcomes(indices: np.ndarray, n: int, qubits) -> np.ndarray:
    """Basis indices of an n-qubit register -> outcomes over ``qubits`` (``qubits[0]`` the MSB)."""
    k = len(qubits)
    if list(qubits) == list(range(n)):
        return indices
    out = np.zeros(len(indices), dtype=np.int64)
    for j, q in enumerate(qubits):
        out |= ((indices >> (n - 1 - q)) & 1) << (k - 1 - j)
    return out


def _to_device(x, backend) -> DeviceState:
    return x if isinstance(x, DeviceState) else DeviceState.from_numpy(x, backend)


def device_fidelity(a, b) -> float:
    """npq.fidelity (DV/numpy_quantum.py:148-161) with at least one device operand."""
    backend = a.backend if isinstance(a, DeviceState) else b.backend
    a_nd, b_nd = a.ndim, b.ndim
    if a_nd == 2 and b_nd == 2:
        # needs eigenvalues: small host LAPACK problem, as in the reference
        ha = a.to_numpy(mirror_dtype=False) if isinstance(a, DeviceState) else a
        hb = b.to_numpy(mirror_dtype=False) if isinstance(b, DeviceState) else b
        ev = np.clip(np.linalg.eigvals(ha @ hb).real, 0.0, None)
        return float(np.sum(np.sqrt(ev)) ** 2)
    da, db = _to_device(a, backend), _to_device(b, backend)
    if a_nd == 1 and b_nd == 1:
        return abs(da.inner(db)) ** 2
    if a_nd == 1:
        return db.expect_ket(da).real
    return da.expect_ket(db).real


# ---- operations on device states ----------------------------------------------------------
def apply_lowered(state: DeviceState, ops, options: dict | None = None) -> dict:
    """Apply a list of ``(targets, matrix)`` gates (targets in buffer-qubit
    numbering) in place as one fused plan; returns the plan statistics."""
    if not ops:
        return {}
    plan = Plan(state.backend, state.n_bits, ops, options)
    plan.execute(state.buf)
    return plan.stats


def measure(state: DeviceState, qubit: int, vec0: np.ndarray, vec1: np.ndarray, forced=None):
    """M.apply (DV/gates.py:165-186) on a device ket: GPU reduction for the two
    norms, the outcome drawn on the host from NumPy's *global* legacy generator
    exactly as the reference does, then a compacting collapse kernel."""
    if state.ndim != 1:
        return _measure_dm(state, qubit, vec0, vec1, forced)
    be, lib = state.backend, state.backend.lib
    n = state.n_bits
    if not 0 <= qubit < n:
        raise ValueError("new_ordering must be a permutation of all qubits")
    b0, b1 = _as_c128(vec0), _as_c128(vec1)
    probs = np.zeros(2, dtype=np.float64)
    _capi.check(lib, lib.qsim_measure_probs(be.ptr(state.buf), n, int(qubit), _dptr(b0.view(np.float64)),
                                            _dptr(b1.view(np.float64)), _dptr(probs), be.stream()))
    norm0, norm1 = np.sqrt(probs[0]), np.sqrt(probs[1])
    if forced is None:
        s = int(np.random.choice([0, 1], p=[norm0 ** 2, norm1 ** 2]))
    else:
        s = forced
    out = be.empty(1 << (n - 1))
    bra = (b0, b1)[s]
    _capi.check(lib, lib.qsim_collapse(be.ptr(state.buf), be.ptr(out), n, int(qubit),
                                       _dptr(bra.view(np.float64)), float((norm0, norm1)[s]), be.stream()))
    collapsed = DeviceState(be, out, n - 1, 1, np.complex128)
    collapsed.scalar_shape = (n == 1)
    return collapsed, s


def _measure_dm(state: DeviceState, qubit: int, vec0, vec1, forced):
    """Measurement of a density matrix.  The reference leaves this undefined
    (its M.apply computes a one-sided product on a 2-D array, SURVEY.md 3.3); we
    define it as the ket rule lifted to rho: rho_s = (v_s . rho . conj(v_s)) on
    the measured qubit, p_s = tr rho_s, result rho_s / p_s."""
    be, lib = state.backend, state.backend.lib
    N = state.n_bits // 2
    if not 0 <= qubit < N:
        raise ValueError("new_ordering must be a permutation of all qubits")
    results = []
    for v in (vec0, vec1):
        v = _as_c128(v)
        vc = np.conjugate(v)
        mid = be.empty(1 << (2 * N - 1))
        _capi.check(lib, lib.qsim_collapse(be.ptr(state.buf), be.ptr(mid), 2 * N, int(qubit),
                                           _dptr(v.view(np.float64)), 1.0, be.stream()))
        fin = be.empty(1 << (2 * N - 2))
        # after removing row qubit `qubit`, column qubit `qubit` sits at N - 1 + qubit
        _capi.check(lib, lib.qsim_collapse(be.ptr(mid), be.ptr(fin), 2 * N - 1, N - 1 + int(qubit),
                                           _dptr(vc.view(np.float64)), 1.0, be.stream()))
        results.append(DeviceState(be, fin, 2 * N - 2, 2, np.complex128))
    p0, p1 = results[0].trace().real, results[1].trace().real
    if forced is None:
        s = int(np.random.choice([0, 1], p=[p0, p1]))
    else:
        s = forced
    chosen = results[s]
    be.divide_(chosen.buf, (p0, p1)[s])
    return chosen, s


def insert(state: DeviceState, position: int, vec: np.ndarray) -> DeviceState:
    """Insert.apply (DV/gates.py:145-153): grow the register by one qubit."""
    be, lib = state.backend, state.backend.lib
    v = _as_c128(vec)
    dtype = np.result_type(state.host_dtype, np.asarray(vec).dtype)
    if state.ndim == 1:
        n = state.n_bits
        if not 0 <= position <= n:
            raise ValueError("new_ordering must be a permutation of all qubits")
        out = be.empty(1 << (n + 1))
        _capi.check(lib, lib.qsim_insert(be.ptr(state.buf), be.ptr(out), n, int(position),
                                         _dptr(v.view(np.float64)), be.stream()))
        return DeviceState(be, out, n + 1, 1, dtype)
    # density matrix: rho (x) |v><v| with the new qubit at `position` in rows and columns
    N = state.n_bits // 2
    if not 0 <= position <= N:
        raise ValueError("new_ordering must be a permutation of all qubits")
    mid = be.empty(1 << (2 * N + 1))
    _capi.check(lib, lib.qsim_insert(be.ptr(state.buf), be.ptr(mid), 2 * N, int(position),
                                     _dptr(v.view(np.float64)), be.stream()))
    vc = np.conjugate(v)
    out = be.empty(1 << (2 * N + 2))
    _capi.check(lib, lib.qsim_insert(be.ptr(mid), be.ptr(out), 2 * N + 1, N + 1 + int(position),
                                     _dptr(vc.view(np.float64)), be.stream()))
    return DeviceState(be, out, 2 * N + 2, 2, dtype)
