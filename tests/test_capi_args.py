"""Argument checks of the compute entry points of the C ABI, in both libraries.

Every call below is invalid, so it must be refused before any work is done: the
CUDA library returns its error without touching CUDA (there is no GPU in the CPU
suite; a check behind the device binding would answer QSIM_ERR_CUDA instead), and
the host emulator returns the same code and the same message.  The buffers are
small host arrays; no call here is ever valid."""
import ctypes as C

import numpy as np
import pytest

from quantum_computations_b200 import _capi, build_native

ARG, UNSUPPORTED = -1, -3


def _load(path):
    lib = C.CDLL(path)
    _capi.declare(lib)
    return lib


@pytest.fixture(scope="module", params=["cuda", "emu"])
def lib(request):
    return _load(build_native.build_cuda() if request.param == "cuda" else build_native.build_emu())


def D(a):
    return a.ctypes.data_as(_capi.c_double_p)


def I(a):
    return a.ctypes.data_as(_capi.c_int_p)


def V(a):
    return a.ctypes.data


ST = np.zeros(64, dtype=np.complex128)           # stands for every state, shard and buffer
OUT = np.zeros(64, dtype=np.float64)
H = (np.array([[1, 1], [1, -1]]) / np.sqrt(2)).astype(np.complex128).view(np.float64).copy()
H2 = np.kron(H.view(np.complex128), H.view(np.complex128)).view(np.float64).copy()
M16 = np.eye(16, dtype=np.complex128).view(np.float64).copy()      # superoperator of one qubit
NAN = H.reshape(-1).copy()
NAN[3] = np.nan
DIAG1 = np.array([1, 0, 1, 0], dtype=np.float64)
DIAG_NAN = np.array([1, 0, np.inf, 0], dtype=np.float64)
Q0 = np.array([0], dtype=np.int32)
Q01 = np.array([0, 1], dtype=np.int32)
Q00 = np.array([0, 0], dtype=np.int32)
QNEG = np.array([-1], dtype=np.int32)
Q3 = np.array([3], dtype=np.int32)
PERM_ID = np.array([0, 1], dtype=np.int32)
PERM_DUP = np.array([0, 0], dtype=np.int32)
PERM_BIG = np.array([0, 2], dtype=np.int32)
PERM_NEG = np.array([-1, 0], dtype=np.int32)
BRA = np.array([1, 0, 0, 0], dtype=np.float64)
AMPS = np.array([1, 0, 0, 0] * 41, dtype=np.float64)
MASK0 = np.array([0], dtype=np.uint64)
MASK1 = np.array([1], dtype=np.uint64)
MASK8 = np.array([8], dtype=np.uint64)          # bit 3: at n = 3 it is out of range
MASK31 = np.array([1 << 31], dtype=np.uint64)   # valid at n = 32
CODES = np.zeros(4, dtype=np.uint16)
OFFS = np.array([0, 1], dtype=np.int64)
OPS = np.zeros(8, dtype=np.int32)
FLIPS = np.zeros(8, dtype=np.uint8)
BITS0 = np.array([0], dtype=np.int32)
BITS00 = np.array([0, 0], dtype=np.int32)
BITS2 = np.array([2], dtype=np.int32)
BITSNEG = np.array([-1], dtype=np.int32)


def plan_for(L, n):
    c = C.c_void_p()
    assert L.qsim_circuit_create(n, C.byref(c)) == 0
    assert L.qsim_circuit_add_matrix(c, 1, I(Q0), D(H)) == 0
    p = C.c_void_p()
    assert L.qsim_plan_compile(c, None, C.byref(p)) == 0
    L.qsim_circuit_destroy(c)
    return p


def execute(L, n, state=True):
    p = plan_for(L, 3)
    try:
        return L.qsim_plan_execute(p, V(ST) if state else None, n, None, None)
    finally:
        L.qsim_plan_destroy(p)


def rb(L, nq=1, n_seq=1, n_opcodes=4, null=None):
    a = [V(CODES), V(OFFS), V(OUT), V(OUT), V(OUT), V(OUT), V(OUT), V(OUT)]
    if null is not None:
        a[null] = None
    return L.qsim_rb_batch(nq, n_seq, a[0], a[1], n_opcodes, a[2], a[3], a[4], a[5], a[6], a[7], None, None)


def traj(L, n=2, shots=1, n_ops=1, fps=2, null=None):
    a = [V(OPS), V(OUT), V(FLIPS), V(ST)]
    if null is not None:
        a[null] = None
    return L.qsim_traj_batch(n, shots, n_ops, a[0], a[1], a[2], fps, a[3], None, V(OUT), None, None, None)


def swap(L, fn, shard=True, buf=True, n_local=4, nbits=1, qubits=Q0, bits=BITS0, first=0, count=1):
    return getattr(L, fn)(V(ST) if shard else None, V(ST) if buf else None, n_local, nbits,
                          None if qubits is None else I(qubits), None if bits is None else I(bits),
                          first, count, None)


def pauli(L, fn, state=True, n=3, n_terms=1, x=MASK1, z=MASK0, out=True):
    return getattr(L, fn)(V(ST) if state else None, n, n_terms, None if x is None else V(x),
                          None if z is None else V(z), D(OUT) if out else None, None)


def _cases():
    cs = []

    def case(name, call, code, msg):
        cs.append(pytest.param(call, code, msg, id=name))

    # qsim_plan_execute
    m = "qsim_plan_execute: null argument"
    case("execute-null-plan", lambda L: L.qsim_plan_execute(None, V(ST), 3, None, None), ARG, m)
    case("execute-null-state", lambda L: execute(L, 3, state=False), ARG, m)
    case("execute-wrong-n", lambda L: execute(L, 4), ARG,
         "qsim_plan_execute: plan was compiled for a different qubit count")

    # qsim_apply_matrix (checks of the one-gate circuit included)
    m = "qsim_apply_matrix: null argument"
    case("matrix-null-state", lambda L: L.qsim_apply_matrix(None, 3, I(Q0), 1, D(H), None, None), ARG, m)
    case("matrix-null-targets", lambda L: L.qsim_apply_matrix(V(ST), 3, None, 1, D(H), None, None), ARG, m)
    case("matrix-null-matrix", lambda L: L.qsim_apply_matrix(V(ST), 3, I(Q0), 1, None, None, None), ARG, m)
    m = "qsim_circuit_create: n_qubits must be in [1, 40]"
    case("matrix-n0", lambda L: L.qsim_apply_matrix(V(ST), 0, I(Q0), 1, D(H), None, None), ARG, m)
    case("matrix-n41", lambda L: L.qsim_apply_matrix(V(ST), 41, I(Q0), 1, D(H), None, None), ARG, m)
    m = "qsim_circuit_add_matrix: k must be in [1, min(10, n)]"
    case("matrix-k0", lambda L: L.qsim_apply_matrix(V(ST), 3, I(Q0), 0, D(H), None, None), ARG, m)
    case("matrix-k11", lambda L: L.qsim_apply_matrix(V(ST), 12, I(Q0), 11, D(H), None, None), ARG, m)
    case("matrix-k-above-n", lambda L: L.qsim_apply_matrix(V(ST), 1, I(Q01), 2, D(H2), None, None), ARG, m)
    m = "qsim_circuit_add_matrix: target out of range"
    case("matrix-target-n", lambda L: L.qsim_apply_matrix(V(ST), 3, I(Q3), 1, D(H), None, None), ARG, m)
    case("matrix-target-neg", lambda L: L.qsim_apply_matrix(V(ST), 3, I(QNEG), 1, D(H), None, None), ARG, m)
    case("matrix-repeated-target", lambda L: L.qsim_apply_matrix(V(ST), 3, I(Q00), 2, D(H2), None, None), ARG,
         "qsim_circuit_add_matrix: targets must be distinct")
    case("matrix-nan", lambda L: L.qsim_apply_matrix(V(ST), 3, I(Q0), 1, D(NAN), None, None), ARG,
         "qsim_circuit_add_matrix: non-finite matrix entry")

    # qsim_apply_diagonal
    m = "qsim_apply_diagonal: null argument"
    case("diagonal-null-state", lambda L: L.qsim_apply_diagonal(None, 3, I(Q0), 1, D(DIAG1), None), ARG, m)
    case("diagonal-null-targets", lambda L: L.qsim_apply_diagonal(V(ST), 3, None, 1, D(DIAG1), None), ARG, m)
    case("diagonal-null-diag", lambda L: L.qsim_apply_diagonal(V(ST), 3, I(Q0), 1, None, None), ARG, m)
    m = "qsim_apply_diagonal: k must be in [1, 4]"
    case("diagonal-k0", lambda L: L.qsim_apply_diagonal(V(ST), 3, I(Q0), 0, D(DIAG1), None), UNSUPPORTED, m)
    case("diagonal-k5", lambda L: L.qsim_apply_diagonal(V(ST), 6, I(Q0), 5, D(DIAG1), None), UNSUPPORTED, m)
    case("diagonal-target-n", lambda L: L.qsim_apply_diagonal(V(ST), 3, I(Q3), 1, D(DIAG1), None), ARG,
         "qsim_circuit_add_matrix: target out of range")
    case("diagonal-inf", lambda L: L.qsim_apply_diagonal(V(ST), 3, I(Q0), 1, D(DIAG_NAN), None), ARG,
         "qsim_circuit_add_matrix: non-finite matrix entry")
    case("diagonal-n0", lambda L: L.qsim_apply_diagonal(V(ST), 0, I(Q0), 1, D(DIAG1), None), ARG,
         "qsim_circuit_create: n_qubits must be in [1, 40]")

    # qsim_apply_permutation
    m = "qsim_apply_permutation: null argument"
    case("permutation-null-state", lambda L: L.qsim_apply_permutation(None, 3, I(Q0), 1, I(PERM_ID), None), ARG, m)
    case("permutation-null-targets", lambda L: L.qsim_apply_permutation(V(ST), 3, None, 1, I(PERM_ID), None), ARG, m)
    case("permutation-null-perm", lambda L: L.qsim_apply_permutation(V(ST), 3, I(Q0), 1, None, None), ARG, m)
    m = "qsim_apply_permutation: k must be in [1, 4]"
    case("permutation-k0", lambda L: L.qsim_apply_permutation(V(ST), 3, I(Q0), 0, I(PERM_ID), None), UNSUPPORTED, m)
    case("permutation-k5", lambda L: L.qsim_apply_permutation(V(ST), 6, I(Q0), 5, I(PERM_ID), None), UNSUPPORTED, m)
    m = "qsim_apply_permutation: not a permutation"
    case("permutation-repeated", lambda L: L.qsim_apply_permutation(V(ST), 3, I(Q0), 1, I(PERM_DUP), None), ARG, m)
    case("permutation-too-big", lambda L: L.qsim_apply_permutation(V(ST), 3, I(Q0), 1, I(PERM_BIG), None), ARG, m)
    case("permutation-negative", lambda L: L.qsim_apply_permutation(V(ST), 3, I(Q0), 1, I(PERM_NEG), None), ARG, m)
    case("permutation-target-neg", lambda L: L.qsim_apply_permutation(V(ST), 3, I(QNEG), 1, I(PERM_ID), None), ARG,
         "qsim_circuit_add_matrix: target out of range")

    # qsim_apply_superop
    m = "qsim_apply_superop: null argument"
    case("superop-null-rho", lambda L: L.qsim_apply_superop(None, 2, I(Q0), 1, D(M16), None, None), ARG, m)
    case("superop-null-targets", lambda L: L.qsim_apply_superop(V(ST), 2, None, 1, D(M16), None, None), ARG, m)
    case("superop-null-superop", lambda L: L.qsim_apply_superop(V(ST), 2, I(Q0), 1, None, None, None), ARG, m)
    m = "qsim_apply_superop: k must be in [1, 5]"
    case("superop-k0", lambda L: L.qsim_apply_superop(V(ST), 2, I(Q0), 0, D(M16), None, None), UNSUPPORTED, m)
    case("superop-k6", lambda L: L.qsim_apply_superop(V(ST), 8, I(Q0), 6, D(M16), None, None), UNSUPPORTED, m)
    m = "qsim_circuit_add_matrix: target out of range"
    case("superop-target-n", lambda L: L.qsim_apply_superop(V(ST), 3, I(Q3), 1, D(M16), None, None), ARG, m)
    case("superop-target-neg", lambda L: L.qsim_apply_superop(V(ST), 3, I(QNEG), 1, D(M16), None, None), ARG, m)
    case("superop-n21", lambda L: L.qsim_apply_superop(V(ST), 21, I(Q0), 1, D(M16), None, None), ARG,
         "qsim_circuit_create: n_qubits must be in [1, 40]")

    # qsim_init_product
    m = "qsim_init_product: bad argument"
    case("product-null-state", lambda L: L.qsim_init_product(None, 3, D(AMPS), None), ARG, m)
    case("product-null-amps", lambda L: L.qsim_init_product(V(ST), 3, None, None), ARG, m)
    case("product-n0", lambda L: L.qsim_init_product(V(ST), 0, D(AMPS), None), ARG, m)
    case("product-n41", lambda L: L.qsim_init_product(V(ST), 41, D(AMPS), None), ARG, m)

    # qsim_measure_probs
    m = "qsim_measure_probs: null argument"
    case("measure-null-state", lambda L: L.qsim_measure_probs(None, 3, 0, D(BRA), D(BRA), D(OUT), None), ARG, m)
    case("measure-null-bra0", lambda L: L.qsim_measure_probs(V(ST), 3, 0, None, D(BRA), D(OUT), None), ARG, m)
    case("measure-null-bra1", lambda L: L.qsim_measure_probs(V(ST), 3, 0, D(BRA), None, D(OUT), None), ARG, m)
    case("measure-null-out", lambda L: L.qsim_measure_probs(V(ST), 3, 0, D(BRA), D(BRA), None, None), ARG, m)
    m = "qsim_measure_probs: qubit out of range"
    case("measure-n0", lambda L: L.qsim_measure_probs(V(ST), 0, 0, D(BRA), D(BRA), D(OUT), None), ARG, m)
    case("measure-qubit-neg", lambda L: L.qsim_measure_probs(V(ST), 3, -1, D(BRA), D(BRA), D(OUT), None), ARG, m)
    case("measure-qubit-n", lambda L: L.qsim_measure_probs(V(ST), 3, 3, D(BRA), D(BRA), D(OUT), None), ARG, m)

    # qsim_collapse
    m = "qsim_collapse: null argument"
    case("collapse-null-in", lambda L: L.qsim_collapse(None, V(ST), 3, 0, D(BRA), 1.0, None), ARG, m)
    case("collapse-null-out", lambda L: L.qsim_collapse(V(ST), None, 3, 0, D(BRA), 1.0, None), ARG, m)
    case("collapse-null-bra", lambda L: L.qsim_collapse(V(ST), V(ST), 3, 0, None, 1.0, None), ARG, m)
    m = "qsim_collapse: qubit out of range"
    case("collapse-n0", lambda L: L.qsim_collapse(V(ST), V(ST), 0, 0, D(BRA), 1.0, None), ARG, m)
    case("collapse-qubit-neg", lambda L: L.qsim_collapse(V(ST), V(ST), 3, -1, D(BRA), 1.0, None), ARG, m)
    case("collapse-qubit-n", lambda L: L.qsim_collapse(V(ST), V(ST), 3, 3, D(BRA), 1.0, None), ARG, m)

    # qsim_insert
    m = "qsim_insert: null argument"
    case("insert-null-in", lambda L: L.qsim_insert(None, V(ST), 3, 0, D(BRA), None), ARG, m)
    case("insert-null-out", lambda L: L.qsim_insert(V(ST), None, 3, 0, D(BRA), None), ARG, m)
    case("insert-null-amp", lambda L: L.qsim_insert(V(ST), V(ST), 3, 0, None, None), ARG, m)
    m = "qsim_insert: position out of range"
    case("insert-n-neg", lambda L: L.qsim_insert(V(ST), V(ST), -1, 0, D(BRA), None), ARG, m)
    case("insert-position-neg", lambda L: L.qsim_insert(V(ST), V(ST), 3, -1, D(BRA), None), ARG, m)
    case("insert-position-above-n", lambda L: L.qsim_insert(V(ST), V(ST), 3, 4, D(BRA), None), ARG, m)

    # reductions
    m = "qsim_reduce_norm2: null argument"
    case("norm2-null-state", lambda L: L.qsim_reduce_norm2(None, 8, D(OUT), None), ARG, m)
    case("norm2-null-out", lambda L: L.qsim_reduce_norm2(V(ST), 8, None, None), ARG, m)
    m = "qsim_reduce_inner: null argument"
    case("inner-null-a", lambda L: L.qsim_reduce_inner(None, V(ST), 8, D(OUT), None), ARG, m)
    case("inner-null-b", lambda L: L.qsim_reduce_inner(V(ST), None, 8, D(OUT), None), ARG, m)
    case("inner-null-out", lambda L: L.qsim_reduce_inner(V(ST), V(ST), 8, None, None), ARG, m)
    m = "qsim_reduce_expect: bad argument"
    case("expect-null-ket", lambda L: L.qsim_reduce_expect(None, V(ST), 2, D(OUT), None), ARG, m)
    case("expect-null-rho", lambda L: L.qsim_reduce_expect(V(ST), None, 2, D(OUT), None), ARG, m)
    case("expect-null-out", lambda L: L.qsim_reduce_expect(V(ST), V(ST), 2, None, None), ARG, m)
    case("expect-n-neg", lambda L: L.qsim_reduce_expect(V(ST), V(ST), -1, D(OUT), None), ARG, m)
    case("expect-n21", lambda L: L.qsim_reduce_expect(V(ST), V(ST), 21, D(OUT), None), ARG, m)
    for fn in ("purity", "trace"):
        name = "qsim_reduce_" + fn
        m = name + ": bad argument"
        case(fn + "-null-rho", lambda L, f=name: getattr(L, f)(None, 2, D(OUT), None), ARG, m)
        case(fn + "-null-out", lambda L, f=name: getattr(L, f)(V(ST), 2, None, None), ARG, m)
        case(fn + "-n-neg", lambda L, f=name: getattr(L, f)(V(ST), -1, D(OUT), None), ARG, m)
        case(fn + "-n21", lambda L, f=name: getattr(L, f)(V(ST), 21, D(OUT), None), ARG, m)

    # Pauli expectation values
    for fn in ("qsim_expect_pauli", "qsim_expect_pauli_dm"):
        tag = fn[5:]
        case(tag + "-terms-neg", lambda L, f=fn: pauli(L, f, n_terms=-1), ARG, fn + ": n_terms < 0")
        m = fn + ": null argument"
        case(tag + "-null-x", lambda L, f=fn: pauli(L, f, x=None), ARG, m)
        case(tag + "-null-z", lambda L, f=fn: pauli(L, f, z=None), ARG, m)
        case(tag + "-null-out", lambda L, f=fn: pauli(L, f, out=False), ARG, m)
        m = fn + ": n_qubits must be in [1, 63]"
        case(tag + "-n0", lambda L, f=fn: pauli(L, f, n=0, x=MASK0), ARG, m)
        case(tag + "-n64", lambda L, f=fn: pauli(L, f, n=64), ARG, m)
        m = fn + ": a Pauli mask has a bit at or above n_qubits"
        case(tag + "-x-mask-high", lambda L, f=fn: pauli(L, f, x=MASK8), ARG, m)
        case(tag + "-z-mask-high", lambda L, f=fn: pauli(L, f, z=MASK8), ARG, m)
        case(tag + "-null-state", lambda L, f=fn: pauli(L, f, state=False), ARG, fn + ": null state")
    case("pauli_dm-n32", lambda L: pauli(L, "qsim_expect_pauli_dm", n=32, x=MASK31), ARG,
         "qsim_expect_pauli_dm: n_qubits must be in [1, 31]")

    # qsim_rb_batch
    for i in range(8):
        case(f"rb-null-{i}", lambda L, i=i: rb(L, null=i), ARG, "qsim_rb_batch: null argument")
    m = "qsim_rb_batch: nq must be 1 or 2"
    case("rb-nq0", lambda L: rb(L, nq=0), UNSUPPORTED, m)
    case("rb-nq3", lambda L: rb(L, nq=3), UNSUPPORTED, m)
    m = "qsim_rb_batch: bad sizes"
    case("rb-nseq-neg", lambda L: rb(L, n_seq=-1), ARG, m)
    case("rb-opcodes0", lambda L: rb(L, n_opcodes=0), ARG, m)
    case("rb-opcodes65537", lambda L: rb(L, n_opcodes=65537), ARG, m)

    # qsim_traj_batch
    for i in range(4):
        case(f"traj-null-{i}", lambda L, i=i: traj(L, null=i), ARG, "qsim_traj_batch: null argument")
    m = "qsim_traj_batch: 1 <= n_qubits <= 12"
    case("traj-n0", lambda L: traj(L, n=0), UNSUPPORTED, m)
    case("traj-n13", lambda L: traj(L, n=13), UNSUPPORTED, m)
    m = "qsim_traj_batch: bad sizes"
    case("traj-shots-neg", lambda L: traj(L, shots=-1), ARG, m)
    case("traj-ops-neg", lambda L: traj(L, n_ops=-1), ARG, m)
    case("traj-flips-neg", lambda L: traj(L, fps=-1), ARG, m)

    # qsim_swap_pack / qsim_swap_unpack
    for fn in ("qsim_swap_pack", "qsim_swap_unpack"):
        tag = fn[5:]
        m = fn + ": null argument"
        case(tag + "-null-shard", lambda L, f=fn: swap(L, f, shard=False), ARG, m)
        case(tag + "-null-buf", lambda L, f=fn: swap(L, f, buf=False), ARG, m)
        m = fn + ": bad bit list"
        case(tag + "-n-local0", lambda L, f=fn: swap(L, f, n_local=0), ARG, m)
        case(tag + "-nbits0", lambda L, f=fn: swap(L, f, nbits=0), ARG, m)
        case(tag + "-nbits9", lambda L, f=fn: swap(L, f, n_local=12, nbits=9), ARG, m)
        case(tag + "-nbits-above-n", lambda L, f=fn: swap(L, f, n_local=1, nbits=2, qubits=Q01, bits=BITS00), ARG, m)
        case(tag + "-null-qubits", lambda L, f=fn: swap(L, f, qubits=None), ARG, m)
        case(tag + "-null-bits", lambda L, f=fn: swap(L, f, bits=None), ARG, m)
        m = fn + ": bad qubit or bit"
        case(tag + "-qubit-neg", lambda L, f=fn: swap(L, f, qubits=QNEG), ARG, m)
        case(tag + "-qubit-n", lambda L, f=fn: swap(L, f, n_local=3, qubits=Q3), ARG, m)
        case(tag + "-bit2", lambda L, f=fn: swap(L, f, bits=BITS2), ARG, m)
        case(tag + "-bit-neg", lambda L, f=fn: swap(L, f, bits=BITSNEG), ARG, m)
        case(tag + "-repeated", lambda L, f=fn: swap(L, f, nbits=2, qubits=Q00, bits=BITS00), ARG,
             fn + ": repeated qubit")
        m = fn + ": chunk out of range"
        case(tag + "-chunk", lambda L, f=fn: swap(L, f, nbits=2, qubits=Q01, bits=BITS00, first=3, count=2), ARG, m)
        case(tag + "-first", lambda L, f=fn: swap(L, f, first=8, count=1), ARG, m)
    return cs


@pytest.mark.parametrize("call, code, message", _cases())
def test_invalid_call_is_refused_before_any_work(lib, call, code, message):
    assert call(lib) == code
    assert lib.qsim_last_error().decode() == message
