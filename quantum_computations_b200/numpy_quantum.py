"""Host-side linear-algebra kit: the drop-in for
``simulators/dv_simulator/numpy_quantum.py`` (reference lines cited per item).

Everything here is small-matrix host code (constants, 2x2 / 4x4 builders,
validators, metrics on NumPy arrays).  The reference's hot routine
``expand_gate`` (numpy_quantum.py:243-247) is kept for API compatibility at
small N but is *not* used by ``Gate.apply`` / ``Simulator.run`` in this
package: those go to the CUDA engine, which never materialises a 2^N x 2^N
operator.  ``fidelity`` / ``purity`` / ``norm`` accept device states
(``engine.DeviceState``) as well and then reduce on the GPU.

Dtypes of the constants match the reference (integer ``ZERO``/``X``/``Z``,
float ``H``/``CZ``/``CX``/``SWAP``, complex ``Y``/``P``/``T``) because result
dtypes follow NumPy promotion (SURVEY.md section 0.4).
"""
from __future__ import annotations

import numpy as np

# ---- constants (numpy_quantum.py:5-25) --------------------------------------
# Integer where the reference is integer, float where it is float, complex where complex:
# result dtypes follow NumPy promotion, so the element types are part of the interface.
_RT2 = np.sqrt(2)
_ket = lambda a, b, scale=1: np.array([a, b]) / scale if scale != 1 else np.array([a, b])   # noqa: E731

ZERO, ONE = _ket(1, 0), _ket(0, 1)
PLUS, MINUS = _ket(1, 1, _RT2), _ket(1, -1, _RT2)
IPLUS, IMINUS = _ket(1, 1j, _RT2), _ket(1, -1j, _RT2)

IDTY = np.identity(2)
X = np.array([[0, 1],
              [1, 0]])
Y = np.array([[0, -1j],
              [1j, 0]])
Z = np.array([[1, 0],
              [0, -1]])
PAULIS = [X, Y, Z]
H = (X + Z) / _RT2

_EYE4 = np.identity(4)
CZ = np.diag([1.0, 1.0, 1.0, -1.0])
CX = _EYE4[[0, 1, 3, 2]]          # permutation matrices, float64 like the reference's
SWAP = _EYE4[[0, 2, 1, 3]]

P = np.diag([1.0, 1.0j])
T = np.diag([1.0, np.exp(0.25j * np.pi)])


# ---- Pauli bookkeeping (numpy_quantum.py:28-76) ------------------------------
class PauliError(ValueError):
    pass


_PAULI_BY_NAME = {"i": 0, "x": 1, "y": 2, "z": 3, "-x": -1, "-y": -2, "-z": -3}
_PAULI_BY_AXIS = {(1, 0, 0): 1, (0, 1, 0): 2, (0, 0, 1): 3,
                  (-1, 0, 0): -1, (0, -1, 0): -2, (0, 0, -1): -3}


def get_pauli_number(pauli_identifier):
    """0 = I, 1..3 = X, Y, Z, negative = the negated operator.  Accepts names
    ('x', 'X', '-z', ...), the numbers themselves, or a unit axis [a, b, c]."""
    found = None
    if isinstance(pauli_identifier, str):
        if len(pauli_identifier) and pauli_identifier[-1].isalpha():
            found = _PAULI_BY_NAME.get(pauli_identifier[:-1] + pauli_identifier[-1].lower())
    elif isinstance(pauli_identifier, (list, tuple)):
        try:
            found = _PAULI_BY_AXIS.get(tuple(pauli_identifier))
        except TypeError:
            found = None
    else:
        try:
            if pauli_identifier in (-3, -2, -1, 0, 1, 2, 3):
                found = int(pauli_identifier)
        except (TypeError, ValueError):
            found = None
    if found is None:
        raise PauliError(f'"{pauli_identifier}" could not be interpreted as a Pauli operator')
    return found


def get_pauli_identifier(pauli_identifier):
    names = {-3: "-Z", -2: "-Y", -1: "-X", 0: "I", 1: "X", 2: "Y", 3: "Z"}
    return names[get_pauli_number(pauli_identifier)]


def is_pauli(case):
    """Whether ``case`` names a (possibly negated) Pauli operator or the identity."""
    try:
        get_pauli_number(case)
        return True
    except PauliError:
        return False


def get_pauli_operator(pauli_identifier):
    number = get_pauli_number(pauli_identifier)
    return PAULIS[number - 1]


def get_pauli_states(pauli_identifier):
    eigenbases = ([PLUS, MINUS], [IPLUS, IMINUS], [ZERO, ONE])
    return eigenbases[get_pauli_number(pauli_identifier) - 1]


def get_pauli_state(pauli_identifier, state_index):
    basis = get_pauli_states(pauli_identifier)
    return basis[state_index]


# ---- state builders (numpy_quantum.py:79-101) ---------------------------------
def basis_state(identifier, N: int | None = None) -> np.ndarray:
    """Computational-basis ket from an int (needs N), a bit string, or a
    sequence of bits."""
    if isinstance(identifier, (list, tuple)):
        return basis_state("".join(str(b) for b in identifier))
    if isinstance(identifier, str):
        return basis_state(int(identifier, 2), len(identifier))
    if isinstance(identifier, (int, np.integer)):
        ket = np.zeros(2 ** N)
        ket[identifier] = 1
        return ket
    raise NotImplementedError(
        f"Could not generate basis state from identifier of type {type(identifier)}")


def qubit_from_polar(theta: float, phi: float) -> np.ndarray:
    half = theta / 2
    return np.array([np.cos(half), np.exp(1j * phi) * np.sin(half)])


def qubit_from_axis(axis) -> np.ndarray:
    ax, ay, az = axis[0], axis[1], axis[-1]
    polar = np.arccos(az / np.sqrt(sum(a ** 2 for a in axis)))
    return qubit_from_polar(polar, np.arctan2(ay, ax))


# ---- small-matrix builders (numpy_quantum.py:100-109, :250-251) ---------------
def phase_gate(theta):
    return np.diag([1, np.exp(1j * theta)])


def axis_rotation(theta: float, axis) -> np.ndarray:
    """exp(-i theta/2 n.sigma).  The DV gate classes RZ/P/Pdg/T/Tdg are built
    from this, *not* from the constants ``P``/``T`` above (global phase)."""
    n_sigma = sum(component * pauli for component, pauli in zip(axis, PAULIS))
    half = theta / 2
    return np.cos(half) * IDTY - 1j * np.sin(half) * n_sigma


def euler_rotation(theta1, theta2, theta3):
    rx = lambda t: axis_rotation(t, [1, 0, 0])
    return rx(theta3) @ axis_rotation(theta2, [0, 0, 1]) @ rx(theta1)


def add_control(gate):
    """|0><0| (x) 1 + |1><1| (x) gate."""
    dim = gate.shape[0]
    out = np.zeros((2 * dim, 2 * dim), dtype=np.result_type(gate.dtype, np.float64))
    out[:dim, :dim] = np.identity(dim)
    out[dim:, dim:] = gate
    return out


# ---- ket / density-matrix helpers (numpy_quantum.py:112-166) -------------------
def _is_device(obj) -> bool:
    return hasattr(obj, "_qsim_device_state")


def ket2dm(ket):
    if ket.ndim != 1:
        raise TypeError("state is not a ket")
    return ket[:, None] * np.conjugate(ket)[None, :]


def dm2ket(dm: np.ndarray, strict: bool = True) -> np.ndarray:
    if not is_hermitian(dm):
        raise TypeError("input is not a density matrix")
    evals, evecs = np.linalg.eigh(dm)
    if strict and not np.allclose(evals[:-1], 0):
        raise TypeError("density matrix does not represent a pure state")
    return normalise(evecs[:, -1])


def norm(ket) -> float:
    if _is_device(ket):
        return ket.norm()
    return np.linalg.norm(np.asarray(ket))


def normalise(state):
    """Unit 2-norm for kets, unit trace for density matrices."""
    scale = {1: np.linalg.norm, 2: np.trace}.get(state.ndim)
    if scale is None:
        raise ValueError("State not ket nor density matrix.")
    return state / scale(state)


def compare_kets(a, b):
    """Equality up to a global phase (and normalisation)."""
    rho_a, rho_b = (ket2dm(normalise(k)) for k in (a, b))
    return np.allclose(rho_a, rho_b)


def fidelity(a, b) -> float:
    """|<a|b>|^2, <psi|rho|psi>, or (tr sqrt(a b))^2 (numpy_quantum.py:148-161).
    Matrices are assumed Hermitian.  Device states reduce on the GPU except for
    the matrix-matrix case, which needs eigenvalues and stays on the host."""
    if _is_device(a) or _is_device(b):
        from .engine import device_fidelity
        return device_fidelity(a, b)
    a_ket, b_ket = a.ndim == 1, b.ndim == 1
    if a_ket and b_ket:
        return np.abs(a.conj() @ b).real ** 2
    # same expressions (hence the same summation order) as the reference, numpy_quantum.py:153-156
    if a_ket:
        return (a.conj() @ b @ a).real
    if b_ket:
        return (b.conj() @ a @ b).real
    spectrum = np.clip(np.linalg.eigvals(a @ b).real, 0.0, None)
    return np.sum(np.sqrt(spectrum)) ** 2


def purity(rho) -> float:
    if _is_device(rho):
        return rho.purity()
    return np.trace(rho @ rho).real          # the reference's expression (numpy_quantum.py:166)


# ---- tensor-product plumbing (numpy_quantum.py:169-258) ------------------------
def tensor(*arrays):
    out = 1
    for factor in arrays:
        out = np.kron(out, factor)
    return out


def is_power_of_two(n):
    return (n & (n - 1) == 0) and n != 0


def is_qubit_operator(oper):
    return oper.ndim == 2 and oper.shape[0] == oper.shape[1] and is_power_of_two(oper.shape[0])


def is_qubit_state(state):
    return state.ndim == 1 and is_power_of_two(len(state))


def is_hermitian(oper):
    return np.allclose(oper, oper.conj().T)


def expect(oper, state):
    """<state| oper |state>.  A ``observables.PauliSum`` operator is evaluated on the GPU for a
    device ket or density matrix, a sharded ket or a host array; a dense operator with a device
    ket reduces on the GPU too (n <= 20)."""
    if getattr(oper, "_qsim_pauli_sum", False):
        from .observables import expect as pauli_expect
        return pauli_expect(oper, state)
    if _is_device(state):
        if state.ndim != 1:
            raise TypeError("incompatible operator and state vector")
        from .engine import DeviceState
        oper = np.asarray(oper)
        if not (is_qubit_operator(oper) and oper.shape[0] == 1 << state.n_bits):
            raise TypeError("incompatible operator and state vector")
        return DeviceState.from_numpy(oper, state.backend).expect_ket(state)
    compatible = is_qubit_operator(oper) and is_qubit_state(state) and oper.shape[0] == state.shape[0]
    if not compatible:
        raise TypeError("incompatible operator and state vector")
    return np.vdot(state, oper @ state)


def expecth(oper, state):
    """Real part of the expectation value (Hermitian operators)."""
    value = expect(oper, state)
    return value.real


def rand_ket(d=2):
    real, imag = np.random.rand(d), np.random.rand(d)       # two draws from the global generator, in this order
    return normalise(real + 1j * imag)


def dagger(array):
    return array.conj().T


def num_qubits(arr) -> int:
    """log2 of a dimension (given directly or as the leading extent of an array)."""
    return int(np.log2(arr if isinstance(arr, int) else arr.shape[0]))


def permute_tensor_product(array, new_ordering):
    """Move tensor factor j to position ``new_ordering[j]`` (rows, and columns
    too for operators) -- numpy_quantum.py:227-240."""
    if not is_power_of_two(array.shape[0]):
        raise ValueError("Given array is not a qubit state nor operator")
    nq = num_qubits(array)
    if set(new_ordering) != set(range(nq)):
        raise ValueError("new_ordering must be a permutation of all qubits")
    source_of = np.argsort(np.asarray(new_ordering))      # inverse permutation
    if array.ndim == 1:
        return array.reshape((2,) * nq).transpose(source_of).reshape(-1)
    cols = array.shape[1]
    if cols == array.shape[0]:
        cube = array.reshape((2,) * (2 * nq))
        axes = list(source_of) + [nq + s for s in source_of]
        return cube.transpose(axes).reshape(array.shape)
    # rectangular: rows first, then the column space on its own terms
    rows_done = array.reshape((2,) * nq + (cols,)).transpose(list(source_of) + [nq])
    rows_done = rows_done.reshape(array.shape)
    back = rows_done.T.reshape((2,) * nq + (-1,)).transpose(list(source_of) + [nq])
    return back.reshape((2 ** nq, -1)).T


def expand_gate(gate, N, targets):
    """Dense (2^N, 2^N) operator (numpy_quantum.py:243-247).  O(4^N): kept for
    compatibility and small N only; the simulator itself never calls it."""
    targets = list(targets)
    others = [q for q in range(N) if q not in targets]
    padded = tensor(gate, *([IDTY] * len(others)))
    return permute_tensor_product(padded, targets + others)
