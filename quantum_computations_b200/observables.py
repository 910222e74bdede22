"""Expectation values of Pauli sums on device states.

The reference evaluates observables only as dense 2^N x 2^N host matrices
(``numpy_quantum.expect``, DV/numpy_quantum.py:254-264), which stops at a dozen
qubits.  Here an observable is a sum of Pauli strings, and every string is
evaluated on the GPU in a read-only pass over the state (``qsim_expect_pauli``):
strings are grouped by their X/Y support, so one read of the state serves up to
32 strings whose X masks span at most four dimensions, and an all-Z observable
costs a single read.  Density matrices (``qsim_expect_pauli_dm``) and sharded
kets (``sharded.ShardedState.expect_pauli``) take the same masks.

The same masks drive evolution: ``evolve`` applies a Trotterised exp(-i H t) for a
``PauliSum`` H as a list of rotations exp(-i theta/2 P) (``apply_pauli_rotations`` of a
device or sharded state, ``qsim_apply_pauli_rotations``), up to 32 rotations per read
and write of the state.

``apply`` gives H|psi> (or H rho) for a ``PauliSum`` on the device (``qsim_apply_pauli_sum``), and
``expect_and_gradient`` gives <H> after a rotation list together with its gradient with respect to
every angle, by the adjoint method (``qsim_pauli_rotations_adjoint``).

Convention: a string is a pair of masks ``(x, z)`` with bit q for reference
qubit q; I = (0, 0), X = (1, 0), Z = (0, 1), Y = (1, 1), and the operator is
``i^popc(x & z) X^x Z^z`` (Z first), so every string is Hermitian.
"""
from __future__ import annotations

import numpy as np

from . import numpy_quantum as npq
from .numpy_quantum import PauliError

_LETTER = "IXYZ"
_NUMBER = {(0, 0): 0, (1, 0): 1, (1, 1): 2, (0, 1): 3}      # (x bit, z bit) -> Pauli number
_SINGLE = {0: np.eye(2, dtype=np.complex128), 1: npq.X.astype(np.complex128),
           2: npq.Y.astype(np.complex128), 3: npq.Z.astype(np.complex128)}


class PauliSum:
    """sum_t c_t P_t over Pauli strings P_t.

    ``terms`` is an iterable of ``(coeff, paulis)``; ``paulis`` is either a string with
    one letter per qubit, qubit 0 first (``"XIZ"``, as in ``npq.tensor``), or a dict
    ``{qubit: identifier}`` with anything ``npq.get_pauli_number`` accepts.  A negated
    identifier ("-x", -3, [0, 0, -1]) folds its sign into the coefficient.  Identical
    strings are merged (first appearance keeps its place)."""

    _qsim_pauli_sum = True

    def __init__(self, terms):
        index = {}
        xs, zs, coeffs = [], [], []
        nq = 0
        for item in terms:
            try:
                coeff, paulis = item
            except (TypeError, ValueError):
                raise PauliError(f"a term must be a pair (coeff, paulis), got {item!r}") from None
            if isinstance(paulis, str):
                factors = {q: npq.get_pauli_number(ch) for q, ch in enumerate(paulis)}
                width = len(paulis)
            elif isinstance(paulis, dict):
                factors = {}
                for q, ident in paulis.items():
                    if not isinstance(q, (int, np.integer)) or q < 0:
                        raise PauliError(f"qubit {q!r} is not a non-negative integer")
                    factors[int(q)] = npq.get_pauli_number(ident)
                width = max(factors) + 1 if factors else 0
            else:
                raise PauliError(f"{paulis!r} is neither a Pauli string nor a {{qubit: Pauli}} dict")
            c = complex(coeff)
            x = z = 0
            for q, number in factors.items():
                if number < 0:
                    c, number = -c, -number
                if number in (1, 2):
                    x |= 1 << q
                if number in (2, 3):
                    z |= 1 << q
            nq = max(nq, width)
            key = (x, z)
            if key in index:
                coeffs[index[key]] += c
            else:
                index[key] = len(xs)
                xs.append(x)
                zs.append(z)
                coeffs.append(c)
        if nq > 63:
            raise PauliError("Pauli strings on more than 63 qubits are not supported")
        self.x_masks = np.array(xs, dtype=np.uint64)
        self.z_masks = np.array(zs, dtype=np.uint64)
        self.coeffs = np.array(coeffs, dtype=np.complex128)
        self.num_qubits = nq

    def __len__(self) -> int:
        return len(self.coeffs)

    def _letters(self, t: int, n: int):
        """Pauli numbers (0 = I, 1..3 = X, Y, Z) of term t on qubits 0 .. n-1."""
        x, z = int(self.x_masks[t]), int(self.z_masks[t])
        return [_NUMBER[((x >> q) & 1, (z >> q) & 1)] for q in range(n)]

    def __repr__(self) -> str:
        body = ", ".join(f"({c!r}, {''.join(_LETTER[p] for p in self._letters(t, self.num_qubits))!r})"
                         for t, c in enumerate(self.coeffs))
        return f"PauliSum([{body}])"

    def matrix(self, n: int | None = None) -> np.ndarray:
        """Dense 2^n x 2^n host matrix (qubit 0 is the first Kronecker factor); small n only."""
        n = self.num_qubits if n is None else int(n)
        if n < self.num_qubits:
            raise ValueError(f"the observable acts on {self.num_qubits} qubits, more than n = {n}")
        out = np.zeros((1 << n, 1 << n), dtype=np.complex128)
        for t, c in enumerate(self.coeffs):
            out += c * npq.tensor(*[_SINGLE[p] for p in self._letters(t, n)])
        return out


def _sharded_type():
    try:
        from .sharded import ShardedState
    except ImportError:                      # pragma: no cover - sharded needs nothing optional
        return ()
    return ShardedState


def expect(observable: PauliSum, state, *, per_term: bool = False):
    """sum_t c_t <P_t> as a Python complex, or with ``per_term`` the array of <P_t>
    (real for kets, complex tr(rho P_t) for density matrices).

    ``state``: an ``engine.DeviceState`` (ket or density matrix), a
    ``sharded.ShardedState`` (collective: every rank calls it and gets the same result) or
    a host ndarray, which is uploaded to the default CUDA backend first -- there is no
    CPU path."""
    if not isinstance(observable, PauliSum):
        raise TypeError("expect needs a PauliSum observable")
    from . import engine
    sharded_type = _sharded_type()
    if isinstance(state, sharded_type):
        values = state.expect_pauli(observable.x_masks, observable.z_masks)
    else:
        if not isinstance(state, engine.DeviceState):
            state = engine.DeviceState.from_numpy(np.asarray(state))
        if observable.num_qubits > state.num_qubits:
            raise ValueError(f"the observable acts on {observable.num_qubits} qubits, "
                             f"the state has {state.num_qubits}")
        values = state.expect_pauli(observable.x_masks, observable.z_masks)
    if per_term:
        return values
    return complex(np.dot(observable.coeffs, values))


def _device_state(state, num_qubits: int, what: str):
    """``state`` itself if sharded or on the device, else uploaded; refuses a sharded density matrix and
    an operator wider than the state."""
    from . import engine
    if isinstance(state, _sharded_type()):
        if state.is_density:
            raise NotImplementedError(f"a {what} on a sharded density matrix is not implemented")
        width = state.n
    else:
        if not isinstance(state, engine.DeviceState):
            state = engine.DeviceState.from_numpy(np.asarray(state))
        width = state.num_qubits
    if num_qubits > width:
        raise ValueError(f"the {what} acts on {num_qubits} qubits, the state has {width}")
    return state


def apply(operator: PauliSum, state):
    """H|psi> for a ket, H rho for a density matrix, as a new state (``qsim_apply_pauli_sum``: one
    read of the state and one write of the result per pass of up to 32 strings); the state is
    unchanged.  ``state``: an ``engine.DeviceState``, a ``sharded.ShardedState`` ket (collective, a new
    sharded ket; a sharded density matrix raises NotImplementedError) or a host ndarray, uploaded first.  Complex coefficients are allowed."""
    if not isinstance(operator, PauliSum):
        raise TypeError("apply needs a PauliSum operator")
    state = _device_state(state, operator.num_qubits, "operator")
    return state.apply_pauli_sum(operator.x_masks, operator.z_masks, operator.coeffs)


def _vec_identity(backend, n: int):
    """vec(I) of an n-qubit identity on the device: |+>^n (unnormalised) on the row qubits, |0>^n on
    the column qubits, then a CNOT from every row qubit to its column qubit."""
    from . import engine
    ket = engine.DeviceState.product([np.array([1.0, 1.0])] * n + [np.array([1.0, 0.0])] * n, backend)
    cnot = np.eye(4, dtype=np.complex128)[[0, 1, 3, 2]]
    engine.apply_lowered(ket, [([q, q + n], cnot) for q in range(n)])
    return engine.DeviceState(backend, ket.buf, 2 * n, 2)


def expect_and_gradient(hamiltonian: PauliSum, rotations, state):
    """(E, dE/dtheta) for E(theta) = <H> on U(theta) state, U = R_{k-1} ... R_0 the rotation list
    ``rotations = (x_masks, z_masks, angles)`` of ``trotter_rotations`` / ``apply_pauli_rotations``,
    by the adjoint method: one forward sweep, one application of H and one backward sweep
    (``qsim_pauli_rotations_adjoint``), whatever k is.  E is a float, the gradient a float64 array in
    caller order.  Parameters shared between rotations (QAOA's gamma on every ZZ term) are the
    caller's chain rule: sum the entries of the rotations that share one.

    ``state``: a ket or density matrix (``engine.DeviceState``, or a host ndarray, uploaded first) or
    a ``sharded.ShardedState`` ket (collective; a sharded density matrix raises NotImplementedError).  It is left unchanged: the work happens on two
    scratch states of its size, psi = U state and lam = H psi (for a density matrix lam = vec(H)).
    H must have real coefficients."""
    if not isinstance(hamiltonian, PauliSum):
        raise TypeError("expect_and_gradient needs a PauliSum Hamiltonian")
    if np.any(hamiltonian.coeffs.imag != 0):
        raise ValueError("the Hamiltonian has a coefficient with a nonzero imaginary part (not Hermitian)")
    x, z, angles = rotations
    state = _device_state(state, hamiltonian.num_qubits, "Hamiltonian")
    if getattr(state, "ndim", 1) == 1:
        psi = state.copy().apply_pauli_rotations(x, z, angles)
        lam = psi.apply_pauli_sum(hamiltonian.x_masks, hamiltonian.z_masks, hamiltonian.coeffs)
        value = psi.inner(lam).real
    else:
        from . import engine
        # vec(H) first, so that vec(I) is gone before the copy of rho is made
        lam = _vec_identity(state.backend, state.num_qubits).apply_pauli_sum(
            hamiltonian.x_masks, hamiltonian.z_masks, hamiltonian.coeffs)
        psi = state.copy().apply_pauli_rotations(x, z, angles)
        as_ket = lambda s: engine.DeviceState(s.backend, s.buf, s.n_bits, 1)     # noqa: E731
        value = as_ket(lam).inner(as_ket(psi)).real                              # Re tr(H^dagger rho)
    grad = psi.pauli_rotations_adjoint(lam, x, z, angles)
    if isinstance(state, _sharded_type()):
        # after the sweep's all-reduce no rank exchanges with these shards any more: release their
        # exchange staging and peer mappings now rather than whenever they are collected
        psi.close()
        lam.close()
    return float(value), grad


def trotter_rotations(hamiltonian: PauliSum, time: float, steps: int = 1, order: int = 1):
    """The rotation list ``(x_masks, z_masks, angles)`` of a Trotterised exp(-i H time): ``steps``
    first-order steps (terms in the sum's order, angle 2 c_t time / steps) or symmetric second-order
    (Strang) steps (every term but the last at half the angle, forward then backward).  Adjacent
    rotations about the same string are merged, which is exact."""
    if not isinstance(hamiltonian, PauliSum):
        raise TypeError("evolve needs a PauliSum Hamiltonian")
    if order not in (1, 2):
        raise ValueError("order must be 1 or 2")
    steps = int(steps)
    if steps < 1:
        raise ValueError("steps must be at least 1")
    if np.any(hamiltonian.coeffs.imag != 0):
        raise ValueError("the Hamiltonian has a coefficient with a nonzero imaginary part (not Hermitian)")
    full = 2.0 * hamiltonian.coeffs.real * (float(time) / steps)
    terms = list(range(len(hamiltonian)))
    if order == 1:
        one = [(t, full[t]) for t in terms]
    else:
        one = [(t, 0.5 * full[t]) for t in terms[:-1]] + [(t, full[t]) for t in terms[-1:]] + \
              [(t, 0.5 * full[t]) for t in reversed(terms[:-1])]
    merged = []
    for t, angle in one * steps:
        if merged and merged[-1][0] == t:
            merged[-1][1] += angle
        else:
            merged.append([t, angle])
    index = np.array([t for t, _ in merged], dtype=np.int64)
    return (hamiltonian.x_masks[index], hamiltonian.z_masks[index],
            np.array([a for _, a in merged], dtype=np.float64))


def evolve(hamiltonian: PauliSum, state, time: float, *, steps: int = 1, order: int = 1):
    """Trotterised exp(-i H time) applied in place to ``state`` (an ``engine.DeviceState`` ket or
    density matrix, or a ``sharded.ShardedState``, collectively); returns the state.  H must have
    real coefficients.  The identity term is kept as a global phase, so a ket matches
    ``expm(-1j * H * time)`` including its phase when the terms commute.  All rotations go to
    ``apply_pauli_rotations`` in one call (see ``trotter_rotations``)."""
    x, z, angles = trotter_rotations(hamiltonian, time, steps, order)
    if not isinstance(state, _sharded_type()) and hamiltonian.num_qubits > state.num_qubits:
        raise ValueError(f"the Hamiltonian acts on {hamiltonian.num_qubits} qubits, "
                         f"the state has {state.num_qubits}")
    return state.apply_pauli_rotations(x, z, angles)
