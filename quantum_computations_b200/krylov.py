"""Lanczos ground-state energies and Krylov time evolution under a Pauli sum, on device states.

Both methods run the Lanczos recurrence of a Hermitian Pauli sum H on the device and keep only the
tridiagonal matrix T on the host (numpy ``eigh`` on at most a few hundred rows).  No basis vector is
stored: a quantity that needs one (the ground-state vector, exp(-iHt)|psi>) comes from a second pass
that regenerates the same vectors bit for bit and accumulates the result on the way.  That is exact
because every reduction of the two kernels behind it uses a fixed grid and a fixed summation tree.

Write u_j for the buffer that holds v_j s_j, s_j a host scalar known at that point (s_0 = |psi|,
s_j = beta_j).  Iteration j is two calls, each ending in one synchronisation:

1. ``qsim_lanczos_apply``: out <- p prev + sum_t (c_t / s_j) P_t u_j with p = -beta_j / s_{j-1}, which
   also returns Re <u_j|out> = alpha_j s_j;
2. ``qsim_lanczos_step``: out <- out - (alpha_j / s_j) u_j, optionally y <- y + (b_j / s_j) u_j, which
   returns |out|^2 = beta_{j+1}^2; out is then u_{j+1}.

The caller's state is read (as ``in`` of iteration 0 and ``prev`` of iteration 1) but never written
during a pass, and two scratch buffers ping-pong after that.  Nothing normalises, copies or scales a
whole state: a ground energy needs three state buffers including the caller's, the ground-state
vector and time evolution four.
"""
from __future__ import annotations

import math

import numpy as np

from . import engine

MAX_SUBSTEP_DIM = 30          # Krylov dimension cap of one evolve_krylov substep
BREAKDOWN = 1e-14             # beta <= BREAKDOWN * |T|: an invariant subspace (happy breakdown)


def tridiagonal(alphas, betas) -> np.ndarray:
    """T_k of k alphas and the betas beta_1 .. beta_{k-1} (``betas[:k-1]``)."""
    k = len(alphas)
    t = np.diag(np.asarray(alphas, dtype=np.float64))
    if k > 1:
        off = np.asarray(betas[:k - 1], dtype=np.float64)
        t += np.diag(off, 1) + np.diag(off, -1)
    return t


class Recurrence:
    """The Lanczos recurrence of the real-coefficient Pauli sum (x, z, c) from the buffer ``start`` (of
    norm ``s0``) on 2^n_bits amplitudes, with the two scratch buffers ``work``."""

    def __init__(self, backend, n_bits: int, x, z, c, start, s0: float, work):
        self.be, self.n_bits = backend, int(n_bits)
        self.x = np.ascontiguousarray(x, dtype=np.uint64)
        self.z = np.ascontiguousarray(z, dtype=np.uint64)
        self.c = np.ascontiguousarray(c, dtype=np.complex128)
        self.start, self.s0, self.work = start, float(s0), work

    def _iterations(self, count, betas):
        """Yields (j, in, prev, out, s_j, p) for j < count; betas[j - 1] is beta_j, known when j runs."""
        cur, prev, out = self.start, None, self.work[0]
        s_prev = s = self.s0
        for j in range(count):
            p = -betas[j - 1] / s_prev if j else 0.0
            yield j, cur, prev, out, s, p
            s_prev, s = s, betas[j]
            prev, cur, out = cur, out, (self.work[1] if j == 0 else cur)

    def first_pass(self, max_dim: int, stop):
        """Runs until ``stop(alphas, betas)`` is true or ``max_dim`` iterations; returns the alphas and
        betas (betas[j] = beta_{j+1}).  ``stop`` sees every prefix."""
        alphas, betas = [], []
        na = 1 << self.n_bits
        for j, cur, prev, out, s, p in self._iterations(max_dim, betas):
            dot = engine.lanczos_apply(self.be, cur, prev, out, self.n_bits, self.x, self.z, self.c / s, p)
            alpha = dot / s
            beta = math.sqrt(max(engine.lanczos_step(self.be, out, cur, None, na, alpha / s), 0.0))
            alphas.append(alpha)
            betas.append(beta)
            if stop(alphas, betas):
                break
        return alphas, betas

    def second_pass(self, alphas, betas, y, coeffs):
        """Regenerates v_0 .. v_{m-1} (m = len(coeffs)) with the first pass's alphas and betas and
        adds y <- y + coeffs[j] v_j on the way.  Returns |y|^2 after the last update and the
        (alpha, beta) pairs the pass recomputed, which equal the first pass's bit for bit."""
        m = len(coeffs)
        na = 1 << self.n_bits
        again = []
        cur, s = self.start, self.s0
        for j, cur, prev, out, s, p in self._iterations(m - 1, betas):
            dot = engine.lanczos_apply(self.be, cur, prev, out, self.n_bits, self.x, self.z, self.c / s, p)
            b2 = engine.lanczos_step(self.be, out, cur, y, na, alphas[j] / s, coeffs[j] / s)
            again.append((dot / s, math.sqrt(max(b2, 0.0))))
        if m > 1:                       # the last vector is the buffer the last step wrote
            cur, s = out, betas[m - 2]
        norm2 = engine.lanczos_step(self.be, None, cur, y, na, 0.0, coeffs[m - 1] / s)
        return norm2, again


def _ket_view(state):
    return engine.DeviceState(state.backend, state.buf, state.n_bits, 1)


def _real_coeffs(hamiltonian) -> np.ndarray:
    if np.any(hamiltonian.coeffs.imag != 0):
        raise ValueError("the Hamiltonian has a coefficient with a nonzero imaginary part (not Hermitian)")
    return hamiltonian.coeffs.real


def ground_state(hamiltonian, state, *, tol: float = 1e-10, max_iter: int = 300, return_state: bool = False,
                 _passes=None):
    """See ``observables.ground_state``.  ``_passes``: a list that receives the first pass's
    (alphas, betas) and, with ``return_state``, the second pass's recomputed pairs (tests)."""
    if state.ndim != 1:
        raise ValueError("ground_state needs a ket; a density matrix has no ground-state vector")
    c = _real_coeffs(hamiltonian)
    if int(max_iter) < 1:
        raise ValueError("max_iter must be at least 1")
    be, n = state.backend, state.n_bits
    s0 = state.norm()
    if not s0 > 0.0:
        raise ValueError("the start state is zero")
    work = (be.empty(1 << n), be.empty(1 << n))
    rec = Recurrence(be, n, hamiltonian.x_masks, hamiltonian.z_masks, c, state.buf, s0, work)
    found = {}

    def stop(alphas, betas):
        theta, vecs = np.linalg.eigh(tridiagonal(alphas, betas))
        found.update(energy=float(theta[0]), residual=float(betas[-1] * abs(vecs[-1, 0])), vec=vecs[:, 0])
        scale = float(np.max(np.abs(theta)))
        return found["residual"] <= tol or betas[-1] <= BREAKDOWN * scale

    alphas, betas = rec.first_pass(int(max_iter), stop)
    if _passes is not None:
        _passes.append((alphas, betas))
    if not return_state:
        return found["energy"], found["residual"]
    y = be.empty(1 << n)
    y[...] = 0
    _norm2, again = rec.second_pass(alphas, betas, y, found["vec"])
    if _passes is not None:
        _passes.append(again)
    return found["energy"], found["residual"], engine.DeviceState(be, y, n, 1)


def _saad_error(theta, vecs, beta, dt) -> float:
    """beta_m |[exp(-i T_m dt)]_{m-1, 0}| (times |psi| by the caller) from T_m = vecs diag(theta) vecs^T."""
    return float(beta * abs(np.dot(vecs[-1, :] * np.exp(-1j * theta * dt), vecs[0, :])))


def evolve_krylov(hamiltonian, state, time: float, *, tol: float = 1e-12, _substeps=None):
    """See ``observables.evolve_krylov``.  ``_substeps``: a list that receives (m, dt) per substep
    (tests)."""
    from .observables import PauliSum
    c = _real_coeffs(hamiltonian)
    x, z = hamiltonian.x_masks, hamiltonian.z_masks
    if state.ndim == 2:
        # vec(e^{-iHt} rho e^{iHt}) = exp(-iLt) vec(rho), L = H (x) I - I (x) H^T on the 2N vec qubits
        op = PauliSum._from_masks(x, z, c, hamiltonian.num_qubits).liouvillian(state.num_qubits)
        x, z, c = op.x_masks, op.z_masks, op.coeffs.real
        phase = 0.0
    else:
        ident = (x == 0) & (z == 0)
        phase = float(c[ident].sum())               # the identity term: a global phase
        x, z, c = x[~ident], z[~ident], c[~ident]
    ket = _ket_view(state)
    be, n = ket.backend, ket.n_bits
    total = abs(float(time))
    sign = 1.0 if time >= 0 else -1.0
    if total == 0.0:
        return state
    s0 = ket.norm()
    if s0 == 0.0:
        return state
    work = (be.empty(1 << n), be.empty(1 << n))
    start, y = ket.buf, be.empty(1 << n)
    left = total
    while left > 0.0:
        rec = Recurrence(be, n, x, z, c, start, s0, work)
        seen = {}

        def stop(alphas, betas):
            theta, vecs = np.linalg.eigh(tridiagonal(alphas, betas))
            seen.update(theta=theta, vecs=vecs, beta=betas[-1])
            seen["exact"] = betas[-1] <= BREAKDOWN * float(np.max(np.abs(theta)))
            return seen["exact"] or s0 * _saad_error(theta, vecs, betas[-1], left) <= tol * left / total

        alphas, betas = rec.first_pass(MAX_SUBSTEP_DIM, stop)
        theta, vecs, beta = seen["theta"], seen["vecs"], seen["beta"]

        def fits(dt):
            return s0 * _saad_error(theta, vecs, beta, dt) <= tol * dt / total

        dt = left
        if not seen["exact"] and not fits(left):
            lo, hi = 0.0, left                       # the longest step whose error fits its share
            for _ in range(60):
                mid = 0.5 * (lo + hi)
                lo, hi = (mid, hi) if fits(mid) else (lo, mid)
            dt = lo
            if dt <= 0.0:
                raise RuntimeError("evolve_krylov: no substep meets the tolerance; raise tol")
        # y = s0 e^{-i phase dt} V_m exp(-i T_m dt) e_0
        coeffs = s0 * np.exp(-1j * sign * phase * dt) * (vecs @ (np.exp(-1j * sign * theta * dt) * vecs[0, :]))
        y[...] = 0
        norm2, _again = rec.second_pass(alphas, betas, y, coeffs)
        if _substeps is not None:
            _substeps.append((len(alphas), dt))
        s0 = math.sqrt(norm2)
        start, y = y, start
        left = left - dt if dt < left else 0.0
    if start is not ket.buf:
        ket.buf[...] = start                        # the one copy back into the caller's buffer
    state.host_dtype = np.dtype(np.complex128)
    return state
