"""State vectors larger than one GPU: shard by g qubits, exchange them in stages.

The reference has no distributed path at all (SURVEY.md section 2.1); this module
is what ``BASELINE.json`` configuration C5 (34 qubits over 8 B200s) needs.

Layout.  A register of ``n`` qubits over ``P = 2^g`` ranks: rank ``r`` holds the
``2^(n-g)`` amplitudes whose top ``g`` *physical* index bits equal ``r``.  Physical
bits ``0 .. n-g-1`` are local, bits ``n-g .. n-1`` are the rank number.  A table maps
every logical index bit (reference qubit ``q`` is logical bit ``n-1-q``) to the
physical bit it currently occupies, and every rank bit carries a *flip* flag: with
the flag set, rank bit value ``b`` stands for logical value ``1-b``.

Execution.  The circuit is cut into *stages*; inside a stage the set of rank qubits
is fixed and everything runs on the shard through the single-GPU fused planner:

* diagonal gates (Z, RZ, P, T, CZ, ...) never need communication: for the bits that
  live in the rank number the diagonal is restricted to this rank's values and
  becomes a smaller diagonal gate (or a scalar) on the shard;
* an antidiagonal single-qubit gate (X, Y, ...) on a rank qubit only relabels the
  ranks: the shard is scaled by one matrix entry and the flip flag toggles;
* any other gate on a rank qubit blocks, and so does whatever depends on it.  When
  nothing more can run, the next stage's rank qubits are chosen -- the ``g`` qubits
  whose next blocking gate lies farthest ahead -- and all of them trade places with
  local qubits in ONE all-to-all exchange: with ``k`` qubits moving, every rank keeps
  ``1/2^k`` of its shard and sends ``1/2^k`` to each of the ``2^k - 1`` ranks that
  differ in those rank bits (0.875 of a shard for k = 3, where three single swaps
  would move 1.5).  ``qsim_swap_pack`` / ``qsim_swap_unpack`` gather and scatter the
  travelling blocks; the transfer is a copy-engine push over NVLink (CUDA IPC) on
  GPUs and a send/recv elsewhere.  The first stage costs nothing: the initial product
  state is built directly in the layout the schedule wants.

``ShardedSimulator.run_circuit`` adds measurements, insertions and classical control
(``Simulator.run`` semantics); ``density=True`` shards a vectorised density matrix.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _capi, engine


def _is_diagonal(m: np.ndarray) -> bool:
    return not np.any(m - np.diag(np.diagonal(m)))


class Comm:
    """Thin wrapper over ``torch.distributed`` point-to-point exchange of
    complex128 buffers (moved as float64 pairs so gloo works too)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.size = dist.get_world_size(group)
        if self.size & (self.size - 1):
            raise ValueError("the number of ranks must be a power of two")
        self.bytes_exchanged = 0

    def exchange(self, send_t, recv_t, partner: int) -> None:
        """Send ``send_t`` to and receive ``recv_t`` from ``partner`` (torch tensors)."""
        import torch
        dist = self.dist
        s = torch.view_as_real(send_t) if send_t.is_complex() else send_t
        r = torch.view_as_real(recv_t) if recv_t.is_complex() else recv_t
        ops = [dist.P2POp(dist.isend, s, partner, self.group), dist.P2POp(dist.irecv, r, partner, self.group)]
        for req in dist.batch_isend_irecv(ops):
            req.wait()
        self.bytes_exchanged += s.numel() * s.element_size()

    def allgather_object(self, obj) -> list:
        out = [None] * self.size
        self.dist.all_gather_object(out, obj, group=self.group)
        return out

    def allreduce_sum(self, values: np.ndarray) -> np.ndarray:
        import torch
        t = torch.from_numpy(np.ascontiguousarray(values, dtype=np.float64))
        dev = getattr(self, "device", None)
        if dev is not None:
            t = t.to(dev)
        self.dist.all_reduce(t, group=self.group)
        return t.cpu().numpy()


class ShardedState:
    """One rank's shard plus the logical->physical bit table (same on all ranks)."""

    def __init__(self, n: int, comm: Comm, backend=None, as_torch=None, buf=None):
        self.n = int(n)
        self.comm = comm
        self.g = comm.size.bit_length() - 1
        if self.g >= self.n:
            raise ValueError("more ranks than amplitudes")
        self.n_local = self.n - self.g
        self.backend = backend or engine.get_backend()
        self.phys = list(range(self.n))           # phys[logical bit] = physical bit
        self.flip = [0] * self.g                  # flip[i]: rank bit i holds the complemented logical value
        self.buf = self.backend.empty(1 << self.n_local) if buf is None else buf
        self.swaps = 0
        self.swap_seconds = 0.0
        self.amps_sent = 0
        self._peer = None
        self._p2p = None                          # peers' shards mapped through CUDA IPC (fused exchange)
        self._swap_events = []                    # CUDA event pairs of the fused exchanges (timed lazily)
        self.is_density = False                   # set by ShardedSimulator(density=True): vec(rho), 2N bits
        # how to view a backend buffer as a torch tensor for the communicator
        self._as_torch = as_torch or (lambda b: b)

    # -- initial states ---------------------------------------------------------------------
    def rank_value(self, phys_bit: int) -> int:
        """Logical value this rank holds for the qubit living in rank bit ``phys_bit``."""
        i = phys_bit - self.n_local
        return ((self.comm.rank >> i) & 1) ^ self.flip[i]

    def set_product(self, vectors, phys=None) -> None:
        """|psi> = kron of single-qubit kets (qubit 0 first), laid out as ``phys``
        (default: identity).  The rank bits select one amplitude of each rank qubit's
        ket: a scalar on this rank."""
        vecs = [np.asarray(v, dtype=np.complex128) for v in vectors]
        assert len(vecs) == self.n
        self.phys = list(phys) if phys is not None else list(range(self.n))
        assert sorted(self.phys) == list(range(self.n))
        self.flip = [0] * self.g
        where = {p: l for l, p in enumerate(self.phys)}            # physical bit -> logical bit
        scale = 1.0 + 0.0j
        for p in range(self.n_local, self.n):
            scale *= vecs[self.n - 1 - where[p]][self.rank_value(p)]
        # local reference-style qubit j of the shard is physical bit n_local-1-j
        local = [vecs[self.n - 1 - where[self.n_local - 1 - j]].copy() for j in range(self.n_local)]
        local[0] = local[0] * scale
        amps = np.ascontiguousarray(np.stack(local))
        be = self.backend
        _capi.check(be.lib, be.lib.qsim_init_product(
            be.ptr(self.buf), self.n_local, amps.view(np.float64).ctypes.data_as(_capi.c_double_p), be.stream()))

    # -- reductions ---------------------------------------------------------------------------
    def norm(self) -> float:
        be = self.backend
        out = np.zeros(2)
        _capi.check(be.lib, be.lib.qsim_reduce_norm2(be.ptr(self.buf), C.c_uint64(1 << self.n_local),
                                                     out.ctypes.data_as(_capi.c_double_p), be.stream()))
        return float(np.sqrt(self.comm.allreduce_sum(out[:1])[0]))

    def inner(self, other: "ShardedState") -> complex:
        """<self|other> (conjugate-linear in self): local reduction + all-reduce of two doubles.
        Both states must be in the same layout (same schedule, or both freshly prepared alike)."""
        if other.n != self.n or other.phys != self.phys or other.flip != self.flip:
            raise ValueError("the two sharded states are laid out differently")
        be = self.backend
        out = np.zeros(2)
        _capi.check(be.lib, be.lib.qsim_reduce_inner(be.ptr(self.buf), be.ptr(other.buf), C.c_uint64(1 << self.n_local),
                                                     out.ctypes.data_as(_capi.c_double_p), be.stream()))
        total = self.comm.allreduce_sum(out)
        return complex(total[0], total[1])

    def fidelity(self, other: "ShardedState") -> float:
        """|<self|other>|^2 (npq.fidelity, ket-ket branch, DV/numpy_quantum.py:148-161)."""
        return abs(self.inner(other)) ** 2

    # -- observables ---------------------------------------------------------------------------
    def expect_pauli(self, x_masks, z_masks) -> np.ndarray:
        """<P_t> of Pauli strings (bit q of the masks = reference qubit q, operator
        i^popc(x & z) X^x Z^z) as a float64 array; a collective, identical on every rank.

        Z factors on rank qubits become a per-rank sign (the logical value, flip flags
        included).  X/Y factors must be local: rank qubits in an X support are first traded,
        in one exchange, against local qubits outside every X support still to evaluate
        (a string whose X/Y support does not fit in a shard is refused).  Every rank evaluates
        its shard with ``qsim_expect_pauli`` and the per-term vector is all-reduced once.  The
        logical state is unchanged; the layout may differ afterwards (``phys`` / ``flip``
        record it, so ``gather_numpy`` and later schedules see the same state)."""
        if self.is_density:
            raise NotImplementedError("Pauli expectation values of a sharded density matrix are not implemented")
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        if x.shape != z.shape:
            raise ValueError("x_masks and z_masks must have the same length")
        n = self.n
        if len(x) and (int(x.max()) >> n or int(z.max()) >> n):
            raise ValueError("a Pauli mask has a bit at or above the number of qubits")
        # logical bit l = n-1-q of reference qubit q
        xs = [{n - 1 - q for q in range(n) if int(v) >> q & 1} for v in x]
        zs = [{n - 1 - q for q in range(n) if int(v) >> q & 1} for v in z]
        values = np.zeros(len(x), dtype=np.float64)
        remaining = list(range(len(x)))
        while remaining:
            chosen, support = self._next_batch(remaining, xs)
            self._localise(support)
            self._expect_local(sorted(chosen), x, xs, zs, values)
            done = set(chosen)
            remaining = [t for t in remaining if t not in done]
        return self.comm.allreduce_sum(values)

    def _next_batch(self, remaining, xs):
        """The terms of ``remaining`` (order free: they commute) that one ``_localise`` can serve: those
        whose X support is local already, then any whose support still fits; and their joint support."""
        n = self.n
        is_local = lambda bits: all(self.phys[l] < self.n_local for l in bits)   # noqa: E731
        chosen = [t for t in remaining if is_local(xs[t])]
        support = set().union(*[xs[t] for t in chosen])
        for t in remaining:
            if t in chosen:
                continue
            wider = support | xs[t]
            need = [l for l in wider if self.phys[l] >= self.n_local]
            free = [l for l in range(n) if self.phys[l] < self.n_local and l not in wider]
            if len(need) <= len(free):
                chosen.append(t)
                support = wider
        if not chosen:
            raise NotImplementedError("a Pauli string's X/Y support is wider than a shard; use fewer ranks")
        return chosen, support

    def _pauli_args(self, x_masks, z_masks, values, what: str):
        """Checks the masks of a collective Pauli call against ``values`` (its coefficients or angles) and
        returns the logical bits of every X and Z mask (logical bit l = n-1-q of reference qubit q)."""
        if self.is_density:
            raise NotImplementedError(f"{what} of a sharded density matrix are not implemented")
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        if x.shape != z.shape or x.shape != values.shape:
            raise ValueError("the masks and the coefficients or angles must have the same length")
        n = self.n
        if len(x) and (int(x.max()) >> n or int(z.max()) >> n):
            raise ValueError("a Pauli mask has a bit at or above the number of qubits")
        xs = [{n - 1 - q for q in range(n) if int(v) >> q & 1} for v in x]
        zs = [{n - 1 - q for q in range(n) if int(v) >> q & 1} for v in z]
        return xs, zs

    def _local_masks(self, terms, xs, zs):
        """Shard masks of ``terms`` (X supports local) and the sign (-1)^v that their Z factors on rank
        qubits contribute on this rank, v the logical values (flip flags included)."""
        nl = self.n_local
        lx = np.zeros(len(terms), dtype=np.uint64)
        lz = np.zeros(len(terms), dtype=np.uint64)
        sign = np.ones(len(terms))
        for k, t in enumerate(terms):
            for l in xs[t]:
                lx[k] |= np.uint64(1 << (nl - 1 - self.phys[l]))         # shard reference qubit
            for l in zs[t]:
                p = self.phys[l]
                if p < nl:
                    lz[k] |= np.uint64(1 << (nl - 1 - p))
                elif self.rank_value(p):
                    sign[k] = -sign[k]
        return lx, lz, sign

    def empty_like(self, buf=None) -> "ShardedState":
        """A state of the same kind (ket or vec of a density matrix), register and ranks in the same
        layout (``phys`` / ``flip``) on ``buf`` (default: a new shard, uninitialised)."""
        out = ShardedState(self.n, self.comm, self.backend, self._as_torch, buf)
        out.phys, out.flip = list(self.phys), list(self.flip)
        out.is_density = self.is_density
        return out

    def copy(self) -> "ShardedState":
        return self.empty_like(self.backend.clone(self.buf))

    def apply_pauli_sum(self, x_masks, z_masks, coeffs) -> "ShardedState":
        """H|psi> with H = sum_t coeffs[t] P_t (``engine.DeviceState.apply_pauli_sum``) as a new sharded
        ket; a collective.  This state is logically unchanged (its layout may change, as in
        ``expect_pauli``); the result ends in the same layout.

        Terms are taken in batches that one ``_localise`` serves, with this state and the result
        localised in lockstep.  A Z factor on a rank qubit becomes a sign on the coefficient.  The first
        batch is written by ``qsim_apply_pauli_sum``, every later one is added to the result in place by
        ``qsim_accumulate_pauli_sum``."""
        c = np.ascontiguousarray(coeffs, dtype=np.complex128).reshape(-1)
        xs, zs = self._pauli_args(x_masks, z_masks, c, "Pauli sums")
        if not np.all(np.isfinite(c)):
            raise ValueError("non-finite coefficient")
        be = self.backend
        out = None
        remaining = list(range(len(c)))
        while out is None or remaining:
            chosen, support = self._next_batch(remaining, xs) if remaining else ([], set())
            self._localise(support)
            if out is None:
                out = self.empty_like()
                fn = be.lib.qsim_apply_pauli_sum
            else:
                out._localise(support)
                fn = be.lib.qsim_accumulate_pauli_sum
            terms = sorted(chosen)
            lx, lz, sign = self._local_masks(terms, xs, zs)
            lc = np.ascontiguousarray(c[terms] * sign, dtype=np.complex128)
            _capi.check(be.lib, fn(be.ptr(self.buf), be.ptr(out.buf), self.n_local, len(terms), lx.ctypes.data,
                                   lz.ctypes.data, lc.ctypes.data, be.stream()))
            done = set(chosen)
            remaining = [t for t in remaining if t not in done]
        return out

    def pauli_rotations_adjoint(self, lam: "ShardedState", x_masks, z_masks, angles) -> np.ndarray:
        """The adjoint sweep (``engine.DeviceState.pauli_rotations_adjoint``) on this ket (psi = U psi0
        on entry, psi0 on return) and ``lam`` (U^dagger lam on return), a collective; returns
        Im<lam_t|P_t|psi_t> for every rotation in caller order, identical on every rank.

        ``lam`` must be laid out as this state (``inner`` accepts the pair).  The rotations are cut,
        from the last one back, into runs whose joint X/Y support fits in a shard; both states are made
        local in lockstep (``_localise`` is deterministic) and swept with one
        ``qsim_pauli_rotations_adjoint`` call per run.  A Z factor on a rank qubit negates the angle and
        the overlap where its logical value is 1.  The gradients are all-reduced once."""
        a = np.ascontiguousarray(angles, dtype=np.float64).reshape(-1)
        xs, zs = self._pauli_args(x_masks, z_masks, a, "Pauli rotations")
        if lam.n != self.n or lam.phys != self.phys or lam.flip != self.flip:
            raise ValueError("psi and lam are laid out differently")
        if not np.all(np.isfinite(a)):
            raise ValueError("non-finite angle")
        if any(len(s) > self.n_local for s in xs):
            raise NotImplementedError("a Pauli string's X/Y support is wider than a shard; use fewer ranks")
        n, be = self.n, self.backend
        grads = np.zeros(len(a), dtype=np.float64)
        end = len(a)
        while end > 0:
            support, start = set(xs[end - 1]), end - 1
            while start > 0:
                wider = support | xs[start - 1]
                need = [l for l in wider if self.phys[l] >= self.n_local]
                free = [l for l in range(n) if self.phys[l] < self.n_local and l not in wider]
                if len(need) > len(free):
                    break
                support, start = wider, start - 1
            self._localise(support)
            lam._localise(support)
            run = list(range(start, end))
            lx, lz, sign = self._local_masks(run, xs, zs)
            la = np.ascontiguousarray(a[run] * sign)
            out = np.zeros(len(run), dtype=np.float64)
            _capi.check(be.lib, be.lib.qsim_pauli_rotations_adjoint(
                be.ptr(self.buf), be.ptr(lam.buf), self.n_local, len(run), lx.ctypes.data, lz.ctypes.data,
                la.ctypes.data, out.ctypes.data, be.stream()))
            grads[start:end] = sign * out
            end = start
        return self.comm.allreduce_sum(grads)

    def expect(self, observable, per_term: bool = False):
        """``observables.expect`` on this sharded ket (collective)."""
        from .observables import expect
        return expect(observable, self, per_term=per_term)

    def apply_pauli_rotations(self, x_masks, z_masks, angles) -> "ShardedState":
        """In place, collective: the ket becomes R_{k-1} ... R_0 |psi> with R_t = exp(-i angles[t]/2 P_t)
        (``engine.DeviceState.apply_pauli_rotations``).  Returns ``self``.

        The rotations are cut, in order, into runs whose joint X/Y support fits in a shard; each run
        is made local with one exchange (``_localise``) and applied with one
        ``qsim_apply_pauli_rotations`` call.  A Z factor on a rank qubit acts as the scalar (-1)^v on
        this shard, v its logical value (flip flags included), so it leaves the shard's mask and
        negates the angle where v = 1.  A string whose X/Y support does not fit in a shard is refused.
        The layout may differ afterwards (``phys`` / ``flip`` record it)."""
        if self.is_density:
            raise NotImplementedError("Pauli rotations of a sharded density matrix are not implemented")
        x = np.ascontiguousarray(x_masks, dtype=np.uint64).reshape(-1)
        z = np.ascontiguousarray(z_masks, dtype=np.uint64).reshape(-1)
        a = np.ascontiguousarray(angles, dtype=np.float64).reshape(-1)
        if x.shape != z.shape or x.shape != a.shape:
            raise ValueError("x_masks, z_masks and angles must have the same length")
        n = self.n
        if len(x) and (int(x.max()) >> n or int(z.max()) >> n):
            raise ValueError("a Pauli mask has a bit at or above the number of qubits")
        if not np.all(np.isfinite(a)):
            raise ValueError("non-finite angle")
        xs = [{n - 1 - q for q in range(n) if int(v) >> q & 1} for v in x]
        zs = [{n - 1 - q for q in range(n) if int(v) >> q & 1} for v in z]
        if any(len(s) > self.n_local for s in xs):
            raise NotImplementedError("a Pauli string's X/Y support is wider than a shard; use fewer ranks")
        start = 0
        while start < len(x):
            support, end = set(xs[start]), start + 1
            while end < len(x):
                wider = support | xs[end]
                need = [l for l in wider if self.phys[l] >= self.n_local]
                free = [l for l in range(n) if self.phys[l] < self.n_local and l not in wider]
                if len(need) > len(free):
                    break
                support, end = wider, end + 1
            self._localise(support)
            self._rotate_local(range(start, end), xs, zs, a)
            start = end
        return self

    def _rotate_local(self, run, xs, zs, angles) -> None:
        """The rotations ``run`` (X supports local) on this shard, Z factors on rank qubits as signs."""
        run = list(run)
        lx, lz, sign = self._local_masks(run, xs, zs)
        la = np.ascontiguousarray(angles[run] * sign)
        be = self.backend
        _capi.check(be.lib, be.lib.qsim_apply_pauli_rotations(be.ptr(self.buf), self.n_local, len(run), lx.ctypes.data,
                                                              lz.ctypes.data, la.ctypes.data, be.stream()))

    def _localise(self, support) -> None:
        """Make the logical bits in ``support`` local with one exchange against the highest
        local bits outside it.  A bit that arrives complemented (its rank bit carried the flip
        flag) is put right with an X on the shard, and the flag is cleared, so that the layout
        tables describe the same logical state as before."""
        need = sorted((l for l in support if self.phys[l] >= self.n_local), key=lambda l: self.phys[l])
        if not need:
            return
        free = sorted((l for l in range(self.n) if self.phys[l] < self.n_local and l not in support),
                      key=lambda l: -self.phys[l])
        pairs = [(self.phys[a], self.phys[b]) for a, b in zip(need, free)]
        complemented = []
        for gp, lp in pairs:
            i = gp - self.n_local
            if self.flip[i]:
                complemented.append(lp)            # the arriving bit lands on physical bit lp
                self.flip[i] = 0
        self.exchange(pairs)
        if complemented:
            x_gate = np.array([[0, 1], [1, 0]], dtype=np.complex128)
            ops = [([self.n_local - 1 - lp], x_gate) for lp in complemented]
            engine.Plan(self.backend, self.n_local, ops).execute(self.buf)

    def _expect_local(self, terms, x, xs, zs, values) -> None:
        """values[t] += this rank's share of <P_t> for terms whose X support is local."""
        lx, lz, sign = self._local_masks(terms, xs, zs)
        be = self.backend
        out = np.zeros(len(terms), dtype=np.float64)
        _capi.check(be.lib, be.lib.qsim_expect_pauli(be.ptr(self.buf), self.n_local, len(terms), lx.ctypes.data, lz.ctypes.data,
                                                     out.ctypes.data_as(_capi.c_double_p), be.stream()))
        values[terms] += sign * out

    # -- measurement statistics -----------------------------------------------------------------
    def probabilities(self, qubits=None) -> np.ndarray:
        """Marginal distribution over ``qubits`` (default: all; ``qubits[0]`` the most significant
        bit of the bin number), float64, not normalised; a collective, identical on every rank.

        The local qubits of the set go to ``qsim_marginal_probs`` on the shard (in shard
        numbering); the shard's bins are placed at this rank's logical values of the set's rank
        qubits (flip flags included) and the 2^k vector is all-reduced once.  No exchange."""
        if self.is_density:
            raise NotImplementedError("marginals of a sharded density matrix are not implemented")
        n, nl = self.n, self.n_local
        q = engine._qubit_list(qubits, n)
        k = len(q)
        local_j = [j for j, v in enumerate(q) if self.phys[n - 1 - v] < nl]
        shard_q = [nl - 1 - self.phys[n - 1 - q[j]] for j in local_j]
        part = np.asarray(self.backend.download(engine.marginal_probs(self.backend, self.buf, nl, shard_q)))
        fixed = 0
        for j, v in enumerate(q):
            p = self.phys[n - 1 - v]
            if p >= nl and self.rank_value(p):
                fixed |= 1 << (k - 1 - j)
        m = len(local_j)
        loc = np.arange(1 << m, dtype=np.int64)
        bins = np.full(1 << m, fixed, dtype=np.int64)
        for i, j in enumerate(local_j):
            bins |= ((loc >> (m - 1 - i)) & 1) << (k - 1 - j)
        full = np.zeros(1 << k, dtype=np.float64)
        full[bins] = part
        return self.comm.allreduce_sum(full)

    def sample(self, shots: int, qubits=None, rng=None) -> np.ndarray:
        """``shots`` outcomes over ``qubits`` (default: all; ``qubits[0]`` the most significant
        bit) as int64; a collective, identical on every rank.

        Rank 0 draws the uniforms (``rng.random(shots)``; ``rng`` a Generator, a seed or None) and
        shares them.  The ranks all-gather their shard totals; a shot goes to the rank whose slice
        of the global CDF holds u * total (ranks in rank order, strict ``>``, so a rank without
        mass gets none), is rescaled to that shard and sampled there with ``qsim_sample``, and the
        physical index is mapped to the logical one through ``phys`` and ``flip``.  One reduction
        of the outcome vector completes the call.  The outcomes therefore equal inverse-CDF
        sampling over the state in rank-major physical order (rank number, then the shard's
        index), up to shots within rounding of a boundary; their distribution is the logical one."""
        if self.is_density:
            raise NotImplementedError("sampling a sharded density matrix is not implemented")
        n, nl, size, rank = self.n, self.n_local, self.comm.size, self.comm.rank
        q = engine._qubit_list(qubits, n)
        shots = int(shots)
        u = None
        if rank == 0:
            gen = rng if isinstance(rng, np.random.Generator) else np.random.default_rng(rng)
            u = gen.random(shots)
        u = self.comm.allgather_object(u)[0]
        mass = float(np.asarray(self.backend.download(engine.marginal_probs(self.backend, self.buf, nl, [])))[0])
        totals = np.array(self.comm.allgather_object(mass), dtype=np.float64)
        cum = np.cumsum(totals)
        if not cum[-1] > 0:
            raise ValueError("the state has no probability mass")
        target = u * cum[-1]
        owner = np.searchsorted(cum, target, side="right")
        owner[owner >= size] = max(r for r in range(size) if totals[r] > 0)
        outcomes = np.zeros(shots, dtype=np.float64)
        mine = np.nonzero(owner == rank)[0]
        if len(mine):
            start = cum[rank - 1] if rank else 0.0
            local_u = np.clip((target[mine] - start) / totals[rank], 0.0, np.nextafter(1.0, 0.0))
            idx, _ = engine.sample_indices(self.backend, self.buf, nl, local_u)
            outcomes[mine] = engine.project_outcomes(self._logical_indices(idx), n, q)
        return self.comm.allreduce_sum(outcomes).astype(np.int64)

    def _logical_indices(self, local_idx: np.ndarray) -> np.ndarray:
        """Shard indices of this rank -> logical basis indices (``phys`` and ``flip``)."""
        out = np.zeros(len(local_idx), dtype=np.int64)
        for l in range(self.n):
            p = self.phys[l]
            bit = (local_idx >> p) & 1 if p < self.n_local else np.int64(self.rank_value(p))
            out |= bit << l
        return out

    # -- swaps -----------------------------------------------------------------------------------
    import os as _os
    # amplitudes per pipeline chunk: 512 MiB measured best (614 GB/s per direction on two B200s;
    # 580 at 256 MiB, 557 at 1 GiB, 539 at 2 GiB)
    CHUNK_LOG2 = int(_os.environ.get("QSIM_SWAP_CHUNK_LOG2", "25"))

    def _peer_setup(self, chunk: int):
        """Allocate the four staging chunks with the library (plain cudaMalloc, so they can be
        exported through CUDA IPC) and open every other rank's receive chunks once."""
        be, lib = self.backend, self.backend.lib
        if self._peer is not None and self._peer["chunk"] == chunk:
            return self._peer
        if self._peer is not None:                # another chunk size: give the old staging back first
            p2p = self._p2p
            self._p2p = None
            self.close()
            self._p2p = p2p
        use_ipc = getattr(be, "name", "") == "cuda" and os.environ.get("QSIM_SWAP_IPC", "1") != "0"
        peer = {"chunk": chunk, "ipc": use_ipc}
        if not use_ipc:
            peer["send"] = [be.empty(chunk) for _ in range(2)]
            peer["recv"] = [be.empty(chunk) for _ in range(2)]
            self._peer = peer
            return peer
        import torch
        dev = be.device.index
        ptrs = []
        for _ in range(4):
            out = C.c_void_p()
            _capi.check(lib, lib.qsim_peer_alloc(dev, C.c_uint64(16 * chunk), C.byref(out)))
            ptrs.append(out.value)
        peer["send_ptr"], peer["recv_ptr"] = ptrs[:2], ptrs[2:]
        handles = []
        for p in peer["recv_ptr"]:
            h = C.create_string_buffer(64)
            _capi.check(lib, lib.qsim_ipc_export(C.c_void_p(p), h))
            handles.append(h.raw)
        gathered = [None] * self.comm.size
        self.comm.dist.all_gather_object(gathered, handles, group=self.comm.group)
        peer["remote_recv"] = {}
        for r, hs in enumerate(gathered):
            if r == self.comm.rank:
                continue
            opened = []
            for h in hs:
                out = C.c_void_p()
                _capi.check(lib, lib.qsim_ipc_import(dev, h, C.byref(out)))
                opened.append(out.value)
            peer["remote_recv"][r] = opened
        peer["token_out"] = torch.zeros(2, dtype=torch.float64, device=be.device)
        peer["token_in"] = torch.zeros(2, dtype=torch.float64, device=be.device)
        self._peer = peer
        return peer

    # -- fused exchange over NVLink peer memory (GPUs) ---------------------------------------------
    def _use_fused(self, block: int) -> bool:
        return (getattr(self.backend, "name", "") == "cuda" and os.environ.get("QSIM_SWAP_FUSED", "1") != "0"
                and os.environ.get("QSIM_SWAP_IPC", "1") != "0" and block >= 64)

    def _p2p_setup(self):
        """Map every other rank's shard into this process (CUDA IPC), once per shard buffer."""
        be, lib = self.backend, self.backend.lib
        key = (be.ptr(self.buf), self.n_local)
        if self._p2p is not None and self._p2p["key"] == key:
            return self._p2p
        self._p2p_release()
        import torch
        h = C.create_string_buffer(64)
        off = C.c_uint64(0)
        _capi.check(lib, lib.qsim_ipc_export_ex(C.c_void_p(key[0]), h, C.byref(off)))
        gathered = self.comm.allgather_object((h.raw, int(off.value), key[1]))
        if any(item[2] != self.n_local for item in gathered):
            raise RuntimeError("the ranks disagree on the shard size")
        shards, opened = {}, []
        for r, (handle, offset, _nl) in enumerate(gathered):
            if r == self.comm.rank:
                continue
            out = C.c_void_p()
            _capi.check(lib, lib.qsim_ipc_import(be.device.index, handle, C.byref(out)))
            opened.append(out.value)
            shards[r] = out.value + offset
        self._p2p = {"key": key, "shards": shards, "opened": opened,
                     "token": torch.zeros(1, dtype=torch.float32, device=be.device)}
        return self._p2p

    def _p2p_release(self):
        p2p, self._p2p = self._p2p, None
        if p2p is None:
            return
        self.backend.synchronize()
        for ptr in p2p["opened"]:
            self.backend.lib.qsim_ipc_release(C.c_void_p(ptr))

    def _rank_barrier(self, token) -> None:
        """Stream-ordered barrier over the ranks: a one-element all-reduce on the compute stream."""
        self.comm.dist.all_reduce(token, group=self.comm.group)

    def _exchange_fused(self, pairs, gis, qubits, mine, block: int) -> None:
        """The whole exchange as one kernel per rank (``qsim_exchange_p2p``): gather, NVLink
        transfer and scatter fused, in place in both shards, bracketed by two stream-ordered
        barriers.  Nothing here synchronises the host."""
        import torch
        be, lib = self.backend, self.backend.lib
        k = len(pairs)
        p2p = self._p2p_setup()
        peers = (C.c_void_p * (1 << k))()
        lower = (C.c_int * (1 << k))()
        for d in range(1, 1 << k):
            partner = self.comm.rank
            for i in range(k):
                partner ^= ((d >> i) & 1) << gis[i]
            peers[d] = p2p["shards"][partner]
            lower[d] = 1 if partner < self.comm.rank else 0
        my_bits = (C.c_int * k)(*mine)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self._rank_barrier(p2p["token"])           # every rank has finished the passes before the exchange
        ev0.record()                               # (waiting for the slowest rank's passes is not exchange time)
        _capi.check(lib, lib.qsim_exchange_p2p(be.ptr(self.buf), peers, self.n_local, k, qubits, my_bits, lower,
                                               be.stream()))
        self._rank_barrier(p2p["token"])           # every rank's kernel is done: the shards are whole again
        ev1.record()
        self._swap_events.append((ev0, ev1))
        self.swaps += 1
        self.amps_sent += ((1 << k) - 1) * block
        self.comm.bytes_exchanged += 16 * ((1 << k) - 1) * block
        for gp, lp in pairs:
            la, lb = self.phys.index(gp), self.phys.index(lp)
            self.phys[la], self.phys[lb] = lp, gp

    def collect_swap_time(self) -> float:
        """Fold the device time of the fused exchanges issued so far into ``swap_seconds``
        (synchronises)."""
        if self._swap_events:
            self.backend.synchronize()
            for ev0, ev1 in self._swap_events:
                self.swap_seconds += 1e-3 * ev0.elapsed_time(ev1)
            self._swap_events = []
        return self.swap_seconds

    def close(self) -> None:
        """Release the peer mappings and the staging buffers of the exchanges."""
        self._p2p_release()
        peer, self._peer = self._peer, None
        if peer is not None and peer.get("ipc"):
            lib = self.backend.lib
            self.backend.synchronize()
            for opened in peer.get("remote_recv", {}).values():
                for ptr in opened:
                    lib.qsim_ipc_release(C.c_void_p(ptr))
            for ptr in peer.get("send_ptr", []) + peer.get("recv_ptr", []):
                lib.qsim_peer_free(C.c_void_p(ptr))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def swap(self, global_phys: int, local_phys: int) -> None:
        """Exchange one rank bit with one local bit (half a shard travels)."""
        self.exchange([(global_phys, local_phys)])

    def exchange(self, pairs) -> None:
        """Exchange the physical rank bits with the physical local bits of ``pairs``
        (``[(global_phys, local_phys), ...]``), all at once.

        With k pairs the 2^k ranks that differ in those rank bits form a group; in round
        d = 1 .. 2^k-1 every rank trades one block of 2^(n_local-k) amplitudes with the
        partner whose rank bits differ by the pattern d: it sends the block whose k local
        bits spell the partner's rank bits and receives into the same positions.  Blocks
        are cut into chunks that flow through a three-stage pipeline on three streams:
        gather (``qsim_swap_pack``) into a staging chunk, transfer, scatter
        (``qsim_swap_unpack``).  On GPUs the transfer is a copy-engine PUSH into the
        partner's staging chunk over NVLink (CUDA IPC + ``qsim_peer_copy``), fenced on both
        sides by tiny stream-ordered NCCL token exchanges with that partner, so no SM is
        spent on communication; elsewhere (gloo tests) it is a send/recv.  Flip flags are
        the caller's business: the bits move as stored."""
        import time
        be, lib = self.backend, self.backend.lib
        k = len(pairs)
        if k == 0:
            return
        gis = [gp - self.n_local for gp, _lp in pairs]                 # bits of the rank number
        if len(set(gis)) != k or len({lp for _gp, lp in pairs}) != k or \
                any(not 0 <= gi < self.g for gi in gis) or any(not 0 <= lp < self.n_local for _gp, lp in pairs):
            raise ValueError("exchange: bad bit pairs")
        qubits = (C.c_int * k)(*[self.n_local - 1 - lp for _gp, lp in pairs])   # local reference-style numbers
        mine = [(self.comm.rank >> gi) & 1 for gi in gis]
        block = 1 << (self.n_local - k)
        chunk = min(block, 1 << self.CHUNK_LOG2)
        per_block = block // chunk
        items = []                                   # (partner, bit values of the travelling block, first)
        for d in range(1, 1 << k):
            partner = self.comm.rank
            vals = []
            for i in range(k):
                di = (d >> i) & 1
                partner ^= di << gis[i]
                vals.append(mine[i] ^ di)
            for c in range(per_block):
                items.append((partner, (C.c_int * k)(*vals), c * chunk))
        if self._use_fused(block):
            self._exchange_fused(pairs, gis, qubits, mine, block)
            return
        peer = self._peer_setup(chunk)
        ipc = peer["ipc"]
        be.synchronize()                           # so the timer below sees the exchange alone
        t0 = time.perf_counter()
        if ipc:
            send_ptr, recv_ptr = peer["send_ptr"], peer["recv_ptr"]
        else:
            send_ptr = [be.ptr(b) for b in peer["send"]]
            recv_ptr = [be.ptr(b) for b in peer["recv"]]
        pipe = be.pipeline(3)                      # stream contexts + events (no-ops on the host emulator)
        packed, moved, unpacked = {}, {}, {}

        def token(partner):                        # both ranks have reached this point of their comm streams
            self.comm.exchange(peer["token_out"], peer["token_in"], partner)

        def pack(c):
            _partner, vals, first = items[c]
            with pipe.stage(0):
                if c >= 2:
                    pipe.wait(moved[c - 2])        # send[c%2] has left (our own push / send of item c-2)
                _capi.check(lib, lib.qsim_swap_pack(be.ptr(self.buf), C.c_void_p(send_ptr[c % 2]), self.n_local,
                                                    k, qubits, vals, C.c_uint64(first), C.c_uint64(chunk),
                                                    be.stream()))
                packed[c] = pipe.record()

        def unpack(c):
            _partner, vals, first = items[c]
            with pipe.stage(2):
                pipe.wait(moved[c])
                _capi.check(lib, lib.qsim_swap_unpack(be.ptr(self.buf), C.c_void_p(recv_ptr[c % 2]), self.n_local,
                                                      k, qubits, vals, C.c_uint64(first), C.c_uint64(chunk),
                                                      be.stream()))
                unpacked[c] = pipe.record()

        for c, (partner, _vals, _first) in enumerate(items):
            pack(c)
            with pipe.stage(1):
                pipe.wait(packed[c])
                if c >= 2:
                    pipe.wait(unpacked[c - 2])     # our recv[c%2] is free again
                if ipc:
                    # first token: both items c are packed and both recv[c%2] are free -> PUSH ours
                    # into the partner's staging with the copy engine (writes are the fast
                    # direction of NVLink P2P); second token: both pushes have landed
                    token(partner)
                    _capi.check(lib, lib.qsim_peer_copy(C.c_void_p(peer["remote_recv"][partner][c % 2]),
                                                        C.c_void_p(send_ptr[c % 2]),
                                                        C.c_uint64(16 * chunk), be.stream()))
                    token(partner)
                    self.comm.bytes_exchanged += 16 * chunk
                else:
                    self.comm.exchange(self._as_torch(peer["send"][c % 2]), self._as_torch(peer["recv"][c % 2]),
                                       partner)
                moved[c] = pipe.record()
            unpack(c)
        pipe.join()
        be.synchronize()
        self.swap_seconds += time.perf_counter() - t0
        self.swaps += 1
        self.amps_sent += len(items) * chunk
        # the logical bits trade places (flip flags stay with the rank bits)
        for gp, lp in pairs:
            la, lb = self.phys.index(gp), self.phys.index(lp)
            self.phys[la], self.phys[lb] = lp, gp

    # -- measurement and insertion (DV/gates.py:145-186 on a sharded ket) ----------------------------
    def _make_local(self, logical: int) -> bool:
        """Bring a rank qubit into the shard (one single-qubit exchange with the top local bit).
        Returns True when the qubit arrives complemented (its rank bit carried the flip flag;
        the flag is cleared, the new occupant of the rank bit is stored as it is)."""
        p = self.phys[logical]
        if p < self.n_local:
            return False
        i = p - self.n_local
        self.exchange([(p, self.n_local - 1)])
        complemented = bool(self.flip[i])
        self.flip[i] = 0
        return complemented

    def measure(self, qubit: int, vec0, vec1, forced=None) -> int:
        """M.apply (DV/gates.py:165-186): contract reference qubit ``qubit`` with the
        un-conjugated vectors, draw the outcome on rank 0 from NumPy's global legacy generator
        (like the reference) and share it, collapse and renormalise.  The register loses the
        qubit; every rank's shard halves."""
        if self.n_local < 2:
            raise ValueError("shards of a single amplitude cannot be measured; use fewer ranks")
        if not 0 <= qubit < self.n:
            raise ValueError("new_ordering must be a permutation of all qubits")
        be, lib = self.backend, self.backend.lib
        logical = self.n - 1 - qubit
        complemented = self._make_local(logical)
        p = self.phys[logical]                       # local now
        vecs = [np.ascontiguousarray(np.asarray(vec0, dtype=np.complex128).reshape(2)),
                np.ascontiguousarray(np.asarray(vec1, dtype=np.complex128).reshape(2))]
        if complemented:                             # contracting a complemented bit = swapping the bra's entries
            vecs = [v[::-1].copy() for v in vecs]
        j = self.n_local - 1 - p
        part = np.zeros(2)
        _capi.check(lib, lib.qsim_measure_probs(be.ptr(self.buf), self.n_local, int(j),
                                                vecs[0].view(np.float64).ctypes.data_as(_capi.c_double_p),
                                                vecs[1].view(np.float64).ctypes.data_as(_capi.c_double_p),
                                                part.ctypes.data_as(_capi.c_double_p), be.stream()))
        probs = self.comm.allreduce_sum(part)
        norm0, norm1 = np.sqrt(probs[0]), np.sqrt(probs[1])
        # rank 0 draws (same generator, same stream consumption and same ValueError as the
        # reference, DV/gates.py:183); a failure there is shared so that every rank raises
        # instead of the others waiting in the next collective
        pick = np.zeros(2)
        error = None
        if self.comm.rank == 0:
            try:
                pick[0] = forced if forced is not None else int(np.random.choice([0, 1], p=[norm0 ** 2, norm1 ** 2]))
            except ValueError as exc:
                pick[1], error = 1.0, exc
        pick = self.comm.allreduce_sum(pick)
        if pick[1] > 0:
            raise error if error is not None else ValueError("probabilities do not sum to 1")
        outcome = int(round(pick[0]))
        out = be.empty(1 << (self.n_local - 1))
        bra = vecs[outcome]
        _capi.check(lib, lib.qsim_collapse(be.ptr(self.buf), be.ptr(out), self.n_local, int(j),
                                           bra.view(np.float64).ctypes.data_as(_capi.c_double_p),
                                           float((norm0, norm1)[outcome]), be.stream()))
        self.buf = out
        # the qubit is gone: logical bits above it and physical bits above its position move down
        new_phys = []
        for l, q in enumerate(self.phys):
            if l == logical:
                continue
            new_phys.append(q - 1 if q > p else q)
        self.phys = new_phys
        self.n -= 1
        self.n_local -= 1
        return outcome

    def insert(self, position: int, amp) -> None:
        """Insert.apply (DV/gates.py:145-153): a new qubit in state ``amp`` at reference
        position ``position``.  It becomes the top local bit of every shard, which doubles."""
        if not 0 <= position <= self.n:
            raise ValueError("new_ordering must be a permutation of all qubits")
        be, lib = self.backend, self.backend.lib
        v = np.ascontiguousarray(np.asarray(amp, dtype=np.complex128).reshape(2))
        out = be.empty(1 << (self.n_local + 1))
        _capi.check(lib, lib.qsim_insert(be.ptr(self.buf), be.ptr(out), self.n_local, 0,
                                         v.view(np.float64).ctypes.data_as(_capi.c_double_p), be.stream()))
        self.buf = out
        new_logical = self.n - position                  # in the grown register
        top = self.n_local                               # physical position of the new bit
        grown = [q + 1 if q >= top else q for q in self.phys]
        self.phys = grown[:new_logical] + [top] + grown[new_logical:]
        self.n += 1
        self.n_local += 1

    # -- gathering (tests / small registers only) -----------------------------------------------------
    def gather_numpy(self) -> np.ndarray:
        """Full state in logical order on every rank."""
        import torch
        local = torch.view_as_real(self._as_torch(self.buf)).contiguous()
        parts = [torch.empty_like(local) for _ in range(self.comm.size)]
        self.comm.dist.all_gather(parts, local, group=self.comm.group)
        flipmask = sum(f << i for i, f in enumerate(self.flip))
        # rank r holds the logical rank value r ^ flipmask
        full = np.concatenate([torch.view_as_complex(parts[r ^ flipmask]).cpu().numpy()
                               for r in range(self.comm.size)])                         # physical order
        # physical index -> logical index: move physical bit phys[l] to logical bit l
        cube = full.reshape((2,) * self.n)                    # axis a <-> physical bit n-1-a
        axes = [self.n - 1 - self.phys[self.n - 1 - a] for a in range(self.n)]   # logical axis a takes that physical axis
        return np.ascontiguousarray(cube.transpose(axes)).reshape(-1)


def _kind(bits, m: np.ndarray) -> str:
    if _is_diagonal(m):
        return "diag"
    if len(bits) == 1 and m[0, 0] == 0 and m[1, 1] == 0:
        return "anti"                                # relabels the ranks when it sits on a rank qubit
    return "full"


class ShardedSimulator:
    """Runs a list of matrix gates (this package's ``Gate`` objects) on a ShardedState.

    ``compile()`` builds the stage schedule; ``prepare(vectors)`` builds the product
    state in the layout the first stage wants; ``run()`` executes."""

    def __init__(self, circuit, state: ShardedState, plan_options=None, density: bool = False):
        """``density``: the state is vec(rho) of an N = state.n / 2 qubit register (row qubits
        first, column qubits after them, as everywhere in this package): unitaries act as
        U on q and conj(U) on q + N, Kraus channels as one superoperator on (q, q + N), and
        the sharding is the same -- the first row qubits are the rank qubits to begin with."""
        self.circuit = circuit
        self.state = state
        self.plan_options = plan_options
        self.density = bool(density)
        if self.density and state.n % 2:
            raise ValueError("a vectorised density matrix has an even number of index bits")
        if self.density:
            state.is_density = True
        self.stats = {"segments": 0, "passes": 0, "swaps": 0, "local_gates": 0, "exchange_units": 0.0,
                      "relabels": 0, "carried_common": 0, "carried_signs": 0, "carried_controlled": 0}
        self._schedule = None
        self.initial_phys = list(range(state.n))
        self.final_flip = [0] * state.g

    # ---- scheduling helpers ---------------------------------------------------------------------
    def _lower(self):
        """[(logical_bits (factor order), matrix, kind)]"""
        n = self.state.n
        nq = n // 2 if self.density else n
        out = []
        for gate in self.circuit:
            fusable = getattr(gate, "_fusable", False) and hasattr(gate, "lowered")
            if not fusable:
                raise NotImplementedError(f"ShardedSimulator runs matrix gates and channels only (no measurement, "
                                          f"insertion or classical control yet); got {gate!r}")
            for targets, matrix in gate.lowered(nq, self.density):
                m = np.asarray(matrix, dtype=np.complex128)
                bits = [n - 1 - q for q in targets]
                out.append((bits, m, _kind(bits, m)))
        return out

    def _rank_value(self, phys_bit: int, flip) -> int:
        st = self.state
        i = phys_bit - st.n_local
        return ((st.comm.rank >> i) & 1) ^ flip[i]

    def _restrict_diagonal(self, bits_phys, matrix, flip):
        """Diagonal gate with some targets in the rank number: keep this rank's entries."""
        st = self.state
        k = len(bits_phys)
        diag = np.diagonal(matrix).reshape((2,) * k)
        index, local_bits = [], []
        for p in bits_phys:
            if p >= st.n_local:
                index.append(self._rank_value(p, flip))
            else:
                index.append(slice(None))
                local_bits.append(p)
        sub = np.asarray(diag[tuple(index)]).reshape(-1)
        if not local_bits:                           # pure scalar: put it on local bit 0
            return [0], np.diag([sub[0], sub[0]])
        return local_bits, np.diag(sub)

    defer_tails = True      # leave each stage's trailing single-qubit phases to the next stage's plan
    dense_caps = (18, 20, 22, 24)   # matrices-per-pass caps tried for every stage (0 entries: planner default)

    def _best_plan(self, nloc, segment, options):
        """A stage is a short circuit, and its last pass is often nearly empty; planning costs
        tens of milliseconds, so try a few caps on the matrices per pass and keep the cheapest
        plan under the measured cost model of DESIGN.md section 5 (3.0 ms per pass + 0.80 ms per
        shared-memory round trip, per 2^30 amplitudes; the matrices cost the same under every cap).  Ranks may decide differently (their
        restricted diagonals differ) -- which is fine, plans are local."""
        if options.get("max_dense_ops") or not self.dense_caps:
            return engine.Plan(self.state.backend, nloc, segment, options)
        best = None
        for cap in self.dense_caps:
            plan = engine.Plan(self.state.backend, nloc, segment, dict(options, max_dense_ops=cap))
            key = 3.0 * plan.stats["n_passes"] + 0.80 * plan.stats["n_steps"]
            if best is None or key < best[0]:
                best = (key, plan)
        return best[1]

    def _carry_controlled(self, out, leaving, l, mats):
        """The general case: a single-qubit gate on ``l`` selected by the ``leaving`` qubits."""
        k = len(leaving)
        full = np.zeros((2 << k, 2 << k), dtype=np.complex128)
        for x, m in enumerate(mats):
            full[2 * x:2 * x + 2, 2 * x:2 * x + 2] = m
        out.append((list(leaving) + [l], full))
        self.stats["carried_controlled"] += 1

    def _carry_residuals(self, residual, leaving, leaving_phys, phys):
        """Gates that stand for the unapplied leftovers (``qsim_plan_residual``) of the plan
        before an exchange, as ``[(logical bits, matrix)]`` for the next stage.

        The leftovers differ from rank to rank (restricted diagonals depend on the rank
        bits), and after the exchange a shard holds data from all 2^k ranks of its group:
        the amplitudes whose now-local qubits ``leaving`` read x came from the rank whose
        bits ``leaving_phys`` were x.  So the leftover on a qubit is a gate controlled by the
        ``leaving`` qubits.  Almost always the 2^k versions differ by scalars only (left
        phases of the same rotation) or by a Z as well (a trailing CZ with a rank qubit): then
        one common 2x2 goes to the qubit, the scalars collect into a single k-qubit diagonal and
        the Z's come back as the CZ gates they were; otherwise the qubit gets its own
        (k+1)-qubit gate, block diagonal in the ``leaving`` qubits.  Qubits that become rank
        qubits in this exchange have nothing left over (``apply_tail_mask``)."""
        st = self.state
        nloc, k = st.n_local, len(leaving)
        gather = getattr(st.comm, "allgather_object", None)
        everyone = gather(residual) if gather else [residual] * st.comm.size     # (ranks, nloc, 2, 2)
        sources = []
        for x in range(1 << k):                       # x: factor order = `leaving` order, first most significant
            r = st.comm.rank
            for i, gp in enumerate(leaving_phys):
                bit = (x >> (k - 1 - i)) & 1
                r = (r & ~(1 << (gp - nloc))) | (bit << (gp - nloc))
            sources.append(everyone[r])
        where = {p: l for l, p in enumerate(phys)}
        eye = np.eye(2)
        x_gate = np.array([[0, 1], [1, 0]], dtype=np.complex128)
        cz_gate = np.diag([1, 1, 1, -1]).astype(np.complex128)
        scalars = np.ones(1 << k, dtype=np.complex128)
        out = []
        for q in range(nloc):
            mats = [src[q] for src in sources]
            if all(np.array_equal(m, eye) for m in mats):
                continue
            l = where[nloc - 1 - q]
            base = mats[0]
            anti = base[0, 0] == 0 and base[1, 1] == 0
            if any((m[0, 0] == 0 and m[1, 1] == 0) != anti for m in mats):
                # H Z^v H = X^v: a rank-dependent Z between two gates turned into a bit flip
                self._carry_controlled(out, leaving, l, mats)
                continue
            # the two non-zero entries: row 0 and row 1 (a Z on the qubit negates row 1)
            top = [m[0, 1] if anti else m[0, 0] for m in mats]
            bot = [m[1, 0] if anti else m[1, 1] for m in mats]
            ratios = np.asarray([t / top[0] for t in top])                       # scalar per source rank
            twist = np.asarray([(b / bot[0]) / r for b, r in zip(bot, ratios)])  # what is left on row 1
            if np.allclose(twist, 1.0, rtol=0, atol=1e-14):
                scalars *= ratios
                out.append(([l], base))
                self.stats["carried_common"] += 1
                continue
            # signs that are linear in x are CZ gates between the qubit and the `leaving` qubits
            coeff = [int(np.real(twist[1 << (k - 1 - i)]) < 0) for i in range(k)]
            linear = np.asarray([(-1.0) ** sum(c * ((x >> (k - 1 - i)) & 1) for i, c in enumerate(coeff))
                                 for x in range(1 << k)])
            if np.allclose(twist, linear, rtol=0, atol=1e-14):
                scalars *= ratios
                out.append(([l], base))
                for i, c in enumerate(coeff):
                    if c:
                        out.append(([leaving[i], l], cz_gate))
                self.stats["carried_signs"] += 1
                continue
            self._carry_controlled(out, leaving, l, mats)
        if not np.array_equal(scalars, np.ones(1 << k)):
            out.append((list(leaving), np.diag(scalars)))
        return out

    @staticmethod
    def _choose_rank_qubits(ops, pending, current, n, g, local_now=()):
        """The g logical bits whose first blocking gate among ``pending`` lies farthest
        ahead (never blocked at all is best); ties keep what is a rank qubit already.
        ``local_now``: bits that must be local in the next stage (progress guarantee)."""
        dist = {b: -1 for b in local_now}
        for pos, idx in enumerate(pending):
            bits, _m, kind = ops[idx]
            if kind == "full":
                for b in bits:
                    dist.setdefault(b, pos)
        order = sorted(range(n), key=lambda l: (-dist.get(l, 1 << 60), 0 if l in current else 1, -l))
        return set(order[:g])

    def compile(self, fixed_layout: bool = False):
        """Cut the circuit into stages (see the module docstring) and build one fused
        local plan per stage, separated by multi-qubit exchanges.  With ``fixed_layout`` the
        schedule starts from the state's current layout and flip flags (a circuit that continues
        on a live state); otherwise the first stage picks its own rank qubits and ``prepare``
        builds the product state accordingly."""
        st = self.state
        ops = self._lower()
        n, g, nloc = st.n, st.g, st.n_local
        x_gate = np.array([[0, 1], [1, 0]], dtype=np.complex128)
        schedule = []

        pending = list(range(len(ops)))
        if fixed_layout:
            phys = list(st.phys)
            glob = {l for l in range(n) if phys[l] >= nloc}
            flip = list(st.flip)
        else:
            # stage 0: the product state can be built in any layout, so choose before moving anything
            glob = self._choose_rank_qubits(ops, pending, set(), n, g)
            phys = [0] * n
            for i, l in enumerate(sorted(glob)):
                phys[l] = nloc + i
            for i, l in enumerate(l for l in range(n) if l not in glob):
                phys[l] = i
            flip = [0] * g
        self.initial_phys = list(phys)
        self.initial_flip = list(flip)
        carry = []                                   # [(logical bits, matrix)] to run before anything else

        while True:
            # What can run in this layout.  A gate that cannot (neither diagonal nor a
            # single-qubit antidiagonal, and on a rank qubit) blocks its qubits; gates behind it
            # are held back only if they do not commute with what is blocked (diagonal gates
            # commute with each other).
            ready, deferred = [], []
            blocked_full, blocked_diag = set(), set()
            for idx in pending:
                bits, _m, kind = ops[idx]
                sb = set(bits)
                is_diag = kind == "diag"
                free = not (blocked_full & sb) and (is_diag or not (blocked_diag & sb))
                if free and (kind != "full" or all(phys[b] < nloc for b in bits)):
                    ready.append(idx)
                else:
                    deferred.append(idx)
                    (blocked_diag if is_diag else blocked_full).update(bits)

            head = deferred[0] if deferred else None          # the first gate that could not run

            # carried gates first: X fix-ups of qubits that arrived complemented and the
            # diagonal / antidiagonal leftovers of the previous plan (qsim_plan_residual)
            segment = []

            def emit(bits, m, kind):
                p_bits = [phys[b] for b in bits]
                if kind == "diag" and any(p >= nloc for p in p_bits):
                    p_bits, m = self._restrict_diagonal(p_bits, m, flip)
                elif kind == "anti" and p_bits[0] >= nloc:
                    v = self._rank_value(p_bits[0], flip)          # this rank's data becomes the 1-v branch
                    scalar = m[1 - v, v]
                    flip[p_bits[0] - nloc] ^= 1
                    self.stats["relabels"] += 1
                    p_bits, m = [0], np.diag([scalar, scalar])
                segment.append(([nloc - 1 - p for p in p_bits], m))

            for bits, m in carry:
                emit(bits, m, _kind(bits, m))
            carry = []
            for idx in ready:
                emit(*ops[idx])
            # the next stage's rank qubits are chosen before this stage's plan is built: a qubit
            # that is about to become a rank qubit must not leave anything unapplied behind
            if deferred:
                new_glob = self._choose_rank_qubits(ops, deferred, glob, n, g, ops[head][0])
                leaving = sorted(glob - new_glob, key=lambda l: phys[l])
                entering = sorted(new_glob - glob, key=lambda l: phys[l])
                assert leaving, "the scheduler made no progress"
                pairs = [(phys[a], phys[b]) for a, b in zip(leaving, entering)]
            want_residual = bool(deferred) and self.defer_tails      # the same on every rank
            residual = np.tile(np.eye(2, dtype=np.complex128), (nloc, 1, 1)) if want_residual else None
            if segment:
                options = dict(self.plan_options or {})
                if want_residual:
                    options["defer_tail"] = 1
                    options["apply_tail_mask"] = sum(1 << (nloc - 1 - lp) for _gp, lp in pairs)
                plan = self._best_plan(nloc, segment, options)
                schedule.append(("plan", plan))
                self.stats["segments"] += 1
                self.stats["passes"] += plan.stats["n_passes"]
                self.stats["local_gates"] += len(segment)
                if want_residual:
                    residual = plan.residual_array()
            if not deferred:
                break

            if residual is not None:
                carry = self._carry_residuals(residual, leaving[:len(pairs)], [gp for gp, _lp in pairs], phys)
            schedule.append(("exchange", pairs))
            self.stats["swaps"] += 1
            self.stats["exchange_units"] += 1.0 - 0.5 ** len(pairs)
            for a, b in zip(leaving, entering):
                i = phys[a] - nloc
                if flip[i]:                          # a's bit is stored complemented: fix it locally
                    carry.append(([a], x_gate))
                    flip[i] = 0
                phys[a], phys[b] = phys[b], phys[a]
            glob = new_glob
            pending = deferred

        self.final_flip = list(flip)
        self.final_phys = list(phys)
        self._schedule = schedule
        return schedule

    def run_circuit(self, vectors) -> ShardedState:
        """``Simulator.run`` semantics (DV/simulator.py:36-53) on a sharded ket, for circuits
        that also measure, insert qubits and feed results forward: maximal runs of matrix
        gates go through the stage scheduler (the first one picks the layout the product state
        is built in, the later ones continue from the live layout), ``M`` / ``Insert`` /
        ``ClassicalControl`` act in between.  Outcomes end up in ``self.results``."""
        from .gates import Insert, M
        from .simulator import ClassicalControl
        if self.density:
            raise NotImplementedError("measurements on a sharded density matrix are not defined (SURVEY 3.3)")
        st = self.state
        vecs = [np.asarray(v, dtype=np.complex128) for v in vectors]
        self.results = []
        segment, prepared = [], False

        def flush():
            nonlocal prepared
            sub = None
            if segment:
                sub = ShardedSimulator(list(segment), st, self.plan_options)
                sub.compile(fixed_layout=prepared)
            if not prepared:
                st.set_product(vecs, sub.initial_phys if sub else None)
                prepared = True
            if sub:
                sub.run()
                for key, val in sub.stats.items():
                    self.stats[key] = self.stats.get(key, 0) + val
            segment.clear()

        for gate in self.circuit:
            if isinstance(gate, ClassicalControl):
                if not gate.eval(self.results):          # every M before it has run: it ended a segment
                    continue
                gate = gate.gate
            if isinstance(gate, M):
                flush()
                v0, v1 = gate.vectors()
                self.results.append(st.measure(gate.indices[0], v0, v1, gate.result))
            elif isinstance(gate, Insert):
                flush()
                st.insert(gate.indices[0], gate.state.get())
            elif getattr(gate, "_fusable", False):
                segment.append(gate)
            else:
                raise NotImplementedError(f"ShardedSimulator cannot run {gate!r}")
        flush()
        return st

    def prepare(self, vectors) -> ShardedState:
        """Product state (qubit 0 first) in the layout the first stage runs in; with
        ``density`` the N kets give rho = |psi><psi|, i.e. vec(rho) = psi (x) conj(psi)."""
        if self._schedule is None:
            self.compile()
        vecs = [np.asarray(v, dtype=np.complex128) for v in vectors]
        if self.density:
            vecs = vecs + [np.conjugate(v) for v in vecs]
        self.state.set_product(vecs, self.initial_phys)
        return self.state

    def run(self) -> ShardedState:
        """Execute the schedule on the state, which must be in the schedule's initial
        layout (``prepare``)."""
        st = self.state
        if self._schedule is None:
            self.compile()
        if st.phys != self.initial_phys or list(st.flip) != list(getattr(self, "initial_flip", [0] * st.g)):
            raise ValueError("the state is not in the schedule's initial layout; call prepare() first")
        for item in self._schedule:
            if item[0] == "plan":
                item[1].execute(st.buf)
            else:
                st.exchange(item[1])
        assert st.phys == self.final_phys
        st.flip = list(self.final_flip)
        return st
