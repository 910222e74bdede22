"""Parity checks shared by the CPU (host-emulator backend) and GPU (CUDA backend)
test modules.  Every function takes the backend to run the package on and
compares with the golden vectors produced by the real reference
(tests/golden/make_golden.py) and/or with the CPU oracle.

Tolerance: the north star asks for <= 1e-10 relative in complex128; the checks
use RTOL = 1e-12 on max|diff| / max|ref| unless stated otherwise.
"""
from __future__ import annotations

import json
import os

import numpy as np

from golden.specs import as_oracle_ops, from_spec
from oracle import dense_ref, gkp_noise, strided
from quantum_computations_b200 import channels, engine, gates, simulator, states, workloads
from quantum_computations_b200 import numpy_quantum as npq
from quantum_computations_b200.batched import BatchedSimulator
from quantum_computations_b200.simulator import Simulator
from quantum_computations_b200.states import State

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-12


def load(name):
    z = np.load(os.path.join(GOLDEN, name))
    return json.loads(str(z["meta"])), z


def rel_err(got, ref) -> float:
    """max |got - ref| / max |ref|: the error relative to the LARGEST reference entry (a norm-wise
    bound, not element-wise relative error -- an amplitude that is 1e-6 of the largest one is
    only checked to RTOL * 1e6 of its own size).  This is the sense in which the north star's
    "<= 1e-10 relative" is asserted throughout, with RTOL = 1e-12."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    scale = max(float(np.abs(ref).max()), 1e-300)
    return float(np.abs(got - ref).max()) / scale


def mk(spec, z):
    return from_spec(spec, gates, simulator, z, channels, states)


def dev(arr, backend):
    return engine.DeviceState.from_numpy(arr, backend)


# ---- single gates ------------------------------------------------------------------------
def check_single_gates(backend):
    meta, z = load("single_gates.npz")
    worst = 0.0
    for rec in meta:
        gate = mk(rec["gate"], z)
        got = gate.apply(dev(z[rec["in"]], backend)).to_numpy()
        ref = z[rec["out"]]
        worst = max(worst, rel_err(got, ref))
        if "dtype" in rec:
            assert str(got.dtype) == rec["dtype"], (rec, got.dtype)
    assert worst < RTOL, worst
    return worst


def check_density_gates(backend):
    meta, z = load("density_gates.npz")
    worst = 0.0
    for rec in meta:
        got = mk(rec["gate"], z).apply(dev(z[rec["in"]], backend)).to_numpy()
        worst = max(worst, rel_err(got, z[rec["out"]]))
    assert worst < RTOL, worst
    return worst


def check_measure(backend):
    meta, z = load("measure.npz")
    worst = 0.0
    for rec in meta:
        if "stream" in rec:
            psi = z[rec["in"]]
            np.random.seed(rec["seed"])
            d = dev(psi, backend)
            got = [int(gates.MZ(rec["q"]).apply(d)[1]) for _ in range(len(rec["stream"]))]
            assert got == rec["stream"]          # bit-exact outcome stream
            continue
        m = gates.M(rec["q"], rec["theta"], rec["phi"], result=rec["forced"])
        if rec["seed"] is not None:
            np.random.seed(rec["seed"])
        out, s = m.apply(dev(z[rec["in"]], backend))
        assert s == rec["s"], rec
        worst = max(worst, rel_err(out.to_numpy(), z[rec["out"]]))
    assert worst < RTOL, worst
    return worst


def check_insert(backend):
    meta, z = load("insert.npz")
    worst = 0.0
    for rec in meta:
        out = gates.Insert(rec["pos"], State[rec["state"]]).apply(dev(z[rec["in"]], backend))
        ref = z[rec["out"]]
        got = out.to_numpy()
        worst = max(worst, rel_err(got, ref))
        assert got.dtype == ref.dtype, (rec, got.dtype, ref.dtype)
    assert worst < RTOL, worst
    return worst


def check_kraus(backend):
    meta, z = load("kraus.npz")
    worst = 0.0
    for rec in meta:
        ch = channels.Channel(rec["indices"], list(z[rec["kraus"]]))
        got = ch.apply(dev(z[rec["in"]], backend)).to_numpy()
        worst = max(worst, rel_err(got, z[rec["out"]]))
    assert worst < RTOL, worst
    return worst


def check_metrics(backend):
    meta, z = load("metrics.npz")
    for rec in meta:
        n = rec["n"]
        a, b, ra, rb = (z[f"{k}{n}"] for k in ("a", "b", "ra", "rb"))
        da, db_, dra, drb = (dev(x, backend) for x in (a, b, ra, rb))
        assert abs(npq.fidelity(da, db_) - rec["f_kk"]) < 1e-12
        assert abs(npq.fidelity(da, drb) - rec["f_kr"]) < 1e-12
        assert abs(npq.fidelity(dra, db_) - rec["f_rk"]) < 1e-12
        assert abs(npq.fidelity(dra, drb) - rec["f_rr"]) < 1e-9     # eigvals branch (host LAPACK)
        assert abs(npq.fidelity(a, drb) - rec["f_kr"]) < 1e-12       # mixed host/device operands
        assert abs(npq.purity(dra) - rec["purity"]) < 1e-12
        assert abs(npq.norm(dev(3.0 * a, backend)) - rec["norm"]) < 1e-12


# ---- circuits ---------------------------------------------------------------------------------
def check_sv_circuits(backend, plan_options=None, max_n=13):
    meta, z = load("circuits.npz")
    worst = 0.0
    for rec in meta:
        if rec["n"] > max_n:
            continue
        circ = workloads.sv_random_circuit(rec["n"], rec["depth"], rec["seed"])
        assert len(circ) == rec["ngates"]
        got = Simulator(circ, backend=backend, plan_options=plan_options).run([State.ZERO] * rec["n"])
        worst = max(worst, rel_err(got, z[rec["out"]]))
    # the same generator from random kets: every amplitude of these vectors is distinct
    meta, z = load("circuits_rand.npz")
    for rec in meta:
        if rec["n"] > max_n:
            continue
        circ = workloads.sv_random_circuit(rec["n"], rec["depth"], rec["seed"])
        assert len(circ) == rec["ngates"]
        got = Simulator(circ, backend=backend, plan_options=plan_options).run(z[rec["in"]])
        worst = max(worst, rel_err(got, z[rec["out"]]))
    assert worst < RTOL, worst
    return worst


def check_grover(backend):
    meta, z = load("grover.npz")
    worst = 0.0
    for rec in meta:
        circ = [mk(s, z) for s in rec["circuit"]]
        init = None if rec["kind"] == "full" else [State[s] for s in rec["init"]]
        got = Simulator(circ, backend=backend).run(init)
        ref = z[rec["out"]]
        worst = max(worst, rel_err(got, ref))
        probs = np.abs(got) ** 2
        for t in rec["tagged"]:                       # ideal Grover: 1/2 on each tagged state
            assert abs(probs[t] - 0.5) < 1e-12
    assert worst < RTOL, worst
    return worst


def check_noisy_grover(backend):
    meta, z = load("noisy_grover.npz")
    worst = 0.0
    for rec in meta:
        circ = [mk(s, z) for s in rec["circuit"]]
        noise = channels.GKPNoise(rec["db"])
        psi0 = npq.tensor(*(State[s].get() for s in rec["init"])).astype(np.complex128)
        rho0 = npq.ket2dm(psi0)
        got = Simulator(noise.noisy(circ), backend=backend).run(rho0)
        worst = max(worst, rel_err(got, z[rec["out"]]))
        success = sum(got[t, t].real for t in rec["tagged"])
        assert abs(success - rec["success"]) < 1e-12
    assert worst < RTOL, worst
    return worst


def check_sim_measure(backend):
    meta, z = load("sim_measure.npz")
    circ = [mk(s, z) for s in meta["circuit"]]
    worst = 0.0
    for run in meta["runs"]:
        np.random.seed(run["seed"])
        sim = Simulator(circ, backend=backend)
        got = sim.run(None)
        assert sim.results == run["results"], (sim.results, run["results"])
        worst = max(worst, rel_err(got, z[run["out"]]))
    assert worst < RTOL, worst
    return worst


def check_rb(backend):
    """Circuit generator equality, ideal kets vs the reference, and the batched
    noisy executor vs the oracle's density-matrix path."""
    meta, z = load("rb.npz")
    rng = np.random.default_rng(meta["seed"])
    circuits = []
    for i, rec in enumerate(meta["samples"]):
        circ = workloads.rb_random_circuit(2, rec["depth"], rng)
        want = [mk(s, z) for s in rec["circuit"]]
        assert [repr(g) for g in circ] == [repr(g) for g in want], i     # same draws, same circuit
        got = Simulator(circ, backend=backend).run([State.ZERO] * 2)
        assert rel_err(got, z[rec["out"]]) < RTOL
        circuits.append(circ)
    db = 10.0
    noise = channels.GKPNoise(db)
    res = BatchedSimulator(2, noise, backend=backend).run(circuits, return_rho=True)
    for i, circ in enumerate(circuits):
        rho = np.zeros((4, 4), dtype=np.complex128)
        rho[0, 0] = 1.0
        for gate in circ:
            rho = dense_ref.apply_matrix(rho, gate.indices, gate.matrix)
            for q, (px, pz) in zip(gate.indices, noise.flips_for(gate)):
                rho = dense_ref.apply_kraus(rho, [q], gkp_noise.pauli_flip_kraus(px, pz))
        ideal = z[meta["samples"][i]["out"]]
        assert rel_err(res["rho"][i], rho) < RTOL
        assert abs(res["fidelity"][i] - dense_ref.fidelity(rho, ideal)) < 1e-12
        assert abs(res["purity"][i] - dense_ref.purity(rho)) < 1e-12
    # noise-free batch reproduces fidelity 1, purity 1
    clean = BatchedSimulator(2, None, backend=backend).run(circuits)
    assert np.allclose(clean["fidelity"], 1.0, atol=1e-12) and np.allclose(clean["purity"], 1.0, atol=1e-12)


# ---- randomised differential test against the oracle ------------------------------------------------
def random_circuit(n, length, rng):
    circ = []
    for _ in range(length):
        r = int(rng.integers(0, 13))
        q = int(rng.integers(0, n))
        others = [x for x in range(n) if x != q]
        q2 = int(rng.choice(others)) if others else None
        if r == 0 or q2 is None and r >= 4 and r not in (7, 8, 9):
            circ.append(gates.H(q))
        elif r == 1:
            circ.append(gates.T(q))
        elif r == 2:
            circ.append(gates.X(q))
        elif r == 3:
            circ.append(gates.RZ(q, float(rng.uniform(0, 2 * np.pi))))
        elif r == 4:
            circ.append(gates.CZ(q, q2))
        elif r == 5:
            circ.append(gates.CX(q, q2))
        elif r == 6:
            circ.append(gates.SWAP(q, q2))
        elif r == 7:
            circ.append(gates.Z(q))
        elif r == 8:
            circ.append(gates.Y(q))
        elif r == 9:
            circ.append(gates.P(q))
        elif r == 10:
            m = rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4))
            circ.append(gates.Gate([q, q2], m / 2))
        elif r == 11:
            rest = [x for x in others if x != q2]
            if rest:
                q3 = int(rng.choice(rest))
                m = rng.normal(size=(8, 8)) + 1j * rng.normal(size=(8, 8))
                circ.append(gates.Gate([q2, q, q3], m / 3))
        else:
            d = np.exp(1j * rng.uniform(0, 2 * np.pi, size=4))
            circ.append(gates.Gate([q, q2], np.diag(d)))
    return circ


def check_random_vs_oracle(backend, trials, n_range, tile_range, seed):
    rng = np.random.default_rng(seed)
    worst = 0.0
    for _ in range(trials):
        n = int(rng.integers(n_range[0], n_range[1] + 1))
        opts = dict(tile_bits=int(rng.integers(tile_range[0], tile_range[1] + 1)),
                    low_bits=int(rng.integers(0, 5)), max_group=int(rng.integers(1, 5)),
                    max_dense_ops=int(rng.integers(1, 24)), merge_1q=int(rng.integers(1, 3)),
                    cta_log2=int(rng.choice([0, 7, 8])))
        psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        psi /= np.linalg.norm(psi)
        circ = random_circuit(n, int(rng.integers(1, 80)), rng)
        got = Simulator(circ, backend=backend, plan_options=opts).run(psi)
        ref, _ = strided.run(as_oracle_ops(circ), psi)
        err = rel_err(got, ref)
        assert err < RTOL, (n, opts, err)
        worst = max(worst, err)
    return worst


def check_edge_cases(backend):
    """The corners: empty and diagonal-only circuits, registers of one qubit, gates on the
    whole register, gates wider than a step (in-place dense-block kernel, k = 5 .. 10; from
    k = 9 on its tile needs more than 48 KiB of shared memory),
    cancelling CZ pairs, reversed / scattered targets, empty and zero-length RB batches."""
    rng = np.random.default_rng(99)

    def rand_state(n):
        psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        return psi / np.linalg.norm(psi)

    def rand_unitary(k):
        return np.linalg.qr(rng.normal(size=(2 ** k, 2 ** k)) + 1j * rng.normal(size=(2 ** k, 2 ** k)))[0]

    def run_both(circ, psi, **opts):
        got = Simulator(circ, backend=backend, plan_options=opts or None).run(psi)
        ref, _ = strided.run(as_oracle_ops(circ), psi)
        return got, ref

    # empty circuit: a copy of the input, not the input itself
    psi = rand_state(5)
    out = Simulator([], backend=backend).run(psi)
    assert out is not psi and np.array_equal(out, psi)
    assert np.array_equal(Simulator([], backend=backend).run([State.ZERO, State.ONE]), np.array([0, 1, 0, 0]))

    # one qubit: gate, then the measurement that leaves a 0-d array (reference quirk)
    one = Simulator([gates.H(0)], backend=backend).run(np.array([1.0, 0.0]))
    assert rel_err(one, np.array([1.0, 1.0]) / np.sqrt(2)) < RTOL
    np.random.seed(5)
    sim = Simulator([gates.H(0), gates.MZ(0)], backend=backend)
    left = sim.run(np.array([1.0, 0.0]))
    assert np.shape(left) == () and sim.results[0] in (0, 1) and abs(abs(left) - 1.0) < 1e-12

    # diagonal gates only (no matrix step at all), with CZ pairs that cancel and Z Z = 1
    n = 7
    psi = rand_state(n)
    circ = [gates.T(0), gates.CZ(0, 6), gates.RZ(3, 0.7), gates.CZ(6, 0), gates.CZ(2, 5), gates.Z(4), gates.Z(4),
            gates.P(6), gates.CZ(1, 2), gates.Tdg(2), gates.CZ(2, 5), gates.Pdg(1)]
    got, ref = run_both(circ, psi, tile_bits=5, low_bits=2)
    assert rel_err(got, ref) < RTOL

    # a gate on the whole register, targets reversed and scattered
    for n, idx in ((2, [1, 0]), (3, [2, 0, 1]), (4, [3, 1, 0, 2])):
        psi = rand_state(n)
        got, ref = run_both([gates.Gate(list(idx), rand_unitary(n))], psi)
        assert rel_err(got, ref) < RTOL
    psi = rand_state(9)
    circ = [gates.Gate([7, 2], rand_unitary(2)), gates.Gate([8, 0, 4], rand_unitary(3)),
            gates.Gate([5, 3, 6, 1], rand_unitary(4)), gates.H(8), gates.Gate([0, 8], rand_unitary(2))]
    got, ref = run_both(circ, psi, tile_bits=6, low_bits=1)
    assert rel_err(got, ref) < RTOL

    # wider than a step: the in-place dense-block kernel (DMMA), between fused segments
    for k, n in ((5, 7), (6, 8), (7, 7)):
        psi = rand_state(n)
        idx = [int(q) for q in rng.permutation(n)[:k]]
        circ = [gates.H(0), gates.CZ(0, n - 1), gates.Gate(idx, rand_unitary(k)), gates.T(idx[0]), gates.H(n - 1)]
        got, ref = run_both(circ, psi)
        assert rel_err(got, ref) < RTOL, (k, n)
    # ... on registers with many tiles; targets on the lowest index bits (qubits n-1, n-2, n-3), on the
    # highest, scattered; the same plan executed twice (the device copy of the matrix is reused)
    for k, n, idx in ((5, 12, [11, 10, 9, 0, 4]), (5, 13, [0, 1, 2, 3, 4]), (6, 12, None), (7, 12, None),
                      (8, 11, None), (5, 5, None), (6, 7, [6, 5, 4, 3, 2, 1]), (9, 12, None),
                      (9, 9, [8, 7, 6, 5, 4, 3, 2, 1, 0]), (10, 13, None), (10, 11, [0, 1, 2, 3, 4, 5, 6, 7, 8, 9])):
        psi = rand_state(n)
        if idx is None:
            idx = [int(q) for q in rng.permutation(n)[:k]]
        u = rand_unitary(k)
        circ = [gates.Gate(idx, u), gates.CZ(0, n - 1), gates.Gate(idx, u.conj().T @ u @ u)]
        sim = Simulator(circ, backend=backend)
        ref, _ = strided.run(as_oracle_ops(circ), psi)
        for _ in range(2):
            assert rel_err(sim.run(psi), ref) < RTOL, (k, n, idx)

    # density matrix with a channel on a one-qubit register
    rho = np.array([[0.75, 0.1 - 0.2j], [0.1 + 0.2j, 0.25]])
    noise = channels.GKPNoise(9.0)
    circ = noise.noisy([gates.H(0), gates.T(0)])
    got = Simulator(circ, backend=backend).run(rho)
    want = rho
    for g in (gates.H(0), gates.T(0)):
        want = dense_ref.apply_matrix(want, g.indices, g.matrix)
        for q, (px, pz) in zip(g.indices, noise.flips_for(g)):
            want = dense_ref.apply_kraus(want, [q], gkp_noise.pauli_flip_kraus(px, pz))
    assert rel_err(got, want) < RTOL

    # batched executor: nothing to do, and sequences without gates
    empty = BatchedSimulator(2, None, backend=backend).run([])
    assert empty["fidelity"].shape == (0,) and empty["purity"].shape == (0,)
    idle = BatchedSimulator(2, channels.GKPNoise(10.0), backend=backend).run([[], [gates.H(0)], []])
    assert np.allclose(idle["fidelity"][[0, 2]], 1.0, atol=1e-15) and np.allclose(idle["purity"][[0, 2]], 1.0, atol=1e-15)
    assert idle["fidelity"][1] < 1.0


def check_swap_pack_unpack(backend):
    """qsim_swap_pack / _unpack (the gather / scatter of a k-qubit exchange block) against
    NumPy indexing, chunked like the pipeline does."""
    import ctypes as C
    from quantum_computations_b200 import _capi
    rng = np.random.default_rng(17)
    n = 11
    lib = backend.lib
    for trial in range(12):
        k = int(rng.integers(1, 5))
        qubits = [int(q) for q in rng.choice(n, size=k, replace=False)]
        values = [int(v) for v in rng.integers(0, 2, size=k)]
        shard = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        # reference: amplitudes whose qubit q (bit n-1-q) equals its value, in index order
        idx = np.arange(2 ** n)
        sel = np.ones(2 ** n, dtype=bool)
        for q, v in zip(qubits, values):
            sel &= ((idx >> (n - 1 - q)) & 1) == v
        want = shard[sel]
        block = 2 ** (n - k)
        assert want.size == block
        d_shard = backend.upload(shard)
        d_buf = backend.upload(np.zeros(block, dtype=np.complex128))
        cq, cv = (C.c_int * k)(*qubits), (C.c_int * k)(*values)
        chunk = block // 4 if block >= 4 else block
        for first in range(0, block, chunk):
            _capi.check(lib, lib.qsim_swap_pack(backend.ptr(d_shard), backend.ptr(d_buf), n, k, cq, cv,
                                                C.c_uint64(first), C.c_uint64(chunk), backend.stream()))
            got = backend.download(d_buf)[:chunk]
            assert np.array_equal(got, want[first:first + chunk]), (trial, qubits, values, first)
        # scatter new data into the same positions
        fresh = rng.normal(size=block) + 1j * rng.normal(size=block)
        expect = shard.copy()
        expect[sel] = fresh
        for first in range(0, block, chunk):
            d_part = backend.upload(fresh[first:first + chunk])
            _capi.check(lib, lib.qsim_swap_unpack(backend.ptr(d_shard), backend.ptr(d_part), n, k, cq, cv,
                                                  C.c_uint64(first), C.c_uint64(chunk), backend.stream()))
        assert np.array_equal(backend.download(d_shard), expect)
    # argument checks
    d = backend.upload(np.zeros(8, dtype=np.complex128))
    two = (C.c_int * 2)(1, 1)
    assert lib.qsim_swap_pack(backend.ptr(d), backend.ptr(d), 3, 2, two, two, C.c_uint64(0), C.c_uint64(1),
                              backend.stream()) != 0             # repeated qubit


def check_plan_cache(backend):
    """Simulator keeps compiled plans between runs, keyed by the content of the segment:
    a second run must not plan again, and a gate mutated in between must be noticed."""
    from quantum_computations_b200 import engine
    n = 9
    rng = np.random.default_rng(3)
    circ = random_circuit(n, 60, rng)
    psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
    psi /= np.linalg.norm(psi)
    sim = Simulator(circ, backend=backend)
    made = []
    real_plan = engine.Plan

    class CountingPlan(real_plan):
        def __init__(self, *a, **k):
            made.append(1)
            super().__init__(*a, **k)

    engine.Plan = CountingPlan
    try:
        first = sim.run(psi)
        n_first = len(made)
        second = sim.run(psi)
        assert len(made) == n_first and n_first >= 1
        assert np.array_equal(first, second)
        ref, _ = strided.run(as_oracle_ops(circ), psi)
        assert rel_err(first, ref) < RTOL
        k = next(i for i, g in enumerate(circ) if len(g.indices) == 1)
        circ[k].matrix = np.asarray(circ[k].matrix) @ np.diag([1.0, 1j])
        third = sim.run(psi)
        assert len(made) > n_first
        ref3, _ = strided.run(as_oracle_ops(circ), psi)
        assert rel_err(third, ref3) < RTOL
    finally:
        engine.Plan = real_plan


def check_deferred_tails(backend, trials, seed):
    """options.defer_tail: the plan leaves trailing diagonal / antidiagonal single-qubit
    products unapplied and reports them (qsim_plan_residual); plan + leftovers must equal
    the circuit, and qubits in apply_tail_mask must have nothing left over."""
    from quantum_computations_b200 import engine, workloads
    rng = np.random.default_rng(seed)
    seen = 0
    for t in range(trials):
        n = int(rng.integers(3, 11))
        circ = workloads.sv_random_circuit(n, int(rng.integers(1, 6)), seed + t) + random_circuit(n, 6, rng)
        ops = []
        for g in circ:
            ops.extend(g.lowered(n, False))
        psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        psi /= np.linalg.norm(psi)
        ref, _ = strided.run(as_oracle_ops(circ), psi)
        mask = int(rng.integers(0, 1 << n))
        opts = dict(tile_bits=int(rng.integers(5, 9)), low_bits=2, defer_tail=1, apply_tail_mask=mask)
        state = dev(psi, backend)
        plan = engine.Plan(backend, n, ops, opts)
        plan.execute(state.buf)
        left = plan.residual()
        for q, m in left:
            assert not (mask >> q) & 1
            assert (m[0, 1] == 0 and m[1, 0] == 0) or (m[0, 0] == 0 and m[1, 1] == 0)
        seen += len(left)
        if left:
            engine.apply_lowered(state, [([q], m) for q, m in left], dict(tile_bits=opts["tile_bits"], low_bits=2))
        err = rel_err(state.to_numpy(), ref)
        assert err < RTOL, (n, opts, err)
    assert seen > 0


def check_dm_layers_vs_oracle(backend, n, depth, seed, db=10.0):
    """Config C3 at small N: noisy layered Clifford+T circuit on a density matrix."""
    noise = channels.GKPNoise(db)
    layers = workloads.dm_random_layers(n, depth, seed)
    circ = noise.noisy([g for layer in layers for g in layer])
    rho0 = np.zeros((2 ** n, 2 ** n), dtype=np.complex128)
    rho0[0, 0] = 1.0
    got = Simulator(circ, backend=backend).run(rho0)
    ref, _ = strided.run(as_oracle_ops(circ), rho0)
    err = rel_err(got, ref)
    assert err < RTOL, err
    assert abs(np.trace(got).real - 1.0) < 1e-12
    return err


def check_planner_features(backend):
    """The planner features of round 2, each with the condition that makes it fire:
    paired dense blocks (two (q, q+N) channels per round trip), rotations beyond 45 degrees
    (quarter turn left in the Pauli frame), narrow steps widened to the widest group of a
    pass, both CTA sizes -- all against the CPU oracle."""
    # 1. paired dense layers: a noisy density-matrix circuit needs fewer round trips than blocks
    n = 5
    noise = channels.GKPNoise(10.0)
    layers = workloads.dm_random_layers(n, 4, 3)
    circ = noise.noisy([g for layer in layers for g in layer])
    rho0 = np.zeros((2 ** n, 2 ** n), dtype=np.complex128)
    rho0[0, 0] = 1.0
    sim = Simulator(circ, backend=backend)
    got = sim.run(rho0)
    ref, _ = strided.run(as_oracle_ops(circ), rho0)
    assert rel_err(got, ref) < RTOL
    stats = sim.last_stats[0]
    assert stats["n_steps"] < stats["n_dense"], stats            # some blocks share a step
    # 2. rotations by every angle (RY-like real rotations and general unitaries), CZ in between
    rng = np.random.default_rng(77)
    n = 9
    for cta in (0, 7, 8):
        circ = []
        for layer in range(6):
            for q in range(n):
                th = rng.uniform(-np.pi, np.pi)
                c, s_ = np.cos(th / 2), np.sin(th / 2)
                ph = np.exp(1j * rng.uniform(-np.pi, np.pi))
                m = np.array([[c, -s_ * ph], [s_, c * ph]], dtype=np.complex128)
                circ.append(gates.Gate([q], m))
            for q in range(layer % 2, n - 1, 2):
                circ.append(gates.CZ(q, q + 1))
        psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        psi /= np.linalg.norm(psi)
        got = Simulator(circ, backend=backend, plan_options={"cta_log2": cta, "tile_bits": 8}).run(psi)
        ref, _ = strided.run(as_oracle_ops(circ), psi)
        assert rel_err(got, ref) < RTOL, cta
    # 3. a pass with one wide and several narrow steps (gates on 4 + 1 + 2 qubits, chained by CZ)
    n = 10
    circ = [gates.H(q) for q in range(4)] + [gates.CZ(0, 4), gates.H(4), gates.CZ(4, 5), gates.CZ(1, 6),
                                             gates.H(5), gates.H(6), gates.CZ(5, 6), gates.H(0)]
    psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
    psi /= np.linalg.norm(psi)
    got = Simulator(circ, backend=backend).run(psi)
    ref, _ = strided.run(as_oracle_ops(circ), psi)
    assert rel_err(got, ref) < RTOL


# ---- SURVEY section 8f rows, on the device: trajectories (f1), MB layering (f2), Cliffords (f3) ---
def _oracle_rho(circ, noise, n):
    """rho after the noisy circuit by the CPU oracle: dense operators and Kraus sums."""
    rho = np.zeros((2 ** n, 2 ** n), dtype=np.complex128)
    rho[0, 0] = 1.0
    for g in circ:
        rho = dense_ref.apply_matrix(rho, g.indices, g.matrix)
        for q, (px, pz) in zip(g.indices, noise.flips_for(g)):
            rho = dense_ref.apply_kraus(rho, [q], gkp_noise.pauli_flip_kraus(px, pz))
    return rho


def check_trajectories(backend, shots=4000):
    """f1: the batched Pauli-trajectory executor (qsim_traj_batch).
    (1) deterministic: every shot's ket equals the CPU oracle's run of the circuit with that
        shot's X / Z flips inserted as gates;
    (2) the batched and the shot-by-shot path draw the same trajectories from one seed;
    (3) statistical: the shot average converges to the ORACLE's density matrix (4 sigma)."""
    from quantum_computations_b200 import trajectories
    noise = channels.GKPNoise(7.0)                       # strong noise: errors in most shots
    n = 4
    circ = [gates.H(0), gates.CZ(0, 1), gates.T(1), gates.H(1), gates.CZ(1, 2), gates.P(2), gates.H(2),
            gates.SWAP(0, 2), gates.H(0), gates.CX(3, 1), gates.RZ(3, 0.37), gates.H(3), gates.CZ(3, 0), gates.Tdg(2)]
    psi0 = np.zeros(2 ** n, dtype=np.complex128)
    psi0[0] = 1.0
    ideal, _ = strided.run(as_oracle_ops(circ), psi0)
    # (1)
    rng = np.random.default_rng(5)
    flips = trajectories.sample_flips(circ, noise, 24, rng)
    res = trajectories.run_batch(circ, flips, psi0, backend=backend, observable=ideal, return_states=True)
    assert flips.any()
    for s in range(flips.shape[0]):
        explicit, col = [], 0
        for g in circ:
            explicit.append(g)
            for q in g.indices:
                if flips[s, col]:
                    explicit.append(gates.X(q))
                if flips[s, col + 1]:
                    explicit.append(gates.Z(q))
                col += 2
        ref, _ = strided.run(as_oracle_ops(explicit), psi0)
        assert rel_err(res["states"][s], ref) < RTOL, s
        assert abs(res["fidelities"][s] - abs(np.vdot(ideal, ref)) ** 2) < 1e-12
    # (2)
    a = trajectories.run_trajectories(circ, noise, [State.ZERO] * n, 12, np.random.default_rng(9), backend=backend,
                                      observable=ideal, batch=True)
    b = trajectories.run_trajectories(circ, noise, [State.ZERO] * n, 12, np.random.default_rng(9), backend=backend,
                                      observable=ideal, batch=False)
    assert np.abs(a["probabilities"] - b["probabilities"]).max() < 1e-12 and abs(a["fidelity"] - b["fidelity"]) < 1e-12
    # (3)
    rho = _oracle_rho(circ, noise, n)
    res = trajectories.run_trajectories(circ, noise, [State.ZERO] * n, shots, np.random.default_rng(7),
                                        backend=backend, observable=ideal)
    want_p = np.real(np.diagonal(rho))
    want_f = float(np.real(np.vdot(ideal, rho @ ideal)))
    tol = 4.0 * 0.5 / np.sqrt(shots)                      # binomial standard error <= 0.5 / sqrt(shots)
    assert np.max(np.abs(res["probabilities"] - want_p)) < tol
    assert abs(res["fidelity"] - want_f) < tol
    assert abs(res["probabilities"].sum() - 1.0) < 1e-12


def check_layered_noise(backend):
    """f2: a circuit scheduled into measurement-based layers (idle qubits charged with identity
    steps, Pauli gates as byproducts) and simulated with the per-layer GKP channel, against
    the CPU oracle's Kraus sums on the same scheduled circuit."""
    from quantum_computations_b200 import layering
    noise = channels.GKPNoise(9.0)
    n = 4
    circ = [gates.H(0), gates.CZ(0, 1), gates.X(2), gates.H(2), gates.T(3), gates.CZ(2, 3), gates.P(1),
            gates.SWAP(1, 2), gates.H(3), gates.Pdg(0), gates.CZ(0, 1), gates.H(1)]
    noisy = layering.noisy_circuit(circ, noise, n)
    lay = layering.MBLayering.of(circ, n)
    assert lay.depth() >= 4
    rho0 = np.zeros((2 ** n, 2 ** n), dtype=np.complex128)
    rho0[0, 0] = 1.0
    got = Simulator(noisy, backend=backend).run(rho0)
    ref, _ = strided.run(as_oracle_ops(noisy), rho0)
    assert rel_err(got, ref) < RTOL
    assert abs(np.trace(got).real - 1.0) < 1e-12


def check_clifford_rb(backend):
    """f3: uniform two-qubit Clifford RB (720 classes mod Paulis) through the batched executor:
    the inverse brings |00> back exactly; with the GKP channel the survival decays to 1/4;
    single sequences agree with the CPU oracle."""
    from quantum_computations_b200 import cliffords
    rng = np.random.default_rng(11)
    seqs = cliffords.clifford_rb_sequences(40, 6, rng)
    clean = BatchedSimulator(2, None, backend=backend).run(seqs)
    assert np.allclose(clean["fidelity"], 1.0, atol=1e-12)
    noise = channels.GKPNoise(6.0)
    noisy = BatchedSimulator(2, noise, backend=backend).run(seqs)
    for i in (0, 7, 23):
        rho = _oracle_rho(seqs[i], noise, 2)
        psi = np.array([1, 0, 0, 0], dtype=np.complex128)
        for g in seqs[i]:
            psi = dense_ref.apply_matrix(psi, g.indices, g.matrix)
        assert abs(noisy["fidelity"][i] - dense_ref.fidelity(rho, psi)) < 1e-12
        assert abs(noisy["purity"][i] - dense_ref.purity(rho)) < 1e-12
    long_seqs = cliffords.clifford_rb_sequences(40, 40, rng)
    f_long = BatchedSimulator(2, noise, backend=backend).run(long_seqs)["fidelity"].mean()
    assert abs(f_long - 0.25) < 0.03                                  # PAPER/plot_data.ipynb:188-189 asymptote


def check_nonblocking_run(backend):
    """Simulator.run(..., out=pinned, block=False): results of overlapping calls land in their own
    buffers and equal the blocking result."""
    n = 12
    circ = workloads.sv_random_circuit(n, 3, 5)
    sim = Simulator(circ, backend=backend)
    want = sim.run([State.ZERO] * n)
    outs = [backend.pinned_empty(1 << n) for _ in range(3)]
    pending = [sim.run([State.ZERO] * n, out=o, block=False) for o in outs]
    for p, o in zip(pending, outs):
        got = p.result()
        assert got is not None and np.shares_memory(got, o)
        assert rel_err(got, want) < 1e-15
        assert p.done()
    try:
        sim.run([State.ZERO] * n, block=False)
    except ValueError:
        pass
    else:
        raise AssertionError("block=False without out must raise")
