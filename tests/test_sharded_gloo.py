"""Multi-rank path on CPU: world_size 2, 4 and 8 over the gloo backend, every rank
running the host emulator on its shard.  Checks the stage scheduling, the multi-qubit
exchange (pack/unpack index arithmetic, pairing of the ranks), the diagonal-gate
restriction to rank bits, the rank relabelling by antidiagonal gates (flip flags) and
the final gather against the single-process oracle."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module", autouse=True)
def _emulator_built_once():
    """Build the emulator library in the parent, so that the spawned ranks only load it."""
    sys.path.insert(0, ROOT)
    from quantum_computations_b200.build_native import build_emu
    build_emu()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _leftover_circuit(gates, n, g):
    """Qubits 0..g-1 see only diagonal gates for a while, so the scheduler makes them the
    rank qubits; the other qubits end their first stage with leftovers that depend on the
    rank bits in all three ways: a scalar (left phases after CZ . H), a sign (CZ after the
    last H) and a bit flip (H . CZ . H)."""
    circ = []
    for q in range(g, n):
        a = (q - g) % g
        circ.append(gates.H(q))
        circ.append(gates.T(q))
        circ.append(gates.CZ(a, q))
        if q % 3 == 0:
            circ.append(gates.H(q))                    # H Z^v H = X^v
        elif q % 3 == 1:
            circ += [gates.RZ(q, 0.3 + q), gates.CZ((a + 1) % g, q)]
        else:
            circ += [gates.H(q), gates.T(q), gates.CZ((a + 1) % g, q)]
    circ += [gates.T(a) for a in range(g)] + [gates.H(a) for a in range(g)]       # ends the stage
    circ += [gates.H(q) for q in range(n)] + [gates.CZ(q, (q + 1) % n) for q in range(n)]
    return circ


def _worker(rank, world, port, n, depth, seed, out_dir):
    for p in (ROOT, HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from emu_backend import emu
        from golden.specs import as_oracle_ops
        from oracle import strided
        from parity_cases import random_circuit
        from quantum_computations_b200 import gates, sharded, workloads
        from quantum_computations_b200.states import State

        be = emu()
        comm = sharded.Comm()
        rng = np.random.default_rng(seed)                 # same circuit on every rank
        if depth == 0:
            circ = _leftover_circuit(gates, n, world.bit_length() - 1)
        else:
            circ = workloads.sv_random_circuit(n, depth, seed) + random_circuit(n, 25, rng)
        # leave every rank qubit complemented (and phased) at the end: the gather must undo it
        circ += [gates.Y(q) for q in range(n)] + [gates.CZ(0, n - 1), gates.T(1)]
        vecs = [State.PLUS.get(), State.T.get()] + [State.ZERO.get()] * (n - 2)
        st = sharded.ShardedState(n, comm, backend=be, as_torch=torch.from_numpy)
        sharded.ShardedState.CHUNK_LOG2 = 4                 # several chunks per block even at this size
        sim = sharded.ShardedSimulator(circ, st, plan_options=dict(tile_bits=6, low_bits=2))
        sim.prepare(vecs)
        sim.run()
        nrm = st.norm()
        got = st.gather_numpy()
        if rank == 0:
            psi0 = np.ones(1)
            for v in vecs:
                psi0 = np.kron(psi0, v)
            ref, _ = strided.run(as_oracle_ops(circ), psi0.astype(np.complex128))
            err = float(np.abs(got - ref).max() / np.abs(ref).max())
            np.save(os.path.join(out_dir, "result.npy"),
                    np.array([err, nrm, np.linalg.norm(ref), sim.stats["swaps"], comm.bytes_exchanged,
                              sim.stats["exchange_units"], sim.stats["relabels"],
                              sim.stats["carried_common"], sim.stats["carried_controlled"],
                              sim.stats["carried_signs"]]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 9), (4, 10), (8, 10)])
def test_sharded_matches_oracle(tmp_path, world, n):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, n, 12, 34, str(tmp_path)), nprocs=world, join=True)
    err, nrm, ref_norm, swaps, nbytes, units, flips, common, controlled, signs = np.load(tmp_path / "result.npy")
    print("exchanges", swaps, "units", units, "relabels", flips, "carried", common, signs, controlled)
    assert err < 1e-12
    assert abs(nrm - ref_norm) < 1e-12
    assert swaps > 0 and nbytes > 0                      # the rank-qubit path was exercised
    assert flips > 0                                     # the relabelling path was exercised
    assert common > 0                                    # leftovers of a plan were carried across an exchange


def _density_worker(rank, world, port, nq, out_dir):
    for p in (ROOT, HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from emu_backend import emu
        from oracle import dense_ref, gkp_noise
        from quantum_computations_b200 import channels, sharded, workloads
        from quantum_computations_b200.states import State

        comm = sharded.Comm()
        noise = channels.GKPNoise(9.0)
        layers = workloads.dm_random_layers(nq, 5, 21)
        clean = [g for layer in layers for g in layer]
        circ = noise.noisy(clean)                               # every gate followed by its Kraus channel(s)
        kets = [State.PLUS.get(), State.T.get()] + [State.ZERO.get()] * (nq - 2)
        st = sharded.ShardedState(2 * nq, comm, backend=emu(), as_torch=torch.from_numpy)
        sharded.ShardedState.CHUNK_LOG2 = 4
        sim = sharded.ShardedSimulator(circ, st, plan_options=dict(tile_bits=6, low_bits=2), density=True)
        sim.prepare(kets)
        sim.run()
        got = st.gather_numpy().reshape(2 ** nq, 2 ** nq)
        if rank == 0:
            psi = np.ones(1)
            for v in kets:
                psi = np.kron(psi, v)
            rho = np.outer(psi, np.conjugate(psi))
            for g in clean:
                rho = dense_ref.apply_matrix(rho, g.indices, g.matrix)
                for q, (px, pz) in zip(g.indices, noise.flips_for(g)):
                    rho = dense_ref.apply_kraus(rho, [q], gkp_noise.pauli_flip_kraus(px, pz))
            err = float(np.abs(got - rho).max() / np.abs(rho).max())
            np.save(os.path.join(out_dir, "density.npy"),
                    np.array([err, abs(np.trace(got) - 1.0), sim.stats["swaps"], sim.stats["passes"]]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,nq", [(2, 4), (4, 5)])
def test_sharded_density_matrix_matches_oracle(tmp_path, world, nq):
    """SURVEY 8e, second row: a vectorised density matrix (2N index bits) sharded by its
    first row qubits, with Kraus channels after every gate, against the oracle's
    U rho U^dagger / sum K rho K^dagger path."""
    port = _free_port()
    mp.spawn(_density_worker, args=(world, port, nq, str(tmp_path)), nprocs=world, join=True)
    err, trace_err, swaps, passes = np.load(tmp_path / "density.npy")
    assert err < 1e-12 and trace_err < 1e-12
    assert swaps > 0 and passes > 0


def _feedforward_circuit(gates, workloads, ClassicalControl, State, n):
    """Measurements of rank and local qubits, a qubit insertion, feed-forward, and random
    layers in between so that exchanges happen on the live layout."""
    circ = [gates.H(0), gates.CX(0, 1), gates.H(2), gates.CZ(2, 3), gates.T(3)]
    circ += workloads.sv_random_circuit(n, 3, 5)
    circ += [gates.MZ(0),                                     # reference qubit 0 starts as a rank qubit
             ClassicalControl(gates.X(0), [0]),               # (qubit numbers shift after a measurement)
             gates.Insert(2, State.PLUS), gates.H(3)]
    circ += workloads.sv_random_circuit(n, 2, 6)
    circ += [gates.MX(n - 1), ClassicalControl(gates.Z(1), [], [1]), gates.M(4, 0.3, 1.1)]
    circ += workloads.sv_random_circuit(n - 2, 3, 7)
    circ += [gates.Insert(0, State.T), gates.MZ(1), ClassicalControl(gates.H(0), [-1])]
    return circ


def _feedforward_worker(rank, world, port, n, out_dir):
    for p in (ROOT, HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from emu_backend import emu
        from quantum_computations_b200 import gates, sharded, workloads
        from quantum_computations_b200.simulator import ClassicalControl, Simulator
        from quantum_computations_b200.states import State

        be = emu()
        comm = sharded.Comm()
        circ = _feedforward_circuit(gates, workloads, ClassicalControl, State, n)
        kets = [State.PLUS.get(), State.T.get()] + [State.ZERO.get()] * (n - 2)
        worst, all_results = 0.0, []
        for seed in (1, 2, 3):
            st = sharded.ShardedState(n, comm, backend=be, as_torch=torch.from_numpy)
            sharded.ShardedState.CHUNK_LOG2 = 4
            sim = sharded.ShardedSimulator(circ, st, plan_options=dict(tile_bits=5, low_bits=1))
            np.random.seed(seed)                               # only rank 0 draws
            sim.run_circuit(kets)
            got = st.gather_numpy()
            if rank == 0:
                psi0 = np.ones(1)
                for v in kets:
                    psi0 = np.kron(psi0, v)
                np.random.seed(seed)
                single = Simulator(circ, backend=be)
                ref = single.run(psi0.astype(np.complex128))
                assert sim.results == single.results, (sim.results, single.results)
                assert got.shape == ref.shape
                worst = max(worst, float(np.abs(got - ref).max() / np.abs(ref).max()))
                all_results.append(tuple(sim.results))
        if rank == 0:
            np.save(os.path.join(out_dir, "feedforward.npy"),
                    np.array([worst, len(set(all_results)), sim.stats["swaps"], st.n]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 8), (4, 9)])
def test_sharded_measurement_insertion_feedforward(tmp_path, world, n):
    """Simulator.run semantics on a sharded ket: M on rank and local qubits (same outcome
    stream as the single-process simulator from the same seed), Insert, ClassicalControl."""
    port = _free_port()
    mp.spawn(_feedforward_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    worst, distinct, swaps, n_final = np.load(tmp_path / "feedforward.npy")
    assert worst < 1e-12
    assert n_final == n - 2                              # four measurements, two insertions
    assert distinct >= 2                                 # the seeds did not all give the same outcomes


def _exchange_worker(rank, world, port, n, out_dir):
    for p in (ROOT, HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from emu_backend import emu
        from quantum_computations_b200 import sharded

        comm = sharded.Comm()
        st = sharded.ShardedState(n, comm, backend=emu(), as_torch=torch.from_numpy)
        sharded.ShardedState.CHUNK_LOG2 = 3
        size = 1 << st.n_local
        st.buf[:] = np.arange(rank * size, (rank + 1) * size) * (1 + 0.5j)   # psi[i] = i (1 + i/2), identity layout
        want = np.arange(1 << n) * (1 + 0.5j)
        bad = 0
        nl, g = st.n_local, st.g
        plans = [[(nl, 0)], [(nl + g - 1, nl - 1)], [(nl + i, 2 * i + 1) for i in range(g)],
                 [(nl + i, nl - 2 - i) for i in range(g - 1, -1, -1)], [(nl, 3), (nl + g - 1, 0)][:g]]
        for pairs in plans:
            st.exchange(pairs)
            if not np.array_equal(st.gather_numpy(), want):              # the logical state never changes
                bad += 1
        # reductions over ranks: <a|b> and |<a|b>|^2 of two states in the same (permuted) layout
        other = sharded.ShardedState(n, comm, backend=emu(), as_torch=torch.from_numpy)
        other.phys, other.flip = list(st.phys), list(st.flip)
        rng = np.random.default_rng(5)
        full_b = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
        # lay `full_b` (logical order) out like st: physical index p takes logical index l with bit moves
        idx = np.arange(1 << n)
        logical_of_phys = np.zeros_like(idx)
        for l, p in enumerate(st.phys):
            logical_of_phys |= ((idx >> p) & 1) << l
        other.buf[:] = full_b[logical_of_phys][rank * size:(rank + 1) * size]
        inner = st.inner(other)
        want_inner = np.vdot(want, full_b)
        if abs(inner - want_inner) > 1e-9 * abs(want_inner) or abs(st.fidelity(other) - abs(want_inner) ** 2) > 1e-9 * abs(want_inner) ** 2:
            bad += 1
        if rank == 0:
            np.save(os.path.join(out_dir, "exchange.npy"), np.array([bad, st.swaps, sorted(st.phys) == list(range(n))]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 7), (4, 9), (8, 11)])
def test_multi_qubit_exchange_is_a_bit_permutation(tmp_path, world, n):
    """k rank bits <-> k local bits in one all-to-all (k = 1 .. log2 world): the data
    moves, the logical state does not."""
    port = _free_port()
    mp.spawn(_exchange_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    bad, swaps, ok = np.load(tmp_path / "exchange.npy")
    assert bad == 0 and swaps == 5 and ok


@pytest.mark.parametrize("world,n", [(2, 8), (4, 9), (8, 10)])
def test_leftovers_cross_an_exchange(tmp_path, world, n):
    """What a stage's plan leaves unapplied (qsim_plan_residual) depends on the rank bits;
    after the exchange it must come back as gates controlled by the qubits that were rank
    qubits: scalars, signs (CZ) and bit flips (block-diagonal gate)."""
    port = _free_port()
    mp.spawn(_worker, args=(world, port, n, 0, 5, str(tmp_path)), nprocs=world, join=True)
    err, nrm, ref_norm, swaps, nbytes, units, flips, common, controlled, signs = np.load(tmp_path / "result.npy")
    print("exchanges", swaps, "units", units, "carried", common, signs, controlled)
    assert err < 1e-12
    assert abs(nrm - ref_norm) < 1e-12
    assert signs > 0 and controlled > 0                 # (the scalar-only case is covered by the random circuits)


def test_sharded_simulator_refuses_non_matrix_gates(emu_backend):
    import types
    from quantum_computations_b200 import gates, sharded
    state = types.SimpleNamespace(n=5, g=1, n_local=4, backend=emu_backend, phys=list(range(5)), flip=[0],
                                  comm=types.SimpleNamespace(rank=0, size=2))
    with pytest.raises(NotImplementedError):
        sharded.ShardedSimulator([gates.H(0), gates.MZ(1)], state).compile()
    sim = sharded.ShardedSimulator([gates.H(0), gates.CZ(0, 4), gates.X(2)], state)
    assert [kind for kind, *_ in sim.compile()] == ["plan"]      # qubit 0 is made local by the initial layout
    assert sim.initial_phys != list(range(5)) and sim.stats["swaps"] == 0


# ---- SURVEY section 8e row 3: batches of independent RB circuits shard trivially ------------------
def _replica_worker(rank, world, port, out_dir):
    for p in (ROOT, HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from emu_backend import emu
        from quantum_computations_b200 import batched, channels, sharded, workloads

        comm = sharded.Comm()
        rng = np.random.default_rng(99)                   # the same batch on every rank
        circuits = [workloads.rb_random_circuit(2, (8, 10, 15, 20)[i % 4], rng) for i in range(37)]   # ragged split
        sim = batched.BatchedSimulator(2, channels.GKPNoise(10.0), backend=emu())
        joined = batched.run_replicas(sim, circuits, rank=rank, world=world, gather=comm.allgather_object)
        local = batched.run_replicas(sim, circuits, rank=rank, world=world)
        lo, hi = local["slice"]
        assert np.array_equal(joined["fidelity"][lo:hi], local["fidelity"])
        if rank == 0:
            whole = sim.run(circuits)                     # one process, whole batch
            np.save(os.path.join(out_dir, "replicas.npy"),
                    np.array([np.abs(joined["fidelity"] - whole["fidelity"]).max(),
                              np.abs(joined["purity"] - whole["purity"]).max(), len(joined["fidelity"])]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_rb_batch_splits_over_ranks_without_communication(tmp_path, world):
    """Every rank runs its contiguous slice of the batch; the gathered results equal the
    single-process run element for element (bit-exact: the same kernel on the same inputs)."""
    mp.spawn(_replica_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d0, d1, count = np.load(os.path.join(str(tmp_path), "replicas.npy"))
    assert count == 37
    assert d0 == 0.0 and d1 == 0.0
