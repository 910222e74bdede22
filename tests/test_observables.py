"""Pauli-sum expectation values (observables.py, qsim_expect_pauli / _dm): parsing of
PauliSum, kets and density matrices against a dense oracle on the host emulator and on the
GPU, the grouping of the terms into passes (launch counts), the npq.expect / expecth
dispatch, the sharded collective over gloo, and at 26 / 30 qubits on the GPU checks against
independent routes (the string applied as gates, product states)."""
import ctypes
import itertools
import os
import socket
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

from quantum_computations_b200 import engine, numpy_quantum as npq, observables  # noqa: E402
from quantum_computations_b200.observables import PauliError, PauliSum  # noqa: E402

_P = {"I": np.eye(2), "X": np.array([[0, 1], [1, 0]]), "Y": np.array([[0, -1j], [1j, 0]]),
      "Z": np.array([[1, 0], [0, -1]])}


# ---- dense oracle ------------------------------------------------------------------------
def dense(label: str) -> np.ndarray:
    out = np.ones((1, 1), dtype=np.complex128)
    for ch in label:
        out = np.kron(out, _P[ch])
    return out


def ket_ref(psi, labels):
    return np.array([np.vdot(psi, dense(s) @ psi) for s in labels])


def dm_ref(rho, labels):
    return np.array([np.trace(rho @ dense(s)) for s in labels])


def rel_err(got, ref) -> float:
    return float(np.abs(np.asarray(got) - np.asarray(ref)).max() / max(np.abs(ref).max(), 1e-300))


def rand_ket(n, rng):
    psi = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    return psi / np.linalg.norm(psi)


def labels_for(n, rng, count=60):
    if n <= 3:
        return ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    found = dict.fromkeys("".join(rng.choice(list("IXYZ"), n)) for _ in range(count))
    found.update(dict.fromkeys(["I" * n, "Z" * n, "X" * n, "Y" * n, "X" + "I" * (n - 2) + "Y"]))
    return list(found)


def launches(be) -> int:
    return int(be.lib.qsim_launch_count())


# ---- PauliSum ---------------------------------------------------------------------------------
def test_paulisum_parsing_and_merging():
    ps = PauliSum([(0.5, "XIZ"), (2, {0: "x", 2: "Z"}), (1j, {1: "-y"}), (3, {2: [0, 0, -1]}), (1, {0: -1})])
    assert len(ps) == 4 and ps.num_qubits == 3
    assert ps.coeffs[0] == 2.5                        # "XIZ" and {0: x, 2: Z} merged
    assert list(ps.x_masks) == [0b001, 0b010, 0, 0b001] and list(ps.z_masks) == [0b100, 0b010, 0b100, 0]
    assert ps.coeffs[1] == -1j and ps.coeffs[2] == -3 and ps.coeffs[3] == -1
    assert ps.x_masks.dtype == np.uint64 and ps.coeffs.dtype == np.complex128
    assert "XIZ" in repr(ps)
    for bad in ([(1, "XQ")], [(1, {0: "w"})], [(1, {-1: "x"})], [(1, 5)], [1.0]):
        with pytest.raises(PauliError):
            PauliSum(bad)


def test_paulisum_matrix_is_the_kronecker_product():
    ps = PauliSum([(0.3, "XYZ"), (-1.5, "IZI"), (0.25j, {3: "Y"})])
    want = 0.3 * np.kron(dense("XYZ"), np.eye(2)) - 1.5 * dense("IZII") + 0.25j * dense("IIIY")
    assert np.array_equal(ps.matrix(4), want)
    assert np.array_equal(PauliSum([(1, "Y")]).matrix(), _P["Y"])
    with pytest.raises(ValueError):
        ps.matrix(2)


# ---- check functions, run on both backends ----------------------------------------------------------
def check_kets(be, sizes, seed=3):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi = rand_ket(n, rng)
        labels = labels_for(n, rng)
        ps = PauliSum([(1.0, s) for s in labels])
        st = engine.DeviceState.from_numpy(psi, be)
        got = observables.expect(ps, st, per_term=True)
        assert got.dtype == np.float64                       # real by construction
        ref = ket_ref(psi, labels)
        assert np.abs(ref.imag).max() < 1e-12
        assert rel_err(got, ref.real) <= 1e-12, n
        again = st.expect_pauli(ps.x_masks, ps.z_masks)
        assert np.array_equal(got, again)                    # bit-identical repeat
        coeffs = rng.normal(size=len(labels))
        total = observables.expect(PauliSum(zip(coeffs, labels)), st)
        assert abs(total - np.dot(coeffs, ref.real)) <= 1e-12 * np.abs(coeffs).sum()


def check_density_matrices(be, sizes, seed=4):
    rng = np.random.default_rng(seed)
    for N in sizes:
        psi = rand_ket(N, rng)
        rho = np.outer(psi, psi.conj())
        skew = rho + 0.3 * (rng.normal(size=rho.shape) + 1j * rng.normal(size=rho.shape))   # not Hermitian
        labels = labels_for(N, rng, 40)
        ps = PauliSum([(1.0, s) for s in labels])
        for mat in (rho, skew):
            st = engine.DeviceState.from_numpy(mat, be)
            got = observables.expect(ps, st, per_term=True)
            assert got.dtype == np.complex128
            assert rel_err(got, dm_ref(mat, labels)) <= 1e-12, N


def check_grouping(be):
    rng = np.random.default_rng(7)
    n = 10
    psi = rand_ket(n, rng)
    st = engine.DeviceState.from_numpy(psi, be)

    def run(ps):
        before = launches(be)
        got = st.expect_pauli(ps.x_masks, ps.z_masks)
        return got, launches(be) - before

    # all Z strings: one pass + the final sum
    zonly = PauliSum([(1, {q: "Z"}) for q in range(n)] + [(1, {q: "Z", q + 1: "Z"}) for q in range(n - 1)])
    got, count = run(zonly)
    assert count == 2
    # every X mask inside qubits {2, 3, 5, 8} (a 4-dimensional span), with Z strings: one pass
    sub = [2, 3, 5, 8]
    labels = []
    for k in range(1, 16):
        chosen = [sub[i] for i in range(4) if k >> i & 1]
        labels.append({q: ("Y" if q == chosen[0] else "X") for q in chosen} | {0: "Z"})
    labels.append({1: "Z", 9: "Z"})
    got, count = run(PauliSum([(1, lab) for lab in labels]))
    assert count == 2
    ref = ket_ref(psi, [observables.PauliSum([(1, lab)])._label_n(n) for lab in labels])
    assert rel_err(got, ref.real) <= 1e-12
    # 200 terms over 40 X masks: several passes, caller order
    masks = rng.choice(1 << n, size=40, replace=False)
    terms = []
    for t in range(200):
        x, z = int(masks[t % 40]), int(rng.integers(1 << n))
        terms.append({q: "IXZY"[((x >> q) & 1) | (((z >> q) & 1) << 1)] for q in range(n)})
    ps = PauliSum([(1, lab) for lab in terms])
    got, count = run(ps)
    assert 3 <= count - 1 <= len(set(int(v) for v in ps.x_masks))
    assert rel_err(got, ket_ref(psi, [ps._label_n(n, t) for t in range(len(ps))]).real) <= 1e-12
    # the lowest and highest index bits, the identity, an empty call
    edge = PauliSum([(1, {0: "X"}), (1, {n - 1: "Y"}), (1, {0: "Y", n - 1: "X"}), (1, {}), (1, "Z" * n)])
    got, _ = run(edge)
    assert rel_err(got, ket_ref(psi, [edge._label_n(n, t) for t in range(len(edge))]).real) <= 1e-12
    assert abs(got[3] - 1.0) < 1e-12
    got, count = run(PauliSum([]))
    assert count == 0 and got.shape == (0,)
    rc = be.lib.qsim_expect_pauli(be.ptr(st.buf), n, 0, None, None, None, be.stream())
    assert rc == 0
    # masks at or above n, and n out of range
    for x, z in ((1 << n, 0), (0, 1 << n), (1 << 63, 0)):
        with pytest.raises(ValueError):
            st.expect_pauli([x], [z])
    out = np.zeros(1)
    one = np.ones(1, dtype=np.uint64)
    assert be.lib.qsim_expect_pauli(be.ptr(st.buf), 64, 1, one.ctypes.data, one.ctypes.data,
                                    out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), be.stream()) == -1


def check_against_measure_probs(be):
    rng = np.random.default_rng(11)
    n = 9
    psi = rand_ket(n, rng)
    st = engine.DeviceState.from_numpy(psi, be)
    zs = st.expect_pauli([0] * n, [1 << q for q in range(n)])
    from quantum_computations_b200 import _capi
    for q in range(n):
        probs = np.zeros(2)
        b0, b1 = np.array([1, 0], dtype=np.complex128), np.array([0, 1], dtype=np.complex128)
        _capi.check(be.lib, be.lib.qsim_measure_probs(be.ptr(st.buf), n, q, b0.view(np.float64).ctypes.data_as(_capi.c_double_p),
                                                      b1.view(np.float64).ctypes.data_as(_capi.c_double_p),
                                                      probs.ctypes.data_as(_capi.c_double_p), be.stream()))
        assert abs(zs[q] - (probs[0] - probs[1])) <= 1e-12


def check_npq_dispatch(be):
    rng = np.random.default_rng(12)
    n = 6
    psi = rand_ket(n, rng)
    st = engine.DeviceState.from_numpy(psi, be)
    ps = PauliSum([(0.7, "XXIIZY"), (-0.2, "ZIIIII"), (1.5j, "IYYIII")])
    host = st.to_numpy(mirror_dtype=False)
    want = np.vdot(host, ps.matrix(n) @ host)
    assert abs(npq.expect(ps, st) - want) <= 1e-12
    assert abs(npq.expecth(ps, st) - want.real) <= 1e-12
    oper = rng.normal(size=(1 << n, 1 << n)) + 1j * rng.normal(size=(1 << n, 1 << n))
    assert abs(npq.expect(oper, st) - np.vdot(host, oper @ host)) <= 1e-12 * np.abs(oper).sum()
    assert abs(npq.expecth(oper, st) - np.vdot(host, oper @ host).real) <= 1e-12 * np.abs(oper).sum()
    dm = engine.DeviceState.from_numpy(np.outer(psi, psi.conj()), be)
    with pytest.raises(TypeError):
        npq.expect(oper, dm)
    with pytest.raises(TypeError):
        npq.expect(np.eye(4), st)
    assert abs(npq.expect(ps, dm) - want) <= 1e-12


def _label_n(self, n, t=0):
    return "".join("IXYZ"[p] for p in self._letters(t, n))


PauliSum._label_n = _label_n          # test helper: the dense-oracle label of term t on n qubits


# ---- emulator ------------------------------------------------------------------------------------
def test_kets_emulator(emu_backend):
    check_kets(emu_backend, range(1, 13))


def test_density_matrices_emulator(emu_backend):
    check_density_matrices(emu_backend, range(1, 7))


def test_grouping_emulator(emu_backend):
    check_grouping(emu_backend)


def test_against_measure_probs_emulator(emu_backend):
    check_against_measure_probs(emu_backend)


def test_npq_dispatch_emulator(emu_backend):
    check_npq_dispatch(emu_backend)


def test_host_ndarray_host_operator_unchanged():
    psi = np.array([0.6, 0.8j])
    assert npq.expect(_P["Y"], psi) == np.vdot(psi, _P["Y"] @ psi)


# ---- GPU -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_kets_gpu(cuda_backend):
    check_kets(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_density_matrices_gpu(cuda_backend):
    check_density_matrices(cuda_backend, range(1, 7))


@pytest.mark.gpu
def test_grouping_gpu(cuda_backend):
    check_grouping(cuda_backend)


@pytest.mark.gpu
def test_against_measure_probs_gpu(cuda_backend):
    check_against_measure_probs(cuda_backend)


@pytest.mark.gpu
def test_npq_dispatch_gpu(cuda_backend):
    check_npq_dispatch(cuda_backend)
    psi = rand_ket(5, np.random.default_rng(2))
    ps = PauliSum([(1, "XZIIY")])
    assert abs(npq.expect(ps, psi) - np.vdot(psi, dense("XZIIY") @ psi)) <= 1e-12     # host array is uploaded


@pytest.mark.gpu
@pytest.mark.parametrize("n", [26, 30])
def test_large_states_gpu(cuda_backend, n):
    """No oracle at this size: <P> against inner(psi, P psi) with P psi from the fused gate path,
    product states with known values, bit-identical repeats."""
    import torch
    from quantum_computations_b200 import workloads
    be = cuda_backend
    st = engine.DeviceState.product([np.array([1, 0], dtype=np.complex128)] * n, be)
    circ = workloads.sv_random_circuit(n, 2, 5)
    for g in circ:
        st = g.apply(st)
    strings = [{0: "X", 1: "Y", n - 1: "Z"}, {3: "Y", 17: "Y"}, {q: "X" for q in range(0, n, 3)},
               {q: "Z" for q in range(n)}, {5: "Z", 6: "Z"}, {n - 1: "X", n - 2: "Y"}]
    ps = PauliSum([(1, s) for s in strings])
    got = st.expect_pauli(ps.x_masks, ps.z_masks)
    assert np.array_equal(got, st.expect_pauli(ps.x_masks, ps.z_masks))
    for t, s in enumerate(strings):
        moved = st.copy()
        engine.apply_lowered(moved, [([q], _P[ch].astype(np.complex128)) for q, ch in sorted(s.items())])
        want = st.inner(moved)
        del moved
        torch.cuda.empty_cache()
        assert abs(want.imag) < 1e-9
        assert abs(got[t] - want.real) <= 1e-12 * max(1.0, abs(want.real)) + 1e-13, (s, got[t], want)
    del st
    torch.cuda.empty_cache()
    plus = np.array([1, 1], dtype=np.complex128) / np.sqrt(2)
    zero = np.array([1, 0], dtype=np.complex128)
    prod = engine.DeviceState.product([plus if q % 2 == 0 else zero for q in range(n)], be)
    checks = PauliSum([(1, {0: "X"}), (1, {1: "Z"}), (1, {0: "X", 1: "Z", n - 2: "X"}), (1, {0: "Z"}),
                       (1, {1: "X"}), (1, {0: "Y"})])
    vals = prod.expect_pauli(checks.x_masks, checks.z_masks)
    assert abs(vals[0] - 1) < 1e-12 and abs(vals[1] - 1) < 1e-12 and abs(vals[2] - 1) < 1e-12
    assert abs(vals[3]) < 1e-12 and abs(vals[4]) < 1e-12 and abs(vals[5]) < 1e-12


# ---- sharded collective over gloo --------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _sharded_worker(rank, world, port, n, out_dir):
    import torch
    import torch.distributed as dist
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

        comm = sharded.Comm()
        rng = np.random.default_rng(21)
        circ = workloads.sv_random_circuit(n, 6, 8) + random_circuit(n, 15, rng)
        circ += [gates.Y(q) for q in range(n)] + [gates.CZ(0, n - 1), gates.T(1)]   # flipped rank qubits
        vecs = [State.PLUS.get(), State.T.get()] + [State.ZERO.get()] * (n - 2)
        st = sharded.ShardedState(n, comm, backend=emu(), as_torch=torch.from_numpy)
        sharded.ShardedState.CHUNK_LOG2 = 4
        opts = dict(tile_bits=6, low_bits=2)
        sim = sharded.ShardedSimulator(circ, st, plan_options=opts)
        sim.prepare(vecs)
        sim.run()
        rank_q = [n - 1 - l for l in range(n) if st.phys[l] >= st.n_local]
        relabel = [gates.Y(q) for q in rank_q]              # antidiagonal on rank qubits: flip flags
        pre = sharded.ShardedSimulator(relabel, st, plan_options=opts)
        pre.compile(fixed_layout=True)
        pre.run()
        circ = circ + relabel
        flipped = sum(st.flip)
        before = st.gather_numpy()
        local_q = [n - 1 - l for l in range(n) if st.phys[l] < st.n_local]
        r0, r1 = rank_q[0], rank_q[-1]
        terms = [{r0: "X", local_q[0]: "Z"}, {r1: "Y", local_q[1]: "X"}, {r0: "Z", local_q[2]: "Y"},
                 {r0: "Z", r1: "Z"}, {r0: "X", r1: "Y", local_q[3]: "Z"}, {local_q[0]: "X", local_q[4]: "Y"},
                 {r1: "Z"}, {}]
        for _ in range(10):
            qs = rng.choice(n, size=3, replace=False)
            terms.append({int(q): "XYZ"[int(rng.integers(3))] for q in qs})
        ps = PauliSum([(rng.normal(), t) for t in terms])
        swaps0 = st.swaps
        got = st.expect(ps, per_term=True)
        total = st.expect(ps)
        after = st.gather_numpy()
        everyone = comm.allgather_object(got.tobytes())
        more = workloads.sv_random_circuit(n, 2, 9)
        sub = sharded.ShardedSimulator(more, st, plan_options=opts)
        sub.compile(fixed_layout=True)
        sub.run()
        final = st.gather_numpy()
        if rank == 0:
            labels = ["".join("IXYZ"[p] for p in ps._letters(t, n)) for t in range(len(ps))]
            ref = ket_ref(before, labels).real
            psi0 = np.ones(1)
            for v in vecs:
                psi0 = np.kron(psi0, v)
            want_final, _ = strided.run(as_oracle_ops(circ + more), psi0.astype(np.complex128))
            np.save(os.path.join(out_dir, "sharded.npy"),
                    np.array([rel_err(got, ref), abs(total - np.dot(ps.coeffs, ref)),
                              float(all(b == everyone[0] for b in everyone)),
                              rel_err(after, before), rel_err(final, want_final), st.swaps - swaps0, flipped]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 9), (4, 10), (8, 10)])
def test_sharded_expect_matches_oracle(tmp_path, world, n):
    import torch.multiprocessing as mp
    from quantum_computations_b200.build_native import build_emu
    build_emu()
    mp.spawn(_sharded_worker, args=(world, _free_port(), n, str(tmp_path)), nprocs=world, join=True)
    err, total_err, same, moved, final_err, swaps, flipped = np.load(tmp_path / "sharded.npy")
    assert err <= 1e-12 and total_err <= 1e-12
    assert same == 1.0                                   # identical on every rank
    assert moved <= 1e-12                                # the logical state did not change
    assert final_err <= 1e-12                            # and later gates still see the right state
    assert swaps >= 1 and flipped >= 1                   # rank qubits were exchanged, some complemented


def test_sharded_density_matrix_is_refused(emu_backend):
    import types
    from quantum_computations_b200 import sharded
    st = sharded.ShardedState.__new__(sharded.ShardedState)
    st.is_density = True
    with pytest.raises(NotImplementedError):
        st.expect_pauli([0], [1])
    state = types.SimpleNamespace(n=4, g=1, n_local=3, backend=emu_backend, phys=list(range(4)), flip=[0],
                                  comm=types.SimpleNamespace(rank=0, size=2))
    sharded.ShardedSimulator([], state, density=True)
    assert state.is_density
