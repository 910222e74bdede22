"""Pauli-string rotations (qsim_apply_pauli_rotations / _dm, DeviceState.apply_pauli_rotations,
ShardedState.apply_pauli_rotations) and Trotterised evolution (observables.evolve): kets and
density matrices against dense exp(-i theta/2 P) products on the host emulator and on the GPU,
the packing of rotations into passes (launch counts), argument checks of both libraries, the
sharded collective over gloo, and on the GPU checks at 26 to 30 qubits against closed forms and
against the same evolution lowered to gates through the planner."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import scipy.linalg

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

from quantum_computations_b200 import _capi, build_native, engine, observables  # noqa: E402
from quantum_computations_b200.observables import PauliSum  # noqa: E402

CAP = 32                                     # QS_PAULI_ROT_MAX (plan.h)


# ---- dense oracle ------------------------------------------------------------------------
def masks_of(labels):
    ps = [PauliSum([(1, lab)]) for lab in labels]
    return (np.array([int(p.x_masks[0]) if len(p) else 0 for p in ps], dtype=np.uint64),
            np.array([int(p.z_masks[0]) if len(p) else 0 for p in ps], dtype=np.uint64))


def pauli_apply(psi, x, z, n):
    """P psi for the string (x, z) (bit q = reference qubit q = index bit n-1-q), P = i^popc(x&z) X^x Z^z."""
    xi = sum(1 << (n - 1 - q) for q in range(n) if int(x) >> q & 1)
    zi = sum(1 << (n - 1 - q) for q in range(n) if int(z) >> q & 1)
    idx = np.arange(1 << n)
    par = np.array([bin(v).count("1") & 1 for v in range(1 << n)])
    src = idx ^ xi
    return (1j ** (bin(int(x) & int(z)).count("1") % 4)) * np.where(par[src & zi], -1, 1) * psi[src]


def rotate_ref(psi, labels, angles, n):
    """exp(-i theta/2 P) = cos(theta/2) - i sin(theta/2) P (P^2 = 1), in caller order."""
    x, z = masks_of(labels)
    out = psi.copy()
    for xv, zv, th in zip(x, z, angles):
        out = np.cos(th / 2) * out - 1j * np.sin(th / 2) * pauli_apply(out, xv, zv, n)
    return out


def dense_unitary(labels, angles, n):
    u = np.eye(1 << n, dtype=np.complex128)
    for lab, th in zip(labels, angles):
        u = scipy.linalg.expm(-0.5j * th * PauliSum([(1, lab)]).matrix(n)) @ u
    return u


def rel_err(got, ref) -> float:
    return float(np.abs(np.asarray(got) - np.asarray(ref)).max() / max(np.abs(ref).max(), 1e-300))


def rand_ket(n, rng):
    psi = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    return psi / np.linalg.norm(psi)


def rotation_list(n, rng, count=14):
    """Identity, Z-only, Y-heavy, wide-X and random strings; angles with 0, +-pi and 2 pi."""
    labels = ["I" * n, "Z" * n, "Y" * n, "X" * n, "X" + "I" * (n - 1), "I" * (n - 1) + "Y"]
    labels += ["".join(rng.choice(list("IXYZ"), n)) for _ in range(count - len(labels))]
    angles = list(rng.uniform(-4, 4, size=len(labels)))
    for k, special in enumerate((0.0, np.pi, -np.pi, 2 * np.pi)):
        angles[(3 * k + 1) % len(labels)] = special
    return labels, np.array(angles)


def launches(be) -> int:
    return int(be.lib.qsim_launch_count())


def heisenberg(n, jx=1.0, jy=0.8, jz=0.6, h=0.3):
    terms = []
    for q in range(n - 1):
        for p, j in (("X", jx), ("Y", jy), ("Z", jz)):
            terms.append((j, {q: p, q + 1: p}))
    terms += [(h * (1 + 0.1 * q), {q: "Z"}) for q in range(n)]
    return PauliSum(terms)


# ---- check functions, run on both backends ----------------------------------------------------------
def check_kets(be, sizes, seed=5):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi = rand_ket(n, rng)
        labels, angles = rotation_list(n, rng)
        x, z = masks_of(labels)
        st = engine.DeviceState.from_numpy(psi, be)
        assert st.apply_pauli_rotations(x, z, angles) is st
        want = dense_unitary(labels, angles, n) @ psi if n <= 6 else rotate_ref(psi, labels, angles, n)
        assert rel_err(st.to_numpy(), want) <= 1e-12, n
        if n <= 6:
            assert rel_err(rotate_ref(psi, labels, angles, n), want) <= 1e-13
        if n >= 2:                                  # caller order matters: X_0 and Z_0 do not commute
            lab = ["X" + "I" * (n - 1), "Z" + "Y" * (n - 1)]
            xs, zs = masks_of(lab)
            fwd = engine.DeviceState.from_numpy(psi, be).apply_pauli_rotations(xs, zs, [0.7, 1.1]).to_numpy()
            bwd = engine.DeviceState.from_numpy(psi, be).apply_pauli_rotations(xs[::-1], zs[::-1],
                                                                               [1.1, 0.7]).to_numpy()
            assert rel_err(fwd, rotate_ref(psi, lab, [0.7, 1.1], n)) <= 1e-12
            assert np.abs(fwd - bwd).max() > 1e-3


def check_density_matrices(be, sizes, seed=6):
    rng = np.random.default_rng(seed)
    for N in sizes:
        a = rng.normal(size=(1 << N, 1 << N)) + 1j * rng.normal(size=(1 << N, 1 << N))
        rho = a @ a.conj().T
        rho /= np.trace(rho)
        labels, angles = rotation_list(N, rng, 10)
        x, z = masks_of(labels)
        st = engine.DeviceState.from_numpy(rho, be).apply_pauli_rotations(x, z, angles)
        got = st.to_numpy()
        u = dense_unitary(labels, angles, N)
        assert rel_err(got, u @ rho @ u.conj().T) <= 1e-12, N
        assert abs(np.trace(got) - 1.0) <= 1e-12
        assert np.abs(got - got.conj().T).max() <= 1e-13


def check_packing(be):
    rng = np.random.default_rng(8)
    n = 10
    st = engine.DeviceState.from_numpy(rand_ket(n, rng), be)

    def count(x, z, angles=None, state=st):
        angles = rng.uniform(0.1, 1.0, size=len(x)) if angles is None else angles
        before = launches(be)
        state.apply_pauli_rotations(x, z, angles)
        return launches(be) - before

    zmasks = rng.integers(1, 1 << n, size=2 * CAP + 1).astype(np.uint64)
    zero = np.zeros_like(zmasks)
    assert count(zero[:CAP], zmasks[:CAP]) == 1                  # cap-many Z-only rotations: one pass
    assert count(zero[:CAP + 1], zmasks[:CAP + 1]) == 2          # the cap is respected
    assert count(zero, zmasks) == 3
    # X masks in the span of qubits {2, 3, 5, 8}: one pass
    sub = [2, 3, 5, 8]
    xs = [sum(1 << sub[i] for i in range(4) if k >> i & 1) for k in range(1, 16)] * 2
    assert count(np.array(xs, dtype=np.uint64), rng.integers(0, 1 << n, size=len(xs)).astype(np.uint64)) == 1
    # single X on qubits 0..4, then 0..3 again: runs stay contiguous (no reordering), at most four
    # generators each: [x0 x1 x2 x3] [x4 x0 x1 x2] [x3]
    seq = [1 << q for q in range(5)] + [1 << q for q in range(4)]
    assert count(np.array(seq, dtype=np.uint64), np.zeros(len(seq), dtype=np.uint64)) == 3
    # angle 0 is the identity: nothing to launch
    assert count(np.array([1, 3], dtype=np.uint64), np.array([2, 0], dtype=np.uint64), np.zeros(2)) == 0
    # density matrix: each rotation's row and column halves share a pass (two generators per X mask)
    N = 5
    dm = engine.DeviceState.from_numpy(np.eye(1 << N) / (1 << N), be)
    single = np.array([1 << q for q in range(3)], dtype=np.uint64)
    assert count(single[:1], np.zeros(1, dtype=np.uint64), state=dm) == 1
    assert count(single[:2], np.zeros(2, dtype=np.uint64), state=dm) == 1
    assert count(single, np.zeros(3, dtype=np.uint64), state=dm) == 2
    assert count(np.zeros(CAP // 2, dtype=np.uint64), np.arange(1, CAP // 2 + 1, dtype=np.uint64), state=dm) == 1
    assert count(np.zeros(CAP // 2 + 1, dtype=np.uint64), np.arange(1, CAP // 2 + 2, dtype=np.uint64),
                 state=dm) == 2


def check_edges(be):
    rng = np.random.default_rng(9)
    n = 7
    st = engine.DeviceState.from_numpy(rand_ket(n, rng), be)
    before = be.download(st.buf).copy()
    assert be.lib.qsim_apply_pauli_rotations(be.ptr(st.buf), n, 0, None, None, None, be.stream()) == 0
    assert be.lib.qsim_apply_pauli_rotations(None, n, 0, None, None, None, be.stream()) == 0
    st.apply_pauli_rotations([], [], [])
    assert np.array_equal(be.download(st.buf).view(np.uint64), before.view(np.uint64))
    st.apply_pauli_rotations([3, 0, 1 << (n - 1)], [1, 5, 0], [0.0, 0.0, -0.0])
    assert np.array_equal(be.download(st.buf).view(np.uint64), before.view(np.uint64))
    # the global phase of the identity string
    st.apply_pauli_rotations([0], [0], [0.8])
    assert rel_err(be.download(st.buf), np.exp(-0.4j) * before) <= 1e-15
    with pytest.raises(ValueError):
        st.apply_pauli_rotations([1], [0], [0.1, 0.2])
    for x, z, a in (([1 << n], [0], [0.1]), ([0], [1 << n], [0.1]), ([1], [0], [np.nan]), ([1], [0], [np.inf])):
        with pytest.raises(ValueError):
            st.apply_pauli_rotations(x, z, a)


def check_evolve(be):
    n = 4
    h = heisenberg(n)
    rng = np.random.default_rng(10)
    psi = rand_ket(n, rng)
    t = 0.9
    hm = h.matrix(n)
    exact = scipy.linalg.expm(-1j * t * hm) @ psi
    terms = [h.coeffs[k].real * PauliSum([(1, h._label_n(n, k))]).matrix(n) for k in range(len(h))]
    errs = {1: [], 2: []}
    for order in (1, 2):
        for steps in (4, 8, 16):
            dt = t / steps
            step = [scipy.linalg.expm(-1j * dt * m) for m in terms]
            if order == 2:
                half = [scipy.linalg.expm(-0.5j * dt * m) for m in terms]
                step = half[:-1] + step[-1:] + half[:-1][::-1]
            u = np.eye(1 << n, dtype=np.complex128)
            for _ in range(steps):
                for g in step:
                    u = g @ u
            got = observables.evolve(h, engine.DeviceState.from_numpy(psi, be), t, steps=steps, order=order)
            assert rel_err(got.to_numpy(), u @ psi) <= 1e-12, (order, steps)
            errs[order].append(np.abs(got.to_numpy() - exact).max())
    r1 = errs[1][0] / errs[1][2]
    r2 = errs[2][0] / errs[2][2]
    assert 3.0 < r1 < 5.5, errs                # 1/steps: four times the steps, a quarter of the error
    assert 12.0 < r2 < 20.0, errs              # 1/steps^2
    # commuting terms (identity included): exact, phase and all
    zz = PauliSum([(0.7, "ZZII"), (-0.4, "IIZZ"), (1.3, "IIII"), (0.2, "ZIIZ")])
    got = observables.evolve(zz, engine.DeviceState.from_numpy(psi, be), 1.7)
    assert rel_err(got.to_numpy(), scipy.linalg.expm(-1.7j * zz.matrix(n)) @ psi) <= 1e-12
    rho = np.outer(psi, psi.conj())
    got = observables.evolve(h, engine.DeviceState.from_numpy(rho, be), t, steps=3, order=2).to_numpy()
    want = observables.evolve(h, engine.DeviceState.from_numpy(psi, be), t, steps=3, order=2).to_numpy()
    assert rel_err(got, np.outer(want, want.conj())) <= 1e-12
    with pytest.raises(ValueError):
        observables.evolve(PauliSum([(1j, "XX")]), engine.DeviceState.from_numpy(psi, be), 0.1)
    with pytest.raises(ValueError):
        observables.evolve(h, engine.DeviceState.from_numpy(psi, be), 0.1, order=3)
    with pytest.raises(ValueError):
        observables.evolve(heisenberg(n + 1), engine.DeviceState.from_numpy(psi, be), 0.1)
    # <Z_q> = cos(theta) after exp(-i theta/2 Y_q) on |0...0>
    zero = np.zeros(1 << 5, dtype=np.complex128)
    zero[0] = 1.0
    for q, th in ((0, 0.3), (2, 2.0), (4, -1.2)):
        st = engine.DeviceState.from_numpy(zero, be).apply_pauli_rotations([1 << q], [1 << q], [th])
        assert abs(observables.expect(PauliSum([(1, {q: "Z"})]), st) - np.cos(th)) <= 1e-14


def test_trotter_rotations_merge_and_order():
    h = PauliSum([(0.5, "XX"), (0.25, "ZI"), (-1.0, "IY")])
    x, z, a = observables.trotter_rotations(h, 0.4, steps=2, order=1)
    assert list(x) == list(h.x_masks) * 2 and np.allclose(a, [0.2, 0.1, -0.4] * 2)
    x, z, a = observables.trotter_rotations(h, 0.4, steps=2, order=2)
    # XX/2 ZI/2 IY ZI/2 XX/2 | XX/2 ... : the two XX halves between the steps merge
    assert list(x) == [int(h.x_masks[k]) for k in (0, 1, 2, 1, 0, 1, 2, 1, 0)]
    assert np.allclose(a, [0.1, 0.05, -0.4, 0.05, 0.2, 0.05, -0.4, 0.05, 0.1])
    x, z, a = observables.trotter_rotations(PauliSum([(1.0, "Z")]), 1.0, steps=5, order=2)
    assert len(a) == 1 and np.isclose(a[0], 2.0)
    with pytest.raises(ValueError):
        observables.trotter_rotations(h, 1.0, steps=0)


# ---- emulator ------------------------------------------------------------------------------------
def test_kets_emulator(emu_backend):
    check_kets(emu_backend, range(1, 13))


def test_density_matrices_emulator(emu_backend):
    check_density_matrices(emu_backend, range(1, 7))


def test_packing_emulator(emu_backend):
    check_packing(emu_backend)


def test_edges_emulator(emu_backend):
    check_edges(emu_backend)


def test_evolve_emulator(emu_backend):
    check_evolve(emu_backend)


@pytest.fixture(scope="module", params=["cuda", "emu"])
def lib(request):
    lib = ctypes.CDLL(build_native.build_cuda() if request.param == "cuda" else build_native.build_emu())
    _capi.declare(lib)
    return lib


def test_argument_checks(lib):
    """Both libraries refuse the same calls with the same message, before any device work (the
    buffers are host arrays)."""
    st = np.zeros(64, dtype=np.complex128)
    one = np.ones(1, dtype=np.uint64)
    zero = np.zeros(1, dtype=np.uint64)
    big = np.array([1 << 6], dtype=np.uint64)
    ang = np.array([0.5])
    p = st.ctypes.data
    cases = [
        (lib.qsim_apply_pauli_rotations, (p, 6, 1, one.ctypes.data, zero.ctypes.data, None), "null argument"),
        (lib.qsim_apply_pauli_rotations, (p, 6, 1, None, zero.ctypes.data, ang.ctypes.data), "null argument"),
        (lib.qsim_apply_pauli_rotations, (p, 6, 1, one.ctypes.data, None, ang.ctypes.data), "null argument"),
        (lib.qsim_apply_pauli_rotations, (None, 6, 1, one.ctypes.data, zero.ctypes.data, ang.ctypes.data),
         "null state"),
        (lib.qsim_apply_pauli_rotations, (p, 6, 1, big.ctypes.data, zero.ctypes.data, ang.ctypes.data),
         "at or above"),
        (lib.qsim_apply_pauli_rotations, (p, 6, 1, zero.ctypes.data, big.ctypes.data, ang.ctypes.data),
         "at or above"),
        (lib.qsim_apply_pauli_rotations, (p, 0, 1, zero.ctypes.data, zero.ctypes.data, ang.ctypes.data), "[1, 63]"),
        (lib.qsim_apply_pauli_rotations, (p, 64, 1, zero.ctypes.data, zero.ctypes.data, ang.ctypes.data), "[1, 63]"),
        (lib.qsim_apply_pauli_rotations, (p, 6, -1, one.ctypes.data, zero.ctypes.data, ang.ctypes.data), "< 0"),
        (lib.qsim_apply_pauli_rotations_dm, (p, 32, 1, one.ctypes.data, zero.ctypes.data, ang.ctypes.data),
         "[1, 31]"),
        (lib.qsim_apply_pauli_rotations_dm, (None, 3, 1, one.ctypes.data, zero.ctypes.data, ang.ctypes.data),
         "null state"),
    ]
    for bad in (np.nan, np.inf, -np.inf):
        a = np.array([bad])
        for fn in (lib.qsim_apply_pauli_rotations, lib.qsim_apply_pauli_rotations_dm):
            cases.append((fn, (p, 3, 1, one.ctypes.data, zero.ctypes.data, a.ctypes.data), "non-finite angle"))
    for fn, args, text in cases:
        assert fn(*args, None) == -1, (fn, args)
        assert text.encode() in lib.qsim_last_error(), (lib.qsim_last_error(), text)
    for fn in (lib.qsim_apply_pauli_rotations, lib.qsim_apply_pauli_rotations_dm):
        assert fn(None, 6, 0, None, None, None, None) == 0


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
        from quantum_computations_b200 import gates, sharded, workloads
        from quantum_computations_b200.states import State

        comm = sharded.Comm()
        rng = np.random.default_rng(31)
        circ = workloads.sv_random_circuit(n, 4, 8)
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
        flipped = sum(st.flip)
        before = st.gather_numpy()
        local_q = [n - 1 - l for l in range(n) if st.phys[l] < st.n_local]
        r0, r1 = rank_q[0], rank_q[-1]
        terms = [{r0: "Z", local_q[0]: "X"}, {r0: "Z", r1: "Z"}, {r1: "Z"}, {r0: "X", local_q[1]: "Z"},
                 {r1: "Y", local_q[2]: "X", r0: "Z"}, {}, {local_q[0]: "Y", local_q[3]: "Y"},
                 {r0: "Y", r1: "X", local_q[4]: "Z"}]
        for _ in range(12):
            qs = rng.choice(n, size=3, replace=False)
            terms.append({int(q): "XYZ"[int(rng.integers(3))] for q in qs})
        x, z = masks_of([PauliSum([(1, t)])._label_n(n) for t in terms])
        angles = rng.uniform(-3, 3, size=len(terms))
        swaps0 = st.swaps
        assert st.apply_pauli_rotations(x, z, angles) is st
        after = st.gather_numpy()
        wide = False
        try:
            st.apply_pauli_rotations([(1 << (st.n_local + 1)) - 1], [0], [0.3])
        except NotImplementedError:
            wide = True
        if rank == 0:
            ref = engine.DeviceState.from_numpy(before, emu()).apply_pauli_rotations(x, z, angles).to_numpy()
            np.save(os.path.join(out_dir, "sharded.npy"),
                    np.array([rel_err(after, ref), st.swaps - swaps0, flipped, float(wide)]))
    finally:
        dist.destroy_process_group()


def _label_n(self, n, t=0):
    return "".join("IXYZ"[p] for p in self._letters(t, n))


PauliSum._label_n = _label_n          # test helper: the dense-oracle label of term t on n qubits


@pytest.mark.parametrize("world,n", [(2, 9), (4, 10), (8, 10)])
def test_sharded_rotations_match_single_process(tmp_path, world, n):
    import torch.multiprocessing as mp
    build_native.build_emu()
    mp.spawn(_sharded_worker, args=(world, _free_port(), n, str(tmp_path)), nprocs=world, join=True)
    err, swaps, flipped, wide = np.load(tmp_path / "sharded.npy")
    assert err <= 1e-12
    assert swaps >= 1 and flipped >= 1                   # rank qubits were exchanged, some complemented
    assert wide == 1.0                                   # a support wider than a shard is refused


def test_sharded_density_matrix_is_refused():
    from quantum_computations_b200 import sharded
    st = sharded.ShardedState.__new__(sharded.ShardedState)
    st.is_density = True
    with pytest.raises(NotImplementedError):
        st.apply_pauli_rotations([1], [0], [0.5])


# ---- GPU -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_kets_gpu(cuda_backend):
    check_kets(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_density_matrices_gpu(cuda_backend):
    check_density_matrices(cuda_backend, range(1, 7))


@pytest.mark.gpu
def test_packing_gpu(cuda_backend):
    check_packing(cuda_backend)


@pytest.mark.gpu
def test_edges_gpu(cuda_backend):
    check_edges(cuda_backend)


@pytest.mark.gpu
def test_evolve_gpu(cuda_backend):
    check_evolve(cuda_backend)


@pytest.mark.gpu
def test_emulator_and_cuda_agree(cuda_backend, emu_backend):
    rng = np.random.default_rng(12)
    for n in (5, 11, 16):
        psi = rand_ket(n, rng)
        labels, angles = rotation_list(n, rng, 60)
        x, z = masks_of(labels)
        got = engine.DeviceState.from_numpy(psi, cuda_backend).apply_pauli_rotations(x, z, angles).to_numpy()
        want = engine.DeviceState.from_numpy(psi, emu_backend).apply_pauli_rotations(x, z, angles).to_numpy()
        assert rel_err(got, want) <= 1e-14, n
        rho = np.outer(psi[:1 << (n // 2)], psi[:1 << (n // 2)].conj())
        got = engine.DeviceState.from_numpy(rho, cuda_backend).apply_pauli_rotations(
            x & ((1 << (n // 2)) - 1), z & ((1 << (n // 2)) - 1), angles).to_numpy()
        want = engine.DeviceState.from_numpy(rho, emu_backend).apply_pauli_rotations(
            x & ((1 << (n // 2)) - 1), z & ((1 << (n // 2)) - 1), angles).to_numpy()
        assert rel_err(got, want) <= 1e-14, n


@pytest.mark.gpu
def test_x_string_on_30_qubits_gpu(cuda_backend):
    import torch
    n, th = 30, 0.73
    st = engine.DeviceState.product([np.array([1, 0], dtype=np.complex128)] * n, cuda_backend)
    st.apply_pauli_rotations([(1 << n) - 1], [0], [th])
    buf = st.buf
    assert abs(complex(buf[0].item()) - np.cos(th / 2)) <= 1e-15
    assert abs(complex(buf[-1].item()) - (-1j * np.sin(th / 2))) <= 1e-15
    assert int(torch.count_nonzero(buf).item()) == 2                # every other amplitude exactly 0
    del st, buf
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_inverse_returns_the_state_gpu(cuda_backend):
    import torch
    from quantum_computations_b200 import workloads
    n = 28
    rng = np.random.default_rng(13)
    st = engine.DeviceState.product([np.array([1, 0], dtype=np.complex128)] * n, cuda_backend)
    ops = [op for g in workloads.sv_random_circuit(n, 2, 3) for op in g.lowered(n, False)]
    engine.Plan(cuda_backend, n, ops).execute(st.buf)
    start = st.buf.clone()
    labels, angles = rotation_list(n, rng, 100)
    x, z = masks_of(labels)
    st.apply_pauli_rotations(x, z, angles)
    assert float((st.buf - start).abs().max().item()) > 1e-6
    st.apply_pauli_rotations(x[::-1], z[::-1], -angles[::-1])
    assert float((st.buf - start).abs().max().item()) <= 1e-13
    del st, start
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_heisenberg_step_matches_planner_gates_gpu(cuda_backend):
    import torch
    from quantum_computations_b200 import workloads
    n, dt = 26, 0.05
    h = heisenberg(n)
    st = engine.DeviceState.product([np.array([1, 0], dtype=np.complex128)] * n, cuda_backend)
    ops = [op for g in workloads.sv_random_circuit(n, 2, 4) for op in g.lowered(n, False)]
    engine.Plan(cuda_backend, n, ops).execute(st.buf)
    gates_st = st.copy()
    observables.evolve(h, st, dt)
    lowered = []
    for k in range(len(h)):
        qs = [q for q in range(n) if (int(h.x_masks[k]) | int(h.z_masks[k])) >> q & 1]
        sub = PauliSum([(1, {i: h._letters(k, n)[q] for i, q in enumerate(qs)})]).matrix(len(qs))
        lowered.append((qs, scipy.linalg.expm(-1j * dt * h.coeffs[k].real * sub)))
    engine.apply_lowered(gates_st, lowered)
    assert float((st.buf - gates_st.buf).abs().max().item()) <= 1e-12
    del st, gates_st
    torch.cuda.empty_cache()
