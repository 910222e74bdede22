"""Lanczos ground-state energies and Krylov time evolution (qsim_lanczos_apply, qsim_lanczos_step,
krylov.py, observables.ground_state / evolve_krylov): the two primitives against NumPy, bit-exact
regeneration of the Lanczos vectors, ground energies against dense and sparse eigensolvers, evolution
against expm for kets and density matrices, launch counts, argument checks of both libraries, and on
the GPU the 20-, 28- and 30-qubit cases with their memory bounds.  Each check runs on the host
emulator and again on the GPU."""
import ctypes

import numpy as np
import pytest
import scipy.linalg

from quantum_computations_b200 import _capi, build_native, engine, krylov, observables
from quantum_computations_b200.observables import PauliSum
from test_pauli_gradients import heisenberg, launches, norm_err, rand_ket, rand_rho, rand_sum, sum_apply


def ising(n, j=1.0, h=0.7):
    return PauliSum([(-j, {q: "Z", q + 1: "Z"}) for q in range(n - 1)] + [(-h, {q: "X"}) for q in range(n)])


def real_sum(n, rng, count=40):
    h = rand_sum(n, rng, count)
    return PauliSum._from_masks(h.x_masks, h.z_masks, h.coeffs.real, h.num_qubits)


def bits_equal(a, b) -> bool:
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.uint64), np.asarray(b, dtype=np.float64).view(np.uint64))


def lanczos_apply_raw(be, inp, prev, out, n, h, scale):
    return engine.lanczos_apply(be, inp.buf, None if prev is None else prev.buf, out.buf, n, h.x_masks, h.z_masks,
                                h.coeffs, scale)


# ---- check functions, run on both backends -----------------------------------------------------------
def check_primitives(be, sizes, seed=71):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi, old, base = rand_ket(n, rng), rand_ket(n, rng), rand_ket(n, rng)
        for h in (rand_sum(n, rng, 3), rand_sum(n, rng, 90)):        # one pass, several passes
            hpsi = sum_apply(h, psi, n)
            for scale in (0.0, -0.75, 1.5):
                inp = engine.DeviceState.from_numpy(psi, be)
                prev = engine.DeviceState.from_numpy(old, be)
                # prev null
                out = engine.DeviceState.from_numpy(base, be)
                dot = lanczos_apply_raw(be, inp, None, out, n, h, scale)
                got = out.to_numpy()
                assert norm_err(got, hpsi) <= 1e-12, n
                assert abs(dot - np.vdot(psi, got).real) <= 1e-12 * max(1.0, abs(dot)), n
                # prev != out
                out = engine.DeviceState.from_numpy(base, be)
                dot = lanczos_apply_raw(be, inp, prev, out, n, h, scale)
                got = out.to_numpy()
                assert norm_err(got, scale * old + hpsi) <= 1e-12, n
                assert abs(dot - np.vdot(psi, got).real) <= 1e-12 * max(1.0, abs(dot)), n
                assert np.array_equal(prev.to_numpy(), old) and np.array_equal(inp.to_numpy(), psi)
                # prev == out, twice: bit-identical outputs and dots
                runs = []
                for _ in range(2):
                    out = engine.DeviceState.from_numpy(old, be)
                    runs.append((lanczos_apply_raw(be, inp, out, out, n, h, scale), out.to_numpy()))
                assert norm_err(runs[0][1], scale * old + hpsi) <= 1e-12, n
                assert bits_equal([runs[0][0]], [runs[1][0]])
                assert bits_equal(runs[0][1].view(np.float64), runs[1][1].view(np.float64))
        # no terms: out = p prev and its dot
        inp = engine.DeviceState.from_numpy(psi, be)
        prev = engine.DeviceState.from_numpy(old, be)
        out = engine.DeviceState.from_numpy(base, be)
        dot = engine.lanczos_apply(be, inp.buf, prev.buf, out.buf, n, [], [], [], -2.0)
        assert np.array_equal(out.to_numpy(), -2.0 * old)
        assert abs(dot - np.vdot(psi, -2.0 * old).real) <= 1e-12
        # the step: with and without y, and y alone
        w0, v0, y0 = rand_ket(n, rng), rand_ket(n, rng), rand_ket(n, rng)
        a, b = 0.37, complex(-0.4, 1.3)
        runs = []
        for _ in range(2):
            w, v, y = (engine.DeviceState.from_numpy(s, be) for s in (w0, v0, y0))
            r = engine.lanczos_step(be, w.buf, v.buf, y.buf, 1 << n, a, b)
            runs.append((r, w.to_numpy(), y.to_numpy()))
        r, wg, yg = runs[0]
        assert norm_err(wg, w0 - a * v0) <= 1e-14 and norm_err(yg, y0 + b * v0) <= 1e-14
        assert abs(r - np.linalg.norm(w0 - a * v0) ** 2) <= 1e-12
        assert bits_equal([r], [runs[1][0]]) and np.array_equal(wg, runs[1][1]) and np.array_equal(yg, runs[1][2])
        w, v = engine.DeviceState.from_numpy(w0, be), engine.DeviceState.from_numpy(v0, be)
        assert engine.lanczos_step(be, w.buf, v.buf, None, 1 << n, a, norm=False) is None
        assert norm_err(w.to_numpy(), w0 - a * v0) <= 1e-14
        v, y = engine.DeviceState.from_numpy(v0, be), engine.DeviceState.from_numpy(y0, be)
        r = engine.lanczos_step(be, None, v.buf, y.buf, 1 << n, 0.0, b)
        assert norm_err(y.to_numpy(), y0 + b * v0) <= 1e-14
        assert abs(r - np.linalg.norm(y0 + b * v0) ** 2) <= 1e-12


def check_regeneration_is_exact(be, seed=72):
    rng = np.random.default_rng(seed)
    for n, h in ((7, heisenberg(7)), (9, real_sum(9, rng, 60)), (10, ising(10))):
        passes = []
        st = engine.DeviceState.from_numpy(rand_ket(n, rng), be)
        krylov.ground_state(h, st, tol=0.0, max_iter=25, return_state=True, _passes=passes)
        (alphas, betas), again = passes
        assert len(alphas) == 25 and len(again) == 24
        assert bits_equal([p[0] for p in again], alphas[:24])
        assert bits_equal([p[1] for p in again], betas[:24])


def check_ground_energies(be, sizes, seed=73):
    rng = np.random.default_rng(seed)
    for n in sizes:
        for h in (real_sum(n, rng, 20), heisenberg(n), ising(n)):
            evals, evecs = np.linalg.eigh(h.matrix(n))
            psi = rand_ket(n, rng)
            st = engine.DeviceState.from_numpy(psi, be)
            energy, residual = observables.ground_state(h, st)
            assert abs(energy - evals[0]) <= 1e-9 * max(1.0, abs(evals[0])), (n, energy, evals[0])
            assert abs(energy - evals[0]) <= residual + 1e-12                # the residual bounds the error
            # a gap below 1e-3 (one random sum at n = 11) needs more than the default 300 iterations
            assert residual <= 1e-10 or evals[1] - evals[0] < 1e-3, (n, residual)
            assert np.array_equal(st.to_numpy(), psi)                   # the start state is unchanged
            if len(evals) > 1 and evals[1] - evals[0] > 1e-3:
                _e, _r, g = observables.ground_state(h, st, return_state=True)
                v = g.to_numpy()
                fid = abs(np.vdot(evecs[:, 0], v)) ** 2 / np.vdot(v, v).real
                assert fid >= 1 - 1e-8, (n, fid)


def check_happy_breakdown(be):
    n = 6
    h = PauliSum([(0.5, "ZIIIII"), (-1.25, "IZZIII"), (0.3, "IIIZZZ"), (2.0, "IIIIII")])
    psi = np.zeros(1 << n, dtype=np.complex128)
    psi[0b101100] = 1.0
    passes = []
    energy, residual = krylov.ground_state(h, engine.DeviceState.from_numpy(psi, be), _passes=passes)
    assert len(passes[0][0]) == 1 and passes[0][1] == [0.0]
    assert abs(energy - np.vdot(psi, h.matrix(n) @ psi).real) <= 1e-12 and residual == 0.0
    with pytest.raises(ValueError):
        observables.ground_state(h, engine.DeviceState.from_numpy(rand_rho(2, np.random.default_rng(0)), be))


def check_evolve_kets(be, sizes, seed=74):
    rng = np.random.default_rng(seed)
    for n in sizes:
        if n % 2:                                       # a chain plus an identity term (a global phase)
            hz = heisenberg(n)
            h = PauliSum._from_masks(np.append(hz.x_masks, 0), np.append(hz.z_masks, 0), np.append(hz.coeffs, 0.4), n)
        else:
            h = real_sum(n, rng, 15)
        psi = rand_ket(n, rng)
        t = 8.0
        st = engine.DeviceState.from_numpy(psi, be)
        subs = []
        assert krylov.evolve_krylov(h, st, t, tol=1e-11, _substeps=subs) is st
        want = scipy.linalg.expm(-1j * h.matrix(n) * t) @ psi
        assert norm_err(st.to_numpy(), want) <= 1e-10, (n, subs)
        if n >= 6:                                      # more dimensions than one substep's 30
            assert len(subs) >= 2
        back = observables.evolve_krylov(h, st, -t, tol=1e-11)
        assert norm_err(back.to_numpy(), psi) <= 1e-10


def check_evolve_density_matrices(be, sizes, seed=75):
    rng = np.random.default_rng(seed)
    for N in sizes:
        h = real_sum(N, rng, 10)
        rho = rand_rho(N, rng)
        t = 1.7
        st = engine.DeviceState.from_numpy(rho, be)
        observables.evolve_krylov(h, st, t, tol=1e-11)
        u = scipy.linalg.expm(-1j * h.matrix(N) * t)
        got = st.to_numpy()
        assert norm_err(got, u @ rho @ u.conj().T) <= 1e-10, N
        assert abs(np.trace(got) - 1.0) <= 1e-12
        assert np.abs(got - got.conj().T).max() <= 1e-12
    h = real_sum(3, rng, 6)
    lv = h.liouvillian(3).matrix(6)
    m = h.matrix(3)
    assert np.allclose(lv, np.kron(m, np.eye(8)) - np.kron(np.eye(8), m.T), atol=1e-13)


def check_evolve_commuting_and_trotter(be, seed=76):
    rng = np.random.default_rng(seed)
    n = 8
    h = PauliSum([(rng.normal(), {q: "Z"}) for q in range(n)] + [(rng.normal(), {q: "Z", q + 1: "Z"})
                                                                   for q in range(n - 1)] + [(0.9, "I" * n)])
    psi = rand_ket(n, rng)
    a = observables.evolve_krylov(h, engine.DeviceState.from_numpy(psi, be), 3.1)
    b = observables.evolve(h, engine.DeviceState.from_numpy(psi, be), 3.1)
    assert norm_err(a.to_numpy(), b.to_numpy()) <= 1e-11
    # the Trotter error of evolve against evolve_krylov falls as 1 / steps^2 for order 2
    n = 6
    h = heisenberg(n)
    psi = rand_ket(n, rng)
    exact = observables.evolve_krylov(h, engine.DeviceState.from_numpy(psi, be), 1.0).to_numpy()
    errs = [norm_err(observables.evolve(h, engine.DeviceState.from_numpy(psi, be), 1.0, steps=s, order=2)
                     .to_numpy(), exact) for s in (4, 8, 16)]
    for e0, e1 in zip(errs, errs[1:]):
        assert 3.6 <= e0 / e1 <= 4.4, errs


def check_launch_counts(be):
    rng = np.random.default_rng(77)
    n = 9
    h = real_sum(n, rng, 70)
    st = engine.DeviceState.from_numpy(rand_ket(n, rng), be)
    before = launches(be)
    st.apply_pauli_sum(h.x_masks, h.z_masks, h.coeffs)
    passes = launches(be) - before
    assert passes >= 3
    k = 7
    before = launches(be)
    krylov.ground_state(h, st, tol=0.0, max_iter=k)
    # the norm (pass + final sum), then per iteration the apply passes, one step and two final sums
    assert launches(be) - before == 2 + k * (passes + 3)
    before = launches(be)
    krylov.ground_state(h, st, tol=0.0, max_iter=k, return_state=True)
    # the second pass: k - 1 iterations, then the step that adds the last vector (pass + final sum)
    assert launches(be) - before == 2 + k * (passes + 3) + (k - 1) * (passes + 3) + 2


# ---- emulator ------------------------------------------------------------------------------------------
def test_primitives_emulator(emu_backend):
    check_primitives(emu_backend, range(1, 13))


def test_regeneration_is_exact_emulator(emu_backend):
    check_regeneration_is_exact(emu_backend)


def test_ground_energies_emulator(emu_backend):
    check_ground_energies(emu_backend, range(1, 11))


def test_happy_breakdown_emulator(emu_backend):
    check_happy_breakdown(emu_backend)


def test_evolve_kets_emulator(emu_backend):
    check_evolve_kets(emu_backend, range(1, 11))


def test_evolve_density_matrices_emulator(emu_backend):
    check_evolve_density_matrices(emu_backend, range(1, 7))


def test_evolve_commuting_and_trotter_emulator(emu_backend):
    check_evolve_commuting_and_trotter(emu_backend)


def test_launch_counts_emulator(emu_backend):
    check_launch_counts(emu_backend)


def test_refusals(emu_backend):
    rng = np.random.default_rng(78)
    st = engine.DeviceState.from_numpy(rand_ket(3, rng), emu_backend)
    with pytest.raises(ValueError):
        observables.ground_state(PauliSum([(1j, "XYZ")]), st)
    with pytest.raises(ValueError):
        observables.evolve_krylov(PauliSum([(1j, "XYZ")]), st, 1.0)
    with pytest.raises(ValueError):
        observables.evolve_krylov(PauliSum([(1.0, "XYZZ")]), st, 1.0)
    from quantum_computations_b200 import sharded
    sh = sharded.ShardedState.__new__(sharded.ShardedState)
    sh.is_density = False
    with pytest.raises(NotImplementedError):
        observables.ground_state(PauliSum([(1.0, "Z")]), sh)
    with pytest.raises(NotImplementedError):
        observables.evolve_krylov(PauliSum([(1.0, "Z")]), sh, 1.0)


# ---- argument checks of both libraries ---------------------------------------------------------------
def _argument_cases(lib):
    a, b, c = (np.zeros(64, dtype=np.complex128) for _ in range(3))
    pa, pb, pc = a.ctypes.data, b.ctypes.data, c.ctypes.data
    one, zero, big = (np.array([v], dtype=np.uint64) for v in (1, 0, 1 << 6))
    coef, dot, bb = np.array([0.5, 0.25]), np.zeros(1), np.array([0.5, -1.0])
    o, z, bg, cf = (v.ctypes.data for v in (one, zero, big, coef))
    pd, pbb = (v.ctypes.data_as(_capi.c_double_p) for v in (dot, bb))
    la, ls = lib.qsim_lanczos_apply, lib.qsim_lanczos_step
    cases = [
        (la, (None, pc, pb, 6, 1, o, z, cf, 0.5, pd), "null state"),
        (la, (pa, pc, None, 6, 1, o, z, cf, 0.5, pd), "null state"),
        (la, (pa, pc, pb, 6, 1, o, z, cf, 0.5, None), "null argument"),
        (la, (pa, pc, pa, 6, 1, o, z, cf, 0.5, pd), "in and out must be different buffers"),
        (la, (pa, pa, pb, 6, 1, o, z, cf, 0.5, pd), "in and prev must be different buffers"),
        (la, (pa, pc, pb, 6, 1, None, z, cf, 0.5, pd), "null argument"),
        (la, (pa, pc, pb, 6, 1, o, z, None, 0.5, pd), "null argument"),
        (la, (pa, pc, pb, 6, 1, bg, z, cf, 0.5, pd), "at or above"),
        (la, (pa, pc, pb, 0, 1, z, z, cf, 0.5, pd), "[1, 63]"),
        (la, (pa, pc, pb, 64, 0, None, None, None, 0.5, pd), "[1, 63]"),
        (la, (pa, pc, pb, 6, -1, o, z, cf, 0.5, pd), "< 0"),
        (ls, (pa, None, pc, 64, 0.5, pbb, pd), "null v"),
        (ls, (None, pb, None, 64, 0.5, pbb, pd), "both null"),
        (ls, (pa, pb, pc, 64, 0.5, None, pd), "null b_re_im"),
        (ls, (pa, pa, pc, 64, 0.5, pbb, pd), "different buffers"),
        (ls, (pa, pb, pb, 64, 0.5, pbb, pd), "different buffers"),
        (ls, (pa, pb, pa, 64, 0.5, pbb, pd), "different buffers"),
        (ls, (pa, pb, pc, 0, 0.5, pbb, pd), "n_amps must be positive"),
    ]
    keep = [a, b, c, one, zero, big, coef, dot, bb]
    for bad in (np.nan, np.inf, -np.inf):
        cases.append((la, (pa, pc, pb, 6, 1, o, z, cf, bad, pd), "non-finite prev_scale"))
        cb = np.array([0.5, bad])
        keep.append(cb)
        cases.append((la, (pa, pc, pb, 6, 1, o, z, cb.ctypes.data, 0.5, pd), "non-finite coefficient"))
        cases.append((ls, (pa, pb, pc, 64, bad, pbb, pd), "non-finite coefficient"))
        cases.append((ls, (pa, pb, pc, 64, 0.5, cb.ctypes.data_as(_capi.c_double_p), pd), "non-finite coefficient"))
    return cases, keep


@pytest.fixture(scope="module", params=["cuda", "emu"])
def lib(request):
    lib = ctypes.CDLL(build_native.build_cuda() if request.param == "cuda" else build_native.build_emu())
    _capi.declare(lib)
    return lib


def test_argument_checks(lib):
    """Both libraries refuse the same calls with the same message, before any device work (the
    buffers are host arrays)."""
    cases, _keep = _argument_cases(lib)
    for fn, args, text in cases:
        assert fn(*args, None) == -1, (fn, args)
        assert text.encode() in lib.qsim_last_error(), (lib.qsim_last_error(), text)


def test_both_libraries_give_the_same_codes_and_messages():
    results = []
    for path in (build_native.build_cuda(), build_native.build_emu()):
        lib = ctypes.CDLL(path)
        _capi.declare(lib)
        cases, _keep = _argument_cases(lib)
        results.append([(fn(*args, None), lib.qsim_last_error()) for fn, args, _text in cases])
    assert results[0] == results[1]


# ---- GPU -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_primitives_gpu(cuda_backend):
    check_primitives(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_regeneration_is_exact_gpu(cuda_backend):
    check_regeneration_is_exact(cuda_backend)


@pytest.mark.gpu
def test_ground_energies_gpu(cuda_backend):
    check_ground_energies(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_happy_breakdown_gpu(cuda_backend):
    check_happy_breakdown(cuda_backend)


@pytest.mark.gpu
def test_evolve_kets_gpu(cuda_backend):
    check_evolve_kets(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_evolve_density_matrices_gpu(cuda_backend):
    check_evolve_density_matrices(cuda_backend, range(1, 7))


@pytest.mark.gpu
def test_evolve_commuting_and_trotter_gpu(cuda_backend):
    check_evolve_commuting_and_trotter(cuda_backend)


@pytest.mark.gpu
def test_launch_counts_gpu(cuda_backend):
    check_launch_counts(cuda_backend)


def sparse_hamiltonian(h, n):
    """scipy.sparse CSR matrix of h on n qubits, built from the strings (bit q of the index = qubit q)."""
    import scipy.sparse
    idx = np.arange(1 << n, dtype=np.int64)
    total = None
    for x, z, c in zip(h.x_masks, h.z_masks, h.coeffs):
        x, z = int(x), int(z)
        par = np.zeros(1 << n, dtype=np.int64)
        zz = idx & z
        for q in range(n):
            par ^= (zz >> q) & 1
        val = c * (1j ** (bin(x & z).count("1") % 4)) * np.where(par, -1.0, 1.0)
        # P|j> = phase(j) |j ^ x>: column j, row j ^ x
        m = scipy.sparse.csr_matrix((val, (idx ^ x, idx)), shape=(1 << n, 1 << n))
        total = m if total is None else total + m
    return total


@pytest.mark.gpu
def test_heisenberg_20_qubits_against_eigsh_gpu(cuda_backend):
    import scipy.sparse.linalg
    n = 20
    h = heisenberg(n)
    want = scipy.sparse.linalg.eigsh(sparse_hamiltonian(h, n), k=1, which="SA", tol=1e-13)[0][0]
    rng = np.random.default_rng(79)
    kets = [rand_ket(1, rng) for _ in range(n)]
    energy, residual = observables.ground_state(h, engine.DeviceState.product(kets, cuda_backend))
    assert residual <= 1e-10
    assert abs(energy - want) <= 1e-9 * abs(want), (energy, want)


@pytest.mark.gpu
def test_evolution_28_qubits_conserves_energy_and_norm_gpu(cuda_backend):
    n = 28
    h = heisenberg(n)
    rng = np.random.default_rng(80)
    st = engine.DeviceState.product([rand_ket(1, rng) for _ in range(n)], cuda_backend)
    e0, nrm0 = observables.expect(h, st).real, st.norm()
    observables.evolve_krylov(h, st, 0.5)
    assert abs(st.norm() - nrm0) <= 1e-10
    assert abs(observables.expect(h, st).real - e0) <= 1e-10 * max(1.0, abs(e0))


@pytest.mark.gpu
def test_memory_at_30_qubits_gpu(cuda_backend):
    import torch
    n = 30
    h = heisenberg(n)
    rng = np.random.default_rng(81)
    kets = [rand_ket(1, rng) for _ in range(n)]
    state_bytes = 16 << n
    slack = 64 << 20
    st = engine.DeviceState.product(kets, cuda_backend)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated() - state_bytes
    energy, residual = observables.ground_state(h, st, tol=1e-3, max_iter=12)
    assert np.isfinite(energy) and residual > 0
    assert torch.cuda.max_memory_allocated() - base <= 3 * state_bytes + slack
    torch.cuda.reset_peak_memory_stats()
    nrm0 = st.norm()
    observables.evolve_krylov(h, st, 0.05, tol=1e-8)
    assert torch.cuda.max_memory_allocated() - base <= 4 * state_bytes + slack
    assert abs(st.norm() - nrm0) <= 1e-8
