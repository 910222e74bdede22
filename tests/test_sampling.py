"""Measurement statistics (qsim_marginal_probs / qsim_sample and their _dm variants,
DeviceState.probabilities / sample, ShardedState.probabilities / sample): marginals and
inverse-CDF sampling against NumPy oracles on the host emulator and on the GPU, zero
probabilities around chunk and sub-tile boundaries, repeatability and fixed launch counts,
argument checks of both libraries, the sharded collectives over gloo, and 30-qubit checks
on the GPU against independent routes (torch on the same buffer, product states, basis
and GHZ states)."""
import ctypes as C
import os
import socket
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

from quantum_computations_b200 import _capi, build_native, engine  # noqa: E402

CHUNK, SUB = 1 << 16, 1 << 8


# ---- oracles ----------------------------------------------------------------------------------
def marg_ref(p, n, qubits):
    k = len(qubits)
    idx = np.arange(1 << n, dtype=np.int64)
    b = np.zeros(1 << n, dtype=np.int64)
    for j, q in enumerate(qubits):
        b |= ((idx >> (n - 1 - q)) & 1) << (k - 1 - j)
    return np.bincount(b, weights=p, minlength=1 << k)


def rel_err(got, ref) -> float:
    return float(np.abs(np.asarray(got) - np.asarray(ref)).max() / max(np.abs(ref).max(), 1e-300))


def rand_ket(n, rng):
    return rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)


def qubit_sets(n, rng):
    sets = [[], list(range(n)), list(range(n))[::-1]]
    for k in range(1, n + 1):
        sets += [list(range(k)), list(range(n - k, n)), [int(v) for v in rng.permutation(n)[:k]]]
    return sets


def check_samples(p, u, idx, total):
    """Every shot against searchsorted(cumsum(p), u * total, side='right'): equal unless u * total
    lies within 1e-12 (relative) of a CDF boundary, and never an index of probability 0."""
    cdf = np.cumsum(p)
    target = u * total
    ref = np.minimum(np.searchsorted(cdf, target, side="right"), len(p) - 1)
    assert (p[idx] > 0).all(), "a zero-probability index was drawn"
    diff = np.nonzero(idx != ref)[0]
    for s in diff:
        lo, hi = min(idx[s], ref[s]), max(idx[s], ref[s])
        edges = cdf[max(lo - 1, 0):hi + 1]
        assert np.abs(edges - target[s]).min() <= 1e-12 * total, (s, idx[s], ref[s])
    return len(diff)


def launches(be) -> int:
    return int(be.lib.qsim_launch_count())


# ---- checks, run on both backends ----------------------------------------------------------------
def check_ket_marginals(be, sizes, seed=5):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi = rand_ket(n, rng) * 3.7                      # not normalised
        st = engine.DeviceState.from_numpy(psi, be)
        p = np.abs(psi) ** 2
        for qs in qubit_sets(n, rng):
            got = st.probabilities(qs)
            assert got.dtype == np.float64 and got.shape == (1 << len(qs),)
            assert rel_err(got, marg_ref(p, n, qs)) <= 1e-12, (n, qs)
        top = list(range(max(1, n // 2)))
        assert np.array_equal(st.probabilities(top), st.probabilities(top))     # bit-identical repeat
        assert np.array_equal(st.to_numpy(mirror_dtype=False), psi)              # state untouched


def check_dm_marginals(be, sizes, seed=6):
    rng = np.random.default_rng(seed)
    for N in sizes:
        a = rng.normal(size=(1 << N, 1 << N)) + 1j * rng.normal(size=(1 << N, 1 << N))
        rho = a @ a.conj().T
        skew = rho + (rng.normal(size=rho.shape) + 1j * rng.normal(size=rho.shape))   # negative diagonal entries too
        for mat in (rho, skew):
            st = engine.DeviceState.from_numpy(mat, be)
            d = np.diagonal(mat).real.copy()
            for qs in qubit_sets(N, rng):
                assert rel_err(st.probabilities(qs), marg_ref(d, N, qs)) <= 1e-12, (N, qs)


def sparse_ket(n, rng):
    """A ket with zero amplitudes inside chunks and sub-tiles and around their boundaries."""
    psi = rand_ket(n, rng)
    psi[rng.random(1 << n) < 0.3] = 0
    for step in (SUB, CHUNK):
        for b in range(step, 1 << n, step):
            psi[b - 3:b + 2] = 0
    if n > 16:
        psi[CHUNK:3 * CHUNK] = 0                           # two empty chunks
        psi[5 * SUB:9 * SUB] = 0                           # empty sub-tiles
    return psi


def run_sample(be, st, u):
    idx, total = engine.sample_indices(be, st.buf, st.num_qubits, u, st.ndim == 2)
    return idx, total


def check_sampling(be, sizes, shots=20000, seed=7):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi = sparse_ket(n, rng)
        st = engine.DeviceState.from_numpy(psi, be)
        p = np.abs(psi) ** 2
        cdf = np.cumsum(p)
        u = rng.random(shots)
        u[:4] = [0.0, np.nextafter(1.0, 0.0), 0.5, 1e-300]
        u[4:40] = cdf[rng.integers(0, 1 << n, 36)] / cdf[-1]          # uniforms on CDF boundaries
        idx, total = run_sample(be, st, u)
        assert abs(total - cdf[-1]) <= 1e-12 * cdf[-1]
        check_samples(p, u, idx, total)
        again, total2 = run_sample(be, st, u)
        assert np.array_equal(idx, again) and total == total2
        assert np.array_equal(st.to_numpy(mirror_dtype=False), psi)


def check_many_shots_no_zero(be, n=18, seed=8):
    rng = np.random.default_rng(seed)
    psi = sparse_ket(n, rng)
    st = engine.DeviceState.from_numpy(psi, be)
    p = np.abs(psi) ** 2
    u = rng.random(100000)
    idx, total = run_sample(be, st, u)
    assert (p[idx] > 0).all()
    check_samples(p, u, idx, total)


def check_one_amplitude(be):
    for n, where in ((1, 1), (7, 77), (17, (1 << 17) - 1), (18, 3 * CHUNK + 5)):
        psi = np.zeros(1 << n, dtype=np.complex128)
        psi[where] = 0.3 - 0.4j
        st = engine.DeviceState.from_numpy(psi, be)
        u = np.concatenate([[0.0, np.nextafter(1.0, 0.0)], np.random.default_rng(n).random(5000)])
        idx, total = run_sample(be, st, u)
        assert (idx == where).all() and abs(total - 0.25) < 1e-15
        assert (st.sample(100, rng=1) == where).all()


def check_dm_sampling(be, sizes=range(1, 7), seed=9):
    rng = np.random.default_rng(seed)
    for N in sizes:
        a = rng.normal(size=(1 << N, 1 << N)) + 1j * rng.normal(size=(1 << N, 1 << N))
        rho = a @ a.conj().T
        rho[0, 0] = -0.5                                   # a negative diagonal entry counts as 0
        if N > 1:
            rho[2, 2] = 0.0
        st = engine.DeviceState.from_numpy(rho, be)
        d = np.clip(np.diagonal(rho).real, 0.0, None)
        u = rng.random(5000)
        idx, total = run_sample(be, st, u)
        assert abs(total - d.sum()) <= 1e-12 * d.sum()
        check_samples(d, u, idx, total)


def check_launches_and_projection(be):
    rng = np.random.default_rng(10)
    n = 11
    psi = rand_ket(n, rng)
    st = engine.DeviceState.from_numpy(psi, be)
    counts = []
    for shots in (1, 1000, 30000):
        before = launches(be)
        run_sample(be, st, rng.random(shots))
        counts.append(launches(be) - before)
    assert counts == [6, 6, 6]                             # independent of the number of shots
    before = launches(be)
    run_sample(be, st, np.zeros(0))
    assert launches(be) == before
    # outcomes over a subset = the same draws projected
    full = st.sample(4000, rng=3)
    qs = [7, 0, 4]
    sub = st.sample(4000, qs, rng=3)
    assert np.array_equal(sub, engine.project_outcomes(full, n, qs))
    assert np.array_equal(st.sample(10, rng=np.random.default_rng(3)), full[:10])
    # a marginal as a device array
    dev = st.probabilities([2, 5], device=True)
    assert np.array_equal(be.download(dev), st.probabilities([2, 5]))
    with pytest.raises(ValueError):
        st.probabilities([0, 0])
    with pytest.raises(ValueError):
        st.sample(3, [n])


def check_zero_mass(be):
    st = engine.DeviceState.from_numpy(np.zeros(1 << 5, dtype=np.complex128), be)
    with pytest.raises(ValueError, match="qsim_sample: the state has no probability mass"):
        st.sample(4)
    rho = np.zeros((4, 4), dtype=np.complex128)
    rho[1, 1] = -1.0
    dm = engine.DeviceState.from_numpy(rho, be)
    with pytest.raises(ValueError, match="qsim_sample_dm: the state has no probability mass"):
        dm.sample(4)


# ---- emulator ------------------------------------------------------------------------------------
def test_ket_marginals_emulator(emu_backend):
    check_ket_marginals(emu_backend, range(1, 13))


def test_dm_marginals_emulator(emu_backend):
    check_dm_marginals(emu_backend, range(1, 7))


def test_sampling_emulator(emu_backend):
    check_sampling(emu_backend, [1, 2, 5, 9, 12, 17, 18, 20])


def test_many_shots_never_draw_zero_emulator(emu_backend):
    check_many_shots_no_zero(emu_backend)


def test_one_amplitude_emulator(emu_backend):
    check_one_amplitude(emu_backend)


def test_dm_sampling_emulator(emu_backend):
    check_dm_sampling(emu_backend)


def test_launches_and_projection_emulator(emu_backend):
    check_launches_and_projection(emu_backend)


def test_zero_mass_emulator(emu_backend):
    check_zero_mass(emu_backend)


# ---- argument checks of both libraries (no GPU needed: refused before any CUDA call) -----------
def _load(path):
    lib = C.CDLL(path)
    _capi.declare(lib)
    return lib


@pytest.fixture(scope="module", params=["cuda", "emu"])
def lib(request):
    return _load(build_native.build_cuda() if request.param == "cuda" else build_native.build_emu())


ST = np.zeros(64, dtype=np.complex128)
OUT = np.zeros(64, dtype=np.float64)
U = np.zeros(64, dtype=np.float64)
IDX = np.zeros(64, dtype=np.uint64)
WS = np.zeros(1 << 16, dtype=np.uint8)
TOT = np.zeros(1, dtype=np.float64)


def _q(*v):
    return np.array(v, dtype=np.int32)


def marg(L, fn="qsim_marginal_probs", state=True, n=3, k=2, qubits=_q(0, 1), out=True):
    return getattr(L, fn)(ST.ctypes.data if state else None, n, k,
                          None if qubits is None else qubits.ctypes.data_as(_capi.c_int_p),
                          OUT.ctypes.data if out else None, None)


def samp(L, fn="qsim_sample", state=True, n=3, shots=4, u=True, out=True, total=True, ws=True, ws_bytes=None):
    nbytes = C.c_uint64()
    L.qsim_sample_workspace_bytes(3, 4, C.byref(nbytes))
    return getattr(L, fn)(ST.ctypes.data if state else None, n, shots, U.ctypes.data if u else None,
                          IDX.ctypes.data if out else None, TOT.ctypes.data_as(_capi.c_double_p) if total else None,
                          WS.ctypes.data if ws else None, nbytes.value if ws_bytes is None else ws_bytes, None)


def _cases():
    cs = []

    def case(name, call, msg):
        cs.append(pytest.param(call, msg, id=name))

    for fn, max_n in (("qsim_marginal_probs", 40), ("qsim_marginal_probs_dm", 31)):
        t = fn[5:]
        m = fn + ": null argument"
        case(t + "-null-state", lambda L, f=fn: marg(L, f, state=False), m)
        case(t + "-null-qubits", lambda L, f=fn: marg(L, f, qubits=None), m)
        case(t + "-null-out", lambda L, f=fn: marg(L, f, out=False), m)
        m = f"{fn}: n_qubits must be in [1, {max_n}]"
        case(t + "-n0", lambda L, f=fn: marg(L, f, n=0, k=0), m)
        case(t + "-n-big", lambda L, f=fn, b=max_n + 1: marg(L, f, n=b, k=1, qubits=_q(0)), m)
        m = fn + ": k must be in [0, n_qubits]"
        case(t + "-k-neg", lambda L, f=fn: marg(L, f, k=-1), m)
        case(t + "-k-above-n", lambda L, f=fn: marg(L, f, k=4, qubits=_q(0, 1, 2, 0)), m)
        m = fn + ": qubit out of range"
        case(t + "-qubit-n", lambda L, f=fn: marg(L, f, qubits=_q(0, 3)), m)
        case(t + "-qubit-neg", lambda L, f=fn: marg(L, f, qubits=_q(-1, 0)), m)
        case(t + "-duplicate", lambda L, f=fn: marg(L, f, qubits=_q(2, 2)), fn + ": qubits must be distinct")
    for fn, max_n in (("qsim_sample", 40), ("qsim_sample_dm", 31)):
        t = fn[5:]
        m = fn + ": null argument"
        for arg in ("state", "u", "out", "total", "ws"):
            case(f"{t}-null-{arg}", lambda L, f=fn, a=arg: samp(L, f, **{a: False}), m)
        m = fn + ": shots must be in [0, 2^31)"
        case(t + "-shots-neg", lambda L, f=fn: samp(L, f, shots=-1), m)
        case(t + "-shots-2^31", lambda L, f=fn: samp(L, f, shots=1 << 31), m)
        m = f"{fn}: n_qubits must be in [1, {max_n}]"
        case(t + "-n0", lambda L, f=fn: samp(L, f, n=0), m)
        case(t + "-n-big", lambda L, f=fn, b=max_n + 1: samp(L, f, n=b), m)
        case(t + "-short-workspace", lambda L, f=fn: samp(L, f, ws_bytes=1000),
             None)                                     # message carries the size, checked below
    m = "qsim_sample_workspace_bytes: "
    case("workspace-null", lambda L: L.qsim_sample_workspace_bytes(3, 4, None), m + "null argument")
    case("workspace-n0", lambda L: L.qsim_sample_workspace_bytes(0, 4, C.byref(C.c_uint64())),
         m + "n_qubits must be in [1, 40]")
    case("workspace-shots-neg", lambda L: L.qsim_sample_workspace_bytes(3, -1, C.byref(C.c_uint64())),
         m + "shots must be in [0, 2^31)")
    return cs


@pytest.mark.parametrize("call, message", _cases())
def test_invalid_call_is_refused_before_any_work(lib, call, message):
    assert call(lib) == -1
    text = lib.qsim_last_error().decode()
    if message is None:
        assert text.endswith("workspace too small (" + str(_need(lib)) + " bytes needed)"), text
    else:
        assert text == message


def _need(L):
    nbytes = C.c_uint64()
    assert L.qsim_sample_workspace_bytes(3, 4, C.byref(nbytes)) == 0
    return nbytes.value


def test_empty_work_returns_at_once(lib):
    before = lib.qsim_launch_count()
    assert samp(lib, shots=0, state=False, u=False, out=False, total=False, ws=False) == 0
    assert lib.qsim_launch_count() == before
    assert lib.qsim_version() == 102


def test_workspace_size_grows_with_shots_and_chunks(lib):
    def need(n, shots):
        v = C.c_uint64()
        assert lib.qsim_sample_workspace_bytes(n, shots, C.byref(v)) == 0
        return v.value
    assert need(30, 10 ** 6) - need(30, 0) >= 16 * 10 ** 6
    assert need(30, 0) >= 8 * (1 << 22)                     # the sub-tile masses: 2^(n-8) doubles
    assert need(10, 0) == need(16, 0) < need(17, 0)


# ---- sharded collectives over gloo ----------------------------------------------------------------
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
        from parity_cases import random_circuit
        from quantum_computations_b200 import gates, sharded, workloads
        from quantum_computations_b200.states import State

        comm = sharded.Comm()
        rng = np.random.default_rng(31)
        circ = workloads.sv_random_circuit(n, 6, 8) + random_circuit(n, 15, rng)
        circ += [gates.Y(q) for q in range(n)] + [gates.CZ(0, n - 1), gates.T(1)]
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
        logical = st.gather_numpy()
        local_q = [n - 1 - l for l in range(n) if st.phys[l] < st.n_local]
        sets = [list(range(n)), rank_q, [rank_q[0], local_q[0]], [local_q[2], rank_q[-1], local_q[0]],
                list(range(n))[::-1], [], [int(v) for v in rng.permutation(n)[:5]]]
        margs = [st.probabilities(qs) for qs in sets]
        # shards in rank-major physical order (what the documented sampling order refers to)
        shards = comm.allgather_object(np.asarray(st.buf).copy())
        u_seed = 77
        shots = 20000
        outcomes = st.sample(shots, rng=u_seed)
        sub_q = [rank_q[0], local_q[1], local_q[3]]
        sub = st.sample(shots, sub_q, rng=u_seed)
        everyone = comm.allgather_object((outcomes.tobytes(), b"".join(m.tobytes() for m in margs)))
        if rank == 0:
            p = np.abs(logical) ** 2
            marg_err = max(rel_err(m, marg_ref(p, n, qs)) for m, qs in zip(margs, sets))
            phys_p = np.abs(np.concatenate(shards)) ** 2
            u = np.random.default_rng(u_seed).random(shots)
            cdf = np.cumsum(phys_p)
            ref_phys = np.minimum(np.searchsorted(cdf, u * cdf[-1], side="right"), len(cdf) - 1)
            # physical index -> logical index
            nl = st.n_local
            ref = np.zeros(shots, dtype=np.int64)
            for l in range(n):
                pb = st.phys[l]
                bit = (ref_phys >> pb) & 1
                if pb >= nl:
                    bit = bit ^ st.flip[pb - nl]
                ref |= bit << l
            mismatch = int((outcomes != ref).sum())
            zero = int((p[outcomes] == 0).sum())
            proj_ok = float(np.array_equal(sub, engine.project_outcomes(outcomes, n, sub_q)))
            np.save(os.path.join(out_dir, "sharded.npy"),
                    np.array([marg_err, mismatch, zero, float(all(e == everyone[0] for e in everyone)), proj_ok,
                              flipped, st.swaps]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 9), (4, 10), (8, 10)])
def test_sharded_marginals_and_samples_match_oracle(tmp_path, world, n):
    import torch.multiprocessing as mp
    build_native.build_emu()
    mp.spawn(_sharded_worker, args=(world, _free_port(), n, str(tmp_path)), nprocs=world, join=True)
    marg_err, mismatch, zero, same, proj_ok, flipped, swaps = np.load(tmp_path / "sharded.npy")
    assert marg_err <= 1e-12
    assert mismatch <= 2 and zero == 0                   # outcome for outcome, up to boundary shots
    assert same == 1.0 and proj_ok == 1.0                # identical on every rank
    assert flipped >= 1 and swaps >= 1                   # rank qubits were exchanged, some complemented


def test_sharded_density_matrix_is_refused():
    from quantum_computations_b200 import sharded
    st = sharded.ShardedState.__new__(sharded.ShardedState)
    st.is_density = True
    with pytest.raises(NotImplementedError):
        st.probabilities([0])
    with pytest.raises(NotImplementedError):
        st.sample(3)


# ---- GPU -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ket_marginals_gpu(cuda_backend):
    check_ket_marginals(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_dm_marginals_gpu(cuda_backend):
    check_dm_marginals(cuda_backend, range(1, 7))


@pytest.mark.gpu
def test_sampling_gpu(cuda_backend):
    check_sampling(cuda_backend, [1, 2, 5, 9, 12, 17, 18, 20, 22])


@pytest.mark.gpu
def test_many_shots_never_draw_zero_gpu(cuda_backend):
    check_many_shots_no_zero(cuda_backend)


@pytest.mark.gpu
def test_one_amplitude_gpu(cuda_backend):
    check_one_amplitude(cuda_backend)


@pytest.mark.gpu
def test_dm_sampling_gpu(cuda_backend):
    check_dm_sampling(cuda_backend)


@pytest.mark.gpu
def test_launches_and_projection_gpu(cuda_backend):
    check_launches_and_projection(cuda_backend)


@pytest.mark.gpu
def test_zero_mass_gpu(cuda_backend):
    check_zero_mass(cuda_backend)


@pytest.mark.gpu
def test_emulator_and_gpu_agree(cuda_backend, emu_backend):
    rng = np.random.default_rng(12)
    for n in (9, 18, 20):
        psi = sparse_ket(n, rng)
        u = rng.random(50000)
        a, ta = run_sample(emu_backend, engine.DeviceState.from_numpy(psi, emu_backend), u)
        g = engine.DeviceState.from_numpy(psi, cuda_backend)
        b, tb = run_sample(cuda_backend, g, u)
        # same summation orders; |psi|^2 may round differently (FMA), so only boundary shots may differ
        p = np.abs(psi) ** 2
        check_samples(p, u, a, ta)
        check_samples(p, u, b, tb)
        assert abs(ta - tb) <= 1e-14 * ta and (a != b).sum() <= 5
        qs = [n - 1, 0, 3]
        assert rel_err(g.probabilities(qs), engine.DeviceState.from_numpy(psi, emu_backend).probabilities(qs)) <= 1e-14


def _big_state(be, n):
    from quantum_computations_b200 import workloads
    st = engine.DeviceState.product([np.array([1, 0], dtype=np.complex128)] * n, be)
    for g in workloads.sv_random_circuit(n, 2, 5):
        st = g.apply(st)
    return st


@pytest.mark.gpu
def test_30_qubit_marginals_and_state_unchanged_gpu(cuda_backend):
    import torch
    n = 30
    st = _big_state(cuda_backend, n)
    keep = st.buf.clone()
    p = torch.view_as_real(st.buf).pow(2).sum(-1)           # |psi|^2 by torch, same buffer
    top = st.probabilities(list(range(20)))
    want = p.view(1 << 20, 1 << 10).sum(1).cpu().numpy()
    assert rel_err(top, want) <= 1e-12
    scattered = [29, 3, 17, 0, 11, 24]
    got = st.probabilities(scattered)
    cube = p.view((2,) * n)
    rest = tuple(a for a in range(n) if a not in scattered)
    want = cube.sum(dim=rest).permute(*[sorted(scattered).index(q) for q in scattered]).reshape(-1).cpu().numpy()
    assert rel_err(got, want) <= 1e-12
    full = st.probabilities(device=True)
    assert torch.allclose(full, p, rtol=1e-15, atol=0)
    del full
    assert rel_err(st.probabilities([]), [p.sum().item()]) <= 1e-12
    idx, _total = engine.sample_indices(cuda_backend, st.buf, n, np.random.default_rng(4).random(10 ** 6))
    assert (p[torch.from_numpy(idx).cuda()] > 0).all()
    assert torch.equal(torch.view_as_real(st.buf), torch.view_as_real(keep))   # bit for bit
    del p, keep, cube, st
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_30_qubit_product_state_samples_gpu(cuda_backend):
    """Outcomes against the closed-form CDF of a product state shot for shot, and per-qubit
    frequencies within 5 sigma."""
    import torch
    n, shots = 30, 10 ** 6
    rng = np.random.default_rng(13)
    p1 = rng.uniform(0.05, 0.95, n)                         # P(qubit q = 1)
    vecs = [np.array([np.sqrt(1 - a), np.sqrt(a) * np.exp(1j * rng.uniform(0, 6))]) for a in p1]
    st = engine.DeviceState.product(vecs, cuda_backend)
    u = rng.random(shots)
    idx, total = engine.sample_indices(cuda_backend, st.buf, n, u)
    assert abs(total - 1.0) < 1e-12
    bits = (idx[:, None] >> (n - 1 - np.arange(n))[None, :]) & 1      # column q = qubit q
    # cdf_excl(i) = sum over qubits q with bit 1 of P(prefix) * P(q = 0); p(i) = prod of P(bit)
    pb = np.where(bits == 1, p1[None, :], 1 - p1[None, :])
    prefix = np.cumprod(np.concatenate([np.ones((shots, 1)), pb[:, :-1]], axis=1), axis=1)
    lo = (bits * prefix * (1 - p1)[None, :]).sum(1)
    hi = lo + pb.prod(1)
    target = u * total
    inside = (target >= lo - 1e-12) & (target < hi + 1e-12)
    assert inside.all(), int((~inside).sum())
    freq = bits.mean(0)
    sigma = np.sqrt(p1 * (1 - p1) / shots)
    assert (np.abs(freq - p1) <= 5 * sigma).all()
    del st
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_30_qubit_basis_and_ghz_states_gpu(cuda_backend):
    import torch
    n = 30
    be = cuda_backend
    where = 0b101100111000111100001111000011
    buf = torch.zeros(1 << n, dtype=torch.complex128, device=be.device)
    buf[where] = 1j
    st = engine.DeviceState(be, buf, n, 1)
    idx, total = engine.sample_indices(be, buf, n, np.random.default_rng(14).random(10 ** 7))
    assert total == 1.0 and (idx == where).all()
    buf.zero_()
    buf[0] = buf[(1 << n) - 1] = 1 / np.sqrt(2)
    out = st.sample(10 ** 6, rng=15)
    assert set(np.unique(out).tolist()) == {0, (1 << n) - 1}
    assert abs((out == 0).mean() - 0.5) < 5 * 0.5 / np.sqrt(10 ** 6)
    marg = st.probabilities([0, 29])
    assert np.allclose(marg, [0.5, 0, 0, 0.5], rtol=1e-15, atol=0)
    del st, buf
    torch.cuda.empty_cache()
