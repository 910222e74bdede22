"""H|psi> for a Pauli sum (qsim_apply_pauli_sum, DeviceState / ShardedState.apply_pauli_sum,
observables.apply) and adjoint gradients over Pauli-rotation circuits (qsim_pauli_rotations_adjoint
/ _dm, observables.expect_and_gradient): kets and density matrices against dense products and the
exact parameter-shift rule on the host emulator and on the GPU, pass counts from launch counts,
argument checks of both libraries, the sharded collectives over gloo, and on the GPU checks at 28
and 30 qubits against parameter shift through the existing calls and against a closed form."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

from quantum_computations_b200 import _capi, build_native, engine, observables  # noqa: E402
from quantum_computations_b200.observables import PauliSum  # noqa: E402

CAP = 32                                     # QS_PAULI_MAX_TERMS = QS_PAULI_ROT_MAX (plan.h)
ADJ_D = 3                                    # QS_PAULI_ADJ_MAX_D (plan.h)


# ---- dense oracle ------------------------------------------------------------------------
def masks_of(labels):
    ps = [PauliSum([(1, lab)]) for lab in labels]
    return (np.array([int(p.x_masks[0]) for p in ps], dtype=np.uint64),
            np.array([int(p.z_masks[0]) for p in ps], dtype=np.uint64))


def pauli_apply(psi, x, z, n):
    """P psi for the string (x, z) (bit q = reference qubit q = index bit n-1-q), P = i^popc(x&z) X^x Z^z."""
    xi = sum(1 << (n - 1 - q) for q in range(n) if int(x) >> q & 1)
    zi = sum(1 << (n - 1 - q) for q in range(n) if int(z) >> q & 1)
    idx = np.arange(1 << n)
    src = idx ^ xi
    par = np.array([bin(v).count("1") & 1 for v in (src & zi)])
    return (1j ** (bin(int(x) & int(z)).count("1") % 4)) * np.where(par, -1, 1) * psi[src]


def sum_apply(h, psi, n):
    return sum(c * pauli_apply(psi, x, z, n) for x, z, c in zip(h.x_masks, h.z_masks, h.coeffs))


def rotate(psi, x, z, angles, n):
    out = psi.copy()
    for xv, zv, th in zip(x, z, angles):
        out = np.cos(th / 2) * out - 1j * np.sin(th / 2) * pauli_apply(out, xv, zv, n)
    return out


def rotate_dm(rho, x, z, angles, n):
    """U rho U^dagger: U on the columns of rho, then U on the columns of (U rho)^dagger."""
    left = np.stack([rotate(rho[:, j], x, z, angles, n) for j in range(1 << n)], axis=1)
    return np.stack([rotate(left.conj()[i], x, z, angles, n) for i in range(1 << n)], axis=0).conj()


def energy(h, psi0, x, z, angles, n):
    v = rotate(psi0, x, z, angles, n)
    return float(np.vdot(v, sum_apply(h, v, n)).real)


def energy_dm(hm, rho0, x, z, angles, n):
    return float(np.trace(hm @ rotate_dm(rho0, x, z, angles, n)).real)


def shift_gradient(f, angles):
    """Exact parameter-shift rule of exp(-i theta/2 P), P^2 = 1."""
    g = np.zeros(len(angles))
    for t in range(len(angles)):
        up, dn = angles.copy(), angles.copy()
        up[t] += np.pi / 2
        dn[t] -= np.pi / 2
        g[t] = (f(up) - f(dn)) / 2
    return g


def norm_err(got, ref) -> float:
    return float(np.linalg.norm(np.asarray(got) - np.asarray(ref)) / max(np.linalg.norm(ref), 1e-300))


def rand_ket(n, rng):
    psi = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    return psi / np.linalg.norm(psi)


def rand_rho(n, rng):
    a = rng.normal(size=(1 << n, 1 << n)) + 1j * rng.normal(size=(1 << n, 1 << n))
    rho = a @ a.conj().T
    return rho / np.trace(rho)


def rand_sum(n, rng, count=40):
    """Complex coefficients; the identity, Y-heavy and full-width X strings, and random strings (more
    distinct X masks than one pass holds)."""
    labels = ["I" * n, "Y" * n, "X" * n, "Z" * n, "Y" * (n - 1) + "X"]
    labels += ["".join(rng.choice(list("IXYZ"), n, p=[0.2, 0.2, 0.4, 0.2])) for _ in range(count)]
    return PauliSum([(complex(rng.normal(), rng.normal()), lab) for lab in labels])


def rand_hamiltonian(n, rng, count=12):
    labels = ["".join(rng.choice(list("IXYZ"), n)) for _ in range(count)] + ["Z" * n, "I" * n]
    return PauliSum([(rng.normal(), lab) for lab in labels])


def rotation_list(n, rng, count=45):
    """Identity, Z-only, Y-heavy, wide-X, repeated and random non-commuting strings over several spans;
    angles with 0, +-pi; more rotations than one sweep pass holds."""
    labels = ["I" * n, "Z" * n, "Y" * n, "X" * n, "X" + "I" * (n - 1), "I" * (n - 1) + "Y"]
    labels += ["".join(rng.choice(list("IXYZ"), n)) for _ in range(count - len(labels) - 3)]
    labels += [labels[4], labels[-1], labels[2]]
    angles = rng.uniform(-3, 3, size=len(labels))
    angles[[1, 7]] = 0.0
    angles[3], angles[9] = np.pi, -np.pi
    x, z = masks_of(labels)
    return x, z, angles


def launches(be) -> int:
    return int(be.lib.qsim_launch_count())


def heisenberg(n, jx=1.0, jy=0.8, jz=0.6, h=0.3):
    terms = []
    for q in range(n - 1):
        for p, j in (("X", jx), ("Y", jy), ("Z", jz)):
            terms.append((j, {q: p, q + 1: p}))
    terms += [(h * (1 + 0.1 * q), {q: "Z"}) for q in range(n)]
    return PauliSum(terms)


def qaoa(n, gammas, betas):
    """MaxCut on the ring with weights 1 + q/n: per layer exp(-i gamma w ZZ) on every edge, then
    exp(-i beta X) on every qubit.  Returns the cost PauliSum, the rotation list and, per rotation,
    its parameter (gamma_l = 2l, beta_l = 2l + 1) and d theta / d parameter."""
    edges = [(q, (q + 1) % n, 1.0 + q / n) for q in range(n)]
    cost = PauliSum([(0.5 * w, {a: "Z", b: "Z"}) for a, b, w in edges])
    xs, zs, angles, param, dtheta = [], [], [], [], []
    for layer, (g, b) in enumerate(zip(gammas, betas)):
        for a, c, w in edges:
            xs.append(0)
            zs.append((1 << a) | (1 << c))
            angles.append(2 * g * w)
            param.append(2 * layer)
            dtheta.append(2 * w)
        for q in range(n):
            xs.append(1 << q)
            zs.append(0)
            angles.append(2 * b)
            param.append(2 * layer + 1)
            dtheta.append(2.0)
    return (cost, (np.array(xs, dtype=np.uint64), np.array(zs, dtype=np.uint64), np.array(angles)),
            np.array(param), np.array(dtheta))


# ---- check functions, run on both backends ----------------------------------------------------------
def check_apply_kets(be, sizes, seed=41):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi = rand_ket(n, rng)
        h = rand_sum(n, rng)
        st = engine.DeviceState.from_numpy(psi, be)
        got = observables.apply(h, st)
        assert got is not st and got.ndim == 1
        # PauliSum.matrix(n) @ psi up to n = 8; beyond, a dense 2^n x 2^n matrix per term costs more than the
        # test is worth, so the reference is sum_apply (term by term, independent of the library), which
        # is itself checked against the matrix for every n <= 8 just below
        want = h.matrix(n) @ psi if n <= 8 else sum_apply(h, psi, n)
        assert norm_err(got.to_numpy(), want) <= 1e-12, n
        if n <= 8:
            assert norm_err(sum_apply(h, psi, n), want) <= 1e-13
        assert np.array_equal(st.to_numpy(), psi)                      # the input is unchanged
        out = engine.DeviceState.from_numpy(np.full(1 << n, np.nan + 0j), be)
        assert st.apply_pauli_sum(h.x_masks, h.z_masks, h.coeffs, out=out) is out
        assert norm_err(out.to_numpy(), want) <= 1e-12, n


def check_apply_density_matrices(be, sizes, seed=42):
    rng = np.random.default_rng(seed)
    for N in sizes:
        rho = rand_rho(N, rng)
        h = rand_sum(N, rng, 20)
        got = observables.apply(h, engine.DeviceState.from_numpy(rho, be))
        assert got.ndim == 2 and got.shape == rho.shape
        assert norm_err(got.to_numpy(), h.matrix(N) @ rho) <= 1e-12, N
    with pytest.raises(ValueError):                     # a column qubit is not part of the operator
        engine.DeviceState.from_numpy(rand_rho(2, rng), be).apply_pauli_sum([4], [0], [1.0])


def check_apply_passes_and_edges(be):
    rng = np.random.default_rng(43)
    n = 10
    st = engine.DeviceState.from_numpy(rand_ket(n, rng), be)

    def count(x, z):
        c = rng.normal(size=len(x)) + 1j * rng.normal(size=len(x))
        before = launches(be)
        st.apply_pauli_sum(x, z, c)
        return launches(be) - before

    def expect_passes(x, z):
        before = launches(be)
        st.expect_pauli(x, z)
        return launches(be) - before - 1                   # minus the final sum

    zmasks = rng.integers(1, 1 << n, size=2 * CAP + 1).astype(np.uint64)
    zero = np.zeros_like(zmasks)
    assert count(zero[:CAP], zmasks[:CAP]) == 1
    assert count(zero[:CAP + 1], zmasks[:CAP + 1]) == 2
    sub = [2, 3, 5, 8]                                  # X masks in a span of four generators: one pass
    xs = np.array([sum(1 << sub[i] for i in range(4) if k >> i & 1) for k in range(1, 16)] * 2, dtype=np.uint64)
    assert count(xs, rng.integers(0, 1 << n, size=len(xs)).astype(np.uint64)) == 1
    single = np.array([1 << q for q in range(5)], dtype=np.uint64)
    assert count(single, np.zeros(5, dtype=np.uint64)) == 2
    for _ in range(3):                                  # the expectation values' packing, pass for pass
        h = rand_sum(n, rng, 70)
        assert count(h.x_masks, h.z_masks) == expect_passes(h.x_masks, h.z_masks) >= 3
    # qsim_accumulate_pauli_sum: the same passes, every one adding to out
    lib = be.lib
    psi = rand_ket(n, rng)
    base = rand_ket(n, rng)
    h = rand_sum(n, rng, 70)
    src = engine.DeviceState.from_numpy(psi, be)
    acc = engine.DeviceState.from_numpy(base, be)
    c = np.ascontiguousarray(h.coeffs)
    before = launches(be)
    assert lib.qsim_accumulate_pauli_sum(be.ptr(src.buf), be.ptr(acc.buf), n, len(h), h.x_masks.ctypes.data,
                                         h.z_masks.ctypes.data, c.ctypes.data, be.stream()) == 0
    assert launches(be) - before == expect_passes(h.x_masks, h.z_masks)
    assert norm_err(acc.to_numpy(), base + sum_apply(h, psi, n)) <= 1e-12
    kept = acc.to_numpy()
    before = launches(be)
    assert lib.qsim_accumulate_pauli_sum(be.ptr(src.buf), be.ptr(acc.buf), n, 0, None, None, None, be.stream()) == 0
    assert launches(be) == before and np.array_equal(acc.to_numpy(), kept)
    # no terms: one pass that writes zeros, whatever the input holds
    bad = engine.DeviceState.from_numpy(np.full(1 << n, np.nan + 1j), be)
    out = bad.apply_pauli_sum([], [], [])
    assert np.array_equal(out.to_numpy(), np.zeros(1 << n))
    x1 = np.ones(1, dtype=np.uint64)
    c1 = np.ones(2)
    assert lib.qsim_apply_pauli_sum(be.ptr(st.buf), be.ptr(st.buf), n, 1, x1.ctypes.data, x1.ctypes.data,
                                    c1.ctypes.data, be.stream()) == -1
    assert b"different buffers" in lib.qsim_last_error()
    with pytest.raises(ValueError):
        st.apply_pauli_sum([1], [0], [np.nan])
    with pytest.raises(ValueError):
        st.apply_pauli_sum([1], [0], [1.0, 2.0])


def check_gradients_kets(be, sizes, seed=44):
    rng = np.random.default_rng(seed)
    for n in sizes:
        psi0 = rand_ket(n, rng)
        h = rand_hamiltonian(n, rng)
        x, z, angles = rotation_list(n, rng)
        st = engine.DeviceState.from_numpy(psi0, be)
        raw = be.download(st.buf).copy()
        value, grad = observables.expect_and_gradient(h, (x, z, angles), st)
        assert np.array_equal(be.download(st.buf).view(np.uint64), raw.view(np.uint64))   # bit for bit
        assert grad.dtype == np.float64 and grad.shape == angles.shape
        want = shift_gradient(lambda a: energy(h, psi0, x, z, a, n), angles)
        assert np.abs(grad - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), n
        assert abs(value - energy(h, psi0, x, z, angles, n)) <= 1e-12
        rotated = engine.DeviceState.from_numpy(psi0, be).apply_pauli_rotations(x, z, angles)
        assert abs(value - observables.expect(h, rotated).real) <= 1e-12
        # the low-level sweep: psi returns to psi0, lam becomes U^dagger lam
        lam0 = rand_ket(n, rng)
        lam = engine.DeviceState.from_numpy(lam0, be)
        rotated.pauli_rotations_adjoint(lam, x, z, angles)
        assert np.abs(rotated.to_numpy() - psi0).max() <= 1e-12
        back = rotate(lam0, x[::-1], z[::-1], -angles[::-1], n)
        assert np.abs(lam.to_numpy() - back).max() <= 1e-12


def check_gradients_density_matrices(be, sizes, seed=45):
    rng = np.random.default_rng(seed)
    for N in sizes:
        rho0 = rand_rho(N, rng)
        h = rand_hamiltonian(N, rng, 8)
        hm = h.matrix(N)
        x, z, angles = rotation_list(N, rng, 36)
        st = engine.DeviceState.from_numpy(rho0, be)
        value, grad = observables.expect_and_gradient(h, (x, z, angles), st)
        assert np.array_equal(st.to_numpy(), rho0)
        want = shift_gradient(lambda a: energy_dm(hm, rho0, x, z, a, N), angles)
        assert np.abs(grad - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), N
        assert abs(value - energy_dm(hm, rho0, x, z, angles, N)) <= 1e-12
        rotated = engine.DeviceState.from_numpy(rho0, be).apply_pauli_rotations(x, z, angles)
        assert abs(value - observables.expect(h, rotated).real) <= 1e-12
        lam = engine.DeviceState.from_numpy(rand_rho(N, rng), be)
        rotated.pauli_rotations_adjoint(lam, x, z, angles)
        assert np.abs(rotated.to_numpy() - rho0).max() <= 1e-12


def check_qaoa(be):
    n = 6
    gammas, betas = np.array([0.4, -0.7]), np.array([0.3, 1.1])
    cost, rot, param, dtheta = qaoa(n, gammas, betas)
    plus = np.full(1 << n, 2 ** (-n / 2), dtype=np.complex128)
    value, grad = observables.expect_and_gradient(cost, rot, engine.DeviceState.from_numpy(plus, be))
    per_param = np.bincount(param, weights=grad * dtheta, minlength=4)      # chain rule over shared parameters
    x, z, angles = rot
    shifted = shift_gradient(lambda a: energy(cost, plus, x, z, a, n), angles)
    assert np.abs(per_param - np.bincount(param, weights=shifted * dtheta, minlength=4)).max() <= 1e-12

    def e_params(p):
        return energy(cost, plus, *qaoa(n, p[0::2], p[1::2])[1], n)
    p0 = np.array([gammas[0], betas[0], gammas[1], betas[1]])
    fd = np.array([(e_params(p0 + 1e-5 * np.eye(4)[k]) - e_params(p0 - 1e-5 * np.eye(4)[k])) / 2e-5
                   for k in range(4)])
    assert np.abs(per_param - fd).max() <= 1e-7
    assert abs(value - e_params(p0)) <= 1e-12


def check_sweep_launches(be):
    rng = np.random.default_rng(46)
    n = 9
    psi = engine.DeviceState.from_numpy(rand_ket(n, rng), be)
    lam = engine.DeviceState.from_numpy(rand_ket(n, rng), be)

    def count(x, z, angles):
        before = launches(be)
        out = psi.pauli_rotations_adjoint(lam, x, z, angles)
        return launches(be) - before, out

    zm = rng.integers(1, 1 << n, size=CAP + 1).astype(np.uint64)
    zero = np.zeros_like(zm)
    assert count(zero[:CAP], zm[:CAP], rng.uniform(-1, 1, CAP))[0] == 1 + 1
    assert count(zero, zm, rng.uniform(-1, 1, CAP + 1))[0] == 2 + 1
    # single X on qubits 0..3, swept from qubit 3 back: [x3 x2 x1] [x0] (three generators per pass)
    single = np.array([1 << q for q in range(ADJ_D + 1)], dtype=np.uint64)
    assert count(single, np.zeros(len(single), dtype=np.uint64), np.ones(len(single)))[0] == 2 + 1
    # angle-0 rotations are swept (they carry a derivative)
    k, g = count(np.array([1, 2], dtype=np.uint64), np.array([2, 1], dtype=np.uint64), np.zeros(2))
    assert k == 1 + 1 and np.all(np.isfinite(g))
    # a density matrix's row and column halves share a pass
    N = 5
    dpsi = engine.DeviceState.from_numpy(rand_rho(N, rng), be)
    dlam = engine.DeviceState.from_numpy(rand_rho(N, rng), be)
    before = launches(be)
    dpsi.pauli_rotations_adjoint(dlam, np.zeros(CAP // 2, dtype=np.uint64), np.arange(1, CAP // 2 + 1, dtype=np.uint64),
                                 np.ones(CAP // 2))
    assert launches(be) - before == 1 + 1
    # two calls on the same inputs: bit-identical
    x, z, angles = rotation_list(n, rng, 70)
    psi0, lam0 = rand_ket(n, rng), rand_ket(n, rng)
    runs = []
    for _ in range(2):
        p = engine.DeviceState.from_numpy(psi0, be).apply_pauli_rotations(x, z, angles)
        runs.append(p.pauli_rotations_adjoint(engine.DeviceState.from_numpy(lam0, be), x, z, angles))
    assert np.array_equal(runs[0].view(np.uint64), runs[1].view(np.uint64))
    with pytest.raises(ValueError):
        psi.pauli_rotations_adjoint(dlam, [1], [0], [0.1])        # not the same kind of state
    with pytest.raises(ValueError):
        observables.expect_and_gradient(PauliSum([(1j, "ZZ")]), (x, z, angles), rand_ket(n, rng))


def test_apply_kets_emulator(emu_backend):
    check_apply_kets(emu_backend, range(1, 13))


def test_apply_density_matrices_emulator(emu_backend):
    check_apply_density_matrices(emu_backend, range(1, 7))


def test_apply_passes_and_edges_emulator(emu_backend):
    check_apply_passes_and_edges(emu_backend)


def test_gradients_kets_emulator(emu_backend):
    check_gradients_kets(emu_backend, range(1, 11))


def test_gradients_density_matrices_emulator(emu_backend):
    check_gradients_density_matrices(emu_backend, range(1, 6))


def test_qaoa_shared_parameters_emulator(emu_backend):
    check_qaoa(emu_backend)


def test_sweep_launches_emulator(emu_backend):
    check_sweep_launches(emu_backend)


# ---- argument checks of both libraries ---------------------------------------------------------------
@pytest.fixture(scope="module", params=["cuda", "emu"])
def lib(request):
    lib = ctypes.CDLL(build_native.build_cuda() if request.param == "cuda" else build_native.build_emu())
    _capi.declare(lib)
    return lib


def _argument_cases(lib):
    a = np.zeros(64, dtype=np.complex128)
    b = np.zeros(64, dtype=np.complex128)
    pa, pb = a.ctypes.data, b.ctypes.data
    one = np.ones(1, dtype=np.uint64)
    zero = np.zeros(1, dtype=np.uint64)
    big = np.array([1 << 6], dtype=np.uint64)
    coef = np.array([0.5, 0.25])
    ang = np.array([0.5])
    out = np.zeros(1)
    o, z, bg, c, an, po = one.ctypes.data, zero.ctypes.data, big.ctypes.data, coef.ctypes.data, ang.ctypes.data, \
        out.ctypes.data
    ap, adj, adm = lib.qsim_apply_pauli_sum, lib.qsim_pauli_rotations_adjoint, lib.qsim_pauli_rotations_adjoint_dm
    cases = [
        (ap, (None, pb, 6, 1, o, z, c), "null state"),
        (ap, (pa, None, 6, 1, o, z, c), "null state"),
        (ap, (pa, None, 6, 0, None, None, None), "null state"),
        (ap, (pa, pa, 6, 1, o, z, c), "in and out must be different buffers"),
        (ap, (pa, pb, 6, 1, None, z, c), "null argument"),
        (ap, (pa, pb, 6, 1, o, None, c), "null argument"),
        (ap, (pa, pb, 6, 1, o, z, None), "null argument"),
        (ap, (pa, pb, 6, 1, bg, z, c), "at or above"),
        (ap, (pa, pb, 6, 1, z, bg, c), "at or above"),
        (ap, (pa, pb, 0, 1, z, z, c), "[1, 63]"),
        (ap, (pa, pb, 64, 0, None, None, None), "[1, 63]"),
        (ap, (pa, pb, 6, -1, o, z, c), "< 0"),
    ]
    bad_coefs = [np.array(bad) for bad in ((np.nan, 0.0), (0.0, np.inf), (-np.inf, 1.0))]
    for cb in bad_coefs:
        cases.append((ap, (pa, pb, 6, 1, o, z, cb.ctypes.data), "non-finite coefficient"))
    acc = lib.qsim_accumulate_pauli_sum                 # the same checks as qsim_apply_pauli_sum
    cases += [(acc, args, text) for fn, args, text in list(cases) if fn is ap]
    for fn in (adj, adm):
        cases += [
            (fn, (None, pb, 3, 1, o, z, an, po), "null state"),
            (fn, (pa, None, 3, 1, o, z, an, po), "null state"),
            (fn, (pa, pb, 3, 1, o, z, an, None), "null argument"),
            (fn, (pa, pb, 3, 1, None, z, an, po), "null argument"),
            (fn, (pa, pb, 3, 1, o, z, None, po), "null argument"),
            (fn, (pa, pa, 3, 1, o, z, an, po), "psi and lam must be different buffers"),
            (fn, (pa, pb, 3, 1, bg, z, an, po), "at or above"),
            (fn, (pa, pb, 0, 1, z, z, an, po), "[1, 63]"),
            (fn, (pa, pb, 3, -1, o, z, an, po), "< 0"),
        ]
        for bad in (np.nan, np.inf, -np.inf):
            ab = np.array([bad])
            cases.append((fn, (pa, pb, 3, 1, o, z, ab.ctypes.data, po), "non-finite angle"))
    cases.append((adm, (pa, pb, 32, 1, o, z, an, po), "[1, 31]"))
    return cases, (a, b, one, zero, big, coef, ang, out, bad_coefs)


def test_argument_checks(lib):
    """Both libraries refuse the same calls with the same message, before any device work (the
    buffers are host arrays)."""
    cases, _keep = _argument_cases(lib)
    for fn, args, text in cases:
        assert fn(*args, None) == -1, (fn, args)
        assert text.encode() in lib.qsim_last_error(), (lib.qsim_last_error(), text)
    for fn in (lib.qsim_pauli_rotations_adjoint, lib.qsim_pauli_rotations_adjoint_dm):
        assert fn(None, None, 6, 0, None, None, None, None, None) == 0


def test_both_libraries_give_the_same_codes_and_messages():
    libs = []
    for path in (build_native.build_cuda(), build_native.build_emu()):
        lib = ctypes.CDLL(path)
        _capi.declare(lib)
        libs.append(lib)
    results = []
    for lib in libs:
        cases, _keep = _argument_cases(lib)
        results.append([(fn(*args, None), lib.qsim_last_error()) for fn, args, _text in cases])
    assert results[0] == results[1]


# ---- sharded collectives over gloo --------------------------------------------------------------------
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
        rng = np.random.default_rng(51)
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
        for _ in range(10):
            qs = rng.choice(n, size=3, replace=False)
            terms.append({int(q): "XYZ"[int(rng.integers(3))] for q in qs})
        h = PauliSum([(complex(rng.normal(), rng.normal()), t) for t in terms])
        hr = PauliSum([(rng.normal(), t) for t in terms[:9]])
        x, z = h.x_masks, h.z_masks
        angles = rng.uniform(-3, 3, size=len(x))
        angles[2] = 0.0
        x_bits = set().union(*[{q for q in range(n) if int(v) >> q & 1} for v in x])
        several_batches = len(x_bits) > st.n_local          # no one layout serves every term
        swaps0 = st.swaps
        applied = observables.apply(h, st)
        assert isinstance(applied, sharded.ShardedState)
        after_apply = applied.gather_numpy()
        unchanged = st.gather_numpy()
        raw = st.buf.copy()
        value, grad = observables.expect_and_gradient(hr, (x, z, angles), st)
        same_buf = np.array_equal(st.buf.view(np.uint64), raw.view(np.uint64))
        # the low-level sweep: psi back to psi0
        psi = st.copy().apply_pauli_rotations(x, z, angles)
        lam = psi.apply_pauli_sum(hr.x_masks, hr.z_masks, hr.coeffs)
        g2 = psi.pauli_rotations_adjoint(lam, x, z, angles)
        back = psi.gather_numpy()
        # a sharded density matrix is refused through observables too, and its copies stay density matrices
        dm = sharded.ShardedState(6, comm, backend=emu(), as_torch=torch.from_numpy)
        sharded.ShardedSimulator([], dm, density=True)
        refused = 0
        for call in (lambda: observables.expect_and_gradient(PauliSum([(1.0, "ZZZ")]), ([1], [0], [0.3]), dm),
                     lambda: observables.apply(PauliSum([(1.0, "XZ")]), dm),
                     lambda: dm.copy().apply_pauli_rotations([1], [0], [0.3]),
                     lambda: dm.copy().apply_pauli_sum([1], [0], [1.0])):
            try:
                call()
            except NotImplementedError:
                refused += 1
        dm_copy_is_density = dm.copy().is_density and dm.empty_like().is_density
        if rank == 0:
            e = emu()
            ref_apply = engine.DeviceState.from_numpy(before, e).apply_pauli_sum(h.x_masks, h.z_masks, h.coeffs)
            ref_value, ref_grad = observables.expect_and_gradient(hr, (x, z, angles),
                                                                  engine.DeviceState.from_numpy(before, e))
            np.save(os.path.join(out_dir, "sharded.npy"),
                    np.array([norm_err(after_apply, ref_apply.to_numpy()), np.abs(unchanged - before).max(),
                              abs(value - ref_value), np.abs(grad - ref_grad).max(), np.abs(g2 - ref_grad).max(),
                              np.abs(back - before).max(), float(same_buf), st.swaps - swaps0, flipped,
                              float(several_batches), refused, float(dm_copy_is_density)]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 9), (4, 10), (8, 10)])
def test_sharded_apply_and_gradient_match_single_process(tmp_path, world, n):
    import torch.multiprocessing as mp
    build_native.build_emu()
    mp.spawn(_sharded_worker, args=(world, _free_port(), n, str(tmp_path)), nprocs=world, join=True)
    err_apply, err_state, err_value, err_grad, err_grad2, err_back, same, swaps, flipped, several, refused, \
        dm_copy = np.load(tmp_path / "sharded.npy")
    assert err_apply <= 1e-12
    assert err_state <= 1e-12
    assert err_value <= 1e-12 and err_grad <= 1e-12 and err_grad2 <= 1e-12
    assert err_back <= 1e-12
    assert same == 1.0                                   # the caller's shard is untouched
    assert swaps >= 1 and flipped >= 1                   # rank qubits were exchanged, some complemented
    assert several == 1.0                                # the sum was accumulated over several layouts
    assert refused == 4 and dm_copy == 1.0               # sharded density matrices: refused, copies included


def test_sharded_density_matrix_is_refused():
    from quantum_computations_b200 import sharded
    st = sharded.ShardedState.__new__(sharded.ShardedState)
    st.is_density = True
    with pytest.raises(NotImplementedError):
        st.apply_pauli_sum([1], [0], [0.5])
    with pytest.raises(NotImplementedError):
        st.pauli_rotations_adjoint(st, [1], [0], [0.5])


# ---- GPU -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_apply_kets_gpu(cuda_backend):
    check_apply_kets(cuda_backend, range(1, 13))


@pytest.mark.gpu
def test_apply_density_matrices_gpu(cuda_backend):
    check_apply_density_matrices(cuda_backend, range(1, 7))


@pytest.mark.gpu
def test_apply_passes_and_edges_gpu(cuda_backend):
    check_apply_passes_and_edges(cuda_backend)


@pytest.mark.gpu
def test_gradients_kets_gpu(cuda_backend):
    check_gradients_kets(cuda_backend, range(1, 11))


@pytest.mark.gpu
def test_gradients_density_matrices_gpu(cuda_backend):
    check_gradients_density_matrices(cuda_backend, range(1, 6))


@pytest.mark.gpu
def test_qaoa_shared_parameters_gpu(cuda_backend):
    check_qaoa(cuda_backend)


@pytest.mark.gpu
def test_sweep_launches_gpu(cuda_backend):
    check_sweep_launches(cuda_backend)


@pytest.mark.gpu
def test_emulator_and_cuda_agree(cuda_backend, emu_backend):
    rng = np.random.default_rng(52)
    for n in (5, 11, 16):
        psi0 = rand_ket(n, rng)
        h = rand_sum(n, rng, 60)
        got = engine.DeviceState.from_numpy(psi0, cuda_backend).apply_pauli_sum(h.x_masks, h.z_masks, h.coeffs)
        want = engine.DeviceState.from_numpy(psi0, emu_backend).apply_pauli_sum(h.x_masks, h.z_masks, h.coeffs)
        assert norm_err(got.to_numpy(), want.to_numpy()) <= 1e-14, n
        hr = rand_hamiltonian(n, rng)
        rot = rotation_list(n, rng, 80)
        vg, gg = observables.expect_and_gradient(hr, rot, engine.DeviceState.from_numpy(psi0, cuda_backend))
        ve, ge = observables.expect_and_gradient(hr, rot, engine.DeviceState.from_numpy(psi0, emu_backend))
        assert abs(vg - ve) <= 1e-13 and np.abs(gg - ge).max() <= 1e-13, n
        N = n // 2
        rho0 = rand_rho(N, rng)
        hN = rand_hamiltonian(N, rng)
        rotN = rotation_list(N, rng, 40)
        vg, gg = observables.expect_and_gradient(hN, rotN, engine.DeviceState.from_numpy(rho0, cuda_backend))
        ve, ge = observables.expect_and_gradient(hN, rotN, engine.DeviceState.from_numpy(rho0, emu_backend))
        assert abs(vg - ve) <= 1e-13 and np.abs(gg - ge).max() <= 1e-13, n


@pytest.mark.gpu
@pytest.mark.parametrize("n", [28, 30])
def test_qaoa_gradient_matches_parameter_shift_gpu(cuda_backend, n):
    import torch
    cost, rot, _param, _dtheta = qaoa(n, [0.37], [0.61])
    x, z, angles = rot
    plus = np.array([1.0, 1.0]) / np.sqrt(2)
    st = engine.DeviceState.product([plus] * n, cuda_backend)
    value, grad = observables.expect_and_gradient(cost, rot, st)

    def e(a):
        s = st.copy().apply_pauli_rotations(x, z, a)
        v = observables.expect(cost, s).real
        del s
        return v
    assert abs(value - e(angles)) <= 1e-10
    for t in (0, n // 2, n - 1, n, n + 7, 2 * n - 1):              # ZZ and X rotations
        up, dn = angles.copy(), angles.copy()
        up[t] += np.pi / 2
        dn[t] -= np.pi / 2
        assert abs(grad[t] - (e(up) - e(dn)) / 2) <= 1e-10, t
    del st
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_heisenberg_norm_on_product_state_30_qubits_gpu(cuda_backend):
    """||H psi||^2 = sum_{s,t} c_s c_t <P_s P_t> on a product state, <P_s P_t> the product over the
    qubits of the single-qubit expectation values of sigma_s sigma_t."""
    import torch
    n = 30
    h = heisenberg(n)
    rng = np.random.default_rng(53)
    kets = [rand_ket(1, rng) for _ in range(n)]
    st = engine.DeviceState.product(kets, cuda_backend)
    hpsi = observables.apply(h, st)
    got = hpsi.norm() ** 2
    del hpsi
    torch.cuda.empty_cache()
    sig = [np.eye(2), np.array([[0, 1], [1, 0]]), np.array([[0, -1j], [1j, 0]]), np.diag([1.0, -1.0])]
    letters = np.array([h._letters(t, n) for t in range(len(h))])             # [term][qubit]
    # e[q][a][b] = <phi_q| sigma_a sigma_b |phi_q>
    e = np.array([[[np.vdot(k, sig[a] @ sig[b] @ k) for b in range(4)] for a in range(4)] for k in kets])
    c = h.coeffs.real
    total = 0.0 + 0.0j
    for s in range(len(h)):
        prod = np.ones(len(h), dtype=np.complex128)
        for q in range(n):
            prod *= e[q, letters[s, q], letters[:, q]]
        total += c[s] * np.dot(c, prod)
    assert abs(total.imag) <= 1e-10
    assert abs(got - total.real) <= 1e-10 * total.real
    del st
    torch.cuda.empty_cache()
