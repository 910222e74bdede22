"""Code that only the CUDA library runs, each path against a plain NumPy reference:

- the fused peer-to-peer exchange (``qsim_exchange_p2p``, ``k_exchange_p2p``), with a world of
  2^g ranks played by 2^g shards of one GPU, and its argument checks;
- the one-gate entry points (``qsim_apply_matrix``, ``_diagonal``, ``_permutation``,
  ``_superop``) by value, on the host emulator and on the GPU: k = 5 .. 10 is the in-place
  dense-block kernel, whose tile needs more than 48 KiB of shared memory from k = 9 on;
- the tile pass with its tile loaded through TMA boxes against the same pass with plain loads.

The launch variants of the tile pass (plain loads and the dense variants) are A/B switches that
only the development build of the library reads from the environment, once per process.  Each
setting therefore runs in a child process -- this file run as a script with the development
build -- which prints one JSON line; the parent asserts on it.  The child also lists the kernels
it launched, so that a setting which did not take effect fails instead of repeating the default."""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from golden.specs import as_oracle_ops  # noqa: E402
from oracle import strided  # noqa: E402
from parity_cases import RTOL, rel_err  # noqa: E402
from quantum_computations_b200 import _capi, build_native, engine, gates  # noqa: E402

ARG, UNSUPPORTED = -1, -3
EXCH_SPLIT_BIT = 5          # kExchSplitBit (kernels.cu): which of the two ranks moves a pair


# ---- the fused exchange ----------------------------------------------------------------------------
def exchange_ref(x, g, n_local, gis, qubits):
    """The exchange as a bit permutation of the global state (index R << n_local | L): global bit
    n_local + gis[i] trades places with local index bit n_local - 1 - qubits[i]."""
    idx = np.arange(1 << (g + n_local), dtype=np.int64)
    src = idx.copy()
    for gi, q in zip(gis, qubits):
        a, b = n_local + gi, n_local - 1 - q
        flip = ((idx >> a) ^ (idx >> b)) & 1
        src ^= (flip << a) | (flip << b)
    return x.reshape(-1)[src]


def exchange_cases():
    """(g, n_local, rank bits gis, local qubits): k = 1 .. 8 at the smallest n_local (k + 6),
    rank bits a random subset of g > k in random order, local index bits below, at and above
    EXCH_SPLIT_BIT in random order, and one shard of 2^23 amplitudes (2^21 pairs per rank: several
    grid-stride trips at the default launch)."""
    rng = np.random.default_rng(11)
    shapes = [(k, k, k + 6) for k in range(1, 9)]
    shapes += [(1, 3, 9), (2, 4, 10), (3, 5, 12), (3, 6, 9), (5, 7, 12), (2, 2, 16), (1, 1, 23)]
    cases = []
    for k, g, n_local in shapes:
        gis = [int(v) for v in rng.permutation(g)[:k]]
        edge = [int(rng.integers(0, EXCH_SPLIT_BIT)), EXCH_SPLIT_BIT, int(rng.integers(EXCH_SPLIT_BIT + 1, n_local))]
        pos = {int(v) for v in rng.permutation(edge)[:k]}
        while len(pos) < k:
            pos.add(int(rng.integers(0, n_local)))
        qubits = [n_local - 1 - p for p in rng.permutation(sorted(pos))]
        cases.append((g, n_local, gis, qubits))
    return cases


def exchange_all(lib, x, g, n_local, gis, qubits, ranks):
    """Every rank's qsim_exchange_p2p, as sharded._exchange_fused makes it, on the current stream
    of the (2^g, 2^n_local) device tensor x; every shard's partners are the other rows of x."""
    import torch
    k = len(gis)
    base, shard_bytes = x.data_ptr(), 16 << n_local
    peers = (C.c_void_p * (1 << k))()
    lower = (C.c_int * (1 << k))()
    local = (C.c_int * k)(*qubits)
    stream = torch.cuda.current_stream().cuda_stream
    for r in ranks:
        for d in range(1, 1 << k):
            partner = r
            for i in range(k):
                partner ^= ((d >> i) & 1) << gis[i]
            peers[d] = base + partner * shard_bytes
            lower[d] = 1 if partner < r else 0
        mine = (C.c_int * k)(*[(r >> gi) & 1 for gi in gis])
        _capi.check(lib, lib.qsim_exchange_p2p(C.c_void_p(base + r * shard_bytes), peers, n_local, k, local, mine,
                                               lower, C.c_void_p(stream)))
    torch.cuda.synchronize()


def run_exchange_cases(lib):
    """For every case: all ranks in order, all ranks in reverse order (each pair is moved by one
    of its two ranks, so the order cannot matter) and the same exchange twice (an involution).
    Returns one failure description per wrong result; the data is pure movement, so every
    comparison is bit-exact."""
    import torch
    failures = []
    rng = np.random.default_rng(12)
    for g, n_local, gis, qubits in exchange_cases():
        size = 1 << (g + n_local)
        x0 = rng.random(size) + 1j * rng.random(size)
        want = exchange_ref(x0, g, n_local, gis, qubits)
        tag = f"g={g} n_local={n_local} gis={gis} qubits={qubits}"
        x = torch.from_numpy(x0.reshape(1 << g, 1 << n_local)).cuda()
        exchange_all(lib, x, g, n_local, gis, qubits, range(1 << g))
        if not np.array_equal(x.cpu().numpy().reshape(-1), want):
            failures.append(tag + ": ranks in order")
        exchange_all(lib, x, g, n_local, gis, qubits, range(1 << g))
        if not np.array_equal(x.cpu().numpy().reshape(-1), x0):
            failures.append(tag + ": twice is not the identity")
        x.copy_(torch.from_numpy(x0.reshape(1 << g, 1 << n_local)))
        exchange_all(lib, x, g, n_local, gis, qubits, reversed(range(1 << g)))
        if not np.array_equal(x.cpu().numpy().reshape(-1), want):
            failures.append(tag + ": ranks in reverse order")
        del x
    return failures


@pytest.mark.gpu
def test_exchange_matches_bit_permutation(cuda_backend):
    assert run_exchange_cases(cuda_backend.lib) == []


def _exch(L, null=None, n_local=12, nbits=1, qubits=(0,), bits=(0,), drop_peer=None):
    st = np.zeros(64, dtype=np.complex128)
    a = {"shard": st.ctypes.data, "peers": (C.c_void_p * 256)(*([st.ctypes.data] * 256)),
         "qubits": (C.c_int * 9)(*qubits), "bits": (C.c_int * 9)(*bits), "lower": (C.c_int * 256)()}
    if drop_peer is not None:
        a["peers"][drop_peer] = None
    if null is not None:
        a[null] = None
    return L.qsim_exchange_p2p(a["shard"], a["peers"], n_local, nbits, a["qubits"], a["bits"], a["lower"], None)


def _exch_arg_cases():
    cs = []

    def case(name, kw, msg):
        cs.append(pytest.param(kw, "qsim_exchange_p2p: " + msg, id=name))

    for what in ("shard", "peers", "qubits", "bits", "lower"):
        case("null-" + what, dict(null=what), "null argument")
    m = "bad sizes (blocks must hold at least 64 amplitudes)"
    case("nbits0", dict(nbits=0), m)
    case("nbits9", dict(n_local=20, nbits=9, qubits=range(9), bits=[0] * 9), m)
    case("block-32-amplitudes-k1", dict(n_local=6, nbits=1), m)
    case("block-32-amplitudes-k3", dict(n_local=8, nbits=3, qubits=(0, 1, 2), bits=(0, 0, 0)), m)
    m = "bad qubit or bit"
    case("bit2", dict(bits=(2,)), m)
    case("bit-neg", dict(bits=(-1,)), m)
    case("qubit-neg", dict(qubits=(-1,)), m)
    case("qubit-n-local", dict(qubits=(12,)), m)
    case("qubit-n-local-second", dict(nbits=2, qubits=(3, 12), bits=(0, 1)), m)
    case("repeated", dict(nbits=2, qubits=(4, 4), bits=(0, 1)), "repeated qubit")
    case("missing-peer", dict(nbits=2, qubits=(4, 7), bits=(0, 1), drop_peer=2), "missing peer pointer")
    case("missing-last-peer", dict(nbits=3, qubits=(4, 7, 1), bits=(0, 1, 1), drop_peer=7), "missing peer pointer")
    return cs


@pytest.fixture(scope="module")
def cuda_lib():
    lib = C.CDLL(build_native.build_cuda())
    _capi.declare(lib)
    return lib


@pytest.mark.parametrize("kw, message", _exch_arg_cases())
def test_exchange_refuses_bad_arguments_before_any_cuda_call(cuda_lib, kw, message):
    """Host arrays and no GPU: a check that came after the device binding would answer
    QSIM_ERR_CUDA instead."""
    assert _exch(cuda_lib, **kw) == ARG
    assert cuda_lib.qsim_last_error().decode() == message


def test_exchange_is_unsupported_on_the_emulator(emu_backend):
    assert _exch(emu_backend.lib) == UNSUPPORTED
    assert b"no peer memory" in emu_backend.lib.qsim_last_error()


# ---- the one-gate entry points ---------------------------------------------------------------------
class _OneGate:
    """Runs one entry point on a copy of a host state: host arrays on the emulator; on the GPU a
    device buffer and a stream of its own, read back only after the call has returned."""

    def __init__(self, name, lib, torch=None):
        self.name, self.lib, self.torch = name, lib, torch

    def __call__(self, fn, state, *args):
        if self.torch is None:
            buf = np.array(state, dtype=np.complex128, copy=True)
            _capi.check(self.lib, getattr(self.lib, fn)(buf.ctypes.data, *args))
            return buf
        torch = self.torch
        buf = torch.from_numpy(np.ascontiguousarray(state, dtype=np.complex128)).cuda()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        _capi.check(self.lib, getattr(self.lib, fn)(buf.data_ptr(), *args[:-1], C.c_void_p(side.cuda_stream)))
        side.synchronize()
        return buf.cpu().numpy()


@pytest.fixture(scope="module", params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def one_gate(request):
    if request.param == "emu":
        return _OneGate("emu", request.getfixturevalue("emu_backend").lib)
    import torch
    return _OneGate("cuda", request.getfixturevalue("cuda_backend").lib, torch)


def D(a):
    return np.ascontiguousarray(a, dtype=np.complex128).view(np.float64).ctypes.data_as(_capi.c_double_p)


def I(a):
    return np.ascontiguousarray(a, dtype=np.int32).ctypes.data_as(_capi.c_int_p)


def rand_ket(n, rng):
    return rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)


def rand_matrix(k, rng):
    return (rng.normal(size=(1 << k, 1 << k)) + 1j * rng.normal(size=(1 << k, 1 << k))) / np.sqrt(1 << k)


def target_sets(n, k, rng):
    """Reversed, scattered, on the lowest index bits (qubits n-1, n-2, ...: bits 0..2 included)
    and on the highest (bits 0..2 avoided once n - k >= 3)."""
    return [list(range(k))[::-1], [int(q) for q in rng.permutation(n)[:k]],
            list(range(n - 1, n - 1 - k, -1)), [int(q) for q in rng.permutation(k)]]


def _apply_matrix(run, psi, n, targets, m):
    return run("qsim_apply_matrix", psi, n, I(targets), len(targets), D(m), None, None)


@pytest.mark.parametrize("k", range(1, 11))
def test_apply_matrix_values(one_gate, k):
    """n = k .. k + 3: from k = 5 on, the dense block with 0 .. 3 column bits in its tile."""
    rng = np.random.default_rng(100 + k)
    for n in range(k, k + 4):
        psi = rand_ket(n, rng)
        for targets in target_sets(n, k, rng):
            m = rand_matrix(k, rng)
            got = _apply_matrix(one_gate, psi, n, targets, m)
            assert rel_err(got, strided.apply_matrix(psi, targets, m)) < RTOL, (one_gate.name, n, targets)


@pytest.mark.parametrize("k", [1, 3, 4, 5, 8, 9, 10])
def test_apply_matrix_many_tiles(one_gate, k):
    rng = np.random.default_rng(200 + k)
    n = 16
    psi = rand_ket(n, rng)
    for targets in target_sets(n, k, rng)[1:]:
        m = rand_matrix(k, rng)
        got = _apply_matrix(one_gate, psi, n, targets, m)
        assert rel_err(got, strided.apply_matrix(psi, targets, m)) < RTOL, (one_gate.name, targets)


@pytest.mark.parametrize("k", range(1, 5))
def test_apply_diagonal_and_permutation_values(one_gate, k):
    rng = np.random.default_rng(300 + k)
    dim = 1 << k
    for n in (k, k + 2, 9):
        psi = rand_ket(n, rng)
        for targets in target_sets(n, k, rng):
            d = rng.normal(size=dim) + 1j * rng.normal(size=dim)
            got = one_gate("qsim_apply_diagonal", psi, n, I(targets), k, D(d), None)
            assert rel_err(got, strided.apply_matrix(psi, targets, np.diag(d))) < RTOL, (one_gate.name, n, targets)
            # from k = 2 on not its own inverse, so that a permutation read as its inverse fails
            perm = rng.permutation(dim)
            while k > 1 and np.array_equal(perm[perm], np.arange(dim)):
                perm = rng.permutation(dim)
            p = np.zeros((dim, dim))
            p[perm, np.arange(dim)] = 1.0                  # column c has its 1 in row perm[c]
            got = one_gate("qsim_apply_permutation", psi, n, I(targets), k, I(perm), None)
            assert rel_err(got, strided.apply_matrix(psi, targets, p)) < RTOL, (one_gate.name, n, targets, perm)


@pytest.mark.parametrize("k", range(1, 6))
def test_apply_superop_values(one_gate, k):
    """S = sum_j kron(K_j, conj K_j) on the row-major vec(rho), against sum_j K_j rho K_j^+;
    k = 5 is the dense block on all 10 index bits of a 5-qubit vec(rho)."""
    rng = np.random.default_rng(400 + k)
    for n in range(k, 7):
        rho = rand_ket(2 * n, rng).reshape(1 << n, 1 << n)
        for targets in target_sets(n, k, rng)[:3]:
            kraus = [rand_matrix(k, rng) for _ in range(3)]
            s = sum(np.kron(kj, kj.conj()) for kj in kraus)
            got = one_gate("qsim_apply_superop", rho.reshape(-1), n, I(targets), k, D(s), None, None)
            want = strided.apply_kraus(rho, targets, kraus)
            assert rel_err(got.reshape(rho.shape), want) < RTOL, (one_gate.name, n, targets)


# ---- TMA against plain tile loads --------------------------------------------------------------------
def tile_cases():
    """(n, plan options, index bits the circuit acts on).  The tile of a pass holds its lowest
    low_bits index bits and grows with bits the circuit uses, so each bit set shapes the tile:
    one run longer than a TMA box (8 bits), two to four runs, more than four runs (the boxes
    cover only the lowest four), a tile without bits 1 and 2 (plain loads), and registers no
    larger than the tile."""
    rng = np.random.default_rng(31)
    cases = []

    def add(n, tile, low, cta, bits):
        bits = sorted({int(b) for b in bits if b < n})
        cases.append((n, dict(tile_bits=tile, low_bits=low, cta_log2=cta), bits))

    for n, tile, low, cta in ((14, 12, 4, 8), (17, 13, 3, 7), (20, 13, 4, 8), (13, 12, 2, 7)):
        add(n, tile, low, cta, range(tile))                          # one long run from bit 0
    for n, tile, low, cta, runs in ((12, 8, 3, 8, [(0, 4), (6, 9)]), (15, 10, 4, 7, [(0, 3), (5, 8), (11, 14)]),
                                    (18, 11, 4, 8, [(0, 4), (6, 8), (10, 12), (14, 17)]),
                                    (16, 6, 1, 7, [(0, 3), (9, 12)]), (19, 12, 2, 8, [(0, 5), (8, 12), (15, 19)]),
                                    (20, 9, 3, 7, [(0, 3), (4, 6), (13, 16), (18, 20)])):
        add(n, tile, low, cta, [b for lo, hi in runs for b in range(lo, hi)])
    for n, tile, low, cta in ((16, 10, 3, 8), (18, 12, 4, 7), (20, 13, 4, 8), (14, 8, 2, 8), (17, 13, 1, 7)):
        add(n, tile, low, cta, [0, 1, 2] + list(range(4, n, 2)))    # isolated bits: many runs
    for n, tile, low, cta in ((12, 6, 1, 8), (15, 9, 1, 7), (19, 12, 2, 8), (13, 7, 2, 7)):
        add(n, tile, low, cta, [0] + [int(b) for b in rng.permutation(range(3, n))[:tile]])
    for n, tile, low, cta in ((12, 12, 4, 8), (12, 13, 2, 7), (13, 13, 3, 8)):
        add(n, tile, low, cta, range(n))
    for _ in range(6):                                               # anything else
        n = int(rng.integers(12, 21))
        tile = int(rng.integers(6, 14))
        bits = [int(b) for b in rng.permutation(n)[:int(rng.integers(tile, n + 1))]]
        add(n, tile, int(rng.integers(1, 5)), int(rng.choice([7, 8])), bits)
    return cases


def confined_circuit(n, bits, length, rng):
    """Random one- to four-qubit gates, dense and diagonal, on the qubits of the given index bits."""
    qs = [n - 1 - b for b in bits]
    circ = []
    for _ in range(length):
        r = int(rng.integers(0, 9))
        k = 1 if r < 3 else 2 if r < 6 else 3 if r < 8 else 4
        k = min(k, len(qs))
        t = [int(q) for q in rng.permutation(qs)[:k]]
        if r == 0:
            circ.append(gates.H(t[0]))
        elif r == 1:
            circ.append(gates.RZ(t[0], float(rng.uniform(0, 2 * np.pi))))
        elif r == 3 and k == 2:
            circ.append(gates.CX(t[0], t[1]))
        elif r == 4 and k == 2:
            circ.append(gates.CZ(t[0], t[1]))
        elif r == 5 and k == 2:
            circ.append(gates.Gate(t, np.diag(np.exp(1j * rng.uniform(0, 2 * np.pi, size=4)))))
        else:
            circ.append(gates.Gate(t, np.linalg.qr(rand_matrix(k, rng))[0]))
    return circ


def run_tile_cases(backend):
    from quantum_computations_b200.simulator import Simulator
    rng = np.random.default_rng(32)
    outs = []
    for n, opts, bits in tile_cases():
        psi = rand_ket(n, rng)
        psi /= np.linalg.norm(psi)
        circ = confined_circuit(n, bits, 40, rng)
        outs.append((psi, circ, Simulator(circ, backend=backend, plan_options=opts).run(psi)))
    return outs


KNOBS = ("QSIM_NO_TMA", "QSIM_FORCE_DENSE_VARIANT")


def run_child(env_knobs, outdir):
    """This file as a script with the development build and one setting of the switches."""
    build_native.build_cuda(dev_knobs=True)        # no-op when tests/_build is up to date
    env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    env.update(env_knobs, QSIM_LIB=build_native.CUDA_KNOBS_LIB)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [__file__, str(outdir)]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    return json.loads(lines[-1])


def _kernels(fn):
    """fn() under torch.profiler: its result and {kernel name: largest grid} of what it launched."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with tempfile.TemporaryDirectory() as d:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            result = fn()
            torch.cuda.synchronize()
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    seen = {}
    for e in events:
        if e.get("cat") == "kernel":
            seen[e["name"]] = max(seen.get(e["name"], 0), int(e.get("args", {}).get("grid", [0])[0]))
    return result, seen


def _child_main(outdir):
    import torch
    be = engine.get_backend()
    assert os.path.samefile(engine._LIB_PATH, build_native.CUDA_KNOBS_LIB)
    torch.cuda.reset_peak_memory_stats()
    outs, kernels = _kernels(lambda: run_tile_cases(be))
    np.savez(os.path.join(outdir, "tiles.npz"), *[o[2] for o in outs])
    modes = re.findall(r"k_tile_pass<\s*\d+\s*,\s*(\d+)\s*,\s*\d+\s*>", " ".join(kernels))
    report = {"dense_modes": sorted({int(m) for m in modes}), "peak_bytes": int(torch.cuda.max_memory_allocated())}
    print(json.dumps(report))


@pytest.fixture(scope="module")
def tile_outputs(cuda_backend):
    outs = run_tile_cases(cuda_backend)
    refs = [strided.run(as_oracle_ops(circ), psi)[0] for psi, circ, _ in outs]
    for (_psi, _circ, got), ref, case in zip(outs, refs, tile_cases()):
        assert rel_err(got, ref) < RTOL, case
    return [o[2] for o in outs], refs


@pytest.mark.gpu
def test_plain_tile_loads_match_tma_bit_for_bit(tile_outputs, tmp_path):
    """Both paths fill the same swizzled tile slots and run the same steps on them."""
    rep = run_child({"QSIM_NO_TMA": "1"}, tmp_path)
    assert rep["peak_bytes"] < 1 << 30
    plain = np.load(tmp_path / "tiles.npz")
    tma, refs = tile_outputs
    for i, case in enumerate(tile_cases()):
        assert rel_err(plain[f"arr_{i}"], refs[i]) < RTOL, case
        assert np.array_equal(plain[f"arr_{i}"], tma[i]), case


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2])
def test_forced_dense_variants_match_oracle(tile_outputs, tmp_path, variant):
    rep = run_child({"QSIM_FORCE_DENSE_VARIANT": str(variant)}, tmp_path)
    # variant 1 raises passes without dense steps to mode 1; passes of mostly dense steps keep mode 2
    assert rep["dense_modes"][0] == variant and set(rep["dense_modes"]) <= {1, 2}
    got = np.load(tmp_path / "tiles.npz")
    _tma, refs = tile_outputs
    for i, case in enumerate(tile_cases()):
        assert rel_err(got[f"arr_{i}"], refs[i]) < RTOL, case


if __name__ == "__main__":
    _child_main(sys.argv[1])
