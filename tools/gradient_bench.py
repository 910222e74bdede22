"""H|psi> for a Pauli sum and adjoint gradients over Pauli rotations at 30 qubits on one GPU
(qsim_apply_pauli_sum, qsim_pauli_rotations_adjoint, observables.expect_and_gradient).

The state is the one a ``workloads.sv_random_circuit(n, 2, seed)`` run leaves behind.  Kernel
calls are timed with CUDA events (warm-up, then --reps calls), whole gradients with a host clock
around calls that end in a synchronise; one JSON line is printed per measurement.  Pass times are
given against an in-process device-to-device copy of the state (``x_copy``; the copy reads and
writes the state once):

1. one apply pass of 1 and 32 terms (X masks in a four-generator span, and Z-only) and H|psi> for
   the Heisenberg chain (XX + YY + ZZ on every bond and Z on every site, 87 terms);
2. one sweep pass of k = 1, 4, 8, 16, 32 rotations (X masks in a three-generator span) against two
   copies (``x_two_copies``), since the sweep reads and writes two states;
3. the full gradient of a first-order Heisenberg Trotter step (87 rotations) and of a QAOA MaxCut
   circuit on the ring (p = 2, 120 rotations) by ``expect_and_gradient``, against the parameter-shift
   rule through the existing calls (copy, ``apply_pauli_rotations``, ``expect``) for --shift-params
   of the rotations (``shift_params_timed``); the per-rotation cost times the rotation count is
   reported as ``shift_ms_all_extrapolated``.

The GPU name, power limit and max SM clock are read in the same run.

    python tools/gradient_bench.py [--qubits 30] [--reps 10] [--out FILE.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from expect_bench import gpu_info, observables, time_events  # noqa: E402


def qaoa_ring(n: int, gammas, betas):
    from quantum_computations_b200.observables import PauliSum
    edges = [(q, (q + 1) % n) for q in range(n)]
    cost = PauliSum([(0.5, {a: "Z", b: "Z"}) for a, b in edges])
    xs, zs, angles = [], [], []
    for g, b in zip(gammas, betas):
        for a, c in edges:
            xs.append(0)
            zs.append((1 << a) | (1 << c))
            angles.append(2 * g)
        for q in range(n):
            xs.append(1 << q)
            zs.append(0)
            angles.append(2 * b)
    return cost, (np.array(xs, dtype=np.uint64), np.array(zs, dtype=np.uint64), np.array(angles))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--seed", type=int, default=20251021)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--shift-params", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("gradient_bench needs a CUDA device")
    from quantum_computations_b200 import _capi, build_native, engine, workloads
    from quantum_computations_b200 import observables as obs
    from quantum_computations_b200.states import State
    build_native.build_cuda()
    torch.cuda.set_device(0)
    be = engine.get_backend(0)
    lib = be.lib
    n = args.qubits
    info = gpu_info()
    lines = []

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)

    state = engine.DeviceState.product([State.ZERO.get()] * n, be)
    ops = [op for g in workloads.sv_random_circuit(n, 2, args.seed) for op in g.lowered(n, False)]
    engine.Plan(be, n, ops).execute(state.buf)
    work = torch.empty_like(state.buf)
    copy_ms = time_events(lambda: work.copy_(state.buf), 20)
    emit({"metric": "d2d_copy_of_state", "qubits": n, "bytes": 2 * 16 * (1 << n), "ms": copy_ms,
          "gbs": 2 * 16 * (1 << n) / copy_ms / 1e6})
    rng = np.random.default_rng(args.seed)

    def launches(fn):
        before = lib.qsim_launch_count()
        fn()
        return int(lib.qsim_launch_count() - before)

    # 1. apply passes
    def apply(x, z, c):
        _capi.check(lib, lib.qsim_apply_pauli_sum(state.buf.data_ptr(), work.data_ptr(), n, len(x), x.ctypes.data,
                                                  z.ctypes.data, c.ctypes.data, be.stream()))
    span4 = [1 << q for q in (0, 9, 18, n - 1)]
    for kind in ("span4", "z_only"):
        for k in (1, 32):
            if kind == "span4":
                x = np.array([sum(span4[i] for i in range(4) if c >> i & 1) for c in rng.integers(1, 16, size=k)],
                             dtype=np.uint64)
            else:
                x = np.zeros(k, dtype=np.uint64)
            z = rng.integers(0, 1 << n, size=k).astype(np.uint64)
            c = np.ascontiguousarray(rng.normal(size=k) + 1j * rng.normal(size=k))
            ms = time_events(lambda: apply(x, z, c), args.reps)
            emit({"metric": "apply_pass", "kind": kind, "terms": k, "qubits": n, "passes": launches(lambda: apply(x, z, c)),
                  "ms": ms, "x_copy": ms / copy_ms, "reps": args.reps})
    heis = observables(n, args.seed)["c_heisenberg"]
    hc = np.ascontiguousarray(heis.coeffs)
    ms = time_events(lambda: apply(heis.x_masks, heis.z_masks, hc), args.reps)
    npass = launches(lambda: apply(heis.x_masks, heis.z_masks, hc))
    emit({"metric": "apply_heisenberg", "qubits": n, "terms": len(heis), "passes": npass, "ms": ms,
          "ms_per_pass": ms / npass, "x_copy_per_pass": ms / npass / copy_ms, "reps": args.reps})

    # 2. sweep passes (both states are rotated back and forth; norms stay 1)
    lam = torch.empty_like(state.buf)
    lam.copy_(state.buf)
    work.copy_(state.buf)
    span3 = [1 << q for q in (0, 15, n - 1)]
    for k in (1, 4, 8, 16, 32):
        x = np.array([sum(span3[i] for i in range(3) if c >> i & 1) for c in rng.integers(1, 8, size=k)],
                     dtype=np.uint64)
        z = rng.integers(0, 1 << n, size=k).astype(np.uint64)
        a = rng.uniform(0.1, 3.0, size=k)
        out = np.zeros(k)

        def sweep():
            _capi.check(lib, lib.qsim_pauli_rotations_adjoint(work.data_ptr(), lam.data_ptr(), n, k, x.ctypes.data,
                                                              z.ctypes.data, a.ctypes.data, out.ctypes.data,
                                                              be.stream()))
        ms = time_events(sweep, args.reps)
        emit({"metric": "adjoint_pass", "rotations": k, "qubits": n, "launches": launches(sweep), "ms": ms,
              "x_two_copies": ms / (2 * copy_ms), "reps": args.reps})
    del lam

    # 3. full gradients against parameter shift through the existing calls
    def e_shift(h, x, z, a):
        s = state.copy().apply_pauli_rotations(x, z, a)
        v = obs.expect(h, s).real
        del s
        return v

    cases = [("heisenberg_trotter_step", heis, obs.trotter_rotations(heis, 0.05)),
             ("qaoa_ring_p2",) + qaoa_ring(n, [0.4, 0.7], [0.3, 0.9])]
    for name, h, (x, z, a) in cases:
        obs.expect_and_gradient(h, (x, z, a), state)                  # warm-up
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            value, grad = obs.expect_and_gradient(h, (x, z, a), state)
        grad_ms = (time.perf_counter() - t0) * 1e3 / reps
        params = list(range(0, len(a), max(1, len(a) // args.shift_params)))[:args.shift_params]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        worst = 0.0
        for t in params:
            up, dn = a.copy(), a.copy()
            up[t] += np.pi / 2
            dn[t] -= np.pi / 2
            worst = max(worst, abs(grad[t] - (e_shift(h, x, z, up) - e_shift(h, x, z, dn)) / 2))
        torch.cuda.synchronize()
        shift_ms = (time.perf_counter() - t0) * 1e3
        emit({"metric": "full_gradient", "case": name, "qubits": n, "rotations": len(a), "terms": len(h),
              "adjoint_ms": grad_ms, "adjoint_reps": reps, "shift_params_timed": len(params), "shift_ms": shift_ms,
              "shift_ms_per_rotation": shift_ms / len(params),
              "shift_ms_all_extrapolated": shift_ms / len(params) * len(a),
              "max_abs_diff_vs_shift": worst, "value": value})

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
