"""Pauli-string rotations at 30 qubits on one GPU (qsim_apply_pauli_rotations).

The state is the one a ``workloads.sv_random_circuit(n, 2, seed)`` run leaves behind.  Every call
is timed with CUDA events (warm-up, then --reps calls) and one JSON line is printed per
measurement.  Pass times are given against an in-process device-to-device copy of the state
(``x_copy`` = pass time / copy time; the copy reads and writes the state once, as a pass does):

1. one pass of k = 1, 4, 8, 16, 32 rotations whose X masks span four dimensions, and the same
   counts Z-only (the sweep behind QS_PAULI_ROT_MAX), and for k = 1 and 32 the blocks per SM of
   the launch (through the development build, whose QSIM_ROT_BLOCKS_PER_SM the library reads);
2. one first-order Trotter step of the Heisenberg chain (XX + YY + ZZ on every bond, 87 terms at
   30 sites) against the same step lowered to 4x4 gates through the planner: time and the largest
   difference of the two states;
3. 16 random weight-n strings against a lowering to gates that exists only here: a basis change
   per qubit, a CNOT ladder, RZ, and both undone, through the planner.

The GPU name, power limit and max SM clock are read in the same run.

    python tools/rotation_bench.py [--qubits 30] [--reps 10] [--out FILE.jsonl]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from expect_bench import gpu_info, observables, time_events  # noqa: E402

H = np.array([[1, 1], [1, -1]], dtype=np.complex128) / np.sqrt(2)
SDG = np.diag([1, -1j]).astype(np.complex128)
CNOT = np.eye(4, dtype=np.complex128)[[0, 1, 3, 2]]


def ladder_gates(n: int, letters: dict, theta: float) -> list:
    """exp(-i theta/2 P) for P = prod_q letters[q] as (targets, matrix) gates: V P V^dagger = Z^w with
    V = H (X) or H S^dagger (Y) per qubit, then a CNOT ladder, RZ(theta) and the ladder undone."""
    qs = sorted(letters)
    basis = [([q], H if letters[q] == "X" else H @ SDG) for q in qs if letters[q] in "XY"]
    ladder = [([qs[i], qs[i + 1]], CNOT) for i in range(len(qs) - 1)]
    rz = ([qs[-1]], np.diag([np.exp(-0.5j * theta), np.exp(0.5j * theta)]))
    undo = [(t, m.conj().T) for t, m in basis]
    return basis + ladder + [rz] + ladder[::-1] + undo


def pauli_gates(ps, angles) -> list:
    """Each rotation as one dense gate on its support (2 qubits for the Heisenberg terms)."""
    import scipy.linalg
    from quantum_computations_b200.observables import PauliSum
    out = []
    for k in range(len(ps)):
        letters = ps._letters(k, ps.num_qubits)
        qs = [q for q in range(ps.num_qubits) if letters[q]]
        sub = PauliSum([(1, {i: "IXYZ"[letters[q]] for i, q in enumerate(qs)})]).matrix(len(qs))
        out.append((qs, scipy.linalg.expm(-0.5j * angles[k] * sub)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--seed", type=int, default=20251021)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rotation_bench needs a CUDA device")
    from quantum_computations_b200 import _capi, build_native, engine, workloads
    from quantum_computations_b200.observables import PauliSum, trotter_rotations
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

    def rotate(x, z, a, target=None, which=lib):
        buf = work if target is None else target
        _capi.check(which, which.qsim_apply_pauli_rotations(buf.data_ptr(), n, len(x), x.ctypes.data, z.ctypes.data,
                                                            a.ctypes.data, be.stream()))

    def passes(x, z, a):
        before = lib.qsim_launch_count()
        rotate(x, z, a)
        return int(lib.qsim_launch_count() - before)

    # 1. rotations per pass
    rng = np.random.default_rng(args.seed)
    span = [1 << q for q in (0, 9, 18, n - 1)]
    knobs = C.CDLL(build_native.build_cuda(dev_knobs=True))
    _capi.declare(knobs)
    for kind in ("span4", "z_only"):
        for k in (1, 4, 8, 16, 32):
            if kind == "span4":
                x = np.array([sum(span[i] for i in range(4) if c >> i & 1) for c in rng.integers(1, 16, size=k)],
                             dtype=np.uint64)
            else:
                x = np.zeros(k, dtype=np.uint64)
            z = rng.integers(0, 1 << n, size=k).astype(np.uint64)
            a = rng.uniform(0.1, 3.0, size=k)
            work.copy_(state.buf)
            ms = time_events(lambda: rotate(x, z, a), args.reps)
            emit({"metric": "rotation_pass", "kind": kind, "rotations": k, "qubits": n, "passes": passes(x, z, a),
                  "ms": ms, "x_copy": ms / copy_ms, "reps": args.reps})
            if kind == "span4" and k in (1, 32):
                for per_sm in (1, 2, 4, 8):
                    os.environ["QSIM_ROT_BLOCKS_PER_SM"] = str(per_sm)
                    ms = time_events(lambda: rotate(x, z, a, which=knobs), args.reps)
                    emit({"metric": "rotation_pass_blocks", "kind": kind, "rotations": k, "blocks_per_sm": per_sm,
                          "threads_per_block": 128, "qubits": n, "ms": ms, "x_copy": ms / copy_ms,
                          "reps": args.reps})
                os.environ.pop("QSIM_ROT_BLOCKS_PER_SM")

    # 2. a first-order Trotter step of the Heisenberg chain
    heis = observables(n, args.seed)["c_heisenberg"]
    dt = 0.05
    x, z, a = trotter_rotations(heis, dt)
    plan = engine.Plan(be, n, pauli_gates(heis, a))
    gates_out = torch.empty_like(state.buf)
    ms_rot = time_events(lambda: rotate(x, z, a), args.reps)
    ms_gates = time_events(lambda: plan.execute(gates_out), args.reps)
    work.copy_(state.buf)
    gates_out.copy_(state.buf)
    npass = passes(x, z, a)
    plan.execute(gates_out)
    diff = float((work - gates_out).abs().max().item())
    emit({"metric": "heisenberg_trotter_step", "qubits": n, "terms": len(heis), "rotation_passes": npass,
          "rotations_ms": ms_rot, "rotations_x_copy": ms_rot / copy_ms, "planner_gates": len(heis),
          "planner_passes": int(plan.stats["n_passes"]), "planner_ms": ms_gates, "planner_x_copy": ms_gates / copy_ms,
          "max_abs_diff": diff, "reps": args.reps})
    del plan

    # 3. random weight-n strings
    labels = [{q: "XYZ"[int(v)] for q, v in enumerate(rng.integers(3, size=n))} for _ in range(16)]
    ps = PauliSum([(1, lab) for lab in labels])
    a = rng.uniform(0.1, 3.0, size=len(ps))
    x, z = ps.x_masks.copy(), ps.z_masks.copy()
    gates = [g for lab, th in zip(labels, a) for g in ladder_gates(n, lab, th)]
    plan = engine.Plan(be, n, gates)
    ms_rot = time_events(lambda: rotate(x, z, a), args.reps)
    ms_gates = time_events(lambda: plan.execute(gates_out), args.reps)
    work.copy_(state.buf)
    gates_out.copy_(state.buf)
    npass = passes(x, z, a)
    plan.execute(gates_out)
    diff = float((work - gates_out).abs().max().item())
    emit({"metric": "weight_n_strings", "qubits": n, "strings": len(ps), "rotation_passes": npass,
          "rotations_ms": ms_rot, "rotations_x_copy": ms_rot / copy_ms, "planner_gates": len(gates),
          "planner_passes": int(plan.stats["n_passes"]), "planner_ms": ms_gates, "planner_x_copy": ms_gates / copy_ms,
          "max_abs_diff": diff, "reps": args.reps})

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
