"""Pauli-sum expectation values at 30 qubits on one GPU (qsim_expect_pauli).

The state is the one a ``workloads.sv_random_circuit`` run leaves behind.  For each
observable the script prints one JSON line: terms, passes (launches of the call minus the
final sum), ms per evaluation from CUDA events (warm-up, then --reps evaluations), the bytes
the passes read (passes x 16 B x 2^n) over that time, and that rate as a fraction of a
device-to-device copy measured in the same process (read + write bytes of torch's copy_).
For comparison it times the only route that exists without the kernel for one Heisenberg
term: copy the state, apply the string as gates, take inner().  The GPU name and power limit
are read in the same run.

    python tools/expect_bench.py [--qubits 30] [--reps 20] [--out FILE.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        power, clock = [v.strip() for v in out.split(",")[:2]]
        info.update(power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except Exception as exc:                      # the numbers are reported without it, marked so
        info["power_limit_w"] = f"unavailable ({exc.__class__.__name__})"
    return info


def observables(n: int, seed: int):
    from quantum_computations_b200.observables import PauliSum
    rng = np.random.default_rng(seed)
    zz = [(1.0, {q: "Z", q + 1: "Z"}) for q in range(n - 1)]
    out = {
        "a_z_and_zz": PauliSum([(1.0, {q: "Z"}) for q in range(n)] + zz),
        "b_tfim": PauliSum(zz + [(0.7, {q: "X"}) for q in range(n)]),
        "c_heisenberg": PauliSum([(1.0, {q: p, q + 1: p}) for q in range(n - 1) for p in "XYZ"]),
    }
    rand = []
    while len(rand) < 100:
        qs = rng.choice(n, size=4, replace=False)
        rand.append((float(rng.normal()), {int(q): "XYZ"[int(rng.integers(3))] for q in qs}))
    out["d_random_4local"] = PauliSum(rand)
    return out


def time_events(fn, reps: int, warmup: int = 2) -> float:
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--depth", type=int, default=2)
    ap.add_argument("--seed", type=int, default=20251020)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 20:
        ap.error("--reps must be at least 20")

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("expect_bench needs a CUDA device")
    from quantum_computations_b200 import build_native, engine, workloads
    from quantum_computations_b200.states import State
    build_native.build_cuda()
    torch.cuda.set_device(0)
    be = engine.get_backend(0)
    n = args.qubits
    info = gpu_info()
    lines = []

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)

    # device-to-device copy peak on a buffer far larger than L2
    src = torch.empty(1 << 28, dtype=torch.complex128, device=be.device)
    dst = torch.empty_like(src)
    copy_ms = time_events(lambda: dst.copy_(src), args.reps)
    copy_gbs = 2 * src.numel() * 16 / copy_ms / 1e6
    del src, dst
    torch.cuda.empty_cache()
    emit({"metric": "d2d_copy", "bytes": 2 * (1 << 28) * 16, "ms": copy_ms, "gbs": copy_gbs})

    state = engine.DeviceState.product([State.ZERO.get()] * n, be)
    circuit = workloads.sv_random_circuit(n, args.depth, args.seed)
    ops = [op for g in circuit for op in g.lowered(n, False)]
    engine.Plan(be, n, ops).execute(state.buf)
    torch.cuda.synchronize()

    for name, obs in observables(n, args.seed).items():
        x, z = obs.x_masks, obs.z_masks
        before = engine.launch_count(be)
        first = state.expect_pauli(x, z)
        passes = engine.launch_count(be) - before - 1
        ms = time_events(lambda: state.expect_pauli(x, z), args.reps)
        again = state.expect_pauli(x, z)
        read = passes * 16 * (1 << n)
        gbs = read / ms / 1e6
        emit({"metric": "expect_pauli", "observable": name, "qubits": n, "terms": len(obs), "passes": passes,
              "ms": ms, "ms_per_pass": ms / passes, "bytes_read": read, "gbs": gbs,
              "fraction_of_copy_peak": gbs / copy_gbs, "repeat_bit_identical": bool(np.array_equal(first, again)),
              "value": float(np.dot(obs.coeffs, first).real), "reps": args.reps})

    # the route without the kernel: copy, apply X_0 X_1 as gates, inner()
    xgate = np.array([[0, 1], [1, 0]], dtype=np.complex128)
    plan = engine.Plan(be, n, [([0], xgate), ([1], xgate)])

    def by_gates():
        moved = state.copy()
        plan.execute(moved.buf)
        return state.inner(moved)

    ms = time_events(by_gates, args.reps)
    kernel = state.expect_pauli([0b11], [0])
    emit({"metric": "copy_gates_inner", "observable": "X0X1", "qubits": n, "ms": ms,
          "kernel_ms": time_events(lambda: state.expect_pauli([0b11], [0]), args.reps),
          "agree": float(abs(by_gates().real - kernel[0])), "reps": args.reps})

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
