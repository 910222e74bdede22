"""Lanczos iterations, ground energies and Krylov evolution at 30 qubits on one GPU
(qsim_lanczos_apply, qsim_lanczos_step, observables.ground_state / evolve_krylov).

H is the Heisenberg chain of the earlier benches (XX + YY + ZZ on every bond, 87 terms at 30
qubits); the start state is a random product state (seeded).  Kernel calls are timed with CUDA
events (warm-up, then --reps calls), whole solves with a host clock around calls that end in a
synchronise.  One JSON line is printed per measurement:

1. one Lanczos iteration (``qsim_lanczos_apply`` + ``qsim_lanczos_step``) against
   ``qsim_apply_pauli_sum`` alone plus one 3-read / 1-write pass, costed as 2 in-process state
   copies (``x_copy``: a copy reads and writes the state once);
2. ``k_lanczos_step`` alone (w <- w - a v and |w|^2: 2 reads, 1 write; with y: 3 reads, 2 writes) as
   a fraction of the in-process copy's rate;
3. the time to a 1e-10 ground energy, and to ``evolve_krylov`` of t = 1 (tol 1e-10) against
   second-order ``evolve`` at the number of steps that reaches the same error.  That step count is
   extrapolated from the Trotter errors measured at --trotter-steps (error ~ C / steps^2, errors
   from |a - b|^2 = |a|^2 + |b|^2 - 2 Re <a|b> against the Krylov result), and its time from the
   measured time per step.

The GPU name, power limit and max SM clock are read in the same run.

    python tools/krylov_bench.py [--qubits 30] [--reps 5] [--out FILE.jsonl]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from expect_bench import gpu_info, observables, time_events  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--seed", type=int, default=20251022)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--time", type=float, default=1.0)
    ap.add_argument("--tol", type=float, default=1e-10)
    ap.add_argument("--trotter-steps", default="4,8,16")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("krylov_bench needs a CUDA device")
    from quantum_computations_b200 import build_native, engine
    from quantum_computations_b200 import observables as obs
    build_native.build_cuda()
    torch.cuda.set_device(0)
    be = engine.get_backend(0)
    n = args.qubits
    na = 1 << n
    info = gpu_info()
    lines = []

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)

    rng = np.random.default_rng(args.seed)
    kets = []
    for _ in range(n):
        v = rng.normal(size=2) + 1j * rng.normal(size=2)
        kets.append(v / np.linalg.norm(v))
    heis = obs.PauliSum([(1.0, {q: p, q + 1: p}) for q in range(n - 1) for p in "XYZ"])
    assert len(heis) == len(observables(n, args.seed)["c_heisenberg"])
    x, z, c = heis.x_masks, heis.z_masks, np.ascontiguousarray(heis.coeffs)
    psi = engine.DeviceState.product(kets, be)
    a, b = be.empty(na), be.empty(na)
    a.copy_(psi.buf)
    b.copy_(psi.buf)
    state_gb = 16 * na / 1e9

    copy_ms = time_events(lambda: a.copy_(psi.buf), args.reps)
    copy_gbs = 2 * state_gb / (copy_ms / 1e3)
    emit({"metric": "x_copy", "qubits": n, "ms": copy_ms, "gb_s": copy_gbs})

    apply_ms = time_events(lambda: psi.apply_pauli_sum(x, z, c, out=engine.DeviceState(be, a, n, 1)), args.reps)
    emit({"metric": "apply_pauli_sum", "qubits": n, "terms": len(heis), "ms": apply_ms})

    def iteration():
        dot = engine.lanczos_apply(be, psi.buf, b, a, n, x, z, c, -0.5)
        engine.lanczos_step(be, a, psi.buf, None, na, dot)
    it_ms = time_events(iteration, args.reps)
    target = apply_ms + 2 * copy_ms
    emit({"metric": "lanczos_iteration", "qubits": n, "terms": len(heis), "ms": it_ms,
          "apply_plus_3r1w_pass_ms": target, "ratio": it_ms / target, "over_apply_ms": it_ms - apply_ms})

    step_ms = time_events(lambda: engine.lanczos_step(be, a, psi.buf, None, na, 1e-3), args.reps)
    emit({"metric": "lanczos_step", "qubits": n, "with_y": False, "ms": step_ms,
          "gb_s": 3 * state_gb / (step_ms / 1e3), "fraction_of_copy_rate": 3 * state_gb / (step_ms / 1e3) / copy_gbs})
    step_y_ms = time_events(lambda: engine.lanczos_step(be, a, psi.buf, b, na, 1e-3, 1e-3j), args.reps)
    emit({"metric": "lanczos_step", "qubits": n, "with_y": True, "ms": step_y_ms,
          "gb_s": 5 * state_gb / (step_y_ms / 1e3),
          "fraction_of_copy_rate": 5 * state_gb / (step_y_ms / 1e3) / copy_gbs})
    del a, b
    torch.cuda.empty_cache()

    from quantum_computations_b200 import krylov
    passes = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    energy, residual = krylov.ground_state(heis, psi, tol=args.tol, max_iter=300, _passes=passes)
    ground_s = time.perf_counter() - t0
    iters = len(passes[0][0])
    emit({"metric": "ground_state", "qubits": n, "tol": args.tol, "energy": energy, "residual": residual,
          "iterations": iters, "s": ground_s, "ms_per_iteration": 1e3 * ground_s / iters})

    subs = []
    evolved = psi.copy()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    krylov.evolve_krylov(heis, evolved, args.time, tol=args.tol, _substeps=subs)
    torch.cuda.synchronize()
    krylov_s = time.perf_counter() - t0
    emit({"metric": "evolve_krylov", "qubits": n, "time": args.time, "tol": args.tol, "s": krylov_s,
          "substeps": len(subs), "iterations": [m for m, _dt in subs], "norm": evolved.norm()})

    errs, per_step = [], []
    for steps in [int(s) for s in args.trotter_steps.split(",")]:
        trot = psi.copy()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        obs.evolve(heis, trot, args.time, steps=steps, order=2)
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        d2 = trot.norm() ** 2 + evolved.norm() ** 2 - 2 * trot.inner(evolved).real
        err = math.sqrt(max(d2, 0.0))
        errs.append((steps, err))
        per_step.append(secs / steps)
        emit({"metric": "evolve_trotter2", "qubits": n, "time": args.time, "steps": steps, "s": secs, "error": err})
        del trot
    # error ~ C / steps^2: the constant from the finest measured step count
    steps_f, err_f = errs[-1]
    need = math.ceil(steps_f * math.sqrt(err_f / args.tol))
    trot_s = need * float(np.median(per_step))
    emit({"metric": "trotter2_at_same_error", "qubits": n, "time": args.time, "error": args.tol,
          "steps_extrapolated": need, "s_extrapolated": trot_s, "krylov_s": krylov_s,
          "krylov_speedup": trot_s / krylov_s})

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
