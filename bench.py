#!/usr/bin/env python
"""Benchmark of the gate-application hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo, on GPUs
    python bench.py --impl reference [--steps K] [--warmup W]    # reference CPU algorithm
    python bench.py --steps K --dump-outputs DIR                 # also write the results (one GPU)

Workload (N=1): config C4 -- the 30-qubit complex128 random circuit, depth 200
(200 x (30 single-qubit gates from {H,T,RZ,X,P} + 15 CZ on a random perfect
matching) = 9000 gates, ``workloads.sv_random_circuit(30, 200, seed=30)``).
One *step* = the whole circuit applied to |0...0>.  Every timed loop (kernel-only,
HBM-roof operating point, end to end) runs exactly --steps steps.

--dump-outputs DIR writes, after the timed steps, what the last step computed, as
float64 .npy files (48 MiB at n = 30), so that two builds can be compared output for
output; the circuit and the sample are seeded, so the same arguments give the same inputs:
  state_sample_index  2^20 basis-state indices drawn without replacement (seed DUMP_SEED)
  state_sample        the final amplitudes of the kernel-only path at those indices, (k, 2) = (re, im)
  state_marginal      probabilities of the 2^20 basis states of qubits 0..19 (summed over the
                      other qubits): every amplitude of the state contributes
  e2e_sample          the array Simulator.run returned in the last end-to-end step, at the same
                      indices (unless the end-to-end run is skipped)

Reported on one JSON line:
  value      gates/s with the state resident in HBM and the fused plan compiled
             (the timed region is the tile-pass kernels only, CUDA events).
  e2e        gates/s through the public API ``Simulator(circuit).run([ZERO]*n, out=pinned)``:
             host circuit objects in; lowering, plan lookup (the plan compiled by the
             warm-up run is reused through the simulator's content-keyed cache, compile
             time is config.plan_seconds), product state, launches and the device->host
             copy of the final 2^n amplitudes inside the timed region.
  roofline   k_tile_pass: algorithmic bytes per launch = 2 x 16 B x 2^n (one read and
             one write of the state) over the mean launch time, against the measured
             HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the reference's own algorithm (oracle/dense_ref.py: dense 2^N x 2^N
             operator per gate) timed on the host cores on a bounded sample of the
             same generator at the largest N that fits the time budget.

The state (16 GiB at n=30) is far larger than the 126 MB L2, so every pass
streams from HBM; no L2 flush is needed between iterations.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "gates/sec (30q c128 random circuit, depth 200)"
METRIC_SHARDED = "gates/sec (34q c128 random circuit, depth 200, sharded over the GPUs)"


def metric_sharded(n: int, depth: int) -> str:
    return f"gates/sec ({n}q c128 random circuit, depth {depth}, sharded over the GPUs)"
ALT_MAX_DENSE = 10           # matrices per pass of the HBM-roof operating point (roofline_hbm_point); measured
ALT_MAX_GROUP = 0            # curve (DESIGN.md section 5): 8 -> 0.79, 10 -> 0.73, 12 -> 0.69, 16 -> 0.59, 20 -> 0.54
PASS_PARAM_BYTES = 28672     # sizeof(QsPass) + tensor map + geometry: kernel parameters per tile-pass launch
# dram__bytes_read.sum + dram__bytes_write.sum per k_tile_pass launch at n = 30, default plan options, from the
# `ncu --set full` captures summarised in profiles/r2_ncu_full_k_tile_pass_p16.csv (17.18 GB + 17.12 GB)
NCU_TRAFFIC_N30 = 34.30e9


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--qubits", type=int, default=0, help="0 = 30 on one GPU, 34 sharded over N > 1 GPUs")
    ap.add_argument("--depth", type=int, default=200)
    ap.add_argument("--seed", type=int, default=30)
    ap.add_argument("--tile-bits", type=int, default=0)
    ap.add_argument("--low-bits", type=int, default=0)
    ap.add_argument("--max-group", type=int, default=0)
    ap.add_argument("--max-dense", type=int, default=0)
    ap.add_argument("--lookahead", type=int, default=0)
    ap.add_argument("--max-layers", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the HBM-roof operating point")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C1-C3 secondary entries")
    ap.add_argument("--rb-sequences", type=int, default=10000)
    ap.add_argument("--no-check", action="store_true", help="sharded: skip the circuit-then-inverse check")
    ap.add_argument("--check-depth", type=int, default=30)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per k_tile_pass launch from an ncu --set full capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is implemented for the single-GPU run")
    return args


# ---- helpers ---------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self) -> dict:
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def cpu_baseline(seconds: float, seed: int) -> dict:
    """Time the reference's algorithm (dense operator per gate, oracle/dense_ref.py)
    on the same generator at N=12, for about ``seconds`` of CPU work."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from golden.specs import as_oracle_ops
    from oracle import dense_ref
    from quantum_computations_b200 import workloads
    n = 12
    ops = as_oracle_ops(workloads.sv_random_circuit(n, 200, seed))
    state = np.zeros(2 ** n, dtype=np.complex128)
    state[0] = 1.0
    done, t0 = 0, time.perf_counter()
    while done < len(ops):
        state, _ = dense_ref.run([ops[done]], state)
        done += 1
        if time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "gates/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"first {done} gates of the same generator at N={n} (the reference's dense 2^N x 2^N "
                      f"operator path cannot hold N=30); numpy {np.__version__}",
            "seconds": dt}


def plan_options(args) -> dict:
    return {"tile_bits": args.tile_bits, "low_bits": args.low_bits, "max_group": args.max_group,
            "max_dense_ops": args.max_dense, "lookahead": args.lookahead, "max_layers": args.max_layers}


# ---- secondary configurations (BASELINE.json configs C1-C3) ---------------------------------------------
RB_DEPTHS = (8, 10, 15, 20)


def rb_circuits(count: int, seed: int = 20251018):
    from quantum_computations_b200 import workloads
    rng = np.random.default_rng(seed)
    return [workloads.rb_random_circuit(2, RB_DEPTHS[i % 4], rng) for i in range(count)]


def _rb_cpu_sequence(spec):
    """One RB sequence by the reference's algorithm (oracle/dense_ref.py): dense operators on the
    2-qubit density matrix, Kraus sums for the GKP channel.  Returns (fidelity, purity)."""
    sys.path.insert(0, ROOT)
    from oracle import dense_ref, gkp_noise
    from quantum_computations_b200 import channels, gates
    noise = channels.GKPNoise(10.0)
    rho = np.zeros((4, 4), dtype=np.complex128)
    rho[0, 0] = 1.0
    psi = np.array([1, 0, 0, 0], dtype=np.complex128)
    for name, idx in spec:
        g = getattr(gates, name)(*idx)
        rho = dense_ref.apply_matrix(rho, g.indices, g.matrix)
        psi = dense_ref.apply_matrix(psi, g.indices, g.matrix)
        for q, (px, pz) in zip(g.indices, noise.flips_for(g)):
            rho = dense_ref.apply_kraus(rho, [q], gkp_noise.pauli_flip_kraus(px, pz))
    return float(dense_ref.fidelity(rho, psi)), float(dense_ref.purity(rho))


def _rb_cpu_chunk(specs):
    return [_rb_cpu_sequence(s) for s in specs]


def secondary_rb(sequences: int, cpu_seconds: float, rank: int = 0, world: int = 1, gather=None) -> dict:
    """C2: `sequences` two-qubit RB sequences (the reference's random_circ generator, depths
    8/10/15/20) as density matrices with the 10 dB GKP channel after every gate."""
    import multiprocessing as mp
    import torch
    from quantum_computations_b200 import batched, channels
    t0 = time.perf_counter()
    circuits = rb_circuits(sequences)
    gen_s = time.perf_counter() - t0
    ngates = sum(len(c) for c in circuits)
    sim = batched.BatchedSimulator(2, channels.GKPNoise(10.0))

    def once():
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = batched.run_replicas(sim, circuits, rank=rank, world=world, gather=gather)
        torch.cuda.synchronize()
        return r, time.perf_counter() - t

    res, cold_s = once()                       # first sight of the gate objects: opcodes are worked out
    res, warm_s = once()
    res, warm2_s = once()
    warm_s = min(warm_s, warm2_s)
    out = {"config": "C2", "workload": f"{sequences} two-qubit RB sequences (depths {list(RB_DEPTHS)}), density "
                                       "matrix + GKP channel at 10 dB", "gates": ngates,
           "sequences_per_s": sequences / warm_s, "seconds_e2e": warm_s, "seconds_e2e_first_call": cold_s,
           "note": "host circuit objects in, fidelity/purity arrays out; the first call also derives the opcode of "
                   "every gate object, later calls read it back from the objects",
           "circuit_generation_seconds": gen_s, "n_gpus": world}
    if rank == 0:
        specs = [[(type(g).__name__, list(g.indices)) for g in c] for c in circuits]
        # one process
        n1, t = 0, time.perf_counter()
        worst = 0.0
        while n1 < len(specs) and time.perf_counter() - t < cpu_seconds / 2:
            f, pu = _rb_cpu_sequence(specs[n1])
            if world == 1 or gather is not None:
                worst = max(worst, abs(res["fidelity"][n1] - f), abs(res["purity"][n1] - pu))
            n1 += 1
        one = n1 / (time.perf_counter() - t)
        # multiprocessing.Pool over the host cores (PAPER/average_clifford_fidelity.py:212-214)
        cores = os.cpu_count() or 1
        per = max(8, int(one * cpu_seconds / 2))
        chunks = [specs[(i * per) % len(specs):][:per] for i in range(cores)]
        try:
            with mp.get_context("spawn").Pool(cores) as pool:
                pool.map(_rb_cpu_chunk, [c[:2] for c in chunks])      # start the workers
                t = time.perf_counter()
                pool.map(_rb_cpu_chunk, chunks)
                many = sum(len(c) for c in chunks) / (time.perf_counter() - t)
        except Exception as exc:                                       # pragma: no cover
            many = None
            out["cpu_pool_error"] = repr(exc)
        out.update({"cpu_port_sequences_per_s_1_process": one, "cpu_port_sequences_per_s_pool": many,
                    "cpu_cores": cores, "cpu_sample": n1,
                    "speedup_vs_1_process": sequences / warm_s / one,
                    "speedup_vs_pool": (sequences / warm_s / many) if many else None,
                    "max_abs_diff_fidelity_purity_vs_oracle": worst,
                    "mean_fidelity": float(np.mean(res["fidelity"])), "mean_purity": float(np.mean(res["purity"]))})
    return out


def secondary_grover() -> dict:
    """C1: the reference's 3-qubit Grover circuit on rho with the GKP channel, checked against
    vectors produced by the reference itself (tests/golden/noisy_grover.npz)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from golden.specs import from_spec
    from quantum_computations_b200 import channels, gates, simulator, states
    from quantum_computations_b200.simulator import Simulator
    z = np.load(os.path.join(ROOT, "tests", "golden", "noisy_grover.npz"))
    meta = json.loads(str(z["meta"]))
    worst, secs, nops = 0.0, [], 0
    for rec in meta:
        circ = [from_spec(s, gates, simulator, z, channels, states) for s in rec["circuit"]]
        noisy = channels.GKPNoise(rec["db"]).noisy(circ)
        rho0 = np.zeros((8, 8), dtype=np.complex128)
        rho0[0, 0] = 1.0
        sim = Simulator(noisy)
        sim.run(rho0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = sim.run(rho0)
        torch.cuda.synchronize()
        secs.append(time.perf_counter() - t0)
        worst = max(worst, float(np.abs(got - z[rec["out"]]).max() / np.abs(z[rec["out"]]).max()))
        nops = len(noisy)
    return {"config": "C1", "workload": "3-qubit Grover search on rho with the GKP finite-squeezing channel",
            "runs": len(meta), "ops_per_run": nops, "seconds_per_run": float(np.mean(secs)),
            "max_rel_err_vs_reference_vectors": worst}


def secondary_dm(n: int = 12, depth: int = 100, plan_opts: dict | None = None) -> dict:
    """C3: n-qubit density matrix (2n-bit vec), layered Clifford+T circuit, a GKP channel after
    every gate; parity of the same generator at n = 6 against the CPU oracle."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from golden.specs import as_oracle_ops
    from oracle import strided
    from quantum_computations_b200 import channels, engine, workloads
    from quantum_computations_b200.simulator import Simulator
    from quantum_computations_b200.states import State
    noise = channels.GKPNoise(10.0)
    layers = workloads.dm_random_layers(n, depth, 12)
    circ = noise.noisy([g for layer in layers for g in layer])
    be = engine.get_backend()
    ops = []
    for g in circ:
        ops.extend(g.lowered(n, True))
    t0 = time.perf_counter()
    plan = engine.Plan(be, 2 * n, ops, plan_opts or {})
    plan_s = time.perf_counter() - t0

    def fresh():
        st = engine.DeviceState.product([State.ZERO.get()] * (2 * n), be)
        st.ndim = 2
        return st

    state = fresh()
    plan.execute(state.buf)
    torch.cuda.synchronize()
    best = None
    for _ in range(3):
        state = fresh()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        plan.execute(state.buf)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    # parity at a size the oracle reaches
    ns = 6
    small = noise.noisy([g for layer in workloads.dm_random_layers(ns, 20, 12) for g in layer])
    rho0 = np.zeros((2 ** ns, 2 ** ns), dtype=np.complex128)
    rho0[0, 0] = 1.0
    got = Simulator(small).run(rho0)
    ref, _ = strided.run(as_oracle_ops(small), rho0)
    err = float(np.abs(got - ref).max() / np.abs(ref).max())
    passes = plan.stats["n_passes"]
    return {"config": "C3", "workload": f"{n}-qubit noisy density matrix ({2 * n}-bit vec), Clifford+T depth {depth}, "
                                        "per-gate GKP channels", "ops_with_channels": len(circ), "plan": plan.stats,
            "plan_seconds": plan_s, "ms_total": best, "ms_per_pass": best / max(1, passes),
            "us_per_gate_or_channel": 1e3 * best / len(circ), "trace": float(state.trace().real),
            "purity": float(state.purity()), "parity_rel_err_vs_oracle_n6": err}


# ---- reference arm -----------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = None
    for _ in range(max(1, args.warmup) - 1):
        cpu_baseline(min(2.0, args.cpu_seconds), args.seed)
    vals = []
    t_all = time.perf_counter()
    for _ in range(max(1, args.steps)):
        base = cpu_baseline(args.cpu_seconds, args.seed)
        vals.append(base["value"])
    total = time.perf_counter() - t_all
    value = float(np.mean(vals))
    base["value"] = value
    metric = METRIC if args.gpus == 1 else METRIC_SHARDED
    line = {"impl": "reference", "metric": metric, "value": value, "unit": "gates/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak" if args.gpus == 1 else "strong", "vs_baseline": None,
            "dtype": "c128", "data": "synthetic",
            "config": {"workload": "C4 generator (sv_random_circuit, depth 200, seed 30) run by the reference's "
                                   "dense-operator algorithm at N=12; it cannot hold N=30 or N=34",
                       "same_config": False},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "gates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---- B200 arm ---------------------------------------------------------------------------------------------
def time_plan(backend, plan, state, reset, steps: int):
    """CUDA-event time of `steps` executions of a resident plan (ms, total)."""
    import torch
    total = 0.0
    for _ in range(steps):
        reset()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        plan.execute(state.buf)
        ev1.record()
        torch.cuda.synchronize()
        total += ev0.elapsed_time(ev1)
    return total


DUMP_SEED = 20251020
DUMP_SAMPLE_LOG2 = 20
DUMP_MARGINAL_QUBITS = 20


def dump_sample_index(n: int) -> np.ndarray:
    """The sorted basis-state indices whose amplitudes --dump-outputs writes (every index up to n = 20)."""
    size = 1 << min(n, DUMP_SAMPLE_LOG2)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(1 << n, size=size, replace=False))


def as_re_im(amps: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(amps, dtype=np.complex128).view(np.float64).reshape(-1, 2)


def dump_device_state(out_dir: str, buf, n: int) -> None:
    """Sample and qubit-0..19 marginal of the 2^n device state ``buf`` (torch complex128)."""
    import torch
    idx = dump_sample_index(n)
    np.save(os.path.join(out_dir, "state_sample_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "state_sample.npy"),
            as_re_im(buf[torch.from_numpy(idx).to(buf.device)].cpu().numpy()))
    m = min(n, DUMP_MARGINAL_QUBITS)
    rows = buf.reshape(1 << m, -1)                    # row r: the basis states whose qubits 0..m-1 read r
    chunk = max(1, (1 << 26) // rows.shape[1])        # bounds the temporary to 1 GiB
    marginal = torch.cat([torch.view_as_real(rows[r:r + chunk]).square().sum(dim=(1, 2))
                          for r in range(0, rows.shape[0], chunk)])
    np.save(os.path.join(out_dir, "state_marginal.npy"), marginal.cpu().numpy())


def run_b200(args):
    import torch
    from quantum_computations_b200 import _capi, engine, workloads
    from quantum_computations_b200.simulator import Simulator
    from quantum_computations_b200.states import State

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        from bench_sharded import run_sharded
        return run_sharded(args, world, rank, local_rank)

    n = args.qubits or 30
    backend = engine.get_backend(local_rank)
    opts = plan_options(args)
    circuit = workloads.sv_random_circuit(n, args.depth, args.seed)
    ngates = len(circuit)

    # compile once (resident plan) for the kernel-only number
    t0 = time.perf_counter()
    ops = []
    for g in circuit:
        ops.extend(g.lowered(n, False))
    plan = engine.Plan(backend, n, ops, opts)
    plan_seconds = time.perf_counter() - t0
    stats = plan.stats
    passes = stats["n_passes"]

    state = engine.DeviceState.product([State.ZERO.get()] * n, backend)
    amps = np.ascontiguousarray(np.stack([np.asarray(State.ZERO.get(), dtype=np.complex128)] * n))

    def reset():
        _capi.check(backend.lib, backend.lib.qsim_init_product(
            backend.ptr(state.buf), n, amps.view(np.float64).ctypes.data_as(_capi.c_double_p), backend.stream()))

    for _ in range(args.warmup):
        reset()
        plan.execute(state.buf)
    torch.cuda.synchronize()

    launches0 = engine.launch_count(backend)
    with ClockSampler(local_rank) as clocks:
        kernel_ms = time_plan(backend, plan, state, reset, args.steps)
    launches = engine.launch_count(backend) - launches0 - args.steps      # minus the reset kernels
    norm = state.norm()
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        dump_device_state(args.dump_outputs, state.buf, n)
    value = args.steps * ngates / (kernel_ms * 1e-3)
    ms_per_step = kernel_ms / args.steps

    peak, peak_src = measured_peaks()
    bytes_per_launch = 2.0 * 16.0 * (2.0 ** n)
    launch_ms = kernel_ms / max(1, args.steps * passes)
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    traffic = args.traffic_bytes
    if traffic is None and n == 30:
        traffic = NCU_TRAFFIC_N30
    roofline = {"bound": "hbm", "kernel": "k_tile_pass", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "bytes_per_launch": bytes_per_launch, "launches_per_step": passes,
                "mean_launch_ms": launch_ms,
                "operating_point": "default plan: as many gates per HBM pass as the SM absorbs (max gates/s)"}

    # the same circuit planned for the HBM roof instead of for gates/s: fewer gates per pass
    roofline_hbm_point = None
    if not args.no_alt and not any(opts.values()):
        alt_opts = dict(opts, max_dense_ops=ALT_MAX_DENSE, max_group=ALT_MAX_GROUP)
        alt = engine.Plan(backend, n, ops, alt_opts)
        reset()
        alt.execute(state.buf)
        alt_steps = args.steps
        alt_ms = time_plan(backend, alt, state, reset, alt_steps)
        alt_launch = alt_ms / (alt_steps * alt.stats["n_passes"])
        alt_ach = bytes_per_launch / (alt_launch * 1e-3) / 1e9
        roofline_hbm_point = {"bound": "hbm", "kernel": "k_tile_pass", "achieved": alt_ach, "peak": peak,
                              "unit": "GB/s", "frac": alt_ach / peak, "traffic": None,
                              "plan_options": alt_opts, "launches_per_step": alt.stats["n_passes"],
                              "mean_launch_ms": alt_launch, "gates_per_s": alt_steps * ngates / (alt_ms * 1e-3),
                              "final_norm": state.norm(),
                              "operating_point": f"at most {ALT_MAX_DENSE} matrices per pass: the pass runs near the "
                                                 "HBM roof, the circuit needs more passes"}
        del alt

    # end to end through the public API, host buffers on both sides
    e2e = None
    if not args.no_e2e:
        import psutil
        need = 16 << n
        if psutil.virtual_memory().available > need * 1.5:
            outs = [backend.pinned_empty(1 << n), backend.pinned_empty(1 << n)] \
                if psutil.virtual_memory().available > need * 2.6 else [backend.pinned_empty(1 << n)]
            init = [State.ZERO] * n
            del state
            torch.cuda.empty_cache()
            sim = Simulator(circuit, plan_options=opts)
            sim.run(init, out=outs[0])                          # warm-up
            # one call after the other, each blocking until its result is in host memory
            e2e_steps = args.steps
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                sim.run(init, out=outs[0])
            torch.cuda.synchronize()
            dt_serial = (time.perf_counter() - t0) / e2e_steps
            # the same calls with block=False: step k+1 computes while the result of step k crosses
            # PCIe (two device states, two pinned buffers); every result is waited for inside the
            # timed region
            dt = dt_serial
            piped_steps = 0
            if len(outs) == 2:
                piped_steps = args.steps
                t0 = time.perf_counter()
                pending = None
                for k in range(piped_steps):
                    nxt = sim.run(init, out=outs[k % 2], block=False)
                    if pending is not None:
                        pending.result()
                    pending = nxt
                pending.result()
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t0) / piped_steps
            out = outs[(piped_steps - 1) % 2] if piped_steps else outs[0]     # the result of the last step
            assert abs(np.vdot(out[:1 << 20], out[:1 << 20]).real) >= 0.0
            if args.dump_outputs:
                np.save(os.path.join(args.dump_outputs, "e2e_sample.npy"), as_re_im(out[dump_sample_index(n)]))
            h2d = passes * PASS_PARAM_BYTES + 64 * n            # kernel-parameter blocks + product-state amplitudes
            e2e = {"value": ngates / dt, "unit": "gates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": need,
                   "seconds_per_step": dt, "steps": piped_steps or e2e_steps,
                   "blocking_calls": {"value": ngates / dt_serial, "seconds_per_step": dt_serial, "steps": e2e_steps},
                   "note": "Simulator(circuit).run([ZERO]*n, out=pinned, block=False), result() of step k taken "
                           "after step k+1 is queued: lowering, plan lookup (the plan compiled by the warm-up run is "
                           "reused through the simulator's content-keyed cache; compiling takes config.plan_seconds), "
                           "product state, all passes, 2^n x 16 B device-to-host copy of EVERY step inside the timed "
                           "region, the copy of step k overlapping the passes of step k+1 (the copy of the last step is "
                           "exposed: 0.34 s over `steps` steps); blocking_calls is the same loop with block=True "
                           "(no overlap)"}
            del out, outs, sim
        else:
            e2e = {"value": None, "unit": "gates/s", "skipped": "host memory too small for the 2^n output buffer"}
    torch.cuda.empty_cache()

    secondary = []
    if not args.no_secondary:
        for fn in (secondary_grover, lambda: secondary_rb(args.rb_sequences, args.cpu_seconds), secondary_dm):
            try:
                secondary.append(fn())
            except Exception as exc:                             # a secondary line must not sink the headline
                secondary.append({"error": repr(exc)})

    base = None
    if not args.no_cpu_baseline:
        base = cpu_baseline(args.cpu_seconds, args.seed)

    line = {"metric": METRIC, "value": value, "unit": "gates/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "c128", "data": "synthetic",
            "config": {"workload": f"C4: {n}-qubit complex128 random circuit, depth {args.depth}, "
                                   f"{ngates} gates (sv_random_circuit seed {args.seed}); state 2^{n} x 16 B "
                                   "exceeds L2, no flush needed",
                       "plan": stats, "plan_options": opts, "plan_seconds": plan_seconds,
                       "gates_per_pass": ngates / max(1, passes), "final_norm": norm},
            "roofline": roofline, "roofline_hbm_point": roofline_hbm_point, "cpu_baseline": base, "e2e": e2e,
            "secondary": secondary, "gpu_launches": int(launches), "clocks": clocks.summary()}
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    main()
