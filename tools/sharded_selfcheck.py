#!/usr/bin/env python
"""Full-size parity property for the sharded path (torchrun, one rank per GPU, exchanges over
CUDA-IPC mapped peer shards): a random circuit followed by its gate-by-gate inverse must bring
|0...0> back.  No oracle can hold 2^34 amplitudes; this checks the whole chain -- stage
scheduler, rank relabelling, leftovers across exchanges, the exchange kernel, tile passes -- on
the real interconnect.  Prints one JSON line on rank 0.

    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/sharded_selfcheck.py --qubits 34 --depth 60
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from quantum_computations_b200 import engine, sharded, workloads  # noqa: E402
from quantum_computations_b200.states import State  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=0)
    ap.add_argument("--depth", type=int, default=60)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--feedforward", action="store_true",
                    help="(<= 28 qubits) a circuit with measurements, insertions and classical control through "
                         "run_circuit, against the single-GPU Simulator from the same seed")
    ap.add_argument("--compare-single", action="store_true",
                    help="(<= 28 qubits) run the forward circuit only and compare the gathered state element by "
                         "element with the single-GPU Simulator on rank 0")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    g = world.bit_length() - 1
    n = args.qubits or 30 + g
    backend = engine.get_backend(local)
    comm = sharded.Comm()
    comm.device = torch.device("cuda", local)
    forward = workloads.sv_random_circuit(n, args.depth, args.seed)
    if args.feedforward:
        from quantum_computations_b200 import gates
        from quantum_computations_b200.simulator import ClassicalControl, Simulator
        circ = [gates.H(0), gates.CX(0, 1), gates.H(2), gates.CZ(2, 3), gates.T(3)]
        circ += workloads.sv_random_circuit(n, 6, 5)
        circ += [gates.MZ(0), ClassicalControl(gates.X(0), [0]), gates.Insert(2, State.PLUS), gates.H(3)]
        circ += workloads.sv_random_circuit(n, 6, 6)
        circ += [gates.MX(n - 1), ClassicalControl(gates.Z(1), [], [1]), gates.M(4, 0.3, 1.1)]
        circ += workloads.sv_random_circuit(n - 2, 6, 7)
        circ += [gates.Insert(0, State.T), gates.MZ(1), ClassicalControl(gates.H(0), [-1])]
        kets = [State.PLUS.get(), State.T.get()] + [State.ZERO.get()] * (n - 2)
        state = sharded.ShardedState(n, comm, backend=backend)
        sim = sharded.ShardedSimulator(circ, state)
        np.random.seed(args.seed)
        sim.run_circuit(kets)
        got = state.gather_numpy()
        if rank == 0:
            psi0 = np.ones(1, dtype=np.complex128)
            for k in kets:
                psi0 = np.kron(psi0, np.asarray(k, dtype=np.complex128))
            np.random.seed(args.seed)
            single = Simulator(circ, backend=backend)
            ref = single.run(psi0)
            err = float(np.abs(got - ref).max() / np.abs(ref).max())
            print(json.dumps({"check": "run_circuit (M, Insert, ClassicalControl) sharded vs single-GPU", "qubits": n,
                              "gpus": world, "gates": len(circ), "results": sim.results,
                              "same_outcomes": sim.results == single.results, "max_rel_err": err,
                              "exchanges": state.swaps, "ok": bool(err < 1e-12 and sim.results == single.results)}))
        dist.destroy_process_group()
        return
    if args.compare_single:
        if n > 28:
            raise SystemExit("--compare-single gathers the state on the host: at most 28 qubits")
        kets = [State.PLUS.get(), State.T.get()] + [State.ZERO.get()] * (n - 2)
        state = sharded.ShardedState(n, comm, backend=backend)
        sim = sharded.ShardedSimulator(forward, state)
        sim.prepare(kets)
        sim.run()
        got = state.gather_numpy()
        if rank == 0:
            from quantum_computations_b200.simulator import Simulator
            psi0 = np.ones(1, dtype=np.complex128)
            for k in kets:
                psi0 = np.kron(psi0, np.asarray(k, dtype=np.complex128))
            ref = Simulator(forward, backend=backend).run(psi0)
            err = float(np.abs(got - ref).max() / np.abs(ref).max())
            print(json.dumps({"check": "sharded vs single-GPU, element by element", "qubits": n,
                              "gpus": world, "depth": args.depth, "gates": len(forward), "max_rel_err": err,
                              "plan": sim.stats, "exchanges": state.swaps, "ok": bool(err < 1e-12)}))
        dist.destroy_process_group()
        return
    circuit = forward + workloads.inverse_circuit(forward)
    state = sharded.ShardedState(n, comm, backend=backend)
    sim = sharded.ShardedSimulator(circuit, state)
    sim.compile()
    sim.prepare([State.ZERO.get()] * n)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    sim.run()
    torch.cuda.synchronize()
    dist.barrier()
    seconds = time.perf_counter() - t0
    norm = state.norm()
    # logical index 0: every logical bit 0 -> the rank whose bits equal the flip flags, local index 0
    owner = sum(f << i for i, f in enumerate(state.flip))
    amp0 = np.zeros(2)
    if rank == owner:
        v = state.buf[:1].cpu().numpy()[0]
        amp0[:] = [v.real, v.imag]
    amp0 = comm.allreduce_sum(amp0)
    if rank == 0:
        overlap = float(amp0[0] ** 2 + amp0[1] ** 2)
        print(json.dumps({"check": "circuit . inverse on |0...0>", "qubits": n, "gpus": world, "depth": args.depth,
                          "gates": len(circuit), "seconds": seconds, "norm": norm, "overlap_with_zero_state": overlap,
                          "one_minus_overlap": 1.0 - overlap, "plan": sim.stats, "exchanges": state.swaps,
                          "ok": bool(abs(norm - 1.0) < 1e-9 and abs(overlap - 1.0) < 1e-9)}))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
