#!/usr/bin/env python
"""Development tool (torchrun, one rank per GPU): time k-qubit exchanges of a sharded ket.

    torchrun --nproc-per-node 2 tools/exchange_bench.py [--shard-qubits 30] [--reps 6]

Prints, on rank 0, ms per exchange and GB/s per direction and GPU for k = 1 .. log2(ranks)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from quantum_computations_b200 import engine, sharded  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shard-qubits", dest="local", type=int, default=30)
    ap.add_argument("--reps", type=int, default=6)
    args = ap.parse_args()
    rank, world, local_rank = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    g = world.bit_length() - 1
    n = args.local + g
    be = engine.get_backend(local_rank)
    comm = sharded.Comm()
    comm.device = torch.device("cuda", local_rank)
    st = sharded.ShardedState(n, comm, backend=be)
    st.set_product([np.array([0.6, 0.8j])] * n)
    out = []
    for k in range(1, g + 1):
        pairs = [(st.n_local + i, st.n_local - 1 - i) for i in range(k)]
        st.exchange(pairs)                      # warm-up (IPC mapping)
        st.collect_swap_time()
        st.swap_seconds, st.swaps, st.amps_sent = 0.0, 0, 0
        for _ in range(args.reps):
            st.exchange(pairs)
        secs = st.collect_swap_time()
        t = torch.tensor([secs], device=comm.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = 1e3 * float(t.item()) / args.reps
        sent = 16.0 * st.amps_sent / args.reps
        out.append({"k": k, "ms": round(ms, 3), "GBps_each_way": round(sent / (ms * 1e-3) / 1e9, 1),
                    "shard_fraction": sent / (16.0 * 2.0 ** st.n_local)})
    norm = st.norm()
    if rank == 0:
        print(json.dumps({"ranks": world, "n_local": st.n_local, "exchanges": out, "norm": norm}))
    st.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
