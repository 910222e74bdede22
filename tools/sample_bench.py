"""Measurement statistics at 30 qubits on one GPU (qsim_marginal_probs, qsim_sample).

The state is the one a ``workloads.sv_random_circuit(n, 2, seed)`` run leaves behind.  Every
call is timed whole with CUDA events (warm-up, then --reps calls) on preallocated device
buffers, and one JSON line is printed per measurement:

* marginals for k = 1, 4, 10, 20 on the top qubits, the bottom qubits and a scattered set,
  plus k = n: read bytes (16 B x 2^n) + written bytes (8 B x 2^k) over the time, and that rate
  as a fraction of a device-to-device copy measured in the same process (read + write bytes);
* sampling 10^3, 10^6 and 10^7 shots (device uniforms), and 10^7 shots on a basis state: time
  against the time of one read of the state (the k = 0 marginal) and against 16 B x 2^n at the
  copy rate;
* the routes that exist without the feature, timed once: the pinned download of the state plus a
  host cumsum / searchsorted for 10^6 shots, and k separate qsim_measure_probs calls against one
  k-qubit marginal.

The GPU name, power limit and max SM clock are read in the same run.

    python tools/sample_bench.py [--qubits 30] [--reps 10] [--out FILE.jsonl]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from expect_bench import gpu_info, time_events  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--seed", type=int, default=20251020)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench needs a CUDA device")
    from quantum_computations_b200 import _capi, build_native, engine, workloads
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

    src = torch.empty(1 << 28, dtype=torch.complex128, device=be.device)
    dst = torch.empty_like(src)
    copy_ms = time_events(lambda: dst.copy_(src), 20)
    copy_gbs = 2 * src.numel() * 16 / copy_ms / 1e6
    del src, dst
    torch.cuda.empty_cache()
    emit({"metric": "d2d_copy", "bytes": 2 * (1 << 28) * 16, "ms": copy_ms, "gbs": copy_gbs})

    state = engine.DeviceState.product([State.ZERO.get()] * n, be)
    ops = [op for g in workloads.sv_random_circuit(n, 2, args.seed) for op in g.lowered(n, False)]
    engine.Plan(be, n, ops).execute(state.buf)
    torch.cuda.synchronize()
    state_bytes = 16 * (1 << n)
    out = torch.empty(1 << n, dtype=torch.float64, device=be.device)

    def marginal(buf, qubits):
        q = np.ascontiguousarray(qubits, dtype=np.int32)
        _capi.check(lib, lib.qsim_marginal_probs(buf.data_ptr(), n, len(q), q.ctypes.data_as(_capi.c_int_p),
                                                 out.data_ptr(), be.stream()))

    rng = np.random.default_rng(args.seed)
    read_ms = time_events(lambda: marginal(state.buf, []), args.reps)
    emit({"metric": "marginal", "layout": "norm", "k": 0, "qubits": n, "ms": read_ms,
          "gbs": state_bytes / read_ms / 1e6, "fraction_of_copy_peak": state_bytes / read_ms / 1e6 / copy_gbs})
    for k in (1, 4, 10, 20, n):
        layouts = {"top": list(range(k)), "bottom": list(range(n - k, n)),
                   "scattered": sorted(int(v) for v in rng.permutation(n)[:k])} if k < n else {"all": list(range(n))}
        for name, qs in layouts.items():
            if name == "scattered":
                rng.shuffle(qs)
            ms = time_events(lambda: marginal(state.buf, qs), args.reps)
            first = out[:1 << k].clone()
            marginal(state.buf, qs)
            moved = state_bytes + 8 * (1 << k)
            gbs = moved / ms / 1e6
            emit({"metric": "marginal", "layout": name, "k": k, "qubits": n, "ms": ms, "bytes": moved, "gbs": gbs,
                  "fraction_of_copy_peak": gbs / copy_gbs,
                  "repeat_bit_identical": bool(torch.equal(first, out[:1 << k])), "reps": args.reps})

    def sampler(buf, shots):
        need = C.c_uint64()
        _capi.check(lib, lib.qsim_sample_workspace_bytes(n, shots, C.byref(need)))
        ws = torch.empty(int(need.value), dtype=torch.uint8, device=be.device)
        u = torch.from_numpy(np.random.default_rng(shots).random(shots)).to(be.device)
        res = torch.empty(shots, dtype=torch.int64, device=be.device)
        total = C.c_double()

        def call():
            _capi.check(lib, lib.qsim_sample(buf.data_ptr(), n, shots, u.data_ptr(), res.data_ptr(), C.byref(total),
                                             ws.data_ptr(), need.value, be.stream()))
        return call, res, int(need.value)

    del out
    torch.cuda.empty_cache()
    for label, shots in (("random", 10 ** 3), ("random", 10 ** 6), ("random", 10 ** 7)):
        call, res, ws_bytes = sampler(state.buf, shots)
        ms = time_events(call, args.reps)
        first = res.clone()
        call()
        emit({"metric": "sample", "state": label, "qubits": n, "shots": shots, "ms": ms,
              "x_one_read": ms / read_ms, "x_one_read_at_copy_rate": ms / (state_bytes / copy_gbs / 1e6),
              "workspace_bytes": ws_bytes, "repeat_identical": bool(torch.equal(first, res)), "reps": args.reps})
        del call, res, first
        torch.cuda.empty_cache()

    # routes without the feature, timed once
    shots = 10 ** 6
    host = torch.empty(1 << n, dtype=torch.complex128, pin_memory=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host.copy_(state.buf)
    t1 = time.perf_counter()
    p = np.abs(host.numpy())
    p *= p
    np.cumsum(p, out=p)
    u = np.random.default_rng(shots).random(shots)
    idx = np.searchsorted(p, u * p[-1], side="right")
    t2 = time.perf_counter()
    emit({"metric": "host_route", "qubits": n, "shots": shots, "download_s": t1 - t0, "host_cumsum_search_s": t2 - t1,
          "total_s": t2 - t0, "first_outcome": int(idx[0])})
    del host, p, idx
    k = 10
    bra0, bra1 = np.array([1, 0, 0, 0], dtype=np.float64), np.array([0, 0, 1, 0], dtype=np.float64)
    probs = np.zeros(2)

    def per_qubit():
        for q in range(k):
            _capi.check(lib, lib.qsim_measure_probs(state.buf.data_ptr(), n, q, bra0.ctypes.data_as(_capi.c_double_p),
                                                    bra1.ctypes.data_as(_capi.c_double_p),
                                                    probs.ctypes.data_as(_capi.c_double_p), be.stream()))
    out = torch.empty(1 << k, dtype=torch.float64, device=be.device)
    ms_sep = time_events(per_qubit, 3, warmup=1)
    ms_one = time_events(lambda: marginal(state.buf, list(range(k))), 3, warmup=1)
    emit({"metric": "measure_probs_route", "qubits": n, "k": k, "separate_calls_ms": ms_sep, "one_marginal_ms": ms_one,
          "note": "the separate calls give only the k one-qubit marginals, not the joint distribution"})

    # a basis state: every shot lands in one chunk
    del state, out
    torch.cuda.empty_cache()
    basis = torch.zeros(1 << n, dtype=torch.complex128, device=be.device)
    where = (1 << n) // 3
    basis[where] = 1.0
    call, res, ws_bytes = sampler(basis, 10 ** 7)
    ms = time_events(call, args.reps)
    emit({"metric": "sample", "state": "basis", "qubits": n, "shots": 10 ** 7, "ms": ms, "x_one_read": ms / read_ms,
          "x_one_read_at_copy_rate": ms / (state_bytes / copy_gbs / 1e6), "workspace_bytes": ws_bytes,
          "all_at_index": bool((res == where).all().item()), "reps": args.reps})

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
