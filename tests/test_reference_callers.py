"""REFERENCE callers on top of this package (drop-in claim, SURVEY.md section 8b).

``compat.install()`` registers this package as ``simulators.dv_simulator``, the import path the
reference's scripts use.  The scripts themselves are not part of this repository, so what they
built and computed is replayed from the vectors recorded from them by tests/golden/make_golden.py:
the circuits of ``randomised_benchmarking.random_circ`` with the depth its ``MBGKPCircuit``
reported (rb.npz), and the circuits of ``dv_circuits.grover`` with their output kets
(grover.npz).  Rebuilt from the classes found under the reference's import path, they must be
this package's classes, draw the same gates as ``workloads.rb_random_circuit`` and reproduce the
recorded results."""
import pickle

import numpy as np

import parity_cases as pc
from golden.specs import as_oracle_ops, from_spec
from oracle import strided
from quantum_computations_b200 import compat, gates, layering, simulator, workloads


def test_recorded_reference_callers_run_on_this_package(emu_backend):
    compat.install()
    from simulators.dv_simulator import gates as dv_gates
    from simulators.dv_simulator import simulator as dv_simulator
    from simulators.dv_simulator import states as dv_states
    assert dv_gates is gates and dv_simulator.Simulator is simulator.Simulator

    # 1. the reference's RB generator: the same draws as workloads.rb_random_circuit, and the
    #    measurement-based depth its MBGKPCircuit reported is the layer depth of this package
    meta, z = pc.load("rb.npz")
    rng = np.random.default_rng(meta["seed"])
    for i, rec in enumerate(meta["samples"]):
        dv_circ = [from_spec(s, dv_gates, dv_simulator, z, states=dv_states) for s in rec["circuit"]]
        assert all(type(g).__module__ == gates.__name__ for g in dv_circ)
        mine = workloads.rb_random_circuit(2, rec["depth"], rng)
        assert [(type(g).__name__, list(g.indices)) for g in dv_circ] == \
               [(type(g).__name__, list(g.indices)) for g in mine], i
        assert layering.MBLayering.of(dv_circ, 2).depth() == rec["mb_depth"] == rec["depth"], i

    # 2. the reference's Grover circuit, simulated by this package (host emulator backend) ==
    #    the reference's own output == CPU oracle
    meta, z = pc.load("grover.npz")
    full = [rec for rec in meta if rec["kind"] == "full"]
    assert len(full) >= 2
    for rec in full:
        gcirc = [from_spec(s, dv_gates, dv_simulator, z, states=dv_states) for s in rec["circuit"]]
        assert all(type(g).__module__ in (gates.__name__, simulator.__name__) for g in gcirc)
        out = dv_simulator.Simulator(gcirc, backend=emu_backend).run(None)
        assert pc.rel_err(out, z[rec["out"]]) < pc.RTOL
        ref, _ = strided.run(as_oracle_ops(gcirc), np.ones(1, dtype=np.complex128))
        assert np.abs(out - ref).max() < 1e-12
        probs = np.abs(out) ** 2
        assert all(abs(probs[t] - 0.5) < 1e-12 for t in rec["tagged"])

    # 3. gate objects survive pickling (the reference farms samples out with multiprocessing)
    g2 = pickle.loads(pickle.dumps([gates.H(0), gates.RZ(1, 0.3), gates.CZ(0, 1)]))
    assert [type(g).__name__ for g in g2] == ["H", "RZ", "CZ"] and np.allclose(g2[1].matrix, gates.RZ(1, 0.3).matrix)
