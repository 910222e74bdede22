"""B200-native gate-application engine with the API of the reference's
``simulators.dv_simulator`` (frederik-kofoed-marqversen/quantum_computations).

Sub-modules mirror the reference package one to one:

    numpy_quantum   constants and small-matrix helpers      (DV/numpy_quantum.py)
    states          ``State`` enum                            (DV/states.py)
    gates           gate classes, ``M``, ``Insert``          (DV/gates.py)
    simulator       ``Simulator``, ``ClassicalControl``      (DV/simulator.py)

plus what the hot path needs on a GPU:

    engine          ctypes binding of csrc/libqsim_b200.so, ``DeviceState``
    channels        ``Channel`` (Kraus) and the GKP finite-squeezing noise model
    batched         ``BatchedSimulator`` for many small independent circuits
    sharded         state sharded over ranks with global-qubit swaps
    observables     Pauli-sum expectation values (``PauliSum``, ``expect``) on the GPU
    trajectories    Pauli-trajectory sampling of noisy circuits on kets
    layering        measurement-based layer scheduling           (GKP/circuit.py)
    cliffords       two-qubit Clifford table and Clifford RB    (PAPER/average_clifford_fidelity.py)
    tomography      process tomography, Kraus fit of a circuit   (PAPER/tomography.py)
    compat          ``install()`` exposes the package as ``simulators.dv_simulator``

Importing the package is cheap and needs neither torch nor a GPU; the CUDA
library is bound on first use and there is no CPU fallback.
"""
from . import numpy_quantum, states, gates, simulator  # noqa: F401
from .states import State  # noqa: F401
from .simulator import Simulator, ClassicalControl  # noqa: F401

__all__ = ["numpy_quantum", "states", "gates", "simulator", "State", "Simulator", "ClassicalControl"]
__version__ = "0.1.0"
