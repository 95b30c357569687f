"""qubism_b200 -- B200-native state-vector backend behind qubism's Haskell API.

Re-export facade in the spirit of src/Qubism.hs:1-16: the state-vector and gate modules.
Importing this package does not touch the GPU; creating a Context does, and fails loudly
if libqubism_sv.so has not been built or no CUDA device is usable (there is no CPU path).
"""
from . import capi  # noqa: F401
from .qgate import (QGate, apply, cnot, controlled, gate, hadamard, ident, ifBit, kronecker, onEvery, onJust,  # noqa: F401
                    onRange, pauliX, pauliY, pauliZ, unitary, unitary_matrix)
from .statevec import (Context, StateVec, collapse, dimension, expectPauli, measure, measureQubit, mkQubit,  # noqa: F401
                       mkStateVec, normalize, pauliEvolve, pauliRotate, pauliRotGrad, pauliSum, tensor, zero)

__version__ = "0.1.0"
