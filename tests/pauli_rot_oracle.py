"""Test helper: the host oracle for Pauli rotations (qb_apply_pauli_rot), by bit operations.

Written with the same bit operations as tests/pauli_oracle.py (the expectation-value oracle) and pinned to
scipy.linalg.expm of the dense string for every string at n <= 4 in tests/test_pauli_rot_cpu.py."""
import numpy as np


def pauli_rot(n: int, x: int, z: int, theta: float, v: np.ndarray) -> np.ndarray:
    """``exp(-i theta/2 p) #> v`` = cos(theta/2) v - i sin(theta/2) (p #> v) for the Pauli string p with X on
    the qubits of ``x`` only, Z on ``z`` only, Y on both (bit q = qubit q, QGate.hs:90-108): pauliY =
    i pauliX pauliZ, so (p #> v)_j = i^popc(x & z) (-1)^popc((j ^ x') & z') v_(j ^ x'), with x', z' the masks
    on index bits (qubit q = bit n-1-q, StateVec.hs:65-67)."""
    xb = sum(1 << (n - 1 - q) for q in range(n) if (x >> q) & 1)
    zb = sum(1 << (n - 1 - q) for q in range(n) if (z >> q) & 1)
    idx = np.arange(1 << n, dtype=np.uint64) ^ np.uint64(xb)
    sign = 1 - 2 * (np.bitwise_count(idx & np.uint64(zb)).astype(np.int64) & 1)
    pv = (1j ** bin(x & z).count("1")) * sign * v[idx]
    return np.cos(theta / 2) * v - 1j * np.sin(theta / 2) * pv
