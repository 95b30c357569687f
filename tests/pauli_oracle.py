"""Test helper: the host oracle for Pauli expectation values (qb_expect_pauli), by bit operations.

It is pinned to the reference's literal form -- realPart (v <.> (p #> v)) with p multiplied out of
onJust q pauliX / pauliY / pauliZ as dense matrices (oracle.dense) -- for every string at n <= 5 in
tests/test_expect_cpu.py, which fixes the Y phase and the qubit <-> index-bit order of QGate.hs."""
import numpy as np


def expect_pauli(n: int, x: int, z: int, v: np.ndarray) -> float:
    """``realPart (v <.> (p #> v))`` for the Pauli string p with X on the qubits of ``x`` only, Z on ``z``
    only, Y on both (bit q = qubit q, QGate.hs:90-108): pauliY = i pauliX pauliZ, so
    (p #> v)_j = i^popc(x & z) (-1)^popc((j ^ x') & z') v_(j ^ x'), with x', z' the masks on index bits
    (qubit q = bit n-1-q, StateVec.hs:65-67).  Not normalised."""
    xb = sum(1 << (n - 1 - q) for q in range(n) if (x >> q) & 1)
    zb = sum(1 << (n - 1 - q) for q in range(n) if (z >> q) & 1)
    idx = np.arange(1 << n, dtype=np.uint64) ^ np.uint64(xb)
    sign = 1 - 2 * (np.bitwise_count(idx & np.uint64(zb)).astype(np.int64) & 1)
    pv = (1j ** bin(x & z).count("1")) * sign * v[idx]
    return float(np.vdot(v, pv).real)
