"""Test helper: the host oracle for Pauli sums (qb_pauli_sum) and adjoint gradients (qb_pauli_rot_grad).

Written with the bit operations of tests/pauli_oracle.py and tests/pauli_rot_oracle.py, and pinned in
tests/test_pauli_grad_cpu.py at n <= 4 to the dense string (every string) and to the parameter-shift rule
over scipy.linalg.expm of the dense strings."""
import numpy as np

from pauli_rot_oracle import pauli_rot


def pauli_apply(n: int, x: int, z: int, v: np.ndarray) -> np.ndarray:
    """``p #> v`` for the Pauli string p with X on the qubits of ``x`` only, Z on ``z`` only, Y on both (bit q =
    qubit q, QGate.hs:90-108): (p #> v)_j = i^popc(x & z) (-1)^popc((j ^ x') & z') v_(j ^ x'), with x', z' the
    masks on index bits (qubit q = bit n-1-q, StateVec.hs:65-67)."""
    xb = sum(1 << (n - 1 - q) for q in range(n) if (x >> q) & 1)
    zb = sum(1 << (n - 1 - q) for q in range(n) if (z >> q) & 1)
    idx = np.arange(1 << n, dtype=np.uint64) ^ np.uint64(xb)
    sign = 1 - 2 * (np.bitwise_count(idx & np.uint64(zb)).astype(np.int64) & 1)
    return (1j ** bin(x & z).count("1")) * sign * v[idx]


def pauli_sum(n: int, xs, zs, coefs, v: np.ndarray) -> np.ndarray:
    """``sum_t coefs[t] (p_t #> v)``."""
    out = np.zeros_like(v, dtype=np.complex128)
    for x, z, c in zip(xs, zs, coefs):
        out += c * pauli_apply(n, int(x), int(z), v)
    return out


def energy(n: int, hx, hz, hc, v: np.ndarray) -> float:
    """``sum_t hc[t] realPart (v <.> (h_t #> v))``, not normalised."""
    return float(np.vdot(v, pauli_sum(n, hx, hz, hc, v)).real)


def rotate(n: int, rx, rz, thetas, v: np.ndarray) -> np.ndarray:
    """``R_{K-1} ... R_0 v`` with R_k = exp(-i thetas[k]/2 p_k)."""
    for x, z, th in zip(rx, rz, thetas):
        v = pauli_rot(n, int(x), int(z), float(th), v)
    return v


def rot_grad(n: int, rx, rz, thetas, hx, hz, hc, v: np.ndarray):
    """``(E, grad)`` of E(theta) = energy(rotate(theta) v) by the adjoint method: lam = H psi_K, then for
    k = K-1 .. 0: grad[k] = Im <lam|p_k|psi>, psi <- R_k^dagger psi, lam <- R_k^dagger lam."""
    psi = rotate(n, rx, rz, thetas, v)
    lam = pauli_sum(n, hx, hz, hc, psi)
    e = float(np.vdot(psi, lam).real)
    grad = np.zeros(len(thetas))
    for k in range(len(thetas) - 1, -1, -1):
        x, z, th = int(rx[k]), int(rz[k]), float(thetas[k])
        if x | z:
            grad[k] = float(np.vdot(lam, pauli_apply(n, x, z, psi)).imag)
        psi = pauli_rot(n, x, z, -th, psi)
        lam = pauli_rot(n, x, z, -th, lam)
    return e, grad
