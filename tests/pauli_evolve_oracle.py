"""Test helper: the host oracle for exact time evolution under Pauli sums (qb_pauli_evolve).

The same Chebyshev expansion the device runs, written with the Pauli sum of tests/pauli_grad_oracle.py and the
Bessel functions of scipy.special.jv, and pinned in tests/test_pauli_evolve_cpu.py to scipy.linalg.expm of the
dense Hamiltonian at n <= 4 and to scipy.sparse.linalg.expm_multiply at n = 10:

    exp(-itH) v = e^{-itc} sum_{k=0..K} a_k T_k(H') v,  H' = (H - c) / r,  a_0 = J_0(tau), a_k = 2 (-i)^k J_k(tau)

with c the identity strings' coefficient sum, r = sum |h| over the merged non-identity strings and tau = t r."""
import numpy as np
import scipy.special

from pauli_grad_oracle import pauli_sum

EPS = 2.0 ** -53


def k_steps(tau: float) -> int:
    """The smallest k >= 1 with 2 sum_{j > k} |J_j(tau)| <= 2^-53 (the truncation bound, ||T_k(H')|| <= 1)."""
    at = abs(float(tau))
    top = int(np.ceil(at + 20.0 * np.cbrt(at))) + 60
    tail = np.abs(scipy.special.jv(np.arange(top + 1), at))[::-1].cumsum()[::-1]  # tail[k] = sum_{j >= k}
    ok = 2.0 * tail[2:] <= EPS  # ok[k - 1]: the bound after k steps
    return int(np.argmax(ok)) + 1


def merge(xs, zs, coefs):
    """(c, [(x, z, h)]): the identity strings' sum and the other strings with equal ones added (first
    appearance order), zero sums dropped."""
    c = 0.0
    acc = {}
    for x, z, h in zip(xs, zs, coefs):
        x, z = int(x), int(z)
        if x == 0 and z == 0:
            c += float(h)
        else:
            acc[(x, z)] = acc.get((x, z), 0.0) + float(h)
    return c, [(x, z, h) for (x, z), h in acc.items() if h != 0.0]


def evolve(n: int, xs, zs, coefs, t: float, v: np.ndarray):
    """``(exp(-i t H) v, K)`` with H = sum_t coefs[t] P_t (real coefficients)."""
    v = np.asarray(v, dtype=np.complex128)
    c, terms = merge(xs, zs, coefs)
    phase = np.exp(-1j * t * c)
    if t == 0 or not terms:
        return phase * v, 0
    r = sum(abs(h) for _, _, h in terms)
    tx = [x for x, _, _ in terms]
    tz = [z for _, z, _ in terms]
    th = [h / r for _, _, h in terms]
    tau = t * r
    K = k_steps(tau)
    J = scipy.special.jv(np.arange(K + 1), tau)
    a = 2.0 * (-1j) ** np.arange(K + 1) * J
    a[0] = J[0]
    prev, cur = v, pauli_sum(n, tx, tz, th, v)
    out = a[0] * prev + a[1] * cur
    for k in range(2, K + 1):
        prev, cur = cur, 2.0 * pauli_sum(n, tx, tz, th, cur) - prev
        out = out + a[k] * cur
    return phase * out, K
