"""Test helper: the host oracle for Lanczos ground states of Pauli sums (qb_pauli_ground).

The same recurrence, stopping rule and two-pass Ritz vector the device runs, written with the Pauli sum of
tests/pauli_grad_oracle.py and the string merge of tests/pauli_evolve_oracle.py, and pinned in
tests/test_pauli_ground_cpu.py to numpy.linalg.eigh of the dense Hamiltonian and to the exact ground energy of
open transverse-field Ising chains.  Plain Lanczos in Paige's A(2,7) form on H' = H - c (c the identity strings'
coefficient sum), from v_0 = v / ||v||:

    w = H' v_k - beta_k v_{k-1},  alpha_k = Re <v_k|w>,  w -= alpha_k v_k,  beta_{k+1} = ||w||,  v_{k+1} = w / beta_{k+1}

stopping after the step with beta_m |y_m| <= tol, beta_m <= 2^-40 r (r = sum |h| over the merged non-identity
strings) or m = maxiter, theta and y the lowest eigenpair of the tridiagonal T_m (y_0 >= 0)."""
import numpy as np
import scipy.linalg

from pauli_evolve_oracle import merge
from pauli_grad_oracle import pauli_sum

BREAKDOWN = 2.0 ** -40


def lowest(al, be):
    """``(theta, y)``: the lowest eigenvalue of the tridiagonal with diagonal al and off-diagonal be (len(al) - 1)
    and its unit eigenvector with y[0] >= 0."""
    if len(al) == 1:
        return float(al[0]), np.ones(1)
    w, Y = scipy.linalg.eigh_tridiagonal(np.asarray(al, float), np.asarray(be, float), select="i",
                                         select_range=(0, 0))
    y = Y[:, 0]
    return float(w[0]), (-y if y[0] < 0 else y)


def ground(n: int, xs, zs, coefs, v: np.ndarray, tol: float, maxiter: int, vector: bool = False):
    """``(energy, resid, m, alpha, beta, x)``: alpha (of H, c included) and beta of the m steps taken, x the
    normalised Ritz vector (vector=True; otherwise None)."""
    v = np.asarray(v, dtype=np.complex128)
    nrm = float(np.linalg.norm(v))
    if not (np.isfinite(nrm) and nrm > 0):
        raise ValueError("start vector of zero or non-finite norm")
    c, terms = merge(xs, zs, coefs)
    if not terms:
        return c, 0.0, 0, np.zeros(0), np.zeros(0), (v / nrm if vector else None)
    r = sum(abs(h) for _, _, h in terms)
    tx = [x for x, _, _ in terms]
    tz = [z for _, z, _ in terms]
    th = [h for _, _, h in terms]
    v0 = v / nrm
    al, be = [], []
    vp, vk = None, v0
    for k in range(maxiter):
        w = pauli_sum(n, tx, tz, th, vk)
        if k:
            w = w - be[-1] * vp
        a = float(np.vdot(vk, w).real)
        w = w - a * vk
        b = float(np.linalg.norm(w))
        al.append(a)
        be.append(b)
        theta, y = lowest(al, be[:-1])
        resid = b * abs(y[-1])
        if resid <= tol or b <= BREAKDOWN * r:
            break
        vp, vk = vk, w / b
    m = len(al)
    x = None
    if vector:
        x = y[0] * v0
        vp, vk = None, v0
        for k in range(m - 1):
            w = pauli_sum(n, tx, tz, th, vk)
            if k:
                w = w - be[k - 1] * vp
            w = w - al[k] * vk
            vp, vk = vk, w / be[k]
            x = x + y[k + 1] * vk
        x = x / np.linalg.norm(x)
    return theta + c, resid, m, np.asarray(al) + c, np.asarray(be), x
