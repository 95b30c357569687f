"""Lanczos ground states of Pauli sums without a device: the Lanczos oracle (tests/pauli_ground_oracle.py) against
numpy.linalg.eigh of the dense Hamiltonian and against the exact ground energy of open transverse-field Ising
chains, its sector minimum from a start state inside a parity sector, argument checks of qb_pauli_ground, and the
register budget of its kernels."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dense_h(n, xs, zs, hs):
    from pauli_grad_oracle import pauli_apply
    cols = np.eye(1 << n, dtype=complex)
    Hd = np.zeros((1 << n, 1 << n), dtype=complex)
    for x, z, h in zip(xs, zs, hs):
        Hd += h * np.stack([pauli_apply(n, int(x), int(z), cols[:, j]) for j in range(1 << n)], axis=1)
    return Hd


def tfim(n, J, g):
    """Open chain H = -sum J_i Z_i Z_{i+1} - sum g_i X_i as masks (bit q = qubit q) and its exact ground energy:
    minus the sum of the singular values of the bidiagonal matrix with diagonal g and superdiagonal J."""
    xs = [0] * (n - 1) + [1 << q for q in range(n)]
    zs = [(1 << q) | (1 << (q + 1)) for q in range(n - 1)] + [0] * n
    hs = list(-np.asarray(J)) + list(-np.asarray(g))
    M = np.diag(g) + np.diag(J, 1)
    return xs, zs, hs, -float(np.linalg.svd(M, compute_uv=False).sum())


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
def test_oracle_is_the_dense_minimum(n):
    """Random sums with identity strings and duplicates; the Ritz vector's true residual is the estimate."""
    from oracle import structured as S
    from pauli_ground_oracle import ground
    rng = np.random.default_rng(7000 + n)
    for trial in range(3):
        k = 4 + 3 * trial + n
        xs = list(rng.integers(0, 1 << n, size=k)) + [0, 0]
        zs = list(rng.integers(0, 1 << n, size=k)) + [0, 0]
        xs += [xs[0], xs[1]]
        zs += [zs[0], zs[1]]
        hs = rng.normal(size=len(xs))
        Hd = _dense_h(n, xs, zs, hs)
        lam = np.linalg.eigvalsh(Hd)[0]
        r = float(sum(abs(h) for x, z, h in zip(xs, zs, hs) if x or z))  # (an upper bound of the merged r)
        v = S.gen_state(n, rng, normalized=False) * 2.5
        e, res, m, al, be, x = ground(n, xs, zs, hs, v, 1e-10 * r, 4000, vector=True)
        assert abs(e - lam) <= 1e-10 * r, (trial, e, lam, m)
        true = float(np.linalg.norm(Hd @ x - e * x))
        assert abs(np.linalg.norm(x) - 1.0) <= 1e-13
        assert true <= res + 1e-9 * r, (true, res)
        assert np.vdot(v, x).real > 0 and abs(np.vdot(v, x).imag) <= 1e-12 * np.linalg.norm(v)
        if n <= 2:  # the Krylov space is all there is: breakdown, m <= 2^n
            assert m <= 1 << n and be[-1] <= 2.0 ** -40 * r


@pytest.mark.parametrize("n", [12, 13, 14])
def test_oracle_is_the_free_fermion_energy(n):
    from pauli_ground_oracle import ground
    rng = np.random.default_rng(7100 + n)
    J, g = rng.uniform(0.5, 1.5, n - 1), rng.uniform(0.5, 1.5, n)
    xs, zs, hs, exact = tfim(n, J, g)
    r = float(np.abs(hs).sum())
    v = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    e, res, m, al, be, _ = ground(n, xs, zs, hs, v, 1e-10 * r, 2000)
    assert res <= 1e-10 * r and 20 < m < 200, (res, m)
    assert abs(e - exact) <= 1e-12 * r, (e, exact)


@pytest.mark.parametrize("n", [4, 6, 8])
def test_oracle_finds_the_sector_minimum(n):
    """The parity P = prod X_i commutes with the Ising chain: from a start state with P = -1 the answer is the odd
    sector's minimum, above the (even) ground energy."""
    from oracle import structured as S
    from pauli_grad_oracle import pauli_apply
    from pauli_ground_oracle import ground
    rng = np.random.default_rng(7200 + n)
    J, g = rng.uniform(0.5, 1.5, n - 1), rng.uniform(0.5, 1.5, n)
    xs, zs, hs, exact = tfim(n, J, g)
    r = float(np.abs(hs).sum())
    Hd = _dense_h(n, xs, zs, hs)
    P = np.stack([pauli_apply(n, (1 << n) - 1, 0, c) for c in np.eye(1 << n, dtype=complex)], axis=1)
    for sign in (1, -1):
        proj = 0.5 * (np.eye(1 << n) + sign * P)
        ev, U = np.linalg.eigh(proj)
        B = U[:, ev > 0.5]  # an orthonormal basis of the sector
        want = np.linalg.eigvalsh(B.conj().T @ Hd @ B)[0]
        v = proj @ S.gen_state(n, rng)
        e, res, m, al, be, x = ground(n, xs, zs, hs, v, 1e-10 * r, 4000, vector=True)
        assert abs(e - want) <= 1e-10 * r, (sign, e, want)
        assert np.abs(P @ x - sign * x).max() <= 1e-10
        if sign == 1:
            assert abs(e - exact) <= 1e-10 * r
        else:
            assert e > exact + 1e-3


def test_argument_errors_need_no_device():
    from qubism_b200 import capi
    L = capi.lib()
    x = (C.c_uint64 * 1)(1)
    z = (C.c_uint64 * 1)(0)
    h = (C.c_double * 1)(0.5)
    e, res, m = C.c_double(), C.c_double(), C.c_int64()
    assert L.qb_pauli_ground(None, x, z, h, 1, 1e-8, 10, 0, C.byref(e), C.byref(res), C.byref(m), None, None) == capi.QB_ERR_ARG
    assert L.qb_pauli_ground(None, x, z, h, -1, 1e-8, 10, 0, C.byref(e), C.byref(res), C.byref(m), None, None) == capi.QB_ERR_ARG
    assert L.qb_pauli_ground(None, None, None, None, 0, 0.0, 1, 1, None, None, None, None, None) == capi.QB_ERR_ARG


def test_lanczos_kernels_do_not_spill():
    """Both instantiations of the Chebyshev tile kernel (evolve, Lanczos) fit three 256-thread CTAs per SM, and the
    update sweep spills nothing."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "qubism_b200", "csrc", "qb_kernels.cu")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    blocks = re.split(r"ptxas info\s*: Compiling entry function ", r.stderr)
    seen = {"cheb_false": 0, "cheb_true": 0, "update": 0}
    for b in blocks:
        head = b.split("\n", 1)[0]
        if "k_pauli_cheb_tile" in head:
            key = "cheb_true" if "Lb1E" in head else "cheb_false"
        elif "k_lanczos_update" in head:
            key = "update"
        else:
            continue
        seen[key] += 1
        assert "0 bytes spill stores, 0 bytes spill loads" in b, b
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        if key != "update":
            assert regs * 256 * 3 <= 65536, f"{regs} registers do not fit three CTAs of 256 threads per SM"
    assert all(seen.values()), seen
