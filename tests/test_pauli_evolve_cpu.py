"""Exact time evolution under Pauli sums without a device: the Chebyshev oracle (tests/pauli_evolve_oracle.py)
against scipy.linalg.expm of the dense Hamiltonian and against scipy.sparse.linalg.expm_multiply, its step
rule against a brute-force Bessel tail, argument checks of qb_pauli_evolve, and the register budget of its
kernel."""
import ctypes as C
import itertools
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse
import scipy.sparse.linalg
import scipy.special

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TIMES = [0.01, -0.01, 0.7, -0.7, 5.0, -5.0]


def _dense(n, x, z):
    from oracle import dense as D
    one = {(1, 0): D.pauliX(), (1, 1): D.pauliY(), (0, 1): D.pauliZ()}
    M = D.ident(n)
    for q in range(n):
        k = ((x >> q) & 1, (z >> q) & 1)
        if k != (0, 0):
            M = D.onJust(n, q, one[k]) @ M
    return M


def _hamiltonian(n, xs, zs, hs):
    return sum(h * _dense(n, int(x), int(z)) for x, z, h in zip(xs, zs, hs))


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_oracle_is_the_dense_expm_for_every_string(n):
    from oracle import structured as S
    from pauli_evolve_oracle import evolve
    from qubism_b200.statevec import pauli_masks
    rng = np.random.default_rng(4000 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.3
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    xs, zs = pauli_masks(strings, n)
    for s, x, z in zip(strings, xs, zs):
        h = float(rng.normal())
        P = _dense(n, int(x), int(z))
        for t in TIMES:
            got, _ = evolve(n, [x], [z], [h], t, v)
            want = scipy.linalg.expm(-1j * t * h * P) @ v
            assert np.abs(got - want).max() <= 1e-13 * max(1.0, float(np.abs(v).max())), (s, t)


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_oracle_is_the_dense_expm_for_random_sums(n):
    """Identity strings and duplicates included: they merge exactly as the device merges them."""
    from oracle import structured as S
    from pauli_evolve_oracle import evolve
    rng = np.random.default_rng(4100 + n)
    for trial in range(6):
        k = 3 + 3 * trial
        xs = list(rng.integers(0, 1 << n, size=k)) + [0, 0]
        zs = list(rng.integers(0, 1 << n, size=k)) + [0, 0]
        xs += [xs[0], xs[1]]  # duplicates
        zs += [zs[0], zs[1]]
        hs = rng.normal(size=len(xs))
        Hd = _hamiltonian(n, xs, zs, hs)
        v = S.gen_state(n, rng, normalized=False)
        for t in TIMES:
            got, K = evolve(n, xs, zs, hs, t, v)
            want = scipy.linalg.expm(-1j * t * Hd) @ v
            assert np.abs(got - want).max() <= 1e-12 * max(1.0, float(np.abs(v).max())), (trial, t, K)


def test_oracle_cancelling_terms_leave_only_the_phase():
    from pauli_evolve_oracle import evolve
    v = np.array([0.6, 0.8j], dtype=complex)
    got, K = evolve(1, [1, 0, 1], [0, 0, 0], [0.5, 0.25, -0.5], 3.0, v)
    assert K == 0 and np.abs(got - np.exp(-0.75j) * v).max() <= 1e-15


def test_oracle_is_expm_multiply_at_large_tau():
    """n = 10, a Heisenberg ring in a random field with tau ~ 800: 900-odd Chebyshev steps."""
    from oracle import structured as S
    from pauli_evolve_oracle import evolve, k_steps
    n = 10
    rng = np.random.default_rng(4200)
    xs, zs, hs = [], [], []
    for q in range(n):
        p = 1 << q | 1 << ((q + 1) % n)
        for x, z in ((p, 0), (p, p), (0, p)):  # XX, YY, ZZ
            xs.append(x)
            zs.append(z)
            hs.append(1.0)
        xs.append(0)
        zs.append(1 << q)
        hs.append(float(rng.uniform(-1, 1)))
    r = sum(abs(h) for h in hs)
    t = 800.0 / r
    v = S.gen_state(n, rng)
    got, K = evolve(n, xs, zs, hs, t, v)
    assert K == k_steps(t * r) and 850 < K < 1000
    from pauli_grad_oracle import pauli_apply
    cols = np.eye(1 << n, dtype=complex)
    Hd = np.zeros((1 << n, 1 << n), dtype=complex)
    for x, z, h in zip(xs, zs, hs):
        Hd += h * np.stack([pauli_apply(n, x, z, cols[:, j]) for j in range(1 << n)], axis=1)
    want = scipy.sparse.linalg.expm_multiply(-1j * t * scipy.sparse.csr_matrix(Hd), v)
    assert np.abs(got - want).max() <= 1e-10, np.abs(got - want).max()
    assert abs(np.linalg.norm(got) - 1.0) <= 1e-11


def test_step_rule_against_a_brute_force_bessel_tail():
    """K for the taus of the design notes, and the rule itself: the bound holds after K steps, not after K - 1."""
    from pauli_evolve_oracle import EPS, k_steps
    table = {0.05: 7, 1.0: 14, 10.0: 35, 30.0: 65, 87.0: 136, 300.0: 374, 870.0: 975}
    for tau, K in table.items():
        assert k_steps(tau) == K and k_steps(-tau) == K, tau
    for tau in [1e-12, 1e-6, 0.3, 2.5, 17.0, 123.4, 640.0]:
        K = k_steps(tau)
        J = np.abs(scipy.special.jv(np.arange(K + 400), tau))
        tail = lambda k: 2.0 * sum(J[k + 1:][::-1])  # noqa: E731
        assert tail(K) <= EPS, tau
        assert K == 1 or tail(K - 1) > EPS, tau


def test_argument_errors_need_no_device():
    from qubism_b200 import capi
    L = capi.lib()
    x = (C.c_uint64 * 1)(1)
    z = (C.c_uint64 * 1)(0)
    h = (C.c_double * 1)(0.5)
    k = C.c_int64(7)
    assert L.qb_pauli_evolve(None, x, z, h, 1, 0.5, C.byref(k)) == capi.QB_ERR_ARG
    assert k.value == 0
    assert L.qb_pauli_evolve(None, x, z, h, -1, 0.5, None) == capi.QB_ERR_ARG
    assert L.qb_pauli_evolve(None, None, None, None, 0, 0.0, None) == capi.QB_ERR_ARG


def test_chebyshev_kernel_does_not_spill():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "qubism_b200", "csrc", "qb_kernels.cu")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    blocks = re.split(r"ptxas info\s*: Compiling entry function ", r.stderr)
    seen = False
    for b in blocks:
        if "k_pauli_cheb_tile" not in b.split("\n", 1)[0]:
            continue
        seen = True
        assert "0 bytes spill stores, 0 bytes spill loads" in b, b
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        assert regs * 256 * 3 <= 65536, f"{regs} registers do not fit three CTAs of 256 threads per SM"
    assert seen
