"""Pauli sums and adjoint gradients without a device: the oracle (tests/pauli_grad_oracle.py) against the dense
strings and against the parameter-shift rule over scipy.linalg.expm, argument checks of qb_pauli_sum and
qb_pauli_rot_grad, and the register budget of their kernels."""
import ctypes as C
import itertools
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dense(n, x, z):
    from oracle import dense as D
    one = {(1, 0): D.pauliX(), (1, 1): D.pauliY(), (0, 1): D.pauliZ()}
    M = D.ident(n)
    for q in range(n):
        k = ((x >> q) & 1, (z >> q) & 1)
        if k != (0, 0):
            M = D.onJust(n, q, one[k]) @ M
    return M


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_oracle_applies_every_string_as_the_dense_matrix(n):
    from oracle import structured as S
    from pauli_grad_oracle import pauli_apply, pauli_sum
    from qubism_b200.statevec import pauli_masks
    rng = np.random.default_rng(170 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.7
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    xs, zs = pauli_masks(strings, n)
    tol = 1e-12 * max(1.0, float(np.abs(v).max()))
    H = np.zeros((1 << n, 1 << n), dtype=np.complex128)
    cs = rng.normal(size=len(strings)) + 1j * rng.normal(size=len(strings))
    for s, x, z, c in zip(strings, xs, zs, cs):
        P = _dense(n, int(x), int(z))
        assert np.abs(pauli_apply(n, int(x), int(z), v) - P @ v).max() <= tol, s
        H += c * P
    assert np.abs(pauli_sum(n, xs, zs, cs, v) - H @ v).max() <= 1e-12 * np.abs(H @ v).max() * len(strings)


def _random_strings(n, k, rng):
    xs = rng.integers(0, 1 << n, size=k)
    zs = rng.integers(0, 1 << n, size=k)
    return xs, zs


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_oracle_gradient_is_the_dense_parameter_shift(n):
    from oracle import structured as S
    from pauli_grad_oracle import rot_grad
    rng = np.random.default_rng(180 + n)
    v = S.gen_state(n, rng, normalized=False)
    for trial in range(4):
        K, M = 3 + 2 * trial, 2 + trial
        rx, rz = _random_strings(n, K, rng)
        rx[0] = rz[0] = 0  # the identity string: gradient 0
        hx, hz = _random_strings(n, M, rng)
        th = rng.uniform(-np.pi, np.pi, size=K)
        hc = rng.normal(size=M)
        Ps = [_dense(n, int(x), int(z)) for x, z in zip(rx, rz)]
        H = sum(c * _dense(n, int(x), int(z)) for x, z, c in zip(hx, hz, hc))

        def E(t):
            psi = v
            for P, a in zip(Ps, t):
                psi = scipy.linalg.expm(-0.5j * a * P) @ psi
            return float(np.vdot(psi, H @ psi).real)

        want = np.array([(E(th + np.pi / 2 * np.eye(K)[k]) - E(th - np.pi / 2 * np.eye(K)[k])) / 2 for k in range(K)])
        e, g = rot_grad(n, rx, rz, th, hx, hz, hc, v)
        scale = max(1.0, float(np.abs(hc).sum() * np.vdot(v, v).real))
        assert abs(e - E(th)) <= 1e-12 * scale
        assert np.abs(g - want).max() <= 1e-12 * scale, (g, want)
        assert g[0] == 0.0


def test_argument_errors_need_no_device():
    from qubism_b200 import capi
    L = capi.lib()
    x = (C.c_uint64 * 1)(1)
    z = (C.c_uint64 * 1)(0)
    cf = (C.c_double * 2)(0.5, 0.0)
    th = (C.c_double * 1)(0.5)
    e = C.c_double()
    g = (C.c_double * 1)()
    out = C.c_void_p()
    assert L.qb_pauli_sum(None, x, z, cf, 1, C.byref(out)) == capi.QB_ERR_ARG
    assert L.qb_pauli_sum(None, x, z, cf, -1, C.byref(out)) == capi.QB_ERR_ARG
    assert L.qb_pauli_sum(None, None, None, None, 0, None) == capi.QB_ERR_ARG
    assert L.qb_pauli_rot_grad(None, x, z, th, 1, x, z, th, 1, C.byref(e), g) == capi.QB_ERR_ARG
    assert L.qb_pauli_rot_grad(None, x, z, th, -1, x, z, th, 1, C.byref(e), g) == capi.QB_ERR_ARG
    assert L.qb_pauli_rot_grad(None, None, None, None, 0, None, None, None, 0, None, None) == capi.QB_ERR_ARG


def test_pauli_sum_and_adjoint_kernels_do_not_spill():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "qubism_b200", "csrc", "qb_kernels.cu")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    blocks = re.split(r"ptxas info\s*: Compiling entry function ", r.stderr)
    budget = {"k_pauli_sum_tile": 256 * 3, "k_pauli_rot_adjoint_tile": 512}  # threads resident per SM as launched
    seen = set()
    for b in blocks:
        head = b.split("\n", 1)[0]
        for name, threads in budget.items():
            if name not in head:
                continue
            seen.add(name)
            assert "0 bytes spill stores, 0 bytes spill loads" in b, b
            regs = int(re.search(r"Used (\d+) registers", b).group(1))
            assert regs * threads <= 65536, f"{name}: {regs} registers do not fit {threads} threads per SM"
    assert seen == set(budget)
