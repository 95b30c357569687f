"""Pauli expectation values without a device: the bit-operation oracle (tests/pauli_oracle.py) against the
reference's literal form, argument checks of qb_expect_pauli, and the register budget of its kernel."""
import ctypes as C
import itertools
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _literal(n, s, v):
    """realPart (v <.> (p #> v)) with p = onJust q pauliX/Y/Z multiplied out as dense matrices."""
    from oracle import dense as D
    one = {"X": D.pauliX(), "Y": D.pauliY(), "Z": D.pauliZ()}
    M = D.ident(n)
    for q, ch in enumerate(s):
        if ch != "I":
            M = D.onJust(n, q, one[ch]) @ M
    return D.inner(v, D.apply(M, v)).real


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5])
def test_oracle_matches_the_literal_form_on_every_string(n):
    from oracle import structured as S
    from pauli_oracle import expect_pauli
    from qubism_b200.statevec import pauli_masks
    rng = np.random.default_rng(40 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.7
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    xs, zs = pauli_masks(strings, n)
    for s, x, z in zip(strings, xs, zs):
        want = _literal(n, s, v)
        got = expect_pauli(n, int(x), int(z), v)
        assert abs(got - want) <= 1e-12 * max(1.0, float(np.vdot(v, v).real)), (s, got, want)


def test_pauli_masks_spellings():
    from qubism_b200.statevec import pauli_masks
    xs, zs = pauli_masks(["XYZI", (5, 6), "iiii"], 4)
    assert list(xs) == [0b0011, 5, 0] and list(zs) == [0b0110, 6, 0]
    with pytest.raises(ValueError):
        pauli_masks(["XYZ"], 4)
    with pytest.raises(ValueError):
        pauli_masks(["XYZA"], 4)


def test_argument_errors_need_no_device():
    from qubism_b200 import capi
    L = capi.lib()
    x = (C.c_uint64 * 1)(1)
    z = (C.c_uint64 * 1)(0)
    out = (C.c_double * 1)()
    assert L.qb_expect_pauli(None, x, z, 1, out) == capi.QB_ERR_ARG
    assert L.qb_expect_pauli(None, x, z, -1, out) == capi.QB_ERR_ARG
    assert L.qb_expect_pauli(None, None, None, 0, None) == capi.QB_ERR_ARG


def test_expect_kernels_do_not_spill():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "qubism_b200", "csrc", "qb_kernels.cu")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    blocks = re.split(r"ptxas info\s*: Compiling entry function ", r.stderr)
    seen = 0
    for b in blocks:
        if "k_expect" not in b.split("\n", 1)[0]:
            continue
        seen += 1
        assert "0 bytes spill stores, 0 bytes spill loads" in b, b
    assert seen >= 8  # the final stage and the partial stage for 1, 2, 4, ..., 64 terms
