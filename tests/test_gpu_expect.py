"""Pauli expectation values on the device (qb_expect_pauli) against the bit-operation oracle
(tests/pauli_oracle.py, itself pinned to the literal dense form in tests/test_expect_cpu.py) and against
the reference route realPart (sv <.> (p #> sv)) through the lazy clone.  Every comparison uses the
tolerance 1e-12 * max(1, |psi|^2)."""
import itertools

import numpy as np
import pytest

from conftest import note_error
from vrank import run_group

pytestmark = pytest.mark.gpu


def _tol(v):
    return 1e-12 * max(1.0, float(np.vdot(v, v).real))


def _oracle(n, xs, zs, v):
    from pauli_oracle import expect_pauli
    return np.array([expect_pauli(n, int(x), int(z), v) for x, z in zip(xs, zs)])


def _check(got, want, tol):
    err = float(np.abs(np.asarray(got) - np.asarray(want)).max()) if len(want) else 0.0
    note_error(err, tol)
    assert err <= tol, (err, tol)


def _random_terms(n, k, rng, max_x=None):
    terms = []
    while len(terms) < k:
        s = "".join(rng.choice(list("IXYZ"), n))
        if max_x is None or sum(ch in "XY" for ch in s) <= max_x:
            terms.append(s)
    return terms


def _pauli_ops(s):
    from oracle import dense as D
    m = {"X": D.pauliX(), "Y": D.pauliY(), "Z": D.pauliZ()}
    return [("U", q, m[ch]) for q, ch in enumerate(s) if ch != "I"]


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_every_string_on_small_states(ctx, n):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.statevec import pauli_masks
    v = S.gen_state(n, np.random.default_rng(70 + n), normalized=False) * 1.9
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    sv = Q.StateVec.from_host(v, ctx=ctx)
    got = sv.expect_pauli(strings)
    _check(got, _oracle(n, *pauli_masks(strings, n), v), _tol(v))


@pytest.mark.parametrize("n", [12, 20])
def test_random_strings(ctx, n):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.statevec import pauli_masks
    rng = np.random.default_rng(80 + n)
    v = S.gen_state(n, rng, normalized=False) * 0.6
    terms = _random_terms(n, 200, rng)
    got = Q.expectPauli(terms, Q.StateVec.from_host(v, ctx=ctx))
    _check(got, _oracle(n, *pauli_masks(terms, n), v), _tol(v))


@pytest.mark.parametrize("jit", [0, 1])
@pytest.mark.parametrize("oop", [0, 1, 2])
@pytest.mark.parametrize("circuit", ["mixed", "layers"])
def test_after_circuits_in_permuted_layouts(ctx, default_opts, circuit, oop, jit):
    """Out-of-place passes leave the qubits in a permuted layout; both routes must see the reference's qubits."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops, random_layers, random_mixed
    from qubism_b200.statevec import pauli_masks
    n = 14
    ctx.set_option("oop", oop)
    ctx.set_option("jit", jit)
    ops = random_mixed(n, 120, seed=11 + oop) if circuit == "mixed" else qft_ops(n) + random_layers(n, 3, seed=12 + oop)
    rng = np.random.default_rng(90 + oop + 3 * jit)
    v = S.gen_state(n, rng, normalized=False) * 1.3
    ref = S.run_ops(n, ops, v)
    terms = _random_terms(n, 40, rng) + ["Z" * n, "X" * n, "I" * n]
    sv = Q.StateVec.from_host(v, ctx=ctx)
    sv.submit(ops)
    got = sv.expect_pauli(terms)
    _check(got, _oracle(n, *pauli_masks(terms, n), ref), _tol(ref))
    route = [sv.inner(sv.apply_pure(_pauli_ops(s))).real for s in terms[:8]]
    _check(got[:8], route, _tol(ref))


def test_known_support_costs_nothing(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.statevec import pauli_masks
    n = 10
    # fresh |0...0> under a queued scalar
    sv = Q.mkStateVec(n, ctx)
    sv.scale_(0.5 - 2j)
    ctx.reset_stats()
    flips = ["X" + "I" * (n - 1), "IYZ" + "I" * (n - 3), "XX" + "Z" * (n - 2)]
    got = sv.expect_pauli(flips)
    assert list(got) == [0.0, 0.0, 0.0]
    assert ctx.stats()["reduce_launches"] == 0
    got = sv.expect_pauli(["Z" * n, "I" * n])
    _check(got, [4.25, 4.25], 1e-12 * 4.25)
    # after a collapse: qubit 3 is known to be 1
    rng = np.random.default_rng(5)
    v = S.gen_state(n, rng)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    sv.collapse_(3, 1)
    ref = S.collapse(n, 3, 1, v)
    terms = _random_terms(n, 60, rng)
    dead = [t for t in terms if t[3] in "XY"]
    live = [t for t in terms if t[3] not in "XY"]
    ctx.reset_stats()
    assert list(sv.expect_pauli(dead)) == [0.0] * len(dead)
    assert ctx.stats()["reduce_launches"] == 0
    _check(sv.expect_pauli(live), _oracle(n, *pauli_masks(live, n), ref), _tol(ref))


def test_deterministic_read_only_and_one_sweep_per_group(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops
    n = 16
    rng = np.random.default_rng(6)
    v = S.gen_state(n, rng, normalized=False)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    sv.submit(qft_ops(n))
    before = sv.to_host()
    # 3 X masks: 1 term, 70 terms (two chunks of <= 64), 5 terms; plus the diagonal group
    xs = [0b101] + [0b110] * 70 + [1 << 15] * 5 + [0] * 3
    zs = [int(z) for z in rng.integers(0, 1 << n, len(xs))]
    ctx.reset_stats()
    a = sv.expect_pauli(list(zip(xs, zs)))
    assert ctx.stats()["reduce_launches"] == 2 * (1 + 2 + 1 + 1)
    b = sv.expect_pauli(list(zip(xs, zs)))
    assert a.tobytes() == b.tobytes()
    assert sv.to_host().tobytes() == before.tobytes()
    _check(a, _oracle(n, xs, zs, before), _tol(before))


def test_argument_errors(ctx):
    import qubism_b200 as Q
    from qubism_b200 import capi
    sv = Q.mkStateVec(4, ctx)
    with pytest.raises(capi.QbError) as e:
        sv.expect_pauli([(1 << 4, 0)])
    assert e.value.code == capi.QB_ERR_ARG
    assert sv.expect_pauli([]).shape == (0,)


@pytest.fixture(scope="module")
def groups():
    import qubism_b200 as Q
    made = {}

    def get(P):
        if P not in made:
            made[P] = Q.Context.group([0] * P)
        return made[P]

    yield get
    for ctxs in made.values():
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("P,n", [(2, 12), (4, 13), (8, 12), (8, 16)])
def test_virtual_ranks(ctx, groups, P, n):
    """X / Y on global qubits swap them into the shard; every rank gets every value."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import random_layers
    from qubism_b200.statevec import pauli_masks
    ctxs = groups(P)
    pbits = P.bit_length() - 1
    L = n - pbits
    rng = np.random.default_rng(100 + P + n)
    full = S.gen_state(n, rng)
    ops = random_layers(n, 2, seed=n)
    ref = S.run_ops(n, ops, full)
    terms = _random_terms(n, 40, rng, max_x=L) + ["X" * pbits + "I" * (n - pbits), "Y" * (pbits + 1) + "Z" * (n - pbits - 1),
                                                  "Z" * n, "X" * L + "I" * pbits]
    xs, zs = pauli_masks(terms, n)
    one = Q.StateVec.from_host(full, ctx=ctx)
    one.submit(ops)
    single = one.expect_pauli(terms)

    def work(r, c):
        sv = Q.StateVec.from_host(full[r << L:(r + 1) << L], n=n, ctx=c)
        sv.submit(ops)
        got = sv.expect_pauli(terms)
        return got, sv.to_host()

    res = run_group(ctxs, work)
    for got, _ in res[1:]:
        assert got.tobytes() == res[0][0].tobytes()
    tol = _tol(ref)
    _check(res[0][0], _oracle(n, xs, zs, ref), tol)
    _check(res[0][0], single, tol)
    for _, amps in res:
        err = float(np.abs(amps - ref).max())
        note_error(err, 1e-12)
        assert err <= 1e-12


def test_virtual_ranks_reject_a_string_wider_than_the_shard(groups):
    import qubism_b200 as Q
    from qubism_b200 import capi
    ctxs = groups(8)
    n = 8  # 5 local qubits

    def work(r, c):
        sv = Q.StateVec.from_host(np.full(1 << 5, 0.1, dtype=complex), n=n, ctx=c)
        try:
            sv.expect_pauli(["X" * n])
        except capi.QbError as e:
            return e.code
        return 0

    assert run_group(ctxs, work) == [capi.QB_ERR_UNSUPPORTED] * 8


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_expectation_over_nccl(world):
    """One process per GPU (torchrun): scripts/expect_dist_check.py.  Skipped on a box with fewer GPUs."""
    import os
    import socket
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(root, "scripts", "expect_dist_check.py")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "EXPECT DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
