"""Pauli rotations exp(-i theta/2 P) on the device (qb_apply_pauli_rot) against the bit-operation oracle
(tests/pauli_rot_oracle.py, itself pinned to scipy.linalg.expm of the dense string in
tests/test_pauli_rot_cpu.py) and against the same evolution decomposed into existing gates (basis changes,
a CX ladder and a diagonal gate) through qb_submit.  Every comparison uses the tolerance
1e-12 * max(1, |psi|^2)."""
import itertools

import numpy as np
import pytest

from conftest import note_error
from vrank import run_group

pytestmark = pytest.mark.gpu

R2 = 1 / np.sqrt(2)
H = np.array([[R2, R2], [R2, -R2]], dtype=complex)
SDG = np.diag([1, -1j])


def _tol(v):
    return 1e-12 * max(1.0, float(np.vdot(v, v).real))


def _check(got, want, tol=None):
    tol = _tol(want) if tol is None else tol
    err = float(np.abs(np.asarray(got) - np.asarray(want)).max()) if np.size(want) else 0.0
    note_error(err, tol)
    assert err <= tol, (err, tol)


def _oracle(n, terms, thetas, v):
    from pauli_rot_oracle import pauli_rot
    from qubism_b200.statevec import pauli_masks
    xs, zs = pauli_masks(terms, n)
    for x, z, th in zip(xs, zs, thetas):
        v = pauli_rot(n, int(x), int(z), float(th), v)
    return v


def _random_terms(n, k, rng, max_x=12, min_x=0):
    terms = []
    while len(terms) < k:
        s = "".join(rng.choice(list("IXYZ"), n, p=[0.7, 0.1, 0.1, 0.1] if n > 8 else None))
        if min_x <= sum(ch in "XY" for ch in s) <= max_x:
            terms.append(s)
    return terms


def _decomposed(s, theta):
    """exp(-i theta/2 P) as existing gates: B on the support (B P_q B^+ = Z), a CX ladder onto the last
    support qubit, diag(e^{-i theta/2}, e^{i theta/2}) there, the ladder back, B^+."""
    sup = [q for q, ch in enumerate(s) if ch != "I"]
    if not sup:
        return [("U", 0, np.exp(-0.5j * theta) * np.eye(2))]
    basis = {"X": H, "Y": H @ SDG, "Z": np.eye(2)}
    pre = [("U", q, basis[s[q]]) for q in sup if s[q] != "Z"]
    post = [("U", q, basis[s[q]].conj().T) for q in sup if s[q] != "Z"]
    ladder = [("CX", sup[i], sup[i + 1]) for i in range(len(sup) - 1)]
    mid = [("U", sup[-1], np.diag([np.exp(-0.5j * theta), np.exp(0.5j * theta)]))]
    return pre + ladder + mid + ladder[::-1] + post


def _run(sv, n, steps, v):
    """Apply a mixed list of steps to the device state and the host reference."""
    from oracle import structured as S
    for st in steps:
        if st[0] == "PAULI":
            sv.pauli_rot_(st[1], st[2])
            v = _oracle(n, st[1], st[2], v)
        elif st[0] == "SCALE":
            sv.scale_(st[1])
            v = v * st[1]
        else:
            sv.run_ops([st])
            v = S.run_ops(n, [st], v)
    return v


def _random_steps(n, rng, count, max_x=12):
    from conftest import rand_unitary_ref
    steps = []
    for _ in range(count):
        k = rng.integers(0, 8)
        if k <= 3:
            m = int(rng.integers(1, 6))
            steps.append(("PAULI", _random_terms(n, m, rng, max_x=max_x), rng.uniform(-4, 4, m)))
        elif k == 4:
            steps.append(("U", int(rng.integers(n)), rand_unitary_ref(rng)))
        elif k == 5:
            c, t = rng.choice(n, 2, replace=False)
            steps.append(("CX", int(c), int(t)))
        elif k == 6:
            c, t = rng.choice(n, 2, replace=False)
            steps.append(("CU", [int(c)], int(t), rand_unitary_ref(rng)))
        else:
            qs = [int(q) for q in rng.choice(n, 2, replace=False)]
            a = rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4))
            steps.append(("KQ", qs, np.linalg.qr(a)[0]))
    return steps


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_every_string_on_small_states(ctx, n):
    import qubism_b200 as Q
    from oracle import structured as S
    rng = np.random.default_rng(200 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.7
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    thetas = rng.uniform(-7, 7, len(strings))
    src = Q.StateVec.from_host(v, ctx=ctx)
    for s, th in zip(strings, thetas):
        _check(Q.pauliRotate([s], [th], src).to_host(), _oracle(n, [s], [th], v))
    _check(src.to_host(), v)  # the source of the pure applications kept its value
    _check(Q.StateVec.from_host(v, ctx=ctx).pauli_rot_(strings, thetas).to_host(), _oracle(n, strings, thetas, v))


@pytest.mark.parametrize("n", [12, 20])
def test_random_sequences_among_other_gates(ctx, n):
    import qubism_b200 as Q
    from oracle import structured as S
    rng = np.random.default_rng(300 + n)
    v = S.gen_state(n, rng, normalized=False) * 0.8
    sv = Q.StateVec.from_host(v, ctx=ctx)
    steps = _random_steps(n, rng, 60)
    steps.insert(20, ("COLLAPSE", 2, 1))
    steps.insert(40, ("SCALE", 0.5 - 1.5j))
    steps.append(("PAULI", ["X" * 12 + "Z" * (n - 12)], [0.3]))
    ref = _run(sv, n, steps, v)
    _check(sv.to_host(), ref)


@pytest.mark.parametrize("n", [24, 26])
def test_against_the_decomposed_evolution(ctx, n):
    import qubism_b200 as Q
    rng = np.random.default_rng(400 + n)
    v = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)) * (1 / np.sqrt(1 << n))
    terms = _random_terms(n, 24, rng, max_x=12) + ["Z" * n, "Y" * 12 + "I" * (n - 12)]
    thetas = rng.uniform(-4, 4, len(terms))
    native = Q.StateVec.from_host(v, ctx=ctx).pauli_rot_(terms, thetas).to_host()
    dec = Q.StateVec.from_host(v, ctx=ctx)
    dec.submit([op for s, th in zip(terms, thetas) for op in _decomposed(s, th)])
    _check(native, dec.to_host(), _tol(v))


OPTION_SETS = [(dict(oop=0), 14), (dict(oop=1), 14), (dict(oop=2), 14), (dict(fuse=0), 14), (dict(jit=0), 14),
               (dict(jit=1), 14), (dict(tile_bits=10), 14), (dict(support=0), 14), (dict(support=1, oop=1), 14),
               (dict(), 9)]  # (n = 9: a shard below the fused tile, the unfused path)


@pytest.mark.parametrize("opts,n", OPTION_SETS,
                         ids=lambda o: ",".join(f"{k}={v}" for k, v in o.items()) or "unfused" if isinstance(o, dict) else f"n{o}")
def test_planner_options_and_permuted_layouts(ctx, default_opts, opts, n):
    """Out-of-place passes before and between the rotations leave the qubits in a permuted layout."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops, random_mixed
    saved = {k: ctx.get_option(k) for k in opts}
    try:
        for k, val in opts.items():
            ctx.set_option(k, val)
        rng = np.random.default_rng(500 + len(str(opts)))
        v = S.gen_state(n, rng, normalized=False) * 1.2
        sv = Q.StateVec.from_host(v, ctx=ctx)
        steps = list(random_mixed(n, 80, seed=21)) + [("PAULI", _random_terms(n, 30, rng), rng.uniform(-3, 3, 30))]
        steps += list(qft_ops(n)) + [("PAULI", _random_terms(n, 70, rng), rng.uniform(-3, 3, 70))]
        steps += list(random_mixed(n, 40, seed=22))
        for _ in range(2):  # the second round runs with whatever layout the first left
            v = _run(sv, n, steps, v)
            _check(sv.to_host(), v)
    finally:
        for k, val in saved.items():
            ctx.set_option(k, val)


def test_lazy_clones_pure_pattern_and_linear(ctx, default_opts):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 13
    rng = np.random.default_rng(600)
    v = S.gen_state(n, rng)
    src = Q.StateVec.from_host(v, ctx=ctx)
    src.submit([("U", 3, H)])
    v = S.run_ops(n, [("U", 3, H)], v)
    terms = _random_terms(n, 10, rng)
    thetas = rng.uniform(-3, 3, 10)
    rot = Q.pauliRotate(terms, thetas, src)
    _check(rot.to_host(), _oracle(n, terms, thetas, v))
    _check(src.to_host(), v)  # the source is unchanged
    # the interpreter's per-op pure pattern: every step a new value
    sv, ref = src, v
    for i in range(12):
        if i % 3 == 2:
            sv = sv.apply_pure([("CX", i % n, (i + 5) % n)])
            ref = S.run_ops(n, [("CX", i % n, (i + 5) % n)], ref)
        else:
            t = _random_terms(n, 1, rng)
            th = rng.uniform(-3, 3, 1)
            sv = Q.pauliRotate(t, th, sv)
            ref = _oracle(n, t, th, ref)
    _check(sv.to_host(), ref)
    _check(src.to_host(), v)
    ctx.set_option("linear", 1)
    try:
        a = Q.StateVec.from_host(v, ctx=ctx)
        b = Q.pauliRotate(terms, thetas, a)
        c = Q.pauliRotate(terms[::-1], -thetas[::-1], b)
        _check(b.to_host(), _oracle(n, terms, thetas, v))
        _check(c.to_host(), v)
    finally:
        ctx.set_option("linear", 0)


def test_known_qubits_from_zero_and_after_a_collapse(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 12
    rng = np.random.default_rng(700)
    terms = ["X" + "I" * (n - 1), "IYZ" + "I" * (n - 3), "ZZ" + "I" * (n - 2), "XX" + "Y" * (n - 2)]
    thetas = rng.uniform(-3, 3, len(terms))
    sv = Q.mkStateVec(n, ctx)
    sv.scale_(0.5 - 2j)
    sv.pauli_rot_(terms, thetas)
    e0 = np.zeros(1 << n, dtype=complex)
    e0[0] = 0.5 - 2j
    _check(sv.to_host(), _oracle(n, terms, thetas, e0))
    v = S.gen_state(n, rng)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    sv.collapse_(3, 1)
    t2 = ["IIIX" + "I" * (n - 4), "IIIZ" + "Z" * (n - 4), "XIIY" + "I" * (n - 4)]
    th2 = rng.uniform(-3, 3, 3)
    sv.pauli_rot_(t2, th2)
    sv.collapse_(5, 0)
    _check(sv.to_host(), S.collapse(n, 5, 0, _oracle(n, t2, th2, S.collapse(n, 3, 1, v))))


def test_launch_counts(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 16
    rng = np.random.default_rng(800)
    v = S.gen_state(n, rng)
    # 130 rotations with X / Y inside nine qubits (+ the three low bits: one tile) -> 3 launches of <= 64
    sv = Q.StateVec.from_host(v, ctx=ctx)
    xs = [int(x) << (n - 9) for x in rng.integers(0, 1 << 9, 130)]
    zs = [int(z) for z in rng.integers(0, 1 << n, 130)]
    th = rng.uniform(-3, 3, 130)
    ctx.reset_stats()
    sv.pauli_rot_(list(zip(xs, zs)), th).flush()
    assert ctx.stats()["simple_launches"] == 3
    _check(sv.to_host(), _oracle(n, list(zip(xs, zs)), th, v))
    # the identity string: a global factor, no launch
    sv = Q.StateVec.from_host(v, ctx=ctx)
    ctx.reset_stats()
    sv.pauli_rot_(["I" * n] * 3, [0.4, 1.0, -2.0])
    _check(sv.expect_pauli(["I" * n]), [np.vdot(v, v).real], _tol(v))  # (observes; keeps the scalar pending)
    assert ctx.stats()["simple_launches"] == 0 and ctx.stats()["passes"] == 0
    _check(sv.to_host(), v * np.exp(-0.5j * (0.4 + 1.0 - 2.0)))
    # X on every qubit in turn: qubits 0..8 (bits 15..7) fill the tile with the three low bits, the rest
    # (bits 6..0) start a second launch
    sv = Q.StateVec.from_host(v, ctx=ctx)
    terms = ["I" * q + "X" + "I" * (n - 1 - q) for q in range(n)]
    ctx.reset_stats()
    sv.pauli_rot_(terms, np.full(n, 0.3)).flush()
    assert ctx.stats()["simple_launches"] == 2
    _check(sv.to_host(), _oracle(n, terms, np.full(n, 0.3), v))


def test_deterministic_and_expectation_preserved(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops
    n = 18
    rng = np.random.default_rng(900)
    v = S.gen_state(n, rng, normalized=False)
    terms = _random_terms(n, 40, rng)
    th = rng.uniform(-3, 3, 40)
    outs = []
    for _ in range(2):
        sv = Q.StateVec.from_host(v, ctx=ctx)
        sv.submit(qft_ops(n))
        sv.pauli_rot_(terms, th)
        outs.append(sv.to_host())
    assert outs[0].tobytes() == outs[1].tobytes()
    sv = Q.StateVec.from_host(v, ctx=ctx)
    for s, t in zip(terms[:10], th[:10]):
        before = sv.expect_pauli([s])
        sv.pauli_rot_([s], [t])
        _check(sv.expect_pauli([s]), before, _tol(v))


def test_round_trip_at_26_qubits(ctx):
    import qubism_b200 as Q
    n = 26
    rng = np.random.default_rng(1000)
    v = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)) * (1 / np.sqrt(1 << n))
    terms = _random_terms(n, 40, rng, max_x=12)
    th = rng.uniform(-4, 4, 40)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    sv.pauli_rot_(terms, th).pauli_rot_(terms[::-1], -th[::-1])
    _check(sv.to_host(), v, _tol(v))


def test_rejected_calls_leave_the_state_untouched(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200 import capi
    n = 14
    rng = np.random.default_rng(1100)
    v = S.gen_state(n, rng)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    ops = [("U", 2, H), ("CX", 2, 5)]
    sv.submit(ops)
    for terms, th, code in [(["X" * 13 + "I"], [0.1], capi.QB_ERR_UNSUPPORTED),
                            (["XZ" + "I" * 12, "Y" * 13 + "I"], [0.1, 0.2], capi.QB_ERR_UNSUPPORTED),
                            (["XZ" + "I" * 12, "ZZ" + "I" * 12], [0.1, np.nan], capi.QB_ERR_ARG),
                            ([(1 << n, 0)], [0.1], capi.QB_ERR_ARG)]:
        with pytest.raises(capi.QbError) as e:
            sv.pauli_rot_(terms, th)
        assert e.value.code == code
    _check(sv.to_host(), S.run_ops(n, ops, v))
    sv.pauli_rot_(["X" * 12 + "II"], [0.5])  # the widest string the tile holds
    _check(sv.to_host(), _oracle(n, ["X" * 12 + "II"], [0.5], S.run_ops(n, ops, v)))


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
    """X / Y on global qubits swap them into the shard; Z on global qubits is a per-rank sign."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import random_layers
    ctxs = groups(P)
    pbits = P.bit_length() - 1
    L = n - pbits
    rng = np.random.default_rng(1200 + P + n)
    full = S.gen_state(n, rng)
    ops = random_layers(n, 2, seed=n)
    terms = _random_terms(n, 30, rng, max_x=min(12, L)) + ["X" * pbits + "I" * (n - pbits),
                                                           "Y" * (pbits + 1) + "Z" * (n - pbits - 1), "Z" * n,
                                                           "X" * min(12, L) + "I" * (n - min(12, L))]
    th = rng.uniform(-3, 3, len(terms))
    ref = _oracle(n, terms, th, S.run_ops(n, ops, full))
    ref = S.run_ops(n, ops, ref)

    def work(r, c):
        sv = Q.StateVec.from_host(full[r << L:(r + 1) << L], n=n, ctx=c)
        sv.submit(ops)
        sv.pauli_rot_(terms, th)
        sv.submit(ops)
        return sv.to_host()

    res = run_group(ctxs, work)
    for amps in res:
        _check(amps, ref)


def test_virtual_ranks_reject_a_string_wider_than_the_shard(groups):
    import qubism_b200 as Q
    from qubism_b200 import capi
    ctxs = groups(8)
    n = 8  # 5 local qubits

    def work(r, c):
        sv = Q.StateVec.from_host(np.full(1 << 5, 0.1, dtype=complex), n=n, ctx=c)
        try:
            sv.pauli_rot_(["X" * 6 + "II"], [0.1])
        except capi.QbError as e:
            return e.code, sv.local_to_host().tobytes() == np.full(1 << 5, 0.1, dtype=complex).tobytes()
        return 0, False

    assert run_group(ctxs, work) == [(capi.QB_ERR_UNSUPPORTED, True)] * 8


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_rotations_over_nccl(world):
    """One process per GPU (torchrun): scripts/pauli_rot_dist_check.py.  Skipped on a box with fewer GPUs."""
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
                          os.path.join(root, "scripts", "pauli_rot_dist_check.py")], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0 and "PAULI ROT DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
