"""Exact time evolution exp(-itH) under Pauli sums (qb_pauli_evolve) on the device: against the Chebyshev oracle
(tests/pauli_evolve_oracle.py, pinned to scipy's expm in tests/test_pauli_evolve_cpu.py), against exact products
of commuting rotations at 26 qubits, through the identities any exact evolution satisfies at 26-30 qubits,
against second-order Trotter, and across cheap cases, pending scalars, known qubits, layouts, lazy clones,
launch counts, rejected calls and virtual ranks."""
import ctypes as C

import numpy as np
import pytest

from conftest import note_error
from vrank import run_group

pytestmark = pytest.mark.gpu

R2 = 1 / np.sqrt(2)
H = np.array([[R2, R2], [R2, -R2]], dtype=complex)


def _check(got, want, tol):
    err = float(np.abs(np.asarray(got) - np.asarray(want)).max()) if np.size(want) else 0.0
    note_error(err, tol)
    assert err <= tol, (err, tol)


def _masks(terms, n):
    from qubism_b200.statevec import pauli_masks
    return pauli_masks(terms, n)


def _evolve(sv, terms, coefs, t):
    """qb_pauli_evolve on sv in place; returns the number of Chebyshev steps it took."""
    from qubism_b200 import capi
    xs, zs = _masks(terms, sv.n)
    cf = np.ascontiguousarray(coefs, dtype=np.float64)
    k = C.c_int64(-1)
    P64 = C.POINTER(C.c_uint64)
    capi.check(sv.ctx.L.qb_pauli_evolve(sv._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64),
                                        cf.ctypes.data_as(C.POINTER(C.c_double)), len(xs), float(t), C.byref(k)))
    return k.value


def _oracle(n, terms, coefs, t, v):
    from pauli_evolve_oracle import evolve
    xs, zs = _masks(terms, n)
    return evolve(n, xs, zs, coefs, t, v)


def _tol(v, K):
    return 1e-12 * max(1.0, float(np.abs(v).max())) * max(1, K)


def _random_terms(n, k, rng, max_x=12):
    terms = []
    while len(terms) < k:
        s = "".join(rng.choice(list("IXYZ"), n, p=[0.7, 0.1, 0.1, 0.1] if n > 8 else None))
        if sum(ch in "XY" for ch in s) <= max_x:
            terms.append(s)
    return terms


def _one(n, q, p):
    return "I" * q + p + "I" * (n - q - len(p))


def _heisenberg(n, rng, field=True):
    terms, coefs = [], []
    for q in range(n - 1):
        for p in ("XX", "YY", "ZZ"):
            terms.append(_one(n, q, p))
            coefs.append(1.0)
    if field:
        for q in range(n):
            terms.append(_one(n, q, "Z"))
            coefs.append(float(rng.uniform(-1, 1)))
    return terms, np.array(coefs)


def _dist(a, b):  # ||a - b||_2 on the device
    return (a - b).norm2()


@pytest.mark.parametrize("n", list(range(1, 13)))
def test_parity_with_the_oracle(ctx, n):
    """Random sums with identity strings, duplicates and X on a qubit of known value, at several times."""
    import qubism_b200 as Q
    from oracle import structured as S
    rng = np.random.default_rng(5000 + n)
    terms = _random_terms(n, 10 + n, rng) + ["I" * n, "I" * n, "Z" * n, _one(n, 0, "X"), _one(n, 0, "X")]
    coefs = rng.normal(size=len(terms))
    v = S.gen_state(n, rng, normalized=False) * 1.2
    for t in (0.3, -1.1, 4.0):
        sv = Q.StateVec.from_host(v, ctx=ctx)
        K = _evolve(sv, terms, coefs, t)
        want, Kw = _oracle(n, terms, coefs, t, v)
        assert abs(K - Kw) <= 1
        _check(sv.to_host(), want, _tol(v, K))
    if n > 1:  # qubit 0 collapsed: known, and X on it
        sv = Q.StateVec.from_host(v, ctx=ctx).collapse_(0, 1)
        w = S.collapse(n, 0, 1, v)
        K = _evolve(sv, terms, coefs, 0.8)
        want, _ = _oracle(n, terms, coefs, 0.8, w)
        _check(sv.to_host(), want, _tol(w, K))
    out = Q.pauliEvolve(terms, coefs, 0.5, Q.StateVec.from_host(v, ctx=ctx))
    _check(out.to_host(), _oracle(n, terms, coefs, 0.5, v)[0], _tol(v, 20))


def test_parity_at_large_tau(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from pauli_evolve_oracle import k_steps
    n = 10
    rng = np.random.default_rng(5100)
    terms, coefs = _heisenberg(n, rng)
    terms += _random_terms(n, 8, rng)
    coefs = np.concatenate([coefs, rng.normal(size=8)])
    r = float(np.abs(coefs).sum())
    t = 800.0 / r
    v = S.gen_state(n, rng)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    K = _evolve(sv, terms, coefs, t)
    assert abs(K - k_steps(t * r)) <= 1 and K > 850
    want, _ = _oracle(n, terms, coefs, t, v)
    _check(sv.to_host(), want, 1e-10)


def test_commuting_cluster_hamiltonian_is_the_rotation_product(ctx):
    """Z_{i-1} X_i Z_{i+1} commute: exp(-itH) = prod_i exp(-i t h_i P_i), each the rotation R_P(2 t h_i)."""
    import qubism_b200 as Q
    n = 26
    rng = np.random.default_rng(5200)
    terms = [_one(n, 0, "XZ")] + [_one(n, i - 1, "ZXZ") for i in range(1, n - 1)] + [_one(n, n - 2, "ZX")]
    h = rng.uniform(0.5, 1.5, size=len(terms))
    v = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)) * (1 / np.sqrt(2 << n))
    for t in (0.37, -1.3):
        sv = Q.StateVec.from_host(v, ctx=ctx)
        K = _evolve(sv, terms, h, t)
        ref = Q.StateVec.from_host(v, ctx=ctx).pauli_rot_(terms, 2 * t * h)
        err = _dist(sv, ref)
        note_error(err, 1e-11 * K)
        assert err <= 1e-11 * K, (err, K)


@pytest.fixture(scope="module")
def heis26():
    rng = np.random.default_rng(5300)
    return _heisenberg(26, rng)


def _random_state(n, seed, ctx):
    import qubism_b200 as Q
    rng = np.random.default_rng(seed)
    v = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)) * (1 / np.sqrt(2 << n))
    return Q.StateVec.from_host(v, ctx=ctx)


def test_non_commuting_identities_at_26_qubits(ctx, heis26):
    """Heisenberg chain in a random field: back and forth is the identity, the norm and <H> are conserved,
    and evolve(t1) evolve(t2) = evolve(t1 + t2)."""
    n = 26
    terms, coefs = heis26
    v = _random_state(n, 5301, ctx)
    nv = v.norm2()
    e0 = float(np.dot(coefs, v.expect_pauli(terms)))
    a = v.clone()
    _evolve(a, terms, coefs, 0.6)
    _check([a.norm2()], [nv], 1e-12)
    _check([float(np.dot(coefs, a.expect_pauli(terms)))], [e0], 1e-10 * float(np.abs(coefs).sum()))
    assert _dist(a, v) > 0.1  # (it did move)
    b = a.clone()
    _evolve(b, terms, coefs, -0.6)
    err = _dist(b, v)
    note_error(err, 1e-10)
    assert err <= 1e-10
    _evolve(a, terms, coefs, 0.25)
    c = v.clone()
    _evolve(c, terms, coefs, 0.85)
    err = _dist(a, c)
    note_error(err, 1e-10)
    assert err <= 1e-10


def test_round_trip_at_30_qubits(ctx):
    import qubism_b200 as Q
    n = 30
    rng = np.random.default_rng(5400)
    terms, coefs = _heisenberg(n, rng)
    v = Q.mkStateVec(n, ctx)
    v.pauli_rot_([_one(n, q, "Y") for q in range(n)], rng.uniform(0, np.pi, n))
    v.flush()
    a = v.clone()
    K = _evolve(a, terms, coefs, 0.05)
    assert K > 5
    _check([a.norm2()], [1.0], 1e-12)
    _evolve(a, terms, coefs, -0.05)
    err = _dist(a, v)
    note_error(err, 1e-11)
    assert err <= 1e-11


def test_second_order_trotter_converges_to_it(ctx):
    """Doubling the Trotter steps divides the error against the exact evolution by about 4."""
    n = 20
    rng = np.random.default_rng(5500)
    terms, coefs = _heisenberg(n, rng)
    t = 1.0
    v = _random_state(n, 5501, ctx)
    exact = v.clone()
    _evolve(exact, terms, coefs, t)
    errs = []
    for steps in (8, 16):
        dt = t / steps
        rots = (terms + terms[::-1]) * steps
        ang = np.concatenate([coefs * dt, coefs[::-1] * dt] * steps)  # exp(-i dt/2 h P) = R_P(dt h)
        tr = v.clone().pauli_rot_(rots, ang)
        errs.append(_dist(tr, exact))
    ratio = errs[0] / errs[1]
    assert errs[1] > 1e-8 and 3.6 < ratio < 4.4, errs


def test_cheap_cases_launch_nothing(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 12
    rng = np.random.default_rng(5600)
    v = S.gen_state(n, rng)
    ops = [("U", 2, H), ("CX", 2, 5)]
    want = S.run_ops(n, ops, v)
    ref = Q.StateVec.from_host(v, ctx=ctx).submit(ops).to_host()
    terms = _random_terms(n, 6, rng)
    for call in (lambda s: _evolve(s, terms, np.ones(6), 0.0), lambda s: _evolve(s, [], [], 1.5),
                 lambda s: _evolve(s, terms + terms, np.concatenate([np.ones(6), -np.ones(6)]), 0.7)):
        sv = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
        ctx.reset_stats()
        assert call(sv) == 0
        st = ctx.stats()
        assert st["simple_launches"] == 0 and st["passes"] == 0
        assert sv.to_host().tobytes() == ref.tobytes()
    # identity strings only: the phase, deferred
    sv = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    ctx.reset_stats()
    assert _evolve(sv, ["I" * n, "I" * n], [0.4, 0.9], 2.0) == 0
    st = ctx.stats()
    assert st["simple_launches"] == 0 and st["passes"] == 0
    _check(sv.to_host(), np.exp(-2.6j) * want, 1e-14)
    # identity strings beside others: the same phase on top of the evolution
    terms = _random_terms(n, 5, rng)
    c = rng.normal(size=5)
    a = Q.StateVec.from_host(v, ctx=ctx)
    _evolve(a, terms + ["I" * n], np.append(c, 1.7), 0.9)
    b = Q.StateVec.from_host(v, ctx=ctx)
    _evolve(b, terms, c, 0.9)
    _check(a.to_host(), np.exp(-1.53j) * b.to_host(), 1e-14)


def test_pending_scalars(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 11
    rng = np.random.default_rng(5700)
    v = S.gen_state(n, rng)
    terms = _random_terms(n, 9, rng) + ["I" * n]
    coefs = rng.normal(size=len(terms))
    z = 0.7 - 1.9j
    sv = Q.StateVec.from_host(v, ctx=ctx).scale_(z)
    K = _evolve(sv, terms, coefs, 1.3)
    want, _ = _oracle(n, terms, coefs, 1.3, z * v)
    _check(sv.to_host(), want, _tol(z * v, K))
    bad = Q.StateVec.from_host(v, ctx=ctx).scale_(complex(np.nan, 0.0))
    _evolve(bad, terms, coefs, 0.4)
    assert np.isnan(bad.to_host()).all()
    inf = Q.StateVec.from_host(v, ctx=ctx).collapse_(3, 0).scale_(np.inf)
    _evolve(inf, [_one(n, 5, "X")], [1.0], 0.4)
    got = inf.to_host()
    assert not np.isfinite(got).any()  # inf * 0 is NaN: nothing may still claim to be exactly zero


@pytest.mark.parametrize("support", [1, 0])
def test_known_support_of_the_result(ctx, default_opts, support):
    """Qubits collapsed before the call stay known unless a term has X on them: reads, sumsq and measurement."""
    import qubism_b200 as Q
    from oracle import structured as S
    n = 13
    rng = np.random.default_rng(5800 + support)
    saved = ctx.get_option("support")
    ctx.set_option("support", support)
    try:
        v = S.gen_state(n, rng, normalized=False)
        w = S.collapse(n, 9, 0, S.collapse(n, 2, 1, v))
        terms = ["I" * n] + _random_terms(n, 10, rng) + [_one(n, 2, "Z"), _one(n, 3, "XY")]
        terms = [s[:9] + ("Z" if s[9] in "XY" else s[9]) + s[10:] for s in terms]  # no X on qubit 9
        terms.append(_one(n, 2, "X"))  # X on qubit 2: it is forgotten
        coefs = rng.normal(size=len(terms))
        e0 = np.zeros(1 << n, dtype=complex)
        e0[0] = 1.0
        for name, sv, start in (("collapsed", Q.StateVec.from_host(v, ctx=ctx).collapse_(2, 1).collapse_(9, 0), w),
                                ("zero", Q.mkStateVec(n, ctx), e0)):
            ref, K = _oracle(n, terms, coefs, 0.7, start)
            _evolve(sv, terms, coefs, 0.7)
            rtol = 1e-10 * max(1.0, float(np.vdot(ref, ref).real))
            for q in (2, 9, 0):
                _check(sv.sumsq(q), S.sumsq(n, q, ref), rtol)
            assert sv.sumsq(9)[1] == 0.0, name  # no term moves qubit 9: exact zeros stay exact
            _check(sv.to_host(), ref, _tol(ref, K))
            bit, _ = sv.measure_qubit_(n - 1, 0.5)
            b_ref, after, _ = S.measure_qubit(n, n - 1, 0.5, ref)
            assert bit == b_ref
            _check(sv.to_host(), after, 1e-9)
    finally:
        ctx.set_option("support", saved)


OPTION_SETS = [dict(oop=0), dict(oop=1), dict(oop=2), dict(fuse=0), dict(tile_bits=10)]


@pytest.mark.parametrize("opts", OPTION_SETS, ids=lambda o: ",".join(f"{k}={v}" for k, v in o.items()))
def test_planner_options_and_permuted_layouts(ctx, default_opts, opts):
    """Fused passes before the call leave the qubits in a permuted layout; pending gates are flushed first."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops, random_mixed
    for k, val in opts.items():
        ctx.set_option(k, val)
    n = 14
    rng = np.random.default_rng(5900 + len(str(opts)))
    v = S.gen_state(n, rng, normalized=False)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    ops = list(random_mixed(n, 80, seed=41)) + list(qft_ops(n))
    sv.submit(ops).flush()
    v = S.run_ops(n, ops, v)
    ops2 = list(random_mixed(n, 30, seed=42))
    sv.submit(ops2)
    v = S.run_ops(n, ops2, v)
    terms = _random_terms(n, 30, rng) + ["X" * 12 + "II"]
    coefs = rng.normal(size=len(terms))
    K = _evolve(sv, terms, coefs, 0.45)
    want, _ = _oracle(n, terms, coefs, 0.45, v)
    _check(sv.to_host(), want, _tol(v, K))
    sv.submit([("U", 4, H)])  # the evolved state goes on like any other
    _check(sv.to_host(), S.run_ops(n, [("U", 4, H)], want), _tol(v, K))


@pytest.mark.parametrize("linear", [0, 1])
def test_lazy_clones_and_linear(ctx, default_opts, linear):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200 import capi
    n = 13
    rng = np.random.default_rng(6000 + linear)
    v = S.gen_state(n, rng)
    ops = [("U", 3, H), ("CX", 3, 7)]
    ctx.set_option("linear", linear)
    base = Q.StateVec.from_host(v, ctx=ctx).submit(ops).to_host()
    src = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    clone = src.clone()
    terms = _random_terms(n, 12, rng)
    coefs = rng.normal(size=len(terms))
    K = _evolve(src, terms, coefs, 0.9)
    _check(src.to_host(), _oracle(n, terms, coefs, 0.9, S.run_ops(n, ops, v))[0], _tol(v, K))
    if linear:
        with pytest.raises(capi.QbError) as e:
            clone.to_host()
        assert e.value.code == capi.QB_ERR_STATE
    else:
        assert clone.to_host().tobytes() == base.tobytes()
    pure = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    out = Q.pauliEvolve(terms, coefs, 0.9, pure)
    assert out.to_host().tobytes() == src.to_host().tobytes()
    if not linear:
        assert pure.to_host().tobytes() == base.tobytes()


def test_launch_counts_steps_and_determinism(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from pauli_evolve_oracle import k_steps
    n = 16
    rng = np.random.default_rng(6100)
    v = S.gen_state(n, rng)
    zz = [_one(n, q, "ZZ") for q in range(n - 1)]
    xs = [_one(n, q, "X") for q in range(n)]
    extra = [s for s in dict.fromkeys(_random_terms(n, 70, rng)) if s != "I" * n]  # distinct, no identity
    for terms in (zz + xs, zz + xs + extra):
        coefs = rng.normal(size=len(terms))
        ctx.reset_stats()
        Q.StateVec.from_host(v, ctx=ctx).pauli_sum(terms, coefs)
        L = ctx.stats()["simple_launches"]
        assert L >= 2
        outs = []
        for t in (0.7, 0.7, -2.2):
            sv = Q.StateVec.from_host(v, ctx=ctx)
            ctx.reset_stats()
            K = _evolve(sv, terms + ["I" * n], np.append(coefs, 0.3), t)
            st = ctx.stats()
            assert st["simple_launches"] == K * L and st["reduce_launches"] == 0
            assert abs(K - k_steps(t * float(np.abs(coefs).sum()))) <= 1
            outs.append(sv.to_host())
        assert outs[0].tobytes() == outs[1].tobytes()


def test_rejected_calls_leave_the_state_untouched(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200 import capi
    n = 14
    rng = np.random.default_rng(6200)
    v = S.gen_state(n, rng)
    ops = [("U", 2, H), ("CX", 2, 5)]
    ref = Q.StateVec.from_host(v, ctx=ctx).submit(ops).to_host()
    sv = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    ok = ["XZ" + "I" * 12]
    bad = [(["X" * 13 + "I"], [0.1], 0.5, capi.QB_ERR_UNSUPPORTED), (ok, [np.inf], 0.5, capi.QB_ERR_ARG),
           (ok, [np.nan], 0.5, capi.QB_ERR_ARG), ([(1 << n, 0)], [0.1], 0.5, capi.QB_ERR_ARG),
           ([(0, 1 << n)], [0.1], 0.5, capi.QB_ERR_ARG), (ok, [1.0], np.inf, capi.QB_ERR_ARG),
           (ok, [1.0], np.nan, capi.QB_ERR_ARG), (ok, [1.0], 2.0e6, capi.QB_ERR_ARG),
           (ok + ["I" * n], [1.0, 1e308], 1e10, capi.QB_ERR_ARG)]
    ctx.reset_stats()
    for terms, coefs, t, code in bad:
        with pytest.raises(capi.QbError) as e:
            _evolve(sv, terms, coefs, t)
        assert e.value.code == code, (terms, coefs, t)
    st = ctx.stats()
    assert st["simple_launches"] == 0 and st["passes"] == 0  # the queued gates are still queued
    assert sv.to_host().tobytes() == ref.tobytes()
    wide = ["X" * 12 + "II"]  # the widest string the tile holds
    K = _evolve(sv, wide + ok, [1.0, -0.5], 0.3)
    want = S.run_ops(n, ops, v)
    _check(sv.to_host(), _oracle(n, wide + ok, [1.0, -0.5], 0.3, want)[0], _tol(want, K))


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
    """X / Y on global qubits swap them into the shard (the other two states follow); every rank ends with the
    single-GPU state."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import random_layers
    ctxs = groups(P)
    pbits = P.bit_length() - 1
    L = n - pbits
    rng = np.random.default_rng(6300 + P + n)
    full = S.gen_state(n, rng)
    ops = random_layers(n, 2, seed=n)
    w = min(12, L)
    terms = _random_terms(n, 14, rng, max_x=w) + ["X" * pbits + "Z" * (n - pbits), "Z" * n, "I" * (n - 1) + "X"]
    terms += ["Y" * w + "I" * (n - w), "I" * n]
    coefs = rng.normal(size=len(terms))
    start = S.run_ops(n, ops, full)
    one = Q.StateVec.from_host(full, ctx=ctx).submit(ops)
    K1 = _evolve(one, terms, coefs, 0.8)
    single = one.to_host()
    _check(single, _oracle(n, terms, coefs, 0.8, start)[0], _tol(start, K1))

    def work(r, c):
        sv = Q.StateVec.from_host(full[r << L:(r + 1) << L], n=n, ctx=c)
        sv.submit(ops)
        K = _evolve(sv, terms, coefs, 0.8)
        return K, sv.to_host()

    for K, amps in run_group(ctxs, work):
        assert K == K1
        _check(amps, single, _tol(start, K1))


def test_virtual_ranks_reject_a_term_wider_than_the_shard(groups):
    import qubism_b200 as Q
    from qubism_b200 import capi
    ctxs = groups(8)
    n = 8  # 5 local qubits

    def work(r, c):
        sv = Q.StateVec.from_host(np.full(1 << 5, 0.1, dtype=complex), n=n, ctx=c)
        try:
            _evolve(sv, ["X" * 6 + "II"], [1.0], 0.5)
            code = 0
        except capi.QbError as e:
            code = e.code
        return code, sv.local_to_host().tobytes() == np.full(1 << 5, 0.1, dtype=complex).tobytes()

    assert run_group(ctxs, work) == [(capi.QB_ERR_UNSUPPORTED, True)] * 8


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_evolution_over_nccl(world):
    """One process per GPU (torchrun): scripts/pauli_evolve_dist_check.py.  Skipped on a box with fewer GPUs."""
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
                          os.path.join(root, "scripts", "pauli_evolve_dist_check.py")], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0 and "PAULI EVOLVE DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
