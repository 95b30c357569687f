"""Pauli sums H|psi> (qb_pauli_sum) and adjoint gradients of Pauli-sum energies over Pauli rotations
(qb_pauli_rot_grad) on the device, against the host oracle (tests/pauli_grad_oracle.py, pinned to the dense
strings and to the dense parameter-shift rule in tests/test_pauli_grad_cpu.py), against the parameter-shift
rule computed with the device's own rotations and expectation values, and across layouts, planner options,
lazy clones and virtual ranks."""
import itertools

import numpy as np
import pytest

from conftest import note_error
from vrank import run_group

pytestmark = pytest.mark.gpu

R2 = 1 / np.sqrt(2)
H = np.array([[R2, R2], [R2, -R2]], dtype=complex)


def _check(got, want, tol):
    if tol == 0.0:  # an exact comparison: nothing to report
        assert np.asarray(got).tobytes() == np.asarray(want, dtype=np.asarray(got).dtype).tobytes()
        return
    err = float(np.abs(np.asarray(got) - np.asarray(want)).max()) if np.size(want) else 0.0
    note_error(err, tol)
    assert err <= tol, (err, tol)


def _vtol(v):
    return 1e-12 * max(1.0, float(np.abs(v).max()))


def _gtol(v, hc):
    return 1e-12 * max(1.0, float(np.abs(hc).sum() * np.vdot(v, v).real))


def _masks(terms, n):
    from qubism_b200.statevec import pauli_masks
    return pauli_masks(terms, n)


def _random_terms(n, k, rng, max_x=12):
    terms = []
    while len(terms) < k:
        s = "".join(rng.choice(list("IXYZ"), n, p=[0.7, 0.1, 0.1, 0.1] if n > 8 else None))
        if sum(ch in "XY" for ch in s) <= max_x:
            terms.append(s)
    return terms


def _rotation_list(n, k, rng, max_x=12):
    """I, Z-only, Y-only and random strings up to weight max_x"""
    terms = ["I" * n, "Z" * n, "Y" + "I" * (n - 1), "I" * (n - 1) + "Y"] + _random_terms(n, k - 4, rng, max_x)
    w = min(n, max_x)
    terms.append("Y" * w + "Z" * (n - w))
    return terms


def _sum_oracle(n, terms, coefs, v):
    from pauli_grad_oracle import pauli_sum
    xs, zs = _masks(terms, n)
    return pauli_sum(n, xs, zs, coefs, v)


def _grad_oracle(n, rots, th, hterms, hc, v):
    from pauli_grad_oracle import rot_grad
    rx, rz = _masks(rots, n)
    hx, hz = _masks(hterms, n)
    return rot_grad(n, rx, rz, th, hx, hz, hc, v)


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_pauli_sum_of_every_string_on_small_states(ctx, n):
    import qubism_b200 as Q
    from oracle import structured as S
    rng = np.random.default_rng(2000 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.4
    sv = Q.StateVec.from_host(v, ctx=ctx)
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    for s in strings:
        c = complex(rng.normal(), rng.normal())
        _check(sv.pauli_sum([s], [c]).to_host(), _sum_oracle(n, [s], [c], v), _vtol(v))
    cs = rng.normal(size=len(strings)) + 1j * rng.normal(size=len(strings))
    out = Q.pauliSum(strings, cs, sv)
    want = _sum_oracle(n, strings, cs, v)
    _check(out.to_host(), want, 1e-12 * max(1.0, float(np.abs(want).max())) * len(strings))
    _check(sv.to_host(), v, 0.0)


@pytest.mark.parametrize("n", [5, 9, 12])
def test_pauli_sum_random_sums_and_the_output_support(ctx, default_opts, n):
    """The identity, duplicate strings, and X on qubits of known value; the output's support is checked by
    reading, measuring and taking expectation values of it."""
    import qubism_b200 as Q
    from oracle import structured as S
    from pauli_oracle import expect_pauli
    rng = np.random.default_rng(2100 + n)
    terms = _random_terms(n, 20, rng) + ["I" * n, "X" + "I" * (n - 1), "X" + "I" * (n - 1), "Z" * n]
    terms += ["I" * (n - 1) + "Y", "Y" + "I" * (n - 2) + "X"]
    cs = rng.normal(size=len(terms)) + 1j * rng.normal(size=len(terms))
    e0 = np.zeros(1 << n, dtype=complex)
    e0[0] = 1.0
    vr = S.gen_state(n, rng, normalized=False)
    cases = [("random", Q.StateVec.from_host(vr, ctx=ctx), vr), ("zero", Q.mkStateVec(n, ctx), e0)]
    sv = Q.StateVec.from_host(vr, ctx=ctx)
    q = n // 2
    sv.collapse_(q, 1)
    cases.append(("collapsed", sv, S.collapse(n, q, 1, vr)))
    obs = _random_terms(n, 6, rng) + ["Z" * n]
    ox, oz = _masks(obs, n)
    saved = ctx.get_option("support")
    for support in (1, 0):
        ctx.set_option("support", support)
        for name, src, v in cases:
            want = _sum_oracle(n, terms, cs, v)
            tol = 1e-12 * max(1.0, float(np.abs(want).max())) * len(terms)
            out = src.pauli_sum(terms, cs)
            rtol = 1e-10 * max(1.0, float(np.vdot(want, want).real))
            ev = out.expect_pauli(obs)
            _check(ev, [expect_pauli(n, int(x), int(z), want) for x, z in zip(ox, oz)], rtol)
            for k in range(n):
                _check(out.sumsq(k), S.sumsq(n, k, want), rtol)
            _check(out.to_host(), want, tol)
            bit, _ = out.measure_qubit_(n - 1, 0.5)
            _check(out.to_host(), S.measure_qubit(n, n - 1, 0.5, want)[1], 1e-9)
            assert bit == S.measure_qubit(n, n - 1, 0.5, want)[0], name
    ctx.set_option("support", saved)
    zero = cases[0][1].pauli_sum([], [])
    _check(zero.to_host(), np.zeros(1 << n), 0.0)


@pytest.mark.parametrize("n", list(range(1, 13)))
def test_gradient_parity_with_the_oracle(ctx, n):
    import qubism_b200 as Q
    from oracle import structured as S
    rng = np.random.default_rng(2200 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.1
    rots = _rotation_list(n, 24, rng)
    th = rng.uniform(-np.pi, np.pi, len(rots))
    hterms = _random_terms(n, 12, rng) + ["I" * n, "Z" * n]
    hc = rng.normal(size=len(hterms))
    sv = Q.StateVec.from_host(v, ctx=ctx)
    e, g = Q.pauliRotGrad(rots, th, hterms, hc, sv)
    we, wg = _grad_oracle(n, rots, th, hterms, hc, v)
    tol = _gtol(v, hc)
    _check([e], [we], tol)
    _check(g, wg, tol)
    assert g[0] == 0.0  # the identity string
    # the energy is sum_t hc[t] <H_t> of the rotated state
    psi = Q.pauliRotate(rots, th, sv)
    _check([e], [float(np.dot(hc, psi.expect_pauli(hterms)))], tol)


@pytest.mark.parametrize("n", [20, 26])
def test_parameter_shift_with_the_device_rotations(ctx, n):
    """Several tiles and launches: every component against (E(theta + pi/2) - E(theta - pi/2)) / 2, each E one
    clone + pauli_rot_ + expect_pauli on the device."""
    import qubism_b200 as Q
    rng = np.random.default_rng(2300 + n)
    v = (rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)) * (1 / np.sqrt(1 << n))
    rots = _random_terms(n, 5, rng, max_x=12) + ["X" * 12 + "I" * (n - 12), "I" * (n - 3) + "YXZ"]
    rots += ["Z" * n, "I" * (n // 2) + "XY" + "I" * (n - n // 2 - 2)]
    th = rng.uniform(-np.pi, np.pi, len(rots))
    hterms = [("I" * q + "ZZ" + "I" * (n - q - 2)) for q in range(n - 1)] + ["I" * q + "X" + "I" * (n - q - 1) for q in range(n)]
    hterms += _random_terms(n, 6, rng)
    hc = rng.normal(size=len(hterms))
    sv = Q.StateVec.from_host(v, ctx=ctx)
    e, g = sv.pauli_rot_grad(rots, th, hterms, hc)

    def E(t):
        return float(np.dot(hc, sv.clone().pauli_rot_(rots, t).expect_pauli(hterms)))

    shift = np.array([(E(th + np.pi / 2 * np.eye(len(th))[k]) - E(th - np.pi / 2 * np.eye(len(th))[k])) / 2
                      for k in range(len(th))])
    scale = float(np.abs(hc).sum())
    _check(g, shift, 1e-10 * scale)
    _check([e], [E(th)], 1e-10 * scale)


OPTION_SETS = [dict(oop=0), dict(oop=1), dict(oop=2), dict(tile_bits=10), dict(fuse=0), dict(support=0)]


@pytest.mark.parametrize("opts", OPTION_SETS, ids=lambda o: ",".join(f"{k}={v}" for k, v in o.items()))
def test_planner_options_and_permuted_layouts(ctx, default_opts, opts):
    """Fused passes before the call leave the qubits in a permuted layout; pending gates ride in the copy."""
    saved = {k: ctx.get_option(k) for k in opts}
    try:
        for k, val in opts.items():
            ctx.set_option(k, val)
        _options_case(ctx, opts)
    finally:
        for k, val in saved.items():
            ctx.set_option(k, val)


def _options_case(ctx, opts):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops, random_mixed
    n = 14
    rng = np.random.default_rng(2400 + len(str(opts)))
    v = S.gen_state(n, rng, normalized=False)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    ops = list(random_mixed(n, 80, seed=31)) + list(qft_ops(n))
    sv.submit(ops).flush()
    v = S.run_ops(n, ops, v)
    ops2 = list(random_mixed(n, 30, seed=32))
    sv.submit(ops2)  # pending when the gradient is asked for
    v = S.run_ops(n, ops2, v)
    rots = _rotation_list(n, 40, rng)
    th = rng.uniform(-3, 3, len(rots))
    hterms = _random_terms(n, 20, rng)
    hc = rng.normal(size=len(hterms))
    e, g = sv.pauli_rot_grad(rots, th, hterms, hc)
    we, wg = _grad_oracle(n, rots, th, hterms, hc, v)
    _check([e], [we], _gtol(v, hc))
    _check(g, wg, _gtol(v, hc))
    _check(sv.to_host(), v, _vtol(v))
    cs = rng.normal(size=len(hterms)) + 1j * rng.normal(size=len(hterms))
    want = _sum_oracle(n, hterms, cs, v)
    _check(sv.pauli_sum(hterms, cs).to_host(), want, 1e-12 * max(1.0, float(np.abs(want).max())) * len(hterms))


def test_pending_scalar(ctx):
    """A pending scalar z on s: psi = z psi_dev, energy and gradient scale by |z|^2; H psi by z."""
    import qubism_b200 as Q
    from oracle import structured as S
    n = 11
    rng = np.random.default_rng(2500)
    v = S.gen_state(n, rng)
    z = 0.7 - 1.9j
    rots = _rotation_list(n, 16, rng)
    th = rng.uniform(-3, 3, len(rots))
    hterms = _random_terms(n, 9, rng)
    hc = rng.normal(size=len(hterms))
    sv = Q.StateVec.from_host(v, ctx=ctx)
    sv.scale_(z)
    e, g = sv.pauli_rot_grad(rots, th, hterms, hc)
    we, wg = _grad_oracle(n, rots, th, hterms, hc, z * v)
    _check([e], [we], _gtol(z * v, hc))
    _check(g, wg, _gtol(z * v, hc))
    e1, g1 = Q.StateVec.from_host(v, ctx=ctx).pauli_rot_grad(rots, th, hterms, hc)
    _check(g, g1 * abs(z) ** 2, _gtol(z * v, hc))
    want = _sum_oracle(n, hterms, hc, z * v)
    _check(sv.pauli_sum(hterms, hc).to_host(), want, 1e-12 * max(1.0, float(np.abs(want).max())) * len(hterms))


@pytest.mark.parametrize("linear", [0, 1])
def test_source_bitwise_unchanged_and_clones_valid(ctx, default_opts, linear):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 13
    rng = np.random.default_rng(2600 + linear)
    v = S.gen_state(n, rng)
    ctx.set_option("linear", linear)
    src = Q.StateVec.from_host(v, ctx=ctx)
    src.submit([("U", 3, H), ("CX", 3, 7)])  # pending in the lineage
    v1 = S.run_ops(n, [("U", 3, H), ("CX", 3, 7)], v)
    clone = src.clone()
    rots = _rotation_list(n, 20, rng)
    th = rng.uniform(-3, 3, len(rots))
    hterms = _random_terms(n, 10, rng)
    hc = rng.normal(size=len(hterms))
    r1 = src.pauli_rot_grad(rots, th, hterms, hc)
    r2 = clone.pauli_rot_grad(rots, th, hterms, hc)
    out = src.pauli_sum(hterms, hc)
    assert r1[0] == r2[0] and r1[1].tobytes() == r2[1].tobytes()
    we, wg = _grad_oracle(n, rots, th, hterms, hc, v1)
    _check(r1[1], wg, _gtol(v1, hc))
    # the same value through the same kernels, never passed to the new calls
    got = src.to_host()
    assert got.tobytes() == Q.StateVec.from_host(v, ctx=ctx).submit([("U", 3, H), ("CX", 3, 7)]).to_host().tobytes()
    assert clone.to_host().tobytes() == got.tobytes()
    _check(out.to_host(), _sum_oracle(n, hterms, hc, v1), 1e-11)
    # a second gradient on the same source: the first left it untouched bit for bit
    assert src.pauli_rot_grad(rots, th, hterms, hc)[1].tobytes() == r1[1].tobytes()
    assert src.to_host().tobytes() == got.tobytes()


def test_deterministic(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 18
    rng = np.random.default_rng(2700)
    v = S.gen_state(n, rng, normalized=False)
    rots = _rotation_list(n, 90, rng)
    th = rng.uniform(-3, 3, len(rots))
    hterms = _random_terms(n, 70, rng)
    hc = rng.normal(size=len(hterms))
    res = [Q.StateVec.from_host(v, ctx=ctx).pauli_rot_grad(rots, th, hterms, hc) for _ in range(2)]
    assert res[0][0] == res[1][0] and res[0][1].tobytes() == res[1][1].tobytes()
    outs = [Q.StateVec.from_host(v, ctx=ctx).pauli_sum(hterms, hc).to_host() for _ in range(2)]
    assert outs[0].tobytes() == outs[1].tobytes()


def test_launch_counts_on_a_tfim_chain(ctx):
    """Forward launches F (the rotation cut), sum launches S (the term cut), backward launches F again: the
    gradient costs 2F + S tile launches and F + S second stages."""
    import qubism_b200 as Q
    from oracle import structured as S
    n = 16
    rng = np.random.default_rng(2800)
    v = S.gen_state(n, rng)
    zz = ["I" * q + "ZZ" + "I" * (n - q - 2) for q in range(n - 1)]
    xs = ["I" * q + "X" + "I" * (n - q - 1) for q in range(n)]
    rots = (zz + xs) * 2
    th = rng.uniform(-1, 1, len(rots))
    hterms, hc = zz + xs, np.concatenate([np.ones(n - 1), np.full(n, 0.7)])
    sv = Q.StateVec.from_host(v, ctx=ctx)
    ctx.reset_stats()
    Q.StateVec.from_host(v, ctx=ctx).pauli_rot_(rots, th).flush()
    F = ctx.stats()["simple_launches"]
    ctx.reset_stats()
    sv.pauli_sum(hterms, hc)
    S_ = ctx.stats()["simple_launches"]
    assert ctx.stats()["reduce_launches"] == 0
    # rotations: the ZZ and X on qubits 0..8 (bits 15..7, with the three low bits 12), then X on qubits 9..15,
    # the second layer's ZZ and X on qubits 0..4, then X on qubits 5..15.  Terms sorted by X mask: the ZZ and X
    # on bits 0..11, then X on bits 12..15
    assert (F, S_) == (3, 2)
    ctx.reset_stats()
    e, g = sv.pauli_rot_grad(rots, th, hterms, hc)
    st = ctx.stats()
    assert st["simple_launches"] == 2 * F + S_ and st["reduce_launches"] == F + S_
    we, wg = _grad_oracle(n, rots, th, hterms, hc, v)
    _check(g, wg, _gtol(v, hc))


def test_rejected_calls_leave_the_state_untouched(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200 import capi
    n = 14
    rng = np.random.default_rng(2900)
    v = S.gen_state(n, rng)
    sv = Q.StateVec.from_host(v, ctx=ctx)
    ops = [("U", 2, H), ("CX", 2, 5)]
    sv.submit(ops)
    ok = ["XZ" + "I" * 12]
    bad_rot = [(["X" * 13 + "I"], [0.1], capi.QB_ERR_UNSUPPORTED), (ok, [np.inf], capi.QB_ERR_ARG),
               ([(1 << n, 0)], [0.1], capi.QB_ERR_ARG)]
    bad_h = [(["Y" * 13 + "I"], [1.0], capi.QB_ERR_UNSUPPORTED), (ok, [np.nan], capi.QB_ERR_ARG),
             ([(0, 1 << n)], [1.0], capi.QB_ERR_ARG)]
    for terms, th, code in bad_rot:
        with pytest.raises(capi.QbError) as e:
            sv.pauli_rot_grad(terms, th, ok, [1.0])
        assert e.value.code == code
    for terms, hc, code in bad_h:
        with pytest.raises(capi.QbError) as e:
            sv.pauli_rot_grad(ok, [0.3], terms, hc)
        assert e.value.code == code
        with pytest.raises(capi.QbError) as e:
            sv.pauli_sum(terms, np.asarray(hc, dtype=complex))
        assert e.value.code == code
    with pytest.raises(capi.QbError) as e:
        sv.pauli_sum(ok, [complex(1.0, np.inf)])
    assert e.value.code == capi.QB_ERR_ARG
    want = S.run_ops(n, ops, v)
    _check(sv.to_host(), want, _vtol(want))
    wide = ["X" * 12 + "II"]  # the widest string the tile holds
    e, g = sv.pauli_rot_grad(wide, [0.5], wide + ok, [1.0, -0.5])
    we, wg = _grad_oracle(n, wide, [0.5], wide + ok, [1.0, -0.5], want)
    _check(g, wg, _gtol(want, [1.0, 0.5]))


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
    """X / Y on global qubits swap them into the shard (the second state follows); Z on global qubits is a
    per-rank sign.  Every rank gets the single-GPU energy and gradient."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import random_layers
    ctxs = groups(P)
    pbits = P.bit_length() - 1
    L = n - pbits
    rng = np.random.default_rng(3000 + P + n)
    full = S.gen_state(n, rng)
    ops = random_layers(n, 2, seed=n)
    w = min(12, L)
    rots = _rotation_list(n, 30, rng, max_x=w) + ["X" * pbits + "I" * (n - pbits), "Y" * (pbits + 1) + "Z" * (n - pbits - 1)]
    rots += ["X" * w + "I" * (n - w)]
    th = rng.uniform(-3, 3, len(rots))
    hterms = _random_terms(n, 12, rng, max_x=w) + ["X" * pbits + "Z" * (n - pbits), "Z" * n, "I" * (n - 1) + "X"]
    hc = rng.normal(size=len(hterms))
    start = S.run_ops(n, ops, full)
    one = Q.StateVec.from_host(full, ctx=ctx)
    one.submit(ops)
    e1, g1 = one.pauli_rot_grad(rots, th, hterms, hc)
    we, wg = _grad_oracle(n, rots, th, hterms, hc, start)
    tol = _gtol(start, hc)
    _check(g1, wg, tol)
    cs = rng.normal(size=len(hterms)) + 1j * rng.normal(size=len(hterms))
    hsum = _sum_oracle(n, hterms, cs, start)

    def work(r, c):
        sv = Q.StateVec.from_host(full[r << L:(r + 1) << L], n=n, ctx=c)
        sv.submit(ops)
        e, g = sv.pauli_rot_grad(rots, th, hterms, hc)
        out = sv.pauli_sum(hterms, cs)
        return e, g, out.to_host(), sv.to_host()

    for e, g, out, amps in run_group(ctxs, work):
        _check([e], [e1], tol)
        _check(g, g1, tol)
        _check(out, hsum, 1e-12 * max(1.0, float(np.abs(hsum).max())) * len(hterms))
        _check(amps, start, _vtol(start))


def test_virtual_ranks_reject_a_term_wider_than_the_shard(groups):
    import qubism_b200 as Q
    from qubism_b200 import capi
    ctxs = groups(8)
    n = 8  # 5 local qubits

    def work(r, c):
        sv = Q.StateVec.from_host(np.full(1 << 5, 0.1, dtype=complex), n=n, ctx=c)
        codes = []
        for call in (lambda: sv.pauli_rot_grad(["Z" * n], [0.1], ["X" * 6 + "II"], [1.0]),
                     lambda: sv.pauli_sum(["X" * 6 + "II"], [1.0])):
            try:
                call()
                codes.append(0)
            except capi.QbError as e:
                codes.append(e.code)
        return codes, sv.local_to_host().tobytes() == np.full(1 << 5, 0.1, dtype=complex).tobytes()

    assert run_group(ctxs, work) == [([capi.QB_ERR_UNSUPPORTED] * 2, True)] * 8


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_gradients_over_nccl(world):
    """One process per GPU (torchrun): scripts/pauli_grad_dist_check.py.  Skipped on a box with fewer GPUs."""
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
                          os.path.join(root, "scripts", "pauli_grad_dist_check.py")], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0 and "PAULI GRAD DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
