"""Lanczos ground states of Pauli sums (qb_pauli_ground) on the device: against the Lanczos oracle
(tests/pauli_ground_oracle.py, pinned to numpy's eigh in tests/test_pauli_ground_cpu.py) and the dense minimum
at n <= 12, against the exact free-fermion energy of Ising chains at 26 and 30 qubits, the Ritz vector's true
residual, Heisenberg chains, symmetry sectors, pending scalars, layouts, lazy clones, launch counts, rejected
calls and virtual ranks."""
import ctypes as C

import numpy as np
import pytest

from conftest import note_error
from vrank import run_group

pytestmark = pytest.mark.gpu

BREAKDOWN = 2.0 ** -40


def _check(got, want, tol):
    err = float(np.abs(np.asarray(got) - np.asarray(want)).max()) if np.size(want) else 0.0
    note_error(err, tol)
    assert err <= tol, (err, tol)


def _masks(terms, n):
    from qubism_b200.statevec import pauli_masks
    return pauli_masks(terms, n)


def _ground(sv, terms, coefs, tol, maxiter=2000, vector=0):
    """qb_pauli_ground through the C ABI: (energy, resid, m, alpha[:m], beta[:m])."""
    from qubism_b200 import capi
    xs, zs = _masks(terms, sv.n)
    cf = np.ascontiguousarray(coefs, dtype=np.float64)
    al, be = np.full(maxiter, -7.0), np.full(maxiter, -7.0)
    e, res, m = C.c_double(), C.c_double(), C.c_int64(-1)
    P64, PD = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
    capi.check(sv.ctx.L.qb_pauli_ground(sv._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64), cf.ctypes.data_as(PD),
                                        len(xs), float(tol), maxiter, vector, C.byref(e), C.byref(res), C.byref(m),
                                        al.ctypes.data_as(PD), be.ctypes.data_as(PD)))
    k = m.value
    assert (al[k:] == 0).all() and (be[k:] == 0).all()
    return e.value, res.value, k, al[:k], be[:k]


def _oracle(n, terms, coefs, v, tol, maxiter=2000, vector=False):
    from pauli_ground_oracle import ground
    xs, zs = _masks(terms, n)
    return ground(n, xs, zs, coefs, v, tol, maxiter, vector)


def _r(terms, coefs):
    from pauli_evolve_oracle import merge
    xs, zs = _masks(terms, len(terms[0]))
    return sum(abs(h) for _, _, h in merge(xs, zs, coefs)[1])


def _sparse_h(n, terms, coefs):
    import scipy.sparse as sp
    from pauli_grad_oracle import pauli_apply
    xs, zs = _masks(terms, n)
    N = 1 << n
    H = sp.csr_matrix((N, N), dtype=complex)
    j = np.arange(N)
    for x, z, h in zip(xs, zs, coefs):
        col = pauli_apply(n, int(x), int(z), np.ones(N, dtype=complex))  # (P 1)_i = phase_i, from index i ^ x'
        xb = sum(1 << (n - 1 - q) for q in range(n) if (int(x) >> q) & 1)
        H = H + h * sp.csr_matrix((col, (j, j ^ xb)), shape=(N, N))
    return H


def _min_eig(n, terms, coefs):
    H = _sparse_h(n, terms, coefs)
    if n <= 8:
        return float(np.linalg.eigvalsh(H.toarray())[0])
    import scipy.sparse.linalg as sl
    return float(sl.eigsh(H, k=1, which="SA", tol=1e-14, ncv=40)[0][0])


def _random_terms(n, k, rng, max_x=12):
    terms = []
    while len(terms) < k:
        s = "".join(rng.choice(list("IXYZ"), n, p=[0.7, 0.1, 0.1, 0.1] if n > 8 else None))
        if sum(ch in "XY" for ch in s) <= max_x:
            terms.append(s)
    return terms


def _one(n, q, p):
    return "I" * q + p + "I" * (n - q - len(p))


def _tfim(n, rng):
    """Open Ising chain -sum J_i Z_i Z_{i+1} - sum g_i X_i with random J, g and its free-fermion ground energy.  The
    field is the larger (g > J everywhere): a gapped chain, so that Lanczos needs tens of steps at 30 qubits and not
    the thousands a disordered critical chain's tiny gaps would take."""
    J, g = rng.uniform(0.3, 0.8, n - 1), rng.uniform(1.0, 1.5, n)
    terms = [_one(n, q, "ZZ") for q in range(n - 1)] + [_one(n, q, "X") for q in range(n)]
    coefs = np.concatenate([-J, -g])
    exact = -float(np.linalg.svd(np.diag(g) + np.diag(J, 1), compute_uv=False).sum())
    return terms, coefs, exact


def _heisenberg(n):
    terms = [_one(n, q, p) for q in range(n - 1) for p in ("XX", "YY", "ZZ")]
    return terms, np.ones(len(terms))


def _product_state(n, rng, ctx):
    import qubism_b200 as Q
    return Q.mkStateVec(n, ctx).pauli_rot_([_one(n, q, "Y") for q in range(n)], rng.uniform(0.3, 2.8, n)).flush()


@pytest.mark.parametrize("n", list(range(1, 13)))
def test_parity_with_the_oracle(ctx, n):
    """Random sums with identity strings, duplicates and X on a collapsed qubit: alpha and beta of the first steps,
    the step count, and the energy against the true minimum."""
    import qubism_b200 as Q
    from oracle import structured as S
    rng = np.random.default_rng(9000 + n)
    terms = _random_terms(n, 10 + n, rng) + ["I" * n, "I" * n, "Z" * n, _one(n, 0, "X"), _one(n, 0, "X")]
    coefs = rng.normal(size=len(terms))
    r = _r(terms, coefs)
    lam = _min_eig(n, terms, coefs)
    v = S.gen_state(n, rng, normalized=False) * 1.7
    starts = [(Q.StateVec.from_host(v, ctx=ctx), v)]
    if n > 1:  # qubit 0 collapsed: known, and X on it
        starts.append((Q.StateVec.from_host(v, ctx=ctx).collapse_(0, 1), S.collapse(n, 0, 1, v)))
    tol = 0.0 if n <= 2 else 1e-10 * r
    for sv, start in starts:
        e, res, m, al, be = _ground(sv, terms, coefs, tol)
        we, wres, wm, wal, wbe, _ = _oracle(n, terms, coefs, start, tol)
        assert abs(m - wm) <= 1, (m, wm)
        k = min(m, wm, 20, max(1, (1 << n) // 2))  # (as the Krylov space nears 2^n, beta is rounding noise)
        _check(al[:k], wal[:k], 1e-12 * r)
        _check(be[:k], wbe[:k], 1e-12 * r)
        _check([e], [lam], 1e-10 * r)
        if n <= 2:
            assert m <= 1 << n and be[-1] <= BREAKDOWN * r and res <= BREAKDOWN * r
        else:
            assert res <= tol
    e2, x = Q.pauliGround(terms, coefs, Q.StateVec.from_host(v, ctx=ctx), 1e-10 * r)
    _check([e2], [lam], 1e-10 * r)
    _check([x.norm2()], [1.0], 1e-13)


@pytest.mark.parametrize("n", [26, 30])
def test_ising_chain_free_fermion_energy(ctx, n):
    rng = np.random.default_rng(9100 + n)
    terms, coefs, exact = _tfim(n, rng)
    r = float(np.abs(coefs).sum())
    sv = _product_state(n, rng, ctx)
    e, res, m, al, be = _ground(sv, terms, coefs, 1e-10 * r, 1000)
    assert res <= 1e-10 * r and m < 1000, (res, m)
    _check([e], [exact], 1e-10 * r)


def test_ritz_vector_at_26_qubits(ctx):
    """x has norm 1, <s|x> > 0, its true residual ||Hx - theta x|| is the estimate, <x|H|x> = theta, and the
    energy-only run gives the same alpha, beta and energy bit for bit."""
    n = 26
    rng = np.random.default_rng(9200)
    terms, coefs, exact = _tfim(n, rng)
    r = float(np.abs(coefs).sum())
    s = _product_state(n, rng, ctx).scale_(0.8)
    before = s.local_to_host(0, 4096).tobytes()
    a = _ground(s, terms, coefs, 1e-8 * r, 1000)
    assert s.local_to_host(0, 4096).tobytes() == before  # (energy only: s unchanged)
    x = s.clone()
    b = _ground(x, terms, coefs, 1e-8 * r, 1000, vector=1)
    assert a[2] == b[2] and a[0] == b[0] and a[1] == b[1]
    assert a[3].tobytes() == b[3].tobytes() and a[4].tobytes() == b[4].tobytes()
    e, res = b[0], b[1]
    _check([x.norm2()], [1.0], 1e-13)
    ov = s.inner(x)
    assert ov.real > 0 and abs(ov.imag) <= 1e-13
    hx = x.pauli_sum(terms, coefs)
    hx.axpy_(-e, x)
    true = hx.norm2()
    note_error(abs(true - res), 1e-3 * res + 1e-12 * r)
    assert abs(true - res) <= 1e-3 * res + 1e-12 * r, (true, res)
    _check([float(np.dot(coefs, x.expect_pauli(terms)))], [e], 1e-10 * r)
    _check([e], [exact], 1e-10 * r)


def test_heisenberg_chain(ctx):
    """|0...0> is an eigenvector (m = 1, beta exactly 0); from a Neel state at 26 qubits the energy lies below the
    Neel energy and below what a few steps of VQE with adjoint gradients reach."""
    import qubism_b200 as Q
    n = 12
    terms, coefs = _heisenberg(n)
    sv = Q.mkStateVec(n, ctx)
    e, res, m, al, be = _ground(sv, terms, coefs, 1e-10, vector=1)
    assert m == 1 and be[0] == 0.0 and res == 0.0 and e == n - 1 and al[0] == n - 1
    want = np.zeros(1 << n, dtype=complex)
    want[0] = 1.0
    assert sv.to_host().tobytes() == want.tobytes()
    n = 26
    terms, coefs = _heisenberg(n)
    odd = [_one(n, q, "X") for q in range(1, n, 2)]
    s = Q.mkStateVec(n, ctx).pauli_rot_(odd, np.full(len(odd), np.pi)).flush()  # (-i X on every odd qubit: Neel)
    e_neel = float(np.dot(coefs, s.expect_pauli(terms)))
    assert abs(e_neel + (n - 1)) <= 1e-12
    bonds = [_one(n, q, "XY") for q in range(n - 1)]  # real exchange between the two spins of a bond
    th = np.full(len(bonds), 0.1)
    vqe = []
    for _ in range(6):
        ev, g = s.pauli_rot_grad(bonds, th, terms, coefs)
        vqe.append(ev)
        th = th - 0.1 * g
    e, res, m, al, be = _ground(s, terms, coefs, 1e-6 * 3 * (n - 1), 400)
    assert e < min(vqe) - 1.0 and e < e_neel - 1.0
    assert e >= -3.0 * (n - 1)  # (no bond goes below -3)


@pytest.mark.parametrize("n", [6, 10])
def test_symmetry_sectors(ctx, n):
    """From a start state of parity -1 (prod X) under the Ising chain the answer is the odd sector's minimum."""
    import qubism_b200 as Q
    from oracle import structured as S
    from pauli_grad_oracle import pauli_apply
    rng = np.random.default_rng(9300 + n)
    terms, coefs, exact = _tfim(n, rng)
    r = float(np.abs(coefs).sum())
    Hd = _sparse_h(n, terms, coefs).toarray()
    allx = (1 << n) - 1
    for sign in (1, -1):
        P = np.stack([pauli_apply(n, allx, 0, c) for c in np.eye(1 << n, dtype=complex)], axis=1)
        proj = 0.5 * (np.eye(1 << n) + sign * P)
        ev, U = np.linalg.eigh(proj)
        B = U[:, ev > 0.5]
        want = float(np.linalg.eigvalsh(B.conj().T @ Hd @ B)[0])
        v = proj @ S.gen_state(n, rng)
        sv = Q.StateVec.from_host(v, ctx=ctx)
        e, res, m, al, be = _ground(sv, terms, coefs, 1e-10 * r, vector=1)
        _check([e], [want], 1e-10 * r)
        x = sv.to_host()
        _check(P @ x, sign * x, 1e-9)
    assert abs(want - exact) > 1e-3  # (the odd sector's minimum is not the ground energy)


def test_pending_scalars(ctx):
    """A positive real scalar leaves the vector as it is; a phase rotates it."""
    import qubism_b200 as Q
    from oracle import structured as S
    n = 11
    rng = np.random.default_rng(9400)
    v = S.gen_state(n, rng)
    terms = _random_terms(n, 12, rng) + ["I" * n]
    coefs = rng.normal(size=len(terms))
    r = _r(terms, coefs)
    base = Q.StateVec.from_host(v, ctx=ctx)
    e0, _, m0, _, _ = _ground(base, terms, coefs, 1e-10 * r, vector=1)
    x0 = base.to_host()
    for z in (3.5, 0.7 - 1.9j):
        sv = Q.StateVec.from_host(v, ctx=ctx).scale_(z)
        e, res, m, al, be = _ground(sv, terms, coefs, 1e-10 * r, vector=1)
        _check([e], [e0], 1e-10 * r)
        _check(sv.to_host(), (z / abs(z)) * x0, 1e-6)
    want = _oracle(n, terms, coefs, v, 1e-10 * r, vector=True)[5]
    _check(x0, want, 1e-6)


OPTION_SETS = [dict(oop=0), dict(oop=1), dict(fuse=0), dict(tile_bits=10)]


@pytest.mark.parametrize("opts", OPTION_SETS, ids=lambda o: ",".join(f"{k}={v}" for k, v in o.items()))
def test_planner_options_and_permuted_layouts(ctx, default_opts, opts):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import qft_ops, random_mixed
    for k, val in opts.items():
        ctx.set_option(k, val)
    n = 14
    rng = np.random.default_rng(9500 + len(str(opts)))
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
    r = _r(terms, coefs)
    e, res, m, al, be = _ground(sv, terms, coefs, 1e-10 * r, vector=1)
    we, _, wm, wal, wbe, wx = _oracle(n, terms, coefs, v, 1e-10 * r, vector=True)
    assert abs(m - wm) <= 1
    _check([e], [we], 1e-10 * r)
    _check(sv.to_host(), wx, 1e-6)
    sv.submit([("U", 4, np.array([[1, 1], [1, -1]]) / np.sqrt(2))])  # the Ritz vector goes on like any other state
    _check([sv.norm2()], [1.0], 1e-13)


@pytest.mark.parametrize("linear", [0, 1])
def test_lazy_clones_and_linear(ctx, default_opts, linear):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200 import capi
    n = 13
    rng = np.random.default_rng(9600 + linear)
    v = S.gen_state(n, rng)
    ops = [("U", 3, np.array([[1, 1], [1, -1]]) / np.sqrt(2)), ("CX", 3, 7)]
    ctx.set_option("linear", linear)
    base = Q.StateVec.from_host(v, ctx=ctx).submit(ops).to_host()
    terms = _random_terms(n, 12, rng)
    coefs = rng.normal(size=len(terms))
    r = _r(terms, coefs)
    # energy only: s and its clones keep their values, also with "linear"
    src = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    clone = src.clone()
    e, *_ = _ground(src, terms, coefs, 1e-10 * r)
    assert src.to_host().tobytes() == base.tobytes() and clone.to_host().tobytes() == base.tobytes()
    # the vector: in place; clones keep the old value, or are consumed with "linear"
    src = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    clone = src.clone()
    ev, *_ = _ground(src, terms, coefs, 1e-10 * r, vector=1)
    assert ev == e
    want = _oracle(n, terms, coefs, S.run_ops(n, ops, v), 1e-10 * r, vector=True)[5]
    _check(src.to_host(), want, 1e-6)
    if linear:
        with pytest.raises(capi.QbError) as exc:
            clone.to_host()
        assert exc.value.code == capi.QB_ERR_STATE
    else:
        assert clone.to_host().tobytes() == base.tobytes()
    pure = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    e2, x = Q.pauliGround(terms, coefs, pure, 1e-10 * r)
    assert e2 == e and x.to_host().tobytes() == src.to_host().tobytes()
    if not linear:
        assert pure.to_host().tobytes() == base.tobytes()


def test_launch_counts_determinism_and_cheap_cases(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    n = 16
    rng = np.random.default_rng(9700)
    v = S.gen_state(n, rng)
    terms, coefs, _ = _tfim(n, rng)
    extra = [s for s in dict.fromkeys(_random_terms(n, 70, rng)) if s != "I" * n and s not in terms]
    for tt, cc in ((terms, coefs), (terms + extra, np.concatenate([coefs, 0.1 * rng.normal(size=len(extra))]))):
        r = float(np.abs(cc).sum())
        ctx.reset_stats()
        Q.StateVec.from_host(v, ctx=ctx).pauli_sum(tt, cc)
        L = ctx.stats()["simple_launches"]
        outs = []
        for vector in (0, 0, 1, 1):
            sv = Q.StateVec.from_host(v, ctx=ctx)
            ctx.reset_stats()
            e, res, m, al, be = _ground(sv, tt + ["I" * n], np.append(cc, 0.3), 1e-9 * r, vector=vector)
            st = ctx.stats()
            steps = m + (m - 1 if vector else 0)
            assert st["simple_launches"] == steps * (L + 1), (st, m, L)
            assert st["reduce_launches"] == 2 * m + 2 + (2 if vector else 0), (st, m)
            outs.append((e, res, m, al.tobytes(), be.tobytes(), sv.to_host().tobytes() if vector else b""))
        assert outs[0] == outs[1] and outs[2] == outs[3] and outs[0][:5] == outs[2][:5]
    # identity strings only (or no terms): energy = c, no step, one norm sweep; the vector is s / ||s||
    w = 2.0 * v
    for tt, cc, c in ((["I" * n, "I" * n], [0.4, 0.9], 0.4 + 0.9), ([], [], 0.0), ([_one(n, 2, "X")] * 2, [1.0, -1.0], 0.0)):
        for vector in (0, 1):
            sv = Q.StateVec.from_host(w, ctx=ctx)
            ctx.reset_stats()
            e, res, m, al, be = _ground(sv, tt, cc, 1e-9, vector=vector)
            st = ctx.stats()
            assert (e, res, m) == (c, 0.0, 0) and st["simple_launches"] == 0 and st["reduce_launches"] == 2
            _check(sv.to_host(), v if vector else w, 1e-15)


def test_rejected_calls_leave_the_state_untouched(ctx):
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200 import capi
    n = 14
    rng = np.random.default_rng(9800)
    v = S.gen_state(n, rng)
    ops = [("U", 2, np.array([[1, 1], [1, -1]]) / np.sqrt(2)), ("CX", 2, 5)]
    ref = Q.StateVec.from_host(v, ctx=ctx).submit(ops).to_host()
    sv = Q.StateVec.from_host(v, ctx=ctx).submit(ops)
    ok = ["XZ" + "I" * 12]
    bad = [(["X" * 13 + "I"], [0.1], 1e-8, 10, capi.QB_ERR_UNSUPPORTED), (ok, [np.inf], 1e-8, 10, capi.QB_ERR_ARG),
           (ok, [np.nan], 1e-8, 10, capi.QB_ERR_ARG), ([(1 << n, 0)], [0.1], 1e-8, 10, capi.QB_ERR_ARG),
           ([(0, 1 << n)], [0.1], 1e-8, 10, capi.QB_ERR_ARG), (ok, [1.0], np.nan, 10, capi.QB_ERR_ARG),
           (ok, [1.0], -1e-3, 10, capi.QB_ERR_ARG), (ok, [1.0], 1e-8, 0, capi.QB_ERR_ARG),
           (ok, [1.0], 1e-8, 65537, capi.QB_ERR_ARG)]
    ctx.reset_stats()
    for terms, coefs, tol, maxiter, code in bad:
        with pytest.raises(capi.QbError) as e:
            _ground(sv, terms, coefs, tol, maxiter)
        assert e.value.code == code, (terms, coefs, tol, maxiter)
    st = ctx.stats()
    assert st["simple_launches"] == 0 and st["passes"] == 0 and st["reduce_launches"] == 0  # still queued
    assert sv.to_host().tobytes() == ref.tobytes()
    for start in (Q.StateVec.from_host(np.zeros(1 << n, dtype=complex), ctx=ctx),
                  Q.StateVec.from_host(v, ctx=ctx).scale_(0.0)):
        before = start.local_to_host().tobytes()
        ctx.reset_stats()
        with pytest.raises(capi.QbError) as e:
            _ground(start, ok, [1.0], 1e-8, 10, vector=1)
        assert e.value.code == capi.QB_ERR_ARG
        assert ctx.stats()["simple_launches"] == 0 and start.local_to_host().tobytes() == before
    e, res, m, al, be = _ground(sv, ok, [1.0], 0.0, 10)
    assert abs(e + 1.0) <= 1e-14 and m <= 2


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


@pytest.mark.parametrize("P,n", [(2, 12), (4, 13), (8, 12)])
def test_virtual_ranks(ctx, groups, P, n):
    """X / Y on global qubits swap them into the shard (the other states follow); every rank receives the
    single-GPU energy, coefficients and Ritz vector."""
    import qubism_b200 as Q
    from oracle import structured as S
    from qubism_b200.circuits import random_layers
    ctxs = groups(P)
    pbits = P.bit_length() - 1
    L = n - pbits
    rng = np.random.default_rng(9900 + P + n)
    full = S.gen_state(n, rng)
    ops = random_layers(n, 2, seed=n)
    w = min(12, L)
    terms = _random_terms(n, 14, rng, max_x=w) + ["X" * pbits + "Z" * (n - pbits), "Z" * n, "I" * (n - 1) + "X"]
    terms += ["Y" * w + "I" * (n - w), "I" * n]
    coefs = rng.normal(size=len(terms))
    r = _r(terms, coefs)
    one = Q.StateVec.from_host(full, ctx=ctx).submit(ops)
    e1, res1, m1, al1, be1 = _ground(one, terms, coefs, 1e-10 * r, vector=1)
    single = one.to_host()

    def work(rk, c):
        sv = Q.StateVec.from_host(full[rk << L:(rk + 1) << L], n=n, ctx=c)
        sv.submit(ops)
        out = _ground(sv, terms, coefs, 1e-10 * r, vector=1)
        return out, sv.to_host()

    res = run_group(ctxs, work)
    for (e, rs, m, al, be), amps in res:
        assert abs(m - m1) <= 1 and m == res[0][0][2]
        assert e == res[0][0][0]  # every rank alike
        k = min(m, m1, 20)
        _check(al[:k], al1[:k], 1e-12 * r)
        _check(be[:k], be1[:k], 1e-12 * r)
        _check([e], [e1], 1e-10 * r)
        _check(amps, single, 1e-6)


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_ground_state_over_nccl(world):
    """One process per GPU (torchrun): scripts/pauli_ground_dist_check.py.  Skipped on a box with fewer GPUs."""
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
                          os.path.join(root, "scripts", "pauli_ground_dist_check.py")], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0 and "PAULI GROUND DIST CHECK PASSED" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
