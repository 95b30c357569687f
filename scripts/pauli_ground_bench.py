"""Lanczos ground states on a 30-qubit state (qb_pauli_ground): the Krylov dimension reached, time per call and per
step, the bytes a step moves and the rate achieved, with a qb_pauli_sum and a qb_norm2 sweep of the same size for
scale.

    python scripts/pauli_ground_bench.py [--n 30] [--tol 1e-9] [--maxiter 1000] --out FILE.json

Hamiltonians: the open transverse-field Ising chain -sum J_i Z_i Z_{i+1} - sum g_i X_i (J_i in [0.3, 0.8], g_i in
[1, 1.5], seeded: 59 terms at n = 30; its exact ground energy is minus the sum of the singular values of the
bidiagonal matrix with diagonal g and superdiagonal J) from a product state, and the open Heisenberg chain (XX, YY,
ZZ on every bond, unit couplings: 87 terms) from the Neel state.  tol is relative to r = sum |h|.  Each is run
energy-only and with the Ritz vector (which runs the recurrence a second time).  Each state (16 GiB at n = 30) is
far larger than the L2, so every sweep reads and writes HBM.  Times are host clocks around one call that ends in a
device synchronise; the kernels were loaded by a qb_pauli_sum and a short call before.

Bytes per step, from the kernels' accesses, with L launches per H pass: every launch reads v_k and the old w and
writes w (48 B per amplitude); the update sweep reads v_k and w and writes w (48 B), in the vector run it also reads
and writes the Ritz vector (80 B).  Step 0 reads no old w and writes the copy of v_0 (the same 48 B in its first
launch)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def one(n, q, p):
    return "I" * q + p + "I" * (n - q - len(p))


def ground(sv, terms, coefs, tol, maxiter, vector):
    from qubism_b200 import capi
    from qubism_b200.statevec import pauli_masks
    xs, zs = pauli_masks(terms, sv.n)
    cf = np.ascontiguousarray(coefs, dtype=np.float64)
    e, res, m = C.c_double(), C.c_double(), C.c_int64()
    P64, PD = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
    capi.check(sv.ctx.L.qb_pauli_ground(sv._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64), cf.ctypes.data_as(PD),
                                        len(xs), float(tol), int(maxiter), int(vector), C.byref(e), C.byref(res),
                                        C.byref(m), None, None))
    return e.value, res.value, m.value


def timed(fn, ctx, reps=1):
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ctx.sync()
        ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.mean(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=30)
    ap.add_argument("--tol", type=float, default=1e-9)
    ap.add_argument("--maxiter", type=int, default=1000)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import qubism_b200 as Q
    ctx = Q.Context.default()
    n = a.n
    amps = 1 << n
    state = 16 * amps
    res = {"card": card(), "n": n, "state_GiB": state / 2**30, "tol_rel": a.tol, "maxiter": a.maxiter,
           "workloads": {}}
    rng = np.random.default_rng(2026)
    J, g = rng.uniform(0.3, 0.8, n - 1), rng.uniform(1.0, 1.5, n)
    tfim = ([one(n, q, "ZZ") for q in range(n - 1)] + [one(n, q, "X") for q in range(n)], np.concatenate([-J, -g]))
    tfim_exact = -float(np.linalg.svd(np.diag(g) + np.diag(J, 1), compute_uv=False).sum())
    heis = ([one(n, q, p) for q in range(n - 1) for p in ("XX", "YY", "ZZ")], np.ones(3 * (n - 1)))
    product = Q.mkStateVec(n, ctx).pauli_rot_([one(n, q, "Y") for q in range(n)], rng.uniform(0.3, 2.8, n)).flush()
    odd = [one(n, q, "X") for q in range(1, n, 2)]
    neel = Q.mkStateVec(n, ctx).pauli_rot_(odd, np.full(len(odd), np.pi)).flush()
    ctx.sync()
    res["norm2_ms"] = timed(product.norm2, ctx, 3)
    res["norm2_read_TBps"] = state / res["norm2_ms"] / 1e9
    for name, (terms, coefs), start, exact in (("tfim", tfim, product, tfim_exact), ("heisenberg", heis, neel, None)):
        r = float(np.abs(coefs).sum())
        product.pauli_sum(terms, coefs).flush()  # (loads the kernels)
        ground(start, terms, coefs, 0.0, 2, 0)
        ctx.sync()
        res[f"pauli_sum_{name}_ms"] = timed(lambda: start.pauli_sum(terms, coefs).flush(), ctx, 3)
        ctx.reset_stats()
        start.pauli_sum(terms, coefs).flush()
        L = ctx.stats()["simple_launches"]
        res[f"pauli_sum_{name}_launches"] = L
        for vector in (0, 1):
            w = start.clone()
            out = {}
            ctx.reset_stats()
            ms = timed(lambda: out.update(zip(("energy", "resid", "m"), ground(w, terms, coefs, a.tol * r, a.maxiter,
                                                                                vector))), ctx)
            st = ctx.stats()
            m = out["m"]
            steps = m + (m - 1 if vector else 0)
            step_bytes = (48 * L + 48) * amps
            total_bytes = (48 * L + 48) * m * amps + ((48 * L + 80) * (m - 1) * amps if vector else 0)
            rec = {"terms": len(terms), "r": r, "energy": out["energy"], "resid": out["resid"], "m": m,
                   "steps_run": steps, "launches_per_step": (st["simple_launches"] / steps) if steps else 0.0,
                   "reduce_launches": st["reduce_launches"], "call_ms": ms, "step_ms": ms / max(1, steps),
                   "bytes_per_energy_step_GB": step_bytes / 1e9, "achieved_TBps": total_bytes / ms / 1e9}
            if exact is not None:
                rec["exact_energy"] = exact
                rec["energy_error_over_r"] = abs(out["energy"] - exact) / r
            if vector:
                rec["norm_of_vector"] = w.norm2()
                rec["expect_H_of_vector"] = float(np.dot(coefs, w.expect_pauli(terms)))
            res["workloads"][f"{name}_{'vector' if vector else 'energy'}"] = rec
            print(name, vector, json.dumps(rec), flush=True)
            del w
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "workloads"}))


if __name__ == "__main__":
    main()
