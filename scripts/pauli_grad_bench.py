"""Adjoint gradients of Pauli-sum energies on a 30-qubit state: qb_pauli_rot_grad against one energy evaluation
and against the parameter-shift rule, qb_pauli_sum alone, and the per-launch times of the two new kernels.

    python scripts/pauli_grad_bench.py [--n 30] [--reps 3] [--warmup 1] --out FILE.json

Hamiltonians: the Heisenberg chain (XX, YY, ZZ on every bond: 87 terms at n = 30) and the transverse-field
Ising chain (ZZ on every bond, X on every qubit: 59 terms).  Ansatz: 1 and 2 layers of the matching Trotter
step (one rotation per term and layer, seeded random angles), so K = 87 / 174 and 59 / 118 angles.

- energy_eval_ms: one energy evaluation as an optimiser without gradients makes it: clone, the K rotations,
  expect_pauli over H.  The parameter-shift gradient is 2K such evaluations: param_shift_ms is 2K times
  that measured time (the 2K evaluations themselves are not run).
- pauli_sum_ms: H psi alone (qb_pauli_sum, a new state).
- grad_ms: qb_pauli_rot_grad (energy and all K components).
Each state (16 GiB at n = 30) is far larger than the L2, so every sweep reads and writes HBM.  Times are host
clocks around `reps` calls that end in a device synchronise, after `warmup` calls of the same workload.

Kernel times come from a separate profiled run (torch.profiler, CUDA activities) of one gradient per
Hamiltonian: the mean time per launch of k_pauli_sum_tile, k_pauli_rot_adjoint_tile and k_pauli_rot_tile,
and the bytes each launch must move over that time (sum: read psi, write H psi, later launches also read it;
adjoint: read and write psi and lam).  For scale: a qb_norm2 sweep (one state read) and a qb_axpy sweep (two
states read, one written) of the same size, host-timed."""
import argparse
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


def hamiltonians(n):
    def s(ch_at):
        t = ["I"] * n
        for q, ch in ch_at:
            t[q] = ch
        return "".join(t)
    heis = [s([(q, p), (q + 1, p)]) for q in range(n - 1) for p in "XYZ"]
    tfim = [s([(q, "Z"), (q + 1, "Z")]) for q in range(n - 1)] + [s([(q, "X")]) for q in range(n)]
    return {"heisenberg": (heis, np.ones(len(heis))),
            "tfim": (tfim, np.concatenate([np.ones(n - 1), np.full(n, 0.8)]))}


def timed(fn, reps, warmup, ctx):
    for _ in range(warmup):
        fn()
    ctx.sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    ctx.sync()
    return (time.perf_counter() - t0) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import qubism_b200 as Q
    from qubism_b200.circuits import qft_ops, random_layers
    ctx = Q.Context.default()
    n = a.n
    state = 16 << n
    res = {"card": card(), "n": n, "state_GiB": state / 2**30, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    sv = Q.mkStateVec(n, ctx).submit(qft_ops(n) + random_layers(n, 2, seed=3)).flush()
    ctx.sync()
    res["norm2_ms"] = timed(sv.norm2, a.reps, a.warmup, ctx)
    res["norm2_read_GBps"] = state / res["norm2_ms"] / 1e6
    y = sv.clone().scale_(0.5).flush()
    res["axpy_ms"] = timed(lambda: y.axpy_(1e-3, sv), a.reps, a.warmup, ctx)
    res["axpy_GBps"] = 3 * state / res["axpy_ms"] / 1e6
    del y
    rng = np.random.default_rng(5)
    ham = hamiltonians(n)
    for name, (hterms, hc) in ham.items():
        res["pauli_sum_" + name + "_ms"] = timed(lambda: sv.pauli_sum(hterms, hc).flush(), a.reps, a.warmup, ctx)
        ctx.reset_stats()
        sv.pauli_sum(hterms, hc).flush()
        res["pauli_sum_" + name + "_launches"] = ctx.stats()["simple_launches"]
        for layers in (1, 2):
            rots = hterms * layers
            th = rng.uniform(-0.3, 0.3, len(rots))
            K = len(rots)

            def energy():
                return float(np.dot(hc, sv.clone().pauli_rot_(rots, th).expect_pauli(hterms)))

            out = {}

            def grad():
                out["eg"] = sv.pauli_rot_grad(rots, th, hterms, hc)

            e_ms = timed(energy, a.reps, a.warmup, ctx)
            g_ms = timed(grad, a.reps, a.warmup, ctx)
            ctx.reset_stats()
            grad()
            st = ctx.stats()
            e, g = out["eg"]
            w = {"angles": K, "terms": len(hterms), "energy": e, "energy_check": energy(),
                 "energy_eval_ms": e_ms, "grad_ms": g_ms, "grad_over_energy_eval": g_ms / e_ms,
                 "param_shift_ms": 2 * K * e_ms, "speedup_over_param_shift": 2 * K * e_ms / g_ms,
                 "grad_tile_launches": st["simple_launches"], "grad_second_stages": st["reduce_launches"],
                 "grad_norm": float(np.linalg.norm(g))}
            res["workloads"][f"{name}_{layers}layer"] = w
            print(name, layers, json.dumps(w), flush=True)
    # kernel times: a profiled run of its own
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for name, (hterms, hc) in ham.items():
        th = rng.uniform(-0.3, 0.3, len(hterms))
        sv.pauli_rot_grad(hterms, th, hterms, hc)
        ctx.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sv.pauli_rot_grad(hterms, th, hterms, hc)
            ctx.sync()
        for ev in prof.key_averages():
            for k in ("k_pauli_sum_tile", "k_pauli_rot_adjoint_tile", "k_pauli_rot_tile"):
                if k in ev.key:
                    us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                    d = kern.setdefault(name, {}).setdefault(k, {"launches": 0, "total_ms": 0.0})
                    d["launches"] += ev.count
                    d["total_ms"] += us / 1e3
    for name, ks in kern.items():
        for k, d in ks.items():
            d["ms_per_launch"] = d["total_ms"] / max(1, d["launches"])
            moved = {"k_pauli_sum_tile": (2 + 3 * max(0, d["launches"] - 1)) / d["launches"],
                     "k_pauli_rot_adjoint_tile": 4, "k_pauli_rot_tile": 2}[k] * state
            d["GBps"] = moved / d["ms_per_launch"] / 1e6
    res["kernels_profiled"] = kern
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "workloads"}))


if __name__ == "__main__":
    main()
