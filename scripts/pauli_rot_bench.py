"""Trotter steps of Pauli rotations on a 30-qubit state: qb_apply_pauli_rot against the same evolution
decomposed into existing gates (basis changes, CX ladder, diagonal gate, ladder back) through qb_submit,
and against a qb_norm2 sweep of the same state for scale.

    python scripts/pauli_rot_bench.py [--n 30] [--reps 5] [--warmup 6] --out FILE.json

Workloads (one Trotter step each): a transverse-field Ising chain (ZZ on every bond, then X on every
qubit), a Heisenberg chain (XX, YY, ZZ on every bond) and a QAOA-style cost layer (ZZ on 3n random
edges, Z only).  Each state (16 GiB at n = 30) is far larger than the L2, so every sweep reads and writes
HBM.  Times are host clocks around `reps` steps that end in a device synchronise, after `warmup` steps of
the same workload (the decomposed route needs them: its repeated pass structures are compiled by NVRTC
on their second sighting).  Both routes run the same number of steps from the same state; the largest
|native - decomposed| is taken over a seeded sample of amplitudes."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

R2 = 1 / np.sqrt(2)
H = np.array([[R2, R2], [R2, -R2]], dtype=complex)
BASIS = {"X": H, "Y": H @ np.diag([1, -1j])}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def workloads(n, rng, dt=0.05):
    def s(ch_at):
        t = ["I"] * n
        for q, ch in ch_at:
            t[q] = ch
        return "".join(t)
    tfim = [s([(q, "Z"), (q + 1, "Z")]) for q in range(n - 1)] + [s([(q, "X")]) for q in range(n)]
    heis = [s([(q, p), (q + 1, p)]) for q in range(n - 1) for p in "XYZ"]
    edges = set()
    while len(edges) < 3 * n:
        a, b = sorted(int(x) for x in rng.choice(n, 2, replace=False))
        edges.add((a, b))
    qaoa = [s([(a, "Z"), (b, "Z")]) for a, b in sorted(edges)]
    return {name: (terms, rng.uniform(0.5, 1.5, len(terms)) * 2 * dt)
            for name, terms in (("tfim", tfim), ("heisenberg", heis), ("qaoa_cost", qaoa))}


def decomposed(s, theta):
    """exp(-i theta/2 P) as existing gates (the diagonal gate written out: the reference's rz is a scalar)."""
    sup = [q for q, ch in enumerate(s) if ch != "I"]
    pre = [("U", q, BASIS[s[q]]) for q in sup if s[q] != "Z"]
    post = [("U", q, BASIS[s[q]].conj().T) for q in sup if s[q] != "Z"]
    ladder = [("CX", sup[i], sup[i + 1]) for i in range(len(sup) - 1)]
    mid = [("U", sup[-1], np.diag([np.exp(-0.5j * theta), np.exp(0.5j * theta)]))]
    return pre + ladder + mid + ladder[::-1] + post


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=30)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import qubism_b200 as Q
    from qubism_b200 import capi
    from qubism_b200.circuits import qft_ops, random_layers
    ctx = Q.Context.default()
    n = a.n
    prep = qft_ops(n) + random_layers(n, 2, seed=3)
    bytes_sweep = 16 << n
    res = {"card": card(), "n": n, "state_GiB": bytes_sweep / 2**30, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    rng = np.random.default_rng(1)
    for name, (terms, thetas) in workloads(n, rng).items():
        native = Q.mkStateVec(n, ctx).submit(prep).flush()
        dec = Q.mkStateVec(n, ctx).submit(prep).flush()
        ctx.sync()
        if "norm2_ms" not in res:
            t0 = time.perf_counter()
            for _ in range(a.reps):
                native.norm2()
            res["norm2_ms"] = (time.perf_counter() - t0) * 1e3 / a.reps
            res["norm2_read_GBps"] = bytes_sweep / res["norm2_ms"] / 1e6
        ops = capi.pack_ops([op for s, th in zip(terms, thetas) for op in decomposed(s, th)])

        def run(step, sv):
            for _ in range(a.warmup):
                step()
            sv.flush()
            ctx.sync()
            ctx.reset_stats()
            t0 = time.perf_counter()
            for _ in range(a.reps):
                step()
            sv.flush()
            ctx.sync()
            ms = (time.perf_counter() - t0) * 1e3 / a.reps
            return ms, ctx.stats()

        nat_ms, nst = run(lambda: native.pauli_rot_(terms, thetas).flush(), native)
        dec_ms, dst = run(lambda: dec.submit(ops).flush(), dec)
        srng = np.random.default_rng(7)
        diff = 0.0
        for first in srng.integers(0, (1 << n) - 4096, 8):
            diff = max(diff, float(np.abs(native.to_host(int(first), 4096) - dec.to_host(int(first), 4096)).max()))
        w = {"rotations": len(terms), "native_ms_per_step": nat_ms,
             "native_launches_per_step": nst["simple_launches"] / a.reps,
             "native_sweeps_over_norm2": nat_ms / res["norm2_ms"],
             "decomposed_ms_per_step": dec_ms, "decomposed_gates_per_step": len(ops),
             "decomposed_passes_per_step": dst["passes"] / a.reps,
             "decomposed_simple_launches_per_step": dst["simple_launches"] / a.reps,
             "decomposed_jit_launches_per_step": dst.get("jit_launches", 0) / a.reps,
             "speedup_native_over_decomposed": dec_ms / nat_ms, "max_abs_native_minus_decomposed": diff}
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        del native, dec
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "workloads"}))


if __name__ == "__main__":
    main()
