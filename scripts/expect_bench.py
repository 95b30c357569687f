"""Pauli expectation values on a 30-qubit state: qb_expect_pauli against a qb_norm2 sweep of the same state
and against the reference route realPart (sv <.> (p #> sv)) (lazy clone + fused pass + qb_dotc per term).

    python scripts/expect_bench.py [--n 30] [--reps 10] --out FILE.json

The state (QFT plus two random layers from |0...0>, 16 GiB at n = 30) is far larger than the L2, so every
sweep reads HBM.  Times are host clocks around calls that end in a device synchronise (every
qb_expect_pauli call reads its values back), after one warm-up call of each workload."""
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


def workloads(n, rng):
    def s(ch_at):
        t = ["I"] * n
        for q, ch in ch_at:
            t[q] = ch
        return "".join(t)
    tfim = [s([(q, "Z"), (q + 1, "Z")]) for q in range(n - 1)] + [s([(q, "X")]) for q in range(n)]
    heis = [s([(q, p), (q + 1, p)]) for q in range(n - 1) for p in "XYZ"]
    out = {"tfim": tfim, "heisenberg": heis}
    x = (1 << 3) | (1 << 17)
    for k in (1, 8, 32, 64):
        out[f"group{k}"] = [(x, int(z)) for z in rng.integers(0, 1 << n, k)]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import qubism_b200 as Q
    from oracle import dense as D
    from qubism_b200.circuits import qft_ops, random_layers
    ctx = Q.Context.default()
    n = a.n
    sv = Q.mkStateVec(n, ctx)
    sv.submit(qft_ops(n) + random_layers(n, 2, seed=3))
    sv.flush()
    ctx.sync()
    bytes_sweep = 16 << n

    def timed(fn, reps):
        fn()
        ctx.sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        ctx.sync()
        return (time.perf_counter() - t0) * 1e3 / reps, r

    norm_ms, _ = timed(sv.norm2, a.reps)
    pm = {"X": D.pauliX(), "Y": D.pauliY(), "Z": D.pauliZ()}
    res = {"card": card(), "n": n, "state_GiB": bytes_sweep / 2**30, "reps": a.reps, "norm2_ms": norm_ms,
           "norm2_read_GBps": bytes_sweep / norm_ms / 1e6, "workloads": {}}
    for name, terms in workloads(n, np.random.default_rng(1)).items():
        ctx.reset_stats()
        sv.expect_pauli(terms)
        sweeps = ctx.stats()["reduce_launches"] // 2
        ms, vals = timed(lambda: sv.expect_pauli(terms), a.reps)
        # the reference route on the first 8 terms: p #> sv (lazy clone, one fused pass with its copy), then <.>
        strs = terms[:8]
        def route():
            out = []
            for t in strs:
                if isinstance(t, tuple):
                    x, z = t
                    t = "".join("Y" if (x >> q) & (z >> q) & 1 else "X" if (x >> q) & 1 else "Z" if (z >> q) & 1 else "I"
                                for q in range(n))
                ops = [("U", q, pm[ch]) for q, ch in enumerate(t) if ch != "I"]
                out.append(sv.inner(sv.apply_pure(ops)).real)
            return out
        route_ms, rv = timed(route, max(1, a.reps // 5))
        diff = float(np.abs(np.asarray(rv) - vals[:len(rv)]).max())
        w = {"terms": len(terms), "sweeps": sweeps, "ms": ms, "ms_per_sweep": ms / sweeps,
             "read_GBps": sweeps * bytes_sweep / ms / 1e6, "per_sweep_over_norm2": ms / sweeps / norm_ms,
             "route_first8_ms": route_ms, "route_first8_terms": len(strs),
             "max_route_diff": diff}
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
    res["norm2_state"] = sv.norm2()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "workloads"}))


if __name__ == "__main__":
    main()
