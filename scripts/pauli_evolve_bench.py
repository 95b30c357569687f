"""Exact time evolution exp(-itH) on a 30-qubit state (qb_pauli_evolve): time per call and per Chebyshev step,
the bytes a step moves and the rate achieved, with a qb_pauli_sum and a qb_norm2 sweep of the same size for scale.

    python scripts/pauli_evolve_bench.py [--n 30] [--reps 1] [--warmup 1] --out FILE.json

Hamiltonians: the Heisenberg chain (XX, YY, ZZ on every bond, unit couplings: 87 terms at n = 30, r = 87) and
the transverse-field Ising chain (ZZ on every bond, 0.8 X on every qubit: 59 terms, r = 53.2), at t = 0.1 and 1.
Each state (16 GiB at n = 30) is far larger than the L2, so every sweep reads and writes HBM.  Times are host
clocks around `reps` calls that each end in a device synchronise, after `warmup` calls of the same workload.

Bytes per step, from the kernel's accesses: every launch reads T_k and T_{k-1} and writes T_{k+1} (48 B per
amplitude); the step's last launch also reads and writes the sum (32 B).  Step 1 reads neither the sum nor
T_{k-1}.  Kernel
times per launch come from a separate profiled run (torch.profiler, CUDA activities) of the t = 0.1 calls."""
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


def evolve(sv, terms, coefs, t):
    from qubism_b200 import capi
    from qubism_b200.statevec import pauli_masks
    xs, zs = pauli_masks(terms, sv.n)
    cf = np.ascontiguousarray(coefs, dtype=np.float64)
    k = C.c_int64()
    P64 = C.POINTER(C.c_uint64)
    capi.check(sv.ctx.L.qb_pauli_evolve(sv._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64),
                                        cf.ctypes.data_as(C.POINTER(C.c_double)), len(xs), float(t), C.byref(k)))
    return k.value


def timed(fn, reps, warmup, ctx):
    for _ in range(warmup):
        fn()
        ctx.sync()
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
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import qubism_b200 as Q
    from qubism_b200.circuits import qft_ops, random_layers
    ctx = Q.Context.default()
    n = a.n
    amps = 1 << n
    state = 16 * amps
    res = {"card": card(), "n": n, "state_GiB": state / 2**30, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    sv = Q.mkStateVec(n, ctx).submit(qft_ops(n) + random_layers(n, 2, seed=3)).flush()
    ctx.sync()
    res["norm2_ms"] = timed(sv.norm2, max(3, a.reps), a.warmup, ctx)
    res["norm2_read_TBps"] = state / res["norm2_ms"] / 1e9
    ham = hamiltonians(n)
    for name, (terms, coefs) in ham.items():
        res[f"pauli_sum_{name}_ms"] = timed(lambda: sv.pauli_sum(terms, coefs).flush(), max(3, a.reps), a.warmup, ctx)
        ctx.reset_stats()
        sv.pauli_sum(terms, coefs).flush()
        L = ctx.stats()["simple_launches"]
        res[f"pauli_sum_{name}_launches"] = L
        for t in (0.1, 1.0):
            w = sv.clone()
            K = {}
            ms = timed(lambda: K.update(k=evolve(w, terms, coefs, t)), a.reps, a.warmup, ctx)
            ctx.reset_stats()
            evolve(w, terms, coefs, t)
            launches = ctx.stats()["simple_launches"]
            k = K["k"]
            step_bytes = (48 * L + 32) * amps
            total_bytes = ((48 * L + 32) * k - 32) * amps  # (step 1 reads neither T_{-1} nor the sum)
            r = {"terms": len(terms), "r": float(np.abs(coefs).sum()), "tau": t * float(np.abs(coefs).sum()),
                 "steps": k, "launches_per_step": launches / k, "call_ms": ms, "step_ms": ms / k,
                 "bytes_per_step_GB": step_bytes / 1e9, "achieved_TBps": total_bytes / ms / 1e9,
                 "norm": w.norm2()}
            res["workloads"][f"{name}_t{t}"] = r
            print(name, t, json.dumps(r), flush=True)
            del w
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for name, (terms, coefs) in ham.items():
        w = sv.clone()
        evolve(w, terms, coefs, 0.1)
        ctx.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            evolve(w, terms, coefs, 0.1)
            ctx.sync()
        for ev in prof.key_averages():
            if "k_pauli_cheb_tile" in ev.key:
                us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                d = kern.setdefault(name, {"launches": 0, "total_ms": 0.0})
                d["launches"] += ev.count
                d["total_ms"] += us / 1e3
        del w
    for name, d in kern.items():
        d["ms_per_launch"] = d["total_ms"] / max(1, d["launches"])
        d["TBps_at_48B_per_amp"] = 48 * amps / d["ms_per_launch"] / 1e9
    res["kernels_profiled"] = kern
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "workloads"}))


if __name__ == "__main__":
    main()
