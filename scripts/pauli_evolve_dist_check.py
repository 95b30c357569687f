"""Exact time evolution under Pauli sums on a sharded state over NCCL: run under torchrun, one rank per GPU.
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/pauli_evolve_dist_check.py
exp(-itH) psi (terms with X / Y and Z on global qubits included) must equal the oracle's on every rank."""
import os, sys
import ctypes as C
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
import torch.distributed as dist
import qubism_b200 as Q
from qubism_b200 import capi
from oracle import structured as S
from qubism_b200.circuits import random_layers, qft_ops
from qubism_b200.statevec import pauli_masks
from pauli_evolve_oracle import evolve

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
if rank == 0:
    idbuf.copy_(torch.frombuffer(bytearray(Q.Context.unique_id()), dtype=torch.uint8))
dist.broadcast(idbuf, 0)
ctx = Q.Context(lr, rank, world, bytes(idbuf.cpu().numpy().tobytes()))
pbits = world.bit_length() - 1
ok = True


def strings(n, k, wmax, rng):
    out = []
    while len(out) < k:
        s = "".join(rng.choice(list("IXYZ"), n))
        if sum(ch in "XY" for ch in s) <= wmax:
            out.append(s)
    return out


for n in (pbits + 8, 16):
    L = n - pbits
    wmax = min(12, L)
    rng = np.random.default_rng(31 + n)  # same seed on every rank: same state, same strings
    full = S.gen_state(n, rng)
    ops = qft_ops(n) + random_layers(n, 2, seed=n)
    terms = strings(n, 20, wmax, rng) + ["X" * wmax + "I" * (n - wmax), "X" * pbits + "Z" * (n - pbits), "Z" * n, "I" * n]
    hc = rng.normal(size=len(terms))
    t = 0.9
    xs, zs = pauli_masks(terms, n)
    start = S.run_ops(n, ops, full)
    want, wk = evolve(n, xs, zs, hc, t, start)
    sv = Q.StateVec.from_host(full[rank << L:(rank + 1) << L], n=n, ctx=ctx)
    sv.submit(ops)
    ctx.reset_stats()
    k = C.c_int64()
    P64 = C.POINTER(C.c_uint64)
    capi.check(ctx.L.qb_pauli_evolve(sv._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64),
                                     hc.ctypes.data_as(C.POINTER(C.c_double)), len(xs), t, C.byref(k)))
    got = sv.to_host(0, 1 << n)
    st = ctx.stats()
    err = float(np.abs(got - want).max())
    tol = 1e-12 * max(1, k.value)
    good = err <= tol and abs(k.value - wk) <= 1
    ok = ok and good
    if rank == 0:
        print(f"n={n} world={world}: {len(terms)} terms, {k.value} Chebyshev steps, err {err:.2e} (tol {tol:.1e}), "
              f"tile launches {st['simple_launches']}, exchanges {st['exchanges']} -> {'OK' if good else 'FAIL'}",
              flush=True)
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
ctx.barrier()
if rank == 0:
    print("PAULI EVOLVE DIST CHECK PASSED" if flag.item() == 1 else "PAULI EVOLVE DIST CHECK FAILED", flush=True)
del sv
ctx.close()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
