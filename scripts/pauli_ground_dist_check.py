"""Lanczos ground states of Pauli sums on a sharded state over NCCL: run under torchrun, one rank per GPU.
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/pauli_ground_dist_check.py
The energy, the Lanczos coefficients and the Ritz vector (terms with X / Y and Z on global qubits included) must
equal the oracle's on every rank."""
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
from pauli_ground_oracle import ground

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


for n in (pbits + 8, 14):
    L = n - pbits
    wmax = min(12, L)
    rng = np.random.default_rng(41 + n)  # same seed on every rank: same state, same strings
    full = S.gen_state(n, rng)
    ops = qft_ops(n) + random_layers(n, 2, seed=n)
    terms = strings(n, 20, wmax, rng) + ["X" * wmax + "I" * (n - wmax), "X" * pbits + "Z" * (n - pbits), "Z" * n, "I" * n]
    hc = rng.normal(size=len(terms))
    xs, zs = pauli_masks(terms, n)
    r = float(np.abs(hc[:-1]).sum())
    tol, maxiter = 1e-10 * r, 2000
    start = S.run_ops(n, ops, full)
    we, _, wm, wal, wbe, wx = ground(n, xs, zs, hc, start, tol, maxiter, vector=True)
    sv = Q.StateVec.from_host(full[rank << L:(rank + 1) << L], n=n, ctx=ctx)
    sv.submit(ops)
    ctx.reset_stats()
    e, res, m = C.c_double(), C.c_double(), C.c_int64()
    al, be = np.zeros(maxiter), np.zeros(maxiter)
    P64, PD = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
    capi.check(ctx.L.qb_pauli_ground(sv._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64), hc.ctypes.data_as(PD),
                                     len(xs), tol, maxiter, 1, C.byref(e), C.byref(res), C.byref(m),
                                     al.ctypes.data_as(PD), be.ctypes.data_as(PD)))
    got = sv.to_host(0, 1 << n)
    st = ctx.stats()
    k = min(m.value, wm, 20)
    err_c = max(float(np.abs(al[:k] - wal[:k]).max()), float(np.abs(be[:k] - wbe[:k]).max()))
    err_e = abs(e.value - we)
    err_x = float(np.abs(got - wx).max())
    good = abs(m.value - wm) <= 1 and err_c <= 1e-12 * r and err_e <= 1e-10 * r and err_x <= 1e-6
    ok = ok and good
    if rank == 0:
        print(f"n={n} world={world}: {len(terms)} terms, m = {m.value} (oracle {wm}), energy err {err_e:.2e}, "
              f"coefficient err {err_c:.2e}, vector err {err_x:.2e}, launches {st['simple_launches']}, "
              f"exchanges {st['exchanges']} -> {'OK' if good else 'FAIL'}", flush=True)
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
ctx.barrier()
if rank == 0:
    print("PAULI GROUND DIST CHECK PASSED" if flag.item() == 1 else "PAULI GROUND DIST CHECK FAILED", flush=True)
del sv
ctx.close()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
