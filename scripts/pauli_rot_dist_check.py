"""Pauli rotations on a sharded state over NCCL: run under torchrun, one rank per GPU.
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/pauli_rot_dist_check.py
The state after gates, rotations (X / Y and Z on global qubits included) and more gates must equal the
oracle's on every rank."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
import torch.distributed as dist
import qubism_b200 as Q
from oracle import structured as S
from qubism_b200.circuits import random_layers, qft_ops
from qubism_b200.statevec import pauli_masks
from pauli_rot_oracle import pauli_rot

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
for n in (pbits + 8, 16):
    L = n - pbits
    wmax = min(12, L)
    rng = np.random.default_rng(17 + n)  # same seed on every rank: same state, same rotations
    full = S.gen_state(n, rng)
    ops = qft_ops(n) + random_layers(n, 2, seed=n)
    terms = []
    while len(terms) < 60:
        s = "".join(rng.choice(list("IXYZ"), n))
        if sum(ch in "XY" for ch in s) <= wmax:
            terms.append(s)
    terms += ["X" * pbits + "I" * (n - pbits), "Y" * (pbits + 1) + "Z" * (n - pbits - 1), "X" * wmax + "I" * (n - wmax)]
    th = rng.uniform(-3, 3, len(terms))
    xs, zs = pauli_masks(terms, n)
    ref = S.run_ops(n, ops, full)
    for x, z, t in zip(xs, zs, th):
        ref = pauli_rot(n, int(x), int(z), float(t), ref)
    ref = S.run_ops(n, ops, ref)
    sv = Q.StateVec.from_host(full[rank << L:(rank + 1) << L], n=n, ctx=ctx)
    sv.submit(ops)
    ctx.reset_stats()
    sv.pauli_rot_(terms, th)
    sv.submit(ops)
    got = sv.to_host(0, 1 << n)
    st = ctx.stats()
    tol = 1e-12 * max(1.0, float(np.vdot(ref, ref).real))
    err = float(np.abs(got - ref).max())
    good = err <= tol
    ok = ok and good
    if rank == 0:
        print(f"n={n} world={world}: {len(terms)} rotations, max err {err:.2e} (tol {tol:.1e}), "
              f"rotation launches {st['simple_launches']}, exchanges {st['exchanges']} -> {'OK' if good else 'FAIL'}",
              flush=True)
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
ctx.barrier()
if rank == 0:
    print("PAULI ROT DIST CHECK PASSED" if flag.item() == 1 else "PAULI ROT DIST CHECK FAILED", flush=True)
del sv
ctx.close()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
