"""Pauli expectation values on a sharded state over NCCL: run under torchrun, one rank per GPU.
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/expect_dist_check.py
Every rank must receive the same values, equal to the oracle's; X / Y on global qubits included, and the
state must read back unchanged afterwards."""
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
from pauli_oracle import expect_pauli

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
    rng = np.random.default_rng(7 + n)  # same seed on every rank: same state, same terms
    full = S.gen_state(n, rng)
    ops = qft_ops(n) + random_layers(n, 2, seed=n)
    ref = S.run_ops(n, ops, full)
    terms = []
    while len(terms) < 60:
        s = "".join(rng.choice(list("IXYZ"), n))
        if sum(ch in "XY" for ch in s) <= L:
            terms.append(s)
    terms += ["X" * pbits + "I" * (n - pbits), "Y" * (pbits + 1) + "Z" * (n - pbits - 1), "X" * L + "I" * pbits]
    xs, zs = pauli_masks(terms, n)
    sv = Q.StateVec.from_host(full[rank << L:(rank + 1) << L], n=n, ctx=ctx)
    sv.submit(ops)
    ctx.reset_stats()
    got = sv.expect_pauli(terms)
    st = ctx.stats()
    want = np.array([expect_pauli(n, int(x), int(z), ref) for x, z in zip(xs, zs)])
    tol = 1e-12 * max(1.0, float(np.vdot(ref, ref).real))
    err = float(np.abs(got - want).max())
    mine = torch.tensor(got, device="cuda")
    first = mine.clone()
    dist.broadcast(first, 0)
    same = bool(torch.equal(mine, first))
    amp_err = float(np.abs(sv.to_host(0, 1 << n) - ref).max())
    good = err <= tol and same and amp_err < 1e-12
    ok = ok and good
    if rank == 0:
        print(f"n={n} world={world}: {len(terms)} terms, max err {err:.2e} (tol {tol:.1e}), same on every rank {same}, "
              f"state err {amp_err:.2e}, sweeps {st['reduce_launches'] // 2}, exchanges {st['exchanges']} -> "
              f"{'OK' if good else 'FAIL'}", flush=True)
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
ctx.barrier()
if rank == 0:
    print("EXPECT DIST CHECK PASSED" if flag.item() == 1 else "EXPECT DIST CHECK FAILED", flush=True)
del sv
ctx.close()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
