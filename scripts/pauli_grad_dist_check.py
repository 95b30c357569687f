"""Pauli sums and adjoint gradients on a sharded state over NCCL: run under torchrun, one rank per GPU.
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/pauli_grad_dist_check.py
The energy and gradient (rotations and terms with X / Y and Z on global qubits included) and H psi must equal
the oracle's on every rank."""
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
from pauli_grad_oracle import pauli_sum, rot_grad

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
    rng = np.random.default_rng(29 + n)  # same seed on every rank: same state, same strings
    full = S.gen_state(n, rng)
    ops = qft_ops(n) + random_layers(n, 2, seed=n)
    rots = strings(n, 40, wmax, rng) + ["I" * n, "X" * pbits + "I" * (n - pbits), "Y" * (pbits + 1) + "Z" * (n - pbits - 1)]
    hterms = strings(n, 20, wmax, rng) + ["X" * wmax + "I" * (n - wmax), "Z" * n]
    th = rng.uniform(-3, 3, len(rots))
    hc = rng.normal(size=len(hterms))
    rx, rz = pauli_masks(rots, n)
    hx, hz = pauli_masks(hterms, n)
    start = S.run_ops(n, ops, full)
    we, wg = rot_grad(n, rx, rz, th, hx, hz, hc, start)
    whs = pauli_sum(n, hx, hz, hc, start)
    sv = Q.StateVec.from_host(full[rank << L:(rank + 1) << L], n=n, ctx=ctx)
    sv.submit(ops)
    ctx.reset_stats()
    e, g = sv.pauli_rot_grad(rots, th, hterms, hc)
    hs = sv.pauli_sum(hterms, hc).to_host(0, 1 << n)
    st = ctx.stats()
    tol = 1e-12 * max(1.0, float(np.abs(hc).sum()))
    err = max(abs(e - we), float(np.abs(g - wg).max()))
    herr = float(np.abs(hs - whs).max())
    good = err <= tol and herr <= 1e-12 * len(hterms) * max(1.0, float(np.abs(whs).max()))
    ok = ok and good
    if rank == 0:
        print(f"n={n} world={world}: {len(rots)} rotations, {len(hterms)} terms, gradient err {err:.2e} (tol {tol:.1e}), "
              f"H psi err {herr:.2e}, tile launches {st['simple_launches']}, exchanges {st['exchanges']} -> "
              f"{'OK' if good else 'FAIL'}", flush=True)
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
ctx.barrier()
if rank == 0:
    print("PAULI GRAD DIST CHECK PASSED" if flag.item() == 1 else "PAULI GRAD DIST CHECK FAILED", flush=True)
del sv
ctx.close()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
