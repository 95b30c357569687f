#!/usr/bin/env python
"""bench.py -- amplitude-updates/s of the qubism state-vector hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload qft_rand|adder32|general] [--qubits n] [--dump-outputs DIR]

One STEP = one pass of the hot path over one batch of synthetic input: the whole primitive
op stream of the workload circuit applied to an n-qubit device-resident state through the C
ABI (libqubism_sv.so).  One amplitude-update = one amplitude visited by one primitive op of
the reference evaluator's op stream (a U on one qubit or a CX, after qelib1.inc expansion);
a primitive op on an n-qubit state is 2^n amplitude-updates no matter how the backend fuses
or folds it (SURVEY.md 8d).

Workload (BASELINE.json):  N = 1: 30 qubits, QFT-30 (2,207 ops, examples/fourier.qasm pattern)
followed by 20 random layers (30 U + 15 CX each, 900 ops).  N > 1: the same family on
n = 31 + log2(N) qubits (32 GiB of amplitudes per GPU; N = 8 is the 34-qubit configuration),
sharded one rank per GPU with global<->local qubit swaps over NCCL/NVLink.

Other workloads (profiles/ keeps their lines): --workload adder32 = examples/rippleCarryAdder.qasm
widened to 32 qubits (BASELINE.json config 4, meant for 2 and 4 GPUs); --workload general = 20
layers of true SU(2) matrices (the general complex gate class); --qubits overrides n (36 = the
capacity stretch point on 8 GPUs).

The JSON line carries: value (device-timed, inputs resident in HBM), e2e (through the C ABI
from HOST buffers the way the reference interpreter drives it: pinned state upload, then per
primitive op one PURE application sv' = g #> sv -- qb_state_apply_pure on the current value, the
old value freed, QASM/Simulation.hs:94-122 -- then reductions and a readback, all inside the
timed region), roofline (HBM, for the fused-pass kernel, measured live with CUDA events on
the launching stream), cpu_baseline (the oracle's C/OpenMP port on the host cores, bounded
sample), clocks (nvidia-smi during the timed region).

--dump-outputs DIR writes what the last timed step left in the state (a fixed, seeded sample of
its amplitudes in index order, DIR/state.npy with their indices in DIR/state_index.npy) and what
the last end-to-end step handed back (DIR/e2e_sumsq.npy, DIR/e2e_window.npy), all float64 with
(re, im) in the last axis, 24 MiB at most.  The warm-up then always takes its longest length,
so the timed steps start from the same state whatever the settling needed, and two builds can be
compared output for output on the same arguments.

--impl reference times the reference's CPU path.  The Haskell reference cannot be built here
(no GHC) and its literal dense algorithm cannot reach 24 qubits on any machine (one gate
matrix would be 4.5 PB, SURVEY.md section 0), so this arm runs the oracle's structured
C/OpenMP restatement (oracle/csrc/sv_struct.c, kind "port") with all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line: NCCL's banner / debug output goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

METRIC = "amplitude_updates_per_s"
UNIT = "amplitude-updates/s"
CPU_SAMPLE_N = 24


def workload(n: int, kind: str = "qft_rand"):
    from qubism_b200.circuits import adder_ops, proper_unitary_layers, qft_ops, random_layers
    if kind == "adder32":
        return adder_ops((n - 2) // 2)
    if kind == "general":
        return proper_unitary_layers(n, 20, seed=3000)
    return qft_ops(n) + random_layers(n, 20, seed=1000)


def workload_name(n: int, kind: str = "qft_rand") -> str:
    if kind == "adder32":
        return (f"adder{n}: examples/rippleCarryAdder.qasm widened to {(n - 2) // 2}-bit operands on one qreg q[{n}] "
                "(ccx = 9 U + 6 CX through qelib1.inc)")
    if kind == "general":
        return f"general20x{n}: 20 layers of true SU(2) matrices (general complex class) + CX pairs ({20 * (n + n // 2)} ops)"
    return f"qft{n}+rand20x{n}: QFT-{n} ({n + 5 * n * (n - 1) // 2 + 2} ops) + 20 random U/CX layers ({20 * (n + n // 2)} ops)"


def inverse_ops(ops):
    """C^-1 for a stream of (near-)unitary U and CX ops: reversed, matrices conjugate-transposed."""
    import numpy as np
    return [op if op[0] == "CX" else ("U", op[1], np.asarray(op[2]).conj().T) for op in reversed(ops)]


# ------------------------------------------------------------------------------ --dump-outputs
DUMP_WINDOW, DUMP_WINDOWS = 4096, 256  # 2^20 amplitudes: 16 MiB of (re, im) pairs + 8 MiB of indices


def state_sample(sv, n: int):
    """The same seeded sample of the 2^n logical amplitudes whatever the build: DUMP_WINDOWS windows
    of DUMP_WINDOW consecutive amplitudes (the whole state when it is smaller).  A collective on a
    sharded state: every rank calls it."""
    import numpy as np
    w = min(DUMP_WINDOW, 1 << n)
    nwin = (1 << n) // w
    starts = np.sort(np.random.default_rng(0).choice(nwin, min(DUMP_WINDOWS, nwin), replace=False)) * w
    amps = np.concatenate([sv.to_host(int(s), w) for s in starts])
    index = (starts[:, None] + np.arange(w)).reshape(-1)
    return {"state": amps.view(np.float64).reshape(-1, 2), "state_index": index.astype(np.float64)}


def write_outputs(out_dir: str, arrays: dict):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        """The timed region starts now: only samples taken from here on count."""
        self.t0 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = getattr(self, "t0", 0.0)
        for stamp, ln in self.lines:
            if stamp < t0:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------ CPU arm
def cpu_threads() -> int:
    """All host threads the process may use.  torch.distributed.run exports OMP_NUM_THREADS=1 to its
    workers; the CPU arm overrides that explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_sample_ops(n: int):
    from qubism_b200.circuits import qft_ops, random_layers
    return qft_ops(n) + random_layers(n, 2, seed=1000)


def cpu_run(n: int, steps: int, warmup: int, budget_s: float = 150.0, keep_first: bool = False):
    """Times the oracle's C/OpenMP port (one sweep per primitive op, no fusion) on the host: `steps`
    timed steps after at most `warmup` untimed ones (the warm-up stops after `budget_s` / 3 seconds)."""
    import numpy as np
    from oracle import cport
    cport.lib().sv_set_threads(cpu_threads())
    ops = cpu_sample_ops(n)
    packed = cport.pack_ops(ops)
    v = np.zeros(1 << n, dtype=np.complex128)
    v[0] = 1.0
    first = None
    t_w = time.perf_counter()
    for i in range(warmup):
        cport.run_ops_inplace(n, packed, v)
        if keep_first and first is None:
            first = v.copy()
        if time.perf_counter() - t_w > budget_s / 3:
            break
    t0 = time.perf_counter()
    for _ in range(steps):
        cport.run_ops_inplace(n, packed, v)
        if keep_first and first is None:
            first = v.copy()
    dt = time.perf_counter() - t0
    cores = int(cport.lib().sv_num_threads())
    aups = len(ops) * (1 << n) * steps / dt
    sample = (f"QFT-{n} + 2 random layers at n={n} ({len(ops)} primitive ops, {(16 << n) >> 20} MiB state), "
              f"{steps} step(s), one sweep per op, OpenMP x{cores}")
    return aups, dt / steps, cores, sample, steps, first


def literal_dense_sample():
    """The reference's REAL algorithm (dense kron / matmul, oracle.dense) at the largest size
    that finishes in seconds: shows its O(8^n) wall next to the structured port."""
    import numpy as np
    from oracle import dense as D
    n = 10
    v = D.mkStateVec(n)
    t0 = time.perf_counter()
    nops = 0
    for q in range(3):
        v = D.apply(D.onJust(n, q, D.hadamard()), v)
        v = D.apply(D.cnot(n, q, q + 1), v)
        nops += 2
    dt = time.perf_counter() - t0
    return {"n": n, "ops": nops, "value": nops * (1 << n) / dt, "unit": UNIT,
            "what": "literal dense restatement of QGate.hs:121-154 (numpy/BLAS), 3 H + 3 CX"}


def bench_n(args, world: int) -> int:
    if args.qubits:
        return args.qubits
    if args.workload == "adder32":
        return 32
    return 30 if world == 1 else 31 + (world.bit_length() - 1)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["OMP_NUM_THREADS"] = str(cpu_threads())
    aups, step_s, cores, sample, done, _ = cpu_run(CPU_SAMPLE_N, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": aups, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "complex128 (f64)", "data": "synthetic",
        "config": {"workload": workload_name(bench_n(args, args.gpus), args.workload), "sample": sample},
        "cpu_baseline": {"value": aups, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": aups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import ctypes as C
    import numpy as np
    import torch
    import qubism_b200 as Q
    from qubism_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idbuf.copy_(torch.frombuffer(bytearray(Q.Context.unique_id()), dtype=torch.uint8))
        dist.broadcast(idbuf, 0)
        ctx = Q.Context(local_rank, rank, world, bytes(idbuf.cpu().numpy().tobytes()))
    else:
        ctx = Q.Context(local_rank)
    n = int(os.environ.get("QB_BENCH_N", bench_n(args, world)))
    L = n - (world.bit_length() - 1)
    ops = workload(n, args.workload)
    packed = capi.pack_ops(ops)
    nops = len(ops)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def mark(what):
        if os.environ.get("QB_BENCH_TRACE"):
            print(f"[bench rank {rank}] {what}", file=sys.stderr, flush=True)

    sv = Q.StateVec.create(n, True, ctx)
    ctx.set_option("time_kernels", 1)
    mark("state created")

    # ---------------- device-resident throughput (`value`)
    def step():
        sv.submit(packed)
        sv.flush()

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()  # nvidia-smi takes a moment to start: launch it before the warm-up
    # the very first step of the process: no pass structure has been seen, every pass runs the
    # generic kernels (what a one-shot program -- the interpreter's usual use -- gets); from a
    # fresh |0...0>, so the early passes also skip the all-zero tiles
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    f0.record(stream)
    step()
    f1.record(stream)
    barrier()
    first_step_ms = max_over_ranks(f0.elapsed_time(f1))
    mark("first step done")
    for _ in range(max(0, args.warmup - 1)):
        step()
    # pass structures that came back during the warm-up are being compiled into specialised
    # kernels on background threads: let that finish, and give the next sighting (which loads
    # the modules) its own untimed steps -- the timed region measures the steady state
    # (the qubit layout of the state cycles with a period of a few steps -- 2 on one GPU, where every
    #  pass re-sorts it; 2-3 sharded -- and a structure has to come round twice before it is compiled)
    for _ in range(6 if world == 1 else 8):
        ctx.jit_wait()
        step()
    # ... and keep going until the steady state is really there: `need` steps in a row in which every
    # pass of every rank ran as a specialised kernel (sharded layouts take 6-10 steps to settle into
    # their cycle of period <= 6 and every structure of the cycle has to come round twice), at most
    # 32 more steps.  All ranks take the same number of steps (the steps hold collectives).
    settle_steps, good, need, max_settle = 0, 0, (2 if world == 1 else 6), 32
    while ctx.get_option("jit") > 0 and good < need and settle_steps < max_settle:
        ctx.jit_wait()
        ctx.reset_stats()
        step()
        stw = ctx.stats()
        generic = 1.0 if stw["jit_launches"] < stw["passes"] else 0.0
        ctx.sync()  # (the library's own collectives have drained before torch's all-reduce is enqueued)
        good = good + 1 if max_over_ranks(generic) == 0.0 else 0
        settle_steps += 1
    if args.dump_outputs:
        # the longest settling on every run: the timed steps start from the same state
        for _ in range(max_settle - settle_steps):
            step()
    barrier()
    mark(f"warm-up done ({settle_steps} settling steps)")
    ctx.reset_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.mark()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    elapsed = e0.elapsed_time(e1) / 1e3
    st = ctx.stats()
    mark("timed steps done")
    outputs = state_sample(sv, n) if args.dump_outputs else {}  # (before the steps below change the state)
    if world == 1 and elapsed < 1.5:
        # nvidia-smi samples every 100 ms: keep the same load running (outside the timed region,
        # after the counters were read) until it has seen at least 1.5 s of it
        t_more = time.time()
        while time.time() - t_more < 1.5 - elapsed:
            step()
        ctx.sync()
    clk = clocks.stop() if rank == 0 else None
    elapsed = max_over_ranks(elapsed)
    value = nops * float(1 << n) * args.steps / elapsed
    passes = st["passes"] / args.steps
    fused_ms = st["fused_ms"] / max(1, st["fused_timed"])  # average launch duration
    launches = (st["passes"] + st["simple_launches"] + st["reduce_launches"])
    ops_exec = st["ops_executed"] / args.steps
    ops_fold = st["ops_folded"] / args.steps
    ctx.set_option("time_kernels", 0)

    # ---------------- sharded runs: an untimed inverse-circuit round trip, C^-1 C |0...0> = |0...0>
    round_trip = None
    if world > 1 or args.round_trip:
        rt = Q.StateVec.create(n, True, ctx)
        rt.submit(packed)
        rt.flush()
        rt.submit(capi.pack_ops(inverse_ops(ops)))
        head = rt.to_host(0, min(1 << n, 1 << 20))
        nrm = rt.norm2()
        head[0] -= 1.0
        round_trip = {"max_abs_diff_vs_basis_state": float(np.abs(head).max()), "amplitudes_checked": int(head.size),
                      "norm_minus_one": nrm - 1.0,
                      "what": "fresh |0...0> -> workload -> inverse workload, first 2^20 logical amplitudes + the norm"}
        rt.free()
        barrier()
        mark("round trip done")

    # ---------------- end to end through the C ABI from host buffers (`e2e`)
    # every step: upload this rank's shard from pinned host memory, then drive the boundary the way
    # the reference interpreter does -- per primitive op ONE pure application sv' = g #> sv on the
    # current value (qb_state_apply_pure: lazy clone + enqueue), the old value dropped
    # (QASM/Simulation.hs:94-122) -- then flush, three measurement reductions and a window of amplitudes.
    shard = 1 << L
    chunk = min(shard, 1 << 28)  # 4 GiB of pinned host memory per rank, re-sent to fill the shard
    host = torch.empty(2 * chunk, dtype=torch.float64, pin_memory=True)
    host.zero_()
    one = torch.zeros(2, dtype=torch.float64, pin_memory=True)
    one[0] = 1.0
    win = min(4096, shard)
    lib = ctx.L
    op_ptrs = [C.cast(C.byref(packed, i * C.sizeof(capi.QbOp)), C.POINTER(capi.QbOp)) for i in range(nops)]
    cur = {"sv": sv}

    def e2e_step():
        s0 = cur["sv"]
        for off in range(0, shard, chunk):
            s0.write_local((host.data_ptr(), chunk), first=off)
        # (every rank makes the same calls: an upload into a state that was ever cloned agrees on its
        #  handles across ranks, i.e. it is a collective)
        s0.write_local((one.data_ptr() if rank == 0 else host.data_ptr(), 1), first=0)
        h = s0._h
        for ptr in op_ptrs:
            nh = C.c_void_p()
            rc = lib.qb_state_apply_pure(h, ptr, 1, C.byref(nh))
            if rc != 0:
                capi.check(rc)
            lib.qb_state_free(h)  # the interpreter's map entry is overwritten: the old value is garbage
            h = nh
        s0._h = None
        s1 = Q.StateVec(h, ctx)
        cur["sv"] = s1
        s1.flush()
        red = [s1.sumsq(q) for q in (0, n // 2, n - 1)]
        w = s1.local_to_host(0, win)
        return red, w

    mark("e2e: buffers ready")
    e2e_step()
    mark("e2e: first step done")
    ctx.jit_wait()
    e2e_step()
    barrier()
    mark("e2e: warm-up done")
    ctx.reset_stats()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 2))
    for _ in range(e2e_steps):
        red, w = e2e_step()
    barrier()
    e2e_dt = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    st_e2e = ctx.stats()
    e2e_value = nops * float(1 << n) / e2e_dt
    h2d = 16 * shard + nops * 80
    d2h = 3 * 16 + 16 * win
    if args.dump_outputs:
        outputs["e2e_sumsq"] = np.array(red)  # (S0, S1) of qubits 0, n // 2, n - 1
        outputs["e2e_window"] = w.view(np.float64).reshape(-1, 2)  # rank 0: the first `win` of its shard

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (k_fused_pass), HBM-bound
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "B200_PROFILING.md fallback 6650 GB/s (of fallback)"
    alg_bytes = 32.0 * float(1 << L)  # 16 B read + 16 B written per local amplitude per pass
    achieved = alg_bytes / (fused_ms / 1e3) / 1e9 if fused_ms > 0 else None
    traffic, traffic_src = None, None
    for tag in ("r02c", "r02", "r01e", "r01d"):  # newest ncu --set full capture of the dominant kernel
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", f"{tag}_fused_pass_summary.json")))
            traffic = prof.get("dram_bytes_per_launch_scaled_to", {}).get(str(L))
            traffic_src = f"profiles/{tag}_fused_pass_summary.json (ncu --set full capture of an earlier run of this command, not measured in this run)"
            break
        except (OSError, ValueError):
            continue
    jit_share = st["jit_launches"] / max(1, st["passes"])
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": ("qb_jit_pass (k_fused_pass specialised per pass structure with NVRTC)" if jit_share > 0.5
                           else "k_fused_pass"),
                "specialised_share_of_launches": jit_share,
                "launches_per_step": passes, "avg_launch_ms": fused_ms,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "kernel_share_of_step": (st["fused_ms"] / 1e3) / elapsed if elapsed > 0 else None,
                # what the ops that REACH a kernel would move one sweep per op (SURVEY.md 8d): may exceed
                # the HBM peak, which is the point of fusing.  Folded ops are not counted here.
                "unfused_equivalent_gbs_executed_ops": ops_exec * float(1 << n) / (elapsed / args.steps) / world * 32.0 / 1e9,
                "gates_per_launch": ops_exec / max(1.0, passes),
                "note": "frac is per launch: a plan that packs the same gates into fewer, denser passes lowers it while the "
                        "step gets faster (DESIGN.md section 6); the memory side of a pass alone (its loads, L2 prefetch and "
                        "stores, no gates) takes 7.1-7.6 ms per 34 GB on this pool's boxes (profiles/r02z_density.txt)"}
    if world > 1:
        # SURVEY.md 8d: T_roof(P) = passes x 32 B x 2^L / HBM  +  bytes sent per GPU / NVLink per direction
        nvl = 770.0  # GB/s per direction, measured peer copy on this pool (SURVEY.md 8d; 900 nominal)
        xb = st["exchange_bytes"] / args.steps
        t_roof = passes * alg_bytes / (peak * 1e9) + xb / (nvl * 1e9)
        roofline["sharded"] = {"t_roof_ms": t_roof * 1e3, "t_measured_ms": elapsed / args.steps * 1e3,
                               "efficiency": t_roof / (elapsed / args.steps),
                               "hbm_term_ms": passes * alg_bytes / (peak * 1e9) * 1e3, "nvlink_term_ms": xb / (nvl * 1e9) * 1e3,
                               "nvlink_gbs_per_direction": nvl,
                               "what": "SURVEY.md 8d: sum of the passes at the HBM peak plus the exchanged bytes at the "
                                       "measured NVLink rate, over the measured step"}

    # ---------------- CPU baseline (rank 0, N = 1 only): the oracle's C port, bounded sample, and the
    # same sample on the GPU: max |amplitude difference| (BASELINE.md section 4)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        aups, _, cores, sample, _, cpu_first = cpu_run(CPU_SAMPLE_N, 1, 0, keep_first=True)
        g = Q.StateVec.create(CPU_SAMPLE_N, True, ctx)
        g.submit(cpu_sample_ops(CPU_SAMPLE_N))
        diff = float(np.abs(g.to_host() - cpu_first).max())
        g.free()
        cpu = {"value": aups, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
               "max_abs_amplitude_diff_gpu_vs_port": diff, "diff_what": f"all 2^{CPU_SAMPLE_N} amplitudes after the sample circuit from |0...0>",
               "literal_dense": literal_dense_sample()}

    step_s = elapsed / args.steps
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "complex128 (f64)", "data": "synthetic",
        # the same time split by what happened to the ops (SURVEY.md 7.2): `value` counts every primitive
        # op submitted; `value_executed` only those that reached a kernel (the host peephole folds scalar
        # u1-type gates, merges runs on one qubit and cancels CX pairs before anything is planned)
        "by_class": {"value_executed": ops_exec * float(1 << n) / step_s, "ops_submitted_per_step": nops,
                     "ops_executed_per_step": ops_exec, "ops_folded_per_step": ops_fold,
                     "folded_share": ops_fold / max(1, nops)},
        # the same step the first time the process sees it: no specialised kernel exists yet
        "first_step": {"ms": first_step_ms, "value": nops * float(1 << n) / (first_step_ms / 1e3),
                       "what": "step 1 of the process from a fresh |0...0>: generic kernels (nothing compiled yet), "
                               "all-zero tiles skipped; steady state = `value`"},
        "config": {"workload": workload_name(n, args.workload), "qubits": n, "local_qubits": L, "primitive_ops_per_step": nops,
                   "state_bytes_per_gpu": 16 << L, "l2_policy": "inputs larger than L2 (state >= 16 GiB >> 126 MB)",
                   "parallelism": f"shard{world}" if world > 1 else "single",
                   "planner": {k: ctx.get_option(k) for k in ("tile_bits", "reg_bits", "low_bits", "lane_fixed", "max_rounds", "peephole", "rot", "lite", "jit", "tma", "oop", "oop_low_bits", "l2_prefetch")},
                   "specialised_kernels": {"compiled": st["jit_compiled"], "compile_ms_total": st["jit_compile_ms"],
                                           "launches_in_timed_region": st["jit_launches"],
                                           "toolchain": lib.qb_jit_toolchain().decode(),
                                           "note": "pass structures seen twice are compiled with NVRTC on background threads during "
                                                   "the warm-up steps (W + 6 untimed steps on one GPU, W + 8 sharded, then until every pass of `need` steps "
                                                   "in a row ran specialised on every rank: `settling_steps`); the timed steps hit the cache",
                                           "settling_steps": settle_steps},
                   "ops_executed_per_step": ops_exec, "ops_folded_per_step": ops_fold,
                   "passes_per_step": passes, "rounds_per_step": st["rounds"] / args.steps,
                   "exchanges_per_step": st["exchanges"] / args.steps,
                   # of those: swaps carried by the stores of the pass before them (option fuse_exchange: that pass
                   # writes over NVLink peer memory into the next owner's second shard; no exchange sweep)
                   "exchanges_fused_per_step": st.get("exchanges_fused", 0) / args.steps,
                   "exchange_bytes_per_gpu_per_step": st["exchange_bytes"] / args.steps,
                   "plan_ms_per_step": st["plan_ms"] / args.steps},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_dt * 1e3, "ffi_calls_per_step": 2 * nops + 8,
                "pattern": "per primitive op: qb_state_apply_pure (sv' = g #> sv) + qb_state_free (old value), "
                           "QASM/Simulation.hs:94-122; lazy clones keep the ops fused",
                "clones_per_step": st_e2e["clones"] / e2e_steps, "passes_per_step": st_e2e["passes"] / e2e_steps,
                "copies_per_step": (st_e2e["cow_fused"] + st_e2e["cow_copies"]) / e2e_steps,
                "check": {"s1_q0": red[0][1], "amp0": [float(w[0].real), float(w[0].imag)]}},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if round_trip:
        line["round_trip"] = round_trip
    if cpu:
        line["cpu_baseline"] = cpu
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="qft_rand", choices=["qft_rand", "adder32", "general"])
    ap.add_argument("--qubits", type=int, default=0)
    ap.add_argument("--round-trip", action="store_true", help="also at 1 GPU: the untimed inverse-circuit check")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed (--impl ours)")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3  # timing rule: at least three warm-up steps
        run_ours(args)


if __name__ == "__main__":
    main()
