"""Pauli rotations without a device: the bit-operation oracle (tests/pauli_rot_oracle.py) against
scipy.linalg.expm of the dense Pauli string, argument checks of qb_apply_pauli_rot, the register budget
of its kernel, and the host op queue's handling of rotations (qb_planner.cpp, compiled on its own)."""
import ctypes as C
import itertools
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import scipy.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THETAS = [0.0, np.pi / 3, -np.pi / 3, np.pi, 2 * np.pi, 0.77]


def _dense(n, s):
    from oracle import dense as D
    one = {"X": D.pauliX(), "Y": D.pauliY(), "Z": D.pauliZ()}
    M = D.ident(n)
    for q, ch in enumerate(s):
        if ch != "I":
            M = D.onJust(n, q, one[ch]) @ M
    return M


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_oracle_matches_expm_on_every_string(n):
    from oracle import structured as S
    from pauli_rot_oracle import pauli_rot
    from qubism_b200.statevec import pauli_masks
    rng = np.random.default_rng(140 + n)
    v = S.gen_state(n, rng, normalized=False) * 1.3
    strings = ["".join(p) for p in itertools.product("IXYZ", repeat=n)]
    xs, zs = pauli_masks(strings, n)
    tol = 1e-12 * max(1.0, float(np.vdot(v, v).real))
    for s, x, z in zip(strings, xs, zs):
        P = _dense(n, s)
        for th in THETAS:
            want = scipy.linalg.expm(-1j * th / 2 * P) @ v
            got = pauli_rot(n, int(x), int(z), th, v)
            assert np.abs(got - want).max() <= tol, (s, th)


def test_argument_errors_need_no_device():
    from qubism_b200 import capi
    L = capi.lib()
    x = (C.c_uint64 * 1)(1)
    z = (C.c_uint64 * 1)(0)
    th = (C.c_double * 1)(0.5)
    assert L.qb_apply_pauli_rot(None, x, z, th, 1) == capi.QB_ERR_ARG
    assert L.qb_apply_pauli_rot(None, x, z, th, -1) == capi.QB_ERR_ARG
    assert L.qb_apply_pauli_rot(None, None, None, None, 0) == capi.QB_ERR_ARG


def test_pauli_rot_kernel_does_not_spill():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "qubism_b200", "csrc", "qb_kernels.cu")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    blocks = re.split(r"ptxas info\s*: Compiling entry function ", r.stderr)
    seen = 0
    for b in blocks:
        if "k_pauli_rot_tile" not in b.split("\n", 1)[0]:
            continue
        seen += 1
        assert "0 bytes spill stores, 0 bytes spill loads" in b, b
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        assert regs * 256 * 3 <= 65536, f"{regs} registers: fewer than 3 CTAs of 256 threads per SM"
    assert seen >= 1


_HARNESS = r"""
#include <cstdio>
#include "qb_internal.h"
using namespace qb;
static int live(const OpQueue &q) { int k = 0; for (auto &o : q.ops) k += !o.dead; return k; }
int main() {
  const double h[8] = {0.7071067811865476, 0, 0.7071067811865476, 0, 0.7071067811865476, 0, -0.7071067811865476, 0};
  const double x[8] = {0, 0, 1, 0, 1, 0, 0, 0};
  OpQueue q;
  q.reset(6, true);
  q.push_1q(2, 0, h);
  q.push_1q(2, 0, h);                 // H H merges into a scalar: nothing left
  printf("hh %d\n", live(q));
  q.reset(6, true);
  q.push_1q(2, 0, h);
  q.push_pauli(1ull << 2, 1ull << 0, 0.8, 0.6);
  q.push_1q(2, 0, h);                 // no merge across the rotation
  printf("hrh %d kind %d nprev %d px %llu pz %llu c %.2f s %.2f\n", live(q), q.ops[1].kind, q.ops[1].nprev,
         (unsigned long long)q.ops[1].px, (unsigned long long)q.ops[1].pz, q.ops[1].m[0], q.ops[1].m[1]);
  q.reset(6, true);
  q.push_1q(3, 1ull << 1, x);
  q.push_pauli(0, 1ull << 3, 0.8, 0.6);
  q.push_1q(3, 1ull << 1, x);         // no CX . CX cancellation across the rotation
  printf("cxrcx %d\n", live(q));
  for (int peep = 0; peep < 2; ++peep) {
    OpQueue qi;
    qi.reset(6, peep != 0);
    qi.push_pauli(0, 0, 0.8, 0.6);    // the identity string: exp(-i theta/2) into the deferred scalar
    printf("ident%d %d %.2f %.2f %llu %llu\n", peep, (int)qi.ops.size(), qi.gscale[0], qi.gscale[1],
           (unsigned long long)qi.folded, (unsigned long long)qi.submitted);
  }
  std::vector<int> perm = {0, 1, 2, 3, 4, 5};  // logical bit = physical bit; 4 local bits
  HostOp r;
  r.kind = 3;
  r.px = 0b110000;
  r.pz = 0b001000;
  std::vector<const HostOp *> p1 = {&r};
  printf("xswaps");
  for (const auto &s : choose_swaps(6, 4, perm, p1, false)) printf(" %d", s.gbit);
  HostOp zr;
  zr.kind = 3;
  zr.pz = 0b110000;
  std::vector<const HostOp *> p2 = {&zr};
  printf("\nzswaps %d\n", (int)choose_swaps(6, 4, perm, p2, false).size());
  // Belady: of the local bits >= 5 the one whose qubit a rotation needs soonest is evicted last
  std::vector<int> perm8 = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9};
  HostOp g, a, b2;
  g.kind = 0; g.type = G_GENERAL; g.target = 9;
  a.kind = 3; a.px = 1ull << 8;
  b2.kind = 3; b2.px = 1ull << 7;
  std::vector<const HostOp *> p3 = {&g, &a, &b2};
  for (const auto &s : choose_swaps(10, 9, perm8, p3, true)) printf("evict %d\n", s.lbit);
}
"""


def test_op_queue_and_swap_choice_on_the_host(tmp_path):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    (tmp_path / "main.cpp").write_text(_HARNESS)
    csrc = os.path.join(ROOT, "qubism_b200", "csrc")
    exe = tmp_path / "harness"
    subprocess.check_call([gxx, "-std=c++17", "-O1", "-I", csrc, str(tmp_path / "main.cpp"),
                           os.path.join(csrc, "qb_planner.cpp"), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    assert out[0] == "hh 0"
    assert out[1] == "hrh 3 kind 3 nprev 7 px 4 pz 1 c 0.80 s 0.60"
    assert out[2] == "cxrcx 3"
    assert out[3] == "ident0 0 0.80 -0.60 1 1" and out[4] == "ident1 0 0.80 -0.60 1 1"
    assert out[5] == "xswaps 4 5"  # X qubits on global bits are needed in the shard ...
    assert out[6] == "zswaps 0"    # ... Z on global qubits is not
    # qubit 9 (global) comes in; the victim is the local bit >= 5 whose qubit is needed furthest ahead:
    # the rotations need bits 8 and 7, so the highest unused one goes
    assert out[7] == "evict 6"
