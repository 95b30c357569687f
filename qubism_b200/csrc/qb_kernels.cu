// CUDA kernels of the qubism state-vector backend, written for sm_100a (B200).
//
// Hot path (SURVEY.md 8a rows a4-a9, a12-a13): k_fused_pass applies a whole *program* of
// queued gates in ONE read + ONE write of the amplitude shard.  A CTA owns a tile of 2^T
// amplitudes selected by T arbitrary physical index bits (the low bits always included so
// every global access is a run of full 128-byte lines).  Each thread keeps 2^R amplitudes
// in registers; a "round" fixes which R tile bits are register-resident, every gate whose
// target is one of them is pure register arithmetic, and between rounds the tile is
// transposed through XOR-swizzled shared memory (conflict-free 128-bit accesses).
// Controls never constrain the tile: they are predicates on register index, thread id or
// tile base.  Diagonal gates can sit on ANY bit.  The kernel is HBM-bound by design:
// 32 B moved per amplitude per pass no matter how many gates the pass carries.
//
// Everything else here is plumbing around that kernel: unfused kernels for shards smaller
// than a tile and for dense k-qubit blocks, deterministic two-stage reductions for
// measurement (a13) and <.> (a15), element-wise vector-space kernels (a15/a16).
#include <cuda_runtime.h>

#include <algorithm>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "qb_internal.h"
#include "qb_kernels.h"

namespace qb {

static int grid_for(uint64_t work, int threads, int sm_count, int per_sm);

__device__ __forceinline__ uint32_t swz(uint32_t u) {
  return u ^ ((u >> 3) & 7u) ^ ((u >> 6) & 7u) ^ ((u >> 9) & 7u) ^ ((u >> 12) & 7u);
}

// ---------------------------------------------------------------- register-resident gates
// Every gate body exists twice: CTRL = false is the common uncontrolled case (straight-line
// DFMA code, nothing predicated); CTRL = true predicates each pair on the control masks.
// ---- the flip mask ------------------------------------------------------------------------
// An X / CX whose controls are NOT register bits never moves data: it toggles bit J of the
// per-thread mask `f`, meaning "the amplitude in register i belongs to logical register index
// i ^ f".  Gates that follow on bit J use the matrix with rows and columns exchanged (one
// select per entry, per thread); controls on register bits test (i ^ f); and at the end of the
// round f folds into the transpose / store ADDRESS as a single XOR (the index maps are linear
// over XOR).  This turns the ~150 ALU instructions of a register-level conditional swap into 3.
//
// Gate bodies come in three flavours (FL): 0 = uncontrolled, no flip possible on this bit
// (planner guarantees it): straight-line DFMA code on uniform-register operands;
// 1 = uncontrolled, flip-aware; 2 = controlled (always flip-aware).
//
// The arithmetic is ordered so that the LAST fused multiply-add of every component reads the
// old value of the register it overwrites: new values never need a second live register, and
// the switch arms leave every amplitude in the register it came in (no shuffle MOVs between
// gates -- they were 55% of all executed instructions in the first version, ncu r01).
template <int R, int J, int FL>
__device__ __forceinline__ void gate_general_m(double (&re)[1 << R], double (&im)[1 << R], const double *m, uint32_t creg_in,
                                               bool ok_thr, uint32_t f) {
  double Ar = m[0], Ai = m[1], Br = m[2], Bi = m[3];
  double Cr = m[4], Ci = m[5], Dr = m[6], Di = m[7];
  if (FL != 0 && ((f >> J) & 1u)) {  // logical pair order is reversed in this thread
    double t;
    t = Ar; Ar = Dr; Dr = t;
    t = Ai; Ai = Di; Di = t;
    t = Br; Br = Cr; Cr = t;
    t = Bi; Bi = Ci; Ci = t;
  }
  const uint32_t creg = (FL == 2) ? creg_in : 0u;
#pragma unroll
  for (int p = 0; p < (1 << (R - 1)); ++p) {
    const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1));
    const int i1 = i0 | (1 << J);
    if (FL != 2 || (ok_thr && (((uint32_t(i0) ^ f) & creg) == creg))) {
      // partial sums that need the OLD x0 / x1
      double P = -Ai * im[i0];
      double Q = Ai * re[i0];
      double Tr = Cr * re[i0];
      double Ti = Cr * im[i0];
      P = fma(Br, re[i1], P);
      Q = fma(Br, im[i1], Q);
      Tr = fma(-Ci, im[i0], Tr);
      Ti = fma(Ci, re[i0], Ti);
      P = fma(-Bi, im[i1], P);
      Q = fma(Bi, re[i1], Q);
      Tr = fma(-Di, im[i1], Tr);
      Ti = fma(Di, re[i1], Ti);
      // in-place finishers
      re[i0] = fma(Ar, re[i0], P);
      im[i0] = fma(Ar, im[i0], Q);
      re[i1] = fma(Dr, re[i1], Tr);
      im[i1] = fma(Dr, im[i1], Ti);
    }
  }
}

template <int R, int J, int FL>
__device__ __forceinline__ void gate_general(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g,
                                             bool ok_thr, uint32_t f) {
  gate_general_m<R, J, FL>(re, im, g.m, g.creg, ok_thr, f);
}

// general complex 2x2 scaled to m00 = 1 (uncontrolled, no flip pending): 12 instead of 16 FP64
// operations per pair
template <int R, int J>
__device__ __forceinline__ void gate_general1_m(double (&re)[1 << R], double (&im)[1 << R], const double *m) {
  const double Br = m[2], Bi = m[3], Cr = m[4], Ci = m[5], Dr = m[6], Di = m[7];
#pragma unroll
  for (int p = 0; p < (1 << (R - 1)); ++p) {
    const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1));
    const int i1 = i0 | (1 << J);
    double Tr = Cr * re[i0];
    double Ti = Cr * im[i0];
    double P = fma(Br, re[i1], re[i0]);
    double Q = fma(Br, im[i1], im[i0]);
    Tr = fma(-Ci, im[i0], Tr);
    Ti = fma(Ci, re[i0], Ti);
    Tr = fma(-Di, im[i1], Tr);
    Ti = fma(Di, re[i1], Ti);
    re[i0] = fma(-Bi, im[i1], P);
    im[i0] = fma(Bi, re[i1], Q);
    re[i1] = fma(Dr, re[i1], Tr);
    im[i1] = fma(Dr, im[i1], Ti);
  }
}

template <int R, int J, int FL>
__device__ __forceinline__ void gate_real_m(double (&re)[1 << R], double (&im)[1 << R], double a, double b, double c,
                                            double d, uint32_t creg_in, bool ok_thr, uint32_t f) {
  if (FL != 0 && ((f >> J) & 1u)) {
    double t;
    t = a; a = d; d = t;
    t = b; b = c; c = t;
  }
  const uint32_t creg = (FL == 2) ? creg_in : 0u;
#pragma unroll
  for (int p = 0; p < (1 << (R - 1)); ++p) {
    const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1));
    const int i1 = i0 | (1 << J);
    if (FL != 2 || (ok_thr && (((uint32_t(i0) ^ f) & creg) == creg))) {
      const double Tr = c * re[i0];
      const double Ti = c * im[i0];
      const double Pr = b * re[i1];
      const double Pi = b * im[i1];
      re[i0] = fma(a, re[i0], Pr);
      im[i0] = fma(a, im[i0], Pi);
      re[i1] = fma(d, re[i1], Tr);
      im[i1] = fma(d, im[i1], Ti);
    }
  }
}

template <int R, int J, int FL>
__device__ __forceinline__ void gate_real(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g,
                                          bool ok_thr, uint32_t f) {
  gate_real_m<R, J, FL>(re, im, g.m[0], g.m[2], g.m[4], g.m[6], g.creg, ok_thr, f);
}

// Conditional swap IN PLACE with the masked-XOR trick (t = (a ^ b) & m; a ^= t; b ^= t), in
// inline PTX so that the optimiser cannot turn it back into selects.  A C++ select
// (a = ok ? b : a ...) makes the compiler rename registers inside the arm, and the resulting
// permutation was repaired with ~64 MOVs around EVERY switch arm of the kernel.
__device__ __forceinline__ void cswap_inplace(double &a, double &b, unsigned long long m) {
  asm volatile(
      "{ .reg .b64 t;\n"
      "  xor.b64 t, %0, %1;\n"
      "  and.b64 t, t, %2;\n"
      "  xor.b64 %0, %0, t;\n"
      "  xor.b64 %1, %1, t;\n"
      "}"
      : "+d"(a), "+d"(b)
      : "l"(m));
}

// X / CX with a control on a REGISTER bit: data really moves (only this flavour exists; the
// others are flip-mask toggles handled in apply_gate)
template <int R, int J, int FL>
__device__ __forceinline__ void gate_swap(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g,
                                          bool ok_thr, uint32_t f) {
  const uint32_t creg = g.creg;
#pragma unroll
  for (int p = 0; p < (1 << (R - 1)); ++p) {
    const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1));
    const int i1 = i0 | (1 << J);
    const bool ok = ok_thr && (((uint32_t(i0) ^ f) & creg) == creg);
    const unsigned long long m = ok ? ~0ull : 0ull;
    cswap_inplace(re[i0], re[i1], m);
    cswap_inplace(im[i0], im[i1], m);
  }
}

// diagonal gate whose target is register bit J
template <int R, int J, int FL>
__device__ __forceinline__ void gate_diag_reg(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g,
                                              bool ok_thr, uint32_t f) {
  double d0r = g.m[0], d0i = g.m[1], d1r = g.m[6], d1i = g.m[7];
  if (FL != 0 && ((f >> J) & 1u)) {
    double t;
    t = d0r; d0r = d1r; d1r = t;
    t = d0i; d0i = d1i; d1i = t;
  }
  const uint32_t creg = (FL == 2) ? g.creg : 0u;
#pragma unroll
  for (int i = 0; i < (1 << R); ++i) {
    const double dr = ((i >> J) & 1) ? d1r : d0r, di = ((i >> J) & 1) ? d1i : d0i;
    if (FL != 2 || (ok_thr && (((uint32_t(i) ^ f) & creg) == creg))) {
      const double t = -di * im[i];
      im[i] = fma(dr, im[i], di * re[i]);
      re[i] = fma(dr, re[i], t);
    }
  }
}

// diagonal gate whose target is a thread-id bit or lies outside the tile: one factor per thread
template <int R>
__device__ __forceinline__ void gate_diag_thr(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g,
                                              bool ok_thr, bool one, uint32_t f) {
  const double dr = one ? g.m[6] : g.m[0], di = one ? g.m[7] : g.m[1];
  const uint32_t creg = g.creg;
#pragma unroll
  for (int i = 0; i < (1 << R); ++i) {
    if (ok_thr && (((uint32_t(i) ^ f) & creg) == creg)) {
      const double t = -di * im[i];
      im[i] = fma(dr, im[i], di * re[i]);
      re[i] = fma(dr, re[i], t);
    }
  }
}

// Rotation [[c,-s],[s,c]], c >= 0, as three shears applied IN PLACE:
//   x0 += t x1;  x1 += s x0;  x0 += t x1      (t = -tan(theta/2), |t| <= 1;  s = sin(theta))
// 3 DFMA per component pair instead of 4 (a DFMA holds the issue port for two cycles on this
// machine, so FP64 instructions are the unit of cost), no temporaries, and each of the three
// sweeps is 2^R independent operations, far longer than the DFMA latency.  With the pair
// order reversed (flip mask) the same rotation is the one by -theta: both coefficients change sign.
template <int R, int J, int FL>
__device__ __forceinline__ void gate_rot(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g,
                                         bool ok_thr, uint32_t f) {
  double t = g.m[0], s = g.m[1];
  if (FL != 0) {
    const long long sg = (long long)((unsigned long long)((f >> J) & 1u) << 63);
    t = __longlong_as_double(__double_as_longlong(t) ^ sg);
    s = __longlong_as_double(__double_as_longlong(s) ^ sg);
  }
  if (FL != 2) {
#pragma unroll
    for (int p = 0; p < (1 << (R - 1)); ++p) {
      const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
      re[i0] = fma(t, re[i1], re[i0]);
      im[i0] = fma(t, im[i1], im[i0]);
    }
#pragma unroll
    for (int p = 0; p < (1 << (R - 1)); ++p) {
      const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
      re[i1] = fma(s, re[i0], re[i1]);
      im[i1] = fma(s, im[i0], im[i1]);
    }
#pragma unroll
    for (int p = 0; p < (1 << (R - 1)); ++p) {
      const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
      re[i0] = fma(t, re[i1], re[i0]);
      im[i0] = fma(t, im[i1], im[i0]);
    }
  } else {
    const uint32_t creg = g.creg;
#pragma unroll
    for (int p = 0; p < (1 << (R - 1)); ++p) {
      const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
      if (ok_thr && (((uint32_t(i0) ^ f) & creg) == creg)) {
        re[i0] = fma(t, re[i1], re[i0]);
        im[i0] = fma(t, im[i1], im[i0]);
        re[i1] = fma(s, re[i0], re[i1]);
        im[i1] = fma(s, im[i0], im[i1]);
        re[i0] = fma(t, re[i1], re[i0]);
        im[i0] = fma(t, im[i1], im[i0]);
      }
    }
  }
}

// One opcode per gate, DENSE for this R (planner-assigned, qb_internal.h): a single jump-table
// dispatch.  The control predicate (thread-id / external masks) is only evaluated in the arms
// that need it.  Labels for J >= R do not exist for this instantiation: they are pushed out of
// the dense range and compile to nothing.
#define QB_LABEL(CLS, FL, JJ) ((JJ) < R ? op_arith(R, CLS, FL, JJ) : 0x1000u + ((CLS) * 3u + (FL)) * 8u + (JJ))
#define QB_ARM(CLS, FN, FL, JJ)                                                                       \
  case QB_LABEL(CLS, FL, JJ):                                                                         \
    if constexpr (JJ < R) FN<R, JJ, FL>(re, im, g, (FL == 2) ? ok_thr(g, tid, basefull) : true, f);   \
    break;
#define QB_ARMS_FL(CLS, FN, FL) QB_ARM(CLS, FN, FL, 0) QB_ARM(CLS, FN, FL, 1) QB_ARM(CLS, FN, FL, 2) QB_ARM(CLS, FN, FL, 3) QB_ARM(CLS, FN, FL, 4)
#define QB_ARMS(CLS, FN) QB_ARMS_FL(CLS, FN, 0) QB_ARMS_FL(CLS, FN, 1) QB_ARMS_FL(CLS, FN, 2)
#define QB_SWAP_ARM(JJ)                                                                \
  case ((JJ) < R ? op_swap_reg(R, JJ) : 0x2000u + (JJ)):                               \
    if constexpr (JJ < R) gate_swap<R, JJ, 2>(re, im, g, ok_thr(g, tid, basefull), f); \
    break;

__device__ __forceinline__ bool ok_thr(const DevGate &g, uint32_t tid, uint64_t basefull) {
  return ((tid & g.cthr) == g.cthr) && ((basefull & g.cext) == g.cext);
}

template <int R>
__device__ __forceinline__ void apply_gate(double (&re)[1 << R], double (&im)[1 << R], const DevGate &g, uint32_t tid,
                                           uint64_t basefull, uint32_t &f) {
  switch (g.op) {
    QB_ARMS(C_GENERAL, gate_general)
    QB_ARMS(C_REAL, gate_real)
    QB_ARMS(C_ROT, gate_rot)
    QB_ARMS(C_DIAG_REG, gate_diag_reg)
    QB_SWAP_ARM(0) QB_SWAP_ARM(1) QB_SWAP_ARM(2) QB_SWAP_ARM(3) QB_SWAP_ARM(4)
    case op_toggle(R):  // flip-mask toggle: no data movement
      f ^= ok_thr(g, tid, basefull) ? (1u << (g.treg & 0xffu)) : 0u;
      break;
    case op_diag_thr(R): {
      const bool one = ((tid & g.dthr) != 0) || ((basefull & g.dext) != 0);
      gate_diag_thr<R>(re, im, g, ok_thr(g, tid, basefull), one, f);
    } break;
    default: break;
  }
}

// ---- LITE passes: uncontrolled rotations and X / CX only (what circuits of U(theta,phi,0) and CX
// layers compile to).  The planner packed each round into DevSteps; a step is straight-line
// code behind uniform skip-branches: no opcode fetch, no dispatch tree, no jump table.
template <int R, int J>
__device__ __forceinline__ void step_rot(double (&re)[1 << R], double (&im)[1 << R], const DevStep &S, uint32_t f,
                                         bool flip) {
  {
    const double t = S.slot[J][0], s = S.slot[J][1];
    if (flip) {  // a flip may be pending on this bit: per-thread sign
      const long long sg = (long long)((unsigned long long)((f >> J) & 1u) << 63);
      const double tv = __longlong_as_double(__double_as_longlong(t) ^ sg);
      const double sv = __longlong_as_double(__double_as_longlong(s) ^ sg);
#pragma unroll
      for (int p = 0; p < (1 << (R - 1)); ++p) {
        const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
        re[i0] = fma(tv, re[i1], re[i0]);
        im[i0] = fma(tv, im[i1], im[i0]);
      }
#pragma unroll
      for (int p = 0; p < (1 << (R - 1)); ++p) {
        const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
        re[i1] = fma(sv, re[i0], re[i1]);
        im[i1] = fma(sv, im[i0], im[i1]);
      }
#pragma unroll
      for (int p = 0; p < (1 << (R - 1)); ++p) {
        const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
        re[i0] = fma(tv, re[i1], re[i0]);
        im[i0] = fma(tv, im[i1], im[i0]);
      }
    } else {  // coefficients straight from the uniform datapath
#pragma unroll
      for (int p = 0; p < (1 << (R - 1)); ++p) {
        const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
        re[i0] = fma(t, re[i1], re[i0]);
        im[i0] = fma(t, im[i1], im[i0]);
      }
#pragma unroll
      for (int p = 0; p < (1 << (R - 1)); ++p) {
        const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
        re[i1] = fma(s, re[i0], re[i1]);
        im[i1] = fma(s, im[i0], im[i1]);
      }
#pragma unroll
      for (int p = 0; p < (1 << (R - 1)); ++p) {
        const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
        re[i0] = fma(t, re[i1], re[i0]);
        im[i0] = fma(t, im[i1], im[i0]);
      }
    }
  }
}

// the 1-qubit slot of register bit J: uniform branches on the slot kind
// (ROT_ONLY: the instantiation for passes whose slots are all rotations -- a third of the code)
template <int R, int J, bool ROT_ONLY>
__device__ __forceinline__ void step_slot(double (&re)[1 << R], double (&im)[1 << R], const DevStep &S, uint32_t kinds,
                                          uint32_t f) {
  const uint32_t kind = (kinds >> (4 * J)) & 15u;
  if (kind == SLOT_NONE) return;
  const bool flip = (kind & SLOT_FLIP) != 0;
  const uint32_t cls = kind & SLOT_CLASS;
  if (ROT_ONLY || cls == SLOT_ROT) {
    step_rot<R, J>(re, im, S, f, flip);
  } else if (cls == SLOT_GENERAL1) {
    gate_general1_m<R, J>(re, im, S.slot[J]);
  } else if (cls == SLOT_REAL) {
    const double a = S.slot[J][0], b = S.slot[J][1], c = S.slot[J][2], d = S.slot[J][3];
    if (flip) gate_real_m<R, J, 1>(re, im, a, b, c, d, 0u, true, f);
    else gate_real_m<R, J, 0>(re, im, a, b, c, d, 0u, true, f);
  } else {
    if (flip) gate_general_m<R, J, 1>(re, im, S.slot[J], 0u, true, f);
    else gate_general_m<R, J, 0>(re, im, S.slot[J], 0u, true, f);
  }
}

template <int R, int J>
__device__ __forceinline__ void step_swap(double (&re)[1 << R], double (&im)[1 << R], const DevStep &S, uint32_t tid,
                                          uint64_t basefull, uint32_t f) {
  const bool okt = ((tid & S.swap_cthr) == S.swap_cthr) && ((basefull & S.swap_cext) == S.swap_cext);
  const uint32_t creg = S.swap_creg;
#pragma unroll
  for (int p = 0; p < (1 << (R - 1)); ++p) {
    const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
    const bool ok = okt && (((uint32_t(i0) ^ f) & creg) == creg);
    const unsigned long long m = ok ? ~0ull : 0ull;
    cswap_inplace(re[i0], re[i1], m);
    cswap_inplace(im[i0], im[i1], m);
  }
}

// XOR swap in place (inline PTX so that the optimiser cannot rename the registers: a renamed
// arm is repaired with moves at the join)
__device__ __forceinline__ void swap_inplace(double &a, double &b) {
  asm volatile(
      "xor.b64 %0, %0, %1;\n"
      "xor.b64 %1, %1, %0;\n"
      "xor.b64 %0, %0, %1;"
      : "+d"(a), "+d"(b));
}

template <int R, int J, int K>
__device__ __forceinline__ void step_swap_static(double (&re)[1 << R], double (&im)[1 << R]) {
#pragma unroll
  for (int p = 0; p < (1 << (R - 1)); ++p) {
    const int i0 = ((p >> J) << (J + 1)) | (p & ((1 << J) - 1)), i1 = i0 | (1 << J);
    if ((i0 >> K) & 1) {
      swap_inplace(re[i0], re[i1]);
      swap_inplace(im[i0], im[i1]);
    }
  }
}

template <int R>
__device__ __forceinline__ void step_swap_static_dispatch(double (&re)[1 << R], double (&im)[1 << R], uint32_t jk) {
#define QB_SS(JJ, KK)                                                             \
  case (JJ) * 8 + (KK):                                                           \
    if constexpr ((JJ) < R && (KK) < R && (JJ) != (KK)) step_swap_static<R, JJ, KK>(re, im); \
    break;
  switch (jk) {
    QB_SS(0, 1) QB_SS(0, 2) QB_SS(0, 3) QB_SS(0, 4) QB_SS(1, 0) QB_SS(1, 2) QB_SS(1, 3) QB_SS(1, 4) QB_SS(2, 0) QB_SS(2, 1)
    QB_SS(2, 3) QB_SS(2, 4) QB_SS(3, 0) QB_SS(3, 1) QB_SS(3, 2) QB_SS(3, 4) QB_SS(4, 0) QB_SS(4, 1) QB_SS(4, 2) QB_SS(4, 3)
    default: break;
  }
#undef QB_SS
}

template <int R, bool ROT_ONLY>
__device__ __forceinline__ void apply_step(double (&re)[1 << R], double (&im)[1 << R], const DevStep &S, uint32_t tid,
                                           uint64_t basefull, uint32_t &f) {
  const uint32_t kinds = S.kinds;
  step_slot<R, 0, ROT_ONLY>(re, im, S, kinds, f);
  step_slot<R, 1, ROT_ONLY>(re, im, S, kinds, f);
  step_slot<R, 2, ROT_ONLY>(re, im, S, kinds, f);
  if constexpr (R > 3) step_slot<R, 3, ROT_ONLY>(re, im, S, kinds, f);
  if constexpr (R > 4) step_slot<R, 4, ROT_ONLY>(re, im, S, kinds, f);
  const uint32_t ntog = S.ntog;
#pragma unroll
  for (int k = 0; k < kStepToggles; ++k) {
    if (k < ntog) {
      const bool ok = ((tid & S.tog[k].cthr) == S.tog[k].cthr) && ((basefull & S.tog[k].cext) == S.tog[k].cext);
      f ^= ok ? (1u << S.tog[k].bit) : 0u;
    }
  }
  const uint32_t sj = S.swap_j;
  if (sj != 0xffu) {
    if (sj & 16u) {  // static: the pairs whose index has control bit K set swap, in every thread
      const uint32_t jk = (sj & 7u) * 8u + (uint32_t)(__ffs((int)S.swap_creg) - 1);
      step_swap_static_dispatch<R>(re, im, jk);
    } else {
      const uint32_t j = sj & 7u;
      if (j == 0) step_swap<R, 0>(re, im, S, tid, basefull, f);
      else if (j == 1) step_swap<R, 1>(re, im, S, tid, basefull, f);
      else if (j == 2) step_swap<R, 2>(re, im, S, tid, basefull, f);
      else if (j == 3) { if constexpr (R > 3) step_swap<R, 3>(re, im, S, tid, basefull, f); }
      else { if constexpr (R > 4) step_swap<R, 4>(re, im, S, tid, basefull, f); }
    }
  }
}

// ---------------------------------------------------------------- the fused pass
template <int T, int R>
__device__ __forceinline__ uint32_t thread_sidx(const DevRound &rd, uint32_t tid) {
  uint32_t u = 0;
#pragma unroll
  for (int j = 0; j < T - R; ++j) u |= ((tid >> j) & 1u) << rd.tid_pos[j];
  return swz(u);
}

template <int T, int R>
__device__ __forceinline__ uint64_t thread_goff(const DevPass &P, const DevRound &rd, uint32_t tid) {
  uint64_t o = 0;
#pragma unroll
  for (int j = 0; j < T - R; ++j) o |= uint64_t((tid >> j) & 1u) << P.tile_pos[rd.tid_pos[j]];
  return o;
}

// The pass program (header + gates) travels as a __grid_constant__ kernel parameter: it lives
// in the constant bank, is read through the uniform datapath (warp-uniform indices), costs no
// shared memory, no upload, and no shared-memory round trip per gate.
struct PassProgram {
  DevPass hdr;
  union {
    DevGate gates[kMaxPassGates];
    DevStep steps[kMaxSteps];  // lite passes
  };
};
static_assert(sizeof(PassProgram) <= 32000, "kernel parameter space");

// 256-bit global accesses (sm_100: LDG.256 / STG.256): when tile bit 0 is a REGISTER bit of the
// load / store round, the two registers of a pair are one whole 32-byte sector of the same
// thread -- one instruction instead of two, and no half-sector requests.
__device__ __forceinline__ void ld_pair256(const double2 *p, double &a0, double &a1, double &b0, double &b1) {
  asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a0), "=d"(a1), "=d"(b0), "=d"(b1) : "l"(p));
}
__device__ __forceinline__ void st_pair256(double2 *p, double a0, double a1, double b0, double b1) {
  asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a0), "d"(a1), "d"(b0), "d"(b1) : "memory");
}

template <int T, int R>
__host__ __device__ constexpr size_t fused_smem_bytes() {
  return (size_t(16) << T) + size_t(kMaxRounds) * (size_t(1) << (T - R)) * sizeof(uint16_t) +
         size_t(2) * (size_t(1) << (T - R)) * sizeof(uint64_t) + (size_t(1) << (T - 3)) * sizeof(uint32_t);
}

template <int T, int R, int MINB, int LITE>
__global__ void __launch_bounds__(1 << (T - R), MINB)
    k_fused_pass(double2 *amps, const double2 *src_amps, unsigned long long ntiles, const __grid_constant__ PassProgram prog) {
  // src_amps == amps: in place (the normal case).  Otherwise the pass reads the tiles of src_amps
  // and writes amps: the copy-on-write of a lazily cloned state rides on its first pass.
  constexpr int NR = 1 << R;
  constexpr int NT = 1 << (T - R);
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const uint32_t tid = threadIdx.x;
  // after the tile: for every round, each thread's swizzled shared-memory index (computed once
  // per kernel; the persistent tile loop then needs one 16-bit load per transpose side)
  uint16_t *sidx_tab = reinterpret_cast<uint16_t *>(smem_raw + (size_t(16) << T));
  const DevPass &P = prog.hdr;
  const DevGate *G = prog.gates;
  const uint32_t nrounds = P.nrounds;
  for (uint32_t r = 0; r < nrounds; ++r) sidx_tab[r * NT + tid] = (uint16_t)thread_sidx<T, R>(P.rounds[r], tid);
  // (each thread only ever reads its own entries: no barrier needed)
  // ... and its element offset inside a tile for the load and the store layout (kept in shared
  // memory, not in four registers: the gate loop needs every register it can get)
  uint64_t *goff_tab = reinterpret_cast<uint64_t *>(sidx_tab + kMaxRounds * NT);
  goff_tab[tid] = thread_goff<T, R>(P, P.rounds[0], tid);
  {  // the store layout: where the planner sends each tile bit (out_pos == tile_pos for an in-place pass)
    uint64_t o = 0;
#pragma unroll
    for (int j = 0; j < T - R; ++j) o |= uint64_t((tid >> j) & 1u) << P.out_pos[P.rounds[nrounds - 1].tid_pos[j]];
    goff_tab[NT + tid] = o;
  }
  // ... and the 128-byte lines of a tile this thread prefetches (offsets in units of 8 elements)
  constexpr int LPT = 1 << (R - 3);  // lines per thread
  uint32_t *line_tab = reinterpret_cast<uint32_t *>(goff_tab + 2 * NT);
#pragma unroll
  for (int k = 0; k < LPT; ++k) {
    const uint32_t l = tid + k * NT;
    uint64_t o = 0;
#pragma unroll
    for (int j = 0; j < T - 3; ++j) o |= uint64_t((l >> j) & 1u) << P.tile_pos[3 + j];
    line_tab[k * NT + tid] = (uint32_t)(o >> 3);
  }

  const uint32_t ntiles32 = (uint32_t)ntiles;
  const uint32_t stride = gridDim.x;
  const uint32_t first = blockIdx.x;
  const uint32_t iters = (ntiles32 + stride - 1) / stride;
  double re[NR], im[NR];
  uint32_t f = 0;  // flip mask: register i holds logical register index i ^ f
  uint64_t base = 0, next_base = 0;
  for (uint32_t it = 0; it <= iters; ++it) {
    const uint32_t tile_id = first + it * stride;
    // ---------------- store the finished tile, then load the next one
    const uint32_t dbg = P.dbg_skip;  // profiling switches (0 in production)
    if (it > 0 && tile_id - stride < ntiles32 && !(dbg & 2u)) {
      // coalesced store with the last round's layout (register strides are distinct bits, so
      // the pending flip mask is one XOR on the element index)
      uint64_t st[R];
      uint64_t fx = 0;
#pragma unroll
      for (int j = 0; j < R; ++j) {
        st[j] = 1ull << P.out_pos[P.rounds[nrounds - 1].reg_pos[j]];
        fx |= ((f >> j) & 1u) ? st[j] : 0ull;
      }
      // out of place: tile number t is block t of the destination (its qubits now sit on the low bits)
      uint64_t obase = base;
      if (P.oop) {  // block address: the tile number's bits, group by group, at their new places
        obase = 0;
        uint64_t t = tile_id - stride;
        const uint32_t nor = P.onruns;
        for (uint32_t k = 0; k < nor; ++k) {
          const uint32_t len = P.orun_len[k];
          obase |= (t & ((1ull << len) - 1ull)) << P.orun_shift[k];
          t >>= len;
        }
      }
      // the stores carry a global<->local swap: every amplitude goes to the rank that owns it after it,
      // over NVLink (the victims' bits of its address pick the rank and take this rank's old values)
      const bool xch = P.oop && P.xch.n != 0;
      auto dst_of = [&](uint64_t a) -> double2 * {
        if (!xch) return amps + a;
        uint32_t rr = P.xch.rbase;
        for (uint32_t k = 0; k < P.xch.n; ++k) rr |= uint32_t((a >> P.xch.lbit[k]) & 1ull) << P.xch.rbit[k];
        return reinterpret_cast<double2 *>(P.xch.peer[rr]) + ((a & ~P.xch.vmask) | P.xch.vconst);
      };
      if (st[0] == 1ull) {  // register bit 0 is physical bit 0: 32-byte stores of register pairs
        const uint64_t at = (obase + goff_tab[NT + tid]) ^ (fx & ~1ull);
        const bool sw = (f & 1u) != 0;  // pending flip on that bit: the pair goes out in reverse order
#pragma unroll
        for (int i = 0; i < NR; i += 2) {
          uint64_t off = 0;
#pragma unroll
          for (int j = 1; j < R; ++j)
            if ((i >> j) & 1) off |= st[j];
          st_pair256(dst_of(at ^ off), sw ? re[i + 1] : re[i], sw ? im[i + 1] : im[i], sw ? re[i] : re[i + 1],
                     sw ? im[i] : im[i + 1]);
        }
      } else {
        const uint64_t at = (obase + goff_tab[NT + tid]) ^ fx;
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          uint64_t off = 0;
#pragma unroll
          for (int j = 0; j < R; ++j)
            if ((i >> j) & 1) off |= st[j];
          __stcs(dst_of(at ^ off), make_double2(re[i], im[i]));
        }
      }
    }
    const bool active = it < iters && tile_id < ntiles32;
    if (active) {
      // deposit the tile id into the free non-tile bit positions (the prefetch of the previous
      // iteration already did it for this tile)
      if (it > 0 && P.l2_prefetch == 1 && !(dbg & 1u)) {
        base = next_base;
      } else {
        base = 0;
        uint64_t t = tile_id;
        const uint32_t nruns = P.nruns;
        for (uint32_t k = 0; k < nruns; ++k) {
          const uint32_t len = P.run_len[k];
          base |= (t & ((1ull << len) - 1ull)) << P.run_shift[k];
          t >>= len;
        }
        base |= P.base_fixed;  // only live tiles are enumerated (qb_planner.cpp, "dead tiles")
      }
      // coalesced load: lanes walk the low tile bits, registers stride over the round-0 bits
      const uint64_t goff_ld = goff_tab[tid];
      const double2 *src = src_amps + base + goff_ld;
      uint64_t st[R];
#pragma unroll
      for (int j = 0; j < R; ++j) st[j] = 1ull << P.tile_pos[P.rounds[0].reg_pos[j]];
      if (!(dbg & 1u)) {
        if (st[0] == 1ull) {  // register bit 0 is physical bit 0: 32-byte loads of register pairs
#pragma unroll
          for (int i = 0; i < NR; i += 2) {
            uint64_t off = 0;
#pragma unroll
            for (int j = 1; j < R; ++j)
              if ((i >> j) & 1) off += st[j];
            ld_pair256(src + off, re[i], im[i], re[i + 1], im[i + 1]);
          }
        } else {
#pragma unroll
          for (int i = 0; i < NR; ++i) {
            uint64_t off = 0;
#pragma unroll
            for (int j = 0; j < R; ++j)
              if ((i >> j) & 1) off += st[j];
            const double2 a = __ldcs(src + off);
            re[i] = a.x;
            im[i] = a.y;
          }
        }
      }
      // While this tile is in registers, pull the group's NEXT tile from HBM into L2 (one request
      // per 128-byte line): its loads then hit L2 instead of waiting on DRAM, which overlaps
      // the memory phase of tile k+1 with the gate / transpose phases of tile k.
      const uint32_t next_id = tile_id + stride * P.l2_prefetch;  // prefetch distance in tiles of this CTA
      if (P.l2_prefetch && next_id < ntiles32 && !(dbg & 1u)) {
        uint64_t nbase = 0;
        uint64_t t = next_id;
        const uint32_t nruns = P.nruns;
        for (uint32_t k = 0; k < nruns; ++k) {
          const uint32_t len = P.run_len[k];
          nbase |= (t & ((1ull << len) - 1ull)) << P.run_shift[k];
          t >>= len;
        }
        nbase |= P.base_fixed;
        next_base = nbase;
#pragma unroll
        for (int k = 0; k < LPT; ++k)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(src_amps + nbase + (uint64_t(line_tab[k * NT + tid]) << 3)));
      }
    }
    if (!active) break;
    const uint64_t basefull = base | P.rank_bits;
    f = 0;
    for (uint32_t r = 0; r < nrounds; ++r) {
      const DevRound &RD = P.rounds[r];
      if (r > 0) {  // transpose through swizzled shared memory: new register-resident bits
        if (!(dbg & 4u)) {
          const DevRound &PR = P.rounds[r - 1];
          // byte offsets throughout: address = tile + (thread part ^ register part)
          uint32_t us = uint32_t(sidx_tab[(r - 1) * NT + tid]) << 4;
          uint32_t sx[R];
#pragma unroll
          for (int j = 0; j < R; ++j) {
            sx[j] = PR.reg_sx[j] << 4;
            us ^= ((f >> j) & 1u) ? sx[j] : 0u;  // fold the flip mask into the address
          }
          f = 0;
          // A warp-local transpose only touches this warp's own slots: the barriers shrink to
          // __syncwarp() and the warps of the CTA stay decoupled.  For a CTA-wide transpose the
          // barrier that frees the buffer ("everyone finished reading the previous layout") was
          // taken EARLY, right after the previous transpose's loads (below), when the warps had
          // just left a barrier together: taking it here would make every warp wait for the
          // slowest one's whole gate phase and then send all the stores to the LSU at once.
          const bool local = RD.warp_local != 0;
          if (local) __syncwarp();
#pragma unroll
          for (int i = 0; i < NR; ++i) {
            uint32_t c = 0;  // uniform: folds at compile time into one XOR operand per register
#pragma unroll
            for (int j = 0; j < R; ++j)
              if ((i >> j) & 1) c ^= sx[j];
            *reinterpret_cast<double2 *>(smem_raw + (us ^ c)) = make_double2(re[i], im[i]);
          }
          if (local) __syncwarp(); else __syncthreads();
          const uint32_t ul = uint32_t(sidx_tab[r * NT + tid]) << 4;
#pragma unroll
          for (int j = 0; j < R; ++j) sx[j] = RD.reg_sx[j] << 4;
#pragma unroll
          for (int i = 0; i < NR; ++i) {
            uint32_t c = 0;
#pragma unroll
            for (int j = 0; j < R; ++j)
              if ((i >> j) & 1) c ^= sx[j];
            const double2 a = *reinterpret_cast<const double2 *>(smem_raw + (ul ^ c));
            re[i] = a.x;
            im[i] = a.y;
          }
          // free the buffer for the next CTA-wide transpose (of this tile, or the first one of the
          // next tile) now
          // (wrapping to the next tile: also when the warps' slot regions change between the last
          //  and the first round -- rounds[0].warp_local == 0 -- or a fast warp's first local
          //  transpose of the next tile would overwrite slots a slow warp is still reading here)
          if (r + 1 < nrounds ? P.rounds[r + 1].warp_local == 0
                              : (P.rounds[1].warp_local == 0 || P.rounds[0].warp_local == 0))
            __syncthreads();
        }
      }
      const uint32_t wb = LITE != 0 ? RD.step_begin : RD.gate_begin, we = LITE != 0 ? RD.step_end : RD.gate_end;
      if (wb < we && !(dbg & 8u)) {
        if constexpr (LITE != 0) {
          for (uint32_t si = wb; si < we; ++si) apply_step<R, LITE == 1>(re, im, prog.steps[si], tid, basefull, f);
        } else {
          for (uint32_t gi = wb; gi < we; ++gi) apply_gate<R>(re, im, G[gi], tid, basefull, f);
        }
      }
    }
    // deferred global scalar (folded u1-type phases, qb_scale); exactly 1 is skipped: it is the
    // identity, and 0 * inf must not turn an infinite amplitude into NaN
    if (P.has_gscale && !(P.gscale[0] == 1.0 && P.gscale[1] == 0.0)) {
      const double sr = P.gscale[0], si = P.gscale[1];
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        const double xr = re[i], xi = im[i];
        re[i] = sr * xr - si * xi;
        im[i] = sr * xi + si * xr;
      }
    }
  }
}

struct FusedVariant {
  int T, R, threads;
  int minb, minb_lite;   // resident CTAs per SM each instantiation is compiled for
  const void *fn[3];     // [0] interpreter (every gate class), [1] steps of rotations and X / CX, [2] steps of
                         // rotation / real / general slots and X / CX
  size_t smem;
};

// MINB_ / MINBL_: the interpreter wants occupancy (its arms are short dependent chains); the
// step kernels want registers (128: no spills, every sweep is 2^R independent DFMAs) -- measured.
#define QB_VARIANT(T_, R_, MINB_, MINBL_)                                                          \
  {T_, R_, 1 << (T_ - R_), MINB_, MINBL_,                                                          \
   {(const void *)&k_fused_pass<T_, R_, MINB_, 0>, (const void *)&k_fused_pass<T_, R_, MINBL_, 1>, \
    (const void *)&k_fused_pass<T_, R_, MINBL_, 2>},                                               \
   fused_smem_bytes<T_, R_>()}

#ifdef QB_QUICK_COMPILE  // developer switch: only the default instantiation (fast ptxas experiments)
static const FusedVariant kVariants[] = {QB_VARIANT(12, 4, 3, 2)};
#else
static const FusedVariant kVariants[] = {
    QB_VARIANT(10, 3, 4, 4), QB_VARIANT(10, 4, 4, 4), QB_VARIANT(11, 3, 3, 3), QB_VARIANT(11, 4, 4, 4),
    QB_VARIANT(11, 5, 6, 6), QB_VARIANT(12, 3, 2, 2), QB_VARIANT(12, 4, 3, 2), QB_VARIANT(12, 5, 3, 3),
    QB_VARIANT(13, 4, 1, 1), QB_VARIANT(13, 5, 1, 1),
};
#endif

static const FusedVariant *find_variant(int T, int R) {
  for (const auto &v : kVariants)
    if (v.T == T && v.R == R) return &v;
  return nullptr;
}

bool fused_variant_supported(int tile_bits, int reg_bits) { return find_variant(tile_bits, reg_bits) != nullptr; }
#ifndef QB_QUICK_COMPILE
static_assert(sizeof(kVariants) / sizeof(kVariants[0]) == sizeof(kFusedVariants) / sizeof(kFusedVariants[0]), "variant tables out of sync");
#endif

cudaError_t launch_fused_pass(double2 *amps, const double2 *src, const uint8_t *blob, uint32_t blob_bytes, int tile_bits,
                              int reg_bits, uint64_t ntiles, int sm_count, cudaStream_t stream, int *grid_out) {
  const FusedVariant *v = find_variant(tile_bits, reg_bits);
  if (!v) return cudaErrorInvalidValue;
  if (blob_bytes > sizeof(PassProgram) || blob_bytes < sizeof(DevPass)) return cudaErrorInvalidValue;
  static thread_local PassProgram prog;  // the launch copies it into the command buffer
  memcpy(&prog, blob, blob_bytes);
  const void *fn = v->fn[prog.hdr.lite <= 2 ? prog.hdr.lite : 0];
  const size_t smem = v->smem;
  const int threads = v->threads;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, threads, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorLaunchOutOfResources;
  uint64_t grid = uint64_t(sm_count) * uint64_t(occ);
  if (grid > ntiles) grid = ntiles;
  if (grid_out) *grid_out = (int)grid;
  unsigned long long nt = ntiles;
  if (!src) src = amps;
  void *args[] = {(void *)&amps, (void *)&src, (void *)&nt, (void *)&prog};
  return cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(threads), args, smem, stream);
}

// ---------------------------------------------------------------- unfused kernels
// One gate, one sweep: shards smaller than a tile, and the `fuse = 0` reference schedule.
__global__ void __launch_bounds__(256) k_simple_gate(double2 *__restrict__ amps, uint64_t npairs, int tbit,
                                                     uint64_t cmask, uint64_t rank_bits, uint32_t type,
                                                     double ar, double ai, double br, double bi, double cr,
                                                     double ci, double dr, double di) {
  const uint64_t stride = 1ull << tbit;
  for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < npairs;
       p += uint64_t(gridDim.x) * blockDim.x) {
    const uint64_t i0 = ((p >> tbit) << (tbit + 1)) | (p & (stride - 1));
    if (((i0 | rank_bits) & cmask) != cmask) continue;
    const uint64_t i1 = i0 | stride;
    const double2 x0 = amps[i0], x1 = amps[i1];
    double2 y0, y1;
    if (type == G_SWAP) {
      y0 = x1;
      y1 = x0;
    } else {
      y0.x = ar * x0.x - ai * x0.y + br * x1.x - bi * x1.y;
      y0.y = ar * x0.y + ai * x0.x + br * x1.y + bi * x1.x;
      y1.x = cr * x0.x - ci * x0.y + dr * x1.x - di * x1.y;
      y1.y = cr * x0.y + ci * x0.x + dr * x1.y + di * x1.x;
    }
    amps[i0] = y0;
    amps[i1] = y1;
  }
}

// diagonal gate / controlled scalar with the target anywhere (local or rank bit)
__global__ void __launch_bounds__(256) k_simple_diag(double2 *__restrict__ amps, uint64_t n, uint64_t tmask,
                                                     uint64_t cmask, uint64_t rank_bits, double d0r, double d0i,
                                                     double d1r, double d1i) {
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const uint64_t full = i | rank_bits;
    if ((full & cmask) != cmask) continue;
    const bool one = (full & tmask) != 0;
    const double dr = one ? d1r : d0r, di = one ? d1i : d0i;
    const double2 x = amps[i];
    amps[i] = make_double2(dr * x.x - di * x.y, dr * x.y + di * x.x);
  }
}

// dense 2^K x 2^K block on K arbitrary local bits (QGate.hs:58-59,142-144: kronecker / <> blocks)
template <int K>
__global__ void __launch_bounds__(128) k_simple_kq(double2 *__restrict__ amps, uint64_t ngroups, const int *__restrict__ bits_sorted,
                                                   const int *__restrict__ bits_order, const double2 *__restrict__ mat,
                                                   uint64_t cmask, uint64_t rank_bits) {
  constexpr int D = 1 << K;
  __shared__ double2 ms[D * D];
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) ms[i] = mat[i];
  __syncthreads();
  int sb[K], ob[K];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    sb[j] = bits_sorted[j];  // ascending physical positions
    ob[j] = bits_order[j];   // position of matrix index bit j (bit 0 = least significant)
  }
  for (uint64_t gidx = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; gidx < ngroups;
       gidx += uint64_t(gridDim.x) * blockDim.x) {
    uint64_t base = gidx;
#pragma unroll
    for (int j = 0; j < K; ++j) base = ((base >> sb[j]) << (sb[j] + 1)) | (base & ((1ull << sb[j]) - 1));
    if (((base | rank_bits) & cmask) != cmask) continue;
    double2 x[D];
#pragma unroll
    for (int a = 0; a < D; ++a) {
      uint64_t off = 0;
#pragma unroll
      for (int j = 0; j < K; ++j)
        if ((a >> j) & 1) off |= 1ull << ob[j];
      x[a] = amps[base | off];
    }
#pragma unroll 1
    for (int row = 0; row < D; ++row) {
      double yr = 0.0, yi = 0.0;
#pragma unroll
      for (int a = 0; a < D; ++a) {
        const double2 mm = ms[row * D + a];
        yr += mm.x * x[a].x - mm.y * x[a].y;
        yi += mm.x * x[a].y + mm.y * x[a].x;
      }
      uint64_t off = 0;
#pragma unroll
      for (int j = 0; j < K; ++j)
        if ((row >> j) & 1) off |= 1ull << ob[j];
      amps[base | off] = make_double2(yr, yi);
    }
  }
}

static int grid_for(uint64_t work, int threads, int sm_count, int per_sm) {
  uint64_t g = (work + threads - 1) / threads;
  uint64_t cap = uint64_t(sm_count) * per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

cudaError_t launch_simple_gate(double2 *amps, int local_bits, int tbit, uint64_t cmask, uint64_t rank_bits,
                               uint32_t type, const double m[8], int sm_count, cudaStream_t stream) {
  const uint64_t npairs = 1ull << (local_bits - 1);
  k_simple_gate<<<grid_for(npairs, 256, sm_count, 8), 256, 0, stream>>>(amps, npairs, tbit, cmask, rank_bits, type,
                                                                       m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7]);
  return cudaGetLastError();
}

cudaError_t launch_simple_diag(double2 *amps, int local_bits, uint64_t tmask, uint64_t cmask, uint64_t rank_bits,
                               const double d0[2], const double d1[2], int sm_count, cudaStream_t stream) {
  const uint64_t n = 1ull << local_bits;
  k_simple_diag<<<grid_for(n, 256, sm_count, 8), 256, 0, stream>>>(amps, n, tmask, cmask, rank_bits, d0[0], d0[1],
                                                                  d1[0], d1[1]);
  return cudaGetLastError();
}

cudaError_t launch_simple_kq(double2 *amps, int local_bits, int k, const int *bits_sorted_dev,
                             const int *bits_order_dev, const double2 *mat_dev, uint64_t cmask, uint64_t rank_bits,
                             int sm_count, cudaStream_t stream) {
  const uint64_t ngroups = 1ull << (local_bits - k);
  const int g = grid_for(ngroups, 128, sm_count, 8);
  switch (k) {
    case 1: k_simple_kq<1><<<g, 128, 0, stream>>>(amps, ngroups, bits_sorted_dev, bits_order_dev, mat_dev, cmask, rank_bits); break;
    case 2: k_simple_kq<2><<<g, 128, 0, stream>>>(amps, ngroups, bits_sorted_dev, bits_order_dev, mat_dev, cmask, rank_bits); break;
    case 3: k_simple_kq<3><<<g, 128, 0, stream>>>(amps, ngroups, bits_sorted_dev, bits_order_dev, mat_dev, cmask, rank_bits); break;
    case 4: k_simple_kq<4><<<g, 128, 0, stream>>>(amps, ngroups, bits_sorted_dev, bits_order_dev, mat_dev, cmask, rank_bits); break;
    case 5: k_simple_kq<5><<<g, 128, 0, stream>>>(amps, ngroups, bits_sorted_dev, bits_order_dev, mat_dev, cmask, rank_bits); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------- global<->local qubit swap
// In-place pairwise exchange over NVLink peer memory (SURVEY.md 8e, no NCCL in the data path,
// no bounce buffer): thread t reads its own element and the partner GPU's element through the
// IPC-mapped peer pointer, and writes each where the other was.  The two ranks of a pair split
// the index range in halves, so both GPUs' SMs work and both link directions carry the same
// load: per rank (1 - 2^-k) of the shard crosses NVLink each way for a k-bit swap.
struct SwapGeom {
  uint32_t nruns;
  uint32_t run_shift[kMaxRuns];  // deposit of the free index into the non-swapped local bits
  uint32_t run_len[kMaxRuns];
  uint64_t my_place, peer_place; // the swapped local bits: my elements that leave / the peer's that arrive
};

__global__ void __launch_bounds__(256) k_peer_swap(double2 *__restrict__ mine, double2 *__restrict__ peer,
                                                   unsigned long long t_begin, unsigned long long t_end,
                                                   const __grid_constant__ SwapGeom geo) {
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long t0 = t_begin + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; t0 < t_end;
       t0 += 4 * stride) {
    uint64_t im[4], ip[4];
    double2 a[4], b[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const unsigned long long t = t0 + u * stride;
      uint64_t idx = 0, rest = t;
      for (uint32_t k = 0; k < geo.nruns; ++k) {
        idx |= (rest & ((1ull << geo.run_len[k]) - 1ull)) << geo.run_shift[k];
        rest >>= geo.run_len[k];
      }
      im[u] = idx | geo.my_place;
      ip[u] = idx | geo.peer_place;
      if (t < t_end) {
        a[u] = mine[im[u]];
        b[u] = peer[ip[u]];  // NVLink read
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (t0 + u * stride < t_end) {
        mine[im[u]] = b[u];
        peer[ip[u]] = a[u];  // NVLink write
      }
    }
  }
}

cudaError_t launch_peer_swap(double2 *mine, double2 *peer, uint64_t t_begin, uint64_t t_end, int local_bits,
                             uint64_t swapped_mask, uint64_t my_place, uint64_t peer_place, int sm_count,
                             cudaStream_t stream) {
  SwapGeom geo{};
  int b = 0;
  while (b < local_bits) {
    if (swapped_mask & (1ull << b)) {
      ++b;
      continue;
    }
    int e = b;
    while (e < local_bits && !(swapped_mask & (1ull << e))) ++e;
    if (geo.nruns >= kMaxRuns) return cudaErrorInvalidValue;
    geo.run_shift[geo.nruns] = b;
    geo.run_len[geo.nruns] = e - b;
    ++geo.nruns;
    b = e;
  }
  geo.my_place = my_place;
  geo.peer_place = peer_place;
  if (t_end <= t_begin) return cudaSuccess;
  unsigned long long tb = t_begin, te = t_end;
  const int grid = grid_for((te - tb + 3) / 4, 256, sm_count, 8);
  void *args[] = {(void *)&mine, (void *)&peer, (void *)&tb, (void *)&te, (void *)&geo};
  return cudaLaunchKernel((const void *)&k_peer_swap, dim3(grid), dim3(256), args, 0, stream);
}

// ---------------------------------------------------------------- reductions (deterministic)
// Stage 1: fixed grid, grid-stride in a fixed order, warp shuffles, one partial per block.
// Stage 2: one block folds the partials in a fixed tree.  No floating-point atomics, so the
// result is run-to-run identical for a given grid (SURVEY.md 7.2 "determinism").
constexpr int kRedThreads = 256;

template <int NV>
__device__ __forceinline__ void block_reduce_store(double (&v)[NV], double *__restrict__ out) {
  __shared__ double sh[NV][kRedThreads / 32];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) sh[k][w] = v[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      double s = 0.0;
      for (int i = 0; i < kRedThreads / 32; ++i) s += sh[k][i];
      out[k] = s;
    }
  }
}

// partials[block][2] = (S0, S1) by the value of physical bit `bit` (bit < 0: everything in S0)
__global__ void __launch_bounds__(kRedThreads) k_sumsq_partial(const double2 *__restrict__ amps, uint64_t n, int bit,
                                                              double *__restrict__ partials) {
  double acc[2] = {0.0, 0.0};
  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    const double2 z = __ldcs(amps + i);
    const double w = z.x * z.x + z.y * z.y;
    if (bit >= 0 && ((i >> bit) & 1ull)) acc[1] += w; else acc[0] += w;
  }
  block_reduce_store<2>(acc, partials + 2 * blockIdx.x);
}

// a <.> b with the first argument conjugated (StateVec.hs:57-58).  The imaginary part is
// formed from separately rounded products so that <a,b> == conj <b,a> holds EXACTLY
// (test/Qubism/AlgebraTests.hs:43-47): no FMA contraction across the antisymmetric pair.
__global__ void __launch_bounds__(kRedThreads) k_dotc_partial(const double2 *__restrict__ a, const double2 *__restrict__ b,
                                                             uint64_t n, double *__restrict__ partials) {
  double acc[2] = {0.0, 0.0};
  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    const double2 x = __ldcs(a + i), y = __ldcs(b + i);
    acc[0] = __dadd_rn(acc[0], __dadd_rn(__dmul_rn(x.x, y.x), __dmul_rn(x.y, y.y)));
    acc[1] = __dadd_rn(acc[1], __dsub_rn(__dmul_rn(x.x, y.y), __dmul_rn(x.y, y.x)));
  }
  block_reduce_store<2>(acc, partials + 2 * blockIdx.x);
}

__global__ void __launch_bounds__(kRedThreads) k_reduce_final(const double *__restrict__ partials, int nblocks,
                                                             double *__restrict__ out) {
  double acc[2] = {0.0, 0.0};
  for (int i = threadIdx.x; i < nblocks; i += kRedThreads) {
    acc[0] += partials[2 * i];
    acc[1] += partials[2 * i + 1];
  }
  block_reduce_store<2>(acc, out);
}

int reduce_grid(uint64_t n, int sm_count) { return grid_for(n, kRedThreads * 4, sm_count, 8); }

cudaError_t launch_sumsq(const double2 *amps, uint64_t n, int bit, double *partials_dev, double *out_dev, int sm_count,
                         cudaStream_t stream) {
  const int g = reduce_grid(n, sm_count);
  k_sumsq_partial<<<g, kRedThreads, 0, stream>>>(amps, n, bit, partials_dev);
  k_reduce_final<<<1, kRedThreads, 0, stream>>>(partials_dev, g, out_dev);
  return cudaGetLastError();
}

cudaError_t launch_dotc(const double2 *a, const double2 *b, uint64_t n, double *partials_dev, double *out_dev,
                        int sm_count, cudaStream_t stream) {
  const int g = reduce_grid(n, sm_count);
  k_dotc_partial<<<g, kRedThreads, 0, stream>>>(a, b, n, partials_dev);
  k_reduce_final<<<1, kRedThreads, 0, stream>>>(partials_dev, g, out_dev);
  return cudaGetLastError();
}

// ---------------------------------------------------------------- Pauli expectation values
// One launch = one group of terms sharing the physical X mask xp.  With h = the top bit of xp, every
// index i with bit h clear meets its partner j = i ^ xp once; the pair product w = conj(psi_j) psi_i is
// formed once and each term adds (-1)^popc(i & zp) times Re w (even popc(x & z)) or Im w (odd); the host
// applies the factor 2, the phase sign and the global-qubit signs.  xp == 0: every i, w = |psi_i|^2.
// A thread takes kExpU pairs per step, pair numbers p0 + u * kRedThreads: the bits of u are a field of
// their own in p, so popc(i_u & zp) = popc(i_0 & zp) + popc(ins(u << 8) & zp), and the second part is
// the host-made bit u of ExpTerms::rflip.  Per term and step one POPC; per term and pair a few integer
// instructions (the sign goes straight into the high word) and one DADD.
static_assert(kRedThreads == 1 << kExpUShift, "ExpTerms::rflip: u is the pair-number field above the thread index");

__global__ void __launch_bounds__(kRedThreads) k_expect_final(const double *__restrict__ partials, int nblocks, int stride,
                                                             double *__restrict__ out) {
  double acc[1] = {0.0};
  for (int i = threadIdx.x; i < nblocks; i += kRedThreads) acc[0] += partials[size_t(i) * stride + blockIdx.x];
  block_reduce_store<1>(acc, out + blockIdx.x);
}

template <int NT>
__global__ void __launch_bounds__(kRedThreads, NT >= 16 ? 1 : 4) k_expect_pauli_partial(const double2 *__restrict__ amps, uint64_t npairs,
                                                                     const __grid_constant__ ExpTerms terms,
                                                                     double *__restrict__ partials) {
  double acc[NT];
#pragma unroll
  for (int t = 0; t < NT; ++t) acc[t] = 0.0;
  const uint64_t lo = terms.lo_mask, xp = terms.xp;
  const uint64_t stride = uint64_t(gridDim.x) * (kRedThreads * kExpU);
  for (uint64_t p0 = blockIdx.x * uint64_t(kRedThreads * kExpU) + threadIdx.x; p0 < npairs; p0 += stride) {
    double re[kExpU], im[kExpU];
    const uint64_t i0 = (p0 & lo) | ((p0 & ~lo) << 1);
#pragma unroll
    for (int u = 0; u < kExpU; ++u) {
      const uint64_t p = p0 + uint64_t(u) * kRedThreads;
      re[u] = im[u] = 0.0;
      if (p < npairs) {
        const uint64_t i = (p & lo) | ((p & ~lo) << 1);  // bit h inserted (lo_mask = ~0: none)
        const double2 a = __ldcs(amps + i);
        if (xp) {
          const double2 b = __ldcs(amps + (i ^ xp));
          re[u] = __dadd_rn(__dmul_rn(b.x, a.x), __dmul_rn(b.y, a.y));
          im[u] = __dsub_rn(__dmul_rn(b.x, a.y), __dmul_rn(b.y, a.x));
        } else {
          re[u] = __dadd_rn(__dmul_rn(a.x, a.x), __dmul_rn(a.y, a.y));
        }
      }
    }
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const uint32_t base = (0u - (uint32_t(__popcll(i0 & terms.zp[t])) & 1u)) ^ terms.rflip[t];
#pragma unroll
      for (int u = 0; u < kExpU; ++u) {
        const double v = t < terms.neven ? re[u] : im[u];
        const int hi = __double2hiint(v) ^ int((base << (31 - u)) & 0x80000000u);
        acc[t] = __dadd_rn(acc[t], __hiloint2double(hi, __double2loint(v)));
      }
    }
  }
  block_reduce_store<NT>(acc, partials + size_t(NT) * blockIdx.x);
}

template <int NT>
static cudaError_t expect_launch(const double2 *amps, uint64_t npairs, const ExpTerms &terms, double *partials_dev,
                                 double *out_dev, int sm_count, cudaStream_t stream) {
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_expect_pauli_partial<NT>, kRedThreads, 0);
  if (e != cudaSuccess) return e;
  const int g = grid_for(npairs, kRedThreads * kExpU, sm_count, std::max(1, std::min(per_sm, 8)));
  k_expect_pauli_partial<NT><<<g, kRedThreads, 0, stream>>>(amps, npairs, terms, partials_dev);
  // partials[block][NT]: one block of the final stage per term
  k_expect_final<<<terms.nterms, kRedThreads, 0, stream>>>(partials_dev, g, NT, out_dev);
  return cudaGetLastError();
}

cudaError_t launch_expect_pauli(const double2 *amps, int local_bits, const ExpTerms &terms, double *partials_dev,
                                double *out_dev, int sm_count, cudaStream_t stream) {
  if (terms.nterms < 1 || terms.nterms > kExpMaxTerms || terms.neven > terms.nterms) return cudaErrorInvalidValue;
  const uint64_t npairs = terms.xp ? (1ull << (local_bits - 1)) : (1ull << local_bits);
  if (terms.nterms <= 1) return expect_launch<1>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
  if (terms.nterms <= 2) return expect_launch<2>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
  if (terms.nterms <= 4) return expect_launch<4>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
  if (terms.nterms <= 8) return expect_launch<8>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
  if (terms.nterms <= 16) return expect_launch<16>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
  if (terms.nterms <= 32) return expect_launch<32>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
  return expect_launch<64>(amps, npairs, terms, partials_dev, out_dev, sm_count, stream);
}

// ---------------------------------------------------------------- Pauli rotations
// exp(-i theta/2 P) = c I - i s P pairs every amplitude j with exactly one partner j ^ x, so a rotation of
// any weight is one 2x2 update per pair; a CTA that holds every X bit of a run of rotations in its tile
// applies the whole run between one load and one store of that tile.  The tile goes straight from global
// to XOR-swizzled shared memory (cp.async: no register staging), thread t owning tile-local indices
// t + k * kPauliThreads (8 consecutive lanes = one 128-byte line while the low physical bits are tile
// bits).  Consecutive Z-only rotations are one step: a phase per amplitude over the thread's own indices,
// applied in one read and write of each.  A rotation with X is one step of one pair per thread and
// iteration (swz keeps the partners conflict-free, being linear over XOR).  A CTA barrier separates two
// steps unless both are Z-only steps; the store reads the thread's own indices again.
__device__ __forceinline__ void pauli_phases(double2 &v, const PauliRotParam &p, uint32_t u, uint32_t sgn0) {
  const bool neg = (__popc(u & p.zt) ^ sgn0) & 1u;
  const double fr = neg ? p.c - p.ar : p.c + p.ar, fi = neg ? -p.ai : p.ai;
  v = make_double2(fr * v.x - fi * v.y, fr * v.y + fi * v.x);
}

template <int TB>
__global__ void __launch_bounds__(kPauliThreads, 3) k_pauli_rot_tile(double2 *__restrict__ amps, const __grid_constant__ PauliRotArgs a) {
  constexpr int kThrBits = 8;
  static_assert(kPauliThreads == 1 << kThrBits && TB > kThrBits, "tile-local index = thread + k * kPauliThreads");
  constexpr int EPT = 1 << (TB - kThrBits);  // amplitudes per thread
  extern __shared__ double2 tile[];
  const uint32_t tid = threadIdx.x, tb = a.tile_bits, nel = 1u << tb, nrot = a.nrot;
  uint64_t base = 0;  // the block number deposited into the local bits outside the tile
  {
    uint64_t t = blockIdx.x;
    for (uint32_t i = 0; i < a.nruns; ++i) {
      base |= (t & ((1ull << a.run_len[i]) - 1ull)) << a.run_shift[i];
      t >>= a.run_len[i];
    }
  }
  uint64_t off_lo = base, off_hi[TB - kThrBits];
#pragma unroll
  for (int b = 0; b < kThrBits; ++b)
    if (b < (int)tb && ((tid >> b) & 1u)) off_lo |= 1ull << a.tile_pos[b];
#pragma unroll
  for (int b = 0; b < TB - kThrBits; ++b) off_hi[b] = b + kThrBits < (int)tb ? 1ull << a.tile_pos[b + kThrBits] : 0ull;
  auto goff = [&](int k) {
    uint64_t o = off_lo;
#pragma unroll
    for (int b = 0; b < TB - kThrBits; ++b)
      if ((k >> b) & 1) o |= off_hi[b];
    return o;
  };
  auto sign0 = [&](const PauliRotParam &p) { return uint32_t(__popcll(base & p.zout)) & 1u; };
#pragma unroll
  for (int k = 0; k < EPT; ++k)
    if (tid + k * kPauliThreads < nel) {
      const uint32_t sa = uint32_t(__cvta_generic_to_shared(tile + swz(tid + k * kPauliThreads)));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(amps + goff(k)) : "memory");
    }
  asm volatile("cp.async.wait_all;" ::: "memory");  // (own indices: visible to this thread, no barrier)
  bool own = true;  // the last step wrote the thread's own indices only
  for (uint32_t r = 0; r < nrot;) {
    const PauliRotParam &p = a.rot[r];
    if (p.xt == 0) {  // Z-only rotations r .. e
      uint32_t e = r + 1;
      while (e < nrot && a.rot[e].xt == 0) ++e;
      if (!own) __syncthreads();
#pragma unroll 4
      for (int k = 0; k < EPT; ++k) {
        const uint32_t u = tid + k * kPauliThreads;
        if (u >= nel) continue;
        double2 v = tile[swz(u)];
        for (uint32_t z = r; z < e; ++z) pauli_phases(v, a.rot[z], u, sign0(a.rot[z]));
        tile[swz(u)] = v;
      }
      own = true;
      r = e;
      continue;
    }
    __syncthreads();
    const uint32_t h = 31 - __clz(p.xt), lo = (1u << h) - 1u, s0 = sign0(p);  // pairs (j, j ^ xt), bit h of j clear
#pragma unroll 4
    for (int k = 0; k < EPT / 2; ++k) {
      const uint32_t q = tid + k * kPauliThreads;
      if (q >= nel / 2) continue;
      const uint32_t j = ((q & ~lo) << 1) | (q & lo), jx = j ^ p.xt;
      const double2 A = tile[swz(j)], B = tile[swz(jx)];
      const bool nj = (__popc(j & p.zt) ^ s0) & 1u, nk = (__popc(jx & p.zt) ^ s0) & 1u;
      const double br = nk ? -B.x : B.x, bi = nk ? -B.y : B.y, ar = nj ? -A.x : A.x, ai = nj ? -A.y : A.y;
      tile[swz(j)] = make_double2(p.c * A.x + p.ar * br - p.ai * bi, p.c * A.y + p.ar * bi + p.ai * br);
      tile[swz(jx)] = make_double2(p.c * B.x + p.ar * ar - p.ai * ai, p.c * B.y + p.ar * ai + p.ai * ar);
    }
    own = false;
    ++r;
  }
  if (!own) __syncthreads();
#pragma unroll
  for (int k = 0; k < EPT; ++k)
    if (tid + k * kPauliThreads < nel) __stcs(amps + goff(k), tile[swz(tid + k * kPauliThreads)]);
}

cudaError_t launch_pauli_rot(double2 *amps, int local_bits, const PauliRotArgs &args, cudaStream_t stream) {
  if (args.nrot < 1 || args.nrot > (uint32_t)kPauliMaxRot || args.tile_bits > (uint32_t)kPauliTileBits ||
      (int)args.tile_bits > local_bits)
    return cudaErrorInvalidValue;
  const size_t smem = sizeof(double2) << args.tile_bits;
  const auto fn = k_pauli_rot_tile<kPauliTileBits>;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(double2) << kPauliTileBits));
  if (e != cudaSuccess) return e;
  fn<<<unsigned(1ull << (local_bits - args.tile_bits)), kPauliThreads, smem, stream>>>(amps, args);
  return cudaGetLastError();
}

// ---------------------------------------------------------------- live sub-cube kernels
// After a collapse (StateVec.hs:104-114) half of the state is exactly zero, and a fresh
// |0...0> is zero outside one amplitude.  The host tracks the index bits whose value is KNOWN
// for every non-zero amplitude (qb_api.cpp, "support"); measurement then only ever touches the
// live sub-cube {i : i & fixed_mask == fixed_val}: the reduction of `measure` on qubit k reads
// 2^(n-k) amplitudes instead of 2^n, and a collapse is a zero-fill of the half that dies (no
// read, no full pass) plus a deferred scalar.  `measure` on all n qubits is ~3 sweep-equivalents
// instead of 2n.
struct CubeGeom {
  uint32_t nruns;
  uint32_t run_shift[kMaxRuns];  // deposit of the free index into the unknown local bits
  uint32_t run_len[kMaxRuns];
  uint64_t fixed;                // the known local bits, at their known value
};

__device__ __forceinline__ uint64_t cube_index(const CubeGeom &geo, uint64_t j) {
  if (geo.nruns == 1 && geo.run_shift[0] == 0) return j | geo.fixed;  // contiguous block (top bits known)
  uint64_t idx = geo.fixed, rest = j;
  for (uint32_t k = 0; k < geo.nruns; ++k) {
    idx |= (rest & ((1ull << geo.run_len[k]) - 1ull)) << geo.run_shift[k];
    rest >>= geo.run_len[k];
  }
  return idx;
}

__global__ void __launch_bounds__(kRedThreads) k_sumsq_cube(const double2 *__restrict__ amps, uint64_t n, int bit,
                                                           double *__restrict__ partials, const __grid_constant__ CubeGeom geo) {
  double acc[2] = {0.0, 0.0};
  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  for (uint64_t j = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; j < n; j += stride) {
    const uint64_t i = cube_index(geo, j);
    const double2 z = __ldcs(amps + i);
    const double w = z.x * z.x + z.y * z.y;
    if (bit >= 0 && ((i >> bit) & 1ull)) acc[1] += w; else acc[0] += w;
  }
  block_reduce_store<2>(acc, partials + 2 * blockIdx.x);
}

// mode 0: amps[i] = 0;  mode 1: amps[i] *= (zr, zi)
__global__ void __launch_bounds__(256) k_cube_update(double2 *__restrict__ amps, uint64_t n, int mode, double zr, double zi,
                                                    const __grid_constant__ CubeGeom geo) {
  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  for (uint64_t j = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; j < n; j += stride) {
    const uint64_t i = cube_index(geo, j);
    if (mode == 0) {
      amps[i] = make_double2(0.0, 0.0);
    } else {
      const double2 x = amps[i];
      amps[i] = make_double2(zr * x.x - zi * x.y, zr * x.y + zi * x.x);
    }
  }
}

static uint64_t make_cube(int local_bits, uint64_t fixed_mask, uint64_t fixed_val, CubeGeom &geo) {
  geo = CubeGeom{};
  geo.fixed = fixed_val & fixed_mask & ((1ull << local_bits) - 1ull);
  int nfree = 0, b = 0;
  while (b < local_bits) {
    if (fixed_mask & (1ull << b)) {
      ++b;
      continue;
    }
    int e = b;
    while (e < local_bits && !(fixed_mask & (1ull << e))) ++e;
    if (geo.nruns >= (uint32_t)kMaxRuns) return 0;  // cannot happen: at most local_bits / 2 + 1 runs <= 16 for <= 31 bits ... guarded by the caller
    geo.run_shift[geo.nruns] = b;
    geo.run_len[geo.nruns] = e - b;
    ++geo.nruns;
    nfree += e - b;
    b = e;
  }
  if (geo.nruns == 0) {  // a single element
    geo.nruns = 1;
    geo.run_shift[0] = 0;
    geo.run_len[0] = 0;
  }
  return 1ull << nfree;
}

int cube_runs(int local_bits, uint64_t fixed_mask) {
  int runs = 0, b = 0;
  while (b < local_bits) {
    if (fixed_mask & (1ull << b)) {
      ++b;
      continue;
    }
    while (b < local_bits && !(fixed_mask & (1ull << b))) ++b;
    ++runs;
  }
  return runs;
}

cudaError_t launch_sumsq_cube(const double2 *amps, int local_bits, uint64_t fixed_mask, uint64_t fixed_val, int bit,
                              double *partials_dev, double *out_dev, int sm_count, cudaStream_t stream) {
  CubeGeom geo;
  const uint64_t n = make_cube(local_bits, fixed_mask, fixed_val, geo);
  if (n == 0) return cudaErrorInvalidValue;
  const int g = reduce_grid(n, sm_count);
  k_sumsq_cube<<<g, kRedThreads, 0, stream>>>(amps, n, bit, partials_dev, geo);
  k_reduce_final<<<1, kRedThreads, 0, stream>>>(partials_dev, g, out_dev);
  return cudaGetLastError();
}

cudaError_t launch_cube_update(double2 *amps, int local_bits, uint64_t fixed_mask, uint64_t fixed_val, int mode,
                               const double z[2], int sm_count, cudaStream_t stream) {
  CubeGeom geo;
  const uint64_t n = make_cube(local_bits, fixed_mask, fixed_val, geo);
  if (n == 0) return cudaErrorInvalidValue;
  k_cube_update<<<grid_for(n, 256 * 4, sm_count, 8), 256, 0, stream>>>(amps, n, mode, z ? z[0] : 0.0, z ? z[1] : 0.0, geo);
  return cudaGetLastError();
}

// ---------------------------------------------------------------- element-wise kernels
__global__ void __launch_bounds__(256) k_axpy(double2 *__restrict__ y, const double2 *__restrict__ x, uint64_t n,
                                              double zr, double zi) {
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const double2 a = x[i];
    double2 b = y[i];
    b.x += zr * a.x - zi * a.y;
    b.y += zr * a.y + zi * a.x;
    y[i] = b;
  }
}

// out[i * nb + j] = a[i] * b[j]  (StateVec.hs:98-100, flatten (outer a b), no conjugation)
__global__ void __launch_bounds__(256) k_tensor(double2 *__restrict__ out, const double2 *__restrict__ a,
                                                const double2 *__restrict__ b, uint64_t n, int bbits) {
  const uint64_t bmask = (1ull << bbits) - 1;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const double2 x = a[i >> bbits], y = b[i & bmask];
    out[i] = make_double2(x.x * y.x - x.y * y.y, x.x * y.y + x.y * y.x);
  }
}

__global__ void k_set_amp(double2 *amps, uint64_t idx, double re, double im) { amps[idx] = make_double2(re, im); }

// exchange two index bits in place (a change of qubit LAYOUT, no gate): every element whose bits
// (hi, lo) read (1, 0) trades places with its partner (0, 1).  Half of the shard moves.
__global__ void __launch_bounds__(256) k_swap_bits(double2 *__restrict__ amps, uint64_t nquads, int lo, int hi) {
  for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < nquads; p += uint64_t(gridDim.x) * blockDim.x) {
    uint64_t i = ((p >> lo) << (lo + 1)) | (p & ((1ull << lo) - 1));   // insert a 0 at `lo`
    i = ((i >> hi) << (hi + 1)) | (i & ((1ull << hi) - 1));            // ... and at `hi` (hi > lo)
    const uint64_t ia = i | (1ull << hi), ib = i | (1ull << lo);
    const double2 a = amps[ia], b = amps[ib];
    amps[ia] = b;
    amps[ib] = a;
  }
}

// out[i * 2^nb + j] = a[i] * b[j] on a sharded context, both operands in the identity layout: this
// rank's shard of `out` is (this rank's shard of a) x (ALL of b); b[j] lives on rank j >> Lb and is
// read through that rank's mapped shard (StateVec.hs:98-100; ProgState.hs:137-166 fuses registers
// this way)
__global__ void __launch_bounds__(256) k_tensor_sharded(double2 *__restrict__ out, const double2 *__restrict__ a,
                                                        double2 *const *__restrict__ b_shards, uint64_t n, int nb, int Lb) {
  const uint64_t bmask = (1ull << nb) - 1, lmask = (1ull << Lb) - 1;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const uint64_t j = i & bmask;
    const double2 x = a[i >> nb], y = b_shards[j >> Lb][j & lmask];
    out[i] = make_double2(x.x * y.x - x.y * y.y, x.x * y.y + x.y * y.x);
  }
}

// ---- qubit layouts other than the identity (global<->local swaps, out-of-place passes) -------------
// Bit b of an index goes to bit pos[b]: applied to logical indices this is "where does amplitude x
// live", applied to old physical indices it is a change of layout.
struct BitMap {
  uint8_t pos[64];
  int nbits;
};
__device__ __forceinline__ uint64_t map_bits(const BitMap &m, uint64_t x) {
  uint64_t o = 0;
  for (int b = 0; b < m.nbits; ++b) o |= ((x >> b) & 1ull) << m.pos[b];
  return o;
}
// out[i] = amps[where(first + i)]: amplitudes [first, first + count) in INDEX order (Show, :dump, parity)
__global__ void __launch_bounds__(256) k_gather_logical(double2 *__restrict__ out, const double2 *__restrict__ amps,
                                                        uint64_t first, uint64_t count, const __grid_constant__ BitMap m) {
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < count; i += uint64_t(gridDim.x) * blockDim.x)
    out[i] = amps[map_bits(m, first + i)];
}
// dst[move(i)] = src[i] for every local index i: a whole change of layout in one sweep
__global__ void __launch_bounds__(256) k_permute_bits(double2 *__restrict__ dst, const double2 *__restrict__ src, uint64_t n,
                                                      const __grid_constant__ BitMap m) {
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x)
    dst[map_bits(m, i)] = src[i];
}

cudaError_t launch_gather_logical(double2 *out, const double2 *amps, uint64_t first, uint64_t count, const int *pos, int nbits,
                                  int sm_count, cudaStream_t stream) {
  if (nbits > 64) return cudaErrorInvalidValue;
  if (count == 0) return cudaSuccess;
  BitMap m{};
  m.nbits = nbits;
  for (int b = 0; b < nbits; ++b) m.pos[b] = (uint8_t)pos[b];
  k_gather_logical<<<grid_for(count, 256, sm_count, 8), 256, 0, stream>>>(out, amps, first, count, m);
  return cudaGetLastError();
}

cudaError_t launch_permute_bits(double2 *dst, const double2 *src, int local_bits, const int *newpos, int sm_count,
                                cudaStream_t stream) {
  if (local_bits > 64) return cudaErrorInvalidValue;
  BitMap m{};
  m.nbits = local_bits;
  for (int b = 0; b < local_bits; ++b) m.pos[b] = (uint8_t)newpos[b];
  const uint64_t n = 1ull << local_bits;
  k_permute_bits<<<grid_for(n, 256, sm_count, 8), 256, 0, stream>>>(dst, src, n, m);
  return cudaGetLastError();
}

cudaError_t launch_axpy(double2 *y, const double2 *x, uint64_t n, const double z[2], int sm_count,
                        cudaStream_t stream) {
  k_axpy<<<grid_for(n, 256, sm_count, 8), 256, 0, stream>>>(y, x, n, z[0], z[1]);
  return cudaGetLastError();
}

cudaError_t launch_tensor(double2 *out, const double2 *a, const double2 *b, int abits, int bbits, int sm_count,
                          cudaStream_t stream) {
  const uint64_t n = 1ull << (abits + bbits);
  k_tensor<<<grid_for(n, 256, sm_count, 8), 256, 0, stream>>>(out, a, b, n, bbits);
  return cudaGetLastError();
}

cudaError_t launch_swap_bits(double2 *amps, int local_bits, int b1, int b2, int sm_count, cudaStream_t stream) {
  if (b1 == b2) return cudaSuccess;
  if (local_bits < 2) return cudaErrorInvalidValue;
  const uint64_t nquads = 1ull << (local_bits - 2);
  k_swap_bits<<<grid_for(nquads, 256, sm_count, 8), 256, 0, stream>>>(amps, nquads, std::min(b1, b2), std::max(b1, b2));
  return cudaGetLastError();
}

cudaError_t launch_tensor_sharded(double2 *out, const double2 *a, double2 *const *b_shards_dev, int a_local_bits, int bbits,
                                  int b_local_bits, int sm_count, cudaStream_t stream) {
  const uint64_t n = 1ull << (a_local_bits + bbits);
  k_tensor_sharded<<<grid_for(n, 256, sm_count, 8), 256, 0, stream>>>(out, a, b_shards_dev, n, bbits, b_local_bits);
  return cudaGetLastError();
}

cudaError_t launch_set_amp(double2 *amps, uint64_t idx, double re, double im, cudaStream_t stream) {
  k_set_amp<<<1, 1, 0, stream>>>(amps, idx, re, im);
  return cudaGetLastError();
}

}  // namespace qb
