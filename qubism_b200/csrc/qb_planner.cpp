// Host-side pass planner: turns a list of queued gates into fused-pass programs.
//
// The reference evaluator issues one `#>` per primitive op (QASM/Simulation.hs:94-122), each
// a full sweep of the state.  Behind the C ABI the ops are queued and this planner groups
// them so that one sweep of HBM carries as many of them as dependencies and the tile
// geometry allow (SURVEY.md 7.1 step 5).  Pure host logic: unit-tested on the CPU through
// qb_plan_describe and the numpy plan emulator in tests/.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <sstream>

#include "qb_internal.h"

namespace qb {

static inline int popc(uint64_t x) { return __builtin_popcountll(x); }

// --------------------------------------------------------------------- options
bool variant_supported(int T, int R) {
  for (const auto &v : kFusedVariants)
    if (v.T == T && v.R == R) return true;
  return false;
}

bool set_opt(PlanOptions &o, const std::string &name, int64_t v) {
  if (name == "tile_bits") {
    if (v < 10 || v > kMaxTileBits) return false;
    o.tile_bits = (int)v;
  } else if (name == "reg_bits") {
    if (v < 3 || v > kMaxRegBits) return false;
    o.reg_bits = (int)v;
  } else if (name == "low_bits") {
    if (v < kLaneFixedBits || v > 10) return false;
    o.low_bits = (int)v;
  } else if (name == "max_rounds") {
    if (v < 3 || v > kMaxRounds) return false;
    o.max_rounds = (int)v;
  } else if (name == "peephole") {
    o.peephole = v ? 1 : 0;
  } else if (name == "fuse") {
    o.fuse = v ? 1 : 0;
  } else if (name == "max_pass_gates") {
    if (v < 1 || v > kMaxPassGates) return false;
    o.max_pass_gates = (int)v;
  } else if (name == "time_kernels") {
    o.time_kernels = v ? 1 : 0;
  } else if (name == "l2_prefetch") {
    if (v < 0 || v > 4) return false;
    o.l2_prefetch = (int)v;
  } else if (name == "hot_bits") {
    if (v < 0 || v > kMaxTileBits) return false;
    o.hot_bits = (int)v;
  } else if (name == "jit_group") {
    if (v != 1 && v != 2 && v != 4 && v != 8) return false;
    o.jit_group = (int)v;
  } else if (name == "jit_minb") {
    if (v < 0 || v > 8) return false;
    o.jit_minb = (int)v;
  } else if (name == "jit_mem") {
    if (v < 0 || v > 7) return false;
    o.jit_mem = (int)v;
  } else if (name == "jit_pf_last") {
    o.jit_pf_last = v ? 1 : 0;
  } else if (name == "tma") {
    if (v < 0 || v > 3) return false;
    o.tma = (int)v;
  } else if (name == "defer_tail") {
    if (v < 0 || v > kMaxPassGates) return false;
    o.defer_tail = (int)v;
  } else if (name == "fuse_exchange") {
    o.fuse_exchange = v ? 1 : 0;
  } else if (name == "pf_lines") {
    if (v < 0 || v > 4) return false;
    o.pf_lines = (int)v;
  } else if (name == "oop_dist") {
    o.oop_dist = v ? 1 : 0;
  } else if (name == "chunk_lanes") {
    o.chunk_lanes = v ? 1 : 0;
  } else if (name == "oop_low_bits") {
    if (v < kLaneFixedBits || v > 10) return false;
    o.oop_low_bits = (int)v;
  } else if (name == "oop") {
    if (v < 0 || v > 2) return false;  // 1: every qubit re-sorted by next use, 2: only the tile's
    o.oop = (int)v;
  } else if (name == "jit") {
    if (v < 0 || v > 1000000) return false;
    o.jit = (int)v;
  } else if (name == "rot") {
    o.rot = v ? 1 : 0;
  } else if (name == "lite") {
    o.lite = v ? 1 : 0;
  } else if (name == "support") {
    o.support = v ? 1 : 0;
  } else if (name == "skip_dead") {
    o.skip_dead = v ? 1 : 0;
  } else if (name == "known_mask") {
    o.known_mask = (uint64_t)v;
  } else if (name == "known_val") {
    o.known_val = (uint64_t)v;
  } else if (name == "lane_fixed") {
    if (v < 0 || v > kLaneFixedBits) return false;
    o.lane_fixed = (int)v;

  } else if (name == "avoid_regswap") {
    if (v < 0 || v > 2) return false;
    o.avoid_regswap = (int)v;
  } else if (name == "dbg_skip") {
    if (v < 0 || v > 31) return false;  // (bit 4: the switches also apply to the specialised kernels)
    o.dbg_skip = (int)v;
  } else {
    return false;
  }
  return true;
}

int64_t get_opt(const PlanOptions &o, const std::string &name) {
  if (name == "tile_bits") return o.tile_bits;
  if (name == "reg_bits") return o.reg_bits;
  if (name == "low_bits") return o.low_bits;
  if (name == "max_rounds") return o.max_rounds;
  if (name == "peephole") return o.peephole;
  if (name == "fuse") return o.fuse;
  if (name == "max_pass_gates") return o.max_pass_gates;
  if (name == "time_kernels") return o.time_kernels;
  if (name == "l2_prefetch") return o.l2_prefetch;
  if (name == "dbg_skip") return o.dbg_skip;
  if (name == "avoid_regswap") return o.avoid_regswap;
  if (name == "hot_bits") return o.hot_bits;
  if (name == "rot") return o.rot;
  if (name == "jit") return o.jit;
  if (name == "jit_pf_last") return o.jit_pf_last;
  if (name == "tma") return o.tma;
  if (name == "oop") return o.oop;
  if (name == "oop_low_bits") return o.oop_low_bits;
  if (name == "chunk_lanes") return o.chunk_lanes;
  if (name == "oop_dist") return o.oop_dist;
  if (name == "pf_lines") return o.pf_lines;
  if (name == "fuse_exchange") return o.fuse_exchange;
  if (name == "defer_tail") return o.defer_tail;
  if (name == "jit_minb") return o.jit_minb;
  if (name == "jit_mem") return o.jit_mem;
  if (name == "jit_group") return o.jit_group;
  if (name == "lite") return o.lite;
  if (name == "lane_fixed") return o.lane_fixed;
  if (name == "skip_dead") return o.skip_dead;
  if (name == "support") return o.support;
  return -1;
}

// effective (T, R) for a shard with L local bits; T = 0 -> unfused kernels only
void effective_tile(const PlanOptions &o, int L, int &T, int &R) {
  T = std::min(o.tile_bits, L);
  R = o.reg_bits;
  if (T < 10) {
    T = 0;
    return;
  }
  if (variant_supported(T, R)) return;
  for (int r : {4, 3, 5})
    if (variant_supported(T, r)) {
      R = r;
      return;
    }
  T = 0;
}

// --------------------------------------------------------------------- classification
// r = k * [[c,-s],[s,c]] with c >= 0?  (k may be negative.)  Rotations run as three in-place
// shears in the kernel: 3 instead of 4 FP64 operations per component pair, and no temporaries.
// Only exact rotation structure qualifies (entries equal to a few ulp); allow_scale = false
// additionally demands k = 1 (controlled gates cannot shed a scalar).
static bool as_rotation(const double r[4], bool allow_scale, double &k, double &cs, double &sn) {
  double scale = 0.0;
  for (int i = 0; i < 4; ++i) scale = std::max(scale, std::fabs(r[i]));
  if (!(scale > 0.0) || !std::isfinite(scale)) return false;
  const double tol = 8.0 * DBL_EPSILON * scale;
  if (!(std::fabs(r[0] - r[3]) <= tol && std::fabs(r[1] + r[2]) <= tol)) return false;
  const double a = 0.5 * (r[0] + r[3]), c = 0.5 * (r[2] - r[1]);
  double kk = std::hypot(a, c);
  if (!(kk > 0.0) || !std::isfinite(kk)) return false;
  if (!allow_scale) {
    if (a < 0.0 || std::fabs(kk - 1.0) > 8.0 * DBL_EPSILON) return false;
    k = 1.0;
    cs = a;
    sn = c;
    return true;
  }
  if (kk < 0x1p-20 || kk > 0x1p20) return false;  // keep the deferred scalar well inside the exponent range
  if (a < 0.0) kk = -kk;
  k = kk;
  cs = a / kk;
  sn = c / kk;
  return true;
}

static void set_rotation(Classified &c, double k, double cs, double sn) {
  c.type = G_ROT;
  std::memset(c.m, 0, sizeof(c.m));
  c.m[0] = cs;
  c.m[2] = -sn;
  c.m[4] = sn;
  c.m[6] = cs;
  c.phase[0] *= k;
  c.phase[1] *= k;
}

// general complex 2x2 with a well-sized m00: divide by it (6 instead of 8 FP64 operations per
// amplitude where no flip can be pending), the factor goes to the deferred scalar
static Classified as_general1(Classified c, double bigabs) {
  const double ar = c.m[0], ai = c.m[1], a2 = ar * ar + ai * ai;
  if (!(a2 >= 0.25 * bigabs * bigabs) || !std::isfinite(a2)) return c;
  const double mag = std::sqrt(a2);
  if (mag < 0x1p-20 || mag > 0x1p20) return c;
  for (int i = 1; i < 4; ++i) {  // x / a = x * conj(a) / |a|^2
    const double xr = c.m[2 * i], xi = c.m[2 * i + 1];
    c.m[2 * i] = (xr * ar + xi * ai) / a2;
    c.m[2 * i + 1] = (xi * ar - xr * ai) / a2;
  }
  c.m[0] = 1.0;
  c.m[1] = 0.0;
  c.phase[0] = ar;
  c.phase[1] = ai;
  c.type = G_GENERAL1;
  return c;
}

Classified classify_2x2(const double m[8], bool allow_phase_pull, bool allow_scale) {
  Classified c{};
  std::memcpy(c.m, m, sizeof(c.m));
  c.phase[0] = 1.0;
  c.phase[1] = 0.0;
  c.is_scalar = false;
  c.type = G_GENERAL;
  const bool b0 = (m[2] == 0.0 && m[3] == 0.0), c0 = (m[4] == 0.0 && m[5] == 0.0);
  const bool a0 = (m[0] == 0.0 && m[1] == 0.0), d0 = (m[6] == 0.0 && m[7] == 0.0);
  if (b0 && c0) {
    c.type = G_DIAG;
    c.is_scalar = (m[0] == m[6] && m[1] == m[7]);
    return c;
  }
  if (a0 && d0 && m[2] == 1.0 && m[3] == 0.0 && m[4] == 1.0 && m[5] == 0.0) {
    c.type = G_SWAP;
    return c;
  }
  bool all_real = (m[1] == 0.0 && m[3] == 0.0 && m[5] == 0.0 && m[7] == 0.0);
  if (all_real) {
    c.type = G_REAL;
    const double r[4] = {m[0], m[2], m[4], m[6]};
    double k, cs, sn;
    if (as_rotation(r, allow_phase_pull && allow_scale, k, cs, sn)) set_rotation(c, k, cs, sn);
    return c;
  }
  if (!allow_phase_pull) return c;
  // m = s * r with r real?  s = phase of the largest entry; the residual imaginary parts must
  // vanish to a few ulp (they are rounding noise of cis(phi)*cos(theta/2)-style products).
  int big = 0;
  double bigabs = 0.0;
  for (int i = 0; i < 4; ++i) {
    const double a = std::hypot(m[2 * i], m[2 * i + 1]);
    if (a > bigabs) {
      bigabs = a;
      big = i;
    }
  }
  if (!(bigabs > 0.0) || !std::isfinite(bigabs)) return c;
  const double sr = m[2 * big] / bigabs, si = m[2 * big + 1] / bigabs;
  const double tol = 4.0 * DBL_EPSILON * bigabs;
  double r[4];
  for (int i = 0; i < 4; ++i) {
    const double xr = m[2 * i], xi = m[2 * i + 1];
    const double yr = xr * sr + xi * si;   // x * conj(s)
    const double yi = xi * sr - xr * si;
    if (!(std::fabs(yi) <= tol)) return allow_scale ? as_general1(c, bigabs) : c;
    r[i] = yr;
  }
  c.type = G_REAL;
  for (int i = 0; i < 4; ++i) {
    c.m[2 * i] = r[i];
    c.m[2 * i + 1] = 0.0;
  }
  c.phase[0] = sr;
  c.phase[1] = si;
  double k, cs, sn;
  if (as_rotation(r, allow_scale, k, cs, sn)) set_rotation(c, k, cs, sn);
  return c;
}

// --------------------------------------------------------------------- op queue + peephole
void OpQueue::reset(int nqubits, bool peep, bool rot) {
  n = nqubits;
  peephole = peep;
  use_rot = rot;
  clear();
}

void OpQueue::clear() {
  ops.clear();
  last_op.assign(n > 0 ? n : 0, -1);
  gscale[0] = 1.0;
  gscale[1] = 0.0;
}

bool OpQueue::empty() const {
  if (!(gscale[0] == 1.0 && gscale[1] == 0.0)) return false;
  for (const auto &o : ops)
    if (!o.dead) return false;
  return true;
}

void OpQueue::mul_gscale(double re, double im) {
  const double r = gscale[0] * re - gscale[1] * im;
  const double i = gscale[0] * im + gscale[1] * re;
  gscale[0] = r;
  gscale[1] = i;
}

static void link_op(OpQueue &q, HostOp &op, int idx, uint64_t qmask) {
  op.nprev = 0;
  for (uint64_t b = qmask; b; b &= b - 1) {
    const int bit = __builtin_ctzll(b);
    if (op.nprev < 6) {
      op.prev_bit[op.nprev] = bit;
      op.prev_idx[op.nprev] = q.last_op[bit];
      ++op.nprev;
    } else {
      op.nprev = 7;  // too many qubits to unlink later: never cancelled
    }
    q.last_op[bit] = idx;
  }
}

static void unlink_op(OpQueue &q, HostOp &op) {
  op.dead = true;
  for (int i = 0; i < op.nprev && i < 6; ++i) q.last_op[op.prev_bit[i]] = op.prev_idx[i];
}

static void mat2_mul(const double a[8], const double b[8], double out[8]) {  // out = a * b
  auto cm = [](double xr, double xi, double yr, double yi, double &zr, double &zi) {
    zr = xr * yr - xi * yi;
    zi = xr * yi + xi * yr;
  };
  for (int r = 0; r < 2; ++r)
    for (int c = 0; c < 2; ++c) {
      double p0r, p0i, p1r, p1i;
      cm(a[(2 * r) * 2], a[(2 * r) * 2 + 1], b[c * 2], b[c * 2 + 1], p0r, p0i);
      cm(a[(2 * r + 1) * 2], a[(2 * r + 1) * 2 + 1], b[(2 + c) * 2], b[(2 + c) * 2 + 1], p1r, p1i);
      out[(2 * r + c) * 2] = p0r + p1r;
      out[(2 * r + c) * 2 + 1] = p0i + p1i;
    }
}

void OpQueue::push_1q(int target_bit, uint64_t ctrl_mask, const double m[8]) {
  ++submitted;
  // scaled rotations shed their scale into the deferred scalar only while that stays far from
  // the exponent limits (a flush folds it back into the amplitudes)
  const double gmag = std::fabs(gscale[0]) + std::fabs(gscale[1]);
  const bool scale_ok = gmag > 0x1p-400 && gmag < 0x1p400;
  Classified c = classify_2x2(m, peephole && ctrl_mask == 0, scale_ok);
  if (c.type == G_ROT && !use_rot) c.type = G_REAL;
  const uint64_t qmask = ctrl_mask | (1ull << target_bit);
  if (peephole) {
    if (ctrl_mask == 0) {
      if (c.type == G_DIAG && c.is_scalar) {  // scalar * I: a global factor (reference u1 family)
        mul_gscale(m[0], m[1]);
        ++folded;
        return;
      }
      if (!(c.phase[0] == 1.0 && c.phase[1] == 0.0)) mul_gscale(c.phase[0], c.phase[1]);
      const int li = last_op[target_bit];
      if (li >= 0 && !ops[li].dead && ops[li].kind == 0 && ops[li].ctrl == 0 && ops[li].target == target_bit &&
          ops[li].nprev <= 6) {
        double prod[8];
        mat2_mul(c.m, ops[li].m, prod);
        Classified pc = classify_2x2(prod, true, scale_ok);
        if (pc.type == G_ROT && !use_rot) pc.type = G_REAL;
        ++folded;
        if (pc.type == G_DIAG && pc.is_scalar) {
          mul_gscale(prod[0], prod[1]);
          unlink_op(*this, ops[li]);
          ++folded;
        } else {
          if (!(pc.phase[0] == 1.0 && pc.phase[1] == 0.0)) mul_gscale(pc.phase[0], pc.phase[1]);
          std::memcpy(ops[li].m, pc.m, sizeof(pc.m));
          ops[li].type = pc.type;
        }
        return;
      }
    } else if (c.type == G_SWAP) {
      const int li = last_op[target_bit];
      if (li >= 0 && !ops[li].dead && ops[li].kind == 0 && ops[li].type == G_SWAP && ops[li].target == target_bit &&
          ops[li].ctrl == ctrl_mask && ops[li].nprev <= 6) {
        bool adjacent = true;
        for (uint64_t b = ctrl_mask; b; b &= b - 1)
          if (last_op[__builtin_ctzll(b)] != li) adjacent = false;
        if (adjacent) {  // cx . cx = identity
          unlink_op(*this, ops[li]);
          folded += 2;
          return;
        }
      }
    }
  }
  HostOp op;
  op.kind = 0;
  op.type = c.type;
  op.target = target_bit;
  op.ctrl = ctrl_mask;
  std::memcpy(op.m, c.m, sizeof(c.m));
  const int idx = (int)ops.size();
  link_op(*this, op, idx, qmask);
  ops.push_back(std::move(op));
}

void OpQueue::push_kq(const int *bits, int k, const double *m, uint64_t ctrl_mask) {
  ++submitted;
  HostOp op;
  op.kind = 2;
  op.k = k;
  op.ctrl = ctrl_mask;
  uint64_t qmask = ctrl_mask;
  for (int i = 0; i < k; ++i) {
    op.kq_bits[i] = bits[i];
    qmask |= 1ull << bits[i];
  }
  op.target = bits[0];
  op.kq_m.assign(m, m + (size_t(2) << (2 * k)));
  const int idx = (int)ops.size();
  link_op(*this, op, idx, qmask);
  op.nprev = 7;  // never merged / cancelled
  ops.push_back(std::move(op));
}

void OpQueue::push_pauli(uint64_t xmask, uint64_t zmask, double c, double s) {
  ++submitted;
  if (!(xmask | zmask)) {  // exp(-i theta/2 I): a global factor
    mul_gscale(c, -s);
    ++folded;
    return;
  }
  HostOp op;
  op.kind = 3;
  op.px = xmask;
  op.pz = zmask;
  op.m[0] = c;
  op.m[1] = s;
  const int idx = (int)ops.size();
  link_op(*this, op, idx, xmask | zmask);
  op.nprev = 7;  // never merged / cancelled
  ops.push_back(std::move(op));
}

// --------------------------------------------------------------------- multi-GPU swap logic
std::vector<SwapPair> choose_swaps(int n, int L, const std::vector<int> &perm,
                                   const std::vector<const HostOp *> &pending, bool any_local,
                                   const std::vector<const HostOp *> *future) {
  // global physical bits that pending non-diagonal gates target, within a lookahead window
  std::vector<int> need;
  uint64_t seen = 0;
  const size_t window = std::max<size_t>(64, size_t(4) * n);
  for (size_t i = 0; i < pending.size() && i < window; ++i) {
    const HostOp &h = *pending[i];
    if (h.kind == 2) {  // a dense block runs unfused and needs ALL its qubits inside the shard
      for (int j = 0; j < h.k; ++j) {
        const int pb = perm[h.kq_bits[j]];
        if (pb >= L && !(seen & (1ull << pb))) {
          seen |= 1ull << pb;
          need.push_back(pb);
        }
      }
      continue;
    }
    if (h.kind == 3) {  // a Pauli rotation pairs amplitudes across its X qubits: those must be inside the shard
      for (uint64_t m = h.px; m; m &= m - 1) {
        const int pb = perm[__builtin_ctzll(m)];
        if (pb >= L && !(seen & (1ull << pb))) {
          seen |= 1ull << pb;
          need.push_back(pb);
        }
      }
      continue;
    }
    if (h.kind != 0 || h.type == G_DIAG) continue;
    const int pb = perm[h.target];
    if (pb >= L && !(seen & (1ull << pb))) {
      seen |= 1ull << pb;
      need.push_back(pb);
    }
  }
  std::sort(need.begin(), need.end());
  const int k = (int)need.size();
  std::vector<int> evict;
  if (!any_local || L - 5 < k) {
    for (int i = 0; i < k; ++i) evict.push_back(L - 1 - i);
  } else {
    // next use (as a non-diagonal target) of the qubit sitting on each local physical bit
    std::vector<int> logical_of(n, -1);
    for (int q = 0; q < n; ++q) logical_of[perm[q]] = q;
    std::vector<std::pair<long, int>> cand;  // (-next_use, -bit): furthest first, high bits first
    for (int b = 5; b < L; ++b) {
      long next = 1L << 40;
      for (size_t i = 0; i < pending.size(); ++i) {
        const HostOp &h = *pending[i];
        if (h.kind == 0 && h.type != G_DIAG && h.target == logical_of[b]) {
          next = (long)i;
          break;
        }
        if (h.kind == 2)
          for (int j = 0; j < h.k; ++j)
            if (h.kq_bits[j] == logical_of[b]) next = std::min(next, (long)i);
        if (h.kind == 3 && ((h.px >> logical_of[b]) & 1ull)) next = std::min(next, (long)i);
      }
      // not needed again in this flush: if the caller knows what comes after it (the same op
      // stream again, for an iterated circuit), look there -- the qubits that end a step on the
      // rank bits are then the ones the NEXT step needs last, and the layout settles into a cycle
      if (next == (1L << 40) && future)
        for (size_t i = 0; i < future->size(); ++i) {
          const HostOp &h = *(*future)[i];
          if (h.kind == 0 && h.type != G_DIAG && h.target == logical_of[b]) {
            next = (long)(pending.size() + i);
            break;
          }
        }
      cand.emplace_back(-next, -b);
    }
    std::sort(cand.begin(), cand.end());
    for (int i = 0; i < k; ++i) evict.push_back(-cand[i].second);
    std::sort(evict.begin(), evict.end(), std::greater<int>());
  }
  std::vector<SwapPair> out;
  for (int i = 0; i < k; ++i) out.push_back({need[i], evict[i]});
  return out;
}

std::vector<SwapStep> swap_schedule(int rank, int L, const std::vector<SwapPair> &pairs) {
  const int k = (int)pairs.size();
  uint32_t mine = 0;  // my value of the swapped rank bits, as a k-bit selector
  for (int i = 0; i < k; ++i)
    if ((rank >> (pairs[i].gbit - L)) & 1) mine |= 1u << i;
  std::vector<SwapStep> out;
  // XOR order: at step s every rank is paired with the rank whose swapped bits differ by s,
  // so the steps of all ranks match up (no rank waits for a busy peer)
  for (uint32_t s = 1; s < (1u << k); ++s) {
    const uint32_t sel = mine ^ s;  // the peer's value of the swapped rank bits
    int r = rank;
    for (int i = 0; i < k; ++i) {
      const int rb = pairs[i].gbit - L;
      r = (r & ~(1 << rb)) | (int)(((sel >> i) & 1u) << rb);
    }
    out.push_back({r, sel, mine});
  }
  return out;
}

bool fused_exchange_geometry(const DevPass &last, int L, int rank, int nranks, const std::vector<SwapPair> &sw, XchGeom *out) {
  if (!last.oop || sw.empty() || sw.size() > 4 || nranks > kMaxXchRanks) return false;
  for (const SwapPair &sp : sw)
    if (sp.lbit < 1 || sp.lbit >= L || sp.gbit < L) return false;  // (bit 0: a 32-byte store of a register pair stays whole)
  XchGeom X;
  memset(&X, 0, sizeof X);
  X.n = (uint32_t)sw.size();
  X.rbase = (uint32_t)rank;
  for (size_t i = 0; i < sw.size(); ++i) {
    const uint32_t rb = (uint32_t)(sw[i].gbit - L);
    X.lbit[i] = (uint32_t)sw[i].lbit;
    X.rbit[i] = rb;
    X.vmask |= 1ull << sw[i].lbit;
    X.vconst |= uint64_t((rank >> rb) & 1) << sw[i].lbit;
    X.rbase &= ~(1u << rb);
  }
  // per register index of the last round: its store offset (as the kernels form it, out_pos of the round's
  // register bits) seen through the victims' positions
  const DevRound &RL = last.rounds[last.nrounds - 1];
  for (uint32_t i = 0; i < (1u << last.reg_bits) && i < 32u; ++i) {
    uint64_t off = 0;
    for (uint32_t j = 0; j < last.reg_bits; ++j)
      if ((i >> j) & 1u) off |= 1ull << last.out_pos[RL.reg_pos[j]];
    uint32_t d = 0;
    for (uint32_t k = 0; k < X.n; ++k) d |= uint32_t((off >> X.lbit[k]) & 1ull) << X.rbit[k];
    X.dr[i] = (uint8_t)d;
  }
  *out = X;
  return true;
}

uint64_t place_sel(uint32_t sel, const std::vector<SwapPair> &pairs) {
  uint64_t m = 0;
  for (size_t i = 0; i < pairs.size(); ++i)
    if ((sel >> i) & 1u) m |= 1ull << pairs[i].lbit;
  return m;
}

void apply_swaps_to_perm(std::vector<int> &perm, const std::vector<SwapPair> &pairs) {
  for (const SwapPair &sp : pairs) {
    int la = -1, lb = -1;
    for (size_t q = 0; q < perm.size(); ++q) {
      if (perm[q] == sp.gbit) la = (int)q;
      if (perm[q] == sp.lbit) lb = (int)q;
    }
    if (la >= 0 && lb >= 0) std::swap(perm[la], perm[lb]);
  }
}

// --------------------------------------------------------------------- one pass
namespace {

struct RoundTmp {
  uint64_t regmask = 0;          // physical bits
  uint64_t swap_ctrl = 0;        // control bits of the X / CX gates placed in this round
  std::vector<int> ops;          // op indices, program order
};

int tile_local_index(const std::vector<int> &tile_bits, int phys) {
  for (size_t i = 0; i < tile_bits.size(); ++i)
    if (tile_bits[i] == phys) return (int)i;
  return -1;
}

}  // namespace

static bool plan_one_pass(const std::vector<PhysOp> &ops, std::vector<char> &done, int L, int rank,
                          const PlanOptions &opt, PassPlan &out, const std::vector<int> &label, bool layout_unknown,
                          const std::vector<long> &again) {
  const int T = opt.tile_bits, R = opt.reg_bits;
  const int C = std::min(std::max(opt.low_bits, kLaneFixedBits), T);
  const int max_rounds = std::max(1, std::min(opt.max_rounds, kMaxRounds));
  const int max_gates = std::max(1, std::min(opt.max_pass_gates, kMaxPassGates));
  uint64_t tile_mask = (1ull << C) - 1;
  int ntile = C;
  // Out-of-place passes re-sort the qubit layout after every pass, and that layout must depend on the
  // op stream only (an iterated circuit then finds its pass structures again).  Every decision below
  // is therefore taken by qubit LABEL where it used to be taken by position, and the first pass of a
  // plan -- which meets whatever layout history left -- picks its gates as if the low bits were empty:
  // the qubits sitting there are passengers (T - C targets at most, whoever they are).
  const bool by_label = opt.oop != 0;
  const bool passengers = by_label && layout_unknown;
  uint64_t hot_mask = 0;  // bits that carry a non-diagonal gate in this pass
  const int max_hot = (opt.hot_bits > 0 && opt.hot_bits < T) ? opt.hot_bits : 0;
  uint64_t blocked = 0;
  // tile bits that must stay on lanes in the load / store rounds: 3 = whole 128-byte lines per
  // quarter-warp, 1 = whole 32-byte sectors per lane pair (same DRAM traffic, more lines per request)
  const int lane_fixed = std::max(0, std::min(opt.lane_fixed, kLaneFixedBits));
  const uint64_t lowfixed = (1ull << lane_fixed) - 1;
  std::vector<RoundTmp> rounds;
  int lastround[64];
  std::fill(lastround, lastround + 64, 0);
  std::vector<std::pair<int, int>> chosen;  // (op index, round)
  const uint64_t allq = ~0ull;
  (void)allq;

  for (size_t i = 0; i < ops.size() && (int)chosen.size() < max_gates; ++i) {
    if (done[i]) continue;
    const PhysOp &op = ops[i];
    const uint64_t tb = 1ull << op.target;
    const uint64_t qmask = op.ctrl | tb;
    if (qmask & blocked) {
      blocked |= qmask;
      continue;
    }
    int r0 = 0;
    for (uint64_t q = qmask; q; q &= q - 1) r0 = std::max(r0, lastround[__builtin_ctzll(q)]);
    int place = -1;
    if (op.type == G_DIAG) {
      place = r0;
      if ((int)rounds.size() <= place) rounds.resize(place + 1);
    } else {
      if (op.target >= L) {  // needs a global<->local swap first
        blocked |= qmask;
        continue;
      }
      const bool in_tile = (tile_mask & tb) != 0;
      if (!in_tile && ntile >= T) {
        blocked |= qmask;
        continue;
      }
      if (passengers && !(hot_mask & tb) && popc(hot_mask) >= T - C) {
        blocked |= qmask;
        continue;
      }
      if (max_hot > 0 && !(hot_mask & tb) && popc(hot_mask) >= max_hot) {  // too many distinct targets
        blocked |= qmask;
        continue;
      }
      // Two attempts: first refuse rounds where an X / CX would end up with a control on a
      // REGISTER bit (that flavour moves data, ~150 instructions per thread, instead of toggling
      // the flip mask); if no round qualifies, accept such a round.
      // (avoid_regswap = 2: the first attempt only looks at rounds that already exist -- never
      //  pay a new round, i.e. a transpose, to save a register swap)
      const int nexisting = (int)rounds.size();
      for (int attempt = opt.avoid_regswap ? 0 : 1; attempt < 2 && place < 0; ++attempt) {
        for (int r = r0; r < max_rounds; ++r) {
          if (attempt == 0 && opt.avoid_regswap == 2 && r >= std::max(nexisting, 1)) break;
          const bool edge = (r == 0) || (r == max_rounds - 1);  // load round / last possible store round
          if (edge && (tb & lowfixed)) continue;
          while ((int)rounds.size() <= r) rounds.emplace_back();
          RoundTmp &rd = rounds[r];
          if (attempt == 0) {
            if (op.type == G_SWAP && (rd.regmask & op.ctrl)) continue;           // my control is a register bit here
            if (!(rd.regmask & tb) && (rd.swap_ctrl & tb)) continue;             // I would turn a placed CX's control into one
          }
          if ((rd.regmask & tb) || popc(rd.regmask) < R) {
            place = r;
            break;
          }
        }
      }
      if (place < 0) {
        // drop trailing empty rounds the search may have appended
        while (!rounds.empty() && rounds.back().ops.empty() && rounds.back().regmask == 0 &&
               (int)rounds.size() > 1)
          rounds.pop_back();
        blocked |= qmask;
        continue;
      }
      rounds[place].regmask |= tb;
      hot_mask |= tb;
      if (op.type == G_SWAP) rounds[place].swap_ctrl |= op.ctrl;
      if (!in_tile) {
        tile_mask |= tb;
        ++ntile;
      }
    }
    rounds[place].ops.push_back((int)i);
    chosen.emplace_back((int)i, place);
    for (uint64_t q = qmask; q; q &= q - 1) lastround[__builtin_ctzll(q)] = place;
  }
  if (chosen.empty()) return false;
  while ((int)rounds.size() > 1 && rounds.back().ops.empty()) rounds.pop_back();
  // the store round may not keep bits 0..2 in registers
  if (rounds.back().regmask & lowfixed) rounds.emplace_back();
  if (rounds[0].regmask & lowfixed) return false;  // cannot happen (edge rule), defensive

  // what the remaining ops want next: first use of the qubit on each local bit as a non-diagonal target
  const long never = 1L << 40;
  std::vector<long> next_phys(L, never);
  {
    std::vector<char> picked(ops.size(), 0);
    for (auto &pr : chosen) picked[pr.first] = 1;
    for (size_t i = 0; i < ops.size(); ++i) {
      if (done[i] || picked[i]) continue;
      const PhysOp &op = ops[i];
      if (op.type == G_DIAG || op.target >= L) continue;
      if (next_phys[op.target] == never) next_phys[op.target] = (long)i;
    }
  }
  // soonest first.  Qubits nothing waits for any more: as if the same op stream came again (an
  // iterated circuit -- the layout a flush leaves behind is then the one its own first pass wants:
  // low bits plus the run above the block instead of the top bits of the index, 7.3 instead of
  // 10.5 ms for that pass); what the stream never targets, by label.  All of it layout-independent.
  for (int b = 0; b < L; ++b)
    if (next_phys[b] == never && label[b] >= 0 && label[b] < (int)again.size() && again[label[b]] < never)
      next_phys[b] = (long)ops.size() + again[label[b]];
  auto before = [&](int pa, int pb) {
    if (next_phys[pa] != next_phys[pb]) return next_phys[pa] < next_phys[pb];
    return label[pa] < label[pb];
  };
  // fill the tile -- bits whose value is KNOWN for every non-zero amplitude last: outside the tile
  // each of them halves the number of live tiles.  In place: the lowest unused local bits.  Out of
  // place: the qubits needed soonest, wherever they sit (they arrive in the block one pass early).
  {
    std::vector<int> cand;
    for (int b = 0; b < L; ++b)
      if (!(tile_mask & (1ull << b))) cand.push_back(b);
    if (by_label) std::sort(cand.begin(), cand.end(), before);
    for (int pass2 = 0; pass2 < 2; ++pass2)
      for (int b : cand)
        if (ntile < T && !(tile_mask & (1ull << b)) && (pass2 == 1 || !(opt.known_mask & (1ull << b)))) {
          tile_mask |= 1ull << b;
          ++ntile;
        }
  }
  // tile-local bit order: ascending position -- or, by label, the low C bits (the contiguous chunk)
  // followed by the other members in label order: everything the rounds below decide then depends
  // on WHO is in the tile, not on where history put them
  std::vector<int> tile_bits;
  for (int b = 0; b < L; ++b)
    if (tile_mask & (1ull << b)) tile_bits.push_back(b);
  if (by_label)
    std::sort(tile_bits.begin() + std::min<size_t>(C, tile_bits.size()), tile_bits.end(),
              [&](int a, int b) { return label[a] < label[b]; });

  const int nrounds = (int)rounds.size();
  // ---- layout of every round: which tile bits sit in registers / lanes / warp-id bits.
  // A transpose between two rounds whose warp-id bits carry the SAME tile bits is warp-local:
  // each warp reads back exactly the shared-memory slots it wrote, so __syncwarp() replaces the
  // two CTA barriers and the warps of a CTA stay decoupled.  The warp bits are therefore kept
  // as long as no gate needs them in registers, and re-chosen Belady-style (the bits whose next
  // use as a register bit is furthest away) when one does.  Tile-local bits 0..2 are never warp
  // bits: they are the lanes that make global accesses whole 128-byte lines.
  const int nw = std::max(0, T - R - 5);
  auto tl_of = [&](int phys) { return tile_local_index(tile_bits, phys); };
  std::vector<uint32_t> req(nrounds, 0);  // tile-local masks
  for (int r = 0; r < nrounds; ++r)
    for (int i = 0; i < T; ++i)
      if (rounds[r].regmask & (1ull << tile_bits[i])) req[r] |= 1u << i;
  std::vector<std::vector<int>> warp_bits(nrounds), lane_bits(nrounds), reg_bits_v(nrounds), qw_lanes(nrounds);
  {
    // quarter-warp lanes: three tile-local bits with distinct residues mod 3, outside `busy`
    auto pick_qw = [&](uint32_t busy, int out[3]) {
      for (int res = 0; res < 3; ++res) {
        out[res] = -1;
        for (int i = res; i < T; i += 3)
          if (!(busy & (1u << i))) {
            out[res] = i;
            break;
          }
      }
      return out[0] >= 0 && out[1] >= 0 && out[2] >= 0;
    };
    std::vector<int> W;  // current warp bits (tile-local), ascending
    for (int r = 0; r < nrounds; ++r) {
      const bool edge = (r == 0) || (r == nrounds - 1);
      uint32_t wmask = 0;
      for (int w : W) wmask |= 1u << w;
      bool keep = (int)W.size() == nw && !(wmask & req[r]);
      int qw[3];
      if (keep && !pick_qw(req[r] | wmask, qw)) keep = false;  // keeping W would cost bank conflicts
      if (!keep) {
        wmask = 0;
        const bool have_qw = pick_qw(req[r], qw);
        uint32_t busy = req[r];
        if (have_qw) busy |= (1u << qw[0]) | (1u << qw[1]) | (1u << qw[2]);
        // candidates: free bits >= 3, furthest next use as a register first (Belady)
        std::vector<std::pair<int, int>> cand;
        // (out of place: the whole contiguous chunk -- tile-local bits < C -- stays on lanes, so that a
        //  warp's load covers 2^C contiguous amplitudes: measured 6.3 -> 6.0 ms per memory-only pass)
        const int first_warp_cand = (by_label && opt.chunk_lanes && T - C >= nw + R) ? C : kLaneFixedBits;
        for (int i = first_warp_cand; i < T; ++i) {
          if (busy & (1u << i)) continue;
          int next = 1000;
          for (int r2 = r + 1; r2 < nrounds; ++r2)
            if (req[r2] & (1u << i)) {
              next = r2;
              break;
            }
          cand.emplace_back(-next, -i);
        }
        std::sort(cand.begin(), cand.end());
        W.clear();
        for (size_t k = 0; k < cand.size() && (int)W.size() < nw; ++k) W.push_back(-cand[k].second);
        std::sort(W.begin(), W.end());
        for (int w : W) wmask |= 1u << w;
        if (!have_qw) pick_qw(req[r] | wmask, qw);  // best effort
      }
      warp_bits[r] = W;
      uint32_t qmask = 0;
      for (int k = 0; k < 3; ++k)
        if (qw[k] >= 0) {
          qmask |= 1u << qw[k];
          qw_lanes[r].push_back(qw[k]);
        }
      if (qw_lanes[r].size() != 3) {
        qw_lanes[r].clear();
        qmask = 0;
      }
      std::sort(qw_lanes[r].begin(), qw_lanes[r].end());
      // fill the register set to exactly R bits: highest free bits (not warp bits, not the
      // quarter-warp lanes, and never bits 0..2 in a load / store round)
      // Filler bits that are CONTROLS of an X / CX of this round come last: a control that is not
      // a register bit keeps the gate a flip-mask toggle instead of a register swap.
      uint32_t ctl = 0;
      for (int i = 0; i < T; ++i)
        if (rounds[r].swap_ctrl & (1ull << tile_bits[i])) ctl |= 1u << i;
      uint32_t regm = req[r];
      for (int pass2 = 0; pass2 < 3; ++pass2)
        for (int i = T - 1; i >= 0 && popc(regm) < R; --i) {
          if ((regm | wmask) & (1u << i)) continue;
          if (edge && i < lane_fixed) continue;
          if (pass2 == 0 && ((qmask | ctl) & (1u << i))) continue;
          if (pass2 == 1 && (qmask & (1u << i))) continue;
          regm |= 1u << i;
        }
      rounds[r].regmask = 0;
      for (int i = 0; i < T; ++i) {
        if (regm & (1u << i)) {
          reg_bits_v[r].push_back(i);
          rounds[r].regmask |= 1ull << tile_bits[i];
        } else if (!(wmask & (1u << i))) {
          lane_bits[r].push_back(i);
        }
      }
    }
  }
  (void)tl_of;

  out = PassPlan();
  out.tile_bits = T;
  out.reg_bits = R;
  out.nrounds = nrounds;
  out.ngates = (int)chosen.size();
  out.tile_mask = tile_mask;
  // dead tiles: a non-tile bit with a known value selects, for every tile, whether it holds
  // anything but zeros.  Finite gates map zero tiles to zero tiles, so the dead ones are
  // never read or written (a fresh |0...0>, everything after a collapse / reset).
  uint64_t kmask = opt.known_mask & ~tile_mask & ((L >= 64) ? ~0ull : ((1ull << L) - 1ull));
  for (auto &pr : chosen)
    for (int k = 0; k < 8; ++k)
      if (!std::isfinite(ops[pr.first].m[k])) kmask = 0;  // 0 * NaN = NaN: every tile is live
  {
    int nr = 0, b = 0;
    const uint64_t skip = tile_mask | kmask;
    while (b < L) {
      if (skip & (1ull << b)) {
        ++b;
        continue;
      }
      while (b < L && !(skip & (1ull << b))) ++b;
      ++nr;
    }
    if (nr > kMaxRuns) kmask = 0;
  }
  out.ntiles = 1ull << (L - T - popc(kmask));
  out.blob.assign(pass_bytes((uint32_t)chosen.size()), 0);
  DevPass *P = reinterpret_cast<DevPass *>(out.blob.data());
  DevGate *G = reinterpret_cast<DevGate *>(out.blob.data() + sizeof(DevPass));
  P->nrounds = nrounds;
  P->ngates = (uint32_t)chosen.size();
  P->tile_bits = T;
  P->reg_bits = R;
  P->local_bits = L;
  P->rank_bits = uint64_t(rank) << L;
  P->gscale[0] = 1.0;
  P->gscale[1] = 0.0;
  P->has_gscale = 0;
  P->l2_prefetch = (uint32_t)opt.l2_prefetch;
  P->jit_group = (uint32_t)opt.jit_group;
  P->jit_pf_last = (uint32_t)opt.jit_pf_last;
  P->jit_minb = (uint32_t)opt.jit_minb;
  P->jit_mem = (uint32_t)opt.jit_mem;
  P->tma = (uint32_t)opt.tma;
  P->pf_lines = (uint32_t)opt.pf_lines;
  P->dbg_skip = (uint32_t)opt.dbg_skip;
  P->sm_count = 148;
  for (int i = 0; i < T; ++i) P->tile_pos[i] = (uint8_t)tile_bits[i];
  P->base_fixed = opt.known_val & kmask;
  {  // runs of the free (non-tile, not known) local bits, ascending
    uint32_t nruns = 0;
    int b = 0;
    const uint64_t skip = tile_mask | kmask;
    while (b < L) {
      if (skip & (1ull << b)) {
        ++b;
        continue;
      }
      int e = b;
      while (e < L && !(skip & (1ull << e))) ++e;
      P->run_shift[nruns] = b;
      P->run_len[nruns] = e - b;
      ++nruns;
      b = e;
    }
    P->nruns = nruns;
  }

  uint32_t gcount = 0;
  std::vector<int> last_order;  // thread-bit order of the last round (tile-local bits, lanes first)
  for (int r = 0; r < nrounds; ++r) {
    DevRound &RD = P->rounds[r];
    const bool edge = (r == 0) || (r == nrounds - 1);
    RD.nthr_bits = T - R;
    const std::vector<int> &regs = reg_bits_v[r];
    // thread-id bit order: lanes first, warp-id bits last.  Load/store rounds keep the lanes
    // ascending (bits 0..2 first = whole 128-byte lines per quarter-warp).  Inner rounds put
    // three lane positions with distinct residues mod 3 first so that each quarter-warp's
    // 128-bit shared accesses hit 8 distinct bank groups under the XOR swizzle.
    std::vector<int> order;
    {
      std::vector<int> rest = lane_bits[r];
      // (with lane_fixed < 3 the load / store rounds use the same rule: bit 0 is then always the
      //  first lane, and bits 1, 2 follow whenever they are not register bits)
      bool qw_ok = (!edge || lane_fixed < kLaneFixedBits) && qw_lanes[r].size() == 3;
      for (int q : qw_lanes[r])
        if (std::find(rest.begin(), rest.end(), q) == rest.end()) qw_ok = false;  // became a register
      if (qw_ok) {
        for (int q : qw_lanes[r]) rest.erase(std::find(rest.begin(), rest.end(), q));
        order = qw_lanes[r];
      }
      order.insert(order.end(), rest.begin(), rest.end());
      order.insert(order.end(), warp_bits[r].begin(), warp_bits[r].end());
    }
    // round 0 has no transpose into it: its flag says whether the LAST round's warp bits equal the
    // first round's, i.e. whether the first (warp-local) transpose of the NEXT tile only touches
    // slots this warp itself read in the last transpose of this tile.  If not, the kernel must
    // take a CTA barrier after the last transpose's loads even when the next transpose is local.
    RD.warp_local = (r > 0 ? warp_bits[r] == warp_bits[r - 1] : warp_bits[0] == warp_bits[nrounds - 1]) ? 1u : 0u;
    if (r == nrounds - 1) last_order = order;
    for (int j = 0; j < T - R; ++j) RD.tid_pos[j] = (uint8_t)order[j];
    for (int j = 0; j < R; ++j) {
      RD.reg_pos[j] = (uint8_t)regs[j];
      RD.reg_sx[j] = swz_host(1u << regs[j]);
    }
    RD.gate_begin = gcount;
    uint32_t flip_possible = 0;  // register bits an earlier X / CX of this round may have flipped
    for (int oi : rounds[r].ops) {
      const PhysOp &op = ops[oi];
      DevGate &g = G[gcount++];
      std::memcpy(g.m, op.m, sizeof(g.m));
      g.type = op.type;
      auto place_bit = [&](int phys, uint32_t &mreg, uint32_t &mthr, uint64_t &mext) {
        const int tl = (phys < L) ? tile_local_index(tile_bits, phys) : -1;
        if (tl < 0) {
          mext |= 1ull << phys;
          return;
        }
        for (int j = 0; j < R; ++j)
          if (regs[j] == tl) {
            mreg |= 1u << j;
            return;
          }
        for (int j = 0; j < T - R; ++j)
          if (order[j] == tl) {
            mthr |= 1u << j;
            return;
          }
      };
      for (uint64_t q = op.ctrl; q; q &= q - 1) place_bit(__builtin_ctzll(q), g.creg, g.cthr, g.cext);
      if (op.type == G_DIAG) {
        place_bit(op.target, g.dreg, g.dthr, g.dext);
        g.treg = g.dreg ? (uint32_t)__builtin_ctz(g.dreg) : 7u;  // 7: target is not a register bit
      } else {
        uint32_t treg_mask = 0, tthr = 0;
        uint64_t text = 0;
        place_bit(op.target, treg_mask, tthr, text);
        g.treg = treg_mask ? (uint32_t)__builtin_ctz(treg_mask) : 0xffu;  // must be a register bit
      }
      // bit 8 of treg: a flip may be pending on the target register bit (flavour 1 in the kernel)
      if (op.type == G_SWAP && g.creg == 0 && g.treg < 8) {
        flip_possible |= 1u << g.treg;
      } else if (g.treg < 8 && (flip_possible & (1u << g.treg))) {
        g.treg |= 1u << 8;
      }
      // bit 9 of treg: X with exactly one control, a register bit that no earlier toggle of this
      // round can have flipped, and no thread / external controls: WHICH register pairs swap is
      // then the same in every thread (static register swap in the step kernel)
      if (op.type == G_SWAP && popc(g.creg) == 1 && g.cthr == 0 && g.cext == 0 && !(flip_possible & g.creg))
        g.treg |= 1u << 9;
      {  // dense opcode for the kernel's jump table
        const bool ctrl = (g.creg | g.cthr) != 0 || g.cext != 0;
        const uint32_t J = g.treg & 0xffu;
        const uint32_t fl = ctrl ? 2u : ((g.treg >> 8) & 1u);
        if (g.type == G_SWAP) g.op = (g.creg == 0) ? op_toggle(R) : op_swap_reg(R, J);
        else if (g.type == G_DIAG) g.op = (J < 8 && g.dreg) ? op_arith(R, C_DIAG_REG, fl, J) : op_diag_thr(R);
        else g.op = op_arith(R, (g.type == G_GENERAL || g.type == G_GENERAL1) ? C_GENERAL : (g.type == G_ROT ? C_ROT : C_REAL), fl, J);
        if (g.type == G_ROT) {  // shear coefficients from (cos, sin), cos >= 0 by classification
          const double cs = op.m[0], sn = op.m[4];
          std::memset(g.m, 0, sizeof(g.m));
          g.m[0] = -sn / (1.0 + cs);
          g.m[1] = sn;
        }
      }
      out.op_index.push_back(oi);
    }
    RD.gate_end = gcount;
    out.round_regmask.push_back(rounds[r].regmask);
  }
  out.gates.assign(G, G + gcount);
  // ---- where the tile is stored.  In place: where it came from.  Out of place (every tile live):
  // as one contiguous block, tile number = block number; WHICH tile qubit lands on which of the T
  // low bits is free.  Bits 0..2 (one 128-byte line) go to three LANE bits of the last round, so
  // that a quarter warp stores whole lines; among them, and for every other position, the qubits
  // the remaining ops target soonest come first: the next pass always holds the lowest bits in
  // its tile (its loads gather chunks of at least one line), and the longer the run of low bits it
  // really needs, the longer those chunks are.
  for (int i = 0; i < T; ++i) P->out_pos[i] = P->tile_pos[i];
  P->oop = 0;
  P->onruns = 0;
  if (opt.oop && kmask == 0) {
    // a passenger of the first pass that no gate of it touched goes behind the pass's own qubits
    auto plain_passenger = [&](int pb) { return passengers && pb < C && !(hot_mask & (1ull << pb)); };
    auto before_out = [&](int pa, int pb) {
      const bool xa = plain_passenger(pa), xb = plain_passenger(pb);
      if (xa != xb) return xb;
      return before(pa, pb);
    };
    const int nlanes = std::min(5, T - R);
    std::vector<int> lanes(last_order.begin(), last_order.begin() + nlanes);
    std::sort(lanes.begin(), lanes.end(), [&](int a, int b) { return before_out(tile_bits[a], tile_bits[b]); });
    // (only three: all five lanes on the five lowest bits would make a warp's store 512 contiguous
    //  bytes, but the qubits needed next are the last round's REGISTER bits more often than not, and
    //  keeping them off the low bits costs 5 passes in 31)
    std::vector<int> seq(lanes.begin(), lanes.begin() + std::min(3, nlanes));
    std::vector<int> rest;
    for (int i = 0; i < T; ++i)
      if (std::find(seq.begin(), seq.end(), i) == seq.end()) rest.push_back(i);
    std::sort(rest.begin(), rest.end(), [&](int a, int b) { return before_out(tile_bits[a], tile_bits[b]); });
    seq.insert(seq.end(), rest.begin(), rest.end());
    for (int p = 0; p < T; ++p) P->out_pos[seq[p]] = (uint8_t)p;
    P->oop = 1;
    out.newpos.assign(L, -1);
    for (int i = 0; i < T; ++i) out.newpos[tile_bits[i]] = P->out_pos[i];
    // the qubits outside the tile: sorted the same way above bit T (oop = 1), or left in their order
    std::vector<int> outside;
    for (int b = 0; b < L; ++b)
      if (out.newpos[b] < 0) outside.push_back(b);
    std::vector<int> sorted_out = outside;
    if (opt.oop == 1) std::sort(sorted_out.begin(), sorted_out.end(), before);
    for (size_t k = 0; k < sorted_out.size(); ++k) out.newpos[sorted_out[k]] = T + (int)k;
    // ---- the ORDER in which the tile number enumerates the qubits outside the tile.  The CTAs of the
    // persistent grid work on consecutive tile numbers at any one time, so the low bits of the tile
    // number decide which addresses are in flight together -- on the load side through the bit each
    // qubit comes from, on the store side through the bit it goes to.  Bits above the DRAM channel
    // hash (address bit 27 = index bit 23 on B200, measured: scripts/copy_ubench2.cu) map to the same
    // channel: if they vary among concurrent tiles, the whole grid queues on a few channels.  Fast
    // tile-number bits therefore go to qubits that sit LOW on both sides.
    std::vector<int> order = outside;
    std::stable_sort(order.begin(), order.end(),
                     [&](int a, int b) { return std::max(a, out.newpos[a]) < std::max(b, out.newpos[b]); });
    for (int attempt = 0; attempt < 3; ++attempt) {
      // attempt 0: that order; 1: ascending source bits (the in-place enumeration); 2: also the qubits
      // outside the tile keep their order (always fits: one run on the store side)
      if (attempt >= 1) order = outside;
      if (attempt == 2)
        for (size_t k = 0; k < outside.size(); ++k) out.newpos[outside[k]] = T + (int)k;
      uint32_t nin = 0, nout = 0;
      bool fits = true;
      uint32_t in_shift[kMaxRuns], in_len[kMaxRuns];
      for (size_t j = 0; j < order.size() && fits;) {  // load side: runs of consecutive source bits
        size_t e = j + 1;
        while (e < order.size() && order[e] == order[e - 1] + 1) ++e;
        if (nin >= (uint32_t)kMaxRuns) fits = false;
        else {
          in_shift[nin] = (uint32_t)order[j];
          in_len[nin] = (uint32_t)(e - j);
          ++nin;
        }
        j = e;
      }
      for (size_t j = 0; j < order.size() && fits;) {  // store side: runs of consecutive destination bits
        size_t e = j + 1;
        while (e < order.size() && out.newpos[order[e]] == out.newpos[order[e - 1]] + 1) ++e;
        if (nout >= (uint32_t)kMaxOutRuns) fits = false;
        else {
          P->orun_len[nout] = (uint8_t)(e - j);
          P->orun_shift[nout] = (uint8_t)out.newpos[order[j]];
          ++nout;
        }
        j = e;
      }
      if (!fits) continue;
      P->onruns = nout;
      P->nruns = nin;
      for (uint32_t k = 0; k < nin; ++k) {
        P->run_shift[k] = in_shift[k];
        P->run_len[k] = in_len[k];
      }
      break;
    }
  }
  {
    bool lite = opt.lite != 0;
    for (uint32_t gi = 0; gi < gcount && lite; ++gi) {
      const DevGate &g = G[gi];
      const bool ctrl = (g.creg | g.cthr) != 0 || g.cext != 0;
      if (!(g.type == G_SWAP ||
            ((g.type == G_ROT || g.type == G_REAL || g.type == G_GENERAL || g.type == G_GENERAL1) && !ctrl)))
        lite = false;
    }
    std::vector<DevStep> steps;
    if (lite) {
      // ---- pack every round into steps (ASAP list scheduling; ops on disjoint qubits commute).
      // Position = 3 * step + phase, phase 0 = 1-qubit slots, 1 = toggles (list order), 2 = the
      // register-controlled X.  An op goes to the earliest position after the last op that
      // shares a qubit with it.
      for (int r = 0; r < nrounds; ++r) {
        DevRound &RD = P->rounds[r];
        const size_t first = steps.size();
        int last_pos[64];
        std::fill(last_pos, last_pos + 64, -1);
        auto step_at = [&](size_t k) -> DevStep & {
          while (steps.size() <= first + k) {
            DevStep s0{};
            s0.swap_j = 0xffu;  // none
            steps.push_back(s0);
          }
          return steps[first + k];
        };
        for (uint32_t gi = RD.gate_begin; gi < RD.gate_end; ++gi) {
          const DevGate &g = G[gi];
          const PhysOp &op = ops[out.op_index[gi]];
          const uint64_t qmask = op.ctrl | (1ull << op.target);
          int lb = -1;
          for (uint64_t q = qmask; q; q &= q - 1) lb = std::max(lb, last_pos[__builtin_ctzll(q)]);
          const uint32_t J = g.treg & 0xffu;
          int pos;
          if (g.type != G_SWAP) {  // a 1-qubit slot
            int k = (lb < 0) ? 0 : lb / 3 + 1;
            DevStep &S = step_at(k);
            uint32_t kind;
            if (g.type == G_ROT) {
              kind = SLOT_ROT;
              S.slot[J][0] = g.m[0];
              S.slot[J][1] = g.m[1];
              S.slot[J][2] = op.m[0];  // (cos, sin) for the structure-specialised kernels (qb_jit.cpp)
              S.slot[J][3] = op.m[4];
            } else if (g.type == G_REAL) {
              kind = SLOT_REAL;
              for (int e = 0; e < 4; ++e) S.slot[J][e] = g.m[2 * e];
            } else {
              kind = (g.type == G_GENERAL1 && !((g.treg >> 8) & 1u)) ? SLOT_GENERAL1 : SLOT_GENERAL;
              std::memcpy(S.slot[J], g.m, sizeof(g.m));
            }
            if ((g.treg >> 8) & 1u) kind |= SLOT_FLIP;
            S.kinds |= kind << (4 * J);
            pos = 3 * k;
          } else if (g.creg == 0) {  // toggle
            int k = (lb < 0) ? 0 : (lb + 1) / 3;  // smallest k with 3k + 1 >= lb
            while (step_at(k).ntog >= (uint32_t)kStepToggles) ++k;
            DevStep &S = step_at(k);
            S.tog[S.ntog].cthr = g.cthr;
            S.tog[S.ntog].cext = g.cext;
            S.tog[S.ntog].bit = J;
            ++S.ntog;
            pos = 3 * k + 1;
          } else {  // X / CX with a register-bit control: data moves
            int k = (lb < 0) ? 0 : (lb - 2 + 3) / 3;  // smallest k with 3k + 2 > lb
            while (3 * k + 2 <= lb) ++k;
            while (step_at(k).swap_j < 0x80u) ++k;
            DevStep &S = step_at(k);
            S.swap_j = J | (((g.treg >> 9) & 1u) << 4);  // bit 4: static flavour
            S.swap_creg = g.creg;
            S.swap_cthr = g.cthr;
            S.swap_cext = g.cext;
            pos = 3 * k + 2;
          }
          for (uint64_t q = qmask; q; q &= q - 1) last_pos[__builtin_ctzll(q)] = pos;
        }
        RD.step_begin = (uint32_t)first;
        RD.step_end = (uint32_t)steps.size();
      }
      if ((int)steps.size() > kMaxSteps) lite = false;  // (never seen: a pass holds <= 96 gates) -> interpreter
    }
    if (lite) {
      bool rot_only = true;
      for (const DevStep &st : steps)
        for (int J = 0; J < kMaxRegBits; ++J) {
          const uint32_t cls = (st.kinds >> (4 * J)) & SLOT_CLASS;
          if (cls != SLOT_NONE && cls != SLOT_ROT) rot_only = false;
        }
      P->lite = rot_only ? 1u : 2u;  // which step-kernel instantiation (qb_kernels.cu)
      P->nsteps = (uint32_t)steps.size();
      std::vector<uint8_t> blob(sizeof(DevPass) + steps.size() * sizeof(DevStep));
      std::memcpy(blob.data(), out.blob.data(), sizeof(DevPass));
      if (!steps.empty()) std::memcpy(blob.data() + sizeof(DevPass), steps.data(), steps.size() * sizeof(DevStep));
      out.blob.swap(blob);
    }
  }
  for (auto &pr : chosen) done[pr.first] = 1;
  return true;
}

PlanResult plan_passes(const std::vector<PhysOp> &ops_in, int local_bits, int rank, const PlanOptions &opt_in,
                       const double *gscale, const std::vector<int> *labels) {
  PlanResult res;
  std::vector<int> label(local_bits);
  for (int b = 0; b < local_bits; ++b) label[b] = (labels && b < (int)labels->size()) ? (*labels)[b] : b;
  PlanOptions opt = opt_in;  // known_mask / known_val evolve pass by pass
  if (gscale && !(std::isfinite(gscale[0]) && std::isfinite(gscale[1]))) opt.known_mask = 0;
  std::vector<PhysOp> ops = ops_in;  // (an out-of-place pass moves qubits: the ops after it are relabelled)
  // first use of every qubit (by label) in this op stream as a non-diagonal target
  std::vector<long> again;
  {
    int maxl = -1;
    for (int b = 0; b < local_bits; ++b) maxl = std::max(maxl, label[b]);
    again.assign(maxl + 1, 1L << 40);
    for (size_t i = 0; i < ops.size(); ++i) {
      const PhysOp &op = ops[i];
      if (op.type == G_DIAG || op.target >= local_bits) continue;
      const int lb = label[op.target];
      if (lb >= 0 && again[lb] == (1L << 40)) again[lb] = (long)i;
    }
  }
  std::vector<char> done(ops.size(), 0);
  size_t ndone = 0;
  auto relabel_mask = [&](uint64_t m, const std::vector<int> &np) {
    uint64_t o = 0;
    for (uint64_t b = m; b; b &= b - 1) {
      const int bit = __builtin_ctzll(b);
      o |= 1ull << (bit < local_bits ? np[bit] : bit);
    }
    return o;
  };
  while (ndone < ops.size()) {
    if (opt.max_passes > 0 && (int)res.passes.size() >= opt.max_passes) break;
    PassPlan p;
    if (!plan_one_pass(ops, done, local_bits, rank, opt, p, label, res.final_pos.empty() && !opt.layout_known, again)) break;
    ndone += p.op_index.size();
    if (!p.newpos.empty()) {
      // (the support bookkeeping below still reads this pass's ops with their OLD positions)
      for (int oi : p.op_index) {
        const PhysOp &op = ops[oi];
        if (op.type != G_DIAG) opt.known_mask &= ~(1ull << op.target);
        for (int k = 0; k < 8; ++k)
          if (!std::isfinite(op.m[k])) opt.known_mask = 0;
      }
      opt.known_val &= opt.known_mask;
      const std::vector<int> &np = p.newpos;
      for (size_t i = 0; i < ops.size(); ++i) {
        if (done[i]) continue;
        if (ops[i].target < local_bits) ops[i].target = np[ops[i].target];
        ops[i].ctrl = relabel_mask(ops[i].ctrl, np);
      }
      opt.known_val = relabel_mask(opt.known_val, np);
      opt.known_mask = relabel_mask(opt.known_mask, np);
      if (res.final_pos.empty()) {
        res.final_pos.resize(local_bits);
        for (int b = 0; b < local_bits; ++b) res.final_pos[b] = b;
      }
      for (int b = 0; b < local_bits; ++b) res.final_pos[b] = np[res.final_pos[b]];
      {
        std::vector<int> nl(local_bits);
        for (int b = 0; b < local_bits; ++b) nl[np[b]] = label[b];
        label.swap(nl);
      }
      res.passes.push_back(std::move(p));
      continue;
    }
    // a non-diagonal gate forgets its target; a non-finite matrix forgets everything
    for (int oi : p.op_index) {
      const PhysOp &op = ops[oi];
      if (op.type != G_DIAG) opt.known_mask &= ~(1ull << op.target);
      for (int k = 0; k < 8; ++k)
        if (!std::isfinite(op.m[k])) opt.known_mask = 0;
    }
    opt.known_val &= opt.known_mask;
    res.passes.push_back(std::move(p));
  }
  res.consumed = ndone;
  res.done = done;
  res.known_mask = opt.known_mask;
  res.known_val = opt.known_val;
  if (gscale && !res.passes.empty() && !(gscale[0] == 1.0 && gscale[1] == 0.0)) {
    DevPass *P = reinterpret_cast<DevPass *>(res.passes.back().blob.data());
    P->gscale[0] = gscale[0];
    P->gscale[1] = gscale[1];
    P->has_gscale = 1;
  }
  return res;
}

PlanResult plan_passes_until_swap(const std::vector<PhysOp> &ops, int local_bits, int rank, const PlanOptions &opt,
                                  const std::vector<int> *labels) {
  PlanResult plan = plan_passes(ops, local_bits, rank, opt, nullptr, labels);
  if (opt.defer_tail <= 0 || !opt.oop || plan.consumed == ops.size()) return plan;  // (in place: the schedule round 1 measured)
  size_t keep = plan.passes.size();
  while (keep > 1 && plan.passes[keep - 1].ngates <= opt.defer_tail) --keep;
  if (keep == plan.passes.size()) return plan;
  PlanOptions o2 = opt;  // (the passes are planned one after the other: the first `keep` come out the same)
  o2.max_passes = (int)keep;
  return plan_passes(ops, local_bits, rank, o2, nullptr, labels);
}

std::string describe_plan(const PlanResult &r) {
  std::ostringstream os;
  os << "passes=" << r.passes.size() << " scheduled=" << r.consumed << "\n";
  for (size_t i = 0; i < r.passes.size(); ++i) {
    const PassPlan &p = r.passes[i];
    const DevPass *P = reinterpret_cast<const DevPass *>(p.blob.data());
    os << "pass " << i << " T=" << p.tile_bits << " R=" << p.reg_bits << " tiles=" << p.ntiles << " tile=[";
    for (int b = 0; b < p.tile_bits; ++b) os << (b ? "," : "") << (int)P->tile_pos[b];
    os << "] rounds=" << p.nrounds << " gates=" << p.ngates << " gscale=" << P->has_gscale << " lite=" << P->lite
       << " steps=" << P->nsteps;
    if (P->oop) {
      os << " out=[";
      for (int b = 0; b < p.tile_bits; ++b) os << (b ? "," : "") << (int)P->out_pos[b];
      os << "]";
    }
    {
      const DevGate *G = p.gates.data();
      int kinds[8] = {0};
      for (int g = 0; g < p.ngates; ++g) {
        const DevGate &d = G[g];
        const bool ctrl = (d.creg | d.cthr) != 0 || d.cext != 0;
        if (d.type == G_SWAP && d.creg == 0) kinds[0]++;           // flip toggle
        else if (d.type == G_SWAP) kinds[1]++;                     // register-controlled swap (data moves)
        else if (ctrl) kinds[2]++;                                 // controlled non-swap
        else if ((d.treg >> 8) & 1) kinds[3]++;                    // uncontrolled, flip-aware
        else kinds[4]++;                                           // plain
      }
      int types[6] = {0};
      for (int g = 0; g < p.ngates; ++g) types[G[g].type < 6 ? G[g].type : 0]++;
      os << " types[general,real,diag,swap,rot,general1]=" << types[0] << "," << types[1] << "," << types[2] << "," << types[3]
         << "," << types[4] << "," << types[5];
      os << " kinds[toggle,regswap,ctrl,flipaware,plain]=" << kinds[0] << "," << kinds[1] << "," << kinds[2] << ","
         << kinds[3] << "," << kinds[4];
    }
    os << "\n";
    for (int rd = 0; rd < p.nrounds; ++rd) {
      const DevRound &RD = P->rounds[rd];
      os << "  round " << rd << " regs=[";
      for (int j = 0; j < p.reg_bits; ++j) os << (j ? "," : "") << (int)P->tile_pos[RD.reg_pos[j]];
      os << "] local=" << RD.warp_local << " tid=[";
      for (int j = 0; j < p.tile_bits - p.reg_bits; ++j) os << (j ? "," : "") << (int)P->tile_pos[RD.tid_pos[j]];
      os << "] ops=[";
      for (uint32_t g = RD.gate_begin; g < RD.gate_end; ++g) os << (g > RD.gate_begin ? "," : "") << p.op_index[g];
      os << "]\n";
    }
  }
  return os.str();
}

}  // namespace qb
