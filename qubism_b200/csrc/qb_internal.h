// Internal structures shared by the host planner (qb_planner.cpp), the C-ABI layer
// (qb_api.cpp) and the kernels (qb_kernels.cu).  Not installed; the public boundary is
// include/qubism_sv.h.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/qubism_sv.h"

namespace qb {

// ------------------------------------------------------------------ compile-time limits
constexpr int kMaxTileBits = 13;   // 2^13 amplitudes * 16 B = 128 KB of shared memory
constexpr int kMaxRegBits = 5;     // 32 amplitudes (128 32-bit registers) per thread
constexpr int kMaxRounds = 8;      // register-residency rounds per pass
constexpr int kMaxRuns = 16;       // runs of non-tile bits in the tile-index deposit
constexpr int kMaxOutRuns = 32;    // out-of-place passes: runs of tile-number bits in the block address
constexpr int kMaxPassGates = 96;  // gates per pass (bounds the shared-memory program copy)
constexpr int kLaneFixedBits = 3;  // bits 0..2 (one 128-B line) stay on lanes in load/store rounds

// ------------------------------------------------------------------ gate classes
// Classification is by VALUE of the 2x2 the caller passed (SURVEY.md 7.2 "gate
// classification"): it changes instruction count, never results beyond fp64 rounding.
enum GateType : uint32_t {
  G_GENERAL = 0,  // arbitrary complex 2x2                     8 DFMA-slot ops / amplitude
  G_REAL = 1,     // real 2x2 (after pulling a common phase)   4
  G_DIAG = 2,     // diag(d0, d1): target may be ANY bit       4
  G_SWAP = 3,     // [[0,1],[1,0]]: pure permutation           0
  G_ROT = 4,      // rotation [[c,-s],[s,c]], c >= 0 (a scale / sign is pulled into the deferred
                  // scalar): three in-place shears            3
  G_GENERAL1 = 5, // complex 2x2 scaled to m00 = 1 (the scale goes to the deferred scalar): 6 where no
                  // flip can be pending; everywhere else it is just a G_GENERAL matrix
};

// One gate as the fused-pass kernel sees it (per round: register/thread/external split).
struct alignas(16) DevGate {
  double m[8];     // row-major (re,im): a b c d.  G_REAL uses re parts; G_DIAG uses a and d.
                   // G_ROT: m[0] = t = -tan(theta/2), m[1] = s = sin(theta) (the shear coefficients)
  uint32_t type;   // GateType
  uint32_t treg;   // target register bit (GENERAL / REAL / SWAP)
  uint32_t creg;   // controls that are register-index bits   (mask over the 2^R index)
  uint32_t cthr;   // controls that are thread-id bits        (mask over threadIdx.x)
  uint64_t cext;   // controls outside the tile               (mask over the full physical index)
  uint32_t dreg;   // G_DIAG: target as register-index mask   (exactly one of dreg/dthr/dext set)
  uint32_t dthr;   // G_DIAG: target as thread-id mask
  uint64_t dext;   // G_DIAG: target as external mask
  uint32_t op;     // dense kernel opcode (dev_opcode below): one jump-table dispatch per gate
  uint32_t _pad;
};

// Opcode space of k_fused_pass's gate switch, DENSE for a kernel with R register bits (one jump
// table, no decision tree).  FL = flavour: 0 uncontrolled / no flip possible, 1 uncontrolled /
// flip-aware, 2 controlled (flip-aware).  J = target register bit (< R).
#ifdef __CUDACC__
#define QB_HD __host__ __device__
#else
#define QB_HD
#endif
enum GateClass : uint32_t { C_GENERAL = 0, C_REAL = 1, C_ROT = 2, C_DIAG_REG = 3, C_COUNT = 4 };
QB_HD constexpr uint32_t op_arith(int R, uint32_t cls, uint32_t fl, uint32_t J) { return (cls * 3u + fl) * uint32_t(R) + J; }
QB_HD constexpr uint32_t op_swap_reg(int R, uint32_t J) { return C_COUNT * 3u * uint32_t(R) + J; }  // X / CX with a register-bit control
QB_HD constexpr uint32_t op_toggle(int R) { return (C_COUNT * 3u + 1u) * uint32_t(R); }            // X / CX: flip-mask toggle
QB_HD constexpr uint32_t op_diag_thr(int R) { return op_toggle(R) + 1u; }  // diagonal gate, target on a thread bit / outside the tile
QB_HD constexpr uint32_t op_count(int R) { return op_toggle(R) + 2u; }
static_assert(sizeof(DevGate) == 112, "DevGate layout");

// LITE passes (uncontrolled 1-qubit gates of the rotation / real / general class and X / CX only:
// everything the reference interpreter ever sends, QASM/Simulation.hs:94-122,163-171) are not
// interpreted gate by gate: the planner packs each round into STEPS of mutually independent
// work -- one 1-qubit slot per register bit, then up to four flip-mask toggles, then at most one
// register-controlled X --
// which the kernel runs as straight-line code behind a few uniform skip-branches.  No opcode
// fetch, no dispatch tree, no jump table: per step ONE header read, per gate two constants.
constexpr int kStepToggles = 4;
constexpr int kMaxSteps = 72;  // steps per pass (kernel parameter space: 72 * 416 B + header < 32 KB)
// slot kinds (4 bits per register bit in DevStep::kinds): class in bits 0-2, bit 3 = a flip may
// be pending on that register bit (flip-aware flavour)
enum : uint32_t { SLOT_NONE = 0, SLOT_ROT = 1, SLOT_REAL = 2, SLOT_GENERAL = 3, SLOT_GENERAL1 = 4, SLOT_CLASS = 7, SLOT_FLIP = 8 };
struct alignas(16) DevStep {
  double slot[kMaxRegBits][8];  // the 1-qubit gate on register bit J: ROT (t, s); REAL a b c d; GENERAL = DevGate::m
  uint32_t kinds;              // slot kind of register bit J in bits 4J .. 4J+3
  uint32_t _pad;
  uint32_t ntog;               // toggles applied after the slots
  uint32_t swap_j;             // 0xff: none; else bits 0-2 = target register bit of an X / CX with register-bit
                               // control(s), bit 4 = static flavour (one control, a register bit without a
                               // pending flip, no other controls: the same pairs swap in every thread)
  struct Tog {
    uint32_t cthr, bit;
    uint64_t cext;
  } tog[kStepToggles];
  uint32_t swap_creg, swap_cthr;
  uint64_t swap_cext;
};
static_assert(sizeof(DevStep) == 416, "DevStep layout");

// A global<->local swap FUSED into the store of an out-of-place pass (sharded states): the pass
// that precedes the swap writes every tile straight to the rank that owns it afterwards -- into
// that rank's second shard, over NVLink peer memory -- instead of writing locally and exchanging
// in a second sweep.  The k victim qubits sit on bits lbit[i] >= 1 of an amplitude's address in the new
// layout: destination rank = rbase | (their values, on rank bits rbit[i]), destination address =
// the address with those bits replaced by this rank's old rank-bit values.  Worked out store by
// store (the victims are usually the qubits the pass has just finished with: bits INSIDE its block).
constexpr int kMaxXchRanks = 16;
struct XchGeom {
  uint64_t peer[kMaxXchRanks];  // every rank's destination shard as mapped into this process (0 = unused)
  uint64_t vmask, vconst;       // the victims' bits of the block address / what replaces them
  uint32_t n, rbase;            // swapped pairs (0 = plain pass) / this rank with the swapped rank bits cleared
  uint32_t lbit[4], rbit[4];
  // dr[i]: what register index i of the pass's last round adds to the destination rank -- its store offset's
  // bits on the victims' positions, moved to the rank bits.  With it a specialised kernel works out one
  // destination per TILE (from the thread's base address) and one XOR per store instead of shifting
  // run-time bit positions store by store.
  uint8_t dr[32];
  uint32_t _pad[2];
};
static_assert(sizeof(XchGeom) == 224, "XchGeom layout (mirrored by the generated QbjXch)");

struct DevRound {
  uint32_t gate_begin, gate_end;
  uint32_t nthr_bits;                 // T - R
  uint32_t warp_local;                // the transpose INTO this round stays inside each warp
  uint8_t tid_pos[16];                // tile-local bit position carried by thread-id bit j
  uint8_t reg_pos[8];                 // tile-local bit position carried by register bit j
  uint32_t reg_sx[8];                 // swizzled shared-memory index contribution of register bit j
  uint32_t step_begin, step_end;      // lite passes: this round's DevSteps
};
static_assert(sizeof(DevRound) == 80, "DevRound layout");

struct DevPass {
  uint32_t nrounds, ngates, tile_bits, reg_bits;
  uint32_t nruns, local_bits;
  uint64_t rank_bits;                 // rank << local_bits: OR-ed into the tile base for predicates
  uint32_t run_shift[kMaxRuns];       // deposit of the tile id into the non-tile bit runs
  uint32_t run_len[kMaxRuns];
  uint8_t tile_pos[16];               // physical bit position of tile-local bit i
  double gscale[2];                   // deferred global scalar applied on the way out (1,0 = none)
  uint32_t has_gscale;
  uint32_t l2_prefetch;               // prefetch the CTA's next tile into L2 while this one computes
  uint32_t dbg_skip;                  // PROFILING ONLY (results are wrong): bit 0 skip global loads, bit 1 skip
                                      // global stores, bit 2 skip the shared-memory transposes, bit 3 skip gates
  uint32_t sm_count;
  uint32_t lite;                      // 0: rounds index DevGates (interpreter); 1 / 2: DevSteps (1 = every slot is a
                                      // rotation, 2 = rotation / real / general slots)
  uint32_t nsteps;
  uint32_t jit_group;                 // specialised kernels: a CTA takes this many CONSECUTIVE tiles in a row and
                                      // prefetches the next such group with one bulk request per chunk
  uint32_t jit_pf_last;               // ... issued while the LAST (1) or the FIRST (0) tile of the running group computes
  uint64_t base_fixed;                // known non-tile bits at their known value: OR-ed into every live tile's base
  uint32_t jit_minb;                  // specialised kernels: resident CTAs per SM to compile for (0 = automatic)
  uint32_t jit_mem;                   // specialised kernels: cache policy of the global accesses (QBJ_MEM, qb_jit_prelude.cuh)
  uint32_t tma;                       // specialised kernels: 1 = the tile is LOADED with asynchronous bulk copies
                                      // (cp.async.bulk -> shared memory, mbarrier) issued one tile ahead
  uint32_t oop;                       // 1 = OUT OF PLACE with a new qubit layout: every tile is written as ONE
                                      // contiguous block of 2^T amplitudes of the destination shard, tile-local bit i
                                      // at bit out_pos[i] of it (a permutation of 0..T-1); which block: onruns below.
                                      // 0 = the tile goes back where it came from (out_pos == tile_pos).
  uint32_t onruns;                    // oop: the block address of tile number t.  Its bits are taken from the low
                                      // end in onruns groups of orun_len[k] bits, group k placed at bit
                                      // orun_shift[k] (>= T): the qubits outside the tile may be re-ordered too
  uint32_t pf_lines;                  // specialised kernels: lines per thread the L2 prefetch of the next tile covers
                                      // (0 = the whole tile; 1 of 2 = half of it: fewer tiles in flight per SM)
  uint8_t out_pos[16];                // physical bit position tile-local bit i is STORED at
  uint8_t orun_len[kMaxOutRuns];
  uint8_t orun_shift[kMaxOutRuns];
  XchGeom xch;                        // n != 0: this pass's stores carry a global<->local swap (see XchGeom)
  DevRound rounds[kMaxRounds];
  // followed in memory by ngates DevGate records (lite: by nsteps DevStep records)
};
static_assert(sizeof(DevPass) % 16 == 0, "DevPass alignment");

inline size_t pass_bytes(uint32_t ngates) { return sizeof(DevPass) + size_t(ngates) * sizeof(DevGate); }

// shared-memory swizzle: XOR every higher 3-bit group of the tile-local index into the low
// 3 bits (the 16-byte bank group of a 128-bit access).  Linear over XOR.
inline uint32_t swz_host(uint32_t u) {
  return u ^ ((u >> 3) & 7u) ^ ((u >> 6) & 7u) ^ ((u >> 9) & 7u) ^ ((u >> 12) & 7u);
}

// ------------------------------------------------------------------ host-side ops
struct HostOp {
  int kind = 0;             // 0 = (controlled) 1q, 2 = dense kq (barrier op), 3 = Pauli rotation (barrier op)
  uint32_t type = G_GENERAL;
  int target = -1;          // LOGICAL bit position (n-1-q)
  uint64_t ctrl = 0;        // mask over LOGICAL bit positions
  double m[8] = {0};
  // dense kq
  int k = 0;
  int kq_bits[QB_MAX_KQ] = {0};  // logical bit positions, kq_bits[0] = most significant index bit
  std::vector<double> kq_m;
  // Pauli rotation cos(theta/2) I - i sin(theta/2) P: X / Z masks over LOGICAL bit positions; (c, s) in m[0], m[1]
  uint64_t px = 0, pz = 0;
  // peephole bookkeeping
  bool dead = false;
  int nprev = 0;
  int prev_bit[6] = {0};    // for each qubit this op touches: the op that touched it before
  int prev_idx[6] = {0};
};

struct PlanOptions {
  int tile_bits = 12;
  int reg_bits = 4;
  int low_bits = 3;     // low physical bits always in the tile: 3 = one 128-byte line per chunk
                        // (measured: no bandwidth loss vs 512-byte chunks, two more free tile bits)
  int max_rounds = 6;
  int fuse = 1;         // 0: one pass per op
  int peephole = 1;
  int max_pass_gates = kMaxPassGates;
  int time_kernels = 0;
  int l2_prefetch = 1;
  int dbg_skip = 0;       // profiling switches, see DevPass::dbg_skip
  int avoid_regswap = 0;  // planner: refuse rounds where a CX control would be a register bit
  int rot = 1;            // rotations [[c,-s],[s,c]] run as three in-place shears (G_ROT) instead of G_REAL
  int support = 1;          // track the support (known index bits of the non-zero amplitudes): live sub-cube
                            // reductions, collapse = zero-fill + deferred scalar.  0 = A/B baseline
  int skip_dead = 1;        // use the state's support: fused passes skip all-zero tiles
  uint64_t known_mask = 0;  // PHYSICAL local bits whose value is the same for every non-zero amplitude ...
  uint64_t known_val = 0;   // ... and that value: tiles that contradict it are all zero and are skipped
  int lane_fixed = 0;     // low tile bits that stay on lanes in the load / store rounds (1..3)
  int lite = 1;           // passes of rotations and X / CX only use the lean kernel instantiation
  int jit = 2;            // k > 0: a step-pass STRUCTURE seen k times is compiled (NVRTC) into a straight-line
                          // kernel and cached (qb_jit.cpp); 0 = generic kernels only
  int jit_group = 1;      // specialised kernels: tiles a CTA takes in a row (1, 2, 4).  Consecutive tiles are
                          // neighbours in memory, so a group is prefetched as runs of group x chunk bytes:
                          // DRAM sees 256-512 contiguous bytes per row activation instead of 128
  int jit_minb = 0;       // specialised kernels: CTAs per SM to compile for (0 = automatic)
  int jit_mem = 0;        // specialised kernels: cache policy of the global loads / stores (QBJ_MEM)
  int jit_pf_last = 1;    // prefetch the next group during the last (1) / first (0) tile of the running one
  int tma = 0;            // specialised kernels: tile loads / stores as asynchronous bulk copies (cp.async.bulk)
  int hot_bits = 0;       // planner: max distinct TARGET bits per pass (0 = tile_bits).  With
                          // hot_bits <= tile_bits - warp bits every transpose can stay warp-local.
  int oop = 1;            // passes run OUT OF PLACE (second shard) and write every tile as ONE contiguous block:
                          // the tile's qubits move to the low physical bits, the others keep their order above
                          // (measured: the scattered 128-byte STORES of the in-place pass are what holds it at
                          // 0.65 of the HBM roofline; reads gather, writes stream).  The planner relabels the
                          // remaining ops after every pass; the caller tracks the layout (PlanResult::final_pos).
                          // 1: every qubit is re-sorted by its next use (the next tile is then the low bits plus
                          // the run right above the block: 512-byte chunks inside a few 2 MB pages, and the
                          // layout depends on the op stream only, so the structures of an iterated circuit come
                          // back); 2: only the tile's qubits move.  Single-GPU states with room for a second shard.
  int layout_known = 0;   // (set by the caller per plan) the layout this plan starts from was produced by
                          // out-of-place passes of the same flush (a replan after a global<->local swap): its
                          // first pass need not treat the low bits as passengers
  int defer_tail = 12;    // sharded: a plan that ends stuck on global qubits drops its LAST passes while they carry at most
                          // this many gates each -- those gates wait for the plan after the swap, whose first passes
                          // have room for them (a pass costs one sweep of the shard however few gates it carries)
  int max_passes = 0;     // (set by plan_passes_until_swap) stop after this many passes (0 = no limit)
  int fuse_exchange = 1;  // sharded, out of place: the pass before a global<->local swap stores its tiles straight
                          // into the second shard of the rank that owns them after the swap (XchGeom)
  int pf_lines = 0;       // see DevPass::pf_lines
  int oop_dist = 1;       // sharded states run out of place too (second shard peer-mapped like the first)
  int chunk_lanes = 0;    // out of place: the chunk bits are never warp-id bits (a warp's load covers the whole
                          // chunk), at the price of fewer warp-local transposes
  int oop_low_bits = 5;   // low_bits while passes run out of place: the low bits hold the qubits needed next, so
                          // a longer contiguous chunk costs no extra passes there (measured 30-31 passes either way)
};

// (tile bits, register bits, min CTAs/SM) instantiations of k_fused_pass
struct VariantSpec {
  int T, R, minb;
};
constexpr VariantSpec kFusedVariants[] = {{10, 3, 4}, {10, 4, 4}, {11, 3, 3}, {11, 4, 4}, {11, 5, 6},
                                          {12, 3, 2}, {12, 4, 3}, {12, 5, 3}, {13, 4, 1}, {13, 5, 1}};
bool variant_supported(int T, int R);
bool set_opt(PlanOptions &o, const std::string &name, int64_t v);
int64_t get_opt(const PlanOptions &o, const std::string &name);
// effective (T, R) for a shard with L local bits; T = 0 -> unfused kernels only
void effective_tile(const PlanOptions &o, int L, int &T, int &R);

// An op with PHYSICAL bit positions, as the planner consumes it.
struct PhysOp {
  uint32_t type;
  int target;       // physical bit; may be >= local_bits (global) for G_DIAG only
  uint64_t ctrl;    // physical mask (may include global bits)
  double m[8];
};

struct PassPlan {
  std::vector<uint8_t> blob;     // what the kernel receives: DevPass + gates (lite: DevPass + steps)
  std::vector<DevGate> gates;    // the gate records in execution order (also kept for lite passes)
  uint64_t ntiles = 0;
  int tile_bits = 0, reg_bits = 0;
  int nrounds = 0, ngates = 0;
  uint64_t tile_mask = 0;        // physical bits in the tile
  std::vector<int> op_index;     // indices (into the planner input) of the ops in this pass
  std::vector<uint64_t> round_regmask;  // physical-bit mask of the register bits per round
  std::vector<int> newpos;       // out-of-place pass: physical bit b of the input layout is bit newpos[b] of the
                                 // output layout (local bits only; empty = layout unchanged)
};

struct PlanResult {
  std::vector<PassPlan> passes;
  size_t consumed = 0;           // number of input ops that were scheduled
  std::vector<char> done;        // per input op: scheduled?
  uint64_t known_mask = 0, known_val = 0;  // the support after the scheduled passes (PlanOptions::known_*)
  std::vector<int> final_pos;    // out-of-place passes ran: local physical bit b (layout the plan started from)
                                 // ends up at final_pos[b] (empty = layout unchanged)
};

// Plan fused passes for `ops` on a shard with `local_bits` local qubits.  Ops that cannot run
// locally (non-diagonal gate on a global bit) and everything that depends on them are left
// unscheduled: result.consumed < ops.size(), result.done says which.
// gscale (may be null) is folded into the last pass.
// labels (may be null): a layout-independent name for the qubit on each local physical bit (its logical
// bit); out-of-place passes break ties by it, so that the layouts they produce depend on the op stream only.
PlanResult plan_passes(const std::vector<PhysOp> &ops, int local_bits, int rank, const PlanOptions &opt,
                       const double *gscale, const std::vector<int> *labels = nullptr);

// plan_passes for one stretch of a flush: if the plan ends stuck (a global<->local swap follows) and
// option defer_tail is set, the sparse passes at its end are dropped (see PlanOptions::defer_tail).
PlanResult plan_passes_until_swap(const std::vector<PhysOp> &ops, int local_bits, int rank, const PlanOptions &opt,
                                  const std::vector<int> *labels);

std::string describe_plan(const PlanResult &r);

// The per-state op queue with its value-based peephole (host only, device independent):
//   - scalar * I gates (the reference's u1 / z / s / t / rz, SURVEY.md section 0 item 5) fold
//     into the deferred global scalar;
//   - an uncontrolled 1q gate directly following another on the same qubit is merged into it
//     (2x2 product on the host);
//   - a controlled-X directly following the identical controlled-X cancels (cx . cx = I).
// Dense blocks and Pauli rotations are never merged or cancelled; the identity Pauli string is a
// global factor whatever the peephole setting.
struct OpQueue {
  int n = 0;
  bool peephole = true;
  bool use_rot = true;
  std::vector<HostOp> ops;
  std::vector<int> last_op;      // per logical bit: last live op touching it, or -1
  double gscale[2] = {1.0, 0.0};
  uint64_t submitted = 0, folded = 0;

  void reset(int nqubits, bool peep, bool rot = true);
  void clear();
  bool empty() const;            // nothing to execute (no live ops, gscale == 1)
  void mul_gscale(double re, double im);
  void push_1q(int target_bit, uint64_t ctrl_mask, const double m[8]);
  void push_kq(const int *bits, int k, const double *m, uint64_t ctrl_mask);
  void push_pauli(uint64_t xmask, uint64_t zmask, double c, double s);  // logical masks, c = cos(theta/2), s = sin
};

// ------------------------------------------------------------------ multi-GPU host logic
// Global<->local qubit swap (SURVEY.md 8e).  The k global physical bits that pending gates
// target trade places with k local bits in ONE all-to-all step: rank r keeps the elements whose
// swapped local bits already equal its own value of the swapped rank bits, and trades every
// other group of 2^(L-k) elements with exactly one peer.
struct SwapPair {
  int gbit, lbit;   // physical bit positions (gbit >= L > lbit)
};
struct SwapStep {
  int peer;            // the rank I trade with
  uint32_t my_sel;     // value of the k swapped local bits selecting MY elements that go to `peer`
  uint32_t peer_sel;   // ... and the peer's elements that come to me (bit i <-> pairs[i])
};
// Which global bits must become local for `pending` (op pointers in program order), and which
// local bits they evict.  any_local = false: the TOP k local bits (contiguous blocks: what a
// plain send/recv needs).  any_local = true: Belady -- the local bits (>= 5, so that warps still
// see 512 contiguous bytes) whose qubits are needed furthest in the future (peer-memory kernel).
// future (may be null): the ops expected AFTER `pending` (an iterated circuit: the same stream again);
// only consulted for the next use of qubits that `pending` never touches again.
std::vector<SwapPair> choose_swaps(int n, int L, const std::vector<int> &perm,
                                   const std::vector<const HostOp *> &pending, bool any_local,
                                   const std::vector<const HostOp *> *future = nullptr);
// the pairwise exchanges rank `rank` performs, XOR-ordered so all ranks' steps match up
std::vector<SwapStep> swap_schedule(int rank, int L, const std::vector<SwapPair> &pairs);
void apply_swaps_to_perm(std::vector<int> &perm, const std::vector<SwapPair> &pairs);
// scatter the k-bit selector into the local-bit positions of `pairs`
uint64_t place_sel(uint32_t sel, const std::vector<SwapPair> &pairs);
// Can the stores of out-of-place pass `last` (the last pass of a plan; layout after it = the one
// `sw` was chosen on) carry the swap `sw`?  Any victim but bit 0 will do (the destination is worked
// out store by store; 32-byte stores of register pairs must stay whole) as long as the pair count
// fits XchGeom.  On success fills everything of *out except the peer pointers (the caller knows
// where every rank's second shard is mapped).
bool fused_exchange_geometry(const DevPass &last, int L, int rank, int nranks, const std::vector<SwapPair> &sw, XchGeom *out);

// classification of a caller-supplied 2x2 (value-based)
struct Classified {
  uint32_t type;
  double m[8];        // matrix to execute
  double phase[2];    // common phase pulled out (multiply into the deferred scalar); (1,0) if none
  bool is_scalar;     // m == phase * I
};
Classified classify_2x2(const double m[8], bool allow_phase_pull, bool allow_scale = true);

}  // namespace qb
