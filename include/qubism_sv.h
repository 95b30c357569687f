/* qubism_sv.h -- C ABI of the B200-native state-vector backend for qubism.
 *
 * This is the drop-in boundary for the one hot path of qubitrot/qubism: applying
 * single-qubit / controlled / multi-qubit gate matrices to the 2^n Complex-Double
 * amplitude vector, plus the measurement reduction and collapse.  The reference has no
 * FFI of its own (SURVEY.md 8b); the seam is the Haskell module API of
 *     src/Qubism/StateVec.hs:14-25   and   src/Qubism/QGate.hs:14-31,
 * and each entry point below names the reference definition it replaces.  The Haskell
 * side binds these with `foreign import ccall` (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *   - qb_c64 is layout-compatible with Haskell `Storable (Complex Double)` / C99
 *     `double _Complex`: (re, im).
 *   - Qubit indices are REFERENCE indices: qubit 0 is the MOST significant bit of the
 *     amplitude index (StateVec.hs:65-67); qubit i is bit n-1-i.
 *   - 2x2 matrices are row-major [a, b, c, d] exactly as `(2><2) [a,b,c,d]`
 *     (QGate.hs:91-118); 2^k x 2^k blocks are row-major with qs[0] the most significant
 *     index bit (the order `kronecker a b` produces, QGate.hs:142-144).
 *   - Matrices need NOT be unitary and states need NOT be normalised: the reference's
 *     `unitary theta phi lambda` is not unitary in general (SURVEY.md section 0, item 5).
 *   - The device state is uniquely owned and mutated in place; the pure `(#>)` of the
 *     reference (QGate.hs:78-80) is qb_state_clone + an in-place apply.
 *   - Gate calls only ENQUEUE; the library fuses queued gates into few passes over HBM and
 *     runs them at qb_flush or at the first call that observes the state.
 *   - Every function returns QB_OK (0) or a negative qb_status; it never aborts.  The
 *     message for the last failure on the calling thread is at qb_last_error().
 *   - There is no CPU fallback: without a usable CUDA device qb_init fails with
 *     QB_ERR_CUDA.
 */
#ifndef QUBISM_SV_H
#define QUBISM_SV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { double re, im; } qb_c64;
typedef struct qb_ctx qb_ctx;     /* device, stream, scratch, (optional) NCCL communicator */
typedef struct qb_state qb_state; /* n, device amplitudes (a shard when distributed), bit map,
                                     op queue, deferred scalar */

typedef enum {
  QB_OK = 0,
  QB_ERR_ARG = -1,      /* bad qubit index / size / null pointer (Haskell: `finite` error) */
  QB_ERR_OOM = -2,      /* device or host allocation failed */
  QB_ERR_CUDA = -3,     /* CUDA runtime failure, or no device */
  QB_ERR_NCCL = -4,     /* NCCL failure / library not loadable */
  QB_ERR_UNSUPPORTED = -5,
  QB_ERR_STATE = -6     /* operands on different contexts / sizes (hmatrix shape error) */
} qb_status;

/* ---- context ------------------------------------------------------------------------- */
/* One context per process and GPU.  device = CUDA ordinal. */
int qb_init(int device, qb_ctx **out);
/* Distributed context: one process per GPU, rank r of nranks (a power of two) owns the
 * amplitudes whose top log2(nranks) physical index bits equal r (SURVEY.md 8e).  `nccl_id`
 * is the 128-byte ncclUniqueId produced by qb_dist_unique_id on rank 0 and broadcast by the
 * caller (torch.distributed, MPI, a file ...). */
int qb_dist_unique_id(void *id128);
int qb_init_dist(int device, int rank, int nranks, const void *nccl_id, qb_ctx **out);
/* Rank group inside ONE process (no NCCL): out[r] becomes rank r of nranks (a power of two) on
 * CUDA device devices[r].  Distinct devices = P GPUs driven from one process (peer access is
 * enabled; global<->local swaps run over NVLink through the peers' shard pointers); the SAME
 * device repeated = P virtual ranks on one GPU, which is how the sharded path -- swap selection,
 * fused passes with rank-bit predicates, the pairwise swap kernel -- is parity-tested for
 * P = 2 / 4 / 8 on a single-GPU box.  Collective calls (everything that touches a state) must be
 * issued for every rank, each rank from its own host thread. */
int qb_init_group(const int *devices, int nranks, qb_ctx **out);
/* Frees every device resource of the context.  States that are still alive turn invalid (their
 * calls return QB_ERR_STATE); their handles may be freed afterwards. */
int qb_shutdown(qb_ctx *ctx);
int qb_ctx_rank(const qb_ctx *ctx);
int qb_ctx_nranks(const qb_ctx *ctx);
/* Barrier over all ranks of a distributed context (no-op on a single-GPU one). */
int qb_barrier(qb_ctx *ctx);
const char *qb_last_error(void);
/* Library build identification ("qubism_sv <version> sm_100a ..."). */
const char *qb_version(void);

/* One primitive op of a batch (qb_submit, qb_state_apply_pure). */
typedef struct {
  int32_t kind;      /* 0 = (controlled) 1q gate, 1 = cnot */
  int32_t target;
  int32_t nctrl;
  int32_t ctrl[4];
  int32_t _pad;
  qb_c64 m[4];
} qb_op;

/* ---- state creation / lifetime ------------------------------------------------------- */
/* mkStateVec / mkStateVec' (StateVec.hs:78-85): basis != 0 -> |0...0>;
 * zero (StateVec.hs:52): basis == 0 -> all-zero vector. */
int qb_state_create(qb_ctx *ctx, int nqubits, int basis, qb_state **out);
/* LA.fromList (StateVec.hs:89, test generators StateVecSpec.hs:26-28): upload 2^n host
 * amplitudes.  In a distributed context every rank passes its own shard
 * (2^n / nranks amplitudes, the ones it owns). */
int qb_state_from_host(qb_ctx *ctx, int nqubits, const qb_c64 *amps, qb_state **out);
/* Value semantics of the pure (#>) (QGate.hs:78-80; the interpreter builds sv' = g #> sv once per
 * primitive op and writes sv' back, QASM/Simulation.hs:94-122).  LAZY: the clone is a second
 * handle on the same device shard -- no flush, no copy, no allocation -- and gates queued on the
 * source stay queued for both.  Gates applied to either handle extend a shared log; the ops
 * between two observations fuse exactly as for in-place calls, however they were sliced into
 * handles.  Data is copied only when a handle is observed (or changed in place) while another
 * live handle still denotes an OLDER value of the same shard, and then the copy rides on the
 * first fused pass (it reads the old shard and writes the new one).  Option "linear" = 1 declares
 * that values are used linearly (the interpreter's pattern): the older handles are then CONSUMED
 * instead -- any later call on them fails with QB_ERR_STATE, nothing is ever copied. */
int qb_state_clone(qb_state *src, qb_state **out);
/* g #> sv in one crossing: *out = a new state holding `ops` applied to src's value (clone +
 * qb_submit); src stays valid. */
int qb_state_apply_pure(qb_state *src, const qb_op *ops, int64_t nops, qb_state **out);
/* ForeignPtr finalizer; callable from any thread, at any time, also after qb_shutdown.  Never a
 * collective: on a sharded context the shard is only marked released and is retired (reused or
 * freed) at a later collective call once every rank has released it. */
void qb_state_free(qb_state *s);
/* dimension (StateVec.hs:74-75). */
int qb_state_nqubits(const qb_state *s);
/* Number of amplitudes held by this rank (2^n on a single GPU). */
uint64_t qb_state_local_len(const qb_state *s);
/* Show / :dump / parity (StateVec.hs:60-68): copy amplitudes [first, first+count) of the
 * LOGICAL index space to the host.  Forces a flush.  Distributed: a collective -- every
 * rank calls it with the same range and receives the same data. */
int qb_state_read(qb_state *s, uint64_t first, uint64_t count, qb_c64 *out);
/* Copy amplitudes of this rank's shard to the host: bench/e2e only.  Single GPU: the shard is the
 * state, amplitudes in index order (as qb_state_read); sharded: the raw shard in physical order. */
int qb_state_read_local(qb_state *s, uint64_t first, uint64_t count, qb_c64 *out);
/* Overwrite amplitudes [first, first+count) of this rank's shard from a host buffer (pinned
 * memory makes the copy asynchronous to the host).  An upload STARTS at first = 0: queued gates,
 * the deferred scalar and the qubit layout of the old contents are dropped.  A call with
 * first > 0 continues it: the amplitudes it does not touch keep their meaning (anything pending
 * on them is applied first; QB_ERR_STATE if the layout is no longer the identity).  The upload
 * counterpart of qb_state_read_local. */
int qb_state_write_local(qb_state *s, uint64_t first, uint64_t count, const qb_c64 *amps);

/* ---- gates (enqueue) ------------------------------------------------------------------ */
/* onJust q m #> v   (QGate.hs:148-154, 78-80) */
int qb_apply_1q(qb_state *s, int q, const qb_c64 m[4]);
/* onRange qlo qhi m #> v / onEvery m #> v   (QGate.hs:158-165) */
int qb_apply_1q_range(qb_state *s, int qlo, int qhi, const qb_c64 m[4]);
/* controlled c1 (controlled c2 (... (onJust t m))) #> v   (QGate.hs:125-132) */
int qb_apply_ctrl_1q(qb_state *s, const int *ctrls, int nctrl, int t, const qb_c64 m[4]);
/* cnot c t #> v   (QGate.hs:121-122) */
int qb_apply_cnot(qb_state *s, int c, int t);
/* kronecker / (<>) blocks (QGate.hs:58-59, 142-144): dense 2^k x 2^k block on qubits
 * qs[0..k), optionally under nctrl controls.  k <= QB_MAX_KQ. */
#define QB_MAX_KQ 5
int qb_apply_kq(qb_state *s, const int *qs, int k, const qb_c64 *m, const int *ctrls, int nctrl);

/* Batch submission (SURVEY.md 8f rank 1): one FFI crossing for a whole op list. */
int qb_submit(qb_state *s, const qb_op *ops, int64_t nops);

/* Plan and run every queued gate.  Returns after the work is ENQUEUED on the stream;
 * use qb_sync to wait for completion. */
int qb_flush(qb_state *s);
int qb_sync(qb_ctx *ctx);

/* ---- measurement ---------------------------------------------------------------------- */
/* Raw reduction behind pOne (StateVec.hs:124-126): s0 / s1 = sum |z_k|^2 over the
 * amplitudes whose qubit-q bit is 0 / 1.  The reference's decision value is sqrt(s1).
 * Deterministic (fixed-order two-stage reduction); distributed: all-reduced. */
int qb_sumsq(qb_state *s, int q, double *s0, double *s1);
/* collapse q bit (StateVec.hs:104-114): zero the rejected half, divide the kept half by
 * its 2-norm.  A zero-weight outcome yields an all-NaN state, as in the reference. */
int qb_collapse(qb_state *s, int q, int bit);
/* measureQubit q (StateVec.hs:118-129) with the uniform draw r supplied by the caller
 * (the RNG stays in Haskell): *bit = 1 iff r < sqrt(s1); the state collapses to *bit.
 * *pone receives sqrt(s1) (0 where the reference has NaN; both decide Zero). */
int qb_measure_qubit(qb_state *s, int q, double r, int *bit, double *pone);
/* measure (StateVec.hs:133-137): measureQubit 0..n-1 in order with draws rs[0..n). */
int qb_measure_all(qb_state *s, const double *rs, int *bits);

/* ---- vector space / Hilbert space (StateVec.hs:51-58, 91-100; Algebra.hs:17-36) ------- */
int qb_scale(qb_state *s, qb_c64 z);                          /* z .: v                   */
int qb_axpy(qb_state *y, qb_c64 z, qb_state *x);              /* y <- y +: (z .: x)       */
int qb_neg(qb_state *s);                                      /* neg v                    */
/* the same two with the scalar as (re, im) doubles: Haskell's FFI cannot pass structs by value */
int qb_scale_ri(qb_state *s, double re, double im);
int qb_axpy_ri(qb_state *y, double re, double im, qb_state *x);
int qb_dotc(qb_state *a, qb_state *b, qb_c64 *out);           /* a <.> b, conj on a       */
int qb_norm2(qb_state *s, double *out);                       /* LA.norm_2 (NOT squared)  */
int qb_normalize(qb_state *s);                                /* normalize                */
int qb_tensor(qb_state *a, qb_state *b, qb_state **out);      /* a `tensor` b             */

/* ---- observables ----------------------------------------------------------------------- */
/* Expectation values of Pauli strings: out[t] = realPart (sv <.> (P_t #> sv)), where P_t is the
 * product of pauliX / pauliY / pauliZ (QGate.hs:90-108) on the qubits named by term t: bit q of
 * xmask[t] / zmask[t] is REFERENCE qubit q; X = x only, Z = z only, Y = both, I = neither.
 * Not normalised (the reference's <.> is not).  Observes the state (flushes it) and leaves its
 * value unchanged.  Deterministic.  Distributed: a collective; every rank passes the same terms
 * and receives all nterms values.
 * Cost: one read-only sweep of the state per distinct X mask and 64 terms (counted in
 * qb_stats.reduce_launches, two launches per sweep); a term whose X mask flips a qubit of known value
 * (|0...0>, after a collapse) is exactly 0 and costs nothing.  Sharded: X / Y on global qubits first
 * swap those qubits into the shard (QB_ERR_UNSUPPORTED if a string has X / Y on more qubits than a
 * shard holds).  QB_ERR_ARG: a null pointer with nterms > 0, nterms < 0, a mask bit at or above n. */
int qb_expect_pauli(qb_state *s, const uint64_t *xmask, const uint64_t *zmask, int64_t nterms, double *out);

/* ---- Pauli rotations ------------------------------------------------------------------- */
/* s <- R_{P_t}(theta[t]) ... R_{P_0}(theta[0]) s, with R_P(theta) = exp(-i theta/2 P)
 * = cos(theta/2) I - i sin(theta/2) P and P_t named by xmask[t] / zmask[t] exactly as in
 * qb_expect_pauli (bit q = REFERENCE qubit q; X = x only, Z = z only, Y = both; pauliY as in
 * QGate.hs:90-108).  Applied in array order.  Enqueues only, like every gate call; the identity
 * string is a global factor exp(-i theta/2) and launches nothing.
 * Cost: one read + write sweep of the state (counted in qb_stats.simple_launches) per run of
 * consecutive rotations whose X qubits fit one tile of QB_PAULI_ROT_MAX_X qubits together, at most 64
 * rotations each; Z-only rotations fit any run.  A run ends the fused pass before it.  Sharded: X / Y on
 * global qubits first swap those qubits into the shard.
 * Checked before anything is queued (a rejected call leaves the state and its queue untouched):
 * QB_ERR_ARG: a null pointer with nrot > 0, nrot < 0, a mask bit at or above n, a non-finite theta.
 * QB_ERR_UNSUPPORTED: a string with X / Y on more than QB_PAULI_ROT_MAX_X qubits, or on more
 * qubits than a shard holds. */
#define QB_PAULI_ROT_MAX_X 12
int qb_apply_pauli_rot(qb_state *s, const uint64_t *xmask, const uint64_t *zmask, const double *theta, int64_t nrot);

/* ---- introspection (tests, bench, profiling) ------------------------------------------- */
typedef struct {
  uint64_t ops_submitted;   /* primitive ops received through the ABI                     */
  uint64_t ops_folded;      /* removed by the host peephole (scalars, cancelling CX pairs,
                               merged 1q products)                                       */
  uint64_t ops_executed;    /* gates that reached a kernel                                */
  uint64_t passes;          /* fused-pass kernel launches (one read+write of the shard)   */
  uint64_t rounds;          /* register-residency rounds inside those passes              */
  uint64_t simple_launches; /* launches of the unfused small-n / dense-k kernels          */
  uint64_t reduce_launches; /* launches of reduction kernels                              */
  uint64_t exchange_bytes;  /* bytes this rank sent in global<->local qubit swaps         */
  uint64_t exchanges;       /* number of such swaps                                       */
  double plan_ms;           /* host time spent planning                                   */
  double fused_ms;          /* device time inside fused-pass kernels (CUDA events on the
                               launching stream), accumulated while option "time_kernels"=1 */
  uint64_t fused_timed;     /* number of fused launches that were timed                    */
  uint64_t tiles;           /* tiles the fused passes visited (all-zero tiles are skipped)  */
  uint64_t jit_compiled;    /* pass structures compiled into specialised kernels (option "jit") */
  uint64_t jit_launches;    /* fused passes that ran as a specialised kernel                 */
  double jit_compile_ms;    /* host time spent in NVRTC + module load                        */
  uint64_t clones;          /* qb_state_clone calls (all lazy)                               */
  uint64_t cow_fused;       /* copy-on-write copies that rode on a fused pass (no extra traffic) */
  uint64_t cow_copies;      /* copy-on-write / fork copies done as a separate device copy     */
  uint64_t exchanges_fused; /* of `exchanges`: swaps carried by the stores of a fused pass (no sweep of
                               their own: the tiles go straight to their next owner over NVLink) */
} qb_stats;
int qb_get_stats(const qb_ctx *ctx, qb_stats *out);
int qb_reset_stats(qb_ctx *ctx);
/* Raw CUDA stream of the context (cudaStream_t as void*), for event timing by callers. */
void *qb_ctx_stream(qb_ctx *ctx);
/* Tuning knobs: "tile_bits", "reg_bits", "low_bits", "lane_fixed", "max_rounds",
 * "max_pass_gates", "peephole", "fuse" (0 = one pass per op), "rot" (rotations as shears),
 * "lite" (step-packed passes), "skip_dead" (skip all-zero tiles using the tracked support),
 * "time_kernels" (bracket every fused launch with CUDA events), "jit" (k > 0: a pass structure
 * seen k times is compiled with NVRTC into a straight-line kernel -- structure as literals, gate
 * coefficients still kernel parameters -- and cached; k = 1 compiles at first sight in the
 * calling thread, k >= 2 in background threads while the generic kernel keeps running;
 * 0 = generic kernels only), "linear" (see qb_state_clone), "pool" (spare shards kept for reuse),
 * "oop" (1, default: fused passes run OUT OF PLACE into a second shard of the same size, every tile
 * stored as one contiguous block and the qubit layout re-sorted by next use after every pass --
 * invisible through this ABI, which always speaks the reference's qubit numbers and index order;
 * 2: only the tile's qubits move; 0: in place, half the memory), "oop_low_bits", "oop_dist" (sharded
 * states run out of place too), "chunk_lanes", "tma" (tile loads as bulk copies), "l2_prefetch", "fuse_exchange" (1, default: on
 * sharded out-of-place states the pass before a global<->local swap stores every tile straight
 * into the second shard of the rank that owns it after the swap; 0: store locally, then exchange),
 * "defer_tail" (12: the last passes of a plan that is stuck on global qubits are held back while they
 * carry at most this many gates each; their gates run after the swap; 0: off).
 * A state that cannot get its second shard (36 qubits on 8 GPUs) stays in place.  Returns
 * QB_ERR_ARG for unknown names / bad values. */
int qb_set_option(qb_ctx *ctx, const char *name, int64_t value);
int64_t qb_get_option(const qb_ctx *ctx, const char *name);
/* Host-only planner entry point (no device needed): plan `nops` ops for an n-qubit local
 * shard and write a textual plan ("pass tile=.. round regs=.. gates=..") into buf.
 * Returns the number of bytes the full plan needs (snprintf-style) or a negative status. */
int64_t qb_plan_describe(int nlocal, const qb_op *ops, int64_t nops, const char *options,
                         char *buf, int64_t buflen);

/* Block until no background compilation of a specialised kernel is pending (option "jit" >= 2
 * compiles on worker threads while the generic kernels keep running).  Benchmarks call it after
 * their warm-up; nothing else needs it. */
int qb_jit_sync(qb_ctx *ctx);
/* Which NVRTC compiles the specialised kernels in this process and the widest global access it
 * emits ("nvrtc 12.9, 256-bit ..."; a process that loaded an older libnvrtc first gets 128-bit). */
const char *qb_jit_toolchain(void);
/* Host-only check of the specialised-kernel toolchain (no device needed): compile `src` (CUDA C++)
 * with NVRTC for sm_100a; *cubin_bytes = size of the resulting cubin.  QB_ERR_UNSUPPORTED if
 * libnvrtc cannot be loaded, QB_ERR_CUDA if the compilation fails (log in qb_last_error). */
int qb_jit_compile_check(const char *src, int64_t *cubin_bytes);

#ifdef __cplusplus
}
#endif
#endif /* QUBISM_SV_H */
