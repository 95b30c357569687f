// C-ABI layer of the qubism state-vector backend (include/qubism_sv.h): contexts, device
// states, the deferred op queue, flush = plan + launch, measurement, vector-space ops.
// No torch types, no CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "qb_dist.h"
#include "qb_internal.h"
#include "qb_jit.h"
#include "qb_kernels.h"

using namespace qb;

// ------------------------------------------------------------------------- errors
static thread_local std::string g_last_error;

static int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define QB_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess)                                                                \
      return fail(e__ == cudaErrorMemoryAllocation ? QB_ERR_OOM : QB_ERR_CUDA, "%s: %s",  \
                  #expr, cudaGetErrorString(e__));                                         \
  } while (0)

#define QB_TRY(expr)         \
  do {                       \
    int rc__ = (expr);       \
    if (rc__ != QB_OK) return rc__; \
  } while (0)

// ------------------------------------------------------------------------- objects
struct Buffer;

struct qb_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  int rank = 0, nranks = 1, pbits = 0;
  double *red_partials = nullptr;  // device, kExpMaxTerms per block of the largest reduction grid
  double *red_out = nullptr;       // device, kExpMaxTerms doubles
  double *red_host = nullptr;      // pinned, kExpMaxTerms doubles
  uint64_t jit_base_compiled = 0, jit_base_launches = 0;  // qb_reset_stats baselines of the process-wide counters
  double jit_base_ms = 0.0;
  int *kq_bits_dev = nullptr;      // 2 * QB_MAX_KQ ints
  double2 *kq_mat_dev = nullptr;   // 4^QB_MAX_KQ
  double2 **peer_tab_dev = nullptr;  // nranks device pointers (sharded tensor)
  PlanOptions opt;
  int linear = 0;                  // option "linear": 1 = a pure application CONSUMES the older handles of its
                                   // lineage (they turn stale and fail loudly) instead of copying on write
  int pool_max = 2;                // option "pool": spare shards kept for the next clone / copy-on-write / second shard
  qb_stats stats{};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed;  // pending (start, stop) pairs
  std::vector<cudaEvent_t> event_pool;
  std::recursive_mutex mu;
  DistState *dist = nullptr;
  // device shards: in use (creation order), spare (registered with the peers, ready for reuse), and
  // released by their last handle but not yet agreed dead by every rank (sharded contexts: a
  // finalizer may run at a different time on every rank, so nothing collective happens in it)
  std::vector<Buffer *> in_use, pool, graveyard;
  uint64_t next_buffer_id = 0;
  long handles = 0;                // live qb_state handles (a finalizer may run after qb_shutdown)
  bool closed = false;
};

// One entry of a lineage log: what a handle did after the position its buffer stands at.
enum LogKind : int { LOG_1Q = 0, LOG_KQ = 2, LOG_SCALE = 3, LOG_COLLAPSE = 4, LOG_PAULI = 5 };
struct LogOp {
  int kind = LOG_1Q;
  int target = -1;    // 1Q: logical target bit.  COLLAPSE: the logical bit
  uint64_t ctrl = 0;  // 1Q / KQ: logical control mask.  COLLAPSE: the outcome (0 / 1).  PAULI: logical X mask
  uint64_t pz = 0;    // PAULI: logical Z mask
  double m[8] = {0};  // 1Q: the matrix.  SCALE: (re, im).  COLLAPSE: m[0] = weight of the outcome.
                      // PAULI: (cos(theta/2), sin(theta/2))
  int k = 0;
  int kq_bits[QB_MAX_KQ] = {0};
  std::shared_ptr<const std::vector<double>> kq_m;
};

// A device shard plus everything that describes what its amplitudes MEAN, shared by the handles
// of one lineage.  The device data stands at log position `mat`; a handle at position p denotes
// the state "data advanced by log[mat .. p)".  Value semantics of the reference's pure (#>)
// (QGate.hs:78-80; the interpreter builds sv' = g #> sv once per primitive op,
// QASM/Simulation.hs:94-122) therefore cost nothing per op: a clone is a new handle at the same
// position, an apply appends to the log, and the ops between two observations still fuse.
struct Buffer {
  qb_ctx *ctx = nullptr;
  int n = 0, L = 0;
  uint64_t id = 0;
  double2 *amps = nullptr;
  double2 *alt = nullptr;        // second shard of the same size (allocated on first use): out-of-place passes
                                 // read `amps`, write `alt`, and the two trade places (option "oop")
  std::vector<double2 *> peers;  // distributed: every rank's shard (IPC / same process); empty: NCCL swaps
  std::vector<double2 *> peers_alt;  // ... and every rank's SECOND shard (the two tables trade places with the shards)
  bool alt_zero = false;         // the second shard holds only zeros (a rank whose shard is all zero skips its
                                 // passes; the out-of-place ones must still trade two all-zero shards)
  const double2 *cow_src = nullptr;  // copy-on-write in progress: the first full pass reads its tiles here
  std::vector<int> perm;  // logical bit -> physical bit (bits >= L are rank bits)
  // SUPPORT of the amplitudes on the device: every non-zero amplitude has
  // (logical index & zmask) == zval.  |0...0> knows every bit, a collapse learns one, a
  // non-diagonal gate forgets its target.  Measurement works on the live sub-cube only.
  uint64_t zmask = 0, zval = 0;
  // deferred scalar that no pass has taken yet (collapse normalisation, qb_scale on an idle state):
  // true amplitudes = pscale * device amplitudes.  Reductions apply it arithmetically; everything
  // that exposes raw amplitudes forces it first (force_scale).
  double pscale[2] = {1.0, 0.0};
  // real factor the structure-specialised passes of the running flush left out of the device
  // amplitudes (their rotations defer a cosine each, qb_jit.cpp): taken by the flush's last
  // pass, or folded into pscale when the flush ends
  double jit_left = 1.0;
  bool all_finite = false;  // no NaN / inf can be in the amplitudes (created here, only finite gates since)
  std::vector<LogOp> log;   // positions log_base .. log_base + log.size()
  size_t log_base = 0, mat = 0;
  std::vector<qb_state *> handles;
  bool broken = false;      // a flush failed half way: the data matches no position any more
  std::string broken_why;
  bool released = false;    // in the graveyard
  bool ever_shared = false; // a second handle has existed on this shard (clone): liveness questions need the ranks' agreement
  OpQueue q;                // scratch of exec_log

  size_t tip() const { return log_base + log.size(); }
};

struct qb_state {
  qb_ctx *ctx = nullptr;
  Buffer *b = nullptr;
  size_t pos = 0;
  int n = 0;
  bool stale = false;  // option "linear": a later pure application consumed this value
};

extern "C" {
static int localise_x(Buffer *b, uint64_t lx);  // (with the Pauli expectation values, below)
}

namespace {

struct Guard {
  std::lock_guard<std::recursive_mutex> lk;
  explicit Guard(qb_ctx *c) : lk(c->mu) { cudaSetDevice(c->device); }
};

int init_common(qb_ctx *c) {
  QB_CUDA(cudaSetDevice(c->device));
  cudaDeviceProp prop;
  QB_CUDA(cudaGetDeviceProperties(&prop, c->device));
  c->sm_count = prop.multiProcessorCount;
  QB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  const int maxblocks = c->sm_count * 8 + 8;
  QB_CUDA(cudaMalloc(&c->red_partials, sizeof(double) * kExpMaxTerms * maxblocks));
  QB_CUDA(cudaMalloc(&c->red_out, sizeof(double) * kExpMaxTerms));
  QB_CUDA(cudaMallocHost(&c->red_host, sizeof(double) * kExpMaxTerms));
  QB_CUDA(cudaMalloc(&c->kq_bits_dev, sizeof(int) * 2 * QB_MAX_KQ));
  QB_CUDA(cudaMalloc(&c->kq_mat_dev, sizeof(double2) << (2 * QB_MAX_KQ)));
  for (const char *name : {"tile_bits", "reg_bits", "low_bits", "max_rounds", "peephole", "fuse", "max_pass_gates", "l2_prefetch", "avoid_regswap", "hot_bits", "rot", "lite", "dbg_skip", "lane_fixed", "skip_dead", "support", "jit", "jit_group", "jit_pf_last", "jit_minb", "jit_mem", "tma", "oop", "oop_low_bits", "chunk_lanes", "oop_dist", "pf_lines", "fuse_exchange", "defer_tail"}) {
    std::string env = "QB_";
    for (const char *p = name; *p; ++p) env.push_back((char)toupper(*p));
    const char *v = getenv(env.c_str());
    if (v && *v) set_opt(c->opt, name, strtoll(v, nullptr, 10));
  }
  if (const char *v = getenv("QB_LINEAR")) c->linear = atoi(v) ? 1 : 0;
  if (const char *v = getenv("QB_POOL")) c->pool_max = std::max(0, atoi(v));
  return QB_OK;
}

// ---- device shards: allocation, the spare pool, release without collectives --------------------
void free_buffer_memory(Buffer *b) {
  if (b->amps) cudaFree(b->amps);
  if (b->alt) cudaFree(b->alt);
  b->amps = b->alt = nullptr;
}

// the second shard of an out-of-place pass; false (and no error) if the memory is not there -- the
// caller then stays in place
bool ensure_alt(Buffer *b) {
  if (b->alt) return true;
  qb_ctx *c = b->ctx;
  if (c->nranks > 1) {
    // sharded: every rank allocates, all agree on the outcome (one rank out of memory keeps every
    // rank in place), the peers map the new shard like the first one.  Collective: every rank runs
    // the same flush.
    bool ok = cudaMalloc(&b->alt, sizeof(double2) << b->L) == cudaSuccess;
    if (!ok) {
      (void)cudaGetLastError();
      b->alt = nullptr;
    }
    double bad = ok ? 0.0 : 1.0;
    if (dist_allreduce_sum(c->dist, &bad, 1, c->stream) != QB_OK) bad = 1.0;
    if (bad == 0.0) {
      ok = cudaMemsetAsync(b->alt, 0, sizeof(double2) << b->L, c->stream) == cudaSuccess;
      if (dist_register(c->dist, b->alt, b->peers_alt, c->stream) != QB_OK) ok = false;
      if (b->peers_alt.size() != b->peers.size()) ok = false;  // (one shard peer-mapped, the other not: stay in place)
      bad = ok ? 0.0 : 1.0;
      if (dist_allreduce_sum(c->dist, &bad, 1, c->stream) != QB_OK) bad = 1.0;
      if (bad != 0.0 && !b->peers_alt.empty()) dist_unregister(c->dist, b->peers_alt, c->stream);
    }
    if (bad != 0.0) {
      if (b->alt) cudaFree(b->alt);
      b->alt = nullptr;
      b->peers_alt.clear();
      return false;
    }
    b->alt_zero = true;
    return true;
  }
  for (size_t i = 0; i < c->pool.size(); ++i)  // a spare shard of the right size is as good as a new one
    if (c->pool[i]->L == b->L && c->pool[i]->peers.empty()) {
      Buffer *p = c->pool[i];
      c->pool.erase(c->pool.begin() + i);
      b->alt = p->amps;
      p->amps = nullptr;
      free_buffer_memory(p);
      delete p;
      return true;
    }
  if (cudaMalloc(&b->alt, sizeof(double2) << b->L) != cudaSuccess) {
    (void)cudaGetLastError();
    b->alt = nullptr;
    return false;
  }
  return true;
}

// Sharded contexts: which released shards are released on EVERY rank?  Handles die in finalizers,
// at a different moment on every rank; a shard exported to the peers can only be reused or freed
// once all of them are done with it.  Collective; called where every rank is anyway (allocation,
// qb_barrier, qb_shutdown): one all-reduce over the first 64 shards in use, in creation order --
// the same list on every rank, because shards are created and retired collectively.
int drain_graveyard(qb_ctx *c) {
  if (c->nranks == 1) {
    for (Buffer *b : c->graveyard) {
      if ((int)c->pool.size() < c->pool_max) {
        c->pool.push_back(b);
      } else {
        free_buffer_memory(b);
        delete b;
      }
    }
    c->graveyard.clear();
    return QB_OK;
  }
  if (c->in_use.empty()) return QB_OK;
  const int w = (int)std::min<size_t>(64, c->in_use.size());
  double v[64];
  for (int i = 0; i < w; ++i) v[i] = c->in_use[i]->released ? 1.0 : 0.0;
  int rc = dist_allreduce_sum(c->dist, v, w, c->stream);
  if (rc != QB_OK) return fail(rc, "shard release agreement failed: %s", dist_last_error());
  std::vector<Buffer *> keep, gone;
  for (int i = 0; i < (int)c->in_use.size(); ++i)
    (i < w && v[i] == (double)c->nranks ? gone : keep).push_back(c->in_use[i]);
  c->in_use.swap(keep);
  bool any_free = false;
  for (Buffer *b : gone) {
    c->graveyard.erase(std::find(c->graveyard.begin(), c->graveyard.end(), b));
    if (b->alt) {  // the second shard is never pooled (same `gone` and same shards on every rank: collective)
      if (!b->peers_alt.empty()) dist_unregister(c->dist, b->peers_alt, c->stream);
      cudaFree(b->alt);
      b->alt = nullptr;
      b->peers_alt.clear();
    }
    if ((int)c->pool.size() < c->pool_max) {
      c->pool.push_back(b);  // stays mapped by the peers: reuse needs no collective
    } else {
      any_free = true;
      if (!b->peers.empty()) dist_unregister(c->dist, b->peers, c->stream);  // collective (same `gone` on every rank)
    }
  }
  if (any_free)
    for (Buffer *b : gone)
      if (std::find(c->pool.begin(), c->pool.end(), b) == c->pool.end()) {
        free_buffer_memory(b);
        delete b;
      }
  return QB_OK;
}

int new_buffer(qb_ctx *ctx, int n, Buffer **out) {
  if (!ctx || !out) return fail(QB_ERR_ARG, "null argument");
  if (ctx->closed) return fail(QB_ERR_STATE, "context was shut down");
  if (n < 1 || n > 62) return fail(QB_ERR_ARG, "nqubits %d out of range", n);
  if (n < ctx->pbits) return fail(QB_ERR_ARG, "nqubits %d smaller than log2(nranks) = %d", n, ctx->pbits);
  const int L = n - ctx->pbits;
  if (L > 58) return fail(QB_ERR_OOM, "2^%d amplitudes per shard do not fit a size_t", L);
  QB_TRY(drain_graveyard(ctx));
  Buffer *b = nullptr;
  for (size_t i = 0; i < ctx->pool.size(); ++i)
    if (ctx->pool[i]->L == L) {
      b = ctx->pool[i];
      ctx->pool.erase(ctx->pool.begin() + i);
      break;
    }
  if (!b) {
    // (the pool holds other sizes: give their memory back first)
    const size_t bytes = sizeof(double2) << L;
    b = new Buffer();
    b->ctx = ctx;
    cudaError_t e = cudaMalloc(&b->amps, bytes);
    if (e != cudaSuccess && !ctx->pool.empty() && ctx->nranks == 1) {
      (void)cudaGetLastError();
      for (Buffer *p : ctx->pool) {
        free_buffer_memory(p);
        delete p;
      }
      ctx->pool.clear();
      e = cudaMalloc(&b->amps, bytes);
    }
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      delete b;
      return fail(e == cudaErrorMemoryAllocation ? QB_ERR_OOM : QB_ERR_CUDA, "cudaMalloc(%zu bytes): %s", bytes,
                  cudaGetErrorString(e));
    }
    b->id = ctx->next_buffer_id++;
    if (ctx->nranks > 1) {  // collective: map every peer's shard for the NVLink swap kernel
      int rc = dist_register(ctx->dist, b->amps, b->peers, ctx->stream);
      if (rc != QB_OK) {
        free_buffer_memory(b);
        delete b;
        return fail(rc, "peer registration failed: %s", dist_last_error());
      }
    }
  }
  b->n = n;
  b->L = L;
  b->cow_src = nullptr;
  b->perm.resize(n);
  for (int i = 0; i < n; ++i) b->perm[i] = i;
  b->zmask = b->zval = 0;
  b->pscale[0] = 1.0;
  b->pscale[1] = 0.0;
  b->jit_left = 1.0;
  b->all_finite = false;
  b->log.clear();
  b->log_base = b->mat = 0;
  b->handles.clear();
  b->broken = false;
  b->released = false;
  b->ever_shared = false;
  ctx->in_use.push_back(b);
  *out = b;
  return QB_OK;
}

// the last handle of a shard went away (possibly inside a finalizer): nothing collective here
void release_buffer(Buffer *b) {
  qb_ctx *c = b->ctx;
  b->log.clear();
  b->released = true;
  if (b->alt && c->nranks == 1) {  // (nothing collective about it) -> the spare pool, if there is room
    if ((int)c->pool.size() + 1 < c->pool_max) {
      Buffer *p = new Buffer();
      p->ctx = c;
      p->L = b->L;
      p->n = b->n;
      p->amps = b->alt;
      c->pool.push_back(p);
    } else {
      cudaFree(b->alt);
    }
    b->alt = nullptr;
  }
  c->graveyard.push_back(b);
  if (c->nranks == 1) {
    c->in_use.erase(std::find(c->in_use.begin(), c->in_use.end(), b));
    drain_graveyard(c);
  }
}

void attach(qb_state *h, Buffer *b, size_t pos) {
  h->b = b;
  h->pos = pos;
  b->handles.push_back(h);
}

void detach(qb_state *h) {
  Buffer *b = h->b;
  if (!b) return;
  b->handles.erase(std::find(b->handles.begin(), b->handles.end(), h));
  h->b = nullptr;
  if (b->handles.empty()) release_buffer(b);
}

int new_handle(qb_ctx *ctx, Buffer *b, size_t pos, qb_state **out) {
  qb_state *h = new qb_state();
  h->ctx = ctx;
  h->n = b->n;
  attach(h, b, pos);
  ++ctx->handles;
  *out = h;
  return QB_OK;
}

// Sharded contexts: handles die in finalizers, at a different moment on every rank, but whether a
// shard has to be copied (a collective allocation) must be decided alike everywhere: "does ANY
// rank still hold such a handle?".  Only asked for shards that were ever cloned.
int agree_any(qb_ctx *c, const Buffer *b, bool *flag) {
  if (c->nranks == 1 || !b->ever_shared) return QB_OK;
  double v = *flag ? 1.0 : 0.0;
  int rc = dist_allreduce_sum(c->dist, &v, 1, c->stream);
  if (rc != QB_OK) return fail(rc, "handle agreement failed: %s", dist_last_error());
  *flag = v != 0.0;
  return QB_OK;
}

int check_state(const qb_state *s) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  if (s->ctx->closed) return fail(QB_ERR_STATE, "the context of this state was shut down");
  if (s->stale || !s->b)
    return fail(QB_ERR_STATE, "stale handle: a later pure application consumed this value (option \"linear\" = 1)");
  if (s->b->broken) return fail(QB_ERR_STATE, "state lost by an earlier failure: %s", s->b->broken_why.c_str());
  return QB_OK;
}

inline int logical_bit(const qb_state *s, int q) { return s->n - 1 - q; }

int check_qubit(const qb_state *s, int q) {
  if (q < 0 || q >= s->n) return fail(QB_ERR_ARG, "qubit index %d out of range for %d qubits", q, s->n);
  return QB_OK;
}

uint64_t phys_mask(const Buffer *s, uint64_t logical_mask) {
  uint64_t m = 0;
  for (uint64_t b = logical_mask; b; b &= b - 1) m |= 1ull << s->perm[__builtin_ctzll(b)];
  return m;
}

int get_event(qb_ctx *c, cudaEvent_t *out) {
  if (!c->event_pool.empty()) {
    *out = c->event_pool.back();
    c->event_pool.pop_back();
    return QB_OK;
  }
  QB_CUDA(cudaEventCreate(out));
  return QB_OK;
}

// fold finished (start, stop) pairs into stats.fused_ms; waits for the stream
int resolve_timed(qb_ctx *c) {
  if (c->timed.empty()) return QB_OK;
  QB_CUDA(cudaStreamSynchronize(c->stream));
  FILE *plog = nullptr;  // developer switch: one line per fused pass (its CUDA-event time) appended to a file
  if (const char *path = getenv("QB_PASS_LOG")) plog = fopen(path, "a");
  for (auto &pr : c->timed) {
    float ms = 0.f;
    QB_CUDA(cudaEventElapsedTime(&ms, pr.first, pr.second));
    if (plog) fprintf(plog, "%.4f\n", ms);
    c->stats.fused_ms += ms;
    c->stats.fused_timed++;
    c->event_pool.push_back(pr.first);
    c->event_pool.push_back(pr.second);
  }
  if (plog) fclose(plog);
  c->timed.clear();
  return QB_OK;
}

// a copy-on-write whose copy has not happened yet (no full pass has run): do it now
int ensure_inplace(Buffer *s) {
  if (!s->cow_src) return QB_OK;
  QB_CUDA(cudaMemcpyAsync(s->amps, s->cow_src, sizeof(double2) << s->L, cudaMemcpyDeviceToDevice, s->ctx->stream));
  s->cow_src = nullptr;
  s->ctx->stats.cow_copies++;
  return QB_OK;
}

// run one op with the unfused kernels
int run_simple(Buffer *s, const HostOp &op) {
  qb_ctx *c = s->ctx;
  QB_TRY(ensure_inplace(s));
  const uint64_t rank_bits = uint64_t(c->rank) << s->L;
  const uint64_t cmask = phys_mask(s, op.ctrl);
  if (op.kind == 2) {
    int sorted[QB_MAX_KQ] = {0}, order[QB_MAX_KQ] = {0};
    if (op.k < 1 || op.k > QB_MAX_KQ) return fail(QB_ERR_ARG, "bad k");
    for (int j = 0; j < op.k; ++j) {
      const int pb = s->perm[op.kq_bits[op.k - 1 - j]];  // matrix index bit j (LSB first)
      if (pb >= s->L) return fail(QB_ERR_UNSUPPORTED, "internal: dense k-qubit block on a global qubit");
      order[j] = pb;
      sorted[j] = pb;
    }
    std::sort(sorted, sorted + op.k);
    int host[2 * QB_MAX_KQ];
    memcpy(host, sorted, sizeof(sorted));
    memcpy(host + QB_MAX_KQ, order, sizeof(order));
    QB_CUDA(cudaMemcpyAsync(c->kq_bits_dev, host, sizeof(host), cudaMemcpyHostToDevice, c->stream));
    QB_CUDA(cudaMemcpyAsync(c->kq_mat_dev, op.kq_m.data(), sizeof(double) * op.kq_m.size(), cudaMemcpyHostToDevice,
                            c->stream));
    QB_CUDA(launch_simple_kq(s->amps, s->L, op.k, c->kq_bits_dev, c->kq_bits_dev + QB_MAX_KQ, c->kq_mat_dev, cmask,
                             rank_bits, c->sm_count, c->stream));
    // the host vectors above are read by the copies asynchronously (pageable memory is staged at
    // call time) -- and the NEXT dense block must not overwrite the device copies early: same stream
    c->stats.simple_launches++;
    c->stats.ops_executed++;
    return QB_OK;
  }
  const int pt = s->perm[op.target];
  if (op.type == G_DIAG) {
    QB_CUDA(launch_simple_diag(s->amps, s->L, 1ull << pt, cmask, rank_bits, &op.m[0], &op.m[6], c->sm_count,
                               c->stream));
  } else {
    if (pt >= s->L) return fail(QB_ERR_UNSUPPORTED, "internal: unfused gate on a global qubit");
    if (s->L < 1) return fail(QB_ERR_UNSUPPORTED, "shard too small");
    QB_CUDA(launch_simple_gate(s->amps, s->L, pt, cmask, rank_bits, op.type, op.m, c->sm_count, c->stream));
  }
  c->stats.simple_launches++;
  c->stats.ops_executed++;
  return QB_OK;
}

int run_gscale_simple(Buffer *s, const double g[2]) {
  qb_ctx *c = s->ctx;
  QB_TRY(ensure_inplace(s));
  QB_CUDA(launch_simple_diag(s->amps, s->L, 0, 0, 0, g, g, c->sm_count, c->stream));
  c->stats.simple_launches++;
  return QB_OK;
}

// Make the global targets of `pending` (live ops, program order) local: in a distributed context
// one multi-bit swap brings them into the shard.
int make_local(Buffer *s, const std::vector<const HostOp *> &pending) {
  qb_ctx *c = s->ctx;
  if (c->nranks == 1) return fail(QB_ERR_UNSUPPORTED, "internal: planner stuck on a single GPU");
  QB_TRY(ensure_inplace(s));
  // what comes after `pending`: assume the flush's op stream again (an iterated circuit).  Only
  // consulted to order the qubits this flush never touches again, which would otherwise tie: the
  // layout then settles into a short cycle (period 2 at 2 GPUs, 3 at 4 on the benchmark circuit)
  // and the specialised kernels find their structures again
  std::vector<const HostOp *> future;
  for (const auto &op : s->q.ops)
    if (!op.dead && op.kind == 0) future.push_back(&op);
  int rc = dist_make_local(c->dist, s->amps, s->peers, s->n, s->L, s->perm, pending, c->sm_count, c->stream, &c->stats,
                           &future);
  if (rc != QB_OK) return fail(rc, "global<->local swap failed: %s", dist_last_error());
  return QB_OK;
}

// The live sub-cube of this rank's shard in PHYSICAL local bits.  Returns false if the support
// cannot be used (nothing known, or too fragmented for the kernels); *dead = this rank holds
// only zeros (a known global bit has the other value here).
bool live_cube(const Buffer *s, uint64_t *mask, uint64_t *val, bool *dead) {
  *mask = *val = 0;
  *dead = false;
  if (!s->zmask || !s->ctx->opt.support) return false;
  for (int lb = 0; lb < s->n; ++lb) {
    if (!((s->zmask >> lb) & 1ull)) continue;
    const int pb = s->perm[lb];
    const uint64_t v = (s->zval >> lb) & 1ull;
    if (pb < s->L) {
      *mask |= 1ull << pb;
      *val |= v << pb;
    } else if ((uint64_t)((s->ctx->rank >> (pb - s->L)) & 1) != v) {
      *dead = true;
    }
  }
  if (cube_runs(s->L, *mask) > kMaxRuns) {
    *mask = *val = 0;
    return *dead;
  }
  return true;
}

static bool finite8(const double *m) {
  for (int i = 0; i < 8; ++i)
    if (!std::isfinite(m[i])) return false;
  return true;
}

int run_fused_segment(Buffer *s, std::vector<const HostOp *> seg, const double *gscale, bool *gscale_done,
                      bool final_seg = false) {
  qb_ctx *c = s->ctx;
  int T, R;
  effective_tile(c->opt, s->L, T, R);
  PlanOptions opt = c->opt;
  opt.tile_bits = T;
  opt.reg_bits = R;
  if (!opt.fuse) opt.max_pass_gates = 1;
  // out-of-place passes (tiles written as contiguous blocks, qubits relabelled): single-GPU states
  // with room for a second shard
  opt.oop = (c->opt.oop && (c->nranks == 1 || c->opt.oop_dist) && T > 0 && ensure_alt(s)) ? c->opt.oop : 0;
  if (opt.oop && opt.low_bits < c->opt.oop_low_bits) opt.low_bits = std::min(c->opt.oop_low_bits, T);
  while (!seg.empty()) {
    std::vector<PhysOp> pops(seg.size());
    for (size_t i = 0; i < seg.size(); ++i) {
      const HostOp &h = *seg[i];
      pops[i].type = h.type;
      pops[i].target = s->perm[h.target];
      pops[i].ctrl = phys_mask(s, h.ctrl);
      memcpy(pops[i].m, h.m, sizeof(h.m));
    }
    // the support in today's physical bits (it changes with every global<->local swap); a rank
    // whose known global bits contradict its rank number holds only zeros: no pass at all
    bool rank_dead = false;
    {
      uint64_t mask, val;
      opt.known_mask = opt.known_val = 0;
      if (c->opt.skip_dead && live_cube(s, &mask, &val, &rank_dead)) {
        opt.known_mask = mask;
        opt.known_val = val;
      } else {
        rank_dead = false;
      }
      if (gscale && !(std::isfinite(gscale[0]) && std::isfinite(gscale[1]))) {
        opt.known_mask = opt.known_val = 0;
        rank_dead = false;
      }
      for (const auto &po : pops)
        if (!finite8(po.m)) rank_dead = false;
    }
    auto t0 = std::chrono::steady_clock::now();
    std::vector<int> labels(s->L, 0);  // the logical bit on each local physical bit (ties between qubits nothing
    for (int q = 0; q < s->n; ++q)     // waits for: the layouts out-of-place passes produce depend on the ops only)
      if (s->perm[q] < s->L) labels[s->perm[q]] = q;
    PlanResult plan = plan_passes_until_swap(pops, s->L, c->rank, opt, &labels);
    const bool all = plan.consumed == seg.size();
    // ---- a global<->local swap follows this plan (something is left that targets a global qubit):
    // fuse it into the stores of the plan's last pass -- that pass writes every tile straight into
    // the second shard of the rank that owns it after the swap, over NVLink peer memory, instead of
    // a local store plus a separate exchange sweep (XchGeom, qb_internal.h).  Needs: an out-of-place
    // last pass, both shards peer-mapped on every rank, no rank whose shard is known to be all zero
    // (it would skip the pass), no pending copy-on-write, and every victim outside that pass's block.
    std::vector<SwapPair> xsw;
    if (!all && c->nranks > 1 && c->opt.fuse_exchange && !plan.passes.empty() && !plan.final_pos.empty() && s->zmask == 0 &&
        !s->cow_src && s->alt && c->nranks <= kMaxXchRanks && dist_has_peers(c->dist, s->peers) &&
        dist_has_peers(c->dist, s->peers_alt)) {
      DevPass *LP = reinterpret_cast<DevPass *>(plan.passes.back().blob.data());
      if (LP->oop) {
        std::vector<int> perm2 = s->perm;  // the layout after this plan
        for (int &x : perm2)
          if (x < s->L) x = plan.final_pos[x];
        std::vector<const HostOp *> rest0, future;
        for (size_t i = 0; i < seg.size(); ++i)
          if (!plan.done[i]) rest0.push_back(seg[i]);
        for (const auto &op : s->q.ops)
          if (!op.dead && op.kind == 0) future.push_back(&op);
        std::vector<SwapPair> sw = choose_swaps(s->n, s->L, perm2, rest0, true, &future);  // (what make_local would choose)
        // (the destination pointers are filled in at launch: the two shards trade places with every pass before it)
        if (fused_exchange_geometry(*LP, s->L, c->rank, c->nranks, sw, &LP->xch)) xsw.swap(sw);
      }
    }
    c->stats.plan_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    // ---- which passes run as structure-specialised kernels (qb_jit.cpp).  Every rank takes the
    // same decisions (same plans, same sighting counts): the factors those kernels leave out
    // must be the same on every shard, because exchanges move raw device amplitudes.
    const int jit_thr = (c->opt.jit > 0 && (!c->opt.dbg_skip || (c->opt.dbg_skip & 16))) ? c->opt.jit : 0;
    const size_t npass = plan.passes.size();
    // the flush's last pass takes the pending scalar (and whatever the specialised passes leave out)
    const bool finish = all && final_seg && npass > 0;
    double gfin[2] = {1.0, 0.0};
    bool want_gfin = false;
    if (finish && gscale && !*gscale_done) {
      gfin[0] = gscale[0];
      gfin[1] = gscale[1];
      want_gfin = true;
      *gscale_done = true;
    }
    if (finish && jit_thr) want_gfin = true;  // (has_gscale is part of a pass's STRUCTURE: keep it stable)
    if (want_gfin) reinterpret_cast<DevPass *>(plan.passes.back().blob.data())->has_gscale = 1;
    std::vector<void *> jit_handle(npass, nullptr);
    std::vector<JitProgram> jit_prog(npass);
    std::vector<double> mid_scale(npass, 0.0);  // != 0: this (not last) pass applies the running factor (range guard)
    std::vector<double> generic_undo(npass, 0.0);  // != 0: a GENERIC kernel runs a pass that is defined to leave
                                                   // this factor out: it divides by it on the way out
    if (jit_thr) {
      for (size_t i = 0; i < npass; ++i) {
        PassPlan &p = plan.passes[i];
        std::string err;
        if (!jit_quick(p, jit_prog[i], nullptr)) continue;
        DevPass *P = reinterpret_cast<DevPass *>(p.blob.data());
        const bool last = finish && i + 1 == npass;
        if (!last && !P->has_gscale && !(std::fabs(s->jit_left * jit_prog[i].left_out) > 0x1p-300)) {
          // keep the stored amplitudes inside the exponent range: apply the factor here
          P->has_gscale = 1;
          P->gscale[0] = 1.0;
          P->gscale[1] = 0.0;
          if (!jit_quick(p, jit_prog[i], nullptr)) continue;
          mid_scale[i] = 1.0;
        }
        bool requested = false;
        const int jr = jit_lookup(jit_prog[i], p, jit_thr, &jit_handle[i], &err, &requested, c->rank);
        if (jr < 0) jit_handle[i] = nullptr;  // the generic kernel computes the same thing
        // Sharded states: WHICH kernel runs may differ between ranks (background compilation
        // finishes at different times), so there a pass whose structure has reached the
        // threshold -- the same on every rank -- is DEFINED to leave its factor out whichever
        // kernel runs: exchanges move raw device amplitudes, every shard must carry the same
        // pending factor.  On one GPU only a specialised kernel leaves anything out.
        const bool leaves_out = c->nranks > 1 ? requested : jit_handle[i] != nullptr;
        if (!leaves_out) jit_handle[i] = nullptr;
        if (leaves_out) {
          s->jit_left *= jit_prog[i].left_out;
          if (!jit_handle[i]) generic_undo[i] = jit_prog[i].left_out;
          if (mid_scale[i] != 0.0) {
            mid_scale[i] = s->jit_left;
            s->jit_left = 1.0;
          }
        } else if (mid_scale[i] != 0.0) {
          mid_scale[i] = 1.0;  // generic kernel, nothing left out: it scales by one
        }
      }
    }
    if (finish) {
      gfin[0] *= s->jit_left;
      gfin[1] *= s->jit_left;
      s->jit_left = 1.0;
      if (want_gfin) {
        DevPass *P = reinterpret_cast<DevPass *>(plan.passes.back().blob.data());
        P->gscale[0] = gfin[0];
        P->gscale[1] = gfin[1];
      }
    }
    for (size_t i = 0; i < npass; ++i) {  // the scalar each pass applies on its way out
      DevPass *P = reinterpret_cast<DevPass *>(plan.passes[i].blob.data());
      if (mid_scale[i] != 0.0) {
        P->gscale[0] = mid_scale[i];
        P->gscale[1] = 0.0;
      }
      if (generic_undo[i] != 0.0) {
        if (!P->has_gscale) {
          P->has_gscale = 1;
          P->gscale[0] = 1.0;
          P->gscale[1] = 0.0;
        }
        P->gscale[0] /= generic_undo[i];
        P->gscale[1] /= generic_undo[i];
      }
    }
    for (size_t i = 0; i < npass; ++i) {
      PassPlan &p = plan.passes[i];
      const bool xpass = !xsw.empty() && i + 1 == npass;  // this pass's stores carry the swap
      if (xpass) {  // every rank's second shard as of NOW; nobody still reads the shard the peers are about to write
        XchGeom &X = reinterpret_cast<DevPass *>(p.blob.data())->xch;
        for (int r = 0; r < c->nranks; ++r) X.peer[r] = reinterpret_cast<uint64_t>(s->peers_alt[r]);
        int rc = dist_stream_barrier(c->dist, c->stream);
        if (rc != QB_OK) return fail(rc, "barrier before the fused swap failed: %s", dist_last_error());
      }
      cudaEvent_t e0 = nullptr, e1 = nullptr;
      if (c->opt.time_kernels && !xpass) {  // (its duration is NVLink's, not the pass's: not part of fused_ms)
        QB_TRY(get_event(c, &e0));
        QB_TRY(get_event(c, &e1));
        QB_CUDA(cudaEventRecord(e0, c->stream));
      }
      // a pending copy-on-write rides on the first pass that visits every tile: it reads the old
      // shard and writes the new one (no separate copy); anything else copies first
      const double2 *src = nullptr;
      if (s->cow_src) {
        if (!rank_dead && p.ntiles == (1ull << (s->L - p.tile_bits))) {
          src = s->cow_src;
          s->cow_src = nullptr;
          c->stats.cow_fused++;
        } else {
          QB_TRY(ensure_inplace(s));
        }
      }
      // an out-of-place pass writes the other shard (unless it already reads somebody else's: the
      // copy-on-write source) and the two trade places
      const bool oop_pass = reinterpret_cast<const DevPass *>(p.blob.data())->oop != 0;
      double2 *dst = s->amps;
      if (oop_pass && !src) {
        if (!s->alt) return fail(QB_ERR_STATE, "internal: out-of-place pass without a second shard");
        if (rank_dead && !s->alt_zero) {  // this rank's shard is all zero and stays so: the other one must be, too
          QB_CUDA(cudaMemsetAsync(s->alt, 0, sizeof(double2) << s->L, c->stream));
          s->alt_zero = true;
        }
        dst = s->alt;
        src = s->amps;
      }
      if (!rank_dead) {
        if (jit_handle[i]) {
          const DevPass *P = reinterpret_cast<const DevPass *>(p.blob.data());
          double gs[2] = {P->gscale[0], P->gscale[1]};
          if (!P->has_gscale) gs[0] = 1.0, gs[1] = 0.0;
          std::string err;
          const std::vector<uint8_t> args = jit_pack_args(jit_prog[i], gs, P->rank_bits, P->base_fixed, P->xch.n ? &P->xch : nullptr);
          if (jit_launch(jit_handle[i], dst, src, p.ntiles, args, c->sm_count, c->stream, &err) != 0)
            return fail(QB_ERR_CUDA, "%s", err.c_str());
        } else {
          QB_CUDA(launch_fused_pass(dst, src, p.blob.data(), (uint32_t)p.blob.size(), p.tile_bits, p.reg_bits, p.ntiles,
                                    c->sm_count, c->stream, nullptr));
        }
      }
      if (xpass) {  // every rank's tiles have landed before anybody reads its new shard
        int rc = dist_stream_barrier(c->dist, c->stream);
        if (rc != QB_OK) return fail(rc, "barrier after the fused swap failed: %s", dist_last_error());
        c->stats.exchanges++;
        c->stats.exchanges_fused++;
        c->stats.exchange_bytes += ((sizeof(double2) << s->L) >> xsw.size()) * ((1ull << xsw.size()) - 1ull);
      }
      if (dst != s->amps) {
        std::swap(s->amps, s->alt);
        std::swap(s->peers, s->peers_alt);
        if (!rank_dead) s->alt_zero = false;  // (the shard just read holds amplitudes)
      }
      c->stats.tiles += rank_dead ? 0 : p.ntiles;
      if (e0) {
        QB_CUDA(cudaEventRecord(e1, c->stream));
        c->timed.emplace_back(e0, e1);
      }
      c->stats.passes++;
      c->stats.rounds += p.nrounds;
      c->stats.ops_executed += p.ngates;
    }
    if (!plan.final_pos.empty()) {  // the out-of-place passes moved the local qubits
      for (int &x : s->perm)
        if (x < s->L) x = plan.final_pos[x];
      opt.layout_known = 1;  // (a replan after the swap below starts from a layout this flush produced)
    }
    if (!xsw.empty()) apply_swaps_to_perm(s->perm, xsw);  // (the last pass's stores carried it)
    for (size_t i = 0; i < seg.size(); ++i) {  // the scheduled ops now shape the support
      if (!plan.done[i]) continue;
      const HostOp &h = *seg[i];
      if (!finite8(h.m)) s->zmask = 0;
      if (h.type != G_DIAG) s->zmask &= ~(1ull << h.target);
    }
    s->zval &= s->zmask;
    if (all) break;
    std::vector<const HostOp *> rest;
    for (size_t i = 0; i < seg.size(); ++i)
      if (!plan.done[i]) rest.push_back(seg[i]);
    if (xsw.empty()) {
      // whatever is left starts with gates on global qubits: remap them into the shard
      QB_TRY(make_local(s, rest));
    }
    seg.swap(rest);
  }
  return QB_OK;
}

// what one executed op does to the support.  Applied right after the op has run: the NEXT
// segment of the same flush plans its dead tiles from it (a dense block populates its qubits).
void support_after_op(Buffer *s, const HostOp &op) {
  if (op.kind == 3) {  // (a Z-only rotation is a phase: what is zero stays zero)
    s->zmask &= ~op.px;
  } else if (op.kind == 2) {
    for (int j = 0; j < op.k; ++j) s->zmask &= ~(1ull << op.kq_bits[j]);
    for (double x : op.kq_m)
      if (!std::isfinite(x)) {
        s->zmask = 0;
        s->all_finite = false;
      }
  } else {
    if (!finite8(op.m)) {  // 0 * NaN = NaN: nothing stays zero (zero-weight collapse, StateVec.hs:92)
      s->zmask = 0;
      s->all_finite = false;
    }
    if (op.type != G_DIAG) s->zmask &= ~(1ull << op.target);
  }
  s->zval &= s->zmask;
}

// The greedy launch cut of the Pauli kernels (k_pauli_rot_tile, k_pauli_sum_tile, k_pauli_rot_adjoint_tile):
// the launch that starts at string i0 of lx (logical X masks) ends before the returned index.  A string joins
// the running launch while that holds fewer than kPauliMaxRot and its X qubits add nothing to the launch's X
// union or the union with the three low physical bits (one 128-byte line) still fits the tile.  *ux = the
// launch's logical X union.
static_assert(kPauliTileBits == QB_PAULI_ROT_MAX_X, "the tile holds the widest string the header allows");
size_t pauli_cut(const Buffer *s, const std::vector<uint64_t> &lx, size_t i0, uint64_t *ux) {
  const int T = std::min(kPauliTileBits, s->L);
  const uint64_t low = (1ull << std::min(3, s->L)) - 1ull;
  *ux = 0;
  size_t i1 = i0;
  for (; i1 < lx.size() && i1 - i0 < size_t(kPauliMaxRot); ++i1) {
    const uint64_t x = lx[i1];
    if (i1 > i0 && (x & ~*ux) && __builtin_popcountll(phys_mask(s, *ux | x) | low) > T) break;
    *ux |= x;
  }
  return i1;
}

// The tile of a launch whose logical X union is ux (already inside the shard): those physical bits topped up
// with the lowest other local bits.  Fills the tile geometry shared by the Pauli kernels' argument blocks.
template <class A>
int pauli_tile(const Buffer *s, uint64_t ux, A &args) {
  const int L = s->L, T = std::min(kPauliTileBits, L);
  uint64_t tile = phys_mask(s, ux);
  if (__builtin_popcountll(tile) > T || (tile >> L))
    return fail(QB_ERR_UNSUPPORTED, "internal: Pauli strings with X outside the rotation tile");
  for (int b = 0; __builtin_popcountll(tile) < T; ++b) tile |= 1ull << b;
  args.tile_bits = uint32_t(T);
  for (int b = 0, i = 0; b < L; ++b)
    if ((tile >> b) & 1ull) args.tile_pos[i++] = uint8_t(b);
  for (int b = 0; b < L;) {  // runs of the local bits outside the tile
    if ((tile >> b) & 1ull) {
      ++b;
      continue;
    }
    int e = b;
    while (e < L && !((tile >> e) & 1ull)) ++e;
    args.run_shift[args.nruns] = uint8_t(b);
    args.run_len[args.nruns++] = uint8_t(e - b);
    b = e;
  }
  return QB_OK;
}

// a physical mask on the tile-local bits of a launch
template <class A>
uint32_t pauli_tile_local(const A &args, uint64_t m) {
  uint32_t r = 0;
  for (uint32_t i = 0; i < args.tile_bits; ++i) r |= uint32_t((m >> args.tile_pos[i]) & 1ull) << i;
  return r;
}

// A stretch of consecutive Pauli rotations (HostOp kind 3), cut by pauli_cut into launches of
// k_pauli_rot_tile (one read + write sweep each).  Sharded: the launch's X qubits are brought into the shard
// first, and Z on global qubits becomes this rank's sign.
int run_pauli_rots(Buffer *s, const std::vector<const HostOp *> &run) {
  qb_ctx *c = s->ctx;
  QB_TRY(ensure_inplace(s));
  const int L = s->L;
  const uint64_t local = (1ull << L) - 1ull;
  std::vector<uint64_t> lx;
  for (const HostOp *h : run) lx.push_back(h->px);
  for (size_t i0 = 0; i0 < run.size();) {
    uint64_t ux = 0;  // logical X union of the launch
    const size_t i1 = pauli_cut(s, lx, i0, &ux);
    if (c->nranks > 1) QB_TRY(localise_x(s, ux));
    PauliRotArgs args;
    memset(&args, 0, sizeof args);
    args.nrot = uint32_t(i1 - i0);
    QB_TRY(pauli_tile(s, ux, args));
    uint64_t tile = 0;
    for (uint32_t i = 0; i < args.tile_bits; ++i) tile |= 1ull << args.tile_pos[i];
    auto tile_local = [&](uint64_t m) { return pauli_tile_local(args, m); };
    for (size_t i = i0; i < i1; ++i) {
      const HostOp &h = *run[i];
      const uint64_t xp = phys_mask(s, h.px), zp = phys_mask(s, h.pz);
      PauliRotParam &p = args.rot[i - i0];
      p.xt = tile_local(xp);
      p.zt = tile_local(zp);
      p.zout = zp & local & ~tile;
      p.c = h.m[0];
      // the partner's factor -i s i^ph, ph = popc(x & z) mod 4 (P = i^ph X^x Z^z: Y = i X Z)
      const double f = (__builtin_popcountll((zp >> L) & uint64_t(c->rank)) & 1) ? -h.m[1] : h.m[1];
      const int ph = __builtin_popcountll(h.px & h.pz) & 3;
      p.ar = ph == 1 ? f : ph == 3 ? -f : 0.0;
      p.ai = ph == 0 ? -f : ph == 2 ? f : 0.0;
    }
    QB_CUDA(launch_pauli_rot(s->amps, L, args, c->stream));
    c->stats.simple_launches++;
    c->stats.ops_executed += args.nrot;
    i0 = i1;
  }
  return QB_OK;
}

// run the queued ops.  The deferred scalar rides on the last fused pass if there is one;
// otherwise it stays pending in s->pscale (no sweep just to scale).
int exec_queue(Buffer *s) {
  qb_ctx *c = s->ctx;
  OpQueue &q = s->q;
  c->stats.ops_submitted += q.submitted;
  c->stats.ops_folded += q.folded;
  q.submitted = q.folded = 0;
  {  // total pending scalar = state-level * queue-level
    const double r = s->pscale[0] * q.gscale[0] - s->pscale[1] * q.gscale[1];
    const double i = s->pscale[0] * q.gscale[1] + s->pscale[1] * q.gscale[0];
    s->pscale[0] = r;
    s->pscale[1] = i;
    q.gscale[0] = 1.0;
    q.gscale[1] = 0.0;
  }
  if (!(std::isfinite(s->pscale[0]) && std::isfinite(s->pscale[1]))) {
    s->zmask = s->zval = 0;
    s->all_finite = false;
  }
  if (q.empty()) {
    q.clear();
    return QB_OK;
  }
  const bool has_g = !(s->pscale[0] == 1.0 && s->pscale[1] == 0.0);
  const double g[2] = {s->pscale[0], s->pscale[1]};
  bool g_done = !has_g;
  int T, R;
  effective_tile(c->opt, s->L, T, R);
  int rc = QB_OK;
  // ops from index i on that are still to run (swap selection looks ahead over them)
  auto pending_from = [&](size_t i) {
    std::vector<const HostOp *> pend;
    for (size_t j = i; j < q.ops.size(); ++j)
      if (!q.ops[j].dead) pend.push_back(&q.ops[j]);
    return pend;
  };
  // a dense block needs ALL its qubits inside the shard
  auto kq_needs_swap = [&](const HostOp &op) {
    for (int j = 0; j < op.k; ++j)
      if (s->perm[op.kq_bits[j]] >= s->L) return true;
    return false;
  };
  // the stretch of consecutive Pauli rotations that starts at op i; i moves to its last op
  auto pauli_stretch = [&](size_t &i) {
    std::vector<const HostOp *> run;
    size_t j = i;
    for (; j < q.ops.size() && (q.ops[j].dead || q.ops[j].kind == 3); ++j)
      if (!q.ops[j].dead) run.push_back(&q.ops[j]);
    i = j - 1;
    const int r = run_pauli_rots(s, run);
    if (r == QB_OK)
      for (const HostOp *h : run) support_after_op(s, *h);
    return r;
  };
  if (T == 0) {
    for (size_t i = 0; i < q.ops.size(); ++i) {
      const HostOp &op = q.ops[i];
      if (op.dead) continue;
      if (op.kind == 3) {
        if ((rc = pauli_stretch(i)) != QB_OK) break;
        continue;
      }
      if ((op.kind == 0 && op.type != G_DIAG && s->perm[op.target] >= s->L) || (op.kind == 2 && kq_needs_swap(op)))
        if ((rc = make_local(s, pending_from(i))) != QB_OK) break;
      if ((rc = run_simple(s, op)) != QB_OK) break;
      support_after_op(s, op);
    }
  } else {
    std::vector<const HostOp *> seg;
    for (size_t i = 0; i < q.ops.size() && rc == QB_OK; ++i) {
      const HostOp &op = q.ops[i];
      if (op.dead) continue;
      if (op.kind == 0) {
        seg.push_back(&op);
        continue;
      }
      if (!seg.empty()) {
        rc = run_fused_segment(s, seg, nullptr, nullptr);
        seg.clear();
      }
      if (op.kind == 3) {  // (ends the fused segment, as a dense block does)
        if (rc == QB_OK) rc = pauli_stretch(i);
        continue;
      }
      if (rc == QB_OK && kq_needs_swap(op)) rc = make_local(s, pending_from(i));
      if (rc == QB_OK) rc = run_simple(s, op);
      if (rc == QB_OK) support_after_op(s, op);
    }
    if (rc == QB_OK && !seg.empty()) rc = run_fused_segment(s, seg, has_g ? g : nullptr, &g_done, true);
  }
  if (rc == QB_OK && g_done) {
    s->pscale[0] = 1.0;
    s->pscale[1] = 0.0;
  }
  if (s->jit_left != 1.0) {  // specialised passes ran but no last pass took their factor: it stays pending
    s->pscale[0] *= s->jit_left;
    s->pscale[1] *= s->jit_left;
    s->jit_left = 1.0;
  }
  q.clear();
  return rc;
}

// apply the pending scalar to the device amplitudes (live sub-cube only when the support is known)
int force_scale(Buffer *s) {
  if (s->pscale[0] == 1.0 && s->pscale[1] == 0.0) return QB_OK;
  qb_ctx *c = s->ctx;
  uint64_t mask, val;
  bool dead;
  const bool finite = std::isfinite(s->pscale[0]) && std::isfinite(s->pscale[1]);
  if (finite && live_cube(s, &mask, &val, &dead)) {
    if (!dead) {
      QB_CUDA(launch_cube_update(s->amps, s->L, mask, val, 1, s->pscale, c->sm_count, c->stream));
      c->stats.simple_launches++;
    }
  } else {
    if (!finite) s->zmask = s->zval = 0;
    QB_TRY(run_gscale_simple(s, s->pscale));
  }
  s->pscale[0] = 1.0;
  s->pscale[1] = 0.0;
  return QB_OK;
}

// reduce (S0, S1) split by a logical bit (lb < 0: total) into host doubles; all-reduced when
// distributed.  The buffer stands at the position to be measured (materialise() first).
int sumsq_buffer(Buffer *s, int lb, double *s0, double *s1) {
  qb_ctx *c = s->ctx;
  if (!(std::isfinite(s->pscale[0]) && std::isfinite(s->pscale[1]))) QB_TRY(force_scale(s));  // NaN / inf must reach the data
  const int pb = lb < 0 ? -1 : s->perm[lb];
  const bool known = lb >= 0 && ((s->zmask >> lb) & 1ull);
  const int kbit = (pb >= 0 && pb < s->L && !known) ? pb : -1;
  uint64_t mask, val;
  bool dead;
  const bool cube = live_cube(s, &mask, &val, &dead);
  double a0 = 0.0, a1 = 0.0;
  if (!(cube && dead)) {
    if (cube && mask) {
      QB_CUDA(launch_sumsq_cube(s->amps, s->L, mask, val, kbit, c->red_partials, c->red_out, c->sm_count, c->stream));
    } else {
      QB_CUDA(launch_sumsq(s->amps, 1ull << s->L, kbit, c->red_partials, c->red_out, c->sm_count, c->stream));
    }
    c->stats.reduce_launches += 2;
    QB_CUDA(cudaMemcpyAsync(c->red_host, c->red_out, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    QB_CUDA(cudaStreamSynchronize(c->stream));
    a0 = c->red_host[0];
    a1 = c->red_host[1];
  }
  if (known) {  // every live amplitude has the known value of this bit
    if ((s->zval >> lb) & 1ull) {
      a1 = a0;
      a0 = 0.0;
    }
  } else if (pb >= s->L) {  // global bit: this rank's whole shard has one value of it
    if ((c->rank >> (pb - s->L)) & 1) {
      a1 = a0;
      a0 = 0.0;
    }
  }
  if (c->nranks > 1) {
    double v[2] = {a0, a1};
    int rc = dist_allreduce_sum(c->dist, v, 2, c->stream);
    if (rc != QB_OK) return fail(rc, "allreduce failed: %s", dist_last_error());
    a0 = v[0];
    a1 = v[1];
  }
  const double g2 = s->pscale[0] * s->pscale[0] + s->pscale[1] * s->pscale[1];  // the pending scalar, arithmetically
  if (g2 != 1.0) {
    a0 *= g2;
    a1 *= g2;
  }
  if (s0) *s0 = a0;
  if (s1) *s1 = a1;
  return QB_OK;
}

// collapse (StateVec.hs:104-114) as a log entry being executed (everything before it has run, the
// queue is empty): zero-fill the half of the live sub-cube that dies, learn the bit, defer the
// normalisation.  No read, no full pass.  `weight` = the reduction taken when the entry was logged.
int collapse_exec(Buffer *s, int lb, int bit, double weight) {
  qb_ctx *c = s->ctx;
  if (weight == 0.0 || !std::isfinite(weight)) {
    // the reference divides by norm_2 = 0: every amplitude becomes NaN (StateVec.hs:92,107)
    double m[8] = {0};
    m[0] = m[6] = NAN;
    s->q.push_1q(lb, 0, m);
    return QB_OK;
  }
  const double f = 1.0 / std::sqrt(weight);
  if (!c->opt.support) {  // A/B switch: the collapse as a queued diagonal gate (a full pass later)
    double m[8] = {0};
    m[bit ? 6 : 0] = f;
    s->q.push_1q(lb, 0, m);
    return QB_OK;
  }
  const bool known = (s->zmask >> lb) & 1ull;  // then the other value has weight 0 and was handled above
  if (!known) {
    QB_TRY(ensure_inplace(s));
    uint64_t mask, val;
    bool dead;
    const bool cube = live_cube(s, &mask, &val, &dead);
    const int pb = s->perm[lb];
    if (!(cube && dead)) {
      if (pb < s->L) {
        const uint64_t m2 = mask | (1ull << pb), v2 = val | (uint64_t(bit ? 0 : 1) << pb);
        if (cube_runs(s->L, m2) <= kMaxRuns) {
          QB_CUDA(launch_cube_update(s->amps, s->L, m2, v2, 0, nullptr, c->sm_count, c->stream));
        } else {  // too fragmented for the cube kernels: the plain diagonal sweep
          const double d0[2] = {bit ? 0.0 : 1.0, 0.0}, d1[2] = {bit ? 1.0 : 0.0, 0.0};
          QB_CUDA(launch_simple_diag(s->amps, s->L, 1ull << pb, 0, 0, d0, d1, c->sm_count, c->stream));
        }
        c->stats.simple_launches++;
      } else if (((c->rank >> (pb - s->L)) & 1) != bit) {  // this rank holds the half that dies
        QB_CUDA(launch_cube_update(s->amps, s->L, mask, val, 0, nullptr, c->sm_count, c->stream));
        c->stats.simple_launches++;
      }
    }
    s->zmask |= 1ull << lb;
    s->zval = (s->zval & ~(1ull << lb)) | (uint64_t(bit) << lb);
  }
  const double r = s->pscale[0] * f, i = s->pscale[1] * f;
  s->pscale[0] = r;
  s->pscale[1] = i;
  return QB_OK;
}

// ---- lineage: execute log[mat .. upto) on the buffer's device data ------------------------------
// The peephole (qb_planner.cpp, OpQueue) runs here, over the whole stretch between two
// observations, however the caller sliced it into handles.
int exec_log(Buffer *b, size_t upto) {
  qb_ctx *c = b->ctx;
  int rc = QB_OK;
  b->q.reset(b->n, c->opt.peephole != 0, c->opt.rot != 0);
  for (size_t p = b->mat; p < upto && rc == QB_OK; ++p) {
    const LogOp &o = b->log[p - b->log_base];
    switch (o.kind) {
      case LOG_1Q: b->q.push_1q(o.target, o.ctrl, o.m); break;
      case LOG_KQ: b->q.push_kq(o.kq_bits, o.k, o.kq_m->data(), o.ctrl); break;
      case LOG_SCALE: b->q.mul_gscale(o.m[0], o.m[1]); break;
      case LOG_PAULI: b->q.push_pauli(o.ctrl, o.pz, o.m[0], o.m[1]); break;
      case LOG_COLLAPSE:
        rc = exec_queue(b);
        if (rc == QB_OK) rc = collapse_exec(b, o.target, (int)o.ctrl, o.m[0]);
        break;
      default: rc = fail(QB_ERR_ARG, "internal: bad log entry"); break;
    }
  }
  if (rc == QB_OK) rc = exec_queue(b);
  if (rc == QB_OK) rc = ensure_inplace(b);  // (a copy-on-write no pass took along)
  if (rc != QB_OK) {
    b->broken = true;
    b->broken_why = g_last_error;
    b->cow_src = nullptr;
    return rc;
  }
  b->mat = upto;
  return QB_OK;
}

// drop the log entries nobody can ask for any more
void trim_log(Buffer *b) {
  size_t keep = b->mat;
  for (const qb_state *h : b->handles)
    if (!h->stale) keep = std::min(keep, h->pos);
  if (keep > b->log_base) {
    b->log.erase(b->log.begin(), b->log.begin() + (keep - b->log_base));
    b->log_base = keep;
  }
}

void copy_meta(Buffer *dst, const Buffer *src) {
  dst->perm = src->perm;
  dst->zmask = src->zmask;
  dst->zval = src->zval;
  dst->pscale[0] = src->pscale[0];
  dst->pscale[1] = src->pscale[1];
  dst->all_finite = src->all_finite;
}

// Give handle h a shard of its own that stands where h's old shard stands, carrying the log
// entries h still needs.  lazy: the copy itself may ride on the first pass of the caller's exec_log.
int split_off(qb_state *h, bool lazy_copy) {
  Buffer *b = h->b;
  qb_ctx *c = h->ctx;
  Buffer *nb = nullptr;
  QB_TRY(new_buffer(c, b->n, &nb));
  copy_meta(nb, b);
  nb->log.assign(b->log.begin() + (b->mat - b->log_base), b->log.begin() + (h->pos - b->log_base));
  nb->log_base = nb->mat = 0;
  if (lazy_copy) {
    nb->cow_src = b->amps;
  } else {
    cudaError_t e = cudaMemcpyAsync(nb->amps, b->amps, sizeof(double2) << b->L, cudaMemcpyDeviceToDevice, c->stream);
    if (e != cudaSuccess) {
      nb->handles.clear();
      release_buffer(nb);
      return fail(QB_ERR_CUDA, "clone: %s", cudaGetErrorString(e));
    }
    c->stats.cow_copies++;
  }
  const size_t npos = nb->log.size();
  b->handles.erase(std::find(b->handles.begin(), b->handles.end(), h));
  attach(h, nb, npos);
  if (b->handles.empty()) release_buffer(b);  // (cannot happen: a split is only needed while others share b)
  else trim_log(b);
  return QB_OK;
}

// Bring the device data to h's position so that it can be observed.  In place when no live handle
// needs the older data; otherwise h moves to a shard of its own (copy-on-write, the copy riding on
// the first fused pass), or -- option "linear" -- the older handles are consumed.
int materialise(qb_state *h) {
  QB_TRY(check_state(h));
  Buffer *b = h->b;
  if (b->mat == h->pos) return QB_OK;
  bool older = false;
  for (const qb_state *g : b->handles)
    if (g != h && !g->stale && g->pos < h->pos) older = true;
  QB_TRY(agree_any(h->ctx, b, &older));
  if (older && h->ctx->linear) {
    for (qb_state *g : b->handles)
      if (g != h && g->pos < h->pos) g->stale = true;
    older = false;
  }
  if (older) {
    QB_TRY(split_off(h, true));
    b = h->b;
  }
  QB_TRY(exec_log(b, h->pos));
  trim_log(b);
  return QB_OK;
}

// h is about to be changed in place (upload, axpy target): nobody else may see its shard
int make_unique(qb_state *h) {
  QB_TRY(materialise(h));
  Buffer *b = h->b;
  bool shared = false;
  for (const qb_state *g : b->handles)
    if (g != h && !g->stale) shared = true;
  QB_TRY(agree_any(h->ctx, b, &shared));
  if (!shared) return QB_OK;
  if (h->ctx->linear) {
    for (qb_state *g : b->handles)
      if (g != h) g->stale = true;
    return QB_OK;
  }
  return split_off(h, false);
}

// Change the qubit layout of a buffer (logical bit q moves to physical bit want[q]) without
// changing what it means: operands of <.>, +: and tensor must agree on where each qubit lives,
// and independent global<->local swaps make layouts diverge (StateVec.hs:51-58,98-100).  A
// sequence of position swaps: local/local = one in-place kernel over half the shard, global/local
// = one pairwise exchange, global/global = three of those through the top local bit.  Collective
// on a sharded context (every rank holds the same perm and takes the same steps).
int relayout(Buffer *b, const std::vector<int> &want) {
  qb_ctx *c = b->ctx;
  QB_TRY(ensure_inplace(b));
  const int L = b->L;
  {
    bool local_only = true, same = true;
    for (int q = 0; q < b->n; ++q) {
      if (b->perm[q] != want[q]) same = false;
      if ((b->perm[q] >= L) != (want[q] >= L) || (b->perm[q] >= L && b->perm[q] != want[q])) local_only = false;
    }
    if (same) return QB_OK;
    if (local_only && c->nranks == 1 && ensure_alt(b)) {  // dst[new place of i] = src[i]
      std::vector<int> np(L, 0);
      for (int q = 0; q < b->n; ++q)
        if (b->perm[q] < L) np[b->perm[q]] = want[q];
      QB_CUDA(launch_permute_bits(b->alt, b->amps, L, np.data(), c->sm_count, c->stream));
      c->stats.simple_launches++;
      std::swap(b->amps, b->alt);
      b->perm = want;
      return QB_OK;
    }
  }
  const bool peer_path = c->nranks > 1 && dist_has_peers(c->dist, b->peers);
  auto swap_positions = [&](int p1, int p2) -> int {  // physical positions
    if (p1 == p2) return QB_OK;
    if (p1 < p2) std::swap(p1, p2);  // p1 > p2
    if (p1 < L) {
      QB_CUDA(launch_swap_bits(b->amps, L, p1, p2, c->sm_count, c->stream));
      c->stats.simple_launches++;
      for (int &x : b->perm) x = (x == p1) ? p2 : (x == p2 ? p1 : x);
      return QB_OK;
    }
    if (p2 < L) {  // global p1 <-> local p2
      int lb = p2;
      if (!peer_path && lb != L - 1) {  // send/recv moves contiguous blocks: go through the top local bit
        QB_CUDA(launch_swap_bits(b->amps, L, lb, L - 1, c->sm_count, c->stream));
        for (int &x : b->perm) x = (x == lb) ? L - 1 : (x == L - 1 ? lb : x);
        lb = L - 1;
      }
      std::vector<SwapPair> sw{{p1, lb}};
      int rc = dist_swap_pairs(c->dist, b->amps, b->peers, L, b->perm, sw, c->sm_count, c->stream, &c->stats);
      if (rc != QB_OK) return fail(rc, "layout exchange failed: %s", dist_last_error());
      if (lb != p2) {
        QB_CUDA(launch_swap_bits(b->amps, L, p2, L - 1, c->sm_count, c->stream));
        for (int &x : b->perm) x = (x == p2) ? L - 1 : (x == L - 1 ? p2 : x);
      }
      return QB_OK;
    }
    // both global: through the top local bit t: (p1 t)(p2 t)(p1 t)
    const int t = L - 1;
    for (int g : {p1, p2, p1}) {
      std::vector<SwapPair> sw{{g, t}};
      int rc = dist_swap_pairs(c->dist, b->amps, b->peers, L, b->perm, sw, c->sm_count, c->stream, &c->stats);
      if (rc != QB_OK) return fail(rc, "layout exchange failed: %s", dist_last_error());
    }
    return QB_OK;
  };
  for (int q = 0; q < b->n; ++q) {
    // each swap puts at least qubit q where it belongs (the qubit that sat there takes q's old place)
    if (b->perm[q] != want[q]) QB_TRY(swap_positions(b->perm[q], want[q]));
  }
  for (int q = 0; q < b->n; ++q)
    if (b->perm[q] != want[q]) return fail(QB_ERR_STATE, "internal: relayout did not converge");
  return QB_OK;
}

// the device holds the TRUE amplitudes of h (deferred scalar applied)
int flush_locked(qb_state *h) {
  QB_TRY(materialise(h));
  return force_scale(h->b);
}

constexpr size_t kMaxLog = size_t(1) << 20;  // entries a lineage may queue before it is flushed on its own

// append an op to h's lineage.  A handle that is not at the tip of its log (another handle of the
// lineage went on from the same value) starts a lineage of its own first.
int append(qb_state *h, LogOp &&op) {
  QB_TRY(check_state(h));
  Buffer *b = h->b;
  if (h->pos != b->tip()) {
    QB_TRY(split_off(h, false));
    b = h->b;
  }
  b->log.push_back(std::move(op));
  h->pos = b->tip();
  if (b->log.size() > kMaxLog) QB_TRY(materialise(h));
  return QB_OK;
}

void drop_handle(qb_state *s) {
  qb_ctx *c = s->ctx;
  bool last_of_closed;
  {
    Guard g(c);
    if (!c->closed) detach(s);
    last_of_closed = (--c->handles == 0) && c->closed;
  }
  delete s;
  if (last_of_closed) delete c;
}

// reference qubit q is logical bit n - 1 - q
uint64_t logical_mask(int n, uint64_t m) {
  uint64_t r = 0;
  for (; m; m &= m - 1) r |= 1ull << (n - 1 - __builtin_ctzll(m));
  return r;
}

// (re, im) * i^popc(x & z) * this rank's sign of Z on global qubits: the factor of P = i^ph X^x Z^z that the
// tile kernels do not form (Y = i X Z)
void pauli_phase(const Buffer *s, uint64_t lx, uint64_t lz, double re, double im, double *out_re, double *out_im) {
  if (__builtin_popcountll((phys_mask(s, lz) >> s->L) & uint64_t(s->ctx->rank)) & 1) {
    re = -re;
    im = -im;
  }
  switch (__builtin_popcountll(lx & lz) & 3) {
    case 0: *out_re = re; *out_im = im; break;
    case 1: *out_re = -im; *out_im = re; break;
    case 2: *out_re = -re; *out_im = -im; break;
    default: *out_re = im; *out_im = -re; break;
  }
}

// Pauli-sum terms named by logical masks (coef: (re, im) per term), taken in the order of their X masks (a sum
// commutes; a stable sort, so the order is a fixed function of the input): the i-th is term ord[i], its X mask
// sx[i].  run_pauli_sum and the Chebyshev steps of qb_pauli_evolve cut them alike.
struct PauliTerms {
  std::vector<uint64_t> lx, lz;
  std::vector<double> coef;
  std::vector<size_t> ord;
  std::vector<uint64_t> sx;
  PauliTerms(std::vector<uint64_t> x, std::vector<uint64_t> z, std::vector<double> cf)
      : lx(std::move(x)), lz(std::move(z)), coef(std::move(cf)), ord(lx.size()), sx(lx.size()) {
    for (size_t t = 0; t < ord.size(); ++t) ord[t] = t;
    std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return lx[a] < lx[b]; });
    for (size_t t = 0; t < ord.size(); ++t) sx[t] = lx[ord[t]];
  }
};

// The launch of a Pauli sum that starts at sorted term i0: cut by pauli_cut on src's layout, its X qubits brought
// into src's shard (sharded), and its tile and terms filled in for src's layout with the coefficients scaled by
// f.  *i1 = the end of the launch.
int pauli_sum_launch(Buffer *src, const PauliTerms &h, double f, size_t i0, size_t *i1, PauliSumArgs &args) {
  qb_ctx *c = src->ctx;
  uint64_t ux = 0;
  *i1 = pauli_cut(src, h.sx, i0, &ux);
  if (c->nranks > 1) QB_TRY(localise_x(src, ux));
  const uint64_t local = (1ull << src->L) - 1ull;
  memset(&args, 0, sizeof args);
  args.nterms = uint32_t(*i1 - i0);
  QB_TRY(pauli_tile(src, ux, args));
  uint64_t tile = 0;
  for (uint32_t i = 0; i < args.tile_bits; ++i) tile |= 1ull << args.tile_pos[i];
  for (size_t i = i0; i < *i1; ++i) {
    const size_t t = h.ord[i];
    const uint64_t zp = phys_mask(src, h.lz[t]);
    PauliSumParam &p = args.term[i - i0];
    p.xt = pauli_tile_local(args, phys_mask(src, h.lx[t]));
    p.zt = pauli_tile_local(args, zp);
    p.zout = zp & local & ~tile;
    pauli_phase(src, h.lx[t], h.lz[t], f * h.coef[2 * t], f * h.coef[2 * t + 1], &p.cr, &p.ci);
  }
  return QB_OK;
}

// out <- (sum_t coef[t] P_t) src; out is a fresh shard of src's size whose old contents do not matter.  The first
// launch writes every amplitude of out in src's layout; later launches add, out following src's layout
// (localise_x) by relayout.  energy_dev: Re <src| H_launch src> of launch l into energy_dev[l], *nlaunch = the
// number of launches.
int run_pauli_sum(Buffer *src, Buffer *out, const std::vector<uint64_t> &lx, const std::vector<uint64_t> &lz,
                  const std::vector<double> &coef, double *energy_dev, int *nlaunch) {
  qb_ctx *c = src->ctx;
  QB_TRY(ensure_inplace(src));
  const PauliTerms h(lx, lz, coef);
  int nl = 0;
  for (size_t i0 = 0, i1 = 0; i0 < h.sx.size(); ++nl, i0 = i1) {
    PauliSumArgs args;
    QB_TRY(pauli_sum_launch(src, h, 1.0, i0, &i1, args));
    if (nl == 0) out->perm = src->perm;  // (the first launch writes every amplitude: born in src's layout)
    else if (out->perm != src->perm) QB_TRY(relayout(out, src->perm));
    args.first = nl == 0;
    QB_CUDA(launch_pauli_sum(src->amps, out->amps, src->L, args, energy_dev ? c->red_partials : nullptr,
                             energy_dev ? energy_dev + nl : nullptr, c->sm_count, c->stream));
    c->stats.simple_launches++;
    if (energy_dev) c->stats.reduce_launches++;
  }
  if (nlaunch) *nlaunch = nl;
  return QB_OK;
}

// Step k >= 1 of the Chebyshev recurrence of qb_pauli_evolve, one launch per run of the cut of h (H' = f h with
// f = 1 / r; the terms are scaled by f at step 1 and by 2 f later): prev <- H' cur (step 1) or 2 H' cur - prev,
// then acc <- a0 cur + ak prev (step 1) or acc + ak prev.  All three shards end in cur's layout; prev's and
// acc's old contents do not matter at step 1 (their first write is a store).
int run_pauli_cheb_step(Buffer *cur, Buffer *prev, Buffer *acc, const PauliTerms &h, double f, int64_t step,
                        const double a0[2], const double ak[2]) {
  qb_ctx *c = cur->ctx;
  for (size_t i0 = 0, i1 = 0; i0 < h.sx.size(); i0 = i1) {
    PauliChebArgs args;
    QB_TRY(pauli_sum_launch(cur, h, step == 1 ? f : 2.0 * f, i0, &i1, args.sum));
    const bool first = i0 == 0, last = i1 == h.sx.size();
    if (step == 1 && first) prev->perm = cur->perm;
    else if (prev->perm != cur->perm) QB_TRY(relayout(prev, cur->perm));
    if (step == 1) {
      if (last) acc->perm = cur->perm;  // (acc is first written, whole, by step 1's last launch)
    } else if (acc->perm != cur->perm) {
      QB_TRY(relayout(acc, cur->perm));
    }
    args.out_mode = !first ? kChebOutAdd : step == 1 ? kChebOutStore : kChebOutSub;
    args.acc_mode = !last ? kChebAccNone : step == 1 ? kChebAccFirst : kChebAccAdd;
    args.a0r = a0[0];
    args.a0i = a0[1];
    args.akr = ak[0];
    args.aki = ak[1];
    QB_CUDA(launch_pauli_cheb(cur->amps, prev->amps, acc->amps, cur->L, args, c->sm_count, c->stream));
    c->stats.simple_launches++;
  }
  return QB_OK;
}

// The Chebyshev coefficients of exp(-i tau x) on [-1, 1]: a[k] = (re, im) of a_0 = J_0(tau), a_k = 2 (-i)^k J_k(tau)
// for k = 0 .. K, K the smallest k >= 1 whose truncation bound 2 sum_{j > k} |J_j(tau)| is at most 2^-53.
// J_k by Miller's backward recurrence from far above K (rescaled before it can overflow), normalised with
// J_0 + 2 sum_m J_2m = 1; J_k(-tau) = (-1)^k J_k(tau).  false: K would exceed max_k.
bool cheb_coefficients(double tau, int64_t max_k, std::vector<double> &a) {
  const double at = std::fabs(tau);
  if (!(at < double(max_k))) return false;  // (K > |tau| once |tau| is large: no need to look)
  std::vector<double> J;
  int64_t K = 1;
  if (at < 0x1p-30) {  // J_0 = 1 - tau^2 / 4 and J_1 = tau / 2 to double precision; the tail ~ tau^2 / 4
    J = {1.0, 0.5 * at};
  } else {
    const int64_t N = int64_t(std::ceil(at + 20.0 * std::cbrt(at))) + 40;
    J.assign(size_t(N) + 2, 0.0);
    J[N] = 1.0;
    for (int64_t k = N; k >= 1; --k) {
      J[k - 1] = (2.0 * double(k) / at) * J[k] - J[k + 1];
      if (std::fabs(J[k - 1]) > 1e250)
        for (int64_t j = k - 1; j <= N; ++j) J[j] *= 1e-250;
    }
    double norm = J[0];
    for (int64_t k = 2; k <= N; k += 2) norm += 2.0 * J[k];
    for (double &v : J) v /= norm;
    double tail = 0.0;  // sum_{j > k} |J_j|, k falling
    K = N;
    for (int64_t k = N; k >= 1 && 2.0 * tail <= 0x1p-53; --k) {
      K = k;
      tail += std::fabs(J[k]);
    }
    if (K > N - 20) return false;  // (cannot happen: N lies far beyond the point where the tail is negligible)
    if (K > max_k) return false;
  }
  a.assign(2 * size_t(K + 1), 0.0);
  for (int64_t k = 0; k <= K; ++k) {
    const double j = (tau < 0 && (k & 1)) ? -J[k] : J[k], m = k == 0 ? 1.0 : 2.0;
    switch (k & 3) {  // (-i)^k
      case 0: a[2 * k] = m * j; break;
      case 1: a[2 * k + 1] = -m * j; break;
      case 2: a[2 * k] = -m * j; break;
      default: a[2 * k + 1] = m * j; break;
    }
  }
  return true;
}

// The backward pass of the adjoint gradient: psi = the state after the rotations (lx, lz, cos / sin of
// theta / 2 in cs, none the identity), lam = H psi in the same layout.  The cut of pauli_cut is walked from its
// last launch to its first, each launch's rotations from last to first; grad_dev[k] = Im <lam_{k+1}| P_k
// |psi_{k+1}> of rotation k.  psi and lam end with every rotation undone.
int run_pauli_adjoint(Buffer *psi, Buffer *lam, const std::vector<uint64_t> &lx, const std::vector<uint64_t> &lz,
                      const std::vector<double> &cs, double *grad_dev) {
  qb_ctx *c = psi->ctx;
  const uint64_t local = (1ull << psi->L) - 1ull;
  std::vector<std::pair<size_t, uint64_t>> cut;  // (first rotation, X union) of each launch
  for (size_t i0 = 0; i0 < lx.size();) {
    uint64_t ux = 0;
    const size_t i1 = pauli_cut(psi, lx, i0, &ux);
    cut.emplace_back(i0, ux);
    i0 = i1;
  }
  for (size_t l = cut.size(); l-- > 0;) {
    const size_t i0 = cut[l].first, i1 = l + 1 < cut.size() ? cut[l + 1].first : lx.size();
    if (c->nranks > 1) QB_TRY(localise_x(psi, cut[l].second));
    if (lam->perm != psi->perm) QB_TRY(relayout(lam, psi->perm));
    PauliAdjArgs args;
    memset(&args, 0, sizeof args);
    args.nrot = uint32_t(i1 - i0);
    QB_TRY(pauli_tile(psi, cut[l].second, args));
    uint64_t tile = 0;
    for (uint32_t i = 0; i < args.tile_bits; ++i) tile |= 1ull << args.tile_pos[i];
    for (size_t k = i0; k < i1; ++k) {
      const uint64_t zp = phys_mask(psi, lz[k]);
      PauliAdjParam &p = args.rot[k - i0];
      p.xt = pauli_tile_local(args, phys_mask(psi, lx[k]));
      p.zt = pauli_tile_local(args, zp);
      p.zout = zp & local & ~tile;
      p.c = cs[2 * k];
      p.s = cs[2 * k + 1];
      pauli_phase(psi, lx[k], lz[k], 1.0, 0.0, &p.fr, &p.fi);
    }
    QB_CUDA(launch_pauli_rot_adjoint(psi->amps, lam->amps, psi->L, args, c->red_partials, grad_dev + i0, c->sm_count,
                                     c->stream));
    c->stats.simple_launches++;
    c->stats.reduce_launches++;
  }
  return QB_OK;
}

}  // namespace

// ============================================================================ C ABI
extern "C" {

const char *qb_last_error(void) { return g_last_error.c_str(); }

const char *qb_version(void) { return "qubism_sv 0.2 sm_100a fused-pass"; }

int qb_init(int device, qb_ctx **out) {
  if (!out) return fail(QB_ERR_ARG, "null out");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(QB_ERR_CUDA, "no CUDA device (%s); this backend has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= ndev) return fail(QB_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
  qb_ctx *c = new qb_ctx();
  c->device = device;
  int rc = init_common(c);
  if (rc != QB_OK) {
    delete c;
    return rc;
  }
  *out = c;
  return QB_OK;
}

int qb_dist_unique_id(void *id128) {
  if (!id128) return fail(QB_ERR_ARG, "null id");
  int rc = dist_unique_id(id128);
  if (rc != QB_OK) return fail(rc, "ncclGetUniqueId failed: %s", dist_last_error());
  return QB_OK;
}

int qb_init_dist(int device, int rank, int nranks, const void *nccl_id, qb_ctx **out) {
  if (!out || !nccl_id) return fail(QB_ERR_ARG, "null argument");
  if (nranks < 1 || (nranks & (nranks - 1)) || rank < 0 || rank >= nranks)
    return fail(QB_ERR_ARG, "nranks must be a power of two and 0 <= rank < nranks");
  QB_TRY(qb_init(device, out));
  qb_ctx *c = *out;
  if (nranks == 1) return QB_OK;
  c->rank = rank;
  c->nranks = nranks;
  c->pbits = __builtin_ctz((unsigned)nranks);
  int rc = dist_create(&c->dist, device, rank, nranks, nccl_id, c->stream);
  if (rc != QB_OK) {
    std::string msg = dist_last_error();
    qb_shutdown(c);
    *out = nullptr;
    return fail(rc, "distributed init failed: %s", msg.c_str());
  }
  QB_CUDA(cudaMalloc(&c->peer_tab_dev, sizeof(double2 *) * nranks));
  return QB_OK;
}

int qb_init_group(const int *devices, int nranks, qb_ctx **out) {
  if (!devices || !out) return fail(QB_ERR_ARG, "null argument");
  if (nranks < 1 || nranks > 64 || (nranks & (nranks - 1))) return fail(QB_ERR_ARG, "nranks must be a power of two <= 64");
  for (int r = 0; r < nranks; ++r) out[r] = nullptr;
  DistGroup *grp = nranks > 1 ? dist_group_create(nranks) : nullptr;
  int rc = QB_OK;
  for (int r = 0; r < nranks && rc == QB_OK; ++r) {
    rc = qb_init(devices[r], &out[r]);
    if (rc != QB_OK || nranks == 1) continue;
    qb_ctx *c = out[r];
    c->rank = r;
    c->nranks = nranks;
    c->pbits = __builtin_ctz((unsigned)nranks);
    rc = dist_create_group(&c->dist, devices[r], r, grp);
    if (rc != QB_OK) {
      fail(rc, "rank group init failed: %s", dist_last_error());
      continue;
    }
    if (cudaMalloc(&c->peer_tab_dev, sizeof(double2 *) * nranks) != cudaSuccess) rc = fail(QB_ERR_OOM, "cudaMalloc");
    // distinct devices: the swap kernel dereferences the peers' shards directly
    for (int q = 0; q < nranks && rc == QB_OK; ++q) {
      if (devices[q] == devices[r]) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, devices[r], devices[q]);
      if (!can) {
        rc = fail(QB_ERR_UNSUPPORTED, "device %d cannot access device %d", devices[r], devices[q]);
        break;
      }
      cudaSetDevice(devices[r]);
      const cudaError_t e = cudaDeviceEnablePeerAccess(devices[q], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) rc = fail(QB_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
      (void)cudaGetLastError();
    }
  }
  if (rc != QB_OK) {
    const std::string msg = g_last_error;
    for (int r = 0; r < nranks; ++r) {
      if (out[r]) qb_shutdown(out[r]);
      out[r] = nullptr;
    }
    g_last_error = msg;
  }
  return rc;
}

int qb_shutdown(qb_ctx *c) {
  if (!c) return QB_OK;
  bool del;
  {
    std::lock_guard<std::recursive_mutex> lk(c->mu);
    if (c->closed) return QB_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    // every shard goes, whoever still holds a handle (those handles fail with QB_ERR_STATE from now on)
    for (auto *list : {&c->in_use, &c->pool})
      for (Buffer *b : *list) {
        for (qb_state *h : b->handles) h->b = nullptr;
        free_buffer_memory(b);
        delete b;
      }
    c->in_use.clear();
    c->pool.clear();
    c->graveyard.clear();
    if (c->dist) dist_destroy(c->dist);
    c->dist = nullptr;
    for (auto &pr : c->timed) {
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    for (auto e : c->event_pool) cudaEventDestroy(e);
    c->timed.clear();
    c->event_pool.clear();
    cudaFree(c->red_partials);
    cudaFree(c->red_out);
    cudaFreeHost(c->red_host);
    cudaFree(c->kq_bits_dev);
    cudaFree(c->kq_mat_dev);
    cudaFree(c->peer_tab_dev);
    if (c->stream) cudaStreamDestroy(c->stream);
    c->stream = nullptr;
    c->closed = true;
    del = c->handles == 0;  // otherwise the last qb_state_free deletes the context object
  }
  if (del) delete c;
  return QB_OK;
}

int qb_ctx_rank(const qb_ctx *c) { return c ? c->rank : -1; }
int qb_ctx_nranks(const qb_ctx *c) { return c ? c->nranks : -1; }

int qb_barrier(qb_ctx *c) {
  if (!c) return fail(QB_ERR_ARG, "null ctx");
  Guard g(c);
  QB_CUDA(cudaStreamSynchronize(c->stream));
  if (c->nranks > 1) {
    double v = 0.0;
    int rc = dist_allreduce_sum(c->dist, &v, 1, c->stream);
    if (rc != QB_OK) return fail(rc, "barrier failed: %s", dist_last_error());
    QB_TRY(drain_graveyard(c));
  }
  return QB_OK;
}

int qb_state_create(qb_ctx *ctx, int nqubits, int basis, qb_state **out) {
  if (!ctx || !out) return fail(QB_ERR_ARG, "null argument");
  Guard g(ctx);
  Buffer *s = nullptr;
  QB_TRY(new_buffer(ctx, nqubits, &s));
  cudaError_t e = cudaMemsetAsync(s->amps, 0, sizeof(double2) << s->L, ctx->stream);
  if (e == cudaSuccess && basis && ctx->rank == 0) e = launch_set_amp(s->amps, 0, 1.0, 0.0, ctx->stream);
  if (e != cudaSuccess) {
    release_buffer(s);
    return fail(QB_ERR_CUDA, "state init: %s", cudaGetErrorString(e));
  }
  if (basis) {  // |0...0>: every index bit of the one non-zero amplitude is known
    s->zmask = (nqubits >= 64) ? ~0ull : ((1ull << nqubits) - 1ull);
    s->zval = 0;
  }
  s->all_finite = true;
  return new_handle(ctx, s, 0, out);
}

int qb_state_from_host(qb_ctx *ctx, int nqubits, const qb_c64 *amps, qb_state **out) {
  if (!ctx || !amps || !out) return fail(QB_ERR_ARG, "null argument");
  Guard g(ctx);
  Buffer *s = nullptr;
  QB_TRY(new_buffer(ctx, nqubits, &s));
  cudaError_t e = cudaMemcpyAsync(s->amps, amps, sizeof(double2) << s->L, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    release_buffer(s);
    return fail(QB_ERR_CUDA, "upload: %s", cudaGetErrorString(e));
  }
  return new_handle(ctx, s, 0, out);
}

// Lazy: the clone is a second handle on the same shard at the same log position.  No flush, no
// copy, no allocation; the queued gates of the source stay queued -- for both.  Data is copied
// only if one of the two is later observed or changed while the other still needs the old value.
int qb_state_clone(qb_state *src, qb_state **out) {
  if (!src || !out) return fail(QB_ERR_ARG, "null argument");
  Guard g(src->ctx);
  QB_TRY(check_state(src));
  src->ctx->stats.clones++;
  src->b->ever_shared = true;
  return new_handle(src->ctx, src->b, src->pos, out);
}

// g #> sv in ONE call (QGate.hs:78-80): *out = a new handle holding `ops` applied to src's value;
// src stays valid (option "linear" = 1: src is consumed).
int qb_state_apply_pure(qb_state *src, const qb_op *ops, int64_t nops, qb_state **out) {
  if (!src || !out || (!ops && nops)) return fail(QB_ERR_ARG, "null argument");
  qb_state *h = nullptr;
  QB_TRY(qb_state_clone(src, &h));
  int rc = qb_submit(h, ops, nops);
  if (rc != QB_OK) {
    qb_state_free(h);
    return rc;
  }
  *out = h;
  return QB_OK;
}

// ForeignPtr finalizer: any thread, any time, also after qb_shutdown.  Never collective: in a
// sharded context the shard is only marked released here and retired when every rank has done so.
void qb_state_free(qb_state *s) {
  if (!s) return;
  drop_handle(s);
}

int qb_state_nqubits(const qb_state *s) { return s ? s->n : QB_ERR_ARG; }
uint64_t qb_state_local_len(const qb_state *s) { return s ? (1ull << (s->n - s->ctx->pbits)) : 0; }

// amplitudes [first, first + count) of a single-GPU state in INDEX order, whatever its qubit layout
static int read_in_index_order(Buffer *b, uint64_t first, uint64_t count, qb_c64 *out) {
  qb_ctx *c = b->ctx;
  bool ident = true;
  for (int q = 0; q < b->n; ++q)
    if (b->perm[q] != q) ident = false;
  if (ident) {
    QB_CUDA(cudaMemcpyAsync(out, b->amps + first, count * sizeof(double2), cudaMemcpyDeviceToHost, c->stream));
    QB_CUDA(cudaStreamSynchronize(c->stream));
    return QB_OK;
  }
  // gathered on the device into a staging buffer (<= 64 MiB at a time), then copied out
  const uint64_t piece = std::min<uint64_t>(count, 1ull << 22);
  if (piece == 0) return QB_OK;
  double2 *stage = nullptr;
  QB_CUDA(cudaMalloc(&stage, piece * sizeof(double2)));
  cudaError_t e = cudaSuccess;
  for (uint64_t off = 0; off < count && e == cudaSuccess; off += piece) {
    const uint64_t k = std::min(piece, count - off);
    e = launch_gather_logical(stage, b->amps, first + off, k, b->perm.data(), b->n, c->sm_count, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out + off, stage, k * sizeof(double2), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  }
  cudaFree(stage);
  if (e != cudaSuccess) return fail(QB_ERR_CUDA, "layout-aware read: %s", cudaGetErrorString(e));
  return QB_OK;
}

int qb_state_read_local(qb_state *s, uint64_t first, uint64_t count, qb_c64 *out) {
  if (!s || !out) return fail(QB_ERR_ARG, "null argument");
  Guard g(s->ctx);
  QB_TRY(flush_locked(s));
  const uint64_t len = 1ull << s->b->L;
  if (first > len || count > len - first) return fail(QB_ERR_ARG, "range beyond the local shard");
  if (s->ctx->nranks == 1) return read_in_index_order(s->b, first, count, out);  // (the shard IS the state)
  QB_CUDA(cudaMemcpyAsync(out, s->b->amps + first, count * sizeof(double2), cudaMemcpyDeviceToHost, s->ctx->stream));
  QB_CUDA(cudaStreamSynchronize(s->ctx->stream));
  return QB_OK;
}

int qb_state_write_local(qb_state *s, uint64_t first, uint64_t count, const qb_c64 *amps) {
  if (!s || !amps) return fail(QB_ERR_ARG, "null argument");
  Guard g(s->ctx);
  QB_TRY(check_state(s));
  const uint64_t len = 1ull << (s->n - s->ctx->pbits);
  if (first > len || count > len - first) return fail(QB_ERR_ARG, "range beyond the local shard");
  Buffer *b = s->b;
  bool shared = false;
  for (const qb_state *h : b->handles)
    if (h != s && !h->stale) shared = true;
  QB_TRY(agree_any(s->ctx, b, &shared));
  if (first == 0 && !shared) {
    // an upload starts at offset 0: whatever the state held (queued gates, layout, deferred
    // scalar, support) is being replaced
    b->log.clear();
    b->log_base = b->mat = s->pos = 0;
    for (int i = 0; i < b->n; ++i) b->perm[i] = i;
    b->pscale[0] = 1.0;
    b->pscale[1] = 0.0;
  } else {
    // continuing an upload (or writing into a state others share): the untouched amplitudes keep
    // their meaning, so they must be the true ones, in the identity layout
    QB_TRY(make_unique(s));
    b = s->b;
    QB_TRY(force_scale(b));
    if (s->ctx->nranks == 1) {  // (out-of-place passes move qubits: back to the identity layout)
      std::vector<int> ident(b->n);
      for (int i = 0; i < b->n; ++i) ident[i] = i;
      QB_TRY(relayout(b, ident));
    }
    for (int i = 0; i < b->n; ++i)
      if (b->perm[i] != i) return fail(QB_ERR_STATE, "partial upload into a state whose qubit layout has changed");
  }
  b->zmask = b->zval = 0;
  b->all_finite = false;
  QB_CUDA(cudaMemcpyAsync(b->amps + first, amps, count * sizeof(double2), cudaMemcpyHostToDevice, s->ctx->stream));
  return QB_OK;
}

int qb_state_read(qb_state *s, uint64_t first, uint64_t count, qb_c64 *out) {
  if (!s || (!out && count)) return fail(QB_ERR_ARG, "null argument");
  const uint64_t len = 1ull << s->n;
  if (first > len || count > len - first) return fail(QB_ERR_ARG, "range beyond 2^n");
  qb_ctx *c = s->ctx;
  Guard g(c);
  QB_TRY(flush_locked(s));
  Buffer *b = s->b;
  if (c->nranks == 1) return read_in_index_order(b, first, count, out);
  int rc = dist_read_logical(c->dist, b->amps, b->n, b->L, b->perm, first, count, out, c->stream);
  if (rc != QB_OK) return fail(rc, "distributed read failed: %s", dist_last_error());
  return QB_OK;
}

// ---- gates
int qb_apply_ctrl_1q(qb_state *s, const int *ctrls, int nctrl, int t, const qb_c64 m[4]) {
  if (!s || !m || (nctrl > 0 && !ctrls)) return fail(QB_ERR_ARG, "null argument");
  QB_TRY(check_qubit(s, t));
  uint64_t cm = 0;
  for (int i = 0; i < nctrl; ++i) {
    QB_TRY(check_qubit(s, ctrls[i]));
    if (ctrls[i] == t) return fail(QB_ERR_ARG, "control %d equals target", t);
    cm |= 1ull << logical_bit(s, ctrls[i]);
  }
  Guard g(s->ctx);
  LogOp o;
  o.kind = LOG_1Q;
  o.target = logical_bit(s, t);
  o.ctrl = cm;
  memcpy(o.m, m, sizeof(o.m));
  return append(s, std::move(o));
}

int qb_apply_1q(qb_state *s, int q, const qb_c64 m[4]) { return qb_apply_ctrl_1q(s, nullptr, 0, q, m); }

int qb_apply_1q_range(qb_state *s, int qlo, int qhi, const qb_c64 m[4]) {
  if (!s || !m) return fail(QB_ERR_ARG, "null argument");
  QB_TRY(check_qubit(s, qlo));
  QB_TRY(check_qubit(s, qhi));
  // onRange f l m = mconcat [onJust i m | i <- [f..l]] (QGate.hs:164-165): the factors act
  // on distinct qubits and commute; [f..l] is empty when f > l.
  for (int q = qlo; q <= qhi; ++q) QB_TRY(qb_apply_1q(s, q, m));
  return QB_OK;
}

int qb_apply_cnot(qb_state *s, int c, int t) {
  static const qb_c64 X[4] = {{0, 0}, {1, 0}, {1, 0}, {0, 0}};
  return qb_apply_ctrl_1q(s, &c, 1, t, X);
}

int qb_apply_kq(qb_state *s, const int *qs, int k, const qb_c64 *m, const int *ctrls, int nctrl) {
  if (!s || !qs || !m || (nctrl > 0 && !ctrls)) return fail(QB_ERR_ARG, "null argument");
  if (k < 1 || k > QB_MAX_KQ) return fail(QB_ERR_UNSUPPORTED, "dense blocks support 1 <= k <= %d", QB_MAX_KQ);
  if (k == 1) return qb_apply_ctrl_1q(s, ctrls, nctrl, qs[0], m);
  if (k > s->n - s->ctx->pbits) return fail(QB_ERR_UNSUPPORTED, "a %d-qubit block does not fit a shard of %d local qubits", k, s->n - s->ctx->pbits);
  uint64_t seen = 0, cm = 0;
  LogOp o;
  o.kind = LOG_KQ;
  o.k = k;
  for (int i = 0; i < k; ++i) {
    QB_TRY(check_qubit(s, qs[i]));
    o.kq_bits[i] = logical_bit(s, qs[i]);
    if (seen & (1ull << o.kq_bits[i])) return fail(QB_ERR_ARG, "repeated qubit %d", qs[i]);
    seen |= 1ull << o.kq_bits[i];
  }
  for (int i = 0; i < nctrl; ++i) {
    QB_TRY(check_qubit(s, ctrls[i]));
    const uint64_t b = 1ull << logical_bit(s, ctrls[i]);
    if (seen & b) return fail(QB_ERR_ARG, "control %d is also a target", ctrls[i]);
    cm |= b;
  }
  o.ctrl = cm;
  o.target = o.kq_bits[0];
  const double *md = reinterpret_cast<const double *>(m);
  o.kq_m = std::make_shared<const std::vector<double>>(md, md + (size_t(2) << (2 * k)));
  Guard g(s->ctx);
  return append(s, std::move(o));
}

int qb_submit(qb_state *s, const qb_op *ops, int64_t nops) {
  if (!s || (!ops && nops)) return fail(QB_ERR_ARG, "null argument");
  Guard g(s->ctx);
  for (int64_t i = 0; i < nops; ++i) {
    const qb_op &o = ops[i];
    if (o.kind == 1) {
      QB_TRY(qb_apply_cnot(s, o.ctrl[0], o.target));
    } else if (o.kind == 0) {
      if (o.nctrl < 0 || o.nctrl > 4) return fail(QB_ERR_ARG, "op %lld: nctrl out of range", (long long)i);
      QB_TRY(qb_apply_ctrl_1q(s, o.ctrl, o.nctrl, o.target, o.m));
    } else {
      return fail(QB_ERR_ARG, "op %lld: unknown kind %d", (long long)i, o.kind);
    }
  }
  return QB_OK;
}

int qb_flush(qb_state *s) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  Guard g(s->ctx);
  return flush_locked(s);
}

int qb_sync(qb_ctx *c) {
  if (!c) return fail(QB_ERR_ARG, "null ctx");
  Guard g(c);
  QB_CUDA(cudaStreamSynchronize(c->stream));
  return QB_OK;
}

// ---- measurement
int qb_sumsq(qb_state *s, int q, double *s0, double *s1) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  QB_TRY(check_qubit(s, q));
  Guard g(s->ctx);
  QB_TRY(materialise(s));
  return sumsq_buffer(s->b, logical_bit(s, q), s0, s1);
}

// the collapse itself is a log entry (it carries the weight just reduced): executed in place at the
// next observation, or fused away as a queued diagonal gate -- never a reason to copy a shared shard
static int log_collapse(qb_state *s, int lb, int bit, double weight) {
  LogOp o;
  o.kind = LOG_COLLAPSE;
  o.target = lb;
  o.ctrl = (uint64_t)bit;
  o.m[0] = weight;
  return append(s, std::move(o));
}

int qb_collapse(qb_state *s, int q, int bit) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  QB_TRY(check_qubit(s, q));
  if (bit != 0 && bit != 1) return fail(QB_ERR_ARG, "bit must be 0 or 1");
  Guard g(s->ctx);
  double s0, s1;
  QB_TRY(materialise(s));
  QB_TRY(sumsq_buffer(s->b, logical_bit(s, q), &s0, &s1));
  return log_collapse(s, logical_bit(s, q), bit, bit ? s1 : s0);
}

int qb_measure_qubit(qb_state *s, int q, double r, int *bit, double *pone) {
  if (!s || !bit) return fail(QB_ERR_ARG, "null argument");
  QB_TRY(check_qubit(s, q));
  Guard g(s->ctx);
  double s0, s1;
  QB_TRY(materialise(s));
  QB_TRY(sumsq_buffer(s->b, logical_bit(s, q), &s0, &s1));
  // the reference's pOne = sqrt(s1); when s1 == 0 it is NaN there (0/0 in collapse) and
  // `r < NaN` is False for EVERY r, so the outcome is Zero even for an out-of-range draw
  const double p = std::sqrt(s1);
  const int b = (s1 > 0.0 && r < p) ? 1 : 0;
  *bit = b;
  if (pone) *pone = p;
  return log_collapse(s, logical_bit(s, q), b, b ? s1 : s0);
}

int qb_measure_all(qb_state *s, const double *rs, int *bits) {
  if (!s || !rs || !bits) return fail(QB_ERR_ARG, "null argument");
  for (int q = 0; q < s->n; ++q) QB_TRY(qb_measure_qubit(s, q, rs[q], &bits[q], nullptr));
  return QB_OK;
}

// ---- vector space
int qb_scale(qb_state *s, qb_c64 z) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  Guard g(s->ctx);
  LogOp o;
  o.kind = LOG_SCALE;
  o.m[0] = z.re;
  o.m[1] = z.im;
  return append(s, std::move(o));
}

int qb_neg(qb_state *s) { return qb_scale(s, qb_c64{-1.0, 0.0}); }
int qb_scale_ri(qb_state *s, double re, double im) { return qb_scale(s, qb_c64{re, im}); }

static int same_shape(qb_state *a, qb_state *b) {
  if (!a || !b) return fail(QB_ERR_ARG, "null state");
  if (a->ctx != b->ctx) return fail(QB_ERR_STATE, "states live on different contexts");
  if (a->n != b->n) return fail(QB_ERR_STATE, "states have %d and %d qubits", a->n, b->n);
  return QB_OK;
}

int qb_axpy(qb_state *y, qb_c64 z, qb_state *x) {
  QB_TRY(same_shape(y, x));
  qb_ctx *c = y->ctx;
  Guard g(c);
  QB_TRY(flush_locked(x));
  QB_TRY(make_unique(y));   // (x == y, or a clone of it: y moves to its own shard, x keeps the old one)
  QB_TRY(flush_locked(x));  // (no-op unless the split moved things)
  QB_TRY(force_scale(y->b));
  Buffer *yb = y->b, *xb = x->b;
  if (yb->perm != xb->perm) QB_TRY(relayout(xb, yb->perm));
  const double zz[2] = {z.re, z.im};
  QB_CUDA(launch_axpy(yb->amps, xb->amps, 1ull << yb->L, zz, c->sm_count, c->stream));
  // the sum is non-zero only where one of the operands is: keep the bits both know with the same value
  yb->zmask = yb->zmask & xb->zmask & ~(yb->zval ^ xb->zval);
  yb->zval &= yb->zmask;
  yb->all_finite = yb->all_finite && xb->all_finite && std::isfinite(z.re) && std::isfinite(z.im);
  if (!yb->all_finite) yb->zmask = yb->zval = 0;
  return QB_OK;
}

int qb_axpy_ri(qb_state *y, double re, double im, qb_state *x) { return qb_axpy(y, qb_c64{re, im}, x); }

int qb_dotc(qb_state *a, qb_state *b, qb_c64 *out) {
  QB_TRY(same_shape(a, b));
  if (!out) return fail(QB_ERR_ARG, "null out");
  qb_ctx *c = a->ctx;
  Guard g(c);
  QB_TRY(flush_locked(a));
  QB_TRY(flush_locked(b));
  QB_TRY(flush_locked(a));  // (b's flush may have split a lineage the two share; idempotent)
  Buffer *ab = a->b, *bb = b->b;
  if (ab->perm != bb->perm) QB_TRY(relayout(bb, ab->perm));
  QB_CUDA(launch_dotc(ab->amps, bb->amps, 1ull << ab->L, c->red_partials, c->red_out, c->sm_count, c->stream));
  c->stats.reduce_launches += 2;
  QB_CUDA(cudaMemcpyAsync(c->red_host, c->red_out, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  QB_CUDA(cudaStreamSynchronize(c->stream));
  double v[2] = {c->red_host[0], c->red_host[1]};
  if (c->nranks > 1) {
    int rc = dist_allreduce_sum(c->dist, v, 2, c->stream);
    if (rc != QB_OK) return fail(rc, "allreduce failed: %s", dist_last_error());
  }
  out->re = v[0];
  out->im = v[1];
  return QB_OK;
}

int qb_norm2(qb_state *s, double *out) {
  if (!s || !out) return fail(QB_ERR_ARG, "null argument");
  Guard g(s->ctx);
  double s0 = 0, s1 = 0;
  QB_TRY(materialise(s));
  QB_TRY(sumsq_buffer(s->b, -1, &s0, &s1));
  *out = std::sqrt(s0 + s1);
  return QB_OK;
}

// ---- Pauli expectation values
// Sharded states: an X / Y on a global qubit pairs amplitudes of two ranks, so the qubits of the logical
// X mask lx are brought into the shard first.  One multi-bit swap through make_local; where its victims
// carried one of those qubits out again (the victim choice knows only the qubits it brings in), a
// relayout trades it for a local qubit outside lx.
static int localise_x(Buffer *b, uint64_t lx) {
  if (!(phys_mask(b, lx) >> b->L)) return QB_OK;
  if (__builtin_popcountll(lx) > b->L)
    return fail(QB_ERR_UNSUPPORTED, "a Pauli string with X / Y on %d qubits does not fit a shard of %d qubits",
                __builtin_popcountll(lx), b->L);
  std::vector<HostOp> ops;
  for (uint64_t m = lx; m; m &= m - 1) {
    HostOp h;
    h.target = __builtin_ctzll(m);
    ops.push_back(h);
  }
  std::vector<const HostOp *> pending;
  for (const HostOp &h : ops) pending.push_back(&h);
  QB_TRY(make_local(b, pending));
  if (!(phys_mask(b, lx) >> b->L)) return QB_OK;
  std::vector<int> want = b->perm, logical_of(b->n);
  for (int q = 0; q < b->n; ++q) logical_of[want[q]] = q;
  int spare = b->L - 1;  // highest local bit not holding a qubit of lx
  for (uint64_t m = lx; m; m &= m - 1) {
    const int q = __builtin_ctzll(m);
    if (want[q] < b->L) continue;
    while ((lx >> logical_of[spare]) & 1ull) --spare;  // (popc(lx) <= L: one is left)
    const int o = logical_of[spare];
    std::swap(want[q], want[o]);
    logical_of[want[q]] = q;
    logical_of[want[o]] = o;
  }
  return relayout(b, want);
}

int qb_expect_pauli(qb_state *s, const uint64_t *xmask, const uint64_t *zmask, int64_t nterms, double *out) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  if (nterms < 0) return fail(QB_ERR_ARG, "nterms %lld < 0", (long long)nterms);
  if (nterms == 0) return QB_OK;
  if (!xmask || !zmask || !out) return fail(QB_ERR_ARG, "null argument");
  const int n = s->n;
  for (int64_t t = 0; t < nterms; ++t)
    if ((xmask[t] | zmask[t]) >> n) return fail(QB_ERR_ARG, "term %lld names a qubit >= %d", (long long)t, n);
  qb_ctx *c = s->ctx;
  Guard g(c);
  QB_TRY(materialise(s));
  Buffer *b = s->b;
  if (!(std::isfinite(b->pscale[0]) && std::isfinite(b->pscale[1]))) QB_TRY(force_scale(b));  // NaN / inf must reach the data
  auto logical = [n](uint64_t m) {  // reference qubit q is logical bit n - 1 - q
    uint64_t r = 0;
    for (; m; m &= m - 1) r |= 1ull << (n - 1 - __builtin_ctzll(m));
    return r;
  };
  std::vector<uint64_t> lx(nterms), lz(nterms);
  std::map<uint64_t, std::vector<int64_t>> groups;  // logical X mask -> its terms in caller order (same on every rank)
  for (int64_t t = 0; t < nterms; ++t) {
    lx[t] = logical(xmask[t]);
    lz[t] = logical(zmask[t]);
    out[t] = 0.0;
    // an X on a qubit of known value pairs every non-zero amplitude with a zero one: exactly 0
    if (c->opt.support && (lx[t] & b->zmask)) continue;
    groups[lx[t]].push_back(t);
  }
  const double g2 = b->pscale[0] * b->pscale[0] + b->pscale[1] * b->pscale[1];  // the pending scalar, arithmetically
  const uint64_t local = (1ull << b->L) - 1ull;
  for (const auto &grp : groups) {
    const uint64_t x = grp.first;
    const std::vector<int64_t> &terms = grp.second;
    if (c->nranks > 1) QB_TRY(localise_x(b, x));
    const uint64_t xp = phys_mask(b, x);
    const uint64_t lo = xp ? (1ull << (63 - __builtin_clzll(xp))) - 1ull : ~0ull;
    for (size_t k0 = 0; k0 < terms.size(); k0 += kExpMaxTerms) {
      const size_t k1 = std::min(terms.size(), k0 + size_t(kExpMaxTerms));
      ExpTerms et;
      memset(&et, 0, sizeof et);
      et.xp = xp;
      et.lo_mask = lo;
      int64_t order[kExpMaxTerms];
      double post[kExpMaxTerms];
      for (int odd = 0; odd < 2; ++odd)  // real parts (even popc(x & z)) first
        for (size_t k = k0; k < k1; ++k)
          if ((__builtin_popcountll(x & lz[terms[k]]) & 1) == odd) order[et.nterms++] = terms[k];
      for (int j = 0; j < et.nterms; ++j) {
        const int64_t t = order[j];
        const int ph = __builtin_popcountll(x & lz[t]) & 3;  // P = i^ph X^x Z^z (Y = i X Z)
        if (!(ph & 1)) et.neven = j + 1;
        const uint64_t zp = phys_mask(b, lz[t]);
        et.zp[j] = zp & local;
        for (uint32_t u = 0; u < (uint32_t)kExpU; ++u) {
          const uint64_t p = uint64_t(u) << kExpUShift, i = (p & lo) | ((p & ~lo) << 1);
          if (__builtin_popcountll(i & et.zp[j]) & 1) et.rflip[j] |= 1u << u;
        }
        // Re(i^ph (w + (-1)^ph conj w)) = 2 * (+1, -1, -1, +1)[ph] * (Re w | Im w) over a pair; one
        // amplitude (xp == 0) counts once.  Z on global qubits: this rank's value of them
        double f = (ph == 1 || ph == 2) ? -1.0 : 1.0;
        if (xp) f *= 2.0;
        if (__builtin_popcountll((zp >> b->L) & uint64_t(c->rank)) & 1) f = -f;
        post[j] = f;
      }
      QB_CUDA(launch_expect_pauli(b->amps, b->L, et, c->red_partials, c->red_out, c->sm_count, c->stream));
      c->stats.reduce_launches += 2;
      QB_CUDA(cudaMemcpyAsync(c->red_host, c->red_out, sizeof(double) * et.nterms, cudaMemcpyDeviceToHost, c->stream));
      QB_CUDA(cudaStreamSynchronize(c->stream));
      double v[kExpMaxTerms];
      for (int j = 0; j < et.nterms; ++j) v[j] = c->red_host[j] * post[j];
      if (c->nranks > 1) {
        int rc = dist_allreduce_sum(c->dist, v, et.nterms, c->stream);
        if (rc != QB_OK) return fail(rc, "allreduce failed: %s", dist_last_error());
      }
      for (int j = 0; j < et.nterms; ++j) out[order[j]] = g2 != 1.0 ? v[j] * g2 : v[j];
    }
  }
  return QB_OK;
}

// ---- Pauli rotations
// The checks of count strings for the tile kernels, made before anything is queued or allocated: the masks
// name qubits of s, the values v[t * nv .. t * nv + nv) are finite, and X / Y fit the rotation tile.
static int check_pauli_strings(const qb_state *s, const char *what, const char *value, const uint64_t *xmask,
                               const uint64_t *zmask, const double *v, int nv, int64_t count) {
  const int n = s->n, T = std::min(kPauliTileBits, s->n - s->ctx->pbits);
  for (int64_t t = 0; t < count; ++t) {
    if ((xmask[t] | zmask[t]) >> n) return fail(QB_ERR_ARG, "%s %lld names a qubit >= %d", what, (long long)t, n);
    for (int j = 0; j < nv; ++j)
      if (!std::isfinite(v[t * nv + j])) return fail(QB_ERR_ARG, "%s %lld: %s is not finite", what, (long long)t, value);
    if (__builtin_popcountll(xmask[t]) > T)
      return fail(QB_ERR_UNSUPPORTED, "%s %lld has X / Y on %d qubits; at most %d fit the rotation tile", what,
                  (long long)t, __builtin_popcountll(xmask[t]), T);
  }
  return QB_OK;
}

// append rotations (already checked) to s's lineage
static int log_pauli_rots(qb_state *s, const uint64_t *xmask, const uint64_t *zmask, const double *theta, int64_t nrot) {
  for (int64_t t = 0; t < nrot; ++t) {
    LogOp o;
    o.kind = LOG_PAULI;
    o.ctrl = logical_mask(s->n, xmask[t]);
    o.pz = logical_mask(s->n, zmask[t]);
    o.m[0] = std::cos(0.5 * theta[t]);
    o.m[1] = std::sin(0.5 * theta[t]);
    QB_TRY(append(s, std::move(o)));
  }
  return QB_OK;
}

int qb_apply_pauli_rot(qb_state *s, const uint64_t *xmask, const uint64_t *zmask, const double *theta, int64_t nrot) {
  if (!s) return fail(QB_ERR_ARG, "null state");
  if (nrot < 0) return fail(QB_ERR_ARG, "nrot %lld < 0", (long long)nrot);
  if (nrot == 0) return QB_OK;
  if (!xmask || !zmask || !theta) return fail(QB_ERR_ARG, "null argument");
  QB_TRY(check_pauli_strings(s, "rotation", "theta", xmask, zmask, theta, 1, nrot));
  Guard g(s->ctx);
  QB_TRY(check_state(s));
  return log_pauli_rots(s, xmask, zmask, theta, nrot);
}

// ---- Pauli sums
int qb_pauli_sum(qb_state *src, const uint64_t *xmask, const uint64_t *zmask, const qb_c64 *coef, int64_t nterms,
                 qb_state **out) {
  if (!src || !out) return fail(QB_ERR_ARG, "null argument");
  if (nterms < 0) return fail(QB_ERR_ARG, "nterms %lld < 0", (long long)nterms);
  if (nterms > 0 && (!xmask || !zmask || !coef)) return fail(QB_ERR_ARG, "null argument");
  static_assert(sizeof(qb_c64) == 2 * sizeof(double), "qb_c64 is (re, im)");
  QB_TRY(check_pauli_strings(src, "term", "coefficient", xmask, zmask, reinterpret_cast<const double *>(coef), 2, nterms));
  qb_ctx *c = src->ctx;
  Guard g(c);
  QB_TRY(materialise(src));
  Buffer *b = src->b;
  if (!(std::isfinite(b->pscale[0]) && std::isfinite(b->pscale[1]))) QB_TRY(force_scale(b));  // NaN / inf must reach the data
  Buffer *ob = nullptr;
  QB_TRY(new_buffer(c, src->n, &ob));
  std::vector<uint64_t> lx(nterms), lz(nterms);
  std::vector<double> cf(2 * nterms);
  uint64_t xunion = 0;
  for (int64_t t = 0; t < nterms; ++t) {
    lx[t] = logical_mask(src->n, xmask[t]);
    lz[t] = logical_mask(src->n, zmask[t]);
    xunion |= lx[t];
    cf[2 * t] = coef[t].re * b->pscale[0] - coef[t].im * b->pscale[1];  // the pending scalar rides on the coefficients
    cf[2 * t + 1] = coef[t].re * b->pscale[1] + coef[t].im * b->pscale[0];
  }
  int rc = QB_OK;
  if (nterms == 0) {
    ob->perm = b->perm;
    if (cudaMemsetAsync(ob->amps, 0, sizeof(double2) << ob->L, c->stream) != cudaSuccess) rc = fail(QB_ERR_CUDA, "zero fill");
  } else {
    rc = run_pauli_sum(b, ob, lx, lz, cf, nullptr, nullptr);
  }
  if (rc != QB_OK) {
    release_buffer(ob);
    return rc;
  }
  // P_t moves amplitude j to j ^ x_t: what the source knows outside every X mask still holds (§3.3b)
  ob->all_finite = b->all_finite;
  ob->zmask = ob->all_finite ? b->zmask & ~xunion : 0;
  ob->zval = b->zval & ob->zmask;
  return new_handle(c, ob, 0, out);
}

// ---- adjoint gradients of Pauli-sum energies
int qb_pauli_rot_grad(qb_state *s, const uint64_t *rx, const uint64_t *rz, const double *theta, int64_t nrot,
                      const uint64_t *hx, const uint64_t *hz, const double *hcoef, int64_t nterms, double *energy,
                      double *grad) {
  if (!s || !energy) return fail(QB_ERR_ARG, "null argument");
  if (nrot < 0) return fail(QB_ERR_ARG, "nrot %lld < 0", (long long)nrot);
  if (nterms < 0) return fail(QB_ERR_ARG, "nterms %lld < 0", (long long)nterms);
  if (nrot > 0 && (!rx || !rz || !theta || !grad)) return fail(QB_ERR_ARG, "null argument");
  if (nterms > 0 && (!hx || !hz || !hcoef)) return fail(QB_ERR_ARG, "null argument");
  QB_TRY(check_pauli_strings(s, "rotation", "theta", rx, rz, theta, 1, nrot));
  QB_TRY(check_pauli_strings(s, "term", "coefficient", hx, hz, hcoef, 1, nterms));
  qb_ctx *c = s->ctx;
  Guard g(c);
  QB_TRY(check_state(s));
  *energy = 0.0;
  for (int64_t k = 0; k < nrot; ++k) grad[k] = 0.0;
  if (nterms == 0) return QB_OK;  // H = 0
  // psi: a copy of s that owns its shard (s keeps its value and its handle, also with option "linear")
  qb_state *w = nullptr;
  QB_TRY(qb_state_clone(s, &w));
  Buffer *lam = nullptr;
  double *dres = nullptr;
  auto done = [&](int rc) {
    if (dres) cudaFree(dres);
    if (lam) release_buffer(lam);
    drop_handle(w);
    return rc;
  };
  int rc = split_off(w, false);
  if (rc == QB_OK) rc = log_pauli_rots(w, rx, rz, theta, nrot);
  if (rc == QB_OK) rc = materialise(w);
  if (rc != QB_OK) return done(rc);
  Buffer *psi = w->b;
  if (!(std::isfinite(psi->pscale[0]) && std::isfinite(psi->pscale[1]))) {
    if ((rc = force_scale(psi)) != QB_OK) return done(rc);
  }
  if ((rc = new_buffer(c, s->n, &lam)) != QB_OK) return done(rc);
  // the rotations the backward pass walks: every one but the identity string (a global phase, gradient 0)
  std::vector<int64_t> idx;
  std::vector<uint64_t> lx, lz, hlx(nterms), hlz(nterms);
  std::vector<double> cs, hc(2 * nterms);
  for (int64_t k = 0; k < nrot; ++k)
    if (rx[k] | rz[k]) {
      idx.push_back(k);
      lx.push_back(logical_mask(s->n, rx[k]));
      lz.push_back(logical_mask(s->n, rz[k]));
      cs.push_back(std::cos(0.5 * theta[k]));
      cs.push_back(std::sin(0.5 * theta[k]));
    }
  for (int64_t t = 0; t < nterms; ++t) {
    hlx[t] = logical_mask(s->n, hx[t]);
    hlz[t] = logical_mask(s->n, hz[t]);
    hc[2 * t] = hcoef[t];
    hc[2 * t + 1] = 0.0;
  }
  const size_t nres = idx.size() + size_t(nterms);  // gradient of each walked rotation, energy of each sum launch
  if (cudaMalloc(&dres, sizeof(double) * nres) != cudaSuccess) {
    (void)cudaGetLastError();
    dres = nullptr;
    return done(fail(QB_ERR_OOM, "gradient scratch"));
  }
  int nl = 0;
  if (cudaMemsetAsync(dres, 0, sizeof(double) * nres, c->stream) != cudaSuccess) return done(fail(QB_ERR_CUDA, "memset"));
  if ((rc = run_pauli_sum(psi, lam, hlx, hlz, hc, dres + idx.size(), &nl)) != QB_OK) return done(rc);
  if ((rc = run_pauli_adjoint(psi, lam, lx, lz, cs, dres)) != QB_OK) return done(rc);
  std::vector<double> v(idx.size() + 1);
  std::vector<double> host(nres);
  if (cudaMemcpyAsync(host.data(), dres, sizeof(double) * nres, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
      cudaStreamSynchronize(c->stream) != cudaSuccess)
    return done(fail(QB_ERR_CUDA, "gradient read-back"));
  for (size_t i = 0; i < idx.size(); ++i) v[i] = host[i];
  double e = 0.0;
  for (int l = 0; l < nl; ++l) e += host[idx.size() + l];  // (launch order: fixed)
  v[idx.size()] = e;
  if (c->nranks > 1) {
    rc = dist_allreduce_sum(c->dist, v.data(), (int)v.size(), c->stream);
    if (rc != QB_OK) return done(fail(rc, "allreduce failed: %s", dist_last_error()));
  }
  // the pending scalar z of psi, arithmetically: psi = z psi_dev, so both scale by |z|^2
  const double g2 = psi->pscale[0] * psi->pscale[0] + psi->pscale[1] * psi->pscale[1];
  for (size_t i = 0; i < idx.size(); ++i) grad[idx[i]] = v[i] * g2;
  *energy = v[idx.size()] * g2;
  return done(QB_OK);
}

// ---- exact time evolution under Pauli sums
constexpr int64_t kEvolveMaxSteps = int64_t(1) << 20;  // bounds the coefficient table and the time of one call

int qb_pauli_evolve(qb_state *s, const uint64_t *hx, const uint64_t *hz, const double *hcoef, int64_t nterms, double t,
                    int64_t *nsteps) {
  if (nsteps) *nsteps = 0;
  if (!s) return fail(QB_ERR_ARG, "null state");
  if (nterms < 0) return fail(QB_ERR_ARG, "nterms %lld < 0", (long long)nterms);
  if (nterms > 0 && (!hx || !hz || !hcoef)) return fail(QB_ERR_ARG, "null argument");
  if (!std::isfinite(t)) return fail(QB_ERR_ARG, "t is not finite");
  QB_TRY(check_pauli_strings(s, "term", "coefficient", hx, hz, hcoef, 1, nterms));
  qb_ctx *c = s->ctx;
  Guard g(c);
  QB_TRY(check_state(s));
  if (t == 0.0 || nterms == 0) return QB_OK;
  // H = cid I + h: equal strings merged (caller order), zero coefficients dropped, the identity apart
  double cid = 0.0, r = 0.0;
  std::vector<uint64_t> lx, lz;
  std::vector<double> cf;
  std::map<std::pair<uint64_t, uint64_t>, size_t> seen;
  for (int64_t k = 0; k < nterms; ++k) {
    if (!(hx[k] | hz[k])) {
      cid += hcoef[k];
      continue;
    }
    const auto it = seen.emplace(std::make_pair(hx[k], hz[k]), lx.size());
    if (it.second) {
      lx.push_back(logical_mask(s->n, hx[k]));
      lz.push_back(logical_mask(s->n, hz[k]));
      cf.push_back(hcoef[k]);
      cf.push_back(0.0);
    } else {
      cf[2 * it.first->second] += hcoef[k];
    }
  }
  uint64_t xunion = 0;
  size_t nh = 0;
  for (size_t k = 0; k < lx.size(); ++k) {
    if (cf[2 * k] == 0.0) continue;
    r += std::fabs(cf[2 * k]);
    xunion |= lx[k];
    lx[nh] = lx[k];
    lz[nh] = lz[k];
    cf[2 * nh] = cf[2 * k];
    ++nh;
  }
  lx.resize(nh);
  lz.resize(nh);
  cf.resize(2 * nh);
  const double tc = t * cid;
  if (!std::isfinite(tc)) return fail(QB_ERR_ARG, "t times the identity coefficient is not finite");
  const double phase[2] = {std::cos(tc), -std::sin(tc)};  // e^{-itc}
  if (r == 0.0) {  // H = cid I: a global phase, deferred like qb_scale
    if (phase[0] == 1.0 && phase[1] == 0.0) return QB_OK;
    LogOp o;
    o.kind = LOG_SCALE;
    o.m[0] = phase[0];
    o.m[1] = phase[1];
    return append(s, std::move(o));
  }
  const double tau = t * r;
  std::vector<double> a;
  if (!std::isfinite(tau) || !cheb_coefficients(tau, kEvolveMaxSteps, a))
    return fail(QB_ERR_ARG, "|t| * sum |h| = %g needs more than %lld Chebyshev steps", std::fabs(tau),
                (long long)kEvolveMaxSteps);
  const int64_t K = int64_t(a.size() / 2) - 1;
  // two temporaries before anything is touched: out of memory leaves s as it was
  Buffer *tmp[2] = {nullptr, nullptr};
  auto done = [&](int rc) {
    for (Buffer *b : tmp)
      if (b) release_buffer(b);
    return rc;
  };
  for (Buffer *&b : tmp) {
    const int rc = new_buffer(c, s->n, &b);
    if (rc != QB_OK) return done(rc);
  }
  // s's shard is about to hold T_k: nobody else may see it (a clone of the old value moves to a copy)
  int rc = make_unique(s);
  if (rc != QB_OK) return done(rc);
  Buffer *sb = s->b;
  if (!(std::isfinite(sb->pscale[0]) && std::isfinite(sb->pscale[1]))) {  // NaN / inf must reach the data
    if ((rc = force_scale(sb)) != QB_OK) return done(rc);
  }
  const PauliTerms h(std::move(lx), std::move(lz), std::move(cf));
  // cur = T_{k-1}, prev = T_{k-2} (becomes T_k), acc = sum_{j < k} a_j T_j; the pending scalar rides along
  Buffer *cur = sb, *prev = tmp[0], *acc = tmp[1];
  for (int64_t k = 1; k <= K && rc == QB_OK; ++k) {
    rc = run_pauli_cheb_step(cur, prev, acc, h, 1.0 / r, k, &a[0], &a[2 * k]);
    std::swap(cur, prev);
  }
  if (rc != QB_OK) {
    sb->broken = true;
    sb->broken_why = g_last_error;
    return done(rc);
  }
  // s takes acc's shard (and its peer table); tmp[1] leaves with s's old one
  std::swap(sb->amps, acc->amps);
  std::swap(sb->peers, acc->peers);
  sb->perm = acc->perm;
  const double pr = sb->pscale[0] * phase[0] - sb->pscale[1] * phase[1];
  sb->pscale[1] = sb->pscale[0] * phase[1] + sb->pscale[1] * phase[0];
  sb->pscale[0] = pr;
  // every T_k(H') moves amplitude j only to j ^ (X masks of h): what s knew outside them still holds (§3.3b)
  sb->zmask = sb->all_finite ? sb->zmask & ~xunion : 0;
  sb->zval &= sb->zmask;
  if (nsteps) *nsteps = K;
  return done(QB_OK);
}

int qb_normalize(qb_state *s) {
  double nrm = 0;
  QB_TRY(qb_norm2(s, &nrm));
  return qb_scale(s, qb_c64{1.0 / nrm, 0.0});  // 0 -> inf -> 0 * inf = NaN, as LA.normalize
}

int qb_tensor(qb_state *a, qb_state *b, qb_state **out) {
  if (!a || !b || !out) return fail(QB_ERR_ARG, "null argument");
  if (a->ctx != b->ctx) return fail(QB_ERR_STATE, "states live on different contexts");
  qb_ctx *c = a->ctx;
  Guard g(c);
  QB_TRY(flush_locked(a));
  QB_TRY(flush_locked(b));
  QB_TRY(flush_locked(a));
  Buffer *ab = a->b, *bb = b->b;
  {
    // both operands in the identity layout (global<->local swaps and out-of-place passes move qubits).
    // Sharded: a's qubits are the high ones (StateVec.hs:98-100), so rank r's shard of the product is
    // (r's shard of a) x (ALL of b): b is read through the peers' mapped shards, a local fill
    // otherwise (SURVEY.md 8e)
    std::vector<int> ident(ab->n);
    for (int i = 0; i < ab->n; ++i) ident[i] = i;
    if (ab->perm != ident) QB_TRY(relayout(ab, ident));
    ident.resize(bb->n);
    for (int i = 0; i < bb->n; ++i) ident[i] = i;
    if (bb->perm != ident) QB_TRY(relayout(bb, ident));
    if (c->nranks > 1 && (int)bb->peers.size() != c->nranks)
      return fail(QB_ERR_UNSUPPORTED, "tensor of distributed states needs peer-mapped shards (CUDA IPC or a rank group)");
  }
  Buffer *s = nullptr;
  QB_TRY(new_buffer(c, ab->n + bb->n, &s));
  cudaError_t e;
  if (c->nranks > 1) {
    e = cudaMemcpyAsync(c->peer_tab_dev, bb->peers.data(), sizeof(double2 *) * c->nranks, cudaMemcpyHostToDevice, c->stream);
    // every rank's b must be final before anyone reads it, and nobody may change b before all are done
    if (e == cudaSuccess && qb_barrier(c) != QB_OK) e = cudaErrorUnknown;
    if (e == cudaSuccess)
      e = launch_tensor_sharded(s->amps, ab->amps, c->peer_tab_dev, ab->L, bb->n, bb->L, c->sm_count, c->stream);
    if (e == cudaSuccess && qb_barrier(c) != QB_OK) e = cudaErrorUnknown;
  } else {
    e = launch_tensor(s->amps, ab->amps, bb->amps, ab->n, bb->n, c->sm_count, c->stream);
  }
  if (e != cudaSuccess) {
    release_buffer(s);
    return fail(QB_ERR_CUDA, "tensor: %s", cudaGetErrorString(e));
  }
  // a's bits are the high ones (StateVec.hs:98-100); a known zero stays zero only against finite factors
  s->all_finite = ab->all_finite && bb->all_finite;
  if (s->all_finite) {
    s->zmask = (ab->zmask << bb->n) | bb->zmask;
    s->zval = (ab->zval << bb->n) | bb->zval;
  }
  return new_handle(c, s, 0, out);
}

// ---- introspection
int qb_get_stats(const qb_ctx *cc, qb_stats *out) {
  if (!cc || !out) return fail(QB_ERR_ARG, "null argument");
  qb_ctx *c = const_cast<qb_ctx *>(cc);
  Guard g(c);
  QB_TRY(resolve_timed(c));
  *out = c->stats;
  const JitStats js = jit_stats();  // (process-wide counters: one process per GPU; reset = new baseline)
  out->jit_compiled = js.compiled - c->jit_base_compiled;
  out->jit_launches = js.launches - c->jit_base_launches;
  out->jit_compile_ms = js.compile_ms - c->jit_base_ms;
  return QB_OK;
}

int qb_reset_stats(qb_ctx *c) {
  if (!c) return fail(QB_ERR_ARG, "null ctx");
  Guard g(c);
  QB_TRY(resolve_timed(c));
  c->stats = qb_stats{};
  const JitStats js = jit_stats();
  c->jit_base_compiled = js.compiled;
  c->jit_base_launches = js.launches;
  c->jit_base_ms = js.compile_ms;
  return QB_OK;
}

void *qb_ctx_stream(qb_ctx *c) { return c ? (void *)c->stream : nullptr; }

int qb_set_option(qb_ctx *c, const char *name, int64_t value) {
  if (!c || !name) return fail(QB_ERR_ARG, "null argument");
  std::lock_guard<std::recursive_mutex> lk(c->mu);
  if (!strcmp(name, "linear")) {
    c->linear = value ? 1 : 0;
    return QB_OK;
  }
  if (!strcmp(name, "pool")) {
    if (value < 0 || value > 8) return fail(QB_ERR_ARG, "bad option pool=%lld", (long long)value);
    c->pool_max = (int)value;
    return QB_OK;
  }
  if (!set_opt(c->opt, name, value)) return fail(QB_ERR_ARG, "bad option %s=%lld", name, (long long)value);
  return QB_OK;
}

int64_t qb_get_option(const qb_ctx *c, const char *name) {
  if (!c || !name) return QB_ERR_ARG;
  if (!strcmp(name, "linear")) return c->linear;
  if (!strcmp(name, "pool")) return c->pool_max;
  return get_opt(c->opt, name);
}

int qb_jit_sync(qb_ctx *c) {
  if (!c) return fail(QB_ERR_ARG, "null ctx");
  jit_wait();
  return QB_OK;
}

const char *qb_jit_toolchain(void) {
  static thread_local std::string s;
  s = jit_toolchain();
  return s.c_str();
}

int qb_jit_compile_check(const char *src, int64_t *cubin_bytes) {
  if (!src) return fail(QB_ERR_ARG, "null argument");
  std::string why;
  size_t nbytes = 0;
  if (!jit_compile_only(src, &nbytes, &why)) {
    const bool missing = why.find("libnvrtc") != std::string::npos;
    return fail(missing ? QB_ERR_UNSUPPORTED : QB_ERR_CUDA, "%s", why.c_str());
  }
  if (cubin_bytes) *cubin_bytes = (int64_t)nbytes;
  return QB_OK;
}

int64_t qb_plan_describe(int nlocal, const qb_op *ops, int64_t nops, const char *options, char *buf,
                         int64_t buflen) {
  if (nlocal < 1 || nlocal > 62 || (!ops && nops)) return fail(QB_ERR_ARG, "bad argument");
  PlanOptions opt;
  if (options) {
    std::string o(options);
    size_t pos = 0;
    while (pos < o.size()) {
      size_t e = o.find(',', pos);
      if (e == std::string::npos) e = o.size();
      std::string kv = o.substr(pos, e - pos);
      size_t eq = kv.find('=');
      if (eq != std::string::npos && !set_opt(opt, kv.substr(0, eq), strtoll(kv.c_str() + eq + 1, nullptr, 10)))
        return fail(QB_ERR_ARG, "bad option %s", kv.c_str());
      pos = e + 1;
    }
  }
  OpQueue q;
  q.reset(nlocal, opt.peephole != 0, opt.rot != 0);
  for (int64_t i = 0; i < nops; ++i) {
    const qb_op &o = ops[i];
    uint64_t cm = 0;
    if (o.target < 0 || o.target >= nlocal) return fail(QB_ERR_ARG, "op %lld: bad target", (long long)i);
    const int nc = o.kind == 1 ? 1 : o.nctrl;
    for (int k = 0; k < nc; ++k) {
      if (o.ctrl[k] < 0 || o.ctrl[k] >= nlocal || o.ctrl[k] == o.target)
        return fail(QB_ERR_ARG, "op %lld: bad control", (long long)i);
      cm |= 1ull << (nlocal - 1 - o.ctrl[k]);
    }
    static const double X[8] = {0, 0, 1, 0, 1, 0, 0, 0};
    q.push_1q(nlocal - 1 - o.target, cm, o.kind == 1 ? X : reinterpret_cast<const double *>(o.m));
  }
  int T, R;
  effective_tile(opt, nlocal, T, R);
  std::string text;
  char head[160];
  snprintf(head, sizeof head, "submitted=%llu folded=%llu gscale=(%.17g,%.17g)\n", (unsigned long long)q.submitted,
           (unsigned long long)q.folded, q.gscale[0], q.gscale[1]);
  text = head;
  if (T == 0) {
    text += "unfused (shard smaller than a tile)\n";
  } else {
    opt.tile_bits = T;
    opt.reg_bits = R;
    if (!opt.fuse) opt.max_pass_gates = 1;
    if (opt.oop && opt.low_bits < opt.oop_low_bits) opt.low_bits = std::min(opt.oop_low_bits, T);  // (as a flush does)
    std::vector<PhysOp> pops;
    for (const auto &h : q.ops) {
      if (h.dead) continue;
      PhysOp p;
      p.type = h.type;
      p.target = h.target;
      p.ctrl = h.ctrl;
      memcpy(p.m, h.m, sizeof(h.m));
      pops.push_back(p);
    }
    PlanResult r = plan_passes(pops, nlocal, 0, opt, q.gscale);
    text += describe_plan(r);
  }
  if (buf && buflen > 0) {
    const size_t ncopy = std::min<size_t>(text.size(), (size_t)buflen - 1);
    memcpy(buf, text.data(), ncopy);
    buf[ncopy] = 0;
  }
  return (int64_t)text.size() + 1;
}

}  // extern "C"
