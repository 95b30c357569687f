// Host-callable launchers for the kernels in qb_kernels.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace qb {

bool fused_variant_supported(int tile_bits, int reg_bits);

// One fused pass: `blob` is the planner's HOST DevPass blob (header + gates); it is passed to
// the kernel by value as a __grid_constant__ parameter.  Persistent grid = SMs x resident
// CTAs/SM (capped at ntiles).
// src: where the tiles are READ (null / == amps: in place; else the pass doubles as the copy of
// a copy-on-write: every tile must be visited).
cudaError_t launch_fused_pass(double2 *amps, const double2 *src, const uint8_t *blob, uint32_t blob_bytes, int tile_bits,
                              int reg_bits, uint64_t ntiles, int sm_count, cudaStream_t stream, int *grid_out);

cudaError_t launch_simple_gate(double2 *amps, int local_bits, int tbit, uint64_t cmask, uint64_t rank_bits,
                               uint32_t type, const double m[8], int sm_count, cudaStream_t stream);
cudaError_t launch_simple_diag(double2 *amps, int local_bits, uint64_t tmask, uint64_t cmask, uint64_t rank_bits,
                               const double d0[2], const double d1[2], int sm_count, cudaStream_t stream);
cudaError_t launch_simple_kq(double2 *amps, int local_bits, int k, const int *bits_sorted_dev,
                             const int *bits_order_dev, const double2 *mat_dev, uint64_t cmask, uint64_t rank_bits,
                             int sm_count, cudaStream_t stream);

// In-place exchange with one peer GPU over IPC-mapped memory: free indices [t_begin, t_end) of the
// 2^(L-k) elements whose swapped local bits (swapped_mask) equal my_place / peer_place.
cudaError_t launch_peer_swap(double2 *mine, double2 *peer, uint64_t t_begin, uint64_t t_end, int local_bits,
                             uint64_t swapped_mask, uint64_t my_place, uint64_t peer_place, int sm_count,
                             cudaStream_t stream);

int reduce_grid(uint64_t n, int sm_count);
// out_dev[0..1] = (S0, S1) split by physical bit `bit` (bit < 0: total in S0).
cudaError_t launch_sumsq(const double2 *amps, uint64_t n, int bit, double *partials_dev, double *out_dev, int sm_count,
                         cudaStream_t stream);
// out_dev[0..1] = (re, im) of sum conj(a_k) b_k.
cudaError_t launch_dotc(const double2 *a, const double2 *b, uint64_t n, double *partials_dev, double *out_dev,
                        int sm_count, cudaStream_t stream);

// Expectation values of up to kExpMaxTerms Pauli strings that share one X mask, in one read-only sweep
// (qb_expect_pauli).  out_dev[t] = sum over the pairs (i, i ^ xp), bit h of i clear (h = top bit of xp), of
// (-1)^popc(i & zp[t]) * (t < neven ? Re : Im) conj(amps[i ^ xp]) amps[i]; xp == 0: sum over every i of
// (-1)^popc(i & zp[t]) |amps[i]|^2.  Deterministic (fixed grid per device, fixed-order two-stage sum).
constexpr int kExpMaxTerms = 64;
constexpr int kExpU = 4;          // pairs per thread and step: pair numbers p0 + u * 256 (u at bit kExpUShift)
constexpr int kExpUShift = 8;
struct ExpTerms {
  uint64_t xp;       // physical X mask (local bits)
  uint64_t lo_mask;  // bits below h ((1 << h) - 1); ~0 when xp == 0
  int32_t nterms, neven;
  uint64_t zp[kExpMaxTerms];     // physical Z mask (local bits) per term
  uint32_t rflip[kExpMaxTerms];  // bit u: popc(deposit(u << kExpUShift) & zp[t]) is odd (deposit = insert a 0 at bit h)
};
cudaError_t launch_expect_pauli(const double2 *amps, int local_bits, const ExpTerms &terms, double *partials_dev,
                                double *out_dev, int sm_count, cudaStream_t stream);

// Pauli rotations exp(-i theta/2 P) in place (qb_apply_pauli_rot): up to kPauliMaxRot rotations in ONE
// read + write sweep.  A CTA owns a tile of 2^tile_bits amplitudes on the physical bits tile_pos[] (every X
// bit of the launch is one of them); rotation r, for every tile-local index j, sets
//   psi'_j = c psi_j + (ar + i ai) (-1)^popc((j ^ xt) & zt) (-1)^popc(base & zout) psi_(j ^ xt)
// with base = the tile's non-tile bits.  The host folds -i sin(theta/2) i^popc(x & z) and the sign of Z on
// global qubits into (ar, ai).  xt == 0 (Z only) is a per-amplitude phase.
constexpr int kPauliTileBits = 12;  // 64 KB of shared memory per CTA
constexpr int kPauliMaxRot = 64;
constexpr int kPauliThreads = 256;
struct PauliRotParam {
  uint64_t zout;       // Z mask on the local bits outside the tile (physical)
  double c, ar, ai;    // cos(theta/2); the partner's factor
  uint32_t xt, zt;     // X / Z masks on the tile-local bits
};
struct PauliRotArgs {
  uint32_t nrot, tile_bits, nruns, _pad;
  uint8_t tile_pos[16];                 // physical bit of tile-local bit i, ascending
  uint8_t run_shift[16], run_len[16];   // the tile number deposited into the local bits outside the tile
  PauliRotParam rot[kPauliMaxRot];
};
cudaError_t launch_pauli_rot(double2 *amps, int local_bits, const PauliRotArgs &args, cudaStream_t stream);

// A Pauli sum applied to a state (qb_pauli_sum): out (+)= sum_t (cr + i ci)_t (-1)^popc((j ^ xt) & zt)
// (-1)^popc(base & zout) src_(j ^ xt) for up to kPauliMaxRot terms whose X bits fit one tile (the tile geometry
// of PauliRotArgs).  first != 0: out is stored, else added to.  partials != null: each block also leaves
// Re sum_j conj(src_j) (this launch's part of out)_j in partials[block], reduced into *energy_dev in a fixed
// order.  A fixed grid walks the tiles in a fixed order: deterministic.
struct PauliSumParam {
  uint64_t zout;
  double cr, ci;      // the term's coefficient times i^popc(x & z) and the sign of Z on global qubits
  uint32_t xt, zt;
};
struct PauliSumArgs {
  uint32_t nterms, tile_bits, nruns, first;
  uint8_t tile_pos[16];
  uint8_t run_shift[16], run_len[16];
  PauliSumParam term[kPauliMaxRot];
};
cudaError_t launch_pauli_sum(const double2 *src, double2 *out, int local_bits, const PauliSumArgs &args,
                             double *partials_dev, double *energy_dev, int sm_count, cudaStream_t stream);

// One launch of a Chebyshev step of exp(-itH) (qb_pauli_evolve): hs = sum over the run's terms as in
// launch_pauli_sum (the host folds 1/r, or 2/r after step 1, into the coefficients), applied to cur; then
//   out = hs (kChebOutStore, step 1's first launch) | hs - out (kChebOutSub, a later step's first launch)
//       | out + hs (kChebOutAdd, every other launch);
// and in the step's last launch acc = a0 cur + ak out (kChebAccFirst, step 1) | acc + ak out (kChebAccAdd).
// cur, out and acc are three shards in one layout.  Deterministic (fixed grid, fixed term order).
enum : uint32_t { kChebOutStore = 0, kChebOutSub = 1, kChebOutAdd = 2 };
enum : uint32_t { kChebAccNone = 0, kChebAccFirst = 1, kChebAccAdd = 2 };
struct PauliChebArgs {
  PauliSumArgs sum;  // tile geometry and terms (sum.first unused)
  uint32_t out_mode, acc_mode;
  double a0r, a0i, akr, aki;
};
cudaError_t launch_pauli_cheb(const double2 *cur, double2 *out, double2 *acc, int local_bits, const PauliChebArgs &args,
                              int sm_count, cudaStream_t stream);

// The backward pass of the adjoint gradient (qb_pauli_rot_grad) over one launch of rotations: psi and lam
// (same layout) are walked through rotations nrot-1 .. 0; for each, grad_dev[r] = Im sum_j conj(lam_j) (P_r psi)_j,
// then psi <- R_r^dagger psi and lam <- R_r^dagger lam with R_r^dagger = c I + i s P_r.  (P psi)_j =
// (fr + i fi) (-1)^popc((j ^ xt) & zt) (-1)^popc(base & zout) psi_(j ^ xt).  Per-block partials of each rotation
// are reduced in a fixed order (partials[block * kPauliMaxRot + r]), then into grad_dev by k_expect_final.
constexpr int kPauliAdjThreads = 512;
struct PauliAdjParam {
  uint64_t zout;
  double c, s, fr, fi;
  uint32_t xt, zt;
};
struct PauliAdjArgs {
  uint32_t nrot, tile_bits, nruns, _pad;
  uint8_t tile_pos[16];
  uint8_t run_shift[16], run_len[16];
  PauliAdjParam rot[kPauliMaxRot];
};
cudaError_t launch_pauli_rot_adjoint(double2 *psi, double2 *lam, int local_bits, const PauliAdjArgs &args,
                                     double *partials_dev, double *grad_dev, int sm_count, cudaStream_t stream);

// Live sub-cube {i : i & fixed_mask == fixed_val} of the shard (see "support" in qb_api.cpp): the
// reduction of launch_sumsq restricted to it, and zero-fill (mode 0) / scaling (mode 1) of it.
int cube_runs(int local_bits, uint64_t fixed_mask);  // must be <= kMaxRuns for the launchers below
cudaError_t launch_sumsq_cube(const double2 *amps, int local_bits, uint64_t fixed_mask, uint64_t fixed_val, int bit,
                              double *partials_dev, double *out_dev, int sm_count, cudaStream_t stream);
cudaError_t launch_cube_update(double2 *amps, int local_bits, uint64_t fixed_mask, uint64_t fixed_val, int mode,
                               const double z[2], int sm_count, cudaStream_t stream);

cudaError_t launch_axpy(double2 *y, const double2 *x, uint64_t n, const double z[2], int sm_count,
                        cudaStream_t stream);
cudaError_t launch_tensor(double2 *out, const double2 *a, const double2 *b, int abits, int bbits, int sm_count,
                          cudaStream_t stream);
// exchange local index bits b1 and b2 in place (layout change)
cudaError_t launch_swap_bits(double2 *amps, int local_bits, int b1, int b2, int sm_count, cudaStream_t stream);
// sharded a `tensor` b: out shard = (a shard) x (all of b, read through the ranks' mapped shards)
cudaError_t launch_tensor_sharded(double2 *out, const double2 *a, double2 *const *b_shards_dev, int a_local_bits, int bbits,
                                  int b_local_bits, int sm_count, cudaStream_t stream);
cudaError_t launch_set_amp(double2 *amps, uint64_t idx, double re, double im, cudaStream_t stream);
// out[i] = amps[index whose bit pos[b] is bit b of (first + i)], i < count: a range of amplitudes in index order from a
// shard whose qubit layout is not the identity (pos = logical bit -> physical bit, nbits of them)
cudaError_t launch_gather_logical(double2 *out, const double2 *amps, uint64_t first, uint64_t count, const int *pos, int nbits,
                                  int sm_count, cudaStream_t stream);
// dst[index with bit b moved to newpos[b]] = src[index]: a change of layout in one out-of-place sweep
cudaError_t launch_permute_bits(double2 *dst, const double2 *src, int local_bits, const int *newpos, int sm_count,
                                cudaStream_t stream);

}  // namespace qb
