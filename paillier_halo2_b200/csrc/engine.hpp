// engine.hpp — internal interfaces between the C ABI (capi.cu) and the CUDA engines.
#pragma once
#include <atomic>
#include <cstdint>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "host_bigint.hpp"
#include "simple64.cuh"

namespace pb200 {

extern std::atomic<uint64_t> g_kernel_launches;
inline void count_launch(uint64_t n = 1) { g_kernel_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- simple64 engine launchers (simple64_kernels.cu) ---------------------------------------
// All pointers are device pointers; work is enqueued on `st`.
cudaError_t simple_gchain(const SimpleConsts* dK, u64* d_gchain /* n_bits * 2k */, int n_bits, cudaStream_t st);
cudaError_t simple_encrypt(const SimpleConsts* dK, const u64* d_gchain, const u64* d_m, const u64* d_r, size_t count,
                           u64* d_c /*nullable*/, u64* d_records /*nullable*/, const u64* d_offsets /*nullable*/,
                           u64* d_digest /*nullable*/, int* d_flags, cudaStream_t st);
cudaError_t simple_add(const SimpleConsts* dK, const u64* d_c1, const u64* d_c2, int c_words, size_t count,
                       u64* d_out, u64* d_q /*nullable*/, int* d_flags, cudaStream_t st);
// product of `count` values (k words each) -> d_out (k words); d_scratch: at least simple_tally_scratch_words(k) words
size_t simple_tally_scratch_words(int k);
cudaError_t simple_tally(const SimpleConsts* dK, int k, const u64* d_c, size_t count, u64* d_out, u64* d_scratch,
                         int* d_flags, cudaStream_t st);
cudaError_t repack_limbs(const u64* d_vals, size_t count, int words_per_value, int value_bits, int limb_bits,
                         u64* d_out, cudaStream_t st);
// decryption pieces on the simple engine: x = base^e mod n^2 (exponent words on the device), and m = (x - 1) / n * mu mod n with
// the constants of the modulus n (mu in their g slot); flag bit 3 when x != 1 (mod n).  e_stride = 0: one exponent for every unit
// (decryption's lambda); e_stride > 0: unit u's exponent starts at word u * e_stride, and the base is reduced mod n^2 first (scalar
// multiplication accepts any words_out-word value); reduce: the base is reduced with e_stride = 0 too (partial decryption)
cudaError_t simple_pow(const SimpleConsts* dK, const u64* d_base, int base_words, const u64* d_e, int e_bits, int e_stride, size_t count,
                       u64* d_out, int* d_flags, cudaStream_t st, bool reduce = false);
cudaError_t simple_lfunc(const SimpleConsts* dKn, const u64* d_x, size_t count, u64* d_m, int* d_flags, cudaStream_t st);

// ---- inverse mod n^2 (inverse_kernels.cu): safegcd mod n, then one Hensel step --------------------------------------------
#define PB200_INV_MAXL 67   // signed 62-bit limbs of the safegcd state at |n| = 4096 (n_bits / 62 + 1)
struct InvConsts {
    SimpleConsts n;         // Barrett constants of the modulus n (k = words_in): c mod n
    int L, batches;         // limbs, batches of 62 divsteps (Bernstein-Yang's bound for an n_bits-bit modulus)
    u64 ninv62;             // n^-1 mod 2^62
    long long n62[PB200_INV_MAXL];
    u64 n2[PB200_SIMPLE_MAXK];
};
// the safegcd fields of an odd n (the caller fills the Barrett constants of n)
void inverse_consts(const BigInt& n, uint32_t n_bits, InvConsts* h);
// out_u = c_u^-1 mod n^2, or c1_u * c_u^-1 mod n^2 when d_c1 is given; a unit with gcd(c_u, n) != 1 gets 0 and raises PB200_FLAG_NOT_INVERTIBLE.  d_neg
// non-null: only units with d_neg[u] != 0 and a non-zero magnitude (kw words at d_mag + u kw) are inverted, the others keep their value
// (d_c == d_out is allowed)
cudaError_t simple_inverse(const SimpleConsts* dK, const InvConsts* dI, const u64* d_c, const u64* d_c1, const uint8_t* d_neg, const u64* d_mag,
                           int kw, size_t count, u64* d_out, int* d_flags, cudaStream_t st);

// running-tally trace (pb200_tally_trace): level l holds n[l] entries per chain in chunks of s[l]; n[l + 1] = ceil(n[l] / s[l]) and the
// last level has one chunk per chain.  Level 0 is the steps themselves.
struct TracePlan { std::vector<size_t> n, s; };
// phases 1 and 2 on simple64: d_tmp (simple_trace_scan_words) ends with the canonical carry-in of every level-0 chunk at its start
size_t simple_trace_scan_words(const TracePlan& P, size_t chains, int k);
cudaError_t simple_trace_scan(const SimpleConsts* dK, int k, const TracePlan& P, const u64* d_init, const u64* d_c, size_t chains,
                              u64* d_tmp, cudaStream_t st);
// phase 3 on simple64: one thread per level-0 chunk (d_carry: carry-in of chunk b >= 1 at (b * chains + j) * k; null with one chunk)
cudaError_t simple_trace_chain(const SimpleConsts* dK, const u64* d_init, const u64* d_c, const u64* d_carry, size_t count, size_t chains,
                               size_t s, u64* d_acc, u64* d_q /*nullable*/, int* d_flags, cudaStream_t st);

// ---- block28 engine (block28_kernels.cu) ----------------------------------------------------
struct Block28Key;  // opaque per-key state of the fast engine
// returns nullptr (and leaves *why) when no compiled configuration covers the key size
Block28Key* block28_create(const BigInt& n, const BigInt& g, uint32_t n_bits, int device, cudaStream_t st,
                           std::string* why, cudaError_t* cuda_err);
void block28_destroy(Block28Key*);
const char* block28_name(const Block28Key*);
// 0: every phase on IMAD (block28), 1: constant-operand phases on mma.sync (block28t), 2: on tcgen05 + TMEM with 32 ciphertexts per
// CTA (block28u), 3: with 64 per CTA (block28u2); each falls back to the next lower one the key size has; -1: fastest available.
// Returns the engine in effect.
int block28_set_engine(Block28Key*, int eng);
// whether the key's configuration compiles engine eng (0..3 as above; no fallback)
bool block28_has_engine(const Block28Key*, int eng);
void block28_chain_counts(const Block28Key*, uint64_t* n_sqr, uint64_t* n_mul);
cudaError_t block28_encrypt(Block28Key*, const u64* d_m, const u64* d_r, size_t count, u64* d_c, cudaStream_t st);
cudaError_t block28_tally(Block28Key*, const u64* d_c, size_t count, u64* d_out, cudaStream_t st);
// out = base^e mod n^2 for a per-key exponent e (sliding-window schedule built by block28_pow_prepare), one schedule per slot:
// POW_LAMBDA the decryption's c^lambda, POW_SHARE a trustee's partial decryption c^(2 Delta s_i)
enum { POW_LAMBDA = 0, POW_SHARE = 1, POW_SLOTS = 2 };
cudaError_t block28_pow_prepare(Block28Key*, int slot, const BigInt& e, cudaStream_t st);
cudaError_t block28_pow(Block28Key*, int slot, const u64* d_base, int base_words, size_t count, u64* d_out, cudaStream_t st);
// out_u = prod_j b_(j, u)^(e_j) mod n^2 for k <= 32 exponents shared by the batch (k_multipow, Straus): b_(j, u) at d_base +
// (pos[j] * stride + u) * words_out.  block28_multipow_prepare builds the merged schedule and uploads it on st; the plan (and its
// host copy of the schedule) must live until st has run every launch that uses it.
struct MultiPow {
    int k = 0, h = 0, first_idx = -1;   // bases, odd powers per base (2^(w - 1)), first table entry of the chain
    std::vector<int> pos;               // share position of each base
    std::vector<int2> ops;              // (squarings, table entry or -1), as PowSched
    int2* d_ops = nullptr; int* d_pos = nullptr;
    uint64_t n_sqr = 0, n_mul = 0;      // squarings / multiplications per unit (table and chain)
};
cudaError_t block28_multipow_prepare(const std::vector<BigInt>& e, const std::vector<int>& pos, MultiPow* P, cudaStream_t st);
void block28_multipow_free(MultiPow* P);
cudaError_t block28_multipow(Block28Key*, const MultiPow& P, const u64* d_base, size_t stride, size_t count, u64* d_out, cudaStream_t st);
// out_i = c_i^(k_i) mod n^2 with a scalar per unit (PB200_WORDS(k_bits) words each; c_i: words_out words, any value): fixed-window
// chain per lane, window width chosen from k_bits; no per-key preparation
cudaError_t block28_scalar(Block28Key*, const u64* d_c, const u64* d_k, uint32_t k_bits, size_t count, u64* d_out, cudaStream_t st);
// matvec (pb200_matvec): the planner's choice for one call.  method 0 = chain (per row and sign: scalar products + tally), 1 = bucket.
// Bucket passes cover rb rows x jg windows x nc ciphertexts (both signs); mulmod counts are upper bounds for dense weights.
struct MatvecPlan {
    int method = 0, c = 0, J = 0, nseg = 0, lseg = 0, nsign = 1;
    size_t rb = 0, jg = 0, nc = 0;
    uint64_t passes = 0, acc = 0, red = 0, horner = 0, sign = 0, chain = 0, bytes = 0;
};
// temporary device memory every matvec stays within: 3 * 2^18 ciphertexts' worth (384 MB at |n| = 2048)
size_t matvec_budget(uint32_t n_bits);
// bucket_ok: the key runs a block28 engine.  PB200_MATVEC_METHOD=chain|bucket forces the method, PB200_MATVEC_PASS_ENTRIES caps the
// sort entries of one pass.  Host only.
MatvecPlan matvec_plan(uint32_t n_bits, int sms, size_t rows, size_t count, uint32_t k_bits, bool has_neg, bool bucket_ok);
// bucket method on the block28 engine: out (rows * words_out) canonical; arena: P.bytes of device memory; d_nm1: plan.rb copies of
// n - 1 (PB200_WORDS(n_bits) words each) when P.nsign == 2
cudaError_t block28_matvec(Block28Key*, const MatvecPlan& P, const u64* d_c, size_t count, const u64* d_w, uint32_t k_bits, const uint8_t* d_neg,
                           size_t rows, u64* d_out, void* arena, const u64* d_nm1, cudaStream_t st);
// plain helpers of the chain method: out <- the magnitudes of sign sgn (others 0); n values of wo words <- 1
cudaError_t matvec_mask(const u64* d_w, const uint8_t* d_neg, size_t n, int kw, int sgn, u64* d_out, cudaStream_t st);
cudaError_t matvec_ones(u64* d_out, size_t n, int wo, cudaStream_t st);
// multi-GPU tally: one launch per GPU, partials exchanged through peer-mapped mailboxes inside the kernel (collective call)
cudaError_t block28_tally_peer(Block28Key*, const u64* d_c, size_t count, u64* d_out, cudaStream_t st);
cudaError_t block28_mailbox(Block28Key*, u64** d_mail, cudaStream_t st);
size_t block28_mailbox_bytes();
int block28_max_world();
int block28_peer_world(const Block28Key*);
cudaError_t block28_tally_peer_connect(Block28Key*, int rank, int world, u64* const* mail, void* const* opened, int* d_flags);
// witness engine: the reference's chain with exact (q, rem) per mul_mod (block28t arithmetic + exact tail)
bool block28_witness_supported(const Block28Key*);
// d_gchain: n_bits records (q, rem) of the g-chain squarings; gchain_ready = false lets the witness engine produce them
cudaError_t block28_witness_prepare(Block28Key*, u64* d_gchain, bool gchain_ready, cudaStream_t st);
cudaError_t block28_witness(Block28Key*, const u64* d_m, const u64* d_r, size_t count, u64* d_c /*nullable*/,
                            u64* d_records /*nullable*/, const u64* d_offsets /*nullable*/, u64* d_digest /*nullable*/,
                            cudaStream_t st);

// one exact mul_mod per pair on the witness engine (requires block28_witness_prepare); range flag bit 0 when q does not fit
cudaError_t block28_add(Block28Key*, const u64* d_c1, const u64* d_c2, int c_words, size_t count, u64* d_out, u64* d_q /*nullable*/,
                        int* d_flags, cudaStream_t st);

// running-tally trace.  Lanes of one wave of the tally's CTA shape (32 x resident CTAs per SM x SMs).
size_t block28_lanes(const Block28Key*);
// phases 1 and 2 on the key's tally engine: d_carry (P.n[1] * chains * words_out words) <- the canonical carry-in of every level-0
// chunk; tmp: block28_trace_scan_bytes of device memory.  Nothing to do when P has a single level.
size_t block28_trace_scan_bytes(const Block28Key*, const TracePlan& P, size_t chains);
cudaError_t block28_trace_scan(Block28Key*, const TracePlan& P, const u64* d_init, const u64* d_c, size_t chains, void* tmp, u64* d_carry,
                               cudaStream_t st);
// phase 3 on the witness engine (requires block28_witness_prepare); d_carry as simple_trace_chain
cudaError_t block28_trace_chain(Block28Key*, const u64* d_init, const u64* d_c, const u64* d_carry, size_t count, size_t chains, size_t s,
                                u64* d_acc, u64* d_q /*nullable*/, int* d_flags, cudaStream_t st);

// diagnostic: one CTA's modular multiplication on raw lazy digits (shared-memory image layout), see k_mulmod_dbg
cudaError_t block28_debug_mulmod(Block28Key*, int eng, const int* h_v, const int* h_y, int reps, int* h_vout, int* h_t, unsigned* h_rows,
                                 cudaStream_t st);
void block28_shape(const Block28Key*, int* G, int* BL);
// 20 layout constants of the block28u variant <G, BL> with lg lane groups per CTA (wit: witness layout); false for unknown shapes
bool block28_umma_layout(int G, int BL, int lg, int wit, int* out);
// diagnostic: cycles of phase A / phases B + C / the whole loop per CTA over `reps` squarings on `ctas` CTAs (|n| = 2048 configuration)
cudaError_t block28_debug_time(Block28Key*, int eng, const int* h_v, int ctas, int reps, int stagger, long long* h_cyc, cudaStream_t st);

}  // namespace pb200
