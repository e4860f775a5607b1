/* paillier_b200.h — C ABI of the B200-native batched Paillier hot path.
 *
 * Drop-in boundary for ONE path of aerius-labs/paillier-halo2: batched encryption
 * c = g^m * r^n mod n^2, homomorphic addition c1*c2 mod n^2, their N-ary fold (tally) and the
 * per-step (q, rem) witness values that PaillierChip::encrypt/add assign through BigUintChip.
 * The reference has no FFI of its own; each entry point below names the reference interface it
 * replaces (paths into the reference repository).  The Rust-side binding a maintainer would add
 * is shown in INTEGRATION.md.
 *
 * Conventions
 *   - all integers are little-endian arrays of uint64_t words ("u64 limbs"); word i has weight
 *     2^(64 i), the same order PaillierChip::get_biguint folds (src/paillier.rs:22-30);
 *   - a value of b bits occupies  PB200_WORDS(b) = ceil(b/64) words; unused high bits are zero;
 *   - batches are unit-major and contiguous: unit u starts at word u * words_per_value;
 *   - every function returns 0 (PB200_OK) or a negative pb200_status; nothing throws or aborts
 *     across the ABI (maps to Result<_, Error> on the Rust side, src/paillier.rs:38,68); entry points
 *     run on the key's device and restore the caller's current CUDA device before returning;
 *   - the caller owns every buffer it passes; the library owns a pb200_key until
 *     pb200_key_destroy;  a key is bound to one CUDA device and one internal stream; calls on one
 *     key are serialised by the caller (mirrors &mut Context<F>), different keys may be used from
 *     different threads;
 *   - functions with the suffix _dev take DEVICE pointers (resident in the key's device) and
 *     enqueue on the key's stream without a final synchronise unless stated; the others take HOST
 *     pointers and return when the result is in the output buffer;
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry point returns
 *     PB200_ERR_CUDA.
 */
#ifndef PAILLIER_B200_H
#define PAILLIER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB200_WORDS(bits) (((bits) + 63) / 64)

typedef enum pb200_status {
    PB200_OK = 0,
    PB200_ERR_INVALID_ARG = -1,   /* null pointer, zero sizes, n_bits % limb_bits != 0 (assign_integer's assert) */
    PB200_ERR_ZERO_MODULUS = -2,  /* n == 0: num-bigint modpow / % panic (src/paillier.rs:89-91,96) */
    PB200_ERR_EVEN_MODULUS = -3,  /* only from pb200_inverse_batch*, pb200_sub_batch*, pb200_scalar_mul_signed_batch* with signs and
                                     pb200_combine_shares_batch* with a negative coefficient (their algorithm needs an odd n); every
                                     other entry point accepts an even n, as the reference
                                     does, whose tests draw n = rng.gen_biguint(bits) (src/paillier.rs:173,251) */
    PB200_ERR_RANGE = -4,         /* an input does not fit its declared bit width (range check would fail) */
    PB200_ERR_UNSUPPORTED = -5,   /* key size larger than the largest compiled engine */
    PB200_ERR_CUDA = -6,          /* CUDA runtime failure; pb200_last_cuda_error() has the text */
    PB200_ERR_NOMEM = -7,
    PB200_ERR_SINK = -8,          /* the witness sink callback returned non-zero */
    PB200_ERR_CONSTRAINT = -9,    /* a supplied (q, rem) does not satisfy a*b = q*n^2 + rem (mul_mod's equality would fail) */
    PB200_ERR_PEER = -10,         /* multi-GPU tally: a peer's partial did not arrive within the kernel's time-out */
    PB200_ERR_DECRYPT = -11,      /* c^lambda mod n^2 is not 1 modulo n: not a valid ciphertext for this key */
    PB200_ERR_NOT_INVERTIBLE = -12 /* gcd(c mod n^2, n) != 1: the value has no inverse mod n^2 (0, n, a multiple of p or q) */
} pb200_status;

/* bits of the per-key device flag word (pb200_key_take_flags) */
#define PB200_FLAG_RANGE 1u       /* -> PB200_ERR_RANGE */
#define PB200_FLAG_CONSTRAINT 2u  /* -> PB200_ERR_CONSTRAINT */
#define PB200_FLAG_PEER_TIMEOUT 4u /* a peer GPU's tally partial did not arrive (pb200_tally_peer_dev / pb200_tally_multi) */
#define PB200_FLAG_DECRYPT 8u     /* -> PB200_ERR_DECRYPT */
#define PB200_FLAG_NOT_INVERTIBLE 16u /* -> PB200_ERR_NOT_INVERTIBLE */

typedef struct pb200_key pb200_key;

/* ---- library ------------------------------------------------------------------------------ */
const char* pb200_strerror(int status);
const char* pb200_last_cuda_error(void);      /* thread-local text of the last CUDA failure */
const char* pb200_version(void);
int pb200_device_count(void);                 /* number of visible CUDA devices, 0 if none */
/* number of kernel launches issued by this library since load (all threads); bench.py reports it */
uint64_t pb200_kernel_launches(void);

/* ---- key ------------------------------------------------------------------------------------
 * Replaces: EncryptionPublicKeyAssigned{n,g} + PaillierChip::construct (src/paillier.rs:6-20) and
 * the per-call recomputation of n^2 by square+refresh (src/paillier.rs:39-45, :69-75) / n*n
 * (:88, :95).  n_bits = enc_bits of the reference (bit width n, g, m, r are assigned with,
 * src/bench.rs:44-60); limb_bits = BigUintChip limb width (64 and 88 in the reference's tests),
 * only used to format witness limbs.  n and g are PB200_WORDS(n_bits) words each. */
int pb200_key_create(int device, uint32_t n_bits, uint32_t limb_bits,
                     const uint64_t* n_le, const uint64_t* g_le, pb200_key** out);
void pb200_key_destroy(pb200_key* key);
uint32_t pb200_key_n_bits(const pb200_key* key);
uint32_t pb200_key_words_in(const pb200_key* key);   /* PB200_WORDS(n_bits)   : n, g, m, r        */
uint32_t pb200_key_words_out(const pb200_key* key);  /* PB200_WORDS(2*n_bits) : n^2, c, q, rem    */
int pb200_key_device(const pb200_key* key);
/* n^2 (words_out words) — value of the Fresh n2 of src/paillier.rs:45 */
int pb200_key_n2(const pb200_key* key, uint64_t* n2_out);
/* name of the arithmetic engine selected for this key size, e.g. "block28<8,19>" or "simple64" */
const char* pb200_key_engine(const pb200_key* key);
/* choose the engine explicitly: 0 = automatic (fastest available), 1 = simple64 (thread per
 * ciphertext, always available, used as the on-GPU cross-check), 2 = block28 (warp-role Barrett, all
 * products on the IMAD pipe), 3 = block28t (same, constant-operand Barrett phases on the tensor pipe with mma.sync), 4 = block28u
 * (the same phases on tcgen05.mma with TMEM accumulators, 32 ciphertexts per CTA; the automatic choice where it exists), 5 = block28u2
 * (tcgen05 with 64 ciphertexts per CTA and half the tensor-core work per ciphertext; kept for A/B).  4 and 5 return
 * PB200_ERR_UNSUPPORTED for key sizes without that variant */
int pb200_key_set_engine(pb200_key* key, int engine);
void* pb200_key_stream(const pb200_key* key);        /* cudaStream_t the key enqueues on */
/* modular squarings and multiplications the selected engine executes per encryption (the chain the
 * roofline's algorithmic work is counted on; excludes the engine's internal canonicalisation) */
int pb200_key_chain_counts(const pb200_key* key, uint64_t* n_sqr, uint64_t* n_mul);
int pb200_key_sync(pb200_key* key);                  /* cudaStreamSynchronize on that stream */
/* _dev entry points report range / constraint failures only through a per-key flag word on the device.  This call synchronises
 * the key's stream, returns the word (PB200_FLAG_*) and clears it.  Host entry points clear it when they start and map it to
 * their return status, so a _dev failure never leaks into a later host call. */
int pb200_key_take_flags(pb200_key* key, uint32_t* flags_out);

/* Diagnostics of the fast engine (block28 family).  pb200_key_shape: G blocks of BL signed 28-bit digits per value.
 * pb200_debug_mulmod: ONE CTA's (32 lanes) lazy modular multiplication V <- V * Y (y_in null: V^2), repeated `reps` times, on
 * engine 2, 3, 4 or 5, on raw digit images in the engine's shared-memory layout ([block][chunk of 4 digits][lane][4] int32,
 * G * ceil(BL / 4) * 32 * 4 words).  t_out non-null: phase A only, the 2L-digit product image (twice that many words).  Otherwise
 * v_out receives the lazy result and qhat_rows (nullable, 32 * G * BL words) the quotient estimate's packed s8 digits.  The
 * engines are specified to agree digit for digit; the parity tests check exactly that. */
int pb200_key_shape(const pb200_key* key, int* g_out, int* bl_out);
/* layout constants of the block28u variant for values of G blocks x BL digits with `lane_groups` (1 or 2) groups of 32 ciphertexts
 * per CTA (witness != 0: the witness engine's layout): out20 = {supported, digits per range, columns per tile, MMA N, tiles of
 * phase B, tiles of phase C, zero chunks in front, behind, k offset, chunk bytes, operand-row bytes, z0 of the two Toeplitz tables,
 * their entry counts, shared-memory bytes, CTAs per SM, TMEM columns, gap bytes, first column of phase B}.  Host only (no device
 * needed): tests/test_umma_layout.py checks its CPU model of the tcgen05 data path against them.  PB200_ERR_UNSUPPORTED for shapes
 * that are not compiled. */
int pb200_umma_layout(int g, int bl, int lane_groups, int witness, int32_t* out20);
int pb200_debug_mulmod(pb200_key* key, int engine, const int32_t* v_in, const int32_t* y_in, int reps, int32_t* v_out, int32_t* t_out,
                       uint32_t* qhat_rows);
/* `reps` lazy squarings on each of `ctas` CTAs (engine 3, 4 or 5, |n| = 2048 configuration); cycles_out[3 cta + {0, 1, 2}] = SM cycles
 * spent in phase A, in phases B + C, in the whole loop.  stagger_cycles > 0 delays every second CTA by that many cycles first. */
int pb200_debug_mulmod_cycles(pb200_key* key, int engine, const int32_t* v_in, int ctas, int reps, int stagger_cycles, int64_t* cycles_out);

/* ---- encrypt --------------------------------------------------------------------------------
 * Replaces: paillier_enc_native (src/paillier.rs:87-92) for `count` independent (m, r) pairs, and
 * the VALUE returned by PaillierChip::encrypt (src/paillier.rs:32-60).
 * m, r: count * words_in words; c_out: count * words_out words, canonical (< n^2).
 * PB200_ERR_RANGE if any m or r has bits at or above n_bits (host variant only). */
int pb200_encrypt_batch(pb200_key* key, const uint64_t* m_le, const uint64_t* r_le, size_t count,
                        uint64_t* c_out_le);
int pb200_encrypt_batch_dev(pb200_key* key, const uint64_t* d_m_le, const uint64_t* d_r_le,
                            size_t count, uint64_t* d_c_out_le);

/* ---- add ------------------------------------------------------------------------------------
 * Replaces: paillier_add_native (src/paillier.rs:94-97) and PaillierChip::add (:62-85) for `count`
 * pairs.  c_words = words per input ciphertext: words_out for real ciphertexts, words_in for the
 * half-width values the reference's tests assign (src/paillier.rs:216-221; extend_limbs at :79-80
 * zero-pads them).  out: count * words_out words.  q_out (nullable): floor(c1*c2 / n^2), the mul_mod
 * quotient witness, count * words_out words. */
int pb200_add_batch(pb200_key* key, const uint64_t* c1_le, const uint64_t* c2_le, uint32_t c_words,
                    size_t count, uint64_t* out_le, uint64_t* q_out_le);
int pb200_add_batch_dev(pb200_key* key, const uint64_t* d_c1_le, const uint64_t* d_c2_le, uint32_t c_words,
                        size_t count, uint64_t* d_out_le, uint64_t* d_q_out_le);

/* ---- tally ----------------------------------------------------------------------------------
 * Replaces: the N-ary fold of paillier_add_native (BASELINE.json config 3).  Product of `count`
 * ciphertexts (words_out words each) mod n^2 on the key's device; count == 0 gives 1 mod n^2.
 * The product is commutative and associative, so the result is independent of the tree shape.
 * _dev: d_c on the key's device, d_partial_out receives one words_out-word value on the device. */
int pb200_tally(pb200_key* key, const uint64_t* c_le, size_t count, uint64_t* out_le);
int pb200_tally_dev(pb200_key* key, const uint64_t* d_c_le, size_t count, uint64_t* d_partial_out_le);
/* combine `n_partials` per-shard partial products (host memory, e.g. gathered by the caller) into the final product on the
 * key's device: the same fold on the key's own engine */
int pb200_tally_combine(pb200_key* key, const uint64_t* partials_le, size_t n_partials, uint64_t* out_le);

/* ---- running-tally trace ------------------------------------------------------------------------
 * The witness of a circuit that proves a running tally: PaillierChip::add(acc, c_i) once per ballot, each step taking the previous
 * step's rem.  For every chain j < chains and step i < count:
 *   a = (i == 0 ? init_j : acc_(i-1, j)),  b = c_(i, j),  q_(i, j) = floor(a b / n^2),  acc_(i, j) = a b mod n^2
 * exactly the values pb200_add_batch(a, b, c_words = words_out, .., q_out) returns for that pair.  A K-option ballot is K chains.
 * Layout: step-major, one ballot per row: entry (i, j) of c, acc and q at (i * chains + j) * words_out words; init: chains *
 * words_out words.  Inputs are any words_out-word values (reduced or not, as for pb200_add_batch): step 0 uses init exactly as given,
 * every later a is canonical, so a q that does not fit words_out words (PB200_ERR_RANGE, host variant; PB200_FLAG_RANGE, _dev) can
 * only come from step 0 with an unreduced init.  q_out == NULL skips the quotients (the prefix products alone).  count == 0 or
 * chains == 0 does nothing; PB200_ERR_INVALID_ARG for null pointers where data is needed.
 *
 * Work: the chains are cut into chunks of about count * chains / lanes steps (lanes = 32 x resident CTAs per SM x SMs, one wave).
 * Phase 1 multiplies each chunk into a total on the tally's engine, level after level over the totals; phase 2 turns them into every
 * chunk's carry-in, init_j * the totals before it; phase 3 runs each chunk's exact chain on the witness engine.  About one fast and
 * one exact multiplication per step; no host synchronise.  Temporary device memory does not depend on count: one buffer per level
 * below the top, sum over l of ceil(n_l / s_l) * chains values, at most 3 * (lanes + chains) lazy values of the block28
 * configuration (slightly more than words_out words each; canonical values on simple64), plus lanes + chains canonical carries
 * (derivation in DESIGN.md §9c); the host variant's staged init, c, acc and q come on top.  PB200_TRACE_LANES=<n> replaces the
 * wave size (a test and diagnostic switch: small waves reach every chunk and level boundary with few steps; output is the same).
 *
 * Contiguous operands for the advice cells: allocate (count + 1) * chains values, put init in row 0 and pass acc_out one row in
 * (buf + chains * words_out).  Then (buf, c, q, buf + chains * words_out) are the (a, b, q, rem) arrays of pb200_mulmod_cells_batch
 * for the count * chains steps, and the cells of the whole trace come from that one call.
 * _dev: device pointers on the key's device, enqueued on the key's stream, no final synchronise. */
int pb200_tally_trace(pb200_key* key, const uint64_t* init_le, const uint64_t* c_le, size_t count, size_t chains,
                      uint64_t* acc_out_le, uint64_t* q_out_le /* nullable */);
int pb200_tally_trace_dev(pb200_key* key, const uint64_t* d_init_le, const uint64_t* d_c_le, size_t count, size_t chains,
                          uint64_t* d_acc_out_le, uint64_t* d_q_out_le /* nullable */);

/* ---- multi-GPU tally (BASELINE.json configs[2]; SURVEY.md 8b pb200_tally(keys[], n_gpus, ..)) --------------------------------
 * Replaces: the fold of paillier_add_native (src/paillier.rs:94-97) over ciphertexts that are sharded across the GPUs of one
 * NVLink/NVSwitch domain.  ONE kernel launch per GPU: every GPU folds its shard, stores its 2|n|/8-byte partial into every
 * peer's mailbox through peer-mapped memory, waits for the peers' partials in its own mailbox and combines them — no NCCL call,
 * no host hop, no second launch; every GPU ends with the full product (bit-identical: the product is commutative).
 *
 * Single process, one key per device: keys[i] must hold the same n; d_c[i] is the shard resident on keys[i]'s device
 * (counts[i] ciphertexts of words_out words); out_le (host) receives the product.  Peer access is enabled on first use; when
 * the devices cannot reach each other the partials are gathered through the host and combined on keys[0] instead. */
int pb200_tally_multi(pb200_key* const* keys, int n_gpus, const uint64_t* const* d_c, const size_t* counts, uint64_t* out_le);

/* One process per GPU (torchrun / MPI): each rank exports a handle to its mailbox, the ranks exchange the 64-byte handles by
 * any means (e.g. an all-gather on the host), each rank connects, and from then on pb200_tally_peer_dev is a COLLECTIVE call:
 * every rank calls it once per tally, in the same order, on its own shard.  d_out (device, words_out words) receives the full
 * product on every rank; enqueued on the key's stream, no synchronise.  A rank whose peers never arrive gives up after a few
 * seconds and raises PB200_FLAG_PEER_TIMEOUT in the key's flag word.  world <= 8. */
typedef struct pb200_ipc_handle { unsigned char bytes[64]; } pb200_ipc_handle;
int pb200_tally_peer_export(pb200_key* key, pb200_ipc_handle* out);
int pb200_tally_peer_connect(pb200_key* key, int rank, int world, const pb200_ipc_handle* handles /* world entries */);
int pb200_tally_peer_dev(pb200_key* key, const uint64_t* d_c_le, size_t count, uint64_t* d_out_le);

/* ---- decryption (SURVEY.md 8f-4) ---------------------------------------------------------------
 * The reference states decryption (README.md:5-22 there: m = L(c^lambda mod n^2) * mu mod n, L(x) = (x - 1) / n) and never
 * implements it; it is the natural end of a tally pipeline (decrypt the product).  pb200_key_set_private attaches the private
 * part to a key: lambda = lcm(p - 1, q - 1) and mu = L(g^lambda mod n^2)^-1 mod n, words_in words each.  c^lambda runs on the
 * key's engine (block28: sliding window over the per-key exponent, like r^n), the L function and the multiplication by mu on
 * 64-bit limbs, one thread per ciphertext.  c: count * words_out words; m_out: count * words_in words.
 * PB200_ERR_DECRYPT when some c^lambda mod n^2 is not 1 modulo n (that unit's output is zero). */
int pb200_key_set_private(pb200_key* key, const uint64_t* lambda_le, const uint64_t* mu_le);
int pb200_decrypt_batch(pb200_key* key, const uint64_t* c_le, size_t count, uint64_t* m_out_le);
int pb200_decrypt_batch_dev(pb200_key* key, const uint64_t* d_c_le, size_t count, uint64_t* d_m_out_le);

/* ---- homomorphic scalar multiplication and the weighted tally -----------------------------------------------------------
 * Multiplying a ciphertext by a plaintext: Dec(c^k mod n^2) = k * Dec(c) mod n, and prod c_i^(k_i) encrypts sum k_i m_i (weighted
 * votes, "against" votes with k = n - 1, encrypted dot products with a plaintext vector).  Runs on the key's engine (block28: a
 * fixed-window chain per ciphertext, as long as the longest scalar among the 32 or 64 ciphertexts of a CTA; simple64: LSB-first
 * square-and-multiply); needs no private part and no per-key preparation.
 *
 * out_i = c_i^(k_i) mod n^2 (Dec(out_i) = k_i * Dec(c_i) mod n).  c: count * words_out words (any value, reduced mod n^2);
 * k: count * PB200_WORDS(k_bits) words, 1 <= k_bits <= n_bits (a negative scalar -s is n - s); out: count * words_out, canonical.
 * PB200_ERR_INVALID_ARG for null pointers, k_bits == 0 or k_bits > n_bits; PB200_ERR_RANGE (host variant) when some scalar has a
 * bit at or above k_bits.  _dev: device pointers on the key's device, enqueued on the key's stream, no final synchronise, scalars
 * are not range-checked (the host variant checks them against k_bits). */
int pb200_scalar_mul_batch(pb200_key* key, const uint64_t* c_le, const uint64_t* k_le, uint32_t k_bits, size_t count, uint64_t* out_le);
int pb200_scalar_mul_batch_dev(pb200_key* key, const uint64_t* d_c_le, const uint64_t* d_k_le, uint32_t k_bits, size_t count,
                               uint64_t* d_out_le);
/* prod c_i^(k_i) mod n^2 = Enc(sum k_i m_i); count == 0 gives 1 mod n^2.  Same arguments and checks as pb200_scalar_mul_batch;
 * works in chunks of 2^18 ciphertexts (scalar products, then the tally's fold of each chunk, then the fold of the partials), so
 * its temporary device memory is bounded (128 MB at |n| = 2048).  _dev: d_out receives words_out words on the device; enqueued
 * on the key's stream, no final synchronise, scalars are not range-checked. */
int pb200_tally_weighted(pb200_key* key, const uint64_t* c_le, const uint64_t* k_le, uint32_t k_bits, size_t count, uint64_t* out_le);
int pb200_tally_weighted_dev(pb200_key* key, const uint64_t* d_c_le, const uint64_t* d_k_le, uint32_t k_bits, size_t count,
                             uint64_t* d_out_le);

/* ---- ciphertext inverse, homomorphic subtraction and signed scalars -----------------------------------------------------
 * c^-1 mod n^2 encrypts -Dec(c), so negation, subtraction and negative scalars cost one inversion instead of a full-width exponent
 * n - 1.  The inverse is a per-ciphertext Bernstein-Yang safegcd mod n (a fixed number of batches of 62 divsteps, so no warp diverges
 * on data) followed by one Hensel step to n^2, one thread per ciphertext, on every engine; it needs no private part.
 *
 *   pb200_inverse_batch:            out_i = c_i^-1 mod n^2                      Dec(out_i) = -Dec(c_i) mod n
 *   pb200_sub_batch:                out_i = c1_i * c2_i^-1 mod n^2              Dec(out_i) = Dec(c1_i) - Dec(c2_i) mod n
 *   pb200_scalar_mul_signed_batch:  out_i = c_i^(k_i) mod n^2, k_i = (k_neg[i] ? -1 : +1) * mag_i, c^-s = (c^-1)^s
 *                                                                               Dec(out_i) = k_i * Dec(c_i) mod n
 * c, c1, c2: count * words_out words, any value (reduced mod n^2); out: count * words_out words, canonical.  k_mag: count *
 * PB200_WORDS(k_bits) words, 1 <= k_bits <= n_bits; k_neg: nullable, one byte per unit, non-zero = negative.  k_neg == NULL gives
 * exactly pb200_scalar_mul_batch; a negative sign with magnitude 0 is k = 0 (output 1, no error, even for c = 0).  The scalars are
 * not reduced mod n: the output is c^k mod n^2 exactly.
 * A unit whose inverse does not exist (gcd(c mod n^2, n) != 1; for sub the c2 operand) gets 0; the others are still computed.  The host
 * variants copy every output back and then return PB200_ERR_NOT_INVERTIBLE; _dev raises PB200_FLAG_NOT_INVERTIBLE in the flag word.
 * PB200_ERR_EVEN_MODULUS for an even n (pb200_scalar_mul_signed_batch* only when k_neg is non-null).  PB200_ERR_INVALID_ARG for null
 * pointers where data is needed, k_bits == 0 or k_bits > n_bits; PB200_ERR_RANGE (host variant) when a magnitude has a bit at or above
 * k_bits.  count == 0 does nothing.  The first call prepares the per-key constants on the device (synchronises once).
 * _dev: device pointers on the key's device, enqueued on the key's stream, no final synchronise, magnitudes are not range-checked. */
int pb200_inverse_batch(pb200_key* key, const uint64_t* c_le, size_t count, uint64_t* out_le);
int pb200_inverse_batch_dev(pb200_key* key, const uint64_t* d_c_le, size_t count, uint64_t* d_out_le);
int pb200_sub_batch(pb200_key* key, const uint64_t* c1_le, const uint64_t* c2_le, size_t count, uint64_t* out_le);
int pb200_sub_batch_dev(pb200_key* key, const uint64_t* d_c1_le, const uint64_t* d_c2_le, size_t count, uint64_t* d_out_le);
int pb200_scalar_mul_signed_batch(pb200_key* key, const uint64_t* c_le, const uint64_t* k_mag_le, const uint8_t* k_neg, uint32_t k_bits,
                                  size_t count, uint64_t* out_le);
int pb200_scalar_mul_signed_batch_dev(pb200_key* key, const uint64_t* d_c_le, const uint64_t* d_k_mag_le, const uint8_t* d_k_neg,
                                      uint32_t k_bits, size_t count, uint64_t* d_out_le);

/* ---- threshold decryption (Fouque-Poupard-Stern 2000, Shoup 2000, Damgard-Jurik 2001) --------------------------------------------
 * The decryption key is split among l = parties trustees so that any t + 1 of them decrypt and t learn nothing; no party holds lambda.
 * With M = n lambda, Delta = l! and L(x) = (x - 1) / n, a dealer (host key material, not in the library) takes d = lambda (lambda^-1 mod n)
 * (d = 0 mod lambda, d = 1 mod n), a random polynomial f(X) = d + a_1 X + .. + a_t X^t mod M, the shares s_i = f(i) for i = 1 .. l, and
 * phi = L(g^(4 Delta^2 d) mod n^2)^-1 mod n (for g = n + 1: (4 Delta^2)^-1 mod n).
 *   pb200_partial_decrypt_batch:  trustee i, out_u = c_u^(2 Delta s_i) mod n^2
 *   pb200_combine_shares_batch:   over a set S of distinct indices, mu_j = Delta prod_(j' in S, j' != j) j' / (j' - j) (an integer, may be
 *                                 negative), P = prod_(mu_j > 0) c_j^(2 mu_j), N = prod_(mu_j < 0) c_j^(2 |mu_j|) mod n^2, m = L(P N^-1 mod n^2) phi mod n
 * With |S| >= t + 1 honest shares m = Dec(c) for any g; with t shares or a corrupted one P N^-1 is not 1 mod n (except with negligible
 * probability) and the unit raises PB200_ERR_DECRYPT.  Shares are not verified: a malicious trustee can shift m undetected.
 *
 * pb200_key_set_threshold: parties (1 .. 32) and phi (words_in words); clears any share set on the key.  PB200_ERR_INVALID_ARG for
 * parties 0 or > 32, PB200_ERR_RANGE for phi >= 2^n_bits.  pb200_key_set_share: trustee `index` (1 .. parties, after set_threshold,
 * else PB200_ERR_INVALID_ARG) and its share s (words_out words, any value); the library forms 2 Delta s and prepares its schedule.  A key
 * can hold the private part and a share together.
 * pb200_partial_decrypt_batch: c: count * words_out words (any value); out: count * words_out words, canonical.  Runs on the key's engine
 * (block28: sliding window over the per-key exponent, as decryption).  PB200_ERR_INVALID_ARG when no share is set.
 * pb200_combine_shares_batch: indices: k host integers (a host array in _dev too); shares: share-major, share j of unit u at
 * (j * count + u) * words_out words; m_out: count * words_in words.  On a block28 key one multi-exponentiation per sign (Straus's
 * method: one squaring chain for all the shares of a unit), then one inverse mod n^2 when some mu_j < 0, then L and phi.
 * PB200_ERR_INVALID_ARG without set_threshold, for k == 0, an index 0 or > parties or an index given twice; PB200_ERR_EVEN_MODULUS for
 * an even n when some mu_j < 0.  A unit whose N has no inverse gets m = 0 and raises PB200_FLAG_NOT_INVERTIBLE; an inexact L gives
 * m = 0 and raises PB200_FLAG_DECRYPT.  The host variant copies every output back, then returns the status of the flags.  count == 0
 * does nothing.  The first call on an index set prepares its schedules on the device (and, with a negative mu_j, the inverse's
 * constants once per key); later _dev calls on the set enqueue without a synchronise.
 * _dev: device pointers on the key's device, enqueued on the key's stream, no final synchronise; failures only raise flags. */
int pb200_key_set_threshold(pb200_key* key, uint32_t parties, const uint64_t* phi_le);
int pb200_key_set_share(pb200_key* key, uint32_t index, const uint64_t* s_le);
int pb200_partial_decrypt_batch(pb200_key* key, const uint64_t* c_le, size_t count, uint64_t* out_le);
int pb200_partial_decrypt_batch_dev(pb200_key* key, const uint64_t* d_c_le, size_t count, uint64_t* d_out_le);
int pb200_combine_shares_batch(pb200_key* key, const uint32_t* indices, uint32_t k, const uint64_t* shares_le, size_t count, uint64_t* m_out_le);
int pb200_combine_shares_batch_dev(pb200_key* key, const uint32_t* indices, uint32_t k, const uint64_t* d_shares_le, size_t count,
                                   uint64_t* d_m_out_le);

/* ---- encrypted matrix-vector product with a signed plaintext matrix ------------------------------------------------------
 * Enc(W m) from Enc(m): private scoring with a linear model, multi-question ballots, PIR-style selection.  On a block28 engine a
 * bucket (Pippenger) multi-exponentiation shared by all the ciphertexts of a row (about ceil(k_bits / c) multiplications per
 * ciphertext and row, c <= 16), else per row and sign the weighted tally's chains (the "chain" method; simple64 keys always).
 *
 * out_r = P_r * N_r^(n-1) mod n^2 for r < rows, where
 *   P_r = prod_{i: w_ri > 0} c_i^|w_ri| mod n^2,   N_r = prod_{i: w_ri < 0} c_i^|w_ri| mod n^2   (empty product = 1)
 * so that Dec(out_r) = sum_i w_ri * Dec(c_i) mod n.  c: count * words_out words (any value, reduced mod n^2);
 * w_mag: rows * count * PB200_WORDS(k_bits) words, row-major (entry (r, i) at (r * count + i) * PB200_WORDS(k_bits));
 * w_neg: nullable, rows * count bytes, non-zero = that weight is negative;  out: rows * words_out words, canonical.
 * A row without negative weights equals pb200_tally_weighted of that row bit for bit.  count == 0 gives 1 for every row, rows == 0
 * does nothing.  PB200_ERR_INVALID_ARG for null pointers where data is needed, k_bits == 0 or k_bits > n_bits; PB200_ERR_RANGE
 * (host variant) when a magnitude has a bit at or above k_bits.  Temporary device memory stays within 3 * 2^18 * 8 * words_out bytes
 * (384 MB at |n| = 2048) whatever rows, count and k_bits (work proceeds in passes; the host variant's staged inputs come on top).
 * _dev: device pointers, enqueued on the key's stream, no final synchronise, magnitudes are not range-checked; the sign step runs
 * whenever d_w_neg is non-null.  The first call with negative weights prepares copies of n - 1 on the device (synchronises once). */
int pb200_matvec(pb200_key* key, const uint64_t* c_le, size_t count, const uint64_t* w_mag_le, const uint8_t* w_neg,
                 uint32_t k_bits, size_t rows, uint64_t* out_le);
int pb200_matvec_dev(pb200_key* key, const uint64_t* d_c_le, size_t count, const uint64_t* d_w_mag_le, const uint8_t* d_w_neg,
                     uint32_t k_bits, size_t rows, uint64_t* d_out_le);
/* host only, no device needed: the plan pb200_matvec would use for a key of n_bits on a GPU of `sms` SMs running a block28 engine
 * (the same planner; PB200_MATVEC_METHOD and PB200_MATVEC_PASS_ENTRIES apply).  out11: method (0 chain, 1 bucket), window width c,
 * windows J, passes, bucket segments per window, then upper bounds for dense weights of the multiplications of accumulation,
 * reduction, Horner and the sign step, the longest sequential chain of multiplications, and the temporary device bytes. */
int pb200_matvec_plan(uint32_t n_bits, int sms, size_t rows, size_t count, uint32_t k_bits, int has_neg, uint64_t* out11);

/* ---- witness --------------------------------------------------------------------------------
 * Replaces: the witness generation inside BigUintChip::pow_mod_fixed_exp / mul_mod that
 * PaillierChip::encrypt drives (src/paillier.rs:51,55,57).  Every mul_mod(a, b, n^2) of the chain
 * contributes one RECORD = q (words_out words) followed by rem (words_out words) with
 * q = floor(a*b / n^2), rem = a*b mod n^2.  Chain order per unit (SURVEY.md Appendix A.5):
 *   g-chain : for bit i of m, low to high:  sqr_i = (g^(2^i))^2 ;  if bit set: mul = acc * g^(2^i)
 *   r-chain : for bit i of n, low to high:  sqr_i = (r^(2^i))^2 ;  if bit set: mul = acc * r^(2^i)
 *   final   : gm * rn
 * The g-chain squarings depend on the key only; they are produced once per key
 * (pb200_key_g_chain) and are NOT repeated in the per-unit stream.  The per-unit stream therefore
 * holds, in order: popcount(m) g-chain mul records, bits(n)+popcount(n) r-chain records (sqr and
 * mul interleaved as above), 1 final record. */
typedef struct pb200_witness_chunk {
    size_t first_unit;             /* index of the first unit in this chunk                        */
    size_t n_units;                /* units in this chunk                                          */
    uint32_t words_out;            /* words per q / per rem                                        */
    const uint64_t* offsets;       /* n_units+1 record offsets into `records` (unit u: [off[u], off[u+1])) */
    const uint64_t* records;       /* records, each 2*words_out words: q then rem                  */
    const uint32_t* g_mul_counts;  /* n_units: number of g-chain mul records at the head of each unit */
} pb200_witness_chunk;

/* called on the calling thread; chunk memory (pinned host memory owned by the library) is valid only during the call;
 * return 0 to continue */
typedef int (*pb200_witness_sink_fn)(void* user, const pb200_witness_chunk* chunk);

/* Delivery: the stream does not fit anywhere whole (4 MB per unit at |n| = 2048), so it is produced on the device in chunks
 * (two record buffers sized from the free device memory: the kernel of the next chunk runs while this one drains) and handed
 * to the sink in pieces of whole units through a ring of four pinned staging slots filled by a second stream — while the sink
 * works on one piece the next three are crossing PCIe.  max_chunk_units bounds the units per sink call (0: as many as fit a
 * staging slot, 256 MiB unless PB200_WITNESS_SLOT_BYTES says otherwise; PB200_WITNESS_CHUNK_BYTES bounds a device chunk).
 * c_out (nullable) receives the ciphertexts of a chunk before its first piece is delivered. */
int pb200_encrypt_witness_batch(pb200_key* key, const uint64_t* m_le, const uint64_t* r_le, size_t count,
                                uint64_t* c_out_le /* nullable */, size_t max_chunk_units,
                                pb200_witness_sink_fn sink, void* user);

/* number of records unit (m) contributes to the per-unit stream: popcount(m) + bits(n) + popcount(n) + 1 */
uint64_t pb200_witness_records_for(const pb200_key* key, const uint64_t* m_le);

/* 64-bit digest of each unit's record stream, computed on the device without materialising the
 * witness on the host: digest_out[count].  Per record H = sum_j w_j * C^(j+1) mod 2^64 over its
 * 2*words_out words (q then rem), C = 0x9E3779B97F4A7C15; per unit D = 0xcbf29ce484222325, then
 * D = (D ^ H) * 0x100000001b3 mod 2^64 for each record in stream order. */
int pb200_encrypt_witness_digest(pb200_key* key, const uint64_t* m_le, const uint64_t* r_le, size_t count,
                                 uint64_t* c_out_le /* nullable */, uint64_t* digest_out);

/* device-resident variant: d_m, d_r (count * words_in words), d_c_out (nullable, count * words_out words) and
 * d_digest_out (count words) on the key's device; enqueued on the key's stream, no final synchronise, inputs
 * are not range-checked (the host variant checks them against n_bits) */
int pb200_encrypt_witness_digest_dev(pb200_key* key, const uint64_t* d_m_le, const uint64_t* d_r_le, size_t count,
                                     uint64_t* d_c_out_le /* nullable */, uint64_t* d_digest_out);
/* name of the engine that produces this key's witnesses: "block28w" (block28t arithmetic with an exact
 * canonicalising tail per mul_mod) when the fast engine is selected and n has exactly n_bits bits, else "simple64" */
const char* pb200_key_witness_engine(pb200_key* key);

/* per-key g-chain squarings: record i (i < n_bits) = (q, rem) of (g^(2^i) mod n^2)^2 mod n^2.
 * out: n_bits * 2 * words_out words. */
int pb200_key_g_chain(pb200_key* key, uint64_t* records_out);

/* ---- limb formatting (K5) ------------------------------------------------------------------
 * Replaces: decompose_biguint inside BigUintChip::assign_integer for limb_bits != 64
 * (src/paillier.rs:187 uses 88).  Pure bit repack, host-side convenience over a device kernel:
 * values of `value_bits` bits (PB200_WORDS words each) -> value_bits/limb_bits limbs, each limb
 * stored in 2 words (low, high) so that 64 < limb_bits <= 128 fits. */
int pb200_repack_limbs(pb200_key* key, const uint64_t* values_le, size_t count, uint32_t value_bits,
                       uint32_t limb_bits, uint64_t* limbs_out /* count * (value_bits/limb_bits) * 2 words */);

/* ---- advice cells (K4) -----------------------------------------------------------------------
 * Replaces: the witness-cell arithmetic BigUintChip performs around every mul_mod that PaillierChip::encrypt/add
 * issue (src/paillier.rs:51,55,57,81), of assign_integer (src/bench.rs:44-66) and of the square+refresh of n
 * (src/paillier.rs:39-45, :69-75); semantics in SURVEY.md Appendix A.1-A.4, A.6.  A CELL is one BN254 Fr advice
 * value = 4 little-endian u64 words: the canonical integer (montgomery = 0; the values never wrap the field) or
 * its Montgomery form x * 2^256 mod p (montgomery = 1), the in-memory representation of halo2curves' Fr.
 * lookup_bits = RangeChip lookup width (15 and 13 in the reference, src/paillier.rs:169, src/bench.rs:163);
 * 0 omits the range-check decomposition cells.
 *
 * Cell order of one mul_mod(a, b, n^2) group (L = 2*n_bits/limb_bits limbs):
 *   q    : per limb [limb, ceil(limb_bits/lookup_bits) chunks (low to high), top chunk << pad if limb_bits % lookup_bits]
 *   rem  : same
 *   ab   : 2L-1 no-carry columns  sum_j a_j b_(i-j)
 *   qn   : 2L-1 columns of q * n^2
 *   qn+r : 2L-1 sums (rem_i added for i < L)
 *   eq   : per column i: carry_(i+1), cs_i, q_acc_i, mod_acc_i, then (i < 2L-2) the chunks of carry_(i+1) at carry_bits
 *   1 cell: the is_equal_muled flag (1). */
typedef struct pb200_cell_layout {
    uint32_t limbs;              /* L */
    uint32_t cells_per_limb;     /* 1 + chunks + (limb_bits % lookup_bits != 0) */
    uint32_t carry_bits;
    uint32_t cells_per_mulmod;
    uint32_t cells_n2;           /* cells of square(n) + refresh */
    uint32_t off_rem, off_ab, off_qn, off_qn_rem, off_eq, eq_stride;
} pb200_cell_layout;
int pb200_cells_layout(pb200_key* key, uint32_t lookup_bits, pb200_cell_layout* out);
/* a, b, q, rem: count * words_out words each (q, rem as produced by the witness stream / pb200_add_batch);
 * cells_out: count * cells_per_mulmod * 4 words.  PB200_ERR_CONSTRAINT if some (q, rem) does not satisfy
 * a*b = q*n^2 + rem (the chip's equality constraint would fail).  _dev: device pointers, no synchronise,
 * no check. */
int pb200_mulmod_cells_batch(pb200_key* key, const uint64_t* a_le, const uint64_t* b_le, const uint64_t* q_le,
                             const uint64_t* rem_le, size_t count, uint32_t lookup_bits, int montgomery,
                             uint64_t* cells_out);
int pb200_mulmod_cells_batch_dev(pb200_key* key, const uint64_t* d_a_le, const uint64_t* d_b_le, const uint64_t* d_q_le,
                                 const uint64_t* d_rem_le, size_t count, uint32_t lookup_bits, int montgomery,
                                 uint64_t* d_cells_out);
/* assign_integer(value, value_bits) for `count` values of PB200_WORDS(value_bits) words:
 * cells_out: count * (value_bits/limb_bits) * cells_per_limb * 4 words */
int pb200_assign_cells_batch(pb200_key* key, const uint64_t* values_le, size_t count, uint32_t value_bits,
                             uint32_t lookup_bits, int montgomery, uint64_t* cells_out);
/* square(n) columns, the refresh div/mod chain, the range-check chunks of the refreshed n^2 limbs:
 * cells_out: cells_n2 * 4 words */
int pb200_key_n2_cells(pb200_key* key, uint32_t lookup_bits, int montgomery, uint64_t* cells_out);

#ifdef __cplusplus
}
#endif
#endif /* PAILLIER_B200_H */
