// capi.cu — the C ABI declared in include/paillier_b200.h.
//
// Host-side glue only: validation (the reference's range checks / panics mapped to status codes),
// per-key constant setup, staging copies and engine dispatch.  All arithmetic per ciphertext runs in
// CUDA kernels (block28_kernels.cu, simple64_kernels.cu); there is no CPU fallback.
#include "../../include/paillier_b200.h"
#include "engine.hpp"
#include "cells.hpp"
#include <cstring>
#include <cstdlib>
#include <map>
#include <memory>
#include <mutex>
#include <new>

using namespace pb200;

static thread_local std::string t_cuda_error;

static int cuda_fail(cudaError_t e, const char* where) {
    t_cuda_error = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return PB200_ERR_NOMEM; }
    return PB200_ERR_CUDA;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(e_, #call); } while (0)

// Nothing may unwind through an extern "C" frame: every entry point is a function-try-block ending in PB200_CATCH.
#define PB200_CATCH \
    catch (const std::bad_alloc&) { t_cuda_error = "host allocation failed"; return PB200_ERR_NOMEM; } \
    catch (const std::exception& ex_) { t_cuda_error = std::string("internal: ") + ex_.what(); return PB200_ERR_UNSUPPORTED; } \
    catch (...) { t_cuda_error = "internal: unknown exception"; return PB200_ERR_UNSUPPORTED; }

// Entry points run on the key's device and put the caller's current device back when they return.
struct DevGuard {
    int prev = -1; bool changed = false;
    cudaError_t set(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; }
        if (prev == dev) return cudaSuccess;
        cudaError_t e = cudaSetDevice(dev);
        changed = e == cudaSuccess;
        return e;
    }
    ~DevGuard() { if (changed && prev >= 0) cudaSetDevice(prev); }
};
#define USE_DEVICE(k) DevGuard dev_guard_; CU(dev_guard_.set((k)->device))

struct DevBuf {  // grow-only device buffer
    void* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct pb200_key {
    int device = 0;
    cudaStream_t stream = nullptr;
    uint32_t n_bits = 0, limb_bits = 0, words_in = 0, words_out = 0;
    BigInt n, g, n2;
    SimpleConsts* d_simple = nullptr;
    u64* d_gchain = nullptr;        // lazy: n_bits records
    int* d_flags = nullptr;
    Block28Key* fast = nullptr;
    std::string fast_why;
    int engine = 0;                 // 0 auto, 1 simple64, 2 block28, 3 block28t, 4 block28u, 5 block28u2
    DevBuf in_a, in_b, out_a, out_b, scratch, offs;
    DevBuf wt_chunk, wt_part;               // weighted tally: one chunk's scalar products, the per-chunk partial products
    DevBuf mv_arena, mv_neg, mv_nm1;        // matvec: temporary memory of the plan, staged signs, copies of n - 1 for the sign step
    size_t mv_nm1_units = 0;
    DevBuf tr_tmp;                          // running-tally trace: per-level chunk totals and the leaf chunks' carries
    std::string engine_name;
    // K4 cell expansion: per lookup_bits layout + device constants (n^2 limbs, word_max, q_acc, mod_acc), refresh spill vector
    struct CellCtx { CellLayout Y; u64* d_consts = nullptr; int* d_inc = nullptr; u64* d_mtab = nullptr; int n_out = 0; int n2_cells = 0; };
    std::map<uint32_t, CellCtx> cells;
    DevBuf cin_a, cin_b, cin_q, cin_r;
    int sms = 148;
    std::vector<pb200_key*> group;          // pb200_tally_multi: the peer group this key is connected to (single process)
    // private part (pb200_key_set_private): constants of the modulus n with mu in their g slot, lambda's words for the simple pow
    SimpleConsts* d_simple_n = nullptr; u64* d_lambda = nullptr; int lambda_bits = 0; bool has_private = false;
    // witness delivery pipeline (pb200_encrypt_witness_batch): created on first use
    struct Pipe {
        static const int NS = 4;             // pinned staging slots
        cudaStream_t copy = nullptr;
        cudaEvent_t kern_done[2] = {}, buf_free[2] = {}, slot_done[NS] = {};
        void* pinned[NS] = {}; size_t slot_bytes = 0;
        DevBuf rec[2], cbuf[2], offs[2], m_in[2], r_in[2];
        bool ready = false;
    } pipe;
};

static bool use_fast(const pb200_key* k) { return k->fast && k->engine != 1; }

extern "C" {

const char* pb200_strerror(int s) {
    switch (s) {
        case PB200_OK: return "ok";
        case PB200_ERR_INVALID_ARG: return "invalid argument";
        case PB200_ERR_ZERO_MODULUS: return "modulus n is zero (num-bigint would panic)";
        case PB200_ERR_EVEN_MODULUS: return "modulus n is even (reserved; even n is accepted)";
        case PB200_ERR_RANGE: return "input does not fit its declared bit width (range check fails)";
        case PB200_ERR_UNSUPPORTED: return "key size not supported by any compiled engine";
        case PB200_ERR_CUDA: return "CUDA failure";
        case PB200_ERR_NOMEM: return "out of memory";
        case PB200_ERR_SINK: return "witness sink aborted";
        case PB200_ERR_PEER: return "a peer GPU's tally partial did not arrive (every rank of the group must make the same call)";
        case PB200_ERR_DECRYPT: return "not a valid ciphertext for this key: c^lambda mod n^2 is not 1 modulo n";
        case PB200_ERR_CONSTRAINT: return "(q, rem) do not satisfy a*b = q*n^2 + rem (the chip's equality constraint fails)";
        default: return "unknown status";
    }
}
const char* pb200_last_cuda_error(void) { return t_cuda_error.c_str(); }
const char* pb200_version(void) { return "paillier_b200 0.1 (sm_100a)"; }
int pb200_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; } return n; }
uint64_t pb200_kernel_launches(void) { return g_kernel_launches.load(); }

static bool fits(const uint64_t* v, uint32_t words, uint32_t bits) {
    for (uint32_t i = 0; i < words; i++) {
        uint32_t lo = i * 64;
        if (lo >= bits) { if (v[i]) return false; }
        else if (bits - lo < 64) { if (v[i] >> (bits - lo)) return false; }
    }
    return true;
}

int pb200_key_create(int device, uint32_t n_bits, uint32_t limb_bits, const uint64_t* n_le, const uint64_t* g_le,
                     pb200_key** out) try {
    if (!out) return PB200_ERR_INVALID_ARG;
    *out = nullptr;
    if (!n_le || !g_le || n_bits == 0 || limb_bits == 0 || limb_bits > 128) return PB200_ERR_INVALID_ARG;
    if (n_bits % limb_bits != 0) return PB200_ERR_INVALID_ARG;  // assign_integer asserts bit_len % limb_bits == 0
    uint32_t win = PB200_WORDS(n_bits), wout = PB200_WORDS(2 * n_bits);
    if (wout > PB200_SIMPLE_MAXK) return PB200_ERR_UNSUPPORTED;
    if (!fits(n_le, win, n_bits) || !fits(g_le, win, n_bits)) return PB200_ERR_RANGE;
    BigInt n = BigInt::from_u64_le(n_le, win), g = BigInt::from_u64_le(g_le, win);
    if (n.is_zero()) return PB200_ERR_ZERO_MODULUS;
    // even n is accepted: the reference's own tests draw n = rng.gen_biguint(bits) (src/paillier.rs:173,251) and nothing in the
    // Barrett engines needs an odd modulus (PB200_ERR_EVEN_MODULUS stays in the enum for ABI stability, never returned)
    int ndev = pb200_device_count();
    if (device < 0 || device >= ndev) { t_cuda_error = "no such CUDA device"; return PB200_ERR_CUDA; }
    DevGuard dev_guard_; CU(dev_guard_.set(device));
    pb200_key* k = new (std::nothrow) pb200_key();
    if (!k) return PB200_ERR_NOMEM;
    struct KeyOwner { pb200_key* k; ~KeyOwner() { if (k) pb200_key_destroy(k); } } owner{k};   // released on success
    k->device = device; k->n_bits = n_bits; k->limb_bits = limb_bits; k->words_in = win; k->words_out = wout;
    k->n = n; k->g = g; k->n2 = BigInt::mul(n, n);
    SimpleConsts* h = new SimpleConsts();
    memset(h, 0, sizeof(*h));
    h->k = (int)wout; h->kin = (int)win; h->n_bits = (int)n_bits; h->exp_bits = (int)n.bits();
    h->s = (int)(64 * wout - k->n2.bits());
    BigInt Nt = BigInt::shl(k->n2, h->s);
    BigInt mu = BigInt::div(BigInt::pow2(128 * (size_t)wout), Nt);
    Nt.to_u64_le(h->Nt, wout); mu.to_u64_le(h->mu, wout + 1);
    n.to_u64_le(h->n, win); g.to_u64_le(h->g, win);
    cudaError_t e = cudaStreamCreateWithFlags(&k->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&k->d_simple, sizeof(SimpleConsts));
    if (e == cudaSuccess) e = cudaMalloc(&k->d_flags, sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpyAsync(k->d_simple, h, sizeof(SimpleConsts), cudaMemcpyHostToDevice, k->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(k->d_flags, 0, sizeof(int), k->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(k->stream);
    delete h;
    if (e != cudaSuccess) return cuda_fail(e, "pb200_key_create");
    cudaError_t fe = cudaSuccess;
    { cudaDeviceProp prop; if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) k->sms = prop.multiProcessorCount; }
    k->fast = block28_create(n, g, n_bits, device, k->stream, &k->fast_why, &fe);
    if (fe != cudaSuccess) return cuda_fail(fe, "block28_create");
    k->engine_name = k->fast ? block28_name(k->fast) : "simple64";
    owner.k = nullptr;
    *out = k;
    return PB200_OK;
} PB200_CATCH

void pb200_key_destroy(pb200_key* k) {
    if (!k) return;
    DevGuard dev_guard_; dev_guard_.set(k->device);
    if (k->stream) cudaStreamSynchronize(k->stream);
    if (k->fast) block28_destroy(k->fast);
    if (k->d_simple) cudaFree(k->d_simple);
    if (k->d_gchain) cudaFree(k->d_gchain);
    if (k->d_flags) cudaFree(k->d_flags);
    if (k->d_simple_n) cudaFree(k->d_simple_n);
    if (k->d_lambda) cudaFree(k->d_lambda);
    k->in_a.release(); k->in_b.release(); k->out_a.release(); k->out_b.release(); k->scratch.release(); k->offs.release();
    k->wt_chunk.release(); k->wt_part.release();
    k->mv_arena.release(); k->mv_neg.release(); k->mv_nm1.release();
    k->tr_tmp.release();
    k->cin_a.release(); k->cin_b.release(); k->cin_q.release(); k->cin_r.release();
    if (k->pipe.ready) {
        if (k->pipe.copy) { cudaStreamSynchronize(k->pipe.copy); cudaStreamDestroy(k->pipe.copy); }
        for (int i = 0; i < 2; i++) {
            if (k->pipe.kern_done[i]) cudaEventDestroy(k->pipe.kern_done[i]);
            if (k->pipe.buf_free[i]) cudaEventDestroy(k->pipe.buf_free[i]);
            k->pipe.rec[i].release(); k->pipe.cbuf[i].release(); k->pipe.offs[i].release(); k->pipe.m_in[i].release(); k->pipe.r_in[i].release();
        }
        for (int i = 0; i < pb200_key::Pipe::NS; i++) {
            if (k->pipe.slot_done[i]) cudaEventDestroy(k->pipe.slot_done[i]);
            if (k->pipe.pinned[i]) cudaFreeHost(k->pipe.pinned[i]);
        }
    }
    for (auto& kv : k->cells) { if (kv.second.d_consts) cudaFree(kv.second.d_consts); if (kv.second.d_inc) cudaFree(kv.second.d_inc); if (kv.second.d_mtab) cudaFree(kv.second.d_mtab); }
    if (k->stream) cudaStreamDestroy(k->stream);
    delete k;
}
uint32_t pb200_key_n_bits(const pb200_key* k) { return k ? k->n_bits : 0; }
uint32_t pb200_key_words_in(const pb200_key* k) { return k ? k->words_in : 0; }
uint32_t pb200_key_words_out(const pb200_key* k) { return k ? k->words_out : 0; }
int pb200_key_device(const pb200_key* k) { return k ? k->device : -1; }
int pb200_key_n2(const pb200_key* k, uint64_t* out) try {
    if (!k || !out) return PB200_ERR_INVALID_ARG;
    k->n2.to_u64_le(out, k->words_out);
    return PB200_OK;
} PB200_CATCH
const char* pb200_key_engine(const pb200_key* k) {
    if (!k) return "";
    return use_fast(k) ? k->engine_name.c_str() : "simple64";
}
// internal numbering of the block28 family: 0 block28, 1 block28t, 2 block28u (32 ciphertexts per CTA), 3 block28u2 (64).
// *eng <- the internal number of public engine 2..5; false when the key has no block28 engine or its configuration lacks that one.
static bool fast_engine(const pb200_key* k, int engine, int* eng) {
    *eng = engine - 2;
    return k->fast && block28_has_engine(k->fast, *eng);
}
int pb200_key_set_engine(pb200_key* k, int engine) try {
    if (!k || engine < 0 || engine > 5) return PB200_ERR_INVALID_ARG;
    int eng = -1;                   // 0 (automatic) and 1 (simple64) leave the fastest block28 engine selected on the key
    if (engine >= 2 && !fast_engine(k, engine, &eng)) return PB200_ERR_UNSUPPORTED;
    k->engine = engine;
    if (k->fast) { block28_set_engine(k->fast, eng); k->engine_name = block28_name(k->fast); }
    return PB200_OK;
} PB200_CATCH
void* pb200_key_stream(const pb200_key* k) { return k ? (void*)k->stream : nullptr; }
int pb200_key_chain_counts(const pb200_key* k, uint64_t* n_sqr, uint64_t* n_mul) try {
    if (!k || !n_sqr || !n_mul) return PB200_ERR_INVALID_ARG;
    if (use_fast(k)) { block28_chain_counts(k->fast, n_sqr, n_mul); return PB200_OK; }
    // simple64 runs the reference's LSB-first chain: bits(n) squarings; popcount(n) + ~popcount(m) + 1 multiplications
    uint64_t pn = 0; for (size_t i = 0; i < k->n.w.size(); i++) pn += (uint64_t)__builtin_popcount(k->n.w[i]);
    *n_sqr = k->n.bits(); *n_mul = pn + k->n_bits / 2 + 1;
    return PB200_OK;
} PB200_CATCH
int pb200_key_sync(pb200_key* k) try {
    if (!k) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    CU(cudaStreamSynchronize(k->stream));
    return PB200_OK;
} PB200_CATCH

// The per-key device flag word: bit 0 (PB200_FLAG_RANGE) a quotient / input outside its declared width, bit 1
// (PB200_FLAG_CONSTRAINT) a (q, rem) that does not satisfy a*b = q*n^2 + rem.  Host entry points clear it when they start
// (clear_flags) and turn it into a status when they end (take_flags); _dev callers read it with pb200_key_take_flags.
static int clear_flags(pb200_key* k) {
    CU(cudaMemsetAsync(k->d_flags, 0, sizeof(int), k->stream));
    return PB200_OK;
}
static int read_flags(pb200_key* k, int* f) {
    *f = 0;
    CU(cudaMemcpyAsync(f, k->d_flags, sizeof(int), cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    if (*f) CU(cudaMemsetAsync(k->d_flags, 0, sizeof(int), k->stream));
    return PB200_OK;
}
static int take_flags(pb200_key* k) {
    int f = 0;
    int rc = read_flags(k, &f); if (rc) return rc;
    if (f & PB200_FLAG_CONSTRAINT) return PB200_ERR_CONSTRAINT;
    if (f & PB200_FLAG_DECRYPT) return PB200_ERR_DECRYPT;
    if (f & ~(PB200_FLAG_CONSTRAINT | PB200_FLAG_DECRYPT)) return PB200_ERR_RANGE;
    return PB200_OK;
}
int pb200_key_take_flags(pb200_key* k, uint32_t* flags_out) try {
    if (!k || !flags_out) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    int f = 0;
    int rc = read_flags(k, &f); if (rc) return rc;
    *flags_out = (uint32_t)f;
    return PB200_OK;
} PB200_CATCH

// Diagnostic entry: one CTA (32 lanes) of the fast engine's modular multiplication on raw lazy digits, on engine 2 / 3 / 4.
int pb200_debug_mulmod(pb200_key* k, int engine, const int32_t* v_in, const int32_t* y_in, int reps, int32_t* v_out, int32_t* t_out,
                       uint32_t* qhat_rows) try {
    if (!k || !v_in || engine < 2 || engine > 5 || (!v_out && !t_out) || reps < 1) return PB200_ERR_INVALID_ARG;
    int eng;
    if (!fast_engine(k, engine, &eng)) return PB200_ERR_UNSUPPORTED;
    USE_DEVICE(k);
    CU(block28_debug_mulmod(k->fast, eng, v_in, y_in, reps, v_out, t_out, qhat_rows, k->stream));
    return PB200_OK;
} PB200_CATCH
int pb200_debug_mulmod_cycles(pb200_key* k, int engine, const int32_t* v_in, int ctas, int reps, int stagger_cycles, int64_t* cycles_out) try {
    if (!k || !v_in || !cycles_out || engine < 3 || engine > 5 || ctas < 1 || reps < 1) return PB200_ERR_INVALID_ARG;
    int eng;
    if (!fast_engine(k, engine, &eng)) return PB200_ERR_UNSUPPORTED;
    { int g = 0, bl = 0; block28_shape(k->fast, &g, &bl); if (g != 8) return PB200_ERR_UNSUPPORTED; }      // the |n| = 2048 configuration only
    USE_DEVICE(k);
    CU(block28_debug_time(k->fast, eng, v_in, ctas, reps, stagger_cycles, (long long*)cycles_out, k->stream));
    return PB200_OK;
} PB200_CATCH
int pb200_umma_layout(int g, int bl, int lane_groups, int witness, int32_t* out20) try {
    if (!out20) return PB200_ERR_INVALID_ARG;
    return block28_umma_layout(g, bl, lane_groups, witness, out20) ? PB200_OK : PB200_ERR_UNSUPPORTED;
} PB200_CATCH
int pb200_key_shape(const pb200_key* k, int* g_out, int* bl_out) {
    if (!k || !g_out || !bl_out) return PB200_ERR_INVALID_ARG;
    if (!k->fast) return PB200_ERR_UNSUPPORTED;
    block28_shape(k->fast, g_out, bl_out);
    return PB200_OK;
}

// per-key g-chain records: by the witness engine when it serves this key (it builds its table in the same pass), else by
// simple64 (one thread, the reference's chain)
static int ensure_gchain(pb200_key* k) {
    if (k->d_gchain) return PB200_OK;
    CU(cudaMalloc(&k->d_gchain, (size_t)k->n_bits * 2 * k->words_out * sizeof(u64)));
    if (use_fast(k) && block28_witness_supported(k->fast)) CU(block28_witness_prepare(k->fast, k->d_gchain, false, k->stream));
    else CU(simple_gchain(k->d_simple, k->d_gchain, (int)k->n_bits, k->stream));
    return PB200_OK;
}

// witness producer for this key: the block28t witness engine when the fast engine is selected and n fills its
// declared width, else simple64 (both on the GPU).  Prepares the per-key tables on first use.
static int witness_engine(pb200_key* k, bool* fast) {
    *fast = false;
    int rc = ensure_gchain(k); if (rc) return rc;
    if (!use_fast(k) || !block28_witness_supported(k->fast)) return PB200_OK;
    CU(block28_witness_prepare(k->fast, k->d_gchain, true, k->stream));
    *fast = true;
    return PB200_OK;
}
static int run_witness(pb200_key* k, const u64* d_m, const u64* d_r, size_t count, u64* d_c, u64* d_records,
                       const u64* d_offsets, u64* d_digest) {
    bool fast = false;
    int rc = witness_engine(k, &fast); if (rc) return rc;
    if (fast) CU(block28_witness(k->fast, d_m, d_r, count, d_c, d_records, d_offsets, d_digest, k->stream));
    else CU(simple_encrypt(k->d_simple, k->d_gchain, d_m, d_r, count, d_c, d_records, d_offsets, d_digest, k->d_flags, k->stream));
    return PB200_OK;
}

// ---- encrypt --------------------------------------------------------------------------------
int pb200_encrypt_batch_dev(pb200_key* k, const uint64_t* d_m, const uint64_t* d_r, size_t count, uint64_t* d_c) try {
    if (!k || (count && (!d_m || !d_r || !d_c))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    if (use_fast(k)) { CU(block28_encrypt(k->fast, (const u64*)d_m, (const u64*)d_r, count, (u64*)d_c, k->stream)); return PB200_OK; }
    int rc = ensure_gchain(k); if (rc) return rc;
    CU(simple_encrypt(k->d_simple, k->d_gchain, (const u64*)d_m, (const u64*)d_r, count, (u64*)d_c, nullptr, nullptr,
                      nullptr, k->d_flags, k->stream));
    return PB200_OK;
} PB200_CATCH

static int check_inputs(const pb200_key* k, const uint64_t* v, size_t count) {
    for (size_t u = 0; u < count; u++) if (!fits(v + u * k->words_in, k->words_in, k->n_bits)) return PB200_ERR_RANGE;
    return PB200_OK;
}

int pb200_encrypt_batch(pb200_key* k, const uint64_t* m, const uint64_t* r, size_t count, uint64_t* c_out) try {
    if (!k || (count && (!m || !r || !c_out))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    if (k->n_bits % 64) { int rc = check_inputs(k, m, count); if (rc) return rc; rc = check_inputs(k, r, count); if (rc) return rc; }
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    size_t bin = count * k->words_in * sizeof(u64), bout = count * k->words_out * sizeof(u64);
    CU(k->in_a.reserve(bin)); CU(k->in_b.reserve(bin)); CU(k->out_a.reserve(bout));
    CU(cudaMemcpyAsync(k->in_a.p, m, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->in_b.p, r, bin, cudaMemcpyHostToDevice, k->stream));
    int rc = pb200_encrypt_batch_dev(k, (const uint64_t*)k->in_a.p, (const uint64_t*)k->in_b.p, count, (uint64_t*)k->out_a.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(c_out, k->out_a.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return use_fast(k) ? PB200_OK : take_flags(k);
} PB200_CATCH

// ---- add ------------------------------------------------------------------------------------
int pb200_add_batch_dev(pb200_key* k, const uint64_t* d_c1, const uint64_t* d_c2, uint32_t c_words, size_t count,
                        uint64_t* d_out, uint64_t* d_q) try {
    if (!k || (count && (!d_c1 || !d_c2 || !d_out)) || c_words == 0 || c_words > k->words_out) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    bool fast = false;
    int rc = witness_engine(k, &fast); if (rc) return rc;
    if (fast) CU(block28_add(k->fast, (const u64*)d_c1, (const u64*)d_c2, (int)c_words, count, (u64*)d_out, (u64*)d_q, k->d_flags, k->stream));
    else CU(simple_add(k->d_simple, (const u64*)d_c1, (const u64*)d_c2, (int)c_words, count, (u64*)d_out, (u64*)d_q, k->d_flags, k->stream));
    return PB200_OK;
} PB200_CATCH
int pb200_add_batch(pb200_key* k, const uint64_t* c1, const uint64_t* c2, uint32_t c_words, size_t count, uint64_t* out,
                    uint64_t* q_out) try {
    if (!k || (count && (!c1 || !c2 || !out)) || c_words == 0 || c_words > k->words_out) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    size_t bin = count * c_words * sizeof(u64), bout = count * k->words_out * sizeof(u64);
    CU(k->in_a.reserve(bin)); CU(k->in_b.reserve(bin)); CU(k->out_a.reserve(bout));
    if (q_out) CU(k->out_b.reserve(bout));
    CU(cudaMemcpyAsync(k->in_a.p, c1, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->in_b.p, c2, bin, cudaMemcpyHostToDevice, k->stream));
    int rc = pb200_add_batch_dev(k, (const uint64_t*)k->in_a.p, (const uint64_t*)k->in_b.p, c_words, count,
                                 (uint64_t*)k->out_a.p, q_out ? (uint64_t*)k->out_b.p : nullptr);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, k->out_a.p, bout, cudaMemcpyDeviceToHost, k->stream));
    if (q_out) CU(cudaMemcpyAsync(q_out, k->out_b.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

// ---- tally ----------------------------------------------------------------------------------
static int tally_dev_impl(pb200_key* k, const uint64_t* d_c, size_t count, uint64_t* d_out, bool collective) {
    if (use_fast(k)) {
        if (collective) CU(block28_tally_peer(k->fast, (const u64*)d_c, count, (u64*)d_out, k->stream));
        else CU(block28_tally(k->fast, (const u64*)d_c, count, (u64*)d_out, k->stream));
        return PB200_OK;
    }
    CU(k->scratch.reserve(simple_tally_scratch_words((int)k->words_out) * sizeof(u64)));
    CU(simple_tally(k->d_simple, (int)k->words_out, (const u64*)d_c, count, (u64*)d_out, (u64*)k->scratch.p, k->d_flags, k->stream));
    return PB200_OK;
}
int pb200_tally_dev(pb200_key* k, const uint64_t* d_c, size_t count, uint64_t* d_out) try {
    if (!k || !d_out || (count && !d_c)) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    return tally_dev_impl(k, d_c, count, d_out, false);
} PB200_CATCH
int pb200_tally(pb200_key* k, const uint64_t* c, size_t count, uint64_t* out) try {
    if (!k || !out || (count && !c)) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    size_t bin = count * k->words_out * sizeof(u64), bout = k->words_out * sizeof(u64);
    CU(k->in_a.reserve(bin ? bin : 8)); CU(k->out_b.reserve(bout));
    if (bin) CU(cudaMemcpyAsync(k->in_a.p, c, bin, cudaMemcpyHostToDevice, k->stream));
    int rc = tally_dev_impl(k, (const uint64_t*)k->in_a.p, count, (uint64_t*)k->out_b.p, false);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, k->out_b.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH
int pb200_tally_combine(pb200_key* k, const uint64_t* partials, size_t n_partials, uint64_t* out) try {
    // the combine of per-shard partials is the same fold, on the key's own engine
    return pb200_tally(k, partials, n_partials, out);
} PB200_CATCH

// ---- running-tally trace: every step (q_i, acc_i) = divmod(acc_(i-1) * c_i, n^2) of `chains` chains ---------------------------------
// Level 0 cuts every chain into chunks of s_0 steps, about one wave of lanes over all the chains; every level above cuts the chunk
// totals of the one below the same way, with at least TRACE_MIN_S per chunk, until one chunk covers a chain.  Every level's size
// follows from (count, chains, lanes), so the whole trace is enqueued without a host synchronise.  PB200_TRACE_LANES replaces the
// wave (a development switch: a small wave gives many levels on few steps).
static const size_t TRACE_MIN_S = 4;
static TracePlan trace_plan(size_t count, size_t chains, size_t lanes) {
    TracePlan P;
    size_t n = count, s = (count * chains + lanes - 1) / lanes;
    if (s < 1) s = 1;
    for (;;) {
        P.n.push_back(n); P.s.push_back(s);
        n = (n + s - 1) / s;
        if (n <= 1) return P;
        s = (n * chains + lanes - 1) / lanes;
        if (s < TRACE_MIN_S) s = TRACE_MIN_S;
    }
}
static int trace_dev_impl(pb200_key* k, const u64* d_init, const u64* d_c, size_t count, size_t chains, u64* d_acc, u64* d_q) {
    const size_t wo = k->words_out;
    // phases 1 and 2 on the tally's engine, phase 3 on the witness engine (both simple64 when the key runs no block28 engine)
    const bool fast_scan = use_fast(k), fast_chain = fast_scan && block28_witness_supported(k->fast);
    if (fast_chain) { bool f = false; int rc = witness_engine(k, &f); if (rc) return rc; }
    size_t lanes = fast_scan ? block28_lanes(k->fast) : (size_t)k->sms * 64;
    if (const char* e = getenv("PB200_TRACE_LANES")) { const long long v = atoll(e); if (v >= 1) lanes = (size_t)v; }
    const TracePlan P = trace_plan(count, chains, lanes);
    u64* d_carry = nullptr;                                           // carry-in of level-0 chunk b >= 1; none with one chunk per chain
    if (P.n.size() > 1) {
        if (fast_scan) {
            const size_t scan = block28_trace_scan_bytes(k->fast, P, chains);
            CU(k->tr_tmp.reserve(scan + P.n[1] * chains * wo * sizeof(u64)));
            d_carry = (u64*)((unsigned char*)k->tr_tmp.p + scan);
            CU(block28_trace_scan(k->fast, P, d_init, d_c, chains, k->tr_tmp.p, d_carry, k->stream));
        } else {
            CU(k->tr_tmp.reserve(simple_trace_scan_words(P, chains, (int)wo) * sizeof(u64)));
            d_carry = (u64*)k->tr_tmp.p;
            CU(simple_trace_scan(k->d_simple, (int)wo, P, d_init, d_c, chains, d_carry, k->stream));
        }
    }
    if (fast_chain) CU(block28_trace_chain(k->fast, d_init, d_c, d_carry, count, chains, P.s[0], d_acc, d_q, k->d_flags, k->stream));
    else CU(simple_trace_chain(k->d_simple, d_init, d_c, d_carry, count, chains, P.s[0], d_acc, d_q, k->d_flags, k->stream));
    return PB200_OK;
}
// count * chains * words_out words must be addressable
static bool trace_size_ok(const pb200_key* k, size_t count, size_t chains) {
    return chains <= SIZE_MAX / count / (k->words_out * sizeof(u64)) / 2;
}
int pb200_tally_trace_dev(pb200_key* k, const uint64_t* d_init, const uint64_t* d_c, size_t count, size_t chains, uint64_t* d_acc,
                          uint64_t* d_q) try {
    if (!k || (count && chains && (!d_init || !d_c || !d_acc))) return PB200_ERR_INVALID_ARG;
    if (!count || !chains) return PB200_OK;
    if (!trace_size_ok(k, count, chains)) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    return trace_dev_impl(k, (const u64*)d_init, (const u64*)d_c, count, chains, (u64*)d_acc, (u64*)d_q);
} PB200_CATCH
int pb200_tally_trace(pb200_key* k, const uint64_t* init, const uint64_t* c, size_t count, size_t chains, uint64_t* acc_out,
                      uint64_t* q_out) try {
    if (!k || (count && chains && (!init || !c || !acc_out))) return PB200_ERR_INVALID_ARG;
    if (!count || !chains) return PB200_OK;
    if (!trace_size_ok(k, count, chains)) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    const size_t bi = chains * k->words_out * sizeof(u64), bc = count * bi;
    CU(k->in_a.reserve(bi)); CU(k->in_b.reserve(bc)); CU(k->out_a.reserve(bc));
    if (q_out) CU(k->out_b.reserve(bc));
    CU(cudaMemcpyAsync(k->in_a.p, init, bi, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->in_b.p, c, bc, cudaMemcpyHostToDevice, k->stream));
    int rc = trace_dev_impl(k, (const u64*)k->in_a.p, (const u64*)k->in_b.p, count, chains, (u64*)k->out_a.p, q_out ? (u64*)k->out_b.p : nullptr);
    if (rc) return rc;
    CU(cudaMemcpyAsync(acc_out, k->out_a.p, bc, cudaMemcpyDeviceToHost, k->stream));
    if (q_out) CU(cudaMemcpyAsync(q_out, k->out_b.p, bc, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

// ---- multi-GPU tally ------------------------------------------------------------------------------------
static int peer_status(int flags) { return (flags & (int)PB200_FLAG_PEER_TIMEOUT) ? PB200_ERR_PEER : PB200_OK; }

int pb200_tally_peer_export(pb200_key* k, pb200_ipc_handle* out) try {
    if (!k || !out) return PB200_ERR_INVALID_ARG;
    if (!k->fast) return PB200_ERR_UNSUPPORTED;
    USE_DEVICE(k);
    u64* mail = nullptr;
    CU(block28_mailbox(k->fast, &mail, k->stream));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, mail));
    static_assert(sizeof(h) == sizeof(out->bytes), "cudaIpcMemHandle_t is 64 bytes");
    memcpy(out->bytes, &h, sizeof(h));
    return PB200_OK;
} PB200_CATCH

int pb200_tally_peer_connect(pb200_key* k, int rank, int world, const pb200_ipc_handle* handles) try {
    if (!k || world < 1 || rank < 0 || rank >= world || (world > 1 && !handles)) return PB200_ERR_INVALID_ARG;
    if (!k->fast || world > block28_max_world()) return PB200_ERR_UNSUPPORTED;
    USE_DEVICE(k);
    CU(cudaStreamSynchronize(k->stream));
    u64* mails[16] = {}; void* opened[16] = {};
    CU(block28_mailbox(k->fast, &mails[rank], k->stream));
    for (int i = 0; i < world; i++) {
        if (i == rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles[i].bytes, sizeof(h));
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int j = 0; j < i; j++) if (opened[j]) cudaIpcCloseMemHandle(opened[j]);
            return cuda_fail(e, "cudaIpcOpenMemHandle");
        }
        mails[i] = (u64*)p; opened[i] = p;
    }
    CU(block28_tally_peer_connect(k->fast, rank, world, mails, opened, k->d_flags));
    k->group.clear();
    return PB200_OK;
} PB200_CATCH

int pb200_tally_peer_dev(pb200_key* k, const uint64_t* d_c, size_t count, uint64_t* d_out) try {
    if (!k || !d_out || (count && !d_c)) return PB200_ERR_INVALID_ARG;
    if (!use_fast(k) || block28_peer_world(k->fast) < 1) return PB200_ERR_UNSUPPORTED;
    USE_DEVICE(k);
    return tally_dev_impl(k, d_c, count, d_out, true);
} PB200_CATCH

int pb200_tally_multi(pb200_key* const* keys, int n_gpus, const uint64_t* const* d_c, const size_t* counts, uint64_t* out) try {
    if (!keys || n_gpus < 1 || !d_c || !counts || !out) return PB200_ERR_INVALID_ARG;
    for (int i = 0; i < n_gpus; i++) {
        if (!keys[i] || (counts[i] && !d_c[i])) return PB200_ERR_INVALID_ARG;
        if (keys[i]->n_bits != keys[0]->n_bits || !(keys[i]->n == keys[0]->n)) return PB200_ERR_INVALID_ARG;
        for (int j = 0; j < i; j++) if (keys[j] == keys[i] || keys[j]->device == keys[i]->device) return PB200_ERR_INVALID_ARG;
    }
    DevGuard dev_guard_;
    CU(dev_guard_.set(keys[0]->device));
    const size_t bout = keys[0]->words_out * sizeof(u64);
    bool peer_ok = n_gpus <= block28_max_world();
    for (int i = 0; i < n_gpus; i++) peer_ok = peer_ok && use_fast(keys[i]);
    if (peer_ok && n_gpus > 1) {
        std::vector<pb200_key*> want(keys, keys + n_gpus);
        bool connected = true;
        for (int i = 0; i < n_gpus; i++) connected = connected && keys[i]->group == want;
        if (!connected) {
            for (int i = 0; i < n_gpus && peer_ok; i++)
                for (int j = 0; j < n_gpus && peer_ok; j++) {
                    if (i == j) continue;
                    int can = 0;
                    CU(cudaDeviceCanAccessPeer(&can, keys[i]->device, keys[j]->device));
                    if (!can) { peer_ok = false; break; }
                    CU(cudaSetDevice(keys[i]->device));
                    cudaError_t e = cudaDeviceEnablePeerAccess(keys[j]->device, 0);
                    if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                    else if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
                }
            if (peer_ok) {
                u64* mails[16] = {};
                for (int i = 0; i < n_gpus; i++) {
                    CU(cudaSetDevice(keys[i]->device));
                    CU(cudaStreamSynchronize(keys[i]->stream));
                    CU(block28_mailbox(keys[i]->fast, &mails[i], keys[i]->stream));
                }
                for (int i = 0; i < n_gpus; i++) {
                    CU(cudaSetDevice(keys[i]->device));
                    CU(block28_tally_peer_connect(keys[i]->fast, i, n_gpus, mails, nullptr, keys[i]->d_flags));
                    keys[i]->group = want;
                }
            }
        }
    }
    if (n_gpus == 1 || peer_ok) {
        // one launch per GPU; the partials cross NVLink inside the kernels and every GPU ends with the full product
        for (int i = 0; i < n_gpus; i++) {
            CU(cudaSetDevice(keys[i]->device));
            int rc = clear_flags(keys[i]); if (rc) return rc;
            CU(keys[i]->out_b.reserve(bout));
            rc = tally_dev_impl(keys[i], d_c[i], counts[i], (uint64_t*)keys[i]->out_b.p, n_gpus > 1);
            if (rc) return rc;
        }
        CU(cudaSetDevice(keys[0]->device));
        CU(cudaMemcpyAsync(out, keys[0]->out_b.p, bout, cudaMemcpyDeviceToHost, keys[0]->stream));
        int status = PB200_OK;
        for (int i = 0; i < n_gpus; i++) {
            CU(cudaSetDevice(keys[i]->device));
            int f = 0;
            int rc = read_flags(keys[i], &f); if (rc) return rc;
            if (f & (int)PB200_FLAG_PEER_TIMEOUT) status = PB200_ERR_PEER;
            else if (f && status == PB200_OK) status = PB200_ERR_RANGE;
        }
        return status;
    }
    // no peer access between these devices (or an engine without the fused kernel): per-GPU partials, gathered through the host,
    // combined on keys[0] — the host only moves bytes, every multiplication still runs on a GPU
    std::vector<uint64_t> partials((size_t)n_gpus * keys[0]->words_out);
    for (int i = 0; i < n_gpus; i++) {
        CU(cudaSetDevice(keys[i]->device));
        int rc = clear_flags(keys[i]); if (rc) return rc;
        CU(keys[i]->out_b.reserve(bout));
        rc = tally_dev_impl(keys[i], d_c[i], counts[i], (uint64_t*)keys[i]->out_b.p, false);
        if (rc) return rc;
        CU(cudaMemcpyAsync(partials.data() + (size_t)i * keys[0]->words_out, keys[i]->out_b.p, bout, cudaMemcpyDeviceToHost, keys[i]->stream));
    }
    for (int i = 0; i < n_gpus; i++) {
        CU(cudaSetDevice(keys[i]->device));
        int rc = take_flags(keys[i]); if (rc) return rc;
    }
    return pb200_tally(keys[0], partials.data(), (size_t)n_gpus, out);
} PB200_CATCH

// ---- decryption (SURVEY.md 8f-4) -----------------------------------------------------------------------------------------
int pb200_key_set_private(pb200_key* k, const uint64_t* lambda_le, const uint64_t* mu_le) try {
    if (!k || !lambda_le || !mu_le) return PB200_ERR_INVALID_ARG;
    if (!fits(lambda_le, k->words_in, k->n_bits) || !fits(mu_le, k->words_in, k->n_bits)) return PB200_ERR_RANGE;
    USE_DEVICE(k);
    CU(cudaStreamSynchronize(k->stream));
    const uint32_t win = k->words_in;
    BigInt lambda = BigInt::from_u64_le(lambda_le, win), mu = BigInt::from_u64_le(mu_le, win);
    std::unique_ptr<SimpleConsts> h(new SimpleConsts());
    memset(h.get(), 0, sizeof(SimpleConsts));
    h->k = (int)win; h->kin = (int)win; h->n_bits = (int)k->n_bits; h->exp_bits = 0;
    h->s = (int)(64 * win - k->n.bits());
    BigInt Nt = BigInt::shl(k->n, h->s);
    BigInt bmu = BigInt::div(BigInt::pow2(128 * (size_t)win), Nt);
    Nt.to_u64_le(h->Nt, win); bmu.to_u64_le(h->mu, win + 1);
    k->n.to_u64_le(h->n, win);
    BigInt::mod(mu, k->n).to_u64_le(h->g, win);                 // the L-function kernel multiplies by this slot
    if (!k->d_simple_n) CU(cudaMalloc(&k->d_simple_n, sizeof(SimpleConsts)));
    if (!k->d_lambda) CU(cudaMalloc(&k->d_lambda, win * sizeof(u64)));
    CU(cudaMemcpyAsync(k->d_simple_n, h.get(), sizeof(SimpleConsts), cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->d_lambda, lambda_le, win * sizeof(u64), cudaMemcpyHostToDevice, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    k->lambda_bits = (int)lambda.bits();
    if (k->fast) CU(block28_pow_prepare(k->fast, lambda, k->stream));
    k->has_private = true;
    return PB200_OK;
} PB200_CATCH

int pb200_decrypt_batch_dev(pb200_key* k, const uint64_t* d_c, size_t count, uint64_t* d_m) try {
    if (!k || (count && (!d_c || !d_m))) return PB200_ERR_INVALID_ARG;
    if (!k->has_private) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    CU(k->scratch.reserve(count * k->words_out * sizeof(u64)));
    u64* d_x = (u64*)k->scratch.p;                               // x = c^lambda mod n^2
    if (use_fast(k)) CU(block28_pow(k->fast, (const u64*)d_c, (int)k->words_out, count, d_x, k->stream));
    else CU(simple_pow(k->d_simple, (const u64*)d_c, (int)k->words_out, k->d_lambda, k->lambda_bits, 0, count, d_x, k->d_flags, k->stream));
    CU(simple_lfunc(k->d_simple_n, d_x, count, (u64*)d_m, k->d_flags, k->stream));
    return PB200_OK;
} PB200_CATCH

int pb200_decrypt_batch(pb200_key* k, const uint64_t* c, size_t count, uint64_t* m_out) try {
    if (!k || (count && (!c || !m_out))) return PB200_ERR_INVALID_ARG;
    if (!k->has_private) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    const size_t bin = count * k->words_out * sizeof(u64), bout = count * k->words_in * sizeof(u64);
    CU(k->in_a.reserve(bin)); CU(k->out_a.reserve(bout));
    CU(cudaMemcpyAsync(k->in_a.p, c, bin, cudaMemcpyHostToDevice, k->stream));
    int rc = pb200_decrypt_batch_dev(k, (const uint64_t*)k->in_a.p, count, (uint64_t*)k->out_a.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(m_out, k->out_a.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

// ---- homomorphic scalar multiplication and the weighted tally --------------------------------------------------------------
static bool scalar_args_ok(const pb200_key* k, uint32_t k_bits) { return k && k_bits != 0 && k_bits <= k->n_bits; }
static int check_scalars(const uint64_t* ks, uint32_t k_bits, size_t count) {
    const uint32_t kw = PB200_WORDS(k_bits);
    for (size_t u = 0; u < count; u++) if (!fits(ks + u * kw, kw, k_bits)) return PB200_ERR_RANGE;
    return PB200_OK;
}
static int scalar_dev_impl(pb200_key* k, const u64* d_c, const u64* d_k, uint32_t k_bits, size_t count, u64* d_out) {
    if (!count) return PB200_OK;
    if (use_fast(k)) CU(block28_scalar(k->fast, d_c, d_k, k_bits, count, d_out, k->stream));
    else CU(simple_pow(k->d_simple, d_c, (int)k->words_out, d_k, (int)k_bits, (int)PB200_WORDS(k_bits), count, d_out, k->d_flags, k->stream));
    return PB200_OK;
}
// chunks of at most 2^18 units: scalar products into wt_chunk, their tally into one slot of wt_part, then the tally of the partials
// (128 MB of temporary memory at |n| = 2048 whatever the count)
static const size_t WT_CHUNK = (size_t)1 << 18;
static int tally_weighted_dev_impl(pb200_key* k, const u64* d_c, const u64* d_k, uint32_t k_bits, size_t count, u64* d_out) {
    if (!count) return tally_dev_impl(k, nullptr, 0, (uint64_t*)d_out, false);
    const size_t wo = k->words_out, kw = PB200_WORDS(k_bits), chunks = (count + WT_CHUNK - 1) / WT_CHUNK;
    CU(k->wt_chunk.reserve((count < WT_CHUNK ? count : WT_CHUNK) * wo * sizeof(u64)));
    if (chunks > 1) CU(k->wt_part.reserve(chunks * wo * sizeof(u64)));
    u64* prod = (u64*)k->wt_chunk.p;
    for (size_t i = 0; i < chunks; i++) {
        const size_t u0 = i * WT_CHUNK, n = count - u0 < WT_CHUNK ? count - u0 : WT_CHUNK;
        int rc = scalar_dev_impl(k, d_c + u0 * wo, d_k + u0 * kw, k_bits, n, prod); if (rc) return rc;
        u64* dst = chunks > 1 ? (u64*)k->wt_part.p + i * wo : d_out;                 // one chunk: its tally is the result
        rc = tally_dev_impl(k, (const uint64_t*)prod, n, (uint64_t*)dst, false); if (rc) return rc;
    }
    if (chunks > 1) return tally_dev_impl(k, (const uint64_t*)k->wt_part.p, chunks, (uint64_t*)d_out, false);
    return PB200_OK;
}

int pb200_scalar_mul_batch_dev(pb200_key* k, const uint64_t* d_c, const uint64_t* d_k, uint32_t k_bits, size_t count, uint64_t* d_out) try {
    if (!scalar_args_ok(k, k_bits) || (count && (!d_c || !d_k || !d_out))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    return scalar_dev_impl(k, (const u64*)d_c, (const u64*)d_k, k_bits, count, (u64*)d_out);
} PB200_CATCH
int pb200_scalar_mul_batch(pb200_key* k, const uint64_t* c, const uint64_t* ks, uint32_t k_bits, size_t count, uint64_t* out) try {
    if (!scalar_args_ok(k, k_bits) || (count && (!c || !ks || !out))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    int rc = check_scalars(ks, k_bits, count); if (rc) return rc;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    const size_t bc = count * k->words_out * sizeof(u64), bk = count * PB200_WORDS(k_bits) * sizeof(u64);
    CU(k->in_a.reserve(bc)); CU(k->in_b.reserve(bk)); CU(k->out_a.reserve(bc));
    CU(cudaMemcpyAsync(k->in_a.p, c, bc, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->in_b.p, ks, bk, cudaMemcpyHostToDevice, k->stream));
    rc = scalar_dev_impl(k, (const u64*)k->in_a.p, (const u64*)k->in_b.p, k_bits, count, (u64*)k->out_a.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, k->out_a.p, bc, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH
int pb200_tally_weighted_dev(pb200_key* k, const uint64_t* d_c, const uint64_t* d_k, uint32_t k_bits, size_t count, uint64_t* d_out) try {
    if (!scalar_args_ok(k, k_bits) || !d_out || (count && (!d_c || !d_k))) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    return tally_weighted_dev_impl(k, (const u64*)d_c, (const u64*)d_k, k_bits, count, (u64*)d_out);
} PB200_CATCH
int pb200_tally_weighted(pb200_key* k, const uint64_t* c, const uint64_t* ks, uint32_t k_bits, size_t count, uint64_t* out) try {
    if (!scalar_args_ok(k, k_bits) || !out || (count && (!c || !ks))) return PB200_ERR_INVALID_ARG;
    int rc = check_scalars(ks, k_bits, count); if (rc) return rc;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    const size_t bc = count * k->words_out * sizeof(u64), bk = count * PB200_WORDS(k_bits) * sizeof(u64), bout = k->words_out * sizeof(u64);
    CU(k->in_a.reserve(bc ? bc : 8)); CU(k->in_b.reserve(bk ? bk : 8)); CU(k->out_b.reserve(bout));
    if (bc) CU(cudaMemcpyAsync(k->in_a.p, c, bc, cudaMemcpyHostToDevice, k->stream));
    if (bk) CU(cudaMemcpyAsync(k->in_b.p, ks, bk, cudaMemcpyHostToDevice, k->stream));
    rc = tally_weighted_dev_impl(k, (const u64*)k->in_a.p, (const u64*)k->in_b.p, k_bits, count, (u64*)k->out_b.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, k->out_b.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

// ---- matvec: out_r = P_r * N_r^(n-1), P_r / N_r the products of c_i^|w_ri| over the positive / negative weights ---------------
// `units` copies of n - 1 (the sign step's scalar), prepared once per key
static int mv_nm1(pb200_key* k, size_t units) {
    if (k->mv_nm1_units >= units) return PB200_OK;
    const size_t kwn = PB200_WORDS(k->n_bits);
    std::vector<u64> h(units * kwn);
    const BigInt nm1 = BigInt::sub(k->n, BigInt(1));
    for (size_t u = 0; u < units; u++) nm1.to_u64_le(h.data() + u * kwn, (uint32_t)kwn);
    CU(k->mv_nm1.reserve(h.size() * sizeof(u64)));
    CU(cudaMemcpyAsync(k->mv_nm1.p, h.data(), h.size() * sizeof(u64), cudaMemcpyHostToDevice, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    k->mv_nm1_units = units;
    return PB200_OK;
}
// chain method: per row and sign, the weighted tally of the masked magnitudes (chunks of 2^18 ciphertexts, partials folded into the
// row's value); then per block of rows N^(n-1) in one scalar launch and P * N^(n-1) by a tally of the pair
static int matvec_chain(pb200_key* k, const MatvecPlan& P, const u64* d_c, size_t count, const u64* d_w, uint32_t k_bits, const uint8_t* d_neg,
                        size_t rows, u64* d_out) {
    const size_t wo = k->words_out, kw = PB200_WORDS(k_bits), CH = WT_CHUNK, chunk = count < CH ? count : CH, rbc = P.rb;
    CU(k->mv_arena.reserve((chunk * kw + (4 + 2 * rbc) * wo) * sizeof(u64)));
    u64* masked = (u64*)k->mv_arena.p;
    u64* acc = masked + chunk * kw;                   // [running product, chunk partial]
    u64* pair = acc + 2 * wo;                         // [P_r, N_r^(n-1)]
    u64* nb = pair + 2 * wo;                          // N of the row block
    u64* np = nb + rbc * wo;                          // N^(n-1) of the row block
    int rc;
    for (size_t r0 = 0; r0 < rows; r0 += rbc) {
        const size_t rb = rows - r0 < rbc ? rows - r0 : rbc;
        for (size_t r = 0; r < rb; r++)
            for (int sgn = 0; sgn < P.nsign; sgn++) {
                u64* dst = sgn ? nb + r * wo : d_out + (r0 + r) * wo;
                for (size_t i0 = 0; i0 < count; i0 += CH) {
                    const size_t n = count - i0 < CH ? count - i0 : CH, e = (r0 + r) * count + i0;
                    CU(matvec_mask(d_w + e * kw, d_neg ? d_neg + e : nullptr, n, (int)kw, sgn, masked, k->stream));
                    if (!i0) { rc = tally_weighted_dev_impl(k, d_c, masked, k_bits, n, dst); if (rc) return rc; continue; }
                    rc = tally_weighted_dev_impl(k, d_c + i0 * wo, masked, k_bits, n, acc + wo); if (rc) return rc;
                    CU(cudaMemcpyAsync(acc, dst, wo * sizeof(u64), cudaMemcpyDeviceToDevice, k->stream));
                    rc = tally_dev_impl(k, acc, 2, dst, false); if (rc) return rc;
                }
            }
        if (P.nsign == 1) continue;
        rc = scalar_dev_impl(k, nb, (const u64*)k->mv_nm1.p, k->n_bits, rb, np); if (rc) return rc;
        for (size_t r = 0; r < rb; r++) {
            u64* out = d_out + (r0 + r) * wo;
            CU(cudaMemcpyAsync(pair, out, wo * sizeof(u64), cudaMemcpyDeviceToDevice, k->stream));
            CU(cudaMemcpyAsync(pair + wo, np + r * wo, wo * sizeof(u64), cudaMemcpyDeviceToDevice, k->stream));
            rc = tally_dev_impl(k, pair, 2, out, false); if (rc) return rc;
        }
    }
    return PB200_OK;
}
static int matvec_dev_impl(pb200_key* k, const u64* d_c, size_t count, const u64* d_w, const uint8_t* d_neg, uint32_t k_bits, size_t rows,
                           u64* d_out) {
    if (!rows) return PB200_OK;
    if (!count) { CU(matvec_ones(d_out, rows, (int)k->words_out, k->stream)); return PB200_OK; }
    const MatvecPlan P = matvec_plan(k->n_bits, k->sms, rows, count, k_bits, d_neg != nullptr, use_fast(k));
    if (P.nsign == 2) { int rc = mv_nm1(k, P.rb); if (rc) return rc; }
    if (P.method == 0) return matvec_chain(k, P, d_c, count, d_w, k_bits, d_neg, rows, d_out);
    CU(k->mv_arena.reserve(P.bytes));                 // the plan's bytes include the copies of n - 1 (held in mv_nm1): a small margin
    CU(block28_matvec(k->fast, P, d_c, count, d_w, k_bits, d_neg, rows, d_out, k->mv_arena.p, (const u64*)k->mv_nm1.p, k->stream));
    return PB200_OK;
}
static bool matvec_args_ok(const pb200_key* k, const void* c, size_t count, const void* w, uint32_t k_bits, size_t rows, const void* out) {
    return scalar_args_ok(k, k_bits) && (!rows || out) && (!rows || !count || (c && w));
}
int pb200_matvec_dev(pb200_key* k, const uint64_t* d_c, size_t count, const uint64_t* d_w, const uint8_t* d_neg, uint32_t k_bits, size_t rows,
                     uint64_t* d_out) try {
    if (!matvec_args_ok(k, d_c, count, d_w, k_bits, rows, d_out)) return PB200_ERR_INVALID_ARG;
    if (!rows) return PB200_OK;
    USE_DEVICE(k);
    return matvec_dev_impl(k, (const u64*)d_c, count, (const u64*)d_w, d_neg, k_bits, rows, (u64*)d_out);
} PB200_CATCH
int pb200_matvec(pb200_key* k, const uint64_t* c, size_t count, const uint64_t* w, const uint8_t* neg, uint32_t k_bits, size_t rows,
                 uint64_t* out) try {
    if (!matvec_args_ok(k, c, count, w, k_bits, rows, out)) return PB200_ERR_INVALID_ARG;
    if (!rows) return PB200_OK;
    int rc = check_scalars(w, k_bits, rows * count); if (rc) return rc;
    bool any_neg = false;
    if (neg) for (size_t e = 0; e < rows * count && !any_neg; e++) any_neg = neg[e] != 0;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    const size_t bc = count * k->words_out * sizeof(u64), bw = rows * count * PB200_WORDS(k_bits) * sizeof(u64), bo = rows * k->words_out * sizeof(u64);
    CU(k->in_a.reserve(bc ? bc : 8)); CU(k->in_b.reserve(bw ? bw : 8)); CU(k->out_a.reserve(bo));
    if (bc) CU(cudaMemcpyAsync(k->in_a.p, c, bc, cudaMemcpyHostToDevice, k->stream));
    if (bw) CU(cudaMemcpyAsync(k->in_b.p, w, bw, cudaMemcpyHostToDevice, k->stream));
    if (any_neg) {                                    // rows without a negative weight give P_r * 1^(n-1) = P_r: only stage signs when some exist
        CU(k->mv_neg.reserve(rows * count));
        CU(cudaMemcpyAsync(k->mv_neg.p, neg, rows * count, cudaMemcpyHostToDevice, k->stream));
    }
    rc = matvec_dev_impl(k, (const u64*)k->in_a.p, count, (const u64*)k->in_b.p, any_neg ? (const uint8_t*)k->mv_neg.p : nullptr, k_bits, rows,
                         (u64*)k->out_a.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, k->out_a.p, bo, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH
int pb200_matvec_plan(uint32_t n_bits, int sms, size_t rows, size_t count, uint32_t k_bits, int has_neg, uint64_t* out11) try {
    if (!out11 || n_bits == 0 || k_bits == 0 || k_bits > n_bits || sms < 1) return PB200_ERR_INVALID_ARG;
    const MatvecPlan P = matvec_plan(n_bits, sms, rows, count, k_bits, has_neg != 0, true);
    const uint64_t v[11] = {(uint64_t)P.method, (uint64_t)P.c, (uint64_t)P.J, P.passes, (uint64_t)P.nseg, P.acc, P.red, P.horner, P.sign, P.chain, P.bytes};
    for (int i = 0; i < 11; i++) out11[i] = v[i];
    return PB200_OK;
} PB200_CATCH

// ---- witness --------------------------------------------------------------------------------
static uint64_t popcount_words(const uint64_t* v, uint32_t words) {
    uint64_t c = 0; for (uint32_t i = 0; i < words; i++) c += (uint64_t)__builtin_popcountll(v[i]); return c;
}
uint64_t pb200_witness_records_for(const pb200_key* k, const uint64_t* m) {
    if (!k || !m) return 0;
    uint64_t pn = 0; for (size_t i = 0; i < k->n.w.size(); i++) pn += (uint64_t)__builtin_popcount(k->n.w[i]);
    return popcount_words(m, k->words_in) + k->n.bits() + pn + 1;
}

int pb200_key_g_chain(pb200_key* k, uint64_t* records_out) try {
    if (!k || !records_out) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    int rc = ensure_gchain(k); if (rc) return rc;
    CU(cudaMemcpyAsync(records_out, k->d_gchain, (size_t)k->n_bits * 2 * k->words_out * sizeof(u64), cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

// Delivery pipeline of the witness stream.  The stream is ~4 MB per unit at |n| = 2048, so it is produced in device CHUNKS
// (two record buffers: the kernel of chunk c+1 runs while chunk c drains) and drained in PIECES through a ring of pinned staging
// slots on a second stream (piece i+1..i+3 are in flight on the copy engine while the caller's sink consumes piece i).  The
// sink always reads pinned host memory and is called on the calling thread.
static size_t env_bytes(const char* name, size_t dflt) {
    const char* e = getenv(name);
    if (!e || !*e) return dflt;
    const double v = atof(e);
    return v >= 1.0 ? (size_t)v : dflt;
}

static int pipe_init(pb200_key* k, size_t slot_bytes) {
    pb200_key::Pipe& P = k->pipe;
    if (!P.ready) {
        CU(cudaStreamCreateWithFlags(&P.copy, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaEventCreateWithFlags(&P.kern_done[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&P.buf_free[i], cudaEventDisableTiming));
        }
        for (int i = 0; i < pb200_key::Pipe::NS; i++) CU(cudaEventCreateWithFlags(&P.slot_done[i], cudaEventDisableTiming));
        P.ready = true;
    }
    if (slot_bytes > P.slot_bytes) {
        for (int i = 0; i < pb200_key::Pipe::NS; i++) {
            if (P.pinned[i]) { cudaFreeHost(P.pinned[i]); P.pinned[i] = nullptr; }
        }
        P.slot_bytes = 0;
        for (int i = 0; i < pb200_key::Pipe::NS; i++) CU(cudaHostAlloc(&P.pinned[i], slot_bytes, cudaHostAllocDefault));
        P.slot_bytes = slot_bytes;
    }
    return PB200_OK;
}

int pb200_encrypt_witness_batch(pb200_key* k, const uint64_t* m, const uint64_t* r, size_t count, uint64_t* c_out,
                                size_t max_chunk_units, pb200_witness_sink_fn sink, void* user) try {
    if (!k || !sink || (count && (!m || !r))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    int rc = check_inputs(k, m, count); if (rc) return rc;
    rc = check_inputs(k, r, count); if (rc) return rc;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    const size_t wo = k->words_out, wi = k->words_in, rec_bytes = 2 * wo * sizeof(u64);
    const uint64_t fixed = pb200_witness_records_for(k, m) - popcount_words(m, k->words_in);  // bits(n) + popcount(n) + 1
    // record offsets of every unit (in records) and the g-chain multiplication counts
    std::vector<uint64_t> offsets(count + 1, 0);
    std::vector<uint32_t> gcounts(count);
    uint64_t max_unit = 0;
    for (size_t u = 0; u < count; u++) {
        const uint64_t pc = popcount_words(m + u * wi, k->words_in);
        gcounts[u] = (uint32_t)pc;
        offsets[u + 1] = offsets[u] + pc + fixed;
        if (pc + fixed > max_unit) max_unit = pc + fixed;
    }
    // sizes: a pinned slot holds at least one unit; a device chunk is bounded by the free memory (two record buffers)
    size_t slot_bytes = env_bytes("PB200_WITNESS_SLOT_BYTES", (size_t)256 << 20);
    if (slot_bytes < max_unit * rec_bytes) slot_bytes = (size_t)max_unit * rec_bytes;
    if (slot_bytes > offsets[count] * rec_bytes) slot_bytes = (size_t)offsets[count] * rec_bytes;
    // a chunk's kernel takes the latency of ONE unit's chain whatever its size (about 0.15 s at |n| = 2048), and the first piece
    // can leave only when the first chunk's kernel has ended: chunks of 8 GiB keep that start-up short while one chunk's drain
    // (8 GiB over PCIe, ~0.15 s) still covers the next chunk's kernel
    // (the chain latency grows with the square of the key size: 0.15 s at 2048, 0.3 s at 3072)
    size_t chunk_bytes = (size_t)(8.0 * 1073741824.0 * ((double)k->n_bits / 2048.0) * ((double)k->n_bits / 2048.0));
    if (chunk_bytes < ((size_t)1 << 30)) chunk_bytes = (size_t)1 << 30;
    { size_t fr = 0, tot = 0; if (cudaMemGetInfo(&fr, &tot) == cudaSuccess) { size_t third = fr / 3; if (third < chunk_bytes) chunk_bytes = third; } }
    chunk_bytes = env_bytes("PB200_WITNESS_CHUNK_BYTES", chunk_bytes);
    if (chunk_bytes < max_unit * rec_bytes) chunk_bytes = (size_t)max_unit * rec_bytes;
    // chunks: [cu0[c], cu0[c+1]) greedy by bytes;  pieces inside a chunk: greedy by slot bytes and max_chunk_units
    struct Piece { size_t u0, u1; int chunk; bool first, last; };
    std::vector<size_t> cu0{0};
    std::vector<Piece> pieces;
    {
        size_t u = 0;
        while (u < count) {
            size_t e = u + 1;
            while (e < count && (offsets[e + 1] - offsets[u]) * rec_bytes <= chunk_bytes) e++;
            const int c = (int)cu0.size() - 1;
            size_t p0 = u;
            while (p0 < e) {
                size_t p1 = p0 + 1;
                while (p1 < e && (offsets[p1 + 1] - offsets[p0]) * rec_bytes <= slot_bytes && (!max_chunk_units || p1 - p0 < max_chunk_units)) p1++;
                pieces.push_back(Piece{p0, p1, c, p0 == u, p1 == e});
                p0 = p1;
            }
            cu0.push_back(e);
            u = e;
        }
    }
    const int nchunks = (int)cu0.size() - 1;
    rc = pipe_init(k, slot_bytes); if (rc) return rc;
    pb200_key::Pipe& P = k->pipe;
    constexpr int NS = pb200_key::Pipe::NS;
    // inputs and the (absolute) record offsets of ALL units go up once, before the pipeline starts: a pageable host-to-device
    // copy synchronises its stream first, which inside the loop would stall the thread that feeds the copy engine
    CU(k->in_a.reserve(count * wi * sizeof(u64))); CU(k->in_b.reserve(count * wi * sizeof(u64))); CU(k->offs.reserve((count + 1) * sizeof(u64)));
    CU(cudaMemcpyAsync(k->in_a.p, m, count * wi * sizeof(u64), cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->in_b.p, r, count * wi * sizeof(u64), cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->offs.p, offsets.data(), (count + 1) * sizeof(u64), cudaMemcpyHostToDevice, k->stream));
    {   // the two record buffers at their final size (cudaMalloc inside the loop would synchronise the device)
        size_t need_rec[2] = {0, 0}, need_c[2] = {0, 0};
        for (int c = 0; c < nchunks; c++) {
            const size_t recs = (size_t)(offsets[cu0[c + 1]] - offsets[cu0[c]]), nu = cu0[c + 1] - cu0[c];
            if (recs * rec_bytes > need_rec[c & 1]) need_rec[c & 1] = recs * rec_bytes;
            if (nu * wo * sizeof(u64) > need_c[c & 1]) need_c[c & 1] = nu * wo * sizeof(u64);
        }
        for (int b = 0; b < 2; b++) if (need_rec[b]) { CU(P.rec[b].reserve(need_rec[b])); CU(P.cbuf[b].reserve(need_c[b])); }
    }
    // fallible steps of the pipeline; every exit path below drains both streams first (the sink's memory must not be in flight)
    auto launch_chunk = [&](int c) -> int {
        const int b = c & 1;
        const size_t u0 = cu0[c], nu = cu0[c + 1] - u0;
        if (c >= 2) CU(cudaStreamWaitEvent(k->stream, P.buf_free[b], 0));        // chunk c-2 has left this buffer
        // the kernels address records as base + offsets[unit] * record words with ABSOLUTE offsets: shift the base
        u64* rec_base = (u64*)P.rec[b].p - (size_t)offsets[u0] * 2 * wo;
        int rcw = run_witness(k, (const u64*)k->in_a.p + u0 * wi, (const u64*)k->in_b.p + u0 * wi, nu, (u64*)P.cbuf[b].p, rec_base,
                              (const u64*)k->offs.p + u0, nullptr);
        if (rcw) return rcw;
        CU(cudaEventRecord(P.kern_done[b], k->stream));
        return PB200_OK;
    };
    int next_chunk = 0;
    auto issue = [&](size_t p) -> int {
        const Piece& pc = pieces[p];
        const int b = pc.chunk & 1, slot = (int)(p % NS);
        const size_t cu = cu0[pc.chunk];
        if (pc.first) {
            CU(cudaStreamWaitEvent(P.copy, P.kern_done[b], 0));
            if (c_out) CU(cudaMemcpyAsync(c_out + cu * wo, P.cbuf[b].p, (cu0[pc.chunk + 1] - cu) * wo * sizeof(u64), cudaMemcpyDeviceToHost, P.copy));
        }
        const size_t r0 = (size_t)(offsets[pc.u0] - offsets[cu]), nrec = (size_t)(offsets[pc.u1] - offsets[pc.u0]);
        CU(cudaMemcpyAsync(P.pinned[slot], (const char*)P.rec[b].p + r0 * rec_bytes, nrec * rec_bytes, cudaMemcpyDeviceToHost, P.copy));
        CU(cudaEventRecord(P.slot_done[slot], P.copy));
        if (pc.last) {
            CU(cudaEventRecord(P.buf_free[b], P.copy));
            if (next_chunk < nchunks) { int rcl = launch_chunk(next_chunk++); if (rcl) return rcl; }
        }
        return PB200_OK;
    };
    auto drain = [&]() { cudaStreamSynchronize(k->stream); cudaStreamSynchronize(P.copy); };
    rc = launch_chunk(next_chunk++);
    if (!rc && next_chunk < nchunks) rc = launch_chunk(next_chunk++);
    if (rc) { drain(); return rc; }
    size_t issued = 0;
    std::vector<uint64_t> poffs;
    for (size_t i = 0; i < pieces.size(); i++) {
        while (issued < pieces.size() && issued < i + NS) {
            rc = issue(issued++);
            if (rc) { drain(); return rc; }
        }
        cudaError_t e = cudaEventSynchronize(P.slot_done[i % NS]);
        if (e != cudaSuccess) { drain(); return cuda_fail(e, "witness pipeline"); }
        const Piece& pc = pieces[i];
        poffs.resize(pc.u1 - pc.u0 + 1);
        for (size_t u = pc.u0; u <= pc.u1; u++) poffs[u - pc.u0] = offsets[u] - offsets[pc.u0];
        pb200_witness_chunk ch;
        ch.first_unit = pc.u0; ch.n_units = pc.u1 - pc.u0; ch.words_out = k->words_out;
        ch.offsets = poffs.data(); ch.records = (const uint64_t*)P.pinned[i % NS]; ch.g_mul_counts = gcounts.data() + pc.u0;
        if (sink(user, &ch) != 0) { drain(); return PB200_ERR_SINK; }
    }
    CU(cudaStreamSynchronize(P.copy));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

int pb200_encrypt_witness_digest(pb200_key* k, const uint64_t* m, const uint64_t* r, size_t count, uint64_t* c_out,
                                 uint64_t* digest_out) try {
    if (!k || !digest_out || (count && (!m || !r))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    int rc = check_inputs(k, m, count); if (rc) return rc;
    rc = check_inputs(k, r, count); if (rc) return rc;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    size_t bin = count * k->words_in * sizeof(u64), bout = count * k->words_out * sizeof(u64);
    CU(k->in_a.reserve(bin)); CU(k->in_b.reserve(bin)); CU(k->out_a.reserve(bout)); CU(k->out_b.reserve(count * sizeof(u64)));
    CU(cudaMemcpyAsync(k->in_a.p, m, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->in_b.p, r, bin, cudaMemcpyHostToDevice, k->stream));
    rc = run_witness(k, (const u64*)k->in_a.p, (const u64*)k->in_b.p, count, (u64*)k->out_a.p, nullptr, nullptr, (u64*)k->out_b.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(digest_out, k->out_b.p, count * sizeof(u64), cudaMemcpyDeviceToHost, k->stream));
    if (c_out) CU(cudaMemcpyAsync(c_out, k->out_a.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);
} PB200_CATCH

int pb200_encrypt_witness_digest_dev(pb200_key* k, const uint64_t* d_m, const uint64_t* d_r, size_t count, uint64_t* d_c,
                                     uint64_t* d_digest) try {
    if (!k || !d_digest || (count && (!d_m || !d_r))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    return run_witness(k, (const u64*)d_m, (const u64*)d_r, count, (u64*)d_c, nullptr, nullptr, (u64*)d_digest);
} PB200_CATCH
const char* pb200_key_witness_engine(pb200_key* k) {
    if (!k) return "";
    return (use_fast(k) && block28_witness_supported(k->fast)) ? "block28w" : "simple64";
}

// ---- K4: advice cells ------------------------------------------------------------------------------------
static BigInt low_bits(const BigInt& v, size_t bits) { return BigInt::sub(v, BigInt::shl(BigInt::shr(v, bits), bits)); }
static void put128(std::vector<u64>& dst, const BigInt& v) { u64 w[2]; v.to_u64_le(w, 2); dst.push_back(w[0]); dst.push_back(w[1]); }

static int cell_ctx(pb200_key* k, uint32_t lookup_bits, pb200_key::CellCtx** out) {
    if (lookup_bits > 32) return PB200_ERR_INVALID_ARG;
    auto it = k->cells.find(lookup_bits);
    if (it != k->cells.end()) { *out = &it->second; return PB200_OK; }
    pb200_key::CellCtx C;
    CellLayout& Y = C.Y;
    const int lb = (int)k->limb_bits, L = (int)(2 * k->n_bits / k->limb_bits), NC = 2 * L - 1, kn = (int)(k->n_bits / k->limb_bits);
    Y.L = L; Y.limb_bits = lb; Y.lookup_bits = (int)lookup_bits;
    BigInt B1 = BigInt::sub(BigInt::pow2(lb), BigInt(1));
    BigInt word_max = BigInt::add(BigInt::mul(BigInt((uint64_t)L), BigInt::mul(B1, B1)), B1);       // A.6
    Y.carry_bits = (int)BigInt::shl(word_max, 1).bits() - lb;
    Y.kl = lookup_bits ? (lb + (int)lookup_bits - 1) / (int)lookup_bits : 0;
    Y.xl = lookup_bits && (lb % (int)lookup_bits) ? 1 : 0;
    Y.cpl = 1 + Y.kl + Y.xl;
    Y.kc = lookup_bits ? (Y.carry_bits + (int)lookup_bits - 1) / (int)lookup_bits : 0;
    Y.xc = lookup_bits && (Y.carry_bits % (int)lookup_bits) ? 1 : 0;
    Y.off_rem = L * Y.cpl; Y.off_ab = 2 * L * Y.cpl; Y.off_qn = Y.off_ab + NC; Y.off_qnp = Y.off_qn + NC; Y.off_eq = Y.off_qnp + NC;
    Y.eq_stride = 4 + Y.kc + Y.xc;
    Y.n_cells = Y.off_eq + (NC - 1) * Y.eq_stride + 4 + 1;
    std::vector<u64> h;
    for (int i = 0; i < L; i++) put128(h, low_bits(BigInt::shr(k->n2, (size_t)i * lb), lb));
    { u64 w[4]; word_max.to_u64_le(w, 4); h.insert(h.end(), w, w + 4); }
    std::vector<u64> qa, ma;
    BigInt acc;
    for (int i = 0; i < NC; i++) {
        acc = BigInt::add(acc, word_max);
        BigInt qacc = BigInt::shr(acc, lb), macc = low_bits(acc, lb);
        put128(qa, qacc); put128(ma, macc);
        acc = qacc;
    }
    h.insert(h.end(), qa.begin(), qa.end()); h.insert(h.end(), ma.begin(), ma.end());
    {   // Montgomery forms (x * 2^256 mod p, BN254 Fr) of the per-key q_acc / mod_acc cells; 32-byte aligned in the buffer
        static const uint64_t FRP[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
        BigInt P = BigInt::from_u64_le(FRP, 4);
        for (int which = 0; which < 2; which++)
            for (int i = 0; i < NC; i++) {
                const std::vector<u64>& src = which ? ma : qa;
                u64 w2[2] = {src[2 * i], src[2 * i + 1]};
                BigInt m = BigInt::mod(BigInt::shl(BigInt::from_u64_le(w2, 2), 256), P);
                u64 w4[4]; m.to_u64_le(w4, 4);
                h.insert(h.end(), w4, w4 + 4);
            }
    }
    // RefreshAux::new(limb_bits, kn, kn) (A.3): how far each column of n*n can spill
    std::vector<BigInt> vals(2 * kn - 1);
    for (int i = 0; i < kn; i++) for (int j = 0; j < kn; j++) vals[i + j] = BigInt::add(vals[i + j], BigInt::mul(B1, B1));
    std::vector<int> inc;
    for (size_t i = 0; i < vals.size(); i++) {
        BigInt v = vals[i], carry = BigInt::shr(v, lb);
        int cnt = 0; size_t kk = 1;
        while (!carry.is_zero()) {
            if (i + kk >= vals.size()) vals.push_back(BigInt());
            vals[i + kk] = BigInt::add(vals[i + kk], low_bits(carry, lb));
            carry = BigInt::shr(carry, lb); cnt++; kk++;
        }
        vals[i] = low_bits(v, lb);
        inc.push_back(cnt);
    }
    C.n_out = (int)inc.size();
    C.n2_cells = (2 * kn - 1) + (lookup_bits ? C.n_out * (Y.kl + Y.xl) : 0);
    for (int i = 0; i < 2 * kn - 1; i++) C.n2_cells += 2 * (inc[i] + 1);
    CU(cudaMalloc(&C.d_consts, h.size() * sizeof(u64)));
    CU(cudaMemcpy(C.d_consts, h.data(), h.size() * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&C.d_inc, inc.size() * sizeof(int)));
    CU(cudaMemcpy(C.d_inc, inc.data(), inc.size() * sizeof(int), cudaMemcpyHostToDevice));
    if (lookup_bits >= 1 && lookup_bits <= 16) {       // chunk-value table for the Montgomery output (2 MB at 16 bits)
        CU(cudaMalloc(&C.d_mtab, ((size_t)32) << lookup_bits));
        CU(cells_mont_table((int)lookup_bits, C.d_mtab, k->stream));
        CU(cudaStreamSynchronize(k->stream));
    }
    k->cells[lookup_bits] = C;
    *out = &k->cells[lookup_bits];
    return PB200_OK;
}

int pb200_cells_layout(pb200_key* k, uint32_t lookup_bits, pb200_cell_layout* out) try {
    if (!k || !out) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    pb200_key::CellCtx* C = nullptr;
    int rc = cell_ctx(k, lookup_bits, &C); if (rc) return rc;
    out->limbs = (uint32_t)C->Y.L; out->cells_per_limb = (uint32_t)C->Y.cpl; out->carry_bits = (uint32_t)C->Y.carry_bits;
    out->cells_per_mulmod = (uint32_t)C->Y.n_cells; out->cells_n2 = (uint32_t)C->n2_cells;
    out->off_rem = (uint32_t)C->Y.off_rem; out->off_ab = (uint32_t)C->Y.off_ab; out->off_qn = (uint32_t)C->Y.off_qn;
    out->off_qn_rem = (uint32_t)C->Y.off_qnp; out->off_eq = (uint32_t)C->Y.off_eq; out->eq_stride = (uint32_t)C->Y.eq_stride;
    return PB200_OK;
} PB200_CATCH

int pb200_mulmod_cells_batch_dev(pb200_key* k, const uint64_t* d_a, const uint64_t* d_b, const uint64_t* d_q, const uint64_t* d_rem,
                                 size_t count, uint32_t lookup_bits, int montgomery, uint64_t* d_cells) try {
    if (!k || (count && (!d_a || !d_b || !d_q || !d_rem || !d_cells))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    pb200_key::CellCtx* C = nullptr;
    int rc = cell_ctx(k, lookup_bits, &C); if (rc) return rc;
    CU(cells_mulmod(C->Y, C->d_consts, (const u64*)d_a, (const u64*)d_b, (const u64*)d_q, (const u64*)d_rem, count, (int)k->words_out,
                    montgomery ? 1 : 0, (u64*)d_cells, k->d_flags, k->sms, C->d_mtab, k->stream));
    return PB200_OK;
} PB200_CATCH

int pb200_mulmod_cells_batch(pb200_key* k, const uint64_t* a, const uint64_t* b, const uint64_t* q, const uint64_t* rem, size_t count,
                             uint32_t lookup_bits, int montgomery, uint64_t* cells_out) try {
    if (!k || (count && (!a || !b || !q || !rem || !cells_out))) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    pb200_key::CellCtx* C = nullptr;
    int rc = cell_ctx(k, lookup_bits, &C); if (rc) return rc;
    const size_t bin = count * k->words_out * sizeof(u64), bout = count * (size_t)C->Y.n_cells * 32;
    CU(k->cin_a.reserve(bin)); CU(k->cin_b.reserve(bin)); CU(k->cin_q.reserve(bin)); CU(k->cin_r.reserve(bin)); CU(k->scratch.reserve(bout));
    CU(cudaMemcpyAsync(k->cin_a.p, a, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->cin_b.p, b, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->cin_q.p, q, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cudaMemcpyAsync(k->cin_r.p, rem, bin, cudaMemcpyHostToDevice, k->stream));
    rc = pb200_mulmod_cells_batch_dev(k, (const uint64_t*)k->cin_a.p, (const uint64_t*)k->cin_b.p, (const uint64_t*)k->cin_q.p,
                                      (const uint64_t*)k->cin_r.p, count, lookup_bits, montgomery, (uint64_t*)k->scratch.p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(cells_out, k->scratch.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return take_flags(k);      // PB200_ERR_CONSTRAINT: (q, rem) do not satisfy a*b = q*n^2 + rem
} PB200_CATCH

int pb200_assign_cells_batch(pb200_key* k, const uint64_t* values, size_t count, uint32_t value_bits, uint32_t lookup_bits,
                             int montgomery, uint64_t* cells_out) try {
    if (!k || !values || !cells_out || value_bits == 0 || value_bits % k->limb_bits || lookup_bits > 32) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    const int lb = (int)k->limb_bits, nl = (int)(value_bits / k->limb_bits);
    const int kl = lookup_bits ? (lb + (int)lookup_bits - 1) / (int)lookup_bits : 0, xl = lookup_bits && (lb % (int)lookup_bits) ? 1 : 0;
    const int cpl = 1 + kl + xl, words = (int)PB200_WORDS(value_bits);
    const size_t bin = count * words * sizeof(u64), bout = count * (size_t)nl * cpl * 32;
    CU(k->cin_a.reserve(bin)); CU(k->scratch.reserve(bout));
    CU(cudaMemcpyAsync(k->cin_a.p, values, bin, cudaMemcpyHostToDevice, k->stream));
    CU(cells_assign((const u64*)k->cin_a.p, count, words, nl, lb, (int)lookup_bits, kl, cpl, montgomery ? 1 : 0, (u64*)k->scratch.p, k->stream));
    CU(cudaMemcpyAsync(cells_out, k->scratch.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return PB200_OK;
} PB200_CATCH

int pb200_key_n2_cells(pb200_key* k, uint32_t lookup_bits, int montgomery, uint64_t* cells_out) try {
    if (!k || !cells_out) return PB200_ERR_INVALID_ARG;
    USE_DEVICE(k);
    { int rc0_ = clear_flags(k); if (rc0_) return rc0_; }
    pb200_key::CellCtx* C = nullptr;
    int rc = cell_ctx(k, lookup_bits, &C); if (rc) return rc;
    std::vector<u64> nw(k->words_in);
    k->n.to_u64_le(nw.data(), k->words_in);
    const size_t bout = (size_t)C->n2_cells * 32;
    CU(k->cin_a.reserve(nw.size() * sizeof(u64))); CU(k->scratch.reserve(bout)); CU(k->offs.reserve(sizeof(int)));
    CU(cudaMemcpyAsync(k->cin_a.p, nw.data(), nw.size() * sizeof(u64), cudaMemcpyHostToDevice, k->stream));
    CU(cells_n2((const u64*)k->cin_a.p, (int)k->words_in, (int)(k->n_bits / k->limb_bits), (int)k->limb_bits, (int)lookup_bits, C->Y.kl,
                C->Y.xl, C->d_inc, C->n_out, montgomery ? 1 : 0, (u64*)k->scratch.p, (int*)k->offs.p, k->d_flags, k->stream));
    int written = 0;
    CU(cudaMemcpyAsync(&written, k->offs.p, sizeof(int), cudaMemcpyDeviceToHost, k->stream));
    CU(cudaMemcpyAsync(cells_out, k->scratch.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    if (written != C->n2_cells) { t_cuda_error = "n2 cell count mismatch"; return PB200_ERR_CUDA; }
    return take_flags(k);
} PB200_CATCH

// ---- limb formatting ------------------------------------------------------------------------
int pb200_repack_limbs(pb200_key* k, const uint64_t* values, size_t count, uint32_t value_bits, uint32_t limb_bits,
                       uint64_t* limbs_out) try {
    if (!k || !values || !limbs_out || limb_bits == 0 || limb_bits > 128 || value_bits % limb_bits) return PB200_ERR_INVALID_ARG;
    if (!count) return PB200_OK;
    USE_DEVICE(k);
    uint32_t wpv = PB200_WORDS(value_bits), nl = value_bits / limb_bits;
    size_t bin = count * wpv * sizeof(u64), bout = count * nl * 2 * sizeof(u64);
    CU(k->in_a.reserve(bin)); CU(k->out_a.reserve(bout));
    CU(cudaMemcpyAsync(k->in_a.p, values, bin, cudaMemcpyHostToDevice, k->stream));
    CU(repack_limbs((const u64*)k->in_a.p, count, (int)wpv, (int)value_bits, (int)limb_bits, (u64*)k->out_a.p, k->stream));
    CU(cudaMemcpyAsync(limbs_out, k->out_a.p, bout, cudaMemcpyDeviceToHost, k->stream));
    CU(cudaStreamSynchronize(k->stream));
    return PB200_OK;
} PB200_CATCH

}  // extern "C"
