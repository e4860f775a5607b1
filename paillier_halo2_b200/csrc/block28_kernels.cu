// block28_kernels.cu — kernels and host driver of the block28 engine (device arithmetic in block28.cuh).
//
// Replaces, for `count` independent units: g.modpow(m, n2), r.modpow(n, n2) and the final product of
// paillier_enc_native (/root/reference/src/paillier.rs:87-92), and the fold of paillier_add_native
// (:94-97).  Chain per unit (all modulo Nt, a multiple of n^2):
//   r^n : left-to-right sliding window (w = 6) over the per-key exponent n; the 32 odd powers of r live in
//         a per-CTA global scratch table (L2-resident), the window schedule is computed once per key;
//   g^m : fixed-base comb, w-bit windows (w = 12 for |n| >= 1024, else 8): product of TG[i][digit_i(m)],
//         TG[i][d] = g^(d * 2^(w i)) mod Nt, built once per key by this engine (k_gtable_*);
//   c   : gm * rn, then one exact canonicalisation (finalize) and the shift back from Nt to n^2.
#include "engine.hpp"
#include "block28.cuh"
#include "block28u.cuh"
#include <cstdio>
#include <vector>
#include <cstring>
#include <cstdlib>
#include <algorithm>

namespace pb200 {
using namespace b28;

constexpr int WIN = 6;                 // sliding window of the r-chain (6: 293 + 31 multiplications at |n| = 2048; 5: 341 + 15)
constexpr int TABN = 1 << (WIN - 1);   // odd powers r^1, r^3, ..., r^(2*TABN-1)
constexpr int SCRATCH_ENTRIES = TABN + 2;   // + r^2 (table build) + rn (kept while g^m is computed)

// left-to-right sliding-window schedule of a fixed exponent (window_schedule): the chain starts from odd-power table entry first_idx
// (-1: the exponent is 0), then runs n_ops steps (number of squarings, table index to multiply by or -1)
struct PowSched { const int2* ops; int n_ops; int first_idx; };

struct B28Dev {            // per-key device-side descriptor (same for every configuration)
    const int4* consts;    // mu, Nt, two_sh : 3 * ENTRY4 int4
    const int4* uconsts2;  // the same for the two-lane-group variant
    const int4* uconsts;   // block28u: constants + CM tables (UL<C>::KEY_BYTES), null when the configuration has no tcgen05 variant
    PowSched rn;           // r-chain schedule (the exponent n)
    const int4* tg;        // comb table: [window][2^comb_bits][ENTRY4]
    int n_windows;
    int comb_bits;         // window width of the fixed-base comb for g^m
    const int4* n_entry;   // g == n + 1 (the standard Paillier generator): strict digits of n, g^m = 1 + m n (mod n^2); else null
    int words_in, words_out;
    int sh;                // Nt = n2 << sh
    unsigned nt_top;       // floor(Nt / 2^(28(L-2)))
    unsigned sms;
};

// ---- device helpers --------------------------------------------------------------------------
__device__ __forceinline__ unsigned smid() { unsigned v; asm volatile("mov.u32 %0, %%smid;" : "=r"(v)); return v; }
template <class C>
__device__ __forceinline__ int& digit_ref(int4* buf, int p, int lane) {
    int blk = p / C::BL, k = p % C::BL;
    return ((int*)(buf + blk * C::BLK4 + (k >> 2) * 32 + lane))[k & 3];
}

// The digit loader: the strict digit of (value << shl) at bit position bit = 28 p - shl of the value, from the 28-bit field there
// plus the carry out of the digit below (updated).  The value is the unsigned integer word(0 .. nwords), u64 little-endian, read
// through the accessor `word`, so every caller keeps its own load flavour and layout.
template <class F>
__device__ __forceinline__ int strict_digit(const F& word, int nwords, int bit, int& carry) {
    u64 v = 0;
    if (bit >= 0) {
        const int wi = bit >> 6, sh = bit & 63;
        const u64 lo = wi < nwords ? word(wi) : 0, hi = wi + 1 < nwords ? word(wi + 1) : 0;
        v = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
    } else if (bit > -W) {
        v = word(0) << (-bit);
    }
    const int t = (int)(v & ((1u << W) - 1)) + carry;
    const int d = sgxt28(t);
    carry = (t - d) >> W;
    return d;
}
// per-lane buffer <- strict digits of (value << shl), value = word(0 .. nwords) (see strict_digit); the carry out of a block is added
// to the first digit of the next one
template <class C, class F>
__device__ __forceinline__ void load_words(int4* buf, const F& word, int nwords, int shl, int role, int lane) {
    int a[C::CH * 4];
    int carry = 0;
#pragma unroll
    for (int k = 0; k < C::BL; k++) a[k] = strict_digit(word, nwords, W * (role * C::BL + k) - shl, carry);
#pragma unroll
    for (int k = C::BL; k < C::CH * 4; k++) a[k] = 0;
    store_block<C>(blk_ptr<C>(buf, role, lane), a);
    __syncthreads();
    if (role + 1 < C::G) *(int*)blk_ptr<C>(buf, role + 1, lane) += carry;
    __syncthreads();
}
// per-lane buffer <- strict digits of (src[0..nwords) << shl) (u64 little-endian)
template <class C>
__device__ __forceinline__ void load_value(int4* buf, const u64* src, int nwords, int role, int lane, int shl = 0) {
    load_words<C>(buf, [src](int i) { return src[i]; }, nwords, shl, role, lane);
}

// The 32 inputs of a CTA step are contiguous in global memory: copy them with coalesced loads into a word-major staging area
// ([word][lane], row stride 33 to spread the transposing stores over the banks) and cut the digits out of shared memory
// (a lane reading its own 512-byte ciphertext word by word touches 32 different lines per instruction).
template <class C>
__device__ __forceinline__ void stage_words(u64* stage, const u64* src, int units_avail, int nwords) {
    const int total = 32 * nwords;
    for (int idx = threadIdx.x; idx < total; idx += C::THREADS) {
        const int l = idx / nwords, wi = idx - l * nwords;
        stage[wi * 33 + l] = l < units_avail ? src[(size_t)l * nwords + wi] : 0;
    }
    __syncthreads();
}
template <class C>
__device__ __forceinline__ void load_value_staged(int4* buf, const u64* stage, int nwords, int role, int lane) {
    load_words<C>(buf, [stage, lane](int i) { return stage[i * 33 + lane]; }, nwords, 0, role, lane);
}

// per-lane buffer <- 1 where cond (the others keep their value); barrier
template <class C>
__device__ __forceinline__ void set_one_where(int4* buf, bool cond, int role, int lane) {
    if (cond) {
        int a[C::CH * 4];
#pragma unroll
        for (int k = 0; k < C::CH * 4; k++) a[k] = 0;
        if (role == 0) a[0] = 1;
        store_block<C>(blk_ptr<C>(buf, role, lane), a);
    }
    __syncthreads();
}

// smem per-lane value <-> global [entry][blk][chunk][lane] (coalesced)
template <class C>
__device__ __forceinline__ void copy_to_global(int4* g, const int4* buf, int role, int lane) {
#pragma unroll
    for (int c = 0; c < C::CH; c++) g[(role * C::CH + c) * 32 + lane] = buf[(role * C::CH + c) * 32 + lane];
}
template <class C>
__device__ __forceinline__ void copy_from_global(int4* buf, const int4* g, int role, int lane) {
#pragma unroll
    for (int c = 0; c < C::CH; c++) buf[(role * C::CH + c) * 32 + lane] = g[(role * C::CH + c) * 32 + lane];
    __syncthreads();
}
// smem per-lane value <- one table entry per lane ([blk][chunk] int4, gathered)
template <class C>
__device__ __forceinline__ void gather_entry(int4* buf, const int4* entry, int role, int lane) {
#pragma unroll
    for (int c = 0; c < C::CH; c++) buf[(role * C::CH + c) * 32 + lane] = __ldg(entry + role * C::CH + c);
    __syncthreads();
}
template <class C>
__device__ __forceinline__ void scatter_entry(int4* entry, const int4* buf, int role, int lane) {
#pragma unroll
    for (int c = 0; c < C::CH; c++) entry[role * C::CH + c] = buf[(role * C::CH + c) * 32 + lane];
}

template <class C>
__device__ __forceinline__ void load_consts(int4* smem_base, const B28Dev& K) {
    int4* k = smem_base + 5 * C::VAL4;
    for (int i = threadIdx.x; i < 3 * C::ENTRY4 + 2 * C::RTAB4; i += C::THREADS) k[i] = K.consts[i];
    __syncthreads();
}


// ---- engine selection: 0 = block28 (all phases on IMAD), 1 = block28t (mma.sync for phases B, C), 2 = block28u (tcgen05) ----------
// SUPPORTED: the configuration compiles this engine (the host instantiates and launches only those)
template <class C, int ENG> struct View {
    typedef Smem<C> type;
    static constexpr bool SUPPORTED = true;
    static constexpr size_t BYTES = C::SMEM_BYTES;
    static constexpr int PER_SM = C::CTAS_PER_SM;
    static constexpr int LG = 1, THREADS = C::THREADS;
};
template <class C> struct View<C, 2> {            // block28u, one lane group per CTA
    typedef SmemU<C, 1> type;
    static constexpr bool SUPPORTED = UL<C, 1>::SUPPORTED;
    static constexpr size_t BYTES = UL<C, 1>::SMEM_BYTES;
    static constexpr int PER_SM = UL<C, 1>::CTAS_PER_SM;
    static constexpr int LG = 1, THREADS = C::THREADS;
};
template <class C> struct View<C, 4> : View<C, 2> {};      // block28u as the tally runs it: MMAs issued by thread 0 (see phases_bc_umma)
template <class C> struct View<C, 3> {            // block28u, two lane groups (64 ciphertexts) per CTA
    typedef SmemU<C, 2> type;
    static constexpr bool SUPPORTED = UL<C, 1>::SUPPORTED && UL<C, 2>::SUPPORTED;
    static constexpr size_t BYTES = UL<C, 2>::SMEM_BYTES;
    static constexpr int PER_SM = UL<C, 2>::CTAS_PER_SM;
    static constexpr int LG = 2, THREADS = 2 * C::THREADS;
};
template <class C, bool SQR, int ENG, class SV>
__device__ __forceinline__ void mm(SV& S, const int4* Y, int role, int lane) {
    if constexpr (ENG >= 2) mulmod_u<C, View<C, ENG>::LG, SQR, ENG != 4>(S, Y);
    else mulmod<C, SQR, ENG == 1>(S, Y, role, lane);
}
// Per-key constants into shared memory (+ TMEM and mbarriers for block28u), by the kernel's shared-memory view: Smem<C> (IMAD and
// mma.sync phases) takes the constant block, SmemU<C, LG, WIT> (tcgen05 phases) its layout's image, the two-lane-group one for LG 2
// (K.uconsts of the witness engine's descriptor is the witness modulus's image)
template <class C>
__device__ __forceinline__ void cta_begin(Smem<C>&, int4* smem_base, const B28Dev& K) { load_consts<C>(smem_base, K); }
template <class C, int LG, bool WIT>
__device__ __forceinline__ void cta_begin(SmemU<C, LG, WIT>& S, int4* smem_base, const B28Dev& K) {
    typedef UL<C, LG, WIT> U;
    int4* dst = (int4*)((unsigned char*)smem_base + U::OFF_CONST);
    const int4* src = LG == 2 ? K.uconsts2 : K.uconsts;
    for (int i = threadIdx.x; i < U::KEY_BYTES / 16; i += U::THREADS) dst[i] = src[i];
    umma_setup(S);
}
template <class C>
__device__ __forceinline__ void cta_end(Smem<C>&) {}
template <class C, int LG, bool WIT>
__device__ __forceinline__ void cta_end(SmemU<C, LG, WIT>& S) { umma_teardown(S); }

// The unit of a lane: the 32 lanes of lane group grp take consecutive units from first + 32 grp (first: the CTA's first unit, LG
// groups of 32 per CTA).  A lane past `count` works on unit count - 1 and is not active: it multiplies like the others, stores nothing.
struct LaneUnit { size_t unit; bool active; };
template <int LG = 1>
__device__ __forceinline__ LaneUnit lane_unit(size_t count, int lane, int grp = 0, size_t first = (size_t)blockIdx.x * (32 * LG)) {
    const size_t u = first + grp * 32 + lane;
    return {u < count ? u : count - 1, u < count};
}

// V <- V * (constant in shared memory, ENTRY4 int4, broadcast)
template <class C, int ENG, class SV>
__device__ __forceinline__ void mulmod_const(SV& S, const int4* cst, int role, int lane) {
    // expand the constant into the per-lane B buffer (keeps phase_product on one code path)
#pragma unroll
    for (int c = 0; c < C::CH; c++) S.B[(role * C::CH + c) * 32 + lane] = cst[role * C::CH + c];
    __syncthreads();
    mm<C, false, ENG>(S, S.B, role, lane);
}

// Exact canonicalisation of the lazy value in V (one thread per lane, role 0): out = ((V * 2^sh) mod Nt) >> sh,
// written as words_out u64 words.  V must already have been multiplied by two_sh.
template <class C>
__device__ void canonical_out(int4* V, const int4* NtC, const B28Dev& K, u64* out, int lane) {
    constexpr int L = C::L;
    const int* nt = (const int*)NtC;
    auto NT = [&](int p) { return nt[(p / C::BL) * C::CH * 4 + (p % C::BL)]; };
    auto D = [&](int p) -> int& { return digit_ref<C>(V, p, lane); };
    // full ripple to strict centred digits
    int carry = 0;
    for (int p = 0; p < L; p++) { int t = D(p) + carry; int d = sgxt28(t); carry = (t - d) >> W; D(p) = d; }
    // quotient estimate from the two top digits
    long long vt = ((long long)D(L - 1) << W) + D(L - 2);
    long long q = vt / (long long)K.nt_top;
    if (vt < 0 && vt % (long long)K.nt_top) q -= 1;           // floor division
    // v -= q * Nt, then fix up into [0, Nt)
    long long c64 = 0;
    for (int p = 0; p < L; p++) {
        long long t = (long long)D(p) - q * (long long)NT(p) + c64;
        int d = sgxt28((int)t); c64 = (t - d) >> W; D(p) = d;
    }
    for (int it = 0; it < 6; it++) {
        int top = 0;
        for (int p = L - 1; p >= 0; p--) { top = D(p); if (top) break; }
        int dir;
        if (top < 0) dir = 1;                                  // negative: add Nt
        else {
            // v >= Nt ?  compare via sign of v - Nt
            int cc = 0, last = 0; bool nonzero = false;
            for (int p = 0; p < L; p++) { int t = D(p) - NT(p) + cc; int d = sgxt28(t); cc = (t - d) >> W; if (d) { last = d; nonzero = true; } }
            dir = (!nonzero || last > 0) ? -1 : 0;             // v - Nt >= 0: subtract
        }
        if (dir == 0) break;
        int cc = 0;
        for (int p = 0; p < L; p++) { int t = D(p) + dir * NT(p) + cc; int d = sgxt28(t); cc = (t - d) >> W; D(p) = d; }
    }
    // unsigned digits (value is now in [0, Nt))
    carry = 0;
    for (int p = 0; p < L; p++) { int t = D(p) + carry; D(p) = t & ((1 << W) - 1); carry = t >> W; }
    // shift right by sh and pack into 64-bit words
    for (int j = 0; j < K.words_out; j++) {
        u64 w = 0;
        int bit0 = 64 * j + K.sh;
        int p0 = bit0 / W;
        for (int p = p0; p < p0 + 4 && p < L; p++) {
            int off = W * p - bit0;                           // position of digit p relative to the word
            u64 d = (u64)(unsigned)D(p);
            if (off >= 64) break;
            w |= off >= 0 ? d << off : d >> (-off);
        }
        out[j] = w;
    }
}

template <class C, int ENG, class SV>
__device__ __forceinline__ void finalize(SV& S, const B28Dev& K, u64* out, bool active, int role, int lane) {
    mulmod_const<C, ENG>(S, S.two_sh, role, lane);
    if (role == 0 && active) canonical_out<C>(S.V, S.Nt, K, out, lane);
    __syncthreads();
}

// ---- kernels ---------------------------------------------------------------------------------
// comb table, stage 1: bases[i] = g^(2^(w i)) mod Nt, i < n_windows (one CTA; every lane computes the same value)
template <class C>
__global__ void __launch_bounds__(C::THREADS, 1) k_gtable_bases(B28Dev K, const u64* g_words, int4* bases) {
    extern __shared__ int4 smem[];
    Smem<C> S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    load_consts<C>(smem, K);
    load_value<C>(S.V, g_words, K.words_in, role, lane);
    for (int i = 0; i < K.n_windows; i++) {
        if (lane == 0) scatter_entry<C>(bases + (size_t)i * C::ENTRY4, S.V, role, lane);
        __syncthreads();
        if (i + 1 < K.n_windows)
            for (int s = 0; s < K.comb_bits; s++) mulmod<C, true>(S, nullptr, role, lane);
    }
}
// comb table, stage 2: lane = window; TG[i][d] = bases[i]^d, d < 2^w
template <class C>
__global__ void __launch_bounds__(C::THREADS, 1) k_gtable_fill(B28Dev K, const int4* bases, int4* tg) {
    extern __shared__ int4 smem[];
    Smem<C> S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    load_consts<C>(smem, K);
    int win = blockIdx.x * 32 + lane;
    bool active = win < K.n_windows;
    if (!active) win = K.n_windows - 1;
    const int nd = 1 << K.comb_bits;
    int4* row = tg + (size_t)win * nd * C::ENTRY4;
    set_one_where<C>(S.V, true, role, lane);
    if (active) scatter_entry<C>(row, S.V, role, lane);
    gather_entry<C>(S.V, bases + (size_t)win * C::ENTRY4, role, lane);
    gather_entry<C>(S.B, bases + (size_t)win * C::ENTRY4, role, lane);
    for (int d = 1; d < nd; d++) {
        if (active) scatter_entry<C>(row + (size_t)d * C::ENTRY4, S.V, role, lane);
        __syncthreads();
        if (d + 1 < nd) mulmod<C, false>(S, S.B, role, lane);
    }
}

// Per-CTA global scratch is sized by the CTAs that can be RESIDENT, not by the grid: a CTA takes one of the `per_sm` slots of the
// SM it runs on (a bit of masks[%smid], atomicCAS) and gives it back when it ends.  per_sm is the occupancy the runtime reports
// for the kernel, so a free bit always exists; the loop still re-reads the mask should that ever not hold.
struct SlotPool { unsigned* masks; int per_sm; };
__device__ __forceinline__ int slot_acquire(const SlotPool& P) {
    unsigned* mk = P.masks + smid();
    const unsigned full = P.per_sm >= 32 ? 0xffffffffu : ((1u << P.per_sm) - 1u);
    for (;;) {
        const unsigned cur = *(volatile unsigned*)mk;
        const unsigned free_bits = ~cur & full;
        if (!free_bits) { __nanosleep(100); continue; }
        const int b = __ffs((int)free_bits) - 1;
        if (atomicCAS(mk, cur, cur | (1u << b)) == cur) return (int)smid() * P.per_sm + b;
    }
}
__device__ __forceinline__ void slot_release(const SlotPool& P, int slot) {
    atomicAnd(P.masks + slot / P.per_sm, ~(1u << (slot % P.per_sm)));
}
__global__ void k_nsmid(unsigned* out) { unsigned v; asm volatile("mov.u32 %0, %%nsmid;" : "=r"(v)); *out = v; }

// the slots of a CTA's LG lane groups, s_slot[g] in shared memory: thread 0 takes them before cta_begin (whose barrier publishes
// them) and gives them back when the CTA ends
template <int LG>
__device__ __forceinline__ void slots_acquire(const SlotPool& P, int* s_slot) {
    if (threadIdx.x == 0) for (int g = 0; g < LG; g++) s_slot[g] = slot_acquire(P);
}
template <int LG>
__device__ __forceinline__ void slots_release(const SlotPool& P, const int* s_slot) {
    if (threadIdx.x == 0) for (int g = 0; g < LG; g++) slot_release(P, s_slot[g]);
}

// V <- x^e for the x in V (each lane its own), e given by its sliding-window schedule E; e == 0 gives 1.  The odd powers x, x^3, ..,
// x^(2 TABN - 1) go to tab[0 .. TABN) of the CTA's scratch slot, x^2 to tab[TABN].
template <class C, int ENG, class SV>
__device__ __forceinline__ void window_pow(SV& S, const PowSched& E, int4* tab, int role, int lane) {
    copy_to_global<C>(tab, S.V, role, lane);                                        // tab[0] = x
    mm<C, true, ENG>(S, nullptr, role, lane);                                   // x^2
    copy_to_global<C>(tab + (size_t)TABN * C::VAL4, S.V, role, lane);
    __syncthreads();
    copy_from_global<C>(S.V, tab, role, lane);
    for (int j = 1; j < TABN; j++) {
        copy_from_global<C>(S.B, tab + (size_t)TABN * C::VAL4, role, lane);
        mm<C, false, ENG>(S, S.B, role, lane);                                  // x^(2j+1)
        copy_to_global<C>(tab + (size_t)j * C::VAL4, S.V, role, lane);
    }
    __syncthreads();
    if (E.first_idx < 0) set_one_where<C>(S.V, true, role, lane);                   // e == 0
    else copy_from_global<C>(S.V, tab + (size_t)E.first_idx * C::VAL4, role, lane);
    for (int o = 0; o < E.n_ops; o++) {
        const int2 op = E.ops[o];
        for (int s_ = 0; s_ < op.x; s_++) mm<C, true, ENG>(S, nullptr, role, lane);
        if (op.y >= 0) {
            copy_from_global<C>(S.B, tab + (size_t)op.y * C::VAL4, role, lane);
            mm<C, false, ENG>(S, S.B, role, lane);
        }
    }
}

// c-bit window i (c <= 16) of the unsigned integer w[0 .. nwords) (u64 little-endian): bits [i c, i c + c)
__device__ __forceinline__ int window_digit(const u64* w, int nwords, int i, int c) {
    const int bit = i * c, wi = bit >> 6, sft = bit & 63;
    u64 v = w[wi] >> sft;
    if (sft + c > 64 && wi + 1 < nwords) v |= w[wi + 1] << (64 - sft);
    return (int)(v & ((1u << c) - 1));
}

template <class C, int ENG>
__global__ void __launch_bounds__(View<C, ENG>::THREADS, View<C, ENG>::PER_SM) k_encrypt(B28Dev K, const u64* __restrict__ m, const u64* __restrict__ r,
                                                            size_t count, u64* __restrict__ c_out, int4* scratch, SlotPool pool) {
    extern __shared__ int4 smem[];
    __shared__ int s_slot[2];
    constexpr int LG = View<C, ENG>::LG;
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = (threadIdx.x >> 5) % C::G, grp = (threadIdx.x >> 5) / C::G;      // grp: lane group (LG per CTA)
    slots_acquire<LG>(pool, s_slot);
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit<LG>(count, lane, grp);
    int4* tab = scratch + (size_t)s_slot[grp] * SCRATCH_ENTRIES * C::VAL4;
    // ---- r^n: odd powers table, then the per-key window schedule
    load_value<C>(S.V, r + unit * K.words_in, K.words_in, role, lane);
    window_pow<C, ENG>(S, K.rn, tab, role, lane);
    copy_to_global<C>(tab + (size_t)(TABN + 1) * C::VAL4, S.V, role, lane);    // rn
    __syncthreads();
    // ---- g^m: comb over the bytes of m
    const u64* mw = m + unit * K.words_in;
    const int cb = K.comb_bits;
    if (K.n_entry) {
        // g = n + 1: (1 + n)^m = 1 + m n (mod n^2) — one multiplication by the per-key constant n instead of the comb
        load_value<C>(S.V, mw, K.words_in, role, lane);
        mulmod_const<C, ENG>(S, K.n_entry, role, lane);
        if (role == 0) ((int*)blk_ptr<C>(S.V, 0, lane))[0] += 1;
        __syncthreads();
    } else {
        gather_entry<C>(S.V, K.tg + (size_t)window_digit(mw, K.words_in, 0, cb) * C::ENTRY4, role, lane);
        for (int i = 1; i < K.n_windows; i++) {
            gather_entry<C>(S.B, K.tg + (((size_t)i << cb) + window_digit(mw, K.words_in, i, cb)) * C::ENTRY4, role, lane);
            mm<C, false, ENG>(S, S.B, role, lane);
        }
    }
    // ---- c = gm * rn, canonical
    copy_from_global<C>(S.B, tab + (size_t)(TABN + 1) * C::VAL4, role, lane);
    mm<C, false, ENG>(S, S.B, role, lane);
    finalize<C, ENG>(S, K, c_out + unit * K.words_out, active, role, lane);
    slots_release<LG>(pool, s_slot);
    cta_end(S);
}

// out = base^e mod n^2 for a per-key exponent e: the r-chain of k_encrypt (window_pow) with its own schedule.  Decryption's
// c^lambda mod n^2 (SURVEY.md 8f-4).
template <class C, int ENG>
__global__ void __launch_bounds__(View<C, ENG>::THREADS, View<C, ENG>::PER_SM) k_pow(B28Dev K, PowSched E, const u64* __restrict__ base, int base_words,
                                                                    size_t count, u64* __restrict__ out, int4* scratch, SlotPool pool) {
    extern __shared__ int4 smem[];
    __shared__ int s_slot[2];
    constexpr int LG = View<C, ENG>::LG;
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = (threadIdx.x >> 5) % C::G, grp = (threadIdx.x >> 5) / C::G;      // grp: lane group (LG per CTA)
    slots_acquire<LG>(pool, s_slot);
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit<LG>(count, lane, grp);
    int4* tab = scratch + (size_t)s_slot[grp] * SCRATCH_ENTRIES * C::VAL4;
    load_value<C>(S.V, base + unit * base_words, base_words, role, lane);
    window_pow<C, ENG>(S, E, tab, role, lane);
    finalize<C, ENG>(S, K, out + unit * K.words_out, active, role, lane);
    slots_release<LG>(pool, s_slot);
    cta_end(S);
}

// out = c^k mod n^2 with its own scalar k per lane: homomorphic scalar multiplication, Dec(c^k) = k Dec(c) mod n.  Fixed window of
// w bits aligned to bit 0; the table x^0 .. x^(2^w - 1) lives in the CTA's scratch slot.  Every lane runs the same sequence of
// multiplications (w squarings, then one multiplication by its own table entry; digit 0 multiplies by the stored 1), so control flow
// never depends on the lane and the lanes of a CTA share every mulmod.  The chain is as long as the CTA's longest scalar.
constexpr int SCALAR_MAXW = 5;
static_assert((1 << SCALAR_MAXW) <= SCRATCH_ENTRIES, "the scalar window's table must fit the CTA's scratch slot");

template <class C, int ENG>
__global__ void __launch_bounds__(View<C, ENG>::THREADS, View<C, ENG>::PER_SM) k_scalar(B28Dev K, const u64* __restrict__ c, const u64* __restrict__ k,
                                                                       int k_words, int w, size_t count, u64* __restrict__ out,
                                                                       int4* scratch, SlotPool pool) {
    extern __shared__ int4 smem[];
    __shared__ int s_slot[2];
    __shared__ int s_bits;
    constexpr int LG = View<C, ENG>::LG;
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = (threadIdx.x >> 5) % C::G, grp = (threadIdx.x >> 5) / C::G;      // grp: lane group (LG per CTA)
    slots_acquire<LG>(pool, s_slot);
    if (threadIdx.x == 0) s_bits = 0;
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit<LG>(count, lane, grp);
    int4* tab = scratch + (size_t)s_slot[grp] * SCRATCH_ENTRIES * C::VAL4;
    const u64* kw = k + unit * k_words;
    // chain length: bits of the CTA's longest scalar (over both lane groups)
    if (role == 0 && active) {
        int b = 0;
        for (int i = k_words - 1; i >= 0; i--) if (kw[i]) { b = 64 * i + 64 - __clzll((long long)kw[i]); break; }
        if (b) atomicMax(&s_bits, b);
    }
    // table: tab[0] = 1, tab[1] = x, tab[e] = x^e (even e by squaring x^(e/2), odd e as x^(e-1) * x)
    load_value<C>(S.V, c + unit * K.words_out, K.words_out, role, lane);
    copy_to_global<C>(tab + C::VAL4, S.V, role, lane);
    set_one_where<C>(S.B, true, role, lane);
    copy_to_global<C>(tab, S.B, role, lane);
    for (int e = 2; e < (1 << w); e++) {
        if (e & 1) {
            copy_from_global<C>(S.B, tab + C::VAL4, role, lane);
            mm<C, false, ENG>(S, S.B, role, lane);
        } else {
            copy_from_global<C>(S.V, tab + (size_t)(e >> 1) * C::VAL4, role, lane);
            mm<C, true, ENG>(S, nullptr, role, lane);
        }
        copy_to_global<C>(tab + (size_t)e * C::VAL4, S.V, role, lane);
    }
    __syncthreads();
    // the chain: window digits straight from the scalar, table entries from this lane's own column
    const int nwin = (s_bits + w - 1) / w;
    if (nwin == 0) set_one_where<C>(S.V, true, role, lane);                            // every scalar of the CTA is 0
    else copy_from_global<C>(S.V, tab + (size_t)window_digit(kw, k_words, nwin - 1, w) * C::VAL4, role, lane);
    for (int i = nwin - 2; i >= 0; i--) {
        for (int s_ = 0; s_ < w; s_++) mm<C, true, ENG>(S, nullptr, role, lane);
        copy_from_global<C>(S.B, tab + (size_t)window_digit(kw, k_words, i, w) * C::VAL4, role, lane);
        mm<C, false, ENG>(S, S.B, role, lane);
    }
    finalize<C, ENG>(S, K, out + unit * K.words_out, active, role, lane);
    slots_release<LG>(pool, s_slot);
    cta_end(S);
}

// ---- tally: the N-ary fold of paillier_add_native (/root/reference/src/paillier.rs:94-97) in ONE launch per GPU -------------------
// 1. every lane of every CTA folds a strided subset of the inputs (main loop, all lanes useful);
// 2. the CTAs fold pairwise up a binary tree by "last arriver continues": a CTA stores its 32 lane values in its node slot, bumps
//    the node counter and leaves if its sibling has not arrived yet; the one that arrives second loads the sibling's values and
//    multiplies (32 useful lanes per multiplication, no spinning, no co-residency assumption);
// 3. the one surviving CTA folds its 32 lanes (5 steps) and canonicalises;
// 4. multi-GPU (world > 1): it stores the canonical partial into every peer's mailbox over NVLink (plain stores to mapped peer
//    memory, then a release flag at system scope), waits for the peers' partials in its own mailbox, folds the `world` partials
//    (3 steps at 8 GPUs) and canonicalises again — every GPU ends with the full product, no host hop and no second launch.
constexpr int TALLY_MAXW = 8;                          // GPUs of one NVSwitch domain
constexpr int MAIL_WORDS = 160;                        // one partial as lazy digits: ENTRY4 int4 = up to 16 blocks x 5 chunks x 16 B = 1280 B
constexpr size_t MAIL_FLAG_OFF = (size_t)2 * TALLY_MAXW * MAIL_WORDS;      // u64 index of flags[parity][src]
constexpr size_t MAIL_U64 = MAIL_FLAG_OFF + 2 * TALLY_MAXW;
struct TallyPeer {
    int world, rank;
    unsigned long long epoch;          // sequence number of this collective call (>= 1); parity selects the mailbox half
    u64* mail[TALLY_MAXW];             // every rank's mailbox as mapped on THIS device (mail[rank] is the local one)
    int* flags;                        // the key's flag word (bit 2: a peer's partial did not arrive)
};

template <class C>
__device__ __forceinline__ void copy_from_global_cg(int4* buf, const int4* g, int role, int lane) {     // written by another SM: L2 only
#pragma unroll
    for (int c = 0; c < C::CH; c++) buf[(role * C::CH + c) * 32 + lane] = __ldcg(g + (role * C::CH + c) * 32 + lane);
    __syncthreads();
}
// V[lane] <- product over the lanes of its aligned group of `width` lanes (width a power of two <= 32)
template <class C, int ENG, class SV>
__device__ __forceinline__ void fold_lanes(SV& S, int width, int role, int lane) {
    for (int off = width >> 1; off >= 1; off >>= 1) {
#pragma unroll
        for (int ch = 0; ch < C::CH; ch++) S.B[(role * C::CH + ch) * 32 + lane] = S.V[(role * C::CH + ch) * 32 + (lane ^ off)];
        __syncthreads();
        mm<C, false, ENG>(S, S.B, role, lane);
    }
}

template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_tally(B28Dev K, const u64* __restrict__ c, size_t count, u64* __restrict__ out,
                                                                      int4* nodes, unsigned* node_cnt, TallyPeer P) {
    extern __shared__ int4 smem[];
    __shared__ int s_first;
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    // ---- 1. main loop
    const size_t stride = (size_t)gridDim.x * 32;
    const size_t first = (size_t)blockIdx.x * 32 + lane;
    const size_t max_iters = (count + stride - 1) / stride;
    set_one_where<C>(S.V, true, role, lane);
    for (size_t it = 0; it < max_iters; it++) {
        const size_t u = first + it * stride;
        const size_t base = (size_t)blockIdx.x * 32 + it * stride;                  // first unit of this CTA step
        stage_words<C>((u64*)S.T, c + base * K.words_out, base < count ? (int)(count - base < 32 ? count - base : 32) : 0, K.words_out);
        load_value_staged<C>(S.B, (const u64*)S.T, K.words_out, role, lane);
        set_one_where<C>(S.B, u >= count, role, lane);                               // lanes without an input multiply by one
        mm<C, false, ENG>(S, S.B, role, lane);
    }
    // ---- 2. tree over the CTAs
    {
        int idx = blockIdx.x, n = gridDim.x;
        size_t node_base = 0;
        while (n > 1) {
            const int j = idx >> 1;
            if ((idx ^ 1) < n) {
                int4* slot = nodes + (node_base + j) * 2 * (size_t)C::VAL4;
                copy_to_global<C>(slot + (size_t)(idx & 1) * C::VAL4, S.V, role, lane);
                __threadfence();
                __syncthreads();
                if (threadIdx.x == 0) s_first = atomicAdd(node_cnt + node_base + j, 1u) == 0u;
                __syncthreads();
                if (s_first) { cta_end(S); return; }                                              // the sibling will pick this value up
                if (threadIdx.x == 0) node_cnt[node_base + j] = 0;                   // both arrived: ready for the next launch
                __threadfence();
                copy_from_global_cg<C>(S.B, slot + (size_t)((idx & 1) ^ 1) * C::VAL4, role, lane);
                mm<C, false, ENG>(S, S.B, role, lane);
            }
            node_base += (size_t)((n + 1) >> 1);
            idx = j; n = (n + 1) >> 1;
        }
    }
    // ---- 3. the surviving CTA: fold its lanes, canonical partial
    fold_lanes<C, ENG>(S, 32, role, lane);
    if (P.world <= 1) { finalize<C, ENG>(S, K, out, lane == 0, role, lane); cta_end(S); return; }
    // ---- 4. exchange over peer memory and combine.  What crosses NVLink is lane 0's LAZY value (strict digits, ENTRY4 int4): the
    // receivers multiply digit arrays directly, so neither a canonicalisation before the exchange nor a digit conversion after it
    const int par = (int)(P.epoch & 1);
    {
        const int4* v0 = S.V;                                   // lane 0's chunks: S.V[(block * CH + chunk) * 32 + 0]
        for (int idx = threadIdx.x; idx < P.world * C::ENTRY4; idx += C::THREADS) {
            const int peer = idx / C::ENTRY4, e = idx - peer * C::ENTRY4;
            int4* dst = reinterpret_cast<int4*>(P.mail[peer] + ((size_t)par * TALLY_MAXW + P.rank) * MAIL_WORDS) + e;
            *dst = v0[e * 32];
        }
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < P.world && (int)threadIdx.x != P.rank) {
        // publish: my partial is in peer t's mailbox;   then wait for peer t's partial in mine
        u64* theirs = P.mail[threadIdx.x] + MAIL_FLAG_OFF + (size_t)par * TALLY_MAXW + P.rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(theirs), "l"(P.epoch) : "memory");
        const u64* flag = P.mail[P.rank] + MAIL_FLAG_OFF + (size_t)par * TALLY_MAXW + threadIdx.x;
        const long long t0 = clock64();
        for (;;) {
            unsigned long long v;
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
            if (v >= P.epoch) break;
            if (clock64() - t0 > 6000000000ll) { atomicOr(P.flags, 4); break; }      // ~3 s: a peer never called
            __nanosleep(200);
        }
    }
    __syncthreads();
    {
        const int src = lane < P.world ? lane : P.world - 1;
        const int4* e = reinterpret_cast<const int4*>(P.mail[P.rank] + ((size_t)par * TALLY_MAXW + src) * MAIL_WORDS);
#pragma unroll
        for (int c = 0; c < C::CH; c++) S.V[(role * C::CH + c) * 32 + lane] = __ldcg(e + role * C::CH + c);
        __syncthreads();
    }
    set_one_where<C>(S.V, lane >= P.world, role, lane);
    int width = 1; while (width < P.world) width <<= 1;
    fold_lanes<C, ENG>(S, width, role, lane);
    finalize<C, ENG>(S, K, out, lane == 0, role, lane);
    cta_end(S);
}

// ---- matvec: bucket (Pippenger) multi-exponentiation, DESIGN.md §9b ------------------------------------------------------------
// The engine kernels below run the tally's CTA shape (32 lanes, ENG 0 / 1 / 4).  Values between them are either canonical words
// (words_out u64, read with load_value, written by finalize) or lazy digits (ENTRY4 int4 per value, gather_entry / scatter_entry).
template <class C>
__device__ __forceinline__ void scatter_one(int4* entry, int role) {
#pragma unroll
    for (int c = 0; c < C::CH; c++) entry[role * C::CH + c] = make_int4(role == 0 && c == 0 ? 1 : 0, 0, 0, 0);
}

// Reduce-by-key of a key-sorted list: out[key] = product of the values with that key (lazy digits).  Lane l takes the slice
// [l * ls, (l + 1) * ls) and multiplies every value of it into its accumulator, restarting at 1 on a key change (one multiplication
// per entry on every lane, padding multiplies by 1).  Runs that start and end inside the slice are complete and stored; the first and
// the last run of a slice may continue into a neighbour, so they go to the carry list as pieces 2l and 2l + 1 (a slice of one run
// emits it and a 1), which is again key-sorted and is folded by the next launch.  A launch whose list fits one slice stores every run.
// Level 0 gathers its values from words (src + idx[t] * src_words), later levels from the lazy pieces of the previous one.
// n: *d_n entries when d_n is set (counted on the device), else n_fixed; *d_n_next: entries of the carry list (0 when complete).
template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_bucket_fold(B28Dev K, const unsigned* __restrict__ keys, const unsigned* __restrict__ idx,
                                                                            const u64* __restrict__ src, int src_words, const int4* __restrict__ src_lazy,
                                                                            const unsigned* __restrict__ d_n, size_t n_fixed, int ls, int4* __restrict__ out,
                                                                            unsigned* __restrict__ keys_next, int4* __restrict__ vals_next, unsigned* __restrict__ d_n_next) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const size_t n = d_n ? *d_n : n_fixed;
    const size_t lanes = (n + ls - 1) / ls;
    const bool last = lanes <= 1;
    if (blockIdx.x == 0 && threadIdx.x == 0) *d_n_next = last ? 0u : (unsigned)(2 * lanes);
    if ((size_t)blockIdx.x * 32 >= lanes) return;                                   // the whole CTA is past the list
    cta_begin(S, smem, K);
    const size_t l = (size_t)blockIdx.x * 32 + lane, a = l * ls;
    const bool active = l < lanes;
    unsigned cur = active ? keys[a] : 0u;
    bool head = true;
    set_one_where<C>(S.V, true, role, lane);
    for (int it = 0; it < ls; it++) {
        const size_t t = a + it;
        const bool real = active && t < n;
        const unsigned kt = real ? keys[t] : cur;
        const bool brk = kt != cur;
        if (brk) {                                                                      // the run ending at t is finished
            if (head && !last) { scatter_entry<C>(vals_next + 2 * l * C::ENTRY4, S.V, role, lane); if (role == 0) keys_next[2 * l] = cur; }
            else scatter_entry<C>(out + (size_t)cur * C::ENTRY4, S.V, role, lane);
            head = false; cur = kt;
        }
        set_one_where<C>(S.V, brk, role, lane);
        const size_t ts = real ? t : n - 1;
        if (src) load_value<C>(S.B, src + (size_t)idx[ts] * src_words, src_words, role, lane);
        else gather_entry<C>(S.B, src_lazy + ts * C::ENTRY4, role, lane);
        set_one_where<C>(S.B, !real, role, lane);
        mm<C, false, ENG>(S, S.B, role, lane);
    }
    if (active) {
        if (last) scatter_entry<C>(out + (size_t)cur * C::ENTRY4, S.V, role, lane);
        else {
            scatter_entry<C>(vals_next + (2 * l + 1) * C::ENTRY4, S.V, role, lane);
            if (head) scatter_one<C>(vals_next + 2 * l * C::ENTRY4, role);
            if (role == 0) { keys_next[2 * l + 1] = cur; if (head) keys_next[2 * l] = cur; }
        }
    }
    cta_end(S);
}

// Buckets B_1 .. B_(2^c - 1) of a set -> per segment [a, a + lseg): T = prod B_d^(d - a + 1) and A = prod B_d, as running products from
// the top (A *= B_d, T *= A: two multiplications per bucket, buckets past 2^c - 1 are 1).  One lane per (set, segment); the set's
// W = prod B_d^d is then prod_s T_s * A_s^(a_s - 1), with a_exp[unit] = a - 1 the scalar of k_scalar.  T rests in the CTA's scratch
// while A is multiplied and the other way round.
template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_bucket_reduce(B28Dev K, const int4* __restrict__ buckets, int c, int nseg, int lseg,
                                                                              size_t units, u64* __restrict__ t_out, u64* __restrict__ a_out,
                                                                              u64* __restrict__ a_exp, int4* scratch) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit(units, lane);
    const size_t set = unit / nseg;
    const int a = 1 + (int)(unit % nseg) * lseg, dmax = (1 << c) - 1;
    const int4* bk = buckets + (set << c) * C::ENTRY4;
    int4* sa = scratch + (size_t)blockIdx.x * 2 * C::VAL4;
    int4* stt = sa + C::VAL4;
    set_one_where<C>(S.V, true, role, lane);
    copy_to_global<C>(sa, S.V, role, lane);                                             // A = 1, T = 1 (in V)
    for (int it = lseg - 1; it >= 0; it--) {
        const int d = a + it;
        copy_to_global<C>(stt, S.V, role, lane);
        copy_from_global<C>(S.V, sa, role, lane);
        gather_entry<C>(S.B, bk + (size_t)(d <= dmax ? d : dmax) * C::ENTRY4, role, lane);
        set_one_where<C>(S.B, d > dmax, role, lane);
        mm<C, false, ENG>(S, S.B, role, lane);                                          // A *= B_d
        copy_to_global<C>(sa, S.V, role, lane);
#pragma unroll
        for (int ch = 0; ch < C::CH; ch++) S.B[(role * C::CH + ch) * 32 + lane] = S.V[(role * C::CH + ch) * 32 + lane];
        __syncthreads();
        copy_from_global<C>(S.V, stt, role, lane);
        mm<C, false, ENG>(S, S.B, role, lane);                                          // T *= A
    }
    finalize<C, ENG>(S, K, t_out + unit * K.words_out, active, role, lane);
    copy_from_global<C>(S.V, sa, role, lane);
    finalize<C, ENG>(S, K, a_out + unit * K.words_out, active, role, lane);
    if (active && threadIdx.x < 32) a_exp[unit] = (u64)(a - 1);
    cta_end(S);
}

// x_u <- x_u^(2^(c * jg)) * prod_jl W_(u, jl)^(2^(c * jl)) (Horner over a group of windows, most significant first), one lane per
// (sign, row); x and W canonical, x updated in place
template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_horner(B28Dev K, u64* x, const u64* __restrict__ w, size_t units, int jg, int c) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit(units, lane);
    load_value<C>(S.V, x + unit * K.words_out, K.words_out, role, lane);
    for (int jl = jg - 1; jl >= 0; jl--) {
        for (int s_ = 0; s_ < c; s_++) mm<C, true, ENG>(S, nullptr, role, lane);
        load_value<C>(S.B, w + (unit * jg + jl) * K.words_out, K.words_out, role, lane);
        mm<C, false, ENG>(S, S.B, role, lane);
    }
    finalize<C, ENG>(S, K, x + unit * K.words_out, active, role, lane);
    cta_end(S);
}

// lazy digits -> canonical words, one lane per value
template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_lazy_canon(B28Dev K, const int4* __restrict__ in, size_t count, u64* __restrict__ out) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit(count, lane);
    gather_entry<C>(S.V, in + unit * C::ENTRY4, role, lane);
    finalize<C, ENG>(S, K, out + unit * K.words_out, active, role, lane);
    cta_end(S);
}

// Digits of one pass (rows [r0, r0 + rb), ciphertexts [i0, i0 + nc), windows [j0, j0 + jg)), one thread per (row, ciphertext): every
// non-zero c-bit digit d becomes one entry with key ((sign * rb + row) * jg + window) * 2^c + d and value i - i0.  keys == nullptr:
// histogram into cursor; else scatter to the positions cursor holds (its exclusive scan), order inside a bucket arbitrary.
__global__ void k_mv_digits(const u64* __restrict__ w, const uint8_t* __restrict__ neg, size_t count, int kw, size_t r0, size_t rb, size_t i0,
                            size_t nc, int c, int j0, int jg, unsigned* __restrict__ cursor, unsigned* __restrict__ keys, unsigned* __restrict__ idx) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rb * nc) return;
    const size_t r = t / nc, i = t - r * nc, e = (r0 + r) * count + i0 + i;
    const u64* m = w + e * kw;
    const unsigned sgn = neg && neg[e] ? 1u : 0u;
    for (int jl = 0; jl < jg; jl++) {
        const unsigned d = (unsigned)window_digit(m, kw, j0 + jl, c);
        if (!d) continue;
        const unsigned key = (((sgn * (unsigned)rb + (unsigned)r) * (unsigned)jg + (unsigned)jl) << c) + d;
        const unsigned p = atomicAdd(cursor + key, 1u);
        if (keys) { keys[p] = key; idx[p] = (unsigned)i; }
    }
}

// in-place exclusive scan of n counters, one CTA of 1024 threads (each a contiguous slice); *total = the sum
__global__ void __launch_bounds__(1024) k_mv_scan(unsigned* v, size_t n, unsigned* total) {
    __shared__ unsigned s[1024];
    const int tid = threadIdx.x;
    const size_t per = (n + 1023) / 1024, b = tid * per, e = b + per < n ? b + per : n;
    unsigned sum = 0;
    for (size_t i = b; i < e; i++) sum += v[i];
    s[tid] = sum;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        const unsigned x = tid >= off ? s[tid - off] : 0u;
        __syncthreads();
        s[tid] += x;
        __syncthreads();
    }
    unsigned run = s[tid] - sum;
    for (size_t i = b; i < e; i++) { const unsigned x = v[i]; v[i] = run; run += x; }
    if (tid == 1023) *total = s[1023];
}

// n lazy values (e4 int4 each) <- 1
__global__ void k_mv_one_lazy(int4* p, size_t n, int e4) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n * e4) p[t] = make_int4(t % e4 == 0 ? 1 : 0, 0, 0, 0);
}
// n canonical values (wo words each) <- 1
__global__ void k_mv_one_words(u64* p, size_t n, int wo) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n * wo) p[t] = t % wo == 0 ? 1 : 0;
}
// entry lists of the per-set fold: set s owns per = 2m (+ 1) entries, values at s*m + l (l < m), sets*m + s*m + l - m (l < 2m),
// 2*sets*m + s (l = 2m) of a [T | A' | W] block
__global__ void k_mv_block_entries(unsigned* keys, unsigned* idx, size_t sets, int m, int per) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= sets * per) return;
    const size_t s = t / per; const int l = (int)(t - s * per);
    keys[t] = (unsigned)s;
    idx[t] = (unsigned)(l < m ? s * m + l : l < 2 * m ? sets * m + s * m + (l - m) : 2 * sets * m + s);
}
// the magnitudes of one sign (the others 0): chain method
__global__ void k_mv_mask(const u64* __restrict__ w, const uint8_t* __restrict__ neg, size_t n, int kw, int sgn, u64* __restrict__ out) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * kw) return;
    const int s = neg && neg[t / kw] ? 1 : 0;
    out[t] = s == sgn ? w[t] : 0;
}



// ---- diagnostic: one modular multiplication on raw lazy digits, on a chosen engine ---------------------------------------------
// v_in / y_in / v_out: one CTA's values in the shared-memory image layout ([block][chunk][lane] int4, VAL4 int4); t_out: the 2L-digit
// product after phase A (2 VAL4 int4); rows_out: the q-hat digits as packed s8 words, [lane][L].  Used by the parity tests to compare
// the engines digit for digit (the lazy digits of block28t and block28u are specified to be identical).
template <class C, int ENG>
__global__ void __launch_bounds__(View<C, ENG>::THREADS, View<C, ENG>::PER_SM) k_mulmod_dbg(B28Dev K, const int4* v_in, const int4* y_in, int reps,
                                                                                 int4* v_out, int4* t_out, unsigned* rows_out) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    constexpr int LG = View<C, ENG>::LG;
    const int lane = threadIdx.x & 31, role = (threadIdx.x >> 5) % C::G, grp = (threadIdx.x >> 5) / C::G;      // every lane group works on the same input
    cta_begin(S, smem, K);
    copy_from_global<C>(S.V, v_in, role, lane);
    if (t_out) {            // phase A alone
        if (y_in) copy_from_global<C>(S.B, y_in, role, lane);
        if constexpr (ENG >= 2) phase_product_u<C, LG>(smem, S.B, y_in ? 0 : 1, S.tmem);
        else if constexpr (ENG == 1) phase_product<C>(S.V, S.B, y_in ? 0 : 1);
        else run_phase<C>(S.V, S.B, y_in ? PH_MUL : PH_SQR);
        if constexpr (ENG >= 2) {
            if (grp == LG - 1) for (int i = threadIdx.x % C::THREADS; i < 2 * C::VAL4; i += C::THREADS) t_out[i] = *(S.tblk(i / C::BLK4, 0) + i % C::BLK4);
        } else for (int i = threadIdx.x; i < 2 * C::VAL4; i += C::THREADS) t_out[i] = S.T[i];
        __syncthreads();
    } else {
        for (int r = 0; r < reps; r++) {
            if (y_in) { copy_from_global<C>(S.B, y_in, role, lane); mm<C, false, ENG>(S, S.B, role, lane); }
            else mm<C, true, ENG>(S, nullptr, role, lane);
        }
        if (grp == LG - 1) copy_to_global<C>(v_out, S.V, role, lane);
        if (rows_out && grp == LG - 1) {
#pragma unroll 1
            for (int k = 0; k < C::BL; k++) {
                const int qd = role * C::BL + k;
                unsigned w = 0;
                if constexpr (ENG >= 2) w = *(const unsigned*)(S.asc() + (UL<C, LG>::FRONT + (qd >> 2)) * UL<C, LG>::CHB + (grp * 32 + lane) * 16 + (qd & 3) * 4);
                else if constexpr (ENG == 1) w = ((const unsigned*)(as_ptr<C>(S) + lane * C::RS))[qd];
                rows_out[lane * C::L + qd] = w;
            }
        }
        __syncthreads();
    }
    cta_end(S);
}


// diagnostic: `reps` modular squarings per CTA on a grid of CTAs, cycles of phase A and of phases B + C accumulated by thread 0
// (cyc[cta] = {phase A, phases B and C, whole loop}); every CTA works on the same input
template <class C, int ENG>
__global__ void __launch_bounds__(View<C, ENG>::THREADS, View<C, ENG>::PER_SM) k_mulmod_time(B28Dev K, const int4* v_in, int reps, int stagger, long long* cyc, unsigned* sm_count) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    constexpr int LG = View<C, ENG>::LG;
    const int lane = threadIdx.x & 31, role = (threadIdx.x >> 5) % C::G;
    cta_begin(S, smem, K);
    copy_from_global<C>(S.V, v_in, role, lane);
    __shared__ unsigned s_order;
    if (threadIdx.x == 0) s_order = atomicAdd(sm_count + smid(), 1u);
    __syncthreads();
    if (stagger > 0 && (s_order & 1)) {             // delay the second CTA of every SM (diagnostic of the A / tensor ping-pong between co-resident CTAs)
        const long long t0 = clock64();
        while (clock64() - t0 < stagger) __nanosleep(200);
        __syncthreads();
    }
    long long ta = 0, tb = 0;
    const long long t_begin = clock64();
    // stagger -2: the first CTA of an SM runs phase A only, the second phases B + C only (interference between the two, no dependency);
    // -3: phase A only everywhere; -4: phases B + C only everywhere
    const bool do_a = stagger == -3 || (stagger == -2 && !(s_order & 1)) || stagger >= 0;
    const bool do_bc = stagger == -4 || (stagger == -2 && (s_order & 1)) || stagger >= 0;
    for (int r = 0; r < reps; r++) {
        const long long t0 = clock64();
        if (do_a) {
            if constexpr (ENG >= 2) phase_product_u<C, LG>(smem, nullptr, 1, S.tmem);
            else phase_product<C>(S.V, nullptr, 1);
        }
        const long long t1 = clock64();
        if (!do_bc) { ta += t1 - t0; continue; }
        if constexpr (ENG >= 2) phases_bc_umma<C, LG>(smem, S.tmem);
        else {
            q1_to_bytes<C>(S, role, lane);
            phase_mma<C, true>(S.V);
            qhat_to_bytes<C>(S, role, lane);
            phase_mma<C, false>(S.V);
            low_to_value<C>(S, role, lane);
        }
        const long long t2 = clock64();
        ta += t1 - t0; tb += t2 - t1;
    }
    if (threadIdx.x == 0) { cyc[3 * blockIdx.x] = ta; cyc[3 * blockIdx.x + 1] = tb; cyc[3 * blockIdx.x + 2] = clock64() - t_begin; }
    cta_end(S);
}

// ---- witness kernels (reference chain with exact (q, rem) per mul_mod) ---------------------------------
struct WitDev {
    const int4* gtab;          // [n_bits][ENTRY4]: strict digits of (g^(2^i) mod n^2) * 2^s   (i = 0: g itself)
    const int4* one_s;         // ENTRY4: 2^s
    const u64* cpow;           // C^(j+1), j < 2*words_out (record hash, include/paillier_b200.h)
    const u64* n_words;        // exponent of the r-chain
    int exp_bits;              // bits(n)
    int sh;                    // Nt_w = n^2 << sh, sh even; chain values carry the factor 2^(sh/2)
    double inv;                // 2^(28(L-2)) / Nt_w
};
struct WitIO {
    const u64* m; const u64* r; size_t count;
    u64* c_out;                // nullable
    u64* records; const u64* offsets;   // nullable: unit u's records start at record index offsets[u]
    u64* digest;               // nullable
    int4* scratch;             // 2 values per CTA: acc of the r-chain, gm
};

// ---- witness engine selection: 0 = block28t arithmetic (mma.sync phases), 1 = block28u arithmetic (tcgen05 phases) ---------------
template <class C, int WENG> struct WView {
    typedef Smem<C> type;
    static constexpr bool SUPPORTED = true;
    static constexpr size_t BYTES = C::SMEM_W_BYTES;
    static constexpr int PER_SM = C::CTAS_PER_SM, THREADS = C::THREADS;
};
template <class C> struct WView<C, 1> {
    typedef SmemU<C, 1, true> type;
    static constexpr bool SUPPORTED = UL<C, 1, true>::SUPPORTED;
    static constexpr size_t BYTES = UL<C, 1, true>::SMEM_BYTES;
    static constexpr int PER_SM = UL<C, 1, true>::CTAS_PER_SM, THREADS = C::THREADS;
};
// q of the last witnessed mul_mod must fit words_out words (range check of assign_integer(q, 2*enc_bits), SURVEY.md A.4): true
// when this thread's block of the canonical q digits, which the step leaves in T, has a bit at or above 64 words_out
template <class C, class SV>
__device__ __forceinline__ bool q_too_wide(const SV& S, int words_out, int role, int lane) {
    const int* Qf = (const int*)S.T + C::L * 32;
    const int qbits = 64 * words_out;
    int bad = 0;
#pragma unroll
    for (int k = 0; k < C::BL; k++) {
        const int p = role * C::BL + k;
        const unsigned d = (unsigned)Qf[p * 32 + lane];
        const int lo = W * p;
        if (lo >= qbits) bad |= d != 0;
        else if (lo + W > qbits) bad |= (d >> (qbits - lo)) != 0;
    }
    return bad;
}
// one witnessed mul_mod (contract of mulmod_w, block28.cuh)
template <class C, int WENG, class SV>
__device__ __forceinline__ u64 wmm(int4* smem_base, SV& S, const int4* Y, int sqr, int4* next_dst, WStep out, int sh, int words_out,
                                   double inv, const u64* cpow) {
    if constexpr (WENG == 1) return mulmod_wu<C>(smem_base, S.tmem, Y, sqr, next_dst, out, sh, words_out, inv, cpow);
    else return mulmod_w<C>(smem_base, Y, sqr, next_dst, out, sh, words_out, inv, cpow);
}

// table entries of the witness chain from 64-bit words: entry i = strict digits of (value_i << shl), one thread per entry.
// value_0 = g (words_in words); value_i = rem of g-chain record i-1 (words_out words at gchain + (i-1)*2*wo + wo)
template <class C>
__global__ void k_wtab(const u64* __restrict__ g_words, int words_in, const u64* __restrict__ gchain, int words_out,
                       int n_entries, int shl, int4* __restrict__ gtab) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_entries) return;
    const u64* src = i == 0 ? g_words : gchain + (size_t)(i - 1) * 2 * words_out + words_out;
    const int nwords = i == 0 ? words_in : words_out;
    int* dst = (int*)(gtab + (size_t)i * C::ENTRY4);
    for (int k = 0; k < C::ENTRY4 * 4; k++) dst[k] = 0;
    int carry = 0;
    for (int p = 0; p < C::L; p++)
        dst[(p / C::BL) * C::CH * 4 + (p % C::BL)] = strict_digit([src](int wi) { return src[wi]; }, nwords, W * p - shl, carry);
}

// per-key g-chain on the witness engine: record i = (q, rem) of (g^(2^i))^2, i < n_bits, and the table entries
// gtab[i] = strict digits of g^(2^i) * 2^s.  One CTA; every lane computes the same value, lane 0 writes.
template <class C, int WENG>
__global__ void __launch_bounds__(C::THREADS, 1) k_gchain_w(B28Dev K, WitDev Wd, const u64* __restrict__ g_words, int n_bits,
                                                            u64* __restrict__ gchain, int4* __restrict__ gtab) {
    extern __shared__ int4 smem[];
    typename WView<C, WENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    load_value<C>(S.V, g_words, K.words_in, role, lane, Wd.sh >> 1);
    for (int i = 0; i < n_bits; i++) {
        if (lane == 0) scatter_entry<C>(gtab + (size_t)i * C::ENTRY4, S.V, role, lane);
        WStep o; o.rec = lane == 0 ? gchain + (size_t)i * 2 * K.words_out : nullptr; o.rem_out = nullptr;
        wmm<C, WENG>(smem, S, nullptr, 1, S.V, o, Wd.sh, K.words_out, Wd.inv, Wd.cpow);
    }
    cta_end(S);
}

// One unit per lane, the reference's chain (src/paillier.rs:51,55,57 -> pow_mod_fixed_exp, SURVEY.md A.5):
//   g-chain: the popcount(m) multiplications acc *= g^(2^i) (the squarings are per key: gtab);
//   r-chain: for every bit i of n, sqr_i = cur^2 and, if the bit is set, acc *= cur; then gm * rn.
// Lanes walk their own set bits of m (inactive lanes multiply by one and emit nothing); the r-chain is uniform.
// In the r-chain the multiplication of an iteration is computed BEFORE its squaring (cur stays in V), the
// records keep the reference's order (sqr_i, then mul_i).
template <class C, int WENG>
__global__ void __launch_bounds__(C::THREADS, WView<C, WENG>::PER_SM) k_witness(B28Dev K, WitDev Wd, WitIO A) {
    extern __shared__ int4 smem[];
    typename WView<C, WENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const auto [unit, active] = lane_unit(A.count, lane);
    const int wo = K.words_out;
    const size_t recw = 2 * (size_t)wo;
    const u64* mw = A.m + unit * K.words_in;
    int pc = 0;
    for (int w = 0; w < K.words_in; w++) pc += __popcll(mw[w]);
    int maxpc = pc;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) maxpc = max(maxpc, __shfl_xor_sync(0xffffffffu, maxpc, off));
    u64* rec = (A.records && active) ? A.records + A.offsets[unit] * recw : nullptr;
    u64 D = PB200_DIGEST_INIT;                                    // running digest of the unit (kept by warp 0)
    int4* sc_acc = A.scratch + (size_t)blockIdx.x * 2 * C::VAL4;
    int4* sc_gm = sc_acc + C::VAL4;
    // ---- g-chain
    gather_entry<C>(S.V, Wd.one_s, role, lane);
    {
        int wi = 0; u64 cur = mw[0];
        for (int t = 0; t < maxpc; t++) {
            const bool act = t < pc;
            const int4* e = Wd.one_s;
            if (act) {
                while (!cur) cur = mw[++wi];
                const int b = __ffsll((long long)cur) - 1;
                cur &= cur - 1;
                e = Wd.gtab + (size_t)(64 * wi + b) * C::ENTRY4;
            }
            gather_entry<C>(S.B, e, role, lane);
            WStep o; o.rec = (act && rec) ? rec + (size_t)t * recw : nullptr; o.rem_out = nullptr;
            const u64 H = wmm<C, WENG>(smem, S, S.B, 0, S.V, o, Wd.sh, wo, Wd.inv, Wd.cpow);
            if (act) D = (D ^ H) * PB200_DIGEST_PRIME;
        }
    }
    copy_to_global<C>(sc_gm, S.V, role, lane);
    // ---- r-chain
    gather_entry<C>(S.B, Wd.one_s, role, lane);
    copy_to_global<C>(sc_acc, S.B, role, lane);
    load_value<C>(S.V, A.r + unit * K.words_in, K.words_in, role, lane, Wd.sh >> 1);
    size_t idx = (size_t)pc;
    for (int i = 0; i < Wd.exp_bits; i++) {
        const bool bit = (Wd.n_words[i >> 6] >> (i & 63)) & 1;
        u64 Hm = 0;
        if (bit) {
            copy_from_global<C>(S.B, sc_acc, role, lane);
            WStep o; o.rec = rec ? rec + (idx + 1) * recw : nullptr; o.rem_out = nullptr;
            Hm = wmm<C, WENG>(smem, S, S.B, 0, S.B, o, Wd.sh, wo, Wd.inv, Wd.cpow);
            copy_to_global<C>(sc_acc, S.B, role, lane);
        }
        WStep o; o.rec = rec ? rec + idx * recw : nullptr; o.rem_out = nullptr;
        const u64 Hs = wmm<C, WENG>(smem, S, nullptr, 1, S.V, o, Wd.sh, wo, Wd.inv, Wd.cpow);
        D = (D ^ Hs) * PB200_DIGEST_PRIME;
        if (bit) D = (D ^ Hm) * PB200_DIGEST_PRIME;
        idx += bit ? 2 : 1;
    }
    // ---- final: mul_mod(gm, rn)
    __syncthreads();
    copy_from_global<C>(S.V, sc_gm, role, lane);
    copy_from_global<C>(S.B, sc_acc, role, lane);
    {
        WStep o; o.rec = rec ? rec + idx * recw : nullptr;
        o.rem_out = (A.c_out && active) ? A.c_out + unit * wo : nullptr;
        const u64 H = wmm<C, WENG>(smem, S, S.B, 0, nullptr, o, Wd.sh, wo, Wd.inv, Wd.cpow);
        D = (D ^ H) * PB200_DIGEST_PRIME;
    }
    if (role == 0 && active && A.digest) A.digest[unit] = D;
    cta_end(S);
}

// paillier_add_native / PaillierChip::add (src/paillier.rs:62-85, :94-97) for `count` pairs on the witness engine:
// one exact mul_mod per lane, rem (and optionally q) as 64-bit words.  Inputs are c_words words each (zero-extended,
// src/paillier.rs:79-80) and need not be reduced; a quotient that does not fit words_out words raises the range flag.
template <class C, int WENG>
__global__ void __launch_bounds__(C::THREADS, WView<C, WENG>::PER_SM) k_add_w(B28Dev K, WitDev Wd, const u64* __restrict__ c1,
                                                                      const u64* __restrict__ c2, int c_words, size_t count,
                                                                      u64* __restrict__ out, u64* __restrict__ q_out, int* flags) {
    extern __shared__ int4 smem[];
    typename WView<C, WENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const int wo = K.words_out;
    for (size_t first = (size_t)blockIdx.x * 32; first < count; first += (size_t)gridDim.x * 32) {
        const auto [unit, active] = lane_unit(count, lane, 0, first);
        load_value<C>(S.V, c1 + unit * c_words, c_words, role, lane, Wd.sh >> 1);
        load_value<C>(S.B, c2 + unit * c_words, c_words, role, lane, Wd.sh >> 1);
        // the record goes through a per-lane staging area only when q is wanted; rem alone is written directly
        WStep o; o.rec = nullptr; o.rem_out = active ? out + unit * wo : nullptr;
        o.q_out = (active && q_out) ? q_out + unit * wo : nullptr;
        wmm<C, WENG>(smem, S, S.B, 0, nullptr, o, Wd.sh, wo, Wd.inv, Wd.cpow);
        if (q_too_wide<C>(S, wo, role, lane) && active) atomicOr(flags, 1);
        __syncthreads();
    }
    cta_end(S);
}

// ---- running-tally trace (pb200_tally_trace, DESIGN.md §9c) --------------------------------------------------------------------
// `chains` chains of n entries each, entry (i, j) of chain j at i * chains + j.  A level cuts every chain into chunks of s
// consecutive entries; lane u = b * chains + j owns chunk b of chain j.  Phase 1 (k_trace_reduce, fast engine) multiplies each chunk
// into a lazy total, level after level; phase 2 (k_trace_apply) turns the totals into exclusive prefixes from the top level down;
// phase 3 (k_trace_w, witness engine) runs the exact chain of every leaf chunk from its carry-in.

// smem per-lane value <- one lazy entry, or 1 where !real (the entry is then not read)
template <class C>
__device__ __forceinline__ void gather_or_one(int4* buf, const int4* entry, bool real, int role, int lane) {
#pragma unroll
    for (int c = 0; c < C::CH; c++)
        buf[(role * C::CH + c) * 32 + lane] = real ? entry[role * C::CH + c] : make_int4(role == 0 && c == 0 ? 1 : 0, 0, 0, 0);
    __syncthreads();
}

// totals[u] = product of chunk b of chain j (lazy).  Level 0 reads words (in_words, words_out each, any value), later levels the lazy
// totals of the level below.  The first entry is loaded, the others multiplied in; entries past the end of the chain multiply by 1.
template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_trace_reduce(B28Dev K, const u64* __restrict__ in_words,
                                                                             const int4* __restrict__ in_lazy, size_t n, size_t chains,
                                                                             size_t s, int4* __restrict__ totals) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const size_t units = (n + s - 1) / s * chains;
    const auto [u, active] = lane_unit(units, lane);
    const size_t b = u / chains, j = u - b * chains;
    for (size_t t = 0; t < s; t++) {
        const size_t i = b * s + t;
        const bool real = i < n;                                                         // always true for t = 0
        const size_t e = (real ? i : n - 1) * chains + j;
        int4* dst = t ? S.B : S.V;
        if (in_words) load_value<C>(dst, in_words + e * K.words_out, K.words_out, role, lane);
        else gather_entry<C>(dst, in_lazy + e * C::ENTRY4, role, lane);
        if (t) {
            set_one_where<C>(S.B, !real, role, lane);
            mm<C, false, ENG>(S, S.B, role, lane);
        }
    }
    if (active) scatter_entry<C>(totals + u * C::ENTRY4, S.V, role, lane);
    cta_end(S);
}

// Exclusive prefix products of one level, in place: entry (b s + t, j) <- carry(b, j) * the entries before it in its chunk.  The carry
// of chunk b is the lazy prefix the level above wrote for it, or init_j at the top level (carry == null: one chunk per chain).
template <class C, int ENG>
__global__ void __launch_bounds__(C::THREADS, View<C, ENG>::PER_SM) k_trace_apply(B28Dev K, const u64* __restrict__ init,
                                                                            const int4* __restrict__ carry, int4* items, size_t n,
                                                                            size_t chains, size_t s) {
    extern __shared__ int4 smem[];
    typename View<C, ENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const size_t units = (n + s - 1) / s * chains;
    const auto [u, active] = lane_unit(units, lane);
    const size_t b = u / chains, j = u - b * chains;
    if (carry) gather_entry<C>(S.V, carry + u * C::ENTRY4, role, lane);
    else load_value<C>(S.V, init + j * K.words_out, K.words_out, role, lane);
    for (size_t t = 0; t < s; t++) {
        const size_t i = b * s + t;
        const bool real = active && i < n;
        int4* e = items + (real ? i * chains + j : 0) * C::ENTRY4;
        gather_or_one<C>(S.B, e, real, role, lane);                                      // the total, read before its slot is overwritten
        if (real) scatter_entry<C>(e, S.V, role, lane);
        if (t + 1 < s) mm<C, false, ENG>(S, S.B, role, lane);                            // the chunk's own product is not needed
    }
    cta_end(S);
}

// The exact chain of every leaf chunk on the witness engine: a <- carry-in (init_j for chunk 0, as given; else carry[u], canonical),
// then per step (q, rem) = divmod(a c_(i, j), n^2), rem to acc (and q to q_out), a <- rem.  Steps past the end multiply by 1 and store
// nothing.  A quotient that does not fit words_out words raises the range flag, as in k_add_w.
template <class C, int WENG>
__global__ void __launch_bounds__(C::THREADS, WView<C, WENG>::PER_SM) k_trace_w(B28Dev K, WitDev Wd, const u64* __restrict__ init,
                                                                        const u64* __restrict__ c, const u64* __restrict__ carry,
                                                                        size_t count, size_t chains, size_t s, u64* __restrict__ acc,
                                                                        u64* __restrict__ q_out, int* flags) {
    extern __shared__ int4 smem[];
    typename WView<C, WENG>::type S(smem);
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    cta_begin(S, smem, K);
    const int wo = K.words_out;
    const size_t units = (count + s - 1) / s * chains;
    const auto [u, active] = lane_unit(units, lane);
    const size_t b = u / chains, j = u - b * chains;
    load_value<C>(S.V, b ? carry + u * wo : init + j * wo, wo, role, lane, Wd.sh >> 1);
    for (size_t t = 0; t < s; t++) {
        const size_t i = b * s + t;
        const bool real = active && i < count;
        const size_t e = (i < count ? i : count - 1) * chains + j;
        load_value<C>(S.B, c + e * wo, wo, role, lane, Wd.sh >> 1);
        if (!real) {
#pragma unroll
            for (int ch = 0; ch < C::CH; ch++) S.B[(role * C::CH + ch) * 32 + lane] = __ldg(Wd.one_s + role * C::CH + ch);
        }
        __syncthreads();
        WStep o; o.rec = nullptr; o.rem_out = real ? acc + e * wo : nullptr;
        o.q_out = (real && q_out) ? q_out + e * wo : nullptr;
        wmm<C, WENG>(smem, S, S.B, 0, S.V, o, Wd.sh, wo, Wd.inv, Wd.cpow);
        if (q_too_wide<C>(S, wo, role, lane) && real) atomicOr(flags, 1);
        __syncthreads();
    }
    cta_end(S);
}

// ---- host side ---------------------------------------------------------------------------------
struct Block28Key {
    int G = 0, BL = 0;
    std::string name;
    B28Dev dev{};
    int4* d_consts = nullptr; int2* d_ops = nullptr; int4* d_tg = nullptr; u64* d_gwords = nullptr; int4* d_nentry = nullptr;
    int4* d_scratch = nullptr; size_t scratch_slots = 0;     // r-power tables, one per resident-CTA slot (SlotPool)
    unsigned* d_slot_masks = nullptr; int nsmid = 0, enc_per_sm = 0;
    int4* d_nodes = nullptr; unsigned* d_node_cnt = nullptr; size_t node_ctas = 0;   // tally tree: 2 values per node, arrival counters
    u64* d_mail = nullptr;                                   // tally mailbox (peer-visible), MAIL_U64 words
    TallyPeer peer{};                                        // world <= 1 until block28_tally_peer_connect
    void* ipc_opened[TALLY_MAXW] = {};                       // peer mailboxes opened with cudaIpcOpenMemHandle
    int device = 0;
    int2* d_pow_ops = nullptr; PowSched pow{};               // decryption exponent (block28_pow_prepare)
    bool pow_ready = false;
    int sms = 148;
    uint64_t n_sqr = 0, n_mul = 0;   // modular squarings / multiplications per encryption
    int eng = 1;                     // 0: all phases on IMAD (block28), 1: phases B, C on mma.sync (block28t), 2: on tcgen05, 32 ciphertexts per
                                     // CTA (block28u), 3: on tcgen05, 64 per CTA (block28u2; the tally and keys without that variant run as 2)
    bool has_u = false;              // a block28u variant is compiled for this configuration
    int4* d_uconsts = nullptr; int4* d_uconsts2 = nullptr; bool has_u2 = false;
    // witness engine (lazy: block28_witness_prepare)
    BigInt n; uint32_t n_bits = 0;
    bool wit_ready = false;
    int4* d_wuconsts = nullptr; bool has_wu = false;     // witness engine on the tcgen05 phases
    int4* d_wconsts = nullptr; int4* d_gtab = nullptr; int4* d_one_s = nullptr; u64* d_cpow = nullptr; u64* d_nwords = nullptr;
    int4* d_wscratch = nullptr; size_t wscratch_ctas = 0;
    B28Dev wdev{}; WitDev wit{};
};

template <class C>
static void to_entry(const BigInt& v, std::vector<int>& out) {   // centred digits in [blk][chunk*4] layout
    out.assign(C::ENTRY4 * 4, 0);
    int carry = 0;
    for (int p = 0; p < C::L; p++) {
        int t = (int)v.bits_at((size_t)W * p, W) + carry;
        int d = ((t + (1 << (W - 1))) & ((1 << W) - 1)) - (1 << (W - 1));
        carry = (t - d) >> W;
        out[(p / C::BL) * C::CH * 4 + (p % C::BL)] = d;
    }
    if (carry != 0 || v.bits() > (size_t)W * C::L - 1) throw std::runtime_error("block28: constant does not fit");
}

// signed 7-bit digits of a constant (4 per 28-bit digit, the top one absorbs the remainder)
template <class C>
static void to_k7(const std::vector<int>& entry, std::vector<signed char>& k7) {
    k7.assign(C::K7, 0);
    for (int p = 0; p < C::L; p++) {
        int d = entry[(p / C::BL) * C::CH * 4 + (p % C::BL)];
        for (int i = 0; i < 3; i++) { int e = ((d + 64) & 127) - 64; k7[4 * p + i] = (signed char)e; d = (d - e) >> 7; }
        if (d < -128 || d > 127) throw std::runtime_error("block28: constant digit does not split into s8");
        k7[4 * p + 3] = (signed char)d;
    }
}
// reversed, zero padded, byte-shifted s8 table of a constant's 7-bit digits (B operand of the IMMA phases)
template <class C>
static void to_rtab(const std::vector<int>& entry, std::vector<int>& out_words) {
    std::vector<signed char> k7;
    to_k7<C>(entry, k7);
    std::vector<signed char> rfull(C::XLEN + 8, 0);
    for (int j = 0; j < C::K7; j++) rfull[C::PAD7 + (C::K7 - 1 - j)] = k7[j];
    std::vector<signed char> tab((size_t)C::RTAB4 * 16, 0);
    for (int sft = 0; sft < 4; sft++)
        for (int x = 0; x < C::XLEN; x++) tab[(size_t)sft * C::XSTR + x] = x + sft < C::XLEN ? rfull[x + sft] : 0;
    out_words.resize((size_t)C::RTAB4 * 4);
    memcpy(out_words.data(), tab.data(), tab.size());
}

// left-to-right sliding window (width WIN) over a fixed exponent: returns the table index the chain starts from (-1 for e == 0)
// and the list of (squarings, table index to multiply by or -1)
static int window_schedule(const BigInt& e, std::vector<int2>& ops) {
    int first_idx = -1;
    int i = (int)e.bits() - 1, pending = 0; bool first = true;
    while (i >= 0) {
        if (!e.bit(i)) { pending++; i--; continue; }
        int j = i - WIN + 1; if (j < 0) j = 0;
        while (!e.bit(j)) j++;
        int val = 0; for (int b = i; b >= j; b--) val = (val << 1) | (e.bit(b) ? 1 : 0);
        int len = i - j + 1;
        if (first) { first_idx = (val - 1) / 2; first = false; }
        else ops.push_back(make_int2(pending + len, (val - 1) / 2));
        pending = 0; i = j - 1;
    }
    if (pending) ops.push_back(make_int2(pending, -1));
    return first_idx;
}

#define CUW(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return e_; } while (0)
#define CUK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { *cuda_err = e_; block28_destroy(key); return nullptr; } } while (0)

static size_t cdiv(size_t a, size_t b) { return (a + b - 1) / b; }

// *d <- a device copy of a host array, which must live until st is synchronised; an empty array still gets an address
template <class T, class E>
static cudaError_t upload(T** d, const std::vector<E>& h, cudaStream_t st) {
    const size_t bytes = h.size() * sizeof(E);
    CUW(cudaMalloc(d, bytes ? bytes : sizeof(E)));
    return bytes ? cudaMemcpyAsync(*d, h.data(), bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
}
// *E <- the sliding-window schedule of the exponent e, its steps uploaded to *d_ops (ops: the host copy, kept by the caller until st
// is synchronised)
static cudaError_t upload_schedule(const BigInt& e, std::vector<int2>& ops, int2** d_ops, PowSched* E, cudaStream_t st) {
    ops.clear();
    const int first_idx = window_schedule(e, ops);
    CUW(upload(d_ops, ops, st));
    *E = PowSched{*d_ops, (int)ops.size(), first_idx};
    return cudaSuccess;
}

// Per-key constants of a modulus Nt: mu = floor(2^(2 BETA) / Nt) and Nt as entries, and the constant block load_consts copies into
// shared memory: mu, Nt, `third` (an entry: 2^sh for the value engine, the unsigned digits of Nt for the witness engine), then the
// reversed s8 tables of mu and Nt
template <class C>
struct KeyConsts {
    std::vector<int> mu, nt, block;
    KeyConsts(const BigInt& Nt, const std::vector<int>& third) {
        to_entry<C>(BigInt::div(BigInt::pow2(2 * (size_t)C::BETA), Nt), mu);
        to_entry<C>(Nt, nt);
        std::vector<int> r_mu, r_nt;
        to_rtab<C>(mu, r_mu); to_rtab<C>(nt, r_nt);
        auto put = [&](const std::vector<int>& v) { block.insert(block.end(), v.begin(), v.end()); };
        put(mu); put(nt); put(third); put(r_mu); put(r_nt);
    }
};
// *d <- block28u's per-key shared-memory image for the layout UL<C, LG, WIT> (from OFF_CONST on): the first three constants of the
// block, then the Toeplitz core-matrix tables of mu and Nt.  Synchronises st (the image is a local).
template <class C, int LG, bool WIT = false>
static cudaError_t upload_u_image(int4** d, const KeyConsts<C>& k, cudaStream_t st) {
    typedef UL<C, LG, WIT> U;
    std::vector<signed char> img(U::KEY_BYTES, 0), k7;
    memcpy(img.data(), k.block.data(), 3 * C::ENTRY4 * 16);
    to_k7<C>(k.mu, k7);
    umma_cm_table<C, LG>(k7.data(), true, img.data() + (U::OFF_CMH - U::OFF_CONST));
    to_k7<C>(k.nt, k7);
    umma_cm_table<C, LG>(k7.data(), false, img.data() + (U::OFF_CML - U::OFF_CONST));
    CUW(upload(d, img, st));
    return cudaStreamSynchronize(st);
}

// The engine kernels need more dynamic shared memory than the default limit; the attribute is per device, so it is set on the
// device of every launch (and before an occupancy query, which counts against the current limit).
template <class V, class... P>
static cudaError_t allow_smem(void (*kern)(P...)) {
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V::BYTES);
}
// launch of an engine kernel: block and dynamic shared memory from its view V (View<C, ENG> or WView<C, WENG>)
template <class V, class... P, class... A>
static cudaError_t launch(void (*kern)(P...), size_t grid, cudaStream_t st, A... args) {
    CUW(allow_smem<V>(kern));
    kern<<<(unsigned)grid, V::THREADS, V::BYTES, st>>>(args...);
    count_launch();
    return cudaGetLastError();
}

// f(std::integral_constant<int, ENG>()) for the ENG of E, ENGS... that equals eng and that the configuration compiles
// (V<C, ENG>::SUPPORTED); cudaErrorInvalidValue when there is none.  The list names the instantiations of one kernel family.
template <template <class, int> class V, class C, int E, int... ENGS, class F>
static cudaError_t with_eng(int eng, F&& f) {
    if constexpr (V<C, E>::SUPPORTED) if (eng == E) return f(std::integral_constant<int, E>());
    if constexpr (sizeof...(ENGS) > 0) return with_eng<V, C, ENGS...>(eng, f);
    else return cudaErrorInvalidValue;
}
// The key's engine per kernel family (block28_set_engine has already fallen back to an engine the configuration compiles):
// k_encrypt, k_pow, k_scalar run key->eng itself (0..3); the tally and the bucket kernels run tcgen05 as 4 and have no 3;
// the witness kernels run tcgen05 (WENG 1) where the key has that variant.
static int tally_eng(const Block28Key* key) { return key->eng >= 2 ? 4 : key->eng; }
static int wit_eng(const Block28Key* key) { return key->has_wu && key->eng >= 2 ? 1 : 0; }

template <class C>
static Block28Key* create_cfg(const BigInt& n, const BigInt& g, uint32_t n_bits, int device, cudaStream_t st, cudaError_t* cuda_err) {
    Block28Key* key = new Block28Key();
    key->G = C::G; key->BL = C::BL;
    key->n = n; key->n_bits = n_bits; key->device = device;
    key->name = "block28t<" + std::to_string(C::G) + "," + std::to_string(C::BL) + ">";      // block28_set_engine(-1) below picks the fastest
    cudaDeviceProp prop;
    CUK(cudaGetDeviceProperties(&prop, device));
    key->sms = prop.multiProcessorCount;
    BigInt n2 = BigInt::mul(n, n);
    int sh = C::KN - (int)n2.bits();
    BigInt Nt = BigInt::shl(n2, sh);
    std::vector<int> e_sh;
    to_entry<C>(BigInt::pow2(sh), e_sh);
    const KeyConsts<C> kc(Nt, e_sh);
    CUK(upload(&key->d_consts, kc.block, st));
    // block28u: the same constants followed by the two Toeplitz core-matrix tables, for one and for two lane groups per CTA
    if constexpr (UL<C, 1>::SUPPORTED) {
        CUK((upload_u_image<C, 1>(&key->d_uconsts, kc, st)));
        key->has_u = true;
    }
    if constexpr (UL<C, 1>::SUPPORTED && UL<C, 2>::SUPPORTED) {
        CUK((upload_u_image<C, 2>(&key->d_uconsts2, kc, st)));
        key->has_u2 = true;
    }
    block28_set_engine(key, -1);
    // sliding-window schedule for the exponent n
    std::vector<int2> ops;
    CUK(upload_schedule(n, ops, &key->d_ops, &key->dev.rn, st));
    int comb_bits = n_bits >= 1024 ? 12 : 8;
    if (const char* e = getenv("PB200_COMB_BITS")) { int v = atoi(e); if (v >= 4 && v <= 16) comb_bits = v; }
    const int n_windows = (int)((n_bits + comb_bits - 1) / comb_bits);
    const bool g_std = g == BigInt::add(n, BigInt(1)) && !getenv("PB200_NO_GSTD");
    key->n_sqr = 1; key->n_mul = (TABN - 1) + (g_std ? 1 : (uint64_t)(n_windows - 1)) + 1;   // r^2; table; comb (or m*n); gm*rn
    for (auto& o : ops) { key->n_sqr += (uint64_t)o.x; if (o.y >= 0) key->n_mul += 1; }
    uint32_t win = (n_bits + 63) / 64;
    std::vector<u64> gw(win);
    g.to_u64_le(gw.data(), win);
    CUK(upload(&key->d_gwords, gw, st));
    if (!g_std) CUK(cudaMalloc(&key->d_tg, ((size_t)n_windows << comb_bits) * C::ENTRY4 * sizeof(int4)));
    if (g_std) {
        std::vector<int> e_n;
        to_entry<C>(n, e_n);
        CUK(upload(&key->d_nentry, e_n, st));
        CUK(cudaStreamSynchronize(st));
    }
    B28Dev& K = key->dev;
    K.n_entry = key->d_nentry;
    K.consts = key->d_consts; K.uconsts = key->d_uconsts; K.uconsts2 = key->d_uconsts2;
    K.tg = key->d_tg; K.n_windows = n_windows; K.comb_bits = comb_bits; K.words_in = (int)win; K.words_out = (int)((2 * n_bits + 63) / 64);
    K.sh = sh;
    K.sms = (unsigned)key->sms;
    K.nt_top = (unsigned)BigInt::shr(Nt, (size_t)W * (C::L - 2)).bits_at(0, 32);
    // comb table
    int4* d_bases = nullptr;
    cudaError_t e = cudaSuccess;
    if (!g_std) {      // the comb table is only needed for a general g
        CUK(cudaMalloc(&d_bases, (size_t)n_windows * C::ENTRY4 * sizeof(int4)));
        e = launch<View<C, 0>>(k_gtable_bases<C>, 1, st, K, key->d_gwords, d_bases);
        if (e == cudaSuccess) e = launch<View<C, 0>>(k_gtable_fill<C>, cdiv(n_windows, 32), st, K, d_bases, key->d_tg);
    }
    const cudaError_t es = cudaStreamSynchronize(st);
    if (d_bases) cudaFree(d_bases);
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) { *cuda_err = e; block28_destroy(key); return nullptr; }
    return key;
}

template <class C>
static cudaError_t ensure_slots(Block28Key* key, cudaStream_t st) {
    if (!key->d_scratch) {
        // slots = SM ids x resident CTAs per SM (occupancy of the kernel as compiled), independent of the batch size
        unsigned* d_n = nullptr; unsigned h_n = 0;
        CUW(cudaMalloc(&d_n, sizeof(unsigned)));
        k_nsmid<<<1, 1, 0, st>>>(d_n); count_launch();
        CUW(cudaMemcpyAsync(&h_n, d_n, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        CUW(cudaStreamSynchronize(st));
        cudaFree(d_n);
        int per_sm = 0;
        CUW((allow_smem<View<C, 1>>(k_encrypt<C, 1>)));
        CUW((cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_encrypt<C, 1>, C::THREADS, C::SMEM_BYTES)));
        if constexpr (UL<C, 1>::SUPPORTED) {
            int per_u = 0;
            CUW((allow_smem<View<C, 2>>(k_encrypt<C, 2>)));
            CUW((cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_u, k_encrypt<C, 2>, C::THREADS, UL<C, 1>::SMEM_BYTES)));
            if (per_u > per_sm) per_sm = per_u;
            if (per_sm < 2) per_sm = 2;       // a CTA of two lane groups takes two slots
        }
        if (per_sm < 1 || per_sm > 32 || h_n == 0) return cudaErrorLaunchOutOfResources;
        key->nsmid = (int)h_n; key->enc_per_sm = per_sm;
        CUW(cudaMalloc(&key->d_slot_masks, h_n * sizeof(unsigned)));
        CUW(cudaMemsetAsync(key->d_slot_masks, 0, h_n * sizeof(unsigned), st));
        const size_t slots = (size_t)h_n * per_sm;
        CUW(cudaMalloc(&key->d_scratch, slots * SCRATCH_ENTRIES * C::VAL4 * sizeof(int4)));
        key->scratch_slots = slots;
    }
    return cudaSuccess;
}

template <class C>
static cudaError_t encrypt_cfg(Block28Key* key, const u64* d_m, const u64* d_r, size_t count, u64* d_c, cudaStream_t st) {
    CUW(ensure_slots<C>(key, st));
    const SlotPool pool{key->d_slot_masks, key->enc_per_sm};
    return with_eng<View, C, 0, 1, 2, 3>(key->eng, [&](auto e) {
        return launch<View<C, e>>(k_encrypt<C, e>, cdiv(count, 32 * View<C, e>::LG), st, key->dev, d_m, d_r, count, d_c, key->d_scratch, pool);
    });
}

template <class C>
static cudaError_t pow_cfg(Block28Key* key, const u64* d_base, int base_words, size_t count, u64* d_out, cudaStream_t st) {
    CUW(ensure_slots<C>(key, st));
    const SlotPool pool{key->d_slot_masks, key->enc_per_sm};
    return with_eng<View, C, 0, 1, 2, 3>(key->eng, [&](auto e) {
        return launch<View<C, e>>(k_pow<C, e>, cdiv(count, 32 * View<C, e>::LG), st, key->dev, key->pow, d_base, base_words, count, d_out,
                                  key->d_scratch, pool);
    });
}

// multiplications of k_scalar's table and chain for k_bits-bit scalars with a w-bit window:
// (2^w - 2) for the table + (ceil(k_bits / w) - 1) * (w + 1) for the chain
static uint64_t scalar_cost(uint32_t k_bits, int w) { return ((1u << w) - 2) + ((k_bits + w - 1) / w - 1) * (uint64_t)(w + 1); }
// window width of the scalar chain for k_bits-bit scalars: the w <= SCALAR_MAXW with the fewest multiplications (5 at 2048 bits, 3 at 32)
static int scalar_window(uint32_t k_bits) {
    int best = 1;
    for (int w = 2; w <= SCALAR_MAXW; w++) if (scalar_cost(k_bits, w) < scalar_cost(k_bits, best)) best = w;
    return best;
}

template <class C>
static cudaError_t scalar_cfg(Block28Key* key, const u64* d_c, const u64* d_k, uint32_t k_bits, size_t count, u64* d_out, cudaStream_t st) {
    CUW(ensure_slots<C>(key, st));
    const SlotPool pool{key->d_slot_masks, key->enc_per_sm};
    const int kw = (int)((k_bits + 63) / 64), w = scalar_window(k_bits);
    return with_eng<View, C, 0, 1, 2, 3>(key->eng, [&](auto e) {
        return launch<View<C, e>>(k_scalar<C, e>, cdiv(count, 32 * View<C, e>::LG), st, key->dev, d_c, d_k, kw, w, count, d_out, key->d_scratch, pool);
    });
}

// nodes of the CTA tree over `n` leaves: sum of ceil(n / 2^l) for l >= 1
static size_t tree_nodes(size_t n) { size_t t = 0; while (n > 1) { n = (n + 1) >> 1; t += n; } return t; }

template <class C>
static cudaError_t tally_cfg(Block28Key* key, const u64* d_c, size_t count, u64* d_out, bool collective, cudaStream_t st) {
    const size_t cap = (size_t)C::CTAS_PER_SM * key->sms;
    size_t ctas = (count + 31) / 32;
    if (ctas > cap) ctas = cap;
    if (ctas < 1) ctas = 1;
    if (!key->d_nodes) {
        const size_t nodes = tree_nodes(cap) + 1;
        CUW(cudaMalloc(&key->d_nodes, nodes * 2 * C::VAL4 * sizeof(int4)));
        CUW(cudaMalloc(&key->d_node_cnt, nodes * sizeof(unsigned)));
        CUW(cudaMemsetAsync(key->d_node_cnt, 0, nodes * sizeof(unsigned), st));
        key->node_ctas = cap;
    }
    TallyPeer P = key->peer;
    if (!collective || P.world <= 1) { P.world = 1; P.rank = 0; }
    else { key->peer.epoch += 1; P.epoch = key->peer.epoch; }
    return with_eng<View, C, 0, 1, 4>(tally_eng(key), [&](auto e) {
        return launch<View<C, e>>(k_tally<C, e>, ctas, st, key->dev, d_c, count, d_out, key->d_nodes, key->d_node_cnt, P);
    });
}


// ---- witness engine: per-key constants and launcher ------------------------------------------------------

template <class C>
static cudaError_t witness_prepare_cfg(Block28Key* key, u64* d_gchain, bool gchain_ready, cudaStream_t st) {
    const BigInt& n = key->n;
    BigInt n2 = BigInt::mul(n, n);
    int sh = C::KN - (int)n2.bits();
    if (sh & 1) sh -= 1;                                   // chain values carry 2^(sh/2)
    BigInt Nt = BigInt::shl(n2, sh);
    std::vector<int> e_ntu(C::ENTRY4 * 4, 0), e_one;
    to_entry<C>(BigInt::pow2(sh / 2), e_one);
    for (int p = 0; p < C::L; p++) e_ntu[(p / C::BL) * C::CH * 4 + (p % C::BL)] = (int)Nt.bits_at((size_t)W * p, W);
    const KeyConsts<C> kc(Nt, e_ntu);                      // the unsigned digits of Nt in the slot the value engine uses for 2^sh
    CUW(upload(&key->d_wconsts, kc.block, st));
    CUW(upload(&key->d_one_s, e_one, st));
    const int wo = key->dev.words_out, wi = key->dev.words_in;
    std::vector<u64> cpow(2 * (size_t)wo);
    { u64 c = PB200_DIGEST_C; for (size_t j = 0; j < cpow.size(); j++) { cpow[j] = c; c *= PB200_DIGEST_C; } }
    CUW(upload(&key->d_cpow, cpow, st));
    std::vector<u64> nw(wi);
    n.to_u64_le(nw.data(), wi);
    CUW(upload(&key->d_nwords, nw, st));
    CUW(cudaMalloc(&key->d_gtab, (size_t)key->n_bits * C::ENTRY4 * sizeof(int4)));
    // 2^(28(L-2)) / Nt_w from the top 52 bits of Nt_w
    BigInt top = BigInt::shr(Nt, (size_t)W * (C::L - 2) - 20);
    double topd = (double)top.bits_at(32, 32) * 4294967296.0 + (double)top.bits_at(0, 32);
    key->wdev = key->dev; key->wdev.consts = key->d_wconsts; key->wdev.sh = sh;
    WitDev& Wd = key->wit;
    Wd.gtab = key->d_gtab; Wd.one_s = key->d_one_s; Wd.cpow = key->d_cpow; Wd.n_words = key->d_nwords;
    Wd.exp_bits = (int)n.bits(); Wd.sh = sh; Wd.inv = 1048576.0 / topd;
    if constexpr (UL<C, 1, true>::SUPPORTED) {
        // the same step on the tcgen05 phases: constants of the witness modulus + their Toeplitz core-matrix tables
        CUW((upload_u_image<C, 1, true>(&key->d_wuconsts, kc, st)));
        key->wdev.uconsts = key->d_wuconsts;
        key->has_wu = !getenv("PB200_NO_UMMA_WITNESS");
    }
    if (gchain_ready) {        // g-chain records already produced (simple64): only convert them into table entries
        k_wtab<C><<<(key->n_bits + 63) / 64, 64, 0, st>>>(key->d_gwords, wi, d_gchain, wo, (int)key->n_bits, sh / 2, key->d_gtab);
        count_launch();
        CUW(cudaGetLastError());
    } else {                   // produce records and table entries with the witness engine itself
        CUW((with_eng<WView, C, 0, 1>(wit_eng(key), [&](auto e) {
            return launch<WView<C, e>>(k_gchain_w<C, e>, 1, st, key->wdev, key->wit, key->d_gwords, (int)key->n_bits, d_gchain, key->d_gtab);
        })));
    }
    CUW(cudaStreamSynchronize(st));                        // the staging vectors above go out of scope
    key->wit_ready = true;
    return cudaSuccess;
}

template <class C>
static cudaError_t witness_cfg(Block28Key* key, const u64* d_m, const u64* d_r, size_t count, u64* d_c, u64* d_records,
                               const u64* d_offsets, u64* d_digest, cudaStream_t st) {
    size_t ctas = (count + 31) / 32;
    if (ctas > key->wscratch_ctas) {
        if (key->d_wscratch) cudaFree(key->d_wscratch);
        key->d_wscratch = nullptr; key->wscratch_ctas = 0;
        CUW(cudaMalloc(&key->d_wscratch, ctas * 2 * C::VAL4 * sizeof(int4)));
        key->wscratch_ctas = ctas;
    }
    WitIO A;
    A.m = d_m; A.r = d_r; A.count = count; A.c_out = d_c; A.records = d_records; A.offsets = d_offsets; A.digest = d_digest;
    A.scratch = key->d_wscratch;
    return with_eng<WView, C, 0, 1>(wit_eng(key), [&](auto e) { return launch<WView<C, e>>(k_witness<C, e>, ctas, st, key->wdev, key->wit, A); });
}

// Compiled configurations <G warps, BL digits per block>: L = G*BL digits of 28 bits; n^2 must fit KN - 2 bits.
typedef Cfg<4, 19> Cfg1024;    // L =  76: n^2 up to 2102 bits (|n| <= 1024 and the reference's default sizes)
typedef Cfg<8, 19> Cfg2048;    // L = 152: n^2 up to 4230 bits (|n| <= 2048)
typedef Cfg<16, 14> Cfg3072;   // L = 224: n^2 up to 6246 bits (|n| <= 3072)
typedef Cfg<16, 19> Cfg4096;   // L = 304: n^2 up to 8486 bits (|n| <= 4096)

template <class C>
static bool covers(uint32_t n_bits) { return 2 * (size_t)n_bits <= (size_t)C::KN - 2 && n_bits % 8 == 0; }

template <class... Cs> struct CfgList {
    // (G, BL) of the first configuration that covers a key of n_bits; false when none does
    static bool shape(uint32_t n_bits, int* G, int* BL) { return ((covers<Cs>(n_bits) ? (*G = Cs::G, *BL = Cs::BL, true) : false) || ...); }
    // f(C()) for the configuration C of shape (G, BL) (a value of the configuration type as its tag): f's result, `none` when no
    // configuration has that shape
    template <class R, class F> static R with(int G, int BL, R none, F&& f) {
        (void)((G == Cs::G && BL == Cs::BL ? (none = f(Cs()), true) : false) || ...);
        return none;
    }
};
typedef CfgList<Cfg1024, Cfg2048, Cfg3072, Cfg4096> Configs;      // in the order a key size picks them
// f(C()) for the key's configuration C
template <class F> static cudaError_t with_cfg(const Block28Key* key, F&& f) { return Configs::with(key->G, key->BL, cudaErrorInvalidValue, f); }

// layout constants of a block28u variant (host only, no device needed): the CPU model of the tcgen05 data path in
// tests/test_umma_layout.py checks its own derivation against these
template <class C, int LG, bool WIT>
static void ul_fill(int* out) {
    typedef UL<C, LG, WIT> U;
    const int v[20] = {(int)U::SUPPORTED, U::RD, U::TCOLS, U::TN, U::NT_H, U::NT_L, U::FRONT, U::BACK, U::KOFF, U::CHB, U::A_BYTES, U::Z0_H, U::Z0_L,
                       U::NCM_H, U::NCM_L, (int)U::SMEM_BYTES, U::CTAS_PER_SM, U::TMEM_COLS, U::GAP, U::P_BASE_H};
    for (int i = 0; i < 20; i++) out[i] = v[i];
}
template <class C>
static bool ul_cfg(int lg, int wit, int* out) {
    if (lg == 1 && !wit) ul_fill<C, 1, false>(out);
    else if (lg == 1 && wit) ul_fill<C, 1, true>(out);
    else if (lg == 2 && !wit) ul_fill<C, 2, false>(out);
    else return false;
    return true;
}
bool block28_umma_layout(int G, int BL, int lg, int wit, int* out) {
    return Configs::with(G, BL, false, [&](auto c) { return ul_cfg<decltype(c)>(lg, wit, out); });
}

Block28Key* block28_create(const BigInt& n, const BigInt& g, uint32_t n_bits, int device, cudaStream_t st,
                           std::string* why, cudaError_t* cuda_err) {
    *cuda_err = cudaSuccess;
    int G = 0, BL = 0;
    if (!Configs::shape(n_bits, &G, &BL)) {
        if (why) *why = "block28: no compiled configuration covers this key size";
        return nullptr;
    }
    return Configs::with(G, BL, (Block28Key*)nullptr, [&](auto c) { return create_cfg<decltype(c)>(n, g, n_bits, device, st, cuda_err); });
}
void block28_destroy(Block28Key* key) {
    if (!key) return;
    if (key->d_consts) cudaFree(key->d_consts);
    if (key->d_uconsts) cudaFree(key->d_uconsts);
    if (key->d_uconsts2) cudaFree(key->d_uconsts2);
    if (key->d_ops) cudaFree(key->d_ops);
    if (key->d_tg) cudaFree(key->d_tg);
    if (key->d_nentry) cudaFree(key->d_nentry);
    if (key->d_gwords) cudaFree(key->d_gwords);
    if (key->d_scratch) cudaFree(key->d_scratch);
    if (key->d_slot_masks) cudaFree(key->d_slot_masks);
    if (key->d_pow_ops) cudaFree(key->d_pow_ops);
    if (key->d_nodes) cudaFree(key->d_nodes);
    if (key->d_node_cnt) cudaFree(key->d_node_cnt);
    for (int i = 0; i < TALLY_MAXW; i++) if (key->ipc_opened[i]) cudaIpcCloseMemHandle(key->ipc_opened[i]);
    if (key->d_mail) cudaFree(key->d_mail);
    if (key->d_wconsts) cudaFree(key->d_wconsts);
    if (key->d_wuconsts) cudaFree(key->d_wuconsts);
    if (key->d_gtab) cudaFree(key->d_gtab);
    if (key->d_one_s) cudaFree(key->d_one_s);
    if (key->d_cpow) cudaFree(key->d_cpow);
    if (key->d_nwords) cudaFree(key->d_nwords);
    if (key->d_wscratch) cudaFree(key->d_wscratch);
    delete key;
}
const char* block28_name(const Block28Key* key) { return key->name.c_str(); }
// eng: 0 = every phase on the IMAD pipe, 1 = constant-operand phases on mma.sync, 2 = on tcgen05 with 32 ciphertexts per CTA,
// 3 = on tcgen05 with 64 per CTA (each falls back to the next lower one this configuration has), -1 = the fastest available (2)
int block28_set_engine(Block28Key* key, int eng) {
    if (eng < 0) eng = getenv("PB200_NO_UMMA") ? 1 : (getenv("PB200_UMMA_LG2") ? 3 : 2);      // measured: 134.9 k enc/s (2) against 129.9 k (3)
    if (eng == 3 && !key->has_u2) eng = 2;
    if (eng == 2 && !key->has_u) eng = 1;
    key->eng = eng;
    key->name = std::string(eng == 3 ? "block28u2<" : eng == 2 ? "block28u<" : eng == 1 ? "block28t<" : "block28<") + std::to_string(key->G) + "," +
                std::to_string(key->BL) + ">";
    return eng;
}
bool block28_has_engine(const Block28Key* key, int eng) { return eng == 0 || eng == 1 || (eng == 2 && key->has_u) || (eng == 3 && key->has_u2); }
void block28_chain_counts(const Block28Key* key, uint64_t* n_sqr, uint64_t* n_mul) { *n_sqr = key->n_sqr; *n_mul = key->n_mul; }
cudaError_t block28_encrypt(Block28Key* key, const u64* d_m, const u64* d_r, size_t count, u64* d_c, cudaStream_t st) {
    return with_cfg(key, [&](auto c) { return encrypt_cfg<decltype(c)>(key, d_m, d_r, count, d_c, st); });
}
cudaError_t block28_pow_prepare(Block28Key* key, const BigInt& e, cudaStream_t st) {
    std::vector<int2> ops;
    if (key->d_pow_ops) { cudaFree(key->d_pow_ops); key->d_pow_ops = nullptr; }
    CUW(upload_schedule(e, ops, &key->d_pow_ops, &key->pow, st));
    CUW(cudaStreamSynchronize(st));
    key->pow_ready = true;
    return cudaSuccess;
}
cudaError_t block28_pow(Block28Key* key, const u64* d_base, int base_words, size_t count, u64* d_out, cudaStream_t st) {
    if (!count) return cudaSuccess;
    if (!key->pow_ready) return cudaErrorInvalidValue;
    return with_cfg(key, [&](auto c) { return pow_cfg<decltype(c)>(key, d_base, base_words, count, d_out, st); });
}
cudaError_t block28_scalar(Block28Key* key, const u64* d_c, const u64* d_k, uint32_t k_bits, size_t count, u64* d_out, cudaStream_t st) {
    if (!count) return cudaSuccess;
    if (k_bits == 0) return cudaErrorInvalidValue;
    return with_cfg(key, [&](auto c) { return scalar_cfg<decltype(c)>(key, d_c, d_k, k_bits, count, d_out, st); });
}

cudaError_t block28_tally(Block28Key* key, const u64* d_c, size_t count, u64* d_out, cudaStream_t st) {
    return with_cfg(key, [&](auto c) { return tally_cfg<decltype(c)>(key, d_c, count, d_out, false, st); });
}
// collective over the connected peer group: every rank calls it once per tally, in the same order
cudaError_t block28_tally_peer(Block28Key* key, const u64* d_c, size_t count, u64* d_out, cudaStream_t st) {
    return with_cfg(key, [&](auto c) { return tally_cfg<decltype(c)>(key, d_c, count, d_out, true, st); });
}
int block28_peer_world(const Block28Key* key) { return key->peer.world; }

// the peer-visible mailbox of this key (allocated on first use, zeroed)
cudaError_t block28_mailbox(Block28Key* key, u64** d_mail, cudaStream_t st) {
    if (!key->d_mail) {
        CUW(cudaMalloc(&key->d_mail, MAIL_U64 * sizeof(u64)));
        CUW(cudaMemsetAsync(key->d_mail, 0, MAIL_U64 * sizeof(u64), st));
        CUW(cudaStreamSynchronize(st));
    }
    *d_mail = key->d_mail;
    return cudaSuccess;
}
size_t block28_mailbox_bytes() { return MAIL_U64 * sizeof(u64); }
int block28_max_world() { return TALLY_MAXW; }
// mail[i]: rank i's mailbox as addressable from this key's device (mail[rank] must be this key's own); opened[i]: non-null when
// the pointer came from cudaIpcOpenMemHandle and must be closed with the key
cudaError_t block28_tally_peer_connect(Block28Key* key, int rank, int world, u64* const* mail, void* const* opened, int* d_flags) {
    if (world < 1 || world > TALLY_MAXW || rank < 0 || rank >= world) return cudaErrorInvalidValue;
    for (int i = 0; i < TALLY_MAXW; i++) {
        if (key->ipc_opened[i]) { cudaIpcCloseMemHandle(key->ipc_opened[i]); key->ipc_opened[i] = nullptr; }
        key->peer.mail[i] = i < world ? mail[i] : nullptr;
        if (opened && i < world) key->ipc_opened[i] = opened[i];
    }
    key->peer.world = world; key->peer.rank = rank; key->peer.epoch = 0; key->peer.flags = d_flags;
    // a reconnect restarts the epochs: the local mailbox flags must restart with them
    if (key->d_mail) CUW(cudaMemset(key->d_mail + MAIL_FLAG_OFF, 0, 2 * TALLY_MAXW * sizeof(u64)));
    return cudaSuccess;
}


template <class C>
static cudaError_t debug_cfg(Block28Key* key, int eng, const int* h_v, const int* h_y, int reps, int* h_vout, int* h_t, unsigned* h_rows, cudaStream_t st) {
    const size_t vb = (size_t)C::VAL4 * 16;
    int4 *d_v = nullptr, *d_y = nullptr, *d_vout = nullptr, *d_t = nullptr; unsigned* d_rows = nullptr;
    cudaError_t e = cudaSuccess;
    auto run = [&]() -> cudaError_t {
        CUW(cudaMalloc(&d_v, vb)); CUW(cudaMalloc(&d_y, vb)); CUW(cudaMalloc(&d_vout, vb)); CUW(cudaMalloc(&d_t, 2 * vb));
        CUW(cudaMalloc(&d_rows, (size_t)32 * C::L * 4));
        CUW(cudaMemset(d_rows, 0, (size_t)32 * C::L * 4));
        CUW(cudaMemcpy(d_v, h_v, vb, cudaMemcpyHostToDevice));
        if (h_y) CUW(cudaMemcpy(d_y, h_y, vb, cudaMemcpyHostToDevice));
        CUW((with_eng<View, C, 0, 1, 2, 3>(eng, [&](auto e) {
            return launch<View<C, e>>(k_mulmod_dbg<C, e>, 1, st, key->dev, d_v, h_y ? d_y : nullptr, reps, d_vout, h_t ? d_t : nullptr, d_rows);
        })));
        CUW(cudaStreamSynchronize(st));
        if (h_t) CUW(cudaMemcpy(h_t, d_t, 2 * vb, cudaMemcpyDeviceToHost));
        else {
            CUW(cudaMemcpy(h_vout, d_vout, vb, cudaMemcpyDeviceToHost));
            if (h_rows) CUW(cudaMemcpy(h_rows, d_rows, (size_t)32 * C::L * 4, cudaMemcpyDeviceToHost));
        }
        return cudaSuccess;
    };
    e = run();
    cudaFree(d_v); cudaFree(d_y); cudaFree(d_vout); cudaFree(d_t); cudaFree(d_rows);
    return e;
}
// eng: 0 block28, 1 block28t, 2 block28u.  h_t non-null: phase A only, the 2L-digit product; else `reps` multiplications, V and q-hat rows
cudaError_t block28_debug_mulmod(Block28Key* key, int eng, const int* h_v, const int* h_y, int reps, int* h_vout, int* h_t, unsigned* h_rows,
                                 cudaStream_t st) {
    return with_cfg(key, [&](auto c) { return debug_cfg<decltype(c)>(key, eng, h_v, h_y, reps, h_vout, h_t, h_rows, st); });
}
void block28_shape(const Block28Key* key, int* G, int* BL) { *G = key->G; *BL = key->BL; }


// eng 1 / 2 / 3; h_cyc: 3 * ctas values
cudaError_t block28_debug_time(Block28Key* key, int eng, const int* h_v, int ctas, int reps, int stagger, long long* h_cyc, cudaStream_t st) {
    typedef Cfg2048 C;
    if (key->G != C::G || key->BL != C::BL) return cudaErrorInvalidValue;
    const size_t vb = (size_t)C::VAL4 * 16;
    int4* d_v = nullptr; long long* d_cyc = nullptr; unsigned* d_cnt = nullptr;
    auto run = [&]() -> cudaError_t {
        CUW(cudaMalloc(&d_v, vb)); CUW(cudaMalloc(&d_cyc, (size_t)ctas * 3 * sizeof(long long)));
        CUW(cudaMalloc(&d_cnt, 1024 * sizeof(unsigned))); CUW(cudaMemset(d_cnt, 0, 1024 * sizeof(unsigned)));
        CUW(cudaMemcpy(d_v, h_v, vb, cudaMemcpyHostToDevice));
        CUW((with_eng<View, C, 1, 2, 3>(eng, [&](auto e) {
            return launch<View<C, e>>(k_mulmod_time<C, e>, ctas, st, key->dev, d_v, reps, stagger, d_cyc, d_cnt);
        })));
        CUW(cudaStreamSynchronize(st));
        CUW(cudaMemcpy(h_cyc, d_cyc, (size_t)ctas * 3 * sizeof(long long), cudaMemcpyDeviceToHost));
        return cudaSuccess;
    };
    cudaError_t e = run();
    cudaFree(d_v); cudaFree(d_cyc); cudaFree(d_cnt);
    return e;
}

template <class C>
static cudaError_t add_cfg(Block28Key* key, const u64* d_c1, const u64* d_c2, int c_words, size_t count, u64* d_out, u64* d_q,
                           int* d_flags, cudaStream_t st) {
    size_t ctas = (count + 31) / 32, cap = (size_t)C::CTAS_PER_SM * key->sms;
    if (ctas > cap) ctas = cap;
    return with_eng<WView, C, 0, 1>(wit_eng(key), [&](auto e) {
        return launch<WView<C, e>>(k_add_w<C, e>, ctas, st, key->wdev, key->wit, d_c1, d_c2, c_words, count, d_out, d_q, d_flags);
    });
}

// The witness engine needs canonical chain values below n^2 from the first step on: n must fill its declared width
// (then g, r < 2^n_bits <= 2n <= n^2).  Other keys keep the simple64 witness path.
bool block28_witness_supported(const Block28Key* key) { return key->eng >= 1 && key->n.bits() == key->n_bits && key->n_bits >= 8; }
cudaError_t block28_witness_prepare(Block28Key* key, u64* d_gchain, bool gchain_ready, cudaStream_t st) {
    if (key->wit_ready) return cudaSuccess;
    try {
        return with_cfg(key, [&](auto c) { return witness_prepare_cfg<decltype(c)>(key, d_gchain, gchain_ready, st); });
    } catch (const std::exception&) { return cudaErrorInvalidValue; }
}
cudaError_t block28_witness(Block28Key* key, const u64* d_m, const u64* d_r, size_t count, u64* d_c, u64* d_records,
                            const u64* d_offsets, u64* d_digest, cudaStream_t st) {
    if (!count) return cudaSuccess;
    return with_cfg(key, [&](auto c) { return witness_cfg<decltype(c)>(key, d_m, d_r, count, d_c, d_records, d_offsets, d_digest, st); });
}

cudaError_t block28_add(Block28Key* key, const u64* d_c1, const u64* d_c2, int c_words, size_t count, u64* d_out, u64* d_q,
                        int* d_flags, cudaStream_t st) {
    if (!count) return cudaSuccess;
    return with_cfg(key, [&](auto c) { return add_cfg<decltype(c)>(key, d_c1, d_c2, c_words, count, d_out, d_q, d_flags, st); });
}

// ---- running-tally trace: driver (DESIGN.md §9c) ----------------------------------------------------------------------------------
// one wave of the trace's scan kernels: 32 lanes x the CTAs per SM of the key's tally engine (View<C, 4> on tcgen05) x SMs
size_t block28_lanes(const Block28Key* key) {
    return Configs::with(key->G, key->BL, (size_t)0, [&](auto c) {
        typedef decltype(c) C;
        return (size_t)(tally_eng(key) == 4 ? View<C, 4>::PER_SM : View<C, 0>::PER_SM) * key->sms * 32;
    });
}
// one buffer of lazy values per level below the top (the totals of its chunks, then in place their carries)
template <class C>
static size_t trace_scan_bytes_cfg(const TracePlan& P, size_t chains) {
    size_t b = 0;
    for (size_t l = 0; l + 1 < P.n.size(); l++) b += P.n[l + 1] * chains * C::ENTRY4 * sizeof(int4);
    return b;
}
size_t block28_trace_scan_bytes(const Block28Key* key, const TracePlan& P, size_t chains) {
    return Configs::with(key->G, key->BL, (size_t)0, [&](auto c) { return trace_scan_bytes_cfg<decltype(c)>(P, chains); });
}
template <class C, int ENG>
static cudaError_t trace_scan_cfg(Block28Key* key, const TracePlan& P, const u64* d_init, const u64* d_c, size_t chains,
                                  unsigned char* tmp, u64* d_carry, cudaStream_t st) {
    typedef View<C, ENG> V;
    const size_t L = P.n.size() - 1;                                 // levels below the top
    std::vector<int4*> buf(L);
    for (size_t l = 0, o = 0; l < L; l++) { buf[l] = (int4*)(tmp + o); o += P.n[l + 1] * chains * C::ENTRY4 * sizeof(int4); }
    for (size_t l = 0; l < L; l++)                                   // phase 1: the totals of every chunk, level after level
        CUW(launch<V>(k_trace_reduce<C, ENG>, cdiv(P.n[l + 1] * chains, 32), st, key->dev, l ? (const u64*)nullptr : d_c,
                      l ? (const int4*)buf[l - 1] : (const int4*)nullptr, P.n[l], chains, P.s[l], buf[l]));
    for (size_t l = L; l >= 1; l--)                                  // phase 2: the carries of level l - 1 from the top down
        CUW(launch<V>(k_trace_apply<C, ENG>, cdiv(cdiv(P.n[l], P.s[l]) * chains, 32), st, key->dev, d_init,
                      l == L ? (const int4*)nullptr : (const int4*)buf[l], buf[l - 1], P.n[l], chains, P.s[l]));
    return launch<V>(k_lazy_canon<C, ENG>, cdiv(P.n[1] * chains, 32), st, key->dev, (const int4*)buf[0], P.n[1] * chains, d_carry);
}
cudaError_t block28_trace_scan(Block28Key* key, const TracePlan& P, const u64* d_init, const u64* d_c, size_t chains, void* tmp, u64* d_carry,
                               cudaStream_t st) {
    if (P.n.size() < 2) return cudaSuccess;
    return with_cfg(key, [&](auto c) {
        typedef decltype(c) C;
        return with_eng<View, C, 0, 1, 4>(tally_eng(key), [&](auto e) {
            return trace_scan_cfg<C, e>(key, P, d_init, d_c, chains, (unsigned char*)tmp, d_carry, st);
        });
    });
}
cudaError_t block28_trace_chain(Block28Key* key, const u64* d_init, const u64* d_c, const u64* d_carry, size_t count, size_t chains, size_t s,
                                u64* d_acc, u64* d_q, int* d_flags, cudaStream_t st) {
    return with_cfg(key, [&](auto c) {
        typedef decltype(c) C;
        return with_eng<WView, C, 0, 1>(wit_eng(key), [&](auto e) {
            return launch<WView<C, e>>(k_trace_w<C, e>, cdiv(cdiv(count, s) * chains, 32), st, key->wdev, key->wit, d_init, d_c, d_carry,
                                       count, chains, s, d_acc, d_q, d_flags);
        });
    });
}

// ---- matvec: planner and driver (DESIGN.md §9b) ---------------------------------------------------------------------------------
// multiplications of k_scalar's chain for k_bits-bit scalars (table, windows, finalize)
static uint64_t scalar_chain(uint32_t k_bits) { return scalar_cost(k_bits, scalar_window(k_bits)) + 1; }
// slice length of a k_bucket_fold launch over n entries: one wave of lanes, at least 8 entries (the carry list shrinks 4x per level)
static int fold_ls(size_t n, size_t lanes) { const size_t l = cdiv(n, lanes); return (int)(l < 8 ? 8 : l); }
// mulmods (upper bound) and sequential chain of the fold of n entries, every carry level included
static void fold_cost(size_t n, size_t lanes, uint64_t* work, uint64_t* chain) {
    for (;;) {
        const int ls = fold_ls(n, lanes);
        const size_t l = cdiv(n, (size_t)ls);
        *work += (uint64_t)l * ls + l; *chain += (uint64_t)ls + 1;
        if (l <= 1) break;
        n = 2 * l;
    }
}
static size_t fold_lanes0(size_t n, size_t lanes) { return cdiv(n, (size_t)fold_ls(n, lanes)); }

struct MvShape { size_t e_bytes = 0, wo = 0, lanes = 0; bool ok = false; };
template <class C>
static MvShape mv_shape_cfg(uint32_t n_bits, int sms) {
    MvShape s; s.e_bytes = (size_t)C::ENTRY4 * 16; s.wo = (2 * (size_t)n_bits + 63) / 64; s.lanes = (size_t)sms * C::CTAS_PER_SM * 32; s.ok = true;
    return s;
}
static MvShape mv_shape(uint32_t n_bits, int sms) {
    int G = 0, BL = 0;
    Configs::shape(n_bits, &G, &BL);
    return Configs::with(G, BL, MvShape(), [&](auto c) { return mv_shape_cfg<decltype(c)>(n_bits, sms); });
}

// the bucket method's arena, carved in this order (every piece 256-byte aligned)
struct MvLayout {
    size_t hist, keys, idx, skeys, sidx, ckeys[2], cvals[2], cnt, buckets, vals, aseg, scal, rscr, wlazy, x, nprime, total;
};
static MvLayout mv_layout(const MatvecPlan& P, const MvShape& S) {
    const size_t sp = P.rb * P.nsign * P.jg, nkeys = sp << P.c, ents = P.rb * P.jg * P.nc, units = sp * P.nseg;
    const size_t sents = std::max(sp * (2 * (size_t)P.nseg + 1), 2 * P.rb);
    const size_t carry = 2 * std::max(fold_lanes0(ents, S.lanes), fold_lanes0(sents, S.lanes));
    const size_t vb = S.wo * 8;
    MvLayout L; size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o += (bytes + 255) & ~(size_t)255; return at; };
    L.hist = take(nkeys * 4); L.keys = take(ents * 4); L.idx = take(ents * 4); L.skeys = take(sents * 4); L.sidx = take(sents * 4);
    for (int i = 0; i < 2; i++) { L.ckeys[i] = take(carry * 4); L.cvals[i] = take(carry * S.e_bytes); }
    L.cnt = take(64 * 4); L.buckets = take(nkeys * S.e_bytes); L.vals = take((2 * units + sp) * vb); L.aseg = take(units * vb);
    L.scal = take(units * 8); L.rscr = take(cdiv(units, 32) * 64 * S.e_bytes); L.wlazy = take(std::max(sp, P.rb) * S.e_bytes);
    L.x = take(P.rb * P.nsign * vb); L.nprime = take(P.rb * vb);
    L.total = o;
    return L;
}

size_t matvec_budget(uint32_t n_bits) { return ((size_t)3 << 18) * 8 * ((2 * (size_t)n_bits + 63) / 64); }

MatvecPlan matvec_plan(uint32_t n_bits, int sms, size_t rows, size_t count, uint32_t k_bits, bool has_neg, bool bucket_ok) {
    const MvShape S = mv_shape(n_bits, sms > 0 ? sms : 1);
    const size_t budget = matvec_budget(n_bits), wo = (2 * (size_t)n_bits + 63) / 64, kw = (k_bits + 63) / 64, kwn = (n_bits + 63) / 64;
    const size_t lanes = S.ok ? S.lanes : (size_t)(sms > 0 ? sms : 1) * 64;
    const int nsign = has_neg ? 2 : 1;
    const char* force = getenv("PB200_MATVEC_METHOD");
    size_t pe = (size_t)1 << 24;
    if (const char* e = getenv("PB200_MATVEC_PASS_ENTRIES")) { const long long v = atoll(e); if (v >= 1 && (size_t)v < pe) pe = (size_t)v; }
    auto waves = [&](size_t u) -> uint64_t { return cdiv(u ? u : 1, lanes); };
    if (!rows || !count) { MatvecPlan z; z.nsign = nsign; return z; }                    // nothing to multiply: every row is 1
    // chain: per row and sign, chunks of 2^18 ciphertexts (masked scalars, scalar products, tally); sign step per block of rows
    MatvecPlan ch;
    {
        const size_t chunk = std::min(count, (size_t)1 << 18), chunks = cdiv(count, (size_t)1 << 18), rbc = std::min(rows, (size_t)4096);
        const uint64_t sk = scalar_chain(k_bits), sn = scalar_chain(n_bits);
        ch.method = 0; ch.nsign = nsign; ch.rb = rbc; ch.nc = chunk; ch.passes = rows * nsign * chunks;
        ch.acc = (uint64_t)rows * nsign * count * sk;
        ch.red = (uint64_t)rows * nsign * (count + 2 * chunks);
        ch.sign = has_neg ? (uint64_t)rows * (sn + 2) : 0;
        ch.chain = ch.passes * (sk + 8) + (has_neg ? cdiv(rows, rbc) * sn + rows * 8 : 0);
        ch.bytes = (chunk * (kw + wo) + (4 + 2 * rbc) * wo + rbc * kwn) * 8;
        if (!S.ok || !bucket_ok || (force && !strcmp(force, "chain"))) return ch;
    }
    const uint64_t slots_chain = (uint64_t)rows * nsign * cdiv(count, (size_t)1 << 18) * (waves(std::min(count, (size_t)1 << 18)) * (scalar_chain(k_bits) + 1) + 8) +
                                 (has_neg ? cdiv(rows, ch.rb) * waves(ch.rb) * scalar_chain(n_bits) + rows * 8 : 0);
    MatvecPlan best; uint64_t best_slots = ~0ull;
    for (int c = 1; c <= 16 && c <= (int)k_bits; c++) {
        MatvecPlan p; p.method = 1; p.c = c; p.J = (int)cdiv(k_bits, c); p.nsign = nsign;
        p.nc = std::min(count, pe);
        const size_t q = std::max((size_t)1, pe / p.nc);
        p.jg = std::min((size_t)p.J, q); p.rb = std::min(rows, std::max((size_t)1, q / p.jg));
        uint64_t slots = 0; bool fit = false;
        for (;;) {
            // segment length: one wave of reduce lanes where possible, fewest slots
            const size_t sp = p.rb * nsign * p.jg, nb = ((size_t)1 << c) - 1;
            uint64_t rs_best = ~0ull;
            for (size_t ls = 1; ls <= nb; ls <<= 1) {
                const size_t nseg = cdiv(nb, ls), units = sp * nseg;
                uint64_t w = 0, fch = 0; fold_cost(sp * (2 * nseg + 1), lanes, &w, &fch);
                const uint64_t rs = waves(units) * (2 * ls + 2 + scalar_chain(c)) + fch;
                if (rs < rs_best) { rs_best = rs; p.lseg = (int)ls; p.nseg = (int)nseg; }
            }
            p.bytes = mv_layout(p, S).total + (has_neg ? p.rb * kwn * 8 : 0);              // + the sign step's copies of n - 1
            if (p.bytes <= budget) { fit = true; break; }
            if (p.rb > 1) p.rb = cdiv(p.rb, 2);
            else if (p.jg > 1) p.jg = cdiv(p.jg, 2);
            else if (p.nc > 1) p.nc = cdiv(p.nc, 2);
            else break;
        }
        if (!fit) continue;
        const size_t sp = p.rb * nsign * p.jg, units = sp * p.nseg, blocks = cdiv(rows, p.rb), groups = cdiv(p.J, p.jg), chunks = cdiv(count, p.nc);
        p.passes = blocks * groups * chunks;
        uint64_t fw = 0, fc = 0, sw = 0, sc = 0, cw = 0, cc = 0;
        fold_cost(p.rb * p.jg * p.nc, lanes, &fw, &fc);
        fold_cost(sp * (2 * (size_t)p.nseg + 1), lanes, &sw, &sc);
        fold_cost(2 * p.rb, lanes, &cw, &cc);
        const uint64_t sn = scalar_chain(n_bits), s_c = scalar_chain(c);
        p.acc = p.passes * fw;
        p.red = p.passes * ((uint64_t)units * (2 * p.lseg + 2) + units * s_c + sw + sp);
        p.horner = (uint64_t)blocks * groups * p.rb * nsign * p.jg * (c + 1) + blocks * p.rb * nsign;
        p.sign = has_neg ? (uint64_t)blocks * p.rb * sn + blocks * cw : 0;
        const uint64_t pass_chain = fc + 2 * p.lseg + 2 + s_c + sc + 1, group_chain = (uint64_t)p.jg * (c + 1) + 1;
        p.chain = p.passes * pass_chain + blocks * groups * group_chain + (has_neg ? blocks * (sn + cc) : 0);
        slots = p.passes * (fc + waves(units) * (2 * p.lseg + 2 + s_c) + sc + 1) +
                blocks * groups * waves(p.rb * nsign) * group_chain + (has_neg ? blocks * (waves(p.rb) * sn + cc) : 0);
        if (slots < best_slots) { best_slots = slots; best = p; }
    }
    if (!best.method) return ch;
    if (force && !strcmp(force, "bucket")) return best;
    return best_slots < slots_chain ? best : ch;
}

// k_bucket_fold over an entry list, level after level until the carry list is empty.  n_dev: the entry count is *cnt (device);
// else n_ub exactly.  Level l reads its count from cnt[l] and writes the next one to cnt[l + 1].
template <class C, int ENG>
static cudaError_t mv_fold(Block28Key* key, const unsigned* keys, const unsigned* idx, const u64* src, bool n_dev, size_t n_ub,
                           int4* out, const MvLayout& L, unsigned char* A, size_t lanes, cudaStream_t st) {
    typedef View<C, ENG> V;
    unsigned* cnt = (unsigned*)(A + L.cnt);
    int lv = 0, ls = fold_ls(n_ub, lanes);
    size_t ln = cdiv(n_ub, (size_t)ls);
    CUW(launch<V>(k_bucket_fold<C, ENG>, cdiv(ln, 32), st, key->dev, keys, idx, src, key->dev.words_out, (const int4*)nullptr,
                      n_dev ? cnt : nullptr, n_ub, ls, out, (unsigned*)(A + L.ckeys[0]), (int4*)(A + L.cvals[0]), cnt + 1));
    while (ln > 1) {
        const size_t n = 2 * ln;
        ls = fold_ls(n, lanes); ln = cdiv(n, (size_t)ls); lv++;
        const int i = (lv - 1) & 1;
        CUW(launch<V>(k_bucket_fold<C, ENG>, cdiv(ln, 32), st, key->dev, (const unsigned*)(A + L.ckeys[i]), (const unsigned*)nullptr,
                      (const u64*)nullptr, 0, (const int4*)(A + L.cvals[i]), cnt + lv, n, ls, out, (unsigned*)(A + L.ckeys[i ^ 1]),
                      (int4*)(A + L.cvals[i ^ 1]), cnt + lv + 1));
        if (lv >= 62) return cudaErrorInvalidValue;
    }
    return cudaSuccess;
}

// ENG: the key's engine as the bucket kernels run it (tally_eng); k_scalar runs the key's own engine
template <class C, int ENG>
static cudaError_t matvec_cfg(Block28Key* key, const MatvecPlan& P, const u64* d_c, size_t count, const u64* d_w, uint32_t k_bits,
                              const uint8_t* d_neg, size_t rows, u64* d_out, unsigned char* A, const u64* d_nm1, cudaStream_t st) {
    typedef View<C, ENG> V;
    CUW(ensure_slots<C>(key, st));
    const MvShape S = mv_shape_cfg<C>(key->n_bits, key->sms);
    const MvLayout L = mv_layout(P, S);
    const int c = P.c, kw = (int)((k_bits + 63) / 64), wo = key->dev.words_out;
    const size_t vb = (size_t)wo;                                   // u64 per canonical value
    u64* vals = (u64*)(A + L.vals); u64* x = (u64*)(A + L.x);
    for (size_t r0 = 0; r0 < rows; r0 += P.rb) {
        const size_t rb = std::min(P.rb, rows - r0), xs = rb * P.nsign;
        k_mv_one_words<<<(unsigned)cdiv(xs * wo, 256), 256, 0, st>>>(x, xs, wo); count_launch();
        for (size_t g = cdiv(P.J, P.jg); g-- > 0;) {
            const int j0 = (int)(g * P.jg), jg = (int)std::min(P.jg, (size_t)P.J - j0);
            const size_t sp = xs * jg, units = sp * P.nseg, nkeys = sp << c;
            u64* w_acc = vals + 2 * units * vb;                                              // the W block of [T | A' | W]
            k_mv_one_words<<<(unsigned)cdiv(sp * wo, 256), 256, 0, st>>>(w_acc, sp, wo); count_launch();
            for (size_t i0 = 0; i0 < count; i0 += P.nc) {
                const size_t nc = std::min(P.nc, count - i0), th = rb * nc;
                unsigned* hist = (unsigned*)(A + L.hist);
                CUW(cudaMemsetAsync(hist, 0, nkeys * 4, st));
                k_mv_digits<<<(unsigned)cdiv(th, 256), 256, 0, st>>>(d_w, d_neg, count, kw, r0, rb, i0, nc, c, j0, jg, hist, nullptr, nullptr);
                k_mv_scan<<<1, 1024, 0, st>>>(hist, nkeys, (unsigned*)(A + L.cnt));
                k_mv_digits<<<(unsigned)cdiv(th, 256), 256, 0, st>>>(d_w, d_neg, count, kw, r0, rb, i0, nc, c, j0, jg, hist,
                                                                    (unsigned*)(A + L.keys), (unsigned*)(A + L.idx));
                k_mv_one_lazy<<<(unsigned)cdiv(nkeys * C::ENTRY4, 256), 256, 0, st>>>((int4*)(A + L.buckets), nkeys, C::ENTRY4);
                count_launch(4);
                CUW(cudaGetLastError());
                CUW((mv_fold<C, ENG>(key, (const unsigned*)(A + L.keys), (const unsigned*)(A + L.idx), d_c + i0 * wo, true, rb * jg * nc,
                                     (int4*)(A + L.buckets), L, A, S.lanes, st)));
                CUW(launch<V>(k_bucket_reduce<C, ENG>, cdiv(units, 32), st, key->dev, (const int4*)(A + L.buckets), c, P.nseg, P.lseg, units, vals,
                              (u64*)(A + L.aseg), (u64*)(A + L.scal), (int4*)(A + L.rscr)));
                CUW(scalar_cfg<C>(key, (const u64*)(A + L.aseg), (const u64*)(A + L.scal), (uint32_t)c, units, vals + units * vb, st));
                const int per = 2 * P.nseg + 1;
                k_mv_block_entries<<<(unsigned)cdiv(sp * per, 256), 256, 0, st>>>((unsigned*)(A + L.skeys), (unsigned*)(A + L.sidx), sp, P.nseg, per);
                count_launch(); CUW(cudaGetLastError());
                CUW((mv_fold<C, ENG>(key, (const unsigned*)(A + L.skeys), (const unsigned*)(A + L.sidx), vals, false, sp * per,
                                     (int4*)(A + L.wlazy), L, A, S.lanes, st)));
                CUW(launch<V>(k_lazy_canon<C, ENG>, cdiv(sp, 32), st, key->dev, (const int4*)(A + L.wlazy), sp, w_acc));
            }
            CUW(launch<V>(k_horner<C, ENG>, cdiv(xs, 32), st, key->dev, x, (const u64*)w_acc, xs, jg, c));
        }
        u64* out = d_out + r0 * vb;
        if (P.nsign == 1) { CUW(cudaMemcpyAsync(out, x, rb * vb * 8, cudaMemcpyDeviceToDevice, st)); continue; }
        // sign step: N^(n-1) next to P, then the fold of the pairs (P_r, N_r^(n-1))
        u64* np = (u64*)(A + L.nprime);
        CUW(scalar_cfg<C>(key, x + rb * vb, d_nm1, key->n_bits, rb, np, st));
        CUW(cudaMemcpyAsync(x + rb * vb, np, rb * vb * 8, cudaMemcpyDeviceToDevice, st));
        k_mv_block_entries<<<(unsigned)cdiv(2 * rb, 256), 256, 0, st>>>((unsigned*)(A + L.skeys), (unsigned*)(A + L.sidx), rb, 1, 2);
        count_launch(); CUW(cudaGetLastError());
        CUW((mv_fold<C, ENG>(key, (const unsigned*)(A + L.skeys), (const unsigned*)(A + L.sidx), x, false, 2 * rb, (int4*)(A + L.wlazy), L, A,
                             S.lanes, st)));
        CUW(launch<V>(k_lazy_canon<C, ENG>, cdiv(rb, 32), st, key->dev, (const int4*)(A + L.wlazy), rb, out));
    }
    return cudaSuccess;
}

cudaError_t block28_matvec(Block28Key* key, const MatvecPlan& P, const u64* d_c, size_t count, const u64* d_w, uint32_t k_bits, const uint8_t* d_neg,
                           size_t rows, u64* d_out, void* arena, const u64* d_nm1, cudaStream_t st) {
    if (!rows || !count || P.method != 1) return cudaErrorInvalidValue;
    unsigned char* A = (unsigned char*)arena;
    return with_cfg(key, [&](auto c) {
        typedef decltype(c) C;
        return with_eng<View, C, 0, 1, 4>(tally_eng(key), [&](auto e) {
            return matvec_cfg<C, e>(key, P, d_c, count, d_w, k_bits, d_neg, rows, d_out, A, d_nm1, st);
        });
    });
}
cudaError_t matvec_mask(const u64* d_w, const uint8_t* d_neg, size_t n, int kw, int sgn, u64* d_out, cudaStream_t st) {
    if (!n) return cudaSuccess;
    k_mv_mask<<<(unsigned)cdiv(n * kw, 256), 256, 0, st>>>(d_w, d_neg, n, kw, sgn, d_out); count_launch();
    return cudaGetLastError();
}
cudaError_t matvec_ones(u64* d_out, size_t n, int wo, cudaStream_t st) {
    if (!n) return cudaSuccess;
    k_mv_one_words<<<(unsigned)cdiv(n * wo, 256), 256, 0, st>>>(d_out, n, wo); count_launch();
    return cudaGetLastError();
}

}  // namespace pb200
