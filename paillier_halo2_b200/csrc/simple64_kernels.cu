// simple64_kernels.cu — kernels of the simple64 engine (see simple64.cuh) + the limb repack kernel.
#include "engine.hpp"

namespace pb200 {

std::atomic<uint64_t> g_kernel_launches{0};

__device__ __forceinline__ void load_ext(u64* dst, const u64* src, int nsrc, int k) {
    for (int i = 0; i < k; i++) dst[i] = i < nsrc ? src[i] : 0;   // extend_limbs (src/paillier.rs:49,53,79-80)
}
__device__ __forceinline__ void set_one(u64* dst, int k) { dst[0] = 1; for (int i = 1; i < k; i++) dst[i] = 0; }
__device__ __forceinline__ int bit_at(const u64* x, int i) { return (int)((x[i >> 6] >> (i & 63)) & 1); }
__device__ __forceinline__ int bit_length(const u64* x, int n) {
    for (int i = n - 1; i >= 0; i--) if (x[i]) return 64 * i + 64 - __clzll((long long)x[i]);
    return 0;
}

// per-key squaring chain of g: record i = (q, rem) of (g^(2^i))^2  (pow_mod_fixed_exp's `squared`)
__global__ void k_simple_gchain(const SimpleConsts* __restrict__ K, u64* __restrict__ gchain, int n_bits) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int k = K->k;
    u64 cur[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK], rem[PB200_SIMPLE_MAXK];
    load_ext(cur, K->g, K->kin, k);
    for (int i = 0; i < n_bits; i++) {
        mulmod_simple(K, q, rem, cur, cur);
        u64* rec = gchain + (size_t)i * 2 * k;
        for (int j = 0; j < k; j++) { rec[j] = q[j]; rec[k + j] = rem[j]; cur[j] = rem[j]; }
    }
}

// one unit per thread, the reference's chain (src/paillier.rs:51,55,57 -> SURVEY.md A.5)
__global__ void __launch_bounds__(32) k_simple_encrypt(const SimpleConsts* __restrict__ K, const u64* __restrict__ gchain,
                                                       const u64* __restrict__ m, const u64* __restrict__ r, size_t count,
                                                       u64* __restrict__ c_out, u64* __restrict__ records,
                                                       const u64* __restrict__ offsets, u64* __restrict__ digest, int* flags) {
    size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= count) return;
    const int k = K->k, kin = K->kin;
    RecordSink sink; sink.k = k; sink.digest = PB200_DIGEST_INIT;
    sink.rec = records ? records + offsets[u] * 2 * (size_t)k : nullptr;
    u64 acc[PB200_SIMPLE_MAXK], cur[PB200_SIMPLE_MAXK], sq[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK], gm[PB200_SIMPLE_MAXK];
    int bad = 0;
    // g-chain: acc *= g^(2^i) for the set bits of m; the squarings are per-key (gchain)
    const u64* mu_ = m + u * kin;
    set_one(acc, k);
    int mbits = bit_length(mu_, kin);
    if (mbits > K->n_bits) { bad = 1; mbits = K->n_bits; }
    for (int i = 0; i < mbits; i++) {
        if (!bit_at(mu_, i)) continue;
        if (i == 0) load_ext(cur, K->g, kin, k);
        else { const u64* rec = gchain + (size_t)(i - 1) * 2 * k + k; for (int j = 0; j < k; j++) cur[j] = rec[j]; }
        bad |= mulmod_simple(K, q, gm, acc, cur);
        sink.emit(q, gm);
        for (int j = 0; j < k; j++) acc[j] = gm[j];
    }
    for (int j = 0; j < k; j++) gm[j] = acc[j];
    // r-chain: full LSB-first chain, exponent n
    set_one(acc, k);
    load_ext(sq, r + u * kin, kin, k);
    if (bit_length(r + u * kin, kin) > K->n_bits) bad = 1;
    for (int i = 0; i < K->exp_bits; i++) {
        for (int j = 0; j < k; j++) cur[j] = sq[j];
        bad |= mulmod_simple(K, q, sq, cur, cur);
        sink.emit(q, sq);
        if (!bit_at(K->n, i)) continue;
        u64 t[PB200_SIMPLE_MAXK];
        bad |= mulmod_simple(K, q, t, acc, cur);
        sink.emit(q, t);
        for (int j = 0; j < k; j++) acc[j] = t[j];
    }
    // final mul_mod(gm, rn)
    bad |= mulmod_simple(K, q, cur, gm, acc);
    sink.emit(q, cur);
    if (c_out) for (int j = 0; j < k; j++) c_out[u * k + j] = cur[j];
    if (digest) digest[u] = sink.digest;
    if (bad) atomicOr(flags, 1);
}

__global__ void __launch_bounds__(32) k_simple_add(const SimpleConsts* __restrict__ K, const u64* __restrict__ c1,
                                                   const u64* __restrict__ c2, int c_words, size_t count,
                                                   u64* __restrict__ out, u64* __restrict__ q_out, int* flags) {
    size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= count) return;
    const int k = K->k;
    u64 a[PB200_SIMPLE_MAXK], b[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK], rem[PB200_SIMPLE_MAXK];
    load_ext(a, c1 + u * c_words, c_words, k);
    load_ext(b, c2 + u * c_words, c_words, k);
    int bad = mulmod_simple(K, q, rem, a, b);
    for (int j = 0; j < k; j++) out[u * k + j] = rem[j];
    if (q_out) for (int j = 0; j < k; j++) q_out[u * k + j] = q[j];
    if (bad) atomicOr(flags, 1);
}

// each thread folds a strided subset: partial[t] = prod_{i = t mod T} c_i mod n2 (inputs reduced first)
__global__ void __launch_bounds__(32) k_simple_tally_partial(const SimpleConsts* __restrict__ K, const u64* __restrict__ c,
                                                             size_t count, u64* __restrict__ partial, int T, int* flags) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int k = K->k;
    u64 acc[PB200_SIMPLE_MAXK], x[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK], rem[PB200_SIMPLE_MAXK];
    set_one(acc, k);
    int bad = 0;
    for (size_t i = t; i < count; i += T) {
        for (int j = 0; j < k; j++) x[j] = c[i * k + j];
        bad |= mulmod_simple(K, q, rem, acc, x);
        for (int j = 0; j < k; j++) acc[j] = rem[j];
    }
    for (int j = 0; j < k; j++) partial[(size_t)t * k + j] = acc[j];
    if (bad) atomicOr(flags, 1);
}
__global__ void k_simple_tally_final(const SimpleConsts* __restrict__ K, const u64* __restrict__ partial, int T,
                                     u64* __restrict__ out, int* flags) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int k = K->k;
    u64 acc[PB200_SIMPLE_MAXK], x[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK], rem[PB200_SIMPLE_MAXK];
    set_one(acc, k);
    // reduce 1 mod n2 (n = 1 gives n2 = 1 and an empty product of 0)
    for (int j = 0; j < k; j++) x[j] = acc[j];
    int bad = mulmod_simple(K, q, rem, acc, x);
    for (int j = 0; j < k; j++) acc[j] = rem[j];
    for (int t = 0; t < T; t++) {
        for (int j = 0; j < k; j++) x[j] = partial[(size_t)t * k + j];
        bad |= mulmod_simple(K, q, rem, acc, x);
        for (int j = 0; j < k; j++) acc[j] = rem[j];
    }
    for (int j = 0; j < k; j++) out[j] = acc[j];
    if (bad) atomicOr(flags, 1);
}

// ---- decryption (SURVEY.md 8f-4; the reference's README.md:5-22 states it, its code never implements it) ------------------------
// x = base^e mod n^2, LSB-first square-and-multiply, exponent words from device memory: the always-available pow for keys the
// block engine does not serve.  e_stride = 0: one exponent for all units (decryption); else unit u's own exponent at u * e_stride
// words, and the base is reduced first (scalar multiplication takes any words_out-word value; squaring an unreduced one would
// overflow the Barrett input)
__global__ void __launch_bounds__(32) k_simple_pow(const SimpleConsts* __restrict__ K, const u64* __restrict__ base, int base_words,
                                                   const u64* __restrict__ e, int e_bits, int e_stride, size_t count, u64* __restrict__ out,
                                                   int* flags) {
    const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= count) return;
    const int k = K->k;
    u64 acc[PB200_SIMPLE_MAXK], sq[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK], t[PB200_SIMPLE_MAXK];
    int bad = 0;
    set_one(acc, k);
    load_ext(sq, base + u * base_words, base_words, k);
    if (e_stride) {
        e += u * (size_t)e_stride;
        bad |= mulmod_simple(K, q, t, sq, acc);
        for (int j = 0; j < k; j++) sq[j] = t[j];
    }
    for (int i = 0; i < e_bits; i++) {
        if (bit_at(e, i)) { bad |= mulmod_simple(K, q, t, acc, sq); for (int j = 0; j < k; j++) acc[j] = t[j]; }
        if (i + 1 < e_bits) { bad |= mulmod_simple(K, q, t, sq, sq); for (int j = 0; j < k; j++) sq[j] = t[j]; }
    }
    if (e_bits == 0) { u64 one[PB200_SIMPLE_MAXK]; set_one(one, k); bad |= mulmod_simple(K, q, t, acc, one); for (int j = 0; j < k; j++) acc[j] = t[j]; }
    for (int j = 0; j < k; j++) out[u * k + j] = acc[j];
    if (bad) atomicOr(flags, 1);
}

// m = L(x) * mu mod n with L(x) = (x - 1) / n (README.md:17-22 of the reference).  Kn: constants of the modulus n (k = words of n),
// its g slot carries mu.  x: 2k words.  Raises flag bit 3 when x is not 1 mod n (not the lambda-th power of a valid ciphertext).
__global__ void __launch_bounds__(32) k_simple_lfunc(const SimpleConsts* __restrict__ Kn, const u64* __restrict__ x, size_t count,
                                                     u64* __restrict__ m_out, int* flags) {
    const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= count) return;
    const int k = Kn->k;
    u64 X[PB200_SIMPLE_MAXK + 1], t[PB200_SIMPLE_MAXK / 2 + 1], rem[PB200_SIMPLE_MAXK / 2 + 1], q[PB200_SIMPLE_MAXK / 2 + 1], m[PB200_SIMPLE_MAXK / 2 + 1];
    u64 borrow = 1;                                       // X = x - 1
    for (int i = 0; i < 2 * k; i++) { const u64 xi = x[u * 2 * k + i]; X[i] = xi - borrow; borrow = xi < borrow; }
    int bad = (int)borrow;                                // x == 0
    bad |= barrett_simple(Kn, t, rem, X);
    for (int i = 0; i < k; i++) bad |= rem[i] != 0;
    mulmod_simple(Kn, q, m, t, Kn->g);
    for (int i = 0; i < k; i++) m_out[u * k + i] = bad ? 0 : m[i];
    if (bad) atomicOr(flags, 8);
}

// ---- running-tally trace (pb200_tally_trace): the three phases of block28_kernels.cu, one thread per chunk, canonical values -------
// totals[u] = product of chunk b of chain j, u = b * chains + j (entries (i, j) at (i * chains + j) * k, any k-word value)
__global__ void __launch_bounds__(32) k_simple_trace_reduce(const SimpleConsts* __restrict__ K, const u64* __restrict__ in, size_t n,
                                                            size_t chains, size_t s, u64* __restrict__ totals) {
    const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= (n + s - 1) / s * chains) return;
    const size_t b = u / chains, j = u - b * chains;
    const int k = K->k;
    u64 acc[PB200_SIMPLE_MAXK], x[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK];
    set_one(acc, k);
    for (size_t i = b * s; i < n && i < (b + 1) * s; i++) {
        for (int w = 0; w < k; w++) x[w] = in[(i * chains + j) * k + w];
        mulmod_simple(K, q, acc, acc, x);                  // acc is canonical: q always fits
    }
    for (int w = 0; w < k; w++) totals[u * k + w] = acc[w];
}
// exclusive prefix products of one level, in place; the carry of chunk b is carry[u], or init_j reduced mod n^2 (carry == null)
__global__ void __launch_bounds__(32) k_simple_trace_apply(const SimpleConsts* __restrict__ K, const u64* __restrict__ init,
                                                           const u64* __restrict__ carry, u64* items, size_t n, size_t chains, size_t s) {
    const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= (n + s - 1) / s * chains) return;
    const size_t b = u / chains, j = u - b * chains;
    const int k = K->k;
    u64 acc[PB200_SIMPLE_MAXK], x[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK];
    if (carry) for (int w = 0; w < k; w++) acc[w] = carry[u * k + w];
    else { set_one(x, k); mulmod_simple(K, q, acc, init + j * k, x); }
    for (size_t i = b * s; i < n && i < (b + 1) * s; i++) {
        u64* e = items + (i * chains + j) * k;
        for (int w = 0; w < k; w++) { x[w] = e[w]; e[w] = acc[w]; }
        mulmod_simple(K, q, acc, acc, x);
    }
}
// the exact chain of every level-0 chunk: a <- init_j (chunk 0, as given) or carry[u]; (q, rem) = divmod(a c_(i, j), n^2), a <- rem
__global__ void __launch_bounds__(32) k_simple_trace_chain(const SimpleConsts* __restrict__ K, const u64* __restrict__ init,
                                                           const u64* __restrict__ c, const u64* __restrict__ carry, size_t count,
                                                           size_t chains, size_t s, u64* __restrict__ acc_out, u64* __restrict__ q_out,
                                                           int* flags) {
    const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= (count + s - 1) / s * chains) return;
    const size_t b = u / chains, j = u - b * chains;
    const int k = K->k;
    u64 a[PB200_SIMPLE_MAXK], x[PB200_SIMPLE_MAXK], q[PB200_SIMPLE_MAXK];
    const u64* a0 = b ? carry + u * k : init + j * k;
    for (int w = 0; w < k; w++) a[w] = a0[w];
    int bad = 0;
    for (size_t i = b * s; i < count && i < (b + 1) * s; i++) {
        const size_t e = (i * chains + j) * k;
        for (int w = 0; w < k; w++) x[w] = c[e + w];
        bad |= mulmod_simple(K, q, a, a, x);
        for (int w = 0; w < k; w++) acc_out[e + w] = a[w];
        if (q_out) for (int w = 0; w < k; w++) q_out[e + w] = q[w];
    }
    if (bad) atomicOr(flags, 1);
}

// K5: value (words_per_value u64 words) -> value_bits/limb_bits limbs, 2 words per limb (lo, hi)
__global__ void k_repack(const u64* __restrict__ vals, size_t count, int wpv, int nl, int limb_bits, u64* __restrict__ out) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= count * (size_t)nl) return;
    size_t u = idx / nl; int l = (int)(idx % nl);
    const u64* v = vals + u * wpv;
    int lo_bit = l * limb_bits;
    u64 w[3];
    for (int j = 0; j < 3; j++) { int wi = (lo_bit >> 6) + j; w[j] = wi < wpv ? v[wi] : 0; }
    int sh = lo_bit & 63;
    u64 lo = sh ? (w[0] >> sh) | (w[1] << (64 - sh)) : w[0];
    u64 hi = sh ? (w[1] >> sh) | (w[2] << (64 - sh)) : w[1];
    if (limb_bits <= 64) { hi = 0; if (limb_bits < 64) lo &= (1ull << limb_bits) - 1; }
    else if (limb_bits < 128) hi &= (1ull << (limb_bits - 64)) - 1;
    out[2 * idx] = lo; out[2 * idx + 1] = hi;
}

// ---- launchers ------------------------------------------------------------------------------
cudaError_t simple_gchain(const SimpleConsts* dK, u64* d_gchain, int n_bits, cudaStream_t st) {
    k_simple_gchain<<<1, 1, 0, st>>>(dK, d_gchain, n_bits); count_launch();
    return cudaGetLastError();
}
cudaError_t simple_encrypt(const SimpleConsts* dK, const u64* d_gchain, const u64* d_m, const u64* d_r, size_t count,
                           u64* d_c, u64* d_records, const u64* d_offsets, u64* d_digest, int* d_flags, cudaStream_t st) {
    if (!count) return cudaSuccess;
    unsigned grid = (unsigned)((count + 31) / 32);
    k_simple_encrypt<<<grid, 32, 0, st>>>(dK, d_gchain, d_m, d_r, count, d_c, d_records, d_offsets, d_digest, d_flags);
    count_launch();
    return cudaGetLastError();
}
cudaError_t simple_add(const SimpleConsts* dK, const u64* d_c1, const u64* d_c2, int c_words, size_t count,
                       u64* d_out, u64* d_q, int* d_flags, cudaStream_t st) {
    if (!count) return cudaSuccess;
    unsigned grid = (unsigned)((count + 31) / 32);
    k_simple_add<<<grid, 32, 0, st>>>(dK, d_c1, d_c2, c_words, count, d_out, d_q, d_flags); count_launch();
    return cudaGetLastError();
}
static const int kTallyT1 = 148 * 32, kTallyT2 = 128;
size_t simple_tally_scratch_words(int k) { return (size_t)(kTallyT1 + kTallyT2) * k; }
cudaError_t simple_tally(const SimpleConsts* dK, int k, const u64* d_c, size_t count, u64* d_out, u64* d_scratch,
                         int* d_flags, cudaStream_t st) {
    // level 1: T1 strided partial products; level 2: T2 partials of those; final: one thread folds T2 values
    int T1 = (int)(count < (size_t)kTallyT1 ? count : (size_t)kTallyT1);
    int T2 = T1 < kTallyT2 ? T1 : kTallyT2;
    u64* p1 = d_scratch;
    u64* p2 = d_scratch + (size_t)kTallyT1 * k;
    if (T1 > 0) {
        k_simple_tally_partial<<<(T1 + 31) / 32, 32, 0, st>>>(dK, d_c, count, p1, T1, d_flags); count_launch();
        k_simple_tally_partial<<<(T2 + 31) / 32, 32, 0, st>>>(dK, p1, (size_t)T1, p2, T2, d_flags); count_launch();
    }
    k_simple_tally_final<<<1, 1, 0, st>>>(dK, p2, T2, d_out, d_flags); count_launch();
    return cudaGetLastError();
}
cudaError_t simple_pow(const SimpleConsts* dK, const u64* d_base, int base_words, const u64* d_e, int e_bits, int e_stride, size_t count,
                       u64* d_out, int* d_flags, cudaStream_t st) {
    if (!count) return cudaSuccess;
    k_simple_pow<<<(unsigned)((count + 31) / 32), 32, 0, st>>>(dK, d_base, base_words, d_e, e_bits, e_stride, count, d_out, d_flags);
    count_launch();
    return cudaGetLastError();
}
cudaError_t simple_lfunc(const SimpleConsts* dKn, const u64* d_x, size_t count, u64* d_m, int* d_flags, cudaStream_t st) {
    if (!count) return cudaSuccess;
    k_simple_lfunc<<<(unsigned)((count + 31) / 32), 32, 0, st>>>(dKn, d_x, count, d_m, d_flags); count_launch();
    return cudaGetLastError();
}
size_t simple_trace_scan_words(const TracePlan& P, size_t chains, int k) {
    size_t w = 0;
    for (size_t l = 0; l + 1 < P.n.size(); l++) w += P.n[l + 1] * chains * k;
    return w;
}
cudaError_t simple_trace_scan(const SimpleConsts* dK, int k, const TracePlan& P, const u64* d_init, const u64* d_c, size_t chains, u64* d_tmp,
                              cudaStream_t st) {
    const size_t L = P.n.size() - 1;
    std::vector<u64*> buf(L);
    for (size_t l = 0, o = 0; l < L; l++) { buf[l] = d_tmp + o; o += P.n[l + 1] * chains * k; }
    for (size_t l = 0; l < L; l++) {
        k_simple_trace_reduce<<<(unsigned)((P.n[l + 1] * chains + 31) / 32), 32, 0, st>>>(dK, l ? buf[l - 1] : d_c, P.n[l], chains, P.s[l], buf[l]);
        count_launch();
    }
    for (size_t l = L; l >= 1; l--) {
        const size_t units = (P.n[l] + P.s[l] - 1) / P.s[l] * chains;
        k_simple_trace_apply<<<(unsigned)((units + 31) / 32), 32, 0, st>>>(dK, d_init, l == L ? nullptr : buf[l], buf[l - 1], P.n[l], chains, P.s[l]);
        count_launch();
    }
    return cudaGetLastError();
}
cudaError_t simple_trace_chain(const SimpleConsts* dK, const u64* d_init, const u64* d_c, const u64* d_carry, size_t count, size_t chains,
                               size_t s, u64* d_acc, u64* d_q, int* d_flags, cudaStream_t st) {
    const size_t units = (count + s - 1) / s * chains;
    k_simple_trace_chain<<<(unsigned)((units + 31) / 32), 32, 0, st>>>(dK, d_init, d_c, d_carry, count, chains, s, d_acc, d_q, d_flags);
    count_launch();
    return cudaGetLastError();
}
cudaError_t repack_limbs(const u64* d_vals, size_t count, int wpv, int value_bits, int limb_bits, u64* d_out, cudaStream_t st) {
    int nl = value_bits / limb_bits;
    size_t total = count * (size_t)nl;
    if (!total) return cudaSuccess;
    k_repack<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_vals, count, wpv, nl, limb_bits, d_out); count_launch();
    return cudaGetLastError();
}

}  // namespace pb200
