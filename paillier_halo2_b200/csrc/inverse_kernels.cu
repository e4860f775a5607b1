// inverse_kernels.cu — c^-1 mod n^2 per ciphertext, one thread each: the kernel of pb200_inverse_batch, pb200_sub_batch and the sign
// step of pb200_scalar_mul_signed_batch.
//
// 1. x0 = c^-1 mod n by Bernstein-Yang safegcd (2019): batches of 62 divsteps on the low 64 bits of (f, g) = (n, c mod n), each
//    giving a transition matrix t with 2^62 (f', g') = t (f, g), applied to (f, g) with an exact division by 2^62 and to (d, e) mod n
//    (n^-1 mod 2^62 cancels the low 62 bits), on signed 62-bit limbs as in libsecp256k1's modinv64.  The batch count is fixed by the
//    iteration bound floor((49 d + 57) / 17) for a d-bit modulus (96 batches at d = 2048), so every lane runs the same loop and no warp
//    diverges on data.  f = +-1 at the end <=> gcd(c, n) = 1.
// 2. x = x0 (2 - c x0) mod n^2, one Hensel step (c x0 = 1 + t n gives c x = 1 - t^2 n^2), on the simple64 Barrett multiplication.
// tests/model_safegcd.py is the limb-exact model of this file.
#include "../../include/paillier_b200.h"
#include "engine.hpp"

namespace pb200 {

typedef long long i64;
typedef __int128 i128;
static const u64 M62 = (1ull << 62) - 1;

// 62 divsteps on the low 64 bits of f (odd) and g; t = (u, v, q, r) with 2^62 (f', g') = (u f + v g, q f + r g).  Branch-free: the
// swap and the odd-g addition are selected by masks (libsecp256k1's divsteps_59 form, with delta in place of zeta).
__device__ __forceinline__ int divsteps_62(int delta, u64 f, u64 g, i64* t) {
    i64 u = 1, v = 0, q = 0, r = 1;
#pragma unroll 2
    for (int i = 0; i < 62; i++) {
        const i64 godd = -(i64)(g & 1);                 // -1 when g is odd
        const i64 c1 = godd & (i64)((-delta) >> 31);    // -1 when delta > 0 and g is odd: swap
        const u64 x = (f ^ (u64)c1) - (u64)c1;          // -f on a swap
        const i64 y = (u ^ c1) - c1, z = (v ^ c1) - c1;
        g += x & (u64)godd; q += y & godd; r += z & godd;
        f += g & (u64)c1; u += q & c1; v += r & c1;     // on a swap f <- old g, (u, v) <- old (q, r)
        delta = ((delta ^ (int)c1) - (int)c1) + 1;      // 1 - delta on a swap, else 1 + delta
        g >>= 1; u += u; v += v;
    }
    t[0] = u; t[1] = v; t[2] = q; t[3] = r;
    return delta;
}

__device__ __forceinline__ u64 low64(const i64* a, int L) { return (u64)a[0] | (L > 1 ? (u64)a[1] << 62 : 0); }

// (f, g) <- t (f, g) / 2^62, exact
__device__ __forceinline__ void update_fg(i64* f, i64* g, int L, const i64* t) {
    const i64 u = t[0], v = t[1], q = t[2], r = t[3];
    i128 cf = (i128)u * f[0] + (i128)v * g[0], cg = (i128)q * f[0] + (i128)r * g[0];
    cf >>= 62; cg >>= 62;
    for (int i = 1; i < L; i++) {
        const i64 fi = f[i], gi = g[i];
        cf += (i128)u * fi + (i128)v * gi;
        cg += (i128)q * fi + (i128)r * gi;
        f[i - 1] = (i64)((u64)cf & M62); g[i - 1] = (i64)((u64)cg & M62);
        cf >>= 62; cg >>= 62;
    }
    f[L - 1] = (i64)cf; g[L - 1] = (i64)cg;
}

// (d, e) <- t (d, e) / 2^62 mod n, both kept in (-2n, n)
__device__ __forceinline__ void update_de(i64* d, i64* e, int L, const i64* t, const InvConsts* __restrict__ I) {
    const i64 u = t[0], v = t[1], q = t[2], r = t[3];
    const i64 sd = d[L - 1] >> 63, se = e[L - 1] >> 63;
    i64 md = (u & sd) + (v & se), me = (q & sd) + (r & se);
    i128 cd = (i128)u * d[0] + (i128)v * e[0], ce = (i128)q * d[0] + (i128)r * e[0];
    md -= (i64)((I->ninv62 * (u64)cd + (u64)md) & M62);
    me -= (i64)((I->ninv62 * (u64)ce + (u64)me) & M62);
    cd += (i128)I->n62[0] * md; ce += (i128)I->n62[0] * me;
    cd >>= 62; ce >>= 62;
    for (int i = 1; i < L; i++) {
        const i64 di = d[i], ei = e[i], ni = I->n62[i];
        cd += (i128)u * di + (i128)v * ei + (i128)ni * md;
        ce += (i128)q * di + (i128)r * ei + (i128)ni * me;
        d[i - 1] = (i64)((u64)cd & M62); e[i - 1] = (i64)((u64)ce & M62);
        cd >>= 62; ce >>= 62;
    }
    d[L - 1] = (i64)cd; e[L - 1] = (i64)ce;
}

// a += b & mask, then a = -a where neg == -1 (every limb (a_i ^ neg) - neg), carries rippled; mask, neg in {0, -1}
__device__ __forceinline__ void add_neg(i64* a, const i64* b, i64 mask, i64 neg, int L) {
    i64 c = 0;
    for (int i = 0; i < L; i++) {
        c += a[i] + (b[i] & mask);
        if (i < L - 1) { a[i] = (i64)((u64)c & M62); c >>= 62; } else a[i] = c;
    }
    c = 0;
    for (int i = 0; i < L; i++) {
        c += (a[i] ^ neg) - neg;
        if (i < L - 1) { a[i] = (i64)((u64)c & M62); c >>= 62; } else a[i] = c;
    }
}

// 64-bit words <-> 62-bit limbs of a value 0 <= x < 2^(62 L)
__device__ __forceinline__ void words_to_62(i64* a, const u64* w, int nw, int L) {
    for (int i = 0; i < L; i++) {
        const int bit = 62 * i, wi = bit >> 6, sh = bit & 63;
        u64 x = wi < nw ? w[wi] >> sh : 0;
        if (sh > 2 && wi + 1 < nw) x |= w[wi + 1] << (64 - sh);
        a[i] = (i64)(x & M62);
    }
}
__device__ __forceinline__ void limbs62_to_words(u64* w, const i64* a, int L, int nw) {
    for (int j = 0; j < nw; j++) {
        const int bit = 64 * j, li = bit / 62, sh = bit - 62 * li;
        u64 x = li < L ? (u64)a[li] >> sh : 0;
        if (li + 1 < L) x |= (u64)a[li + 1] << (62 - sh);
        if (sh > 60 && li + 2 < L) x |= (u64)a[li + 2] << (124 - sh);
        w[j] = x;
    }
}

// whether the nw-word x has a bit at or above `bits`
__device__ __forceinline__ bool wider_than(const u64* x, int nw, int bits) {
    const int w = bits >> 6, b = bits & 63;
    u64 over = w < nw ? x[w] >> b : 0;
    for (int i = w + 1; i < nw; i++) over |= x[i];
    return over != 0;
}

// out_u = c_u^-1 mod n^2 (c1 == null) or c1_u * c_u^-1 mod n^2; 0 and flag PB200_FLAG_NOT_INVERTIBLE when gcd(c_u, n) != 1.  neg != null:
// only the units with neg[u] != 0 and a non-zero magnitude (kw words at mag + u kw) are inverted, the others are left as they are (the
// in-place sign step of the signed scalar multiplication).  Any words_out-word c and c1 (reduced mod n^2).
__global__ void __launch_bounds__(128) k_inverse(const SimpleConsts* __restrict__ K, const InvConsts* __restrict__ I, const u64* c,
                                                 const u64* __restrict__ c1, const uint8_t* __restrict__ neg, const u64* __restrict__ mag,
                                                 int kw, size_t count, u64* out, int* flags) {
    const size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= count) return;
    if (neg) {
        u64 nz = 0;
        for (int i = 0; i < kw; i++) nz |= mag[u * kw + i];
        if (!neg[u] || !nz) return;
    }
    const int k = K->k, kin = K->kin, L = I->L;
    u64 a[PB200_SIMPLE_MAXK], X[2 * PB200_SIMPLE_MAXK + 1], q[PB200_SIMPLE_MAXK], y[PB200_SIMPLE_MAXK], x0[PB200_SIMPLE_MAXK / 2];
    for (int i = 0; i < k; i++) a[i] = c[u * k + i];
    // y = c mod n (Barrett of the modulus n; a value too wide for it is reduced mod n^2 first)
    for (int i = 0; i < 2 * k; i++) X[i] = i < k ? a[i] : 0;     // 2 kin <= 2 k words read below
    if (wider_than(a, k, 128 * kin - I->n.s)) {
        barrett_simple(K, q, y, X);
        for (int i = 0; i < 2 * k; i++) X[i] = i < k ? y[i] : 0;
    }
    barrett_simple(&I->n, q, y, X);
    // safegcd: f = n, g = y, d = 0, e = 1
    i64 f[PB200_INV_MAXL], g[PB200_INV_MAXL], d[PB200_INV_MAXL], e[PB200_INV_MAXL], t[4];
    for (int i = 0; i < L; i++) { f[i] = I->n62[i]; d[i] = 0; e[i] = i == 0; }
    words_to_62(g, y, kin, L);
    int delta = 1;
    for (int b = 0; b < I->batches; b++) {
        delta = divsteps_62(delta, low64(f, L), low64(g, L), t);
        update_fg(f, g, L, t);
        update_de(d, e, L, t, I);
    }
    // f = 1 or f = -1 (normalised limbs: all ones below a top limb of -1)
    bool one = f[0] == 1, mone = L == 1 ? f[0] == -1 : f[0] == (i64)M62;
    for (int i = 1; i < L; i++) { one &= f[i] == 0; mone &= f[i] == (i == L - 1 ? -1 : (i64)M62); }
    const bool bad = !one && !mone;
    // x0 = d sign(f) in [0, n): add n if negative, negate for f = -1, add n if negative
    add_neg(d, I->n62, d[L - 1] >> 63, mone ? -1 : 0, L);
    add_neg(d, I->n62, d[L - 1] >> 63, 0, L);
    limbs62_to_words(x0, d, L, kin);
    // Hensel: y = n^2 + 2 - c x0 mod n^2, x = x0 y mod n^2 (both products kin x k words; y < n^2 + 2 is taken unreduced)
    mul_full(X, a, k, x0, kin);
    for (int i = k + kin; i < 2 * k; i++) X[i] = 0;
    barrett_simple(K, q, y, X);
    u64 cy = 2, br = 0;
    for (int i = 0; i < k; i++) {
        const u64 s = I->n2[i] + cy; cy = s < cy;
        const u64 d1 = s - y[i], b1 = s < y[i], d2 = d1 - br, b2 = d1 < br;
        y[i] = d2; br = b1 | b2;
    }
    mul_full(X, x0, kin, y, k);
    for (int i = k + kin; i < 2 * k; i++) X[i] = 0;
    barrett_simple(K, q, a, X);
    if (c1) {
        for (int i = 0; i < k; i++) y[i] = c1[u * k + i];
        mulmod_simple(K, q, a, y, a);
    }
    for (int i = 0; i < k; i++) out[u * k + i] = bad ? 0 : a[i];
    if (bad) atomicOr(flags, (int)PB200_FLAG_NOT_INVERTIBLE);
}

void inverse_consts(const BigInt& n, uint32_t n_bits, InvConsts* h) {
    const int L = (int)(n_bits / 62 + 1);
    const int steps = n_bits < 46 ? (49 * (int)n_bits + 80) / 17 : (49 * (int)n_bits + 57) / 17;
    h->L = L;
    h->batches = (steps + 61) / 62;
    const uint64_t n0 = (uint64_t)n.w[0] | (n.w.size() > 1 ? (uint64_t)n.w[1] << 32 : 0);
    uint64_t inv = n0;                                  // Newton: inv = n0^-1 mod 2^(3 * 2^i), n0 odd
    for (int i = 0; i < 5; i++) inv *= 2 - n0 * inv;
    h->ninv62 = inv & M62;
    for (int i = 0; i < L; i++) {
        int64_t limb = 0;
        for (int b = 0; b < 62; b++) if (n.bit((size_t)(62 * i + b))) limb |= (int64_t)1 << b;
        h->n62[i] = limb;
    }
    BigInt::mul(n, n).to_u64_le(h->n2, PB200_SIMPLE_MAXK);
}

cudaError_t simple_inverse(const SimpleConsts* dK, const InvConsts* dI, const u64* d_c, const u64* d_c1, const uint8_t* d_neg, const u64* d_mag,
                           int kw, size_t count, u64* d_out, int* d_flags, cudaStream_t st) {
    if (!count) return cudaSuccess;
    k_inverse<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(dK, dI, d_c, d_c1, d_neg, d_mag, kw, count, d_out, d_flags);
    count_launch();
    return cudaGetLastError();
}

}  // namespace pb200
