// matvec_cpu.cpp — OpenSSL BIGNUM reference of the encrypted matrix-vector product (pb200_matvec, include/paillier_b200.h).
// TEST INFRASTRUCTURE ONLY: the parity checks of tests/test_gpu_matvec.py (built by tests/matvec_oracle.py into a temporary
// directory).  Never linked into the product library.  Words are little-endian uint64 (same layout as include/paillier_b200.h).
#include <openssl/bn.h>
#include <atomic>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

static BIGNUM* from_words(const uint64_t* w, int n) {
    std::vector<unsigned char> buf((size_t)n * 8);
    memcpy(buf.data(), w, buf.size());
    return BN_lebin2bn(buf.data(), (int)buf.size(), nullptr);
}
static void to_words(const BIGNUM* b, uint64_t* w, int n) {
    std::vector<unsigned char> buf((size_t)n * 8);
    BN_bn2lebinpad(b, buf.data(), (int)buf.size());
    memcpy(w, buf.data(), buf.size());
}

extern "C" {

// out[r] = P_r * N_r^(n-1) mod n^2 with P_r = prod_{w_ri > 0} c_i^|w_ri|, N_r = prod_{w_ri < 0} c_i^|w_ri| (include/paillier_b200.h,
// pb200_matvec).  c: count * 2 words_in words; w: rows * count * k_words magnitude words, row-major; neg: nullable, rows * count bytes.
// Work items are (row, slice of the ciphertexts); their partial products are folded per row at the end.
int cpu_paillier_matvec(const uint64_t* n_w, int words_in, const uint64_t* c_w, size_t count, const uint64_t* w_w, const uint8_t* neg,
                        int k_words, size_t rows, uint64_t* out_w, int threads) {
    if (threads < 1) threads = 1;
    const int words_out = 2 * words_in;
    const size_t slices = (size_t)threads, items = rows * slices;
    std::vector<uint64_t> part(items * 2 * words_out, 0);
    std::atomic<size_t> next{0};
    std::atomic<int> err{0};
    auto work = [&]() {
        BN_CTX* ctx = BN_CTX_new();
        BIGNUM* n = from_words(n_w, words_in);
        BIGNUM* n2 = BN_new(); BIGNUM* t = BN_new(); BIGNUM* acc[2] = {BN_new(), BN_new()};
        BN_mul(n2, n, n, ctx);
        for (;;) {
            const size_t it = next.fetch_add(1);
            if (it >= items) break;
            const size_t r = it / slices, s = it % slices, i0 = count * s / slices, i1 = count * (s + 1) / slices;
            BN_one(acc[0]); BN_one(acc[1]);
            for (size_t i = i0; i < i1; i++) {
                const size_t e = r * count + i;
                BIGNUM* c = from_words(c_w + i * words_out, words_out);
                BIGNUM* k = from_words(w_w + e * k_words, k_words);
                if (!BN_mod_exp(t, c, k, n2, ctx)) err = 1;
                BIGNUM* a = acc[neg && neg[e] ? 1 : 0];
                if (!BN_mod_mul(a, a, t, n2, ctx)) err = 1;
                BN_free(c); BN_free(k);
            }
            to_words(acc[0], part.data() + it * 2 * words_out, words_out);
            to_words(acc[1], part.data() + it * 2 * words_out + words_out, words_out);
        }
        BN_free(n); BN_free(n2); BN_free(t); BN_free(acc[0]); BN_free(acc[1]); BN_CTX_free(ctx);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    BN_CTX* ctx = BN_CTX_new();
    BIGNUM* n = from_words(n_w, words_in);
    BIGNUM* n2 = BN_new(); BIGNUM* nm1 = BN_dup(n); BIGNUM* P = BN_new(); BIGNUM* N = BN_new();
    BN_mul(n2, n, n, ctx);
    BN_sub_word(nm1, 1);
    for (size_t r = 0; r < rows; r++) {
        BN_one(P); BN_one(N);
        for (size_t s = 0; s < slices; s++) {
            BIGNUM* p = from_words(part.data() + (r * slices + s) * 2 * words_out, words_out);
            BIGNUM* q = from_words(part.data() + (r * slices + s) * 2 * words_out + words_out, words_out);
            if (!BN_mod_mul(P, P, p, n2, ctx) || !BN_mod_mul(N, N, q, n2, ctx)) err = 1;
            BN_free(p); BN_free(q);
        }
        if (!BN_mod_exp(N, N, nm1, n2, ctx) || !BN_mod_mul(P, P, N, n2, ctx)) err = 1;
        BN_nnmod(P, P, n2, ctx);                                   // count == 0: 1 mod n^2
        to_words(P, out_w + r * words_out, words_out);
    }
    BN_free(n); BN_free(n2); BN_free(nm1); BN_free(P); BN_free(N); BN_CTX_free(ctx);
    return err.load();
}


}  // extern "C"
