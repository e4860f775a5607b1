// scalar_cpu.cpp — OpenSSL BIGNUM reference of homomorphic scalar multiplication, out = c^k mod n^2 per unit.
// TEST / MEASUREMENT INFRASTRUCTURE ONLY: the large parity checks of tests/test_gpu_scalar.py and tools/scalar_bench.py.  Never
// linked into the product library.  Words are little-endian uint64 (same layout as include/paillier_b200.h).
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

// out[u] = c[u]^k[u] mod n^2; c: count * 2 words_in words (any value), k: count * k_words words; `threads` worker threads
int cpu_paillier_scalar_batch(const uint64_t* n_w, int words_in, const uint64_t* c_w, const uint64_t* k_w, int k_words, size_t count,
                              uint64_t* out_w, int threads) {
    if (threads < 1) threads = 1;
    const int words_out = 2 * words_in;
    std::atomic<size_t> next{0};
    std::atomic<int> err{0};
    auto work = [&]() {
        BN_CTX* ctx = BN_CTX_new();
        BIGNUM* n = from_words(n_w, words_in);
        BIGNUM* n2 = BN_new(); BIGNUM* r = BN_new();
        BN_mul(n2, n, n, ctx);
        for (;;) {
            const size_t u0 = next.fetch_add(64);
            if (u0 >= count) break;
            for (size_t u = u0; u < count && u < u0 + 64; u++) {
                BIGNUM* c = from_words(c_w + u * words_out, words_out);
                BIGNUM* k = from_words(k_w + u * k_words, k_words);
                if (!BN_mod_exp(r, c, k, n2, ctx)) err = 1;     // reduces c first; c^0 = 1
                to_words(r, out_w + u * words_out, words_out);
                BN_free(c); BN_free(k);
            }
        }
        BN_free(n); BN_free(n2); BN_free(r); BN_CTX_free(ctx);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    return err.load();
}

}  // extern "C"
