"""Ciphertext inverse (c^-1 mod n^2), homomorphic subtraction (c1 c2^-1) and signed scalars (c^k, k of any sign): bit-exact against Python
ints on every key size, non-invertible units and their status / flag, decryption round trips, every engine, small and short keys, an
even modulus and the device-pointer variants."""
import random
from math import gcd

import numpy as np
import pytest

from paillier_halo2_b200 import _lib, workload
from paillier_halo2_b200.api import PaillierKey, Pb200Error, ints_to_words, private_from_primes, words, words_to_ints

gpu = pytest.mark.gpu


def _invert_twice(key, c_w):
    """every call runs twice with identical output"""
    a = key.invert_words(c_w)
    assert (key.invert_words(c_w) == a).all()
    return a


def _edges(n, wo):
    """invertible edge values, reduced and not: 1, 2, n - 1, n + 1, n^2 - 1, n^2 + 1, 2^(64 wo) - 1 and a value with a long run of zero low bits"""
    cs = [1, 2, n - 1, n + 1, n * n - 1, n * n + 1, (1 << (64 * wo)) - 1, (n - 2) << 300]
    return [c for c in cs if gcd(c, n) == 1 and c < 1 << (64 * wo)]


@gpu
@pytest.mark.parametrize("n_bits,count", [(1024, 64 * 32 + 7), (2048, 64 * 16 + 7), (3072, 64 * 4 + 7), (4096, 64 * 4 + 7)])
def test_inverse_parity(built_lib, n_bits, count):
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    n2, wo = n * n, 2 * n_bits // 64
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=41)
    edges = _edges(n, wo)
    c_w[100:100 + len(edges)] = ints_to_words(edges, wo)
    cs = words_to_ints(c_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        got = words_to_ints(_invert_twice(key, c_w))
    assert got == [pow(c, -1, n2) for c in cs]


@gpu
def test_inverse_large_batch(built_lib):
    n_bits, count = 2048, (1 << 18) + 5
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    n2 = n * n
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=42)
    with PaillierKey(n, g, n_bits, 64) as key:
        got = key.invert_words(c_w)
    cs, xs = words_to_ints(c_w), words_to_ints(got)
    assert all(x < n2 and c * x % n2 == 1 for c, x in zip(cs, xs))       # the inverse is unique: this is pow(c, -1, n2)


def _non_invertible(kd, rng):
    n, p, q = kd["n"], kd["p"], kd["q"]
    return [0, n, n * n, p * rng.getrandbits(200), q * rng.getrandbits(200), p, 7 * q]


@gpu
def test_not_invertible_units(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    n2, wo = n * n, 2 * n_bits // 64
    rng = random.Random(43)
    count = 200
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=43)
    bad = [3, 40, 41, 99, 128, 150, 199]
    c_w[bad] = ints_to_words(_non_invertible(kd, rng), wo)
    cs = words_to_ints(c_w)
    want = [0 if i in bad else pow(c, -1, n2) for i, c in enumerate(cs)]
    import torch
    with PaillierKey(n, g, n_bits, 64) as key:
        for _ in range(2):
            with pytest.raises(Pb200Error) as e:
                key.invert_words(c_w)
            assert e.value.status == _lib.PB200_ERR_NOT_INVERTIBLE
            assert words_to_ints(e.value.outputs) == want
        # _dev: the flag, and it does not leak into a later host call
        d_c = torch.from_numpy(c_w.view(np.int64)).cuda()
        d_out = torch.empty_like(d_c)
        key.invert_dev(d_c.data_ptr(), count, d_out.data_ptr())
        assert key.take_flags() == _lib.PB200_FLAG_NOT_INVERTIBLE
        assert words_to_ints(d_out.cpu().numpy().view(np.uint64)) == want
        key.invert_dev(d_c.data_ptr(), count, d_out.data_ptr())
        good = [c for i, c in enumerate(cs) if i not in bad]
        assert key.invert(good) == [pow(c, -1, n2) for c in good]
        assert key.take_flags() == 0
        key.invert_dev(d_c[:3].data_ptr(), 3, d_out.data_ptr())
        assert key.take_flags() == 0 and key.invert([]) == []


@gpu
def test_sub(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    n2, wo = n * n, 2 * n_bits // 64
    count = 64 * 3 + 7
    c1 = words_to_ints(workload.ciphertexts(n_bits, count, n, seed_offset=44))
    c2 = words_to_ints(workload.ciphertexts(n_bits, count, n, seed_offset=45))
    top = (1 << (64 * wo)) - 1
    c1[5], c2[6], c1[7], c2[7] = top, top, n2 + 12345, n2 + 1       # unreduced operands
    c1[8] = 0                                                          # output 0, no error
    with PaillierKey(n, g, n_bits, 64) as key:
        for _ in range(2):
            assert key.sub(c1, c2) == [a * pow(b, -1, n2) % n2 for a, b in zip(c1, c2)]
        c2[9] = kd["p"] * 3
        with pytest.raises(Pb200Error) as e:
            key.sub_words(ints_to_words(c1, wo), ints_to_words(c2, wo))
        assert e.value.status == _lib.PB200_ERR_NOT_INVERTIBLE
        got = words_to_ints(e.value.outputs)
        assert got[9] == 0 and got[:9] + got[10:] == [a * pow(b, -1, n2) % n2 for i, (a, b) in enumerate(zip(c1, c2)) if i != 9]
        assert key.sub([], []) == []


@gpu
def test_scalar_mul_signed(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    n2, wo = n * n, 2 * n_bits // 64
    rng = random.Random(46)
    count = 200
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=46)
    cs = words_to_ints(c_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        for k_bits in (1, 32, 64, 65, n_bits):
            mags = [rng.getrandbits(k_bits) for _ in range(count)]
            mags[3], mags[4], mags[40] = (1 << k_bits) - 1, 0, 1 << (k_bits - 1)
            neg = np.array([rng.random() < 0.5 for _ in range(count)], dtype=np.uint8)
            neg[4] = 1                                                   # -0
            mag_w = ints_to_words(mags, words(k_bits))
            got = words_to_ints(key.scalar_mul_signed_words(c_w, mag_w, neg, k_bits))
            assert got == [pow(c, -m if s else m, n2) for c, m, s in zip(cs, mags, neg)], k_bits
            # k_neg = NULL and all-positive signs: exactly pb200_scalar_mul_batch
            plain = key.scalar_mul_words(c_w, mag_w, k_bits)
            assert (key.scalar_mul_signed_words(c_w, mag_w, None, k_bits) == plain).all()
            assert (key.scalar_mul_signed_words(c_w, mag_w, np.zeros(count, np.uint8), k_bits) == plain).all()
        # mixed signs, short scalars and one full-width lane in the same CTA; -0 with c = 0 gives 1
        ks = [rng.choice([-1, 1]) * rng.getrandbits(rng.choice([1, 5, 32])) for _ in range(count)]
        ks[37] = -(rng.getrandbits(n_bits) | 1 << (n_bits - 1))
        ks[38] = -(n - 1)
        ks[39] = (1 << n_bits) - 1
        cs2 = list(cs)
        cs2[50], ks[50] = 0, 0
        cs2[51], ks[51] = (1 << (64 * wo)) - 1, -3                        # unreduced base
        k_w = ints_to_words([abs(k) for k in ks], words(n_bits))
        neg = np.array([k < 0 for k in ks], dtype=np.uint8)
        neg[50] = 1
        got = words_to_ints(key.scalar_mul_signed_words(ints_to_words(cs2, wo), k_w, neg, n_bits))
        assert got == [pow(c, k, n2) for c, k in zip(cs2, ks)]
        assert got[50] == 1
        assert key.scalar_mul_signed(cs2, ks) == got
        with pytest.raises(Pb200Error) as e:
            key.scalar_mul_signed([cs[0]], [1 << n_bits])
        assert e.value.status == _lib.PB200_ERR_RANGE
        with pytest.raises(Pb200Error) as e:                              # a negative power of a non-invertible value
            key.scalar_mul_signed([cs[0], kd["q"], 0], [-2, -5, -1])
        assert e.value.status == _lib.PB200_ERR_NOT_INVERTIBLE
        assert words_to_ints(e.value.outputs) == [pow(cs[0], -2, n2), 0, 0]
        assert key.scalar_mul_signed([kd["q"]], [5]) == [pow(kd["q"], 5, n2)]
        assert key.scalar_mul_signed([], []) == []


@pytest.mark.parametrize("g_kind", ["g_rand", "g_std"])
@gpu
def test_decryption_round_trips(built_lib, g_kind):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, p, q = kd["n"], kd["p"], kd["q"]
    g = kd["g_rand"] if g_kind == "g_rand" else n + 1
    rng = random.Random(47)
    m_w, r_w = workload.units(n_bits, 100, seed_offset=23)
    ms = words_to_ints(m_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        key.set_private(*private_from_primes(p, q, g))
        cs = words_to_ints(key.encrypt_words(m_w, r_w))
        assert key.decrypt(key.invert(cs)) == [-m % n for m in ms]
        a, b = cs[:50], cs[50:]
        assert key.decrypt(key.sub(a, b)) == [(x - y) % n for x, y in zip(ms[:50], ms[50:])]
        ss = [rng.getrandbits(rng.choice([1, 16, 64, 300])) for _ in ms]
        assert key.decrypt(key.scalar_mul_signed(cs, [-s for s in ss])) == [-s * m % n for s, m in zip(ss, ms)]


@gpu
def test_every_engine_gives_identical_outputs(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(48)
    count = 64 * 3 + 7
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=48)
    cs = words_to_ints(c_w)
    ks = [rng.choice([-1, 1]) * rng.getrandbits(rng.choice([1, 32, n_bits])) for _ in range(count)]
    n2 = n * n
    want_s = [pow(c, k, n2) for c, k in zip(cs, ks)]
    want_i = [pow(c, -1, n2) for c in cs]
    ran = []
    with PaillierKey(n, g, n_bits, 64) as key:
        for engine in (1, 2, 3, 4, 5):
            try:
                key.set_engine(engine)
            except Pb200Error as e:
                assert e.status == _lib.PB200_ERR_UNSUPPORTED
                continue
            assert key.scalar_mul_signed(cs, ks) == want_s, key.engine
            assert key.invert(cs) == want_i, key.engine
            assert key.sub(cs, cs[::-1]) == [a * pow(b, -1, n2) % n2 for a, b in zip(cs, cs[::-1])], key.engine
            ran.append(key.engine)
    assert len(ran) >= 4, ran


@gpu
def test_small_and_short_keys(built_lib):
    """the reference-default key sizes (128 / 64, 264 / 88) on the automatic engine and simple64, and a short n (fewer bits than declared)"""
    rng = random.Random(49)
    cases = [(128, 64, rng.getrandbits(128) | 1 << 127 | 1), (264, 88, rng.getrandbits(264) | 1 << 263 | 1),
             (1024, 64, rng.getrandbits(1000) | 1)]
    for n_bits, limb_bits, n in cases:
        g = rng.getrandbits(n_bits)
        n2, wo = n * n, words(2 * n_bits)
        cs = _edges(n, wo) + [rng.randrange(n2) for _ in range(70)]
        cs = [c for c in cs if gcd(c, n) == 1]
        ks = [rng.choice([-1, 1]) * rng.getrandbits(rng.choice([1, 9, n_bits])) for _ in cs]
        with PaillierKey(n, g, n_bits, limb_bits) as key:
            for engine in (0, 1):
                key.set_engine(engine)
                assert key.invert(cs) == [pow(c, -1, n2) for c in cs], (n_bits, key.engine)
                assert key.sub(cs, cs[::-1]) == [a * pow(b, -1, n2) % n2 for a, b in zip(cs, cs[::-1])], (n_bits, key.engine)
                assert key.scalar_mul_signed(cs, ks) == [pow(c, k, n2) for c, k in zip(cs, ks)], (n_bits, key.engine)


@gpu
def test_even_modulus_and_empty_calls(built_lib):
    rng = random.Random(50)
    n = rng.getrandbits(128) | 1 << 127
    n &= ~1
    n2 = n * n
    cs = [rng.randrange(n2) for _ in range(5)]
    with PaillierKey(n, 3, 128, 64) as key:
        for fn in (lambda: key.invert(cs), lambda: key.sub(cs, cs), lambda: key.scalar_mul_signed(cs, [-1, 2, 3, 4, 5])):
            with pytest.raises(Pb200Error) as e:
                fn()
            assert e.value.status == _lib.PB200_ERR_EVEN_MODULUS
        # without signs the signed entry point is the plain scalar multiplication, which accepts an even n
        assert key.scalar_mul_signed(cs, [1, 2, 3, 4, 5]) == [pow(c, k, n2) for c, k in zip(cs, [1, 2, 3, 4, 5])]
        assert key.invert([]) == [] and key.sub([], []) == [] and key.scalar_mul_signed([], []) == []
        null = None
        assert key._lib.pb200_inverse_batch(key.handle, null, 0, null) == _lib.PB200_OK
        assert key._lib.pb200_sub_batch_dev(key.handle, null, null, 0, null) == _lib.PB200_OK
        assert key._lib.pb200_scalar_mul_signed_batch_dev(key.handle, null, null, null, 8, 0, null) == _lib.PB200_OK


@gpu
def test_dev_variants(built_lib):
    import torch
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(51)
    count = 300
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=51)
    c2_w = workload.ciphertexts(n_bits, count, n, seed_offset=52)
    mag_w = ints_to_words([rng.getrandbits(40) for _ in range(count)], 1)
    neg = np.array([rng.random() < 0.5 for _ in range(count)], dtype=np.uint8)
    with PaillierKey(n, g, n_bits, 64) as key:
        want_i, want_s = key.invert_words(c_w), key.sub_words(c_w, c2_w)
        want_k = key.scalar_mul_signed_words(c_w, mag_w, neg, 40)
        d_c, d_c2 = (torch.from_numpy(a.view(np.int64)).cuda() for a in (c_w, c2_w))
        d_m = torch.from_numpy(mag_w.view(np.int64)).cuda()
        d_neg = torch.from_numpy(neg).cuda()
        d_out = torch.empty_like(d_c)
        for _ in range(2):
            key.invert_dev(d_c.data_ptr(), count, d_out.data_ptr())
            assert key.take_flags() == 0 and (d_out.cpu().numpy().view(np.uint64) == want_i).all()
            key.sub_dev(d_c.data_ptr(), d_c2.data_ptr(), count, d_out.data_ptr())
            assert key.take_flags() == 0 and (d_out.cpu().numpy().view(np.uint64) == want_s).all()
            key.scalar_mul_signed_dev(d_c.data_ptr(), d_m.data_ptr(), d_neg.data_ptr(), 40, count, d_out.data_ptr())
            assert key.take_flags() == 0 and (d_out.cpu().numpy().view(np.uint64) == want_k).all()
        with pytest.raises(Pb200Error) as e:
            key.scalar_mul_signed_words(c_w, mag_w, neg, 39)
        assert e.value.status == _lib.PB200_ERR_RANGE
