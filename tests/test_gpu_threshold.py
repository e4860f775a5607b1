"""Threshold decryption on the GPU: a trustee's partial decryption c^(2 Delta s_i) mod n^2 bit for bit against Python ints (every key size,
ragged counts, values at or above n^2, every engine, simple64 keys), the combination of t + 1 .. l shares in any order against decrypt
under set_private (fresh, tallied and matvec ciphertexts), too few or corrupted shares, the argument checks, and a key holding the
private part and a share together."""
import itertools
import random
from math import factorial

import numpy as np
import pytest

from paillier_halo2_b200 import _lib, workload
from paillier_halo2_b200.api import (PaillierKey, Pb200Error, ints_to_words, private_from_primes, threshold_from_primes, words,
                                     words_to_ints)

gpu = pytest.mark.gpu


def _values(n, n_bits, count, seed):
    """count words_out-word values: random below n^2, and edge values at or above n^2"""
    rng = random.Random(seed)
    top = 1 << (64 * words(2 * n_bits))
    edges = [0, 1, n, n * n - 1, n * n, n * n + 1, top - 1, top - n]
    return [v for v in edges if v < top] + [rng.randrange(n * n) for _ in range(count - len(edges))]


def _partials_all(key, shares, cs):
    """{i: trustee i's partial decryptions of cs}, one set_share per trustee on the same key"""
    out = {}
    for i, s in shares.items():
        key.set_share(i, s)
        out[i] = key.partial_decrypt(cs)
    return out


@gpu
@pytest.mark.parametrize("n_bits,count", [(1024, 64 * 4 + 7), (2048, 64 * 2 + 7), (3072, 64 + 7), (4096, 32 + 7)])
def test_partial_decrypt_parity(built_lib, n_bits, count):
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(n_bits)
    vals = _values(n, n_bits, count, n_bits)
    parties = 9
    s = rng.randrange(n * (n // 2))                          # a share is below n lambda
    e = 2 * factorial(parties) * s
    with PaillierKey(n, g, n_bits, 64) as key:
        key.set_threshold(parties, rng.randrange(1, n))
        key.set_share(4, s)
        got = key.partial_decrypt(vals)
        assert key.partial_decrypt(vals) == got
    assert got == [pow(v, e, n * n) for v in vals]


@gpu
def test_partial_decrypt_every_engine(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    vals = _values(n, n_bits, 64 + 9, 7)
    rng = random.Random(7)
    s = rng.getrandbits(64 * words(2 * n_bits))             # any words_out-word share
    want = [pow(v, 2 * factorial(5) * s, n * n) for v in vals]
    ran = []
    with PaillierKey(n, g, n_bits, 64) as key:
        key.set_threshold(5, 3)
        key.set_share(5, s)
        for engine in (1, 2, 3, 4, 5):
            try:
                key.set_engine(engine)
            except Pb200Error as e:
                assert e.status == _lib.PB200_ERR_UNSUPPORTED
                continue
            assert key.partial_decrypt(vals) == want, key.engine
            ran.append(key.engine)
    assert len(ran) >= 4, ran


@gpu
def test_partial_decrypt_simple64_and_short_keys(built_lib):
    rng = random.Random(8)
    cases = [(260, 65, rng.getrandbits(260) | 1 << 259 | 1), (1024, 64, rng.getrandbits(1000) | 1), (128, 64, rng.getrandbits(128) | 1 << 127 | 1)]
    for n_bits, limb_bits, n in cases:
        vals = _values(n, n_bits, 45, n_bits)
        s = rng.getrandbits(2 * n_bits)
        want = [pow(v, 2 * factorial(3) * s, n * n) for v in vals]
        with PaillierKey(n, rng.getrandbits(n_bits), n_bits, limb_bits) as key:
            key.set_threshold(3, 1)
            key.set_share(2, s)
            for engine in (0, 1):
                key.set_engine(engine)
                assert key.partial_decrypt(vals) == want, (n_bits, key.engine)
            if n_bits == 260:
                assert "simple64" in key.engine


def _setup(n_bits, which, t, parties, seed):
    kd = workload.load_key(n_bits)
    p, q, n = kd["p"], kd["q"], kd["n"]
    g = kd["g_rand"] if which == "rand" else n + 1
    shares, phi = threshold_from_primes(p, q, g, t, parties, rng=random.Random(seed))
    return kd, n, g, shares, phi


@gpu
def test_combination_recovers_the_plaintexts(built_lib):
    n_bits = 2048
    rng = random.Random(11)
    for which, t, parties in (("rand", 2, 5), ("std", 4, 9)):
        kd, n, g, shares, phi = _setup(n_bits, which, t, parties, 11 + parties)
        count = 37
        ms = [rng.randrange(n) for _ in range(count - 3)] + [0, 1, n - 1]
        rs = [rng.randrange(1, n) for _ in ms]
        with PaillierKey(n, g, n_bits, 64) as key:
            cs = key.paillier_enc_native(ms, rs)
            # a tally and two rows of a signed matvec ride along
            W = [[rng.randrange(-1000, 1000) for _ in cs[:10]] for _ in range(2)]
            extra = [key.tally(cs[:10])] + key.matvec(cs[:10], W)
            cs_all = cs + extra
            lam, mu = private_from_primes(kd["p"], kd["q"], g)
            key.set_private(lam, mu)
            want = key.decrypt(cs_all)
            assert want[:count] == ms
            assert want[count] == sum(ms[:10]) % n
            assert want[count + 1:] == [sum(w * m for w, m in zip(row, ms[:10])) % n for row in W]
            key.set_threshold(parties, phi)
            parts = _partials_all(key, shares, cs_all)
            sets = [list(s) for s in itertools.combinations(range(1, parties + 1), t + 1)]
            if parties == 9:
                sets = [sorted(rng.sample(range(1, 10), t + 1)) for _ in range(4)]
            sets.append(list(range(1, parties + 1)))
            for s in sets:
                rng.shuffle(s)
                assert key.combine_shares(s, [parts[i] for i in s]) == want, (which, s)
            # the key's private part is untouched by the threshold set-up
            assert key.decrypt(cs_all) == want


@gpu
def test_combination_every_engine_and_simple64(built_lib):
    n_bits = 2048
    kd, n, g, shares, phi = _setup(n_bits, "rand", 2, 5, 12)
    rng = random.Random(12)
    ms = [rng.randrange(n) for _ in range(33)]
    ran = []
    with PaillierKey(n, g, n_bits, 64) as key:
        cs = key.paillier_enc_native(ms, [rng.randrange(1, n) for _ in ms])
        key.set_threshold(5, phi)
        parts = _partials_all(key, shares, cs)
        for engine in (1, 2, 3, 4, 5):
            try:
                key.set_engine(engine)
            except Pb200Error:
                continue
            for s in ([5, 1, 3], [2, 4, 1, 5, 3]):
                assert key.combine_shares(s, [parts[i] for i in s]) == ms, (key.engine, s)
            ran.append(key.engine)
    assert len(ran) >= 4, ran
    # a key on simple64 only (256 bits on engine 1) and the smallest key on the block engine
    for n_bits in (128, 256):
        kd, n, g, shares, phi = _setup(n_bits, "std", 1, 3, n_bits)
        ms = [rng.randrange(n) for _ in range(20)]
        with PaillierKey(n, g, n_bits, 64) as key:
            cs = key.paillier_enc_native(ms, [rng.randrange(1, n) for _ in ms])
            key.set_threshold(3, phi)
            for engine in (0, 1):
                key.set_engine(engine)
                parts = _partials_all(key, shares, cs)
                for s in ([1, 2], [3, 1], [2, 3], [1, 2, 3]):
                    assert key.combine_shares(s, [parts[i] for i in s]) == ms, (n_bits, key.engine, s)


@gpu
def test_too_few_and_corrupted_shares(built_lib):
    import torch

    n_bits = 2048
    t, parties = 2, 5
    kd, n, g, shares, phi = _setup(n_bits, "rand", t, parties, 13)
    rng = random.Random(13)
    ms = [rng.randrange(n) for _ in range(40)]
    with PaillierKey(n, g, n_bits, 64) as key:
        cs = key.paillier_enc_native(ms, [rng.randrange(1, n) for _ in ms])
        key.set_threshold(parties, phi)
        parts = _partials_all(key, shares, cs)
        few = [2, 5]
        w = np.stack([ints_to_words(parts[i], key.words_out) for i in few])
        with pytest.raises(Pb200Error) as e:
            key.combine_shares_words(few, w)
        assert e.value.status == _lib.PB200_ERR_DECRYPT
        assert e.value.outputs.shape == (len(ms), key.words_in) and not e.value.outputs.any()
        d_w = torch.from_numpy(w.reshape(-1).view(np.int64)).cuda()
        d_m = torch.empty((len(ms), key.words_in), dtype=torch.int64, device="cuda")
        key.combine_shares_dev(few, d_w.data_ptr(), len(ms), d_m.data_ptr())
        assert key.take_flags() == _lib.PB200_FLAG_DECRYPT
        # the flag does not leak into the next host call
        s = [1, 3, 4]
        assert key.combine_shares(s, [parts[i] for i in s]) == ms
        # one unit's share replaced by 0: that unit fails, the others are still recovered
        for bad in (1, 3):                                    # mu_1 > 0 (P = 0), mu_3 < 0 in {1, 3, 4} (N = 0, no inverse)
            sh = {i: list(parts[i]) for i in s}
            sh[bad][7] = 0
            with pytest.raises(Pb200Error) as e:
                key.combine_shares(s, [sh[i] for i in s])
            assert e.value.status in (_lib.PB200_ERR_NOT_INVERTIBLE, _lib.PB200_ERR_DECRYPT)
            out = words_to_ints(e.value.outputs)
            assert out[7] == 0 and out[:7] + out[8:] == ms[:7] + ms[8:]


@gpu
def test_argument_checks(built_lib):
    kd = workload.load_key(1024)
    n, g = kd["n"], kd["g_rand"]
    lib = _lib.load()
    wi, wo = words(1024), words(2048)
    one_in, one_out = ints_to_words([1], wi), ints_to_words([1], wo)
    P = lambda a: a.ctypes.data_as(_lib.u64p)          # noqa: E731
    idx = lambda *v: np.array(v, dtype=np.uint32).ctypes.data_as(__import__("ctypes").c_void_p)      # noqa: E731
    sh = ints_to_words([1] * 4, wo)
    out = np.zeros((2, wi), dtype="<u8")
    with PaillierKey(n, g, 1024, 64) as key:
        h = key.handle
        assert lib.pb200_key_set_share(h, 1, P(one_out)) == _lib.PB200_ERR_INVALID_ARG               # before set_threshold
        assert lib.pb200_combine_shares_batch(h, idx(1, 2), 2, P(sh), 2, P(out)) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_partial_decrypt_batch(h, P(one_out), 1, P(one_out.copy())) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_key_set_threshold(h, 0, P(one_in)) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_key_set_threshold(h, 33, P(one_in)) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_key_set_threshold(h, 3, None) == _lib.PB200_ERR_INVALID_ARG
        big = np.zeros(wi, dtype="<u8")
        big[-1] = 1 << 63
        assert lib.pb200_key_set_threshold(h, 3, P(big)) == _lib.PB200_OK               # 2^1023 < 2^n_bits fits
        with pytest.raises(Pb200Error) as e:
            key.set_threshold(3, 1 << 1024)
        assert e.value.status == _lib.PB200_ERR_RANGE
        assert lib.pb200_key_set_threshold(h, 3, P(one_in)) == _lib.PB200_OK
        for i in (0, 4):
            assert lib.pb200_key_set_share(h, i, P(one_out)) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_partial_decrypt_batch(h, P(one_out), 1, P(one_out.copy())) == _lib.PB200_ERR_INVALID_ARG    # no share yet
        assert lib.pb200_key_set_share(h, 3, P(one_out)) == _lib.PB200_OK
        assert lib.pb200_partial_decrypt_batch(h, None, 0, None) == _lib.PB200_OK
        for args in ((idx(1, 2), 0), (idx(0, 2), 2), (idx(1, 4), 2), (idx(2, 2), 2), (None, 2)):
            assert lib.pb200_combine_shares_batch(h, args[0], args[1], P(sh), 2, P(out)) == _lib.PB200_ERR_INVALID_ARG, args
            assert lib.pb200_combine_shares_batch_dev(h, args[0], args[1], None, 0, None) == _lib.PB200_ERR_INVALID_ARG, args
        assert lib.pb200_combine_shares_batch(h, idx(1, 2), 2, None, 0, None) == _lib.PB200_OK          # count == 0
        # set_threshold clears the share
        assert lib.pb200_key_set_threshold(h, 3, P(one_in)) == _lib.PB200_OK
        assert lib.pb200_partial_decrypt_batch(h, P(one_out), 1, P(one_out.copy())) == _lib.PB200_ERR_INVALID_ARG
    # an even n: only sets with a negative coefficient need the inverse
    rng = random.Random(14)
    ne = (rng.getrandbits(128) | 1 << 127) & ~1
    with PaillierKey(ne, 3, 128, 64) as key:
        key.set_threshold(3, 1)
        w = ints_to_words([5, 7], words(256))
        for s, status in (([1, 2], _lib.PB200_ERR_EVEN_MODULUS), ([2, 1], _lib.PB200_ERR_EVEN_MODULUS)):
            with pytest.raises(Pb200Error) as e:
                key.combine_shares_words(s, np.stack([w[:1], w[1:]]))
            assert e.value.status == status
        try:
            key.combine_shares_words([1], w[:1].reshape(1, 1, -1))                    # mu_1 = Delta > 0: no inverse
        except Pb200Error as e:
            assert e.status == _lib.PB200_ERR_DECRYPT


@gpu
def test_set_share_keeps_decrypt_and_dev_variants(built_lib):
    import torch

    n_bits = 3072
    kd, n, g, shares, phi = _setup(n_bits, "rand", 1, 3, 15)
    rng = random.Random(15)
    count = 64 + 5
    ms = [rng.randrange(n) for _ in range(count)]
    with PaillierKey(n, g, n_bits, 64) as key:
        cs = key.paillier_enc_native(ms, [rng.randrange(1, n) for _ in ms])
        key.set_private(*private_from_primes(kd["p"], kd["q"], g))
        c_w = ints_to_words(cs, key.words_out)
        before = key.decrypt_words(c_w)
        key.set_threshold(3, phi)
        key.set_share(2, shares[2])
        assert (key.decrypt_words(c_w) == before).all()
        # _dev: partial decryption and combination from device memory equal the host calls
        d_c = torch.from_numpy(c_w.view(np.int64)).cuda()
        parts = {}
        for i in (3, 1):
            key.set_share(i, shares[i])
            d_p = torch.empty_like(d_c)
            key.partial_decrypt_dev(d_c.data_ptr(), count, d_p.data_ptr())
            key.sync()
            parts[i] = d_p.cpu().numpy().view("<u8")
            assert (parts[i] == key.partial_decrypt_words(c_w)).all()
        d_sh = torch.from_numpy(np.stack([parts[3], parts[1]]).reshape(-1).view(np.int64)).cuda()
        d_m = torch.empty((count, key.words_in), dtype=torch.int64, device="cuda")
        for _ in range(2):                                     # the second call reuses the cached plan
            key.combine_shares_dev([3, 1], d_sh.data_ptr(), count, d_m.data_ptr())
            assert key.take_flags() == 0
            assert words_to_ints(d_m.cpu().numpy().view("<u8")) == ms
        assert (key.decrypt_words(c_w) == before).all()
