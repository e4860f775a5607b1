"""Homomorphic scalar multiplication (c^k mod n^2, Dec = k m mod n) and the weighted tally (prod c_i^(k_i) = Enc(sum k_i m_i)):
bit-exact against OpenSSL (oracle/scalar_cpu.cpp) and Python pow on every engine and key size, homomorphic round trips through
decryption, the weighted tally's chunk boundaries, the device-pointer variants, argument checks and the SASS of the tcgen05
instantiations."""
import ctypes as C
import random
import re

import numpy as np
import pytest

from oracle import cpu_ref, scalar_oracle
from oracle.paillier_oracle import tally_native
from oracle.scalar_oracle import paillier_scalar_native, tally_weighted_native
from paillier_halo2_b200 import _lib, workload
from paillier_halo2_b200.api import PaillierKey, Pb200Error, ints_to_words, private_from_primes, words, words_to_ints

gpu = pytest.mark.gpu


def _oracle(n, c_w, k_w):
    """OpenSSL c^k mod n^2 per unit (keys whose n fills whole words: words_out = 2 words_in)"""
    return scalar_oracle.scalar_batch(n, c_w.shape[1] // 2, c_w, k_w, threads=cpu_ref.hardware_threads())


def _scalar_twice(key, c_w, k_w, k_bits):
    """every call runs twice with identical output (the CTAs' scratch slots are given back)"""
    a = key.scalar_mul_words(c_w, k_w, k_bits)
    b = key.scalar_mul_words(c_w, k_w, k_bits)
    assert (a == b).all()
    return a


def _edges(n, n_bits, wo, k_bits):
    """(c, k) pairs: k in {0, 1, 2, 2^k_bits - 1, n - 1 (when it fits)} x c in {0, 1, n^2 - 1, 2^(64 wo) - 1 (>= n^2)}"""
    ks = [0, 1, 2, (1 << k_bits) - 1] + ([n - 1] if (n - 1).bit_length() <= k_bits else [])
    cs = [0, 1, n * n - 1, (1 << (64 * wo)) - 1]
    return [(c, k) for c in cs for k in ks]


# ---- oracle parity ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n_bits,count", [(1024, 64 * 32 + 7), (2048, 64 * 16 + 7), (3072, 64 * 4 + 7), (4096, 64 * 4 + 7)])
def test_scalar_parity_vs_openssl(built_lib, n_bits, count):
    """ragged batch, random g, full-width scalars, edge scalars and ciphertexts in the middle of the batch; every unit against
    OpenSSL, a sample against Python pow"""
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    wo = 2 * n_bits // 64
    rng = random.Random(n_bits)
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=31)
    ks = [rng.getrandbits(n_bits) for _ in range(count)]
    edges = _edges(n, n_bits, wo, n_bits)
    c_w[100:100 + len(edges)] = ints_to_words([c for c, _ in edges], wo)
    ks[100:100 + len(edges)] = [k for _, k in edges]
    k_w = ints_to_words(ks, n_bits // 64)
    want = _oracle(n, c_w, k_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        got = _scalar_twice(key, c_w, k_w, n_bits)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, bad[:8]
    cs = words_to_ints(c_w)
    for u in [0, 1, 100, 101, 100 + len(edges) - 1, count - 1]:
        assert words_to_ints(got[u])[0] == pow(cs[u], ks[u], n * n), u


@gpu
def test_mixed_lengths_and_declared_widths(built_lib):
    """one full-width lane among short ones in the same CTA; declared k_bits in {1, 16, 32, 64, 65, n_bits}: every window width,
    one- and two-word scalar layouts"""
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(11)
    c_w = workload.ciphertexts(n_bits, 200, n, seed_offset=32)
    with PaillierKey(n, g, n_bits, 64) as key:
        ks = [rng.getrandbits(rng.choice([0, 1, 3, 9, 17])) for _ in range(200)]
        ks[37] = rng.getrandbits(n_bits) | (1 << (n_bits - 1))          # the CTA of lanes 32..63 runs the full chain
        ks[70] = 0
        k_w = ints_to_words(ks, n_bits // 64)
        assert (_scalar_twice(key, c_w, k_w, n_bits) == _oracle(n, c_w, k_w)).all()
        for k_bits in (1, 16, 32, 64, 65, n_bits):
            ks = [rng.getrandbits(k_bits) for _ in range(200)]
            ks[3], ks[4], ks[40] = (1 << k_bits) - 1, 0, 1 << (k_bits - 1)
            k_w = ints_to_words(ks, words(k_bits))
            got = _scalar_twice(key, c_w, k_w, k_bits)
            assert (got == _oracle(n, c_w, k_w)).all(), k_bits


@gpu
def test_every_engine_gives_identical_outputs(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(12)
    count = 64 * 3 + 7
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=33)
    ks = [rng.getrandbits(n_bits) for _ in range(count)]
    ks[:8] = [k for _, k in _edges(n, n_bits, 2 * n_bits // 64, n_bits)][:8]
    k_w = ints_to_words(ks, n_bits // 64)
    wk = ints_to_words([rng.getrandbits(32) for _ in range(count)], 1)
    want = _oracle(n, c_w, k_w)
    want_t = cpu_ref.tally(n, n_bits // 64, _oracle(n, c_w, wk), threads=8)
    ran = []
    with PaillierKey(n, g, n_bits, 64) as key:
        for engine in (1, 2, 3, 4, 5):
            try:
                key.set_engine(engine)
            except Pb200Error as e:
                assert e.status == _lib.PB200_ERR_UNSUPPORTED
                continue
            assert (_scalar_twice(key, c_w, k_w, n_bits) == want).all(), key.engine
            assert (key.tally_weighted_words(c_w, wk, 32) == want_t).all(), key.engine
            ran.append(key.engine)
    assert len(ran) >= 4, ran


@gpu
def test_simple64_path(built_lib):
    """reference-default key sizes (128 / 64, 264 / 88) on the automatic engine and on simple64, and a 1024-bit key forced to
    simple64"""
    rng = random.Random(13)
    cases = [(128, 64, rng.getrandbits(128) | 1 << 127 | 1), (264, 88, rng.getrandbits(264) | 1 << 263 | 1),
             (1024, 64, workload.load_key(1024)["n"])]
    for n_bits, limb_bits, n in cases:
        g = rng.getrandbits(n_bits)
        wo = words(2 * n_bits)
        edges = _edges(n, n_bits, wo, n_bits)
        cs = [c for c, _ in edges] + [rng.randrange(n * n) for _ in range(40)]
        ks = [k for _, k in edges] + [rng.getrandbits(n_bits) for _ in range(40)]
        want = [paillier_scalar_native(n, c, k) for c, k in zip(cs, ks)]
        with PaillierKey(n, g, n_bits, limb_bits) as key:
            for engine in ((0, 1) if n_bits < 1024 else (1,)):
                key.set_engine(engine)
                for _ in range(2):
                    assert key.scalar_mul(cs, ks) == want, (n_bits, key.engine)
                    assert key.tally_weighted(cs, ks) == tally_weighted_native(n, cs, ks), (n_bits, key.engine)


@pytest.mark.parametrize("g_kind", ["g_rand", "g_std"])
@gpu
def test_homomorphic_round_trips(built_lib, g_kind):
    """Dec(scalar_mul(Enc(m), k)) = k m mod n; Dec(tally_weighted(cs, ks)) = sum k_i m_i mod n with negative weights; all weights
    1 give the plain tally"""
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, p, q = kd["n"], kd["p"], kd["q"]
    g = kd["g_rand"] if g_kind == "g_rand" else n + 1
    rng = random.Random(14)
    m_w, r_w = workload.units(n_bits, 100, seed_offset=19)
    ms = words_to_ints(m_w)
    ks = [rng.getrandbits(rng.choice([1, 8, 32, 200, n_bits])) for _ in ms]
    ks[:4] = [0, 1, n - 1, -1]
    ws = [rng.randrange(-1000, 1000) for _ in ms]
    with PaillierKey(n, g, n_bits, 64) as key:
        key.set_private(*private_from_primes(p, q, g))
        cs = words_to_ints(key.encrypt_words(m_w, r_w))
        assert key.decrypt(key.scalar_mul(cs, ks)) == [k * m % n for k, m in zip(ks, ms)]
        t = key.tally_weighted(cs, ws)
        assert t == tally_weighted_native(n, cs, ws)
        assert key.decrypt([t]) == [sum(w * m for w, m in zip(ws, ms)) % n]
        assert key.tally_weighted(cs, [1] * len(cs)) == key.tally(cs) == tally_native(n, cs)
        assert key.tally_weighted([], []) == 1
        assert key.scalar_mul([], []) == []


@gpu
def test_weighted_tally_chunk_boundaries(built_lib):
    """counts around the 2^18-unit chunk of pb200_tally_weighted (|n| = 1024 keeps the host check short)"""
    n_bits = 1024
    kd = workload.load_key(n_bits)
    n, g, wi = kd["n"], kd["g_rand"], n_bits // 64
    total = (1 << 18) + 1
    c_w = workload.ciphertexts(n_bits, total, n, seed_offset=34)
    k_w = np.random.Generator(np.random.Philox(key=35)).integers(0, 1 << 16, size=(total, 1), dtype=np.uint64)
    prods = _oracle(n, c_w, k_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        for count in (0, 1, (1 << 18) - 1, 1 << 18, total):
            want = cpu_ref.tally(n, wi, prods[:count], threads=cpu_ref.hardware_threads()) if count else ints_to_words([1], 2 * wi)[0]
            for _ in range(2):
                assert (key.tally_weighted_words(c_w[:count], k_w[:count], 16) == want).all(), count


@gpu
def test_dev_variants_and_host_checks(built_lib):
    import torch
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(15)
    count = 300
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=36)
    k_w = ints_to_words([rng.getrandbits(100) for _ in range(count)], 2)
    with PaillierKey(n, g, n_bits, 64) as key:
        want = key.scalar_mul_words(c_w, k_w, 100)
        want_t = key.tally_weighted_words(c_w, k_w, 100)
        d_c = torch.from_numpy(c_w.view(np.int64)).cuda()
        d_k = torch.from_numpy(k_w.view(np.int64)).cuda()
        d_out = torch.empty((count, key.words_out), dtype=torch.int64, device="cuda")
        d_t = torch.empty(key.words_out, dtype=torch.int64, device="cuda")
        for _ in range(2):
            key.scalar_mul_dev(d_c.data_ptr(), d_k.data_ptr(), 100, count, d_out.data_ptr())
            key.tally_weighted_dev(d_c.data_ptr(), d_k.data_ptr(), 100, count, d_t.data_ptr())
            assert key.take_flags() == 0
            assert (d_out.cpu().numpy().view(np.uint64) == want).all()
            assert (d_t.cpu().numpy().view(np.uint64) == want_t).all()
        # argument checks on a live key: k_bits 0 / above n_bits, a scalar wider than declared
        for fn in (key._lib.pb200_scalar_mul_batch, key._lib.pb200_tally_weighted):
            for k_bits in (0, n_bits + 1):
                assert fn(key.handle, c_w.ctypes.data_as(_lib.u64p), k_w.ctypes.data_as(_lib.u64p), k_bits, 1,
                          np.empty(key.words_out * count, dtype="<u8").ctypes.data_as(_lib.u64p)) == _lib.PB200_ERR_INVALID_ARG
        with pytest.raises(Pb200Error) as e:
            key.scalar_mul_words(c_w, k_w, 99)
        assert e.value.status == _lib.PB200_ERR_RANGE
        with pytest.raises(Pb200Error) as e:
            key.tally_weighted_words(c_w, k_w, 99)
        assert e.value.status == _lib.PB200_ERR_RANGE


# ---- CPU-only ----------------------------------------------------------------------------------------------------------------------
def test_null_and_width_arguments_are_rejected(built_lib):
    lib = built_lib
    null = C.c_void_p()
    for k_bits in (1, 0, 1 << 20):
        assert lib.pb200_scalar_mul_batch(null, None, None, k_bits, 1, None) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_scalar_mul_batch_dev(null, None, None, k_bits, 1, None) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_tally_weighted(null, None, None, k_bits, 0, None) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_tally_weighted_dev(null, None, None, k_bits, 0, None) == _lib.PB200_ERR_INVALID_ARG


def test_oracles_agree():
    rng = random.Random(16)
    for n_bits in (128, 1024):
        n = rng.getrandbits(n_bits) | 1 << (n_bits - 1) | 1
        wi = n_bits // 64
        cs = [0, 1, n * n - 1, (1 << (128 * wi)) - 1] + [rng.randrange(n * n) for _ in range(30)]
        ks = [0, 1, n - 1, 2] + [rng.getrandbits(rng.choice([1, 17, n_bits])) % n for _ in range(30)]
        got = words_to_ints(scalar_oracle.scalar_batch(n, wi, ints_to_words(cs, 2 * wi), ints_to_words(ks, wi), threads=2))
        assert got == [paillier_scalar_native(n, c, k) for c, k in zip(cs, ks)] == [pow(c, k, n * n) for c, k in zip(cs, ks)]
        want = tally_native(n, got)
        assert tally_weighted_native(n, cs, ks) == want
        assert tally_weighted_native(n, cs, [k - n for k in ks]) == want       # k and k - n are the same weight
    assert tally_weighted_native(7, [], []) == 1


def test_scalar_kernels_are_tcgen05(built_lib):
    """the k_scalar<..., 2> instantiations at |n| = 2048 / 3072 / 4096 run their phases on tcgen05 (same parse as test_sass.py)"""
    import os
    import shutil
    import subprocess
    exe = next((c for c in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump") if c and os.path.exists(c)), None)
    if not exe:
        pytest.skip("cuobjdump not available")
    out = subprocess.run([exe, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    per, cur = {}, None
    for line in out.split("\n"):
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            per[cur] = {}
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,5}\*/\s+(?:@!?U?P\d\s+)?([A-Z][A-Z0-9_]*)", line)
        if cur and m:
            per[cur][m.group(1)] = per[cur].get(m.group(1), 0) + 1
    for g, bl in ((8, 19), (16, 14), (16, 19)):
        pat = re.compile(rf"\d+k_scalarINS_3b283CfgILi{g}ELi{bl}EEELi2EEEv")
        ks = [v for k, v in per.items() if pat.search(k)]
        assert len(ks) == 1, (g, bl)
        ops = ks[0]
        assert ops.get("UTCIMMA", 0) >= 8 and ops.get("LDTM", 0) >= 2 and ops.get("STTM", 0) >= 1 and ops.get("UTCBAR", 0) >= 2
        assert ops.get("IMMA", 0) == 0
