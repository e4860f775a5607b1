"""Encrypted matrix-vector product with a signed plaintext matrix (pb200_matvec): bit-exact against OpenSSL (tests/matvec_cpu.cpp) and
Python pow on every key size, both methods and every engine; the bucket method's edge cases (one bucket over many CTAs, every bucket
once, digits on segment boundaries, multi-pass); parity with the weighted tally; decryption round trips; the device variant; the
planner's choices and memory budget; argument checks and the SASS of the tcgen05 instantiations."""
import ctypes as C
import random
import re

import numpy as np
import pytest

from oracle import cpu_ref
from oracle.paillier_oracle import tally_native
from paillier_halo2_b200 import _lib, workload
from paillier_halo2_b200.api import (PaillierKey, Pb200Error, ints_to_words, matvec_budget, matvec_plan, matvec_weights,
                                     private_from_primes, words_to_ints)

import matvec_oracle
from matvec_oracle import matvec_native

gpu = pytest.mark.gpu


def _oracle(n, c_w, mag, neg):
    return matvec_oracle.matvec(n, c_w.shape[1] // 2, c_w, mag, neg, threads=cpu_ref.hardware_threads())


def _run(key, c_w, mag, neg, k_bits, monkeypatch=None, method=None):
    """two calls with identical output (repeatability), optionally with the method forced"""
    if monkeypatch is not None:
        if method:
            monkeypatch.setenv("PB200_MATVEC_METHOD", method)
        else:
            monkeypatch.delenv("PB200_MATVEC_METHOD", raising=False)
    a = key.matvec_words(c_w, mag, neg, k_bits)
    b = key.matvec_words(c_w, mag, neg, k_bits)
    assert (a == b).all()
    return a


def _signed(W):
    """rows of Python ints -> (magnitude words, signs, k_bits)"""
    return matvec_weights(W, len(W[0]))


def _edge_matrix(rng, n, n_bits, count, rows, k_bits):
    """random signed weights below 2^k_bits with: an all-zero row, an all-zero column, magnitudes 2^k_bits - 1, an all-negative
    row, and (for the caller's ciphertexts) a repeated ciphertext"""
    top = (1 << k_bits) - 1
    W = [[rng.randint(-top, top) for _ in range(count)] for _ in range(rows)]
    W[0] = [0] * count
    for r in range(rows):
        W[r][3] = 0
        W[r][5] = top if r % 2 else -top
    W[2] = [-rng.randint(1, top) for _ in range(count)]
    return W


def _edge_ciphertexts(n_bits, count, n, wo, seed):
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=seed)
    c_w[7:11] = ints_to_words([0, 1, n * n - 1, (1 << (64 * wo)) - 1], wo)
    c_w[12] = c_w[13]                                                   # a repeated ciphertext
    return c_w


# ---- oracle parity ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n_bits", [1024, 2048, 3072, 4096])
def test_matvec_parity_vs_openssl(built_lib, n_bits, monkeypatch):
    """ragged count, several rows, k_bits in {1, 8, 32, 64, n_bits}, signed weights with edge rows and columns, edge ciphertexts;
    the automatic plan and both forced methods against OpenSSL, one row against Python pow"""
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    wo = 2 * n_bits // 64
    rng = random.Random(n_bits + 1)
    count, rows = 77, 4
    c_w = _edge_ciphertexts(n_bits, count, n, wo, 41)
    cs = words_to_ints(c_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        for k_bits in (1, 8, 32, 64, n_bits):
            W = _edge_matrix(rng, n, n_bits, count, rows, k_bits)
            mag, neg, kb = _signed(W)
            assert kb == k_bits
            want = _oracle(n, c_w, mag, neg)
            for method in (None, "chain", "bucket"):
                got = _run(key, c_w, mag, neg, k_bits, monkeypatch, method)
                bad = np.nonzero((got != want).any(axis=1))[0]
                assert bad.size == 0, (k_bits, method, bad)
            if k_bits <= 64:
                assert words_to_ints(want[1])[0] == matvec_native(n, cs, [W[1]])[0]


@gpu
def test_every_engine_gives_identical_outputs(built_lib, monkeypatch):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(51)
    count, rows = 64 * 3 + 7, 5
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=42)
    W = [[rng.randint(-(1 << 16) + 1, (1 << 16) - 1) for _ in range(count)] for _ in range(rows)]
    mag, neg, k_bits = _signed(W)
    want = _oracle(n, c_w, mag, neg)
    ran = []
    with PaillierKey(n, g, n_bits, 64) as key:
        for engine in (0, 1, 2, 3, 4, 5):
            try:
                key.set_engine(engine)
            except Pb200Error as e:
                assert e.status == _lib.PB200_ERR_UNSUPPORTED
                continue
            for method in ("chain", "bucket"):
                assert (_run(key, c_w, mag, neg, k_bits, monkeypatch, method) == want).all(), (key.engine, method)
            ran.append(key.engine)
    assert len(ran) >= 5, ran


@gpu
def test_reference_key_sizes_and_simple64(built_lib):
    """the reference's default key sizes on the automatic engine and on simple64 (which always takes the chain method), and a key
    size no block engine covers, against Python pow"""
    rng = random.Random(52)
    for n_bits, limb_bits in ((128, 64), (264, 88), (260, 65)):
        n = rng.getrandbits(n_bits) | 1 << (n_bits - 1) | 1
        g = rng.getrandbits(n_bits)
        cs = [0, 1, n * n - 1] + [rng.randrange(n * n) for _ in range(20)]
        W = [[rng.randint(-50, 50) for _ in cs] for _ in range(3)] + [[-1] * len(cs), [rng.getrandbits(n_bits) for _ in cs]]
        with PaillierKey(n, g, n_bits, limb_bits) as key:
            for engine in (0, 1):
                key.set_engine(engine)
                for _ in range(2):
                    assert key.matvec(cs, W) == matvec_native(n, cs, W), (n_bits, key.engine)


# ---- bucket method edge cases ----------------------------------------------------------------------------------------------------
@gpu
def test_bucket_edge_cases(built_lib, monkeypatch):
    """all weights 1 (one bucket over many CTAs and carry levels; the oracle is the plain tally), every bucket of the window used once,
    digits on the reducer's segment boundaries, and multi-pass runs forced by PB200_MATVEC_PASS_ENTRIES"""
    n_bits = 1024
    kd = workload.load_key(n_bits)
    n, g, wi = kd["n"], kd["g_rand"], n_bits // 64
    rng = random.Random(53)
    monkeypatch.setenv("PB200_MATVEC_METHOD", "bucket")
    with PaillierKey(n, g, n_bits, 64) as key:
        count = 20000
        c_w = workload.ciphertexts(n_bits, count, n, seed_offset=43)
        ones = np.ones((1, count), dtype=np.int64)
        got = key.matvec_words(c_w, *matvec_weights(ones, count)[:2], 1)
        assert (got[0] == cpu_ref.tally(n, wi, c_w, threads=cpu_ref.hardware_threads())).all()
        # every 8-bit digit value once (at c = 8 every bucket holds one ciphertext)
        count = 255
        c_w = workload.ciphertexts(n_bits, count, n, seed_offset=44)
        perm = list(range(1, 256))
        rng.shuffle(perm)
        W = [perm, [-v for v in perm]]
        mag, neg, k_bits = _signed(W)
        assert (_run(key, c_w, mag, neg, k_bits) == _oracle(n, c_w, mag, neg)).all()
        # every digit on a segment boundary of the plan in use (sms: the SM count the call plans with)
        import torch
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        for k_bits in (8, 16):
            p = matvec_plan(n_bits, sms, 2, 300, k_bits, True)
            assert p["method"] == 1
            c, J = p["c"], p["windows"]
            lseg = -(-((1 << c) - 1) // p["segments"])
            marks = sorted({v for s in range(p["segments"]) for v in (1 + s * lseg, min(s * lseg + lseg, (1 << c) - 1))})
            ws = [sum(marks[(i + j) % len(marks)] << (c * j) for j in range(J)) & ((1 << k_bits) - 1) for i in range(300)]
            W = [ws, [-w for w in ws[::-1]]]
            c_w = workload.ciphertexts(n_bits, 300, n, seed_offset=45)
            mag, neg, kb = _signed(W)
            assert (_run(key, c_w, mag, neg, kb) == _oracle(n, c_w, mag, neg)).all(), k_bits
        # multi-pass: a few hundred entries per pass over rows, windows and ciphertext chunks
        count, rows = 500, 3
        c_w = workload.ciphertexts(n_bits, count, n, seed_offset=46)
        W = [[rng.randint(-(1 << 40), 1 << 40) for _ in range(count)] for _ in range(rows)]
        mag, neg, k_bits = _signed(W)
        want = _oracle(n, c_w, mag, neg)
        for pe in ("200", "1500", "100000"):
            monkeypatch.setenv("PB200_MATVEC_PASS_ENTRIES", pe)
            assert matvec_plan(n_bits, sms, rows, count, k_bits, True)["passes"] >= (2 if pe != "100000" else 1)
            assert (_run(key, c_w, mag, neg, k_bits) == want).all(), pe


@gpu
def test_parity_with_weighted_tally(built_lib):
    """rows without negative weights equal pb200_tally_weighted bit for bit, across its 2^18-ciphertext chunk boundary"""
    n_bits = 1024
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    count = (1 << 18) + 5
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=47)
    W = np.random.Generator(np.random.Philox(key=48)).integers(0, 1 << 32, size=(2, count), dtype=np.uint64)
    with PaillierKey(n, g, n_bits, 64) as key:
        mag, neg, k_bits = matvec_weights(W, count)
        assert neg is None and k_bits == 32
        got = key.matvec_words(c_w, mag, None, k_bits)
        for r in range(2):
            assert (got[r] == key.tally_weighted_words(c_w, mag[r], k_bits)).all(), r


@pytest.mark.parametrize("g_kind", ["g_rand", "g_std"])
@gpu
def test_decryption_round_trips(built_lib, g_kind):
    """Dec(matvec(Enc(m), W)) = W m mod n for rows of Python ints (any sign and size) and for numpy matrices; empty shapes"""
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, p, q = kd["n"], kd["p"], kd["q"]
    g = kd["g_rand"] if g_kind == "g_rand" else n + 1
    rng = random.Random(54)
    m_w, r_w = workload.units(n_bits, 120, seed_offset=20)
    ms = words_to_ints(m_w)
    W = [[rng.randint(-1000, 1000) for _ in ms] for _ in range(4)] + [[-1] * len(ms), [rng.getrandbits(300) for _ in ms]]
    Wn = np.random.Generator(np.random.Philox(key=49)).integers(-(1 << 62), 1 << 62, size=(3, len(ms)), dtype=np.int64)
    Wn[0, 0] = np.iinfo(np.int64).min
    with PaillierKey(n, g, n_bits, 64) as key:
        key.set_private(*private_from_primes(p, q, g))
        cs = words_to_ints(key.encrypt_words(m_w, r_w))
        got = key.matvec(cs, W)
        assert got == matvec_native(n, cs, W)
        assert key.decrypt(got) == [sum(w * m for w, m in zip(row, ms)) % n for row in W]
        gn = key.matvec(cs, Wn)
        assert gn == key.matvec(cs, Wn.tolist())
        assert key.decrypt(gn) == [sum(int(w) * m for w, m in zip(row, ms)) % n for row in Wn]
        assert key.matvec(cs, [[1] * len(cs)]) == [key.tally(cs)] == [tally_native(n, cs)]
        assert key.matvec([], [[], []]) == [1, 1]
        assert key.matvec(cs, []) == []


@gpu
def test_dev_variant_and_flags(built_lib):
    """pb200_matvec_dev gives the host variant's output and leaves the flag word clean; a sign vector of zeros runs the sign step
    and changes nothing"""
    import torch
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(55)
    count, rows = 300, 3
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=50)
    W = [[rng.randint(-(1 << 20), 1 << 20) for _ in range(count)] for _ in range(rows)]
    mag, neg, k_bits = _signed(W)
    with PaillierKey(n, g, n_bits, 64) as key:
        want = key.matvec_words(c_w, mag, neg, k_bits)
        pos = key.matvec_words(c_w, mag, None, k_bits)
        d_c = torch.from_numpy(c_w.view(np.int64)).cuda()
        d_w = torch.from_numpy(mag.view(np.int64)).cuda()
        d_neg = torch.from_numpy(neg).cuda()
        d_zero = torch.zeros_like(d_neg)
        d_out = torch.empty((rows, key.words_out), dtype=torch.int64, device="cuda")
        for _ in range(2):
            key.matvec_dev(d_c.data_ptr(), count, d_w.data_ptr(), d_neg.data_ptr(), k_bits, rows, d_out.data_ptr())
            key.sync()
            assert key.take_flags() == 0
            assert (d_out.cpu().numpy().view(np.uint64) == want).all()
            key.matvec_dev(d_c.data_ptr(), count, d_w.data_ptr(), d_zero.data_ptr(), k_bits, rows, d_out.data_ptr())
            key.sync()
            assert key.take_flags() == 0
            assert (d_out.cpu().numpy().view(np.uint64) == pos).all()
        with pytest.raises(Pb200Error) as e:
            key.matvec_words(c_w, mag, neg, k_bits - 1)
        assert e.value.status == _lib.PB200_ERR_RANGE
        for kb in (0, n_bits + 1):
            assert key._lib.pb200_matvec(key.handle, c_w.ctypes.data_as(_lib.u64p), count, mag.ctypes.data_as(_lib.u64p), None, kb, rows,
                                         np.empty(rows * key.words_out, dtype="<u8").ctypes.data_as(_lib.u64p)) == _lib.PB200_ERR_INVALID_ARG


# ---- CPU-only ----------------------------------------------------------------------------------------------------------------------
def test_planner_stays_within_the_budget(monkeypatch):
    """extreme shapes, both methods forced, with and without signs"""
    shapes = [(4096, 1, 1 << 32, 4096), (2048, 1 << 20, 2, 32), (2048, 1, 1 << 20, 2048), (2048, 256, 4096, 16), (1024, 1 << 16, 1 << 16, 1),
              (3072, 7, 1 << 24, 64)]
    for method in (None, "chain", "bucket"):
        if method:
            monkeypatch.setenv("PB200_MATVEC_METHOD", method)
        for n_bits, rows, count, k_bits in shapes:
            for has_neg in (False, True):
                p = matvec_plan(n_bits, 148, rows, count, k_bits, has_neg)
                assert 0 < p["temp_bytes"] <= matvec_budget(n_bits), (method, n_bits, rows, count, k_bits, has_neg, p)
                assert p["method"] == (0 if method == "chain" else 1 if method == "bucket" else p["method"])
                if p["method"] == 1:
                    assert 1 <= p["c"] <= 16 and p["windows"] == -(-k_bits // p["c"]) and p["segments"] >= 1
                    assert p["acc_mulmods"] >= rows * count * p["windows"]
                    assert (p["sign_mulmods"] > 0) == has_neg
    assert matvec_budget(2048) == 384 << 20
    assert matvec_plan(2048, 148, 0, 10, 32, True)["temp_bytes"] == matvec_plan(2048, 148, 10, 0, 32, True)["temp_bytes"] == 0


def test_planner_picks_chain_for_tiny_and_bucket_for_large(monkeypatch):
    monkeypatch.delenv("PB200_MATVEC_METHOD", raising=False)
    monkeypatch.delenv("PB200_MATVEC_PASS_ENTRIES", raising=False)
    assert matvec_plan(2048, 148, 1, 2, 32, False)["method"] == 0
    for k_bits, has_neg in ((32, False), (2048, False), (1, True), (16, True)):
        p = matvec_plan(2048, 148, 1, 1 << 20, k_bits, has_neg)
        assert p["method"] == 1, (k_bits, p)
        assert p["acc_mulmods"] + p["reduce_mulmods"] + p["horner_mulmods"] < (1 << 20) * (k_bits + 1), p
    assert matvec_plan(2048, 148, 256, 4096, 16, True)["method"] == 1
    # keys the block engine does not cover always take the chain
    assert matvec_plan(260, 148, 1, 1 << 20, 32, False)["method"] == 0


def test_pass_entries_switch_changes_the_passes(monkeypatch):
    monkeypatch.setenv("PB200_MATVEC_METHOD", "bucket")
    monkeypatch.delenv("PB200_MATVEC_PASS_ENTRIES", raising=False)
    base = matvec_plan(2048, 148, 4, 10000, 64, True)
    monkeypatch.setenv("PB200_MATVEC_PASS_ENTRIES", "1000")
    small = matvec_plan(2048, 148, 4, 10000, 64, True)
    assert base["passes"] == 1 and small["passes"] > base["passes"]


def test_matvec_arguments_are_rejected(built_lib):
    lib = built_lib
    null = C.c_void_p()
    for k_bits in (1, 0, 1 << 20):
        assert lib.pb200_matvec(null, None, 0, None, None, k_bits, 1, None) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_matvec_dev(null, None, 0, None, None, k_bits, 1, None) == _lib.PB200_ERR_INVALID_ARG
    out = np.zeros(11, dtype="<u8")
    for n_bits, k_bits, sms in ((2048, 0, 148), (2048, 2049, 148), (0, 1, 148), (2048, 32, 0)):
        assert lib.pb200_matvec_plan(n_bits, sms, 1, 1, k_bits, 0, out.ctypes.data_as(_lib.u64p)) == _lib.PB200_ERR_INVALID_ARG
    assert lib.pb200_matvec_plan(2048, 148, 1, 1, 32, 0, None) == _lib.PB200_ERR_INVALID_ARG


def test_weight_conversion_and_oracles_agree():
    W = np.array([[3, -5, 0], [np.iinfo(np.int64).min, 1, -1]], dtype=np.int64)
    mag, neg, k_bits = matvec_weights(W, 3)
    assert k_bits == 64 and mag.shape == (2, 3, 1)
    assert mag.reshape(2, 3).tolist() == [[3, 5, 0], [1 << 63, 1, 1]] and neg.tolist() == [[0, 1, 0], [1, 0, 1]]
    m2, n2, k2 = matvec_weights(W.tolist(), 3)
    assert (m2 == mag).all() and (n2 == neg).all() and k2 == k_bits
    mu, nu, ku = matvec_weights(np.array([[1, 2], [3, 4]], dtype=np.uint8), 2)
    assert nu is None and ku == 3
    with pytest.raises(ValueError):
        matvec_weights([[1, 2]], 3)
    rng = random.Random(56)
    for n_bits in (128, 1024):
        n = rng.getrandbits(n_bits) | 1 << (n_bits - 1) | 1
        wi = n_bits // 64
        cs = [0, 1, n * n - 1, (1 << (128 * wi)) - 1] + [rng.randrange(n * n) for _ in range(30)]
        W = [[rng.randint(-(1 << 70), 1 << 70) for _ in cs] for _ in range(3)] + [[0] * len(cs), [-3] * len(cs)]
        mag, neg, k_bits = matvec_weights(W, len(cs))
        got = words_to_ints(matvec_oracle.matvec(n, wi, ints_to_words(cs, 2 * wi), mag, neg, threads=3))
        want = matvec_native(n, cs, W)
        assert got == want
        n2 = n * n
        for row, v in zip(W, want):
            t = 1
            for c, w in zip(cs, row):
                t = t * pow(c, w % n, n2) % n2
            assert v == t                      # c^(n - s) and c^(-s) * ... agree: N^(n-1) is the product with weights n - |w|
    assert words_to_ints(matvec_oracle.matvec(7, 1, np.zeros((0, 2), dtype="<u8"), np.zeros((2, 0, 1), dtype="<u8"), None)) == [1, 1]


def test_matvec_kernels_are_tcgen05(built_lib):
    """the k_bucket_fold / k_bucket_reduce / k_horner / k_lazy_canon instantiations for the tcgen05 engine (tally shape, ENG 4) at
    |n| = 2048 / 3072 / 4096 run their phases on tcgen05 (same parse as test_sass.py)"""
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
    for name in ("k_bucket_fold", "k_bucket_reduce", "k_horner", "k_lazy_canon"):
        for g, bl in ((8, 19), (16, 14), (16, 19)):
            pat = re.compile(rf"\d+{name}INS_3b283CfgILi{g}ELi{bl}EEELi4EEEv")
            ks = [v for k, v in per.items() if pat.search(k)]
            assert len(ks) == 1, (name, g, bl)
            ops = ks[0]
            assert ops.get("UTCIMMA", 0) >= 8 and ops.get("LDTM", 0) >= 2 and ops.get("UTCBAR", 0) >= 2, (name, g, bl)
            assert ops.get("IMMA", 0) == 0
