"""Running-tally trace (pb200_tally_trace): every step (q_i, acc_i) = divmod(acc_(i-1) * c_i, n^2) of every chain, bit-exact against
the Python chain below on every key size, chunk partition and engine; unreduced inputs and the range check; consistency with
pb200_tally and pb200_add_batch; the (q, rem) pairs satisfy the chip's constraints and feed pb200_mulmod_cells_batch through the
contiguous-operand layout; decryption round trips; the device variant; argument checks and the SASS of the new kernels."""
import ctypes as C
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle.paillier_oracle import BigUintChip, Context, EncryptionPublicKeyAssigned, PaillierChip, check_constraints
from paillier_halo2_b200 import _lib, workload
from paillier_halo2_b200.api import PaillierKey, Pb200Error, ints_to_words, private_from_primes, words_to_ints

gpu = pytest.mark.gpu


def trace_native(n, inits, rows):
    """the oracle: per chain j, a = init_j, then (q, a) = divmod(a * c_ij, n^2) for every row i; returns (acc, q) shaped like rows"""
    n2 = n * n
    a = list(inits)
    acc, qs = [], []
    for row in rows:
        qa = [divmod(x * c, n2) for x, c in zip(a, row)]
        qs.append([q for q, _ in qa])
        a = [r for _, r in qa]
        acc.append(list(a))
    return acc, qs


def _rows(rng, n, count, chains, edges=True):
    """random ciphertexts below n^2 with the edge values 1, n^2 - 1 and n spread over the steps and chains, and 0 at the last step
    of chain 0 (a 0 earlier would force every later carry of its chain to 0)"""
    n2 = n * n
    rows = [[rng.randrange(n2) for _ in range(chains)] for _ in range(count)]
    if edges:
        for t, v in enumerate((1, n2 - 1, n)):
            i = (t * 7919) % count
            rows[i][(t + 1) % chains] = v
        rows[count - 1][0] = 0
    return rows


def _check(key, n, inits, rows, want_q=True):
    acc, q = key.tally_trace(inits, rows, want_q=True)
    wa, wq = trace_native(n, inits, rows)
    assert acc == wa
    assert q == wq
    if not want_q:
        assert key.tally_trace(inits, rows, want_q=False) == wa
    return acc, q


# ---- oracle parity ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n_bits", [1024, 2048, 3072, 4096])
def test_trace_parity(built_lib, n_bits, monkeypatch):
    """chains 1, 3, 33; step counts around the chunk length s and around one wave of lanes (a small wave through PB200_TRACE_LANES,
    so the chunking and every scan level are crossed with few steps), a few thousand + 7 on the default wave; edge ciphertexts"""
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(n_bits + 7)
    with PaillierKey(n, g, n_bits, 64) as key:
        monkeypatch.setenv("PB200_TRACE_LANES", "64")
        # chains = 1: s = 1 up to 64 steps, then s = ceil(count / 64) (s - 1, s, s + 1 around s = 2 and 16); levels of 4 above
        for count in (1, 2, 3, 4, 5, 17, 63, 64, 65, 127, 128, 129, 1023, 1024, 1025):
            init = rng.randrange(n * n)
            _check(key, n, [init], _rows(rng, n, count, 1, edges=count >= 4))
        # chains = 3 (a wave of 64 lanes is 21 chunks per chain) and chains = 33 (one chunk per chain from 2 steps on)
        for chains, counts in ((3, (1, 2, 21, 22, 23, 43, 44, 45, 207)), (33, (1, 2, 3, 65))):
            for count in counts:
                inits = [rng.randrange(n * n) for _ in range(chains)]
                _check(key, n, inits, _rows(rng, n, count, chains, edges=count >= 4), want_q=count == counts[-1])
        # one wave of 4096 lanes +- 1 at one chain: s = 1 for 4095 and 4096 steps, 2 for 4097
        monkeypatch.setenv("PB200_TRACE_LANES", "4096")
        for count in (4095, 4096, 4097):
            _check(key, n, [rng.randrange(n * n)], _rows(rng, n, count, 1))
        monkeypatch.delenv("PB200_TRACE_LANES")
        for chains in (1, 3, 33):
            count = 3007 if chains < 33 else 207
            inits = [rng.randrange(n * n) for _ in range(chains)]
            _check(key, n, inits, _rows(rng, n, count, chains))


@gpu
def test_int_api_shapes(built_lib):
    """an int init (Python or numpy) with int steps gives flat lists; a list init gives one list per step"""
    kd = workload.load_key(1024)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(3)
    cs = [rng.randrange(n * n) for _ in range(9)]
    with PaillierKey(n, g, 1024, 64) as key:
        acc, q = key.tally_trace(5, cs)
        wa, wq = trace_native(n, [5], [[c] for c in cs])
        assert acc == [a[0] for a in wa] and q == [x[0] for x in wq]
        assert key.tally_trace(5, cs, want_q=False) == acc
        assert key.tally_trace(np.int64(5), cs) == (acc, q)                  # a numpy integer is one chain too
        acc2, q2 = key.tally_trace([5], [[c] for c in cs])
        assert acc2 == wa and q2 == wq
        assert key.tally_trace([1, 2], []) == ([], [])


# ---- unreduced inputs and the range check ----------------------------------------------------------------------------------------
@gpu
def test_unreduced_inputs_and_range(built_lib, monkeypatch):
    """init and c at or above n^2 (q still fitting words_out words) give the Python chain on several levels; a first pair whose q
    overflows raises PB200_ERR_RANGE, as pb200_add_batch does on the same pair"""
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    n2, wo = n * n, 2 * n_bits // 64
    rng = random.Random(11)
    top = 1 << (64 * wo)
    with PaillierKey(n, g, n_bits, 64) as key:
        for lanes in ("64", None):
            if lanes:
                monkeypatch.setenv("PB200_TRACE_LANES", lanes)
            else:
                monkeypatch.delenv("PB200_TRACE_LANES", raising=False)
            chains, count = 3, 500
            inits = [n2, n2 + 5, top // 2 - 1]
            rows = [[rng.randrange(n2, top // 2) if (i + j) % 3 else rng.randrange(n2) for j in range(chains)] for i in range(count)]
            rows[0] = [n2, top // 2 - 1, 1]
            _check(key, n, inits, rows)
        bad = [[top - 1]]
        with pytest.raises(Pb200Error) as e:
            key.tally_trace([top - 1], bad * 40)
        assert e.value.status == _lib.PB200_ERR_RANGE
        with pytest.raises(Pb200Error) as e2:
            key.paillier_add_native([top - 1], [top - 1], want_q=True)
        assert e2.value.status == _lib.PB200_ERR_RANGE


# ---- consistency with the existing entry points -----------------------------------------------------------------------------------
@gpu
def test_consistent_with_tally_and_add_batch(built_lib):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(12)
    chains, count = 3, 2000
    with PaillierKey(n, g, n_bits, 64) as key:
        inits = [rng.randrange(n * n) for _ in range(chains)]
        rows = _rows(rng, n, count, chains)
        acc, q = key.tally_trace(inits, rows)
        for j in range(chains):
            assert acc[-1][j] == key.tally([inits[j]] + [r[j] for r in rows])
        steps = sorted(rng.sample(range(count), 64))
        a = [inits[0] if i == 0 else acc[i - 1][0] for i in steps]
        b = [rows[i][0] for i in steps]
        ra, rq = key.paillier_add_native(a, b, want_q=True)
        assert ra == [acc[i][0] for i in steps] and rq == [q[i][0] for i in steps]


# ---- engines ----------------------------------------------------------------------------------------------------------------------
@gpu
def test_every_engine_gives_identical_outputs(built_lib, monkeypatch):
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    rng = random.Random(13)
    chains, count = 3, 300
    inits = [rng.randrange(n * n) for _ in range(chains)]
    rows = _rows(rng, n, count, chains)
    want = trace_native(n, inits, rows)
    ran = []
    monkeypatch.setenv("PB200_TRACE_LANES", "64")
    with PaillierKey(n, g, n_bits, 64) as key:
        for engine in (1, 2, 3, 4, 5):
            try:
                key.set_engine(engine)
            except Pb200Error as e:
                assert e.status == _lib.PB200_ERR_UNSUPPORTED
                continue
            assert key.tally_trace(inits, rows) == want, key.engine
            ran.append(key.engine)
    assert len(ran) >= 4, ran


@gpu
def test_simple64_witness_keys(built_lib, monkeypatch):
    """a key whose n is shorter than n_bits (block28 scan, simple64 chain), an even modulus, and a key size no block engine covers
    (simple64 throughout), each on the automatic engine and on simple64"""
    rng = random.Random(14)
    monkeypatch.setenv("PB200_TRACE_LANES", "64")
    for n_bits, limb_bits, n in ((1024, 64, None), (1024, 64, "even"), (260, 65, None)):
        if n is None:
            n = rng.getrandbits(n_bits - (8 if n_bits == 1024 else 0)) | 1 << (n_bits - (9 if n_bits == 1024 else 1)) | 1
        else:
            n = (rng.getrandbits(n_bits) | 1 << (n_bits - 1)) & ~1
        g = rng.getrandbits(n_bits - 1)
        with PaillierKey(n, g, n_bits, limb_bits) as key:
            if n_bits == 1024 and n.bit_length() < n_bits:
                assert key.witness_engine == "simple64" and key.engine != "simple64"
            for engine in (0, 1):
                key.set_engine(engine)
                for chains, count in ((1, 150), (3, 70)):
                    inits = [rng.randrange(n * n) for _ in range(chains)]
                    _check(key, n, inits, _rows(rng, n, count, chains))


# ---- size -------------------------------------------------------------------------------------------------------------------------
@gpu
def test_large_trace(built_lib):
    """2^18 + 5 steps of one chain at |n| = 2048 on the default wave, compared in full; two calls give identical output"""
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    count = (1 << 18) + 5
    c_w = workload.ciphertexts(n_bits, count, n, seed_offset=61)
    init_w = workload.ciphertexts(n_bits, 1, n, seed_offset=62)
    with PaillierKey(n, g, n_bits, 64) as key:
        acc, q = key.tally_trace_words(init_w, c_w.reshape(count, 1, -1))
        acc2, q2 = key.tally_trace_words(init_w, c_w.reshape(count, 1, -1))
        assert (acc == acc2).all() and (q == q2).all()
    n2 = n * n
    a = words_to_ints(init_w)[0]
    cs, got_a, got_q = words_to_ints(c_w), words_to_ints(acc.reshape(count, -1)), words_to_ints(q.reshape(count, -1))
    for i, c in enumerate(cs):
        qi, a = divmod(a * c, n2)
        assert got_a[i] == a and got_q[i] == qi, i


# ---- witness validity -------------------------------------------------------------------------------------------------------------
@gpu
def test_trace_feeds_the_chip_and_the_cells(built_lib):
    """the (q, rem) of 8 steps satisfy the restated PaillierChip::add chain; the contiguous-operand layout (init in row 0, acc one
    row in) gives the (a, b, q, rem) arrays of pb200_mulmod_cells_batch, which accepts them and rejects a tampered q"""
    import torch
    n_bits = 1024
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    wo = 2 * n_bits // 64
    rng = random.Random(15)
    init, cs = rng.randrange(n * n), [rng.randrange(n * n) for _ in range(8)]
    with PaillierKey(n, g, n_bits, 64) as key:
        acc, q = key.tally_trace(init, cs)
        ctx = Context()
        big = BigUintChip(64, 15, witness_source=list(zip(q, acc)))
        chip = PaillierChip.construct(big, n_bits)
        pk = EncryptionPublicKeyAssigned(big.assign_integer(ctx, n, n_bits), big.assign_integer(ctx, g, n_bits))
        a = big.assign_integer(ctx, init, 2 * n_bits)
        for c, want in zip(cs, acc):
            a = chip.add(ctx, pk, a, big.assign_integer(ctx, c, 2 * n_bits))
            assert a.value == want
        check_constraints(ctx)
        # contiguous operands on the device, for 3 chains and 50 steps
        chains, count = 3, 50
        inits = [rng.randrange(n * n) for _ in range(chains)]
        rows = _rows(rng, n, count, chains)
        buf = torch.zeros(((count + 1) * chains, wo), dtype=torch.int64, device="cuda")
        buf[:chains] = torch.from_numpy(ints_to_words(inits, wo).view(np.int64)).cuda()
        d_c = torch.from_numpy(ints_to_words([c for r in rows for c in r], wo).view(np.int64)).cuda()
        d_q = torch.empty((count * chains, wo), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()                                        # the key's stream does not wait for torch's
        key.tally_trace_dev(buf.data_ptr(), d_c.data_ptr(), count, chains, buf[chains:].data_ptr(), d_q.data_ptr())
        key.sync()
        assert key.take_flags() == 0
        lay = key.cells_layout(15)
        cells = torch.empty((count * chains, lay["cells_per_mulmod"], 4), dtype=torch.int64, device="cuda")
        key.mulmod_cells_dev(buf.data_ptr(), d_c.data_ptr(), d_q.data_ptr(), buf[chains:].data_ptr(), count * chains, 15, False, cells.data_ptr())
        key.sync()
        h = buf.cpu().numpy().view(np.uint64)
        qh, ch = d_q.cpu().numpy().view(np.uint64), d_c.cpu().numpy().view(np.uint64)
        want_a, want_q = trace_native(n, inits, rows)
        assert words_to_ints(h[chains:]) == [x for r in want_a for x in r]
        assert words_to_ints(qh) == [x for r in want_q for x in r]
        host = key.mulmod_cells_words(h[:-chains], ch, qh, h[chains:], 15)
        assert (host == cells.cpu().numpy().view(np.uint64).reshape(host.shape)).all()
        bad = qh.copy()
        bad[17, 0] ^= 1
        with pytest.raises(Pb200Error) as e:
            key.mulmod_cells_words(h[:-chains], ch, bad, h[chains:], 15)
        assert e.value.status == _lib.PB200_ERR_CONSTRAINT


# ---- decryption -------------------------------------------------------------------------------------------------------------------
@gpu
def test_decryption_round_trip(built_lib):
    """Dec(acc_i) = m_init + sum_(t <= i) m_t mod n for every step of two chains"""
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, p, q = kd["n"], kd["p"], kd["q"]
    g = kd["g_rand"]
    chains, count = 2, 120
    m_w, r_w = workload.units(n_bits, (count + 1) * chains, seed_offset=30)
    ms = words_to_ints(m_w)
    with PaillierKey(n, g, n_bits, 64) as key:
        key.set_private(*private_from_primes(p, q, g))
        cs = words_to_ints(key.encrypt_words(m_w, r_w))
        inits, rows = cs[:chains], [cs[chains * (i + 1):chains * (i + 2)] for i in range(count)]
        acc = key.tally_trace(inits, rows, want_q=False)
        dec = key.decrypt([x for r in acc for x in r])
        for j in range(chains):
            s = ms[j]
            for i in range(count):
                s = (s + ms[chains * (i + 1) + j]) % n
                assert dec[i * chains + j] == s, (i, j)


# ---- device variant ---------------------------------------------------------------------------------------------------------------
@gpu
def test_dev_variant_and_flags(built_lib):
    """pb200_tally_trace_dev gives the host variant's output with and without q and a clean flag word; an overflowing first q
    raises PB200_FLAG_RANGE; empty shapes do nothing"""
    import torch
    n_bits = 2048
    kd = workload.load_key(n_bits)
    n, g = kd["n"], kd["g_rand"]
    wo = 2 * n_bits // 64
    rng = random.Random(16)
    chains, count = 5, 700
    inits = [rng.randrange(n * n) for _ in range(chains)]
    rows = _rows(rng, n, count, chains)
    with PaillierKey(n, g, n_bits, 64) as key:
        want_a, want_q = key.tally_trace_words(ints_to_words(inits, wo), ints_to_words([c for r in rows for c in r], wo))
        d_i = torch.from_numpy(ints_to_words(inits, wo).view(np.int64)).cuda()
        d_c = torch.from_numpy(ints_to_words([c for r in rows for c in r], wo).view(np.int64)).cuda()
        d_a = torch.empty((count * chains, wo), dtype=torch.int64, device="cuda")
        d_q = torch.empty_like(d_a)
        for with_q in (True, False):
            d_a.zero_()
            torch.cuda.synchronize()                                    # the key's stream does not wait for torch's
            key.tally_trace_dev(d_i.data_ptr(), d_c.data_ptr(), count, chains, d_a.data_ptr(), d_q.data_ptr() if with_q else None)
            key.sync()
            assert key.take_flags() == 0
            assert (d_a.cpu().numpy().view(np.uint64) == want_a.reshape(-1, wo)).all()
            if with_q:
                assert (d_q.cpu().numpy().view(np.uint64) == want_q.reshape(-1, wo)).all()
        top = torch.full((1, wo), -1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        key.tally_trace_dev(top.data_ptr(), top.data_ptr(), 1, 1, d_a.data_ptr(), None)
        key.sync()
        assert key.take_flags() & _lib.PB200_FLAG_RANGE
        lib = key._lib
        assert lib.pb200_tally_trace_dev(key.handle, None, None, 0, chains, None, None) == _lib.PB200_OK
        assert lib.pb200_tally_trace_dev(key.handle, None, None, count, 0, None, None) == _lib.PB200_OK
        assert lib.pb200_tally_trace(key.handle, None, None, 0, 0, None, None) == _lib.PB200_OK
        for args in ((None, d_c.data_ptr(), d_a.data_ptr()), (d_i.data_ptr(), None, d_a.data_ptr()), (d_i.data_ptr(), d_c.data_ptr(), None)):
            assert lib.pb200_tally_trace_dev(key.handle, args[0], args[1], 1, 1, args[2], None) == _lib.PB200_ERR_INVALID_ARG
        u = np.zeros(wo, dtype="<u8")
        assert lib.pb200_tally_trace(key.handle, None, u.ctypes.data_as(_lib.u64p), 1, 1, u.ctypes.data_as(_lib.u64p), None) == \
            _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_tally_trace(key.handle, u.ctypes.data_as(_lib.u64p), u.ctypes.data_as(_lib.u64p), 1, 1, None, None) == \
            _lib.PB200_ERR_INVALID_ARG


# ---- CPU-only ---------------------------------------------------------------------------------------------------------------------
def test_trace_arguments_are_rejected(built_lib):
    """no key: PB200_ERR_INVALID_ARG whatever the sizes"""
    lib = built_lib
    null = C.c_void_p()
    for count, chains in ((0, 0), (1, 0), (0, 1), (3, 2)):
        assert lib.pb200_tally_trace(null, None, None, count, chains, None, None) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_tally_trace_dev(null, None, None, count, chains, None, None) == _lib.PB200_ERR_INVALID_ARG


def test_trace_oracle_matches_pairwise_divmod():
    rng = random.Random(17)
    n = rng.getrandbits(128) | 1 << 127 | 1
    inits = [rng.getrandbits(256) for _ in range(2)]
    rows = [[rng.getrandbits(256) for _ in range(2)] for _ in range(5)]
    acc, q = trace_native(n, inits, rows)
    for j in range(2):
        a = inits[j]
        for i in range(5):
            assert q[i][j] * n * n + acc[i][j] == a * rows[i][j] and 0 <= acc[i][j] < n * n
            a = acc[i][j]


def _sass_ops():
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
    return per


def test_trace_kernels_are_tcgen05(built_lib):
    """the fast-engine trace kernels for the tcgen05 engine (tally shape, ENG 4) at |n| = 2048 / 3072 / 4096 run on tcgen05; the
    witness-chain kernel is compiled for every configuration (WENG 0) and on tcgen05 where the configuration has it (WENG 1)"""
    per = _sass_ops()
    for name in ("k_trace_reduce", "k_trace_apply"):
        for g, bl in ((8, 19), (16, 14), (16, 19)):
            pat = re.compile(rf"\d+{name}INS_3b283CfgILi{g}ELi{bl}EEELi4EEEv")
            ks = [v for k, v in per.items() if pat.search(k)]
            assert len(ks) == 1, (name, g, bl)
            ops = ks[0]
            assert ops.get("UTCIMMA", 0) >= 8 and ops.get("LDTM", 0) >= 2 and ops.get("UTCBAR", 0) >= 2, (name, g, bl)
            assert ops.get("IMMA", 0) == 0
    for g, bl in ((4, 19), (8, 19), (16, 14), (16, 19)):
        pat = re.compile(rf"\d+k_trace_wINS_3b283CfgILi{g}ELi{bl}EEELi0EEEv")
        ks = [v for k, v in per.items() if pat.search(k)]
        assert len(ks) == 1, (g, bl)
        assert ks[0].get("IMMA", 0) > 0
    for g, bl in ((8, 19), (16, 14), (16, 19)):
        pat = re.compile(rf"\d+k_trace_wINS_3b283CfgILi{g}ELi{bl}EEELi1EEEv")
        ks = [v for k, v in per.items() if pat.search(k)]
        assert len(ks) == 1, (g, bl)
        assert ks[0].get("UTCIMMA", 0) >= 8
