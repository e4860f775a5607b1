"""CPU tests of threshold decryption: the dealer (api.threshold_from_primes) and a Python-int restatement of the two steps the library
runs (a trustee's partial decryption c^(2 Delta s_i) mod n^2, the combination L(P N^-1 mod n^2) phi mod n with signed Lagrange
exponents), on the committed keys with a random g and with g = n + 1; plus the compiled k_multipow (no spills, tcgen05 on block28u).
No device needed."""
import itertools
import os
import random
import re
import shutil
import subprocess
from math import factorial

import pytest

from paillier_halo2_b200 import workload
from paillier_halo2_b200.api import threshold_from_primes

SCHEMES = [(1, 3), (2, 5), (4, 9), (7, 32)]
LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "paillier_halo2_b200", "libpaillier_b200.so")


def lagrange(indices, parties):
    """mu_j = Delta prod_(j' != j) j' / (j' - j) as the library forms it: magnitude Delta prod j' // prod |j' - j| (asserted exact), sign
    the parity of the j' < j."""
    delta = factorial(parties)
    out = []
    for j in indices:
        num, den, below = delta, 1, 0
        for jj in indices:
            if jj != j:
                num *= jj
                den *= abs(jj - j)
                below += jj < j
        assert num % den == 0, (indices, j)
        out.append(-(num // den) if below & 1 else num // den)
    return out


def partial(c, share, parties, p, q):
    """c^(2 Delta s) mod n^2 for a c prime to n, by CRT over p^2 and q^2 with the exponent reduced mod p (p - 1) and q (q - 1) (the same
    value as pow(c, 2 Delta s, n^2), several times faster at 3072 bits)"""
    e = 2 * factorial(parties) * share
    p2, q2 = p * p, q * q
    a, b = pow(c, e % (p * (p - 1)), p2), pow(c, e % (q * (q - 1)), q2)
    return (a + p2 * ((b - a) * pow(p2, -1, q2) % q2)) % (p2 * q2)


def combine(indices, shares, parties, n, phi):
    """(m, exact): the combination of one unit's shares; exact is False when P N^-1 is not 1 mod n (the library's DECRYPT flag)."""
    n2 = n * n
    P, N = 1, 1
    for mu, c in zip(lagrange(indices, parties), shares):
        if mu > 0:
            P = P * pow(c, 2 * mu, n2) % n2
        else:
            N = N * pow(c, -2 * mu, n2) % n2
    x = P * pow(N, -1, n2) % n2
    if x % n != 1:
        return 0, False
    return (x - 1) // n * phi % n, True


def _keys():
    for n_bits in (128, 256, 1024, 2048, 3072):
        kd = workload.load_key(n_bits)
        for which in ("rand", "std"):
            yield n_bits, which, kd


def _subsets(parties, size, rng, limit):
    allsets = itertools.combinations(range(1, parties + 1), size) if parties <= 9 else None
    if allsets is not None:
        return [list(s) for s in allsets]
    return [sorted(rng.sample(range(1, parties + 1), size)) for _ in range(limit)]


@pytest.mark.parametrize("t,parties", SCHEMES)
@pytest.mark.parametrize("n_bits,which,kd", list(_keys()), ids=lambda v: str(v) if not isinstance(v, dict) else "key")
def test_dealer_and_combination(n_bits, which, kd, t, parties):
    p, q, n = kd["p"], kd["q"], kd["n"]
    g = kd["g_rand"] if which == "rand" else n + 1
    rng = random.Random(n_bits * 1000 + parties)
    shares, phi = threshold_from_primes(p, q, g, t, parties, rng=rng)
    assert sorted(shares) == list(range(1, parties + 1))
    delta = factorial(parties)
    if which == "std":
        assert phi == pow(4 * delta * delta, -1, n)
    # the exponent bound: 2 Delta s_i < 2^(2 n_bits + bits(2 Delta))
    for s in shares.values():
        assert (2 * delta * s).bit_length() <= 2 * n_bits + (2 * delta).bit_length()
    m = rng.randrange(n)
    c = pow(g, m, n * n) * pow(rng.randrange(1, n), n, n * n) % (n * n)
    cs = {i: partial(c, shares[i], parties, p, q) for i in range(1, parties + 1)}
    assert cs[1] == pow(c, 2 * delta * shares[1], n * n)
    for s in _subsets(parties, t + 1, rng, 12):
        got, ok = combine(s, [cs[i] for i in s], parties, n, phi)
        assert ok and got == m, (s,)
        shuffled = s[:]
        rng.shuffle(shuffled)
        assert combine(shuffled, [cs[i] for i in shuffled], parties, n, phi) == (m, True)
    every = list(range(1, parties + 1))
    assert combine(every, [cs[i] for i in every], parties, n, phi) == (m, True)
    # t shares do not pass the L check
    few = list(range(1, t + 1))
    assert combine(few, [cs[i] for i in few], parties, n, phi)[1] is False


@pytest.mark.parametrize("parties", [3, 5, 9, 32])
def test_lagrange_coefficients_are_integers_and_small(parties):
    rng = random.Random(parties)
    sets = [list(s) for s in itertools.combinations(range(1, parties + 1), min(parties, 5))] if parties <= 9 else []
    sets += [sorted(rng.sample(range(1, parties + 1), k)) for k in (1, 2, parties // 2, parties) for _ in range(5)]
    for s in sets:
        mus = lagrange(s, parties)
        # sum_j mu_j j^e = Delta [e == 0] for e < |S|: the interpolation at 0 of the polynomials 1, X, .., X^(|S|-1)
        for e in range(len(s)):
            assert sum(mu * j ** e for mu, j in zip(mus, s)) == (factorial(parties) if e == 0 else 0)
        assert mus[s.index(min(s))] > 0                  # the smallest index always has a positive coefficient
    if parties == 9:                                     # k_multipow's exponents at ell = 9: at most 30 bits (29 for 5 shares)
        assert max(abs(2 * mu).bit_length() for s in sets for mu in lagrange(s, 9)) <= 30
        assert max(abs(2 * mu).bit_length() for s in itertools.combinations(range(1, 10), 5) for mu in lagrange(list(s), 9)) == 29


def test_dealer_arguments():
    kd = workload.load_key(128)
    with pytest.raises(ValueError):
        threshold_from_primes(kd["p"], kd["q"], kd["n"] + 1, 3, 3)
    with pytest.raises(ValueError):
        threshold_from_primes(kd["p"], kd["q"], kd["n"] + 1, 1, 33)
    a = threshold_from_primes(kd["p"], kd["q"], kd["n"] + 1, 1, 3, rng=random.Random(1))
    b = threshold_from_primes(kd["p"], kd["q"], kd["n"] + 1, 1, 3, rng=random.Random(1))
    assert a == b
    assert threshold_from_primes(kd["p"], kd["q"], kd["n"] + 1, 1, 3)[0] != a[0]      # system randomness by default


def _cuobjdump():
    for c in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if c and os.path.exists(c):
            return c
    return None


def test_k_multipow_local_memory_and_tcgen05(built_lib):
    """k_multipow on the tally's engines: on block28t / block28u (ENG 1 / 4) at most a handful of local-memory instructions (ptxas -v:
    0 to 8 bytes of spill stores, DESIGN.md 9e), fewer than the k_tally it shares the CTA shape with; block28u's instantiations run
    phases B and C on tcgen05 (UTCIMMA, LDTM, STTM) and carry no mma.sync."""
    exe = _cuobjdump()
    if not exe:
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([exe, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    per, cur = {}, None
    for line in sass.split("\n"):
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            per[cur] = {}
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,5}\*/\s+(?:@!?U?P\d\s+)?([A-Z][A-Z0-9_]*)", line)
        if cur and m:
            per[cur][m.group(1)] = per[cur].get(m.group(1), 0) + 1

    def one(name, g, bl, eng):
        pat = re.compile(rf"\d+{name}INS_3b283CfgILi{g}ELi{bl}EEELi{eng}EEEv")
        ks = [v for k, v in per.items() if pat.search(k)]
        assert len(ks) == 1, (name, g, bl, eng, len(ks))
        return ks[0]

    local = lambda ops: ops.get("STL", 0) + ops.get("LDL", 0)      # noqa: E731
    for (g, bl), engs in {(4, 19): (1,), (8, 19): (1, 4), (16, 14): (1, 4), (16, 19): (1, 4)}.items():
        for eng in engs:
            ops = one("k_multipow", g, bl, eng)
            assert local(ops) <= 4 and local(ops) < local(one("k_tally", g, bl, eng)), (g, bl, eng, ops.get("STL"), ops.get("LDL"))
            if eng == 4:
                assert ops.get("UTCIMMA", 0) >= 8 and ops.get("LDTM", 0) >= 2 and ops.get("STTM", 0) >= 1
                assert ops.get("IMMA", 0) == 0
