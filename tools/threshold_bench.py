#!/usr/bin/env python
"""Throughput of threshold decryption on one GPU: a trustee's partial decryption c^(2 Delta s_i) mod n^2 beside decrypt, and the fused
combination of k shares (k_multipow per sign, one inverse, L and phi) beside the route the library offered before it, on the same shares
in the same process.

    python tools/threshold_bench.py --out profiles/threshold_bench_r07.json

Legs (2^16 ciphertexts, random g, |n| = 2048 unless stated):
  (a) pb200_partial_decrypt_batch_dev at l = 9, beside pb200_decrypt_batch_dev of the same ciphertexts
  (b) pb200_partial_decrypt_batch_dev at |n| = 1024, 3072, 4096 (l = 9)
  (c) pb200_combine_shares_batch_dev with k = 2 (l = 3, t = 1), k = 5 and k = 9 (l = 9, t = 4), each beside the composed route:
      pb200_scalar_mul_signed_batch_dev per share (c_j^(2 mu_j), an inverse where mu_j < 0), k - 1 pb200_add_batch_dev folds, then
      pb200_decrypt_batch_dev on a key set up with set_private(1, phi); it yields the same m
Every timed call is enqueued on the key's stream between two CUDA events; each leg is warmed up, then repeated and reported as median /
min / max.  The ciphertexts are real encryptions of seeded plaintexts (workload.units).  Checks: every plaintext of every combination
and of decrypt against the dealer's m; every partial decryption feeds the k = l combinations, and a random 128 of each partial
decryption leg against Python's pow (by CRT over p^2 and q^2).  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import sys
from math import factorial

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from inverse_bench import card, timed  # noqa: E402
from paillier_halo2_b200 import workload  # noqa: E402
from paillier_halo2_b200.api import PaillierKey, ints_to_words, private_from_primes, threshold_from_primes, words_to_ints  # noqa: E402

N_BITS = 2048
UNITS = 1 << 16
SAMPLE = 128


def lagrange(indices, parties):
    delta = factorial(parties)
    out = []
    for j in indices:
        num, den, below = delta, 1, 0
        for jj in indices:
            if jj != j:
                num *= jj
                den *= abs(jj - j)
                below += jj < j
        out.append(-(num // den) if below & 1 else num // den)
    return out


def pow_crt(c: int, e: int, p: int, q: int) -> int:
    """c^e mod (pq)^2 for c prime to pq, over p^2 and q^2 with the exponent reduced mod p (p - 1), q (q - 1)"""
    p2, q2 = p * p, q * q
    a, b = pow(c, e % (p * (p - 1)), p2), pow(c, e % (q * (q - 1)), q2)
    return (a + p2 * ((b - a) * pow(p2, -1, q2) % q2)) % (p2 * q2)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--units", type=int, default=UNITS)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to fall back to")
    U = args.units
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()      # noqa: E731
    host = lambda t: t.cpu().numpy().view(np.uint64)                                    # noqa: E731
    rng = random.Random(20261022)
    rec = {"tool": "tools/threshold_bench.py", "n_bits": N_BITS, "g": "random", "units": U, "card": card(), "reps": args.reps,
           "warmup": args.warmup, "inputs": "encryptions of seeded plaintexts; 2^16 ciphertexts are 32 MiB at |n| = 2048"}
    legs, checks = {}, {}

    def partial_leg(bits, parties, name, with_decrypt):
        kd = workload.load_key(bits)
        n, g, p, q = kd["n"], kd["g_rand"], kd["p"], kd["q"]
        shares, phi = threshold_from_primes(p, q, g, 4, parties, rng=random.Random(bits))
        m_w, r_w = workload.units(bits, U, seed_offset=91)
        with PaillierKey(n, g, bits, 64) as key:
            stream = torch.cuda.ExternalStream(key.stream)
            torch.cuda.set_stream(stream)
            rec.setdefault("engine", {})[bits] = key.engine
            c_w = key.encrypt_words(m_w, r_w)
            d_c = dev(c_w)
            d_out = torch.empty_like(d_c)
            key.set_threshold(parties, phi)
            key.set_share(1, shares[1])
            legs[name] = timed(torch, stream, lambda: key.partial_decrypt_dev(d_c.data_ptr(), U, d_out.data_ptr()), args.reps, args.warmup, U)
            print(name, json.dumps(legs[name]), flush=True)
            key.sync()
            got = host(d_out)
            idx = rng.sample(range(U), SAMPLE)
            e = 2 * factorial(parties) * shares[1]
            checks[name] = sum(pow_crt(c, e, p, q) != x for c, x in zip(words_to_ints(c_w[idx]), words_to_ints(got[idx])))
            if with_decrypt:
                key.set_private(*private_from_primes(p, q, g))
                d_m = torch.empty((U, bits // 64), dtype=torch.int64, device="cuda")
                legs["a_decrypt"] = timed(torch, stream, lambda: key.decrypt_dev(d_c.data_ptr(), U, d_m.data_ptr()), args.reps, args.warmup, U)
                print("a_decrypt", json.dumps(legs["a_decrypt"]), flush=True)
                key.sync()
                checks["a_decrypt"] = int((host(d_m).reshape(U, -1) != m_w).any(axis=1).sum())
            assert key.take_flags() == 0

    partial_leg(N_BITS, 9, "a_partial_l9", True)
    for bits in (1024, 3072, 4096):
        partial_leg(bits, 9, f"b_partial_{bits}", False)

    # (c) combination, fused against composed
    kd = workload.load_key(N_BITS)
    n, g, p, q = kd["n"], kd["g_rand"], kd["p"], kd["q"]
    wi, wo = N_BITS // 64, 2 * N_BITS // 64
    m_w, r_w = workload.units(N_BITS, U, seed_offset=92)
    speed = {}
    for parties, t, ks in ((3, 1, (2,)), (9, 4, (5, 9))):
        shares, phi = threshold_from_primes(p, q, g, t, parties, rng=random.Random(parties))
        with PaillierKey(n, g, N_BITS, 64) as key:
            stream = torch.cuda.ExternalStream(key.stream)
            torch.cuda.set_stream(stream)
            c_w = key.encrypt_words(m_w, r_w)
            d_c = dev(c_w)
            key.set_threshold(parties, phi)
            d_sh = torch.empty((parties, U, wo), dtype=torch.int64, device="cuda")
            for i in range(1, parties + 1):
                key.set_share(i, shares[i])
                key.partial_decrypt_dev(d_c.data_ptr(), U, d_sh[i - 1].data_ptr())
            key.sync()
            key.set_private(1, phi)                            # the composed route: L(x) phi after its own products
            d_m = torch.empty((U, wi), dtype=torch.int64, device="cuda")
            d_acc = torch.empty((2, U, wo), dtype=torch.int64, device="cuda")
            d_tmp = torch.empty((U, wo), dtype=torch.int64, device="cuda")
            for k in ks:
                idx = list(range(1, k + 1)) if k == parties else sorted(rng.sample(range(1, parties + 1), k))
                d_set = torch.stack([d_sh[i - 1] for i in idx]).contiguous()
                mus = lagrange(idx, parties)
                kb = max(abs(2 * mu).bit_length() for mu in mus)
                d_mag = [dev(ints_to_words([abs(2 * mu)] * U, (kb + 63) // 64)) for mu in mus]
                d_neg = [torch.full((U,), 1 if mu < 0 else 0, dtype=torch.uint8, device="cuda") for mu in mus]

                def fused():
                    key.combine_shares_dev(idx, d_set.data_ptr(), U, d_m.data_ptr())

                def composed():
                    for j in range(k):
                        dst = d_acc[0] if j == 0 else d_tmp
                        key.scalar_mul_signed_dev(d_set[j].data_ptr(), d_mag[j].data_ptr(), d_neg[j].data_ptr() if mus[j] < 0 else 0, kb, U,
                                                  dst.data_ptr())
                        if j:
                            key.add_dev(d_acc[(j - 1) % 2].data_ptr(), d_tmp.data_ptr(), wo, U, d_acc[j % 2].data_ptr(), 0)
                    key.decrypt_dev(d_acc[(k - 1) % 2].data_ptr(), U, d_m.data_ptr())

                for name, fn in ((f"c_fused_k{k}", fused), (f"c_composed_k{k}", composed)):
                    d_m.zero_()
                    legs[name] = timed(torch, stream, fn, args.reps, args.warmup, U)
                    legs[name]["indices"] = idx
                    print(name, json.dumps(legs[name]), flush=True)
                    key.sync()
                    checks[name] = int((host(d_m).reshape(U, -1) != m_w).any(axis=1).sum())
                    assert key.take_flags() == 0, name
                speed[f"k{k}"] = legs[f"c_fused_k{k}"]["per_s_median"] / legs[f"c_composed_k{k}"]["per_s_median"]
    rec["legs"] = legs
    rec["checks_mismatches"] = checks
    rec["combination_speedup_fused_over_composed"] = speed
    rec["partial_over_decrypt"] = legs["a_partial_l9"]["per_s_median"] / legs["a_decrypt"]["per_s_median"]
    print(json.dumps(rec))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
    if any(checks.values()):
        raise SystemExit("an output differs from its reference")


if __name__ == "__main__":
    main()
