#!/usr/bin/env python
"""Throughput of the ciphertext inverse, the homomorphic subtraction and signed scalars on one GPU, each beside the route that existed
before them (a full-width exponent n - 1), on the same ciphertexts in the same process.

    python tools/inverse_bench.py --out profiles/inverse_bench_r06.json
    python tools/inverse_bench.py --profile --out profiles/inverse_bench_r06.json     # adds the per-kernel split (a run of its own)

Legs at |n| = 2048, random g (d: other sizes):
  (a) pb200_inverse_batch_dev against pb200_scalar_mul_batch_dev with every k = n - 1, at 2^16 and 2^20 units
  (b) pb200_sub_batch_dev against scalar_mul(c2, n - 1) + pb200_add_batch_dev, 2^16 pairs
  (c) pb200_scalar_mul_signed_batch_dev with 32-bit magnitudes, half of them negative, against pb200_scalar_mul_batch_dev with the same
      weights as n - s (full width), and against the unsigned 32-bit pb200_scalar_mul_batch_dev (the floor)
  (d) pb200_inverse_batch_dev at |n| = 1024, 3072, 4096 (2^16 units)
Every timed call is enqueued on the key's stream between two CUDA events; each leg is warmed up, then repeated and reported as median /
min / max.  Inputs are uniform below n^2 (workload.ciphertexts); 2^16 values of 512 bytes fit the 126 MB L2, 2^20 do not; no flush.
Checks: every output of the 2^16 legs against Python ints (c x = 1 mod n^2 for an inverse, which is unique), and a random 1 000 of each
2^20 leg; the n - 1 routes on a sample (a Python pow with a 2048-bit exponent per unit).  The card's name and power limit are read in the
same run.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from paillier_halo2_b200 import workload  # noqa: E402
from paillier_halo2_b200.api import PaillierKey, ints_to_words, words_to_ints  # noqa: E402

N_BITS = 2048
SMALL, LARGE = 1 << 16, 1 << 20
OLD_SAMPLE = 64          # units of each n - 1 route checked with a full-width Python pow


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.strip().split(",")) if q.returncode == 0 else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(torch, stream, fn, reps: int, warmup: int, units: int) -> dict:
    for _ in range(warmup):
        fn()
    stream.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        ms.append(a.elapsed_time(b))
    med = statistics.median(ms)
    return {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "reps": reps, "units": units, "per_s_median": units / med * 1e3}


def kernel_split(torch, stream, fn) -> dict:
    """GPU milliseconds and launches per kernel name over one call"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        stream.synchronize()
    split = {}
    for ev in prof.key_averages():
        if ev.device_time_total <= 0:
            continue
        name = ev.key.split("(")[0].split("<")[0].replace("void ", "").replace("pb200::", "").strip()
        s = split.setdefault(name, {"ms": 0.0, "launches": 0})
        s["ms"] = round(s["ms"] + ev.device_time_total / 1e3, 3)
        s["launches"] += ev.count
    return split


def host(t, n=None) -> list:
    a = t.cpu().numpy().view(np.uint64)
    return words_to_ints(a if n is None else a[:n])


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON record (default: stdout only); with --profile, the record to add the split to")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--profile", action="store_true", help="only the per-kernel split of one call of each new leg")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to fall back to")
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()      # noqa: E731
    rng = random.Random(20261022)
    kd = workload.load_key(N_BITS)
    n, g = kd["n"], kd["g_rand"]
    n2, wi, wo = n * n, N_BITS // 64, 2 * N_BITS // 64
    c_w = workload.ciphertexts(N_BITS, LARGE, n, seed_offset=81)
    c2_w = workload.ciphertexts(N_BITS, SMALL, n, seed_offset=82)
    mags = [rng.getrandbits(32) for _ in range(SMALL)]
    neg = np.array([i % 2 for i in range(SMALL)], dtype=np.uint8)                         # half negative, interleaved in every CTA
    rec = {"tool": "tools/inverse_bench.py", "n_bits": N_BITS, "g": "random", "card": card(), "reps": args.reps, "warmup": args.warmup,
           "inputs": "uniform below n^2; 2^16 units (32 MiB) fit L2, 2^20 (512 MiB) do not; no flush"}
    with PaillierKey(n, g, N_BITS, 64) as key:
        stream = torch.cuda.ExternalStream(key.stream)
        torch.cuda.set_stream(stream)
        rec["engine"] = key.engine
        d_c, d_c2 = dev(c_w), dev(c2_w)
        d_nm1 = dev(ints_to_words([n - 1] * LARGE, wi))
        d_mag = dev(ints_to_words(mags, 1))
        d_neg = torch.from_numpy(neg).cuda()
        d_nms = dev(ints_to_words([n - m if s else m for m, s in zip(mags, neg)], wi))
        d_out = torch.empty((LARGE, wo), dtype=torch.int64, device="cuda")
        d_tmp = torch.empty((SMALL, wo), dtype=torch.int64, device="cuda")
        c, c2, out, tmp = d_c.data_ptr(), d_c2.data_ptr(), d_out.data_ptr(), d_tmp.data_ptr()
        legs = {
            "a_inverse_2^16": (lambda: key.invert_dev(c, SMALL, out), SMALL),
            "a_nm1_2^16": (lambda: key.scalar_mul_dev(c, d_nm1.data_ptr(), N_BITS, SMALL, out), SMALL),
            "a_inverse_2^20": (lambda: key.invert_dev(c, LARGE, out), LARGE),
            "a_nm1_2^20": (lambda: key.scalar_mul_dev(c, d_nm1.data_ptr(), N_BITS, LARGE, out), LARGE),
            "b_sub_2^16": (lambda: key.sub_dev(c, c2, SMALL, out), SMALL),
            "b_nm1_add_2^16": (lambda: (key.scalar_mul_dev(c2, d_nm1.data_ptr(), N_BITS, SMALL, tmp), key.add_dev(c, tmp, wo, SMALL, out, 0)), SMALL),
            "c_signed_32_2^16": (lambda: key.scalar_mul_signed_dev(c, d_mag.data_ptr(), d_neg.data_ptr(), 32, SMALL, out), SMALL),
            "c_n_minus_s_2^16": (lambda: key.scalar_mul_dev(c, d_nms.data_ptr(), N_BITS, SMALL, out), SMALL),
            "c_unsigned_32_2^16": (lambda: key.scalar_mul_dev(c, d_mag.data_ptr(), 32, SMALL, out), SMALL),
        }
        if args.profile:
            split = {}
            for name in ("a_inverse_2^16", "b_sub_2^16", "c_signed_32_2^16", "a_nm1_2^16"):
                legs[name][0]()
                key.sync()
                split[name] = kernel_split(torch, stream, legs[name][0])
            rec = json.load(open(args.out)) if args.out and os.path.exists(args.out) else {}
            rec["kernel_split_ms"] = split
            rec["kernel_split_card"] = card()
            print(json.dumps(split))
            if args.out:
                json.dump(rec, open(args.out, "w"), indent=1)
            return
        res, checks = {}, {}
        cs = words_to_ints(c_w[:SMALL])
        sample = rng.sample(range(SMALL), OLD_SAMPLE)
        for name, (fn, units) in legs.items():
            res[name] = timed(torch, stream, fn, args.reps, args.warmup, units)
            print(name, json.dumps(res[name]), flush=True)
            fn()
            key.sync()
            if name == "a_inverse_2^16":
                xs = host(d_out, SMALL)
                checks[name] = sum(c * x % n2 != 1 for c, x in zip(cs, xs))
            elif name == "a_inverse_2^20":
                idx = rng.sample(range(LARGE), 1000)
                got = d_out.cpu().numpy().view(np.uint64)
                call = words_to_ints(c_w[idx])
                checks[name] = sum(c * x % n2 != 1 for c, x in zip(call, words_to_ints(got[idx])))
            elif name.startswith("a_nm1"):
                got = d_out.cpu().numpy().view(np.uint64)
                idx = sample if name.endswith("2^16") else rng.sample(range(LARGE), OLD_SAMPLE)
                checks[name] = sum(pow(c, n - 1, n2) != x for c, x in zip(words_to_ints(c_w[idx]), words_to_ints(got[idx])))
            elif name == "b_sub_2^16":
                c2s = words_to_ints(c2_w)
                checks[name] = sum((x * b - a) % n2 != 0 for a, b, x in zip(cs, c2s, host(d_out, SMALL)))
            elif name == "b_nm1_add_2^16":
                c2s = words_to_ints(c2_w)
                got = host(d_out, SMALL)
                checks[name] = sum(got[i] != cs[i] * pow(c2s[i], n - 1, n2) % n2 for i in sample)
            elif name == "c_unsigned_32_2^16":
                checks[name] = sum(pow(c, m, n2) != x for c, m, x in zip(cs, mags, host(d_out, SMALL)))
            elif name == "c_signed_32_2^16":
                got = host(d_out, SMALL)
                checks[name] = sum((x * pow(c, m, n2) % n2 != 1) if s else (x != pow(c, m, n2)) for c, m, s, x in zip(cs, mags, neg, got))
            elif name == "c_n_minus_s_2^16":
                got = host(d_out, SMALL)
                checks[name] = sum(got[i] != pow(cs[i], n - mags[i] if neg[i] else mags[i], n2) for i in sample)
            print(name, "mismatches", checks[name], flush=True)
        assert key.take_flags() == 0
        rec["legs"] = res
        rec["checks_mismatches"] = checks
        rec["checks_units"] = {k: (SMALL if k in ("a_inverse_2^16", "b_sub_2^16", "c_signed_32_2^16", "c_unsigned_32_2^16")
                                   else 1000 if k == "a_inverse_2^20" else OLD_SAMPLE) for k in checks}
        sp = lambda a, b: res[a]["per_s_median"] / res[b]["per_s_median"]      # noqa: E731
        rec["speedup"] = {"a_2^16": sp("a_inverse_2^16", "a_nm1_2^16"), "a_2^20": sp("a_inverse_2^20", "a_nm1_2^20"),
                          "b": sp("b_sub_2^16", "b_nm1_add_2^16"), "c_vs_n_minus_s": sp("c_signed_32_2^16", "c_n_minus_s_2^16"),
                          "c_vs_unsigned_floor": sp("c_signed_32_2^16", "c_unsigned_32_2^16")}
    # (d) other key sizes
    other = {}
    for bits in (1024, 3072, 4096):
        kd = workload.load_key(bits)
        nb, nb2 = kd["n"], kd["n"] * kd["n"]
        cw = workload.ciphertexts(bits, SMALL, nb, seed_offset=83)
        with PaillierKey(nb, kd["g_rand"], bits, 64) as key:
            stream = torch.cuda.ExternalStream(key.stream)
            torch.cuda.set_stream(stream)
            dc = dev(cw)
            do = torch.empty_like(dc)
            t = timed(torch, stream, lambda: key.invert_dev(dc.data_ptr(), SMALL, do.data_ptr()), args.reps, args.warmup, SMALL)
            key.sync()
            t["mismatches"] = sum(c * x % nb2 != 1 for c, x in zip(words_to_ints(cw), host(do)))
            assert key.take_flags() == 0
            other[f"d_inverse_{bits}_2^16"] = t
            print(bits, json.dumps(t), flush=True)
    rec["d_other_sizes"] = other
    print(json.dumps(rec))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
    if any(checks.values()) or any(v["mismatches"] for v in other.values()):
        raise SystemExit("an output differs from its Python reference")


if __name__ == "__main__":
    main()
