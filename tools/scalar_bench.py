#!/usr/bin/env python
"""Throughput of homomorphic scalar multiplication and of the weighted tally on one GPU at |n| = 2048, with the decryption leg
(k_pow, c^lambda mod n^2) and the plain tally of the same process as the A/B reference.

    python tools/scalar_bench.py --out profiles/scalar_bench_r03.json

Every timed call is enqueued on the key's stream between two CUDA events; each leg is warmed up, then repeated and reported as
median / min / max.  Inputs are valid ciphertexts (encrypted on the GPU from the seeded workload units), so the decryption leg
runs on what it is meant for.  Every unit of the timed full-width and 32-bit scalar batches is compared with OpenSSL
(oracle/scalar_cpu.cpp).  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import cpu_ref, scalar_oracle  # noqa: E402
from paillier_halo2_b200 import workload  # noqa: E402
from paillier_halo2_b200.api import PaillierKey, private_from_primes  # noqa: E402

N_BITS = 2048
UNITS = 1 << 16          # scalar multiplications and decryptions per timed call
TALLY_UNITS = 1 << 20    # ciphertexts of the weighted and plain tallies


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.strip().split(",")) if q.returncode == 0 else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(torch, stream, fn, reps: int, warmup: int) -> dict:
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
    return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "reps": reps}


def rate(t: dict, units: int) -> dict:
    return {"per_s_median": units / t["ms_median"] * 1e3, "per_s_min": units / t["ms_max"] * 1e3, "per_s_max": units / t["ms_min"] * 1e3}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON record (default: stdout only)")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to fall back to")
    kd = workload.load_key(N_BITS)
    n, g = kd["n"], kd["g_rand"]
    wi, wo = N_BITS // 64, 2 * N_BITS // 64
    rng = np.random.Generator(np.random.Philox(key=20261020))
    k_full = rng.integers(0, 1 << 64, size=(UNITS, wi), dtype=np.uint64)
    k_32 = rng.integers(0, 1 << 32, size=(UNITS, 1), dtype=np.uint64)
    w_full = rng.integers(0, 1 << 64, size=(TALLY_UNITS, wi), dtype=np.uint64)
    w_32 = rng.integers(0, 1 << 32, size=(TALLY_UNITS, 1), dtype=np.uint64)
    rec = {"tool": "tools/scalar_bench.py", "n_bits": N_BITS, "g": "random", "card": card(), "units": UNITS, "tally_units": TALLY_UNITS}
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()      # noqa: E731
    with PaillierKey(n, g, N_BITS, 64) as key:
        key.set_private(*private_from_primes(kd["p"], kd["q"], g))
        rec["engine"] = key.engine
        stream = torch.cuda.ExternalStream(key.stream)
        # valid ciphertexts: 2^20 encryptions of the seeded workload units; the first 2^16 are the scalar / decrypt batch
        m_w, r_w = workload.units(N_BITS, TALLY_UNITS)
        d_m, d_r = dev(m_w), dev(r_w)
        d_c = torch.empty((TALLY_UNITS, wo), dtype=torch.int64, device="cuda")
        key.encrypt_dev(d_m.data_ptr(), d_r.data_ptr(), TALLY_UNITS, d_c.data_ptr())
        key.sync()
        del d_m, d_r
        d_kf, d_k32, d_wf, d_w32 = dev(k_full), dev(k_32), dev(w_full), dev(w_32)
        d_out = torch.empty((UNITS, wo), dtype=torch.int64, device="cuda")
        d_dec = torch.empty((UNITS, wi), dtype=torch.int64, device="cuda")
        d_t = torch.empty(wo, dtype=torch.int64, device="cuda")
        c, out, t = d_c.data_ptr(), d_out.data_ptr(), d_t.data_ptr()
        legs = {
            "scalar_full": (lambda: key.scalar_mul_dev(c, d_kf.data_ptr(), N_BITS, UNITS, out), UNITS),
            "scalar_32": (lambda: key.scalar_mul_dev(c, d_k32.data_ptr(), 32, UNITS, out), UNITS),
            "decrypt": (lambda: key.decrypt_dev(c, UNITS, d_dec.data_ptr()), UNITS),
            "tally_weighted_32": (lambda: key.tally_weighted_dev(c, d_w32.data_ptr(), 32, TALLY_UNITS, t), TALLY_UNITS),
            "tally_weighted_full": (lambda: key.tally_weighted_dev(c, d_wf.data_ptr(), N_BITS, TALLY_UNITS, t), TALLY_UNITS),
            "tally": (lambda: key.tally_dev(c, TALLY_UNITS, t), TALLY_UNITS),
        }
        res = {}
        for name, (fn, units) in legs.items():
            tm = timed(torch, stream, fn, args.reps, args.warmup)
            res[name] = {**tm, **rate(tm, units)}
            print(name, json.dumps(res[name]), flush=True)
        assert key.take_flags() == 0
        rec["legs"] = res
        rec["scalar_full_over_decrypt"] = res["scalar_full"]["per_s_median"] / res["decrypt"]["per_s_median"]
        # every unit of the timed scalar batches against OpenSSL
        c_host = d_c[:UNITS].cpu().numpy().view(np.uint64)
        threads = cpu_ref.hardware_threads()
        checks = {}
        for name, kw, d_kw, kb in (("scalar_full", k_full, d_kf, N_BITS), ("scalar_32", k_32, d_k32, 32)):
            key.scalar_mul_dev(c, d_kw.data_ptr(), kb, UNITS, out)
            key.sync()
            got = d_out.cpu().numpy().view(np.uint64)
            t0 = time.time()
            want = scalar_oracle.scalar_batch(n, wi, c_host, kw, threads=threads)
            bad = int((got != want).any(axis=1).sum())
            checks[name] = {"units": UNITS, "mismatches": bad, "openssl_threads": threads, "openssl_s": round(time.time() - t0, 1)}
            print(name, "check", json.dumps(checks[name]), flush=True)
        rec["check_vs_openssl"] = checks
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
    if any(v["mismatches"] for v in checks.values()):
        raise SystemExit("scalar batch differs from OpenSSL")


if __name__ == "__main__":
    main()
