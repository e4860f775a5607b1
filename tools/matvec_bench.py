#!/usr/bin/env python
"""Encrypted matrix-vector product (pb200_matvec) on one GPU at |n| = 2048, against the weighted tally and the chain method measured
in the same process.

    python tools/matvec_bench.py --out profiles/matvec_bench_r04.json

Legs (ciphertexts are valid encryptions of the seeded workload units, made on the GPU):
  (a) R = 1, N = 2^20, 32-bit weights          vs pb200_tally_weighted                 bit-exact
  (b) R = 1, N = 2^20, full-width weights      vs pb200_tally_weighted                 bit-exact
  (c) R = 1, N = 2^20, weights in {-1, 0, +1}  vs pb200_tally_weighted with n - 1      decryption equals sum w m
  (d) R = 256, N = 4096, signed 16-bit weights vs 256 one-row calls of the chain method bit-exact
Every timed call is enqueued on the key's stream between two CUDA events, after warm-up; each leg reports median / min / max.  Per
leg: the planner's mulmods (pb200_matvec_plan, dense upper bounds) and the resulting mulmods/s next to the plain tally's fold rate
(one mulmod per ciphertext) of the same run, and the GPU time per kernel of one call (torch.profiler).  The card's name and power
limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from paillier_halo2_b200 import workload  # noqa: E402
from paillier_halo2_b200.api import PaillierKey, matvec_plan, private_from_primes, words_to_ints  # noqa: E402

N_BITS = 2048
N = 1 << 20
R_D, N_D = 256, 4096


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


def kernel_split(torch, stream, fn) -> dict:
    """GPU milliseconds per kernel name over one call"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        stream.synchronize()
    split = {}
    for ev in prof.key_averages():
        if ev.device_time_total <= 0:
            continue
        name = ev.key.split("(")[0].split("<")[0].replace("void ", "").replace("pb200::", "").strip()
        split[name] = round(split.get(name, 0.0) + ev.device_time_total / 1e3, 3)
    return split


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON record (default: stdout only)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to fall back to")
    os.environ.pop("PB200_MATVEC_METHOD", None)
    os.environ.pop("PB200_MATVEC_PASS_ENTRIES", None)
    kd = workload.load_key(N_BITS)
    n, g = kd["n"], kd["g_rand"]
    wi, wo = N_BITS // 64, 2 * N_BITS // 64
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.Generator(np.random.Philox(key=20261021))
    w32 = rng.integers(0, 1 << 32, size=(N, 1), dtype=np.uint64)
    wfull = rng.integers(0, 1 << 64, size=(N, wi), dtype=np.uint64)
    w3 = rng.integers(-1, 2, size=N, dtype=np.int64)
    w3_mag = np.abs(w3).astype(np.uint64).reshape(N, 1)
    w3_neg = (w3 < 0).astype(np.uint8)
    nm1 = np.frombuffer((n - 1).to_bytes(8 * wi, "little"), dtype="<u8")
    w3_tw = np.zeros((N, wi), dtype=np.uint64)                            # the same weights for the weighted tally: -1 as n - 1
    w3_tw[w3 == 1, 0] = 1
    w3_tw[w3 == -1] = nm1
    wd = rng.integers(-(1 << 16) + 1, 1 << 16, size=(R_D, N_D), dtype=np.int64)
    wd_mag = np.abs(wd).astype(np.uint64).reshape(R_D, N_D, 1)
    wd_neg = (wd < 0).astype(np.uint8)
    rec = {"tool": "tools/matvec_bench.py", "n_bits": N_BITS, "g": "random", "card": card(), "sms": sms, "reps": args.reps,
           "warmup": args.warmup}
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64) if a.dtype != np.uint8 else np.ascontiguousarray(a)).cuda()  # noqa: E731
    with PaillierKey(n, g, N_BITS, 64) as key:
        key.set_private(*private_from_primes(kd["p"], kd["q"], g))
        rec["engine"] = key.engine
        stream = torch.cuda.ExternalStream(key.stream)
        m_w, r_w = workload.units(N_BITS, N)
        d_m, d_r = dev(m_w), dev(r_w)
        d_c = torch.empty((N, wo), dtype=torch.int64, device="cuda")
        key.encrypt_dev(d_m.data_ptr(), d_r.data_ptr(), N, d_c.data_ptr())
        key.sync()
        del d_m, d_r
        c = d_c.data_ptr()
        d_w32, d_wf, d_w3, d_w3n, d_w3tw = dev(w32), dev(wfull), dev(w3_mag), dev(w3_neg), dev(w3_tw)
        d_wd, d_wdn = dev(wd_mag), dev(wd_neg)
        d_o = [torch.empty(wo, dtype=torch.int64, device="cuda") for _ in range(2)]
        d_od = torch.empty((R_D, wo), dtype=torch.int64, device="cuda")
        d_odc = torch.empty((R_D, wo), dtype=torch.int64, device="cuda")
        o0, o1 = d_o[0].data_ptr(), d_o[1].data_ptr()
        kw16 = wo                                                            # words per (1, N_D)-row of d_wd: 1 word per weight

        def chain_rows():
            os.environ["PB200_MATVEC_METHOD"] = "chain"
            try:
                for r in range(R_D):
                    key.matvec_dev(c, N_D, d_wd.data_ptr() + r * N_D * 8, d_wdn.data_ptr() + r * N_D, 16, 1, d_odc.data_ptr() + r * kw16 * 8)
            finally:
                os.environ.pop("PB200_MATVEC_METHOD", None)

        legs = {
            "a_32bit": ((lambda: key.matvec_dev(c, N, d_w32.data_ptr(), None, 32, 1, o0)),
                        (lambda: key.tally_weighted_dev(c, d_w32.data_ptr(), 32, N, o1)), (1, N, 32, False)),
            "b_full": ((lambda: key.matvec_dev(c, N, d_wf.data_ptr(), None, N_BITS, 1, o0)),
                       (lambda: key.tally_weighted_dev(c, d_wf.data_ptr(), N_BITS, N, o1)), (1, N, N_BITS, False)),
            "c_pm1": ((lambda: key.matvec_dev(c, N, d_w3.data_ptr(), d_w3n.data_ptr(), 1, 1, o0)),
                      (lambda: key.tally_weighted_dev(c, d_w3tw.data_ptr(), N_BITS, N, o1)), (1, N, 1, True)),
            "d_256x4096": ((lambda: key.matvec_dev(c, N_D, d_wd.data_ptr(), d_wdn.data_ptr(), 16, R_D, d_od.data_ptr())),
                           chain_rows, (R_D, N_D, 16, True)),
        }
        res, checks = {}, {}
        t_tally = timed(torch, stream, lambda: key.tally_dev(c, N, o1), args.reps, args.warmup)
        tally_rate = N / t_tally["ms_median"] * 1e3
        res["tally"] = {**t_tally, "mulmods_per_s": tally_rate}
        print("tally", json.dumps(res["tally"]), flush=True)
        for name, (mv, base, shape) in legs.items():
            plan = matvec_plan(N_BITS, sms, *shape)
            mulmods = plan["acc_mulmods"] + plan["reduce_mulmods"] + plan["horner_mulmods"] + plan["sign_mulmods"]
            t_mv = timed(torch, stream, mv, args.reps, args.warmup)
            t_base = timed(torch, stream, base, args.reps, args.warmup)
            res[name] = {"plan": plan, "matvec": t_mv, "baseline": t_base, "speedup_median": t_base["ms_median"] / t_mv["ms_median"],
                         "plan_mulmods": mulmods, "mulmods_per_s": mulmods / t_mv["ms_median"] * 1e3,
                         "mulmods_per_s_over_tally": mulmods / t_mv["ms_median"] * 1e3 / tally_rate,
                         "kernels_ms": kernel_split(torch, stream, mv)}
            print(name, json.dumps({k: v for k, v in res[name].items() if k != "kernels_ms"}), flush=True)
            print(name, "kernels", json.dumps(res[name]["kernels_ms"]), flush=True)
            # outputs of the last timed calls
            mv(); base()
            key.sync()
            if name == "d_256x4096":
                got, want = d_od.cpu().numpy().view(np.uint64), d_odc.cpu().numpy().view(np.uint64)
                checks[name] = {"rows": R_D, "mismatches": int((got != want).any(axis=1).sum())}
            elif name == "c_pm1":
                got, want = d_o[0].cpu().numpy().view(np.uint64), d_o[1].cpu().numpy().view(np.uint64)
                ms = words_to_ints(m_w)
                expect = sum(int(w) * m for w, m in zip(w3.tolist(), ms)) % n
                dec = key.decrypt(words_to_ints(np.stack([got, want])))
                checks[name] = {"decrypt_matvec_ok": dec[0] == expect, "decrypt_tally_weighted_ok": dec[1] == expect,
                                "mismatches": int(not (dec[0] == expect and dec[1] == expect))}
            else:
                got, want = d_o[0].cpu().numpy().view(np.uint64), d_o[1].cpu().numpy().view(np.uint64)
                checks[name] = {"mismatches": int((got != want).any())}
            print(name, "check", json.dumps(checks[name]), flush=True)
        assert key.take_flags() == 0
        rec["legs"] = res
        rec["checks"] = checks
    print(json.dumps({k: v for k, v in rec.items() if k != "legs"}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
    if any(v["mismatches"] for v in checks.values()):
        raise SystemExit("matvec output check failed")


if __name__ == "__main__":
    main()
