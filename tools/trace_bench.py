#!/usr/bin/env python
"""Running-tally trace (pb200_tally_trace) on one GPU at |n| = 2048, random g, against the tally and the per-step pb200_add_batch
measured in the same process.

    python tools/trace_bench.py --out profiles/trace_bench_r05.json
    python tools/trace_bench.py --profile --out profiles/trace_bench_r05.json     # adds the per-kernel split (a run of its own)

Legs:
  (a) pb200_tally_trace_dev, 2^20 steps x 1 chain, with q
  (b) pb200_tally_trace (host variant) on the same steps: staging, the trace and the device-to-host copy of acc and q (1 GiB)
  (c) pb200_tally_trace_dev, 2^14 steps x 64 chains, with q
  (d) pb200_tally_dev of the same 2^20 ciphertexts: the A/B reference (the same products, without the intermediate values)
  (e) pb200_add_batch_dev once per step, each step's rem the next step's a, for 4096 steps: the sequential baseline, reported per step
      and extrapolated (labelled so) to 2^20 steps
Device legs are timed with CUDA events on the key's stream after warm-up (median, min, max of --reps calls); the host leg with a host
clock around the call, which ends in a synchronise.  Inputs are uniform values below n^2, 512 MiB per 2^20 ciphertexts: larger than
the 126 MB L2, so no flush is needed.  Every leg is checked: the last acc of each chain equals the tally of init and its column, and
1000 random steps (all of (e)) satisfy (q_i, acc_i) = divmod(acc_(i-1) c_i, n^2) in Python ints.  The device-to-host copy bandwidth
(pageable and pinned host memory) is measured in the same run for leg (b).  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from paillier_halo2_b200 import _lib, workload  # noqa: E402
from paillier_halo2_b200.api import PaillierKey, words_to_ints  # noqa: E402

N_BITS = 2048
N = 1 << 20
C_STEPS, C_CHAINS = 1 << 14, 64
E_STEPS = 4096


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


def check_steps(n2: int, init, c_w, acc_w, q_w, chains: int, steps, tallies) -> dict:
    """(q_i, acc_i) = divmod(acc_(i-1) c_i, n^2) on the given (step, chain) pairs; the last acc of every chain equals its tally"""
    count = c_w.shape[0] // chains
    bad = 0
    for i, j in steps:
        e = i * chains + j
        a = init[j] if i == 0 else words_to_ints(acc_w[e - chains:e - chains + 1])[0]
        q, r = divmod(a * words_to_ints(c_w[e:e + 1])[0], n2)
        bad += (q, r) != (words_to_ints(q_w[e:e + 1])[0], words_to_ints(acc_w[e:e + 1])[0])
    last = words_to_ints(acc_w[(count - 1) * chains:count * chains])
    return {"steps_checked": len(steps), "steps_bad": bad, "last_equals_tally": last == tallies}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON record (default: stdout only); with --profile, the record to add the split to")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--profile", action="store_true", help="only the per-kernel split of one call of legs (a) and (c)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to fall back to")
    os.environ.pop("PB200_TRACE_LANES", None)
    kd = workload.load_key(N_BITS)
    n, g = kd["n"], kd["g_rand"]
    n2, wo = n * n, 2 * N_BITS // 64
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    c_w = workload.ciphertexts(N_BITS, N, n, seed_offset=71)
    init_w = workload.ciphertexts(N_BITS, C_CHAINS, n, seed_offset=72)
    init = words_to_ints(init_w)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()  # noqa: E731
    rng = random.Random(20261021)
    with PaillierKey(n, g, N_BITS, 64) as key:
        stream = torch.cuda.ExternalStream(key.stream)
        torch.cuda.set_stream(stream)                                  # torch's own copies and kernels are ordered with the key's work
        d_c, d_i = dev(c_w), dev(init_w)
        d_acc = torch.empty((N, wo), dtype=torch.int64, device="cuda")
        d_q = torch.empty_like(d_acc)
        d_t = torch.empty((C_CHAINS, wo), dtype=torch.int64, device="cuda")
        leg_a = lambda: key.tally_trace_dev(d_i.data_ptr(), d_c.data_ptr(), N, 1, d_acc.data_ptr(), d_q.data_ptr())  # noqa: E731
        leg_c = lambda: key.tally_trace_dev(d_i.data_ptr(), d_c.data_ptr(), C_STEPS, C_CHAINS, d_acc.data_ptr(), d_q.data_ptr())  # noqa: E731
        if args.profile:
            leg_a(); leg_c(); key.sync()                                                   # noqa: E702  warm-up
            split = {"a_2^20x1": kernel_split(torch, stream, leg_a), "c_2^14x64": kernel_split(torch, stream, leg_c)}
            rec = json.load(open(args.out)) if args.out and os.path.exists(args.out) else {}
            rec["kernel_split_ms"] = split
            rec["kernel_split_card"] = card()
            print(json.dumps(split))
            if args.out:
                json.dump(rec, open(args.out, "w"), indent=1)
            return
        rec = {"tool": "tools/trace_bench.py", "n_bits": N_BITS, "g": "random", "card": card(), "sms": sms, "reps": args.reps,
               "warmup": args.warmup, "engine": key.engine, "witness_engine": key.witness_engine,
               "inputs": "uniform below n^2, larger than L2 (512 MiB per 2^20 ciphertexts), no flush"}
        # (d) the tally of init_0 and the 2^20 ciphertexts (the reference: also the check of (a) and (b))
        d_ic = torch.cat([d_i[:1], d_c])
        leg_d = lambda: key.tally_dev(d_ic.data_ptr(), N + 1, d_t.data_ptr())  # noqa: E731
        rec["d_tally_2^20"] = timed(torch, stream, leg_d, args.reps, args.warmup)
        key.sync()
        tally_a = words_to_ints(d_t[:1].cpu().numpy().view(np.uint64))
        # (a)
        rec["a_trace_dev_2^20x1"] = timed(torch, stream, leg_a, args.reps, args.warmup)
        key.sync()
        assert key.take_flags() == 0
        steps = [(0, 0), (N - 1, 0)] + [(rng.randrange(N), 0) for _ in range(998)]
        acc_h, q_h = d_acc.cpu().numpy().view(np.uint64), d_q.cpu().numpy().view(np.uint64)
        rec["a_trace_dev_2^20x1"]["check"] = check_steps(n2, init, c_w, acc_h, q_h, 1, steps, tally_a)
        rec["a_over_d"] = rec["a_trace_dev_2^20x1"]["ms_median"] / rec["d_tally_2^20"]["ms_median"]
        rec["a_ns_per_step"] = rec["a_trace_dev_2^20x1"]["ms_median"] * 1e6 / N
        # (b) host variant, and the device-to-host copy bandwidth of the same run
        out_a, out_q = np.empty((N, 1, wo), dtype="<u8"), np.empty((N, 1, wo), dtype="<u8")
        ms = []
        u64p = lambda a: a.ctypes.data_as(_lib.u64p)  # noqa: E731
        for r in range(args.warmup + args.reps):
            t0 = time.perf_counter()
            rc = key._lib.pb200_tally_trace(key.handle, u64p(init_w), u64p(c_w), N, 1, u64p(out_a), u64p(out_q))
            t1 = time.perf_counter()
            assert rc == 0, rc
            if r >= args.warmup:
                ms.append((t1 - t0) * 1e3)
        bytes_out = 2 * N * wo * 8
        rec["b_trace_host_2^20x1"] = {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "reps": args.reps,
                                     "bytes_in": N * wo * 8, "bytes_out": bytes_out, "clock": "host perf_counter around the call"}
        rec["b_trace_host_2^20x1"]["check"] = check_steps(n2, init, c_w, out_a.reshape(N, wo), out_q.reshape(N, wo), 1, steps, tally_a)
        rec["b_trace_host_2^20x1"]["same_as_a"] = bool((out_a.reshape(N, wo) == acc_h).all() and (out_q.reshape(N, wo) == q_h).all())
        src = torch.empty(bytes_out // 8, dtype=torch.int64, device="cuda")
        for kind, host in (("pageable", torch.empty(bytes_out // 8, dtype=torch.int64)),
                           ("pinned", torch.empty(bytes_out // 8, dtype=torch.int64, pin_memory=True))):
            t = []
            for r in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                host.copy_(src)
                torch.cuda.synchronize()
                t.append(time.perf_counter() - t0)
            rec[f"d2h_copy_{kind}_GBps"] = bytes_out / min(t) / 1e9
            del host
        del src
        # (c) 2^14 steps x 64 chains
        rec["c_trace_dev_2^14x64"] = timed(torch, stream, leg_c, args.reps, args.warmup)
        key.sync()
        assert key.take_flags() == 0
        nc = C_STEPS * C_CHAINS
        acc_c, q_c = d_acc[:nc].cpu().numpy().view(np.uint64), d_q[:nc].cpu().numpy().view(np.uint64)
        tallies = []
        for j in range(C_CHAINS):
            col = torch.cat([d_i[j:j + 1], d_c[:nc].view(C_STEPS, C_CHAINS, wo)[:, j]]).contiguous()
            key.tally_dev(col.data_ptr(), C_STEPS + 1, d_t[j:j + 1].data_ptr())
        key.sync()
        tallies = words_to_ints(d_t.cpu().numpy().view(np.uint64))
        steps_c = [(rng.randrange(C_STEPS), rng.randrange(C_CHAINS)) for _ in range(1000)]
        rec["c_trace_dev_2^14x64"]["check"] = check_steps(n2, init, c_w[:nc], acc_c, q_c, C_CHAINS, steps_c, tallies)
        rec["c_ns_per_step"] = rec["c_trace_dev_2^14x64"]["ms_median"] * 1e6 / nc
        # (e) the sequential baseline: one pb200_add_batch_dev per step
        d_a = torch.empty((E_STEPS + 1, wo), dtype=torch.int64, device="cuda")
        d_eq = torch.empty((E_STEPS, wo), dtype=torch.int64, device="cuda")
        row = wo * 8

        def leg_e():
            d_a[0].copy_(d_i[0])
            for i in range(E_STEPS):
                key.add_dev(d_a.data_ptr() + i * row, d_c.data_ptr() + i * row, wo, 1, d_a.data_ptr() + (i + 1) * row, d_eq.data_ptr() + i * row)
        rec["e_add_batch_per_step_4096"] = timed(torch, stream, leg_e, max(3, args.reps // 2), 1)
        key.sync()
        e_acc, e_q = d_a[1:].cpu().numpy().view(np.uint64), d_eq.cpu().numpy().view(np.uint64)
        rec["e_add_batch_per_step_4096"]["same_as_trace"] = bool((e_acc == acc_h[:E_STEPS]).all() and (e_q == q_h[:E_STEPS]).all())
        rec["e_add_batch_per_step_4096"]["check"] = check_steps(n2, init, c_w[:E_STEPS], e_acc, e_q, 1, [(i, 0) for i in range(E_STEPS)],
                                                                words_to_ints(acc_h[E_STEPS - 1:E_STEPS]))
        rec["e_us_per_step"] = rec["e_add_batch_per_step_4096"]["ms_median"] * 1e3 / E_STEPS
        rec["e_extrapolated_ms_2^20"] = rec["e_us_per_step"] * N / 1e3
        rec["a_speedup_over_e_extrapolated"] = rec["e_extrapolated_ms_2^20"] / rec["a_trace_dev_2^20x1"]["ms_median"]
        # (b) less (a): the staging copies, 512 MiB in and 1 GiB out
        rec["b_transfer_GBps"] = (N * wo * 8 + bytes_out) / (rec["b_trace_host_2^20x1"]["ms_median"] - rec["a_trace_dev_2^20x1"]["ms_median"]) / 1e6
    print(json.dumps(rec, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(rec, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
