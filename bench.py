#!/usr/bin/env python
"""bench.py — Paillier enc/s at |n|=2048 on N B200s (BASELINE.json metric), one JSON line on stdout.

    python bench.py --gpus N --steps K --warmup W            # our arm   (N>1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: CPU path on the host cores

A step is one pass of the hot path over one batch: encrypt 2^16 independent (m, r) pairs under one
2048-bit key (BASELINE.json configs[1]; SURVEY.md §8d inputs: seeded Paillier key, random g in
[2, 2^|n|), full-width Philox m, r).  `value` times the device-resident call (inputs already in HBM) with
CUDA events on the stream the kernel is launched on; `e2e` times the host-buffer C-ABI call
(pb200_encrypt_batch: pinned host -> device, kernel, device -> host) by wall clock around the blocking call.
Multi-GPU: units are independent, so each rank encrypts its own 2^16 units (weak scaling, no data-path
collective); the time is the max over ranks.
`--dump-outputs DIR` writes a fixed sample of the last timed step's ciphertexts (rank 0) to DIR/ciphertexts.npy, so that two
builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The contract is ONE JSON line on stdout.  NCCL prints its version banner to file descriptor 1 when the first communicator is
# created, so everything except the result line is sent to stderr: fd 1 is duplicated for the result, then pointed at fd 2.
_RESULT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict) -> None:
    _RESULT.write(json.dumps(line) + "\n")
    _RESULT.flush()


N_BITS = 2048
UNITS = 1 << 16
# dram__bytes_read.sum + dram__bytes_write.sum of one k_encrypt launch (ncu --set full, profiles/), keyed by (|n|, units)
TRAFFIC_BYTES = {(2048, 1 << 16): 12073794000 + 1481068000}   # profiles/ncu_k_encrypt_r02_block28u_summary.txt (comb-table gathers + r-power scratch)
METRIC = "paillier_enc_per_s_n2048"
UNIT = "enc/s"


def imad_pipe(key, n_sqr, n_mul, units, kernel_s, peak):
    """IMAD.WIDE instructions per lane the fast engines EXECUTE for the per-ciphertext product (phase A): L^2 per multiplication,
    L (L + 1) / 2 per squaring over L = G * BL signed 28-bit digits; None for the other engines"""
    try:
        import ctypes as _C
        g, bl = _C.c_int(), _C.c_int()
        if key._lib.pb200_key_shape(key.handle, _C.byref(g), _C.byref(bl)) != 0 or not key.engine.startswith("block28"):
            return None
        L = g.value * bl.value
        per_enc = n_sqr * (L * (L + 1) // 2) + n_mul * L * L
        rate = units * per_enc / kernel_s
        return {"digits": L, "wide_mac_executed_per_enc": per_enc, "rate_TMAC_s": rate / 1e12, "frac_of_peak": rate / peak,
                "counts": "phase A only (all of it for block28t / block28u; block28 runs the other two products on IMAD as well)"}
    except Exception:      # a reporting extra must never cost the bench line
        return None


def mac_counts(n_bits: int):
    """Algorithmic 32x32->64 MACs per modular multiplication / squaring over n^2 (SURVEY.md §8d):
    W_mul = 2*L32^2 + L32, W_sqr = (L32^2 + L32)/2 + L32^2 + L32, L32 = 2|n|/32."""
    l32 = 2 * n_bits // 32
    return 2 * l32 * l32 + l32, (l32 * l32 + l32) // 2 + l32 * l32 + l32


def imad_peak():
    """P_imad: measured rate of 32x32->64 multiplies (SASS IMAD.WIDE) on this pool's B200, from
    profiles/imad_peak2_r01.json (csrc/microbench/imad_peak2.cu, variant imadw_only: 31.9 per clk per SM,
    half the 32-bit IMAD rate).  MEASURED_PEAKS.json carries no integer-pipe peak."""
    path = os.path.join(ROOT, "profiles", "imad_peak2_r01.json")
    try:
        d = json.load(open(path))
        return max(r["op_per_s"] for r in d["results"] if r["variant"] == "imadw_only"), "profiles/imad_peak2_r01.json (IMAD.WIDE, measured)"
    except Exception:
        return 148 * 32 * 1.965e9, "nominal 148 SM x 32 IMAD.WIDE/clk x 1.965 GHz"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(threads: int, units: int, key: dict):
    """The CPU restatement (oracle/paillier_cpu.cpp: OpenSSL BIGNUM port of src/paillier.rs:87-92) on the
    first `units` units of the same workload, `threads` worker threads.  Returns (enc/s, seconds)."""
    from oracle import cpu_ref
    from paillier_halo2_b200 import workload

    m_w, r_w = workload.units(N_BITS, units)
    t0 = time.perf_counter()
    cpu_ref.enc_batch(key["n"], key["g_rand"], N_BITS // 64, m_w, r_w, threads=threads)
    dt = time.perf_counter() - t0
    return units / dt, dt


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm (OpenSSL port; the Rust original cannot be built
    here) with every host thread, on bounded samples of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_ref
    from paillier_halo2_b200 import workload

    key = workload.load_key(N_BITS)
    threads = cpu_ref.hardware_threads()
    sample = max(64, min(UNITS, 96 * threads))          # ~3 s of CPU work per step at ~35 enc/s/thread
    m_w, r_w = workload.units(N_BITS, sample)
    for _ in range(args.warmup):
        cpu_ref.enc_batch(key["n"], key["g_rand"], N_BITS // 64, m_w[: max(threads, 8)], r_w[: max(threads, 8)], threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_ref.enc_batch(key["n"], key["g_rand"], N_BITS // 64, m_w, r_w, threads=threads)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 (OpenSSL BIGNUM)", "data": "synthetic",
        "config": {"workload": f"batched encrypt |n|={N_BITS}, bounded sample of {sample} units/step of the 2^16-unit batch, random g",
                   "key": "seeded p*q (SURVEY.md 8d)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} units x {args.steps} steps, OpenSSL BN_mod_exp x2 + BN_mod_mul per unit"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def hbm_peak():
    """Measured HBM copy bandwidth of this pool's B200 (driver-written MEASURED_PEAKS.json), else the profiling guide's fallback."""
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def cells_leg(key, kd, n_bits, groups=1 << 16, lookup_bits=15, reps=4):
    """K4 (SURVEY.md 8f-1/2): advice cells of `groups` mul_mod groups, device-resident, CUDA events on the key's stream.
    Algorithmic bytes per group = cells_per_mulmod x 32 B written + 4 x words_out x 8 B read."""
    import numpy as np
    import torch
    from paillier_halo2_b200 import workload
    dev = torch.device("cuda", key.device)
    wo = key.words_out
    c_w = workload.ciphertexts(n_bits, 2 * groups, kd["n"])
    d_a = torch.from_numpy(c_w[:groups].view(np.int64)).to(dev)
    d_b = torch.from_numpy(c_w[groups:].view(np.int64)).to(dev)
    d_rem, d_q = torch.empty_like(d_a), torch.empty_like(d_a)
    key.add_dev(d_a.data_ptr(), d_b.data_ptr(), wo, groups, d_rem.data_ptr(), d_q.data_ptr())
    key.sync()
    per = key.cells_layout(lookup_bits)["cells_per_mulmod"]
    d_cells = torch.empty((groups, per, 4), dtype=torch.int64, device=dev)       # 5.3 GB at |n| = 2048: larger than L2
    stream = torch.cuda.ExternalStream(key.stream, device=dev)
    peak, src = hbm_peak()
    out = {"groups": groups, "lookup_bits": lookup_bits, "cells_per_group": per}
    for mont in (0, 1):
        for _ in range(3):
            key.mulmod_cells_dev(d_a.data_ptr(), d_b.data_ptr(), d_q.data_ptr(), d_rem.data_ptr(), groups, lookup_bits, bool(mont), d_cells.data_ptr())
        key.sync()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            key.mulmod_cells_dev(d_a.data_ptr(), d_b.data_ptr(), d_q.data_ptr(), d_rem.data_ptr(), groups, lookup_bits, bool(mont), d_cells.data_ptr())
            e1.record(stream)
            key.sync()
            ms.append(e0.elapsed_time(e1))
        t = sum(ms) / len(ms) * 1e-3
        gbs = groups * (per * 32 + 4 * wo * 8) / t / 1e9
        out["montgomery" if mont else "canonical"] = {"groups_per_s": groups / t, "ms_per_launch": t * 1e3,
                                                      "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                                                                   "peak_source": src}}
    # parity of one group against the chip restatement (checker only)
    from oracle.paillier_oracle import Assigned, BigUintChip, Context, decompose
    from paillier_halo2_b200.api import _cells_to_ints, words_to_ints
    L = 2 * n_bits // 64
    a0, b0 = words_to_ints(c_w[:1])[0], words_to_ints(c_w[groups:groups + 1])[0]
    n2 = kd["n"] ** 2
    key.mulmod_cells_dev(d_a.data_ptr(), d_b.data_ptr(), d_q.data_ptr(), d_rem.data_ptr(), 1, lookup_bits, False, d_cells.data_ptr())
    key.sync()
    got = _cells_to_ints(d_cells[0].cpu().numpy().view(np.uint64))
    ctx = Context()
    BigUintChip(64, lookup_bits).mul_mod(ctx, Assigned(decompose(a0, L, 64), a0, 64), Assigned(decompose(b0, L, 64), b0, 64),
                                         Assigned(decompose(n2, L, 64), n2, 64))
    out["parity"] = bool(got == ctx.cells)
    del d_cells
    return out


class Ctx:
    """Per-process bench context: rank / world, torch + NCCL, the loaded library."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        from paillier_halo2_b200 import _lib

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the Paillier hot path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.lib = _lib.load()
        self.dev = torch.device("cuda", self.local_rank)
        self.flush_buf = None

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def flush_l2(self):
        if self.flush_buf is None:
            self.flush_buf = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.dev)      # > 126 MB L2
        self.flush_buf.fill_(1)
        self.torch.cuda.synchronize()

    def stream_of(self, key):
        return self.torch.cuda.ExternalStream(key.stream, device=self.dev)

    def launches(self):
        return int(self.lib.pb200_kernel_launches())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def unit_stream(kd, g, m_row, r_row):
    """(q, rem) records of one unit's stream from the Python oracle (checker)."""
    from oracle.paillier_oracle import encrypt_steps
    from paillier_halo2_b200.api import words_to_ints
    mi, ri = words_to_ints(m_row)[0], words_to_ints(r_row)[0]
    c, steps = encrypt_steps(kd["n"], g, mi, ri)
    gs = mi.bit_length() + bin(mi).count("1")
    return c, [(x.q, x.rem) for x in steps[:gs] if x.kind == "mul"] + [(x.q, x.rem) for x in steps[gs:]]


def witness_chain_macs(kd, m_w, n_bits):
    import numpy as np
    from paillier_halo2_b200.api import words_to_ints
    w_mul, w_sqr = mac_counts(n_bits)
    pop_n = bin(kd["n"]).count("1")
    pop_m = float(np.mean([bin(v).count("1") for v in words_to_ints(m_w[:256])]))
    n_sqr, n_mul = kd["n"].bit_length(), pop_n + pop_m + 1
    return n_sqr, n_mul, n_sqr * w_sqr + n_mul * w_mul


class ParityJob:
    """Full-batch witness parity on the host cores, in the background: the CPU chain (oracle/paillier_cpu.cpp: full product +
    div_rem per mul_mod) over the units in index order, in slices, until every unit is done or the time budget is spent.
    A checker: it never feeds the product path."""

    def __init__(self, kd, g, n_bits, m_w, r_w, budget_s, threads):
        self.args = (kd["n"], g, n_bits // 64, m_w, r_w)
        self.budget, self.threads = budget_s, threads
        self.dig, self.cs, self.done, self.backend, self.secs = [], [], 0, None, 0.0
        self.t = threading.Thread(target=self._run, daemon=True)

    def start(self):
        self.t.start()
        return self

    def _run(self):
        import numpy as np
        from oracle import cpu_ref
        n, g, wi, m_w, r_w = self.args
        t0 = time.perf_counter()
        step = max(64, 48 * self.threads)
        rate = None
        while self.done < len(m_w):
            left = self.budget - (time.perf_counter() - t0)
            if left <= 0 or (rate and step / rate > left):
                break
            e = min(len(m_w), self.done + step)
            t1 = time.perf_counter()
            c, d, self.backend = cpu_ref.witness_digest_batch(n, g, wi, m_w[self.done:e], r_w[self.done:e], threads=self.threads)
            rate = (e - self.done) / (time.perf_counter() - t1)
            self.cs.append(c); self.dig.append(d); self.done = e
        self.secs = time.perf_counter() - t0
        self.dig = np.concatenate(self.dig) if self.dig else np.empty(0, dtype="<u8")
        self.cs = np.concatenate(self.cs) if self.cs else np.empty((0, 2 * wi), dtype="<u8")

    def join(self):
        self.t.join()
        return self


def leg_witness(cx, key, kd, g, n_bits, m_w, r_w, d_m, d_r, reps=2):
    """Witness mode, device-resident: the reference's own LSB-first chain with the exact (q, rem) of every mul_mod, digested on the
    device (pb200_encrypt_witness_digest_dev).  Returns (result dict, device digests, device ciphertexts)."""
    torch = cx.torch
    units = m_w.shape[0]
    d_dig = torch.empty(units, dtype=torch.int64, device=cx.dev)
    d_cw = torch.empty((units, key.words_out), dtype=torch.int64, device=cx.dev)
    stream = cx.stream_of(key)
    key.encrypt_witness_digest_dev(d_m.data_ptr(), d_r.data_ptr(), units, d_cw.data_ptr(), d_dig.data_ptr())     # warm-up at full size
    cx.barrier()
    wl0 = cx.launches()
    sampler = ClockSampler(cx.local_rank)
    sampler.start()
    evs = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        key.encrypt_witness_digest_dev(d_m.data_ptr(), d_r.data_ptr(), units, d_cw.data_ptr(), d_dig.data_ptr())
        e1.record(stream)
        evs.append((e0, e1))
    cx.barrier()
    clocks = sampler.stop()
    (w_ms,) = cx.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs) / len(evs))
    n_sqr, n_mul, a_wit = witness_chain_macs(kd, m_w, n_bits)
    peak_w, _ = imad_peak()
    out = {"value": cx.world * units / (w_ms * 1e-3), "unit": "units/s", "engine": key.witness_engine, "arithmetic": key.engine, "ms_per_launch": w_ms,
           "units_per_gpu": units, "records_per_unit": n_sqr + n_mul, "mul_mod_per_s": cx.world * units * (n_sqr + n_mul) / (w_ms * 1e-3),
           "witness_stream_GBps": cx.world * units * (n_sqr + n_mul) * 2 * key.words_out * 8 / (w_ms * 1e-3) / 1e9,
           "chain": {"mod_sqr": n_sqr, "mod_mul": n_mul, "mac_per_unit": a_wit},
           "frac_of_imad_peak": units * a_wit / (w_ms * 1e-3) / peak_w,
           "gpu_launches": int(cx.launches() - wl0), "clocks": clocks, "ms_each": [a.elapsed_time(b) for a, b in evs]}
    return out, d_dig, d_cw


def pcie_d2h_gbs(cx, nbytes=1 << 30):
    """Measured device -> pinned host copy bandwidth of this box (the roof of the witness delivery), best of 3."""
    torch = cx.torch
    src = torch.empty(nbytes, dtype=torch.uint8, device=cx.dev)
    dst = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    best = 0.0
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); dst.copy_(src, non_blocking=True); e1.record()
        torch.cuda.synchronize()
        best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def leg_witness_e2e(cx, key, kd, g, n_bits, m_w, r_w, units, dig_ref=None):
    """The witness DELIVERED: pb200_encrypt_witness_batch with host inputs, every (q, rem) record landing in pinned host memory
    and handed to a sink callback (here: counts bytes, re-hashes the first unit of every 4th piece and compares it with the
    device digest).  Wall clock around the blocking C-ABI call; the roof is the measured device -> host copy bandwidth."""
    import ctypes as C
    import numpy as np
    from paillier_halo2_b200 import _lib
    from paillier_halo2_b200.api import DIGEST_C, DIGEST_INIT, DIGEST_PRIME, MASK64
    wo = key.words_out
    units = min(units, m_w.shape[0])
    cpow = np.empty(2 * wo, dtype=np.uint64)
    c = DIGEST_C
    for j in range(2 * wo):
        cpow[j] = c; c = (c * DIGEST_C) & MASK64
    state = {"bytes": 0, "units": 0, "pieces": 0, "checked": 0, "ok": True}

    def sink(_user, chp):
        ch = chp.contents
        nu = ch.n_units
        offs = np.ctypeslib.as_array(ch.offsets, shape=(nu + 1,))
        total = int(offs[nu])
        state["bytes"] += total * 2 * wo * 8; state["units"] += nu; state["pieces"] += 1
        if dig_ref is not None and state["pieces"] % 4 == 1:
            recs = np.ctypeslib.as_array(ch.records, shape=(total, 2 * wo))[: int(offs[1])]
            with np.errstate(over="ignore"):
                hs = (recs * cpow).sum(axis=1, dtype=np.uint64)
            d = DIGEST_INIT
            for hv in hs.tolist():
                d = ((d ^ hv) * DIGEST_PRIME) & MASK64
            state["checked"] += 1
            state["ok"] = state["ok"] and d == int(dig_ref[ch.first_unit])
        return 0

    cb = _lib.SINK_FN(sink)
    m_h, r_h = np.ascontiguousarray(m_w[:units]), np.ascontiguousarray(r_w[:units])
    c_h = np.empty((units, wo), dtype="<u8")
    p = lambda a: a.ctypes.data_as(_lib.u64p)
    # warm-up: pinned ring, device record buffers and per-key tables are allocated on first use
    _lib.check(cx.lib.pb200_encrypt_witness_batch(key.handle, p(m_h), p(r_h), units, p(c_h), 0, cb, None), "pb200_encrypt_witness_batch")
    d2h = pcie_d2h_gbs(cx)
    for k_ in state:
        state[k_] = True if k_ == "ok" else 0
    cx.barrier()
    t0 = time.perf_counter()
    _lib.check(cx.lib.pb200_encrypt_witness_batch(key.handle, p(m_h), p(r_h), units, p(c_h), 0, cb, None), "pb200_encrypt_witness_batch")
    dt = time.perf_counter() - t0
    dt, d2h_min = cx.max_over_ranks(dt, -d2h)
    gbs = state["bytes"] / dt / 1e9
    return {"value": cx.world * units / dt, "unit": "units/s", "units_per_gpu": units, "seconds": dt, "pieces": state["pieces"],
            "d2h_bytes_per_step": int(state["bytes"] + c_h.nbytes), "h2d_bytes_per_step": int(m_h.nbytes + r_h.nbytes),
            "roofline": {"bound": "pcie_d2h", "achieved": gbs, "peak": -d2h_min, "unit": "GB/s", "frac": gbs / -d2h_min,
                         "peak_source": "device -> pinned host copy of 1 GiB measured in this run (best of 4)"},
            "sink_rehashed_units": state["checked"], "parity": bool(state["ok"] and state["units"] == units)}


def leg_decrypt(cx, key, kd, g, n_bits, d_c, m_w, reps=2):
    """SURVEY.md 8f-4: decrypt the ciphertexts the headline step produced (c^lambda mod n^2 on the key's engine, then the L function
    and the multiplication by mu).  Parity: the round trip must return EVERY plaintext of the batch; a few units against the oracle."""
    import numpy as np
    from paillier_halo2_b200.api import private_from_primes, words_to_ints
    torch = cx.torch
    units = m_w.shape[0]
    lam, mu = private_from_primes(kd["p"], kd["q"], g)
    key.set_private(lam, mu)
    d_m = torch.empty((units, key.words_in), dtype=torch.int64, device=cx.dev)
    stream = cx.stream_of(key)
    key.decrypt_dev(d_c.data_ptr(), units, d_m.data_ptr())
    cx.barrier()
    l0 = cx.launches()
    evs = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); key.decrypt_dev(d_c.data_ptr(), units, d_m.data_ptr()); e1.record(stream)
        evs.append((e0, e1))
    cx.barrier()
    (ms,) = cx.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs) / len(evs))
    flags = key.take_flags()
    got = d_m.cpu().numpy().view(np.uint64)
    ok = bool((got == m_w).all()) and flags == 0
    if cx.rank == 0:
        from oracle.paillier_oracle import paillier_dec_native
        cs = words_to_ints(d_c[:3].cpu().numpy().view(np.uint64))
        ok = ok and words_to_ints(got[:3]) == [paillier_dec_native(kd["n"], lam, mu, c) for c in cs]
    return {"value": cx.world * units / (ms * 1e-3), "unit": "dec/s", "ms_per_launch": ms, "units_per_gpu": units,
            "gpu_launches": int(cx.launches() - l0), "parity": ok, "parity_units": units,
            "note": "m = L(c^lambda mod n^2) * mu mod n; round trip of the headline step's ciphertexts, every plaintext compared"}


DUMP_ROWS = 8192


def dump_ciphertexts(out_dir, c_w):
    """DIR/ciphertexts.npy: DUMP_ROWS ciphertexts spread evenly over the batch (all of them when the batch is smaller), one row
    per ciphertext in little-endian 32-bit limbs stored as float64, which holds every limb exactly (16 MiB at most, |n| = 4096)."""
    import numpy as np
    rows = np.unique(np.linspace(0, c_w.shape[0] - 1, min(DUMP_ROWS, c_w.shape[0])).astype(np.int64))
    limbs = np.ascontiguousarray(c_w[rows], dtype="<u8").view("<u4")
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ciphertexts.npy"), limbs.astype(np.float64))


TALLY_TOTAL = 1 << 20
TALLY_PARTS = 8            # the 2^20 ciphertexts are 8 fixed Philox streams, so the SET is the same for every GPU count


def leg_tally(cx, kd, n_bits, steps, warmup):
    """BASELINE.json configs[2]: product of 2^20 ciphertexts mod n^2 sharded over the GPUs.  Strong scaling (total fixed).  One
    launch per GPU per tally (pb200_tally_peer_dev): shard fold, partials exchanged through peer-mapped memory inside the kernel,
    combine — or, when the peers cannot be mapped, fold + NCCL all-gather + combine."""
    import numpy as np
    from paillier_halo2_b200 import PaillierKey
    from paillier_halo2_b200.shard import connect_tally_peers, tally_sharded_gpu
    torch = cx.torch
    world, rank = cx.world, cx.rank
    key = PaillierKey(kd["n"], kd["g_std"], n_bits, 64, device=cx.local_rank)
    per_part = TALLY_TOTAL // TALLY_PARTS
    from paillier_halo2_b200 import workload
    mine = range(rank * TALLY_PARTS // world, (rank + 1) * TALLY_PARTS // world)
    parts = {s_: workload.ciphertexts(n_bits, per_part, kd["n"], seed_offset=100 + s_) for s_ in (range(TALLY_PARTS) if rank == 0 else mine)}
    shard = np.concatenate([parts[s_] for s_ in mine])
    count = shard.shape[0]
    d_c = torch.from_numpy(shard.view(np.int64)).to(cx.dev)
    out = torch.empty(key.words_out, dtype=torch.int64, device=cx.dev)
    exchange = connect_tally_peers(key, rank, world) if world > 1 else "peer-memory"
    if world == 1:
        key.tally_peer_connect(0, 1, [key.tally_peer_export()])
    stream = cx.stream_of(key)
    for _ in range(max(warmup, 1)):
        tally_sharded_gpu(key, d_c, count, world, exchange=exchange, out=out)
    cx.barrier()
    l0 = cx.launches()
    ms = []
    for _ in range(steps):
        cx.flush_l2()
        cx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        tally_sharded_gpu(key, d_c, count, world, exchange=exchange, out=out)
        e1.record(stream)
        key.sync()
        wall = (time.perf_counter() - t0) * 1e3
        ms.append(cx.max_over_ranks(e0.elapsed_time(e1) if exchange == "peer-memory" else wall)[0])
    launches = cx.launches() - l0
    flags = key.take_flags()
    t = sum(ms) / len(ms) * 1e-3
    res = {"value": TALLY_TOTAL / t, "unit": "ciphertexts/s", "ciphertexts": TALLY_TOTAL, "n_gpus": world, "scaling": "strong",
           "ms_per_tally": t * 1e3, "ms_each": ms, "exchange": exchange, "engine": key.engine, "gpu_launches_per_tally": launches / steps,
           "timing": "CUDA events on the launching stream, max over ranks" if exchange == "peer-memory" else "wall clock around the call, max over ranks",
           "l2": "flushed between tallies (256 MiB write)", "flags": flags}
    if rank == 0:
        from oracle import cpu_ref
        c_all = np.concatenate([parts[s_] for s_ in range(TALLY_PARTS)])
        want = cpu_ref.tally(kd["n"], n_bits // 64, c_all, threads=cpu_ref.hardware_threads())
        res["parity_vs_cpu_fold"] = bool((out.cpu().numpy().view(np.uint64) == want).all())
        w_mul, _ = mac_counts(n_bits)
        peak, src = imad_peak()
        res["roofline"] = {"bound": "imad", "achieved": TALLY_TOTAL * w_mul / t / 1e12, "peak": world * peak / 1e12, "unit": "TMAC/s",
                           "frac": TALLY_TOTAL * w_mul / t / (world * peak), "peak_source": src,
                           "hbm_gbs_achieved": TALLY_TOTAL * key.words_out * 8 / t / 1e9,
                           "note": "whole tally (fold + exchange + combine) against world x P_imad; one modmul per 512 B read (64 MAC/B): "
                                   "compute-bound, HBM GB/s reported because north_star asks for it"}
    key.close()
    return res


def leg_witness_cfg3(cx, steps_units, parity_units=1024):
    """BASELINE.json configs[3]: batched encrypt + full (q, rem) limb witness at |n| = 3072, 2^18 units over 8 GPUs = 32768 units
    per GPU (weak scaling, no collective).  Device digest for every unit; parity: `parity_units` units spread evenly over the
    batch re-derived by the CPU chain; plus the delivery (pb200_encrypt_witness_batch) of a bounded sample."""
    import numpy as np
    from paillier_halo2_b200 import PaillierKey, workload
    torch = cx.torch
    n_bits = 3072
    kd = workload.load_key(n_bits)
    g = kd["g_rand"]
    units = steps_units
    key = PaillierKey(kd["n"], g, n_bits, 64, device=cx.local_rank)
    m_w, r_w = workload.units(n_bits, units, seed_offset=3000 + 1000 * cx.rank)
    d_m = torch.from_numpy(m_w.view(np.int64)).to(cx.dev); d_r = torch.from_numpy(r_w.view(np.int64)).to(cx.dev)
    res, d_dig, d_cw = leg_witness(cx, key, kd, g, n_bits, m_w, r_w, d_m, d_r, reps=2)
    res["config"] = f"|n|=3072, {units} units per GPU ({cx.world * units} in total), (q, rem) of every mul_mod, digested on the device"
    dig = d_dig.cpu().numpy().view(np.uint64)
    res["e2e"] = leg_witness_e2e(cx, key, kd, g, n_bits, m_w, r_w, min(units, 6144), dig)
    if cx.rank == 0:
        from oracle import cpu_ref
        idx = np.unique(np.linspace(0, units - 1, min(parity_units, units)).astype(np.int64))
        t0 = time.perf_counter()
        c, d, backend = cpu_ref.witness_digest_batch(kd["n"], g, n_bits // 64, m_w[idx], r_w[idx], threads=cpu_ref.hardware_threads())
        res["parity"] = bool((d == dig[idx]).all() and (c == d_cw.cpu().numpy().view(np.uint64)[idx]).all())
        res["parity_units"] = int(len(idx))
        res["parity_note"] = f"{len(idx)} units spread evenly over rank 0's batch, CPU chain ({backend}), {time.perf_counter() - t0:.0f} s"
    del d_dig, d_cw, d_m, d_r
    key.close()
    return res


def run_tally(args):
    cx = Ctx()
    from paillier_halo2_b200 import workload
    kd = workload.load_key(N_BITS)
    res = leg_tally(cx, kd, N_BITS, args.steps, args.warmup)
    if cx.rank == 0:
        line = {"metric": f"paillier_tally_ciphertexts_per_s_n{N_BITS}", "value": res["value"], "unit": "ciphertexts/s", "n_gpus": cx.world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_tally"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "int64 accumulators over signed 28-bit digits", "data": "synthetic",
                "config": {"workload": f"product of 2^20 ciphertexts mod n^2, |n|={N_BITS}, sharded over {cx.world} GPU(s) (BASELINE.json configs[2])"},
                "gpu_launches": int(res["gpu_launches_per_tally"] * args.steps), "tally": res, "roofline": res.get("roofline")}
        emit(line)
    cx.close()


def run_witness(args):
    """`--workload witness`: the witness leg alone at --n-bits / --units (key-size sweep of the witness engine)."""
    import numpy as np
    from paillier_halo2_b200 import PaillierKey, workload
    cx = Ctx()
    torch = cx.torch
    kd = workload.load_key(N_BITS)
    g = kd["g_rand"]
    units = args.units
    key = PaillierKey(kd["n"], g, N_BITS, 64, device=cx.local_rank)
    m_w, r_w = workload.units(N_BITS, units, seed_offset=1000 * cx.rank)
    d_m = torch.from_numpy(m_w.view(np.int64)).to(cx.dev); d_r = torch.from_numpy(r_w.view(np.int64)).to(cx.dev)
    res, d_dig, d_cw = leg_witness(cx, key, kd, g, N_BITS, m_w, r_w, d_m, d_r, reps=max(args.steps, 1))
    if cx.rank == 0:
        from oracle import cpu_ref
        idx = np.unique(np.linspace(0, units - 1, min(512, units)).astype(np.int64))
        c, d, backend = cpu_ref.witness_digest_batch(kd["n"], g, N_BITS // 64, m_w[idx], r_w[idx], threads=cpu_ref.hardware_threads())
        res["parity"] = bool((d == d_dig.cpu().numpy().view(np.uint64)[idx]).all() and (c == d_cw.cpu().numpy().view(np.uint64)[idx]).all())
        res["parity_units"] = int(len(idx))
        peak, src = imad_peak()
        line = {"metric": f"paillier_witness_units_per_s_n{N_BITS}", "value": res["value"], "unit": "units/s", "n_gpus": cx.world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_launch"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64 columns over signed 28-bit digits + s8 tensor-core phases, exact (q, rem) tail", "data": "synthetic",
                "config": {"workload": f"batched encrypt + (q, rem) limb witness of every mul_mod, |n|={N_BITS}, {units} units per GPU per step"},
                "gpu_launches": res["gpu_launches"], "clocks": res["clocks"], "parity": res["parity"], "witness": res,
                "roofline": {"bound": "imad", "achieved": res["frac_of_imad_peak"] * peak / 1e12, "peak": peak / 1e12, "unit": "TMAC/s",
                             "frac": res["frac_of_imad_peak"], "peak_source": src, "traffic": None}}
        emit(line)
    key.close()
    cx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--units", type=int, default=UNITS, help="units per GPU per step (default: the BASELINE config, 2^16)")
    ap.add_argument("--g", default="rand", choices=["rand", "std"], help="rand: random g (headline); std: g = n+1")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg and the full-batch CPU witness parity")
    ap.add_argument("--no-witness", action="store_true", help="only the headline encrypt leg (used for ncu captures)")
    ap.add_argument("--skip", default="", help="comma-separated legs to skip: witness,witness_e2e,decrypt,tally,cells,witness3072")
    ap.add_argument("--parity-budget", type=float, default=float(os.environ.get("PB200_PARITY_BUDGET_S", "240")),
                    help="seconds of host time the full-batch CPU witness parity may take (units are checked in index order)")
    ap.add_argument("--engine", type=int, default=0)
    ap.add_argument("--n-bits", type=int, default=2048, help="key size |n| (default 2048, the BASELINE metric; others are the sweep)")
    ap.add_argument("--workload", default="encrypt", choices=["encrypt", "tally", "witness"],
                    help="encrypt: the BASELINE metric with every leg (default); tally: configs[2] alone; witness: the witness leg alone "
                         "at --n-bits / --units")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's ciphertexts to DIR/ciphertexts.npy (encrypt workload, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "encrypt"):
        ap.error("--dump-outputs covers the encrypt workload of --impl ours")
    global N_BITS, METRIC
    N_BITS = args.n_bits
    METRIC = f"paillier_enc_per_s_n{N_BITS}"
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "tally":
        return run_tally(args)
    if args.workload == "witness":
        return run_witness(args)

    import numpy as np

    from paillier_halo2_b200 import PaillierKey, _lib, workload

    cx = Ctx()
    torch, lib, world, rank, local_rank = cx.torch, cx.lib, cx.world, cx.rank, cx.local_rank
    skip = set(x for x in args.skip.split(",") if x)
    if args.no_witness:
        skip |= {"witness", "witness_e2e", "tally", "cells", "witness3072", "decrypt"}
    kd = workload.load_key(N_BITS)
    g = kd["g_rand"] if args.g == "rand" else kd["g_std"]
    units = args.units
    key = PaillierKey(kd["n"], g, N_BITS, 64, device=local_rank)
    if args.engine:
        key.set_engine(args.engine)
    n_sqr, n_mul = key.chain_counts()
    w_mul, w_sqr = mac_counts(N_BITS)
    a_enc = n_sqr * w_sqr + n_mul * w_mul

    # this rank's units: rank r takes the r-th 2^16-unit slice of the Philox stream
    m_w, r_w = workload.units(N_BITS, units, seed_offset=1000 * rank)
    m_pin = torch.from_numpy(m_w.view(np.int64)).pin_memory()
    r_pin = torch.from_numpy(r_w.view(np.int64)).pin_memory()
    c_pin = torch.empty((units, key.words_out), dtype=torch.int64).pin_memory()
    d_m = m_pin.cuda(non_blocking=False)
    d_r = r_pin.cuda(non_blocking=False)
    d_c = torch.empty((units, key.words_out), dtype=torch.int64, device="cuda")
    stream = cx.stream_of(key)
    barrier = cx.barrier

    def step_dev():
        key.encrypt_dev(d_m.data_ptr(), d_r.data_ptr(), units, d_c.data_ptr())

    for _ in range(max(args.warmup, 0)):
        step_dev()
    key.sync()

    # ---- timed: K steps, device-resident inputs, CUDA events on the launching stream, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    launches0 = lib.pb200_kernel_launches()
    barrier()
    sampler.start()
    evs = []
    for _ in range(args.steps):
        cx.flush_l2()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step_dev()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    clocks = sampler.stop()
    launches = lib.pb200_kernel_launches() - launches0
    (dev_ms,) = cx.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))
    value = world * units * args.steps / (dev_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_ciphertexts(args.dump_outputs, d_c.cpu().numpy().view(np.uint64))

    # ---- e2e: the host-buffer C-ABI call, pinned host memory, H2D + kernel + D2H inside the timed region
    import ctypes as C
    hp = [C.cast(t_.data_ptr(), _lib.u64p) for t_ in (m_pin, r_pin, c_pin)]

    def step_host():
        _lib.check(lib.pb200_encrypt_batch(key.handle, hp[0], hp[1], units, hp[2]), "pb200_encrypt_batch")

    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    (e2e_s,) = cx.max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * units * args.steps / e2e_s

    # ---- witness mode (BASELINE.json configs[1]: "witnesses checked bit-exact"), device digests, then the witness delivered
    witness, dig, cw_host, parity_job = None, None, None, None
    if "witness" not in skip:
        witness, d_dig, d_cw = leg_witness(cx, key, kd, g, N_BITS, m_w, r_w, d_m, d_r)
        dig = d_dig.cpu().numpy().view(np.uint64)
        cw_host = d_cw.cpu().numpy().view(np.uint64)
        del d_dig, d_cw
        if "witness_e2e" not in skip:
            witness["e2e"] = leg_witness_e2e(cx, key, kd, g, N_BITS, m_w, r_w, 16384, dig)
    # ---- decryption of the step's ciphertexts (SURVEY.md 8f-4)
    decrypt = leg_decrypt(cx, key, kd, g, N_BITS, d_c, m_w) if "decrypt" not in skip else None
    # ---- tally (configs[2]) before the host cores get busy with the parity job: its launches are sub-millisecond
    tally = leg_tally(cx, kd, N_BITS, 10, 3) if "tally" not in skip else None
    # ---- full-batch witness parity on the host cores, in the background while the remaining GPU legs run
    if witness is not None and rank == 0 and not args.no_cpu:
        from oracle import cpu_ref
        parity_job = ParityJob(kd, g, N_BITS, m_w, r_w, args.parity_budget, cpu_ref.hardware_threads()).start()
    # ---- K4: advice-cell expansion of mul_mod groups (HBM-bound writer), rank 0 only
    cells = cells_leg(key, kd, N_BITS) if ("cells" not in skip and rank == 0) else None
    # ---- configs[3]: |n| = 3072 witness, 32768 units per GPU
    witness3072 = leg_witness_cfg3(cx, 32768) if "witness3072" not in skip else None

    # parity spot check of the last step's output against the CPU port (a checker, never the thing measured)
    parity = None
    if rank == 0:
        from oracle import cpu_ref
        got_dev_all = d_c.cpu().numpy().view(np.uint64)
        if parity_job is not None:
            parity_job.join()
            nd = parity_job.done
            w_ok = bool((parity_job.dig == dig[:nd]).all() and (parity_job.cs == cw_host[:nd]).all())
            fast_ok = bool((parity_job.cs == got_dev_all[:nd]).all() and (cw_host == got_dev_all).all())
            witness["parity"] = w_ok and fast_ok
            witness["parity_units"] = int(nd)
            witness["parity_note"] = (f"digests and ciphertexts of the first {nd} of {units} units re-derived by the CPU chain "
                                      f"(oracle/paillier_cpu.cpp, {parity_job.backend} backend, full product + div_rem per mul_mod, "
                                      f"{parity_job.threads} threads, {parity_job.secs:.0f} s, budget {args.parity_budget:.0f} s); the fast chain's "
                                      f"ciphertexts (k_encrypt) equal them too; all {units} fast-chain and witness-chain ciphertexts agree")
        elif witness is not None:
            idx17 = sorted({0, units - 1} | {(units * t) // 16 for t in range(16)})
            from paillier_halo2_b200.api import witness_digest
            ok = bool((cw_host == got_dev_all).all())
            for i in idx17:
                _, mine = unit_stream(kd, g, m_w[i:i + 1], r_w[i:i + 1])
                ok = ok and int(dig[i]) == witness_digest(mine, key.words_out)
            witness["parity"], witness["parity_units"] = ok, len(idx17)
        idx = [0, 1, units // 2, units - 1]
        want = cpu_ref.enc_batch(kd["n"], g, N_BITS // 64, m_w[idx], r_w[idx], threads=4)
        got_host = c_pin.numpy().view(np.uint64)[idx]
        parity = bool((want == got_dev_all[idx]).all() and (want == got_host).all())

    if rank == 0:
        peak, peak_src = imad_peak()
        kernel_s = dev_ms * 1e-3 / args.steps            # one launch per step per rank
        achieved = units * a_enc / kernel_s
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64 columns over signed 28-bit digits (IMAD.WIDE) + s8 x s8 -> s32 on the tensor core ("
                     + ("tcgen05.mma kind::i8, TMEM accumulators" if key.engine.startswith("block28u") else "mma.sync" if key.engine.startswith("block28t") else "none")
                     + ") for the constant-operand phases", "data": "synthetic",
            "config": {"workload": f"batched encrypt |n|={N_BITS} (4096-bit n^2), {units} units per GPU per step, "
                                   f"{'random g' if args.g == 'rand' else 'g = n+1'}, full-width m and r (BASELINE.json configs[1])",
                       "engine": key.engine, "l2": "flushed between timed steps (256 MiB write)",
                       "chain": {"mod_sqr": n_sqr, "mod_mul": n_mul, "mac_per_enc": a_enc}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(m_pin.numel() * 8 + r_pin.numel() * 8),
                    "d2h_bytes_per_step": int(c_pin.numel() * 8)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "parity_spot_check": parity,
            "witness": witness,
            "tally": tally,
            "witness3072": witness3072,
            "decrypt": decrypt,
            "cells": cells,
            "roofline": {"bound": "imad", "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "TMAC/s (32x32->64 multiply-accumulate)",
                         "frac": achieved / peak, "traffic": TRAFFIC_BYTES.get((N_BITS, units)), "peak_source": peak_src,
                         "note": "algorithmic MACs = units x (mod_sqr x W_sqr + mod_mul x W_mul), W for 32-bit limbs over n^2 "
                                 "(SURVEY.md 8d), against the measured IMAD.WIDE rate; the block28u / block28t engines run the per-ciphertext "
                                 "product on the IMAD pipe and the two constant-operand Barrett products on the tensor core (tcgen05 / "
                                 "mma.sync), so the fraction can exceed what the IMAD pipe alone could deliver; imad_pipe is the share of "
                                 "the measured IMAD.WIDE peak that the 28-bit-digit products of phase A actually executed occupy; "
                                 "HBM is idle by design",
                         "imad_pipe": imad_pipe(key, n_sqr, n_mul, units, kernel_s, peak)},
        }
        if not args.no_cpu and world >= 1:
            from oracle import cpu_ref
            threads = cpu_ref.hardware_threads()
            sample = max(64, min(units, int(256 * threads * (2048 / N_BITS) ** 3)))     # ~3-6 s of CPU work at every key size
            v, dt = cpu_baseline(threads, sample, kd)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"first {sample} units of the same batch, {dt:.1f} s, OpenSSL BIGNUM port of src/paillier.rs:87-92"}
            try:        # second line of SURVEY.md 8d: the Python-int restatement on one core, two units
                from oracle.paillier_oracle import paillier_enc_native as _py_enc
                from paillier_halo2_b200.api import words_to_ints as _w2i
                _ms, _rs = _w2i(m_w[:2]), _w2i(r_w[:2])
                _t0 = time.perf_counter()
                for _m, _r in zip(_ms, _rs):
                    _py_enc(kd["n"], g, _m, _r)
                line["cpu_baseline"]["python_int_enc_per_s_one_core"] = 2 / (time.perf_counter() - _t0)
            except Exception as _e:     # a reporting extra must never cost the bench line
                line["cpu_baseline"]["python_int_enc_per_s_one_core"] = None
        emit(line)
    key.close()
    cx.close()


if __name__ == "__main__":
    main()
