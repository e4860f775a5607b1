"""Reference of homomorphic scalar multiplication and the weighted tally: Python ints, and a threaded OpenSSL batch
(oracle/scalar_cpu.cpp, built into oracle/_build/libscalar_cpu.so) for the large parity checks.

TEST / MEASUREMENT INFRASTRUCTURE ONLY (tests/test_gpu_scalar.py, tools/scalar_bench.py).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "scalar_cpu.cpp")
LIB_PATH = os.path.join(HERE, "_build", "libscalar_cpu.so")
u64p = C.POINTER(C.c_uint64)
_lib = None


def paillier_scalar_native(n: int, c: int, k: int) -> int:
    """c^(k mod n) mod n^2: the ciphertext of k * Dec(c) mod n.  c may be any non-negative value; k is reduced mod n first, so a
    negative weight -s is n - s."""
    n2 = n * n
    if n2 == 0:
        raise ZeroDivisionError("modpow with zero modulus (num-bigint panics)")
    return pow(c, k % n, n2)


def tally_weighted_native(n: int, cs: Sequence[int], ks: Sequence[int]) -> int:
    """prod c_i^(k_i mod n) mod n^2: the ciphertext of sum k_i * m_i mod n; the empty product is 1 mod n^2."""
    n2 = n * n
    acc = 1 % n2
    for c, k in zip(cs, ks, strict=True):
        acc = (acc * paillier_scalar_native(n, c, k)) % n2
    return acc


def build() -> str:
    """Compile the OpenSSL batch when it is missing or older than its source."""
    if not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(SRC):
        os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
        cxx = os.environ.get("CXX", "g++")
        subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-o", LIB_PATH, SRC, "-lcrypto", "-lpthread"],
                       check=True, capture_output=True)
    return LIB_PATH


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        lib = C.CDLL(LIB_PATH)
        lib.cpu_paillier_scalar_batch.restype = C.c_int
        lib.cpu_paillier_scalar_batch.argtypes = [u64p, C.c_int, u64p, u64p, C.c_int, C.c_size_t, u64p, C.c_int]
        _lib = lib
    return _lib


def scalar_batch(n: int, words_in: int, c_w: np.ndarray, k_w: np.ndarray, threads: int = 1) -> np.ndarray:
    """c[u]^k[u] mod n^2 per unit with OpenSSL; c_w: (count, 2 words_in) words, k_w: (count, k_words) words."""
    lib = load()
    c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, 2 * words_in)
    count = c_w.shape[0]
    k_w = np.ascontiguousarray(k_w, dtype="<u8").reshape(count, -1)
    n_w = np.frombuffer(int(n).to_bytes(8 * words_in, "little"), dtype="<u8").copy()
    out = np.empty((count, 2 * words_in), dtype="<u8")
    rc = lib.cpu_paillier_scalar_batch(n_w.ctypes.data_as(u64p), words_in, c_w.ctypes.data_as(u64p), k_w.ctypes.data_as(u64p),
                                       k_w.shape[1], count, out.ctypes.data_as(u64p), threads)
    assert rc == 0
    return out
