"""Reference of the encrypted matrix-vector product (pb200_matvec): Python ints, and a threaded OpenSSL batch (tests/matvec_cpu.cpp)
for the larger parity checks.

TEST INFRASTRUCTURE ONLY (tests/test_gpu_matvec.py).  The OpenSSL batch is compiled on first use into the system's temporary
directory, named by a hash of its source, so the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from typing import Sequence

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "matvec_cpu.cpp")
u64p = C.POINTER(C.c_uint64)
_lib = None


def matvec_native(n: int, cs: Sequence[int], W: Sequence[Sequence[int]]) -> list:
    """Row r: P_r * N_r^(n - 1) mod n^2, P_r = prod_{W[r][i] > 0} c_i^W[r][i], N_r = prod_{W[r][i] < 0} c_i^(-W[r][i]) (the exact
    output of pb200_matvec; the ciphertext of sum_i W[r][i] * m_i mod n)."""
    n2 = n * n
    out = []
    for row in W:
        P, N = 1 % n2, 1 % n2
        for c, w in zip(cs, row, strict=True):
            if w > 0:
                P = P * pow(c, w, n2) % n2
            elif w < 0:
                N = N * pow(c, -w, n2) % n2
        out.append(P * pow(N, n - 1, n2) % n2)
    return out


def build() -> str:
    """Compile the OpenSSL batch unless a build of this exact source exists; returns the library's path."""
    src = open(SRC, "rb").read()
    path = os.path.join(tempfile.gettempdir(), f"pb200_matvec_cpu_{hashlib.sha256(src).hexdigest()[:16]}.so")
    if not os.path.exists(path):
        fd, tmp = tempfile.mkstemp(suffix=".so")
        os.close(fd)
        cxx = os.environ.get("CXX", "g++")
        subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-o", tmp, SRC, "-lcrypto", "-lpthread"], check=True,
                       capture_output=True)
        os.replace(tmp, path)
    return path


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        lib.cpu_paillier_matvec.restype = C.c_int
        lib.cpu_paillier_matvec.argtypes = [u64p, C.c_int, u64p, C.c_size_t, u64p, C.c_void_p, C.c_int, C.c_size_t, u64p, C.c_int]
        _lib = lib
    return _lib


def matvec(n: int, words_in: int, c_w: np.ndarray, w_mag: np.ndarray, w_neg, threads: int = 1) -> np.ndarray:
    """matvec_native with OpenSSL on words: c_w (count, 2 words_in), w_mag (rows, count, k_words), w_neg None or (rows, count)."""
    lib = load()
    c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, 2 * words_in)
    count = c_w.shape[0]
    w_mag = np.ascontiguousarray(w_mag, dtype="<u8")
    rows = w_mag.shape[0]
    k_words = w_mag.size // max(1, rows * count)
    neg = None if w_neg is None else np.ascontiguousarray(w_neg, dtype=np.uint8).reshape(rows, count)
    n_w = np.frombuffer(int(n).to_bytes(8 * words_in, "little"), dtype="<u8").copy()
    out = np.empty((rows, 2 * words_in), dtype="<u8")
    rc = lib.cpu_paillier_matvec(n_w.ctypes.data_as(u64p), words_in, c_w.ctypes.data_as(u64p), count, w_mag.ctypes.data_as(u64p),
                                 None if neg is None else neg.ctypes.data_as(C.c_void_p), max(1, k_words), rows,
                                 out.ctypes.data_as(u64p), threads)
    assert rc == 0
    return out
