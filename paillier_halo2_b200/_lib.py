"""ctypes binding of libpaillier_b200.so (the C ABI in include/paillier_b200.h).

There is no CPU fallback: if the shared library is missing this module raises at import of the
symbol table, and every compute call fails with PB200_ERR_CUDA when no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PB200_LIB") or os.path.join(HERE, "libpaillier_b200.so")   # PB200_LIB: A/B builds (tools/build_variant.py)

PB200_OK = 0
PB200_ERR_INVALID_ARG = -1
PB200_ERR_ZERO_MODULUS = -2
PB200_ERR_EVEN_MODULUS = -3
PB200_ERR_RANGE = -4
PB200_ERR_UNSUPPORTED = -5
PB200_ERR_CUDA = -6
PB200_ERR_NOMEM = -7
PB200_ERR_SINK = -8
PB200_ERR_CONSTRAINT = -9
PB200_ERR_PEER = -10
PB200_ERR_DECRYPT = -11
PB200_ERR_NOT_INVERTIBLE = -12
PB200_FLAG_RANGE, PB200_FLAG_CONSTRAINT, PB200_FLAG_PEER_TIMEOUT, PB200_FLAG_DECRYPT, PB200_FLAG_NOT_INVERTIBLE = 1, 2, 4, 8, 16

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)


class WitnessChunk(C.Structure):
    _fields_ = [
        ("first_unit", C.c_size_t),
        ("n_units", C.c_size_t),
        ("words_out", C.c_uint32),
        ("offsets", u64p),
        ("records", u64p),
        ("g_mul_counts", u32p),
    ]


SINK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(WitnessChunk))

# name -> (restype, argtypes); every symbol include/paillier_b200.h declares
SYMBOLS = {
    "pb200_strerror": (C.c_char_p, [C.c_int]),
    "pb200_last_cuda_error": (C.c_char_p, []),
    "pb200_version": (C.c_char_p, []),
    "pb200_device_count": (C.c_int, []),
    "pb200_kernel_launches": (C.c_uint64, []),
    "pb200_key_create": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32, u64p, u64p, C.POINTER(C.c_void_p)]),
    "pb200_key_destroy": (None, [C.c_void_p]),
    "pb200_key_n_bits": (C.c_uint32, [C.c_void_p]),
    "pb200_key_words_in": (C.c_uint32, [C.c_void_p]),
    "pb200_key_words_out": (C.c_uint32, [C.c_void_p]),
    "pb200_key_device": (C.c_int, [C.c_void_p]),
    "pb200_key_n2": (C.c_int, [C.c_void_p, u64p]),
    "pb200_key_engine": (C.c_char_p, [C.c_void_p]),
    "pb200_key_set_engine": (C.c_int, [C.c_void_p, C.c_int]),
    "pb200_umma_layout": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "pb200_key_shape": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pb200_debug_mulmod_cycles": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "pb200_debug_mulmod": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pb200_key_stream": (C.c_void_p, [C.c_void_p]),
    "pb200_key_sync": (C.c_int, [C.c_void_p]),
    "pb200_key_take_flags": (C.c_int, [C.c_void_p, u32p]),
    "pb200_key_chain_counts": (C.c_int, [C.c_void_p, u64p, u64p]),
    "pb200_encrypt_batch": (C.c_int, [C.c_void_p, u64p, u64p, C.c_size_t, u64p]),
    "pb200_encrypt_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_add_batch": (C.c_int, [C.c_void_p, u64p, u64p, C.c_uint32, C.c_size_t, u64p, u64p]),
    "pb200_add_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t, C.c_void_p, C.c_void_p]),
    "pb200_tally": (C.c_int, [C.c_void_p, u64p, C.c_size_t, u64p]),
    "pb200_tally_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_tally_combine": (C.c_int, [C.c_void_p, u64p, C.c_size_t, u64p]),
    "pb200_tally_trace": (C.c_int, [C.c_void_p, u64p, u64p, C.c_size_t, C.c_size_t, u64p, u64p]),
    "pb200_tally_trace_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]),
    "pb200_tally_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), u64p]),
    "pb200_tally_peer_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pb200_tally_peer_connect": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "pb200_tally_peer_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_key_set_private": (C.c_int, [C.c_void_p, u64p, u64p]),
    "pb200_decrypt_batch": (C.c_int, [C.c_void_p, u64p, C.c_size_t, u64p]),
    "pb200_decrypt_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_scalar_mul_batch": (C.c_int, [C.c_void_p, u64p, u64p, C.c_uint32, C.c_size_t, u64p]),
    "pb200_scalar_mul_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t, C.c_void_p]),
    "pb200_tally_weighted": (C.c_int, [C.c_void_p, u64p, u64p, C.c_uint32, C.c_size_t, u64p]),
    "pb200_tally_weighted_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t, C.c_void_p]),
    "pb200_inverse_batch": (C.c_int, [C.c_void_p, u64p, C.c_size_t, u64p]),
    "pb200_inverse_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_sub_batch": (C.c_int, [C.c_void_p, u64p, u64p, C.c_size_t, u64p]),
    "pb200_sub_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_scalar_mul_signed_batch": (C.c_int, [C.c_void_p, u64p, u64p, C.c_void_p, C.c_uint32, C.c_size_t, u64p]),
    "pb200_scalar_mul_signed_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t, C.c_void_p]),
    "pb200_key_set_threshold": (C.c_int, [C.c_void_p, C.c_uint32, u64p]),
    "pb200_key_set_share": (C.c_int, [C.c_void_p, C.c_uint32, u64p]),
    "pb200_partial_decrypt_batch": (C.c_int, [C.c_void_p, u64p, C.c_size_t, u64p]),
    "pb200_partial_decrypt_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_combine_shares_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, u64p, C.c_size_t, u64p]),
    "pb200_combine_shares_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pb200_matvec": (C.c_int, [C.c_void_p, u64p, C.c_size_t, u64p, C.c_void_p, C.c_uint32, C.c_size_t, u64p]),
    "pb200_matvec_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t, C.c_void_p]),
    "pb200_matvec_plan": (C.c_int, [C.c_uint32, C.c_int, C.c_size_t, C.c_size_t, C.c_uint32, C.c_int, u64p]),
    "pb200_encrypt_witness_batch": (C.c_int, [C.c_void_p, u64p, u64p, C.c_size_t, u64p, C.c_size_t, SINK_FN, C.c_void_p]),
    "pb200_witness_records_for": (C.c_uint64, [C.c_void_p, u64p]),
    "pb200_encrypt_witness_digest": (C.c_int, [C.c_void_p, u64p, u64p, C.c_size_t, u64p, u64p]),
    "pb200_encrypt_witness_digest_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "pb200_key_witness_engine": (C.c_char_p, [C.c_void_p]),
    "pb200_key_g_chain": (C.c_int, [C.c_void_p, u64p]),
    "pb200_cells_layout": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "pb200_mulmod_cells_batch": (C.c_int, [C.c_void_p, u64p, u64p, u64p, u64p, C.c_size_t, C.c_uint32, C.c_int, u64p]),
    "pb200_mulmod_cells_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, C.c_void_p]),
    "pb200_assign_cells_batch": (C.c_int, [C.c_void_p, u64p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_int, u64p]),
    "pb200_key_n2_cells": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, u64p]),
    "pb200_repack_limbs": (C.c_int, [C.c_void_p, u64p, C.c_size_t, C.c_uint32, C.c_uint32, u64p]),
}



class CellLayout(C.Structure):
    """pb200_cell_layout (include/paillier_b200.h)"""
    _fields_ = [(n, C.c_uint32) for n in ("limbs", "cells_per_limb", "carry_bits", "cells_per_mulmod", "cells_n2", "off_rem", "off_ab",
                                          "off_qn", "off_qn_rem", "off_eq", "eq_stride")]


_lib = None


def load() -> C.CDLL:
    """Load the shared library and bind every declared symbol.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m paillier_halo2_b200.build` "
            "(there is no CPU fallback for the Paillier hot path)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and the header drifted apart
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class Pb200Error(RuntimeError):
    def __init__(self, status: int, where: str):
        lib = load()
        msg = lib.pb200_strerror(status).decode()
        if status == PB200_ERR_CUDA:
            msg += ": " + lib.pb200_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} (status {status})")
        self.status = status


def check(status: int, where: str) -> None:
    if status != PB200_OK:
        raise Pb200Error(status, where)
