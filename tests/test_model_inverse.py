"""CPU tests of the inverse mod n^2: the limb-exact model of the kernel (tests/model_safegcd.py) against Python's pow(c, -1, n^2) on the
committed keys and on random odd moduli of 64 ... 4096 bits, adversarial inputs, non-invertible inputs, and the argument checks of the
new entry points (no device needed)."""
import ctypes as C
import random

import pytest

import model_safegcd as M
from paillier_halo2_b200 import _lib, workload


def _want(c, n):
    try:
        return pow(c, -1, n * n)
    except ValueError:
        return None


def _adversarial(n, n_bits, rng):
    wo = (2 * n_bits + 63) // 64
    cs = [1, 2, n - 1, n + 1, 2 * n + 1, n * n - 1, n * n + 1, (1 << (64 * wo)) - 1]
    cs += [1 << b for b in (1, 61, 62, 63, 64, n_bits - 1, n_bits, 2 * n_bits - 1) if b < 64 * wo]
    cs += [(1 << b) - 1 for b in (62, 124, n_bits, n_bits + 1)]
    # long runs of equal low bits: the divstep batches see all-zero or all-one words for many batches
    cs += [((rng.getrandbits(64) | 1) << b) | 1 for b in (124, 248, n_bits - 70) if b > 0]
    cs += [(rng.getrandbits(n_bits) << b) - 1 for b in (186, n_bits // 2)]
    cs += [n - (1 << b) for b in (62, 200) if b < n_bits - 1]
    return cs


@pytest.mark.parametrize("n_bits", [128, 256, 1024, 2048, 3072, 4096])
def test_model_on_committed_keys(n_bits):
    kd = workload.load_key(n_bits)
    n, p, q = kd["n"], kd["p"], kd["q"]
    K = M.Consts(n, n_bits)
    rng = random.Random(n_bits)
    cs = _adversarial(n, n_bits, rng) + [rng.randrange(n * n) for _ in range(6 if n_bits >= 3072 else 20)]
    for c in cs:
        assert M.inverse_mod_n2(K, c) == pow(c, -1, n * n), hex(c)
    # not invertible: 0, n, n^2, multiples of p and q
    for c in (0, n, n * n, p, q, 3 * p, q * rng.getrandbits(n_bits // 2), n * n + p):
        assert M.inverse_mod_n2(K, c) is None, hex(c)


def test_model_on_random_odd_moduli():
    rng = random.Random(7)
    sizes = [64, 65, 100, 124, 127, 128, 186, 200, 256, 512, 777, 1024, 1536, 2048, 4096]
    for n_bits in sizes:
        for trial in range(4 if n_bits <= 1024 else 1):
            n = rng.getrandbits(n_bits) | 1 | (1 << (n_bits - 1))
            if trial == 1:
                n >>= rng.randrange(1, 40)          # a short n in a wider declared size
                n |= 1
            K = M.Consts(n, n_bits)
            cs = _adversarial(n, n_bits, rng) + [rng.randrange(n * n) for _ in range(4)]
            for c in cs:
                assert M.inverse_mod_n2(K, c) == _want(c, n), (n_bits, hex(n), hex(c))


def test_model_small_moduli_exhaustive():
    """every c below n^2 (and a few above) for small odd n, including composite ones with many non-invertible values"""
    for n in (3, 9, 15, 21, 35, 45, 63, 105, 127, 255):
        K = M.Consts(n, 8)
        for c in list(range(n * n + 3)) + [(1 << 64) - 1]:
            assert M.inverse_mod_n2(K, c) == _want(c, n), (n, c)


def test_iteration_bound_and_layout():
    """the fixed iteration count and limb count the kernel uses (96 batches of 62 divsteps, 34 limbs at |n| = 2048; 67 limbs at 4096)"""
    assert M.divsteps_total(2048) == 5906 and M.batches(2048) == 96 and M.limbs(2048) == 34
    assert M.limbs(4096) == 67 and M.limbs(4096) == 4096 // 62 + 1
    assert M.divsteps_total(45) == (49 * 45 + 80) // 17 and M.divsteps_total(46) == (49 * 46 + 57) // 17


def test_matrix_bounds_hold_on_worst_inputs():
    """|u| + |v| <= 2^62 and |q| + |r| <= 2^62 for every batch, so every matrix entry and every limb product fits the kernel's 64- and
    128-bit words"""
    rng = random.Random(9)
    for _ in range(200):
        delta = rng.choice([1, -1, 5, -300, 1000])
        f = rng.getrandbits(64) | 1
        g = rng.choice([0, 1, (1 << 64) - 1, rng.getrandbits(64)])
        _, (u, v, q, r) = M.divsteps_62(delta, f, g)
        assert abs(u) + abs(v) <= 1 << 62 and abs(q) + abs(r) <= 1 << 62
        assert (u * f + v * g) % (1 << 62) == 0 and (q * f + r * g) % (1 << 62) == 0


# ---- argument checks of the C ABI (no device needed) ------------------------------------------------------------------------
def test_null_and_width_arguments_are_rejected(built_lib):
    lib = built_lib
    null = C.c_void_p()
    assert lib.pb200_inverse_batch(null, None, 1, None) == _lib.PB200_ERR_INVALID_ARG
    assert lib.pb200_inverse_batch_dev(null, None, 1, None) == _lib.PB200_ERR_INVALID_ARG
    assert lib.pb200_sub_batch(null, None, None, 1, None) == _lib.PB200_ERR_INVALID_ARG
    assert lib.pb200_sub_batch_dev(null, None, None, 1, None) == _lib.PB200_ERR_INVALID_ARG
    for k_bits in (1, 0, 1 << 20):
        assert lib.pb200_scalar_mul_signed_batch(null, None, None, None, k_bits, 1, None) == _lib.PB200_ERR_INVALID_ARG
        assert lib.pb200_scalar_mul_signed_batch_dev(null, None, None, None, k_bits, 1, None) == _lib.PB200_ERR_INVALID_ARG


def test_status_texts(built_lib):
    assert built_lib.pb200_strerror(_lib.PB200_ERR_NOT_INVERTIBLE) not in (b"", b"unknown status")
    assert b"reserved" not in built_lib.pb200_strerror(_lib.PB200_ERR_EVEN_MODULUS)
    assert (_lib.PB200_ERR_NOT_INVERTIBLE, _lib.PB200_FLAG_NOT_INVERTIBLE) == (-12, 16)
