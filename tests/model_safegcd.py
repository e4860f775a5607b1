"""Limb-exact Python model of the inverse kernel (paillier_halo2_b200/csrc/inverse_kernels.cu).

c^-1 mod n^2 in two steps, as the kernel does them:
  1. x0 = c^-1 mod n by Bernstein-Yang safegcd ("Fast constant-time gcd computation and modular inversion", 2019): a fixed number of
     batches of 62 divsteps on the low 64 bits of (f, g), each batch giving a transition matrix that is applied to (f, g) with an exact
     division by 2^62 and to (d, e) mod n, on signed 62-bit limbs (libsecp256k1's modinv64 layout).  f = +-1 at the end means
     gcd(c, n) = 1.
  2. x = x0 (2 - c x0) mod n^2: one Hensel step, because c x0 = 1 + t n gives c x = 1 - t^2 n^2.

Python ints stand in for the device's 64- and 128-bit words; every limb operation the kernel makes is made here in the same order, with
the same masks and shifts, so the CUDA is a transliteration of this file.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

B = 62                       # divsteps per batch = bits per limb
M62 = (1 << B) - 1
M64 = (1 << 64) - 1


def divsteps_total(d: int) -> int:
    """Bernstein-Yang's iteration bound for f odd, 0 <= g <= f < 2^d: after this many divsteps g = 0 and f = +-gcd(f, g)."""
    return (49 * d + 80) // 17 if d < 46 else (49 * d + 57) // 17


def batches(d: int) -> int:
    return -(-divsteps_total(d) // B)


def limbs(d: int) -> int:
    """signed 62-bit limbs holding values in (-2^(d+1), 2^(d+1)): every limb but the top one in [0, 2^62), the top one a signed int64"""
    return d // B + 1


def to_limbs(x: int, L: int) -> List[int]:
    out = [(x >> (B * i)) & M62 for i in range(L - 1)]
    out.append(x >> (B * (L - 1)))                      # signed top limb
    return out


def from_limbs(a: List[int]) -> int:
    return sum(v << (B * i) for i, v in enumerate(a))


def divsteps_62(delta: int, f0: int, g0: int) -> Tuple[int, Tuple[int, int, int, int]]:
    """62 divsteps on the low 64 bits of f (odd) and g.  Returns the new delta and the matrix t = (u, v, q, r) with
    2^62 (f', g') = (u f + v g, q f + r g) for the full values; |u| + |v| <= 2^62 and |q| + |r| <= 2^62.  Branch-free in the kernel:
    every step makes the same operations, selected by masks."""
    f, g = f0 & M64, g0 & M64
    u, v, q, r = 1, 0, 0, 1
    for _ in range(B):
        swap = delta > 0 and (g & 1)
        if swap:                                        # (delta, f, g) <- (1 - delta, g, (g - f) / 2)
            delta = 1 - delta
            f, g = g, (g - f) & M64
            u, v, q, r = q, r, q - u, r - v
        else:                                           # (delta, f, g) <- (1 + delta, f, (g + (g & 1) f) / 2)
            delta = 1 + delta
            if g & 1:
                g = (g + f) & M64
                q, r = q + u, r + v
        g >>= 1                                         # exact: g is even here
        u, v = u << 1, v << 1
    return delta, (u, v, q, r)


def update_fg(f: List[int], g: List[int], t) -> None:
    """(f, g) <- t (f, g) / 2^62 exactly (the low 62 bits of both products are zero by construction of t)"""
    u, v, q, r = t
    L = len(f)
    cf = u * f[0] + v * g[0]
    cg = q * f[0] + r * g[0]
    assert cf & M62 == 0 and cg & M62 == 0
    cf >>= B
    cg >>= B
    for i in range(1, L):
        cf += u * f[i] + v * g[i]
        cg += q * f[i] + r * g[i]
        f[i - 1], g[i - 1] = cf & M62, cg & M62
        cf >>= B
        cg >>= B
    f[L - 1], g[L - 1] = cf, cg
    assert -(1 << 63) <= cf < (1 << 63) and -(1 << 63) <= cg < (1 << 63)


def update_de(d: List[int], e: List[int], t, n62: List[int], ninv62: int) -> None:
    """(d, e) <- t (d, e) / 2^62 mod n, keeping both in (-2n, n): adds md n and me n, md and me chosen so that the low 62 bits vanish
    (ninv62 = n^-1 mod 2^62), after a sign correction that keeps the range (libsecp256k1 modinv64's update_de)."""
    u, v, q, r = t
    L = len(d)
    sd = -1 if d[L - 1] < 0 else 0
    se = -1 if e[L - 1] < 0 else 0
    md = (u & sd) + (v & se)
    me = (q & sd) + (r & se)
    cd = u * d[0] + v * e[0]
    ce = q * d[0] + r * e[0]
    md -= (ninv62 * (cd & M64) + md) & M62
    me -= (ninv62 * (ce & M64) + me) & M62
    cd += n62[0] * md
    ce += n62[0] * me
    assert cd & M62 == 0 and ce & M62 == 0
    cd >>= B
    ce >>= B
    for i in range(1, L):
        cd += u * d[i] + v * e[i] + n62[i] * md
        ce += q * d[i] + r * e[i] + n62[i] * me
        d[i - 1], e[i - 1] = cd & M62, ce & M62
        cd >>= B
        ce >>= B
    d[L - 1], e[L - 1] = cd, ce
    assert -(1 << 63) <= cd < (1 << 63) and -(1 << 63) <= ce < (1 << 63)


def add_masked(a: List[int], b: List[int], mask: int) -> None:
    """a += b & mask (mask 0 or -1), carries rippled so that every limb but the top one is back in [0, 2^62)"""
    c = 0
    L = len(a)
    for i in range(L):
        c += a[i] + (b[i] & mask)
        if i < L - 1:
            a[i] = c & M62
            c >>= B
        else:
            a[i] = c


def neg_masked(a: List[int], mask: int) -> None:
    """a = -a where mask == -1: every limb becomes (a_i ^ mask) - mask = -a_i, then the carries are rippled as in add_masked"""
    c = 0
    L = len(a)
    for i in range(L):
        c += (a[i] ^ mask) - mask
        if i < L - 1:
            a[i] = c & M62
            c >>= B
        else:
            a[i] = c


def normalize(d: List[int], f_sign_mask: int, n62: List[int]) -> None:
    """d in (-2n, n) -> d * sign(f) in [0, n): add n if negative, negate when f = -1, add n if negative"""
    L = len(d)
    add_masked(d, n62, -1 if d[L - 1] < 0 else 0)
    neg_masked(d, f_sign_mask)
    add_masked(d, n62, -1 if d[L - 1] < 0 else 0)


class Consts:
    """per-key constants of the kernel: the limb count, the batch count, n in 62-bit limbs and n^-1 mod 2^62"""

    def __init__(self, n: int, n_bits: int):
        assert n & 1, "safegcd needs an odd modulus"
        self.n, self.n_bits = n, n_bits
        self.L = limbs(n_bits)
        self.batches = batches(n_bits)
        self.n62 = to_limbs(n, self.L)
        self.ninv62 = pow(n, -1, 1 << B)


def inverse_mod_n(K: Consts, x: int) -> Optional[int]:
    """x^-1 mod n for 0 <= x < n, or None when gcd(x, n) != 1"""
    L = K.L
    f, g = list(K.n62), to_limbs(x, L)
    d, e = [0] * L, to_limbs(1, L)
    delta = 1
    for _ in range(K.batches):
        lo_f = (f[0] | (f[1] << B)) & M64 if L > 1 else f[0] & M64
        lo_g = (g[0] | (g[1] << B)) & M64 if L > 1 else g[0] & M64
        delta, t = divsteps_62(delta, lo_f, lo_g)
        update_fg(f, g, t)
        update_de(d, e, t, K.n62, K.ninv62)
    assert from_limbs(g) == 0
    one = to_limbs(1, L)
    minus_one = to_limbs(-1, L)
    if f != one and f != minus_one:
        return None
    normalize(d, -1 if f == minus_one else 0, K.n62)
    return from_limbs(d)


def inverse_mod_n2(K: Consts, c: int) -> Optional[int]:
    """c^-1 mod n^2 for any c >= 0 (reduced mod n first), or None when gcd(c, n) != 1: the safegcd inverse mod n, then the Hensel step"""
    n, n2 = K.n, K.n * K.n
    x0 = inverse_mod_n(K, c % n)
    if x0 is None:
        return None
    t = c * x0 % n2                                     # = 1 + t' n
    y = n2 + 2 - t                                      # 2 - t (mod n^2), not reduced: the kernel's multiplication takes it as is
    return x0 * y % n2
