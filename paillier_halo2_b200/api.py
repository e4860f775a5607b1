"""Host-side mirror of the reference's interface for the Paillier hot path, over the C ABI.

The reference exposes this path as two pure functions and one chip
(`paillier_enc_native`, `paillier_add_native`, `PaillierChip::{construct, encrypt, add}`;
src/paillier.rs:87-97, :11-85).  The batched equivalents keep the names and argument meaning:

    key = PaillierKey(n, g, enc_bits, limb_bits)          # EncryptionPublicKeyAssigned + construct
    cs  = key.paillier_enc_native(ms, rs)                 # src/paillier.rs:87-92, per (m, r) pair
    ss  = key.paillier_add_native(c1s, c2s)               # src/paillier.rs:94-97, per pair
    t   = key.tally(cs)                                   # N-ary fold of paillier_add_native

Every call goes to CUDA through libpaillier_b200.so; nothing here computes a ciphertext on the CPU.
"""
from __future__ import annotations

import ctypes as C
import numbers
from typing import Callable, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import Pb200Error, check  # noqa: F401


def words(bits: int) -> int:
    return (bits + 63) // 64


def ints_to_words(vals: Sequence[int], nwords: int) -> np.ndarray:
    """Python ints -> (len, nwords) little-endian uint64 array.  Raises OverflowError if one does not fit."""
    out = np.empty((len(vals), nwords), dtype="<u8")
    nbytes = nwords * 8
    for i, v in enumerate(vals):
        out[i] = np.frombuffer(int(v).to_bytes(nbytes, "little"), dtype="<u8")
    return out


def words_to_ints(arr: np.ndarray) -> List[int]:
    arr = np.ascontiguousarray(arr, dtype="<u8")
    if arr.ndim == 1:
        arr = arr.reshape(1, -1)
    return [int.from_bytes(row.tobytes(), "little") for row in arr]


def _p(a: np.ndarray):
    return a.ctypes.data_as(_lib.u64p)


BN254_FR = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def _cells_to_ints(arr: np.ndarray) -> List[int]:
    """(n, 4) u64 cells -> integers (the 4 words little-endian)"""
    raw = np.ascontiguousarray(arr, dtype="<u8").tobytes()
    return [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(len(raw) // 32)]


class CellMixin:
    """K4: advice-cell values (BN254 Fr, 4 x u64) produced on the GPU (include/paillier_b200.h, "advice cells")."""

    def cells_layout(self, lookup_bits: int) -> dict:
        lay = _lib.CellLayout()
        check(self._lib.pb200_cells_layout(self._h, lookup_bits, C.byref(lay)), "pb200_cells_layout")
        return {n: int(getattr(lay, n)) for n, _ in lay._fields_}

    def mulmod_cells_words(self, a_w, b_w, q_w, rem_w, lookup_bits: int, montgomery: bool = False) -> np.ndarray:
        count = a_w.shape[0]
        per = self.cells_layout(lookup_bits)["cells_per_mulmod"]
        out = np.empty((count, per, 4), dtype="<u8")
        check(self._lib.pb200_mulmod_cells_batch(self._h, _p(a_w), _p(b_w), _p(q_w), _p(rem_w), count, lookup_bits, int(montgomery), _p(out)),
              "pb200_mulmod_cells_batch")
        return out

    def mulmod_cells_dev(self, d_a: int, d_b: int, d_q: int, d_rem: int, count: int, lookup_bits: int, montgomery: bool, d_cells: int) -> None:
        """Device-pointer variant (pb200_mulmod_cells_batch_dev): enqueues on the key's stream, no synchronise."""
        check(self._lib.pb200_mulmod_cells_batch_dev(self._h, d_a, d_b, d_q, d_rem, count, lookup_bits, int(montgomery), d_cells),
              "pb200_mulmod_cells_batch_dev")

    def add_dev(self, d_c1: int, d_c2: int, c_words: int, count: int, d_out: int, d_q: int) -> None:
        check(self._lib.pb200_add_batch_dev(self._h, d_c1, d_c2, c_words, count, d_out, d_q or None), "pb200_add_batch_dev")

    def mulmod_cells(self, groups: Sequence[Tuple[int, int, int, int]], lookup_bits: int, montgomery: bool = False) -> List[List[int]]:
        """groups: (a, b, q, rem) per mul_mod -> the group's cells in BigUintChip assignment order."""
        if not groups:
            return []
        cols = [ints_to_words([g[i] for g in groups], self.words_out) for i in range(4)]
        out = self.mulmod_cells_words(*cols, lookup_bits, montgomery)
        return [_cells_to_ints(out[i]) for i in range(len(groups))]

    def assign_cells(self, vals: Sequence[int], value_bits: int, lookup_bits: int, montgomery: bool = False) -> List[List[int]]:
        """assign_integer(v, value_bits) for each value: [limb, range-check chunks...] per limb."""
        v_w = ints_to_words(vals, words(value_bits))
        per = (value_bits // self.limb_bits) * self.cells_layout(lookup_bits)["cells_per_limb"]
        out = np.empty((len(vals), per, 4), dtype="<u8")
        check(self._lib.pb200_assign_cells_batch(self._h, _p(v_w), len(vals), value_bits, lookup_bits, int(montgomery), _p(out)),
              "pb200_assign_cells_batch")
        return [_cells_to_ints(out[i]) for i in range(len(vals))]

    def n2_cells(self, lookup_bits: int, montgomery: bool = False) -> List[int]:
        """square(n) columns + refresh div/mod chain + range-check chunks of the refreshed limbs (src/paillier.rs:39-45)."""
        out = np.empty((self.cells_layout(lookup_bits)["cells_n2"], 4), dtype="<u8")
        check(self._lib.pb200_key_n2_cells(self._h, lookup_bits, int(montgomery), _p(out)), "pb200_key_n2_cells")
        return _cells_to_ints(out)

    def encrypt_cells(self, m: int, r: int, lookup_bits: int, montgomery: bool = False):
        """Every advice cell of the reference's encrypt test flow (src/bench.rs:33-75: assign n, g, m, r; PaillierChip::encrypt;
        assign res) for one unit, all values computed on the GPU: witnesses from the (q, rem) stream, cells from K4.
        Returns (ciphertext, cells in assignment order)."""
        n, g, eb = self.n, self.g, self.enc_bits
        cs, units, _ = self.encrypt_witness([m], [r])
        stream = chip_order(m, n, self.g_chain(), units[0])
        groups = []
        it = iter(stream)
        marks = []          # number of groups before each chain start (acc = assign_constant(1) is loaded there)
        for base, e in ((g, m), (r, n)):
            marks.append(len(groups))
            acc, sq = 1, base
            for i in range(e.bit_length()):
                cur = sq
                q, sq = next(it)
                groups.append((cur, cur, q, sq))
                if (e >> i) & 1:
                    q, rem = next(it)
                    groups.append((acc, cur, q, rem))
                    acc = rem
            if base == g:
                gm = acc
        q, c = next(it)
        groups.append((gm, acc, q, c))
        gcells = self.mulmod_cells(groups, lookup_bits, montgomery)
        one = (1 << 256) % BN254_FR if montgomery else 1
        cells: List[int] = []
        for a in self.assign_cells([n, g, m, r], eb, lookup_bits, montgomery):
            cells += a
        cells += self.n2_cells(lookup_bits, montgomery) + [0]
        for gi, gc in enumerate(gcells):
            cells += [one] * marks.count(gi)
            cells += gc
        cells += self.assign_cells([cs[0]], 2 * eb, lookup_bits, montgomery)[0]
        return cs[0], cells


class PaillierKey(CellMixin):
    """EncryptionPublicKeyAssigned{n, g} (src/paillier.rs:6-9) bound to one CUDA device."""

    def __init__(self, n: int, g: int, enc_bits: int, limb_bits: int = 64, device: int = 0):
        self._lib = _lib.load()
        self.enc_bits = enc_bits
        self.limb_bits = limb_bits
        self.n = n
        self.g = g
        win = words(enc_bits)
        try:
            n_w = ints_to_words([n], win)
            g_w = ints_to_words([g], win)
        except OverflowError:
            raise Pb200Error(_lib.PB200_ERR_RANGE, "PaillierKey")
        h = C.c_void_p()
        check(self._lib.pb200_key_create(device, enc_bits, limb_bits, _p(n_w), _p(g_w), C.byref(h)), "pb200_key_create")
        self._h = h
        self.words_in = self._lib.pb200_key_words_in(h)
        self.words_out = self._lib.pb200_key_words_out(h)
        self.device = device

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.pb200_key_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- properties ---------------------------------------------------------------------------
    @property
    def handle(self):
        return self._h

    @property
    def engine(self) -> str:
        return self._lib.pb200_key_engine(self._h).decode()

    @property
    def witness_engine(self) -> str:
        """Engine that produces this key's witnesses: "block28w" or "simple64"."""
        return self._lib.pb200_key_witness_engine(self._h).decode()

    def set_engine(self, engine: int) -> None:
        check(self._lib.pb200_key_set_engine(self._h, engine), "pb200_key_set_engine")

    def n2(self) -> int:
        out = np.zeros(self.words_out, dtype="<u8")
        check(self._lib.pb200_key_n2(self._h, _p(out)), "pb200_key_n2")
        return words_to_ints(out)[0]

    def chain_counts(self):
        """(modular squarings, modular multiplications) the selected engine executes per encryption."""
        a, b = C.c_uint64(), C.c_uint64()
        check(self._lib.pb200_key_chain_counts(self._h, C.byref(a), C.byref(b)), "pb200_key_chain_counts")
        return int(a.value), int(b.value)

    @property
    def stream(self) -> int:
        return int(self._lib.pb200_key_stream(self._h) or 0)

    def encrypt_dev(self, d_m: int, d_r: int, count: int, d_c: int) -> None:
        """Device-pointer variant (pb200_encrypt_batch_dev): enqueues on the key's stream, no synchronise."""
        check(self._lib.pb200_encrypt_batch_dev(self._h, d_m, d_r, count, d_c), "pb200_encrypt_batch_dev")

    def encrypt_witness_digest_dev(self, d_m: int, d_r: int, count: int, d_c: int, d_digest: int) -> None:
        """Device-pointer variant (pb200_encrypt_witness_digest_dev): enqueues on the key's stream, no synchronise."""
        check(self._lib.pb200_encrypt_witness_digest_dev(self._h, d_m, d_r, count, d_c or None, d_digest),
              "pb200_encrypt_witness_digest_dev")

    def tally_dev(self, d_c: int, count: int, d_out: int) -> None:
        check(self._lib.pb200_tally_dev(self._h, d_c, count, d_out), "pb200_tally_dev")

    def sync(self) -> None:
        check(self._lib.pb200_key_sync(self._h), "pb200_key_sync")

    def take_flags(self) -> int:
        """Synchronise, return and clear the per-key device flag word (PB200_FLAG_*): how _dev callers learn of a failure."""
        f = C.c_uint32()
        check(self._lib.pb200_key_take_flags(self._h, C.byref(f)), "pb200_key_take_flags")
        return int(f.value)

    # -- multi-GPU tally: one process per GPU (pb200_tally_peer_*), or one process driving several keys (tally_multi) ------
    def tally_peer_export(self) -> bytes:
        """64-byte handle of this key's mailbox; the ranks exchange these and pass the list to tally_peer_connect."""
        buf = (C.c_ubyte * 64)()
        check(self._lib.pb200_tally_peer_export(self._h, buf), "pb200_tally_peer_export")
        return bytes(buf)

    def tally_peer_connect(self, rank: int, world: int, handles: Sequence[bytes]) -> None:
        raw = b"".join(handles) if world > 1 else bytes(64)
        assert len(raw) == 64 * max(world, 1)
        buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
        check(self._lib.pb200_tally_peer_connect(self._h, rank, world, buf), "pb200_tally_peer_connect")

    def tally_peer_dev(self, d_c: int, count: int, d_out: int) -> None:
        """Collective: every rank of the connected group calls it once per tally; d_out receives the full product."""
        check(self._lib.pb200_tally_peer_dev(self._h, d_c, count, d_out), "pb200_tally_peer_dev")

    @staticmethod
    def tally_multi(keys: Sequence["PaillierKey"], d_cs: Sequence[int], counts: Sequence[int]) -> int:
        """pb200_tally_multi: keys[i] on distinct devices of one process, d_cs[i] the device pointer of shard i."""
        n = len(keys)
        lib = keys[0]._lib
        hk = (C.c_void_p * n)(*[k._h for k in keys])
        hp = (C.c_void_p * n)(*[C.c_void_p(p) for p in d_cs])
        hc = (C.c_size_t * n)(*counts)
        out = np.empty(keys[0].words_out, dtype="<u8")
        check(lib.pb200_tally_multi(hk, n, hp, hc, _p(out)), "pb200_tally_multi")
        return words_to_ints(out)[0]

    # -- raw array API (uint64 little-endian words, unit-major) -----------------------------
    def encrypt_words(self, m_w: np.ndarray, r_w: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        m_w = np.ascontiguousarray(m_w, dtype="<u8")
        r_w = np.ascontiguousarray(r_w, dtype="<u8")
        count = m_w.shape[0]
        assert m_w.shape == (count, self.words_in) and r_w.shape == m_w.shape
        if out is None:
            out = np.empty((count, self.words_out), dtype="<u8")
        check(self._lib.pb200_encrypt_batch(self._h, _p(m_w), _p(r_w), count, _p(out)), "pb200_encrypt_batch")
        return out

    def add_words(self, c1_w: np.ndarray, c2_w: np.ndarray, want_q: bool = False):
        c1_w = np.ascontiguousarray(c1_w, dtype="<u8")
        c2_w = np.ascontiguousarray(c2_w, dtype="<u8")
        count, cw = c1_w.shape
        assert c2_w.shape == c1_w.shape
        out = np.empty((count, self.words_out), dtype="<u8")
        q = np.empty((count, self.words_out), dtype="<u8") if want_q else None
        check(self._lib.pb200_add_batch(self._h, _p(c1_w), _p(c2_w), cw, count, _p(out), _p(q) if want_q else None),
              "pb200_add_batch")
        return (out, q) if want_q else out

    def tally_words(self, c_w: np.ndarray) -> np.ndarray:
        c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, self.words_out)
        out = np.empty(self.words_out, dtype="<u8")
        check(self._lib.pb200_tally(self._h, _p(c_w) if c_w.shape[0] else None, c_w.shape[0], _p(out)), "pb200_tally")
        return out

    def tally_combine_words(self, partials_w: np.ndarray) -> np.ndarray:
        partials_w = np.ascontiguousarray(partials_w, dtype="<u8").reshape(-1, self.words_out)
        out = np.empty(self.words_out, dtype="<u8")
        check(self._lib.pb200_tally_combine(self._h, _p(partials_w), partials_w.shape[0], _p(out)), "pb200_tally_combine")
        return out

    # -- reference-named API on Python ints ---------------------------------------------------
    def paillier_enc_native(self, ms: Sequence[int], rs: Sequence[int]) -> List[int]:
        """Batched src/paillier.rs:87-92 under this key's (n, g)."""
        try:
            m_w = ints_to_words(ms, self.words_in)
            r_w = ints_to_words(rs, self.words_in)
        except OverflowError:
            raise Pb200Error(_lib.PB200_ERR_RANGE, "paillier_enc_native")
        return words_to_ints(self.encrypt_words(m_w, r_w)) if len(ms) else []

    def paillier_add_native(self, c1s: Sequence[int], c2s: Sequence[int], c_bits: Optional[int] = None,
                            want_q: bool = False):
        """Batched src/paillier.rs:94-97.  c_bits = width the inputs are assigned with (enc_bits in the
        reference's tests, 2*enc_bits for real ciphertexts; default 2*enc_bits)."""
        cw = words(c_bits if c_bits is not None else 2 * self.enc_bits)
        try:
            a = ints_to_words(c1s, cw)
            b = ints_to_words(c2s, cw)
        except OverflowError:
            raise Pb200Error(_lib.PB200_ERR_RANGE, "paillier_add_native")
        if not len(c1s):
            return ([], []) if want_q else []
        if want_q:
            out, q = self.add_words(a, b, True)
            return words_to_ints(out), words_to_ints(q)
        return words_to_ints(self.add_words(a, b))

    def tally(self, cs: Sequence[int]) -> int:
        c_w = ints_to_words(cs, self.words_out) if len(cs) else np.empty((0, self.words_out), dtype="<u8")
        return words_to_ints(self.tally_words(c_w))[0]

    # -- running-tally trace: (q_i, acc_i) = divmod(acc_(i-1) * c_i, n^2) for every step of every chain --------------------------
    def tally_trace_words(self, init_w: np.ndarray, c_w: np.ndarray, want_q: bool = True):
        """init_w: (chains, words_out); c_w: (count, chains, words_out), any values -> acc (and q when want_q), each of shape
        (count, chains, words_out): step i of chain j multiplies acc_(i-1, j) (init_j for i = 0) by c_(i, j) (pb200_tally_trace)."""
        init_w = np.ascontiguousarray(init_w, dtype="<u8").reshape(-1, self.words_out)
        chains = init_w.shape[0]
        c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, chains, self.words_out)
        count = c_w.shape[0]
        acc = np.empty((count, chains, self.words_out), dtype="<u8")
        q = np.empty((count, chains, self.words_out), dtype="<u8") if want_q else None
        if count and chains:
            check(self._lib.pb200_tally_trace(self._h, _p(init_w), _p(c_w), count, chains, _p(acc), _p(q) if want_q else None),
                  "pb200_tally_trace")
        return (acc, q) if want_q else acc

    def tally_trace_dev(self, d_init: int, d_c: int, count: int, chains: int, d_acc: int, d_q: Optional[int] = None) -> None:
        """Device-pointer variant (pb200_tally_trace_dev): enqueues on the key's stream, no synchronise; a quotient that does not fit
        raises PB200_FLAG_RANGE in the flag word (take_flags)."""
        check(self._lib.pb200_tally_trace_dev(self._h, d_init, d_c, count, chains, d_acc, d_q or None), "pb200_tally_trace_dev")

    def tally_trace(self, init, cs: Sequence, want_q: bool = True):
        """Running tally on Python ints.  init: an int (one chain) or a sequence of one int per chain; cs: one element per step,
        an int (one chain) or a sequence of one int per chain.  Returns acc (and q when want_q) as lists shaped like cs."""
        single = isinstance(init, numbers.Integral)
        inits = [int(init)] if single else [int(x) for x in init]
        rows = [[int(c)] if single else [int(x) for x in c] for c in cs]
        assert all(len(r) == len(inits) for r in rows), "every step needs one ciphertext per chain"
        init_w = self._ciphertexts(inits, "tally_trace")
        c_w = self._ciphertexts([c for r in rows for c in r], "tally_trace") if rows else np.empty((0, self.words_out), dtype="<u8")
        res = self.tally_trace_words(init_w, c_w.reshape(len(rows), len(inits), self.words_out), want_q)
        arrs = res if want_q else (res,)
        outs = []
        for a in arrs:
            flat = words_to_ints(a.reshape(-1, self.words_out)) if rows else []
            outs.append([flat[i] for i in range(len(rows))] if single else
                        [flat[i * len(inits):(i + 1) * len(inits)] for i in range(len(rows))])
        return (outs[0], outs[1]) if want_q else outs[0]

    # -- decryption (SURVEY.md 8f-4) -----------------------------------------------------------------------------------
    def set_private(self, lam: int, mu: int) -> None:
        """lambda = lcm(p-1, q-1), mu = L(g^lambda mod n^2)^-1 mod n (private_from_primes gives both)."""
        try:
            a, b = ints_to_words([lam], self.words_in), ints_to_words([mu], self.words_in)
        except OverflowError:
            raise Pb200Error(_lib.PB200_ERR_RANGE, "set_private")
        check(self._lib.pb200_key_set_private(self._h, _p(a), _p(b)), "pb200_key_set_private")

    def decrypt_words(self, c_w: np.ndarray) -> np.ndarray:
        c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, self.words_out)
        out = np.empty((c_w.shape[0], self.words_in), dtype="<u8")
        check(self._lib.pb200_decrypt_batch(self._h, _p(c_w) if c_w.shape[0] else None, c_w.shape[0], _p(out)), "pb200_decrypt_batch")
        return out

    def decrypt(self, cs: Sequence[int]) -> List[int]:
        """m_i = L(c_i^lambda mod n^2) * mu mod n for every ciphertext."""
        if not len(cs):
            return []
        return words_to_ints(self.decrypt_words(ints_to_words(cs, self.words_out)))

    def decrypt_dev(self, d_c: int, count: int, d_m: int) -> None:
        check(self._lib.pb200_decrypt_batch_dev(self._h, d_c, count, d_m), "pb200_decrypt_batch_dev")

    # -- homomorphic scalar multiplication: Dec(c^k mod n^2) = k Dec(c) mod n, prod c_i^(k_i) = Enc(sum k_i m_i) --------------
    def scalar_mul_words(self, c_w: np.ndarray, k_w: np.ndarray, k_bits: int) -> np.ndarray:
        """c_w: (count, words_out) any values; k_w: (count, words(k_bits)) scalars below 2^k_bits -> (count, words_out) c^k mod n^2."""
        c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, self.words_out)
        k_w = np.ascontiguousarray(k_w, dtype="<u8").reshape(-1, words(k_bits))
        count = c_w.shape[0]
        assert k_w.shape[0] == count
        out = np.empty((count, self.words_out), dtype="<u8")
        check(self._lib.pb200_scalar_mul_batch(self._h, _p(c_w), _p(k_w), k_bits, count, _p(out)), "pb200_scalar_mul_batch")
        return out

    def scalar_mul_dev(self, d_c: int, d_k: int, k_bits: int, count: int, d_out: int) -> None:
        """Device-pointer variant (pb200_scalar_mul_batch_dev): enqueues on the key's stream, no synchronise, no range check."""
        check(self._lib.pb200_scalar_mul_batch_dev(self._h, d_c, d_k, k_bits, count, d_out), "pb200_scalar_mul_batch_dev")

    def _scalars(self, ks: Sequence[int]) -> Tuple[np.ndarray, int]:
        """Scalars reduced mod n (a negative weight -s becomes n - s), their words and the declared width (largest bit length)."""
        red = [int(k) % self.n for k in ks]
        k_bits = max([1] + [k.bit_length() for k in red])
        return ints_to_words(red, words(k_bits)), k_bits

    def _ciphertexts(self, cs: Sequence[int], where: str) -> np.ndarray:
        try:
            return ints_to_words(cs, self.words_out)
        except OverflowError:
            raise Pb200Error(_lib.PB200_ERR_RANGE, where)

    def scalar_mul(self, cs: Sequence[int], ks: Sequence[int]) -> List[int]:
        """c_i^(k_i mod n) mod n^2 for every pair: the ciphertext of k_i * m_i mod n."""
        assert len(cs) == len(ks)
        if not len(cs):
            return []
        k_w, k_bits = self._scalars(ks)
        return words_to_ints(self.scalar_mul_words(self._ciphertexts(cs, "scalar_mul"), k_w, k_bits))

    def tally_weighted_words(self, c_w: np.ndarray, k_w: np.ndarray, k_bits: int) -> np.ndarray:
        c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, self.words_out)
        k_w = np.ascontiguousarray(k_w, dtype="<u8").reshape(-1, words(k_bits))
        count = c_w.shape[0]
        assert k_w.shape[0] == count
        out = np.empty(self.words_out, dtype="<u8")
        check(self._lib.pb200_tally_weighted(self._h, _p(c_w) if count else None, _p(k_w) if count else None, k_bits, count, _p(out)),
              "pb200_tally_weighted")
        return out

    def tally_weighted(self, cs: Sequence[int], ks: Sequence[int]) -> int:
        """prod c_i^(k_i mod n) mod n^2: the ciphertext of sum k_i m_i mod n (weights may be negative)."""
        assert len(cs) == len(ks)
        k_w, k_bits = self._scalars(ks)
        c_w = self._ciphertexts(cs, "tally_weighted") if len(cs) else np.empty((0, self.words_out), dtype="<u8")
        return words_to_ints(self.tally_weighted_words(c_w, k_w, k_bits))[0]

    def tally_weighted_dev(self, d_c: int, d_k: int, k_bits: int, count: int, d_out: int) -> None:
        """Device-pointer variant (pb200_tally_weighted_dev): enqueues on the key's stream, no synchronise, no range check."""
        check(self._lib.pb200_tally_weighted_dev(self._h, d_c, d_k, k_bits, count, d_out), "pb200_tally_weighted_dev")

    # -- encrypted matrix-vector product: row r of the result encrypts sum_i W[r, i] * m_i mod n --------------------------------
    def matvec_words(self, c_w: np.ndarray, w_mag_w: np.ndarray, w_neg: Optional[np.ndarray], k_bits: int) -> np.ndarray:
        """c_w: (count, words_out) any values; w_mag_w: (rows, count, words(k_bits)) magnitudes below 2^k_bits; w_neg: None or
        (rows, count), non-zero where the weight is negative -> (rows, words_out) canonical ciphertexts (pb200_matvec)."""
        c_w = np.ascontiguousarray(c_w, dtype="<u8").reshape(-1, self.words_out)
        count, kw = c_w.shape[0], words(k_bits)
        w_mag_w = np.ascontiguousarray(w_mag_w, dtype="<u8")
        rows = w_mag_w.shape[0]
        assert w_mag_w.size == rows * count * kw
        neg = None
        if w_neg is not None:
            neg = np.ascontiguousarray(w_neg, dtype=np.uint8)
            assert neg.size == rows * count
        out = np.empty((rows, self.words_out), dtype="<u8")
        check(self._lib.pb200_matvec(self._h, _p(c_w) if count else None, count, _p(w_mag_w) if w_mag_w.size else None,
                                     neg.ctypes.data_as(C.c_void_p) if neg is not None and neg.size else None, k_bits, rows,
                                     _p(out) if rows else None), "pb200_matvec")
        return out

    def matvec_dev(self, d_c: int, count: int, d_w_mag: int, d_w_neg: Optional[int], k_bits: int, rows: int, d_out: int) -> None:
        """Device-pointer variant (pb200_matvec_dev): enqueues on the key's stream, no synchronise, no range check; the sign step
        runs whenever d_w_neg is given."""
        check(self._lib.pb200_matvec_dev(self._h, d_c, count, d_w_mag, d_w_neg or None, k_bits, rows, d_out), "pb200_matvec_dev")

    def matvec(self, cs: Sequence[int], W) -> List[int]:
        """Enc(W m): W is a sequence of rows of Python ints (any sign) or a 2-D numpy integer array with one column per ciphertext.
        Row r of the result is prod c_i^|W[r, i]| over the positive weights times (the same over the negative ones)^(n - 1)."""
        mag, neg, k_bits = matvec_weights(W, len(cs))
        c_w = self._ciphertexts(cs, "matvec") if len(cs) else np.empty((0, self.words_out), dtype="<u8")
        return words_to_ints(self.matvec_words(c_w, mag, neg, k_bits)) if mag.shape[0] else []

    # -- witness ------------------------------------------------------------------------------
    def g_chain(self) -> List[Tuple[int, int]]:
        """Per-key records (q, rem) of the g-chain squarings, i < enc_bits."""
        out = np.empty((self.enc_bits, 2, self.words_out), dtype="<u8")
        check(self._lib.pb200_key_g_chain(self._h, _p(out)), "pb200_key_g_chain")
        return [(words_to_ints(out[i, 0])[0], words_to_ints(out[i, 1])[0]) for i in range(self.enc_bits)]

    def encrypt_witness(self, ms: Sequence[int], rs: Sequence[int], max_chunk_units: int = 0,
                        on_chunk: Optional[Callable] = None):
        """Returns (ciphertexts, per-unit list of (q, rem) records, per-unit g-chain mul counts).
        With `on_chunk`, chunks are handed to the callback as numpy views and not accumulated."""
        m_w = ints_to_words(ms, self.words_in)
        r_w = ints_to_words(rs, self.words_in)
        count = len(ms)
        c_out = np.empty((count, self.words_out), dtype="<u8")
        units: List[List[Tuple[int, int]]] = []
        gcounts: List[int] = []
        wo = self.words_out

        def sink(_user, chp):
            ch = chp.contents
            nu = ch.n_units
            offs = np.ctypeslib.as_array(ch.offsets, shape=(nu + 1,))
            total = int(offs[nu])
            recs = np.ctypeslib.as_array(ch.records, shape=(total, 2, wo))
            gc = np.ctypeslib.as_array(ch.g_mul_counts, shape=(nu,))
            if on_chunk is not None:
                return int(on_chunk(ch.first_unit, offs, recs, gc) or 0)
            for u in range(nu):
                rr = recs[int(offs[u]):int(offs[u + 1])]
                units.append([(int.from_bytes(x[0].tobytes(), "little"), int.from_bytes(x[1].tobytes(), "little")) for x in rr])
                gcounts.append(int(gc[u]))
            return 0

        cb = _lib.SINK_FN(sink)
        check(self._lib.pb200_encrypt_witness_batch(self._h, _p(m_w), _p(r_w), count, _p(c_out), max_chunk_units, cb, None),
              "pb200_encrypt_witness_batch")
        return words_to_ints(c_out) if count else [], units, gcounts

    def encrypt_witness_digest(self, ms: Sequence[int], rs: Sequence[int]):
        m_w = ints_to_words(ms, self.words_in)
        r_w = ints_to_words(rs, self.words_in)
        count = len(ms)
        c_out = np.empty((count, self.words_out), dtype="<u8")
        dig = np.empty(count, dtype="<u8")
        check(self._lib.pb200_encrypt_witness_digest(self._h, _p(m_w), _p(r_w), count, _p(c_out), _p(dig)),
              "pb200_encrypt_witness_digest")
        return (words_to_ints(c_out) if count else []), [int(d) for d in dig]

    def witness_records_for(self, m: int) -> int:
        return int(self._lib.pb200_witness_records_for(self._h, _p(ints_to_words([m], self.words_in))))

    def repack_limbs(self, vals: Sequence[int], value_bits: int, limb_bits: int) -> List[List[int]]:
        """decompose_biguint for limb_bits != 64 (K5): returns value_bits/limb_bits limbs per value."""
        v_w = ints_to_words(vals, words(value_bits))
        nl = value_bits // limb_bits
        out = np.empty((len(vals), nl, 2), dtype="<u8")
        check(self._lib.pb200_repack_limbs(self._h, _p(v_w), len(vals), value_bits, limb_bits, _p(out)), "pb200_repack_limbs")
        return [[int(out[i, j, 0]) | (int(out[i, j, 1]) << 64) for j in range(nl)] for i in range(len(vals))]


def matvec_weights(W, count: int) -> Tuple[np.ndarray, Optional[np.ndarray], int]:
    """Weights -> (magnitude words (rows, count, words(k_bits)), signs (rows, count) uint8 or None, k_bits = largest bit length, >= 1).
    A numpy integer array is converted without a Python loop; anything else is taken as rows of Python ints."""
    if isinstance(W, np.ndarray) and W.dtype.kind in "iu":
        if W.ndim != 2 or W.shape[1] != count:
            raise ValueError("W must have one column per ciphertext")
        if W.dtype.kind == "u":
            mag, neg = W.astype(np.uint64), None
        else:
            w64 = W.astype(np.int64)
            mag = np.abs(w64).astype(np.uint64)                   # |int64 min| wraps to 2^63 as uint64: exact
            neg = (w64 < 0).astype(np.uint8)
            if not neg.any():
                neg = None
        top = int(mag.max()) if mag.size else 0
        return np.ascontiguousarray(mag.reshape(W.shape[0], count, 1), dtype="<u8"), neg, max(1, top.bit_length())
    rows = [list(r) for r in W]
    if any(len(r) != count for r in rows):
        raise ValueError("every row of W needs one weight per ciphertext")
    flat = [int(v) for r in rows for v in r]
    k_bits = max([1] + [abs(v).bit_length() for v in flat])
    mag = ints_to_words([abs(v) for v in flat], words(k_bits)).reshape(len(rows), count, words(k_bits))
    neg = np.array([v < 0 for v in flat], dtype=np.uint8).reshape(len(rows), count) if any(v < 0 for v in flat) else None
    return mag, neg, k_bits


MATVEC_PLAN_FIELDS = ("method", "c", "windows", "passes", "segments", "acc_mulmods", "reduce_mulmods", "horner_mulmods", "sign_mulmods",
                      "chain", "temp_bytes")


def matvec_budget(n_bits: int) -> int:
    """Temporary device memory a matvec stays within (pb200_matvec): 3 * 2^18 ciphertexts of words_out words."""
    return 3 * (1 << 18) * 8 * words(2 * n_bits)


def matvec_plan(n_bits: int, sms: int, rows: int, count: int, k_bits: int, has_neg: bool) -> dict:
    """The plan pb200_matvec would use on a block28 engine (pb200_matvec_plan, host only): method 0 chain / 1 bucket, window width c,
    windows, passes, bucket segments per window, dense-weight mulmod upper bounds, longest sequential chain, temporary bytes."""
    out = np.zeros(11, dtype="<u8")
    check(_lib.load().pb200_matvec_plan(n_bits, sms, rows, count, k_bits, int(bool(has_neg)), _p(out)), "pb200_matvec_plan")
    return dict(zip(MATVEC_PLAN_FIELDS, (int(v) for v in out)))


def chip_order(m: int, n: int, g_chain: Sequence[Tuple[int, int]], unit_records: Sequence[Tuple[int, int]]):
    """Interleave the per-key g-chain squarings with one unit's record stream into the order in which
    PaillierChip::encrypt issues its mul_mods (src/paillier.rs:51,55,57; INTEGRATION.md §3):
    g-chain: for bit i of m low->high: sqr_i [, mul]; then the unit's r-chain records; then the final one."""
    out = []
    it = iter(unit_records)
    for i in range(m.bit_length()):
        out.append(g_chain[i])
        if (m >> i) & 1:
            out.append(next(it))
    out.extend(it)
    return out


MASK64 = (1 << 64) - 1
DIGEST_INIT = 0xCBF29CE484222325
DIGEST_PRIME = 0x100000001B3
DIGEST_C = 0x9E3779B97F4A7C15


def witness_digest(records: Iterable[Tuple[int, int]], words_out: int) -> int:
    """Host restatement of the device digest (include/paillier_b200.h): per record
    H = sum_j w_j * C^(j+1) mod 2^64 over the 2*words_out words (q then rem); D = (D ^ H) * PRIME."""
    d = DIGEST_INIT
    for q, rem in records:
        h = 0
        c = DIGEST_C
        for v in (q, rem):
            for j in range(words_out):
                h = (h + ((v >> (64 * j)) & MASK64) * c) & MASK64
                c = (c * DIGEST_C) & MASK64
        d = ((d ^ h) * DIGEST_PRIME) & MASK64
    return d


def private_from_primes(p: int, q: int, g: int):
    """(lambda, mu) of the Paillier key n = p*q, g: lambda = lcm(p-1, q-1), mu = L(g^lambda mod n^2)^-1 mod n.  Host-side key
    material preparation (a handful of big-integer operations per KEY, not per ciphertext)."""
    from math import gcd
    n = p * q
    lam = (p - 1) * (q - 1) // gcd(p - 1, q - 1)
    x = pow(g, lam, n * n)
    return lam, pow((x - 1) // n, -1, n)
