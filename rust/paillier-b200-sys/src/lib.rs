//! Raw bindings to `include/paillier_b200.h` plus a thin safe wrapper over word slices.
//!
//! NOT COMPILED IN THE BUILD ENVIRONMENT OF THIS REPOSITORY (no Rust toolchain there): the declarations are kept in step with the
//! header by `tests/test_abi.py::test_rust_sys_crate_declares_every_symbol`; the executable statement of how `PaillierChip`
//! consumes these calls is the C++ mirror `include/paillier_chip_host.hpp` (see INTEGRATION.md §3b).
//!
//! All integers are little-endian `u64` words (`BigUint::to_u64_digits()` order); every function returns 0 or a negative status.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct pb200_key {
    _private: [u8; 0],
}

pub const PB200_OK: c_int = 0;
pub const PB200_ERR_INVALID_ARG: c_int = -1;
pub const PB200_ERR_ZERO_MODULUS: c_int = -2;
pub const PB200_ERR_EVEN_MODULUS: c_int = -3;
pub const PB200_ERR_RANGE: c_int = -4;
pub const PB200_ERR_UNSUPPORTED: c_int = -5;
pub const PB200_ERR_CUDA: c_int = -6;
pub const PB200_ERR_NOMEM: c_int = -7;
pub const PB200_ERR_SINK: c_int = -8;
pub const PB200_ERR_CONSTRAINT: c_int = -9;
pub const PB200_ERR_PEER: c_int = -10;
pub const PB200_ERR_DECRYPT: c_int = -11;
pub const PB200_ERR_NOT_INVERTIBLE: c_int = -12;
pub const PB200_FLAG_RANGE: u32 = 1;
pub const PB200_FLAG_CONSTRAINT: u32 = 2;
pub const PB200_FLAG_PEER_TIMEOUT: u32 = 4;
pub const PB200_FLAG_DECRYPT: u32 = 8;
pub const PB200_FLAG_NOT_INVERTIBLE: u32 = 16;

/// 64-byte handle of a key's tally mailbox (CUDA IPC), exchanged between the ranks of a multi-process tally group
#[repr(C)]
#[derive(Clone, Copy)]
pub struct pb200_ipc_handle {
    pub bytes: [u8; 64],
}

#[repr(C)]
pub struct pb200_witness_chunk {
    pub first_unit: usize,
    pub n_units: usize,
    pub words_out: u32,
    pub offsets: *const u64,
    pub records: *const u64,
    pub g_mul_counts: *const u32,
}
pub type pb200_witness_sink_fn = extern "C" fn(user: *mut c_void, chunk: *const pb200_witness_chunk) -> c_int;

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct pb200_cell_layout {
    pub limbs: u32,
    pub cells_per_limb: u32,
    pub carry_bits: u32,
    pub cells_per_mulmod: u32,
    pub cells_n2: u32,
    pub off_rem: u32,
    pub off_ab: u32,
    pub off_qn: u32,
    pub off_qn_rem: u32,
    pub off_eq: u32,
    pub eq_stride: u32,
}

extern "C" {
    pub fn pb200_strerror(status: c_int) -> *const c_char;
    pub fn pb200_last_cuda_error() -> *const c_char;
    pub fn pb200_version() -> *const c_char;
    pub fn pb200_device_count() -> c_int;
    pub fn pb200_kernel_launches() -> u64;

    pub fn pb200_key_create(device: c_int, n_bits: u32, limb_bits: u32, n_le: *const u64, g_le: *const u64, out: *mut *mut pb200_key) -> c_int;
    pub fn pb200_key_destroy(key: *mut pb200_key);
    pub fn pb200_key_n_bits(key: *const pb200_key) -> u32;
    pub fn pb200_key_words_in(key: *const pb200_key) -> u32;
    pub fn pb200_key_words_out(key: *const pb200_key) -> u32;
    pub fn pb200_key_device(key: *const pb200_key) -> c_int;
    pub fn pb200_key_n2(key: *const pb200_key, n2_out: *mut u64) -> c_int;
    pub fn pb200_key_engine(key: *const pb200_key) -> *const c_char;
    pub fn pb200_key_set_engine(key: *mut pb200_key, engine: c_int) -> c_int;
    pub fn pb200_umma_layout(g: c_int, bl: c_int, lane_groups: c_int, witness: c_int, out20: *mut i32) -> c_int;
    pub fn pb200_key_shape(key: *const pb200_key, g_out: *mut c_int, bl_out: *mut c_int) -> c_int;
    pub fn pb200_debug_mulmod_cycles(key: *mut pb200_key, engine: c_int, v_in: *const i32, ctas: c_int, reps: c_int, stagger_cycles: c_int, cycles_out: *mut i64) -> c_int;
    pub fn pb200_debug_mulmod(key: *mut pb200_key, engine: c_int, v_in: *const i32, y_in: *const i32, reps: c_int, v_out: *mut i32, t_out: *mut i32, qhat_rows: *mut u32) -> c_int;
    pub fn pb200_key_stream(key: *const pb200_key) -> *mut c_void;
    pub fn pb200_key_chain_counts(key: *const pb200_key, n_sqr: *mut u64, n_mul: *mut u64) -> c_int;
    pub fn pb200_key_sync(key: *mut pb200_key) -> c_int;
    pub fn pb200_key_take_flags(key: *mut pb200_key, flags_out: *mut u32) -> c_int;

    pub fn pb200_encrypt_batch(key: *mut pb200_key, m_le: *const u64, r_le: *const u64, count: usize, c_out_le: *mut u64) -> c_int;
    pub fn pb200_encrypt_batch_dev(key: *mut pb200_key, d_m_le: *const u64, d_r_le: *const u64, count: usize, d_c_out_le: *mut u64) -> c_int;

    pub fn pb200_add_batch(key: *mut pb200_key, c1_le: *const u64, c2_le: *const u64, c_words: u32, count: usize, out_le: *mut u64, q_out_le: *mut u64) -> c_int;
    pub fn pb200_add_batch_dev(key: *mut pb200_key, d_c1_le: *const u64, d_c2_le: *const u64, c_words: u32, count: usize, d_out_le: *mut u64, d_q_out_le: *mut u64) -> c_int;

    pub fn pb200_tally(key: *mut pb200_key, c_le: *const u64, count: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_tally_dev(key: *mut pb200_key, d_c_le: *const u64, count: usize, d_partial_out_le: *mut u64) -> c_int;
    pub fn pb200_tally_combine(key: *mut pb200_key, partials_le: *const u64, n_partials: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_tally_trace(key: *mut pb200_key, init_le: *const u64, c_le: *const u64, count: usize, chains: usize, acc_out_le: *mut u64,
                             q_out_le: *mut u64) -> c_int;
    pub fn pb200_tally_trace_dev(key: *mut pb200_key, d_init_le: *const u64, d_c_le: *const u64, count: usize, chains: usize,
                                 d_acc_out_le: *mut u64, d_q_out_le: *mut u64) -> c_int;
    pub fn pb200_tally_multi(keys: *const *mut pb200_key, n_gpus: c_int, d_c: *const *const u64, counts: *const usize, out_le: *mut u64) -> c_int;
    pub fn pb200_tally_peer_export(key: *mut pb200_key, out: *mut pb200_ipc_handle) -> c_int;
    pub fn pb200_tally_peer_connect(key: *mut pb200_key, rank: c_int, world: c_int, handles: *const pb200_ipc_handle) -> c_int;
    pub fn pb200_tally_peer_dev(key: *mut pb200_key, d_c_le: *const u64, count: usize, d_out_le: *mut u64) -> c_int;

    pub fn pb200_key_set_private(key: *mut pb200_key, lambda_le: *const u64, mu_le: *const u64) -> c_int;
    pub fn pb200_decrypt_batch(key: *mut pb200_key, c_le: *const u64, count: usize, m_out_le: *mut u64) -> c_int;
    pub fn pb200_decrypt_batch_dev(key: *mut pb200_key, d_c_le: *const u64, count: usize, d_m_out_le: *mut u64) -> c_int;

    pub fn pb200_scalar_mul_batch(key: *mut pb200_key, c_le: *const u64, k_le: *const u64, k_bits: u32, count: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_scalar_mul_batch_dev(key: *mut pb200_key, d_c_le: *const u64, d_k_le: *const u64, k_bits: u32, count: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_tally_weighted(key: *mut pb200_key, c_le: *const u64, k_le: *const u64, k_bits: u32, count: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_tally_weighted_dev(key: *mut pb200_key, d_c_le: *const u64, d_k_le: *const u64, k_bits: u32, count: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_inverse_batch(key: *mut pb200_key, c_le: *const u64, count: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_inverse_batch_dev(key: *mut pb200_key, d_c_le: *const u64, count: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_sub_batch(key: *mut pb200_key, c1_le: *const u64, c2_le: *const u64, count: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_sub_batch_dev(key: *mut pb200_key, d_c1_le: *const u64, d_c2_le: *const u64, count: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_scalar_mul_signed_batch(key: *mut pb200_key, c_le: *const u64, k_mag_le: *const u64, k_neg: *const u8, k_bits: u32, count: usize,
                                         out_le: *mut u64) -> c_int;
    pub fn pb200_scalar_mul_signed_batch_dev(key: *mut pb200_key, d_c_le: *const u64, d_k_mag_le: *const u64, d_k_neg: *const u8, k_bits: u32,
                                             count: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_key_set_threshold(key: *mut pb200_key, parties: u32, phi_le: *const u64) -> c_int;
    pub fn pb200_key_set_share(key: *mut pb200_key, index: u32, s_le: *const u64) -> c_int;
    pub fn pb200_partial_decrypt_batch(key: *mut pb200_key, c_le: *const u64, count: usize, out_le: *mut u64) -> c_int;
    pub fn pb200_partial_decrypt_batch_dev(key: *mut pb200_key, d_c_le: *const u64, count: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_combine_shares_batch(key: *mut pb200_key, indices: *const u32, k: u32, shares_le: *const u64, count: usize,
                                      m_out_le: *mut u64) -> c_int;
    pub fn pb200_combine_shares_batch_dev(key: *mut pb200_key, indices: *const u32, k: u32, d_shares_le: *const u64, count: usize,
                                          d_m_out_le: *mut u64) -> c_int;
    pub fn pb200_matvec(key: *mut pb200_key, c_le: *const u64, count: usize, w_mag_le: *const u64, w_neg: *const u8, k_bits: u32, rows: usize,
                        out_le: *mut u64) -> c_int;
    pub fn pb200_matvec_dev(key: *mut pb200_key, d_c_le: *const u64, count: usize, d_w_mag_le: *const u64, d_w_neg: *const u8, k_bits: u32,
                            rows: usize, d_out_le: *mut u64) -> c_int;
    pub fn pb200_matvec_plan(n_bits: u32, sms: c_int, rows: usize, count: usize, k_bits: u32, has_neg: c_int, out11: *mut u64) -> c_int;

    pub fn pb200_encrypt_witness_batch(key: *mut pb200_key, m_le: *const u64, r_le: *const u64, count: usize, c_out_le: *mut u64,
                                       max_chunk_units: usize, sink: pb200_witness_sink_fn, user: *mut c_void) -> c_int;
    pub fn pb200_witness_records_for(key: *const pb200_key, m_le: *const u64) -> u64;
    pub fn pb200_encrypt_witness_digest(key: *mut pb200_key, m_le: *const u64, r_le: *const u64, count: usize, c_out_le: *mut u64, digest_out: *mut u64) -> c_int;
    pub fn pb200_encrypt_witness_digest_dev(key: *mut pb200_key, d_m_le: *const u64, d_r_le: *const u64, count: usize, d_c_out_le: *mut u64, d_digest_out: *mut u64) -> c_int;
    pub fn pb200_key_witness_engine(key: *mut pb200_key) -> *const c_char;
    pub fn pb200_key_g_chain(key: *mut pb200_key, records_out: *mut u64) -> c_int;

    pub fn pb200_cells_layout(key: *mut pb200_key, lookup_bits: u32, out: *mut pb200_cell_layout) -> c_int;
    pub fn pb200_mulmod_cells_batch(key: *mut pb200_key, a_le: *const u64, b_le: *const u64, q_le: *const u64, rem_le: *const u64, count: usize,
                                    lookup_bits: u32, montgomery: c_int, cells_out: *mut u64) -> c_int;
    pub fn pb200_mulmod_cells_batch_dev(key: *mut pb200_key, d_a_le: *const u64, d_b_le: *const u64, d_q_le: *const u64, d_rem_le: *const u64, count: usize,
                                        lookup_bits: u32, montgomery: c_int, d_cells_out: *mut u64) -> c_int;
    pub fn pb200_assign_cells_batch(key: *mut pb200_key, values_le: *const u64, count: usize, value_bits: u32, lookup_bits: u32,
                                    montgomery: c_int, cells_out: *mut u64) -> c_int;
    pub fn pb200_key_n2_cells(key: *mut pb200_key, lookup_bits: u32, montgomery: c_int, cells_out: *mut u64) -> c_int;

    pub fn pb200_repack_limbs(key: *mut pb200_key, values_le: *const u64, count: usize, value_bits: u32, limb_bits: u32, limbs_out: *mut u64) -> c_int;
}

/// Owning handle of a `pb200_key` with slice-based calls; `Err(status)` carries the library's negative status code.
pub struct Key {
    raw: *mut pb200_key,
}

// a key is bound to one device and one stream; calls on one key are serialised by `&mut self`
unsafe impl Send for Key {}

impl Key {
    /// `n`, `g`: `ceil(n_bits / 64)` words each (BigUint::to_u64_digits(), zero padded)
    pub fn new(device: i32, n_bits: u32, limb_bits: u32, n: &[u64], g: &[u64]) -> Result<Key, i32> {
        let words = ((n_bits + 63) / 64) as usize;
        if n.len() != words || g.len() != words {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut raw: *mut pb200_key = std::ptr::null_mut();
        let rc = unsafe { pb200_key_create(device, n_bits, limb_bits, n.as_ptr(), g.as_ptr(), &mut raw) };
        if rc == PB200_OK { Ok(Key { raw }) } else { Err(rc) }
    }
    pub fn words_in(&self) -> usize { unsafe { pb200_key_words_in(self.raw) as usize } }
    pub fn words_out(&self) -> usize { unsafe { pb200_key_words_out(self.raw) as usize } }
    pub fn as_ptr(&mut self) -> *mut pb200_key { self.raw }
    /// name of the arithmetic engine in effect ("block28u<8,19>" = tcgen05 + TMEM phases at |n| = 2048, "block28t<..>", "simple64")
    pub fn engine(&self) -> String {
        unsafe { std::ffi::CStr::from_ptr(pb200_key_engine(self.raw)).to_string_lossy().into_owned() }
    }
    /// 0 = automatic (fastest), 1 = simple64, 2 = block28, 3 = block28t (mma.sync), 4 = block28u (tcgen05), 5 = block28u2; every engine
    /// returns the same canonical words, so a host only calls this for A/B measurements
    pub fn set_engine(&mut self, engine: i32) -> Result<(), i32> {
        let rc = unsafe { pb200_key_set_engine(self.raw, engine as c_int) };
        if rc == PB200_OK { Ok(()) } else { Err(rc) }
    }

    /// batched `paillier_enc_native` (src/paillier.rs:87-92): `m`, `r` hold `count * words_in` words, the result `count * words_out`
    pub fn encrypt_batch(&mut self, m: &[u64], r: &[u64]) -> Result<Vec<u64>, i32> {
        let wi = self.words_in();
        if wi == 0 || m.len() != r.len() || m.len() % wi != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let count = m.len() / wi;
        let mut out = vec![0u64; count * self.words_out()];
        let rc = unsafe { pb200_encrypt_batch(self.raw, m.as_ptr(), r.as_ptr(), count, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// batched `paillier_add_native` (src/paillier.rs:94-97) with the mul_mod quotient: returns (c1*c2 mod n^2, floor(c1*c2 / n^2))
    pub fn add_batch(&mut self, c1: &[u64], c2: &[u64]) -> Result<(Vec<u64>, Vec<u64>), i32> {
        let wo = self.words_out();
        if wo == 0 || c1.len() != c2.len() || c1.len() % wo != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let count = c1.len() / wo;
        let (mut out, mut q) = (vec![0u64; c1.len()], vec![0u64; c1.len()]);
        let rc = unsafe { pb200_add_batch(self.raw, c1.as_ptr(), c2.as_ptr(), wo as u32, count, out.as_mut_ptr(), q.as_mut_ptr()) };
        if rc == PB200_OK { Ok((out, q)) } else { Err(rc) }
    }

    /// product of all ciphertexts mod n^2
    pub fn tally(&mut self, c: &[u64]) -> Result<Vec<u64>, i32> {
        let wo = self.words_out();
        if wo == 0 || c.len() % wo != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; wo];
        let rc = unsafe { pb200_tally(self.raw, c.as_ptr(), c.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// homomorphic scalar multiplication: `c` holds `count * words_out` words, `k` `count * ceil(k_bits / 64)` words (scalars below
    /// 2^k_bits, 1 <= k_bits <= n_bits; a negative scalar -s is n - s); returns c_i^(k_i) mod n^2, whose plaintext is k_i * m_i mod n
    pub fn scalar_mul_batch(&mut self, c: &[u64], k: &[u64], k_bits: u32) -> Result<Vec<u64>, i32> {
        let (wo, kw) = (self.words_out(), ((k_bits as usize) + 63) / 64);
        if wo == 0 || kw == 0 || c.len() % wo != 0 || k.len() != c.len() / wo * kw {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; c.len()];
        let rc = unsafe { pb200_scalar_mul_batch(self.raw, c.as_ptr(), k.as_ptr(), k_bits, c.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// weighted tally: prod c_i^(k_i) mod n^2, the ciphertext of sum k_i * m_i mod n (same layout of `c` and `k` as scalar_mul_batch)
    pub fn tally_weighted(&mut self, c: &[u64], k: &[u64], k_bits: u32) -> Result<Vec<u64>, i32> {
        let (wo, kw) = (self.words_out(), ((k_bits as usize) + 63) / 64);
        if wo == 0 || kw == 0 || c.len() % wo != 0 || k.len() != c.len() / wo * kw {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; wo];
        let rc = unsafe { pb200_tally_weighted(self.raw, c.as_ptr(), k.as_ptr(), k_bits, c.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// c_i^-1 mod n^2 for `count * words_out` words of ciphertexts: the ciphertexts of -m_i mod n.  A unit without an inverse
    /// (gcd(c_i, n) != 1) makes the call return `Err(PB200_ERR_NOT_INVERTIBLE)`; `PB200_ERR_EVEN_MODULUS` for an even n
    pub fn inverse_batch(&mut self, c: &[u64]) -> Result<Vec<u64>, i32> {
        let wo = self.words_out();
        if wo == 0 || c.len() % wo != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; c.len()];
        let rc = unsafe { pb200_inverse_batch(self.raw, c.as_ptr(), c.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// homomorphic subtraction: c1_i * c2_i^-1 mod n^2, the ciphertexts of m1_i - m2_i mod n (errors as `inverse_batch`)
    pub fn sub_batch(&mut self, c1: &[u64], c2: &[u64]) -> Result<Vec<u64>, i32> {
        let wo = self.words_out();
        if wo == 0 || c1.len() != c2.len() || c1.len() % wo != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; c1.len()];
        let rc = unsafe { pb200_sub_batch(self.raw, c1.as_ptr(), c2.as_ptr(), c1.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// scalar multiplication with signed scalars: `k_mag` as `k` of scalar_mul_batch, `k_neg` (empty, or one byte per ciphertext,
    /// non-zero = negative); returns c_i^(k_i) mod n^2 exactly (c^-s = (c^-1)^s, scalars not reduced mod n), the ciphertext of k_i * m_i
    pub fn scalar_mul_signed_batch(&mut self, c: &[u64], k_mag: &[u64], k_neg: &[u8], k_bits: u32) -> Result<Vec<u64>, i32> {
        let (wo, kw) = (self.words_out(), ((k_bits as usize) + 63) / 64);
        if wo == 0 || kw == 0 || c.len() % wo != 0 || k_mag.len() != c.len() / wo * kw || (!k_neg.is_empty() && k_neg.len() != c.len() / wo) {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; c.len()];
        let neg = if k_neg.is_empty() { std::ptr::null() } else { k_neg.as_ptr() };
        let rc = unsafe { pb200_scalar_mul_signed_batch(self.raw, c.as_ptr(), k_mag.as_ptr(), neg, k_bits, c.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// threshold decryption: `parties` trustees (1 ..= 32) and phi = L(g^(4 Delta^2 d) mod n^2)^-1 mod n (`words_in` words); clears
    /// any share set on this key
    pub fn set_threshold(&mut self, parties: u32, phi: &[u64]) -> Result<(), i32> {
        if phi.len() != self.words_in() {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let rc = unsafe { pb200_key_set_threshold(self.raw, parties, phi.as_ptr()) };
        if rc == PB200_OK { Ok(()) } else { Err(rc) }
    }

    /// this key's trustee: `index` (1 ..= parties) and its share s_index (`words_out` words)
    pub fn set_share(&mut self, index: u32, share: &[u64]) -> Result<(), i32> {
        if share.len() != self.words_out() {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let rc = unsafe { pb200_key_set_share(self.raw, index, share.as_ptr()) };
        if rc == PB200_OK { Ok(()) } else { Err(rc) }
    }

    /// the trustee's partial decryptions c_i^(2 Delta s) mod n^2 of `count * words_out` words of ciphertexts
    pub fn partial_decrypt_batch(&mut self, c: &[u64]) -> Result<Vec<u64>, i32> {
        let wo = self.words_out();
        if wo == 0 || c.len() % wo != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; c.len()];
        let rc = unsafe { pb200_partial_decrypt_batch(self.raw, c.as_ptr(), c.len() / wo, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// combination of the partial decryptions of the trustees `indices`: `shares` share-major (share j of ciphertext u at
    /// `(j * count + u) * words_out`); returns `count * words_in` words of plaintexts.  `Err(PB200_ERR_DECRYPT)` when too few or wrong
    /// shares leave some unit without an exact L (`PB200_ERR_NOT_INVERTIBLE` when its N has no inverse)
    pub fn combine_shares_batch(&mut self, indices: &[u32], shares: &[u64]) -> Result<Vec<u64>, i32> {
        let (wo, k) = (self.words_out(), indices.len());
        if wo == 0 || k == 0 || shares.len() % (k * wo) != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let count = shares.len() / (k * wo);
        let mut out = vec![0u64; count * self.words_in()];
        let rc = unsafe { pb200_combine_shares_batch(self.raw, indices.as_ptr(), k as u32, shares.as_ptr(), count, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// encrypted matrix-vector product: `c` holds `count * words_out` words, `w_mag` the magnitudes of a `rows x count` weight matrix
    /// row-major (`ceil(k_bits / 64)` words each, below 2^k_bits), `w_neg` (empty, or `rows * count` bytes) marks the negative ones;
    /// returns `rows * words_out` words, row r the ciphertext of sum_i w_ri * m_i mod n
    pub fn matvec(&mut self, c: &[u64], w_mag: &[u64], w_neg: &[u8], k_bits: u32, rows: usize) -> Result<Vec<u64>, i32> {
        let (wo, kw) = (self.words_out(), ((k_bits as usize) + 63) / 64);
        if wo == 0 || kw == 0 || c.len() % wo != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let count = c.len() / wo;
        if w_mag.len() != rows * count * kw || (!w_neg.is_empty() && w_neg.len() != rows * count) {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let mut out = vec![0u64; rows * wo];
        let neg = if w_neg.is_empty() { std::ptr::null() } else { w_neg.as_ptr() };
        let rc = unsafe { pb200_matvec(self.raw, c.as_ptr(), count, w_mag.as_ptr(), neg, k_bits, rows, out.as_mut_ptr()) };
        if rc == PB200_OK { Ok(out) } else { Err(rc) }
    }

    /// running-tally trace: `init` holds `chains * words_out` words, `c` the steps row by row (`count * chains * words_out` words, entry
    /// (i, j) at `(i * chains + j) * words_out`); returns (acc, q), each laid out like `c`, with
    /// (q_ij, acc_ij) = divmod(acc_(i-1)j * c_ij, n^2) and acc_(-1)j = init_j: the (q, rem) of every `PaillierChip::add` of the chains
    pub fn tally_trace(&mut self, init: &[u64], c: &[u64]) -> Result<(Vec<u64>, Vec<u64>), i32> {
        let wo = self.words_out();
        if wo == 0 || init.is_empty() || init.len() % wo != 0 || c.len() % init.len() != 0 {
            return Err(PB200_ERR_INVALID_ARG);
        }
        let (chains, count) = (init.len() / wo, c.len() / init.len());
        let (mut acc, mut q) = (vec![0u64; c.len()], vec![0u64; c.len()]);
        let rc = unsafe { pb200_tally_trace(self.raw, init.as_ptr(), c.as_ptr(), count, chains, acc.as_mut_ptr(), q.as_mut_ptr()) };
        if rc == PB200_OK { Ok((acc, q)) } else { Err(rc) }
    }
}

impl Drop for Key {
    fn drop(&mut self) {
        unsafe { pb200_key_destroy(self.raw) }
    }
}
