//! `extern "C"` binding of libptau_b200.so (include/ptau_b200.h).
//!
//! SOURCE ONLY: there is no Rust toolchain in the build image, so this file has never
//! been compiled.  It is the stub a maintainer of `kzg-setup-powersoftau` would add;
//! see INTEGRATION.md.
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int, c_uint, c_void};

pub const PTAU_G1: c_int = 1;
pub const PTAU_G2: c_int = 2;
pub const PTAU_FMT_ZCASH_UNCOMPRESSED: c_int = 1;
pub const PTAU_FMT_ZCASH_COMPRESSED: c_int = 2;
pub const PTAU_FMT_ARK_UNCOMPRESSED: c_int = 3;
pub const PTAU_FMT_ARK_MONT_LIMBS: c_int = 4;
pub const PTAU_CHECK_ON_CURVE: c_uint = 2;
pub const PTAU_CHECK_SUBGROUP: c_uint = 4;
pub const PTAU_CHECK_REJECT_INFINITY: c_uint = 8;
pub const PTAU_CHECKS_LOAD: c_uint = 0;
pub const PTAU_CHECKS_READ: c_uint = PTAU_CHECK_SUBGROUP;
pub const PTAU_CHECKS_STRICT: c_uint = 14;
pub const PTAU_VARIANT_KGZ: c_int = 1;
pub const PTAU_VARIANT_FASTKGZ: c_int = 2;
pub const PTAU_OK: c_int = 0;
pub const PTAU_BAD_NON_CANONICAL: c_int = 1;
pub const PTAU_BAD_FLAGS: c_int = 2;
pub const PTAU_BAD_INFINITY: c_int = 3;
pub const PTAU_BAD_NOT_ON_CURVE: c_int = 4;
pub const PTAU_BAD_NOT_IN_SUBGROUP: c_int = 5;
pub const PTAU_ERR_SIZE: c_int = -3;
pub const PTAU_ERR_IO: c_int = -5;
pub const PTAU_ERR_DIGEST: c_int = -6;
pub const PTAU_ERR_EXISTS: c_int = -7;
pub const PTAU_FILE_SKIP_DIGEST: c_uint = 1;
pub const PTAU_FILE_NO_UNCOMPRESSED: c_uint = 2;
pub const PTAU_FILE_FSYNC: c_uint = 4;

#[repr(C)]
pub struct ptau_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct ptau_kzg_powers {
    _private: [u8; 0],
}

#[link(name = "ptau_b200")]
extern "C" {
    pub fn ptau_device_count() -> c_int;
    pub fn ptau_create(ctx: *mut *mut ptau_ctx, n_gpus: c_int, device_ids: *const c_int, chunk_points: usize) -> c_int;
    pub fn ptau_destroy(ctx: *mut ptau_ctx);
    pub fn ptau_strerror(code: c_int) -> *const c_char;
    pub fn ptau_last_error(ctx: *mut ptau_ctx) -> *const c_char;
    pub fn ptau_host_alloc(bytes: usize) -> *mut c_void;
    pub fn ptau_host_free(p: *mut c_void);
    pub fn ptau_record_size(group: c_int, fmt: c_int) -> usize;
    pub fn ptau_response_size(n_powers: u64) -> u64;
    pub fn ptau_uncompressed_size(n_powers: u64) -> u64;
    pub fn ptau_setup_size(variant: c_int, n_powers: u64) -> u64;
    pub fn ptau_convert(
        ctx: *mut ptau_ctx, group: c_int, in_fmt: c_int, input: *const c_void, out_fmt: c_int, output: *mut c_void,
        n_points: usize, checks: c_uint, bad_index: *mut u64, bad_kind: *mut c_int,
    ) -> c_int;
    pub fn ptau_preprocess(
        ctx: *mut ptau_ctx, variant: c_int, response: *const c_void, response_len: u64, n_powers: u64,
        setup_out: *mut c_void, setup_len: u64, uncompressed_out: *mut c_void, uncompressed_len: u64, checks: c_uint,
        bad_index: *mut u64, bad_kind: *mut c_int, bad_section: *mut c_int,
    ) -> c_int;
    pub fn ptau_load_setup(
        ctx: *mut ptau_ctx, variant: c_int, setup: *const c_void, setup_len: u64, n_powers: u64, checks: c_uint,
        g1_out: *mut c_void, g1_out_len: u64, g2_out: *mut c_void, g2_out_len: u64, bad_index: *mut u64,
        bad_kind: *mut c_int,
    ) -> c_int;
    pub fn ptau_load_phase1(
        ctx: *mut ptau_ctx, data: *const c_void, len: u64, m: u64, checks: c_uint, g1_out: *mut c_void,
        g1_out_len: u64, g2_out: *mut c_void, g2_out_len: u64, bad_index: *mut u64, bad_kind: *mut c_int,
    ) -> c_int;
    pub fn ptau_preprocess_files(
        ctx: *mut ptau_ctx, variant: c_int, response_path: *const c_char, setup_path: *const c_char,
        uncompressed_path: *const c_char, log2_powers: c_uint, expected_digest_hex: *const c_char, flags: c_uint,
        checks: c_uint, bad_index: *mut u64, bad_kind: *mut c_int, bad_section: *mut c_int,
    ) -> c_int;
    pub fn ptau_load_setup_file(
        ctx: *mut ptau_ctx, variant: c_int, setup_path: *const c_char, n_powers: u64, checks: c_uint,
        g1_out: *mut c_void, g1_out_len: u64, g2_out: *mut c_void, g2_out_len: u64, n_powers_out: *mut u64,
        bad_index: *mut u64, bad_kind: *mut c_int,
    ) -> c_int;
    pub fn ptau_blake2b_file(path: *const c_char, out_hex: *mut c_char) -> c_int;
    pub fn ptau_kzg_commit(ctx: *mut ptau_ctx, powers: *const c_void, coeffs: *const c_void, n: usize, commitment: *mut c_void) -> c_int;
    pub fn ptau_kzg_powers_upload(ctx: *mut ptau_ctx, powers: *const c_void, n: usize, out: *mut *mut ptau_kzg_powers) -> c_int;
    pub fn ptau_kzg_powers_free(powers: *mut ptau_kzg_powers);
    pub fn ptau_kzg_commit_resident(ctx: *mut ptau_ctx, powers: *const ptau_kzg_powers, coeffs: *const c_void, n: usize, commitment: *mut c_void) -> c_int;
    pub fn ptau_kzg_quotient(coeffs: *const c_void, n: usize, point: *const c_void, quotient_out: *mut c_void, value_out: *mut c_void) -> c_int;
    pub fn ptau_kzg_open(
        ctx: *mut ptau_ctx, powers: *const ptau_kzg_powers, gamma_powers: *const ptau_kzg_powers, coeffs: *const c_void,
        n: usize, blinding: *const c_void, n_b: usize, points: *const c_void, k: usize, proofs_out: *mut c_void,
        values_out: *mut c_void, random_v_out: *mut c_void,
    ) -> c_int;
    pub fn ptau_kzg_open_cosets(
        ctx: *mut ptau_ctx, powers: *const ptau_kzg_powers, coeffs: *const c_void, n: usize, log2_k: c_int,
        shifts: *const c_void, m: usize, proofs_out: *mut c_void, values_out: *mut c_void,
    ) -> c_int;
    pub fn ptau_kzg_check_cosets(
        ctx: *mut ptau_ctx, powers: *const ptau_kzg_powers, h: *const c_void, tau_k_h: *const c_void, log2_k: c_int,
        comms: *const c_void, shifts: *const c_void, values: *const c_void, proofs: *const c_void, m: usize,
        seed: *const u8, ok: *mut u8,
    ) -> c_int;
    pub fn ptau_kzg_check(
        ctx: *mut ptau_ctx, vk_g1: *const c_void, vk_g2: *const c_void, comms: *const c_void, points: *const c_void,
        values: *const c_void, proofs_w: *const c_void, random_v: *const c_void, n: usize, ok: *mut u8,
    ) -> c_int;
    pub fn ptau_pairing_product2(
        ctx: *mut ptau_ctx, g1: *const c_void, g2: *const c_void, n: usize, gt_out: *mut c_void, is_one: *mut u8,
    ) -> c_int;
    pub fn ptau_g2_prepare(ctx: *mut ptau_ctx, g2: *const c_void, n: usize, coeffs_out: *mut c_void, infinity_out: *mut u8) -> c_int;
    pub fn ptau_challenge_size(n_powers: u64) -> u64;
    pub fn ptau_contribute(
        ctx: *mut ptau_ctx, challenge: *const c_void, challenge_len: u64, n_powers: u64, secrets: *const u8, checks: c_uint,
        response_out: *mut c_void, response_len: u64, bad_index: *mut u64, bad_kind: *mut c_int, bad_section: *mut c_int,
    ) -> c_int;
    pub fn ptau_verify_contribution(
        ctx: *mut ptau_ctx, challenge: *const c_void, challenge_len: u64, response: *const c_void, response_len: u64,
        n_powers: u64, seed: *const u8, bad_index: *mut u64, bad_kind: *mut c_int, bad_section: *mut c_int,
        bad_relation: *mut c_int,
    ) -> c_int;
}
