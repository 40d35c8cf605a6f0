//! Raw bindings of `include/blsgpu.h` (C ABI of the B200 batch BLS12-381 verification engine).
//! One declaration per entry point; see the header for the reference function each one replaces.
#![allow(non_camel_case_types)]
#![no_std]

use core::ffi::{c_char, c_int, c_void};

#[repr(C)]
pub struct blsgpu_ctx {
    _private: [u8; 0],
}

// engine errors (function results)
pub const BLSGPU_OK: c_int = 0;
pub const BLSGPU_E_ARG: c_int = -1;
pub const BLSGPU_E_CUDA: c_int = -2;
pub const BLSGPU_E_ALLOC: c_int = -3;

// per-item statuses = the reference's outcome for the item
pub const BLSGPU_ST_OK: u8 = 0;
pub const BLSGPU_ST_INVALID_SIGNATURE: u8 = 1;
pub const BLSGPU_ST_SIG_IDENTITY: u8 = 2;
pub const BLSGPU_ST_PK_IDENTITY: u8 = 3;
pub const BLSGPU_ST_DESERIALIZE: u8 = 4;
pub const BLSGPU_ST_LEGACY_FORMAT: u8 = 5;
pub const BLSGPU_ST_INVALID_LENGTH: u8 = 6;
pub const BLSGPU_ST_INVALID_COEFFICIENT: u8 = 7;
pub const BLSGPU_ST_DUPLICATE_MESSAGES: u8 = 8;
pub const BLSGPU_ST_SCHEME: u8 = 9;
pub const BLSGPU_ST_MISMATCHED_LENGTHS: u8 = 10;
pub const BLSGPU_ST_VSSS: u8 = 11;
pub const BLSGPU_ST_INVALID_PROOF: u8 = 12;
pub const BLSGPU_ST_COMMITMENT_IDENTITY: u8 = 13;
pub const BLSGPU_ST_PROOF_IDENTITY: u8 = 14;
pub const BLSGPU_ST_ZERO_CHALLENGE: u8 = 15;

pub const BLSGPU_STAGE_COUNT: usize = 8;
pub const BLSGPU_KERNEL_COUNT: usize = 10;

extern "C" {
    // ---- context -----------------------------------------------------------------------------------------------
    pub fn blsgpu_ctx_create(devices: *const c_int, ndev: c_int, out: *mut *mut blsgpu_ctx) -> c_int;
    pub fn blsgpu_ctx_destroy(ctx: *mut blsgpu_ctx);
    pub fn blsgpu_last_error(ctx: *const blsgpu_ctx) -> *const c_char;
    pub fn blsgpu_ctx_set_stream(ctx: *mut blsgpu_ctx, cuda_stream: *mut c_void) -> c_int;
    pub fn blsgpu_ctx_set_rlc_salt(ctx: *mut blsgpu_ctx, salt: *const u8) -> c_int; // 32 bytes; tests only
    pub fn blsgpu_ctx_set_rlc_bits(ctx: *mut blsgpu_ctx, bits: c_int) -> c_int; // 64 | 128
    pub fn blsgpu_selftest(ctx: *mut blsgpu_ctx) -> c_int;

    // ---- Signature::verify / ProofOfPossession::verify over slices ------------------------------------------------
    pub fn blsgpu_verify_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, n: usize,
        pks: *const u8, sigs: *const u8, msgs: *const u8, msg_off: *const u64, status_out: *mut u8) -> c_int;
    pub fn blsgpu_verify_batch_grouped(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, n: usize,
        pks: *const u8, sigs: *const u8, msg_idx: *const u32, q: usize, msgs: *const u8, msg_off: *const u64,
        status_out: *mut u8) -> c_int;

    // ---- key sets: public keys decoded once, verify calls that name them by index ------------------------------------
    pub fn blsgpu_keyset_create(ctx: *mut blsgpu_ctx, impl_id: c_int, format: c_int, n: usize, pks: *const u8,
        status_out: *mut u8 /* [n] or null */, keyset_out: *mut u64) -> c_int;
    pub fn blsgpu_keyset_destroy(ctx: *mut blsgpu_ctx, keyset: u64) -> c_int;
    pub fn blsgpu_keyset_update(ctx: *mut blsgpu_ctx, keyset: u64, format: c_int, k: usize, key_idx: *const u32, pks: *const u8,
        status_out: *mut u8 /* [k] or null */) -> c_int;
    pub fn blsgpu_keyset_append(ctx: *mut blsgpu_ctx, keyset: u64, format: c_int, k: usize, pks: *const u8,
        status_out: *mut u8 /* [k] or null */) -> c_int;
    pub fn blsgpu_verify_batch_keyed(ctx: *mut blsgpu_ctx, keyset: u64, scheme: c_int, format: c_int, n: usize,
        key_idx: *const u32, sigs: *const u8, msgs: *const u8, msg_off: *const u64, status_out: *mut u8) -> c_int;
    pub fn blsgpu_verify_batch_grouped_keyed(ctx: *mut blsgpu_ctx, keyset: u64, scheme: c_int, format: c_int, n: usize,
        key_idx: *const u32, sigs: *const u8, msg_idx: *const u32, q: usize, msgs: *const u8, msg_off: *const u64,
        status_out: *mut u8) -> c_int;

    pub fn blsgpu_verify_batch_dev(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, n: usize,
        pks_dev: *const u8, sigs_dev: *const u8, msgs_dev: *const u8, msg_off_dev: *const u64,
        status_out_dev: *mut u8) -> c_int;
    pub fn blsgpu_pop_verify_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, format: c_int, n: usize, pks: *const u8,
        sigs: *const u8, status_out: *mut u8) -> c_int;

    // ---- one batch over several GPUs / processes: slice-local partial results, fold, finish -------------------------
    pub fn blsgpu_miller_partial(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, n: usize,
        pks: *const u8, sigs: *const u8, msgs: *const u8, msg_off: *const u64, gt_out: *mut u8 /* 576 */,
        sum_out: *mut u8 /* 96 | 48 */) -> c_int;
    pub fn blsgpu_final_exp_is_one(ctx: *mut blsgpu_ctx, impl_id: c_int, k: usize, partial_gts: *const u8,
        partial_sums: *const u8, is_one_out: *mut c_int) -> c_int;
    pub fn blsgpu_partial_finish(ctx: *mut blsgpu_ctx, batch_ok: c_int, status_out: *mut u8) -> c_int;

    // ---- AggregateSignature::verify, point sums ---------------------------------------------------------------------
    pub fn blsgpu_aggregate_verify(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, n: usize,
        pks: *const u8, msgs: *const u8, msg_off: *const u64, sig: *const u8, status_out: *mut u8,
        index_out: *mut i64 /* [2] */) -> c_int;
    pub fn blsgpu_aggregate_verify_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, q: usize,
        set_off: *const u64, pks: *const u8, msgs: *const u8, msg_off: *const u64, sigs: *const u8, status_out: *mut u8,
        index_out: *mut i64 /* [2 q] or null */) -> c_int;
    pub fn blsgpu_sum_points(ctx: *mut blsgpu_ctx, group: c_int, format: c_int, n: usize, points: *const u8,
        out: *mut u8, status_out: *mut u8, bad_index_out: *mut i64) -> c_int;

    // ---- secure aggregation -------------------------------------------------------------------------------------------
    pub fn blsgpu_verify_secure_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, q: usize,
        key_off: *const u64, pks: *const u8, sigs: *const u8, msgs: *const u8, msg_off: *const u64,
        status_out: *mut u8) -> c_int;
    pub fn blsgpu_aggregate_secure_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, format: c_int, q: usize,
        key_off: *const u64, pks: *const u8, member_sigs: *const u8, out_sigs: *mut u8, status_out: *mut u8) -> c_int;
    pub fn blsgpu_verify_secure_batch_keyed(ctx: *mut blsgpu_ctx, keyset: u64, scheme: c_int, format: c_int, q: usize,
        key_off: *const u64, key_idx: *const u32, sigs: *const u8, msgs: *const u8, msg_off: *const u64,
        status_out: *mut u8) -> c_int;
    pub fn blsgpu_aggregate_secure_batch_keyed(ctx: *mut blsgpu_ctx, keyset: u64, format: c_int, q: usize,
        key_off: *const u64, key_idx: *const u32, member_sigs: *const u8, out_sigs: *mut u8, status_out: *mut u8) -> c_int;

    // ---- multi-signatures over signer subsets ------------------------------------------------------------------------------
    pub fn blsgpu_verify_multisig_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, format: c_int, q: usize,
        key_off: *const u64, pks: *const u8, sigs: *const u8, msgs: *const u8, msg_off: *const u64,
        status_out: *mut u8) -> c_int;
    pub fn blsgpu_verify_multisig_batch_keyed(ctx: *mut blsgpu_ctx, keyset: u64, scheme: c_int, format: c_int, q: usize,
        key_off: *const u64, key_idx: *const u32, sigs: *const u8, msgs: *const u8, msg_off: *const u64,
        status_out: *mut u8) -> c_int;
    pub fn blsgpu_sum_points_batch(ctx: *mut blsgpu_ctx, group: c_int, format: c_int, q: usize, set_off: *const u64,
        points: *const u8, out: *mut u8, status_out: *mut u8, bad_index_out: *mut i64 /* [q] or null */) -> c_int;

    // ---- threshold shares -----------------------------------------------------------------------------------------------
    /// shares: records of 32 + 48|96 bytes = `Vec::<u8>::from(&InnerPointShareG1|G2)` (reference src/lib.rs:150-157)
    pub fn blsgpu_combine_shares_batch(ctx: *mut blsgpu_ctx, group: c_int, q: usize, share_off: *const u64,
        shares: *const u8, out: *mut u8, status_out: *mut u8) -> c_int;
    pub fn blsgpu_verify_share_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, n: usize,
        pk_shares: *const u8, sig_shares: *const u8, msgs: *const u8, msg_off: *const u64, status_out: *mut u8) -> c_int;

    // ---- wire front ends --------------------------------------------------------------------------------------------------
    /// tagged_sigs: n records of 1 + 96|48 bytes = `Vec::<u8>::from(&Signature<C>)` (reference src/signature.rs:112-118)
    pub fn blsgpu_verify_batch_wire(ctx: *mut blsgpu_ctx, impl_id: c_int, n: usize, pks: *const u8,
        tagged_sigs: *const u8, msgs: *const u8, msg_off: *const u64, status_out: *mut u8) -> c_int;
    /// ragged records; scheme_or_tagged < 0: serde_bare tagged signatures, else raw signatures of that scheme in `format`
    pub fn blsgpu_verify_batch_records(ctx: *mut blsgpu_ctx, impl_id: c_int, format: c_int, scheme_or_tagged: c_int,
        n: usize, pk_bytes: *const u8, pk_off: *const u64, sig_bytes: *const u8, sig_off: *const u64,
        msgs: *const u8, msg_off: *const u64, status_out: *mut u8) -> c_int;

    // ---- the other public 2-pairing checks ---------------------------------------------------------------------------------
    pub fn blsgpu_signcrypt_valid_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, n: usize,
        u_points: *const u8, w_points: *const u8, v_bytes: *const u8, v_off: *const u64, ok_out: *mut u8,
        status_out: *mut u8) -> c_int;
    pub fn blsgpu_signcrypt_verify_share_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, n: usize,
        shares: *const u8, pk_shares: *const u8, u_points: *const u8, w_points: *const u8, v_bytes: *const u8,
        v_off: *const u64, ok_out: *mut u8, status_out: *mut u8) -> c_int;
    pub fn blsgpu_pok_verify_batch(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, n: usize,
        commitments: *const u8, proofs: *const u8, pks: *const u8, challenges32: *const u8, msgs: *const u8,
        msg_off: *const u64, status_out: *mut u8) -> c_int;
    pub fn blsgpu_pairing_check_batch(ctx: *mut blsgpu_ctx, q: usize, pair_off: *const u64, g1_points: *const u8,
        g2_points: *const u8, ok_out: *mut u8, status_out: *mut u8) -> c_int;

    // ---- building blocks ---------------------------------------------------------------------------------------------------
    pub fn blsgpu_hash_to_curve_batch(ctx: *mut blsgpu_ctx, group: c_int, n: usize, msgs: *const u8,
        msg_off: *const u64, dst: *const u8, dst_len: usize, out: *mut u8) -> c_int;
    pub fn blsgpu_recode_points(ctx: *mut blsgpu_ctx, group: c_int, format_in: c_int, format_out: c_int, n: usize,
        input: *const u8, out: *mut u8, status_out: *mut u8) -> c_int;
    pub fn blsgpu_fp_mul_batch(ctx: *mut blsgpu_ctx, variant: c_int, n: usize, a: *const u8, b: *const u8,
        out: *mut u8) -> c_int;
    pub fn blsgpu_pairing_product_is_one(ctx: *mut blsgpu_ctx, n: usize, g1_points: *const u8, g2_points: *const u8,
        is_one_out: *mut c_int) -> c_int;
    pub fn blsgpu_testdata_sign(ctx: *mut blsgpu_ctx, impl_id: c_int, scheme: c_int, n: usize, scalars32: *const u8,
        msgs: *const u8, msg_off: *const u64, out_pks: *mut u8, out_sigs: *mut u8) -> c_int;
    pub fn blsgpu_imad_peak(ctx: *mut blsgpu_ctx, mac_per_s_out: *mut f64) -> c_int;
    pub fn blsgpu_plan_msm(n: usize, scalar_bits: c_int, window_bits_out: *mut c_int, windows_out: *mut c_int,
        top_window_bits_out: *mut c_int) -> c_int;
    pub fn blsgpu_plan_shards(sets: usize, set_off: *const u64, ndev: c_int, cut_out: *mut u64) -> c_int;

    // ---- metrics -------------------------------------------------------------------------------------------------------------
    pub fn blsgpu_last_stage_ms(ctx: *const blsgpu_ctx, ms_out: *mut f32 /* [BLSGPU_STAGE_COUNT] */) -> c_int;
    pub fn blsgpu_last_kernel_ms(ctx: *const blsgpu_ctx, ms_out: *mut f32 /* [BLSGPU_KERNEL_COUNT] */,
        launches_out: *mut c_int) -> c_int;
    pub fn blsgpu_launch_count(ctx: *const blsgpu_ctx) -> u64;
}
