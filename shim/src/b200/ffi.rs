//! `extern "C"` declarations of include/milagro_bls_b200.h, one per header entry (tests/test_abi.py keeps the two in step).
//! Comments name the reference item each entry serves (M = /root/reference/src).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct b3_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct b3_keytable {
    _private: [u8; 0],
}
#[repr(C)]
pub struct b3_comm {
    _private: [u8; 0],
}

pub const B3_OK: c_int = 0;
pub const B3_ERR_AGGREGATE_EMPTY_POINTS: c_int = -1;
pub const B3_ERR_INVALID_POINT: c_int = -5;
pub const B3_ERR_INVALID_G1_SIZE: c_int = -6;
pub const B3_ERR_INVALID_G2_SIZE: c_int = -7;
pub const B3_ERR_INVALID_YFLAG: c_int = -8;
pub const B3_ITEM_VERIFY: c_int = 0;
pub const B3_ITEM_FAST_AGGREGATE: c_int = 1;
pub const B3_ITEM_PRE_AGGREGATED: c_int = 2;
pub const B3_PARTIAL_BYTES: usize = 592;

extern "C" {
    // ---- contexts
    pub fn b3_ctx_create(device: c_int, out: *mut *mut b3_ctx) -> c_int;
    pub fn b3_ctx_destroy(ctx: *mut b3_ctx);
    pub fn b3_last_error(ctx: *mut b3_ctx) -> *const c_char;
    pub fn b3_ctx_stream(ctx: *mut b3_ctx) -> *mut c_void;
    pub fn b3_ctx_launch_count(ctx: *mut b3_ctx) -> u64;
    pub fn b3_ctx_last_kernel_ms(ctx: *mut b3_ctx, which: c_int) -> f32;
    pub fn b3_ctx_stage_ms(ctx: *mut b3_ctx, stage: c_int) -> f32;
    pub fn b3_stage_name(stage: c_int) -> *const c_char;
    pub fn b3_stage_count() -> c_int;
    pub fn b3_ctx_set_serial(ctx: *mut b3_ctx, serial: c_int);
    pub fn b3_ctx_set_item_kernel(ctx: *mut b3_ctx, which: c_int);
    pub fn b3_ctx_set_trusted_points(ctx: *mut b3_ctx, trusted: c_int);
    pub fn b3_ctx_set_latency_mode(ctx: *mut b3_ctx, mode: c_int);
    // ---- (de)serialisation: M/keys.rs:140-186, M/signature.rs:43-51, M/aggregates.rs:319-327
    pub fn b3_g1_decompress(ctx: *mut b3_ctx, in48: *const u8, n: usize, validate: c_int, out96: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_g2_decompress(ctx: *mut b3_ctx, in96: *const u8, n: usize, out192: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_g1_compress(ctx: *mut b3_ctx, in96: *const u8, n: usize, out48: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_g2_compress(ctx: *mut b3_ctx, in192: *const u8, n: usize, out96: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_g1_validate(ctx: *mut b3_ctx, in96: *const u8, n: usize, status: *mut i32, valid: *mut i32) -> c_int;
    pub fn b3_g2_subgroup_check(ctx: *mut b3_ctx, in192: *const u8, n: usize, status: *mut i32, ok: *mut i32) -> c_int;
    // ---- aggregation: M/aggregates.rs:29-56, 100-106
    pub fn b3_g1_aggregate(ctx: *mut b3_ctx, pks96: *const u8, off: *const u32, n_sets: usize, out96: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_g2_aggregate(ctx: *mut b3_ctx, sigs192: *const u8, off: *const u32, n_sets: usize, out192: *mut u8, status: *mut i32) -> c_int;
    // ---- M/amcl_utils.rs:33-35
    pub fn b3_hash_to_g2(ctx: *mut b3_ctx, msgs: *const u8, off: *const u32, n: usize, dst: *const u8, dst_len: usize, out192: *mut u8) -> c_int;
    // ---- verification: M/signature.rs:27-40, M/aggregates.rs:130-316
    pub fn b3_verify(ctx: *mut b3_ctx, sig192: *const u8, pk96: *const u8, msg: *const u8, msg_len: usize, accept: *mut c_int, gt576: *mut u8) -> c_int;
    pub fn b3_fast_aggregate_verify(ctx: *mut b3_ctx, sig192: *const u8, pks96: *const u8, n_pks: usize, msg: *const u8, msg_len: usize,
                                    accept: *mut c_int, gt576: *mut u8) -> c_int;
    pub fn b3_fast_aggregate_verify_pre_aggregated(ctx: *mut b3_ctx, sig192: *const u8, apk96: *const u8, msg: *const u8, msg_len: usize,
                                                   accept: *mut c_int, gt576: *mut u8) -> c_int;
    pub fn b3_aggregate_verify(ctx: *mut b3_ctx, sig192: *const u8, pks96: *const u8, msgs: *const u8, msg_off: *const u32, n: usize,
                               accept: *mut c_int, gt576: *mut u8) -> c_int;
    pub fn b3_verify_multiple(ctx: *mut b3_ctx, sigs192: *const u8, pks96: *const u8, pk_off: *const u32, msgs: *const u8, msg_off: *const u32,
                              scalars: *const u64, n: usize, accept: *mut c_int, first_bad: *mut i64, gt576: *mut u8) -> c_int;
    pub fn b3_verify_multiple_dev(ctx: *mut b3_ctx, sigs192_dev: *const u8, pks96_dev: *const u8, pk_off_dev: *const u32, msgs_dev: *const u8,
                                  msg_off_dev: *const u32, scalars_dev: *const u64, n: usize, accept: *mut c_int, first_bad: *mut i64,
                                  gt576: *mut u8) -> c_int;
    pub fn b3_verify_multiple_indexed_dev(ctx: *mut b3_ctx, t: *const b3_keytable, sigs192_dev: *const u8, key_idx_dev: *const u32,
                                          pk_off_dev: *const u32, msgs_dev: *const u8, msg_off_dev: *const u32, scalars_dev: *const u64,
                                          n: usize, accept: *mut c_int, first_bad: *mut i64, gt576: *mut u8) -> c_int;
    // sets naming their message by index: one hash and one Miller pair per distinct message
    pub fn b3_verify_multiple_grouped(ctx: *mut b3_ctx, t: *const b3_keytable, sigs192: *const u8, keys: *const c_void, pk_off: *const u32,
                                      msgs: *const u8, msg_off: *const u32, n_msgs: usize, msg_idx: *const u32, scalars: *const u64,
                                      n: usize, device_pointers: c_int, accept: *mut c_int, first_bad: *mut i64, gt576: *mut u8) -> c_int;
    // per-set verdicts after a rejected whole verify_multiple call on the same context
    pub fn b3_verify_multiple_locate(ctx: *mut b3_ctx, n: usize, valid: *mut i32, n_invalid: *mut usize) -> c_int;
    // two-phase form: the RNG contract of M/aggregates.rs:272-287 without running the subgroup checks twice
    pub fn b3_sig_precheck(ctx: *mut b3_ctx, sigs192: *const u8, n: usize, first_bad: *mut i64) -> c_int;
    pub fn b3_verify_multiple_checked(ctx: *mut b3_ctx, pks96: *const u8, pk_off: *const u32, msgs: *const u8, msg_off: *const u32,
                                      scalars: *const u64, n: usize, accept: *mut c_int, gt576: *mut u8) -> c_int;
    // ---- device-resident key table: PublicKey::from_bytes paid once per validator (M/keys.rs:140-147)
    pub fn b3_keytable_create(ctx: *mut b3_ctx, capacity: usize, out: *mut *mut b3_keytable) -> c_int;
    pub fn b3_keytable_destroy(t: *mut b3_keytable);
    pub fn b3_keytable_size(t: *const b3_keytable) -> usize;
    pub fn b3_keytable_append(ctx: *mut b3_ctx, t: *mut b3_keytable, keys: *const u8, n: usize, compressed: c_int, validate: c_int,
                              status: *mut i32, first_index: *mut usize) -> c_int;
    pub fn b3_keytable_get(ctx: *mut b3_ctx, t: *const b3_keytable, idx: *const u32, n: usize, out96: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_g1_aggregate_indexed(ctx: *mut b3_ctx, t: *const b3_keytable, key_idx: *const u32, off: *const u32, n_sets: usize,
                                   out96: *mut u8, status: *mut i32) -> c_int;
    pub fn b3_verify_multiple_indexed(ctx: *mut b3_ctx, t: *const b3_keytable, sigs192: *const u8, key_idx: *const u32, pk_off: *const u32,
                                      msgs: *const u8, msg_off: *const u32, scalars: *const u64, n: usize, accept: *mut c_int,
                                      first_bad: *mut i64, gt576: *mut u8) -> c_int;
    // ---- n independent items, one accept bit each (locating the bad set after a batch reject)
    pub fn b3_verify_batch(ctx: *mut b3_ctx, mode: c_int, sigs192: *const u8, pks96: *const u8, pk_off: *const u32, msgs: *const u8,
                           msg_off: *const u32, n: usize, accept: *mut i32, status: *mut i32, gt576: *mut u8) -> c_int;
    pub fn b3_verify_batch_dev(ctx: *mut b3_ctx, mode: c_int, sigs192_dev: *const u8, pks96_dev: *const u8, pk_off_dev: *const u32,
                               msgs_dev: *const u8, msg_off_dev: *const u32, n: usize, accept_dev: *mut i32, status_dev: *mut i32,
                               gt576_dev: *mut u8) -> c_int;
    // ---- sharded verify_multiple, one process per GPU (partials + combine; the b3_comm_* entries below do the all-gather too)
    pub fn b3_verify_multiple_partial_dev(ctx: *mut b3_ctx, sigs192_dev: *const u8, pks96_dev: *const u8, pk_off_dev: *const u32,
                                          msgs_dev: *const u8, msg_off_dev: *const u32, scalars_dev: *const u64, n: usize, index_base: i64,
                                          partial_dev: *mut u8) -> c_int;
    pub fn b3_verify_multiple_partial(ctx: *mut b3_ctx, sigs192: *const u8, pks96: *const u8, pk_off: *const u32, msgs: *const u8,
                                      msg_off: *const u32, scalars: *const u64, n: usize, index_base: i64, partial_dev: *mut u8) -> c_int;
    pub fn b3_verify_multiple_indexed_partial(ctx: *mut b3_ctx, t: *const b3_keytable, sigs192: *const u8, key_idx: *const u32,
                                              pk_off: *const u32, msgs: *const u8, msg_off: *const u32, scalars: *const u64, n: usize,
                                              index_base: i64, partial_dev: *mut u8) -> c_int;
    pub fn b3_verify_multiple_indexed_partial_dev(ctx: *mut b3_ctx, t: *const b3_keytable, sigs192_dev: *const u8, key_idx_dev: *const u32,
                                                  pk_off_dev: *const u32, msgs_dev: *const u8, msg_off_dev: *const u32,
                                                  scalars_dev: *const u64, n: usize, index_base: i64, partial_dev: *mut u8) -> c_int;
    pub fn b3_combine_partials_dev(ctx: *mut b3_ctx, partials_dev: *const u8, n_partials: usize, accept: *mut c_int, first_bad: *mut i64,
                                   gt576: *mut u8) -> c_int;
    pub fn b3_hash_to_g2_dev(ctx: *mut b3_ctx, msgs_dev: *const u8, off_dev: *const u32, n: usize, out192_dev: *mut u8) -> c_int;
    pub fn b3_g1_aggregate_dev(ctx: *mut b3_ctx, pks96_dev: *const u8, off_dev: *const u32, n_sets: usize, out96_dev: *mut u8,
                               status_dev: *mut i32) -> c_int;
    // ---- multi-GPU with the NCCL all-gather inside the library (M/aggregates.rs:261-316 over the ranks of one box)
    pub fn b3_nccl_unique_id(id128: *mut u8) -> c_int;
    pub fn b3_comm_create(device: c_int, nranks: c_int, rank: c_int, id128: *const u8, lanes: c_int, out: *mut *mut b3_comm) -> c_int;
    pub fn b3_comm_destroy(c: *mut b3_comm);
    pub fn b3_comm_last_error(c: *mut b3_comm) -> *const c_char;
    pub fn b3_comm_collective_count(c: *mut b3_comm) -> u64;
    pub fn b3_sharded_begin(ctx: *mut b3_ctx, c: *mut b3_comm, lane: c_int, table: *const b3_keytable, sigs192: *const u8, keys: *const c_void,
                            pk_off: *const u32, msgs: *const u8, msg_off: *const u32, scalars: *const u64, n: usize, index_base: i64,
                            device_pointers: c_int, ticket: *mut i64) -> c_int;
    pub fn b3_sharded_finish(ctx: *mut b3_ctx, c: *mut b3_comm, lane: c_int, ticket: i64, accept: *mut c_int, first_bad: *mut i64,
                             gt576: *mut u8) -> c_int;
    pub fn b3_verify_multiple_sharded(ctx: *mut b3_ctx, c: *mut b3_comm, lane: c_int, table: *const b3_keytable, sigs192: *const u8,
                                      keys: *const c_void, pk_off: *const u32, msgs: *const u8, msg_off: *const u32, scalars: *const u64,
                                      n: usize, index_base: i64, device_pointers: c_int, accept: *mut c_int, first_bad: *mut i64,
                                      gt576: *mut u8) -> c_int;
    // ---- input synthesis helpers and the roofline probe (tests / benches only)
    pub fn b3_g1_mul_gen(ctx: *mut b3_ctx, scalars32: *const u8, n: usize, out96: *mut u8) -> c_int;
    pub fn b3_g2_mul(ctx: *mut b3_ctx, pts192: *const u8, scalars32: *const u8, n: usize, out192: *mut u8) -> c_int;
    pub fn b3_imad_peak(ctx: *mut b3_ctx, wide: c_int, ops_per_s: *mut f64) -> c_int;
}
