//! Raw declarations of the C ABI in `include/rofl_b200.h` (kept in the order of the header; no bindgen needed: plain pointers and sizes).
#![allow(non_camel_case_types)]
use libc::{c_char, c_float, c_int, c_long, c_void, size_t};

#[repr(C)]
pub struct rofl_ctx { _private: [u8; 0] }
/// device-resident round accumulator (`rofl_acc_*`); the context it was created on must outlive it
#[repr(C)]
pub struct rofl_acc { _private: [u8; 0] }

pub const ROFL_OK: c_int = 0;
pub const ROFL_ERR_VALUE_OUT_OF_RANGE: c_int = 2;
pub const ROFL_ERR_OVERFLOW: c_int = 3;
pub const ROFL_ERR_NORM_OUT_OF_RANGE: c_int = 4;
pub const ROFL_ERR_FORMAT: c_int = -1;
pub const ROFL_ERR_ARGS: c_int = -2;
pub const ROFL_ERR_GENS: c_int = -3;
pub const ROFL_ERR_POINT: c_int = -4;
pub const ROFL_ERR_DLOG: c_int = -5;
pub const ROFL_ERR_TOO_MANY: c_int = -6;
pub const ROFL_ERR_BITSIZE: c_int = -7;
pub const ROFL_ERR_UNBALANCED: c_int = -8;
pub const ROFL_ERR_NAN: c_int = -98;
pub const ROFL_ERR_PARTITION: c_int = -99;
pub const ROFL_ERR_CUDA: c_int = -100;

extern "C" {
    pub fn rofl_ctx_create(out: *mut *mut rofl_ctx, device: c_int) -> c_int;
    pub fn rofl_ctx_destroy(ctx: *mut rofl_ctx);
    pub fn rofl_last_error() -> *const c_char;
    pub fn rofl_set_host_threads(ctx: *mut rofl_ctx, n: c_int);
    pub fn rofl_set_option(ctx: *mut rofl_ctx, name: *const c_char, value: c_long) -> c_int;
    pub fn rofl_next_pow2(v: size_t) -> size_t;
    pub fn rofl_range_proof_len(n_times_m: size_t) -> size_t;
    pub fn rofl_range_proof_shape(d: size_t, range: c_int, n_partition: size_t, n_proofs: *mut size_t, proof_len: *mut size_t);
    pub fn rofl_f32_to_scalar_vec(ctx: *mut rofl_ctx, v: *const c_float, d: size_t, n_bits: c_int, frac: c_int, out32: *mut u8) -> c_int;
    pub fn rofl_scalar_to_f32_vec(ctx: *mut rofl_ctx, scalars32: *const u8, d: size_t, n_bits: c_int, frac: c_int, out: *mut c_float) -> c_int;
    pub fn rofl_clip_bounds(range: c_int, n_bits: c_int, frac: c_int, mn: *mut c_float, mx: *mut c_float);
    pub fn rofl_l2_clip_bound(range: c_int, n_bits: c_int, frac: c_int) -> c_float;
    pub fn rofl_clip_f32_to_range_vec(v: *const c_float, d: size_t, range: c_int, n_bits: c_int, frac: c_int, out: *mut c_float);
    pub fn rofl_rnd_scalar_vec(seed32: *const u8, d: size_t, out32: *mut u8);
    pub fn rofl_scalar_ops(op: c_int, a32: *const u8, b32: *const u8, n: size_t, out32: *mut u8) -> c_int;
    pub fn rofl_commit(ctx: *mut rofl_ctx, v: *const c_float, blind32: *const u8, d: size_t, n_bits: c_int, frac: c_int, out_l32: *mut u8, out_r32: *mut u8) -> c_int;
    pub fn rofl_range_prove(ctx: *mut rofl_ctx, v: *const c_float, blind32: *const u8, d: size_t, range: c_int, n_partition: size_t, n_bits: c_int, frac: c_int,
                            seed32: *const u8, out_proofs: *mut u8, out_proof_len: *mut size_t, out_n_proofs: *mut size_t, out_commits32: *mut u8) -> c_int;
    pub fn rofl_range_verify(ctx: *mut rofl_ctx, proofs: *const u8, proof_len: size_t, n_proofs: size_t, commits32: *const u8, d: size_t, range: c_int, seed32: *const u8) -> c_int;
    pub fn rofl_range_prove_shard(ctx: *mut rofl_ctx, v: *const c_float, blind32: *const u8, d_shard: size_t, chunk_len: size_t, chunk_begin: size_t, n_chunks: size_t, range: c_int,
                                  n_bits: c_int, frac: c_int, seed32: *const u8, out_proofs: *mut u8, out_proof_len: *mut size_t, out_commits32: *mut u8) -> c_int;
    pub fn rofl_range_verify_shard(ctx: *mut rofl_ctx, proofs: *const u8, proof_len: size_t, n_chunks: size_t, commits32: *const u8, d_shard: size_t, chunk_len: size_t,
                                   chunk_begin: size_t, range: c_int, seed32: *const u8) -> c_int;
    pub fn rofl_range_verify_batch(ctx: *mut rofl_ctx, proofs: *const u8, proof_len: size_t, n_proofs: size_t, commits32: *const u8, d: size_t, n_clients: size_t, range: c_int,
                                   seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_l2_prove(ctx: *mut rofl_ctx, v: *const c_float, blind32: *const u8, d: size_t, range: c_int, n_bits: c_int, frac: c_int, seed32: *const u8,
                         out_proof: *mut u8, out_proof_len: *mut size_t, out_commit32: *mut u8) -> c_int;
    pub fn rofl_l2_verify(ctx: *mut rofl_ctx, proof: *const u8, proof_len: size_t, commit32: *const u8, range: c_int, seed32: *const u8) -> c_int;
    pub fn rofl_square_prove(ctx: *mut rofl_ctx, v: *const c_float, value_com32: *const u8, r1_32: *const u8, r2_32: *const u8, d: size_t, n_bits: c_int, frac: c_int,
                             seed32: *const u8, out_proofs160: *mut u8, out_commits64: *mut u8) -> c_int;
    pub fn rofl_square_verify(ctx: *mut rofl_ctx, proofs160: *const u8, commits64: *const u8, d: size_t) -> c_int;
    pub fn rofl_crp_prove(ctx: *mut rofl_ctx, v: *const c_float, value_com32: *const u8, blind32: *const u8, d: size_t, n_bits: c_int, frac: c_int, seed32: *const u8,
                          out_proof128: *mut u8, out_pairs64: *mut u8) -> c_int;
    pub fn rofl_crp_verify(ctx: *mut rofl_ctx, proof128: *const u8, pairs64: *const u8, d: size_t) -> c_int;
    pub fn rofl_crp_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, proofs128: *const u8, pairs64: *const u8, d: size_t, seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_rand_prove(ctx: *mut rofl_ctx, v: *const c_float, value_com32: *const u8, blind32: *const u8, d: size_t, n_bits: c_int, frac: c_int, seed32: *const u8,
                           out_proofs128: *mut u8, out_pairs64: *mut u8) -> c_int;
    pub fn rofl_rand_verify(ctx: *mut rofl_ctx, proofs128: *const u8, pairs64: *const u8, d: size_t) -> c_int;
    pub fn rofl_square_rand_prove(ctx: *mut rofl_ctx, v: *const c_float, value_com32: *const u8, r1_32: *const u8, r2_32: *const u8, d: size_t, n_bits: c_int, frac: c_int,
                                  seed32: *const u8, out_proofs192: *mut u8, out_commits96: *mut u8) -> c_int;
    pub fn rofl_square_rand_verify(ctx: *mut rofl_ctx, proofs192: *const u8, commits96: *const u8, d: size_t) -> c_int;
    pub fn rofl_enc_l2_compressed_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, enc_values96: *const u8, d: size_t, square_proofs160: *const u8, range_proofs: *const u8,
                                               proof_len: size_t, n_proofs: size_t, square_range_proofs: *const u8, sq_proof_len: size_t, prove_range: c_int, l2_range: c_int,
                                               seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_enc_range_compressed_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, enc_values64: *const u8, d: size_t, rand_proofs128: *const u8, range_proofs: *const u8,
                                                  proof_len: size_t, n_proofs: size_t, prove_range: c_int, check_percentage: c_float, seed32: *const u8,
                                                  out_ok: *mut c_int) -> c_int;
    pub fn rofl_rand_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, proofs128: *const u8, pairs64: *const u8, d: size_t, seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_square_rand_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, proofs192: *const u8, commits96: *const u8, d: size_t, seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_enc_range_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, enc_values64: *const u8, d: size_t, rand_proofs128: *const u8, range_proofs: *const u8,
                                       proof_len: size_t, n_proofs: size_t, prove_range: c_int, check_percentage: c_float, seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_enc_l2_verify_batch(ctx: *mut rofl_ctx, n_clients: size_t, enc_values96: *const u8, d: size_t, square_proofs192: *const u8, range_proofs: *const u8,
                                    proof_len: size_t, n_proofs: size_t, square_range_proofs: *const u8, sq_proof_len: size_t, prove_range: c_int, l2_range: c_int,
                                    seed32: *const u8, out_ok: *mut c_int) -> c_int;
    pub fn rofl_aggregate(ctx: *mut rofl_ctx, points32: *const u8, n_clients: size_t, d: size_t, init_unity: c_int, out32: *mut u8) -> c_int;
    pub fn rofl_dlog(ctx: *mut rofl_ctx, points32: *const u8, d: size_t, table_size: u64, bsgs_bits: c_int, n_bits: c_int, frac: c_int, out_scalars32: *mut u8, out_f32: *mut c_float) -> c_int;
    pub fn rofl_acc_create(ctx: *mut rofl_ctx, d: size_t, rec_bytes: c_int, init_unity: c_int, out: *mut *mut rofl_acc) -> c_int;
    pub fn rofl_acc_destroy(acc: *mut rofl_acc);
    pub fn rofl_acc_reset(acc: *mut rofl_acc) -> c_int;
    pub fn rofl_acc_add(acc: *mut rofl_acc, records: *const u8, n_clients: size_t, mask: *const c_int, out_added: *mut c_int) -> c_int;
    pub fn rofl_acc_add_dev(acc: *mut rofl_acc, records_dev: *const u8, n_clients: size_t, mask: *const c_int, out_added: *mut c_int) -> c_int;
    pub fn rofl_acc_count(acc: *const rofl_acc) -> size_t;
    pub fn rofl_acc_export(acc: *mut rofl_acc, out: *mut u8) -> c_int;
    pub fn rofl_acc_extract(acc: *mut rofl_acc, table_size: u64, bsgs_bits: c_int, n_bits: c_int, frac: c_int, out_scalars32: *mut u8, out_f32: *mut c_float) -> c_int;
    pub fn rofl_ctx_stream(ctx: *mut rofl_ctx) -> *mut c_void;
}
