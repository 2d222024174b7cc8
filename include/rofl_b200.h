/* rofl_b200 -- C ABI of the B200-native implementation of RoFL's rofl_crypto client-prove / server-verify hot path.
 *
 * This header is the drop-in boundary (SURVEY.md section 8b): every entry point replaces one function of the
 * reference's Rust API (the surface rofl_service/src/flserver/params.rs links) and, where one exists, the matching
 * `extern "C"` export of rofl_crypto/src/bindings32.rs.  INTEGRATION.md shows the Rust `-sys` binding and the
 * shim that maps these calls back onto the reference's module paths and types.
 *
 * Conventions
 *   - plain pointers and sizes only; points are 32-byte compressed ristretto255 encodings, scalars are 32-byte
 *     little-endian canonical integers mod l, values are IEEE f32, proofs are the reference's byte serialisations
 *     (RangeProof::to_bytes, SquareProof::to_bytes 160 B, SquareProofCommitments 64 B, ElGamalPair 64 B).
 *   - functions without suffix take HOST buffers (the reference-facing calls; copies are inside the call);
 *     `_dev` variants take DEVICE pointers for every array marked [dev] (inputs already resident in HBM).
 *   - the fixed-point configuration the reference selects with cargo features (rofl_crypto/src/fp.rs:35-137) is the
 *     runtime pair (n_bits in {8,16,32,64}, frac in 0..12).
 *   - every nonce the reference draws from rand::thread_rng() is drawn from ChaCha20 streams derived from `seed`
 *     (32 bytes) in the reference's draw order, so outputs are a pure function of (inputs, seed).
 *     SECURITY: a prover seed must be SECRET and FRESH for every call (the nonces are a function of the seed alone: a repeated or
 *     known seed leaks the witness, exactly like a repeated rng state would in the reference).  Fixed seeds are for parity tests only.
 *     A verifier seed should be fresh too, but the verifier does not rely on it: its batching scalars are derived by Fiat-Shamir from
 *     the seed AND every proof / commitment byte of the call, so a known seed does not help a forger (ts_kernels.cuh, k_verify_keys).
 *   - return codes: prove calls return 0 on success; verify calls return 1 (valid) / 0 (invalid, the reference's
 *     Ok(false)); negative values are errors (the reference's Err(..) or panic), positive prove codes are the
 *     reference's domain errors.  rofl_last_error() gives a message for the calling thread.
 *   - there is no CPU fallback: every call needs a CUDA device (sm_100a) and fails with ROFL_ERR_CUDA otherwise.
 */
#ifndef ROFL_B200_H
#define ROFL_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct rofl_ctx rofl_ctx;

enum {
    ROFL_OK = 0,
    ROFL_ERR_VALUE_OUT_OF_RANGE = 2,   /* RangeProofError::ValueOutOfRangeError (range_proof_vec/errors.rs:5-19)          */
    ROFL_ERR_OVERFLOW = 3,             /* L2RangeProofError::OverflowError      (l2_range_proof_vec/errors.rs:4-31)       */
    ROFL_ERR_NORM_OUT_OF_RANGE = 4,    /* L2RangeProofError::NormOutOfRangeError                                         */
    ROFL_ERR_FORMAT = -1,              /* ProofError::FormatError (malformed proof / non-canonical scalar)               */
    ROFL_ERR_ARGS = -2,                /* bad arguments (null / zero sizes / unsupported fixed-point configuration)      */
    ROFL_ERR_GENS = -3,                /* ProofError::InvalidGeneratorsLength                                             */
    ROFL_ERR_POINT = -4,               /* a commitment does not decode (the reference's decompress().unwrap() panics)    */
    ROFL_ERR_DLOG = -5,                /* no discrete log in range (bsgs32.rs:69-70 unwrap panic)                         */
    ROFL_ERR_TOO_MANY = -6,            /* more than 900 000 pairs in a compressed rand proof (the reference's label table ends there) */
    ROFL_ERR_BITSIZE = -7,             /* ProofError::InvalidBitsize (range not in {8,16,32,64}), prove and verify side   */
    ROFL_ERR_UNBALANCED = -8,          /* an accumulated R is not B at extract (params.rs:133-138, el_gamal.rs:101-103)   */
    ROFL_ERR_NAN = -98,                /* NaN input (Fix::saturating_from_float panics)                                   */
    ROFL_ERR_PARTITION = -99,          /* n_partition gives non power-of-two chunks (range_proof_vec/mod.rs:137-140 panic) */
    ROFL_ERR_CUDA = -100               /* CUDA runtime error / no device                                                   */
};

/* process-wide context: device, stream, cached generator tables and BSGS tables (SURVEY.md section 8b "threading").
 * Thread-safe: concurrent callers of one context run on separate lanes (stream sets, up to "max_lanes", further callers wait);
 * the generator / BSGS tables are cached per DEVICE and shared by every context and caller on it (server.rs:54,84 shares one Arc<BSGSTable>). */
int rofl_ctx_create(rofl_ctx **out, int device);
void rofl_ctx_destroy(rofl_ctx *ctx);
const char *rofl_last_error(void);
void rofl_set_host_threads(rofl_ctx *ctx, int n);          /* host threads used for the per-chunk Merlin transcripts */
/* tuning knobs (results never depend on them): "use_rt" 0/1 generator tables, "rt_unfold" unfolded IPP rounds, "groups" chunk
 * groups on separate queues, "tail_np" largest half-size handled by the fused tail kernel (0 = off), "rt_bits" table radix, "rt_per" table-MSM
 * terms per thread, "tail_ncta" thread blocks (one cluster) per chunk in the tail kernel (1, 2, 4, 8), "frozen" 0/1 frozen-level middle rounds,
 * "nt_unfold" / "nt_unfold_min" unfolded rounds without tables, "ts_host_m" chunk size above which commitments are absorbed on the host,
 * "max_lanes" concurrent callers, "drop_tables", "trim" (hand cached scratch back to CUDA), "sigma_rlc_terms" MSM terms per range of the
 * batched rand / square-rand proof check (1 .. 2^24, the default), "crp_batch_terms" MSM terms per client group of the batched compressed-rand-proof
 * check (1 .. 2^24, the default; a group holds at least one client).
 * returns 0, -2 unknown name */
int rofl_set_option(rofl_ctx *ctx, const char *name, long value);

/* ---- sizes ---------------------------------------------------------------------------------------------------- */
size_t rofl_next_pow2(size_t v);                           /* range_proof_vec/mod.rs:237-246                          */
size_t rofl_range_proof_len(size_t n_times_m);             /* 32*(9 + 2 lg(n*m)) : RangeProof::to_bytes length         */
/* number of proofs and bytes per proof create_rangeproof produces for (D, range, n_partition) */
void rofl_range_proof_shape(size_t D, int range, size_t n_partition, size_t *n_proofs, size_t *proof_len);

/* ---- conversion32.rs / range_proof_vec::clip_f32_to_range_vec -------------------------------------------------- */
/* self test of the device field arithmetic (GF(2^255-19), curve25519-dalek-ng FieldElement semantics): n raw 256-bit inputs,
 * out = n x 6 x 32 canonical encodings of a*b, a^2, a+b, a-b, (a+b)(a-b), 1/a */
int rofl_field_selftest(rofl_ctx *, const uint8_t *a32, const uint8_t *b32, size_t n, uint8_t *out);
/* out: n x 96 bytes = a*b mod l for RAW 256-bit a, b | (a mod l)^-1 (division steps) | (a mod l)^-1 (Fermat); 0 for a = 0 */
int rofl_scalar_selftest(rofl_ctx *, const uint8_t *a32, const uint8_t *b32, size_t n, uint8_t *out);
int rofl_f32_to_scalar_vec(rofl_ctx *, const float *v, size_t D, int n_bits, int frac, uint8_t *out_scalars32);       /* conversion32.rs:11-22 */
int rofl_scalar_to_f32_vec(rofl_ctx *, const uint8_t *scalars32, size_t D, int n_bits, int frac, float *out);         /* conversion32.rs:24-38 */
void rofl_clip_bounds(int range, int n_bits, int frac, float *mn, float *mx);                                        /* conversion32.rs:56-60 */
float rofl_l2_clip_bound(int range, int n_bits, int frac);                                                            /* conversion32.rs:62-64 */
void rofl_clip_f32_to_range_vec(const float *v, size_t D, int range, int n_bits, int frac, float *out);              /* range_proof_vec/mod.rs:104-111 (host; O(D) f32 min/max) */
void rofl_rnd_scalar_vec(const uint8_t seed[32], size_t D, uint8_t *out_scalars32);                                  /* pedersen_ops.rs:124-127, seeded   */
/* element-wise scalar arithmetic mod l (host): op 0 = a + b, 1 = -a   (bindings32.rs:727 `add_scalars`, pedersen_ops.rs:110-122 cancelling blindings) */
int rofl_scalar_ops(int op, const uint8_t *a32, const uint8_t *b32, size_t n, uint8_t *out32);

/* ---- commitments: pedersen_ops::commit_vec / commit_no_blinding_vec (pedersen_ops.rs:9-25) and the ElGamal right
 *      halves R = r*B (el_gamal.rs:57-69, compressed_rand_proof/party.rs:23-24).  blind32 may be NULL (zero blinding,
 *      then out_R32 must be NULL); out_R32 may be NULL.  bindings32.rs:118,130 (`commit_no_blinding`, `commit`). */
int rofl_commit(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int n_bits, int frac, uint8_t *out_L32, uint8_t *out_R32);
int rofl_commit_dev(rofl_ctx *, const float *v /*dev*/, const uint8_t *blind32 /*dev*/, size_t D, int n_bits, int frac, uint8_t *out_L32 /*dev*/, uint8_t *out_R32 /*dev*/);

/* ---- range_proof_vec::create_rangeproof (range_proof_vec/mod.rs:16-102; bindings32.rs:228 `create_rangeproof`).
 *      out_proofs: n_proofs*proof_len bytes (see rofl_range_proof_shape), out_commits32: D*32 bytes. */
int rofl_range_prove(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int range, size_t n_partition, int n_bits, int frac,
                     const uint8_t seed[32], uint8_t *out_proofs, size_t *out_proof_len, size_t *out_n_proofs, uint8_t *out_commits32);
int rofl_range_prove_dev(rofl_ctx *, const float *v /*dev*/, const uint8_t *blind32 /*dev*/, size_t D, int range, size_t n_partition, int n_bits, int frac,
                         const uint8_t seed[32], uint8_t *out_proofs /*host*/, size_t *out_proof_len, size_t *out_n_proofs, uint8_t *out_commits32 /*dev*/);
/* ---- range_proof_vec::verify_rangeproof (range_proof_vec/mod.rs:149-191; bindings32.rs:265 `verify_rangeproof`).
 *      seed feeds the verifier's random batching scalar (RangeProof::verify_multiple draws it from thread_rng). */
int rofl_range_verify(rofl_ctx *, const uint8_t *proofs, size_t proof_len, size_t n_proofs, const uint8_t *commits32, size_t D, int range, const uint8_t seed[32]);
int rofl_range_verify_dev(rofl_ctx *, const uint8_t *proofs /*host*/, size_t proof_len, size_t n_proofs, const uint8_t *commits32 /*dev*/, size_t D, int range, const uint8_t seed[32]);

/* ---- l2_range_proof_vec::{create_rangeproof_l2, verify_rangeproof_l2} (l2_range_proof_vec/mod.rs:15-140,185-228;
 *      bindings32.rs:441,507).  out_proof: rofl_range_proof_len(range) bytes; out_commit32: 32 bytes (not shifted). */
/* chunk-sharded range proofs for multi-GPU (one update, chunk c -> GPU c mod G; range_proof_vec/mod.rs:54-78 makes the chunks
 * independent proofs).  The caller passes the slice of chunks [chunk_begin, chunk_begin + n_chunks) of chunk length chunk_len
 * (= next_pow2(D) / min(next_pow2(D), n_partition)); D_shard = real elements in the slice (the rest is the reference's zero padding).
 * The proofs / commitments are byte-identical to the corresponding rows of the whole-update call. */
int rofl_range_prove_shard(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D_shard, size_t chunk_len, size_t chunk_begin, size_t n_chunks, int range,
                           int n_bits, int frac, const uint8_t seed[32], uint8_t *out_proofs, size_t *out_proof_len, uint8_t *out_commits32);
int rofl_range_verify_shard(rofl_ctx *, const uint8_t *proofs, size_t proof_len, size_t n_chunks, const uint8_t *commits32, size_t D_shard, size_t chunk_len, size_t chunk_begin,
                            int range, const uint8_t seed[32]);
int rofl_l2_prove(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int range, int n_bits, int frac, const uint8_t seed[32],
                  uint8_t *out_proof, size_t *out_proof_len, uint8_t *out_commit32);
int rofl_l2_verify(rofl_ctx *, const uint8_t *proof, size_t proof_len, const uint8_t commit32[32], int range, const uint8_t seed[32]);

/* ---- square_proof_vec::{create_l2rangeproof_vec_existing, verify_l2rangeproof_vec} (square_proof_vec/mod.rs:19-75,130-160).
 *      value_com32: D commitments c_l; r1/r2: D blindings each; out_proofs: D*160; out_commits: D*64 (c_l | c_sq). */
/* compressed_rand_proof::CompressedRandProof::{helper_prove, helper_prove_existing, helper_verify} (compressed_rand_proof/mod.rs:134-158):
 * ONE sigma proof that all D ElGamal pairs (L_i, R_i) = (m_i B + r_i H, r_i B) are well formed; also the call that materialises the
 * R halves (party.rs:23-24,55-56).  value_com32 = the existing L_i (prove_existing) or NULL (L_i = commit(m_i, r_i)).
 * proof128 = C'_L | C'_R | z_m | z_r (mod.rs:108-114), pairs64 = D x (L | R) (el_gamal.rs:105-111).
 * prove: 0 ok, ROFL_ERR_POINT, -6 more than 900 000 pairs (the reference's label table ends there: it panics), ROFL_ERR_NAN.
 * verify: 1 valid, 0 invalid, ROFL_ERR_FORMAT, -6. */
int rofl_crp_prove(rofl_ctx *, const float *v, const uint8_t *value_com32, const uint8_t *blind32, size_t D, int n_bits, int frac, const uint8_t seed[32],
                   uint8_t *out_proof128, uint8_t *out_pairs64);
int rofl_crp_verify(rofl_ctx *, const uint8_t *proof128, const uint8_t *pairs64, size_t D);
/* The un-optimised encodings' per-element proofs (enc types 2 and 3, params.rs:468-511,608-646):
 *   rand_proof_vec::{create_randproof_vec, create_randproof_vec_existing, verify_randproof_vec}  (rand_proof_vec/mod.rs:14-118): RandProof = 128 B
 *       (C'_L | C'_R | z_m | z_r, rand_proof/mod.rs:87-97) over 64-byte ElGamal pairs;
 *   square_rand_proof_vec::{create_l2rangeproof_vec, create_l2rangeproof_vec_existing, verify_l2rangeproof_vec} (square_rand_proof_vec/mod.rs:18-160):
 *       SquareRandProof = 192 B over SquareRandProofCommitments = 96 B (c.L | c.R | c_sq).
 * value_com32 = existing Pedersen commitments (the *_existing variants) or NULL.  prove: 0 ok, ROFL_ERR_POINT, ROFL_ERR_NAN; verify: 1 / 0 / ROFL_ERR_FORMAT. */
int rofl_rand_prove(rofl_ctx *, const float *v, const uint8_t *value_com32, const uint8_t *blind32, size_t D, int n_bits, int frac, const uint8_t seed[32],
                    uint8_t *out_proofs128, uint8_t *out_pairs64);
int rofl_rand_verify(rofl_ctx *, const uint8_t *proofs128, const uint8_t *pairs64, size_t D);
int rofl_square_rand_prove(rofl_ctx *, const float *v, const uint8_t *value_com32, const uint8_t *r1_32, const uint8_t *r2_32, size_t D, int n_bits, int frac,
                           const uint8_t seed[32], uint8_t *out_proofs192, uint8_t *out_commits96);
int rofl_square_rand_verify(rofl_ctx *, const uint8_t *proofs192, const uint8_t *commits96, size_t D);
/* The two optimised encodings of rofl_service end to end, on the wire fields of flservice.proto (the protobuf framing stays on the Rust side):
 *   EncParamsRangeCompressed::{encrypt, verify}  (params.rs:699-743, 236-256)   enc_values = D x 64 (L | R), rand_proof 128 B, range_proof[]
 *   EncParamsL2Compressed::{encrypt, verify}     (params.rs:797-845, 257-290)   enc_values = D x 96 (L | R | c_sq), square_proof D x 160,
 *                                                                               rand_proof 128 B, range_proof[], square_range_proof
 * encrypt: 0 ok or the error of the failing step; verify: 1 accept, 0 reject (an Err of any part is a reject in the reference too), < 0 bad arguments.
 * The deserialisation checks of the reference (`from_bytes`: points decode, scalars canonical) happen on the GPU inside the verify calls;
 * rofl_enc_l2_compressed_verify returns ROFL_ERR_POINT when ANY of the three points of a 96-byte record does not decode -- c.R included, which
 * that arm never uses afterwards (decode_l2enc_vec, params.rs:560-571 -> SquareRandProofCommitments::from_bytes, square_rand_proof/pedersen.rs:33-45
 * -> ElGamalPair::from_bytes, rand_proof/el_gamal.rs:112-123; the reference unwrap()s, i.e. one client's malformed message panics the server task). */
int rofl_enc_range_compressed_encrypt(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int prove_range, size_t n_partition, int n_bits, int frac,
                                      const uint8_t seed[32], uint8_t *out_enc_values64, uint8_t *out_rand_proof128, uint8_t *out_range_proofs, size_t *out_proof_len, size_t *out_n_proofs);
int rofl_enc_range_compressed_verify(rofl_ctx *, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proof128, const uint8_t *range_proofs, size_t proof_len,
                                     size_t n_proofs, int prove_range, float check_percentage, const uint8_t seed[32]);
int rofl_enc_l2_compressed_encrypt(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int prove_range, size_t n_partition, int l2_range, int n_bits, int frac,
                                   const uint8_t seed[32], uint8_t *out_enc_values96, uint8_t *out_square_proofs160, uint8_t *out_rand_proof128, uint8_t *out_range_proofs,
                                   size_t *out_proof_len, size_t *out_n_proofs, uint8_t *out_square_range_proof, size_t *out_sq_proof_len);
int rofl_enc_l2_compressed_verify(rofl_ctx *, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs160, const uint8_t *range_proofs, size_t proof_len,
                                  size_t n_proofs, const uint8_t *square_range_proof, size_t sq_proof_len, int prove_range, int l2_range, const uint8_t seed[32]);
/* The two un-optimised encodings end to end (same conventions as above):
 *   EncParamsRange::{encrypt, verify}  (params.rs:467-510, 186-203)   enc_values = D x 64, rand_proofs = D x 128 (one RandProof per element, over the UNCLIPPED
 *                                       plaintext as in the reference), range proofs over the first round(D * check_percentage) elements (all when >= 1)
 *   EncParamsL2::{encrypt, verify}     (params.rs:607-646, 205-233)   enc_values = D x 96, square_proofs = D x 192 (SquareRandProof), range_proof[], square_range_proof */
int rofl_enc_range_encrypt(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int prove_range, size_t n_partition, float check_percentage, int n_bits, int frac,
                           const uint8_t seed[32], uint8_t *out_enc_values64, uint8_t *out_rand_proofs128, uint8_t *out_range_proofs, size_t *out_proof_len, size_t *out_n_proofs);
int rofl_enc_range_verify(rofl_ctx *, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proofs128, const uint8_t *range_proofs, size_t proof_len, size_t n_proofs,
                          int prove_range, float check_percentage, const uint8_t seed[32]);
int rofl_enc_l2_encrypt(rofl_ctx *, const float *v, const uint8_t *blind32, size_t D, int prove_range, size_t n_partition, int l2_range, int n_bits, int frac,
                        const uint8_t seed[32], uint8_t *out_enc_values96, uint8_t *out_square_proofs192, uint8_t *out_range_proofs, size_t *out_proof_len, size_t *out_n_proofs,
                        uint8_t *out_square_range_proof, size_t *out_sq_proof_len);
int rofl_enc_l2_verify(rofl_ctx *, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs192, const uint8_t *range_proofs, size_t proof_len, size_t n_proofs,
                       const uint8_t *square_range_proof, size_t sq_proof_len, int prove_range, int l2_range, const uint8_t seed[32]);
int rofl_square_prove(rofl_ctx *, const float *v, const uint8_t *value_com32, const uint8_t *r1_32, const uint8_t *r2_32, size_t D, int n_bits, int frac,
                      const uint8_t seed[32], uint8_t *out_proofs160, uint8_t *out_commits64);
int rofl_square_prove_dev(rofl_ctx *, const float *v, const uint8_t *value_com32, const uint8_t *r1_32, const uint8_t *r2_32, size_t D, int n_bits, int frac,
                          const uint8_t seed[32], uint8_t *out_proofs160, uint8_t *out_commits64);     /* all arrays [dev] */
int rofl_square_verify(rofl_ctx *, const uint8_t *proofs160, const uint8_t *commits64, size_t D);
int rofl_square_verify_dev(rofl_ctx *, const uint8_t *proofs160 /*dev*/, const uint8_t *commits64 /*dev*/, size_t D);

/* ---- server side, all clients of a round at once.  rofl_service fans EncModelParams::verify out over a rayon pool, one task per client
 *      (server.rs:516-522,666-667 -> params.rs:181-291); here the n_clients updates of one round (same D, range and partition) share ONE
 *      batched check: one random linear combination over all clients x chunks, one generator MSM, one bucket MSM over all commitments.
 *      Arrays are client-major (proofs: n_clients x n_proofs x proof_len; commits32: n_clients x D x 32; ...).
 *      out_ok[k] = 1 valid, 0 invalid, < 0 the error of that client's update; if the combined check fails the clients are re-checked one by one,
 *      so the result names the offending client exactly like the reference's per-client verdicts.  Return value: 0, or < 0 for bad arguments. */
int rofl_range_verify_batch(rofl_ctx *, const uint8_t *proofs, size_t proof_len, size_t n_proofs, const uint8_t *commits32, size_t D, size_t n_clients, int range,
                            const uint8_t seed[32], int *out_ok);
int rofl_enc_l2_compressed_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs160, const uint8_t *range_proofs,
                                        size_t proof_len, size_t n_proofs, const uint8_t *square_range_proofs, size_t sq_proof_len, int prove_range, int l2_range,
                                        const uint8_t seed[32], int *out_ok);
/* K compressed rand proofs (helper_verify, compressed_rand_proof/mod.rs:149-158) in one batched check.  proofs128: n_clients x 128,
 * pairs64: n_clients x D x 64.  out_ok[k] = exactly what rofl_crp_verify(proofs128[k], pairs64[k], D) returns: 1, 0, ROFL_ERR_FORMAT, -6.
 * Return value: 0, or < 0 for bad arguments. */
int rofl_crp_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *proofs128, const uint8_t *pairs64, size_t D, const uint8_t seed[32], int *out_ok);
/* EncModelParams::verify, EncRangeCompressed arm (params.rs:236-256), for n_clients messages of one shape: enc_values64 n_clients x D x 64,
 * rand_proofs128 n_clients x 128, range_proofs n_clients x n_proofs x proof_len.  out_ok[k] = exactly what rofl_enc_range_compressed_verify(message k,
 * check_percentage, seed) returns (1 / 0).  Return value: 0, or ROFL_ERR_ARGS (D == 0, n_proofs == 0, null out_ok). */
int rofl_enc_range_compressed_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proofs128, const uint8_t *range_proofs,
                                           size_t proof_len, size_t n_proofs, int prove_range, float check_percentage, const uint8_t seed[32], int *out_ok);
/* K x D rand proofs (rand_proof_vec::verify_randproof_vec) / square-rand proofs (square_rand_proof_vec::verify_l2rangeproof_vec) in one batched
 * check.  proofs128 / proofs192: n_clients x D x 128 | 192, pairs64 / commits96: n_clients x D x 64 | 96.  out_ok[k] = exactly what
 * rofl_rand_verify / rofl_square_rand_verify(proofs k, commits k, D) returns: 1, 0, ROFL_ERR_FORMAT (D == 0: 1 for every client).
 * Return value: 0, or ROFL_ERR_ARGS (null out_ok, null buffers). */
int rofl_rand_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *proofs128, const uint8_t *pairs64, size_t D, const uint8_t seed[32], int *out_ok);
int rofl_square_rand_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *proofs192, const uint8_t *commits96, size_t D, const uint8_t seed[32], int *out_ok);
/* EncModelParams::verify, EncRange arm (params.rs:186-203), for n_clients messages of one shape: enc_values64 n_clients x D x 64,
 * rand_proofs128 n_clients x D x 128, range_proofs n_clients x n_proofs x proof_len.  out_ok[k] = exactly what rofl_enc_range_verify(message k,
 * check_percentage, seed) returns (1 / 0).  Return value: 0, or ROFL_ERR_ARGS (D == 0, n_proofs == 0, null out_ok). */
int rofl_enc_range_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proofs128, const uint8_t *range_proofs,
                                size_t proof_len, size_t n_proofs, int prove_range, float check_percentage, const uint8_t seed[32], int *out_ok);
/* EncModelParams::verify, EncL2 arm (params.rs:205-233), for n_clients messages of one shape: enc_values96 n_clients x D x 96, square_proofs192
 * n_clients x D x 192, range_proofs n_clients x n_proofs x proof_len, square_range_proofs n_clients x sq_proof_len.  out_ok[k] = exactly what
 * rofl_enc_l2_verify(message k, ..., seed) returns (1 / 0).  Return value: 0, or ROFL_ERR_ARGS (D == 0, n_proofs == 0, null out_ok). */
int rofl_enc_l2_verify_batch(rofl_ctx *, size_t n_clients, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs192, const uint8_t *range_proofs,
                             size_t proof_len, size_t n_proofs, const uint8_t *square_range_proofs, size_t sq_proof_len, int prove_range, int l2_range,
                             const uint8_t seed[32], int *out_ok);

/* ---- aggregation: EncModelParamsAccumulator::accumulate_other (params.rs:81-124) / pedersen_ops::add_rp_vec_vec
 *      (pedersen_ops.rs:56-69; bindings32.rs:64 `add_commitments`).  points32: n_clients x D encodings, client-major.
 *      init_unity = 1 starts every element at the basepoint (ElGamalPair::unity, el_gamal.rs:83-88), 0 at the identity. */
int rofl_aggregate(rofl_ctx *, const uint8_t *points32, size_t n_clients, size_t D, int init_unity, uint8_t *out32);
int rofl_aggregate_dev(rofl_ctx *, const uint8_t *points32 /*dev*/, size_t n_clients, size_t D, int init_unity, uint8_t *out32 /*dev*/);

/* ---- decryption: pedersen_ops::discrete_log_vec_table + BSGSTable (pedersen_ops.rs:47-53, bsgs32.rs:20-73;
 *      bindings32.rs:213 `extract_values`).  table_size = BSGSTable::new(m); bsgs_bits = width of BSGS_URawFix
 *      (8 for fp8, else 16).  out_scalars32 / out_f32 may be NULL.  The table is built once per (table_size, bsgs_bits). */
int rofl_dlog(rofl_ctx *, const uint8_t *points32, size_t D, uint64_t table_size, int bsgs_bits, int n_bits, int frac, uint8_t *out_scalars32, float *out_f32);
int rofl_dlog_dev(rofl_ctx *, const uint8_t *points32 /*dev*/, size_t D, uint64_t table_size, int bsgs_bits, int n_bits, int frac, uint8_t *out_scalars32 /*dev*/, float *out_f32 /*dev*/);

/* ---- round accumulator: EncModelParamsAccumulator (params.rs:74-148) on the device, for D elements.  Clients are added as they arrive
 *      (accumulate_other, params.rs:81-124); the accumulated points stay in HBM between calls, O(D) state whatever the number of clients.
 *   rec_bytes 32: Pedersen commitments (L only; pedersen_ops::add_rp_vec_vec, pedersen_ops.rs:56-69)
 *             64: ElGamal pairs L | R (EncRange / EncRangeCompressed enc_values)
 *             96: L | R | c_sq (EncL2 / EncL2Compressed enc_values): c_sq must decode, it is not accumulated
 *   init_unity 1: every element starts at ElGamalPair::unity = (B, B) (params.rs:165-179, el_gamal.rs:83-88); 0: at the identity.
 * The state (two extended points per element, one for rec_bytes 32: 256 B / 128 B) is allocated at create and never enters the scratch cache.
 * The accumulator keeps a pointer to its context: the context must outlive it.  Calls on one accumulator from several threads are serialised
 * by the accumulator's own mutex.  Group addition is commutative and export writes canonical encodings, so no result depends on the order
 * of the adds or on how the clients are split over calls.  Return values: 0 / counts as stated, ROFL_ERR_ARGS for bad arguments. */
typedef struct rofl_acc rofl_acc;
int rofl_acc_create(rofl_ctx *, size_t D, int rec_bytes, int init_unity, rofl_acc **out);
void rofl_acc_destroy(rofl_acc *);
int rofl_acc_reset(rofl_acc *);                 /* back to the initial state, count 0, memory kept (the next round) */
/* records: n_clients x D x rec_bytes, client-major.  mask (nullable): add client k only where mask[k] == 1 (the out_ok of a *_verify_batch call
 * can be passed as it is).  out_added (nullable): per client 1 added, 0 skipped by the mask, ROFL_ERR_POINT a point of its record does not decode
 * (then nothing of that client is added: the reference's from_bytes fails before accumulate).  Returns the number of clients added, or < 0. */
int rofl_acc_add(rofl_acc *, const uint8_t *records, size_t n_clients, const int *mask, int *out_added);
int rofl_acc_add_dev(rofl_acc *, const uint8_t *records /*dev*/, size_t n_clients, const int *mask /*host*/, int *out_added /*host*/);
size_t rofl_acc_count(const rofl_acc *);        /* clients added since create / reset */
/* the accumulated values, compressed: D x 32 (rec_bytes 32) or D x 64 (L | R) */
int rofl_acc_export(rofl_acc *, uint8_t *out);
/* EncModelParamsAccumulator::extract (params.rs:126-147): first every accumulated R must equal B (Ristretto equality; not checked for rec_bytes 32),
 * else ROFL_ERR_UNBALANCED and nothing is written; then BSGS on L exactly as rofl_dlog(table_size, bsgs_bits, n_bits, frac): ROFL_ERR_DLOG when
 * an element has no log in range (the reference's unwrap panic).  out_scalars32 (D x 32) / out_f32 (D) nullable.  The accumulator is not changed. */
int rofl_acc_extract(rofl_acc *, uint64_t table_size, int bsgs_bits, int n_bits, int frac, uint8_t *out_scalars32, float *out_f32);

/* ---- measurement hooks (bench.py): CUDA-event time per kernel family and launch counts since the last reset ------- */
enum { ROFL_PROF_FOLD = 0, ROFL_PROF_MSM = 1, ROFL_PROF_COMMIT = 2, ROFL_PROF_SQUARE = 3 };
void rofl_prof_enable(int on);
void rofl_prof_reset(void);
double rofl_prof_ms(int slot);            /* summed device time of that kernel family, milliseconds */
long rofl_prof_launches(int slot);        /* launches of that family; slot -1 = all kernels launched by the library */
double rofl_prof_work(int slot);          /* algorithmic work of that family since the last reset (slot 4, table MSM: mixed point additions) */
double rofl_probe_imad_wide(rofl_ctx *);  /* measured IMAD.WIDE.U32 issue rate of this GPU, multiply-adds per second (roofline denominator) */
void *rofl_ctx_stream(rofl_ctx *);        /* the cudaStream_t the context launches on */
/* ---- test hooks: the warp-cooperative transcript absorb against the sequential code (0 equal / 1 different), and the Fiat-Shamir batching
 *      scalars (c_i | rho_i, 2 x n_proofs x 32 bytes) rofl_range_verify derives for a call (return value as rofl_range_verify) */
int rofl_debug_ts_absorb(rofl_ctx *, const uint8_t *V32, size_t m, int n, int label_id);
int rofl_debug_square_rlc(rofl_ctx *, const uint8_t *proofs160, const uint8_t *commits64, size_t D);   /* the batched square-proof check alone: 1 holds, 0 does not */
/* the batched compressed-rand-proof check of rofl_crp_verify_batch alone: 1 = the combination over all n_clients proofs held and none is malformed, 0 = it did not */
int rofl_debug_crp_rlc(rofl_ctx *, size_t n_clients, const uint8_t *proofs128, const uint8_t *pairs64, size_t D, const uint8_t seed[32]);
/* the batched check of rofl_rand_verify_batch (kind 1) / rofl_square_rand_verify_batch (kind 2) alone, over n_elems elements of one update and at any
 * size: 1 = the combination over all elements held and none is malformed, 0 = it did not */
int rofl_debug_sigma_rlc(rofl_ctx *, int kind, size_t n_elems, const uint8_t *proofs, const uint8_t *commits, const uint8_t seed[32]);
int rofl_debug_verify_weights(rofl_ctx *, const uint8_t *proofs, size_t proof_len, size_t n_proofs, const uint8_t *commits32, size_t D, int range, const uint8_t seed[32], uint8_t *out_weights);
/* the terms of one batched check as its production code computed them (nothing is derived by the hook).  family 0: square proofs (proofs
 * n_clients x D x 160, commits x 64); 1: rand proofs (x 128, x 64); 2: square-rand proofs (x 192, x 96) -- families 0-2 also below the size thresholds of
 * the public calls; 3: compressed rand proofs (proofs n_clients x 128, commits = the pairs n_clients x D x 64, D <= 900 000).
 *   root32: the digest the weights are keyed from; chal32: the challenge of every element (families 0-2, n_clients x D) or client (3, n_clients);
 *   ranges: per range of elements (client group for family 3) 8 int64: i0, n, MSM window width c, weight bits wbits (0 for family 3: 128-bit rho_k),
 *     is_id of output 0 and 1 (-1: no such output), index of its first scalar in scalars32, index of its first flag in bad;
 *   scalars32: the MSM scalars of every range in term order; coef32: per range sB[0], sB[1], sH[0], sH[1] as given to k_finalize (zero where unused);
 *   bad: per range, the bad flags of the clients it touches;
 *   verdicts: per client, what the public batch call returns for it (1 / 0 / -1; family 3 as rofl_crp_verify).
 *   cap / cnt: capacities of ranges, scalars32, bad, and what the call produced.
 * returns 1 = every range's combination held and nothing was malformed, 0 = not, ROFL_ERR_ARGS (also when a capacity is short: cnt tells the need) */
int rofl_debug_rlc_terms(rofl_ctx *, int family, size_t n_clients, size_t D, const uint8_t *proofs, const uint8_t *commits, const uint8_t seed[32],
                         uint8_t *root32, uint8_t *chal32, int64_t *ranges, uint8_t *scalars32, uint8_t *coef32, int *bad, int *verdicts,
                         const size_t cap[3], size_t cnt[3]);
/* the MSM front end alone (production plan / forced window width / generator tables, then k_finalize): out32[k] = sum_t s[k][t] P_t + sB[k] B + sH[k] H.
 * scalars32: n_msm x T canonical scalars; points32: T shared or n_msm x T (points_per_msm) encodings, or NULL for BulletproofGens(gen_n, T / (2 gen_n));
 * path 0 = msm_plan_for(T, n_msm, big_min), 1 = window width c with `knob` slices (c <= 8) / parts (c >= 9), 2 = generator tables.  sB32 / sH32 may be NULL.
 * info (nullable, 3 ints): width, slices / parts / blocks, kernel (0 k_msm, 1 k_bm_*, 2 k_rt_msm).  0 ok, ROFL_ERR_ARGS (non-canonical scalar), ROFL_ERR_POINT */
int rofl_debug_msm(rofl_ctx *, const uint8_t *scalars32, size_t n_msm, size_t T, const uint8_t *points32, int points_per_msm, int gen_n,
                   int path, int c, int knob, size_t big_min, const uint8_t *sB32, const uint8_t *sH32, uint8_t *out32, int *info);
#ifdef __cplusplus
}
#endif
#endif
