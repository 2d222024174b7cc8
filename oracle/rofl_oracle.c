/* ORACLE -- TEST INFRASTRUCTURE ONLY.  CPU restatement of the rofl_crypto hot path (SURVEY.md section 8a),
 * exported as a flat C ABI for ctypes.  Never linked into the product; only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it (as checker / reported baseline).
 *
 * Each function cites the reference file:line it restates (paths relative to /root/reference/rofl_crypto/src).
 * The fixed-point configuration that the reference selects with cargo features (fp.rs:35-137) is a runtime
 * (n_bits, frac) pair here.  Randomness: every nonce the reference draws from rand::thread_rng() is drawn
 * from a ChaCha20 stream keyed by derive_key(seed, domain, index) in the reference's draw order (bp.h).
 *
 * PARITY: proof / commitment bytes are UNPINNED against the real Rust crate (no golden vectors exist in the
 * reference and cargo is absent here).  Pinned layers: field/group/scalar vs libsodium, SHA3/SHAKE vs hashlib,
 * Merlin vs its published vector, fixed-point conversion and accept/reject verdicts vs the reference's
 * literal-value unit tests (tests/test_oracle_*.py).
 */
#include "bp.h"
#include <math.h>
#include <stdio.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define EXPORT __attribute__((visibility("default")))

enum { DOM_RANGE_PROVE = 1, DOM_RANGE_VERIFY = 2, DOM_SQUARE = 3, DOM_L2_PROVE = 4, DOM_L2_VERIFY = 5, DOM_CRP = 6, DOM_RND_VEC = 7, DOM_RANDPROOF = 8, DOM_SQUARE_RAND = 9 };

/* key = SHA3-256(seed || u32le(domain) || u64le(index)) */
EXPORT void orc_derive_key(uint8_t out[32], const uint8_t seed[32], uint32_t domain, uint64_t index) {
    uint8_t buf[44]; memcpy(buf, seed, 32); u32le(buf + 32, domain);
    for (int i = 0; i < 8; i++) buf[36 + i] = (uint8_t)(index >> (8 * i));
    sha3_256(out, buf, 44);
}

static pc_gens_t PC; static int PC_INIT = 0;
static void init_pc(void) {
#pragma omp critical(pcinit)
    { if (!PC_INIT) { pc_gens_default(&PC); PC_INIT = 1; } }
}

/* ============================ primitive exports (used by tests to pin the layers) ============== */
EXPORT void orc_sc_mul(uint8_t o[32], const uint8_t a[32], const uint8_t b[32]) { sc x, y, r; sc_from_bytes_mod_order(&x, a); sc_from_bytes_mod_order(&y, b); sc_mul(&r, &x, &y); sc_tobytes(o, &r); }
EXPORT void orc_sc_add(uint8_t o[32], const uint8_t a[32], const uint8_t b[32]) { sc x, y, r; sc_from_bytes_mod_order(&x, a); sc_from_bytes_mod_order(&y, b); sc_add(&r, &x, &y); sc_tobytes(o, &r); }
EXPORT void orc_sc_sub(uint8_t o[32], const uint8_t a[32], const uint8_t b[32]) { sc x, y, r; sc_from_bytes_mod_order(&x, a); sc_from_bytes_mod_order(&y, b); sc_sub(&r, &x, &y); sc_tobytes(o, &r); }
EXPORT void orc_sc_invert(uint8_t o[32], const uint8_t a[32]) { sc x, r; sc_from_bytes_mod_order(&x, a); sc_invert(&r, &x); sc_tobytes(o, &r); }
EXPORT void orc_sc_reduce_wide(uint8_t o[32], const uint8_t a[64]) { sc r; sc_from_bytes_wide(&r, a); sc_tobytes(o, &r); }
EXPORT int orc_sc_is_canonical(const uint8_t a[32]) { sc r; return sc_from_canonical_bytes(&r, a); }
EXPORT void orc_fe_mul(uint8_t o[32], const uint8_t a[32], const uint8_t b[32]) { fe x, y, r; fe_frombytes(&x, a); fe_frombytes(&y, b); fe_mul(&r, &x, &y); fe_tobytes(o, &r); }
EXPORT void orc_fe_invert(uint8_t o[32], const uint8_t a[32]) { fe x, r; fe_frombytes(&x, a); fe_invert(&r, &x); fe_tobytes(o, &r); }
EXPORT void orc_basepoint(uint8_t o[32]) { ge b; ge_base(&b); ge_compress(o, &b); }
EXPORT void orc_blinding_basepoint(uint8_t o[32]) { init_pc(); ge_compress(o, &PC.B_blinding); }
EXPORT int orc_scalarmult(uint8_t o[32], const uint8_t s[32], const uint8_t p[32]) {
    ge P, R; sc k; if (!ge_decompress(&P, p)) return -1; sc_from_bytes_mod_order(&k, s); ge_scalarmult(&R, &k, &P); ge_compress(o, &R); return 0;
}
EXPORT void orc_scalarmult_base(uint8_t o[32], const uint8_t s[32]) { ge P, R; sc k; ge_base(&P); sc_from_bytes_mod_order(&k, s); ge_scalarmult(&R, &k, &P); ge_compress(o, &R); }
EXPORT int orc_point_add(uint8_t o[32], const uint8_t a[32], const uint8_t b[32]) { ge P, Q, R; if (!ge_decompress(&P, a) || !ge_decompress(&Q, b)) return -1; ge_add(&R, &P, &Q); ge_compress(o, &R); return 0; }
EXPORT int orc_point_sub(uint8_t o[32], const uint8_t a[32], const uint8_t b[32]) { ge P, Q, R; if (!ge_decompress(&P, a) || !ge_decompress(&Q, b)) return -1; ge_sub(&R, &P, &Q); ge_compress(o, &R); return 0; }
EXPORT int orc_point_valid(const uint8_t a[32]) { ge P; return ge_decompress(&P, a); }
EXPORT void orc_from_uniform_bytes(uint8_t o[32], const uint8_t in[64]) { ge P; ge_from_uniform_bytes(&P, in); ge_compress(o, &P); }
EXPORT int orc_msm(uint8_t o[32], const uint8_t *scalars, const uint8_t *points, size_t n) {
    sc *s = malloc(sizeof(sc) * n); ge *p = malloc(sizeof(ge) * n); int rc = 0;
    for (size_t i = 0; i < n; i++) { sc_from_bytes_mod_order(&s[i], scalars + 32 * i); if (!ge_decompress(&p[i], points + 32 * i)) rc = -1; }
    if (!rc) { ge R; ge_msm(&R, s, p, n); ge_compress(o, &R); }
    free(s); free(p); return rc;
}
EXPORT void orc_sha3_512(uint8_t o[64], const uint8_t *in, size_t n) { sha3_512(o, in, n); }
EXPORT void orc_sha3_256(uint8_t o[32], const uint8_t *in, size_t n) { sha3_256(o, in, n); }
EXPORT void orc_shake256(uint8_t *o, size_t on, const uint8_t *in, size_t n) { sponge s; sponge_init(&s, 136); sponge_absorb(&s, in, n); sponge_finish(&s, 0x1f); sponge_squeeze(&s, o, on); }
EXPORT void orc_chacha20_block(uint8_t o[64], const uint8_t key[32], uint64_t ctr) { chacha20_block(o, key, ctr); }
/* Merlin: Transcript::new(proto); append_message(label,msg); challenge_bytes(clabel, n) */
EXPORT void orc_merlin_simple(uint8_t *o, size_t on, const char *proto, const char *label, const uint8_t *msg, size_t n, const char *clabel) {
    transcript t; transcript_init(&t, proto); transcript_append(&t, label, msg, n); transcript_challenge(&t, clabel, o, on);
}
/* BulletproofGens chain: n compressed points of party `party`, which = 'G' or 'H' (SURVEY A.2) */
EXPORT void orc_bp_gens(uint8_t *o, int which, uint32_t party, int n) {
    ge *g = malloc(sizeof(ge) * n); bp_gens_chain(g, (char)which, party, n);
    for (int i = 0; i < n; i++) ge_compress(o + 32 * i, &g[i]);
    free(g);
}
EXPORT void orc_rnd_scalar_vec(uint8_t *o, const uint8_t seed[32], size_t n) {   /* pedersen_ops.rs:124-127 */
    uint8_t key[32]; orc_derive_key(key, seed, DOM_RND_VEC, 0);
    for (size_t i = 0; i < n; i++) { sc s; rng_scalar_at(key, i, &s); sc_tobytes(o + 32 * i, &s); }
}

/* ============================ fixed point (fp.rs, conversion32.rs) ============================= */
static inline uint64_t fix_max(int n_bits) { return n_bits == 64 ? ~0ULL : ((1ULL << n_bits) - 1); }
static int fp_ok(int n_bits, int frac) { return (n_bits == 8 || n_bits == 16 || n_bits == 32 || n_bits == 64) && frac >= 0 && frac <= 12; }
/* Fix::saturating_from_float(|x|).to_bits()  -- round to nearest, ties to even, saturate (conversion32.rs:12) */
static inline int fix_from_f32(uint64_t *raw, float x, int n_bits, int frac) {
    if (isnan(x)) return -1;
    double r = rint((double)fabsf(x) * (double)(1u << frac));
    double lim = ldexp(1.0, n_bits);
    *raw = (r >= lim) ? fix_max(n_bits) : (uint64_t)r;
    return 0;
}
static inline float fix_to_f32(uint64_t raw, int frac) { return (float)raw * (1.0f / (float)(1u << frac)); }
/* conversion32.rs:11-19 */
static inline int f32_to_scalar(sc *s, float x, int n_bits, int frac) {
    uint64_t raw; if (fix_from_f32(&raw, x, n_bits, frac)) return -1;
    sc_from_u64(s, raw); if (x < 0.0f) sc_neg(s, s);
    return 0;
}
static inline uint64_t read_from_bytes(const sc *s, int n_bits) { return s->v[0] & fix_max(n_bits); }   /* fp.rs:42,58,74,95 */
/* conversion32.rs:24-34 */
static inline float scalar_to_f32(const sc *s, int n_bits, int frac) {
    uint8_t b[32]; sc_tobytes(b, s);
    if (b[31] != 0) { sc n; sc_neg(&n, s); return -fix_to_f32(read_from_bytes(&n, n_bits), frac); }
    return fix_to_f32(read_from_bytes(s, n_bits), frac);
}
/* conversion32.rs:56-60: Fix::from_bits(((1u128 << range-1) - 1) as URawFix) */
static inline float clip_max(int range, int n_bits, int frac) {
    uint64_t raw = (range - 1 >= 64) ? ~0ULL : ((1ULL << (range - 1)) - 1);
    return fix_to_f32(raw & fix_max(n_bits), frac);
}
static inline float l2_clip_max(int range, int n_bits, int frac) {          /* conversion32.rs:62-64 */
    uint64_t raw = (range >= 64) ? ~0ULL : ((1ULL << range) - 1);
    return fix_to_f32(raw & fix_max(n_bits), frac);
}
EXPORT int orc_f32_to_scalar_vec(uint8_t *o, const float *v, size_t D, int n_bits, int frac) {
    if (!fp_ok(n_bits, frac)) return -2;
    for (size_t i = 0; i < D; i++) { sc s; if (f32_to_scalar(&s, v[i], n_bits, frac)) return -1; sc_tobytes(o + 32 * i, &s); }
    return 0;
}
EXPORT int orc_scalar_to_f32_vec(float *o, const uint8_t *s32, size_t D, int n_bits, int frac) {
    if (!fp_ok(n_bits, frac)) return -2;
    for (size_t i = 0; i < D; i++) { sc s; sc_from_bytes_mod_order(&s, s32 + 32 * i); o[i] = scalar_to_f32(&s, n_bits, frac); }
    return 0;
}
EXPORT void orc_clip_bounds(float *mn, float *mx, int range, int n_bits, int frac) { *mx = clip_max(range, n_bits, frac); *mn = -*mx; }
EXPORT float orc_l2_clip_bound(int range, int n_bits, int frac) { return l2_clip_max(range, n_bits, frac); }
/* range_proof_vec/mod.rs:104-111 */
EXPORT void orc_clip_f32_to_range_vec(float *o, const float *v, size_t D, int range, int n_bits, int frac) {
    float mx = clip_max(range, n_bits, frac), mn = -mx;
    for (size_t i = 0; i < D; i++) o[i] = fminf(mx, fmaxf(mn, v[i]));
}
/* conversion32.rs:66-89 `square`: returns -1 where the reference panics (checked_mul overflow) */
EXPORT int orc_square(uint8_t o[32], const uint8_t s32[32], int n_bits, int frac) {
    sc s, n; sc_from_bytes_mod_order(&s, s32);
    uint64_t u = (s32[31] != 0) ? (sc_neg(&n, &s), read_from_bytes(&n, n_bits)) : read_from_bytes(&s, n_bits);
    unsigned __int128 p = ((unsigned __int128)u * u) >> frac;
    if (n_bits < 64 ? (p >> n_bits) != 0 : (p >> 64) != 0) return -1;
    sc r; sc_from_u64(&r, (uint64_t)p); sc_tobytes(o, &r); return 0;
}

/* ============================ commitments (pedersen_ops.rs, el_gamal.rs) ======================== */
/* pedersen_ops.rs:18-25 commit_vec over f32_to_scalar_vec(values); blind == NULL -> commit_no_blinding_vec (:9-16) */
EXPORT int orc_commit_f32(uint8_t *o, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac) {
    if (!fp_ok(n_bits, frac)) return -2;
    init_pc(); int rc = 0;
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        sc s, b; ge P; sc_0(&b);
        if (f32_to_scalar(&s, v[i], n_bits, frac)) { rc = -1; continue; }
        if (blind) sc_from_bytes_mod_order(&b, blind + 32 * i);
        pc_commit(&P, &PC, &s, &b); ge_compress(o + 32 * i, &P);
    }
    return rc;
}
EXPORT void orc_commit_scalars(uint8_t *o, const uint8_t *vals, const uint8_t *blind, size_t D) {
    init_pc();
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        sc s, b; ge P; sc_0(&b); sc_from_bytes_mod_order(&s, vals + 32 * i);
        if (blind) sc_from_bytes_mod_order(&b, blind + 32 * i);
        pc_commit(&P, &PC, &s, &b); ge_compress(o + 32 * i, &P);
    }
}
/* el_gamal.rs:57-69: R = blinding * B  (the R halves; compressed_rand_proof/party.rs:23-24) */
EXPORT void orc_elgamal_R(uint8_t *o, const uint8_t *blind, size_t D) {
    init_pc();
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) { sc b; ge P; sc_from_bytes_mod_order(&b, blind + 32 * i); ge_scalarmult(&P, &b, &PC.B); ge_compress(o + 32 * i, &P); }
}

/* ============================ range_proof_vec (range_proof_vec/mod.rs) ========================== */
static size_t next_pow2(size_t v) { if (v <= 1) return 1; size_t n = v - 1; while (n & (n - 1)) n &= n - 1; return n << 1; }  /* :237-246 */
EXPORT size_t orc_next_pow2(size_t v) { return next_pow2(v); }
EXPORT size_t orc_rp_proof_len(size_t N) { return rp_proof_len(N); }

/* create_rangeproof (:16-102).  proofs_out: n_chunks * rp_proof_len(range*chunk) bytes, commits_out: D*32.
 * returns 0 ok, 1 WrongNumBlindingFactors (n/a here), 2 ValueOutOfRangeError, -7 InvalidBitsize,
 * -99 where the reference panics ("Should not get here": non power-of-two chunking), -2 bad fp config */
static int range_prove_impl(uint8_t *proofs_out, uint8_t *commits_out, const float *values, const uint8_t *blind, size_t D,
                            int range, size_t n_partition, int n_bits, int frac, const uint8_t seed[32], const uint8_t *tx_bl_shift32) {
    if (!fp_ok(n_bits, frac) || D == 0 || range < 1 || range > n_bits) return -2;
    init_pc();
    float mx = clip_max(range, n_bits, frac), mn = -mx;
    for (size_t i = 0; i < D; i++) if (mn > values[i] || values[i] > mx) return 2;              /* :26-29,113-116 */
    size_t Dp = next_pow2(D);
    uint64_t *vals = calloc(Dp, sizeof(uint64_t)); sc *bl = calloc(Dp, sizeof(sc));
    sc offset; sc_from_u64(&offset, 1ULL << (range - 1));
    for (size_t i = 0; i < D; i++) {                                                             /* :35-43 */
        sc s; f32_to_scalar(&s, values[i], n_bits, frac); sc_add(&s, &s, &offset);
        vals[i] = read_from_bytes(&s, n_bits);
        sc_from_bytes_mod_order(&bl[i], blind + 32 * i);
    }
    size_t n_chunks = Dp < n_partition ? Dp : n_partition, chunk = Dp / n_chunks;                 /* :54-55 */
    if (!(range == 8 || range == 16 || range == 32 || range == 64)) { free(vals); free(bl); return -7; }
    if (chunk & (chunk - 1) || chunk * n_chunks != Dp) { free(vals); free(bl); return -99; }
    bp_gens_t bg; bp_gens_new(&bg, range, (int)chunk);           /* identical for every chunk (:126 rebuilds it per chunk) */
    size_t plen = rp_proof_len((size_t)range * chunk);
    uint8_t *V = malloc(32 * Dp); int rc = 0;
#pragma omp parallel for schedule(dynamic)
    for (size_t c = 0; c < n_chunks; c++) {                                                      /* :75-78, helper :118-142 */
        transcript t; transcript_init(&t, "RangeProof");
        uint8_t key[32]; rng_t rng; orc_derive_key(key, seed, DOM_RANGE_PROVE, c); rng_init(&rng, key);
        sc shift; if (tx_bl_shift32) sc_from_bytes_mod_order(&shift, tx_bl_shift32 + 32 * c);
        int r = rp_prove_multiple_ex(proofs_out + plen * c, V + 32 * chunk * c, &bg, &PC, &t, vals + chunk * c, bl + chunk * c, (int)chunk, range, &rng,
                                     tx_bl_shift32 ? &shift : NULL);
        if (r) rc = r;
    }
    if (!rc) {
        sc noff; sc_neg(&noff, &offset); ge inv_off; ge_scalarmult(&inv_off, &noff, &PC.B);      /* :96-99 */
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < D; i++) { ge P; ge_decompress(&P, V + 32 * i); ge_add(&P, &P, &inv_off); ge_compress(commits_out + 32 * i, &P); }
    }
    bp_gens_free(&bg); free(V); free(vals); free(bl);
    return rc;
}
EXPORT int orc_range_prove(uint8_t *proofs_out, uint8_t *commits_out, const float *values, const uint8_t *blind, size_t D,
                           int range, size_t n_partition, int n_bits, int frac, const uint8_t seed[32]) {
    return range_prove_impl(proofs_out, commits_out, values, blind, D, range, n_partition, n_bits, frac, seed, NULL);
}
/* the same proofs with t_x_blinding of chunk c shifted by tx_bl_shift32[c] (n_chunks x 32 bytes) before it is absorbed: each chunk's
 * verification equation is then off by exactly -c_verifier shift B_blinding (tests of the batched verifier only) */
EXPORT int orc_range_prove_tx_bl_shifted(uint8_t *proofs_out, uint8_t *commits_out, const float *values, const uint8_t *blind, size_t D,
                                         int range, size_t n_partition, int n_bits, int frac, const uint8_t seed[32], const uint8_t *tx_bl_shift32) {
    return range_prove_impl(proofs_out, commits_out, values, blind, D, range, n_partition, n_bits, frac, seed, tx_bl_shift32);
}
/* verify_rangeproof (:149-191).  returns 1 true, 0 false, <0 error (-1 format, -7 bitsize, -3 gens length, -4 bad point) */
EXPORT int orc_range_verify(const uint8_t *proofs, size_t proof_len, size_t n_proofs, const uint8_t *commits, size_t D,
                            int range, const uint8_t seed[32]) {
    if (D == 0 || n_proofs == 0 || range < 1 || range > 64) return -2;
    init_pc();
    size_t Dp = next_pow2(D), chunk = Dp / n_proofs;
    if (chunk == 0) return -3;
    uint8_t *V = calloc(Dp, 32);                          /* identity encodes as 32 zero bytes (:163-165) */
    sc off; sc_from_u64(&off, 1ULL << (range - 1)); ge offp; ge_scalarmult(&offp, &off, &PC.B);
    int bad = 0;
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) { ge P; if (!ge_decompress(&P, commits + 32 * i)) { bad = 1; continue; } ge_add(&P, &P, &offp); ge_compress(V + 32 * i, &P); }
    if (bad) { free(V); return -4; }
    bp_gens_t bg; bp_gens_new(&bg, range, (int)chunk);
    int res = 1, err = 0;
#pragma omp parallel for schedule(dynamic)
    for (size_t c = 0; c < n_proofs; c++) {
        if ((c + 1) * chunk > Dp) continue;
        transcript t; transcript_init(&t, "RangeProof");
        uint8_t key[32]; rng_t rng; orc_derive_key(key, seed, DOM_RANGE_VERIFY, c); rng_init(&rng, key);
        int r = rp_verify_multiple(proofs + proof_len * c, proof_len, V + 32 * chunk * c, &bg, &PC, &t, (int)chunk, range, &rng);
#pragma omp critical(verres)
        { if (r < 0) { if (!err) err = r; } else res &= r; }
    }
    bp_gens_free(&bg); free(V);
    return err ? err : res;
}

/* the verifier's transcript challenges and batch digest of one range proof (bp.h rp_challenges); V32: its m commitments as the transcript sees them
 * (shifted for L-infinity, padding = identity encodings); label_id 0 "RangeProof", 1 "L2RangeProof" */
EXPORT int orc_rp_challenges(const uint8_t *proof, size_t proof_len, const uint8_t *V32, int n, int m, int label_id, uint8_t *out_chal, uint8_t out_digest[32]) {
    transcript t; transcript_init(&t, label_id ? "L2RangeProof" : "RangeProof");
    return rp_challenges(proof, proof_len, V32, &t, m, n, out_chal, out_digest);
}

/* ============================ l2_range_proof_vec (l2_range_proof_vec/mod.rs) ==================== */
/* create_rangeproof_l2 (:15-140): returns 0 ok, 2 ValueOutOfRange, 3 OverflowError, 4 NormOutOfRange, -7 InvalidBitsize.
 * proof_out: rp_proof_len(range) bytes; commit_out: 32 bytes (NOT shifted) */
EXPORT int orc_l2_prove(uint8_t *proof_out, uint8_t *commit_out, const float *values, const uint8_t *blind, size_t D,
                        int range, int n_bits, int frac, const uint8_t seed[32]) {
    if (!fp_ok(n_bits, frac) || D == 0) return -2;
    init_pc();
    float mx = clip_max(range, n_bits, frac), mn = -mx;
    for (size_t i = 0; i < D; i++) if (mn > values[i] || values[i] > mx) return 2;
    sc val, bsum; sc_0(&val); sc_0(&bsum);
    float shift = (float)(1 << frac), val_float = 0.0f;
    for (size_t i = 0; i < D; i++) {                                                             /* :37-50 */
        sc s, b; f32_to_scalar(&s, values[i], n_bits, frac); sc_muladd(&val, &s, &s, &val);
        float x = scalar_to_f32(&s, n_bits, frac), term = x * x * shift;
        val_float = (i == 0) ? term : val_float + term;
        sc_from_bytes_mod_order(&b, blind + 32 * i); sc_add(&bsum, &bsum, &b);
    }
    float vf = scalar_to_f32(&val, n_bits, frac);
    if (fabsf(vf - val_float) > 1.1920929e-7f) return 3;                                         /* :53-58 */
    if (vf > l2_clip_max(range, n_bits, frac)) return 4;                                         /* :60-64 */
    uint64_t v = read_from_bytes(&val, n_bits);                                                  /* :69-73 */
    if (!(range == 8 || range == 16 || range == 32 || range == 64)) return -7;
    bp_gens_t bg; bp_gens_new(&bg, 64, 1);                                                       /* :162 */
    transcript t; transcript_init(&t, "L2RangeProof");
    uint8_t key[32]; rng_t rng; orc_derive_key(key, seed, DOM_L2_PROVE, 0); rng_init(&rng, key);
    int rc = rp_prove_multiple(proof_out, commit_out, &bg, &PC, &t, &v, &bsum, 1, range, &rng);
    bp_gens_free(&bg);
    return rc;
}
/* verify_rangeproof_l2 (:185-228) */
EXPORT int orc_l2_verify(const uint8_t *proof, size_t proof_len, const uint8_t commit[32], int range, const uint8_t seed[32]) {
    init_pc();
    ge P; if (!ge_decompress(&P, commit)) return -4;
    uint8_t V[32]; ge_compress(V, &P);
    bp_gens_t bg; bp_gens_new(&bg, 64, 1);
    transcript t; transcript_init(&t, "L2RangeProof");
    uint8_t key[32]; rng_t rng; orc_derive_key(key, seed, DOM_L2_VERIFY, 0); rng_init(&rng, key);
    int r = rp_verify_multiple(proof, proof_len, V, &bg, &PC, &t, 1, range, &rng);
    bp_gens_free(&bg);
    return r;
}

/* ============================ square proofs (square_proof/{mod,party,dealer}.rs, square_proof_vec/mod.rs) ======== */
static void sq_transcript_start(transcript *t, const uint8_t cl[32], const uint8_t csq[32]) {     /* dealer.rs:20-27 */
    transcript_init(t, "SquareProof");
    transcript_append(t, "dom-sep", (const uint8_t *)"randomness proof v1", 19);                 /* transcript.rs:20-22 */
    transcript_append(t, "C_eg", cl, 32); transcript_append(t, "C_ped", csq, 32);
}
/* the challenge of one square proof (dealer.rs:20-27,49-53): com64 = c_l | c_sq, cp64 = C'_l | C'_sq */
EXPORT void orc_sq_challenge(uint8_t o[32], const uint8_t com64[64], const uint8_t cp64[64]) {
    transcript t; sc c; sq_transcript_start(&t, com64, com64 + 32);
    transcript_append(&t, "C_prime_eg", cp64, 32); transcript_append(&t, "C_prime_ped", cp64 + 32, 32);
    ts_challenge(&t, "c", &c); sc_tobytes(o, &c);
}
/* create_l2rangeproof_vec_existing (square_proof_vec/mod.rs:19-75) -> SquareProof::prove_existing (square_proof/mod.rs:42-58).
 * proofs_out: D*160 (C'_l|C'_sq|z_m|z_r1|z_r2), commits_out: D*64 (c_l|c_sq).  returns 0, 1 WrongNumBlindingFactors n/a, -4 bad point */
EXPORT int orc_square_prove(uint8_t *proofs_out, uint8_t *commits_out, const float *values, const uint8_t *value_com,
                            const uint8_t *r1v, const uint8_t *r2v, size_t D, int n_bits, int frac, const uint8_t seed[32]) {
    if (!fp_ok(n_bits, frac)) return -2;
    init_pc();
    uint8_t key[32]; orc_derive_key(key, seed, DOM_SQUARE, 0);
    int rc = 0;
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        sc m, r1, r2, msq, mp, r1p, r2p, c, zm, zr1, zr2, tmp;
        ge Cl, Csq, Cp, Csqp, T;
        if (f32_to_scalar(&m, values[i], n_bits, frac) || !ge_decompress(&Cl, value_com + 32 * i)) { rc = -4; continue; }
        sc_from_bytes_mod_order(&r1, r1v + 32 * i); sc_from_bytes_mod_order(&r2, r2v + 32 * i);
        sc_mul(&msq, &m, &m); pc_commit(&Csq, &PC, &msq, &r2);                                   /* party.rs:34-35 */
        rng_scalar_at(key, 3 * i, &mp); rng_scalar_at(key, 3 * i + 1, &r1p); rng_scalar_at(key, 3 * i + 2, &r2p);   /* :40-42 */
        pc_commit(&Cp, &PC, &mp, &r1p);                                                          /* :44 */
        ge_scalarmult(&Csqp, &mp, &Cl); ge_scalarmult(&T, &r2p, &PC.B_blinding); ge_add(&Csqp, &Csqp, &T);   /* :46-50 */
        uint8_t *o = proofs_out + 160 * i, *co = commits_out + 64 * i;
        ge_compress(co, &Cl); ge_compress(co + 32, &Csq); ge_compress(o, &Cp); ge_compress(o + 32, &Csqp);
        transcript t; sq_transcript_start(&t, co, co + 32);
        transcript_append(&t, "C_prime_eg", o, 32); transcript_append(&t, "C_prime_ped", o + 32, 32);   /* dealer.rs:49-53 */
        ts_challenge(&t, "c", &c);
        sc_muladd(&zm, &m, &c, &mp); sc_muladd(&zr1, &r1, &c, &r1p);                             /* party.rs:146-152 */
        sc_mul(&tmp, &m, &r1); sc_sub(&tmp, &r2, &tmp); sc_muladd(&zr2, &tmp, &c, &r2p);
        sc_tobytes(o + 64, &zm); sc_tobytes(o + 96, &zr1); sc_tobytes(o + 128, &zr2);
    }
    return rc;
}
/* RandProof per element (rand_proof/{mod,party,dealer}.rs, rand_proof_vec/mod.rs:14-118).  pairs_out D*64 (L|R), proofs_out D*128 (C'_L|C'_R|z_m|z_r).
 * value_com NULL: Party::new (L = commit(m, r)); else PartyExisting.  0 ok, -4 bad point */
static void rp_challenge(sc *c, const uint8_t pair[64], const uint8_t cp[64]) {
    transcript t; transcript_init(&t, "RandProof");
    transcript_append(&t, "dom-sep", (const uint8_t *)"randomness proof v1", 19);
    transcript_append(&t, "C", pair, 64); transcript_append(&t, "C_prime", cp, 64);               /* dealer.rs:20-21,42 */
    ts_challenge(&t, "c", c);
}
EXPORT void orc_rp_challenge(uint8_t o[32], const uint8_t pair[64], const uint8_t cp[64]) { sc c; rp_challenge(&c, pair, cp); sc_tobytes(o, &c); }
EXPORT int orc_rand_prove(uint8_t *proofs_out, uint8_t *pairs_out, const float *values, const uint8_t *value_com, const uint8_t *rv, size_t D, int n_bits, int frac, const uint8_t seed[32]) {
    if (!fp_ok(n_bits, frac)) return -2;
    init_pc(); uint8_t key[32]; orc_derive_key(key, seed, DOM_RANDPROOF, 0); int rc = 0; ge Bp; ge_base(&Bp);
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        sc m, r, mp, rp, c, zm, zr; ge L, R, Lp, Rp;
        if (f32_to_scalar(&m, values[i], n_bits, frac)) { rc = -98; continue; }
        sc_from_bytes_mod_order(&r, rv + 32 * i);
        if (value_com) { if (!ge_decompress(&L, value_com + 32 * i)) { rc = -4; continue; } } else pc_commit(&L, &PC, &m, &r);
        ge_scalarmult(&R, &r, &Bp);
        rng_scalar_at(key, 2 * i, &mp); rng_scalar_at(key, 2 * i + 1, &rp);                        /* party.rs:23-24 */
        pc_commit(&Lp, &PC, &mp, &rp); ge_scalarmult(&Rp, &rp, &Bp);
        uint8_t *o = proofs_out + 128 * i, *po = pairs_out + 64 * i;
        ge_compress(po, &L); ge_compress(po + 32, &R); ge_compress(o, &Lp); ge_compress(o + 32, &Rp);
        rp_challenge(&c, po, o);
        sc_muladd(&zm, &m, &c, &mp); sc_muladd(&zr, &r, &c, &rp);                                  /* party.rs:76-80 */
        sc_tobytes(o + 64, &zm); sc_tobytes(o + 96, &zr);
    }
    return rc;
}
EXPORT int orc_rand_verify(const uint8_t *proofs, const uint8_t *pairs, size_t D) {              /* rand_proof/mod.rs:64-85, rand_proof_vec/mod.rs:91-118 */
    init_pc(); int res = 1, err = 0; ge Bp; ge_base(&Bp);
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        const uint8_t *o = proofs + 128 * i, *po = pairs + 64 * i;
        ge L, R, Lp, Rp, lhs, rhs, T; sc zm, zr, c;
        if (!ge_decompress(&L, po) || !ge_decompress(&R, po + 32) || !ge_decompress(&Lp, o) || !ge_decompress(&Rp, o + 32) ||
            !sc_from_canonical_bytes(&zm, o + 64) || !sc_from_canonical_bytes(&zr, o + 96)) { err = -1; continue; }
        rp_challenge(&c, po, o);
        int ok = 1;
        pc_commit(&lhs, &PC, &zm, &zr); ge_scalarmult(&T, &c, &L); ge_add(&rhs, &Lp, &T); ok &= ge_eq(&lhs, &rhs);
        ge_scalarmult(&lhs, &zr, &Bp); ge_scalarmult(&T, &c, &R); ge_add(&rhs, &Rp, &T); ok &= ge_eq(&lhs, &rhs);
        if (!ok) res = 0;
    }
    return err ? err : res;
}
/* SquareRandProof per element (square_rand_proof/{mod,party,dealer,constants}.rs, square_rand_proof_vec/mod.rs:18-160).
 * commits_out D*96 (c.L|c.R|c_sq), proofs_out D*192 (C'.L|C'.R|C'_sq|z_m|z_r1|z_r2) */
static void srp_challenge(sc *c, const uint8_t com[96], const uint8_t cp[96]) {
    transcript t; transcript_init(&t, "SquareRandProof");
    transcript_append(&t, "dom-sep", (const uint8_t *)"randomness proof v1", 19);
    transcript_append(&t, "C_eg", com, 64); transcript_append(&t, "C_ped", com + 64, 32);         /* dealer.rs:23-25 */
    transcript_append(&t, "C_prime_eg", cp, 64); transcript_append(&t, "C_prime_ped", cp + 64, 32);
    ts_challenge(&t, "c", c);
}
EXPORT void orc_srp_challenge(uint8_t o[32], const uint8_t com[96], const uint8_t cp[96]) { sc c; srp_challenge(&c, com, cp); sc_tobytes(o, &c); }
EXPORT int orc_square_rand_prove(uint8_t *proofs_out, uint8_t *commits_out, const float *values, const uint8_t *value_com, const uint8_t *r1v, const uint8_t *r2v, size_t D,
                                 int n_bits, int frac, const uint8_t seed[32]) {
    if (!fp_ok(n_bits, frac)) return -2;
    init_pc(); uint8_t key[32]; orc_derive_key(key, seed, DOM_SQUARE_RAND, 0); int rc = 0; ge Bp; ge_base(&Bp);
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        sc m, r1, r2, msq, mp, r1p, r2p, c, zm, zr1, zr2, tmp; ge L, R, Csq, Lp, Rp, Csqp, T;
        if (f32_to_scalar(&m, values[i], n_bits, frac)) { rc = -98; continue; }
        sc_from_bytes_mod_order(&r1, r1v + 32 * i); sc_from_bytes_mod_order(&r2, r2v + 32 * i);
        if (value_com) { if (!ge_decompress(&L, value_com + 32 * i)) { rc = -4; continue; } } else pc_commit(&L, &PC, &m, &r1);
        ge_scalarmult(&R, &r1, &Bp);
        sc_mul(&msq, &m, &m); pc_commit(&Csq, &PC, &msq, &r2);                                      /* party.rs:31-32 */
        rng_scalar_at(key, 3 * i, &mp); rng_scalar_at(key, 3 * i + 1, &r1p); rng_scalar_at(key, 3 * i + 2, &r2p);
        pc_commit(&Lp, &PC, &mp, &r1p); ge_scalarmult(&Rp, &r1p, &Bp);
        ge_scalarmult(&Csqp, &mp, &L); ge_scalarmult(&T, &r2p, &PC.B_blinding); ge_add(&Csqp, &Csqp, &T);
        uint8_t *o = proofs_out + 192 * i, *co = commits_out + 96 * i;
        ge_compress(co, &L); ge_compress(co + 32, &R); ge_compress(co + 64, &Csq); ge_compress(o, &Lp); ge_compress(o + 32, &Rp); ge_compress(o + 64, &Csqp);
        srp_challenge(&c, co, o);
        sc_muladd(&zm, &m, &c, &mp); sc_muladd(&zr1, &r1, &c, &r1p);
        sc_mul(&tmp, &m, &r1); sc_sub(&tmp, &r2, &tmp); sc_muladd(&zr2, &tmp, &c, &r2p);
        sc_tobytes(o + 96, &zm); sc_tobytes(o + 128, &zr1); sc_tobytes(o + 160, &zr2);
    }
    return rc;
}
EXPORT int orc_square_rand_verify(const uint8_t *proofs, const uint8_t *commits, size_t D) {     /* square_rand_proof/mod.rs:76-112 */
    init_pc(); int res = 1, err = 0; ge Bp; ge_base(&Bp);
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        const uint8_t *o = proofs + 192 * i, *co = commits + 96 * i;
        ge L, R, Csq, Lp, Rp, Csqp, lhs, rhs, T; sc zm, zr1, zr2, c;
        if (!ge_decompress(&L, co) || !ge_decompress(&R, co + 32) || !ge_decompress(&Csq, co + 64) || !ge_decompress(&Lp, o) || !ge_decompress(&Rp, o + 32) || !ge_decompress(&Csqp, o + 64) ||
            !sc_from_canonical_bytes(&zm, o + 96) || !sc_from_canonical_bytes(&zr1, o + 128) || !sc_from_canonical_bytes(&zr2, o + 160)) { err = -1; continue; }
        srp_challenge(&c, co, o);
        int ok = 1;
        pc_commit(&lhs, &PC, &zm, &zr1); ge_scalarmult(&T, &c, &L); ge_add(&rhs, &Lp, &T); ok &= ge_eq(&lhs, &rhs);
        ge_scalarmult(&lhs, &zr1, &Bp); ge_scalarmult(&T, &c, &R); ge_add(&rhs, &Rp, &T); ok &= ge_eq(&lhs, &rhs);
        ge_scalarmult(&lhs, &zm, &L); ge_scalarmult(&T, &zr2, &PC.B_blinding); ge_add(&lhs, &lhs, &T);
        ge_scalarmult(&T, &c, &Csq); ge_add(&rhs, &Csqp, &T); ok &= ge_eq(&lhs, &rhs);
        if (!ok) res = 0;
    }
    return err ? err : res;
}
/* CompressedRandProof (compressed_rand_proof/mod.rs:43-102, party.rs:17-100, dealer.rs:20-94, constants.rs:5-7):
 * ONE sigma proof that every ElGamal pair (L_i, R_i) = (m_i B + r_i H, r_i B) of an update is well formed.
 *   pairs_out: D*64 (L|R).  value_com = existing L_i (prove_existing, party.rs:17-45) or NULL (Party::new :50-79: L_i = commit(m_i, r_i)).
 *   proof_out: 128 = C'_L | C'_R | z_m | z_r.   Transcript labels of the pairs: [3i, 3i+1, 3i+2] mod 256 (generate_unique_u8_triplets.py:9-13);
 *   the label table has 900 000 rows, a longer update indexes past its end (panic) -> -6.  returns 0, -4 bad point, -2 bad args */
#define CRP_MAX_D 900000
static void crp_transcript(transcript *t, const uint8_t *pairs, size_t D, const uint8_t cprime[64], sc *c) {
    transcript_init(t, "CompressedRandProof");                                                     /* mod.rs:137,144,153 */
    transcript_append(t, "dom-sep", (const uint8_t *)"randomness proof v1", 19);                   /* rand_proof/transcript.rs:20-22 */
    for (size_t i = 0; i < D; i++) {
        uint8_t lab[3] = {(uint8_t)(3 * i), (uint8_t)(3 * i + 1), (uint8_t)(3 * i + 2)};
        transcript_append_l(t, lab, 3, pairs + 64 * i, 64);                                        /* dealer.rs:27-29 */
    }
    transcript_append(t, "C_prime_eg", cprime, 64);                                                /* dealer.rs:53-54 */
    ts_challenge(t, "c", c);
}
EXPORT void orc_crp_challenge(uint8_t o[32], const uint8_t *pairs, size_t D, const uint8_t cprime[64]) { transcript t; sc c; crp_transcript(&t, pairs, D, cprime, &c); sc_tobytes(o, &c); }
EXPORT int orc_crp_prove(uint8_t proof_out[128], uint8_t *pairs_out, const float *values, const uint8_t *value_com, const uint8_t *rv, size_t D,
                         int n_bits, int frac, const uint8_t seed[32]) {
    if (!fp_ok(n_bits, frac)) return -2;
    if (D > CRP_MAX_D) return -6;
    init_pc();
    sc *m = malloc(sizeof(sc) * (D ? D : 1)), *r = malloc(sizeof(sc) * (D ? D : 1)); int rc = 0;
    ge Bp; ge_base(&Bp);
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        ge Lp, Rp;
        if (f32_to_scalar(&m[i], values[i], n_bits, frac)) { rc = -98; continue; }
        sc_from_bytes_mod_order(&r[i], rv + 32 * i);
        if (value_com) { if (!ge_decompress(&Lp, value_com + 32 * i)) { rc = -4; continue; } }
        else pc_commit(&Lp, &PC, &m[i], &r[i]);
        ge_scalarmult(&Rp, &r[i], &Bp);                                                            /* el_gamal.rs:57-69 */
        ge_compress(pairs_out + 64 * i, &Lp); ge_compress(pairs_out + 64 * i + 32, &Rp);
    }
    if (!rc) {
        uint8_t key[32]; orc_derive_key(key, seed, DOM_CRP, 0);
        sc mp, rp, c, zm, zr, pw, t; ge Cl, Cr;
        rng_scalar_at(key, 0, &mp); rng_scalar_at(key, 1, &rp);                                    /* party.rs:26-29 */
        pc_commit(&Cl, &PC, &mp, &rp); ge_scalarmult(&Cr, &rp, &Bp);
        ge_compress(proof_out, &Cl); ge_compress(proof_out + 32, &Cr);
        transcript tr; crp_transcript(&tr, pairs_out, D, proof_out, &c);
        zm = mp; zr = rp; pw = c;                                                                  /* party.rs:90-100: sum m_i c^(i+1) */
        for (size_t i = 0; i < D; i++) { sc_mul(&t, &m[i], &pw); sc_add(&zm, &zm, &t); sc_mul(&t, &r[i], &pw); sc_add(&zr, &zr, &t); sc_mul(&pw, &pw, &c); }
        sc_tobytes(proof_out + 64, &zm); sc_tobytes(proof_out + 96, &zr);
    }
    free(m); free(r);
    return rc;
}
/* CompressedRandProof::verify (mod.rs:76-102) after from_bytes (:118-134): 1 valid, 0 invalid, -1 FormatError, -6 too long */
EXPORT int orc_crp_verify(const uint8_t proof[128], const uint8_t *pairs, size_t D) {
    if (D > CRP_MAX_D) return -6;
    init_pc();
    ge Cl, Cr, Bp; sc zm, zr, c; ge_base(&Bp);
    if (!ge_decompress(&Cl, proof) || !ge_decompress(&Cr, proof + 32) || !sc_from_canonical_bytes(&zm, proof + 64) || !sc_from_canonical_bytes(&zr, proof + 96)) return -1;
    ge *Lp = malloc(sizeof(ge) * (D ? D : 1)), *Rp = malloc(sizeof(ge) * (D ? D : 1)); sc *pw = malloc(sizeof(sc) * (D ? D : 1)); int bad = 0;
    for (size_t i = 0; i < D; i++) if (!ge_decompress(&Lp[i], pairs + 64 * i) || !ge_decompress(&Rp[i], pairs + 64 * i + 32)) bad = 1;
    int res = -1;
    if (!bad) {
        transcript tr; crp_transcript(&tr, pairs, D, proof, &c);
        sc p = c; for (size_t i = 0; i < D; i++) { pw[i] = p; sc_mul(&p, &p, &c); }
        ge SL, SR, lhsL, lhsR, T;
        ge_msm(&SL, pw, Lp, D); ge_msm(&SR, pw, Rp, D);
        ge_add(&SL, &SL, &Cl); ge_add(&SR, &SR, &Cr);                                              /* C' + sum c^(i+1) C_i */
        pc_commit(&lhsL, &PC, &zm, &zr); ge_scalarmult(&lhsR, &zr, &Bp);                            /* eg_gens.commit(z_m, z_r) */
        (void)T;
        res = (ge_eq(&lhsL, &SL) && ge_eq(&lhsR, &SR)) ? 1 : 0;
    }
    free(Lp); free(Rp); free(pw);
    return res;
}
/* verify_l2rangeproof_vec (square_proof_vec/mod.rs:130-160) -> SquareProof::verify (square_proof/mod.rs:77-112).
 * returns 1 true, 0 false, -1 FormatError (from_bytes :127-146, pedersen.rs:30-45) */
EXPORT int orc_square_verify(const uint8_t *proofs, const uint8_t *commits, size_t D) {
    init_pc(); int res = 1, err = 0;
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        const uint8_t *o = proofs + 160 * i, *co = commits + 64 * i;
        ge Cl, Csq, Cp, Csqp, lhs, rhs, T; sc zm, zr1, zr2, c;
        if (!ge_decompress(&Cl, co) || !ge_decompress(&Csq, co + 32) || !ge_decompress(&Cp, o) || !ge_decompress(&Csqp, o + 32) ||
            !sc_from_canonical_bytes(&zm, o + 64) || !sc_from_canonical_bytes(&zr1, o + 96) || !sc_from_canonical_bytes(&zr2, o + 128)) { err = -1; continue; }
        transcript t; sq_transcript_start(&t, co, co + 32);
        transcript_append(&t, "C_prime_eg", o, 32); transcript_append(&t, "C_prime_ped", o + 32, 32);
        ts_challenge(&t, "c", &c);
        int ok = 1;
        pc_commit(&lhs, &PC, &zm, &zr1); ge_scalarmult(&T, &c, &Cl); ge_add(&rhs, &Cp, &T); ok &= ge_eq(&lhs, &rhs);         /* mod.rs:94-98 */
        ge_scalarmult(&lhs, &zm, &Cl); ge_scalarmult(&T, &zr2, &PC.B_blinding); ge_add(&lhs, &lhs, &T);
        ge_scalarmult(&T, &c, &Csq); ge_add(&rhs, &Csqp, &T); ok &= ge_eq(&lhs, &rhs);                                       /* :101-109 */
        if (!ok) res = 0;
    }
    return err ? err : res;
}

/* ============================ aggregate + decrypt =============================================== */
/* params.rs:81-124 accumulate / pedersen_ops.rs:56-69 add_rp_vec_vec.  clients: n_clients pointers-free layout:
 * pts[client][D] compressed.  init: 0 = identity (add_rp_vec_vec), 1 = basepoint (ElGamalPair::unity, el_gamal.rs:83-88) */
EXPORT int orc_aggregate(uint8_t *o, const uint8_t *pts, size_t n_clients, size_t D, int init) {
    int rc = 0;
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        ge acc, P; if (init) ge_base(&acc); else ge_identity(&acc);
        for (size_t c = 0; c < n_clients; c++) { if (!ge_decompress(&P, pts + 32 * (c * D + i))) { rc = -4; break; } ge_add(&acc, &acc, &P); }
        ge_compress(o + 32 * i, &acc);
    }
    return rc;
}
/* bsgs32.rs:20-73 + pedersen_ops.rs:47-53.  table_size = m, bsgs_bits = BSGS_N_BITS (8 or 16: the width of BSGS_URawFix).
 * out scalars D*32.  returns 0, or -5 where the reference panics (`inv_res.unwrap()` on None, bsgs32.rs:70) */
typedef struct { uint64_t key; uint32_t val; uint32_t used; uint8_t full[32]; } bsgs_ent;
EXPORT int orc_dlog(uint8_t *o, const uint8_t *pts, size_t D, size_t table_size, int bsgs_bits) {
    init_pc();
    uint64_t vmask = (1ULL << bsgs_bits) - 1;
    size_t cap = 1; while (cap < 4 * (table_size + 1)) cap <<= 1;
    bsgs_ent *tab = calloc(cap, sizeof(bsgs_ent));
    size_t distinct = 0;
    ge cur; ge_identity(&cur);
    for (size_t x = 0; x <= table_size; x++) {                    /* bsgs32.rs:26-33: insert overwrites on equal key */
        uint8_t k[32]; ge_compress(k, &cur);
        uint64_t h; memcpy(&h, k, 8); size_t pos = (h * 0x9E3779B97F4A7C15ULL) >> 20 & (cap - 1);
        while (tab[pos].used && memcmp(tab[pos].full, k, 32)) pos = (pos + 1) & (cap - 1);
        if (!tab[pos].used) { distinct++; tab[pos].used = 1; memcpy(tab[pos].full, k, 32); }
        tab[pos].val = (uint32_t)(x & vmask);
        ge_add(&cur, &cur, &PC.B);
    }
    uint64_t size = distinct - 1;                                  /* get_size :44-46 */
    sc msc; sc_from_u64(&msc, table_size & vmask); ge mG; ge_scalarmult(&mG, &msc, &PC.B);   /* :23 */
    uint64_t max_it = size ? (1ULL << bsgs_bits) / size : 0;       /* :60-62 */
    int rc = 0;
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < D; i++) {
        ge M; if (!ge_decompress(&M, pts + 32 * i)) { rc = -4; continue; }
        int found = 0; uint64_t val = 0; sc res;
        for (int sign = 0; sign < 2 && !found; sign++) {
            ge curp; if (sign) ge_neg(&curp, &M); else curp = M;
            for (uint64_t it = 0; it < max_it && !found; it++) {
                uint8_t k[32]; ge_compress(k, &curp);
                uint64_t h; memcpy(&h, k, 8); size_t pos = (h * 0x9E3779B97F4A7C15ULL) >> 20 & (cap - 1);
                while (tab[pos].used && memcmp(tab[pos].full, k, 32)) pos = (pos + 1) & (cap - 1);
                if (tab[pos].used) { found = 1 + sign; val = (it * size + tab[pos].val) & vmask; }
                else ge_sub(&curp, &curp, &mG);
            }
        }
        if (!found) { rc = -5; memset(o + 32 * i, 0xff, 32); continue; }
        sc_from_u64(&res, val); if (found == 2) sc_neg(&res, &res);
        sc_tobytes(o + 32 * i, &res);
    }
    free(tab);
    return rc;
}
EXPORT int orc_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
EXPORT void orc_set_num_threads(int n) {
#ifdef _OPENMP
    omp_set_num_threads(n);
#else
    (void)n;
#endif
}
