/* ORACLE -- TEST INFRASTRUCTURE ONLY (see fe51.h).
 *
 * Restatement of the published Bulletproofs aggregated range proof as implemented by the
 * `bulletproofs 4.0.0` crate (third-party; NOT under /root/reference, Cargo.lock:164-165):
 * PedersenGens / BulletproofGens (generator chain), RangeProof::prove_multiple_with_rng,
 * RangeProof::verify_multiple_with_rng, InnerProductProof::{create, verification_scalars},
 * byte serialisation.  Algorithm as restated in SURVEY.md Appendix A.2-A.4.
 * Reference call sites: range_proof_vec/mod.rs:124-135,200-209, l2_range_proof_vec/mod.rs:162-171,236-246.
 *
 * PARITY UNPINNED against the real crate: the reference holds no golden proof bytes and has no
 * seeded RNG; what IS pinned: group/scalar/hash layers against libsodium + hashlib + the Merlin
 * vector, and prove<->verify self-consistency (tests/).  Nonces come from an injected ChaCha20
 * stream in the draw order of prove_multiple_with_rng, so a Rust harness calling
 * `prove_multiple_with_rng(.., &mut ChaCha20Rng::from_seed(key))` can be compared byte for byte
 * later (INTEGRATION.md).
 */
#ifndef ROFL_ORACLE_BP_H
#define ROFL_ORACLE_BP_H
#include "ge.h"
#include "hash.h"
#include <stdlib.h>

/* ---- deterministic nonce source: draw k == ChaCha20 block k, wide-reduced (A.5) ------------ */
typedef struct { uint8_t key[32]; uint64_t ctr; } rng_t;
static inline void rng_init(rng_t *r, const uint8_t key[32]) { memcpy(r->key, key, 32); r->ctr = 0; }
static inline void rng_scalar(rng_t *r, sc *out) { uint8_t b[64]; chacha20_block(b, r->key, r->ctr++); sc_from_bytes_wide(out, b); }
static inline void rng_scalar_at(const uint8_t key[32], uint64_t idx, sc *out) { uint8_t b[64]; chacha20_block(b, key, idx); sc_from_bytes_wide(out, b); }

/* ---- generators ----------------------------------------------------------------------------- */
typedef struct { ge B, B_blinding; } pc_gens_t;
static inline void pc_gens_default(pc_gens_t *g) {
    uint8_t cb[32], h[64];
    ge_base(&g->B); ge_compress(cb, &g->B);
    sha3_512(h, cb, 32); ge_from_uniform_bytes(&g->B_blinding, h);
}
/* G_j[0..n) / H_j[0..n): SHAKE256("GeneratorsChain" || 'G'|'H' || u32le(j)), 64 bytes per point */
static inline void bp_gens_chain(ge *out, char which, uint32_t party, int n) {
    sponge s; sponge_init(&s, 136);
    uint8_t label[5] = {(uint8_t)which, (uint8_t)party, (uint8_t)(party >> 8), (uint8_t)(party >> 16), (uint8_t)(party >> 24)};
    sponge_absorb(&s, (const uint8_t *)"GeneratorsChain", 15); sponge_absorb(&s, label, 5);
    sponge_finish(&s, 0x1f);
    for (int i = 0; i < n; i++) { uint8_t u[64]; sponge_squeeze(&s, u, 64); ge_from_uniform_bytes(&out[i], u); }
}
typedef struct { int n, m; ge *G, *H; } bp_gens_t;     /* party-major: G[j*n + i] */
static inline void bp_gens_new(bp_gens_t *g, int n, int m) {
    g->n = n; g->m = m; g->G = (ge *)malloc(sizeof(ge) * n * m); g->H = (ge *)malloc(sizeof(ge) * n * m);
    /* the party chains are independent (SURVEY.md A.2); inside a parallel region (one thread per chunk) this loop stays serial */
#pragma omp parallel for schedule(static) if (m >= 64)
    for (int j = 0; j < m; j++) { bp_gens_chain(g->G + (size_t)j * n, 'G', j, n); bp_gens_chain(g->H + (size_t)j * n, 'H', j, n); }
}
static inline void bp_gens_free(bp_gens_t *g) { free(g->G); free(g->H); }

/* ---- multiscalar multiplication --------------------------------------------------------------
 * Straus with signed radix-16 digits and shared doublings (the shape of dalek's
 * `multiscalar_mul`); Pippenger for large sizes (dalek switches at 190 points). */
static inline void ge_msm_straus(ge *r, const sc *s, const ge *p, size_t n) {
    ge *tab = (ge *)malloc(sizeof(ge) * 8 * n); int8_t *e = (int8_t *)malloc(64 * n);
    for (size_t k = 0; k < n; k++) {
        tab[8 * k] = p[k];
        for (int i = 1; i < 8; i++) ge_add(&tab[8 * k + i], &tab[8 * k + i - 1], &p[k]);
        sc_radix16(e + 64 * k, &s[k]);
    }
    ge acc; ge_identity(&acc);
    for (int i = 63; i >= 0; i--) {
        if (i != 63) { ge_dbl(&acc, &acc); ge_dbl(&acc, &acc); ge_dbl(&acc, &acc); ge_dbl(&acc, &acc); }
        for (size_t k = 0; k < n; k++) {
            int d = e[64 * k + i];
            if (d > 0) ge_add(&acc, &acc, &tab[8 * k + d - 1]);
            else if (d < 0) ge_sub(&acc, &acc, &tab[8 * k - d - 1]);
        }
    }
    *r = acc; free(tab); free(e);
}
static inline void ge_msm_pippenger(ge *r, const sc *s, const ge *p, size_t n) {
    int w = n < 500 ? 6 : n < 800 ? 7 : 8;
    int nd = (256 + w - 1) / w + 1, nb = 1 << (w - 1);
    int16_t *dig = (int16_t *)malloc(sizeof(int16_t) * nd * n);
    for (size_t k = 0; k < n; k++) {                      /* signed radix-2^w digits */
        uint8_t b[40] = {0}; sc_tobytes(b, &s[k]);
        int carry = 0;
        for (int i = 0; i < nd; i++) {
            int bit = i * w, v = 0;
            for (int t = 0; t < w; t++) { int bb = bit + t; if (bb < 256) v |= ((b[bb >> 3] >> (bb & 7)) & 1) << t; }
            v += carry; carry = 0;
            if (v > nb) { v -= 1 << w; carry = 1; }
            dig[k * nd + i] = (int16_t)v;
        }
    }
    ge *bk = (ge *)malloc(sizeof(ge) * nb), acc; ge_identity(&acc);
    for (int i = nd - 1; i >= 0; i--) {
        for (int t = 0; t < w; t++) ge_dbl(&acc, &acc);
        for (int t = 0; t < nb; t++) ge_identity(&bk[t]);
        for (size_t k = 0; k < n; k++) {
            int d = dig[k * nd + i];
            if (d > 0) ge_add(&bk[d - 1], &bk[d - 1], &p[k]);
            else if (d < 0) ge_sub(&bk[-d - 1], &bk[-d - 1], &p[k]);
        }
        ge run, sum; ge_identity(&run); ge_identity(&sum);
        for (int t = nb - 1; t >= 0; t--) { ge_add(&run, &run, &bk[t]); ge_add(&sum, &sum, &run); }
        ge_add(&acc, &acc, &sum);
    }
    *r = acc; free(bk); free(dig);
}
static inline void ge_msm(ge *r, const sc *s, const ge *p, size_t n) {
    if (n < 190) { ge_msm_straus(r, s, p, n); return; }
    if (n < 65536) { ge_msm_pippenger(r, s, p, n); return; }
    /* one very large chunk (resnet18-full: 4.2 M points): term slices on the host threads, partial sums added up (same group element) */
    enum { SL = 64 }; ge part[SL]; const size_t per = (n + SL - 1) / SL;
#pragma omp parallel for schedule(dynamic)
    for (int t = 0; t < SL; t++) {
        const size_t b = (size_t)t * per, e = b + per < n ? b + per : n;
        if (b < e) ge_msm_pippenger(&part[t], s + b, p + b, e - b); else ge_identity(&part[t]);
    }
    ge acc; ge_identity(&acc);
    for (int t = 0; t < SL; t++) ge_add(&acc, &acc, &part[t]);
    *r = acc;
}
/* two-term variable-time a*P + b*Q with width-5 NAFs (dalek vartime Straus on 2 points) */
static inline void ge_double_scalarmult(ge *r, const sc *a, const ge *P, const sc *b, const ge *Q) {
    int8_t na[256], nb_[256]; ge tp[8], tq[8], P2, Q2;
    sc_naf(na, a, 5); sc_naf(nb_, b, 5);
    ge_dbl(&P2, P); ge_dbl(&Q2, Q); tp[0] = *P; tq[0] = *Q;
    for (int i = 1; i < 8; i++) { ge_add(&tp[i], &tp[i - 1], &P2); ge_add(&tq[i], &tq[i - 1], &Q2); }
    int i = 255; while (i >= 0 && na[i] == 0 && nb_[i] == 0) i--;
    ge acc; ge_identity(&acc);
    for (; i >= 0; i--) {
        ge_dbl(&acc, &acc);
        if (na[i] > 0) ge_add(&acc, &acc, &tp[na[i] >> 1]); else if (na[i] < 0) ge_sub(&acc, &acc, &tp[(-na[i]) >> 1]);
        if (nb_[i] > 0) ge_add(&acc, &acc, &tq[nb_[i] >> 1]); else if (nb_[i] < 0) ge_sub(&acc, &acc, &tq[(-nb_[i]) >> 1]);
    }
    *r = acc;
}
static inline void pc_commit(ge *r, const pc_gens_t *g, const sc *v, const sc *blind) {
    sc s[2] = {*v, *blind}; ge p[2] = {g->B, g->B_blinding}; ge_msm_straus(r, s, p, 2);
}

/* ---- transcript helpers (bulletproofs `TranscriptProtocol`) ---------------------------------- */
static inline void ts_point(transcript *t, const char *label, const ge *p) { uint8_t b[32]; ge_compress(b, p); transcript_append(t, label, b, 32); }
static inline void ts_scalar(transcript *t, const char *label, const sc *s) { uint8_t b[32]; sc_tobytes(b, s); transcript_append(t, label, b, 32); }
static inline void ts_challenge(transcript *t, const char *label, sc *out) { uint8_t b[64]; transcript_challenge(t, label, b, 64); sc_from_bytes_wide(out, b); }
/* validate_and_append_point: reject the identity encoding (all zero) */
static inline int ts_validate_point(transcript *t, const char *label, const uint8_t b[32]) {
    uint8_t z = 0; for (int i = 0; i < 32; i++) z |= b[i];
    if (!z) return 0;
    transcript_append(t, label, b, 32); return 1;
}

static inline int ilog2(size_t x) { int l = 0; while (((size_t)1 << l) < x) l++; return l; }

/* ---- inner product proof (A.4). Writes 32*(2 lgN + 2) bytes to out. G,H are consumed. ------- */
static inline void ipp_create(uint8_t *out, transcript *t, const ge *Q, const sc *Hfac /* y^-i */,
                              ge *G, ge *H, sc *a, sc *b, size_t N) {
    transcript_append(t, "dom-sep", (const uint8_t *)"ipp v1", 6);
    transcript_append_u64(t, "n", N);
    size_t n = N; int first = 1;
    sc *ms = (sc *)malloc(sizeof(sc) * (N + 1)); ge *mp = (ge *)malloc(sizeof(ge) * (N + 1));
    while (n > 1) {
        n /= 2;
        sc cL, cR; sc_0(&cL); sc_0(&cR);
        for (size_t i = 0; i < n; i++) { sc_muladd(&cL, &a[i], &b[n + i], &cL); sc_muladd(&cR, &a[n + i], &b[i], &cR); }
        ge L, R;
        /* L = <a_L * Gf_R, G_R> + <b_R * Hf_L, H_L> + c_L Q */
        for (size_t i = 0; i < n; i++) {
            ms[i] = a[i]; mp[i] = G[n + i];
            if (first) sc_mul(&ms[n + i], &b[n + i], &Hfac[i]); else ms[n + i] = b[n + i];
            mp[n + i] = H[i];
        }
        ms[2 * n] = cL; mp[2 * n] = *Q; ge_msm(&L, ms, mp, 2 * n + 1);
        for (size_t i = 0; i < n; i++) {
            ms[i] = a[n + i]; mp[i] = G[i];
            if (first) sc_mul(&ms[n + i], &b[i], &Hfac[n + i]); else ms[n + i] = b[i];
            mp[n + i] = H[n + i];
        }
        ms[2 * n] = cR; mp[2 * n] = *Q; ge_msm(&R, ms, mp, 2 * n + 1);
        ge_compress(out, &L); ge_compress(out + 32, &R);
        transcript_append(t, "L", out, 32); transcript_append(t, "R", out + 32, 32); out += 64;
        sc u, ui; ts_challenge(t, "u", &u); sc_invert(&ui, &u);
        for (size_t i = 0; i < n; i++) {
            sc t0, t1;
            sc_mul(&t0, &a[i], &u); sc_mul(&t1, &ui, &a[n + i]); sc_add(&a[i], &t0, &t1);
            sc_mul(&t0, &b[i], &ui); sc_mul(&t1, &u, &b[n + i]); sc_add(&b[i], &t0, &t1);
            ge_double_scalarmult(&G[i], &ui, &G[i], &u, &G[n + i]);        /* G_factors == 1 */
            if (first) { sc_mul(&t0, &u, &Hfac[i]); sc_mul(&t1, &ui, &Hfac[n + i]); ge_double_scalarmult(&H[i], &t0, &H[i], &t1, &H[n + i]); }
            else ge_double_scalarmult(&H[i], &u, &H[i], &ui, &H[n + i]);
        }
        first = 0;
    }
    sc_tobytes(out, &a[0]); sc_tobytes(out + 32, &b[0]);
    free(ms); free(mp);
}

/* proof length in bytes for aggregated size N = n*m */
static inline size_t rp_proof_len(size_t N) { return 32 * (9 + 2 * (size_t)ilog2(N)); }

/* ---- RangeProof::prove_multiple_with_rng (A.3).  values < 2^n, m = power of two.
 * proof_out: rp_proof_len(n*m) bytes; V_out: m*32 bytes compressed commitments.
 * returns 0 ok, -7 invalid bitsize, -2 invalid aggregation ------------------------------------ */
/* tx_bl_shift (nullable, tests only): added to t_x_blinding before it is absorbed -- an otherwise honest proof whose verification equation
 * is off by exactly -c shift B_blinding (the adaptive-forgery tests of the batched verifier) */
static inline int rp_prove_multiple_ex(uint8_t *proof_out, uint8_t *V_out, const bp_gens_t *bg, const pc_gens_t *pc,
                                       transcript *t, const uint64_t *values, const sc *blindings, int m, int n, rng_t *rng, const sc *tx_bl_shift) {
    if (!(n == 8 || n == 16 || n == 32 || n == 64)) return -7;
    if (m <= 0 || (m & (m - 1)) || bg->n < n || bg->m < m) return -2;
    size_t N = (size_t)n * m;
    transcript_append(t, "dom-sep", (const uint8_t *)"rangeproof v1", 13);
    transcript_append_u64(t, "n", n); transcript_append_u64(t, "m", m);
    sc *sL = (sc *)malloc(sizeof(sc) * N), *sR = (sc *)malloc(sizeof(sc) * N);
    sc *a_bl = (sc *)malloc(sizeof(sc) * m), *s_bl = (sc *)malloc(sizeof(sc) * m);
    sc *t1_bl = (sc *)malloc(sizeof(sc) * m), *t2_bl = (sc *)malloc(sizeof(sc) * m);
    ge A, S, Aj, Sj; ge_identity(&A); ge_identity(&S);
    sc *ms = (sc *)malloc(sizeof(sc) * (2 * n + 1)); ge *mp = (ge *)malloc(sizeof(ge) * (2 * n + 1));
    for (int j = 0; j < m; j++) {                       /* Party::new + assign_position_with_rng */
        sc v; sc_from_u64(&v, values[j]);
        ge V; pc_commit(&V, pc, &v, &blindings[j]); ge_compress(V_out + 32 * j, &V);
        const ge *Gj = bg->G + (size_t)j * bg->n, *Hj = bg->H + (size_t)j * bg->n;
        rng_scalar(rng, &a_bl[j]);
        ge_scalarmult(&Aj, &a_bl[j], &pc->B_blinding);
        for (int i = 0; i < n; i++) { if ((values[j] >> i) & 1) ge_add(&Aj, &Aj, &Gj[i]); else ge_sub(&Aj, &Aj, &Hj[i]); }
        rng_scalar(rng, &s_bl[j]);
        for (int i = 0; i < n; i++) rng_scalar(rng, &sL[(size_t)j * n + i]);
        for (int i = 0; i < n; i++) rng_scalar(rng, &sR[(size_t)j * n + i]);
        ms[0] = s_bl[j]; mp[0] = pc->B_blinding;
        for (int i = 0; i < n; i++) { ms[1 + i] = sL[(size_t)j * n + i]; mp[1 + i] = Gj[i]; ms[1 + n + i] = sR[(size_t)j * n + i]; mp[1 + n + i] = Hj[i]; }
        ge_msm_straus(&Sj, ms, mp, 2 * n + 1);
        ge_add(&A, &A, &Aj); ge_add(&S, &S, &Sj);
    }
    for (int j = 0; j < m; j++) transcript_append(t, "V", V_out + 32 * j, 32);
    uint8_t *o = proof_out;
    ge_compress(o, &A); transcript_append(t, "A", o, 32); o += 32;
    ge_compress(o, &S); transcript_append(t, "S", o, 32); o += 32;
    sc y, z; ts_challenge(t, "y", &y); ts_challenge(t, "z", &z);
    /* per-party polynomials */
    sc *l0 = (sc *)malloc(sizeof(sc) * N), *r0 = (sc *)malloc(sizeof(sc) * N), *r1 = (sc *)malloc(sizeof(sc) * N);
    sc zz, one, two; sc_mul(&zz, &z, &z); sc_from_u64(&one, 1); sc_from_u64(&two, 2);
    sc t1s, t2s, t0s; sc_0(&t0s); sc_0(&t1s); sc_0(&t2s);
    sc exp_y; sc_from_u64(&exp_y, 1);
    sc offset_z; sc_from_u64(&offset_z, 1);               /* z^j */
    sc *offset_zz = (sc *)malloc(sizeof(sc) * m);
    ge T1, T2, Tj; ge_identity(&T1); ge_identity(&T2);
    for (int j = 0; j < m; j++) {
        sc_mul(&offset_zz[j], &zz, &offset_z);
        sc exp_2; sc_from_u64(&exp_2, 1);
        sc t0, t1, t2; sc_0(&t0); sc_0(&t1); sc_0(&t2);
        for (int i = 0; i < n; i++) {
            size_t k = (size_t)j * n + i;
            sc aL, aR, tmp; sc_from_u64(&aL, (values[j] >> i) & 1); sc_sub(&aR, &aL, &one);
            sc_sub(&l0[k], &aL, &z);
            sc_add(&tmp, &aR, &z); sc_mul(&r0[k], &exp_y, &tmp); sc_mul(&tmp, &offset_zz[j], &exp_2); sc_add(&r0[k], &r0[k], &tmp);
            sc_mul(&r1[k], &exp_y, &sR[k]);
            sc_muladd(&t0, &l0[k], &r0[k], &t0); sc_muladd(&t2, &sL[k], &r1[k], &t2);
            sc l01, r01; sc_add(&l01, &l0[k], &sL[k]); sc_add(&r01, &r0[k], &r1[k]); sc_muladd(&t1, &l01, &r01, &t1);
            sc_mul(&exp_y, &exp_y, &y); sc_add(&exp_2, &exp_2, &exp_2);
        }
        sc_sub(&t1, &t1, &t0); sc_sub(&t1, &t1, &t2);
        rng_scalar(rng, &t1_bl[j]); rng_scalar(rng, &t2_bl[j]);
        pc_commit(&Tj, pc, &t1, &t1_bl[j]); ge_add(&T1, &T1, &Tj);
        pc_commit(&Tj, pc, &t2, &t2_bl[j]); ge_add(&T2, &T2, &Tj);
        sc_add(&t0s, &t0s, &t0); sc_add(&t1s, &t1s, &t1); sc_add(&t2s, &t2s, &t2);
        sc_mul(&offset_z, &offset_z, &z);
    }
    ge_compress(o, &T1); transcript_append(t, "T_1", o, 32); o += 32;
    ge_compress(o, &T2); transcript_append(t, "T_2", o, 32); o += 32;
    sc x; ts_challenge(t, "x", &x);
    sc xx; sc_mul(&xx, &x, &x);
    sc t_x, t_x_bl, e_bl, tmp; sc_0(&t_x_bl); sc_0(&e_bl);
    sc_mul(&tmp, &t1s, &x); sc_add(&t_x, &t0s, &tmp); sc_mul(&tmp, &t2s, &xx); sc_add(&t_x, &t_x, &tmp);
    sc *l = l0, *r = r0;
    for (int j = 0; j < m; j++) {
        sc_muladd(&t_x_bl, &offset_zz[j], &blindings[j], &t_x_bl);
        sc_muladd(&t_x_bl, &t1_bl[j], &x, &t_x_bl); sc_muladd(&t_x_bl, &t2_bl[j], &xx, &t_x_bl);
        sc_add(&e_bl, &e_bl, &a_bl[j]); sc_muladd(&e_bl, &s_bl[j], &x, &e_bl);
    }
    for (size_t k = 0; k < N; k++) { sc_muladd(&l[k], &sL[k], &x, &l0[k]); sc_muladd(&r[k], &r1[k], &x, &r0[k]); }
    sc_tobytes(o, &t_x); transcript_append(t, "t_x", o, 32); o += 32;
    if (tx_bl_shift) sc_add(&t_x_bl, &t_x_bl, tx_bl_shift);
    sc_tobytes(o, &t_x_bl); transcript_append(t, "t_x_blinding", o, 32); o += 32;
    sc_tobytes(o, &e_bl); transcript_append(t, "e_blinding", o, 32); o += 32;
    sc w; ts_challenge(t, "w", &w);
    ge Q; ge_scalarmult(&Q, &w, &pc->B);
    sc yinv; sc_invert(&yinv, &y);
    sc *Hfac = r1; sc_from_u64(&Hfac[0], 1); for (size_t k = 1; k < N; k++) sc_mul(&Hfac[k], &Hfac[k - 1], &yinv);
    ge *G = (ge *)malloc(sizeof(ge) * N), *H = (ge *)malloc(sizeof(ge) * N);
    for (int j = 0; j < m; j++) { memcpy(G + (size_t)j * n, bg->G + (size_t)j * bg->n, sizeof(ge) * n); memcpy(H + (size_t)j * n, bg->H + (size_t)j * bg->n, sizeof(ge) * n); }
    ipp_create(o, t, &Q, Hfac, G, H, l, r, N);
    free(G); free(H); free(l0); free(r0); free(r1); free(offset_zz); free(ms); free(mp);
    free(sL); free(sR); free(a_bl); free(s_bl); free(t1_bl); free(t2_bl);
    return 0;
}

static inline int rp_prove_multiple(uint8_t *proof_out, uint8_t *V_out, const bp_gens_t *bg, const pc_gens_t *pc,
                                    transcript *t, const uint64_t *values, const sc *blindings, int m, int n, rng_t *rng) {
    return rp_prove_multiple_ex(proof_out, V_out, bg, pc, t, values, blindings, m, n, rng, NULL);
}

/* ---- RangeProof::from_bytes + verify_multiple_with_rng (A.3).
 * returns 1 accept, 0 VerificationError, -1 FormatError, -7 InvalidBitsize, -3 InvalidGeneratorsLength */
static inline int rp_verify_multiple(const uint8_t *proof, size_t proof_len, const uint8_t *V, const bp_gens_t *bg,
                                     const pc_gens_t *pc, transcript *t, int m, int n, rng_t *rng) {
    if (proof_len % 32 || proof_len < 7 * 32) return -1;
    size_t ne = proof_len / 32 - 7;                      /* ipp elements */
    if (ne < 2 || (ne - 2) % 2) return -1;
    size_t lg = (ne - 2) / 2; if (lg >= 32) return -1;
    sc t_x, t_x_bl, e_bl, a, b;
    if (!sc_from_canonical_bytes(&t_x, proof + 128) || !sc_from_canonical_bytes(&t_x_bl, proof + 160) ||
        !sc_from_canonical_bytes(&e_bl, proof + 192)) return -1;
    const uint8_t *ipp = proof + 224;
    if (!sc_from_canonical_bytes(&a, ipp + 64 * lg) || !sc_from_canonical_bytes(&b, ipp + 64 * lg + 32)) return -1;
    if (!(n == 8 || n == 16 || n == 32 || n == 64)) return -7;
    if (bg->n < n || bg->m < m) return -3;
    size_t N = (size_t)n * m;
    transcript_append(t, "dom-sep", (const uint8_t *)"rangeproof v1", 13);
    transcript_append_u64(t, "n", n); transcript_append_u64(t, "m", m);
    for (int j = 0; j < m; j++) transcript_append(t, "V", V + 32 * j, 32);
    if (!ts_validate_point(t, "A", proof) || !ts_validate_point(t, "S", proof + 32)) return 0;
    sc y, z; ts_challenge(t, "y", &y); ts_challenge(t, "z", &z);
    if (!ts_validate_point(t, "T_1", proof + 64) || !ts_validate_point(t, "T_2", proof + 96)) return 0;
    sc x; ts_challenge(t, "x", &x);
    transcript_append(t, "t_x", proof + 128, 32); transcript_append(t, "t_x_blinding", proof + 160, 32);
    transcript_append(t, "e_blinding", proof + 192, 32);
    sc w; ts_challenge(t, "w", &w);
    sc c; rng_scalar(rng, &c);
    /* verification_scalars */
    if (N != ((size_t)1 << lg)) return 0;
    transcript_append(t, "dom-sep", (const uint8_t *)"ipp v1", 6); transcript_append_u64(t, "n", N);
    sc *u_sq = (sc *)malloc(sizeof(sc) * (lg + 1)), *u_inv_sq = (sc *)malloc(sizeof(sc) * (lg + 1));
    sc allinv; sc_from_u64(&allinv, 1);
    for (size_t k = 0; k < lg; k++) {
        if (!ts_validate_point(t, "L", ipp + 64 * k) || !ts_validate_point(t, "R", ipp + 64 * k + 32)) { free(u_sq); free(u_inv_sq); return 0; }
        sc u, ui; ts_challenge(t, "u", &u); sc_invert(&ui, &u);
        sc_mul(&allinv, &allinv, &ui); sc_mul(&u_sq[k], &u, &u); sc_mul(&u_inv_sq[k], &ui, &ui);
    }
    sc *s = (sc *)malloc(sizeof(sc) * N);
    s[0] = allinv;
    for (size_t i = 1; i < N; i++) { int lgi = 0; while (((size_t)2 << lgi) <= i) lgi++; size_t k = (size_t)1 << lgi; sc_mul(&s[i], &s[i - k], &u_sq[(lg - 1) - lgi]); }
    size_t npts = 4 + 2 * lg + 2 + 2 * N + m;
    sc *ms = (sc *)malloc(sizeof(sc) * npts); ge *mp = (ge *)malloc(sizeof(ge) * npts);
    size_t q = 0; int ok = 1;
    sc zz, minus_z, cx, tmp; sc_mul(&zz, &z, &z); sc_neg(&minus_z, &z); sc_mul(&cx, &c, &x);
    sc_from_u64(&ms[q], 1); ok &= ge_decompress(&mp[q++], proof);
    ms[q] = x; ok &= ge_decompress(&mp[q++], proof + 32);
    ms[q] = cx; ok &= ge_decompress(&mp[q++], proof + 64);
    sc_mul(&ms[q], &cx, &x); ok &= ge_decompress(&mp[q++], proof + 96);
    for (size_t k = 0; k < lg; k++) { ms[q] = u_sq[k]; ok &= ge_decompress(&mp[q++], ipp + 64 * k); }
    for (size_t k = 0; k < lg; k++) { ms[q] = u_inv_sq[k]; ok &= ge_decompress(&mp[q++], ipp + 64 * k + 32); }
    sc_mul(&tmp, &c, &t_x_bl); sc_add(&tmp, &tmp, &e_bl); sc_neg(&ms[q], &tmp); mp[q++] = pc->B_blinding;
    /* delta(n,m,y,z) = (z - z^2) sum_{i<N} y^i - z^3 (2^n - 1) sum_{j<m} z^j */
    sc sum_y, ey, sum_z, ez, sum_2, delta; sc_0(&sum_y); sc_from_u64(&ey, 1); sc_0(&sum_z); sc_from_u64(&ez, 1);
    for (size_t i = 0; i < N; i++) { sc_add(&sum_y, &sum_y, &ey); sc_mul(&ey, &ey, &y); }
    for (int j = 0; j < m; j++) { sc_add(&sum_z, &sum_z, &ez); sc_mul(&ez, &ez, &z); }
    sc_from_u64(&sum_2, n == 64 ? ~0ULL : ((1ULL << n) - 1));
    sc_sub(&delta, &z, &zz); sc_mul(&delta, &delta, &sum_y);
    sc_mul(&tmp, &zz, &z); sc_mul(&tmp, &tmp, &sum_2); sc_mul(&tmp, &tmp, &sum_z); sc_sub(&delta, &delta, &tmp);
    sc bs, ab; sc_mul(&ab, &a, &b); sc_sub(&bs, &t_x, &ab); sc_mul(&bs, &w, &bs);
    sc_sub(&tmp, &delta, &t_x); sc_mul(&tmp, &c, &tmp); sc_add(&ms[q], &bs, &tmp); mp[q++] = pc->B;
    for (int j = 0; j < m; j++) for (int i = 0; i < n; i++) { size_t k = (size_t)j * n + i; sc_mul(&tmp, &a, &s[k]); sc_sub(&ms[q], &minus_z, &tmp); mp[q++] = bg->G[(size_t)j * bg->n + i]; }
    sc yinv, eyi, ezj; sc_invert(&yinv, &y); sc_from_u64(&eyi, 1); sc_from_u64(&ezj, 1);
    for (int j = 0; j < m; j++) {
        sc e2; sc_from_u64(&e2, 1);
        for (int i = 0; i < n; i++) {
            size_t k = (size_t)j * n + i;
            sc z2, bsv; sc_mul(&z2, &ezj, &e2); sc_mul(&z2, &zz, &z2);            /* zz * z^j 2^i */
            sc_mul(&bsv, &b, &s[N - 1 - k]); sc_sub(&z2, &z2, &bsv); sc_mul(&z2, &eyi, &z2);
            sc_add(&ms[q], &z, &z2); mp[q++] = bg->H[(size_t)j * bg->n + i];
            sc_mul(&eyi, &eyi, &yinv); sc_add(&e2, &e2, &e2);
        }
        sc_mul(&ezj, &ezj, &z);
    }
    sc_from_u64(&ezj, 1);
    for (int j = 0; j < m; j++) { sc_mul(&tmp, &c, &zz); sc_mul(&ms[q + j], &tmp, &ezj); sc_mul(&ezj, &ezj, &z); }
    { int okv = 1;
#pragma omp parallel for schedule(static) reduction(&: okv) if (m >= 4096)
      for (int j = 0; j < m; j++) okv &= ge_decompress(&mp[q + j], V + 32 * j);
      ok &= okv; q += m; }
    int res = 0;
    if (ok) { ge chk; ge_msm(&chk, ms, mp, npts); res = ge_is_identity(&chk); }
    free(ms); free(mp); free(s); free(u_sq); free(u_inv_sq);
    return res;
}

/* ---- the transcript of rp_verify_multiple alone, replayed over every point also when one is the identity encoding (the batched verifier still
 * draws its challenges then and rejects the chunk separately).  out_chal: y z x w u_0 .. u_(lg-1), 32 bytes each; out_digest: the 32-byte
 * "rofl-batch" challenge drawn after a and b, the per-chunk digest the batched verifier keys its weights from (DESIGN.md §2).
 * returns 1 when every point of the proof is a non-identity encoding, 0 when one is the identity, -1 on a malformed length */
static inline int rp_challenges(const uint8_t *proof, size_t proof_len, const uint8_t *V, transcript *t, int m, int n, uint8_t *out_chal, uint8_t out_digest[32]) {
    if (proof_len % 32 || proof_len < 7 * 32) return -1;
    size_t ne = proof_len / 32 - 7;
    if (ne < 2 || (ne - 2) % 2) return -1;
    size_t lg = (ne - 2) / 2; if (lg >= 32) return -1;
    const uint8_t *ipp = proof + 224;
    int ok = 1; sc ch; int q = 0;
#define RPC_POINT(label, b) do { uint8_t z_ = 0; for (int i_ = 0; i_ < 32; i_++) z_ |= (b)[i_]; ok &= z_ != 0; transcript_append(t, label, b, 32); } while (0)
#define RPC_CHAL(label) do { ts_challenge(t, label, &ch); sc_tobytes(out_chal + 32 * q++, &ch); } while (0)
    transcript_append(t, "dom-sep", (const uint8_t *)"rangeproof v1", 13);
    transcript_append_u64(t, "n", n); transcript_append_u64(t, "m", m);
    for (int j = 0; j < m; j++) transcript_append(t, "V", V + 32 * j, 32);
    RPC_POINT("A", proof); RPC_POINT("S", proof + 32); RPC_CHAL("y"); RPC_CHAL("z");
    RPC_POINT("T_1", proof + 64); RPC_POINT("T_2", proof + 96); RPC_CHAL("x");
    transcript_append(t, "t_x", proof + 128, 32); transcript_append(t, "t_x_blinding", proof + 160, 32); transcript_append(t, "e_blinding", proof + 192, 32);
    RPC_CHAL("w");
    transcript_append(t, "dom-sep", (const uint8_t *)"ipp v1", 6); transcript_append_u64(t, "n", (uint64_t)n * m);
    for (size_t k = 0; k < lg; k++) { RPC_POINT("L", ipp + 64 * k); RPC_POINT("R", ipp + 64 * k + 32); RPC_CHAL("u"); }
    transcript_append(t, "a", ipp + 64 * lg, 32); transcript_append(t, "b", ipp + 64 * lg + 32, 32);
    transcript_challenge(t, "rofl-batch", out_digest, 32);
#undef RPC_POINT
#undef RPC_CHAL
    return ok;
}
#endif
