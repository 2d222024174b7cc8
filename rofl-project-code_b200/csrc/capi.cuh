// extern "C" entry points declared in include/rofl_b200.h.  Host-buffer variants stage through device scratch and call
// the same engine functions as the _dev variants.
#pragma once
#include "engine.cuh"
#include "../../include/rofl_b200.h"

struct rofl_ctx { rofl_engine e; };
static thread_local std::string g_last_error;
// every entry point may be called from any host thread: bind that thread to the context's GPU first
#define API_TRY if (!c) return ROFL_ERR_ARGS; try { rt_set_device(c->e.device);
#define API_CATCH } catch (const std::exception &ex) { g_last_error = ex.what(); return ROFL_ERR_CUDA; }

extern "C" const char *rofl_last_error(void) { return g_last_error.c_str(); }
extern "C" void rofl_set_host_threads(rofl_ctx *c, int n) { if (c && n > 0) c->e.host_threads = n; }
extern "C" int rofl_set_option(rofl_ctx *c, const char *name, long value) {
    if (!c || !name) return ROFL_ERR_ARGS;
    try { rt_set_device(c->e.device); } catch (...) { return ROFL_ERR_CUDA; }
    std::string n(name);
    if (n == "use_rt") c->e.use_rt = value != 0;
    else if (n == "rt_unfold") c->e.rt_unfold = (int)std::max<long>(0, std::min<long>(6, value));
    else if (n == "groups") c->e.groups = (int)std::max<long>(1, std::min<long>(ROFL_MAX_GROUPS, value));
    else if (n == "rt_bits") { c->e.rt_bits = (int)std::max<long>(8, std::min<long>(RT_MAX_BITS, value)); engine_drop_rt(c->e); }      // the cached tables of the device are rebuilt at the new radix on next use
    else if (n == "drop_tables") engine_drop_rt(c->e);
    else if (n == "trim") rt_trim();                                                  // hand the cached scratch blocks of this device back to CUDA
    else if (n == "frozen") c->e.use_frz = value != 0;
    else if (n == "tail_np") c->e.tail_np = (int)std::max<long>(0, std::min<long>(TAIL_MAX_F / 2, value));
    else if (n == "tail_batch_mb") c->e.tail_batch_mb = (int)std::max<long>(1, std::min<long>(65536, value));
    else if (n == "tail_ncta") c->e.tail_ncta = value >= 8 ? 8 : value >= 4 ? 4 : value >= 2 ? 2 : 1;
    else if (n == "rt_per") c->e.rt_per = (int)std::max<long>(0, std::min<long>(64, value));
    else if (n == "nt_unfold") c->e.nt_unfold = (int)std::max<long>(0, std::min<long>(4, value));
    else if (n == "nt_unfold_min") c->e.nt_unfold_min = (int)std::max<long>(2, std::min<long>(1 << 30, value));
    else if (n == "ts_host_m") c->e.ts_host_m = (int)std::max<long>(0, std::min<long>(1 << 30, value));
    else if (n == "max_lanes") c->e.max_lanes = (int)std::max<long>(1, std::min<long>(64, value));
    else if (n == "sigma_rlc_terms") c->e.sigma_rlc_terms = (size_t)std::max<long>(1, std::min<long>(1L << 24, value));
    else if (n == "crp_batch_terms") c->e.crp_batch_terms = (size_t)std::max<long>(1, std::min<long>(1L << 24, value));
    else return ROFL_ERR_ARGS;
    return ROFL_OK;
}
extern "C" size_t rofl_next_pow2(size_t v) { return next_pow2_sz(v); }
extern "C" size_t rofl_range_proof_len(size_t N) { return 32 * (9 + 2 * (size_t)ilog2_sz(N)); }
extern "C" void rofl_range_proof_shape(size_t D, int range, size_t n_partition, size_t *n_proofs, size_t *proof_len) {
    size_t Dp = next_pow2_sz(D ? D : 1), C = std::min(Dp, n_partition ? n_partition : 1), m = Dp / C;
    if (n_proofs) *n_proofs = C;
    if (proof_len) *proof_len = rofl_range_proof_len((size_t)range * m);
}
extern "C" void rofl_clip_bounds(int range, int n_bits, int frac, float *mn, float *mx) { float m = clip_max_f(range, n_bits, frac); if (mx) *mx = m; if (mn) *mn = -m; }
extern "C" float rofl_l2_clip_bound(int range, int n_bits, int frac) { return l2_clip_max_f(range, n_bits, frac); }
extern "C" void rofl_clip_f32_to_range_vec(const float *v, size_t D, int range, int n_bits, int frac, float *out) {
    float mx = clip_max_f(range, n_bits, frac), mn = -mx;
    for (size_t i = 0; i < D; i++) out[i] = fminf(mx, fmaxf(mn, v[i]));
}
extern "C" void rofl_rnd_scalar_vec(const uint8_t seed[32], size_t D, uint8_t *out) {
    uint8_t key[32]; derive_key(key, seed, DOM_RND_VEC, 0); uint32_t kw[8]; key_words(kw, key);
    for (size_t i = 0; i < D; i++) { sc s; nonce_scalar(s, kw, i); sc_tobytes(out + 32 * i, s); }
}

// element-wise scalar arithmetic mod l on the host (bindings32.rs `add_scalars`, pedersen_ops::generate_cancelling_scalar_vec): op 0 = a + b, 1 = -a
extern "C" int rofl_scalar_ops(int op, const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out) {
    if (!a || !out || (op == 0 && !b) || (op != 0 && op != 1)) return ROFL_ERR_ARGS;
    for (size_t i = 0; i < n; i++) {
        sc x, y, r; sc_from_bytes_mod_order(x, a + 32 * i);
        if (op == 0) { sc_from_bytes_mod_order(y, b + 32 * i); sc_add(r, x, y); } else sc_neg(r, x);
        sc_tobytes(out + 32 * i, r);
    }
    return 0;
}

// host <-> device staging helpers
struct staged_in { dev_buf b; staged_in(const void *h, size_t n, cudaStream_t s) : b(n ? n : 16, s) { if (h && n) rt_h2d(b.p, h, n, s); } };

// device field-arithmetic self test (a32, b32: n raw 256-bit little-endian values; out: n x 6 x 32 canonical encodings)
extern "C" int rofl_field_selftest(rofl_ctx *c, const uint8_t *a32, const uint8_t *b32, size_t n, uint8_t *out) {
    API_TRY
    if (!n) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in da(a32, 32 * n, s), db(b32, 32 * n, s); dev_buf o(192 * n, s);
    LAUNCH(k_field_selftest, dim3((unsigned)((n + 127) / 128)), dim3(128), s, o.as<uint8_t>(), da.b.as<uint8_t>(), db.b.as<uint8_t>(), n);
    rt_d2h(out, o.p, 192 * n, s); rt_sync(s);
    return 0;
    API_CATCH
}
// device scalar-arithmetic self test (a32, b32: n raw 256-bit values; out: n x 3 x 32: a*b mod l, (a mod l)^-1 by division steps and by Fermat)
extern "C" int rofl_scalar_selftest(rofl_ctx *c, const uint8_t *a32, const uint8_t *b32, size_t n, uint8_t *out) {
    API_TRY
    if (!n) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in da(a32, 32 * n, s), db(b32, 32 * n, s); dev_buf o(96 * n, s);
    LAUNCH(k_scalar_selftest, dim3((unsigned)((n + 127) / 128)), dim3(128), s, o.as<uint8_t>(), da.b.as<uint8_t>(), db.b.as<uint8_t>(), n);
    rt_d2h(out, o.p, 96 * n, s); rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_f32_to_scalar_vec(rofl_ctx *c, const float *v, size_t D, int n_bits, int frac, uint8_t *out) {
    API_TRY
    if (!fp_ok(n_bits, frac)) return ROFL_ERR_ARGS;
    if (!D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s); dev_buf o(32 * D, s), fl(sizeof(int), s); rt_memset(fl.p, 0, sizeof(int), s);
    LAUNCH(k_f32_to_scalar, dim3((unsigned)((D + 255) / 256)), dim3(256), s, o.as<uint8_t>(), dv.b.as<float>(), D, n_bits, frac, fl.as<int>());
    int f = 0; rt_d2h(out, o.p, 32 * D, s); rt_d2h(&f, fl.p, sizeof(int), s); rt_sync(s);
    return f ? ROFL_ERR_NAN : 0;
    API_CATCH
}
extern "C" int rofl_scalar_to_f32_vec(rofl_ctx *c, const uint8_t *sc32, size_t D, int n_bits, int frac, float *out) {
    API_TRY
    if (!fp_ok(n_bits, frac)) return ROFL_ERR_ARGS;
    if (!D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in ds(sc32, 32 * D, s); dev_buf o(4 * D, s);
    LAUNCH(k_scalar_to_f32, dim3((unsigned)((D + 255) / 256)), dim3(256), s, o.as<float>(), ds.b.as<uint8_t>(), D, n_bits, frac);
    rt_d2h(out, o.p, 4 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_commit_dev(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, uint8_t *L, uint8_t *R) {
    API_TRY return engine_commit(c->e, v, blind, D, n_bits, frac, L, R); API_CATCH
}
extern "C" int rofl_commit(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, uint8_t *L, uint8_t *R) {
    API_TRY
    if (!D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s), db(blind, blind ? 32 * D : 0, s); dev_buf dL(32 * D, s), dR(32 * D, s);
    int rc = engine_commit(c->e, dv.b.as<float>(), blind ? db.b.as<uint8_t>() : nullptr, D, n_bits, frac, dL.as<uint8_t>(), (R && blind) ? dR.as<uint8_t>() : nullptr);
    if (rc) return rc;
    rt_d2h(L, dL.p, 32 * D, s); if (R && blind) rt_d2h(R, dR.p, 32 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_range_prove_dev(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int range, size_t P, int n_bits, int frac, const uint8_t seed[32],
                                    uint8_t *proofs, size_t *plen, size_t *np, uint8_t *commits) {
    API_TRY
    size_t a = 0, b = 0;
    int rc = engine_range_prove(c->e, v, blind, D, range, P, n_bits, frac, seed, proofs, &a, &b, commits);
    if (plen) *plen = a; if (np) *np = b;
    return rc;
    API_CATCH
}
extern "C" int rofl_range_prove(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int range, size_t P, int n_bits, int frac, const uint8_t seed[32],
                                uint8_t *proofs, size_t *plen, size_t *np, uint8_t *commits) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s), db(blind, 32 * D, s); dev_buf dC(32 * D, s);
    size_t a = 0, b = 0;
    int rc = engine_range_prove(c->e, dv.b.as<float>(), db.b.as<uint8_t>(), D, range, P, n_bits, frac, seed, proofs, &a, &b, dC.as<uint8_t>());
    if (plen) *plen = a; if (np) *np = b;
    if (rc) return rc;
    rt_d2h(commits, dC.p, 32 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_range_verify_dev(rofl_ctx *c, const uint8_t *proofs, size_t plen, size_t np, const uint8_t *commits, size_t D, int range, const uint8_t seed[32]) {
    API_TRY return engine_range_verify(c->e, proofs, plen, np, commits, D, range, seed); API_CATCH
}
extern "C" int rofl_range_verify(rofl_ctx *c, const uint8_t *proofs, size_t plen, size_t np, const uint8_t *commits, size_t D, int range, const uint8_t seed[32]) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e);
    staged_in dc(commits, 32 * D, lg.s());
    return engine_range_verify(c->e, proofs, plen, np, dc.b.as<uint8_t>(), D, range, seed);
    API_CATCH
}
// chunk-sharded variants (multi-GPU: chunk c of an update goes to GPU c mod G, SURVEY.md 8e)
extern "C" int rofl_range_prove_shard(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D_shard, size_t chunk_len, size_t chunk_begin, size_t n_chunks, int range,
                                      int n_bits, int frac, const uint8_t seed[32], uint8_t *proofs, size_t *plen, uint8_t *commits) {
    API_TRY
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D_shard, s), db(blind, 32 * D_shard, s); dev_buf dC(32 * (D_shard ? D_shard : 1), s);
    shard_spec sh = {chunk_len, chunk_begin, n_chunks};
    size_t a = 0, b = 0;
    int rc = engine_range_prove(c->e, dv.b.as<float>(), db.b.as<uint8_t>(), D_shard, range, 0, n_bits, frac, seed, proofs, &a, &b, dC.as<uint8_t>(), &sh);
    if (plen) *plen = a;
    if (rc) return rc;
    if (D_shard) rt_d2h(commits, dC.p, 32 * D_shard, s);
    rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_range_verify_shard(rofl_ctx *c, const uint8_t *proofs, size_t plen, size_t n_chunks, const uint8_t *commits, size_t D_shard, size_t chunk_len, size_t chunk_begin,
                                       int range, const uint8_t seed[32]) {
    API_TRY
    lane_guard lg(c->e);
    staged_in dc(commits, 32 * D_shard, lg.s());
    shard_spec sh = {chunk_len, chunk_begin, n_chunks};
    return engine_range_verify(c->e, proofs, plen, n_chunks, dc.b.as<uint8_t>(), D_shard, range, seed, &sh);
    API_CATCH
}
extern "C" int rofl_l2_prove(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int range, int n_bits, int frac, const uint8_t seed[32],
                             uint8_t *proof, size_t *plen, uint8_t *commit) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s), db(blind, 32 * D, s);
    size_t a = 0;
    int rc = engine_l2_prove(c->e, v, dv.b.as<float>(), db.b.as<uint8_t>(), D, range, n_bits, frac, seed, proof, &a, commit);
    if (plen) *plen = a;
    return rc;
    API_CATCH
}
extern "C" int rofl_l2_verify(rofl_ctx *c, const uint8_t *proof, size_t plen, const uint8_t commit[32], int range, const uint8_t seed[32]) {
    API_TRY return engine_l2_verify(c->e, proof, plen, commit, range, seed); API_CATCH
}
// rand_proof_vec (RandProof, 128 B per element over 64-byte ElGamal pairs) and square_rand_proof_vec (SquareRandProof, 192 B over 96-byte commitments)
static int sigma_prove_host(rofl_ctx *c, int kind, const float *v, const uint8_t *vc, const uint8_t *r1, const uint8_t *r2, size_t D, int n_bits, int frac, const uint8_t seed[32],
                            uint8_t *proofs, uint8_t *commits) {
    if (!D) return 0;
    const size_t pw = 32 * sigma_kind_of(kind).pw, cw = 32 * sigma_kind_of(kind).cw;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s), dvc(vc, vc ? 32 * D : 0, s), d1(r1, 32 * D, s), d2(r2, r2 ? 32 * D : 0, s); dev_buf dp(pw * D, s), dc(cw * D, s);
    int rc = engine_sigma_prove(c->e, kind, dv.b.as<float>(), vc ? dvc.b.as<uint8_t>() : nullptr, d1.b.as<uint8_t>(), r2 ? d2.b.as<uint8_t>() : nullptr, D, n_bits, frac, seed, dp.as<uint8_t>(), dc.as<uint8_t>());
    if (rc) return rc;
    rt_d2h(proofs, dp.p, pw * D, s); rt_d2h(commits, dc.p, cw * D, s); rt_sync(s);
    return 0;
}
static int sigma_verify_host(rofl_ctx *c, int kind, const uint8_t *proofs, const uint8_t *commits, size_t D) {
    if (!D) return 1;
    const size_t pw = 32 * sigma_kind_of(kind).pw, cw = 32 * sigma_kind_of(kind).cw;
    lane_guard lg(c->e);
    staged_in dp(proofs, pw * D, lg.s()), dc(commits, cw * D, lg.s());
    return engine_sigma_verify(c->e, kind, dp.b.as<uint8_t>(), dc.b.as<uint8_t>(), D);
}
extern "C" int rofl_rand_prove(rofl_ctx *c, const float *v, const uint8_t *value_com32, const uint8_t *blind32, size_t D, int n_bits, int frac, const uint8_t seed[32],
                               uint8_t *proofs128, uint8_t *pairs64) {
    API_TRY return sigma_prove_host(c, 1, v, value_com32, blind32, nullptr, D, n_bits, frac, seed, proofs128, pairs64); API_CATCH
}
extern "C" int rofl_rand_verify(rofl_ctx *c, const uint8_t *proofs128, const uint8_t *pairs64, size_t D) { API_TRY return sigma_verify_host(c, 1, proofs128, pairs64, D); API_CATCH }
extern "C" int rofl_square_rand_prove(rofl_ctx *c, const float *v, const uint8_t *value_com32, const uint8_t *r1_32, const uint8_t *r2_32, size_t D, int n_bits, int frac,
                                      const uint8_t seed[32], uint8_t *proofs192, uint8_t *commits96) {
    API_TRY return sigma_prove_host(c, 2, v, value_com32, r1_32, r2_32, D, n_bits, frac, seed, proofs192, commits96); API_CATCH
}
extern "C" int rofl_square_rand_verify(rofl_ctx *c, const uint8_t *proofs192, const uint8_t *commits96, size_t D) { API_TRY return sigma_verify_host(c, 2, proofs192, commits96, D); API_CATCH }
// ---- the two optimised encodings end to end (rofl_service/src/flserver/params.rs): client `encrypt`, server `verify` on the wire fields ----------
// EncParamsRangeCompressed::encrypt (params.rs:699-743): range proofs + compressed rand proof.  enc_values = D x 64 (L | R).
extern "C" int rofl_enc_range_compressed_encrypt(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int prove_range, size_t n_partition, int n_bits, int frac,
                                                 const uint8_t seed[32], uint8_t *enc_values64, uint8_t *rand_proof128, uint8_t *range_proofs, size_t *plen, size_t *n_proofs) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    std::vector<float> clipped(D); rofl_clip_f32_to_range_vec(v, D, prove_range, n_bits, frac, clipped.data());                 // :709
    staged_in dv(clipped.data(), 4 * D, s), db(blind, 32 * D, s); dev_buf dC(32 * D, s);
    size_t a = 0, b = 0;
    // the compressed rand proof (helper_prove_existing: one sequential transcript over all D pairs on a host core) as a second caller of the context,
    // beside the range proofs; it commits L = v B + r H itself -- the same points the range proofs publish
    rt_sync(s);
    int rc_crp = 0; std::string err_crp;
    std::thread crp([&] {
        try { rt_set_device(c->e.device); rc_crp = engine_crp_prove(c->e, dv.b.as<float>(), nullptr, db.b.as<uint8_t>(), D, n_bits, frac, seed, rand_proof128, enc_values64); }
        catch (const std::exception &ex) { rc_crp = ROFL_ERR_CUDA; err_crp = ex.what(); }
    });
    struct joiner { std::thread &t; ~joiner() { if (t.joinable()) t.join(); } } jn{crp};
    int rc = engine_range_prove(c->e, dv.b.as<float>(), db.b.as<uint8_t>(), D, prove_range, n_partition, n_bits, frac, seed, range_proofs, &a, &b, dC.as<uint8_t>());
    if (plen) *plen = a; if (n_proofs) *n_proofs = b;
    crp.join();
    if (rc) return rc;
    if (rc_crp == ROFL_ERR_CUDA && !err_crp.empty()) throw std::runtime_error(err_crp);
    return rc_crp;
    API_CATCH
}
// EncModelParams::verify, EncRangeCompressed arm (params.rs:236-256): rand proof over ALL pairs, range proofs over the first
// round(D * check_percentage) Pedersen halves.  1 accept, 0 reject (any Err of the parts is a reject there too), < 0 bad arguments
extern "C" int rofl_enc_range_compressed_verify(rofl_ctx *c, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proof128, const uint8_t *range_proofs, size_t plen,
                                                size_t n_proofs, int prove_range, float check_percentage, const uint8_t seed[32]) {
    API_TRY
    if (!D || !n_proofs) return ROFL_ERR_ARGS;
    int ok = engine_crp_verify(c->e, rand_proof128, enc_values64, D);
    if (ok < 0 && ok != ROFL_ERR_FORMAT && ok != -6) return ok;
    if (ok != 1) return 0;
    const size_t num = (size_t)llroundf((float)D * check_percentage);                                                                   // :243-244
    if (num == 0 || num > D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(enc_values64, 64 * D, s); dev_buf dL(32 * D, s), dR(32 * D, s);
    LAUNCH(k_pairs_split, dim3((unsigned)((D + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dR.as<uint8_t>(), dp.b.as<uint8_t>(), D);
    int rr = engine_range_verify(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), num, prove_range, seed);
    return rr == 1 ? 1 : 0;
    API_CATCH
}
// EncParamsL2Compressed::encrypt (params.rs:797-845): range proofs, the sum-of-squares proof, the compressed rand proof (existing commitments),
// the per-element square proofs; enc_values = D x 96 (L | R | c_sq), square_proofs = D x 160.
extern "C" int rofl_enc_l2_compressed_encrypt(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int prove_range, size_t n_partition, int l2_range, int n_bits, int frac,
                                              const uint8_t seed[32], uint8_t *enc_values96, uint8_t *square_proofs160, uint8_t *rand_proof128, uint8_t *range_proofs, size_t *plen,
                                              size_t *n_proofs, uint8_t *square_range_proof, size_t *sq_plen) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    std::vector<float> clipped(D); rofl_clip_f32_to_range_vec(v, D, prove_range, n_bits, frac, clipped.data());                 // :806
    std::vector<uint8_t> rnd(32 * D); { uint8_t k2[32]; derive_key(k2, seed, DOM_RND_VEC, 1); rofl_rnd_scalar_vec(k2, D, rnd.data()); }   // rand_scalars (:805)
    staged_in dv(clipped.data(), 4 * D, s), db(blind, 32 * D, s), dr(rnd.data(), 32 * D, s); dev_buf dC(32 * D, s), dPairs(64 * D, s), dSp(160 * D, s), dSc(64 * D, s), dEnc(96 * D, s);
    size_t a = 0, b = 0, q = 0;
    // The compressed rand proof (:822-825) absorbs all D pairs into ONE transcript -- 24 000 sequential permutations for 50 000 pairs, ~15 ms of one host
    // core, as in the reference.  It runs as a second caller of this context (its own lane of streams; it commits L = v B + r H itself, the same points
    // the range proofs publish) beside the range / sum / square proofs instead of after them.
    rt_sync(s);                                          // the staged inputs are on the device
    std::vector<uint8_t> pairs(64 * D);
    int rc_crp = 0; std::string err_crp;
    std::thread crp([&] {
        try { rt_set_device(c->e.device); rc_crp = engine_crp_prove(c->e, dv.b.as<float>(), nullptr, db.b.as<uint8_t>(), D, n_bits, frac, seed, rand_proof128, pairs.data()); }
        catch (const std::exception &ex) { rc_crp = ROFL_ERR_CUDA; err_crp = ex.what(); }
    });
    struct joiner { std::thread &t; ~joiner() { if (t.joinable()) t.join(); } } jn{crp};
    int rc = engine_range_prove(c->e, dv.b.as<float>(), db.b.as<uint8_t>(), D, prove_range, n_partition, n_bits, frac, seed, range_proofs, &a, &b, dC.as<uint8_t>());
    if (plen) *plen = a; if (n_proofs) *n_proofs = b;
    if (rc) return rc;
    uint8_t sum_commit[32];
    rc = engine_l2_prove(c->e, clipped.data(), dv.b.as<float>(), dr.b.as<uint8_t>(), D, l2_range, n_bits, frac, seed, square_range_proof, &q, sum_commit);      // :815-821
    if (sq_plen) *sq_plen = q;
    if (rc) return rc;
    rc = engine_square_prove(c->e, dv.b.as<float>(), dC.as<uint8_t>(), db.b.as<uint8_t>(), dr.b.as<uint8_t>(), D, n_bits, frac, seed, dSp.as<uint8_t>(), dSc.as<uint8_t>());   // :826-831
    if (rc) return rc;
    crp.join();
    if (rc_crp == ROFL_ERR_CUDA && !err_crp.empty()) throw std::runtime_error(err_crp);
    if (rc_crp) return rc_crp;
    rt_h2d(dPairs.p, pairs.data(), 64 * D, s);
    LAUNCH(k_join96, dim3((unsigned)((D + 255) / 256)), dim3(256), s, dEnc.as<uint8_t>(), dPairs.as<uint8_t>(), dSc.as<uint8_t>(), D);                           // merge (:774-784)
    rt_d2h(enc_values96, dEnc.p, 96 * D, s); rt_d2h(square_proofs160, dSp.p, 160 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
// EncModelParams::verify, EncL2Compressed arm (params.rs:257-290): square proofs on (c.L, c_sq), range proofs on c.L, the sum proof on sum c_sq.
// (The compressed rand proof is NOT checked by that arm of the reference; rofl_crp_verify is available separately.)
extern "C" int rofl_enc_l2_compressed_verify(rofl_ctx *c, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs160, const uint8_t *range_proofs, size_t plen,
                                             size_t n_proofs, const uint8_t *square_range_proof, size_t sq_plen, int prove_range, int l2_range, const uint8_t seed[32]) {
    API_TRY
    if (!D || !n_proofs) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in de(enc_values96, 96 * D, s), dsp(square_proofs160, 160 * D, s); dev_buf dL(32 * D, s), dSc(64 * D, s), dCsq(32 * D, s), dbad(sizeof(int), s);
    // decode_l2enc_vec (params.rs:560-571): every record must deserialise -- c.L, c_sq and also c.R, which this arm never uses afterwards
    // (SquareRandProofCommitments::from_bytes -> ElGamalPair::from_bytes; the reference unwrap()s = panics, here the message is refused with ROFL_ERR_POINT)
    rt_memset(dbad.p, 0, sizeof(int), s);
    LAUNCH(k_validate_points, dim3((unsigned)((3 * D + 127) / 128)), dim3(128), s, de.b.as<uint8_t>(), (size_t)32, (size_t)0, 3 * D, dbad.as<int>(), (size_t)0);
    LAUNCH(k_split96, dim3((unsigned)((D + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dSc.as<uint8_t>(), dCsq.as<uint8_t>(), de.b.as<uint8_t>(), D);
    int bad = 0; rt_d2h(&bad, dbad.p, sizeof(int), s);
    const int sq = engine_square_verify(c->e, dsp.b.as<uint8_t>(), dSc.as<uint8_t>(), D);               // (synchronises the stream: `bad` is valid afterwards)
    if (bad) return ROFL_ERR_POINT;
    if (sq != 1) return 0;
    const int rr = engine_range_verify(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), D, prove_range, seed);
    if (rr == ROFL_ERR_POINT) return ROFL_ERR_POINT;
    if (rr != 1) return 0;
    uint8_t sum[32];
    if (engine_points_sum(c->e, dCsq.as<uint8_t>(), D, sum) != 0) return ROFL_ERR_POINT;
    return engine_l2_verify(c->e, square_range_proof, sq_plen, sum, l2_range, seed) == 1 ? 1 : 0;
    API_CATCH
}
// ---- the two un-optimised encodings end to end -------------------------------------------------------------------------------------------------
// EncParamsRange::encrypt (params.rs:467-510): range proofs on the clipped values (all of them, or the first round(D * check_percentage)), then one
// RandProof per element over the UNCLIPPED plaintext -- on the range proofs' commitments when everything was range-proved (create_randproof_vec_existing),
// on fresh commitments otherwise (create_randproof_vec).  enc_values = D x 64 (L | R), rand_proofs = D x 128.
extern "C" int rofl_enc_range_encrypt(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int prove_range, size_t n_partition, float check_percentage, int n_bits, int frac,
                                      const uint8_t seed[32], uint8_t *enc_values64, uint8_t *rand_proofs128, uint8_t *range_proofs, size_t *plen, size_t *n_proofs) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    std::vector<float> clipped(D); rofl_clip_f32_to_range_vec(v, D, prove_range, n_bits, frac, clipped.data());                 // :475
    const bool all = check_percentage >= 1.0f;
    const size_t num = all ? D : (size_t)llroundf((float)D * check_percentage);                                                 // :487
    if (num > D) return ROFL_ERR_ARGS;
    staged_in dv(clipped.data(), 4 * D, s), dplain(v, 4 * D, s), db(blind, 32 * D, s); dev_buf dC(32 * D, s), dP(128 * D, s), dE(64 * D, s);
    size_t a = 0, b = 0;
    int rc = engine_range_prove(c->e, dv.b.as<float>(), db.b.as<uint8_t>(), num, prove_range, n_partition, n_bits, frac, seed, range_proofs, &a, &b, dC.as<uint8_t>());
    if (plen) *plen = a; if (n_proofs) *n_proofs = b;
    if (rc) return rc;
    rc = engine_sigma_prove(c->e, 1, dplain.b.as<float>(), all ? dC.as<uint8_t>() : nullptr, db.b.as<uint8_t>(), nullptr, D, n_bits, frac, seed, dP.as<uint8_t>(), dE.as<uint8_t>());   // :498-503
    if (rc) return rc;
    rt_d2h(rand_proofs128, dP.p, 128 * D, s); rt_d2h(enc_values64, dE.p, 64 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
// EncModelParams::verify, EncRange arm (params.rs:186-203): every RandProof, then the range proofs over the first round(D * check_percentage) Pedersen halves
extern "C" int rofl_enc_range_verify(rofl_ctx *c, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proofs128, const uint8_t *range_proofs, size_t plen, size_t n_proofs,
                                     int prove_range, float check_percentage, const uint8_t seed[32]) {
    API_TRY
    if (!D || !n_proofs) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(enc_values64, 64 * D, s), dpf(rand_proofs128, 128 * D, s); dev_buf dL(32 * D, s), dR(32 * D, s);
    const int ok = engine_sigma_verify(c->e, 1, dpf.b.as<uint8_t>(), dp.b.as<uint8_t>(), D);
    if (ok < 0) return 0;                                                                                                      // Err(_) -> false
    const size_t num = (size_t)llroundf((float)D * check_percentage);
    if (num == 0 || num > D) return 0;
    LAUNCH(k_pairs_split, dim3((unsigned)((D + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dR.as<uint8_t>(), dp.b.as<uint8_t>(), D);
    const int rr = engine_range_verify(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), num, prove_range, seed);
    return (ok == 1 && rr == 1) ? 1 : 0;
    API_CATCH
}
// EncParamsL2::encrypt (params.rs:607-646): range proofs, the sum-of-squares proof under fresh rand_scalars, one SquareRandProof per element on the range proofs' commitments.
// enc_values = D x 96 (c.L | c.R | c_sq), square_proofs = D x 192.
extern "C" int rofl_enc_l2_encrypt(rofl_ctx *c, const float *v, const uint8_t *blind, size_t D, int prove_range, size_t n_partition, int l2_range, int n_bits, int frac,
                                   const uint8_t seed[32], uint8_t *enc_values96, uint8_t *square_proofs192, uint8_t *range_proofs, size_t *plen, size_t *n_proofs,
                                   uint8_t *square_range_proof, size_t *sq_plen) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    std::vector<float> clipped(D); rofl_clip_f32_to_range_vec(v, D, prove_range, n_bits, frac, clipped.data());                 // :616
    std::vector<uint8_t> rnd(32 * D); { uint8_t k2[32]; derive_key(k2, seed, DOM_RND_VEC, 1); rofl_rnd_scalar_vec(k2, D, rnd.data()); }   // rand_scalars (:615)
    staged_in dv(clipped.data(), 4 * D, s), db(blind, 32 * D, s), dr(rnd.data(), 32 * D, s); dev_buf dC(32 * D, s), dP(192 * D, s), dE(96 * D, s);
    size_t a = 0, b = 0, q = 0;
    int rc = engine_range_prove(c->e, dv.b.as<float>(), db.b.as<uint8_t>(), D, prove_range, n_partition, n_bits, frac, seed, range_proofs, &a, &b, dC.as<uint8_t>());
    if (plen) *plen = a; if (n_proofs) *n_proofs = b;
    if (rc) return rc;
    uint8_t sum_commit[32];
    rc = engine_l2_prove(c->e, clipped.data(), dv.b.as<float>(), dr.b.as<uint8_t>(), D, l2_range, n_bits, frac, seed, square_range_proof, &q, sum_commit);      // :624-630
    if (sq_plen) *sq_plen = q;
    if (rc) return rc;
    rc = engine_sigma_prove(c->e, 2, dv.b.as<float>(), dC.as<uint8_t>(), db.b.as<uint8_t>(), dr.b.as<uint8_t>(), D, n_bits, frac, seed, dP.as<uint8_t>(), dE.as<uint8_t>());  // :631-637
    if (rc) return rc;
    rt_d2h(square_proofs192, dP.p, 192 * D, s); rt_d2h(enc_values96, dE.p, 96 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
// EncModelParams::verify, EncL2 arm (params.rs:205-233): every SquareRandProof, the range proofs over all c.L, the sum proof over sum c_sq
extern "C" int rofl_enc_l2_verify(rofl_ctx *c, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs192, const uint8_t *range_proofs, size_t plen, size_t n_proofs,
                                  const uint8_t *square_range_proof, size_t sq_plen, int prove_range, int l2_range, const uint8_t seed[32]) {
    API_TRY
    if (!D || !n_proofs) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in de(enc_values96, 96 * D, s), dsp(square_proofs192, 192 * D, s); dev_buf dL(32 * D, s), dSc(64 * D, s), dCsq(32 * D, s);
    const int ok = engine_sigma_verify(c->e, 2, dsp.b.as<uint8_t>(), de.b.as<uint8_t>(), D);
    if (ok < 0) return 0;
    LAUNCH(k_split96, dim3((unsigned)((D + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dSc.as<uint8_t>(), dCsq.as<uint8_t>(), de.b.as<uint8_t>(), D);
    const int rr = engine_range_verify(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), D, prove_range, seed);
    if (rr < 0) return 0;
    uint8_t sum[32];
    if (engine_points_sum(c->e, dCsq.as<uint8_t>(), D, sum) != 0) return 0;
    const int rs = engine_l2_verify(c->e, square_range_proof, sq_plen, sum, l2_range, seed);
    return (ok == 1 && rr == 1 && rs == 1) ? 1 : 0;
    API_CATCH
}
extern "C" int rofl_square_prove_dev(rofl_ctx *c, const float *v, const uint8_t *vc, const uint8_t *r1, const uint8_t *r2, size_t D, int n_bits, int frac,
                                     const uint8_t seed[32], uint8_t *proofs, uint8_t *commits) {
    API_TRY return engine_square_prove(c->e, v, vc, r1, r2, D, n_bits, frac, seed, proofs, commits); API_CATCH
}
extern "C" int rofl_crp_prove(rofl_ctx *c, const float *v, const uint8_t *value_com32, const uint8_t *blind, size_t D, int n_bits, int frac, const uint8_t seed[32],
                              uint8_t *proof128, uint8_t *pairs64) {
    API_TRY
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s), db(blind, 32 * D, s), dc(value_com32, value_com32 ? 32 * D : 0, s);
    return engine_crp_prove(c->e, dv.b.as<float>(), value_com32 ? dc.b.as<uint8_t>() : nullptr, db.b.as<uint8_t>(), D, n_bits, frac, seed, proof128, pairs64);
    API_CATCH
}
extern "C" int rofl_crp_verify(rofl_ctx *c, const uint8_t *proof128, const uint8_t *pairs64, size_t D) {
    API_TRY return engine_crp_verify(c->e, proof128, pairs64, D); API_CATCH
}
extern "C" int rofl_square_prove(rofl_ctx *c, const float *v, const uint8_t *vc, const uint8_t *r1, const uint8_t *r2, size_t D, int n_bits, int frac,
                                 const uint8_t seed[32], uint8_t *proofs, uint8_t *commits) {
    API_TRY
    if (!D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(v, 4 * D, s), dvc(vc, 32 * D, s), d1(r1, 32 * D, s), d2(r2, 32 * D, s); dev_buf dp(160 * D, s), dc(64 * D, s);
    int rc = engine_square_prove(c->e, dv.b.as<float>(), dvc.b.as<uint8_t>(), d1.b.as<uint8_t>(), d2.b.as<uint8_t>(), D, n_bits, frac, seed, dp.as<uint8_t>(), dc.as<uint8_t>());
    if (rc) return rc;
    rt_d2h(proofs, dp.p, 160 * D, s); rt_d2h(commits, dc.p, 64 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_square_verify_dev(rofl_ctx *c, const uint8_t *proofs, const uint8_t *commits, size_t D) {
    API_TRY return engine_square_verify(c->e, proofs, commits, D); API_CATCH
}
extern "C" int rofl_square_verify(rofl_ctx *c, const uint8_t *proofs, const uint8_t *commits, size_t D) {
    API_TRY
    if (!D) return 1;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(proofs, 160 * D, s), dc(commits, 64 * D, s);
    return engine_square_verify(c->e, dp.b.as<uint8_t>(), dc.b.as<uint8_t>(), D);
    API_CATCH
}
extern "C" int rofl_aggregate_dev(rofl_ctx *c, const uint8_t *pts, size_t nc, size_t D, int init, uint8_t *out) {
    API_TRY return engine_aggregate(c->e, pts, nc, D, init, out); API_CATCH
}
extern "C" int rofl_aggregate(rofl_ctx *c, const uint8_t *pts, size_t nc, size_t D, int init, uint8_t *out) {
    API_TRY
    if (!D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(pts, 32 * nc * D, s); dev_buf o(32 * D, s);
    int rc = engine_aggregate(c->e, dp.b.as<uint8_t>(), nc, D, init, o.as<uint8_t>());
    if (rc) return rc;
    rt_d2h(out, o.p, 32 * D, s); rt_sync(s);
    return 0;
    API_CATCH
}
extern "C" int rofl_dlog_dev(rofl_ctx *c, const uint8_t *pts, size_t D, uint64_t ts, int bb, int n_bits, int frac, uint8_t *osc, float *of) {
    API_TRY return engine_dlog(c->e, pts, D, ts, bb, n_bits, frac, osc, of); API_CATCH
}
extern "C" int rofl_dlog(rofl_ctx *c, const uint8_t *pts, size_t D, uint64_t ts, int bb, int n_bits, int frac, uint8_t *osc, float *of) {
    API_TRY
    if (!D) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(pts, 32 * D, s); dev_buf o(32 * D, s), f(4 * D, s);
    int rc = engine_dlog(c->e, dp.b.as<uint8_t>(), D, ts, bb, n_bits, frac, o.as<uint8_t>(), f.as<float>());
    if (osc) rt_d2h(osc, o.p, 32 * D, s); if (of) rt_d2h(of, f.p, 4 * D, s); rt_sync(s);
    return rc;
    API_CATCH
}

// ---- device-resident round accumulator (EncModelParamsAccumulator, params.rs:74-148): one mutex per accumulator serialises its calls,
//      each call runs on a lane of the accumulator's context like every other call
#define ACC_TRY if (!a) return ROFL_ERR_ARGS; try { rt_set_device(a->e->device); std::lock_guard<std::mutex> acc_lk_(a->mu);
extern "C" int rofl_acc_create(rofl_ctx *c, size_t D, int rec_bytes, int init_unity, rofl_acc **out) {
    if (out) *out = nullptr;
    API_TRY
    if (!out || !D || (rec_bytes != 32 && rec_bytes != 64 && rec_bytes != 96) || (init_unity != 0 && init_unity != 1)) return ROFL_ERR_ARGS;
    *out = engine_acc_create(c->e, D, rec_bytes, init_unity);
    return ROFL_OK;
    API_CATCH
}
extern "C" void rofl_acc_destroy(rofl_acc *a) {
    if (!a) return;
    try { rt_set_device(a->e->device); } catch (...) {}
    engine_acc_destroy(a);
}
extern "C" int rofl_acc_reset(rofl_acc *a) {
    ACC_TRY engine_acc_reset(*a); return ROFL_OK; API_CATCH
}
extern "C" size_t rofl_acc_count(const rofl_acc *a) {
    if (!a) return 0;
    std::lock_guard<std::mutex> lk(const_cast<rofl_acc *>(a)->mu); return a->count;
}
extern "C" int rofl_acc_add_dev(rofl_acc *a, const uint8_t *records, size_t n_clients, const int *mask, int *out_added) {
    ACC_TRY
    if (!records) return ROFL_ERR_ARGS;
    return engine_acc_add(*a, records, n_clients, mask, out_added);
    API_CATCH
}
extern "C" int rofl_acc_add(rofl_acc *a, const uint8_t *records, size_t n_clients, const int *mask, int *out_added) {
    ACC_TRY
    if (!records) return ROFL_ERR_ARGS;
    if (!n_clients) return 0;
    lane_guard lg(*a->e);
    staged_in dr(records, (size_t)a->rec_bytes * a->D * n_clients, lg.s());
    return engine_acc_add(*a, dr.b.as<uint8_t>(), n_clients, mask, out_added);
    API_CATCH
}
extern "C" int rofl_acc_export(rofl_acc *a, uint8_t *out) {
    ACC_TRY
    if (!out) return ROFL_ERR_ARGS;
    lane_guard lg(*a->e); cudaStream_t s = lg.s();
    const size_t n = 32 * a->D * a->ncols;
    dev_buf o(n, s);
    engine_acc_export(*a, o.as<uint8_t>());
    rt_d2h(out, o.p, n, s); rt_sync(s);
    return ROFL_OK;
    API_CATCH
}
extern "C" int rofl_acc_extract(rofl_acc *a, uint64_t ts, int bb, int n_bits, int frac, uint8_t *osc, float *of) {
    ACC_TRY
    lane_guard lg(*a->e); cudaStream_t s = lg.s();
    dev_buf o(32 * a->D, s), f(4 * a->D, s);
    int rc = engine_acc_extract(*a, ts, bb, n_bits, frac, o.as<uint8_t>(), f.as<float>());
    if (rc != 0 && rc != ROFL_ERR_DLOG) return rc;
    if (osc) rt_d2h(osc, o.p, 32 * a->D, s); if (of) rt_d2h(of, f.p, 4 * a->D, s); rt_sync(s);
    return rc;
    API_CATCH
}

// ---- server side: all clients of a round in one call (rofl_service/src/flserver/server.rs:516-522,666-667 fans EncModelParams::verify out over a
//      rayon pool, one task per client; on a GPU the clients share ONE batched check instead) ------------------------------------------------------
extern "C" int rofl_range_verify_batch(rofl_ctx *c, const uint8_t *proofs, size_t plen, size_t n_proofs, const uint8_t *commits32, size_t D, size_t n_clients, int range,
                                       const uint8_t seed[32], int *out_ok) {
    API_TRY
    if (!D || !n_clients || !out_ok) return ROFL_ERR_ARGS;
    lane_guard lg(c->e);
    staged_in dc(commits32, 32 * D * n_clients, lg.s());
    return engine_range_verify_batch(c->e, proofs, plen, n_proofs, dc.b.as<uint8_t>(), D, n_clients, range, seed, out_ok);
    API_CATCH
}
// EncModelParams::verify, EncL2Compressed arm (params.rs:257-290), for n_clients messages of the same shape.  out_ok[k]: 1 accept, 0 reject,
// ROFL_ERR_POINT when one of the message's points does not decode.  Every array is client-major.
extern "C" int rofl_enc_l2_compressed_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs160, const uint8_t *range_proofs,
                                                   size_t plen, size_t n_proofs, const uint8_t *square_range_proofs, size_t sq_plen, int prove_range, int l2_range,
                                                   const uint8_t seed[32], int *out_ok) {
    API_TRY
    const size_t K = n_clients;
    if (!D || !n_proofs || !K || !out_ok) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in de(enc_values96, 96 * D * K, s), dsp(square_proofs160, 160 * D * K, s);
    dev_buf dL(32 * D * K, s), dSc(64 * D * K, s), dCsq(32 * D * K, s), dbad(sizeof(int) * K, s), dres(2 * sizeof(int) * K, s);
    std::vector<int> bad(K, 0), res(2 * K), ok_range(K, 0), ok_sum(K, 0);
    for (size_t k = 0; k < K; k++) { res[2 * k] = 1; res[2 * k + 1] = 0; }
    rt_memset(dbad.p, 0, sizeof(int) * K, s); rt_h2d(dres.p, res.data(), sizeof(int) * 2 * K, s);
    LAUNCH(k_validate_points, dim3((unsigned)((3 * D * K + 127) / 128)), dim3(128), s, de.b.as<uint8_t>(), (size_t)32, (size_t)0, 3 * D * K, dbad.as<int>(), 3 * D);
    LAUNCH(k_split96, dim3((unsigned)((D * K + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dSc.as<uint8_t>(), dCsq.as<uint8_t>(), de.b.as<uint8_t>(), D * K);
    sigma_verify_groups(c->e, s, 0, dsp.b.as<uint8_t>(), dSc.as<uint8_t>(), D * K, nullptr, D, dres.as<int>());   // all K x D square proofs in one batched check, else element by element
    // sum_i c_sq,i per client (params.rs:267)
    const int nb = (int)std::max<size_t>(1, std::min<size_t>(64, (D + 127) / 128));
    dev_buf dpart(sizeof(p3_st) * nb * K, s), dbad2(sizeof(int) * K, s), dsum(32 * K, s);
    rt_memset(dbad2.p, 0, sizeof(int) * K, s);
    LAUNCH_COOP(k_points_sum, dim3(nb, (unsigned)K), dim3(128), s, dpart.as<p3_st>(), dCsq.as<uint8_t>(), D, dbad2.as<int>());
    { finalize_args f = {}; f.partial = dpart.as<p3_st>(); f.npartial = nb; f.tabB = c->e.sh->tabB; f.tabH = c->e.sh->tabH; f.out32 = dsum.as<uint8_t>(); f.count = (int)K; run_finalize(s, f); }
    std::vector<uint8_t> sums(32 * K);
    rt_d2h(bad.data(), dbad.p, sizeof(int) * K, s); rt_d2h(res.data(), dres.p, sizeof(int) * 2 * K, s); rt_d2h(sums.data(), dsum.p, 32 * K, s); rt_sync(s);
    int rc = engine_range_verify_batch(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), D, K, prove_range, seed, ok_range.data());
    if (rc < 0) return rc;
    rc = engine_l2_verify_batch(c->e, square_range_proofs, sq_plen, sums.data(), K, l2_range, seed, ok_sum.data());
    if (rc < 0) return rc;
    for (size_t k = 0; k < K; k++) {
        if (bad[k] || ok_range[k] == ROFL_ERR_POINT) out_ok[k] = ROFL_ERR_POINT;
        else out_ok[k] = (res[2 * k] == 1 && res[2 * k + 1] == 0 && ok_range[k] == 1 && ok_sum[k] == 1) ? 1 : 0;
    }
    return 0;
    API_CATCH
}
// K compressed rand proofs (compressed_rand_proof/mod.rs:149-158) in one batched check (engine.cuh, engine_crp_verify_batch).
// out_ok[k] = exactly what rofl_crp_verify(proofs128[k], pairs64[k], D) returns.
extern "C" int rofl_crp_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *proofs128, const uint8_t *pairs64, size_t D, const uint8_t seed[32], int *out_ok) {
    API_TRY return engine_crp_verify_batch(c->e, proofs128, pairs64, nullptr, D, n_clients, seed, out_ok); API_CATCH
}
// EncModelParams::verify, EncRangeCompressed arm (params.rs:236-256), for n_clients messages of one shape: the compressed rand proofs of all
// clients in one batched check, the range proofs over the first round(D * check_percentage) L halves of every client in another
// (engine_range_verify_batch).  The K rand-proof transcripts run on host threads while the range batch runs on this thread.
// out_ok[k] = exactly what rofl_enc_range_compressed_verify(message k, ...) returns (1 / 0).
extern "C" int rofl_enc_range_compressed_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proofs128,
                                                      const uint8_t *range_proofs, size_t plen, size_t n_proofs, int prove_range, float check_percentage,
                                                      const uint8_t seed[32], int *out_ok) {
    API_TRY
    const size_t K = n_clients;
    if (!D || !n_proofs || !out_ok) return ROFL_ERR_ARGS;
    if (!K) return 0;
    if (!enc_values64 || !rand_proofs128) return ROFL_ERR_ARGS;
    const size_t num = (size_t)llroundf((float)D * check_percentage);                                                                   // :243-244
    if (D > CRP_MAX_D || num == 0 || num > D) { for (size_t k = 0; k < K; k++) out_ok[k] = 0; return 0; }
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(enc_values64, 64 * D * K, s); dev_buf dL(32 * num * K, s);
    LAUNCH(k_pairs_gather_L, dim3((unsigned)((num * K + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dp.b.as<uint8_t>(), D, num, K);
    std::vector<int> ok_crp(K, 0), ok_range(K, 0);
    crp_batch b(c->e, s, rand_proofs128, enc_values64, dp.b.as<uint8_t>(), D, K);
    crp_batch_begin(b);
    const int rc = engine_range_verify_batch(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), num, K, prove_range, seed, ok_range.data());
    crp_batch_end(b, seed, ok_crp.data());
    for (size_t k = 0; k < K; k++) out_ok[k] = (rc == 0 && ok_crp[k] == 1 && ok_range[k] == 1) ? 1 : 0;    // a bad range argument is a reject of every message, as there
    return 0;
    API_CATCH
}

// K x D rand proofs (rand_proof_vec::verify_randproof_vec, kind 1) or square-rand proofs (square_rand_proof_vec::verify_l2rangeproof_vec, kind 2)
// in one batched check (engine.cuh, sigma_verify_groups).  out[k] = exactly what sigma_verify_host(kind, proofs k, commits k, D) returns: 1 / 0 / -1.
static int sigma_verify_batch_host(rofl_ctx *c, int kind, size_t K, const uint8_t *proofs, const uint8_t *commits, size_t D, const uint8_t seed[32], int *out) {
    if (!out) return ROFL_ERR_ARGS;
    if (!K) return 0;
    if (!D) { for (size_t k = 0; k < K; k++) out[k] = 1; return 0; }
    if (!proofs || !commits || !seed) return ROFL_ERR_ARGS;
    const size_t pw = 32 * sigma_kind_of(kind).pw, cw = 32 * sigma_kind_of(kind).cw;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(proofs, pw * D * K, s), dc(commits, cw * D * K, s); dev_buf dres(2 * sizeof(int) * K, s);
    std::vector<int> res(2 * K);
    for (size_t k = 0; k < K; k++) { res[2 * k] = 1; res[2 * k + 1] = 0; }
    rt_h2d(dres.p, res.data(), sizeof(int) * 2 * K, s);
    sigma_verify_groups(c->e, s, kind, dp.b.as<uint8_t>(), dc.b.as<uint8_t>(), D * K, seed, D, dres.as<int>());
    rt_d2h(res.data(), dres.p, sizeof(int) * 2 * K, s); rt_sync(s);
    for (size_t k = 0; k < K; k++) out[k] = res[2 * k + 1] ? -1 : res[2 * k] ? 1 : 0;
    return 0;
}
extern "C" int rofl_rand_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *proofs128, const uint8_t *pairs64, size_t D, const uint8_t seed[32], int *out_ok) {
    API_TRY return sigma_verify_batch_host(c, 1, n_clients, proofs128, pairs64, D, seed, out_ok); API_CATCH
}
extern "C" int rofl_square_rand_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *proofs192, const uint8_t *commits96, size_t D, const uint8_t seed[32], int *out_ok) {
    API_TRY return sigma_verify_batch_host(c, 2, n_clients, proofs192, commits96, D, seed, out_ok); API_CATCH
}
// EncModelParams::verify, EncRange arm (params.rs:186-203), for n_clients messages of one shape: the K x D rand proofs in one batched check, the
// range proofs over the first round(D * check_percentage) L halves of every client in another (engine_range_verify_batch).
// out_ok[k] = exactly what rofl_enc_range_verify(message k, ...) returns (1 / 0).
extern "C" int rofl_enc_range_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *enc_values64, size_t D, const uint8_t *rand_proofs128, const uint8_t *range_proofs,
                                           size_t plen, size_t n_proofs, int prove_range, float check_percentage, const uint8_t seed[32], int *out_ok) {
    API_TRY
    const size_t K = n_clients;
    if (!D || !n_proofs || !out_ok) return ROFL_ERR_ARGS;
    if (!K) return 0;
    if (!enc_values64 || !rand_proofs128 || !seed) return ROFL_ERR_ARGS;
    const size_t num = (size_t)llroundf((float)D * check_percentage);
    if (num == 0 || num > D) { for (size_t k = 0; k < K; k++) out_ok[k] = 0; return 0; }
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dpf(rand_proofs128, 128 * D * K, s), dp(enc_values64, 64 * D * K, s); dev_buf dres(2 * sizeof(int) * K, s), dL(32 * num * K, s);
    std::vector<int> res(2 * K), ok_range(K, 0);
    for (size_t k = 0; k < K; k++) { res[2 * k] = 1; res[2 * k + 1] = 0; }
    rt_h2d(dres.p, res.data(), sizeof(int) * 2 * K, s);
    sigma_verify_groups(c->e, s, 1, dpf.b.as<uint8_t>(), dp.b.as<uint8_t>(), D * K, seed, D, dres.as<int>());
    LAUNCH(k_pairs_gather_L, dim3((unsigned)((num * K + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dp.b.as<uint8_t>(), D, num, K);
    rt_d2h(res.data(), dres.p, sizeof(int) * 2 * K, s); rt_sync(s);
    const int rc = engine_range_verify_batch(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), num, K, prove_range, seed, ok_range.data());
    for (size_t k = 0; k < K; k++)                         // a rand-proof format error and a bad range argument are rejects, as there
        out_ok[k] = (rc == 0 && res[2 * k] == 1 && res[2 * k + 1] == 0 && ok_range[k] == 1) ? 1 : 0;
    return 0;
    API_CATCH
}
// EncModelParams::verify, EncL2 arm (params.rs:205-233), for n_clients messages of one shape: the K x D square-rand proofs in one batched check,
// the range proofs over all c.L of every client in another, the sums of c_sq per client, the K sum-of-squares proofs in a third.
// out_ok[k] = exactly what rofl_enc_l2_verify(message k, ...) returns (1 / 0: that arm rejects, rather than refuses, undecodable points).
extern "C" int rofl_enc_l2_verify_batch(rofl_ctx *c, size_t n_clients, const uint8_t *enc_values96, size_t D, const uint8_t *square_proofs192, const uint8_t *range_proofs,
                                        size_t plen, size_t n_proofs, const uint8_t *square_range_proofs, size_t sq_plen, int prove_range, int l2_range,
                                        const uint8_t seed[32], int *out_ok) {
    API_TRY
    const size_t K = n_clients;
    if (!D || !n_proofs || !out_ok) return ROFL_ERR_ARGS;
    if (!K) return 0;
    if (!enc_values96 || !square_proofs192 || !seed) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in de(enc_values96, 96 * D * K, s), dsp(square_proofs192, 192 * D * K, s);
    dev_buf dL(32 * D * K, s), dSc(64 * D * K, s), dCsq(32 * D * K, s), dres(2 * sizeof(int) * K, s);
    std::vector<int> res(2 * K), ok_range(K, 0), ok_sum(K, 0), bad(K, 0);
    for (size_t k = 0; k < K; k++) { res[2 * k] = 1; res[2 * k + 1] = 0; }
    rt_h2d(dres.p, res.data(), sizeof(int) * 2 * K, s);
    sigma_verify_groups(c->e, s, 2, dsp.b.as<uint8_t>(), de.b.as<uint8_t>(), D * K, seed, D, dres.as<int>());
    LAUNCH(k_split96, dim3((unsigned)((D * K + 255) / 256)), dim3(256), s, dL.as<uint8_t>(), dSc.as<uint8_t>(), dCsq.as<uint8_t>(), de.b.as<uint8_t>(), D * K);
    // sum_i c_sq,i per client; a c_sq that does not decode is a reject of its message
    const int nb = (int)std::max<size_t>(1, std::min<size_t>(64, (D + 127) / 128));
    dev_buf dpart(sizeof(p3_st) * nb * K, s), dbad(sizeof(int) * K, s), dsum(32 * K, s);
    rt_memset(dbad.p, 0, sizeof(int) * K, s);
    LAUNCH_COOP(k_points_sum, dim3(nb, (unsigned)K), dim3(128), s, dpart.as<p3_st>(), dCsq.as<uint8_t>(), D, dbad.as<int>());
    { finalize_args f = {}; f.partial = dpart.as<p3_st>(); f.npartial = nb; f.tabB = c->e.sh->tabB; f.tabH = c->e.sh->tabH; f.out32 = dsum.as<uint8_t>(); f.count = (int)K; run_finalize(s, f); }
    std::vector<uint8_t> sums(32 * K);
    rt_d2h(res.data(), dres.p, sizeof(int) * 2 * K, s); rt_d2h(bad.data(), dbad.p, sizeof(int) * K, s); rt_d2h(sums.data(), dsum.p, 32 * K, s); rt_sync(s);
    const int rr = engine_range_verify_batch(c->e, range_proofs, plen, n_proofs, dL.as<uint8_t>(), D, K, prove_range, seed, ok_range.data());
    const int rs = engine_l2_verify_batch(c->e, square_range_proofs, sq_plen, sums.data(), K, l2_range, seed, ok_sum.data());
    for (size_t k = 0; k < K; k++)
        out_ok[k] = (rr == 0 && rs == 0 && res[2 * k] == 1 && res[2 * k + 1] == 0 && ok_range[k] == 1 && !bad[k] && ok_sum[k] == 1) ? 1 : 0;
    return 0;
    API_CATCH
}

// ---- test hooks (tests/test_emul_vs_oracle.py, tests/test_gpu_parity.py, tests/test_msm_kernels.py) -----------------------------------------------
// the warp-cooperative V absorb (ts_kernels.cuh, k_ts_absorbV) against the sequential transcript code for the same m commitments: 0 equal, 1 different
extern "C" int rofl_debug_ts_absorb(rofl_ctx *c, const uint8_t *V32, size_t m, int n, int label_id) {
    API_TRY
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dv(V32, 32 * m, s); dev_buf d_ts(sizeof(transcript), s);
    ts_absorb_args aa = {}; aa.ts = d_ts.as<transcript>(); aa.V32 = dv.b.as<uint8_t>(); aa.m = (uint32_t)m; aa.n = (uint32_t)n; aa.label_id = label_id;
    LAUNCH_COOP(k_ts_absorbV, dim3(1), dim3(TS_THREADS), s, aa);
    transcript got; rt_d2h(&got, d_ts.p, sizeof(transcript), s); rt_sync(s);
    transcript t; transcript_init(t, label_id ? "L2RangeProof" : "RangeProof");
    transcript_append(t, "dom-sep", (const uint8_t *)"rangeproof v1", 13);
    transcript_append_u64(t, "n", (uint64_t)n); transcript_append_u64(t, "m", (uint64_t)m);
    for (size_t j = 0; j < m; j++) transcript_append(t, "V", V32 + 32 * j, 32);
    return (memcmp(t.st, got.st, sizeof(t.st)) || t.pos != got.pos || t.pos_begin != got.pos_begin) ? 1 : 0;
    API_CATCH
}
// the batched square-proof check alone (engine.cuh, sigma_verify_rlc kind 0): 1 = the random linear combination over all D proofs holds and every
// element is well-formed, 0 = it does not or D is below the size threshold (rofl_square_verify then decides element by element).  proofs D x 160,
// commits D x 64, host buffers.
extern "C" int rofl_debug_square_rlc(rofl_ctx *c, const uint8_t *proofs, const uint8_t *commits, size_t D) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    if (D < SIGMA_RLC_MIN) return 0;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(proofs, 160 * D, s), dc(commits, 64 * D, s);
    return sigma_verify_rlc(c->e, s, 0, dp.b.as<uint8_t>(), dc.b.as<uint8_t>(), D, nullptr);
    API_CATCH
}
// the batched compressed-rand-proof check alone (engine.cuh, engine_crp_verify_batch): 1 = the combination over all K proofs held and no proof is
// malformed, 0 = it did not (the verdicts then came from the per-client checks), < 0 as rofl_crp_verify_batch.  Host buffers as there.
extern "C" int rofl_debug_crp_rlc(rofl_ctx *c, size_t n_clients, const uint8_t *proofs128, const uint8_t *pairs64, size_t D, const uint8_t seed[32]) {
    API_TRY
    if (!n_clients || !D || D > CRP_MAX_D) return ROFL_ERR_ARGS;
    std::vector<int> ok(n_clients); int holds = 0;
    const int rc = engine_crp_verify_batch(c->e, proofs128, pairs64, nullptr, D, n_clients, seed, ok.data(), &holds);
    return rc < 0 ? rc : holds;
    API_CATCH
}
// the batched rand-proof (kind 1) / square-rand-proof (kind 2) check of sigma_verify_groups alone, over n_elems elements as one update and without the
// size threshold: 1 = every range's combination held and no element is malformed, 0 = not.  proofs n_elems x 128 | 192, commits n_elems x 64 | 96 (host)
extern "C" int rofl_debug_sigma_rlc(rofl_ctx *c, int kind, size_t n_elems, const uint8_t *proofs, const uint8_t *commits, const uint8_t seed[32]) {
    API_TRY
    if ((kind != 1 && kind != 2) || !n_elems || !proofs || !commits || !seed) return ROFL_ERR_ARGS;
    const size_t pw = 32 * sigma_kind_of(kind).pw, cw = 32 * sigma_kind_of(kind).cw;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in dp(proofs, pw * n_elems, s), dc(commits, cw * n_elems, s);
    return sigma_verify_rlc(c->e, s, kind, dp.b.as<uint8_t>(), dc.b.as<uint8_t>(), n_elems, seed);
    API_CATCH
}
// the terms of one batched check, copied from the buffers of its production code (engine.cuh rlc_tap) and derived by nothing here: family 0 / 1 / 2
// the square / rand / square-rand proofs (sigma_verify_groups, that kind) over n_clients updates of D elements and below its size threshold too,
// 3 the compressed rand proofs of n_clients clients of D pairs (engine_crp_verify_batch; commits = the pairs).  See include/rofl_b200.h.
extern "C" int rofl_debug_rlc_terms(rofl_ctx *c, int family, size_t n_clients, size_t D, const uint8_t *proofs, const uint8_t *commits, const uint8_t seed[32],
                                    uint8_t *root32, uint8_t *chal32, int64_t *ranges, uint8_t *scalars32, uint8_t *coef32, int *bad, int *verdicts,
                                    const size_t cap[3], size_t cnt[3]) {
    API_TRY
    const size_t K = n_clients;
    if (family < 0 || family > 3 || !K || !D || !proofs || !commits || !seed || !root32 || !chal32 || !ranges || !scalars32 || !coef32 || !bad || !verdicts || !cap || !cnt)
        return ROFL_ERR_ARGS;
    if (family == 3 && D > CRP_MAX_D) return ROFL_ERR_ARGS;
    rlc_tap tap;
    if (family == 3) {
        const int rc = engine_crp_verify_batch(c->e, proofs, commits, nullptr, D, K, seed, verdicts, nullptr, &tap);
        if (rc < 0) return rc;
    } else {
        const size_t pw = 32 * sigma_kind_of(family).pw, cw = 32 * sigma_kind_of(family).cw;
        lane_guard lg(c->e); cudaStream_t s = lg.s();
        staged_in dp(proofs, pw * D * K, s), dc(commits, cw * D * K, s); dev_buf dres(2 * sizeof(int) * K, s);
        std::vector<int> res(2 * K);
        for (size_t k = 0; k < K; k++) { res[2 * k] = 1; res[2 * k + 1] = 0; }
        rt_h2d(dres.p, res.data(), sizeof(int) * 2 * K, s);
        sigma_verify_groups(c->e, s, family, dp.b.as<uint8_t>(), dc.b.as<uint8_t>(), D * K, seed, D, dres.as<int>(), &tap);
        rt_d2h(res.data(), dres.p, sizeof(int) * 2 * K, s); rt_sync(s);
        for (size_t k = 0; k < K; k++) verdicts[k] = res[2 * k + 1] ? -1 : res[2 * k] ? 1 : 0;
    }
    size_t nsc = 0, nbad = 0;
    for (const auto &r : tap.ranges) { nsc += r.scal.size(); nbad += r.bad.size(); }
    cnt[0] = tap.ranges.size(); cnt[1] = nsc; cnt[2] = nbad;
    if (cnt[0] > cap[0] || nsc > cap[1] || nbad > cap[2]) return ROFL_ERR_ARGS;
    memcpy(root32, tap.root, 32);
    for (size_t i = 0; i < tap.chal.size(); i++) memcpy(chal32 + 32 * i, &tap.chal[i], 32);
    size_t os = 0, ob = 0;
    for (size_t j = 0; j < tap.ranges.size(); j++) {
        const rlc_tap::range &r = tap.ranges[j];
        const int64_t info[8] = {(int64_t)r.i0, (int64_t)r.n, r.c, r.wbits, r.is_id[0], r.is_id[1], (int64_t)os, (int64_t)ob};
        memcpy(ranges + 8 * j, info, sizeof(info));
        for (size_t t = 0; t < r.scal.size(); t++) memcpy(scalars32 + 32 * (os + t), &r.scal[t], 32);
        const sc_st *cf[4] = {&r.sB[0], &r.sB[1], &r.sH[0], &r.sH[1]};
        for (int q = 0; q < 4; q++) memcpy(coef32 + 128 * j + 32 * q, cf[q], 32);
        memcpy(bad + ob, r.bad.data(), sizeof(int) * r.bad.size());
        os += r.scal.size(); ob += r.bad.size();
    }
    return tap.held;
    API_CATCH
}
// the batching scalars (c_i | rho_i, 2 x n_proofs x 32 bytes) the verifier derives for this call; return value as rofl_range_verify
extern "C" int rofl_debug_verify_weights(rofl_ctx *c, const uint8_t *proofs, size_t plen, size_t np, const uint8_t *commits, size_t D, int range, const uint8_t seed[32], uint8_t *out_weights) {
    API_TRY
    if (!D) return ROFL_ERR_ARGS;
    lane_guard lg(c->e);
    staged_in dc(commits, 32 * D, lg.s());
    return engine_range_verify(c->e, proofs, plen, np, dc.b.as<uint8_t>(), D, range, seed, nullptr, out_weights);
    API_CATCH
}
// the MSM front end alone: out32[k] = sum_t s[k][t] P_t (+ sB[k] B + sH[k] H), k < n_msm, through the production plan / kernels / k_finalize.
//   scalars32: n_msm x T canonical scalars; one >= l is ROFL_ERR_ARGS (the signed recoding and the fat-top-window bound assume reduced scalars).
//   points32: compressed bases, T shared by all instances (points_per_msm = 0) or n_msm x T (1), split into two segments at ceil(T / 2) like the
//     verifier's commitments | proof points; an undecodable one is ROFL_ERR_POINT.  NULL: the generators BulletproofGens(gen_n, T / (2 gen_n)), G then H.
//   path 0: msm_plan_for(T, n_msm, big_min); 1: msm_plan_forced(T, c, knob); 2: the generator tables (k_rt_msm, generators only).
//   sB32 / sH32: n_msm scalars each, or NULL.  info (nullable): window width, slices (k_msm) / parts (k_bm_*) / blocks (k_rt_msm), kernel 0 / 1 / 2.
extern "C" int rofl_debug_msm(rofl_ctx *c, const uint8_t *scalars32, size_t n_msm, size_t T, const uint8_t *points32, int points_per_msm, int gen_n,
                              int path, int cw, int knob, size_t big_min, const uint8_t *sB32, const uint8_t *sH32, uint8_t *out32, int *info) {
    API_TRY
    if (!scalars32 || !out32 || !n_msm || n_msm > 0xffff || !T || n_msm * T > 0x7fffffffu || path < 0 || path > 2) return ROFL_ERR_ARGS;
    if (points32 ? path == 2 : (gen_n <= 0 || T % (2 * (size_t)gen_n))) return ROFL_ERR_ARGS;
    auto canonical = [](std::vector<sc_st> &o, const uint8_t *b, size_t n) {
        o.resize(n);
        for (size_t i = 0; i < n; i++) { sc x; sc_frombytes(x, b + 32 * i); if (!sc_is_canonical(x)) return false; sc_to_st(o[i], x); }
        return true;
    };
    std::vector<sc_st> hs, hB, hH;
    if (!canonical(hs, scalars32, n_msm * T) || (sB32 && !canonical(hB, sB32, n_msm)) || (sH32 && !canonical(hH, sH32, n_msm))) return ROFL_ERR_ARGS;
    lane_guard lg(c->e); cudaStream_t s = lg.s();
    staged_in ds(hs.data(), sizeof(sc_st) * hs.size(), s), dB(hB.data(), sizeof(sc_st) * hB.size(), s), dH(hH.data(), sizeof(sc_st) * hH.size(), s);
    dev_buf dout(32 * n_msm, s);
    finalize_args f = {}; f.sBa = sB32 ? dB.b.as<sc_st>() : nullptr; f.sHa = sH32 ? dH.b.as<sc_st>() : nullptr; f.tabB = c->e.sh->tabB; f.tabH = c->e.sh->tabH;
    f.out32 = dout.as<uint8_t>(); f.count = (int)n_msm;
    int inf[3] = {0, 0, 0};
    msm_args a = {}; a.v[0].scalars = ds.b.as<sc_st>(); a.split = (uint32_t)n_msm; a.T = (uint32_t)T; a.scalar_stride = (uint32_t)T; a.nseg = 2;
    auto msm = [&](const msm_plan &pl) {
        dev_buf d_win(sizeof(p3_st) * pl.out_count(n_msm), s);
        a.out = d_win.as<p3_st>();
        run_msm(c->e, s, a, pl, (uint32_t)n_msm);
        fin_windows(f, d_win.as<p3_st>(), pl);
        run_finalize(s, f);
        rt_d2h(out32, dout.p, 32 * n_msm, s); rt_sync(s);
        inf[0] = pl.c; inf[1] = (int)(pl.big ? pl.parts : pl.slices); inf[2] = pl.big ? 1 : 0;
    };
    const msm_plan pl = path == 1 ? msm_plan_forced(T, cw, knob) : msm_plan_for(T, n_msm, big_min);
    if (points32) {
        const size_t np = points_per_msm ? n_msm * T : T;
        const uint32_t h = (uint32_t)((T + 1) / 2), stride = points_per_msm ? (uint32_t)T : 0;
        staged_in dp(points32, 32 * np, s); dev_buf d_pts(sizeof(p3_st) * np, s), d_bad(sizeof(int), s);
        rt_memset(d_bad.p, 0, sizeof(int), s);
        LAUNCH(k_decompress, dim3((unsigned)((np + 127) / 128)), dim3(128), s, d_pts.as<p3_st>(), (uint8_t *)nullptr, dp.b.as<uint8_t>(), np, np, (const p3_st *)nullptr, d_bad.as<int>(), np);
        int bad = 0; rt_d2h(&bad, d_bad.p, sizeof(int), s); rt_sync(s);
        if (bad) return ROFL_ERR_POINT;
        a.v[0].seg[0] = mk_seg(d_pts.as<p3_st>(), h, stride, 1); a.v[0].seg[1] = mk_seg(d_pts.as<p3_st>() + h, (uint32_t)T - h, stride, 1);
        msm(pl);
    } else {
        const int m = (int)(T / (2 * (size_t)gen_n)); const uint32_t N = (uint32_t)(T / 2);
        tables_use tu(*c->e.sh);
        engine_gens(c->e, tu, s, gen_n, m);
        rt_tables rt; const bool have_rt = path == 2 && engine_rt(c->e, tu, s, gen_n, m, rt);
        const gens_entry g = engine_gens(c->e, tu, s, gen_n, m);
        if (path == 2) {
            if (!have_rt) return ROFL_ERR_ARGS;
            const int nb = rt_blocks(T, (int)n_msm);
            dev_buf d_part(sizeof(p3_st) * (size_t)nb * n_msm, s);
            rt_msm_args ra = {}; ra.scalars = ds.b.as<sc_st>(); ra.T = (uint32_t)T; ra.scalar_stride = (uint32_t)T; ra.nG = N; ra.mode = 0; ra.rt = rt; ra.partial = d_part.as<p3_st>();
            run_rt_msm(c->e, s, ra, nb, (uint32_t)n_msm);
            f.partial = d_part.as<p3_st>(); f.npartial = nb;
            run_finalize(s, f);
            rt_d2h(out32, dout.p, 32 * n_msm, s); rt_sync(s);
            inf[0] = rt.c; inf[1] = nb; inf[2] = 2;
        } else {
            a.v[0].seg[0] = mk_seg(g.G, N, 0, 0); a.v[0].seg[1] = mk_seg(g.H, N, 0, 0);
            msm(pl);
        }
    }
    if (info) memcpy(info, inf, sizeof(inf));
    return 0;
    API_CATCH
}
