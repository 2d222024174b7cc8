// Host orchestration of the rofl_crypto prove / verify hot path on one GPU (C++; the reference's host side is Rust).
// Mirrors, function for function, the vector API that rofl_service links (SURVEY.md section 8b):
//   range_proof_vec::{create_rangeproof, verify_rangeproof}      range_proof_vec/mod.rs:16-102,149-191
//   l2_range_proof_vec::{create_rangeproof_l2, verify_rangeproof_l2}   l2_range_proof_vec/mod.rs:15-140,185-228
//   square_proof_vec::{create_l2rangeproof_vec_existing, verify_l2rangeproof_vec}   square_proof_vec/mod.rs:19-75,130-160
//   pedersen_ops::{commit_vec, add_rp_vec_vec, discrete_log_vec_table}, ElGamal R halves, bsgs32::BSGSTable
// All chunks of one update advance in lock step: one kernel launch per phase covers every chunk, the sequential
// Fiat-Shamir transcripts (Merlin) stay on the host, one small device<->host exchange per challenge.
#pragma once
#include "kernels.cuh"
#include "rt.cuh"
#include <map>
#include <mutex>
#include <shared_mutex>
#include <condition_variable>
#include <thread>
#include <atomic>
#ifndef ROFL_EMUL
#include <sys/resource.h>
#endif
#include <algorithm>
#include <chrono>
#include <cstdio>

enum { ROFL_ERR_BITSIZE_ = -7 };          // include/rofl_b200.h ROFL_ERR_BITSIZE
enum { DOM_RANGE_PROVE = 1, DOM_RANGE_VERIFY = 2, DOM_SQUARE = 3, DOM_L2_PROVE = 4, DOM_L2_VERIFY = 5, DOM_CRP = 6, DOM_RND_VEC = 7, DOM_RANDPROOF = 8, DOM_SQUARE_RAND = 9,
       DOM_CRP_BATCH = 0x62707263 /* "crpb" as LE32: the weights of engine_crp_verify_batch */,
       DOM_SQ_RLC = 0x6c727173 /* "sqrl": the weights of the batched square-proof check (sigma_verify_rlc, kind 0) */,
       DOM_RP_RLC = 0x6c727072 /* "rprl": the same for rand proofs (kind 1) */,
       DOM_SRP_RLC = 0x6c727273 /* "srrl": the same for square-rand proofs (kind 2) */ };
enum { PROF_FOLD = 0, PROF_MSM = 1, PROF_COMMIT = 2, PROF_SQUARE = 3, PROF_RTMSM = 4, PROF_TAIL = 5, PROF_FRZ = 6, PROF_SLOTS = 8 };

struct gens_entry { int n = 0; int cap = 0; niels_st *G = nullptr, *H = nullptr;
                    int rt_cap = 0, rt_c = 8; niels_st *RTG = nullptr, *RTH = nullptr; size_t rt_bytes = 0; uint64_t last_use = 0;
                    int rt_nofit = 0; };     // smallest party count whose tables did NOT fit the device (0 = none yet): not tried again until tables are dropped     // radix-2^rt_c tables (RT path)
struct bsgs_entry { unsigned long long *keys = nullptr; uint32_t *vals = nullptr; uint32_t cap = 0; uint64_t size = 0; };
// Everything that is a function of the DEVICE alone lives once per device and process and is shared by all contexts on it: the fixed-base
// tables of B / B_blinding, the Bulletproofs generators, their radix-2^c tables (tens of GB) and the BSGS tables (server.rs:54,84 shares one
// Arc<BSGSTable> between its workers the same way).  tab_mu: calls hold it SHARED while they use cached tables; building, regrowing or
// dropping a table takes it EXCLUSIVE, i.e. waits until no call is using the old arrays.
struct dev_shared {
    int device = 0, refs = 0;
    niels_st *tabB = nullptr, *tabH = nullptr;
    uint8_t B32[32], H32[32];
    std::map<int, gens_entry> gens;
    std::map<std::pair<uint64_t, int>, bsgs_entry> bsgs;
    std::shared_mutex tab_mu;
    std::atomic<size_t> free_hint{0};     // free device memory when the generator tables were last (re)built: cudaMemGetInfo is NOT for the hot path
    std::atomic<uint64_t> clock{0};       // LRU stamps of the generator tables
};
struct tables_use {
    dev_shared &sh; bool excl = false;
    explicit tables_use(dev_shared &s) : sh(s) { sh.tab_mu.lock_shared(); }
    ~tables_use() { if (excl) sh.tab_mu.unlock(); else sh.tab_mu.unlock_shared(); }
    // not atomic: re-check the condition after it.  There is no way back to shared (that would open a second gap in which another caller
    // could evict what was just built): a call that had to build a table keeps the device's tables to itself until it returns.
    void upgrade() { if (!excl) { sh.tab_mu.unlock_shared(); sh.tab_mu.lock(); excl = true; } }
    tables_use(const tables_use &) = delete; tables_use &operator=(const tables_use &) = delete;
};
// A lane = the streams one caller works on: per chunk group a queue (high-priority stream for the latency-bound Fiat-Shamir chain, normal
// stream for the bulk kernels, rt.cuh `chain`) and a side stream.  Concurrent callers of one context (rofl_service runs one verify() per
// client on a rayon pool, server.rs:516-522,666) get different lanes, i.e. run on different streams; the cached tables are shared.
#define ROFL_MAX_GROUPS 4
struct lane { chain q[ROFL_MAX_GROUPS]; cudaStream_t side[ROFL_MAX_GROUPS]; bool busy = false; };
struct rofl_engine {
    int device = 0;
    dev_shared *sh = nullptr;
    std::mutex lane_mu; std::condition_variable lane_cv; std::vector<lane *> lanes; int max_lanes = 8;
    int host_threads = 8;
    int groups = 3;                       // chunk groups proved concurrently on separate queues (the latency-bound chain of one overlaps the bulk kernels of the others)
    int use_rt = 1;                       // 0: never build generator tables (generic Pippenger / fold path only)
    int rt_unfold = 4;                    // IPP rounds computed over the original generators before the catch-up fold
    int tail_np = 32;                     // IPP rounds with half-size <= tail_np run in the fused on-device tail kernel (0 = off)
    int tail_batch_mb = 2048;             // the tail's per-digit tables (8 MB per chunk) are built and used for this many MB of chunks at a time
    int tail_ncta = 2;                    // thread blocks (one cluster) per chunk in the tail kernel: 1, 2, 4, 8.  Measured with three chunk groups: 2 -> 36.15 ms,
                                          // 1 -> 36.35, 4 -> 38.1 (a 4-block cluster of 544-thread blocks waits for room beside the other groups' bulk kernels)
    std::mutex pin_mu; std::vector<std::pair<void *, size_t>> pins;      // pool of pinned host blocks
    int use_frz = 1;                      // middle IPP rounds over frozen generators with on-the-fly Straus tables (kernels.cuh K6c)
    int rt_bits = RT_MAX_BITS;            // widest generator-table radix to try (8..11)
    double group_w[ROFL_MAX_GROUPS] = {1.0, 1.0, 1.0, 1.0};      // relative chunk counts of the groups
    int nt_unfold = 4, nt_unfold_min = 1 << 16;      // unfolded IPP rounds without generator tables, for chunks of at least that many bit positions
    int ts_host_m = 8192;                 // chunks with more commitments than this absorb them on the host (absorb_commitments)
    int rt_per = 2;                       // table-MSM terms per thread and block: short blocks let the other groups' small kernels in quickly
    double rt_mem_frac = 0.45;            // tables may take this fraction of the free device memory
    size_t sigma_rlc_terms = (size_t)1 << 24;      // MSM terms per range of the batched rand / square-rand proof check (sigma_verify_rlc; not square proofs)
    size_t crp_batch_terms = (size_t)1 << 24;      // MSM terms per client group of the batched compressed-rand-proof check (crp_batch)
};
static thread_local lane *tl_lane = nullptr; static thread_local rofl_engine *tl_lane_engine = nullptr; static thread_local int tl_lane_depth = 0;
static inline lane *lane_new() {
    lane *l = new lane();
    // the short kernels of every group's Fiat-Shamir chain run at the greatest priority, the bulk kernels one level below.  (ROFL_PRIO_ORDERED=1
    // orders the bulk streams of the groups as well -- group 0 races ahead so that its latency-bound last rounds run under the bulk kernels of
    // the groups behind it; measured on B200 it is 3 ms SLOWER per proof than equal priorities: the last group ends up alone.  DESIGN.md section 3)
    static const int ordered = getenv("ROFL_PRIO_ORDERED") ? atoi(getenv("ROFL_PRIO_ORDERED")) : 0, flat = getenv("ROFL_PRIO_FLAT") ? atoi(getenv("ROFL_PRIO_FLAT")) : 0;
    static const int own_side = getenv("ROFL_SIDE") ? atoi(getenv("ROFL_SIDE")) : 1;
    for (int g = 0; g < ROFL_MAX_GROUPS; g++) { cudaStream_t hi = rt_stream_create(flat ? 1 : 0), lo = rt_stream_create(ordered ? 1 + g : 1); l->q[g] = chain(hi, lo); l->side[g] = own_side ? rt_stream_create(0) : hi; }
    return l;
}
static inline void lane_delete(lane *l) { for (int g = 0; g < ROFL_MAX_GROUPS; g++) { rt_stream_destroy(l->q[g].hi); if (l->q[g].lo != l->q[g].hi) rt_stream_destroy(l->q[g].lo); if (l->side[g] != l->q[g].hi) rt_stream_destroy(l->side[g]); } delete l; }
// the calling thread's lane for the duration of an API call (nested engine calls of the same thread share it)
struct lane_guard {
    rofl_engine &e; lane *ln = nullptr;
    explicit lane_guard(rofl_engine &eng) : e(eng) {
        if (tl_lane && tl_lane_engine == &e) { ln = tl_lane; tl_lane_depth++; return; }
        if (tl_lane) throw std::runtime_error("rofl_b200: nested calls into two contexts from one thread");
        std::unique_lock<std::mutex> lk(e.lane_mu);
        for (;;) {
            for (lane *l : e.lanes) if (!l->busy) { ln = l; break; }
            if (ln) break;
            if ((int)e.lanes.size() < e.max_lanes) { ln = lane_new(); e.lanes.push_back(ln); break; }
            e.lane_cv.wait(lk);
        }
        ln->busy = true; tl_lane = ln; tl_lane_engine = &e; tl_lane_depth = 1;
    }
    ~lane_guard() {
        if (--tl_lane_depth > 0) return;
        rt_d2h_finish(std::uncaught_exceptions() > 0);
        { std::lock_guard<std::mutex> lk(e.lane_mu); ln->busy = false; }
        e.lane_cv.notify_one(); tl_lane = nullptr; tl_lane_engine = nullptr;
    }
    cudaStream_t s() const { return ln->q[0].hi; }
    lane_guard(const lane_guard &) = delete; lane_guard &operator=(const lane_guard &) = delete;
};

// pinned host scratch with scope lifetime, recycled through the engine's pool (cudaHostAlloc is far too slow to call per proof)
struct pinned_buf {
    rofl_engine &e; void *p = nullptr; size_t n = 0;
    pinned_buf(rofl_engine &eng, size_t bytes) : e(eng) {
        { std::lock_guard<std::mutex> lk(e.pin_mu);
          for (size_t i = 0; i < e.pins.size(); i++) if (e.pins[i].second >= bytes) { p = e.pins[i].first; n = e.pins[i].second; e.pins.erase(e.pins.begin() + i); break; } }
        if (!p) { n = std::max<size_t>(bytes, 1 << 16); p = rt_host_alloc(n); }
    }
    ~pinned_buf() { std::lock_guard<std::mutex> lk(e.pin_mu); e.pins.emplace_back(p, n); }
    pinned_buf(const pinned_buf &) = delete; pinned_buf &operator=(const pinned_buf &) = delete;
    template <class T> T *as() const { return (T *)p; }
};

// ROFL_TRACE=1: wall-clock phase marks of prove_chunks on stderr (stream synchronised at every mark; debugging aid only)
struct phase_trace {
    bool on; cudaStream_t s; std::chrono::steady_clock::time_point t0; std::string out;
    phase_trace(cudaStream_t st) : on(getenv("ROFL_TRACE") != nullptr), s(st) { if (on) { rt_sync(s); t0 = std::chrono::steady_clock::now(); } }
    void mark(const char *what) { if (!on) return; rt_sync(s); auto t = std::chrono::steady_clock::now(); char b[96]; snprintf(b, sizeof b, " %s=%.2f", what, std::chrono::duration<double, std::milli>(t - t0).count()); out += b; t0 = t; }
    ~phase_trace() { if (on) fprintf(stderr, "[rofl trace]%s\n", out.c_str()); }
};

// ---- small host helpers ---------------------------------------------------------------------------------------------------
static inline size_t next_pow2_sz(size_t v) { if (v <= 1) return 1; size_t n = v - 1; while (n & (n - 1)) n &= n - 1; return n << 1; }   // range_proof_vec/mod.rs:237-246
static inline int ilog2_sz(size_t x) { int l = 0; while (((size_t)1 << l) < x) l++; return l; }
static inline bool fp_ok(int n_bits, int frac) { return (n_bits == 8 || n_bits == 16 || n_bits == 32 || n_bits == 64) && frac >= 0 && frac <= 12; }
static inline float clip_max_f(int range, int n_bits, int frac) {                  // conversion32.rs:56-60
    uint64_t raw = (range - 1 >= 64) ? ~0ULL : ((1ULL << (range - 1)) - 1);
    return fix_to_f32(raw & fix_max(n_bits), frac);
}
static inline float l2_clip_max_f(int range, int n_bits, int frac) {               // conversion32.rs:62-64
    uint64_t raw = (range >= 64) ? ~0ULL : ((1ULL << range) - 1);
    return fix_to_f32(raw & fix_max(n_bits), frac);
}
static inline void derive_key(uint8_t out[32], const uint8_t seed[32], uint32_t domain, uint64_t index) {
    uint8_t buf[44]; memcpy(buf, seed, 32);
    for (int i = 0; i < 4; i++) buf[32 + i] = (uint8_t)(domain >> (8 * i));
    for (int i = 0; i < 8; i++) buf[36 + i] = (uint8_t)(index >> (8 * i));
    sha3_256(out, buf, 44);
}
static inline void key_words(uint32_t w[8], const uint8_t k[32]) { for (int i = 0; i < 8; i++) w[i] = (uint32_t)k[4 * i] | ((uint32_t)k[4 * i + 1] << 8) | ((uint32_t)k[4 * i + 2] << 16) | ((uint32_t)k[4 * i + 3] << 24); }
static inline void sc_to_st(sc_st &o, const sc &s) { for (int i = 0; i < 8; i++) o.w[i] = s.v[i]; }
static inline void st_to_sc(sc &s, const sc_st &o) { for (int i = 0; i < 8; i++) s.v[i] = o.w[i]; }
template <class F> static void parallel_for(size_t n, int threads, F f) {
    rt_host_timer t_(&rt_host_prof::par, "parallel_for");
    if (n <= 1 || threads <= 1) { for (size_t i = 0; i < n; i++) f(i); return; }
    size_t nt = std::min<size_t>(threads, n); std::vector<std::thread> th;
    for (size_t t = 0; t < nt; t++) th.emplace_back([=] { for (size_t i = t; i < n; i += nt) f(i); });
    for (auto &x : th) x.join();
}
// light per-chunk host work (a few Keccak-f per chunk): thread start-up would cost more than the work
template <class F> static void serial_for(size_t n, F f) { rt_host_timer t_(&rt_host_prof::ser, "serial_for"); for (size_t i = 0; i < n; i++) f(i); }
// Montgomery's trick: v[i] <- v[i]^-1 (all non-zero)
static inline void sc_batch_invert(std::vector<sc> &v) {
    size_t n = v.size(); if (!n) return;
    std::vector<sc> pre(n); sc acc; sc_from_u64(acc, 1);
    for (size_t i = 0; i < n; i++) { pre[i] = acc; sc_mul(acc, acc, v[i]); }
    sc inv; sc_invert_vartime(inv, acc);           // public Fiat-Shamir challenges only
    for (size_t i = n; i-- > 0;) { sc t; sc_mul(t, inv, pre[i]); sc_mul(inv, inv, v[i]); v[i] = t; }
}
static inline void ts_challenge_scalar(transcript &t, const char *label, sc &out) { uint8_t b[64]; transcript_challenge(t, label, b, 64); sc_from_bytes_wide(out, b); }
static inline void ts_append_sc(transcript &t, const char *label, const sc &s) { uint8_t b[32]; sc_tobytes(b, s); transcript_append(t, label, b, 32); }
static inline bool is_zero32(const uint8_t *b) { uint8_t z = 0; for (int i = 0; i < 32; i++) z |= b[i]; return z == 0; }
// pow2[b] = s^(2^b), b < 32
static inline void sc_pow2_table(sc_st *tab, const sc &s) { sc c = s; for (int b = 0; b < 32; b++) { sc_to_st(tab[b], c); sc_mul(c, c, c); } }

// ---- engine lifetime ------------------------------------------------------------------------------------------------------
static std::mutex g_shared_mu; static std::map<int, dev_shared *> g_shared;
static inline void engine_init(rofl_engine &e) {
    {
        std::lock_guard<std::mutex> lk(g_shared_mu);
        dev_shared *&sh = g_shared[e.device];
        if (!sh) { sh = new dev_shared(); sh->device = e.device; }
        sh->refs++; e.sh = sh;
    }
    if (e.lanes.empty()) e.lanes.push_back(lane_new());
    dev_shared &sh = *e.sh;
    std::unique_lock<std::shared_mutex> ex(sh.tab_mu);
    if (sh.tabB) return;
    ge_p3 B, H; ge_base(B); ge_compress(sh.B32, B);
    uint8_t h[64]; sha3_512(h, sh.B32, 32); ge_from_uniform_bytes(H, h); ge_compress(sh.H32, H);     // PedersenGens::default / el_gamal.rs:31-40
    cudaStream_t s = e.lanes[0]->q[0].hi;
    sh.free_hint = rt_free_mem();
    sh.tabB = (niels_st *)rt_raw_malloc(sizeof(niels_st) * FB_WINDOWS * FB_ENTRIES);
    sh.tabH = (niels_st *)rt_raw_malloc(sizeof(niels_st) * FB_WINDOWS * FB_ENTRIES);
    dev_buf pts(64, s);
    rt_h2d(pts.as<uint8_t>(), sh.B32, 32, s); rt_h2d(pts.as<uint8_t>() + 32, sh.H32, 32, s);
    int nent = FB_WINDOWS * FB_ENTRIES;
    LAUNCH(k_fb_table_build, dim3((nent + 63) / 64), dim3(64), s, sh.tabB, pts.as<uint8_t>());
    LAUNCH(k_fb_table_build, dim3((nent + 63) / 64), dim3(64), s, sh.tabH, pts.as<uint8_t>() + 32);
    rt_sync(s);
}
static inline void engine_destroy(rofl_engine &e) {
    for (lane *l : e.lanes) { for (int g = 0; g < ROFL_MAX_GROUPS; g++) { rt_sync(l->q[g].hi); rt_sync(l->q[g].lo); rt_sync(l->side[g]); } lane_delete(l); }
    e.lanes.clear();
    for (auto &pp : e.pins) rt_host_free(pp.first);
    e.pins.clear();
    std::lock_guard<std::mutex> lk(g_shared_mu);
    dev_shared *sh = e.sh; e.sh = nullptr;
    if (!sh || --sh->refs > 0) return;
    rt_raw_free(sh->tabB); rt_raw_free(sh->tabH);
    for (auto &g : sh->gens) { rt_raw_free(g.second.G); rt_raw_free(g.second.H); rt_raw_free(g.second.RTG); rt_raw_free(g.second.RTH); }
    for (auto &b : sh->bsgs) { rt_raw_free(b.second.keys); rt_raw_free(b.second.vals); }
    g_shared.erase(sh->device); delete sh;
    rt_trim();
}
// BulletproofGens::new(n, m): cached per n and device, capacity grows (the reference rebuilds them per chunk per call,
// range_proof_vec/mod.rs:126,201).  Returns a copy of the entry; the arrays stay valid while the caller's tables_use is held.
static inline gens_entry engine_gens(rofl_engine &e, tables_use &tu, cudaStream_t s, int n, int m) {
    dev_shared &sh = *e.sh;
    for (;;) {
        auto it = sh.gens.find(n);
        if (it != sh.gens.end() && it->second.cap >= m) return it->second;
        tu.upgrade();
        gens_entry &g = sh.gens[n];
        if (g.cap >= m) continue;
        int newcap = std::max(m, g.cap * 2);
        niels_st *G = (niels_st *)rt_raw_malloc(sizeof(niels_st) * (size_t)n * newcap);
        niels_st *H = (niels_st *)rt_raw_malloc(sizeof(niels_st) * (size_t)n * newcap);
        if (g.cap) { rt_d2d(G, g.G, sizeof(niels_st) * (size_t)n * g.cap, s); rt_d2d(H, g.H, sizeof(niels_st) * (size_t)n * g.cap, s); }
        int cnt = 2 * (newcap - g.cap);
        LAUNCH(k_gens_build, dim3((cnt + 63) / 64), dim3(64), s, G, H, n, g.cap, newcap);
        rt_sync(s);
        rt_raw_free(g.G); rt_raw_free(g.H);
        g.n = n; g.cap = newcap; g.G = G; g.H = H;
    }
}
static inline void rt_fill(rt_tables &t, int c) { t.c = c; t.nw = msm_nw(c); t.B = 1 << (c - 1); msm_recode_const(t.K, c); }
static inline size_t rt_table_bytes(size_t cnt, int c) { return 2 * cnt * (size_t)msm_nw(c) * ((size_t)1 << (c - 1)) * sizeof(niels_st); }
// radix-2^c generator tables for the first m parties of the n-bit generators (c = 11 .. 8: the widest that fits the memory budget; wider =
// fewer additions per term); returns false when not even c = 8 fits.  The tables of other (n, m) are evicted, least recently used first,
// when that lets this one have a wider radix: the current workload gets the best tables the device can hold.
static inline bool engine_rt(rofl_engine &e, tables_use &tu, cudaStream_t s, int n, int m, rt_tables &out) {
    if (!e.use_rt) return false;
    dev_shared &sh = *e.sh;
    for (;;) {
        gens_entry &g = sh.gens[n];                          // exists: engine_gens ran first
        if (g.rt_cap >= m) { g.last_use = ++sh.clock; out.G = g.RTG; out.H = g.RTH; rt_fill(out, g.rt_c); return true; }
        if (g.rt_nofit && m >= g.rt_nofit) return false;         // (resnet18-full chunks: 2^22 generators would need terabytes; asking again would trim the scratch cache on every call)
        if (!tu.excl) { tu.upgrade(); continue; }
        const size_t cnt = (size_t)n * m;
        if ((double)rt_table_bytes(cnt, 8) > 170e9) { g.rt_nofit = m; return false; }          // cannot fit any B200 even at the narrowest radix: keep what is cached
        rt_sync(s); rt_raw_free(g.RTG); rt_raw_free(g.RTH); g.RTG = g.RTH = nullptr; g.rt_cap = 0; g.rt_bytes = 0;
        rt_trim();
        const int want = std::max(8, std::min(RT_MAX_BITS, e.rt_bits));
        int c = 0;
        for (;;) {
            const size_t have = rt_free_mem();
            for (c = want; c >= 8; c--) if ((double)(rt_table_bytes(cnt, c) + cnt * msm_nw(c) * sizeof(p3_st)) <= e.rt_mem_frac * (double)have) break;
            if (c == want) break;
            gens_entry *victim = nullptr;                    // not the widest radix: drop the least recently used tables of another (n, m) and look again
            for (auto &kv : sh.gens) if (&kv.second != &g && kv.second.RTG && (!victim || kv.second.last_use < victim->last_use)) victim = &kv.second;
            if (!victim) break;
            rt_raw_free(victim->RTG); rt_raw_free(victim->RTH); victim->RTG = victim->RTH = nullptr; victim->rt_cap = 0; victim->rt_bytes = 0;
        }
        if (c < 8) { g.rt_nofit = m; sh.free_hint = rt_free_mem(); return false; }
        rt_tables t; rt_fill(t, c);
        const size_t bytes = cnt * rt_row_entries(t) * sizeof(niels_st);
        niels_st *RTG = (niels_st *)rt_raw_malloc(bytes), *RTH = (niels_st *)rt_raw_malloc(bytes);
        {
            dev_buf P(cnt * t.nw * sizeof(p3_st), s);
            const size_t rows = cnt * t.nw, thr = rows * (t.B / 16);
            for (int which = 0; which < 2; which++) {
                LAUNCH(k_rt_shifts, dim3((unsigned)((cnt + 127) / 128)), dim3(128), s, P.as<p3_st>(), which ? g.H : g.G, (uint32_t)cnt, t.c, t.nw);
                LAUNCH(k_rt_rows, dim3((unsigned)((thr + 127) / 128)), dim3(128), s, which ? RTH : RTG, P.as<p3_st>(), rows, t.B);
            }
            rt_sync(s);
        }
        g.RTG = RTG; g.RTH = RTH; g.rt_cap = m; g.rt_c = c; g.rt_bytes = 2 * bytes;
        rt_trim();                                           // the build scratch goes back to CUDA before the free memory is recorded
        sh.free_hint = rt_free_mem();
    }
}
// drop every cached generator table of the device (they are rebuilt on next use)
static inline void engine_drop_rt(rofl_engine &e) {
    std::unique_lock<std::shared_mutex> ex(e.sh->tab_mu);
    for (auto &g : e.sh->gens) { rt_raw_free(g.second.RTG); rt_raw_free(g.second.RTH); g.second.RTG = g.second.RTH = nullptr; g.second.rt_cap = 0; g.second.rt_bytes = 0; g.second.rt_nofit = 0; }
}
// blocks per msm for the direct table MSM: every block of a wave runs ceil(T / (nb*128)) terms per thread, so pick the nb whose
// waves (148 SMs x 4 resident blocks) x terms-per-thread product is smallest (+ a block-sum epilogue worth ~half a term)
static inline int rt_blocks(size_t T, int C, int per_max = 0) {
    const size_t slots = 148 * RTM_BLOCKS, max_nb = std::max<size_t>(1, (T + 127) / 128);
    if (per_max > 0) {           // at most per_max terms per thread: blocks of ~100 us, several waves (the gaps at their ends are filled by the other chunk groups)
        const size_t nb = std::min(max_nb, (T + 128 * (size_t)per_max - 1) / (128 * (size_t)per_max));
        return (int)std::max<size_t>(1, nb);
    }
    const size_t lim = std::max<size_t>(1, std::min(max_nb, slots * 4 / (size_t)C));
    size_t best = 1; double best_cost = 1e300;
    for (size_t nb = 1; nb <= lim; nb++) {
        const double waves = (double)((nb * C + slots - 1) / slots), per = (double)((T + nb * 128 - 1) / (nb * 128));
        const double cost = waves * (per + 0.5);
        if (cost < best_cost * 0.999) { best_cost = cost; best = nb; }
    }
    return (int)best;
}
static inline void run_rt_msm(rofl_engine &e, cudaStream_t s, rt_msm_args a, int nb, uint32_t n_msm) {
    rt_prof_work(PROF_RTMSM, (double)a.T * n_msm * a.rt.nw);          // mixed additions (upper bound: zero digits skip theirs)
    void *tk = rt_prof_begin(PROF_RTMSM, s);
    LAUNCH_COOP(k_rt_msm, dim3(nb, n_msm), dim3(128), s, a);
    rt_prof_end(PROF_RTMSM, tk, s);
}

// ---- MSM front end ----------------------------------------------------------------------------------------------------------
// window width and term slicing for an MSM of T terms run as n_msm independent instances (kernels.cuh, k_msm)
struct msm_plan { int c, nw; uint32_t slices, slice_len; bool big = false; uint32_t parts = 1; size_t out_count(size_t n_msm) const { return n_msm * slices * (size_t)nw; } };
static inline int msm_pick_c(size_t T) {
    int best = 8; double bc = 1e300;
    for (int c = 3; c <= 8; c++) { const double B = (double)(1 << (c - 1)), cost = (double)msm_nw(c) * ((double)T + B * c); if (cost < bc) { bc = cost; best = c; } }
    return best;
}
static inline size_t bm_min_terms() { static const size_t v = getenv("ROFL_BM_MIN") ? (size_t)atoll(getenv("ROFL_BM_MIN")) : (size_t)32768; return v; }
// a forced plan (tests): window width c (clamped to 3 .. 16) and one more knob -- term slices for k_msm (c <= 8, clamped to 1 .. T), parts per
// bucket for k_bm_* (c >= 9, clamped to 1 .. 8)
static inline msm_plan msm_plan_forced(size_t T, int c, int knob) {
    msm_plan p; p.c = std::max(3, std::min(16, c)); p.nw = msm_nw(p.c); p.slices = 1; p.slice_len = (uint32_t)T;
    if (p.c > 8) { p.big = true; p.parts = (uint32_t)std::max(1, std::min(8, knob)); return p; }
    if (T > 0) { p.slices = (uint32_t)std::max<size_t>(1, std::min<size_t>(std::max(knob, 1), T)); p.slice_len = (uint32_t)((T + p.slices - 1) / p.slices); p.slices = (uint32_t)((T + p.slice_len - 1) / p.slice_len); }
    return p;
}
// big_min: smallest T for the sorted wide-window form (0 = the default bm_min_terms(); single verifier-side MSMs pass 2048: k_msm needs 3.6 ms for
// the 10 000 terms of a configs[0] verification -- 76 blocks walking 32 windows -- the sorted form 0.5 ms)
static inline msm_plan msm_plan_for(size_t T, size_t n_msm, size_t big_min = 0) {
    msm_plan p; p.c = msm_pick_c(T); p.slices = 1; p.slice_len = (uint32_t)T;
    if (const char *fc = getenv("ROFL_MSM_C"))         // test hook: force the window width / slicing
        return msm_plan_forced(T, atoi(fc), getenv("ROFL_MSM_SLICES") ? atoi(getenv("ROFL_MSM_SLICES")) : 1);
    if (T >= (big_min ? big_min : bm_min_terms())) {   // wide windows, buckets sorted in global memory (kernels.cuh K4b): ~64 terms per bucket
        p.big = true; p.c = std::max(9, std::min(16, ilog2_sz(T + 1) - 6)); p.nw = msm_nw(p.c);
        const size_t threads = n_msm * (size_t)p.nw * ((size_t)1 << (p.c - 1));
        p.parts = (uint32_t)std::max<size_t>(1, std::min<size_t>(8, (148 * 1024 + threads - 1) / threads));
        return p;
    }
    const size_t wpb = MSM_THREADS >> (p.c - 1), blocks = n_msm * ((msm_nw(p.c) + wpb - 1) / wpb), slots = 148 * 4;
    if (blocks < slots && T >= 4096) {
        p.slices = (uint32_t)std::min<size_t>((slots + blocks - 1) / blocks, T / 2048);
        p.slice_len = (uint32_t)((T + p.slices - 1) / p.slices); p.slices = (uint32_t)((T + p.slice_len - 1) / p.slice_len);
        p.c = msm_pick_c(p.slice_len);
    }
    p.nw = msm_nw(p.c);
    return p;
}
// a: v[], split, nseg, T, scalar_stride, out filled by the caller
static inline void run_msm(rofl_engine &e, cudaStream_t s, msm_args a, const msm_plan &p, uint32_t n_msm) {
    a.c = p.c; a.nw = p.nw; a.slices = p.slices; a.slice_len = p.slice_len; msm_recode_const(a.K, p.c);
    void *tk = rt_prof_begin(PROF_MSM, s);
    if (p.big) {
        const size_t B = (size_t)1 << (p.c - 1), nslot = (size_t)n_msm * p.nw * (B + 1);
        dev_buf d_start(4 * nslot, s), d_cur(4 * nslot, s), d_sorted(4 * (size_t)n_msm * p.nw * a.T, s), d_bkt(sizeof(p3_st) * (size_t)n_msm * p.nw * B * p.parts, s);
        a.bm_start = d_start.as<uint32_t>(); a.bm_cur = d_cur.as<uint32_t>(); a.bm_sorted = d_sorted.as<uint32_t>(); a.bm_bkt = d_bkt.as<p3_st>(); a.parts = p.parts;
        // top window: 254 - c (nw - 1) bits.  Fewer than c - 4 -> at most B / 16 of its buckets can be hit: deal its B * parts threads out over those
        a.top_bits = (uint32_t)(254 - p.c * (p.nw - 1)); a.parts_top = 0;
        if ((int)a.top_bits < p.c - 4) a.parts_top = (uint32_t)((B * p.parts) >> (a.top_bits + 1));
        rt_memset(d_start.p, 0, 4 * nslot, s);
        const dim3 gt((unsigned)((a.T + 255) / 256), n_msm);
        LAUNCH(k_bm_hist, gt, dim3(256), s, a, 0);
        LAUNCH_COOP(k_bm_scan, dim3(p.nw, n_msm), dim3(256), s, a);
        LAUNCH(k_bm_hist, gt, dim3(256), s, a, 1);
        LAUNCH(k_bm_accum, dim3((unsigned)(((size_t)p.nw * B * p.parts + 127) / 128), n_msm), dim3(128), s, a);
        LAUNCH_COOP(k_bm_reduce, dim3(p.nw, n_msm), dim3(128), s, a);
    } else {
        const int wpb = MSM_THREADS >> (p.c - 1);
        LAUNCH_COOP(k_msm, dim3((p.nw + wpb - 1) / wpb, n_msm, p.slices), dim3(MSM_THREADS), s, a);
    }
    rt_prof_end(PROF_MSM, tk, s);
}
static inline msm_seg mk_seg(const void *base, uint32_t count, uint32_t stride, int kind, uint32_t np = 0, int hi = 0) { msm_seg s; s.base = base; s.count = count; s.stride = stride; s.kind = kind; s.np = np; s.hi = hi; return s; }
static inline void run_finalize(cudaStream_t s, const finalize_args &f) { LAUNCH_COOP(k_finalize, dim3(f.count), dim3(FIN_THREADS), s, f); }
static inline void fin_windows(finalize_args &f, const p3_st *win, const msm_plan &p) { f.windows = win; f.c = p.c; f.nw = p.nw; f.slices = p.slices; }


// V_1..V_m into the transcripts of C chunks.  Small chunks: on the device (ts_kernels.cuh, one warp per chunk, ~2.5 us per sponge block).  Large
// chunks (resnet18-full: 2^18 commitments = 65 000 sequential Keccak-f per chunk, only C warps busy): the host's cores are ~5x faster per
// permutation, so the commitments are copied out, absorbed by host threads (one per chunk) and the 208-byte states copied back.
static void absorb_commitments(rofl_engine &e, cudaStream_t s, transcript *d_ts, const uint8_t *d_V32, int label_id, int n, int m, int C) {
    if (m <= e.ts_host_m) {
        ts_absorb_args aa = {}; aa.ts = d_ts; aa.V32 = d_V32; aa.m = (uint32_t)m; aa.n = (uint32_t)n; aa.label_id = label_id;
        LAUNCH_COOP(k_ts_absorbV, dim3(C), dim3(TS_THREADS), s, aa);
        return;
    }
    std::vector<uint8_t> hV(32 * (size_t)C * m); std::vector<transcript> ts(C);
    rt_d2h(hV.data(), d_V32, hV.size(), s); rt_sync(s);
    parallel_for(C, e.host_threads, [&](size_t c) {
        transcript &t = ts[c]; transcript_init(t, label_id ? "L2RangeProof" : "RangeProof");
        transcript_append(t, "dom-sep", (const uint8_t *)"rangeproof v1", 13);
        transcript_append_u64(t, "n", (uint64_t)n); transcript_append_u64(t, "m", (uint64_t)m);
        for (int j = 0; j < m; j++) transcript_append(t, "V", &hV[32 * (c * (size_t)m + j)], 32);
    });
    rt_h2d(d_ts, ts.data(), sizeof(transcript) * (size_t)C, s); rt_sync(s);
}

// =============================================================================================================================
// RangeProof::prove_multiple for C chunks in lock step (SURVEY.md A.3/A.4).  All pointers are device pointers except
// h_proofs (host).  d_vals: C*m shifted values, d_blind: C*m blindings (reduced), d_V32: C*m compressed commitments.
// label = transcript label ("RangeProof" / "L2RangeProof"); keys = C ChaCha20 keys (host).
// =============================================================================================================================
static void prove_chunks(rofl_engine &e, chain &q, cudaStream_t side, int label_id, int n, int m, int C, const gens_entry &g, const rt_tables *rt, const uint64_t *d_vals,
                         const sc_st *d_blind, const uint8_t *d_V32, const std::vector<uint8_t> &keys, uint8_t *h_proofs) {
    const size_t N = (size_t)n * m, NT = N * C;
    const int lgN = ilog2_sz(N);
    const size_t plen = 32 * (9 + 2 * (size_t)lgN);
    phase_trace tr(q.hi);
    // ---- device scratch.  The Merlin transcripts live on the device (ts_kernels.cuh): nothing below waits for the host until the proofs are copied out.
    dev_buf d_ts(sizeof(transcript) * (size_t)C, q), d_proofs(plen * (size_t)C, q);
    rt_stream_after(side, q.small());
    dev_buf d_keys(32 * (size_t)C, q), d_sLR(sizeof(sc_st) * 2 * NT, q), d_sums(sizeof(sc_st) * 5 * C, q);
    { std::vector<uint32_t> kw(8 * (size_t)C); for (int c = 0; c < C; c++) key_words(&kw[8 * c], &keys[32 * c]); rt_h2d(d_keys.p, kw.data(), 32 * (size_t)C, q.small()); }
    LAUNCH(k_nonces, dim3((unsigned)((NT + 255) / 256)), dim3(256), q.big(), d_sLR.as<sc_st>(), d_keys.as<uint32_t>(), n, m, NT);
    const int nbPS = (int)std::max<size_t>(1, std::min<size_t>(64, ((size_t)m + 1023) / 1024));          // blocks per chunk of the per-party sums
    dev_buf d_partPS(sizeof(sc_st) * 3 * (size_t)C * nbPS, q);
    { pow_tab none = {nullptr, 0, 0};
      LAUNCH_COOP(k_party_sums, dim3(nbPS, C), dim3(256), q.small(), d_partPS.as<sc_st>(), d_keys.as<uint32_t>(), d_blind, (const sc_st *)nullptr, none, n, m, 0);
      LAUNCH_COOP(k_sc_sum, dim3(C), dim3(256), q.small(), d_sums.as<sc_st>(), d_partPS.as<sc_st>(), nbPS, 2); }
    // ---- A
    const int nbA = (int)std::min<size_t>(64, (N + 511) / 512);
    dev_buf d_partA(sizeof(p3_st) * (size_t)C * nbA, q), d_AS(64 * (size_t)C, q);
    LAUNCH_COOP(k_bits_sum, dim3(nbA, C), dim3(128), q.big(), d_partA.as<p3_st>(), d_vals, g.G, g.H, n, m);
    {
        finalize_args f = {}; f.partial = d_partA.as<p3_st>(); f.npartial = nbA; f.sHa = d_sums.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
        f.out32 = d_AS.as<uint8_t>(); f.count = C;
        run_finalize(q.small(), f);
    }
    // ---- S = (sum s_bl) H + <s_L, G> + <s_R, H>
    if (rt) {
        const int nbS = rt_blocks(2 * N, C, e.rt_per);
        dev_buf d_partS(sizeof(p3_st) * (size_t)C * nbS, q);
        rt_msm_args a = {}; a.scalars = d_sLR.as<sc_st>(); a.T = (uint32_t)(2 * N); a.scalar_stride = (uint32_t)(2 * N); a.nG = (uint32_t)N; a.mode = 0; a.rt = *rt; a.partial = d_partS.as<p3_st>();
        run_rt_msm(e, q.big(), a, nbS, C);
        finalize_args f = {}; f.partial = d_partS.as<p3_st>(); f.npartial = nbS; f.sHa = d_sums.as<sc_st>() + C; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
        f.out32 = d_AS.as<uint8_t>() + 32 * (size_t)C; f.count = C;
        run_finalize(q.small(), f);
    } else {
        const msm_plan pl = msm_plan_for(2 * N, C);
        dev_buf d_winS(sizeof(p3_st) * pl.out_count(C), q);
        msm_args a = {}; a.v[0].scalars = d_sLR.as<sc_st>(); a.split = (uint32_t)C; a.T = (uint32_t)(2 * N); a.scalar_stride = (uint32_t)(2 * N);
        a.v[0].seg[0] = mk_seg(g.G, (uint32_t)N, 0, 0); a.v[0].seg[1] = mk_seg(g.H, (uint32_t)N, 0, 0); a.nseg = 2; a.out = d_winS.as<p3_st>();
        run_msm(e, q.big(), a, pl, C);
        finalize_args f = {}; fin_windows(f, d_winS.as<p3_st>(), pl); f.sHa = d_sums.as<sc_st>() + C; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
        f.out32 = d_AS.as<uint8_t>() + 32 * (size_t)C; f.count = C;
        run_finalize(q.small(), f);
    }
    // ---- transcripts: V_1..V_m are independent of A and S: absorbed on the side stream while the kernels queued above run
    absorb_commitments(e, side, d_ts.as<transcript>(), d_V32, label_id, n, m, C);
    rt_stream_after(q.small(), side);
    dev_buf d_ypow2(sizeof(sc_st) * 32 * C, q), d_zpow2(sizeof(sc_st) * 32 * C, q), d_yinvpow2(sizeof(sc_st) * 32 * C, q), d_z(sizeof(sc_st) * C, q);
    { ts_yz_args ya = {}; ya.ts = d_ts.as<transcript>(); ya.AS = d_AS.as<uint8_t>(); ya.proofs = d_proofs.as<uint8_t>(); ya.plen = (uint32_t)plen; ya.C = (uint32_t)C;
      ya.ypow2 = d_ypow2.as<sc_st>(); ya.zpow2 = d_zpow2.as<sc_st>(); ya.yinvpow2 = d_yinvpow2.as<sc_st>(); ya.z = d_z.as<sc_st>();
      LAUNCH_COOP(k_ts_yz, dim3(C), dim3(TS_THREADS), q.small(), ya); }
    // ---- polynomials
    const int nbP = (int)std::min<size_t>(256, (N + 255) / 256);
    dev_buf d_a(sizeof(sc_st) * NT, q), d_b(sizeof(sc_st) * NT, q), d_part(sizeof(sc_st) * 3 * (size_t)C * nbP, q), d_tsum(sizeof(sc_st) * 3 * C, q);
    // split power tables for y^k, y^-k (k < N) and z^j (j < m)
    const int lgm = ilog2_sz((size_t)m);
    pow_tab ytab = {nullptr, lgN / 2, lgN - lgN / 2}, yitab = ytab, ztab = {nullptr, lgm / 2, lgm - lgm / 2};
    dev_buf d_ptab(sizeof(sc_st) * (size_t)C * (2 * pow_tab_size(ytab) + pow_tab_size(ztab)), q);
    ytab.tab = d_ptab.as<sc_st>(); yitab.tab = ytab.tab + (size_t)C * pow_tab_size(ytab); ztab.tab = yitab.tab + (size_t)C * pow_tab_size(yitab);
    LAUNCH(k_pow_tables, dim3((pow_tab_size(ytab) + 255) / 256, C), dim3(256), q.small(), (sc_st *)ytab.tab, d_ypow2.as<sc_st>(), ytab.L, ytab.H);
    LAUNCH(k_pow_tables, dim3((pow_tab_size(yitab) + 255) / 256, C), dim3(256), q.small(), (sc_st *)yitab.tab, d_yinvpow2.as<sc_st>(), yitab.L, yitab.H);
    LAUNCH(k_pow_tables, dim3((pow_tab_size(ztab) + 255) / 256, C), dim3(256), q.small(), (sc_st *)ztab.tab, d_zpow2.as<sc_st>(), ztab.L, ztab.H);
    LAUNCH_COOP(k_poly, dim3(nbP, C), dim3(256), q.big(), d_a.as<sc_st>(), d_b.as<sc_st>(), d_sLR.as<sc_st>(), d_part.as<sc_st>(), d_vals, ytab, ztab, d_zpow2.as<sc_st>(), n, m);
    LAUNCH_COOP(k_sc_sum, dim3(C), dim3(256), q.small(), d_tsum.as<sc_st>(), d_part.as<sc_st>(), nbP, 3);
    LAUNCH_COOP(k_party_sums, dim3(nbPS, C), dim3(256), q.small(), d_partPS.as<sc_st>(), d_keys.as<uint32_t>(), d_blind, d_z.as<sc_st>(), ztab, n, m, 1);
    LAUNCH_COOP(k_sc_sum, dim3(C), dim3(256), q.small(), d_sums.as<sc_st>() + 2 * (size_t)C, d_partPS.as<sc_st>(), nbPS, 3);
    dev_buf d_t12(sizeof(sc_st) * 2 * C, q), d_T12(64 * (size_t)C, q);
    LAUNCH(k_ts_t12, dim3((unsigned)((C + 63) / 64)), dim3(64), q.small(), d_t12.as<sc_st>(), d_tsum.as<sc_st>(), (uint32_t)C);
    {
        finalize_args f = {}; f.sBa = d_t12.as<sc_st>(); f.sHa = d_sums.as<sc_st>() + 2 * C; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
        f.out32 = d_T12.as<uint8_t>(); f.count = 2 * C;
        run_finalize(q.small(), f);
    }
    // ---- x, shares, w
    dev_buf d_x(sizeof(sc_st) * C, q), d_w2(sizeof(sc_st) * 2 * C, q), d_yinv(sizeof(sc_st) * NT, q);
    { ts_x_args xa = {}; xa.ts = d_ts.as<transcript>(); xa.T12 = d_T12.as<uint8_t>(); xa.proofs = d_proofs.as<uint8_t>(); xa.plen = (uint32_t)plen; xa.C = (uint32_t)C;
      xa.tsum = d_tsum.as<sc_st>(); xa.sums = d_sums.as<sc_st>(); xa.x = d_x.as<sc_st>(); xa.w2 = d_w2.as<sc_st>(); xa.N = (uint64_t)N;
      LAUNCH_COOP(k_ts_x, dim3(C), dim3(TS_THREADS), q.small(), xa); }
    LAUNCH(k_lr, dim3((unsigned)((NT + 255) / 256)), dim3(256), q.big(), d_a.as<sc_st>(), d_b.as<sc_st>(), d_sLR.as<sc_st>(), d_yinv.as<sc_st>(), d_x.as<sc_st>(), yitab, N, NT);
    tr.mark("pre_ipp");
    // ---- inner product argument
    // folded generators [C][half]; a tail that starts at round 0 keeps all N original generators there instead
    const size_t half = (N / 2 <= (size_t)std::min(e.tail_np, TAIL_MAX_F / 2)) ? N : (N / 2 ? N / 2 : 1);
    dev_buf d_Gf(sizeof(p3_st) * half * C, q), d_Hf(sizeof(p3_st) * half * C, q);
    sc_st *msmL = d_sLR.as<sc_st>(), *msmR = d_sLR.as<sc_st>() + NT;         // s_L / s_R are dead after k_lr: reuse as MSM scalar buffers
    dev_buf d_cLR(sizeof(sc_st) * 2 * C, q), d_LR(64 * (size_t)C, q), d_u2(sizeof(sc_st) * C, q), d_uinv2(sizeof(sc_st) * C, q), d_nafs(512 * (size_t)C, q), d_up(sizeof(sc_st) * 2 * (size_t)C, q);
    { std::vector<sc_st> h_up(2 * (size_t)C); sc one; sc_from_u64(one, 1); for (auto &v : h_up) sc_to_st(v, one); rt_h2d(d_up.p, h_up.data(), sizeof(sc_st) * h_up.size(), q.small()); }
    // RT path: the first r_unf rounds take L/R as table MSMs over the ORIGINAL generators (no generator folding), then one
    // catch-up fold builds G"/H" of length N >> r_unf directly from the tables (DESIGN.md section 3)
    // rounds with half-size <= tail_np run in the fused on-device tail kernel; `pre` rounds come before it
    const size_t tail_np = (size_t)std::min(e.tail_np, TAIL_MAX_F / 2);
    int pre = 0; while (pre < lgN && ((N / 2) >> pre) > tail_np) pre++;
    // without tables (chunks of 2^18 values and more): the same unfolded rounds as wide-window Pippenger MSMs over the original generators, then a
    // joint double-and-add catch-up (k_catchup_naf) -- 2^r bases per output share 252 doublings instead of a fold ladder per base and level
    const int r_unf = rt ? std::min({e.rt_unfold, lgN, pre}) : ((N >= (size_t)e.nt_unfold_min && e.nt_unfold > 0) ? std::min({e.nt_unfold, lgN, pre, 4}) : 0);
    const int nbU = rt ? rt_blocks(N, 2 * C, e.rt_per) : 1;
    const uint32_t cstride = 1u << (r_unf > 0 ? r_unf : 0);
    // coefficient tables of the unfolded rounds [G | H][C][cstride], kept on the device: k_ts_round doubles them after every challenge
    auto coef_init = [&](dev_buf &d, uint32_t stride) {
        std::vector<sc_st> h(2 * (size_t)C * stride); memset(h.data(), 0, sizeof(sc_st) * h.size());
        for (size_t c = 0; c < 2 * (size_t)C; c++) h[c * stride].w[0] = 1;
        rt_h2d(d.p, h.data(), sizeof(sc_st) * h.size(), q.small());
    };
    dev_buf d_cGH(sizeof(sc_st) * 2 * (size_t)C * cstride, q), d_partU(sizeof(p3_st) * 2 * (size_t)C * nbU, q), d_digs(rt ? sizeof(int16_t) * 2 * (size_t)C * cstride * RT_MAXW : 256 * 2 * (size_t)C * cstride, q);
    coef_init(d_cGH, cstride);
    const int nbQ = (int)std::min<size_t>(256, (N / 2 + 255) / 256);
    dev_buf d_partQ(sizeof(sc_st) * 2 * (size_t)C * nbQ, q);
    // frozen level (kernels.cuh K6c): rounds ra .. pre-1 run over the generators as they are at round ra (FA of G" and of H" per chunk)
    int ra = -1; size_t FA = 0; uint32_t cAstride = 1;
    if (e.use_frz) {
        int r = std::max(r_unf, 1);
        while (r < pre && 2 * ((N / 2) >> r) > FRZ_MAX_F) r++;
        const size_t fa = r < lgN ? 2 * ((N / 2) >> r) : 0;
        const double need = (double)C * 2 * fa * FRZ_Q * (FRZ_E + 1) * sizeof(p3_st);
        // (the budget check uses the free memory recorded when the tables were built: cudaMemGetInfo itself blocks for tens of
        //  milliseconds every now and then -- it was the cause of the "slow steps" of DESIGN.md section 7)
        if (e.sh->free_hint.load() == 0) e.sh->free_hint = rt_free_mem();
        if (pre - r >= 2 && fa >= 4 && need < 0.25 * (double)e.sh->free_hint.load()) { ra = r; FA = fa; cAstride = (uint32_t)(FA / ((N / 2) >> (pre - 1))); }
    }
    dev_buf d_cA(sizeof(sc_st) * 2 * (size_t)C * cAstride, q), d_frzV(sizeof(p3_st) * 2 * (size_t)C * 8, q);
    coef_init(d_cA, cAstride);
    dev_buf d_frzT(ra >= 0 ? sizeof(p3_st) * (size_t)C * 2 * FA * FRZ_Q * FRZ_E : 16, q);
    dev_buf d_dg(ra >= 0 ? 2 * (size_t)C * cAstride * 64 : 16, q);             // radix-16 digits of the frozen level's coefficients when it is left
    int round = 0;
    bool tail_done = false;
    for (size_t np = N / 2; np >= 1; np /= 2, round++) {
        if (round == r_unf) tr.mark("unfolded");
        if (round == ra) {           // enter the frozen level: Straus tables of the current G", H"
            dev_buf d_bases(sizeof(p3_st) * (size_t)C * 2 * FA * FRZ_Q, q);      // returned stream-ordered: the kernels below may still be running
            q.big();
            void *tk = rt_prof_begin(PROF_FRZ, q.cur ? q.lo : q.hi);
            LAUNCH(k_frz_bases, dim3((unsigned)((2 * FA + 127) / 128), C), dim3(128), q.big(), d_bases.as<p3_st>(), d_Gf.as<p3_st>(), d_Hf.as<p3_st>(), (uint32_t)FA, (uint32_t)half, (uint32_t)FRZ_Q, 32u);
            const size_t cnt = (size_t)C * 2 * FA * FRZ_Q;
            LAUNCH(k_frz_tables, dim3((unsigned)((cnt + 127) / 128)), dim3(128), q.big(), d_frzT.as<p3_st>(), d_bases.as<p3_st>(), cnt);
            rt_prof_end(PROF_FRZ, tk, q.cur ? q.lo : q.hi);
        }
        const bool frozen = ra >= 0 && round >= ra;
        if (round == pre) tr.mark("middle");
        if (round == pre && frozen) {       // leave the frozen level: the 2*np generators the tail starts from, straight from the tables
            const uint32_t nblk = (uint32_t)(FA / (2 * np));                  // == cAstride: the digits were written by the last frozen round's k_ts_round
            frz_exit_args xa = {}; xa.T = d_frzT.as<p3_st>(); xa.digs = d_dg.as<int8_t>(); xa.Gf = d_Gf.as<p3_st>(); xa.Hf = d_Hf.as<p3_st>();
            xa.F = (uint32_t)FA; xa.Fo = (uint32_t)(2 * np); xa.nblk = nblk; xa.stride = (uint32_t)half;
            dev_buf d_xV(sizeof(p3_st) * (size_t)C * 2 * xa.Fo * 8, q); xa.V = d_xV.as<p3_st>();
            void *tk = rt_prof_begin(PROF_FRZ, q.cur ? q.lo : q.hi);
            LAUNCH_COOP(k_frz_exit, dim3((unsigned)(2 * np), C, 2), dim3(128), q.small(), xa);
            LAUNCH(k_frz_exit_chain, dim3((unsigned)(((size_t)C * 2 * xa.Fo + 127) / 128)), dim3(128), q.small(), xa, (uint32_t)C);
            rt_prof_end(PROF_FRZ, tk, q.cur ? q.lo : q.hi);
        }
        if (round == pre) tr.mark("exit");
        if (round == pre) {          // np <= tail_np: every remaining round in one launch (kernels.cuh, k_ipp_tail)
            // freeze the 2*np generators the tail works on: Straus tables (kernels.cuh K6c), built once for all its rounds
            const uint32_t Ft = (uint32_t)(2 * np);
            if (round == 0) LAUNCH(k_niels_to_p3, dim3((Ft + 127) / 128, C), dim3(128), q.small(), d_Gf.as<p3_st>(), d_Hf.as<p3_st>(), g.G, g.H, Ft, (uint32_t)half);
            // tables of the tail: (k+1) 16^pos P for every radix-16 digit position (TAIL_Q = 64 per point; 8 MB per chunk): a round is then a plain sum
            // of table entries -- the 28-doubling chain per round that octant tables need was 215 k cycles of one lane in each of the six rounds
            // (the tables are built and used for at most Cb chunks at a time: 2 GB of them however many chunks a call has)
            const size_t per_chunk = sizeof(p3_st) * 2 * (size_t)Ft * TAIL_Q * (FRZ_E + 1);
            const size_t Cb = std::max<size_t>(1, std::min<size_t>((size_t)C, ((size_t)e.tail_batch_mb << 20) / per_chunk));
            dev_buf d_tb(sizeof(p3_st) * Cb * 2 * Ft * TAIL_Q, q), d_tT(sizeof(p3_st) * Cb * 2 * Ft * TAIL_Q * FRZ_E, q);
            dev_buf d_tscr(sizeof(p3_st) * 512 * Cb, q), d_gfac(sizeof(sc_st) * 3 * Cb, q);
            static const bool tail_dbg = getenv("ROFL_TAIL_DBG") != nullptr;
            dev_buf d_tdbg(tail_dbg ? 128 * sizeof(long long) : 16, q);
            void *tk = rt_prof_begin(PROF_TAIL, q.cur ? q.lo : q.hi);
            for (size_t c0 = 0; c0 < (size_t)C; c0 += Cb) {
                const unsigned Cn = (unsigned)std::min<size_t>(Cb, (size_t)C - c0);
                const p3_st *Gb = d_Gf.as<p3_st>() + c0 * half, *Hb = d_Hf.as<p3_st>() + c0 * half;
#ifdef ROFL_EMUL
                LAUNCH(k_frz_bases, dim3((2 * Ft + 127) / 128, Cn), dim3(128), q.small(), d_tb.as<p3_st>(), Gb, Hb, Ft, (uint32_t)half, (uint32_t)TAIL_Q, 4u);
#else
                LAUNCH(k_frz_bases4, dim3((4 * 2 * Ft + 127) / 128, Cn), dim3(128), q.small(), d_tb.as<p3_st>(), Gb, Hb, Ft, (uint32_t)half, (uint32_t)TAIL_Q, 4u);
#endif
                LAUNCH(k_frz_tables, dim3((unsigned)(((size_t)Cn * 2 * Ft * TAIL_Q + 127) / 128)), dim3(128), q.small(), d_tT.as<p3_st>(), d_tb.as<p3_st>(), (size_t)Cn * 2 * Ft * TAIL_Q);
                tail_args ta = {}; ta.T = d_tT.as<p3_st>();
                ta.a = d_a.as<sc_st>() + c0 * N; ta.b = d_b.as<sc_st>() + c0 * N; ta.yinv = d_yinv.as<sc_st>() + c0 * N; ta.N = N;
                ta.ts = d_ts.as<transcript>() + c0; ta.w = d_w2.as<sc_st>() + c0; ta.uprod = d_up.as<sc_st>() + c0; ta.uinvprod = d_up.as<sc_st>() + C + c0; ta.tabB = e.sh->tabB;
                ta.scratch = d_tscr.as<p3_st>(); ta.gfac = d_gfac.as<sc_st>();
                ta.out = d_proofs.as<uint8_t>() + c0 * plen + 224 + 64 * (size_t)round; ta.out_stride = (uint32_t)plen; ta.F = Ft;
                if (tail_dbg && c0 == 0) { rt_memset(d_tdbg.p, 0, 128 * sizeof(long long), q.small()); ta.dbg = d_tdbg.as<long long>(); }
#ifdef ROFL_EMUL
                ta.ncta = 1;
#else
                ta.ncta = (uint32_t)e.tail_ncta;
#endif
                LAUNCH_COOP(k_ipp_tail, dim3((unsigned)(Cn * ta.ncta)), dim3(TAIL_THREADS), q.small(), ta);
            }
            if (tail_dbg) {
                long long h[128]; rt_d2h(h, d_tdbg.p, sizeof(h), q.small()); rt_sync(q.small());
                static const char *nm[7] = {"digits", "c_tree", "table_adds", "point_tree", "chain+compress", "transcript+invert", "folds"};
                for (int r = 0; r < 8 && h[8 * r]; r++) { fprintf(stderr, "[rofl tail] round %d:", r); for (int k = 0; k < 7; k++) fprintf(stderr, " %s=%lld", nm[k], h[8 * r + k + 1] - h[8 * r + k]); fprintf(stderr, "\n"); }
                fprintf(stderr, "[rofl tail] round 2, per warp (table loop, shuffle tree):"); for (int w = 0; w < 16; w++) fprintf(stderr, " (%lld, %lld)", h[64 + 2 * w], h[64 + 2 * w + 1]); fprintf(stderr, "  c w B threads: %lld\n", h[96]);
            }
            rt_prof_end(PROF_TAIL, tk, q.cur ? q.lo : q.hi);
            tail_done = true;
            break;
        }
        const int nbI = (int)std::min<size_t>(256, (np + 255) / 256);
        const bool unfolded = round < r_unf;
        if (frozen) {
            const int nbQA = (int)std::min<size_t>(256, (FA / 2 + 255) / 256);
            LAUNCH_COOP(k_ipp_scalars_unf, dim3(nbQA, C), dim3(256), q.small(), d_a.as<sc_st>(), d_b.as<sc_st>(), d_yinv.as<sc_st>(), d_cA.as<sc_st>(), d_cA.as<sc_st>() + (size_t)C * cAstride, cAstride,
                        msmL, msmR, d_partQ.as<sc_st>(), N, (uint32_t)np, (uint32_t)FA);
            LAUNCH_COOP(k_sc_sum, dim3(C), dim3(256), q.small(), d_cLR.as<sc_st>(), d_partQ.as<sc_st>(), nbQA, 2);
            frz_reduce_args ra_ = {}; ra_.T = d_frzT.as<p3_st>(); ra_.msmL = msmL; ra_.msmR = msmR; ra_.V = d_frzV.as<p3_st>(); ra_.F = (uint32_t)FA; ra_.np = (uint32_t)np; ra_.C = (uint32_t)C;
            void *tk = rt_prof_begin(PROF_FRZ, q.cur ? q.lo : q.hi);
            LAUNCH_COOP(k_frz_reduce, dim3(8, 2 * C), dim3(128), q.small(), ra_);
            rt_prof_end(PROF_FRZ, tk, q.cur ? q.lo : q.hi);
            finalize_args f = {}; f.windows = d_frzV.as<p3_st>(); f.c = 4; f.nw = 8; f.slices = 1; f.sBa = d_cLR.as<sc_st>(); f.sBb = d_w2.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
            f.out32 = d_LR.as<uint8_t>(); f.count = 2 * C;
            run_finalize(q.small(), f);
        } else if (unfolded) {
            LAUNCH_COOP(k_ipp_scalars_unf, dim3(nbQ, C), dim3(256), q.big(), d_a.as<sc_st>(), d_b.as<sc_st>(), d_yinv.as<sc_st>(), d_cGH.as<sc_st>(), d_cGH.as<sc_st>() + (size_t)C * cstride, cstride,
                        msmL, msmR, d_partQ.as<sc_st>(), N, (uint32_t)np, (uint32_t)N);
            LAUNCH_COOP(k_sc_sum, dim3(C), dim3(256), q.small(), d_cLR.as<sc_st>(), d_partQ.as<sc_st>(), nbQ, 2);
            if (rt) {
                rt_msm_args aL = {}; aL.scalars = msmL; aL.T = (uint32_t)N; aL.scalar_stride = (uint32_t)N; aL.nG = (uint32_t)(N / 2); aL.np = (uint32_t)np; aL.mode = 1; aL.rt = *rt; aL.partial = d_partU.as<p3_st>();
                rt_msm_args aR = aL; aR.scalars = msmR; aR.mode = 2; aR.partial = d_partU.as<p3_st>() + (size_t)C * nbU;
                run_rt_msm(e, q.big(), aL, nbU, C); run_rt_msm(e, q.big(), aR, nbU, C);
                finalize_args f = {}; f.partial = d_partU.as<p3_st>(); f.npartial = nbU; f.sBa = d_cLR.as<sc_st>(); f.sBb = d_w2.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
                f.out32 = d_LR.as<uint8_t>(); f.count = 2 * C;
                run_finalize(q.small(), f);
            } else {
                // L: G-terms on the hi halves, H-terms on the lo halves of the 2np-blocks of the ORIGINAL generators; R: the other way round
                const msm_plan pl = msm_plan_for(N, 2 * (size_t)C);
                dev_buf d_win(sizeof(p3_st) * pl.out_count(2 * (size_t)C), q);
                msm_args a = {}; a.v[0].scalars = msmL; a.v[1].scalars = msmR; a.split = (uint32_t)C; a.T = (uint32_t)N; a.scalar_stride = (uint32_t)N; a.nseg = 2; a.out = d_win.as<p3_st>();
                a.v[0].seg[0] = mk_seg(g.G, (uint32_t)(N / 2), 0, 0, (uint32_t)np, 1); a.v[0].seg[1] = mk_seg(g.H, (uint32_t)(N / 2), 0, 0, (uint32_t)np, 0);
                a.v[1].seg[0] = mk_seg(g.G, (uint32_t)(N / 2), 0, 0, (uint32_t)np, 0); a.v[1].seg[1] = mk_seg(g.H, (uint32_t)(N / 2), 0, 0, (uint32_t)np, 1);
                run_msm(e, q.big(), a, pl, 2 * (uint32_t)C);
                finalize_args f = {}; fin_windows(f, d_win.as<p3_st>(), pl); f.sBa = d_cLR.as<sc_st>(); f.sBb = d_w2.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
                f.out32 = d_LR.as<uint8_t>(); f.count = 2 * C;
                run_finalize(q.small(), f);
            }
        } else {
            LAUNCH_COOP(k_ipp_scalars, dim3(nbI, C), dim3(256), q.small(), d_a.as<sc_st>(), d_b.as<sc_st>(), d_yinv.as<sc_st>(), msmL, msmR, d_part.as<sc_st>(), N, (uint32_t)np);
            LAUNCH_COOP(k_sc_sum, dim3(C), dim3(256), q.small(), d_cLR.as<sc_st>(), d_part.as<sc_st>(), nbI, 2);
            // L and R of every chunk in one launch: msm = lr*C + c
            const msm_plan pl = msm_plan_for(2 * np, 2 * (size_t)C);
            dev_buf d_win(sizeof(p3_st) * pl.out_count(2 * (size_t)C), q);
            msm_args a = {}; a.v[0].scalars = msmL; a.v[1].scalars = msmR; a.split = (uint32_t)C;
            a.T = (uint32_t)(2 * np); a.scalar_stride = (uint32_t)(2 * np); a.nseg = 2; a.out = d_win.as<p3_st>();
            if (round == 0) {
                a.v[0].seg[0] = mk_seg(g.G + np, (uint32_t)np, 0, 0); a.v[0].seg[1] = mk_seg(g.H, (uint32_t)np, 0, 0);
                a.v[1].seg[0] = mk_seg(g.G, (uint32_t)np, 0, 0);      a.v[1].seg[1] = mk_seg(g.H + np, (uint32_t)np, 0, 0);
            } else {
                a.v[0].seg[0] = mk_seg(d_Gf.as<p3_st>() + np, (uint32_t)np, (uint32_t)half, 1); a.v[0].seg[1] = mk_seg(d_Hf.as<p3_st>(), (uint32_t)np, (uint32_t)half, 1);
                a.v[1].seg[0] = mk_seg(d_Gf.as<p3_st>(), (uint32_t)np, (uint32_t)half, 1);      a.v[1].seg[1] = mk_seg(d_Hf.as<p3_st>() + np, (uint32_t)np, (uint32_t)half, 1);
            }
            run_msm(e, q.big(), a, pl, 2 * (uint32_t)C);
            finalize_args f = {}; fin_windows(f, d_win.as<p3_st>(), pl); f.sBa = d_cLR.as<sc_st>(); f.sBb = d_w2.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
            f.out32 = d_LR.as<uint8_t>(); f.count = 2 * C;
            run_finalize(q.small(), f);
        }
        // ---- L, R -> u on the device, with everything the next kernels need from it (ts_kernels.cuh, k_ts_round)
        const bool catchup = unfolded && round + 1 == r_unf && np >= 2, fold = !frozen && !unfolded && np >= 2;
        {
            ts_round_args t = {}; t.ts = d_ts.as<transcript>(); t.LR = d_LR.as<uint8_t>(); t.proofs = d_proofs.as<uint8_t>(); t.plen = (uint32_t)plen; t.off = (uint32_t)(224 + 64 * round); t.C = (uint32_t)C;
            t.yinvpow2 = d_yinvpow2.as<sc_st>(); t.lgnp = ilog2_sz(np); t.u2 = d_u2.as<sc_st>(); t.uinv2 = d_uinv2.as<sc_st>(); t.up = d_up.as<sc_st>();
            if (frozen) { t.coefG = d_cA.as<sc_st>(); t.coefH = d_cA.as<sc_st>() + (size_t)C * cAstride; t.cstride = cAstride; t.nblk = (uint32_t)(FA / (2 * np)); if (round + 1 == pre && pre < lgN) { t.emit = 3; t.digs8 = d_dg.as<int8_t>(); } }
            else if (unfolded) { t.coefG = d_cGH.as<sc_st>(); t.coefH = d_cGH.as<sc_st>() + (size_t)C * cstride; t.cstride = cstride; t.nblk = 1u << round;
                                 if (catchup && rt) { t.emit = 2; t.digs16 = d_digs.as<int16_t>(); for (int i = 0; i < 9; i++) t.rtK[i] = rt->K[i]; t.rtc = rt->c; t.rtnw = rt->nw; }
                                 else if (catchup) { t.emit = 4; t.nafs = d_digs.as<int8_t>(); } }
            else if (fold) { t.emit = 1; t.nafs = d_nafs.as<int8_t>(); }
            LAUNCH_COOP(k_ts_round, dim3(C), dim3(TS_THREADS), q.small(), t);
        }
        LAUNCH(k_ipp_fold_scalars, dim3((unsigned)((np + 255) / 256), C), dim3(256), q.small(), d_a.as<sc_st>(), d_b.as<sc_st>(), d_u2.as<sc_st>(), d_uinv2.as<sc_st>(), N, (uint32_t)np);
        if (catchup && rt) {         // G", H" of length np straight from the tables
            catchup_args ca = {}; ca.rt = *rt; ca.Gf = d_Gf.as<p3_st>(); ca.Hf = d_Hf.as<p3_st>(); ca.digits = d_digs.as<int16_t>(); ca.nr = (uint32_t)np; ca.nblk = 1u << r_unf; ca.stride = (uint32_t)half;
            q.big();
            void *tk = rt_prof_begin(PROF_FOLD, q.cur ? q.lo : q.hi);
            LAUNCH_COOP(k_rt_catchup, dim3((unsigned)((np + 127) / 128), C, 2), dim3(128), q.big(), ca);
            rt_prof_end(PROF_FOLD, tk, q.cur ? q.lo : q.hi);
        } else if (catchup) {        // ... or by one joint double-and-add over the 2^r_unf original generators of every output
            catchup_naf_args ca = {}; ca.G = g.G; ca.H = g.H; ca.Gf = d_Gf.as<p3_st>(); ca.Hf = d_Hf.as<p3_st>(); ca.nafs = d_digs.as<int8_t>(); ca.nr = (uint32_t)np; ca.nblk = 1u << r_unf; ca.stride = (uint32_t)half;
            q.big();
            void *tk = rt_prof_begin(PROF_FOLD, q.cur ? q.lo : q.hi);
            LAUNCH_COOP(k_catchup_naf, dim3((unsigned)((np + 127) / 128), C, 2), dim3(128), q.big(), ca);
            rt_prof_end(PROF_FOLD, tk, q.cur ? q.lo : q.hi);
        } else if (fold) {
            fold_args fa = {}; fa.Gn = round == 0 ? g.G : nullptr; fa.Hn = round == 0 ? g.H : nullptr;
            fa.Gf = d_Gf.as<p3_st>(); fa.Hf = d_Hf.as<p3_st>(); fa.nafs = d_nafs.as<int8_t>(); fa.np = (uint32_t)np; fa.stride = (uint32_t)half;
            q.big();
            void *tk = rt_prof_begin(PROF_FOLD, q.cur ? q.lo : q.hi);
            LAUNCH_COOP(k_ipp_fold_points, dim3((unsigned)((np + 127) / 128), C, 2), dim3(128), q.big(), fa);
            rt_prof_end(PROF_FOLD, tk, q.cur ? q.lo : q.hi);
        }
    }
    if (!tail_done) {            // final a, b: a = a^ prod u_k, b = b^ prod u_k^-1
        ts_final_args fa = {}; fa.a = d_a.as<sc_st>(); fa.b = d_b.as<sc_st>(); fa.up = d_up.as<sc_st>(); fa.proofs = d_proofs.as<uint8_t>(); fa.plen = (uint32_t)plen; fa.off = (uint32_t)(224 + 64 * lgN); fa.C = (uint32_t)C; fa.N = N;
        LAUNCH(k_ts_final, dim3((unsigned)((C + 63) / 64)), dim3(64), q.small(), fa);
    }
    rt_d2h(h_proofs, d_proofs.p, plen * (size_t)C, q.small());
    rt_sync(q.small());
    tr.mark("ipp");
}


// run f(group, c0, c1, queue, side stream) for `groups` contiguous chunk ranges concurrently (one host thread + one queue per group)
template <class F> static void for_chunk_groups(rofl_engine &e, lane &ln, size_t C, F f) {
    size_t G = std::max<size_t>(1, std::min<size_t>({(size_t)e.groups, (size_t)ROFL_MAX_GROUPS, C}));
    if (G == 1) { f(0, (size_t)0, C, ln.q[0], ln.side[0]); return; }
    // chunk ranges proportional to the group weights: the LAST group's latency-bound end is the only one nothing overlaps, so it gets the fewest chunks
    std::vector<size_t> cut(G + 1, 0); double tot = 0, acc = 0;
    for (size_t gi = 0; gi < G; gi++) tot += e.group_w[gi];
    for (size_t gi = 0; gi < G; gi++) { acc += e.group_w[gi]; cut[gi + 1] = gi + 1 == G ? C : std::min(C, std::max(cut[gi] + 1, (size_t)(acc / tot * (double)C + 0.5))); }
    for (size_t gi = G; gi-- > 0;) if (cut[gi + 1] <= cut[gi]) cut[gi] = cut[gi + 1] - 1;          // every group at least one chunk
    std::vector<std::thread> th; std::vector<std::string> errs(G);
    for (size_t gi = 0; gi < G; gi++) th.emplace_back([&, gi] {
        try { rt_set_device(e.device); f(gi, cut[gi], cut[gi + 1], ln.q[gi], ln.side[gi]); } catch (const std::exception &ex) { errs[gi] = ex.what(); }
    });
    for (auto &t : th) t.join();
    for (auto &m : errs) if (!m.empty()) throw std::runtime_error(m);
}

// =============================================================================================================================
// range_proof_vec::create_rangeproof (range_proof_vec/mod.rs:16-102).  d_values / d_blind / d_commits are device pointers.
// returns 0 ok, 2 ValueOutOfRangeError, -7 InvalidBitsize, -2 bad arguments, -98 NaN input (reference panics),
// -99 non power-of-two chunking (reference panics "Should not get here")
// =============================================================================================================================
// A shard = chunks [chunk_begin, chunk_begin + n_chunks) of a larger update (chunk length m): the caller passes only that
// slice of the values / blindings (D = its real elements, the rest of the m * n_chunks positions is the reference's zero
// padding) and gets exactly the proofs the whole-update call would produce for those chunks (same per-chunk nonce streams).
struct shard_spec { size_t m, chunk_begin, n_chunks; };
static int engine_range_prove(rofl_engine &e, const float *d_values, const uint8_t *d_blind, size_t D, int range, size_t n_partition,
                              int n_bits, int frac, const uint8_t seed[32], uint8_t *h_proofs, size_t *proof_len, size_t *n_proofs, uint8_t *d_commits,
                              const shard_spec *shard = nullptr) {
    if (!fp_ok(n_bits, frac) || range < 1 || range > n_bits) return -2;
    if (shard ? (shard->m == 0 || shard->n_chunks == 0 || D > shard->m * shard->n_chunks) : (D == 0 || n_partition == 0)) return -2;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const size_t Dp = shard ? shard->m * shard->n_chunks : next_pow2_sz(D);
    const size_t C = shard ? shard->n_chunks : std::min(Dp, n_partition), m = Dp / C;                         // :54-55
    const size_t c_off = shard ? shard->chunk_begin : 0;
    const bool bitsize_ok = (range == 8 || range == 16 || range == 32 || range == 64);
    const bool chunk_ok = !(m & (m - 1)) && m * C == Dp;
    dev_buf d_V(32 * Dp, s), d_vals(8 * Dp, s), d_bl(sizeof(sc_st) * Dp, s), d_flags(sizeof(int), s);
    rt_memset(d_flags.p, 0, sizeof(int), s);
    commit_args ca = {}; ca.values = d_values; ca.blind = d_blind; ca.D = D; ca.Dp = Dp; ca.n_bits = n_bits; ca.frac = frac;
    ca.shift_bits = range; ca.mx = clip_max_f(range, n_bits, frac); ca.mn = -ca.mx; ca.tabB = e.sh->tabB; ca.tabH = e.sh->tabH;
    ca.V = d_V.as<uint8_t>(); ca.C = d_commits; ca.vals = d_vals.as<uint64_t>(); ca.blind_sc = d_bl.as<sc_st>(); ca.flags = d_flags.as<int>();
    void *tk = rt_prof_begin(PROF_COMMIT, s);
    LAUNCH(k_commit, dim3((unsigned)((Dp + 127) / 128)), dim3(128), s, ca);
    rt_prof_end(PROF_COMMIT, tk, s);
    int flags = 0; rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    if (flags & 2) return 2;                                                         // :26-29
    if (flags & 1) return -98;
    if (!bitsize_ok) return ROFL_ERR_BITSIZE_;
    if (!chunk_ok) return -99;
    tables_use tu(*e.sh);
    engine_gens(e, tu, s, range, (int)m);
    rt_tables rt; const bool have_rt = engine_rt(e, tu, s, range, (int)m, rt);
    const gens_entry g = engine_gens(e, tu, s, range, (int)m);          // (read after engine_rt: an upgrade of the lock inside it lets others regrow the arrays)
    std::vector<uint8_t> keys(32 * C);
    for (size_t c = 0; c < C; c++) derive_key(&keys[32 * c], seed, DOM_RANGE_PROVE, c_off + c);
    const size_t plen = 32 * (9 + 2 * (size_t)ilog2_sz((size_t)range * m));
    for_chunk_groups(e, *lg.ln, C, [&](size_t, size_t c0, size_t c1, chain &gq, cudaStream_t side) {
        std::vector<uint8_t> k(keys.begin() + 32 * c0, keys.begin() + 32 * c1);
        prove_chunks(e, gq, side, 0, range, (int)m, (int)(c1 - c0), g, have_rt ? &rt : nullptr, d_vals.as<uint64_t>() + c0 * m, d_bl.as<sc_st>() + c0 * m, d_V.as<uint8_t>() + 32 * c0 * m, k, h_proofs + plen * c0);
    });
    *proof_len = plen; *n_proofs = C;
    return 0;
}

// =============================================================================================================================
// RangeProof::verify_multiple for C chunks (SURVEY.md A.3): d_Vp3 / d_V32 hold C*m (shifted) commitments as points / encodings (device).
// The transcripts are replayed on the device (ts_kernels.cuh) and all chunks are checked with ONE random linear combination whose weights
// are derived by Fiat-Shamir from the seed and every proof / commitment of the call.
// verdict[c] = 1 accept / 0 VerificationError.  returns 0 or a negative error (-1 FormatError).  d_xbad (nullable): one more device flag
// word fetched with the result (the caller's "a commitment did not decode").
// =============================================================================================================================
static inline int range_proof_format_check(const uint8_t *h_proofs, size_t plen, size_t C, size_t *lg_out) {       // RangeProof::from_bytes / InnerProductProof::from_bytes
    if (plen % 32 || plen < 7 * 32) return -1;
    const size_t ne = plen / 32 - 7;
    if (ne < 2 || (ne - 2) % 2) return -1;
    const size_t lg = (ne - 2) / 2; if (lg >= 32) return -1;
    for (size_t c = 0; c < C; c++) {
        const uint8_t *p = h_proofs + plen * c; sc t;
        for (size_t off : {(size_t)128, (size_t)160, (size_t)192, 224 + 64 * lg, 224 + 64 * lg + 32}) { sc_frombytes(t, p + off); if (!sc_is_canonical(t)) return -1; }
    }
    if (lg_out) *lg_out = lg;
    return 0;
}
// Test hook (rofl_debug_range_terms): every verify_chunks invocation that builds the batched equation appends one record, copied from the device
// buffers it already filled; nothing is derived here.  With a null tap verify_chunks issues exactly its production launches and copies.
struct range_tap {
    struct rec {
        int C = 0, n = 0, m = 0, lgN = 0; uint64_t c_off = 0; uint32_t dom = 0;
        int rt = 0, c = 0;                              // fixed-generator MSM: 1 generator tables (k_rt_msm), 0 bucket MSM; its window width
        std::vector<sc_st> vch, ccrho, chal, var, gh;   // y z x w u_0.. per chunk | c_i, rho_i | chal blocks | C m commitment + C nsmall small-point scalars | g, h
        std::vector<uint8_t> digest; std::vector<int> bad; int id = 0;
    };
    std::vector<rec> recs;
};
static int verify_chunks(rofl_engine &e, cudaStream_t s, int label_id, int n, int m, int C, const gens_entry &g, const rt_tables *rt, const p3_st *d_Vp3, const uint8_t *d_V32,
                         const uint8_t *h_proofs, size_t plen, const uint8_t seed[32], uint32_t dom, uint64_t c_off, std::vector<int> &verdict, const int *d_xbad = nullptr, int *h_xbad = nullptr,
                         range_tap *tap = nullptr, size_t nx = 1) {
    verdict.assign(C, 0);
    phase_trace tr(s);
    size_t lg = 0;
    if (range_proof_format_check(h_proofs, plen, (size_t)C, &lg)) return -1;
    const size_t N = (size_t)n * m;
    if ((m & (m - 1)) || N != ((size_t)1 << lg)) {                      // verification_scalars: n != 1 << lg_n -> VerificationError (all chunks false)
        if (d_xbad) { rt_d2h(h_xbad, d_xbad, sizeof(int) * nx, s); rt_sync(s); }
        return 0;
    }
    const int lgN = (int)lg, nsmall = 6 + 2 * lgN, lgm = ilog2_sz((size_t)m);
    // all C chunks are checked with ONE equation: sum_c rho_c * (chunk c's mega-check) == identity (kernels.cuh, k_verify_scalars)
    const int chs = 5 + 2 * lgN;
    const uint32_t vstride = (uint32_t)(m + nsmall);
    const vtab_layout vt = vtab_make(lgN, lgm);
    dev_buf d_proofs(plen * (size_t)C, s), d_ts(sizeof(transcript) * (size_t)C, s), d_vch(sizeof(sc_st) * (size_t)C * (4 + lgN), s), d_digest(32 * (size_t)C, s), d_ccrho(sizeof(sc_st) * 2 * (size_t)C, s);
    dev_buf d_chal(sizeof(sc_st) * (size_t)C * chs, s), d_yinvpow2(sizeof(sc_st) * 32 * C, s), d_zpow2(sizeof(sc_st) * 32 * C, s);
    dev_buf d_tab(sizeof(sc_st) * (size_t)C * vt.total, s), d_gh(sizeof(sc_st) * 2 * N, s), d_var(sizeof(sc_st) * (size_t)C * vstride, s);
    dev_buf d_sp32(32 * (size_t)C * nsmall, s), d_sp(sizeof(p3_st) * (size_t)C * nsmall, s), d_bad(sizeof(int) * C, s), d_id(sizeof(int), s), d_fix(sizeof(p3_st), s);
    rt_h2d(d_proofs.p, h_proofs, plen * (size_t)C, s);
    rt_memset(d_bad.p, 0, sizeof(int) * C, s);
    absorb_commitments(e, s, d_ts.as<transcript>(), d_V32, label_id, n, m, C);
    { ts_verify_args va = {}; va.ts = d_ts.as<transcript>(); va.proofs = d_proofs.as<uint8_t>(); va.plen = (uint32_t)plen; va.C = (uint32_t)C; va.lgN = lgN; va.N = (uint64_t)N;
      va.chal = d_vch.as<sc_st>(); va.digest = d_digest.as<uint8_t>(); va.bad = d_bad.as<int>(); va.sp32 = d_sp32.as<uint8_t>(); memcpy(va.B32, e.sh->B32, 32); memcpy(va.H32, e.sh->H32, 32);
      LAUNCH_COOP(k_ts_verify, dim3((unsigned)C), dim3(TS_THREADS), s, va); }
    { verify_keys_args ka = {}; ka.digest = d_digest.as<uint8_t>(); ka.C = (uint32_t)C; ka.dom = dom; ka.c_off = c_off; memcpy(ka.seed, seed, 32); ka.ccrho = d_ccrho.as<sc_st>();
      LAUNCH_COOP(k_verify_keys, dim3(1), dim3(256), s, ka); }
    { verify_prep_args pa = {}; pa.proofs = d_proofs.as<uint8_t>(); pa.plen = (uint32_t)plen; pa.C = (uint32_t)C; pa.lgN = lgN; pa.lgm = lgm; pa.n = n; pa.vch = d_vch.as<sc_st>(); pa.ccrho = d_ccrho.as<sc_st>();
      pa.chal = d_chal.as<sc_st>(); pa.chs = chs; pa.small = d_var.as<sc_st>() + (size_t)C * m; pa.nsmall = nsmall; pa.yinvpow2 = d_yinvpow2.as<sc_st>(); pa.zpow2 = d_zpow2.as<sc_st>();
      LAUNCH_COOP(k_verify_prep, dim3(C), dim3(2 * TS_THREADS), s, pa); }
    tr.mark("v_transcripts");
    LAUNCH(k_verify_tables, dim3((vt.total + m + 255) / 256, C), dim3(256), s, d_tab.as<sc_st>(), vt, d_var.as<sc_st>(), (uint32_t)m, d_chal.as<sc_st>(), chs, d_yinvpow2.as<sc_st>(), d_zpow2.as<sc_st>(), m);
    LAUNCH_COOP(k_verify_scalars, dim3((unsigned)((N + 63) / 64)), dim3(256), s, d_gh.as<sc_st>(), d_tab.as<sc_st>(), vt, d_chal.as<sc_st>(), chs, n, C);
    LAUNCH(k_decompress, dim3((unsigned)(((size_t)C * nsmall + 127) / 128)), dim3(128), s, d_sp.as<p3_st>(), (uint8_t *)nullptr, d_sp32.as<uint8_t>(), (size_t)C * nsmall, (size_t)C * nsmall, (const p3_st *)nullptr, d_bad.as<int>(), (size_t)nsmall);
    tr.mark("v_scalar_kernels");
    // fixed generators: one 2N-term MSM (radix-2^c tables when they exist, bucket MSM otherwise) -> d_fix.  It runs on the lane's side stream,
    // beside the MSM over the commitments and proof points below (both need only the scalars); the last finalize joins them.
    cudaStream_t side = (tl_lane && tl_lane_engine == &e && tl_lane->q[0].hi == s) ? tl_lane->side[0] : s;
    rt_stream_after(side, s);
    const int nbV = rt ? rt_blocks(2 * N, 1) : 0;
    const msm_plan plF = rt ? msm_plan() : msm_plan_for(2 * N, 1);
    dev_buf d_partV(rt ? sizeof(p3_st) * (size_t)nbV : 16, s), d_winF(rt ? 16 : sizeof(p3_st) * plF.out_count(1), s);
    {
        finalize_args f = {}; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.out_p3 = d_fix.as<p3_st>(); f.count = 1;
        if (rt) {
            rt_msm_args ra = {}; ra.scalars = d_gh.as<sc_st>(); ra.T = (uint32_t)(2 * N); ra.scalar_stride = (uint32_t)(2 * N); ra.nG = (uint32_t)N; ra.mode = 0; ra.rt = *rt; ra.partial = d_partV.as<p3_st>();
            run_rt_msm(e, side, ra, nbV, 1);
            f.partial = d_partV.as<p3_st>(); f.npartial = nbV;
            run_finalize(side, f);
        } else {
            msm_args a = {}; a.v[0].scalars = d_gh.as<sc_st>(); a.split = 1; a.T = (uint32_t)(2 * N); a.scalar_stride = (uint32_t)(2 * N); a.nseg = 2; a.out = d_winF.as<p3_st>();
            a.v[0].seg[0] = mk_seg(g.G, (uint32_t)N, 0, 0); a.v[0].seg[1] = mk_seg(g.H, (uint32_t)N, 0, 0);
            run_msm(e, side, a, plF, 1);
            fin_windows(f, d_winF.as<p3_st>(), plF);
            run_finalize(side, f);
        }
    }
    // commitments and proof points of ALL chunks: one sliced MSM over C*m + C*nsmall terms (scalars laid out the same way)
    {
        const uint32_t TV = (uint32_t)((size_t)C * m + (size_t)C * nsmall);
        const msm_plan pl = msm_plan_for(TV, 1, 2048);
        dev_buf d_winV(sizeof(p3_st) * pl.out_count(1), s);
        msm_args a = {}; a.v[0].scalars = d_var.as<sc_st>(); a.split = 1; a.T = TV; a.scalar_stride = TV; a.nseg = 2; a.out = d_winV.as<p3_st>();
        a.v[0].seg[0] = mk_seg(d_Vp3, (uint32_t)((size_t)C * m), 0, 1); a.v[0].seg[1] = mk_seg(d_sp.p, (uint32_t)((size_t)C * nsmall), 0, 1);
        run_msm(e, s, a, pl, 1);
        rt_stream_after(s, side);
        tr.mark("v_msms");
        finalize_args f = {}; fin_windows(f, d_winV.as<p3_st>(), pl);
        f.partial = d_fix.as<p3_st>(); f.npartial = 1; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.is_id = d_id.as<int>(); f.count = 1;
        run_finalize(s, f);
    }
    std::vector<int> h_bad(C); int h_id = 0;
    rt_d2h(&h_id, d_id.p, sizeof(int), s); rt_d2h(h_bad.data(), d_bad.p, sizeof(int) * C, s);
    if (d_xbad) rt_d2h(h_xbad, d_xbad, sizeof(int) * nx, s);
    rt_sync(s);
    tr.mark("v_final");
    if (tap) {
        range_tap::rec r; r.C = C; r.n = n; r.m = m; r.lgN = lgN; r.c_off = c_off; r.dom = dom; r.rt = rt ? 1 : 0; r.c = rt ? rt->c : plF.c; r.id = h_id; r.bad = h_bad;
        auto get = [&](std::vector<sc_st> &v, const dev_buf &d, size_t count) { v.resize(count); rt_d2h(v.data(), d.p, sizeof(sc_st) * count, s); };
        get(r.vch, d_vch, (size_t)C * (4 + lgN)); get(r.ccrho, d_ccrho, 2 * (size_t)C); get(r.chal, d_chal, (size_t)C * chs);
        get(r.var, d_var, (size_t)C * vstride); get(r.gh, d_gh, 2 * N);
        r.digest.resize(32 * (size_t)C); rt_d2h(r.digest.data(), d_digest.p, 32 * (size_t)C, s);
        rt_sync(s);
        tap->recs.push_back(std::move(r));
    }
    int all_ok = h_id;
    for (int c = 0; c < C; c++) all_ok &= h_bad[c] ? 0 : 1;
    for (int c = 0; c < C; c++) verdict[c] = all_ok;
    return 0;
}

// range_proof_vec::verify_rangeproof (range_proof_vec/mod.rs:149-191).  d_commits: D compressed points (device).
// returns 1 true, 0 false, -1 FormatError, -7 InvalidBitsize, -2 bad args, -3 InvalidGeneratorsLength, -4 undecodable commitment
static int engine_range_verify(rofl_engine &e, const uint8_t *h_proofs, size_t plen, size_t n_proofs, const uint8_t *d_commits, size_t D,
                               int range, const uint8_t seed[32], const shard_spec *shard = nullptr, range_tap *tap = nullptr) {
    if (n_proofs == 0 || range < 1 || range > 64) return -2;
    if (shard ? (shard->m == 0 || shard->n_chunks != n_proofs || D > shard->m * shard->n_chunks) : D == 0) return -2;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const size_t Dp = shard ? shard->m * shard->n_chunks : next_pow2_sz(D), m = Dp / n_proofs;                     // :168
    const size_t c_off = shard ? shard->chunk_begin : 0;
    if (m == 0) return -3;
    // RangeProof::from_bytes happens when the caller deserialises (params.rs:444-458): format errors come first
    if (range_proof_format_check(h_proofs, plen, n_proofs, nullptr)) return -1;
    if (!(range == 8 || range == 16 || range == 32 || range == 64)) return ROFL_ERR_BITSIZE_;
    const size_t C = std::min(n_proofs, (Dp + m - 1) / m);                        // zip(proofs, chunks)
    phase_trace tr(s);
    dev_buf d_off(sizeof(p3_st), s), d_offs(sizeof(sc_st), s), d_Vp3(sizeof(p3_st) * Dp, s), d_V32(32 * Dp, s), d_bad(sizeof(int), s);
    { sc o; sc_from_u64(o, 1ULL << (range - 1)); sc_st os; sc_to_st(os, o); rt_h2d(d_offs.p, &os, sizeof(os), s);
      finalize_args f = {}; f.sBa = d_offs.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.out_p3 = d_off.as<p3_st>(); f.count = 1;
      run_finalize(s, f); }
    rt_memset(d_bad.p, 0, sizeof(int), s);
    LAUNCH(k_decompress, dim3((unsigned)((Dp + 127) / 128)), dim3(128), s, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), d_commits, D, Dp, d_off.as<p3_st>(), d_bad.as<int>(), Dp);
    tr.mark("v_decompress");
    tables_use tu(*e.sh);
    engine_gens(e, tu, s, range, (int)m);
    rt_tables rt; const bool have_rt = engine_rt(e, tu, s, range, (int)m, rt);
    const gens_entry g = engine_gens(e, tu, s, range, (int)m);
    // one group: every chunk goes into the same batched check (kernels.cuh, k_verify_scalars), splitting would repeat the generator MSM
    std::vector<int> verdict; int bad = 0;
    const int rc = verify_chunks(e, s, 0, range, (int)m, (int)C, g, have_rt ? &rt : nullptr, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), h_proofs, plen, seed, DOM_RANGE_VERIFY, c_off, verdict, d_bad.as<int>(), &bad, tap);
    if (bad) return -4;
    if (rc < 0) return rc;
    int res = 1; for (int v : verdict) res &= v;                               // :183-190
    return res;
}


// =============================================================================================================================
// Server side: K updates of the same shape (D, range, n_proofs) verified TOGETHER -- one random linear combination over all K x n_proofs
// chunks, ONE generator MSM, one bucket MSM over all commitments (rofl_service verifies the clients one by one on a thread pool,
// server.rs:516-522,666-667 -> params.rs:181-291).  d_commits: K x D encodings (device), h_proofs: K x n_proofs x plen.
// out[k] = 1 valid, 0 invalid, < 0 that update's error.  When the combined check fails (or any update is malformed) the updates are
// re-checked one by one, so that the verdict names the offender exactly as the reference's per-client results do.
// =============================================================================================================================
static int engine_range_verify_batch(rofl_engine &e, const uint8_t *h_proofs, size_t plen, size_t n_proofs, const uint8_t *d_commits, size_t D, size_t K,
                                     int range, const uint8_t seed[32], int *out, range_tap *tap = nullptr) {
    if (n_proofs == 0 || D == 0 || range < 1 || range > 64 || !out) return -2;
    if (K == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const size_t Dp = next_pow2_sz(D), m = Dp / n_proofs;
    bool batch_ok = m != 0 && (range == 8 || range == 16 || range == 32 || range == 64) && n_proofs * m == Dp && K * n_proofs <= (1u << 20);
    for (size_t k = 0; k < K && batch_ok; k++) if (range_proof_format_check(h_proofs + k * n_proofs * plen, plen, n_proofs, nullptr)) batch_ok = false;
    if (batch_ok) {
        dev_buf d_off(sizeof(p3_st), s), d_offs(sizeof(sc_st), s), d_Vp3(sizeof(p3_st) * Dp * K, s), d_V32(32 * Dp * K, s), d_bad(sizeof(int) * K, s);
        { sc o; sc_from_u64(o, 1ULL << (range - 1)); sc_st os; sc_to_st(os, o); rt_h2d(d_offs.p, &os, sizeof(os), s);
          finalize_args f = {}; f.sBa = d_offs.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.out_p3 = d_off.as<p3_st>(); f.count = 1;
          run_finalize(s, f); }
        rt_memset(d_bad.p, 0, sizeof(int) * K, s);
        LAUNCH(k_decompress_batch, dim3((unsigned)((K * Dp + 127) / 128)), dim3(128), s, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), d_commits, D, Dp, K, d_off.as<p3_st>(), d_bad.as<int>());
        tables_use tu(*e.sh);
        engine_gens(e, tu, s, range, (int)m);
        rt_tables rt; const bool have_rt = engine_rt(e, tu, s, range, (int)m, rt);
        const gens_entry g = engine_gens(e, tu, s, range, (int)m);
        std::vector<int> verdict, bad(K, 0);
        const int rc = verify_chunks(e, s, 0, range, (int)m, (int)(K * n_proofs), g, have_rt ? &rt : nullptr, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), h_proofs, plen, seed, DOM_RANGE_VERIFY, 0, verdict,
                                     d_bad.as<int>(), bad.data(), tap, K);
        bool all = rc == 0; for (int v : verdict) all = all && v == 1; for (int b : bad) all = all && !b;
        if (all) { for (size_t k = 0; k < K; k++) out[k] = 1; return 0; }
    }
    for (size_t k = 0; k < K; k++) out[k] = engine_range_verify(e, h_proofs + k * n_proofs * plen, plen, n_proofs, d_commits + 32 * k * D, D, range, seed, nullptr, tap);
    return 0;
}
static int engine_l2_verify(rofl_engine &e, const uint8_t *h_proof, size_t plen, const uint8_t *h_commit, int range, const uint8_t seed[32], range_tap *tap = nullptr);
// K sum-of-squares proofs (l2_range_proof_vec::verify_rangeproof_l2, :185-228) in one batched check; h_commits: K x 32
static int engine_l2_verify_batch(rofl_engine &e, const uint8_t *h_proofs, size_t plen, const uint8_t *h_commits, size_t K, int range, const uint8_t seed[32], int *out,
                                  range_tap *tap = nullptr) {
    if (!out) return -2;
    if (K == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    bool batch_ok = (range == 8 || range == 16 || range == 32 || range == 64) && range_proof_format_check(h_proofs, plen, K, nullptr) == 0;
    if (batch_ok) {
        dev_buf d_c(32 * K, s), d_Vp3(sizeof(p3_st) * K, s), d_V32(32 * K, s), d_bad(sizeof(int) * K, s);
        rt_h2d(d_c.p, h_commits, 32 * K, s); rt_memset(d_bad.p, 0, sizeof(int) * K, s);
        LAUNCH(k_decompress_batch, dim3((unsigned)((K + 127) / 128)), dim3(128), s, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), d_c.as<uint8_t>(), (size_t)1, (size_t)1, K, (const p3_st *)nullptr, d_bad.as<int>());
        tables_use tu(*e.sh);
        const gens_entry g = engine_gens(e, tu, s, range, 1);
        std::vector<int> verdict, bad(K, 0);
        const int rc = verify_chunks(e, s, 1, range, 1, (int)K, g, nullptr, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), h_proofs, plen, seed, DOM_L2_VERIFY, 0, verdict, d_bad.as<int>(), bad.data(), tap, K);
        bool all = rc == 0; for (int v : verdict) all = all && v == 1; for (int b : bad) all = all && !b;
        if (all) { for (size_t k = 0; k < K; k++) out[k] = 1; return 0; }
    }
    for (size_t k = 0; k < K; k++) out[k] = engine_l2_verify(e, h_proofs + k * plen, plen, h_commits + 32 * k, range, seed, tap);
    return 0;
}

// =============================================================================================================================
// l2_range_proof_vec::create_rangeproof_l2 (l2_range_proof_vec/mod.rs:15-140): one m=1 proof on sum x_i^2 with blinding sum r_i.
// h_values is a HOST copy of the values: the reference cross-checks the scalar sum against a sequential f32 fold (:44-58)
// whose rounding depends on the summation order, so that O(D) fold runs on the host exactly as written.
// returns 0 ok, 2 ValueOutOfRange, 3 OverflowError, 4 NormOutOfRange, -7 InvalidBitsize, -2 bad args
// =============================================================================================================================
static int engine_l2_prove(rofl_engine &e, const float *h_values, const float *d_values, const uint8_t *d_blind, size_t D, int range,
                           int n_bits, int frac, const uint8_t seed[32], uint8_t *h_proof, size_t *proof_len, uint8_t *h_commit) {
    if (!fp_ok(n_bits, frac) || D == 0 || range < 1) return -2;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const float mx = clip_max_f(range, n_bits, frac), mn = -mx;
    for (size_t i = 0; i < D; i++) if (mn > h_values[i] || h_values[i] > mx) return 2;
    const int nb = (int)std::min<size_t>(256, (D + 255) / 256);
    dev_buf d_part(sizeof(sc_st) * 2 * nb, s), d_sum(sizeof(sc_st) * 2, s), d_flags(sizeof(int), s);
    rt_memset(d_flags.p, 0, sizeof(int), s);
    LAUNCH_COOP(k_l2_sums, dim3(nb), dim3(256), s, d_part.as<sc_st>(), d_values, d_blind, D, n_bits, frac, d_flags.as<int>());
    LAUNCH_COOP(k_sc_sum, dim3(1), dim3(256), s, d_sum.as<sc_st>(), d_part.as<sc_st>(), nb, 2);
    sc_st hs[2]; int flags = 0;
    rt_d2h(hs, d_sum.p, sizeof(hs), s); rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    if (flags & 1) return -98;
    sc val, bsum; st_to_sc(val, hs[0]); st_to_sc(bsum, hs[1]);
    // :44-58 sequential f32 cross-check
    const float shift = (float)(1 << frac); float val_float = 0.0f;
    for (size_t i = 0; i < D; i++) {
        sc sx; f32_to_scalar(sx, h_values[i], n_bits, frac);
        float xq = scalar_to_f32(sx, n_bits, frac), term = xq * xq * shift;
        val_float = (i == 0) ? term : val_float + term;
    }
    const float vf = scalar_to_f32(val, n_bits, frac);
    if (fabsf(vf - val_float) > 1.1920929e-7f) return 3;
    if (vf > l2_clip_max_f(range, n_bits, frac)) return 4;
    if (!(range == 8 || range == 16 || range == 32 || range == 64)) return ROFL_ERR_BITSIZE_;
    uint64_t v = (((uint64_t)val.v[1] << 32) | val.v[0]) & fix_max(n_bits);      // :69-73 read_from_bytes
    // V = v B + bsum H
    dev_buf d_v(8, s), d_bl(sizeof(sc_st), s), d_vs(sizeof(sc_st), s), d_V(32, s);
    sc vs; sc_from_u64(vs, v); sc_st t; sc_to_st(t, vs); rt_h2d(d_vs.p, &t, sizeof(t), s);
    sc_to_st(t, bsum); rt_h2d(d_bl.p, &t, sizeof(t), s); rt_h2d(d_v.p, &v, 8, s);
    { finalize_args f = {}; f.sBa = d_vs.as<sc_st>(); f.sHa = d_bl.as<sc_st>(); f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.out32 = d_V.as<uint8_t>(); f.count = 1;
      run_finalize(s, f); }
    tables_use tu(*e.sh);
    const gens_entry g = engine_gens(e, tu, s, range, 1);                         // BulletproofGens::new(64, 1) restricted to n = range (:162)
    std::vector<uint8_t> keys(32); derive_key(keys.data(), seed, DOM_L2_PROVE, 0);
    prove_chunks(e, lg.ln->q[0], lg.ln->side[0], 1, range, 1, 1, g, nullptr, d_v.as<uint64_t>(), d_bl.as<sc_st>(), d_V.as<uint8_t>(), keys, h_proof);
    rt_d2h(h_commit, d_V.p, 32, s); rt_sync(s);
    *proof_len = 32 * (9 + 2 * (size_t)ilog2_sz((size_t)range));
    return 0;
}
// verify_rangeproof_l2 (:185-228)
static int engine_l2_verify(rofl_engine &e, const uint8_t *h_proof, size_t plen, const uint8_t *h_commit, int range, const uint8_t seed[32], range_tap *tap) {
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    if (range_proof_format_check(h_proof, plen, 1, nullptr)) return -1;
    dev_buf d_c(32, s), d_Vp3(sizeof(p3_st), s), d_V32(32, s), d_bad(sizeof(int), s);
    rt_h2d(d_c.p, h_commit, 32, s); rt_memset(d_bad.p, 0, sizeof(int), s);
    LAUNCH(k_decompress, dim3(1), dim3(128), s, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), d_c.as<uint8_t>(), (size_t)1, (size_t)1, (const p3_st *)nullptr, d_bad.as<int>(), (size_t)1);
    if (!(range == 8 || range == 16 || range == 32 || range == 64)) {
        int bad = 0; rt_d2h(&bad, d_bad.p, sizeof(int), s); rt_sync(s);
        return bad ? -4 : ROFL_ERR_BITSIZE_;
    }
    tables_use tu(*e.sh);
    const gens_entry g = engine_gens(e, tu, s, range, 1);
    std::vector<int> verdict; int bad = 0;
    const int rc = verify_chunks(e, s, 1, range, 1, 1, g, nullptr, d_Vp3.as<p3_st>(), d_V32.as<uint8_t>(), h_proof, plen, seed, DOM_L2_VERIFY, 0, verdict, d_bad.as<int>(), &bad, tap);
    if (bad) return -4;
    if (rc < 0) return rc;
    return verdict.empty() ? 0 : verdict[0];
}

// =============================================================================================================================
// square_proof_vec::create_l2rangeproof_vec_existing (square_proof_vec/mod.rs:19-75); device pointers.  The verify (engine_square_verify) follows
// the batched check it uses, sigma_verify_groups
// =============================================================================================================================
static int engine_square_prove(rofl_engine &e, const float *d_values, const uint8_t *d_value_com, const uint8_t *d_r1, const uint8_t *d_r2, size_t D,
                               int n_bits, int frac, const uint8_t seed[32], uint8_t *d_proofs, uint8_t *d_commits) {
    if (!fp_ok(n_bits, frac)) return -2;
    if (D == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    dev_buf d_flags(sizeof(int), s); rt_memset(d_flags.p, 0, sizeof(int), s);
    square_args a = {}; a.values = d_values; a.value_com = d_value_com; a.r1 = d_r1; a.r2 = d_r2; a.D = D; a.n_bits = n_bits; a.frac = frac;
    uint8_t key[32]; derive_key(key, seed, DOM_SQUARE, 0); key_words(a.key, key);
    a.tabB = e.sh->tabB; a.tabH = e.sh->tabH; a.proofs = d_proofs; a.commits = d_commits; a.flags = d_flags.as<int>();
    void *tk = rt_prof_begin(PROF_SQUARE, s);
    LAUNCH(k_square_prove, dim3((unsigned)((D + 127) / 128)), dim3(128), s, a);
    rt_prof_end(PROF_SQUARE, tk, s);
    int flags = 0; rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    if (flags & 4) return -4;
    if (flags & 1) return -98;
    return 0;
}
// bits of the batched checks' weights for an MSM of window width c: the smallest c * w - 1 >= 125 (125 .. 134 for c = 3 .. 16), so that the top
// window holds c - 1 uniform bits and the signed recoding never carries out of it (kernels.cuh k_sigma_rlc_scalars).  Not c * ceil(125 / c) - 1:
// that is 124 at c = 5, the width msm_plan_for picks for 157 .. 521 terms (small calls and the last range of a long one).
static inline int rlc_wbits(int c) { return c * ((126 + c - 1) / c) - 1; }
// Test hook (rofl_debug_rlc_terms): copies of what a batched check computed, taken from the buffers it already has.  The checks take a nullable
// pointer to one; with nullptr they issue exactly their production launches and copies.
struct rlc_tap {
    struct range {
        size_t i0 = 0, n = 0; int c = 0, wbits = 0;          // elements (clients for the compressed rand proofs) [i0, i0 + n), MSM window width, weight bits
        int is_id[2] = {-1, -1};                             // k_finalize's identity test per output (-1: no such output)
        std::vector<sc_st> scal; sc_st sB[2] = {}, sH[2] = {};   // MSM scalars in term order, fixed-base coefficients as given to k_finalize
        std::vector<int> bad;                                // bad flags of the clients the range touches
    };
    uint8_t root[32] = {}; std::vector<sc_st> chal; std::vector<range> ranges; int held = 0;
};

// =============================================================================================================================
// compressed_rand_proof::CompressedRandProof::{helper_prove, helper_prove_existing, helper_verify} (compressed_rand_proof/mod.rs:134-158)
//   d_values / d_blind / d_value_com (nullable: L_i = commit(m_i, r_i)) are device pointers; h_proof (128 B) and h_pairs (D x 64) host.
//   returns 0 ok, -4 undecodable existing commitment, -6 more than 900 000 pairs (the reference's label table ends there and it panics), -98 NaN
// =============================================================================================================================
#define CRP_MAX_D 900000
static inline void crp_challenge(sc &c, const uint8_t *h_pairs, size_t D, const uint8_t cprime[64]) {
    transcript t; transcript_init(t, "CompressedRandProof");
    const uint8_t ds[19] = {'r', 'a', 'n', 'd', 'o', 'm', 'n', 'e', 's', 's', ' ', 'p', 'r', 'o', 'o', 'f', ' ', 'v', '1'};
    transcript_append(t, "dom-sep", ds, 19);                                                         // rand_proof/transcript.rs:20-22
    for (size_t i = 0; i < D; i++) {                                                                 // dealer.rs:27-29; labels: generate_unique_u8_triplets.py:9-13
        const uint8_t lab[3] = {(uint8_t)(3 * i), (uint8_t)(3 * i + 1), (uint8_t)(3 * i + 2)};
        transcript_append_l(t, lab, 3, h_pairs + 64 * i, 64);
    }
    transcript_append(t, "C_prime_eg", cprime, 64);                                                  // dealer.rs:53-54
    ts_challenge_scalar(t, "c", c);
}
static inline pow_tab crp_pow_table(rofl_engine &e, cudaStream_t s, const sc &c, size_t D, dev_buf &store) {
    const int bits = std::max(2, ilog2_sz(D + 2));
    pow_tab ct = {nullptr, bits / 2, bits - bits / 2};
    std::vector<sc_st> h_pow2(32); sc_pow2_table(h_pow2.data(), c);
    sc_st *base = store.as<sc_st>();                               // [32 pow2 | table]
    rt_h2d(base, h_pow2.data(), sizeof(sc_st) * 32, s);
    ct.tab = base + 32;
    LAUNCH(k_pow_tables, dim3((pow_tab_size(ct) + 255) / 256, 1), dim3(256), s, base + 32, base, ct.L, ct.H);
    return ct;
}
static int engine_crp_prove(rofl_engine &e, const float *d_values, const uint8_t *d_value_com, const uint8_t *d_blind, size_t D, int n_bits, int frac,
                            const uint8_t seed[32], uint8_t *h_proof, uint8_t *h_pairs) {
    if (!fp_ok(n_bits, frac)) return -2;
    if (D > CRP_MAX_D) return -6;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const size_t Dn = D ? D : 1;
    dev_buf d_L(32 * Dn, s), d_R(32 * Dn, s), d_pairs(64 * Dn, s), d_flags(sizeof(int), s), d_bad(sizeof(int), s);
    rt_memset(d_flags.p, 0, sizeof(int), s); rt_memset(d_bad.p, 0, sizeof(int), s);
    if (D) {
        commit_args ca = {}; ca.values = d_values; ca.blind = d_blind; ca.D = D; ca.Dp = D; ca.n_bits = n_bits; ca.frac = frac;
        ca.tabB = e.sh->tabB; ca.tabH = e.sh->tabH; ca.C = d_value_com ? nullptr : d_L.as<uint8_t>(); ca.R = d_R.as<uint8_t>(); ca.flags = d_flags.as<int>();   // R_i = r_i B (el_gamal.rs:57-69)
        LAUNCH(k_commit, dim3((unsigned)((D + 127) / 128)), dim3(128), s, ca);
        if (d_value_com) {          // prove_existing: the caller's commitments must at least decode (the reference holds RistrettoPoints)
            dev_buf d_tmp(sizeof(p3_st) * D, s);
            LAUNCH(k_decompress, dim3((unsigned)((D + 127) / 128)), dim3(128), s, d_tmp.as<p3_st>(), (uint8_t *)nullptr, d_value_com, D, D, (const p3_st *)nullptr, d_bad.as<int>(), D);
        }
        LAUNCH(k_pairs_join, dim3((unsigned)((D + 255) / 256)), dim3(256), s, d_pairs.as<uint8_t>(), d_value_com ? d_value_com : d_L.as<uint8_t>(), d_R.as<uint8_t>(), D);
        rt_d2h(h_pairs, d_pairs.p, 64 * D, s);
    }
    // C' = (m' B + r' H, r' B), nonces in the draw order of Party::new (party.rs:26-29)
    uint8_t key[32]; derive_key(key, seed, DOM_CRP, 0); uint32_t kw[8]; key_words(kw, key);
    sc mp, rp, zero; nonce_scalar(mp, kw, 0); nonce_scalar(rp, kw, 1); sc_0(zero);
    sc_st h_sB[2], h_sH[2]; sc_to_st(h_sB[0], mp); sc_to_st(h_sH[0], rp); sc_to_st(h_sB[1], rp); sc_to_st(h_sH[1], zero);
    dev_buf d_s(sizeof(sc_st) * 4, s), d_cp(64, s);
    rt_h2d(d_s.p, h_sB, sizeof(h_sB), s); rt_h2d(d_s.as<sc_st>() + 2, h_sH, sizeof(h_sH), s);
    { finalize_args f = {}; f.sBa = d_s.as<sc_st>(); f.sHa = d_s.as<sc_st>() + 2; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.out32 = d_cp.as<uint8_t>(); f.count = 2; run_finalize(s, f); }
    int flags = 0, bad = 0;
    rt_d2h(h_proof, d_cp.p, 64, s); rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_d2h(&bad, d_bad.p, sizeof(int), s);
    rt_sync(s);
    if (flags & 1) return -98;
    if (bad) return -4;
    sc c; crp_challenge(c, h_pairs, D, h_proof);
    sc zm = mp, zr = rp;
    if (D) {
        dev_buf d_ct(sizeof(sc_st) * (32 + ((size_t)2 << ((ilog2_sz(D + 2) + 1) / 2 + 1))), s);
        pow_tab ct = crp_pow_table(e, s, c, D, d_ct);
        const int nb = (int)std::min<size_t>(256, (D + 255) / 256);
        dev_buf d_part(sizeof(sc_st) * 2 * nb, s), d_sum(sizeof(sc_st) * 2, s);
        LAUNCH_COOP(k_crp_sums, dim3(nb), dim3(256), s, d_part.as<sc_st>(), d_values, d_blind, D, n_bits, frac, ct, d_flags.as<int>());
        LAUNCH_COOP(k_sc_sum, dim3(1), dim3(256), s, d_sum.as<sc_st>(), d_part.as<sc_st>(), nb, 2);
        sc_st hs[2]; rt_d2h(hs, d_sum.p, sizeof(hs), s); rt_sync(s);
        sc a, b; st_to_sc(a, hs[0]); st_to_sc(b, hs[1]); sc_add(zm, zm, a); sc_add(zr, zr, b);     // party.rs:93-97
    }
    sc_tobytes(h_proof + 64, zm); sc_tobytes(h_proof + 96, zr);
    return 0;
}
// returns 1 valid, 0 invalid, -1 FormatError (from_bytes: mod.rs:118-134, el_gamal.rs:113-123), -6 too many pairs.
// The check given the challenge: c_known = c when the caller already ran crp_challenge over these pairs (the batched verifier's per-client
// re-check), else it is computed here while the device decompresses; d_pairs = the pairs already on the device (nullable: staged from h_pairs).
static int engine_crp_verify(rofl_engine &e, const uint8_t *h_proof, const uint8_t *h_pairs, size_t D, const sc *c_known = nullptr, const uint8_t *d_pairs_in = nullptr) {
    if (D > CRP_MAX_D) return -6;
    sc zm, zr; sc_frombytes(zm, h_proof + 64); sc_frombytes(zr, h_proof + 96);
    if (!sc_is_canonical(zm) || !sc_is_canonical(zr)) return -1;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const size_t Dn = D ? D : 1;
    dev_buf d_pairs(64 * Dn, s), d_LR32(64 * Dn, s), d_LR(sizeof(p3_st) * 2 * Dn, s), d_cp32(64, s), d_cp(sizeof(p3_st) * 2, s), d_bad(sizeof(int) * 2, s);
    rt_memset(d_bad.p, 0, sizeof(int) * 2, s);
    rt_h2d(d_cp32.p, h_proof, 64, s);
    LAUNCH(k_decompress, dim3(1), dim3(128), s, d_cp.as<p3_st>(), (uint8_t *)nullptr, d_cp32.as<uint8_t>(), (size_t)2, (size_t)2, (const p3_st *)nullptr, d_bad.as<int>(), (size_t)2);
    if (D) {
        if (!d_pairs_in) rt_h2d(d_pairs.p, h_pairs, 64 * D, s);
        LAUNCH(k_pairs_split, dim3((unsigned)((D + 255) / 256)), dim3(256), s, d_LR32.as<uint8_t>(), d_LR32.as<uint8_t>() + 32 * D, d_pairs_in ? d_pairs_in : d_pairs.as<uint8_t>(), D);
        LAUNCH(k_decompress, dim3((unsigned)((2 * D + 127) / 128)), dim3(128), s, d_LR.as<p3_st>(), (uint8_t *)nullptr, d_LR32.as<uint8_t>(), 2 * D, 2 * D, (const p3_st *)nullptr, d_bad.as<int>() + 1, 2 * D);
    }
    sc c; if (c_known) c = *c_known; else crp_challenge(c, h_pairs, D, h_proof);                   // overlaps the decompression
    // sum_i c^(i+1) L_i and sum_i c^(i+1) R_i: two MSMs that share their scalars
    sc nzm, nzr, zero; sc_neg(nzm, zm); sc_neg(nzr, zr); sc_0(zero);
    sc_st h_s[4]; sc_to_st(h_s[0], nzm); sc_to_st(h_s[1], nzr); sc_to_st(h_s[2], nzr); sc_to_st(h_s[3], zero);      // sB = [-z_m, -z_r], sH = [-z_r, 0]
    dev_buf d_s(sizeof(sc_st) * 4, s), d_id(sizeof(int) * 2, s);
    rt_h2d(d_s.p, h_s, sizeof(h_s), s);
    finalize_args f = {}; f.partial = d_cp.as<p3_st>(); f.npartial = 1; f.sBa = d_s.as<sc_st>(); f.sHa = d_s.as<sc_st>() + 2; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
    f.is_id = d_id.as<int>(); f.count = 2;
    if (D) {
        dev_buf d_ct(sizeof(sc_st) * (32 + ((size_t)2 << ((ilog2_sz(D + 2) + 1) / 2 + 1))), s), d_pw(sizeof(sc_st) * D, s);
        pow_tab ct = crp_pow_table(e, s, c, D, d_ct);
        LAUNCH(k_crp_pows, dim3((unsigned)((D + 255) / 256)), dim3(256), s, d_pw.as<sc_st>(), D, ct);
        const msm_plan pl = msm_plan_for(D, 2);
        dev_buf d_win(sizeof(p3_st) * pl.out_count(2), s);
        msm_args a = {}; a.v[0].scalars = d_pw.as<sc_st>(); a.v[1].scalars = d_pw.as<sc_st>(); a.split = 1; a.T = (uint32_t)D; a.scalar_stride = 0; a.nseg = 1; a.out = d_win.as<p3_st>();
        a.v[0].seg[0] = mk_seg(d_LR.as<p3_st>(), (uint32_t)D, 0, 1); a.v[1].seg[0] = mk_seg(d_LR.as<p3_st>() + D, (uint32_t)D, 0, 1);
        run_msm(e, s, a, pl, 2);
        fin_windows(f, d_win.as<p3_st>(), pl);
        run_finalize(s, f);
        int id[2], bad[2]; rt_d2h(id, d_id.p, sizeof(id), s); rt_d2h(bad, d_bad.p, sizeof(bad), s); rt_sync(s);
        if (bad[0] || bad[1]) return -1;
        return (id[0] && id[1]) ? 1 : 0;
    }
    run_finalize(s, f);
    int id[2], bad[2]; rt_d2h(id, d_id.p, sizeof(id), s); rt_d2h(bad, d_bad.p, sizeof(bad), s); rt_sync(s);
    if (bad[0]) return -1;
    return (id[0] && id[1]) ? 1 : 0;
}

// Server side: the compressed rand proofs of K clients in ONE check.  Client k's proof holds iff
//   C'_L,k + sum_i c_k^(i+1) L_k,i - z_m,k B - z_r,k H = 0   and   C'_R,k + sum_i c_k^(i+1) R_k,i - z_r,k B = 0;
// with Fiat-Shamir weights rho_k both are summed over the clients and checked by one MSM with two outputs that share their scalars
// (v[0] over L | C'_L, v[1] over R | C'_R; T = K (D + 1) terms) and one k_finalize whose fixed-base coefficients carry the signs:
//   sB = [-sum rho_k z_m,k, -sum rho_k z_r,k],  sH = [-sum rho_k z_r,k, 0].
// The weights: digest_k = SHA3-256(c_k | z_m,k | z_r,k) (c_k binds client k's pairs and C'), root = SHA3-256(seed | "crpb" | LE64 K | LE64 D |
// digest_0 .. digest_(K-1)), rho_k = the low 128 bits of ChaCha20(SHA3-256(root | LE64 k)) (the next block while they are zero).
// The K transcripts (crp_challenge: one sequential Merlin transcript over all D pairs per client) run on host threads from begin() to end(),
// while the device decompresses and the caller may queue more work on its stream (the whole-message batch runs its range batch there).
// Those threads do host work only: they never take a lane.  Clients are processed in groups of at most e.crp_batch_terms terms (default and
// upper bound CRP_BATCH_TERMS; a group holds at least one client).
// Verdicts: the combined check holds and no client of the group is malformed -> 1; otherwise malformed clients get -1 and every other client
// is re-checked on its own with the challenge already computed (engine_crp_verify given c), so each verdict is exactly rofl_crp_verify's.
#define CRP_BATCH_TERMS ((size_t)1 << 24)
struct crp_batch {
    rofl_engine &e; cudaStream_t s;
    const uint8_t *h_proofs, *h_pairs, *d_pairs; size_t D, K, G;
    std::vector<sc> c; std::vector<uint8_t> fmt;                                   // fmt[k]: z_m or z_r not canonical
    dev_buf d_cp, d_P, d_bad;
    std::thread th; std::string err;
    crp_batch(rofl_engine &eng, cudaStream_t st, const uint8_t *hp, const uint8_t *hpairs, const uint8_t *dpairs, size_t D_, size_t K_)
        : e(eng), s(st), h_proofs(hp), h_pairs(hpairs), d_pairs(dpairs), D(D_), K(K_), G(std::max<size_t>(1, std::min(K_, eng.crp_batch_terms / (D_ + 1)))),
          c(K_), fmt(K_, 0), d_cp(64 * K_, st), d_P(sizeof(p3_st) * 2 * (G * (D_ + 1)), st), d_bad(sizeof(int) * K_, st) {}
    ~crp_batch() { if (th.joinable()) th.join(); }
    crp_batch(const crp_batch &) = delete; crp_batch &operator=(const crp_batch &) = delete;
    void decompress(size_t k0, size_t g) {
        const size_t n = 2 * g * (D + 1);
        LAUNCH(k_crp_batch_points, dim3((unsigned)((n + 127) / 128)), dim3(128), s, d_P.as<p3_st>(), d_pairs + 64 * D * k0, d_cp.as<uint8_t>() + 64 * k0, D, (uint32_t)g, d_bad.as<int>() + k0);
    }
};
// D >= 1, D <= CRP_MAX_D, K >= 1; the caller holds a lane (s is its stream) and has put the K x D pairs at d_pairs
static void crp_batch_begin(crp_batch &b) {
    std::vector<uint8_t> cp(64 * b.K);
    for (size_t k = 0; k < b.K; k++) {
        const uint8_t *p = b.h_proofs + 128 * k; memcpy(&cp[64 * k], p, 64);
        sc zm, zr; sc_frombytes(zm, p + 64); sc_frombytes(zr, p + 96);
        b.fmt[k] = !sc_is_canonical(zm) || !sc_is_canonical(zr);
    }
    rt_h2d(b.d_cp.p, cp.data(), cp.size(), b.s); rt_memset(b.d_bad.p, 0, sizeof(int) * b.K, b.s);
    b.decompress(0, std::min(b.G, b.K));
    b.th = std::thread([&b] {
        try { parallel_for(b.K, b.e.host_threads, [&b](size_t k) { crp_challenge(b.c[k], b.h_pairs + 64 * b.D * k, b.D, b.h_proofs + 128 * k); }); }
        catch (const std::exception &ex) { b.err = ex.what(); }
    });
}
// holds (nullable): 1 when the combined check of every group held, else 0.  tap: the test hook's copies (rlc_tap; the range i0 / n are clients)
static void crp_batch_end(crp_batch &b, const uint8_t seed[32], int *out, int *holds = nullptr, rlc_tap *tap = nullptr) {
    rofl_engine &e = b.e; cudaStream_t s = b.s; const size_t K = b.K, D = b.D;
    b.th.join();
    if (!b.err.empty()) throw std::runtime_error(b.err);
    std::vector<uint8_t> root_in(32 + 4 + 16 + 32 * K);
    memcpy(root_in.data(), seed, 32);
    for (int i = 0; i < 4; i++) root_in[32 + i] = (uint8_t)((uint32_t)DOM_CRP_BATCH >> (8 * i));
    for (int i = 0; i < 8; i++) { root_in[36 + i] = (uint8_t)((uint64_t)K >> (8 * i)); root_in[44 + i] = (uint8_t)((uint64_t)D >> (8 * i)); }
    for (size_t k = 0; k < K; k++) {
        uint8_t m[96]; sc_tobytes(m, b.c[k]); memcpy(m + 32, b.h_proofs + 128 * k + 64, 64);
        sha3_256(&root_in[52 + 32 * k], m, 96);
    }
    uint8_t root[32]; sha3_256(root, root_in.data(), root_in.size());
    if (tap) { memcpy(tap->root, root, 32); tap->chal.resize(K); for (size_t k = 0; k < K; k++) sc_to_st(tap->chal[k], b.c[k]); }
    std::vector<sc> rho(K);
    for (size_t k = 0; k < K; k++) {
        uint8_t kb[40], key[32]; memcpy(kb, root, 32);
        for (int i = 0; i < 8; i++) kb[32 + i] = (uint8_t)((uint64_t)k >> (8 * i));
        sha3_256(key, kb, 40); uint32_t kw[8]; key_words(kw, key);
        for (uint64_t ctr = 0;; ctr++) {
            uint32_t w[16]; chacha20_block_words(w, kw, ctr);
            sc_0(rho[k]); for (int i = 0; i < 4; i++) rho[k].v[i] = w[i];
            if (w[0] | w[1] | w[2] | w[3]) break;
        }
    }
    const int bits = std::max(2, ilog2_sz(D + 2));
    pow_tab ct = {nullptr, bits / 2, bits - bits / 2};
    const size_t tabn = pow_tab_size(ct);
    std::vector<int> bad(K, 0);
    if (holds) *holds = 1;
    if (tap) tap->held = 1;
    for (size_t k0 = 0; k0 < K; k0 += b.G) {
        const size_t g = std::min(b.G, K - k0), n = g * (D + 1);
        bool any_fmt = false; for (size_t k = k0; k < k0 + g; k++) any_fmt = any_fmt || b.fmt[k];
        int id[2] = {0, 0};
        if (!any_fmt) {
            if (k0) b.decompress(k0, g);
            std::vector<sc_st> h_pow2(32 * g), h_rho(g); sc sB0, sB1, t; sc_0(sB0); sc_0(sB1);
            for (size_t j = 0; j < g; j++) {
                const size_t k = k0 + j; sc zm, zr; sc_frombytes(zm, b.h_proofs + 128 * k + 64); sc_frombytes(zr, b.h_proofs + 128 * k + 96);
                sc_pow2_table(&h_pow2[32 * j], b.c[k]); sc_to_st(h_rho[j], rho[k]);
                sc_mul(t, rho[k], zm); sc_add(sB0, sB0, t); sc_mul(t, rho[k], zr); sc_add(sB1, sB1, t);
            }
            sc_neg(sB0, sB0); sc_neg(sB1, sB1); sc zero; sc_0(zero);
            sc_st h_s[4]; sc_to_st(h_s[0], sB0); sc_to_st(h_s[1], sB1); sc_to_st(h_s[2], sB1); sc_to_st(h_s[3], zero);       // sB = [-sum rho z_m, -sum rho z_r], sH = [-sum rho z_r, 0]
            dev_buf d_pow2(sizeof(sc_st) * 32 * g, s), d_tab(sizeof(sc_st) * tabn * g, s), d_rho(sizeof(sc_st) * g, s), d_sc(sizeof(sc_st) * n, s), d_s(sizeof(h_s), s), d_id(sizeof(int) * 2, s);
            rt_h2d(d_pow2.p, h_pow2.data(), sizeof(sc_st) * h_pow2.size(), s); rt_h2d(d_rho.p, h_rho.data(), sizeof(sc_st) * g, s); rt_h2d(d_s.p, h_s, sizeof(h_s), s);
            LAUNCH(k_pow_tables, dim3((unsigned)((tabn + 255) / 256), (unsigned)g), dim3(256), s, d_tab.as<sc_st>(), d_pow2.as<sc_st>(), ct.L, ct.H);
            ct.tab = d_tab.as<sc_st>();
            LAUNCH(k_crp_batch_scalars, dim3((unsigned)((n + 255) / 256)), dim3(256), s, d_sc.as<sc_st>(), D, (uint32_t)g, ct, d_rho.as<sc_st>());
            const msm_plan pl = msm_plan_for(n, 2);
            dev_buf d_win(sizeof(p3_st) * pl.out_count(2), s);
            msm_args a = {}; a.v[0].scalars = d_sc.as<sc_st>(); a.v[1].scalars = d_sc.as<sc_st>(); a.split = 1; a.T = (uint32_t)n; a.scalar_stride = 0; a.nseg = 1; a.out = d_win.as<p3_st>();
            a.v[0].seg[0] = mk_seg(b.d_P.as<p3_st>(), (uint32_t)n, 0, 1); a.v[1].seg[0] = mk_seg(b.d_P.as<p3_st>() + n, (uint32_t)n, 0, 1);
            run_msm(e, s, a, pl, 2);
            finalize_args f = {}; fin_windows(f, d_win.as<p3_st>(), pl); f.sBa = d_s.as<sc_st>(); f.sHa = d_s.as<sc_st>() + 2; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH;
            f.is_id = d_id.as<int>(); f.count = 2;
            run_finalize(s, f);
            rt_d2h(id, d_id.p, sizeof(id), s); rt_d2h(&bad[k0], b.d_bad.as<int>() + k0, sizeof(int) * g, s);
            rlc_tap::range r;
            if (tap) { r.scal.resize(n); rt_d2h(r.scal.data(), d_sc.p, sizeof(sc_st) * n, s); }
            rt_sync(s);
            if (tap) {
                r.i0 = k0; r.n = g; r.c = pl.c; r.is_id[0] = id[0]; r.is_id[1] = id[1]; r.bad.assign(&bad[k0], &bad[k0] + g);
                r.sB[0] = h_s[0]; r.sB[1] = h_s[1]; r.sH[0] = h_s[2]; r.sH[1] = h_s[3]; tap->ranges.push_back(std::move(r));
            }
            bool all = id[0] && id[1]; for (size_t k = k0; k < k0 + g; k++) all = all && !bad[k];
            if (all) { for (size_t k = k0; k < k0 + g; k++) out[k] = 1; continue; }
        }
        if (holds) *holds = 0;
        if (tap) tap->held = 0;
        for (size_t k = k0; k < k0 + g; k++)
            out[k] = b.fmt[k] ? -1 : engine_crp_verify(e, b.h_proofs + 128 * k, b.h_pairs + 64 * D * k, D, &b.c[k], b.d_pairs + 64 * D * k);
    }
}
// K compressed rand proofs (h_proofs K x 128, h_pairs K x D x 64 host; d_pairs the same pairs on the device, nullable) in one batched check;
// out[k] = exactly engine_crp_verify(proof k, pairs k, D).  Returns 0, -2 for bad arguments.  holds: as crp_batch_end (left alone when no check runs)
static int engine_crp_verify_batch(rofl_engine &e, const uint8_t *h_proofs, const uint8_t *h_pairs, const uint8_t *d_pairs, size_t D, size_t K, const uint8_t seed[32], int *out,
                                   int *holds = nullptr, rlc_tap *tap = nullptr) {
    if (!out) return -2;
    if (K == 0) return 0;
    if (!h_proofs || (D && !h_pairs)) return -2;
    if (D > CRP_MAX_D) { for (size_t k = 0; k < K; k++) out[k] = -6; return 0; }
    if (D == 0) { for (size_t k = 0; k < K; k++) out[k] = engine_crp_verify(e, h_proofs + 128 * k, h_pairs, 0); return 0; }
    lane_guard lg(e); cudaStream_t s = lg.s();
    dev_buf d_own(d_pairs ? 16 : 64 * D * K, s);
    if (!d_pairs) rt_h2d(d_own.p, h_pairs, 64 * D * K, s);
    crp_batch b(e, s, h_proofs, h_pairs, d_pairs ? d_pairs : d_own.as<uint8_t>(), D, K);
    crp_batch_begin(b);
    crp_batch_end(b, seed, out, holds, tap);
    return 0;
}

// rand_proof_vec::{create_randproof_vec(_existing), verify_randproof_vec} (kind 1) and square_rand_proof_vec::{create_l2rangeproof_vec(_existing),
// verify_l2rangeproof_vec} (kind 2); device pointers; d_value_com nullable (commit inside).  prove: 0, -4 bad point, -98 NaN; verify: 1 / 0 / -1 FormatError
static int engine_sigma_prove(rofl_engine &e, int kind, const float *d_values, const uint8_t *d_value_com, const uint8_t *d_r1, const uint8_t *d_r2, size_t D,
                              int n_bits, int frac, const uint8_t seed[32], uint8_t *d_proofs, uint8_t *d_commits) {
    if (!fp_ok(n_bits, frac) || (kind != 1 && kind != 2)) return -2;
    if (D == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    dev_buf d_flags(sizeof(int), s); rt_memset(d_flags.p, 0, sizeof(int), s);
    sigma_args a = {}; a.kind = kind; a.values = d_values; a.value_com = d_value_com; a.r1 = d_r1; a.r2 = d_r2; a.D = D; a.n_bits = n_bits; a.frac = frac;
    uint8_t key[32]; derive_key(key, seed, kind == 1 ? DOM_RANDPROOF : DOM_SQUARE_RAND, 0); key_words(a.key, key);
    a.tabB = e.sh->tabB; a.tabH = e.sh->tabH; a.proofs = d_proofs; a.commits = d_commits; a.flags = d_flags.as<int>();
    void *tk = rt_prof_begin(PROF_SQUARE, s);
    LAUNCH(k_sigma_prove, dim3((unsigned)((D + 127) / 128)), dim3(128), s, a);
    rt_prof_end(PROF_SQUARE, tk, s);
    int flags = 0; rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    if (flags & 4) return -4;
    if (flags & 1) return -98;
    return 0;
}
static int engine_sigma_verify(rofl_engine &e, int kind, const uint8_t *d_proofs, const uint8_t *d_commits, size_t D) {
    if (kind != 1 && kind != 2) return -2;
    if (D == 0) return 1;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    dev_buf d_res(2 * sizeof(int), s); int init[2] = {1, 0}; rt_h2d(d_res.p, init, sizeof(init), s);
    LAUNCH(k_sigma_verify, dim3((unsigned)((D + 127) / 128)), dim3(128), s, kind, d_proofs, d_commits, D, e.sh->tabB, e.sh->tabH, d_res.as<int>(), (size_t)0);
    int res[2]; rt_d2h(res, d_res.p, sizeof(res), s); rt_sync(s);
    if (res[1]) return -1;
    return res[0] ? 1 : 0;
}

// calls of fewer elements go straight to the per-element kernel (sigma_verify_groups; rofl_debug_square_rlc answers 0 for them)
#define SIGMA_RLC_MIN 256
// All N square proofs (kind 0), rand proofs (kind 1) or square-rand proofs (kind 2) of a call, in updates of `group` elements, in random linear
// combinations (kernels.cuh, k_sigma_rlc_*): the weights come from one hash tree over all N elements; the elements are then checked in ranges of
// at most e.sigma_rlc_terms MSM terms (np per element, sigma_kind_of), one MSM and one k_finalize per range.  A range may start or end inside an
// update.  Square proofs are checked in ONE range over the whole call, whose MSM's window width sets their weights' width; a call of more than
// 2^31 - 1 of their terms is left to the per-element kernel whole.
// seed: part of every key but kind 0's (nullable there).  failed (nullable) receives the element ranges [i0, i1) whose check did not hold or that
// touch an update with a malformed element.  Returns 1 when every range held and no element is malformed, else 0.  The caller holds a lane; s is
// its stream.  tap: the test hook's copies (rlc_tap)
static int sigma_verify_rlc(rofl_engine &e, cudaStream_t s, int kind, const uint8_t *d_proofs, const uint8_t *d_commits, size_t N, const uint8_t seed[32],
                            size_t group = 0, std::vector<std::pair<size_t, size_t>> *failed = nullptr, rlc_tap *tap = nullptr) {
    if (!group) group = N;
    const sigma_kind sk = sigma_kind_of(kind);
    const size_t np = sk.np, K = (N + group - 1) / group;
    if (kind == 0 && np * N > 0x7fffffffu) { if (failed) failed->push_back({0, N}); return 0; }
    const size_t R = kind == 0 ? N : std::max<size_t>(1, std::min(e.sigma_rlc_terms, CRP_BATCH_TERMS) / np);          // elements per range
    const size_t n1 = (N + 63) / 64, n2 = (n1 + 63) / 64, rmax = std::min(R, N), nbmax = (rmax + 127) / 128;
    dev_buf d_dig(32 * N, s), d_chal(sizeof(sc_st) * N, s), d_l1(32 * n1, s), d_l2(32 * n2, s), d_bad(sizeof(int) * K, s);
    dev_buf d_scal(sizeof(sc_st) * np * rmax, s), d_part(sizeof(sc_st) * 2 * nbmax, s), d_pts(sizeof(p3_st) * np * rmax, s), d_sum(sizeof(sc_st) * 2, s), d_id(sizeof(int), s);
    rt_memset(d_bad.p, 0, sizeof(int) * K, s);
    static const uint32_t tags[3] = {DOM_SQ_RLC, DOM_RP_RLC, DOM_SRP_RLC};
    sigma_rlc_args a = {}; a.kind = kind; a.proofs = d_proofs; a.commits = d_commits; a.N = N; a.group = group; a.tag = tags[kind];
    if (sk.seeded) memcpy(a.seed, seed, 32);
    a.digest = d_dig.as<uint8_t>(); a.chal = d_chal.as<sc_st>(); a.scal = d_scal.as<sc_st>(); a.partial = d_part.as<sc_st>(); a.pts = d_pts.as<p3_st>(); a.bad = d_bad.as<int>();
    LAUNCH(k_sigma_rlc_prep, dim3((unsigned)((N + 127) / 128)), dim3(128), s, a);
    const uint8_t *cur = d_dig.as<uint8_t>(); size_t n = N; uint8_t *bufs[2] = {d_l1.as<uint8_t>(), d_l2.as<uint8_t>()}; int which = 0;
    do {                                                   // hash tree, 64 digests per node
        const size_t nn = (n + 63) / 64;
        LAUNCH(k_hash_tree, dim3((unsigned)((nn + 127) / 128)), dim3(128), s, bufs[which], cur, n);
        cur = bufs[which]; which ^= 1; n = nn;
    } while (n > 1);
    a.root = cur;
    if (tap) { tap->chal.resize(N); rt_d2h(tap->root, cur, 32, s); rt_d2h(tap->chal.data(), d_chal.p, sizeof(sc_st) * N, s); }
    std::vector<int> bad(K);
    int all = 1;
    for (size_t i0 = 0; i0 < N; i0 += R) {
        const size_t r = std::min(R, N - i0), T = np * r, k0 = i0 / group, k1 = (i0 + r - 1) / group + 1;
        const unsigned nb = (unsigned)((r + 127) / 128);
        const msm_plan pl = msm_plan_for(T, 1, 2048);
        a.i0 = i0; a.n = r; a.wbits = rlc_wbits(pl.c);
        LAUNCH_COOP(k_sigma_rlc_scalars, dim3(nb), dim3(128), s, a);
        LAUNCH_COOP(k_sc_sum, dim3(1), dim3(256), s, d_sum.as<sc_st>(), d_part.as<sc_st>(), (int)nb, 2);
        LAUNCH(k_sigma_rlc_points, dim3((unsigned)((T + 127) / 128)), dim3(128), s, a);
        dev_buf d_win(sizeof(p3_st) * pl.out_count(1), s);
        msm_args m = {}; m.v[0].scalars = d_scal.as<sc_st>(); m.split = 1; m.T = (uint32_t)T; m.scalar_stride = (uint32_t)T; m.nseg = 1; m.out = d_win.as<p3_st>();
        m.v[0].seg[0] = mk_seg(d_pts.p, (uint32_t)T, 0, 1);
        run_msm(e, s, m, pl, 1);
        finalize_args f = {}; fin_windows(f, d_win.as<p3_st>(), pl); f.sBa = d_sum.as<sc_st>(); f.sHa = d_sum.as<sc_st>() + 1; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.is_id = d_id.as<int>(); f.count = 1;
        run_finalize(s, f);
        int id = 0; rt_d2h(&id, d_id.p, sizeof(int), s); rt_d2h(&bad[k0], d_bad.as<int>() + k0, sizeof(int) * (k1 - k0), s);
        rlc_tap::range tr;
        if (tap) { tr.scal.resize(T); rt_d2h(tr.scal.data(), d_scal.p, sizeof(sc_st) * T, s); rt_d2h(&tr.sB[0], d_sum.p, sizeof(sc_st), s); rt_d2h(&tr.sH[0], d_sum.as<sc_st>() + 1, sizeof(sc_st), s); }
        rt_sync(s);
        bool ok = id == 1; for (size_t k = k0; k < k1; k++) ok = ok && !bad[k];
        if (!ok) { all = 0; if (failed) failed->push_back({i0, i0 + r}); }
        if (tap) { tr.i0 = i0; tr.n = r; tr.c = pl.c; tr.wbits = a.wbits; tr.is_id[0] = id; tr.bad.assign(&bad[k0], &bad[k0] + (k1 - k0)); tap->ranges.push_back(std::move(tr)); }
    }
    if (tap) tap->held = all;
    return all;
}
// verdicts of the square / rand / square-rand proofs (kind 0 / 1 / 2) of N elements in updates of `group` elements each (group = 0: one update):
// d_res = (all valid, format error) per update, initialised to (1, 0) by the caller -- exactly what the per-element kernel (k_square_verify for
// kind 0, else k_sigma_verify) gives.  Calls of at least SIGMA_RLC_MIN elements go through the batched check first; every update a failed range
// touches is then checked element by element, each update at most once.  tap (test hook): the batched check also runs below SIGMA_RLC_MIN.
static void sigma_verify_groups(rofl_engine &e, cudaStream_t s, int kind, const uint8_t *d_proofs, const uint8_t *d_commits, size_t N, const uint8_t seed[32],
                                size_t group, int *d_res, rlc_tap *tap = nullptr) {
    if (!N) return;
    if (!group) group = N;
    const sigma_kind sk = sigma_kind_of(kind);
    const size_t pw = 32 * sk.pw, cw = 32 * sk.cw;
    void *tk = rt_prof_begin(PROF_SQUARE, s);
    std::vector<std::pair<size_t, size_t>> failed;
    if (N < SIGMA_RLC_MIN && !tap) failed.push_back({0, N});
    else sigma_verify_rlc(e, s, kind, d_proofs, d_commits, N, seed, group, &failed, tap);
    size_t next = 0;                                       // first update not yet checked element by element
    for (const auto &rg : failed) {
        const size_t k0 = std::max(next, rg.first / group), k1 = (rg.second - 1) / group + 1;
        if (k0 >= k1) continue;
        const size_t j0 = k0 * group, n = std::min(N, k1 * group) - j0;
        const dim3 g((unsigned)((n + 127) / 128));
        if (kind == 0) LAUNCH(k_square_verify, g, dim3(128), s, d_proofs + pw * j0, d_commits + cw * j0, n, e.sh->tabB, e.sh->tabH, d_res + 2 * k0, group);
        else LAUNCH(k_sigma_verify, g, dim3(128), s, kind, d_proofs + pw * j0, d_commits + cw * j0, n, e.sh->tabB, e.sh->tabH, d_res + 2 * k0, group);
        next = k1;
    }
    rt_prof_end(PROF_SQUARE, tk, s);
}

// square_proof_vec::verify_l2rangeproof_vec (square_proof_vec/mod.rs:130-160): the square proofs of one update, kind 0 of the batched check
static int engine_square_verify(rofl_engine &e, const uint8_t *d_proofs, const uint8_t *d_commits, size_t D) {
    if (D == 0) return 1;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    dev_buf d_res(2 * sizeof(int), s); int init[2] = {1, 0}; rt_h2d(d_res.p, init, sizeof(init), s);
    sigma_verify_groups(e, s, 0, d_proofs, d_commits, D, nullptr, 0, d_res.as<int>());
    int res[2]; rt_d2h(res, d_res.p, sizeof(res), s); rt_sync(s);
    if (res[1]) return -1;
    return res[0] ? 1 : 0;
}

// sum of D compressed points -> compressed (device in, host out); -4 if one does not decode
static int engine_points_sum(rofl_engine &e, const uint8_t *d_pts, size_t D, uint8_t *h_out32) {
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    const int nb = (int)std::max<size_t>(1, std::min<size_t>(296, (D + 127) / 128));
    dev_buf d_part(sizeof(p3_st) * nb, s), d_bad(sizeof(int), s), d_out(32, s);
    rt_memset(d_bad.p, 0, sizeof(int), s);
    LAUNCH_COOP(k_points_sum, dim3(nb), dim3(128), s, d_part.as<p3_st>(), d_pts, D, d_bad.as<int>());
    finalize_args f = {}; f.partial = d_part.as<p3_st>(); f.npartial = nb; f.tabB = e.sh->tabB; f.tabH = e.sh->tabH; f.out32 = d_out.as<uint8_t>(); f.count = 1;
    run_finalize(s, f);
    int bad = 0; rt_d2h(h_out32, d_out.p, 32, s); rt_d2h(&bad, d_bad.p, sizeof(int), s); rt_sync(s);
    return bad ? -4 : 0;
}

// =============================================================================================================================
// commitments (pedersen_ops.rs:9-25; el_gamal.rs:57-69), aggregation (params.rs:81-124), discrete log (bsgs32.rs, pedersen_ops.rs:47-53)
// =============================================================================================================================
static int engine_commit(rofl_engine &e, const float *d_values, const uint8_t *d_blind, size_t D, int n_bits, int frac, uint8_t *d_L, uint8_t *d_R) {
    if (!fp_ok(n_bits, frac)) return -2;
    if (D == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    dev_buf d_flags(sizeof(int), s); rt_memset(d_flags.p, 0, sizeof(int), s);
    commit_args ca = {}; ca.values = d_values; ca.blind = d_blind; ca.D = D; ca.Dp = D; ca.n_bits = n_bits; ca.frac = frac;
    ca.tabB = e.sh->tabB; ca.tabH = e.sh->tabH; ca.C = d_L; ca.R = d_blind ? d_R : nullptr; ca.flags = d_flags.as<int>();
    void *tk = rt_prof_begin(PROF_COMMIT, s);
    LAUNCH(k_commit, dim3((unsigned)((D + 127) / 128)), dim3(128), s, ca);
    rt_prof_end(PROF_COMMIT, tk, s);
    int flags = 0; rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    return (flags & 1) ? -98 : 0;
}
static int engine_aggregate(rofl_engine &e, const uint8_t *d_pts, size_t n_clients, size_t D, int init_base, uint8_t *d_out) {
    if (D == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    dev_buf d_bad(sizeof(int), s); rt_memset(d_bad.p, 0, sizeof(int), s);
    LAUNCH(k_aggregate, dim3((unsigned)((D + 127) / 128)), dim3(128), s, d_out, d_pts, n_clients, D, init_base, d_bad.as<int>());
    int bad = 0; rt_d2h(&bad, d_bad.p, sizeof(int), s); rt_sync(s);
    return bad ? -4 : 0;
}
static bsgs_entry engine_bsgs(rofl_engine &e, tables_use &tu, cudaStream_t s, uint64_t table_size, int bsgs_bits) {
    dev_shared &sh = *e.sh;
    auto key = std::make_pair(table_size, bsgs_bits);
    for (;;) {
        auto it = sh.bsgs.find(key);
        if (it != sh.bsgs.end()) return it->second;
        if (!tu.excl) { tu.upgrade(); continue; }
        bsgs_entry b; b.cap = 1; while (b.cap < 4 * (table_size + 1)) b.cap <<= 1;
        b.keys = (unsigned long long *)rt_raw_malloc(8 * (size_t)b.cap); b.vals = (uint32_t *)rt_raw_malloc(4 * (size_t)b.cap);
        rt_memset(b.keys, 0xff, 8 * (size_t)b.cap, s); rt_memset(b.vals, 0, 4 * (size_t)b.cap, s);
        dev_buf d_cnt(sizeof(int), s); rt_memset(d_cnt.p, 0, sizeof(int), s);
        LAUNCH(k_bsgs_build, dim3((unsigned)((table_size + 1 + 127) / 128)), dim3(128), s, b.keys, b.vals, b.cap, (uint32_t)table_size, sh.tabB, d_cnt.as<int>());
        int cnt = 0; rt_d2h(&cnt, d_cnt.p, sizeof(int), s); rt_sync(s);
        b.size = (uint64_t)cnt - 1;                                                   // get_size (bsgs32.rs:44-46)
        sh.bsgs[key] = b;
    }
}
// returns 0, -2 bad table or fixed-point format, -4 undecodable point, -5 where the reference panics (no discrete log within range for either
// sign, bsgs32.rs:69-70)
static int engine_dlog(rofl_engine &e, const uint8_t *d_pts, size_t D, uint64_t table_size, int bsgs_bits, int n_bits, int frac, uint8_t *d_out_sc, float *d_out_f32) {
    if (!fp_ok(n_bits, frac) || table_size == 0 || table_size > (1ull << 28) || bsgs_bits < 1 || bsgs_bits > 32) return -2;
    if (D == 0) return 0;
    lane_guard lg(e);
    cudaStream_t s = lg.s();
    tables_use tu(*e.sh);
    const bsgs_entry b = engine_bsgs(e, tu, s, table_size, bsgs_bits);
    uint64_t max_it = b.size ? (1ULL << bsgs_bits) / b.size : 0;                  // bsgs32.rs:60-62
    dev_buf d_flags(sizeof(int), s); rt_memset(d_flags.p, 0, sizeof(int), s);
    LAUNCH(k_bsgs_solve, dim3((unsigned)((D + 127) / 128)), dim3(128), s, d_out_sc, d_out_f32, d_pts, D, b.keys, b.vals, b.cap, (uint32_t)table_size, b.size, max_it,
           bsgs_bits, n_bits, frac, e.sh->tabB, d_flags.as<int>());
    int flags = 0; rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    if (flags & 4) return -4;
    if (flags & 8) return -5;
    return 0;
}

// =============================================================================================================================
// device-resident round accumulator: EncModelParamsAccumulator (params.rs:74-148) -- accumulate_other per arriving client, extract at
// the round's end.  The state (ncols x D extended points, kernels.cuh K9b) is allocated once, outside the scratch cache, so `trim` and
// table eviction never touch it.  Every call holds the accumulator's mutex and ends in a synchronise of its lane, so the next call may
// run on another lane (stream) of the context.
// =============================================================================================================================
enum { ROFL_ERR_UNBALANCED_ = -8 };       // include/rofl_b200.h ROFL_ERR_UNBALANCED
struct rofl_acc {
    rofl_engine *e = nullptr; size_t D = 0; int rec_bytes = 0, ncols = 0, init_unity = 0; size_t count = 0;
    p3_st *st = nullptr; std::mutex mu;
};
static void engine_acc_reset(rofl_acc &a) {
    lane_guard lg(*a.e); cudaStream_t s = lg.s();
    const size_t n = a.D * a.ncols;
    LAUNCH(k_acc_init, dim3((unsigned)((n + 255) / 256)), dim3(256), s, a.st, n, a.init_unity);
    rt_sync(s);
    a.count = 0;
}
static rofl_acc *engine_acc_create(rofl_engine &e, size_t D, int rec_bytes, int init_unity) {
    rofl_acc *a = new rofl_acc();
    a->e = &e; a->D = D; a->rec_bytes = rec_bytes; a->ncols = rec_bytes == 32 ? 1 : 2; a->init_unity = init_unity ? 1 : 0;
    try {
        a->st = (p3_st *)rt_raw_malloc(sizeof(p3_st) * D * a->ncols);
        engine_acc_reset(*a);
    } catch (...) { rt_raw_free(a->st); delete a; throw; }
    return a;
}
static void engine_acc_destroy(rofl_acc *a) { if (a) { rt_raw_free(a->st); delete a; } }
// d_rec: n_clients x D x rec_bytes [dev].  Clients with mask[k] != 1 (mask may be null: all) are skipped; the points of the others are validated
// first (one flag per client), and only clients whose every point decodes are added.  out_added[k]: 1 / 0 skipped / ROFL_ERR_POINT.  Returns the
// number of clients added.
static int engine_acc_add(rofl_acc &a, const uint8_t *d_rec, size_t n_clients, const int *mask, int *out_added) {
    rofl_engine &e = *a.e;
    lane_guard lg(e); cudaStream_t s = lg.s();
    const size_t pts = a.rec_bytes / 32, D = a.D;
    std::vector<int> bad(n_clients, 0);
    dev_buf d_bad(sizeof(int) * (n_clients ? n_clients : 1), s); rt_memset(d_bad.p, 0, sizeof(int) * n_clients, s);
    // validate each run of consecutive selected clients in one launch: the masked-out clients cost nothing
    for (size_t k0 = 0; k0 < n_clients;) {
        if (mask && mask[k0] != 1) { k0++; continue; }
        size_t k1 = k0 + 1; while (k1 < n_clients && (!mask || mask[k1] == 1)) k1++;
        const size_t np = pts * D * (k1 - k0);
        LAUNCH(k_validate_points, dim3((unsigned)((np + 127) / 128)), dim3(128), s, d_rec + a.rec_bytes * D * k0, (size_t)32, (size_t)0, np, d_bad.as<int>() + k0, pts * D);
        k0 = k1;
    }
    rt_d2h(bad.data(), d_bad.p, sizeof(int) * n_clients, s); rt_sync(s);
    std::vector<uint32_t> acc;
    for (size_t k = 0; k < n_clients; k++) {
        const int r = (mask && mask[k] != 1) ? 0 : bad[k] ? -4 : 1;
        if (r == 1) acc.push_back((uint32_t)k);
        if (out_added) out_added[k] = r;
    }
    if (!acc.empty()) {
        dev_buf d_list(sizeof(uint32_t) * acc.size(), s);
        rt_h2d(d_list.p, acc.data(), sizeof(uint32_t) * acc.size(), s);
        LAUNCH(k_acc_add, dim3((unsigned)((D + 127) / 128)), dim3(128), s, a.st, D, a.ncols, d_rec, (size_t)a.rec_bytes, d_list.as<uint32_t>(), (uint32_t)acc.size());
        rt_sync(s);
    }
    a.count += acc.size();
    return (int)acc.size();
}
// d_out: D x 32 ncols [dev], the canonical encodings of the accumulated values
static void engine_acc_export(rofl_acc &a, uint8_t *d_out) {
    lane_guard lg(*a.e); cudaStream_t s = lg.s();
    const size_t n = a.D * a.ncols;
    LAUNCH(k_acc_export, dim3((unsigned)((n + 127) / 128)), dim3(128), s, d_out, a.st, a.D, a.ncols);
}
// EncModelParamsAccumulator::extract: 0, ROFL_ERR_UNBALANCED (some R != B; nothing is written), -5 no discrete log in range (as engine_dlog),
// -2 bad table or fixed-point format
static int engine_acc_extract(rofl_acc &a, uint64_t table_size, int bsgs_bits, int n_bits, int frac, uint8_t *d_out_sc, float *d_out_f32) {
    if (!fp_ok(n_bits, frac) || table_size == 0 || table_size > (1ull << 28) || bsgs_bits < 1 || bsgs_bits > 32) return -2;
    rofl_engine &e = *a.e;
    lane_guard lg(e); cudaStream_t s = lg.s();
    tables_use tu(*e.sh);
    const bsgs_entry b = engine_bsgs(e, tu, s, table_size, bsgs_bits);
    uint64_t max_it = b.size ? (1ULL << bsgs_bits) / b.size : 0;                  // bsgs32.rs:60-62
    dev_buf d_flags(sizeof(int), s); rt_memset(d_flags.p, 0, sizeof(int), s);
    LAUNCH(k_acc_extract, dim3((unsigned)((a.D + 127) / 128)), dim3(128), s, d_out_sc, d_out_f32, a.st, a.D, a.ncols == 2 ? 1 : 0, b.keys, b.vals, b.cap,
           (uint32_t)table_size, b.size, max_it, bsgs_bits, n_bits, frac, e.sh->tabB, d_flags.as<int>());
    int flags = 0; rt_d2h(&flags, d_flags.p, sizeof(int), s); rt_sync(s);
    if (flags & 16) return ROFL_ERR_UNBALANCED_;
    if (flags & 8) return -5;
    return 0;
}
