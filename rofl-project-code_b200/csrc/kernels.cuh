// sm_100a kernels of the rofl_crypto prove / verify hot path (SURVEY.md section 2.3, K0-K11).
//
// Everything in this file is written against plain CUDA C++ (threadIdx/blockIdx, __shared__, __syncthreads,
// shared-memory atomics) so that tests/hostsim/cuda_emul.h can run the very same kernel bodies on CPU threads in
// this GPU-less container; on the device they are compiled by nvcc for sm_100a only.  No CPU path ships in the
// product library.
//
// HBM layout (all arrays 16-byte aligned, one record per point/scalar so gathers touch whole sectors):
//   niels_st   96 B : affine (y+x, y-x, 2dxy), 3 x 8 saturated 32-bit limbs            -- fixed generators, tables
//   p3_st     128 B : extended (X,Y,Z,T), 4 x 8 limbs                                 -- folded generators, partial sums
//   sc        32 B  : canonical scalar, 8 words
#pragma once
#include "devfn.cuh"

#include "rt.cuh"
#ifndef ROFL_EMUL
#define KERNEL extern "C" __global__
#define LB(t, b) __launch_bounds__(t, b)
#define DEV __device__ __forceinline__
// host-side launcher defined next to each kernel (the kernels are split over several translation units, see Makefile)
#define KLAUNCH(k, coop, PARAMS, ARGS) void launch_##k(dim3 g_, dim3 b_, cudaStream_t s_, KL_UNPACK PARAMS) { rt_host_timer t_(&rt_host_prof::launch, #k); void *tl_ = rt_timeline_begin(#k, s_, g_.x * g_.y * g_.z); k<<<g_, b_, 0, s_>>> ARGS; rt_check(cudaGetLastError(), #k); rt_timeline_end(tl_, s_); rt_count_launch(#k); }
#else
#define KERNEL static
#define LB(t, b)
#define DEV inline
#define KLAUNCH(k, coop, PARAMS, ARGS) void launch_##k(dim3 g_, dim3 b_, cudaStream_t s_, KL_UNPACK PARAMS) { (void)s_; emu_launch(g_, b_, coop, [&] { k ARGS; }); }
#endif
#define KL_UNPACK(...) __VA_ARGS__
// kernel groups: a translation unit defines KG_<GROUP> (or KG_ALL) to get the kernel bodies of that group
#if defined(KG_ALL)
#define KG_TABLES 1
#define KG_COMMIT 1
#define KG_SCALAR 1
#define KG_MSM 1
#define KG_FOLD 1
#define KG_SQUARE 1
#define KG_BSGS 1
#define KG_TS 1
#endif
#include "wtranscript.cuh"

// a point operand that is either a fixed generator (niels) or a variable point (p3)
// the sign is applied to the operand (swap y+x / y-x, negate 2dxy resp. X and T) so that lanes of a warp with different
// signs execute ONE addition instead of diverging into add and sub paths
HD void acc_add_niels(ge_p3 &acc, const niels_st *p, bool neg) {
    // -Q = (y-x, y+x, -2dxy): the swap is an address select, the sign of C = T1*2dxy swaps G = D+C and F = D-C afterwards
    const uint4 *q = (const uint4 *)p; ge_niels m;
    ld_fe1(m.yplusx, q + (neg ? 2 : 0)); ld_fe1(m.yminusx, q + (neg ? 0 : 2)); ld_fe1(m.xy2d, q + 4);
    ge_p1p1 t; ge_madd_p1p1(t, acc, m);
    fe z = t.Z; fe_cmov(t.Z, t.T, neg); fe_cmov(t.T, z, neg);
    ge_p1p1_to_p3(acc, t);
}
HD void acc_add_p3(ge_p3 &acc, const p3_st *p, bool neg) {
    ge_p3 q, nq; ld_p3(q, p); ge_neg(nq, q);
    fe_cmov(q.X, nq.X, neg); fe_cmov(q.T, nq.T, neg);
    ge_add(acc, acc, q);
}
// the cached form (Y+X | Y-X | Z | 2dT) in a p3_st record
HD void st_cached(p3_st *p, const ge_cached &c) { uint4 *q = (uint4 *)p; st_fe1(q, c.YplusX); st_fe1(q + 2, c.YminusX); st_fe1(q + 4, c.Z); st_fe1(q + 6, c.T2d); }
HD void ld_cached(ge_cached &c, const p3_st *p) { const uint4 *q = (const uint4 *)p; ld_fe2(c.YplusX, c.YminusX, q); ld_fe2(c.Z, c.T2d, q + 4); }
HD void acc_add_cached(ge_p3 &acc, const p3_st *p, bool neg) { ge_cached c; ld_cached(c, p); ge_add_cached_signed(acc, acc, c, neg); }

// ===================================================================================================================
// K0: tables
// ===================================================================================================================
// fixed-base table of the point with compressed encoding `pt`: entry (w,k) = (k+1) 256^w P  (FB_WINDOWS x FB_ENTRIES)
#ifdef KG_TABLES
KERNEL void k_fb_table_build(niels_st *tab, const uint8_t *pt) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= FB_WINDOWS * FB_ENTRIES) return;
    uint8_t b[32]; for (int i = 0; i < 32; i++) b[i] = pt[i];
    ge_p3 p; ge_decompress(p, b);
    ge_niels n; fb_table_entry(n, p, idx / FB_ENTRIES, idx % FB_ENTRIES);
    st_niels(tab + idx, n);
}
KLAUNCH(k_fb_table_build, false, (niels_st *tab, const uint8_t *pt), (tab, pt))
#endif
// K3: BulletproofGens (range_proof_vec/mod.rs:126,201 rebuild these per chunk per call; here once per (n, capacity)).
// one thread per (party, G|H) chain; writes niels records party-major: G[(j*n + i)]
#ifdef KG_TABLES
KERNEL void k_gens_build(niels_st *G, niels_st *H, int n, int party_begin, int party_end) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int j = party_begin + (idx >> 1);
    if (j >= party_end) return;
    int which = (idx & 1) ? 'H' : 'G';
    niels_st *out = ((idx & 1) ? H : G) + (size_t)j * n;
    gen_chain c; gen_chain_init(c, which, (uint32_t)j);
    for (int i = 0; i < n; i++) {
        ge_p3 p; gen_chain_next(c, p);
        fe zinv; fe_invert(zinv, p.Z);
        ge_niels q; ge_p3_to_niels(q, p, zinv);
        st_niels(out + i, q);
    }
}
KLAUNCH(k_gens_build, false, (niels_st *G, niels_st *H, int n, int party_begin, int party_end), (G, H, n, party_begin, party_end))
#endif

// ===================================================================================================================
// K1 + K2: f32 -> fixed point -> commitments
// ===================================================================================================================
// flags bits: 1 = NaN, 2 = value out of [mn, mx]
struct commit_args {
    const float *values;        // D
    const uint8_t *blind;       // D x 32 or null (zero blinding)
    size_t D, Dp;               // Dp = padded length (>= D); padding = value 0, blinding 0
    int n_bits, frac;
    int shift_bits;             // > 0: range-proof mode, commit to raw + 2^(shift_bits-1) (range_proof_vec/mod.rs:35-43)
    float mn, mx;               // range check bounds (range-proof mode)
    const niels_st *tabB, *tabH;
    uint8_t *V;                 // Dp x 32 compressed commitments to the (shifted) value   (may be null)
    uint8_t *C;                 // D x 32 compressed un-shifted commitments v*B + r*H        (may be null)
    uint8_t *R;                 // D x 32 compressed r*B  (ElGamal right halves, el_gamal.rs:57-69)  (may be null)
    uint64_t *vals;             // Dp shifted values as u64 (may be null)
    sc_st *blind_sc;            // Dp blindings reduced mod l (may be null)
    int *flags;
};
#ifdef KG_COMMIT
KERNEL void LB(128, 1) k_commit(commit_args a) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.Dp) return;
    sc gamma; sc_0(gamma);
    uint64_t raw = 0; bool neg = false; int fl = 0;
    if (i < a.D) {
        float x = a.values[i];
        if (f32_to_fix(&raw, x, a.n_bits, a.frac)) fl |= 1;
        neg = x < 0.0f;
        if (a.shift_bits > 0 && (a.mn > x || x > a.mx)) fl |= 2;
        if (a.blind) { uint8_t b[32]; ld_bytes32(b, a.blind + 32 * i); sc_from_bytes_mod_order(gamma, b); }
    }
    if (fl) atomicOr(a.flags, fl);
    if (a.blind_sc) st_sc(a.blind_sc + i, gamma);
    // gamma * H
    ge_p3 bh; ge_p3_0(bh);
    if (a.blind) fb_mul_acc(bh, a.tabH, gamma, 32);
    if (a.shift_bits > 0) {
        // shifted value: low n_bits of (f32_to_scalar(x) + 2^(shift-1)) mod l
        uint64_t sh = 0;
        if (i < a.D) {
            uint64_t off = 1ULL << (a.shift_bits - 1);
            if (!neg) sh = (raw + off) & fix_max(a.n_bits);
            else if (raw <= off) sh = (off - raw) & fix_max(a.n_bits);
            else { sc s, o; sc_from_u64(s, raw); sc_neg(s, s); sc_from_u64(o, off); sc_add(s, s, o); sh = (((uint64_t)s.v[1] << 32) | s.v[0]) & fix_max(a.n_bits); }
        }
        if (a.vals) a.vals[i] = sh;
        // V = sh B + gamma H ; the returned commitment is V - 2^(shift-1) B exactly as range_proof_vec/mod.rs:96-99 computes it
        // (this reproduces the reference's wrap-around when raw + offset overflows n_bits, e.g. x = +2^24 at fp32 / range 32)
        ge_p3 v = bh; sc s; sc_from_u64(s, sh); fb_mul_acc(v, a.tabB, s, 32);
        if (a.V) { uint8_t out[32]; ge_compress(out, v); st_bytes32(a.V + 32 * i, out); }
        if (i < a.D && a.C) {
            sc o; sc_from_u64(o, 1ULL << (a.shift_bits - 1)); sc_neg(o, o);
            // -2^(shift-1) B = msub of the single non-zero radix-256 digit of 2^(shift-1)
            int sb = a.shift_bits - 1; ge_niels nn; ld_niels(nn, a.tabB + (sb >> 3) * FB_ENTRIES + (1 << (sb & 7)) - 1);
            ge_msub(v, v, nn);
            uint8_t out[32]; ge_compress(out, v); st_bytes32(a.C + 32 * i, out);
        }
    } else if (i < a.D && a.C) {
        ge_p3 v; ge_p3_0(v); sc s; sc_from_u64(s, raw); fb_mul_acc(v, a.tabB, s, 32);
        if (neg) ge_neg(v, v);
        ge_add(v, v, bh);
        uint8_t out[32]; ge_compress(out, v); st_bytes32(a.C + 32 * i, out);
    }
    if (i < a.D && a.R) {
        ge_p3 v; ge_p3_0(v); fb_mul_acc(v, a.tabB, gamma, 32);
        uint8_t out[32]; ge_compress(out, v); st_bytes32(a.R + 32 * i, out);
    }
}
KLAUNCH(k_commit, false, (commit_args a), (a))
#endif

// field self-test (tests/test_gpu_parity.py): raw 256-bit inputs (NOT masked: loose representatives incl. values >= p) ->
// canonical encodings of a*b, a^2, a+b, a-b, (a+b)*(a-b), 1/a computed by the device code paths
#ifdef KG_COMMIT
KERNEL void LB(128, 1) k_field_selftest(uint8_t *out, const uint8_t *a32, const uint8_t *b32, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe a, b, r, s, t;
    for (int k = 0; k < 8; k++) { const uint8_t *pa = a32 + 32 * i + 4 * k, *pb = b32 + 32 * i + 4 * k;
        a.v[k] = (uint32_t)pa[0] | ((uint32_t)pa[1] << 8) | ((uint32_t)pa[2] << 16) | ((uint32_t)pa[3] << 24);
        b.v[k] = (uint32_t)pb[0] | ((uint32_t)pb[1] << 8) | ((uint32_t)pb[2] << 16) | ((uint32_t)pb[3] << 24); }
    uint8_t *o = out + 192 * i;
    fe_mul(r, a, b); fe_tobytes(o, r);
    fe_sq(r, a); fe_tobytes(o + 32, r);
    fe_add(s, a, b); fe_tobytes(o + 64, s);
    fe_sub(t, a, b); fe_tobytes(o + 96, t);
    fe_mul(r, s, t); fe_tobytes(o + 128, r);
    fe_invert(r, a); fe_tobytes(o + 160, r);
}
KLAUNCH(k_field_selftest, false, (uint8_t *out, const uint8_t *a32, const uint8_t *b32, size_t n), (out, a32, b32, n))
// scalar arithmetic mod l as the device computes it: a*b for RAW 256-bit a, b (sc_mul's fold reduction), (a mod l)^-1 by division steps, a^-1 by Fermat
KERNEL void LB(128, 1) k_scalar_selftest(uint8_t *out, const uint8_t *a32, const uint8_t *b32, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sc a, b, r;
    sc_frombytes(a, a32 + 32 * i); sc_frombytes(b, b32 + 32 * i);
    uint8_t *o = out + 96 * i;
    sc_mul(r, a, b); sc_tobytes(o, r);
    sc am; sc_from_bytes_mod_order(am, a32 + 32 * i);
    sc_invert_vartime(r, am); sc_tobytes(o + 32, r);
    sc_invert(r, am); sc_tobytes(o + 64, r);
}
KLAUNCH(k_scalar_selftest, false, (uint8_t *out, const uint8_t *a32, const uint8_t *b32, size_t n), (out, a32, b32, n))
#endif

// ===================================================================================================================
// block-level reductions through shared memory (no warp shuffles: keeps the bodies runnable under cuda_emul.h)
// ===================================================================================================================
// sum of one scalar per thread; result valid in thread 0.  `buf` = blockDim.x records of shared memory.
DEV void block_sum_sc(sc &v, sc_st *buf, int tid, int nthreads) {
    st_sc(buf + tid, v);
    __syncthreads();
    for (int s = nthreads >> 1; s > 0; s >>= 1) {
        if (tid < s) { sc a, b; ld_sc(a, buf + tid); ld_sc(b, buf + tid + s); sc_add(a, a, b); st_sc(buf + tid, a); }
        __syncthreads();
    }
    ld_sc(v, buf);
    __syncthreads();
}
// sum of one point per thread; result valid in thread 0
DEV void block_sum_p3(ge_p3 &v, p3_st *buf, int tid, int nthreads) {
    st_p3(buf + tid, v);
    __syncthreads();
    for (int s = nthreads >> 1; s > 0; s >>= 1) {
        if (tid < s) { ge_p3 a, b; ld_p3(a, buf + tid); ld_p3(b, buf + tid + s); ge_add(a, a, b); st_p3(buf + tid, a); }
        __syncthreads();
    }
    ld_p3(v, buf);
    __syncthreads();
}

// ===================================================================================================================
// K11 + K4/K5 helpers: nonces in the draw order of RangeProof::prove_multiple_with_rng (SURVEY.md A.3, A.5)
//   chunk c uses ChaCha20 key keys[c]; party j draws a_blinding (2n+2)j, s_blinding +1, s_L[i] +2+i, s_R[i] +2+n+i;
//   after all parties: t1_blinding m(2n+2)+2j, t2_blinding +1.
// ===================================================================================================================
// sLR[c][0..N) = s_L, sLR[c][N..2N) = s_R  (one array so that S = <s_L,G> + <s_R,H> is a single 2N-term MSM per chunk)
#ifdef KG_SCALAR
KERNEL void LB(256, 2) k_nonces(sc_st *sLR, const uint32_t *keys, int n, int m, size_t total) {
    size_t gp = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gp >= total) return;
    size_t N = (size_t)n * m;
    size_t c = gp / N, k = gp % N, j = k / n, i = k % n;
    const uint32_t *key = keys + 8 * c;
    uint32_t kk[8]; for (int t = 0; t < 8; t++) kk[t] = key[t];
    sc s;
    nonce_scalar(s, kk, (uint64_t)j * (2 * n + 2) + 2 + i); st_sc(sLR + c * 2 * N + k, s);
    nonce_scalar(s, kk, (uint64_t)j * (2 * n + 2) + 2 + n + i); st_sc(sLR + c * 2 * N + N + k, s);
}
KLAUNCH(k_nonces, false, (sc_st *sLR, const uint32_t *keys, int n, int m, size_t total), (sLR, keys, n, m, total))
#endif
// split power tables: b^e = lo[e & (2^L - 1)] * hi[e >> L] -- one multiplication per position instead of a square-and-multiply.
//   tab[c*(2^L + 2^H) + ..] = lo[2^L] | hi[2^H] for base b_c given as pow2[c*32 + i] = b_c^(2^i)
struct pow_tab { const sc_st *tab; int L, H; };
HD uint32_t pow_tab_size(const pow_tab &t) { return (1u << t.L) + (1u << t.H); }
HD void sc_pow_tab(sc &r, const sc_st *pow2, uint64_t e) {
    sc_from_u64(r, 1);
    for (int b = 0; e; b++, e >>= 1) if (e & 1) { sc t; ld_sc(t, pow2 + b); sc_mul(r, r, t); }
}
HD void pow_tab_get(sc &r, const pow_tab &t, int c, uint64_t e) {
    const sc_st *b = t.tab + (size_t)c * pow_tab_size(t);
    sc lo, hi; ld_sc(lo, b + (e & ((1u << t.L) - 1))); ld_sc(hi, b + (1u << t.L) + (e >> t.L)); sc_mul(r, lo, hi);
}
// per-chunk sums over parties, block partials: partial[(c*gridDim.x + blockIdx.x)*q + s] (grid (blocks, C); k_sc_sum adds the blocks up).
//   phase 0 (q = 2): s=0 sum a_bl, 1 sum s_bl ;  phase 1 (q = 3, needs z and the split power table of z): s=0 sum t1_bl, 1 sum t2_bl, 2 sum z^(j+2) gamma_j
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_party_sums(sc_st *partial, const uint32_t *keys, const sc_st *blind, const sc_st *z, pow_tab ztab, int n, int m, int phase) {
    __shared__ sc_st buf[256];
    int c = blockIdx.y, tid = threadIdx.x;
    uint32_t kk[8]; for (int t = 0; t < 8; t++) kk[t] = keys[8 * c + t];
    sc s0, s1, s2; sc_0(s0); sc_0(s1); sc_0(s2);
    sc zc, zz; sc_0(zc); sc_0(zz);
    if (phase == 1) { ld_sc(zc, z + c); sc_mul(zz, zc, zc); }
    for (int j = blockIdx.x * blockDim.x + tid; j < m; j += gridDim.x * blockDim.x) {
        sc t;
        if (phase == 0) {
            nonce_scalar(t, kk, (uint64_t)j * (2 * n + 2)); sc_add(s0, s0, t);
            nonce_scalar(t, kk, (uint64_t)j * (2 * n + 2) + 1); sc_add(s1, s1, t);
        } else {
            uint64_t base = (uint64_t)m * (2 * n + 2);
            nonce_scalar(t, kk, base + 2 * (uint64_t)j); sc_add(s0, s0, t);
            nonce_scalar(t, kk, base + 2 * (uint64_t)j + 1); sc_add(s1, s1, t);
            sc zj, g; pow_tab_get(zj, ztab, c, (uint64_t)j); sc_mul(zj, zj, zz);
            ld_sc(g, blind + (size_t)c * m + j); sc_mul(g, g, zj); sc_add(s2, s2, g);
        }
    }
    block_sum_sc(s0, buf, tid, blockDim.x); block_sum_sc(s1, buf, tid, blockDim.x);
    if (phase == 1) block_sum_sc(s2, buf, tid, blockDim.x);
    if (tid == 0) {
        const int q = phase == 0 ? 2 : 3;
        sc_st *o = partial + ((size_t)c * gridDim.x + blockIdx.x) * q;
        st_sc(o, s0); st_sc(o + 1, s1); if (phase == 1) st_sc(o + 2, s2);
    }
}
KLAUNCH(k_party_sums, true, (sc_st *partial, const uint32_t *keys, const sc_st *blind, const sc_st *z, pow_tab ztab, int n, int m, int phase), (partial, keys, blind, z, ztab, n, m, phase))
#endif

// ===================================================================================================================
// K4: A = a_bl*H + sum_k (bit_k ? G_k : -H_k)     (bulletproofs Party::assign_position, aggregated over parties)
//   grid (blocks_per_chunk, C); partial[c*gridDim.x + blockIdx.x]
// ===================================================================================================================
#ifdef KG_MSM
KERNEL void LB(128, 2) k_bits_sum(p3_st *partial, const uint64_t *vals, const niels_st *G, const niels_st *H, int n, int m) {
    __shared__ p3_st buf[128];
    int c = blockIdx.y, tid = threadIdx.x;
    size_t N = (size_t)n * m;
    ge_p3 acc; ge_p3_0(acc);
    for (size_t k = (size_t)blockIdx.x * blockDim.x + tid; k < N; k += (size_t)gridDim.x * blockDim.x) {
        size_t j = k / n; int i = (int)(k % n);
        bool bit = (vals[(size_t)c * m + j] >> i) & 1;
        acc_add_niels(acc, (bit ? G : H) + k, !bit);
    }
    block_sum_p3(acc, buf, tid, blockDim.x);
    if (tid == 0) st_p3(partial + (size_t)c * gridDim.x + blockIdx.x, acc);
}
KLAUNCH(k_bits_sum, true, (p3_st *partial, const uint64_t *vals, const niels_st *G, const niels_st *H, int n, int m), (partial, vals, G, H, n, m))
#endif

// ===================================================================================================================
// K4/K6/K7: batched Pippenger multiscalar multiplication with a run-time window width c in [3, 8].
//   digit_w(x) = field_w(x + K) - (B-1),  K = sum_w (B-1) 2^(cw),  B = 2^(c-1):  signed digits in [-(B-1), B] without
//   carries to track.  One block of 128 threads owns 128/B consecutive windows of one (msm, slice): thread (wl, b) owns
//   bucket b+1 of window wl.  Per tile the scalars are read once, the terms are counting-sorted by (window, bucket) in
//   shared memory, each thread walks its own list, then the buckets of every window are combined by a suffix scan + tree
//   sum in shared memory.  Small MSMs pick small c (few buckets to reduce), large ones c = 8; a long MSM can be cut into
//   `slices` term ranges whose window sums k_finalize adds up.
// ===================================================================================================================
#define MSM_THREADS 128
#define MSM_SORT 8192
#define MSM_MAXW 85
struct msm_seg { const void *base; uint32_t count; uint32_t stride; int kind; uint32_t np; int hi; };     // kind 0 = niels_st, 1 = p3_st; stride = records per msm (0: shared)
//   np > 0: term q of the segment is record (q / np) * 2 np + (hi ? np : 0) + q % np -- the hi / lo halves of consecutive 2np-blocks (unfolded IPP round over the original generators)
struct msm_var { const sc_st *scalars; msm_seg seg[4]; };                            // scalars[idx*scalar_stride + t]
struct msm_args {
    msm_var v[2]; uint32_t split;            // msm < split: v[0] with idx = msm; else v[1] with idx = msm - split   (L / R in one launch)
    int nseg; uint32_t T, scalar_stride;
    int c, nw; uint32_t K[9];                // window bits, window count = ceil(254/c), recoding constant
    uint32_t slices, slice_len;              // slice s covers terms [s*slice_len, min(T, (s+1)*slice_len))
    p3_st *out;                              // out[(msm*slices + slice)*nw + w]
    // big-window path (k_bm_*): per (msm, window) B = 2^(c-1) buckets; start[(msm*nw + w)*(B+1) + b], cursors likewise, sorted[(msm*nw + w)*T + ..],
    // bucket sums bkt[((msm*nw + w)*B + b)*parts + part]
    uint32_t *bm_start, *bm_cur, *bm_sorted; p3_st *bm_bkt; uint32_t parts;
    // the TOP window holds only 254 - c (nw-1) bits: when that is far less than c its few buckets are enormous (every term falls into one of
    // 2^top_bits + 1 buckets) -- they are cut into parts_top pieces each instead of `parts` (0 = the top window is treated like the others)
    uint32_t top_bits, parts_top;
};
HD int msm_nw(int c) { return (254 + c - 1) / c; }
HD void msm_recode_const(uint32_t K[9], int c) {
    for (int i = 0; i < 9; i++) K[i] = 0;
    const uint32_t bm1 = (1u << (c - 1)) - 1; const int nw = msm_nw(c);
    for (int w = 0; w < nw; w++) { int bit = c * w; uint64_t v = (uint64_t)bm1 << (bit & 31); K[bit >> 5] |= (uint32_t)v; if ((bit >> 5) + 1 < 9) K[(bit >> 5) + 1] |= (uint32_t)(v >> 32); }
}
HD void msm_recode(uint32_t xk[9], const sc &x, const uint32_t K[9]) {
    uint64_t cy = 0;
    for (int i = 0; i < 8; i++) { cy += (uint64_t)x.v[i] + K[i]; xk[i] = (uint32_t)cy; cy >>= 32; }
    xk[8] = (uint32_t)cy + K[8];
}
HD int msm_digit(const uint32_t xk[9], int w, int c) {
    int bit = c * w, i = bit >> 5, sh = bit & 31;
    uint64_t v = (uint64_t)xk[i] | ((uint64_t)(i + 1 < 9 ? xk[i + 1] : 0) << 32);
    return (int)((v >> sh) & ((1u << c) - 1)) - ((1 << (c - 1)) - 1);
}
// locate the record of term t first, THEN add: lanes whose terms sit in different segments of the same kind must run ONE
// addition together (an add inside the segment loop made them take turns and halved the SIMT efficiency)
HD void msm_add_term(ge_p3 &acc, const msm_var &v, int nseg, uint32_t idx, uint32_t t, bool neg) {
    uint32_t start = 0; const void *base = nullptr; size_t rec = 0; int kind = -1;
    for (int s = 0; s < nseg; s++) {
        const msm_seg &g = v.seg[s];
        const bool here = kind < 0 && t < start + g.count;
        if (here) { const uint32_t q = t - start, j = g.np ? (q / g.np) * 2 * g.np + (g.hi ? g.np : 0) + q % g.np : q; base = g.base; rec = (size_t)idx * g.stride + j; kind = g.kind; }
        start += g.count;
    }
    if (kind == 0) acc_add_niels(acc, (const niels_st *)base + rec, neg);
    else if (kind == 1) acc_add_p3(acc, (const p3_st *)base + rec, neg);
}
#ifdef KG_MSM
KERNEL void LB(MSM_THREADS, 4) k_msm(msm_args a) {
    __shared__ uint16_t sorted[MSM_SORT];
    __shared__ int cnt[MSM_THREADS], off[MSM_THREADS + 1], cur[MSM_THREADS];
    __shared__ p3_st bk[MSM_THREADS];
    const int tid = threadIdx.x, c = a.c, B = 1 << (c - 1), wpb = MSM_THREADS / B;
    const int w0 = blockIdx.x * wpb, wl_mine = tid / B, b_mine = tid & (B - 1);
    const uint32_t msm = blockIdx.y, slice = blockIdx.z;
    const msm_var &v = msm < a.split ? a.v[0] : a.v[1];
    const uint32_t idx = msm < a.split ? msm : msm - a.split;
    const sc_st *scal = v.scalars + (size_t)idx * a.scalar_stride;
    const uint32_t t_begin = slice * a.slice_len, t_end = t_begin + a.slice_len < a.T ? t_begin + a.slice_len : a.T;
    const uint32_t tile_len = MSM_SORT / wpb;
    int nwl = a.nw - w0; if (nwl > wpb) nwl = wpb;                   // windows of this block that exist
    ge_p3 acc; ge_p3_0(acc);
    for (uint32_t tile = t_begin; tile < t_end; tile += tile_len) {
        const uint32_t nt = t_end - tile < tile_len ? t_end - tile : tile_len;
        cnt[tid] = 0;
        __syncthreads();
        for (uint32_t t = tid; t < nt; t += MSM_THREADS) {
            sc x; ld_sc(x, scal + tile + t);
            uint32_t xk[9]; msm_recode(xk, x, a.K);
            for (int wl = 0; wl < nwl; wl++) { int d = msm_digit(xk, w0 + wl, c); if (d != 0) atomicAdd(&cnt[wl * B + (d > 0 ? d : -d) - 1], 1); }
        }
        __syncthreads();
        if (tid == 0) { int o = 0; for (int b = 0; b < MSM_THREADS; b++) { off[b] = o; cur[b] = o; o += cnt[b]; } off[MSM_THREADS] = o; }
        __syncthreads();
        for (uint32_t t = tid; t < nt; t += MSM_THREADS) {
            sc x; ld_sc(x, scal + tile + t);
            uint32_t xk[9]; msm_recode(xk, x, a.K);
            for (int wl = 0; wl < nwl; wl++) {
                int d = msm_digit(xk, w0 + wl, c);
                if (d != 0) { int p = atomicAdd(&cur[wl * B + (d > 0 ? d : -d) - 1], 1); sorted[p] = (uint16_t)(t | (d < 0 ? 0x8000u : 0u)); }
            }
        }
        __syncthreads();
        for (int e = off[tid]; e < off[tid + 1]; e++) {
            uint32_t ent = sorted[e];
            msm_add_term(acc, v, a.nseg, idx, tile + (ent & 0x7fffu), (ent >> 15) != 0);
        }
        __syncthreads();
    }
    // per window: sum_b (b+1) * bucket_b  =  sum of the suffix sums
    st_p3(bk + tid, acc);
    __syncthreads();
    for (int s = 1; s < B; s <<= 1) {
        ge_p3 x, y; const bool act = b_mine + s < B;
        if (act) { ld_p3(x, bk + tid); ld_p3(y, bk + tid + s); ge_add(x, x, y); }
        __syncthreads();
        if (act) st_p3(bk + tid, x);
        __syncthreads();
    }
    for (int s = B >> 1; s > 0; s >>= 1) {
        if (b_mine < s) { ge_p3 x, y; ld_p3(x, bk + tid); ld_p3(y, bk + tid + s); ge_add(x, x, y); st_p3(bk + tid, x); }
        __syncthreads();
    }
    if (b_mine == 0 && wl_mine < nwl) { ge_p3 r; ld_p3(r, bk + tid); st_p3(a.out + ((size_t)msm * a.slices + slice) * a.nw + w0 + wl_mine, r); }
}
KLAUNCH(k_msm, true, (msm_args a), (a))
#endif

// ===================================================================================================================
// K4b: Pippenger with WIDE windows (c = 9 .. 16) for long multiscalar multiplications -- resnet18-full chunks (2^22 generators per
//   chunk: no table fits), the server's batched check over all clients' commitments, the verifier's commitment MSM.
//   k_msm keeps its buckets in one block (c <= 8: 32 additions per term, bucket lists of uneven length walked by the lanes of a warp);
//   here the (term, window) pairs are counting-sorted by bucket in global memory, so that
//     * a term costs ceil(254/c) additions (16 at c = 16 instead of 32),
//     * every thread owns one bucket (or 1/parts of it) and walks a list of Poisson-equal length: lanes of a warp stay in step,
//     * the bucket reduction sum_b b*B_b is a segmented running sum (128 threads per window).
//   k_bm_hist -> k_bm_scan -> k_bm_scatter -> k_bm_accum -> k_bm_reduce; the window sums go to k_finalize like k_msm's (slices = 1).
//   The order of the entries inside a bucket depends on the atomics' timing; the bucket SUM does not (same group element, and every
//   consumer compresses to the canonical encoding).
// ===================================================================================================================
#ifdef KG_MSM
KERNEL void LB(256, 2) k_bm_hist(msm_args a, int scatter) {
    const uint32_t msm = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.T) return;
    const msm_var &v = msm < a.split ? a.v[0] : a.v[1];
    const uint32_t idx = msm < a.split ? msm : msm - a.split, B = 1u << (a.c - 1);
    sc x; ld_sc(x, v.scalars + (size_t)idx * a.scalar_stride + t);
    uint32_t xk[9]; msm_recode(xk, x, a.K);
    for (int w = 0; w < a.nw; w++) {
        const int d = msm_digit(xk, w, a.c);
        if (d == 0) continue;
        const size_t slot = ((size_t)msm * a.nw + w) * (B + 1) + (uint32_t)(d > 0 ? d : -d) - 1;
        if (!scatter) atomicAdd(a.bm_start + slot, 1u);
        else { const uint32_t pos = atomicAdd(a.bm_cur + slot, 1u); a.bm_sorted[((size_t)msm * a.nw + w) * a.T + pos] = t | (d < 0 ? 0x80000000u : 0u); }
    }
}
KLAUNCH(k_bm_hist, false, (msm_args a, int scatter), (a, scatter))
// counts -> exclusive start offsets (B + 1 entries per (msm, window), the last one = number of non-zero digits), copied to the cursors.  grid (nw, n_msm)
KERNEL void LB(256, 1) k_bm_scan(msm_args a) {
    __shared__ uint32_t part[256];
    const uint32_t B = 1u << (a.c - 1), tid = threadIdx.x, per = (B + 1 + 255) / 256;
    uint32_t *st = a.bm_start + ((size_t)blockIdx.y * a.nw + blockIdx.x) * (B + 1), *cu = a.bm_cur + ((size_t)blockIdx.y * a.nw + blockIdx.x) * (B + 1);
    uint32_t sum = 0;
    for (uint32_t i = tid * per; i < (tid + 1) * per && i <= B; i++) sum += i < B ? st[i] : 0;
    part[tid] = sum;
    __syncthreads();
    if (tid == 0) { uint32_t o = 0; for (int i = 0; i < 256; i++) { const uint32_t c = part[i]; part[i] = o; o += c; } }
    __syncthreads();
    uint32_t o = part[tid];
    for (uint32_t i = tid * per; i < (tid + 1) * per && i <= B; i++) { const uint32_t c = i < B ? st[i] : 0; st[i] = o; cu[i] = o; o += c; }
}
KLAUNCH(k_bm_scan, true, (msm_args a), (a))
// one thread per (window, bucket, part): the sum of its share of the bucket's points.  B * parts threads per window; in a "fat" top window they
// are dealt out as parts_top threads for each of its 2^(top_bits + 1) possible buckets.
KERNEL void LB(128, 3) k_bm_accum(msm_args a) {
    const uint32_t msm = blockIdx.y, B = 1u << (a.c - 1);
    const size_t per_w = (size_t)B * a.parts, gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, total = (size_t)a.nw * per_w;
    if (gid >= total) return;
    const uint32_t w = (uint32_t)(gid / per_w), local = (uint32_t)(gid % per_w);
    const bool fat = a.parts_top && w == (uint32_t)a.nw - 1;
    const uint32_t np = fat ? a.parts_top : a.parts, part = local % np, b = local / np;
    const msm_var &v = msm < a.split ? a.v[0] : a.v[1];
    const uint32_t idx = msm < a.split ? msm : msm - a.split;
    const uint32_t *st = a.bm_start + ((size_t)msm * a.nw + w) * (B + 1), *lst = a.bm_sorted + ((size_t)msm * a.nw + w) * a.T;
    ge_p3 acc; ge_p3_0(acc);
    if (b < B) {
        const uint32_t e1 = st[b + 1];
        for (uint32_t e = st[b] + part; e < e1; e += np) { const uint32_t ent = lst[e]; msm_add_term(acc, v, a.nseg, idx, ent & 0x7fffffffu, (ent >> 31) != 0); }
    }
    st_p3(a.bm_bkt + ((size_t)msm * a.nw + w) * per_w + local, acc);
}
KLAUNCH(k_bm_accum, false, (msm_args a), (a))
// out[msm*nw + w] = sum_b (b+1) * bucket_b: thread j takes the buckets [lo, hi) of its segment -- a descending running sum gives
// sum (b - lo + 1) B_b, plus lo * (sum of the segment) by double-and-add -- and the 128 segments are added up by the block.  grid (nw, n_msm)
KERNEL void LB(128, 2) k_bm_reduce(msm_args a) {
    __shared__ p3_st buf[128];
    const uint32_t B = 1u << (a.c - 1), tid = threadIdx.x, w = blockIdx.x, msm = blockIdx.y;
    const bool fat = a.parts_top && w == (uint32_t)a.nw - 1;
    const uint32_t np = fat ? a.parts_top : a.parts, nb = fat ? (2u << a.top_bits) : B;          // buckets that can be non-empty
    const p3_st *bk = a.bm_bkt + ((size_t)msm * a.nw + w) * B * a.parts;
    ge_p3 run, acc; ge_p3_0(run); ge_p3_0(acc);
    if (nb < 128) {
        // few, heavily split buckets (fat top window): 128 / nb threads share a bucket's partial sums, then weight their share with (b + 1)
        const uint32_t tpb = 128 / nb, b = tid / tpb, lane = tid % tpb;
        if (b < nb) {
            for (uint32_t p = lane; p < np; p += tpb) acc_add_p3(run, bk + (size_t)b * np + p, false);
            for (int bit = 15; bit >= 0; bit--) { ge_p3_dbl(acc, acc); if (((b + 1) >> bit) & 1) ge_add(acc, acc, run); }
        }
    } else {
        const uint32_t per = (nb + 127) / 128, lo = tid * per, hi = lo + per < nb ? lo + per : nb;
        for (uint32_t b = hi; b-- > lo;) {
            for (uint32_t p = 0; p < np; p++) acc_add_p3(run, bk + (size_t)b * np + p, false);
            ge_add(acc, acc, run);
        }
        if (lo > 0 && lo < hi) {                       // + lo * run
            ge_p3 m; ge_p3_0(m);
            for (int bit = 15; bit >= 0; bit--) { ge_p3_dbl(m, m); if ((lo >> bit) & 1) ge_add(m, m, run); }
            ge_add(acc, acc, m);
        }
    }
    block_sum_p3(acc, buf, (int)tid, 128);
    if (tid == 0) st_p3(a.out + (size_t)msm * a.nw + w, acc);
}
KLAUNCH(k_bm_reduce, true, (msm_args a), (a))
#endif

// combine, one block per output idx:
//   R = sum_w 2^(cw) (sum_s W[idx][s][w])  +  sum of `npartial` extra points  +  sB*B + sH*H
//   sB = sBa[idx] (* sBb[idx] if sBb), same for sH; any pointer may be null.  The window sums, the extra points and the two
//   fixed-base products are computed by different threads, then four lanes run the doubling chain (one coordinate each) and thread 0 compresses.
//   out32: compressed result (nullable); out_p3: extended result (nullable); is_id: 1 if the result is the identity (nullable)
#define FIN_THREADS 128
struct finalize_args {
    const p3_st *windows; int c, nw; uint32_t slices;      // [count][slices][nw] or null
    const p3_st *partial; int npartial;                    // [count][npartial] or null
    const sc_st *sBa, *sBb, *sHa, *sHb;
    const niels_st *tabB, *tabH;
    uint8_t *out32; p3_st *out_p3; int *is_id;
    int count;
};
#ifdef KG_MSM
KERNEL void LB(FIN_THREADS, 1) k_finalize(finalize_args a) {
    __shared__ p3_st sw[MSM_MAXW + 3];
    __shared__ p3_st ex[96];
    const int idx = blockIdx.x, tid = threadIdx.x;
    if (a.windows && tid < a.nw) {
        const p3_st *src = a.windows + (size_t)idx * a.slices * a.nw + tid;
        ge_p3 r; ld_p3(r, src);
        for (uint32_t s = 1; s < a.slices; s++) acc_add_p3(r, src + (size_t)s * a.nw, false);
        if (tid == a.nw - 1) st_p3(sw + tid, r);                       // the chain starts from the top window (extended), the others are added (cached)
        else { ge_cached cr; ge_p3_to_cached(cr, r); st_cached(sw + tid, cr); }
    }
    // 96 helper threads: one radix-256 window of sB*B each (32), one of sH*H each (32), the extra points (32, strided); then a tree over the 96
    if (tid >= 32) {
        const int j = tid - 32;
        ge_p3 r; ge_p3_0(r);
        if (j < 64) {
            const bool isH = j >= 32; const int w = j & 31;
            const sc_st *sa = isH ? a.sHa : a.sBa, *sb = isH ? a.sHb : a.sBb;
            if (sa) {
                sc s; ld_sc(s, sa + idx); if (sb) { sc t; ld_sc(t, sb + idx); sc_mul(s, s, t); }
                int16_t d[32]; sc_radix256(d, s);
                const int di = d[w];
                if (di != 0) { ge_niels n; ld_niels(n, (isH ? a.tabH : a.tabB) + w * FB_ENTRIES + (di > 0 ? di : -di) - 1); ge_madd_signed(r, r, n, di < 0); }
            }
        } else for (int k = j - 64; k < a.npartial; k += 32) acc_add_p3(r, a.partial + (size_t)idx * a.npartial + k, false);
        st_p3(ex + j, r);
    }
    __syncthreads();
    for (int n = 96; n > 1;) {
        const int half = (n + 1) / 2;
        if (tid < n - half) { ge_p3 x, y; ld_p3(x, ex + tid); ld_p3(y, ex + tid + half); ge_add(x, x, y); st_p3(ex + tid, x); }
        __syncthreads();
        n = half;
    }
#ifdef ROFL_EMUL
    if (tid != 0) return;
    ge_p3 r; ld_p3(r, ex);
    if (a.windows) {
        ge_p3 h; ld_p3(h, sw + a.nw - 1);
        for (int w = a.nw - 2; w >= 0; w--) {
            ge_p2 q; ge_p1p1 t;
            ge_dbl_p1p1(t, h.X, h.Y, h.Z); ge_dbl_fix(t);
            for (int k = 1; k < a.c; k++) { ge_p1p1_to_p2(q, t); ge_dbl_p1p1(t, q.X, q.Y, q.Z); ge_dbl_fix(t); }
            ge_p1p1_to_p3(h, t);
            acc_add_cached(h, sw + w, false);
        }
        ge_add(r, r, h);
    }
#else
    // The chain sum_w 2^(cw) W_w by FOUR lanes (device): lane k owns coordinate k of (X : Y : Z : T).  A doubling is four independent squarings and
    // four independent multiplications, an addition two rounds of four independent multiplications, so the quad needs two multiplication
    // latencies + shuffles per step where one lane needs 7-9 (3076 / 4134 cycles, tools/microbench_lat.cu): the verifier's last finalize
    // (242 doublings) 0.43 -> 0.16 ms.  Warp 0 runs it (the lanes above 3 only keep the shuffles convergent).
    if (tid >= 32) return;
    ge_p3 r; ld_p3(r, ex);
    if (a.windows) {
        const int k = tid & 3, qb = tid & ~3;
        auto bc = [&](const fe &v, int from) { fe o; for (int i = 0; i < 8; i++) o.v[i] = __shfl_sync(0xffffffffu, v.v[i], qb + from); return o; };
        fe mine; { const uint32_t *wp = (const uint32_t *)(sw + a.nw - 1) + 8 * k; for (int i = 0; i < 8; i++) mine.v[i] = wp[i]; }
        for (int w = a.nw - 2; w >= 0; w--) {
            for (int it = 0; it < a.c; it++) {
                const fe X = bc(mine, 0), Y = bc(mine, 1);
                fe in = mine; if (k == 3) fe_add(in, X, Y);
                fe sq; fe_sq(sq, in);                               // XX | YY | ZZ | (X+Y)^2
                const fe xx = bc(sq, 0), yy = bc(sq, 1), zz = bc(sq, 2), xy = bc(sq, 3);
                fe Yp, Zp, Xp, Tp, tt;
                fe_add(Yp, yy, xx); fe_sub(Zp, yy, xx); fe_sub(Xp, xy, Yp);
                fe_add(tt, zz, zz); fe_add(tt, tt, xx); fe_sub(Tp, tt, yy);
                const fe &A = (k == 0 || k == 2) ? Tp : (k == 1 ? Yp : Xp), &B = k == 0 ? Xp : (k == 3 ? Yp : Zp);
                fe_mul(mine, A, B);                                 // X3 = T'X' | Y3 = Y'Z' | Z3 = T'Z' | T3 = X'Y'
            }
            {   // + W_w (cached: Y+X | Y-X | Z | 2dT)
                const fe X = bc(mine, 0), Y = bc(mine, 1);
                fe op1 = mine; if (k == 0) fe_sub(op1, Y, X); else if (k == 1) fe_add(op1, Y, X);
                fe op2; { const uint32_t *wp = (const uint32_t *)(sw + w) + 8 * (k == 0 ? 1 : k == 1 ? 0 : k); for (int i = 0; i < 8; i++) op2.v[i] = wp[i]; }
                fe pr; fe_mul(pr, op1, op2);                        // a = (Y1-X1)(Y2-X2) | b = (Y1+X1)(Y2+X2) | Z1 Z2 | c = T1 2dT2
                const fe pa = bc(pr, 0), pb = bc(pr, 1), pz = bc(pr, 2), pc = bc(pr, 3);
                fe d, E, H, G, F;
                fe_add(d, pz, pz); fe_sub(E, pb, pa); fe_add(H, pb, pa); fe_add(G, d, pc); fe_sub(F, d, pc);
                const fe &A = (k == 0 || k == 2) ? F : (k == 1 ? H : E), &B = k == 0 ? E : (k == 3 ? H : G);
                fe_mul(mine, A, B);                                 // X3 = F E | Y3 = H G | Z3 = F G | T3 = E H
            }
        }
        ge_p3 h; h.X = bc(mine, 0); h.Y = bc(mine, 1); h.Z = bc(mine, 2); h.T = bc(mine, 3);
        if (tid == 0) ge_add(r, r, h);
    }
    if (tid != 0) return;
#endif
    if (a.out32) { uint8_t o[32]; ge_compress(o, r); st_bytes32(a.out32 + 32 * (size_t)idx, o); }
    if (a.out_p3) st_p3(a.out_p3 + idx, r);
    if (a.is_id) a.is_id[idx] = ge_is_identity(r) ? 1 : 0;
}
KLAUNCH(k_finalize, true, (finalize_args a), (a))
#endif

// ===================================================================================================================
// K5: polynomial vectors of the range proof (SURVEY.md A.3 step 4), per position k = j*n + i of chunk c:
//   l0 = aL - z, l1 = sL, r0 = y^k (aL - 1 + z) + z^(j+2) 2^i, r1 = y^k sR;  partial sums t0 = <l0,r0>, t2 = <l1,r1>,
//   t1' = <l0+l1, r0+r1>.   ypow2[c*32+b] = y^(2^b), zpow2 likewise.  r1 overwrites sR.
//   partial[(c*gridDim.x + blockIdx.x)*3 + q]
// ===================================================================================================================
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_pow_tables(sc_st *tab, const sc_st *pow2, int L, int H) {
    const int c = blockIdx.y; const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x, nlo = 1u << L, n = nlo + (1u << H);
    if (e >= n) return;
    sc r; sc_pow_tab(r, pow2 + 32 * c, e < nlo ? (uint64_t)e : (uint64_t)(e - nlo) << L);
    st_sc(tab + (size_t)c * n + e, r);
}
KLAUNCH(k_pow_tables, false, (sc_st *tab, const sc_st *pow2, int L, int H), (tab, pow2, L, H))
#endif
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_poly(sc_st *l0, sc_st *r0, sc_st *sLR, sc_st *partial, const uint64_t *vals,
                             pow_tab ytab, pow_tab ztab, const sc_st *zpow2, int n, int m) {
    __shared__ sc_st buf[256];
    int c = blockIdx.y, tid = threadIdx.x;
    size_t N = (size_t)n * m;
    sc z, zz, one; ld_sc(z, zpow2 + 32 * c); ld_sc(zz, zpow2 + 32 * c + 1); sc_from_u64(one, 1);
    sc t0, t1, t2; sc_0(t0); sc_0(t1); sc_0(t2);
    for (size_t k = (size_t)blockIdx.x * blockDim.x + tid; k < N; k += (size_t)gridDim.x * blockDim.x) {
        size_t j = k / n; int i = (int)(k % n); size_t gp = (size_t)c * N + k;
        sc ey, ozz, aL, a, b, rr0, rr1, ll0, ll1, e2;
        pow_tab_get(ey, ytab, c, k);
        pow_tab_get(ozz, ztab, c, j); sc_mul(ozz, ozz, zz);
        sc_from_u64(aL, (vals[(size_t)c * m + j] >> i) & 1);
        sc_sub(ll0, aL, z);
        sc_sub(a, aL, one); sc_add(a, a, z); sc_mul(rr0, ey, a);
        sc_from_u64(e2, 1ULL << i); sc_mul(b, ozz, e2); sc_add(rr0, rr0, b);
        sc_st *sLc = sLR + (size_t)c * 2 * N, *sRc = sLc + N;
        ld_sc(rr1, sRc + k); sc_mul(rr1, ey, rr1);
        ld_sc(ll1, sLc + k);
        st_sc(l0 + gp, ll0); st_sc(r0 + gp, rr0); st_sc(sRc + k, rr1);
        sc_mul(a, ll0, rr0); sc_add(t0, t0, a);
        sc_mul(a, ll1, rr1); sc_add(t2, t2, a);
        sc_add(a, ll0, ll1); sc_add(b, rr0, rr1); sc_mul(a, a, b); sc_add(t1, t1, a);
    }
    block_sum_sc(t0, buf, tid, blockDim.x); block_sum_sc(t1, buf, tid, blockDim.x); block_sum_sc(t2, buf, tid, blockDim.x);
    if (tid == 0) { sc_st *o = partial + ((size_t)c * gridDim.x + blockIdx.x) * 3; st_sc(o, t0); st_sc(o + 1, t1); st_sc(o + 2, t2); }
}
KLAUNCH(k_poly, true, (sc_st *l0, sc_st *r0, sc_st *sLR, sc_st *partial, const uint64_t *vals, pow_tab ytab, pow_tab ztab, const sc_st *zpow2, int n, int m), (l0, r0, sLR, partial, vals, ytab, ztab, zpow2, n, m))
#endif
// out[s*C + c] = sum_{b < cnt} in[(c*cnt + b)*q + s]   (second stage of the block partial sums; C = gridDim.x)
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_sc_sum(sc_st *out, const sc_st *in, int cnt, int q) {
    __shared__ sc_st buf[256];
    int c = blockIdx.x, tid = threadIdx.x;
    for (int s = 0; s < q; s++) {
        sc acc; sc_0(acc);
        for (int b = tid; b < cnt; b += blockDim.x) { sc t; ld_sc(t, in + ((size_t)c * cnt + b) * q + s); sc_add(acc, acc, t); }
        block_sum_sc(acc, buf, tid, blockDim.x);
        if (tid == 0) st_sc(out + (size_t)s * gridDim.x + c, acc);
    }
}
KLAUNCH(k_sc_sum, true, (sc_st *out, const sc_st *in, int cnt, int q), (out, in, cnt, q))
#endif
// l = l0 + x sL (into l0), r = r0 + x r1 (into r0), yinv[k] = y^-k     (SURVEY.md A.3 step 6)
#ifdef KG_SCALAR
KERNEL void LB(256, 2) k_lr(sc_st *l0, sc_st *r0, const sc_st *sLR, sc_st *yinv, const sc_st *x, pow_tab yitab, size_t N, size_t total) {
    size_t gp = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gp >= total) return;
    size_t c = gp / N, k = gp % N;
    sc xc, a, b; ld_sc(xc, x + c);
    ld_sc(a, sLR + c * 2 * N + k); sc_mul(a, a, xc); ld_sc(b, l0 + gp); sc_add(a, a, b); st_sc(l0 + gp, a);
    ld_sc(a, sLR + c * 2 * N + N + k); sc_mul(a, a, xc); ld_sc(b, r0 + gp); sc_add(a, a, b); st_sc(r0 + gp, a);
    pow_tab_get(a, yitab, (int)c, k); st_sc(yinv + gp, a);
}
KLAUNCH(k_lr, false, (sc_st *l0, sc_st *r0, const sc_st *sLR, sc_st *yinv, const sc_st *x, pow_tab yitab, size_t N, size_t total), (l0, r0, sLR, yinv, x, yitab, N, total))
#endif

// ===================================================================================================================
// K6: inner-product argument, one round for every chunk in lock step (SURVEY.md A.4), in the "lazy factor" form:
//   with fG = prod u_k^-1, fH = prod u_k the true vectors are a = a^ / fG, b = b^ / fH, G = fG G", H_i = y^-i fH H"_i,
//   so  <a_L,b_R> = <a^_L, b^_R>,  L = <a^_L, G"_R> + <b^_R y^-i, H"_L> + c_L w B   and the folds need ONE scalar each:
//   a^ <- a^_L + u^-2 a^_R,  b^ <- b^_L + u^2 b^_R,  G" <- G"_L + u^2 G"_R,  H" <- H"_L + (u^-2 y^-n') H"_R.
//   Every L_k, R_k is the same group element the reference computes, so the compressed proof bytes are identical.
// ===================================================================================================================
// grid (blocks, C): msmL[c*2n' + ..], msmR[...], partial[(c*gridDim.x+blk)*2 + {cL,cR}]
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_ipp_scalars(const sc_st *a, const sc_st *b, const sc_st *yinv, sc_st *msmL, sc_st *msmR, sc_st *partial, size_t N, uint32_t np) {
    __shared__ sc_st buf[256];
    int c = blockIdx.y, tid = threadIdx.x;
    const sc_st *ac = a + (size_t)c * N, *bc = b + (size_t)c * N, *yc = yinv + (size_t)c * N;
    sc cL, cR; sc_0(cL); sc_0(cR);
    for (uint32_t i = blockIdx.x * blockDim.x + tid; i < np; i += gridDim.x * blockDim.x) {
        sc alo, ahi, blo, bhi, ylo, yhi, t;
        ld_sc(alo, ac + i); ld_sc(ahi, ac + np + i); ld_sc(blo, bc + i); ld_sc(bhi, bc + np + i); ld_sc(ylo, yc + i); ld_sc(yhi, yc + np + i);
        sc_mul(t, alo, bhi); sc_add(cL, cL, t);
        sc_mul(t, ahi, blo); sc_add(cR, cR, t);
        st_sc(msmL + (size_t)c * 2 * np + i, alo);
        sc_mul(t, bhi, ylo); st_sc(msmL + (size_t)c * 2 * np + np + i, t);
        st_sc(msmR + (size_t)c * 2 * np + i, ahi);
        sc_mul(t, blo, yhi); st_sc(msmR + (size_t)c * 2 * np + np + i, t);
    }
    block_sum_sc(cL, buf, tid, blockDim.x); block_sum_sc(cR, buf, tid, blockDim.x);
    if (tid == 0) { sc_st *o = partial + ((size_t)c * gridDim.x + blockIdx.x) * 2; st_sc(o, cL); st_sc(o + 1, cR); }
}
KLAUNCH(k_ipp_scalars, true, (const sc_st *a, const sc_st *b, const sc_st *yinv, sc_st *msmL, sc_st *msmR, sc_st *partial, size_t N, uint32_t np), (a, b, yinv, msmL, msmR, partial, N, np))
#endif
// a^[i] += uinv2[c] a^[np+i],  b^[i] += u2[c] b^[np+i]
#ifdef KG_SCALAR
KERNEL void LB(256, 2) k_ipp_fold_scalars(sc_st *a, sc_st *b, const sc_st *u2, const sc_st *uinv2, size_t N, uint32_t np) {
    int c = blockIdx.y;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    sc_st *ac = a + (size_t)c * N, *bc = b + (size_t)c * N;
    sc s, lo, hi;
    ld_sc(s, uinv2 + c); ld_sc(lo, ac + i); ld_sc(hi, ac + np + i); sc_mul(hi, hi, s); sc_add(lo, lo, hi); st_sc(ac + i, lo);
    ld_sc(s, u2 + c); ld_sc(lo, bc + i); ld_sc(hi, bc + np + i); sc_mul(hi, hi, s); sc_add(lo, lo, hi); st_sc(bc + i, lo);
}
KLAUNCH(k_ipp_fold_scalars, false, (sc_st *a, sc_st *b, const sc_st *u2, const sc_st *uinv2, size_t N, uint32_t np), (a, b, u2, uinv2, N, np))
#endif
// generator fold: out[c][i] = P[i] + s_c * P[np + i], s_c given as width-FOLD_W NAF nafs[(c*2 + which)*256 ..]
//   grid (blocks, C, 2): z = 0 folds G (scalar u^2), z = 1 folds H (scalar u^-2 y^-np).
//   first round: in = shared niels generators (in_stride 0); later rounds: in == out (p3, in place, stride = out_stride)
#define FOLD_W 5
struct fold_args {
    const niels_st *Gn, *Hn;       // first round sources (or null)
    p3_st *Gf, *Hf;                // folded generators [C][stride]
    const int8_t *nafs;
    uint32_t np, stride;
};
#ifdef KG_FOLD
KERNEL void LB(128, 4) k_ipp_fold_points(fold_args a) {
    __shared__ int8_t naf[256];
    int c = blockIdx.y, which = blockIdx.z, tid = threadIdx.x;
    for (int t = tid; t < 256; t += blockDim.x) naf[t] = a.nafs[((size_t)c * 2 + which) * 256 + t];
    __syncthreads();
    uint32_t i = blockIdx.x * blockDim.x + tid;
    if (i >= a.np) return;
    ge_p3 lo, hi, r;
    p3_st *dst = (which ? a.Hf : a.Gf) + (size_t)c * a.stride;
    if (a.Gn) {
        const niels_st *src = which ? a.Hn : a.Gn;
        ge_niels nl, nh; ld_niels(nl, src + i); ld_niels(nh, src + a.np + i);
        ge_niels_to_p3(lo, nl); ge_niels_to_p3(hi, nh);
    } else { ld_p3(lo, dst + i); ld_p3(hi, dst + a.np + i); }
    ge_fold(r, naf, lo, hi, FOLD_W);
    st_p3(dst + i, r);
}
KLAUNCH(k_ipp_fold_points, true, (fold_args a), (a))
#endif


// ===================================================================================================================
// K7: verifier side (RangeProof::verify_multiple, SURVEY.md A.3)
// ===================================================================================================================
// decompress `count` encodings; optionally add a fixed point (offset, as p3) -- verify_rangeproof shifts every
// commitment by 2^(n-1) B (range_proof_vec/mod.rs:155-160) and pads with the identity (:163-165).
//   in: count_in encodings; out p3 [count_out] (entries >= count_in are the identity); out32: compressed shifted points
//   bad[i / bad_group] is set to 1 if encoding i fails to decode
#ifdef KG_COMMIT
KERNEL void LB(128, 2) k_decompress(p3_st *out, uint8_t *out32, const uint8_t *in, size_t count_in, size_t count_out, const p3_st *offset, int *bad, size_t bad_group) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count_out) return;
    ge_p3 p; ge_p3_0(p);
    if (i < count_in) {
        uint8_t b[32]; ld_bytes32(b, in + 32 * i);
        if (!ge_decompress(p, b)) { atomicOr(bad + i / bad_group, 1); ge_p3_0(p); }
        if (offset) { ge_p3 o; ld_p3(o, offset); ge_add(p, p, o); }
    }
    st_p3(out + i, p);
    if (out32) { uint8_t o[32]; ge_compress(o, p); st_bytes32(out32 + 32 * i, o); }
}
KLAUNCH(k_decompress, false, (p3_st *out, uint8_t *out32, const uint8_t *in, size_t count_in, size_t count_out, const p3_st *offset, int *bad, size_t bad_group), (out, out32, in, count_in, count_out, offset, bad, bad_group))
// the same for K updates in one launch (server side, one update per client): update k's D encodings start at in + 32 k D and fill entries
// [k Dp, k Dp + D) of the outputs, the rest of its Dp entries is identity padding; bad[k] is set if one of ITS encodings does not decode
KERNEL void LB(128, 2) k_decompress_batch(p3_st *out, uint8_t *out32, const uint8_t *in, size_t D, size_t Dp, size_t K, const p3_st *offset, int *bad) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * Dp) return;
    const size_t k = i / Dp, j = i % Dp;
    ge_p3 p; ge_p3_0(p);
    if (j < D) {
        uint8_t b[32]; ld_bytes32(b, in + 32 * (k * D + j));
        if (!ge_decompress(p, b)) { atomicOr(bad + k, 1); ge_p3_0(p); }
        if (offset) { ge_p3 o; ld_p3(o, offset); ge_add(p, p, o); }
    }
    st_p3(out + i, p);
    if (out32) { uint8_t o[32]; ge_compress(o, p); st_bytes32(out32 + 32 * i, o); }
}
KLAUNCH(k_decompress_batch, false, (p3_st *out, uint8_t *out32, const uint8_t *in, size_t D, size_t Dp, size_t K, const p3_st *offset, int *bad), (out, out32, in, D, Dp, K, offset, bad))
#endif
// Batched verification: all C chunks of a call share the generators, so the verifier takes one random weight rho_c per chunk
// and checks  sum_c rho_c * (chunk c's verification equation) == 0  with ONE 2N-term generator MSM (soundness error 2^-252;
// the reference ANDs the per-chunk verdicts, range_proof_vec/mod.rs:183-190).
// per-chunk challenge block prepared by the host (all canonical scalars):
//   [0] rho z  [1] rho z^2  [2] rho a  [3] rho b  [4] c (the reference's own batching scalar)  [5..5+lgN) u_k  [5+lgN..5+2lgN) u_k^-1
// k_verify_tables builds per-chunk split tables (k = khi 2^L + klo, j = jhi 2^Lm + jlo) so that every per-position factor is
// one product of two table entries instead of a lgN-step square-and-multiply:
//   tab[c] = S_lo[2^L] | S_hi[2^H] | Y_lo[2^L] | Y_hi[2^H] | Z_lo[2^Lm] | Z_hi[2^Hm]
//   s_k = S_lo[klo] S_hi[khi] (= prod_p bit_p(k) ? u_(lgN-1-p) : u^-1_(lgN-1-p)),  y^-k = Y_lo Y_hi,  rho z^2 z^j = Z_lo Z_hi
// and the per-chunk commitment scalars var[c*var_stride + j] = c * rho z^2 z^j.
struct vtab_layout { int lgN, L, H, lgm, Lm, Hm; uint32_t oSlo, oShi, oYlo, oYhi, oZlo, oZhi, total; };
HD vtab_layout vtab_make(int lgN, int lgm) {
    vtab_layout t; t.lgN = lgN; t.L = lgN / 2; t.H = lgN - t.L; t.lgm = lgm; t.Lm = lgm / 2; t.Hm = lgm - t.Lm;
    t.oSlo = 0; t.oShi = t.oSlo + (1u << t.L); t.oYlo = t.oShi + (1u << t.H); t.oYhi = t.oYlo + (1u << t.L);
    t.oZlo = t.oYhi + (1u << t.H); t.oZhi = t.oZlo + (1u << t.Lm); t.total = t.oZhi + (1u << t.Hm);
    return t;
}
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_verify_tables(sc_st *tab, vtab_layout t, sc_st *var, uint32_t var_stride, const sc_st *chal, int chal_stride, const sc_st *yinvpow2, const sc_st *zpow2, int m) {
    const int c = blockIdx.y;
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    const sc_st *ch = chal + (size_t)c * chal_stride;
    sc_st *out = tab + (size_t)c * t.total;
    if (e < t.oYlo) {                                   // S_lo / S_hi
        const bool hi = e >= t.oShi; const uint32_t v = hi ? e - t.oShi : e; const int p0 = hi ? t.L : 0, nb = hi ? t.H : t.L;
        sc s; sc_from_u64(s, 1);
        for (int q = 0; q < nb; q++) { const int tt = t.lgN - 1 - (p0 + q); sc f; ld_sc(f, ((v >> q) & 1) ? ch + 5 + tt : ch + 5 + t.lgN + tt); sc_mul(s, s, f); }
        st_sc(out + e, s);
    } else if (e < t.oZlo) {                            // Y_lo[j] = y^-j, Y_hi[j] = y^-(j 2^L)
        const bool hi = e >= t.oYhi; const uint64_t v = hi ? (uint64_t)(e - t.oYhi) << t.L : e - t.oYlo;
        sc s; sc_pow_tab(s, yinvpow2 + 32 * c, v); st_sc(out + e, s);
    } else if (e < t.total) {                           // Z_lo[j] = rho z^2 z^j, Z_hi[j] = z^(j 2^Lm)
        const bool hi = e >= t.oZhi; const uint64_t v = hi ? (uint64_t)(e - t.oZhi) << t.Lm : e - t.oZlo;
        sc s; sc_pow_tab(s, zpow2 + 32 * c, v);
        if (!hi) { sc r; ld_sc(r, ch + 1); sc_mul(s, s, r); }
        st_sc(out + e, s);
    } else if (e < t.total + (uint32_t)m) {             // commitment scalars
        const uint32_t j = e - t.total;
        sc s, r, cc; sc_pow_tab(s, zpow2 + 32 * c, j); ld_sc(r, ch + 1); ld_sc(cc, ch + 4); sc_mul(s, s, r); sc_mul(s, s, cc);
        st_sc(var + (size_t)c * var_stride + j, s);          // var_stride = m: the commitment scalars of all chunks are contiguous
    }
}
KLAUNCH(k_verify_tables, false, (sc_st *tab, vtab_layout t, sc_st *var, uint32_t var_stride, const sc_st *chal, int chal_stride, const sc_st *yinvpow2, const sc_st *zpow2, int m),
        (tab, t, var, var_stride, chal, chal_stride, yinvpow2, zpow2, m))
// gh[k] = sum_c rho_c g_(c,k) = sum_c -(rho z + rho a s_k);  gh[N + k] = sum_c rho z + y^-k (rho z^2 z^j 2^i - rho b s_k^-1),  k = j n + i
// block = 64 positions x 4 chunk lanes (lane cs takes chunks cs, cs+4, ..), partial sums joined through shared memory: 4x the blocks of a
// thread-per-position layout (N = 16 384 positions would fill only 64 blocks)
KERNEL void LB(256, 1) k_verify_scalars(sc_st *gh, const sc_st *tab, vtab_layout t, const sc_st *chal, int chal_stride, int n, int C) {
    __shared__ sc_st part[2][4][64];
    const size_t N = (size_t)1 << t.lgN;
    const int pl = threadIdx.x & 63, cs = threadIdx.x >> 6;
    const size_t k = (size_t)blockIdx.x * 64 + pl;
    sc g, h; sc_0(g); sc_0(h);
    if (k < N) {
        const uint32_t mL = (1u << t.L) - 1, mH = (1u << t.H) - 1, mLm = (1u << t.Lm) - 1;
        const uint32_t klo = (uint32_t)k & mL, khi = (uint32_t)(k >> t.L);
        const size_t j = k / n; const int i = (int)(k % n);
        sc e2; sc_from_u64(e2, 1ULL << i);
        for (int c = cs; c < C; c += 4) {
            const sc_st *tb = tab + (size_t)c * t.total, *ch = chal + (size_t)c * chal_stride;
            sc a, b, s, sinv, yk, zj, rz, ra, rb, t1;
            ld_sc(a, tb + t.oSlo + klo); ld_sc(b, tb + t.oShi + khi); sc_mul(s, a, b);
            ld_sc(a, tb + t.oSlo + (~klo & mL)); ld_sc(b, tb + t.oShi + (~khi & mH)); sc_mul(sinv, a, b);
            ld_sc(a, tb + t.oYlo + klo); ld_sc(b, tb + t.oYhi + khi); sc_mul(yk, a, b);
            ld_sc(a, tb + t.oZlo + ((uint32_t)j & mLm)); ld_sc(b, tb + t.oZhi + (uint32_t)(j >> t.Lm)); sc_mul(zj, a, b);
            ld_sc(rz, ch); ld_sc(ra, ch + 2); ld_sc(rb, ch + 3);
            sc_mul(t1, ra, s); sc_add(t1, t1, rz); sc_sub(g, g, t1);
            sc_mul(zj, zj, e2); sc_mul(t1, rb, sinv); sc_sub(zj, zj, t1); sc_mul(zj, zj, yk); sc_add(h, h, zj); sc_add(h, h, rz);
        }
    }
    st_sc(&part[0][cs][pl], g); st_sc(&part[1][cs][pl], h);
    __syncthreads();
    if (cs == 0 && k < N) {
        for (int q = 1; q < 4; q++) { sc x; ld_sc(x, &part[0][q][pl]); sc_add(g, g, x); ld_sc(x, &part[1][q][pl]); sc_add(h, h, x); }
        st_sc(gh + k, g); st_sc(gh + N + k, h);
    }
}
KLAUNCH(k_verify_scalars, true, (sc_st *gh, const sc_st *tab, vtab_layout t, const sc_st *chal, int chal_stride, int n, int C), (gh, tab, t, chal, chal_stride, n, C))
#endif

// ===================================================================================================================
// K8: per-element square proofs (square_proof_vec/mod.rs)
// ===================================================================================================================
struct square_args {
    const float *values; const uint8_t *value_com, *r1, *r2; size_t D; int n_bits, frac;
    uint32_t key[8];
    const niels_st *tabB, *tabH;
    uint8_t *proofs, *commits;     // D x 160, D x 64
    int *flags;                    // bit 1 NaN, bit 4 bad point
};
#ifdef KG_SQUARE
KERNEL void LB(128, 1) k_square_prove(square_args a) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.D) return;
    uint8_t cl[32], r1[32], r2[32], proof[160], com[64];
    ld_bytes32(cl, a.value_com + 32 * i); ld_bytes32(r1, a.r1 + 32 * i); ld_bytes32(r2, a.r2 + 32 * i);
    int rc = square_prove_one(proof, com, a.values[i], cl, r1, r2, a.key, (uint64_t)i, a.n_bits, a.frac, a.tabB, a.tabH);
    if (rc) { atomicOr(a.flags, rc == -1 ? 1 : 4); return; }
    for (int k = 0; k < 5; k++) st_bytes32(a.proofs + 160 * i + 32 * k, proof + 32 * k);
    st_bytes32(a.commits + 64 * i, com); st_bytes32(a.commits + 64 * i + 32, com + 32);
}
KLAUNCH(k_square_prove, false, (square_args a), (a))
#endif
// result[0] &= all valid ; result[1] |= format error
#ifdef KG_SQUARE
//   group: elements per update when several updates are checked in one launch (result = 2 ints per update); 0 = one update
KERNEL void LB(128, 1) k_square_verify(const uint8_t *proofs, const uint8_t *commits, size_t D, const niels_st *tabB, const niels_st *tabH, int *result, size_t group) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    if (group) result += 2 * (i / group);
    uint8_t proof[160], com[64];
    for (int k = 0; k < 5; k++) ld_bytes32(proof + 32 * k, proofs + 160 * i + 32 * k);
    ld_bytes32(com, commits + 64 * i); ld_bytes32(com + 32, commits + 64 * i + 32);
    int rc = square_verify_one(proof, com, tabB, tabH);
    if (rc < 0) atomicOr(result + 1, 1);
    else if (rc == 0) atomicAnd(result, 0);
}
KLAUNCH(k_square_verify, false, (const uint8_t *proofs, const uint8_t *commits, size_t D, const niels_st *tabB, const niels_st *tabH, int *result, size_t group), (proofs, commits, D, tabB, tabH, result, group))
#endif

// the un-optimised encodings' per-element proofs (enc types 2 and 3): same shape as K8, one thread per element.
//   kind 1 = RandProof (pair 64 B, proof 128 B), kind 2 = SquareRandProof (commitments 96 B, proof 192 B)
struct sigma_args {
    int kind; const float *values; const uint8_t *value_com, *r1, *r2; size_t D; int n_bits, frac;
    uint32_t key[8]; const niels_st *tabB, *tabH;
    uint8_t *proofs, *commits; int *flags;
};
#ifdef KG_SQUARE
KERNEL void LB(128, 1) k_sigma_prove(sigma_args a) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.D) return;
    uint8_t vc[32], r1[32], r2[32], proof[192], com[96];
    if (a.value_com) ld_bytes32(vc, a.value_com + 32 * i);
    ld_bytes32(r1, a.r1 + 32 * i);
    const int pw = a.kind == 1 ? 4 : 6, cw = a.kind == 1 ? 2 : 3;
    int rc;
    if (a.kind == 1) rc = rand_prove_one(proof, com, a.values[i], a.value_com ? vc : nullptr, r1, a.key, (uint64_t)i, a.n_bits, a.frac, a.tabB, a.tabH);
    else { ld_bytes32(r2, a.r2 + 32 * i); rc = square_rand_prove_one(proof, com, a.values[i], a.value_com ? vc : nullptr, r1, r2, a.key, (uint64_t)i, a.n_bits, a.frac, a.tabB, a.tabH); }
    if (rc) { atomicOr(a.flags, rc == -1 ? 1 : 4); return; }
    for (int k = 0; k < pw; k++) st_bytes32(a.proofs + 32 * (pw * i + k), proof + 32 * k);
    for (int k = 0; k < cw; k++) st_bytes32(a.commits + 32 * (cw * i + k), com + 32 * k);
}
KLAUNCH(k_sigma_prove, false, (sigma_args a), (a))
//   group: elements per update when several updates are checked in one launch (result = 2 ints per update, counted from the launch's first
//   element, which starts an update); 0 = one update
KERNEL void LB(128, 1) k_sigma_verify(int kind, const uint8_t *proofs, const uint8_t *commits, size_t D, const niels_st *tabB, const niels_st *tabH, int *result, size_t group) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    if (group) result += 2 * (i / group);
    uint8_t proof[192], com[96];
    const int pw = kind == 1 ? 4 : 6, cw = kind == 1 ? 2 : 3;
    for (int k = 0; k < pw; k++) ld_bytes32(proof + 32 * k, proofs + 32 * (pw * i + k));
    for (int k = 0; k < cw; k++) ld_bytes32(com + 32 * k, commits + 32 * (cw * i + k));
    const int rc = kind == 1 ? rand_verify_one(proof, com, tabB, tabH) : square_rand_verify_one(proof, com, tabB, tabH);
    if (rc < 0) atomicOr(result + 1, 1);
    else if (rc == 0) atomicAnd(result, 0);
}
KLAUNCH(k_sigma_verify, false, (int kind, const uint8_t *proofs, const uint8_t *commits, size_t D, const niels_st *tabB, const niels_st *tabH, int *result, size_t group),
        (kind, proofs, commits, D, tabB, tabH, result, group))
#endif

// ---- the same verdict for ALL square proofs (kind 0), rand proofs (kind 1) or square-rand proofs (kind 2) of a call with ONE random linear
//        combination per range of elements (engine.cuh, sigma_verify_groups).  Per element, every kind checks the L equation, kind 1 and kind 2
//        the R equation, kind 0 and kind 2 the square equation (square_verify_one, rand_verify_one, square_rand_verify_one; z_r = z_r1, and
//        L = C_l for a square proof):
//          L:  z_m B + z_r H == C'_L + c L          R:  z_r B == C'_R + c R          square:  z_m L + z_r2 H == C'_sq + c C_sq
//   Weighted by a_i (L), b_i (R) and q_i (square) and negated, the sum over the elements of a range is one MSM plus two fixed-base terms:
//     kind 0:  sum_i a C'_l + (a c - q z_m) C_l + q C'_sq + q c C_sq                                   - (sum a z_m) B - (sum a z_r1 + q z_r2) H == 0
//     kind 1:  sum_i a C'_L + a c L + b C'_R + b c R                                                     - (sum a z_m + b z_r) B - (sum a z_r) H == 0
//     kind 2:  sum_i a C'_L + (a c - q z_m) L + b C'_R + b c R + q C'_sq + q c C_sq                    - (sum a z_m + b z_r1) B - (sum a z_r1 + q z_r2) H == 0
//   Weights: key_i = SHA3-256(root | seed | tag | LE64 N | LE64 i) over the N elements of the call (kind 0: no seed), root = the hash tree
//   (k_hash_tree) over leaf_i = SHA3-256(0x00 | commitments_i | proof_i); one ChaCha20 block of key_i gives the weights of the equations the kind
//   checks, in the order a, b, q, from words 0..4, 5..9, 10..14 (kind 0: a = 0..4, q = 5..9), each masked to wbits bits.  They stay short and
//   positive, so that their upper windows are zero digits the MSM skips: the signs live in the fixed-base coefficients only.  (Negated weights
//   l - w share their upper 125 bits: every term fell into the same bucket of the upper windows and one thread added millions of points.)
//   For square proofs one MSM over 4 N points replaces, per element, two fixed-base and two variable-base scalar multiplications (~7 100 field
//   multiplications -> ~1 700 incl. the four decompressions).
//   A malformed element (non-canonical response, undecodable point) sets the bad flag of its update (element i belongs to update i / group).
//   k_sigma_rlc_prep:    format checks, challenge c_i, leaf digest_i                         (one thread per element of the call)
//   k_hash_tree:         out[j] = SHA3-256(0x01 | in[64 j .. 64 j + 63])                    (levels until one digest is left)
//   k_sigma_rlc_scalars: weights, the np point scalars of the element, block sums of the B and H scalars         (elements [i0, i0 + n))
//   k_sigma_rlc_points:  the np points of each element of the range                          (one thread per point)
// The layout of one element of each kind, in 32-byte words, and the equations it checks besides L.  Its np MSM points (and scalars) are, in this
// order, C'_L, L (, C'_R, R) (, C'_sq, C_sq): even ones from the proof, odd ones from the commitments, word w / 2 of each; the responses
// z_m, z_r (, z_r2) are the proof's words np / 2 .. pw - 1.
struct sigma_kind { int cw, pw, np; bool req, sqeq, seeded; };
HD constexpr sigma_kind sigma_kind_of(int kind) {
    return kind == 0 ? sigma_kind{2, 5, 4, false, true, false}       // square proof:      C_l, C_sq      | C'_l, C'_sq, z_m, z_r1, z_r2
         : kind == 1 ? sigma_kind{2, 4, 4, true, false, true}        // rand proof:        L, R           | C'_L, C'_R, z_m, z_r
         :             sigma_kind{3, 6, 6, true, true, true};        // square-rand proof: L, R, C_sq     | C'_L, C'_R, C'_sq, z_m, z_r1, z_r2
}
struct sigma_rlc_args {
    int kind; const uint8_t *proofs, *commits; size_t N, group, i0, n; uint32_t tag; uint8_t seed[32];
    uint8_t *digest; sc_st *chal; const uint8_t *root; sc_st *scal, *partial; p3_st *pts; int *bad; int wbits;
};
#ifdef KG_SQUARE
KERNEL void LB(128, 1) k_sigma_rlc_prep(sigma_rlc_args a) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.N) return;
    const sigma_kind sk = sigma_kind_of(a.kind);
    uint8_t buf[288];                                                              // commitments | proof
    for (int k = 0; k < sk.cw; k++) ld_bytes32(buf + 32 * k, a.commits + 32 * (sk.cw * i + k));
    for (int k = 0; k < sk.pw; k++) ld_bytes32(buf + 32 * (sk.cw + k), a.proofs + 32 * (sk.pw * i + k));
    const uint8_t *com = buf, *proof = buf + 32 * sk.cw;
    sc z; bool ok = true;
    for (int k = sk.np / 2; k < sk.pw; k++) { sc_frombytes(z, proof + 32 * k); ok = ok && sc_is_canonical(z); }
    if (!ok) atomicOr(a.bad + i / a.group, 1);
    sc c;
    if (a.kind == 0) sq_transcript_challenge(c, com, com + 32, proof, proof + 32);
    else if (a.kind == 1) rp_transcript_challenge(c, com, proof);
    else srp_transcript_challenge(c, com, proof);
    st_sc(a.chal + i, c);
    // leaf of the hash tree: tag 0x00 (inner nodes absorb 0x01 first, so that no element's bytes can pass for a node of the tree)
    uint8_t dg[32]; { sponge sp; sponge_init(sp, 136); const uint8_t tag = 0x00; sponge_absorb(sp, &tag, 1); sponge_absorb(sp, buf, 32 * (sk.cw + sk.pw)); sponge_finish(sp, 0x06); sponge_squeeze(sp, dg, 32); }
    st_bytes32(a.digest + 32 * i, dg);
}
KLAUNCH(k_sigma_rlc_prep, false, (sigma_rlc_args a), (a))
KERNEL void LB(128, 1) k_hash_tree(uint8_t *out, const uint8_t *in, size_t n) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x, lo = 64 * j;
    if (lo >= n) return;
    const size_t cnt = n - lo < 64 ? n - lo : 64;
    sponge sp; sponge_init(sp, 136);
    { const uint8_t tag = 0x01; sponge_absorb(sp, &tag, 1); }
    for (size_t k = 0; k < cnt; k++) { uint8_t d[32]; ld_bytes32(d, in + 32 * (lo + k)); sponge_absorb(sp, d, 32); }
    sponge_finish(sp, 0x06);
    uint8_t o[32]; sponge_squeeze(sp, o, 32); st_bytes32(out + 32 * j, o);
}
KLAUNCH(k_hash_tree, false, (uint8_t *out, const uint8_t *in, size_t n), (out, in, n))
KERNEL void LB(128, 1) k_sigma_rlc_scalars(sigma_rlc_args a) {
    __shared__ sc_st buf[128];
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; const int tid = threadIdx.x;
    sc sB, sH; sc_0(sB); sc_0(sH);
    if (t < a.n) {
        const size_t i = a.i0 + t;
        const sigma_kind sk = sigma_kind_of(a.kind);
        uint8_t kb[84], key[32]; ld_bytes32(kb, a.root);
        int kt = 32;                                                               // where the tag goes: after the seed, if the kind has one
        if (sk.seeded) { for (int k = 0; k < 32; k++) kb[32 + k] = a.seed[k]; kt = 64; }
        for (int k = 0; k < 4; k++) kb[kt + k] = (uint8_t)(a.tag >> (8 * k));
        for (int k = 0; k < 8; k++) { kb[kt + 4 + k] = (uint8_t)((uint64_t)a.N >> (8 * k)); kb[kt + 12 + k] = (uint8_t)((uint64_t)i >> (8 * k)); }
        sha3_256(key, kb, kt + 20);
        uint32_t kw[8], w[16];
        for (int k = 0; k < 8; k++) kw[k] = (uint32_t)key[4 * k] | ((uint32_t)key[4 * k + 1] << 8) | ((uint32_t)key[4 * k + 2] << 16) | ((uint32_t)key[4 * k + 3] << 24);
        chacha20_block_words(w, kw, 0);
        // weights of wbits = c * ceil(126 / c) - 1 bits (125 .. 134, engine.cuh rlc_wbits) for the MSM's window width c: their top window then holds c - 1 uniform bits and the
        // recoding never carries out of it.  (With 128-bit weights at c = 16 half of all short scalars got the digit +1 in the window above -- ONE bucket
        // with millions of points, seconds of serial additions; at other widths the few-bit top window had the same effect on a smaller scale.)
        sc wa, wb, wq; sc_0(wa); sc_0(wb); sc_0(wq);                             // weights of the L, R and square equations (0 where the kind has none)
        for (int k = 0; k < 5; k++) {
            wa.v[k] = w[k];
            if (sk.req) wb.v[k] = w[5 + k];
            if (sk.sqeq) wq.v[k] = sk.req ? w[10 + k] : w[5 + k];
        }
        { const int full = a.wbits >> 5, rem = a.wbits & 31;
          for (int k = 0; k < 5; k++) { const uint32_t m = k < full ? 0xffffffffu : (k == full ? ((1u << rem) - 1u) : 0u); wa.v[k] &= m; wb.v[k] &= m; wq.v[k] &= m; } }
        uint8_t zb[32]; sc zm, zr, c, u, v;
        const uint8_t *pf = a.proofs + 32 * (sk.pw * i + sk.np / 2);               // z_m | z_r (| z_r2)
        ld_bytes32(zb, pf); sc_frombytes(zm, zb);
        ld_bytes32(zb, pf + 32); sc_frombytes(zr, zb);
        ld_sc(c, a.chal + i);
        sc_st *o = a.scal + sk.np * t;
        st_sc(o, wa);                                                              // C'_L:  a
        sc_mul(u, wa, c);                                                          // L:     a c (- q z_m)
        sc_mul(sB, wa, zm);                                                        // B:     -(a z_m (+ b z_r))
        sc_mul(sH, wa, zr);                                                        // H:     -(a z_r (+ q z_r2))
        if (sk.req) {
            st_sc(o + 2, wb);                                                      // C'_R:  b
            sc_mul(v, wb, c); st_sc(o + 3, v);                                     // R:     b c
            sc_mul(v, wb, zr); sc_add(sB, sB, v);
        }
        if (sk.sqeq) {
            sc zr2; ld_bytes32(zb, pf + 64); sc_frombytes(zr2, zb);
            sc_mul(v, wq, zm); sc_sub(u, u, v);
            st_sc(o + sk.np - 2, wq);                                              // C'_sq: q
            sc_mul(v, wq, c); st_sc(o + sk.np - 1, v);                             // C_sq:  q c
            sc_mul(v, wq, zr2); sc_add(sH, sH, v);
        }
        st_sc(o + 1, u);
        sc_neg(sB, sB); sc_neg(sH, sH);
    }
    block_sum_sc(sB, buf, tid, 128);
    if (tid == 0) st_sc(a.partial + 2 * (size_t)blockIdx.x, sB);
    block_sum_sc(sH, buf, tid, 128);
    if (tid == 0) st_sc(a.partial + 2 * (size_t)blockIdx.x + 1, sH);
}
KLAUNCH(k_sigma_rlc_scalars, true, (sigma_rlc_args a), (a))
KERNEL void LB(128, 2) k_sigma_rlc_points(sigma_rlc_args a) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const sigma_kind sk = sigma_kind_of(a.kind);
    if (t >= (size_t)sk.np * a.n) return;
    const size_t i = a.i0 + t / sk.np; const int w = (int)(t % sk.np);
    const uint8_t *src = (w & 1) ? a.commits + 32 * (sk.cw * i + (w >> 1)) : a.proofs + 32 * (sk.pw * i + (w >> 1));
    uint8_t enc[32]; ld_bytes32(enc, src);
    ge_p3 P;
    if (!ge_decompress(P, enc)) { atomicOr(a.bad + i / a.group, 1); ge_p3_0(P); }
    st_p3(a.pts + t, P);
}
KLAUNCH(k_sigma_rlc_points, false, (sigma_rlc_args a), (a))
#endif

// ===================================================================================================================
// K9: homomorphic aggregation over clients (params.rs:81-124, pedersen_ops.rs:56-69); pts[client][D] compressed
// ===================================================================================================================
#ifdef KG_COMMIT
KERNEL void LB(128, 2) k_aggregate(uint8_t *out, const uint8_t *pts, size_t n_clients, size_t D, int init_base, int *bad) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    ge_p3 acc; if (init_base) ge_base(acc); else ge_p3_0(acc);
    for (size_t c = 0; c < n_clients; c++) {
        uint8_t b[32]; ld_bytes32(b, pts + 32 * (c * D + i));
        ge_p3 p; if (!ge_decompress(p, b)) { atomicOr(bad, 1); continue; }
        ge_add(acc, acc, p);
    }
    uint8_t o[32]; ge_compress(o, acc); st_bytes32(out + 32 * i, o);
}
KLAUNCH(k_aggregate, false, (uint8_t *out, const uint8_t *pts, size_t n_clients, size_t D, int init_base, int *bad), (out, pts, n_clients, D, init_base, bad))
#endif

// ===================================================================================================================
// K10: baby-step giant-step discrete log (bsgs32.rs:20-73).  The table maps the first 8 bytes of compress(x B) (an
//   injective key with overwhelming probability; the full encoding is stored for an exact compare) to x, in an
//   open-addressing hash table of `cap` (power of two) slots that lives in HBM / L2.
// ===================================================================================================================
// Table = two arrays of `cap` (power of two) slots: keys[] (u64, 0xff..ff = empty) and vals[] (u32, x+1).
#define BSGS_EMPTY 0xffffffffffffffffULL
HD unsigned long long bsgs_key(const ge_p3 &p) {
    uint8_t o[32]; ge_compress(o, p);
    unsigned long long k = 0; for (int i = 0; i < 8; i++) k |= (unsigned long long)o[i] << (8 * i);
    return k == BSGS_EMPTY ? BSGS_EMPTY - 1 : k;
}
HD uint32_t bsgs_hash(unsigned long long k, uint32_t cap) { return (uint32_t)((k * 0x9E3779B97F4A7C15ULL) >> 24) & (cap - 1); }
// entry x in [0, m]: key(compress(x B)) -> x+1.  Later entries overwrite earlier ones on equal keys (HashMap::insert,
// bsgs32.rs:26-33): atomicMax makes that independent of thread order.  distinct counts the occupied slots (table.len()).
#ifdef KG_BSGS
KERNEL void LB(128, 2) k_bsgs_build(unsigned long long *keys, uint32_t *vals, uint32_t cap, uint32_t m, const niels_st *tabB, int *distinct) {
    uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x > m) return;
    ge_p3 p; ge_p3_0(p); sc s; sc_from_u64(s, x); fb_mul_acc(p, tabB, s, 32);
    unsigned long long k = bsgs_key(p);
    uint32_t pos = bsgs_hash(k, cap);
    for (uint32_t probe = 0; probe < cap; probe++) {
        unsigned long long prev = atomicCAS(&keys[pos], BSGS_EMPTY, k);
        if (prev == BSGS_EMPTY) atomicAdd(distinct, 1);
        if (prev == BSGS_EMPTY || prev == k) { atomicMax(&vals[pos], x + 1); return; }
        pos = (pos + 1) & (cap - 1);
    }
}
KLAUNCH(k_bsgs_build, false, (unsigned long long *keys, uint32_t *vals, uint32_t cap, uint32_t m, const niels_st *tabB, int *distinct), (keys, vals, cap, m, tabB, distinct))
#endif
// exact lookup: a key hit is confirmed by recomputing x B and comparing group elements
HD bool bsgs_lookup(uint32_t &val, const unsigned long long *keys, const uint32_t *vals, uint32_t cap, const ge_p3 &p, const niels_st *tabB) {
    unsigned long long k = bsgs_key(p);
    uint32_t pos = bsgs_hash(k, cap);
    for (uint32_t probe = 0; probe < cap; probe++) {
        unsigned long long cur = keys[pos];
        if (cur == BSGS_EMPTY) return false;
        if (cur == k) {
            uint32_t x = vals[pos] - 1;
            ge_p3 q; ge_p3_0(q); sc s; sc_from_u64(s, x); fb_mul_acc(q, tabB, s, 32);
            if (ge_eq(q, p)) { val = x; return true; }
        }
        pos = (pos + 1) & (cap - 1);
    }
    return false;
}
// solve_discrete_log_with_neg (bsgs32.rs:48-73): up to max_it giant steps for M, then for -M.
//   size = distinct - 1 (get_size), mG = (m & vmask) B, result (it*size + val) & vmask; miss on both signs -> flag 8
// Element i of a point M already in extended coordinates: shared by k_bsgs_solve (M decompressed from the wire) and k_acc_extract (M = the
// accumulated L, resident on the device).
DEV void bsgs_solve_point(uint8_t *out_sc, float *out_f32, size_t i, const ge_p3 &M, const unsigned long long *keys, const uint32_t *vals, uint32_t cap,
                         uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags) {
    uint64_t vmask = (1ULL << bsgs_bits) - 1;
    ge_p3 mG; ge_p3_0(mG); { sc s; sc_from_u64(s, (uint64_t)m & vmask); fb_mul_acc(mG, tabB, s, 32); }
    int found = 0; uint64_t val = 0;
    for (int sign = 0; sign < 2 && !found; sign++) {
        ge_p3 cur; if (sign) ge_neg(cur, M); else cur = M;
        for (uint64_t it = 0; it < max_it && !found; it++) {
            uint32_t v;
            if (bsgs_lookup(v, keys, vals, cap, cur, tabB)) { found = 1 + sign; val = (it * size + (v & vmask)) & vmask; }
            else ge_sub(cur, cur, mG);
        }
    }
    sc r; sc_0(r);
    if (!found) { atomicOr(flags, 8); for (int k = 0; k < 8; k++) r.v[k] = 0xffffffffu; }
    else { sc_from_u64(r, val); if (found == 2) sc_neg(r, r); }
    if (out_sc) { uint8_t o[32]; sc_tobytes(o, r); st_bytes32(out_sc + 32 * i, o); }
    if (out_f32) out_f32[i] = found ? scalar_to_f32(r, n_bits, frac) : 0.0f;
}
#ifdef KG_BSGS
KERNEL void LB(128, 2) k_bsgs_solve(uint8_t *out_sc, float *out_f32, const uint8_t *pts, size_t D, const unsigned long long *keys, const uint32_t *vals, uint32_t cap,
                                   uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32]; ld_bytes32(b, pts + 32 * i);
    ge_p3 M; if (!ge_decompress(M, b)) { atomicOr(flags, 4); return; }
    bsgs_solve_point(out_sc, out_f32, i, M, keys, vals, cap, m, size, max_it, bsgs_bits, n_bits, frac, tabB, flags);
}
KLAUNCH(k_bsgs_solve, false, (uint8_t *out_sc, float *out_f32, const uint8_t *pts, size_t D, const unsigned long long *keys, const uint32_t *vals, uint32_t cap, uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags), (out_sc, out_f32, pts, D, keys, vals, cap, m, size, max_it, bsgs_bits, n_bits, frac, tabB, flags))
#endif

// ===================================================================================================================
// K9b / K10b: device-resident round accumulator (EncModelParamsAccumulator, params.rs:74-148).  The state is `ncols` columns of
//   D extended points, column-major: st[col * D + i] (col 0 = L, col 1 = R).  Records are the wire records of the clients
//   (rec_bytes = 32 | 64 | 96, client-major, L at offset 0, R at 32, c_sq at 64 -- c_sq is validated by the caller, never added).
// ===================================================================================================================
#ifdef KG_COMMIT
// every element at the unity (B, B) (ElGamalPair::unity, el_gamal.rs:83-88) or at the identity
KERNEL void LB(256, 2) k_acc_init(p3_st *st, size_t n, int init_base) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_p3 p; if (init_base) ge_base(p); else ge_p3_0(p);
    st_p3(st + i, p);
}
KLAUNCH(k_acc_init, false, (p3_st *st, size_t n, int init_base), (st, n, init_base))
// adds the accepted clients `clients[0 .. n_acc)` of one call: their points were all validated before (k_validate_points), so every
// decompression here succeeds -- a client is added entirely or not at all
KERNEL void LB(128, 2) k_acc_add(p3_st *st, size_t D, int ncols, const uint8_t *rec, size_t rec_bytes, const uint32_t *clients, uint32_t n_acc) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    for (int col = 0; col < ncols; col++) {
        ge_p3 acc; ld_p3(acc, st + col * D + i);
        for (uint32_t c = 0; c < n_acc; c++) {
            uint8_t b[32]; ld_bytes32(b, rec + rec_bytes * ((size_t)clients[c] * D + i) + 32 * col);
            ge_p3 p; ge_decompress(p, b);
            ge_add(acc, acc, p);
        }
        st_p3(st + col * D + i, acc);
    }
}
KLAUNCH(k_acc_add, false, (p3_st *st, size_t D, int ncols, const uint8_t *rec, size_t rec_bytes, const uint32_t *clients, uint32_t n_acc), (st, D, ncols, rec, rec_bytes, clients, n_acc))
// canonical encodings: out[i * 32 ncols + 32 col] = compress(st[col * D + i])  (D x 32 or D x 64 = L | R)
KERNEL void LB(128, 2) k_acc_export(uint8_t *out, const p3_st *st, size_t D, int ncols) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= D * ncols) return;
    const size_t i = t / ncols, col = t % ncols;
    ge_p3 p; ld_p3(p, st + col * D + i);
    uint8_t o[32]; ge_compress(o, p); st_bytes32(out + 32 * t, o);
}
KLAUNCH(k_acc_export, false, (uint8_t *out, const p3_st *st, size_t D, int ncols), (out, st, D, ncols))
#endif
#ifdef KG_BSGS
// EncModelParamsAccumulator::extract (params.rs:126-147): R == B (Ristretto equality, el_gamal.rs:101-103) for every element when check_R,
// else flag 16; then BSGS on the resident L exactly as k_bsgs_solve after its decompression.  Once a wrong R has been seen, later threads
// skip their discrete log (the host returns ROFL_ERR_UNBALANCED and hands out no result).
KERNEL void LB(128, 2) k_acc_extract(uint8_t *out_sc, float *out_f32, const p3_st *st, size_t D, int check_R, const unsigned long long *keys, const uint32_t *vals, uint32_t cap,
                                     uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    if (check_R) {
        ge_p3 R, B; ld_p3(R, st + D + i); ge_base(B);
        if (!ge_eq(R, B)) { atomicOr(flags, 16); return; }
    }
    if (*(volatile int *)flags & 16) return;
    ge_p3 M; ld_p3(M, st + i);
    bsgs_solve_point(out_sc, out_f32, i, M, keys, vals, cap, m, size, max_it, bsgs_bits, n_bits, frac, tabB, flags);
}
KLAUNCH(k_acc_extract, false, (uint8_t *out_sc, float *out_f32, const p3_st *st, size_t D, int check_R, const unsigned long long *keys, const uint32_t *vals, uint32_t cap, uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags), (out_sc, out_f32, st, D, check_R, keys, vals, cap, m, size, max_it, bsgs_bits, n_bits, frac, tabB, flags))
#endif

// K1: conversions exposed on their own (conversion32.rs:11-38, range_proof_vec/mod.rs:104-111)
#ifdef KG_COMMIT
KERNEL void k_f32_to_scalar(uint8_t *out, const float *v, size_t D, int n_bits, int frac, int *flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    sc s; if (f32_to_scalar(s, v[i], n_bits, frac)) { atomicOr(flags, 1); sc_0(s); }
    uint8_t o[32]; sc_tobytes(o, s); st_bytes32(out + 32 * i, o);
}
KLAUNCH(k_f32_to_scalar, false, (uint8_t *out, const float *v, size_t D, int n_bits, int frac, int *flags), (out, v, D, n_bits, frac, flags))
#endif
#ifdef KG_COMMIT
KERNEL void k_scalar_to_f32(float *out, const uint8_t *in, size_t D, int n_bits, int frac) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32]; ld_bytes32(b, in + 32 * i); sc s; sc_from_bytes_mod_order(s, b);
    out[i] = scalar_to_f32(s, n_bits, frac);
}
KLAUNCH(k_scalar_to_f32, false, (float *out, const uint8_t *in, size_t D, int n_bits, int frac), (out, in, D, n_bits, frac))
#endif
// sum of squares of f32_to_scalar(x) mod l and sum of blindings (l2_range_proof_vec/mod.rs:37-42,75-79): block partials
#ifdef KG_COMMIT
KERNEL void LB(256, 1) k_l2_sums(sc_st *partial, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, int *flags) {
    __shared__ sc_st buf[256];
    int tid = threadIdx.x;
    sc sq, bs; sc_0(sq); sc_0(bs);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + tid; i < D; i += (size_t)gridDim.x * blockDim.x) {
        sc s, t; if (f32_to_scalar(s, v[i], n_bits, frac)) { atomicOr(flags, 1); continue; }
        sc_mul(t, s, s); sc_add(sq, sq, t);
        uint8_t b[32]; ld_bytes32(b, blind + 32 * i); sc_from_bytes_mod_order(t, b); sc_add(bs, bs, t);
    }
    block_sum_sc(sq, buf, tid, blockDim.x); block_sum_sc(bs, buf, tid, blockDim.x);
    if (tid == 0) { st_sc(partial + 2 * blockIdx.x, sq); st_sc(partial + 2 * blockIdx.x + 1, bs); }
}
KLAUNCH(k_l2_sums, true, (sc_st *partial, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, int *flags), (partial, v, blind, D, n_bits, frac, flags))
#endif

// ===================================================================================================================
// K9: compressed randomness proof (compressed_rand_proof/mod.rs:43-102, party.rs:90-100): one sigma proof over all D ElGamal pairs
//   z_m = m' + sum_i m_i c^(i+1),  z_r = r' + sum_i r_i c^(i+1);  verify: commit(z_m, z_r) == C' + sum_i c^(i+1) (L_i, R_i)
// ===================================================================================================================
#ifdef KG_COMMIT
// block partial sums of m_i c^(i+1) and r_i c^(i+1); ctab = split power table of c (chunk 0)
KERNEL void LB(256, 1) k_crp_sums(sc_st *partial, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, pow_tab ctab, int *flags) {
    __shared__ sc_st buf[256];
    int tid = threadIdx.x;
    sc sm, sr; sc_0(sm); sc_0(sr);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + tid; i < D; i += (size_t)gridDim.x * blockDim.x) {
        sc m, r, pw, t; if (f32_to_scalar(m, v[i], n_bits, frac)) { atomicOr(flags, 1); continue; }
        uint8_t b[32]; ld_bytes32(b, blind + 32 * i); sc_from_bytes_mod_order(r, b);
        pow_tab_get(pw, ctab, 0, i + 1);
        sc_mul(t, m, pw); sc_add(sm, sm, t); sc_mul(t, r, pw); sc_add(sr, sr, t);
    }
    block_sum_sc(sm, buf, tid, blockDim.x); block_sum_sc(sr, buf, tid, blockDim.x);
    if (tid == 0) { st_sc(partial + 2 * blockIdx.x, sm); st_sc(partial + 2 * blockIdx.x + 1, sr); }
}
KLAUNCH(k_crp_sums, true, (sc_st *partial, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, pow_tab ctab, int *flags), (partial, v, blind, D, n_bits, frac, ctab, flags))
// out[i] = c^(i+1)
KERNEL void LB(256, 2) k_crp_pows(sc_st *out, size_t D, pow_tab ctab) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    sc pw; pow_tab_get(pw, ctab, 0, i + 1); st_sc(out + i, pw);
}
KLAUNCH(k_crp_pows, false, (sc_st *out, size_t D, pow_tab ctab), (out, D, ctab))
// pairs[i] = L[i] | R[i]  (64-byte wire form of an ElGamalPair, el_gamal.rs:105-111) and the reverse
KERNEL void LB(256, 2) k_pairs_join(uint8_t *pairs, const uint8_t *L, const uint8_t *R, size_t D) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32]; ld_bytes32(b, L + 32 * i); st_bytes32(pairs + 64 * i, b); ld_bytes32(b, R + 32 * i); st_bytes32(pairs + 64 * i + 32, b);
}
KLAUNCH(k_pairs_join, false, (uint8_t *pairs, const uint8_t *L, const uint8_t *R, size_t D), (pairs, L, R, D))
KERNEL void LB(256, 2) k_pairs_split(uint8_t *L, uint8_t *R, const uint8_t *pairs, size_t D) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32]; ld_bytes32(b, pairs + 64 * i); st_bytes32(L + 32 * i, b); ld_bytes32(b, pairs + 64 * i + 32); st_bytes32(R + 32 * i, b);
}
KLAUNCH(k_pairs_split, false, (uint8_t *L, uint8_t *R, const uint8_t *pairs, size_t D), (L, R, pairs, D))
// L halves of the first `num` of the D pairs of each of K updates -> out[K x num x 32] (the Pedersen commitments a prefix range check is about)
KERNEL void LB(256, 2) k_pairs_gather_L(uint8_t *out, const uint8_t *pairs, size_t D, size_t num, size_t K) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * num) return;
    const size_t k = i / num, j = i % num;
    uint8_t b[32]; ld_bytes32(b, pairs + 64 * (k * D + j)); st_bytes32(out + 32 * i, b);
}
KLAUNCH(k_pairs_gather_L, false, (uint8_t *out, const uint8_t *pairs, size_t D, size_t num, size_t K), (out, pairs, D, num, K))
// Batched check of G compressed rand proofs (engine.cuh, engine_crp_verify_batch).  Points: n = G D + G terms per side,
//   P[0, n)  = L of every client (client-major) | C'_L of every client,   P[n, 2n) = R ... | C'_R ...
// from pairs[G x D x 64] and cp[G x 64] (C'_L | C'_R); an undecodable encoding sets bad[client] and contributes the identity.
KERNEL void LB(128, 2) k_crp_batch_points(p3_st *P, const uint8_t *pairs, const uint8_t *cp, size_t D, uint32_t G, int *bad) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, GD = (size_t)G * D, n = GD + G;
    if (i >= 2 * n) return;
    const size_t which = i >= n ? 1 : 0, j = i - which * n;
    const bool pair = j < GD;
    const uint8_t *src = pair ? pairs + 64 * j + 32 * which : cp + 64 * (j - GD) + 32 * which;
    uint8_t b[32]; ld_bytes32(b, src);
    ge_p3 p; if (!ge_decompress(p, b)) { atomicOr(bad + (pair ? j / D : j - GD), 1); ge_p3_0(p); }
    st_p3(P + i, p);
}
KLAUNCH(k_crp_batch_points, false, (p3_st *P, const uint8_t *pairs, const uint8_t *cp, size_t D, uint32_t G, int *bad), (P, pairs, cp, D, G, bad))
// the MSM scalars of that check: s[k D + i] = rho_k c_k^(i+1) (the split power table of c_k is table k of ctab), s[G D + k] = rho_k.
// Nothing is negated here: the signs live in the fixed-base coefficients of k_finalize (negated short weights would share one bucket).
KERNEL void LB(256, 2) k_crp_batch_scalars(sc_st *s, size_t D, uint32_t G, pow_tab ctab, const sc_st *rho) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, GD = (size_t)G * D;
    if (i >= GD + G) return;
    sc r;
    if (i < GD) {
        const size_t k = i / D;
        sc pw, w; pow_tab_get(pw, ctab, (int)k, i - k * D + 1); ld_sc(w, rho + k); sc_mul(r, pw, w);
    } else ld_sc(r, rho + (i - GD));
    st_sc(s + i, r);
}
KLAUNCH(k_crp_batch_scalars, false, (sc_st *s, size_t D, uint32_t G, pow_tab ctab, const sc_st *rho), (s, D, G, ctab, rho))
#endif

// ===================================================================================================================
// K12: wire records of the optimised encodings (params.rs:408-458,554-605; SURVEY Appendix C) and the sum of a point vector
// ===================================================================================================================
#ifdef KG_COMMIT
// SquareRandProofCommitments, 96 bytes = c.L | c.R | c_sq (square_rand_proof/pedersen.rs:21-30)
KERNEL void LB(256, 2) k_join96(uint8_t *out96, const uint8_t *pairs64, const uint8_t *sq64, size_t D) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32];
    ld_bytes32(b, pairs64 + 64 * i); st_bytes32(out96 + 96 * i, b);
    ld_bytes32(b, pairs64 + 64 * i + 32); st_bytes32(out96 + 96 * i + 32, b);
    ld_bytes32(b, sq64 + 64 * i + 32); st_bytes32(out96 + 96 * i + 64, b);          // c_sq of SquareProofCommitments (c_l | c_sq)
}
KLAUNCH(k_join96, false, (uint8_t *out96, const uint8_t *pairs64, const uint8_t *sq64, size_t D), (out96, pairs64, sq64, D))
// -> L[D x 32] (the Pedersen halves the range proofs are about), sq64[D x 64] = c_l | c_sq (SquareProofCommitments), csq[D x 32]
KERNEL void LB(256, 2) k_split96(uint8_t *L, uint8_t *sq64, uint8_t *csq, const uint8_t *in96, size_t D) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32];
    ld_bytes32(b, in96 + 96 * i); st_bytes32(L + 32 * i, b); st_bytes32(sq64 + 64 * i, b);
    ld_bytes32(b, in96 + 96 * i + 64); st_bytes32(sq64 + 64 * i + 32, b); st_bytes32(csq + 32 * i, b);
}
KLAUNCH(k_split96, false, (uint8_t *L, uint8_t *sq64, uint8_t *csq, const uint8_t *in96, size_t D), (L, sq64, csq, in96, D))
// from_bytes validation of one column of compressed points inside fixed-width wire records: *bad = 1 if record i's 32 bytes at `offset` do
// not decode (ElGamalPair::from_bytes, rand_proof/el_gamal.rs:112-123; SquareRandProofCommitments::from_bytes, square_rand_proof/pedersen.rs:33-45)
//   group: records per update when several updates are validated in one launch (one flag per update); 0 = one update
KERNEL void LB(128, 2) k_validate_points(const uint8_t *rec, size_t stride, size_t offset, size_t D, int *bad, size_t group) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    uint8_t b[32]; ld_bytes32(b, rec + stride * i + offset);
    ge_p3 p; if (!ge_decompress(p, b)) atomicOr(bad + (group ? i / group : 0), 1);
}
KLAUNCH(k_validate_points, false, (const uint8_t *rec, size_t stride, size_t offset, size_t D, int *bad, size_t group), (rec, stride, offset, D, bad, group))
// partial[blockIdx.x] = sum of this block's share of D compressed points (params.rs:267: enc_values.iter().map(|x| x.c_sq).sum())
//   blockIdx.y = update k when several are summed in one launch: points pts32 + 32 k D, partial[k gridDim.x + blockIdx.x], bad[k]
KERNEL void LB(128, 2) k_points_sum(p3_st *partial, const uint8_t *pts32, size_t D, int *bad) {
    __shared__ p3_st buf[128];
    const int tid = threadIdx.x;
    pts32 += 32 * (size_t)blockIdx.y * D; partial += (size_t)blockIdx.y * gridDim.x; bad += blockIdx.y;
    ge_p3 acc; ge_p3_0(acc);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + tid; i < D; i += (size_t)gridDim.x * blockDim.x) {
        uint8_t b[32]; ld_bytes32(b, pts32 + 32 * i);
        ge_p3 p; if (!ge_decompress(p, b)) { atomicOr(bad, 1); continue; }
        ge_add(acc, acc, p);
    }
    block_sum_p3(acc, buf, tid, blockDim.x);
    if (tid == 0) st_p3(partial + blockIdx.x, acc);
}
KLAUNCH(k_points_sum, true, (p3_st *partial, const uint8_t *pts32, size_t D, int *bad), (partial, pts32, D, bad))
#endif

// ---- launcher declarations (definitions live in the translation unit of each kernel group) ----------------------------
void launch_k_fb_table_build(dim3 g_, dim3 b_, cudaStream_t s_, niels_st *tab, const uint8_t *pt);
void launch_k_gens_build(dim3 g_, dim3 b_, cudaStream_t s_, niels_st *G, niels_st *H, int n, int party_begin, int party_end);
void launch_k_commit(dim3 g_, dim3 b_, cudaStream_t s_, commit_args a);
void launch_k_field_selftest(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const uint8_t *a32, const uint8_t *b32, size_t n);
void launch_k_scalar_selftest(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const uint8_t *a32, const uint8_t *b32, size_t n);
void launch_k_nonces(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *sLR, const uint32_t *keys, int n, int m, size_t total);
void launch_k_party_sums(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *partial, const uint32_t *keys, const sc_st *blind, const sc_st *z, pow_tab ztab, int n, int m, int phase);
void launch_k_bits_sum(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *partial, const uint64_t *vals, const niels_st *G, const niels_st *H, int n, int m);
void launch_k_msm(dim3 g_, dim3 b_, cudaStream_t s_, msm_args a);
void launch_k_bm_hist(dim3 g_, dim3 b_, cudaStream_t s_, msm_args a, int scatter);
void launch_k_bm_scan(dim3 g_, dim3 b_, cudaStream_t s_, msm_args a);
void launch_k_bm_accum(dim3 g_, dim3 b_, cudaStream_t s_, msm_args a);
void launch_k_bm_reduce(dim3 g_, dim3 b_, cudaStream_t s_, msm_args a);
void launch_k_finalize(dim3 g_, dim3 b_, cudaStream_t s_, finalize_args a);
void launch_k_pow_tables(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *tab, const sc_st *pow2, int L, int H);
void launch_k_poly(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *l0, sc_st *r0, sc_st *sLR, sc_st *partial, const uint64_t *vals, pow_tab ytab, pow_tab ztab, const sc_st *zpow2, int n, int m);
void launch_k_sc_sum(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *out, const sc_st *in, int cnt, int q);
void launch_k_lr(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *l0, sc_st *r0, const sc_st *sLR, sc_st *yinv, const sc_st *x, pow_tab yitab, size_t N, size_t total);
void launch_k_ipp_scalars(dim3 g_, dim3 b_, cudaStream_t s_, const sc_st *a, const sc_st *b, const sc_st *yinv, sc_st *msmL, sc_st *msmR, sc_st *partial, size_t N, uint32_t np);
void launch_k_ipp_fold_scalars(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *a, sc_st *b, const sc_st *u2, const sc_st *uinv2, size_t N, uint32_t np);
void launch_k_ipp_fold_points(dim3 g_, dim3 b_, cudaStream_t s_, fold_args a);
void launch_k_decompress_batch(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *out, uint8_t *out32, const uint8_t *in, size_t D, size_t Dp, size_t K, const p3_st *offset, int *bad);
void launch_k_decompress(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *out, uint8_t *out32, const uint8_t *in, size_t count_in, size_t count_out, const p3_st *offset, int *bad, size_t bad_group);
void launch_k_verify_tables(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *tab, vtab_layout t, sc_st *var, uint32_t var_stride, const sc_st *chal, int chal_stride, const sc_st *yinvpow2, const sc_st *zpow2, int m);
void launch_k_verify_scalars(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *gh, const sc_st *tab, vtab_layout t, const sc_st *chal, int chal_stride, int n, int C);
void launch_k_square_prove(dim3 g_, dim3 b_, cudaStream_t s_, square_args a);
void launch_k_sigma_prove(dim3 g_, dim3 b_, cudaStream_t s_, sigma_args a);
void launch_k_sigma_verify(dim3 g_, dim3 b_, cudaStream_t s_, int kind, const uint8_t *proofs, const uint8_t *commits, size_t D, const niels_st *tabB, const niels_st *tabH, int *result, size_t group);
void launch_k_sigma_rlc_prep(dim3 g_, dim3 b_, cudaStream_t s_, sigma_rlc_args a);
void launch_k_sigma_rlc_scalars(dim3 g_, dim3 b_, cudaStream_t s_, sigma_rlc_args a);
void launch_k_sigma_rlc_points(dim3 g_, dim3 b_, cudaStream_t s_, sigma_rlc_args a);
void launch_k_square_verify(dim3 g_, dim3 b_, cudaStream_t s_, const uint8_t *proofs, const uint8_t *commits, size_t D, const niels_st *tabB, const niels_st *tabH, int *result, size_t group);
void launch_k_hash_tree(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const uint8_t *in, size_t n);
void launch_k_aggregate(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const uint8_t *pts, size_t n_clients, size_t D, int init_base, int *bad);
void launch_k_bsgs_build(dim3 g_, dim3 b_, cudaStream_t s_, unsigned long long *keys, uint32_t *vals, uint32_t cap, uint32_t m, const niels_st *tabB, int *distinct);
void launch_k_bsgs_solve(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out_sc, float *out_f32, const uint8_t *pts, size_t D, const unsigned long long *keys, const uint32_t *vals, uint32_t cap, uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags);
void launch_k_acc_init(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *st, size_t n, int init_base);
void launch_k_acc_add(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *st, size_t D, int ncols, const uint8_t *rec, size_t rec_bytes, const uint32_t *clients, uint32_t n_acc);
void launch_k_acc_export(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const p3_st *st, size_t D, int ncols);
void launch_k_acc_extract(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out_sc, float *out_f32, const p3_st *st, size_t D, int check_R, const unsigned long long *keys, const uint32_t *vals, uint32_t cap, uint32_t m, uint64_t size, uint64_t max_it, int bsgs_bits, int n_bits, int frac, const niels_st *tabB, int *flags);
void launch_k_f32_to_scalar(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const float *v, size_t D, int n_bits, int frac, int *flags);
void launch_k_scalar_to_f32(dim3 g_, dim3 b_, cudaStream_t s_, float *out, const uint8_t *in, size_t D, int n_bits, int frac);
void launch_k_l2_sums(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *partial, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, int *flags);
void launch_k_join96(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out96, const uint8_t *pairs64, const uint8_t *sq64, size_t D);
void launch_k_validate_points(dim3 g_, dim3 b_, cudaStream_t s_, const uint8_t *rec, size_t stride, size_t offset, size_t D, int *bad, size_t group);
void launch_k_split96(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *L, uint8_t *sq64, uint8_t *csq, const uint8_t *in96, size_t D);
void launch_k_points_sum(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *partial, const uint8_t *pts32, size_t D, int *bad);
void launch_k_crp_sums(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *partial, const float *v, const uint8_t *blind, size_t D, int n_bits, int frac, pow_tab ctab, int *flags);
void launch_k_crp_pows(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *out, size_t D, pow_tab ctab);
void launch_k_pairs_join(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *pairs, const uint8_t *L, const uint8_t *R, size_t D);
void launch_k_pairs_split(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *L, uint8_t *R, const uint8_t *pairs, size_t D);
void launch_k_pairs_gather_L(dim3 g_, dim3 b_, cudaStream_t s_, uint8_t *out, const uint8_t *pairs, size_t D, size_t num, size_t K);
void launch_k_crp_batch_points(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *P, const uint8_t *pairs, const uint8_t *cp, size_t D, uint32_t G, int *bad);
void launch_k_crp_batch_scalars(dim3 g_, dim3 b_, cudaStream_t s_, sc_st *s, size_t D, uint32_t G, pow_tab ctab, const sc_st *rho);

// ===================================================================================================================
// RT path: per-generator radix-256 tables in HBM (512 KB per generator: 32 windows x 128 affine-Niels multiples).
//   Fixed generators never need doublings, buckets or sorting: s*G_j = sum_w +-RT[j][w][|d_w|-1]  (<= 32 mixed adds).
//   Used for S, the verifier's G/H part, the first IPP rounds in "unfolded" form and the catch-up fold (engine.cuh).
//   Layout: RT[(j*nw + w)*B + k] = (k+1) * 2^(cw) * Gen_j ;  j < n*m for G, then the same for H in a second array.
// ===================================================================================================================
// run-time radix 2^c (c = 8, 9 or 10): nw = ceil(254/c) windows of B = 2^(c-1) multiples; same signed recoding as k_msm
#define RT_MAXW 32
#define RT_MAX_BITS 11                    // widest table radix: 2^11 -> 24 windows of 1024 records (77 GB for 2 x 32768 generators)
struct rt_tables { const niels_st *G, *H; int c, nw, B; uint32_t K[9]; };
HD size_t rt_row_entries(const rt_tables &t) { return (size_t)t.nw * t.B; }      // niels records per generator
#ifdef KG_TABLES
// step 1: P[j*nw + w] = 2^(cw) * Gen_j  (one thread per generator, c doublings per window)
KERNEL void LB(128, 2) k_rt_shifts(p3_st *P, const niels_st *gens, uint32_t count, int c, int nw) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    ge_niels g; ld_niels(g, gens + j);
    ge_p3 p; ge_niels_to_p3(p, g);
    for (int w = 0; w < nw; w++) {
        st_p3(P + (size_t)j * nw + w, p);
        for (int k = 0; k < c; k++) ge_p3_dbl(p, p);
    }
}
KLAUNCH(k_rt_shifts, false, (p3_st *P, const niels_st *gens, uint32_t count, int c, int nw), (P, gens, count, c, nw))
// step 2: one thread per (row = j*nw+w, group of 16 multiples): entries 16g+1 .. 16g+16 of row, converted to affine with
// one shared inversion (Montgomery's trick over the 16 Z's)
KERNEL void LB(128, 2) k_rt_rows(niels_st *RT, const p3_st *P, size_t rows, int B) {
    const int gpr = B / 16;                               // groups per row
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * gpr) return;
    size_t row = idx / gpr; int grp = (int)(idx % gpr);
    ge_p3 base; ld_p3(base, P + row);
    ge_cached cb; ge_p3_to_cached(cb, base);
    // start = (16 grp + 1) * base
    ge_p3 cur; ge_p3_0(cur);
    { uint32_t k = 16 * grp + 1; for (int b = 9; b >= 0; b--) { ge_p3_dbl(cur, cur); if ((k >> b) & 1) ge_add_cached(cur, cur, cb); } }
    ge_p3 pts[16]; fe pre[16], acc; fe_1(acc);
    for (int e = 0; e < 16; e++) { pts[e] = cur; pre[e] = acc; fe_mul(acc, acc, cur.Z); if (e < 15) ge_add_cached(cur, cur, cb); }
    fe inv; fe_invert(inv, acc);
    for (int e = 15; e >= 0; e--) {
        fe zinv; fe_mul(zinv, inv, pre[e]); fe_mul(inv, inv, pts[e].Z);
        ge_niels n; ge_p3_to_niels(n, pts[e], zinv);
        st_niels(RT + row * B + 16 * grp + e, n);
    }
}
KLAUNCH(k_rt_rows, false, (niels_st *RT, const p3_st *P, size_t rows, int B), (RT, P, rows, B))
#endif

// signed digits of a scalar for all nw windows at once (same recoding as k_msm: digit_w = field_w(x + K) - (B-1))
HD void rt_digits(int16_t d[RT_MAXW], const sc &x, const rt_tables &t) {
    uint32_t xk[9]; msm_recode(xk, x, t.K);
    for (int w = 0; w < t.nw; w++) d[w] = (int16_t)msm_digit(xk, w, t.c);
}
HD void rt_mul_acc(ge_p3 &acc, const niels_st *row0, const sc &x, const rt_tables &t) {          // acc += x * Gen ; row0 = RT + j*nw*B
    uint32_t xk[9]; msm_recode(xk, x, t.K);
    for (int w = 0; w < t.nw; w++) {
        const int dw = msm_digit(xk, w, t.c);
        if (dw != 0) acc_add_niels(acc, row0 + (size_t)w * t.B + (dw > 0 ? dw : -dw) - 1, dw < 0);
    }
}
// direct table MSM: out partial[msm*gridDim.x + blockIdx.x] = sum over this block's terms of s_t * Gen_{map(t)}.
//   terms t < T per msm; scalars[msm*scalar_stride + t]; generator of term t:
//     mode 0: t < nG -> G[t], else H[t - nG]                                         (S, verifier: all generators in order)
//     mode 1/2 (unfolded IPP round, np = half block): the G part uses the hi (mode 1, "L") or lo (mode 2, "R") half of every
//       2np block, the H part the opposite half:  q < nG: j = (q/np)*2np + (hiG ? np : 0) + q%np
struct rt_msm_args { const sc_st *scalars; uint32_t T, scalar_stride, nG, np; int mode; rt_tables rt; p3_st *partial; };
// Table records are gathered from ~40 GB of HBM at random: every thread stages its next RTM_STAGES-1 records in its own
// shared-memory slots with cp.async (no registers held across the latency, no block barrier: a thread only reads what it
// copied itself), and the scalar of its next term likewise.  Slot layout [stage][16-byte piece][thread] -> conflict-free LDS.128.
#ifndef RTM_STAGES
#define RTM_STAGES 3
#endif
#ifndef RTM_BLOCKS
#define RTM_BLOCKS 4                     // resident blocks per SM the table kernels are compiled for
#endif
#ifdef ROFL_EMUL
DEV void cp_async16(void *dst, const void *src) { *(uint4 *)dst = *(const uint4 *)src; }
DEV void cp_async_commit() {}
template <int N> DEV void cp_async_wait() {}
#else
DEV void cp_async16(void *dst, const void *src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory"); }
DEV void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> DEV void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
#endif
struct rtm_stage { uint4 rec[RTM_STAGES][6][128]; uint4 scal[2][2][128]; };
struct rtm_cursor { uint32_t xk[9]; const niels_st *row0; uint32_t term, w, flags; };      // producer side of one thread's record stream
// acc +/- the record staged in `slot` of this thread
DEV void rtm_consume(ge_p3 &acc, const rtm_stage &sm, uint32_t slot, int tid, bool neg) {
    const uint4 *q = &sm.rec[slot][0][tid]; const uint32_t op = neg ? 256u : 0u, om = neg ? 0u : 256u;          // -Q: y+x and y-x swap by address
    uint4 v0 = q[op], v1 = q[op + 128], v2 = q[om], v3 = q[om + 128], v4 = q[512], v5 = q[640];
    ge_niels m;
    m.yplusx.v[0] = v0.x; m.yplusx.v[1] = v0.y; m.yplusx.v[2] = v0.z; m.yplusx.v[3] = v0.w; m.yplusx.v[4] = v1.x; m.yplusx.v[5] = v1.y; m.yplusx.v[6] = v1.z; m.yplusx.v[7] = v1.w;
    m.yminusx.v[0] = v2.x; m.yminusx.v[1] = v2.y; m.yminusx.v[2] = v2.z; m.yminusx.v[3] = v2.w; m.yminusx.v[4] = v3.x; m.yminusx.v[5] = v3.y; m.yminusx.v[6] = v3.z; m.yminusx.v[7] = v3.w;
    m.xy2d.v[0] = v4.x; m.xy2d.v[1] = v4.y; m.xy2d.v[2] = v4.z; m.xy2d.v[3] = v4.w; m.xy2d.v[4] = v5.x; m.xy2d.v[5] = v5.y; m.xy2d.v[6] = v5.z; m.xy2d.v[7] = v5.w;
    ge_p1p1 t; ge_madd_p1p1(t, acc, m);
    fe z = t.Z; fe_cmov(t.Z, t.T, neg); fe_cmov(t.T, z, neg);                       // ... and the sign of C swaps G and F
    ge_p1p1_to_p3(acc, t);
}
#ifdef KG_MSM
DEV void rtm_produce(rtm_cursor &p, rtm_stage &sm, const rt_msm_args &a, const sc_st *scal, uint32_t t0, uint32_t stride, uint32_t nterm, uint32_t g, uint32_t total, uint32_t slot, int tid) {
    if (g < total) {
        if (p.w == (uint32_t)a.rt.nw) {                                                     // next term: its scalar was staged one term ago
            sc x; const uint32_t t = t0 + p.term * stride;
            if (p.term == 0) ld_sc(x, scal + t);
            else { uint4 lo = sm.scal[p.term & 1][0][tid], hi = sm.scal[p.term & 1][1][tid]; x.v[0] = lo.x; x.v[1] = lo.y; x.v[2] = lo.z; x.v[3] = lo.w; x.v[4] = hi.x; x.v[5] = hi.y; x.v[6] = hi.z; x.v[7] = hi.w; }
            const bool isG = t < a.nG; const uint32_t q = isG ? t : t - a.nG; uint32_t j = q;
            if (a.mode) { bool hi = (a.mode == 1) == isG; j = (q / a.np) * 2 * a.np + (hi ? a.np : 0) + q % a.np; }
            p.row0 = (isG ? a.rt.G : a.rt.H) + (size_t)j * rt_row_entries(a.rt);
            msm_recode(p.xk, x, a.rt.K);
            p.term++; p.w = 0;
            if (p.term < nterm) { const uint4 *nx = (const uint4 *)(scal + t0 + p.term * stride); cp_async16(&sm.scal[p.term & 1][0][tid], nx); cp_async16(&sm.scal[p.term & 1][1][tid], nx + 1); }
        }
        const int dw = msm_digit(p.xk, (int)p.w, a.rt.c);
        if (dw != 0) {
            const uint4 *src = (const uint4 *)(p.row0 + (size_t)p.w * a.rt.B + (dw > 0 ? dw : -dw) - 1);
            for (int i = 0; i < 6; i++) cp_async16(&sm.rec[slot][i][tid], src + i);
        }
        p.flags = (p.flags & ~(3u << (2 * slot))) | ((uint32_t)(dw != 0) | ((uint32_t)(dw < 0) << 1)) << (2 * slot);
        p.w++;
    }
    cp_async_commit();
}
KERNEL void LB(128, RTM_BLOCKS) k_rt_msm(rt_msm_args a) {
    __shared__ rtm_stage sm;
    const int tid = threadIdx.x; const uint32_t msm = blockIdx.y;
    const sc_st *scal = a.scalars + (size_t)msm * a.scalar_stride;
    const uint32_t stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + tid;
    const uint32_t nterm = t0 < a.T ? (a.T - t0 + stride - 1) / stride : 0, total = nterm * (uint32_t)a.rt.nw;
    rtm_cursor p; p.term = 0; p.w = (uint32_t)a.rt.nw; p.flags = 0; p.row0 = nullptr;
    ge_p3 acc; ge_p3_0(acc);
    uint32_t pslot = 0, cslot = 0;
    for (uint32_t g = 0; g < RTM_STAGES - 1; g++) { rtm_produce(p, sm, a, scal, t0, stride, nterm, g, total, pslot, tid); pslot = pslot + 1 == RTM_STAGES ? 0 : pslot + 1; }
    for (uint32_t k = 0; k < total; k++) {
        rtm_produce(p, sm, a, scal, t0, stride, nterm, k + RTM_STAGES - 1, total, pslot, tid); pslot = pslot + 1 == RTM_STAGES ? 0 : pslot + 1;
        cp_async_wait<RTM_STAGES - 1>();
        const uint32_t f = (p.flags >> (2 * cslot)) & 3u;
        if (f & 1u) rtm_consume(acc, sm, cslot, tid, (f & 2u) != 0);
        cslot = cslot + 1 == RTM_STAGES ? 0 : cslot + 1;
    }
    cp_async_wait<0>();
    __syncthreads();
    block_sum_p3(acc, (p3_st *)&sm, tid, blockDim.x);
    if (tid == 0) st_p3(a.partial + (size_t)msm * gridDim.x + blockIdx.x, acc);
}
KLAUNCH(k_rt_msm, true, (rt_msm_args a), (a))
#endif
void launch_k_rt_shifts(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *P, const niels_st *gens, uint32_t count, int c, int nw);
void launch_k_rt_rows(dim3 g_, dim3 b_, cudaStream_t s_, niels_st *RT, const p3_st *P, size_t rows, int B);
void launch_k_rt_msm(dim3 g_, dim3 b_, cudaStream_t s_, rt_msm_args a);

// unfolded IPP round k (np = N >> (k+1), 2^k blocks of 2np original generators each; coefficient tables cG/cH[c*cstride + t]):
//   L: G-term (t,i) -> a^[i] cG[t] on G[t*2np + np + i];  H-term -> b^[np+i] y^-i cH[t] on H[t*2np + i]
//   R: G-term -> a^[np+i] cG[t] on G[t*2np + i];           H-term -> b^[i] y^-(np+i) cH[t] on H[t*2np + np + i]
//   msmL / msmR: [c][N] scalars laid out for k_rt_msm modes 1 / 2 (N/2 G-terms then N/2 H-terms, term q = t*np + i)
#ifdef KG_SCALAR
KERNEL void LB(256, 1) k_ipp_scalars_unf(const sc_st *a, const sc_st *b, const sc_st *yinv, const sc_st *cG, const sc_st *cH, uint32_t cstride,
                                         sc_st *msmL, sc_st *msmR, sc_st *partial, size_t N, uint32_t np, uint32_t live) {
    // N = stride of a / b / yinv per chunk; live = number of base points the round is expressed over (N for the original generators,
    // F for a frozen level): msmL / msmR are [c][live]
    __shared__ sc_st buf[256];
    int c = blockIdx.y, tid = threadIdx.x;
    const sc_st *ac = a + (size_t)c * N, *bc = b + (size_t)c * N, *yc = yinv + (size_t)c * N;
    sc_st *L = msmL + (size_t)c * live, *R = msmR + (size_t)c * live;
    const uint32_t half = live / 2;
    sc cL, cR; sc_0(cL); sc_0(cR);
    for (uint32_t q = blockIdx.x * blockDim.x + tid; q < half; q += gridDim.x * blockDim.x) {
        uint32_t t = q / np, i = q % np;
        sc alo, ahi, blo, bhi, ylo, yhi, g, h, x;
        ld_sc(alo, ac + i); ld_sc(ahi, ac + np + i); ld_sc(blo, bc + i); ld_sc(bhi, bc + np + i); ld_sc(ylo, yc + i); ld_sc(yhi, yc + np + i);
        ld_sc(g, cG + (size_t)c * cstride + t); ld_sc(h, cH + (size_t)c * cstride + t);
        if (t == 0) { sc_mul(x, alo, bhi); sc_add(cL, cL, x); sc_mul(x, ahi, blo); sc_add(cR, cR, x); }
        sc_mul(x, alo, g); st_sc(L + q, x);
        sc_mul(x, bhi, ylo); sc_mul(x, x, h); st_sc(L + half + q, x);
        sc_mul(x, ahi, g); st_sc(R + q, x);
        sc_mul(x, blo, yhi); sc_mul(x, x, h); st_sc(R + half + q, x);
    }
    block_sum_sc(cL, buf, tid, blockDim.x); block_sum_sc(cR, buf, tid, blockDim.x);
    if (tid == 0) { sc_st *o = partial + ((size_t)c * gridDim.x + blockIdx.x) * 2; st_sc(o, cL); st_sc(o + 1, cR); }
}
KLAUNCH(k_ipp_scalars_unf, true, (const sc_st *a, const sc_st *b, const sc_st *yinv, const sc_st *cG, const sc_st *cH, uint32_t cstride, sc_st *msmL, sc_st *msmR, sc_st *partial, size_t N, uint32_t np, uint32_t live),
        (a, b, yinv, cG, cH, cstride, msmL, msmR, partial, N, np, live))
#endif
// catch-up fold after r unfolded rounds: out[c][i] = sum_{t < nblk} coef[t] * Gen[t*nr + i], i < nr = N >> r, through the RT tables.
//   digits[((c*2 + which)*nblk + t)*32 + w] = radix-256 signed digits of the coefficient (host-computed, uniform per chunk)
//   grid (blocks, C, 2): z = 0 -> G, 1 -> H
struct catchup_args { rt_tables rt; p3_st *Gf, *Hf; const int16_t *digits; uint32_t nr, nblk, stride; };      // digits[((c*2+which)*nblk + t)*RT_MAXW + w]
#ifdef KG_FOLD
KERNEL void LB(128, RTM_BLOCKS) k_rt_catchup(catchup_args a) {
    __shared__ rtm_stage sm;                                    // record staging as in k_rt_msm; the scalar slots hold the digits here
    int16_t *dg = (int16_t *)sm.scal;                           // 64 * RT_MAXW digits = 4 KB
    int c = blockIdx.y, which = blockIdx.z, tid = threadIdx.x;
    for (uint32_t t = tid; t < a.nblk * RT_MAXW; t += blockDim.x) dg[t] = a.digits[((size_t)c * 2 + which) * a.nblk * RT_MAXW + t];
    __syncthreads();
    uint32_t i = blockIdx.x * blockDim.x + tid;
    if (i >= a.nr) return;
    const niels_st *RT = which ? a.rt.H : a.rt.G;
    const size_t rowsz = rt_row_entries(a.rt);
    const uint32_t nw = (uint32_t)a.rt.nw, total = a.nblk * nw;
    ge_p3 acc; ge_p3_0(acc);
    uint32_t pt = 0, pw = 0, flags = 0, pslot = 0, cslot = 0;
    auto produce = [&](uint32_t g) {
        if (g < total) {
            const int d = dg[pt * RT_MAXW + pw];
            if (d != 0) {
                const uint4 *src = (const uint4 *)(RT + ((size_t)pt * a.nr + i) * rowsz + (size_t)pw * a.rt.B + (d > 0 ? d : -d) - 1);
                for (int k = 0; k < 6; k++) cp_async16(&sm.rec[pslot][k][tid], src + k);
            }
            flags = (flags & ~(3u << (2 * pslot))) | ((uint32_t)(d != 0) | ((uint32_t)(d < 0) << 1)) << (2 * pslot);
            if (++pw == nw) { pw = 0; pt++; }
        }
        cp_async_commit();
        pslot = pslot + 1 == RTM_STAGES ? 0 : pslot + 1;
    };
    for (uint32_t g = 0; g < RTM_STAGES - 1; g++) produce(g);
    for (uint32_t k = 0; k < total; k++) {
        produce(k + RTM_STAGES - 1);
        cp_async_wait<RTM_STAGES - 1>();
        const uint32_t f = (flags >> (2 * cslot)) & 3u;
        if (f & 1u) rtm_consume(acc, sm, cslot, tid, (f & 2u) != 0);
        cslot = cslot + 1 == RTM_STAGES ? 0 : cslot + 1;
    }
    st_p3((which ? a.Hf : a.Gf) + (size_t)c * a.stride + i, acc);
}
KLAUNCH(k_rt_catchup, true, (catchup_args a), (a))
#endif
void launch_k_ipp_scalars_unf(dim3 g_, dim3 b_, cudaStream_t s_, const sc_st *a, const sc_st *b, const sc_st *yinv, const sc_st *cG, const sc_st *cH, uint32_t cstride, sc_st *msmL, sc_st *msmR, sc_st *partial, size_t N, uint32_t np, uint32_t live);
void launch_k_rt_catchup(dim3 g_, dim3 b_, cudaStream_t s_, catchup_args a);


// catch-up fold WITHOUT generator tables (chunks too large for them): out[c][i] = sum_{t < nblk} coef[t] * Gen[t*nr + i], i < nr, as ONE joint double-and-add
// per output: the coefficients are the same for every i (and coef[0] = 1), so all lanes follow the same width-3 NAF digit pattern;
// per base only P and 3P are kept.  252 doublings + ~63 additions per base instead of a 253-step fold ladder per base and level.
//   nafs[((c*2 + which)*nblk + t)*256 + bit] (k_ts_round, emit 4).  grid (blocks, C, 2): z = 0 -> G, 1 -> H
#define CATCHUP_MAX_BASES 16
struct catchup_naf_args { const niels_st *G, *H; p3_st *Gf, *Hf; const int8_t *nafs; uint32_t nr, nblk, stride; };
#ifdef KG_FOLD
KERNEL void LB(128, 2) k_catchup_naf(catchup_naf_args a) {
    __shared__ int8_t naf[CATCHUP_MAX_BASES][256];
    const int c = blockIdx.y, which = blockIdx.z, tid = threadIdx.x;
    for (uint32_t t = tid; t < a.nblk * 256; t += blockDim.x) naf[t >> 8][t & 255] = a.nafs[(((size_t)c * 2 + which) * a.nblk) * 256 + t];
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + tid;
    if (i >= a.nr) return;
    const niels_st *src = which ? a.H : a.G;
    ge_cached p1[CATCHUP_MAX_BASES], p3[CATCHUP_MAX_BASES];
    for (uint32_t t = 0; t < a.nblk; t++) {
        ge_niels n; ld_niels(n, src + (size_t)t * a.nr + i);
        ge_p3 P, P2, P3; ge_niels_to_p3(P, n); ge_p3_dbl(P2, P); ge_p3_to_cached(p1[t], P); ge_add_cached(P3, P2, p1[t]); ge_p3_to_cached(p3[t], P3);
    }
    int top = 255;
    for (; top > 0; top--) { bool any = false; for (uint32_t t = 0; t < a.nblk; t++) any = any || naf[t][top] != 0; if (any) break; }
    ge_p3 r; ge_p3_0(r);
    for (int bit = top; bit >= 0; bit--) {
        ge_p3_dbl(r, r);
        for (uint32_t t = 0; t < a.nblk; t++) {
            const int d = naf[t][bit];
            if (d != 0) ge_add_cached_signed(r, r, (d == 1 || d == -1) ? p1[t] : p3[t], d < 0);
        }
    }
    st_p3((which ? a.Hf : a.Gf) + (size_t)c * a.stride + i, r);
}
KLAUNCH(k_catchup_naf, true, (catchup_naf_args a), (a))
#endif
void launch_k_catchup_naf(dim3 g_, dim3 b_, cudaStream_t s_, catchup_naf_args a);

// ===================================================================================================================
// K6c: FROZEN LEVEL.  After the catch-up the folded generators of a chunk (F = N/16 of G" and of H") stay frozen for the
// middle rounds: like the first rounds over the original generators, every later L / R is a sum over ALL frozen points with
// coefficient tables, but the points are new per proof, so their tables are small Straus tables built on the fly:
//   T[p][q][k] = (k+1) * 2^(32 q) * P_p,  q < 8 octants, k < 8  (signed radix-16 digits; 64 cached records = 8 KB per point)
//   s * P_p = sum_{pos<8} 16^pos * sum_{q<8} e[8q+pos] * 2^(32q) P_p       (e = signed radix-16 digits of s)
// so a round is 64 additions per point and its doubling chain has only 28 doublings (k_finalize with c = 4, nw = 8) instead
// of a 253-step fold ladder per point plus a 252-doubling chain per output.
// ===================================================================================================================
#define FRZ_Q 8
#define FRZ_E 8
#define FRZ_MAX_F 1024
struct frz_reduce_args { const p3_st *T; const sc_st *msmL, *msmR; p3_st *V; uint32_t F, np, C; };
struct frz_exit_args { const p3_st *T; const int8_t *digs; p3_st *Gf, *Hf, *V; uint32_t F, Fo, nblk, stride; };
#ifdef KG_FOLD
// bases[(c*2F + p)*8 + q] = 2^(32 q) * P_p ; P = G"[c][0..F) then H"[c][0..F).  grid (blocks, C)
// Q bases per point, `step` doublings apart: (FRZ_Q, 32) for the frozen level, (TAIL_Q, 4) = one base per radix-16 digit for the tail
KERNEL void LB(128, 4) k_frz_bases(p3_st *bases, const p3_st *Gf, const p3_st *Hf, uint32_t F, uint32_t stride, uint32_t Q, uint32_t step) {
    const int c = blockIdx.y; const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= 2 * F) return;
    ge_p3 P; ld_p3(P, (p < F ? Gf + (size_t)c * stride + p : Hf + (size_t)c * stride + (p - F)));
    p3_st *o = bases + ((size_t)c * 2 * F + p) * Q;
    for (uint32_t q = 0; q < Q; q++) {
        st_p3(o + q, P);
        if (q + 1 < Q) for (uint32_t k = 0; k < step; k++) ge_p3_dbl(P, P);
    }
}
KLAUNCH(k_frz_bases, false, (p3_st *bases, const p3_st *Gf, const p3_st *Hf, uint32_t F, uint32_t stride, uint32_t Q, uint32_t step), (bases, Gf, Hf, F, stride, Q, step))
#ifndef ROFL_EMUL
// The same bases with FOUR lanes per point (device only): lane k of a quad owns coordinate k of (X : Y : Z : T).  A doubling is 4 independent
// squarings followed by 4 independent multiplications (ge_dbl_p1p1 / ge_p1p1_to_p3), so the quad does it in the time of one squaring + one
// multiplication + 48 shuffles -- one lane alone needs 3500 cycles per doubling (tools/microbench_lat.cu) and the tail's 252-doubling chain per
// point is pure latency at the exposed end of a proof.  Bit-identical coordinates to k_frz_bases.
KERNEL void LB(128, 4) k_frz_bases4(p3_st *bases, const p3_st *Gf, const p3_st *Hf, uint32_t F, uint32_t stride, uint32_t Q, uint32_t step) {
    const int c = blockIdx.y; const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, k = t & 3;
    const bool live = (t >> 2) < 2 * F; const uint32_t p = live ? (t >> 2) : 2 * F - 1;
    const int qb = (int)(threadIdx.x & 31u) & ~3;
    const p3_st *src = p < F ? Gf + (size_t)c * stride + p : Hf + (size_t)c * stride + (p - F);
    fe mine; { const uint32_t *w = (const uint32_t *)src + 8 * k; for (int i = 0; i < 8; i++) mine.v[i] = w[i]; }
    p3_st *o = bases + ((size_t)c * 2 * F + p) * Q;
    auto bc = [&](const fe &v, int from) { fe r; for (int i = 0; i < 8; i++) r.v[i] = __shfl_sync(0xffffffffu, v.v[i], qb + from); return r; };
    for (uint32_t q = 0; q < Q; q++) {
        if (live) { uint32_t *w = (uint32_t *)(o + q) + 8 * k; for (int i = 0; i < 8; i++) w[i] = mine.v[i]; }
        if (q + 1 < Q) for (uint32_t it = 0; it < step; it++) {
            const fe X = bc(mine, 0), Y = bc(mine, 1);
            fe in = mine; if (k == 3) fe_add(in, X, Y);
            fe sq; fe_sq(sq, in);                                   // XX | YY | ZZ | (X+Y)^2
            const fe xx = bc(sq, 0), yy = bc(sq, 1), zz = bc(sq, 2), xy = bc(sq, 3);
            fe Yp, Zp, Xp, Tp, tt;
            fe_add(Yp, yy, xx); fe_sub(Zp, yy, xx); fe_sub4(Xp, xy, Yp); fe_carry(Xp, Xp);
            fe_add(tt, zz, zz); fe_add(tt, tt, xx); fe_sub(Tp, tt, yy);
            const fe &A = (k == 0 || k == 2) ? Tp : (k == 1 ? Yp : Xp), &B = k == 0 ? Xp : (k == 3 ? Yp : Zp);
            fe_mul(mine, A, B);                                     // X3 = T'X' | Y3 = Y'Z' | Z3 = T'Z' | T3 = X'Y'
        }
    }
}
KLAUNCH(k_frz_bases4, false, (p3_st *bases, const p3_st *Gf, const p3_st *Hf, uint32_t F, uint32_t stride, uint32_t Q, uint32_t step), (bases, Gf, Hf, F, stride, Q, step))
#endif
// T[idx*8 + k] = (k+1) * bases[idx]   (cached form), one thread per (point, octant)
KERNEL void LB(128, 4) k_frz_tables(p3_st *T, const p3_st *bases, size_t count) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= count) return;
    ge_p3 base, cur; ld_p3(base, bases + idx); cur = base;
    ge_cached cb; ge_p3_to_cached(cb, base);
    st_cached(T + idx * FRZ_E, cb);
    for (int k = 1; k < FRZ_E; k++) { ge_add_cached(cur, cur, cb); ge_cached ck; ge_p3_to_cached(ck, cur); st_cached(T + idx * FRZ_E + k, ck); }
}
KLAUNCH(k_frz_tables, false, (p3_st *T, const p3_st *bases, size_t count), (T, bases, count))
// one round: V[(lr*C + c)*8 + pos] = sum over the F terms of side lr (F/2 G-terms then F/2 H-terms, scalars as k_ipp_scalars_unf lays them
// out) and the 8 octants of the table entry selected by digit e[8q + pos].  grid (8, 2C), 128 threads
KERNEL void LB(128, 4) k_frz_reduce(frz_reduce_args a) {
    __shared__ p3_st buf[128];
    const int pos = blockIdx.x, tid = threadIdx.x; const uint32_t lr = blockIdx.y / a.C, c = blockIdx.y % a.C;
    const sc_st *scal = (lr ? a.msmR : a.msmL) + (size_t)c * a.F;
    const uint32_t half = a.F / 2;
    ge_p3 acc; ge_p3_0(acc);
    for (uint32_t k = tid; k < a.F; k += 128) {
        sc x; ld_sc(x, scal + k);
        if (sc_iszero(x)) continue;
        const bool isG = k < half; const uint32_t qk = isG ? k : k - half;
        const bool hi = (lr == 0) == isG;
        const uint32_t j = (qk / a.np) * 2 * a.np + (hi ? a.np : 0) + qk % a.np, p = isG ? j : a.F + j;
        int8_t e[64]; sc_radix16(e, x);
        const p3_st *row = a.T + ((size_t)c * 2 * a.F + p) * FRZ_Q * FRZ_E;
        for (int q = 0; q < FRZ_Q; q++) {
            const int d = e[8 * q + pos];
            if (d != 0) acc_add_cached(acc, row + q * FRZ_E + (d > 0 ? d : -d) - 1, d < 0);
        }
    }
    block_sum_p3(acc, buf, tid, 128);
    if (tid == 0) st_p3(a.V + ((size_t)lr * a.C + c) * 8 + pos, acc);
}
KLAUNCH(k_frz_reduce, true, (frz_reduce_args a), (a))
// leave the level: out[c][i] = sum_{t < nblk} coef[t] * P[t*Fo + i], i < Fo (the folded generators the next stage starts from), through the
// tables.  digs[((c*2 + which)*nblk + t)*64 + ..] = signed radix-16 digits of the coefficient (host).  grid (Fo, C, 2), 128 threads:
// thread (pos = tid % 8, g = tid / 8) sums the (t, q) pairs g, g+16, .. of its digit position; 16-way tree per position; thread 0 runs the
// 28-doubling chain.
KERNEL void LB(128, 4) k_frz_exit(frz_exit_args a) {
    __shared__ p3_st buf[128];
    const uint32_t i = blockIdx.x, c = blockIdx.y, which = blockIdx.z; const int tid = threadIdx.x, pos = tid & 7, g = tid >> 3;
    const int8_t *dg = a.digs + ((size_t)c * 2 + which) * a.nblk * 64;
    ge_p3 acc; ge_p3_0(acc);
    for (uint32_t pr = g; pr < a.nblk * FRZ_Q; pr += 16) {
        const uint32_t t = pr / FRZ_Q, q = pr % FRZ_Q;
        const int d = dg[t * 64 + 8 * q + pos];
        const uint32_t p = which * a.F + t * a.Fo + i;
        if (d != 0) acc_add_cached(acc, a.T + (((size_t)c * 2 * a.F + p) * FRZ_Q + q) * FRZ_E + (d > 0 ? d : -d) - 1, d < 0);
    }
    st_p3(buf + tid, acc);
    __syncthreads();
    for (int s2 = 64; s2 >= 8; s2 >>= 1) {
        if (tid < s2) { ge_p3 x, y; ld_p3(x, buf + tid); ld_p3(y, buf + tid + s2); ge_add(x, x, y); st_p3(buf + tid, x); }
        __syncthreads();
    }
    if (tid < 8) { ge_p3 x; ld_p3(x, buf + tid); st_p3(a.V + ((((size_t)c * 2 + which) * a.Fo + i) * 8 + tid), x); }      // the 8 position sums; chains: k_frz_exit_chain
}
KLAUNCH(k_frz_exit, true, (frz_exit_args a), (a))
// out = sum_pos 16^pos V[pos]: one thread per output so that all 28-doubling chains run side by side (inside k_frz_exit they would keep one
// lane of every block busy for 2/3 of its life)
KERNEL void LB(128, 1) k_frz_exit_chain(frz_exit_args a, uint32_t C) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * 2 * a.Fo) return;
    const uint32_t i = idx % a.Fo, which = (idx / a.Fo) & 1, c = idx / (2 * a.Fo);
    const p3_st *v = a.V + (size_t)idx * 8;
    ge_p3 h; ld_p3(h, v + 7);
    for (int w = 6; w >= 0; w--) { for (int k = 0; k < 4; k++) ge_p3_dbl(h, h); acc_add_p3(h, v + w, false); }
    st_p3((which ? a.Hf : a.Gf) + (size_t)c * a.stride + i, h);
}
KLAUNCH(k_frz_exit_chain, false, (frz_exit_args a, uint32_t C), (a, C))
#endif
void launch_k_frz_bases(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *bases, const p3_st *Gf, const p3_st *Hf, uint32_t F, uint32_t stride, uint32_t Q, uint32_t step);
#ifndef ROFL_EMUL
void launch_k_frz_bases4(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *bases, const p3_st *Gf, const p3_st *Hf, uint32_t F, uint32_t stride, uint32_t Q, uint32_t step);
#endif
void launch_k_frz_tables(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *T, const p3_st *bases, size_t count);
void launch_k_frz_reduce(dim3 g_, dim3 b_, cudaStream_t s_, frz_reduce_args a);
void launch_k_frz_exit(dim3 g_, dim3 b_, cudaStream_t s_, frz_exit_args a);
void launch_k_frz_exit_chain(dim3 g_, dim3 b_, cudaStream_t s_, frz_exit_args a, uint32_t C);

// ===================================================================================================================
// K6b: the last rounds of the inner-product argument (half-size np <= TAIL_MAX_F/2) in ONE launch, one thread-block cluster per chunk,
// nothing leaves the SMs between rounds: the Merlin transcript, the challenge inversion and the scalar folds run on the device.
// The generators are frozen at their F = 2 np0 entry values; their tables T[p][pos][k] = (k+1) 16^pos P_p -- one position per radix-16
// digit, built by k_frz_bases / k_frz_tables right before the launch -- make every round a plain sum of table entries:
//   128 threads recode the scalars of the 2F points into signed radix-16 digits (shared memory);
//   512 threads (side, lane) add up their 16 table entries each (dealt over the blocks of the cluster), shuffle tree per warp,
//   the leader block sums the 8 warp results of a side (shuffle tree over 8 lanes), adds c_L w B / c_R w B (computed meanwhile by a
//   spare warp, one radix-256 window per lane) and compresses; warp 0 appends L, R to the transcript and draws u (wtranscript.cuh);
//   lane 0 inverts it (division steps) and publishes u^2, u^-2, u^-2 y^-np; every block folds its copy of a^, b^ and the coefficients.
//   out[c]: rounds x (L | R) compressed, then a | b (the proof's last two scalars)
// Per round on B200 (ROFL_TAIL_DBG, cycles at 1.965 GHz): table sums 330 k, sums + compress 275 k (the compression alone 186 k), transcript +
// inversion 160 k.  History: octant tables with a 28-doubling Horner chain per round 400 k; one lane walking the 32 windows of c w B 370 k.
// ===================================================================================================================
#define TAIL_MAX_F 64
#define TAIL_Q 64                            // table positions per point in the tail: one per radix-16 digit, so that a round needs NO doubling chain
#define TAIL_THREADS (512 + 32)
struct tail_args {
    const p3_st *T;                          // [C][2F][TAIL_Q][FRZ_E] tables (k+1) 16^pos P of G"[0..F) then H"[0..F)
    const sc_st *a, *b, *yinv; size_t N;     // [C][N] lazy-factor vectors a^, b^ and y^-i (first F entries live)
    const transcript *ts;                    // [C] transcript states after the previous challenge
    const sc_st *w, *uprod, *uinvprod;       // [C] w; products of the earlier u_k and u_k^-1
    const niels_st *tabB;
    p3_st *scratch;                          // [C][512] partial sums
    uint8_t *out; uint32_t out_stride;
    uint32_t F;
    uint32_t ncta;                           // blocks (= cluster size) per chunk: 1, 2, 4 or 8
    sc_st *gfac;                             // [C][3] the round's fold factors, leader -> the other blocks of the cluster
    long long *dbg;                          // diagnostic (ROFL_TAIL_DBG): clock64 of block 0 at the 8 phase boundaries of every round
};
#ifdef KG_FOLD
#if defined(__CUDA_ARCH__)
#define TAIL_STAMP(k) do { if (a.dbg && blockIdx.x == 0 && tid == 0) a.dbg[8 * round + (k)] = clock64(); } while (0)
#else
#define TAIL_STAMP(k) do { } while (0)
#endif
#if defined(__CUDA_ARCH__)
#define TAIL_CSYNC() do { if (ncta > 1) asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory"); else __syncthreads(); } while (0)
#else
#define TAIL_CSYNC() __syncthreads()
#endif
KERNEL void LB(TAIL_THREADS, 1) k_ipp_tail(tail_args a) {
    __shared__ sc_st sa[TAIL_MAX_F], sb[TAIL_MAX_F], sy[TAIL_MAX_F], scg[TAIL_MAX_F], sch[TAIL_MAX_F], red[64], sfac[3];
    __shared__ p3_st ptB[2];
    __shared__ int8_t dig[2 * TAIL_MAX_F][64];
    __shared__ uint8_t side_of[2 * TAIL_MAX_F];                         // 0: the point feeds L this round, 1: R
    // a.ncta blocks (one thread-block cluster) per chunk: the table sums of a round are dealt to all of them, block 0 (the leader) runs the
    // serial part -- chains, compression, transcript -- and publishes the round's three fold factors; every block keeps its own copy of the
    // scalar vectors and folds it.  Two cluster barriers per round order the exchanges through global memory.
    const uint32_t ncta = a.ncta, rank = blockIdx.x % ncta;
    const int c = blockIdx.x / ncta, tid = threadIdx.x;
    const bool leader = rank == 0;
    const uint32_t F = a.F, NP = 2 * F;
    const int tB = 512;                                                // lanes 0 / 1 of the last warp: the c_L w B and c_R w B terms
    p3_st *pts = a.scratch + (size_t)c * 512;                          // [16 warps][32]: slot 32 w + r = warp w's sum of block r
    sc_st *gfac = a.gfac + 3 * (size_t)c;
    const p3_st *T = a.T + (size_t)c * NP * TAIL_Q * FRZ_E;
    for (uint32_t i = tid; i < F; i += TAIL_THREADS) {
        sa[i] = a.a[(size_t)c * a.N + i]; sb[i] = a.b[(size_t)c * a.N + i]; sy[i] = a.yinv[(size_t)c * a.N + i];
    }
    if (tid == 0) { sc one; sc_from_u64(one, 1); st_sc(scg, one); st_sc(sch, one); }
    sc up, uip, wc;
#ifdef ROFL_EMUL
    transcript t;                                                      // (the emulation's warp barrier is the block barrier: one lane runs the transcript there)
    if (tid == 0) t = a.ts[c];
#else
    __shared__ strobe_sh hts;                                          // the transcript is run by warp 0 (wtranscript.cuh)
    wts wt = {0, 0, 0};
    if (leader && tid < TS_THREADS) wt_load(hts, wt, tid, a.ts[c]);
#endif
    if (leader && tid == 0) { ld_sc(up, a.uprod + c); ld_sc(uip, a.uinvprod + c); }
    if (tid >= tB) ld_sc(wc, a.w + c);
    uint8_t *out = a.out + (size_t)c * a.out_stride;
    // accumulation role: side (L / R), digit position, group
    const uint32_t a_side = (uint32_t)tid >> 8, a_lin = (uint32_t)tid & 255, a_g = (uint32_t)tid & 31;
    __syncthreads();
    int round = 0;
    for (uint32_t np = F >> 1; np >= 1; np >>= 1, round++) {
        TAIL_STAMP(0);
        // c_L = <a^_lo, b^_hi>, c_R = <a^_hi, b^_lo>
        if (tid < 64) {
            sc v; sc_0(v);
            const uint32_t i = tid & 31;
            if (i < np) { sc x, y; ld_sc(x, tid < 32 ? sa + i : sa + np + i); ld_sc(y, tid < 32 ? sb + np + i : sb + i); sc_mul(v, x, y); }
            st_sc(red + tid, v);
        }
        // digits of the scalar of every frozen point (points 0..F-1 = G", F..2F-1 = H")
        if ((uint32_t)tid >= 64 && (uint32_t)tid < 64 + NP) {
            const uint32_t p = tid - 64; const bool isH = p >= F; const uint32_t j = isH ? p - F : p;
            const uint32_t tt = j / (2 * np), h = (j / np) & 1, i = j % np;
            sc s, x; bool toL;
            if (!isH) { toL = h == 1; ld_sc(s, toL ? sa + i : sa + np + i); ld_sc(x, scg + tt); sc_mul(s, s, x); }
            else { toL = h == 0; ld_sc(s, toL ? sb + np + i : sb + i); ld_sc(x, toL ? sy + i : sy + np + i); sc_mul(s, s, x); ld_sc(x, sch + tt); sc_mul(s, s, x); }
            int8_t e[64]; sc_radix16(e, s);
            for (int k = 0; k < 64; k++) dig[p][k] = e[k];
            side_of[p] = toL ? 0 : 1;
        }
        __syncthreads();
        TAIL_STAMP(1);
        for (int s2 = 16; s2 > 0; s2 >>= 1) {
            if (tid < 64 && (tid & 31) < s2) { sc x, y; ld_sc(x, red + tid); ld_sc(y, red + tid + s2); sc_add(x, x, y); st_sc(red + tid, x); }
            __syncthreads();
        }
        TAIL_STAMP(2);
        ge_p3 acc; ge_p3_0(acc);
#ifndef ROFL_EMUL
        long long w_t0 = 0, w_t1 = 0; if (a.dbg) w_t0 = clock64();
#endif
        if (tid < 512) {
            // pairs (point, octant) of my side, strided over the 32 groups of my (side, position)
            // the F points of my side (G" blocks with h = 1 and H" blocks with h = 0 feed L, the others R) x 8 octants, dealt to the 32 lanes of
            // my (side, position): 16 pairs each in every round (striding over ALL points and skipping the other side's left half of the lanes
            // idle once np < 4: the last two rounds took twice as long)
            for (uint32_t pr = rank * 256 + a_lin; pr < F * TAIL_Q; pr += 256 * ncta) {
                const uint32_t idx = pr / TAIL_Q, pos = pr % TAIL_Q;
                const bool isH = idx >= F / 2; const uint32_t tt = isH ? idx - F / 2 : idx;
                const uint32_t hsel = isH ? a_side : 1 - a_side;
                const uint32_t j = ((tt / np) * 2 + hsel) * np + tt % np, p = isH ? F + j : j;
                const int d = dig[p][pos];
                if (d != 0) acc_add_cached(acc, T + ((size_t)p * TAIL_Q + pos) * FRZ_E + (d > 0 ? d : -d) - 1, d < 0);
            }
#ifdef ROFL_EMUL
            st_p3(pts + tid, acc);
#else
            if (a.dbg) w_t1 = clock64();
            // 32-way sum of my (side, position) = my warp: shuffle tree, no memory round trips and no block barriers
            for (int s2 = 16; s2 > 0; s2 >>= 1) {
                ge_p3 y;
                for (int k = 0; k < 8; k++) {
                    y.X.v[k] = __shfl_down_sync(0xffffffffu, acc.X.v[k], s2); y.Y.v[k] = __shfl_down_sync(0xffffffffu, acc.Y.v[k], s2);
                    y.Z.v[k] = __shfl_down_sync(0xffffffffu, acc.Z.v[k], s2); y.T.v[k] = __shfl_down_sync(0xffffffffu, acc.T.v[k], s2);
                }
                ge_add(acc, acc, y);
            }
            if (a_g == 0) st_p3(pts + tid + rank, acc);
            if (a.dbg && blockIdx.x == 0 && a_g == 0 && round == 2) { a.dbg[64 + 2 * (tid >> 5)] = w_t1 - w_t0; a.dbg[64 + 2 * (tid >> 5) + 1] = clock64() - w_t1; }
#endif
        } else if (leader) {
#ifdef ROFL_EMUL
          if (tid == tB || tid == tB + 1) {
            sc s; ld_sc(s, red + 32 * (tid - tB)); sc_mul(s, s, wc);
            ge_p3 r; ge_p3_0(r); fb_mul_acc(r, a.tabB, s, 32);
            st_p3(ptB + (tid - tB), r);
          }
#else
            // c_L w B and c_R w B by the whole spare warp: lane i takes radix-256 window i (one table entry), shuffle tree over the 32 windows.
            // (One lane walking the 32 windows was the longest path of this phase: 250-370 k cycles beside 16 busy warps.)
            const int ln = tid - tB;
            for (int lr = 0; lr < 2; lr++) {
                sc s; ld_sc(s, red + 32 * lr); sc_mul(s, s, wc);
                int16_t d[32]; sc_radix256(d, s);
                int di = 0;
#pragma unroll
                for (int i = 0; i < 32; i++) if (i == ln) di = d[i];
                ge_p3 r; ge_p3_0(r);
                if (di != 0) { ge_niels n; ld_niels(n, a.tabB + ln * FB_ENTRIES + (di > 0 ? di : -di) - 1); ge_madd_signed(r, r, n, di < 0); }
                for (int s2 = 16; s2 > 0; s2 >>= 1) {
                    ge_p3 y;
                    for (int k = 0; k < 8; k++) {
                        y.X.v[k] = __shfl_down_sync(0xffffffffu, r.X.v[k], s2); y.Y.v[k] = __shfl_down_sync(0xffffffffu, r.Y.v[k], s2);
                        y.Z.v[k] = __shfl_down_sync(0xffffffffu, r.Z.v[k], s2); y.T.v[k] = __shfl_down_sync(0xffffffffu, r.T.v[k], s2);
                    }
                    ge_add(r, r, y);
                }
                if (ln == 0) st_p3(ptB + lr, r);
            }
#endif
#ifndef ROFL_EMUL
            if (a.dbg && blockIdx.x == 0 && tid == tB && round == 2) a.dbg[64 + 32] = clock64() - w_t0;
#endif
        }
        TAIL_CSYNC();
        if (ncta > 1) {                                       // the leader adds up the blocks' partial sums of every (side, position)
            if (leader && tid < 512 && a_g == 0) { for (uint32_t r = 1; r < ncta; r++) { ge_p3 y; ld_p3(y, pts + tid + r); ge_add(acc, acc, y); } st_p3(pts + tid, acc); }
            __syncthreads();
        }
        TAIL_STAMP(3);
#ifdef ROFL_EMUL
        for (uint32_t s2 = 16; s2 > 0; s2 >>= 1) {          // 32-way tree inside every (side, position) group
            if (tid < 512 && a_g < s2) { ge_p3 x, y; ld_p3(x, pts + tid); ld_p3(y, pts + tid + s2); ge_add(x, x, y); st_p3(pts + tid, x); }
            __syncthreads();
        }
#endif
        TAIL_STAMP(4);
        // my side's 8 warp sums (every table entry already carries its 16^pos), + c w B, compress
#ifdef ROFL_EMUL
        if (leader && (tid == 0 || tid == 256)) {
            const int lr = tid ? 1 : 0;
            ge_p3 h; ld_p3(h, pts + tid);
            for (int w = 1; w < 8; w++) acc_add_p3(h, pts + tid + w * 32, false);
            ge_p3 y; ld_p3(y, ptB + lr); ge_add(h, h, y);
            uint8_t enc[32]; ge_compress(enc, h);
            for (int k = 0; k < 32; k++) out[64 * round + 32 * lr + k] = enc[k];
        }
#else
        if (leader && (tid < 32 || (tid >= 256 && tid < 288))) {
            const int lr = tid >= 256 ? 1 : 0, ln = tid & 31;
            ge_p3 h; if (ln < 8) ld_p3(h, pts + 256 * lr + 32 * ln); else ge_p3_0(h);
            for (int s2 = 4; s2 > 0; s2 >>= 1) {
                ge_p3 y;
                for (int k = 0; k < 8; k++) {
                    y.X.v[k] = __shfl_down_sync(0xffffffffu, h.X.v[k], s2); y.Y.v[k] = __shfl_down_sync(0xffffffffu, h.Y.v[k], s2);
                    y.Z.v[k] = __shfl_down_sync(0xffffffffu, h.Z.v[k], s2); y.T.v[k] = __shfl_down_sync(0xffffffffu, h.T.v[k], s2);
                }
                ge_add(h, h, y);
            }
            if (ln == 0) {
                ge_p3 y; ld_p3(y, ptB + lr); ge_add(h, h, y);
                uint8_t enc[32]; ge_compress(enc, h);
                for (int k = 0; k < 32; k++) out[64 * round + 32 * lr + k] = enc[k];
            }
        }
#endif
        __syncthreads();
        TAIL_STAMP(5);
#ifndef ROFL_EMUL
        sc u;
        if (leader && tid < TS_THREADS) {
            wt_load32(hts, tid, out + 64 * round); wt_append(hts, wt, tid, "L", hts.io, 32);
            wt_load32(hts, tid, out + 64 * round + 32); wt_append(hts, wt, tid, "R", hts.io, 32);
            wt_challenge_sc(hts, wt, tid, "u", u);
        }
#endif
        if (leader && tid == 0) {
            sc ui, u2, ui2, sH, ynp;
#ifdef ROFL_EMUL
            sc u;
            uint8_t lrb[64]; for (int k = 0; k < 64; k++) lrb[k] = out[64 * round + k];
            transcript_append(t, "L", lrb, 32); transcript_append(t, "R", lrb + 32, 32);
            uint8_t ub[64]; transcript_challenge(t, "u", ub, 64);
            sc_from_bytes_wide(u, ub);
#endif
            sc_invert_vartime(ui, u);
            sc_mul(u2, u, u); sc_mul(ui2, ui, ui); ld_sc(ynp, sy + np); sc_mul(sH, ui2, ynp);          // u^-2 y^-np
            sc_mul(up, up, u); sc_mul(uip, uip, ui);
            st_sc(sfac, u2); st_sc(sfac + 1, ui2); st_sc(sfac + 2, sH);
            if (ncta > 1) { st_sc(gfac, u2); st_sc(gfac + 1, ui2); st_sc(gfac + 2, sH); }
        }
        TAIL_CSYNC();
        if (ncta > 1) { if (!leader && tid < 3) sfac[tid] = gfac[tid]; __syncthreads(); }
        TAIL_STAMP(6);
        // fold a^ / b^ and extend the coefficient tables: c'[2t] = c[t], c'[2t+1] = c[t] * s
        sc cgv, chv; const uint32_t nblk = F / (2 * np);
        if ((uint32_t)tid < nblk) { ld_sc(cgv, scg + tid); ld_sc(chv, sch + tid); }
        if ((uint32_t)tid < np) {
            sc f, lo, hi;
            ld_sc(f, sfac + 1); ld_sc(lo, sa + tid); ld_sc(hi, sa + np + tid); sc_mul(hi, hi, f); sc_add(lo, lo, hi); st_sc(sa + tid, lo);
            ld_sc(f, sfac); ld_sc(lo, sb + tid); ld_sc(hi, sb + np + tid); sc_mul(hi, hi, f); sc_add(lo, lo, hi); st_sc(sb + tid, lo);
        }
        __syncthreads();
        if ((uint32_t)tid < nblk) {
            sc f, x;
            ld_sc(f, sfac); sc_mul(x, cgv, f); st_sc(scg + 2 * tid, cgv); st_sc(scg + 2 * tid + 1, x);
            ld_sc(f, sfac + 2); sc_mul(x, chv, f); st_sc(sch + 2 * tid, chv); st_sc(sch + 2 * tid + 1, x);
        }
        __syncthreads();
        TAIL_STAMP(7);
    }
    if (leader && tid == 0) {  // a = a^ prod u_k, b = b^ prod u_k^-1
        sc x, y; ld_sc(x, sa); ld_sc(y, sb); sc_mul(x, x, up); sc_mul(y, y, uip);
        uint8_t e[32]; sc_tobytes(e, x); for (int k = 0; k < 32; k++) out[64 * round + k] = e[k];
        sc_tobytes(e, y); for (int k = 0; k < 32; k++) out[64 * round + 32 + k] = e[k];
    }
}
#ifdef ROFL_EMUL
KLAUNCH(k_ipp_tail, true, (tail_args a), (a))
#else
// launched as thread-block clusters of a.ncta blocks (grid = chunks x ncta)
void launch_k_ipp_tail(dim3 g_, dim3 b_, cudaStream_t s_, tail_args a) {
    rt_host_timer t_(&rt_host_prof::launch, "k_ipp_tail"); void *tl_ = rt_timeline_begin("k_ipp_tail", s_, g_.x * g_.y * g_.z);
    cudaLaunchConfig_t cfg = {}; cfg.gridDim = g_; cfg.blockDim = b_; cfg.dynamicSmemBytes = 0; cfg.stream = s_;
    cudaLaunchAttribute at[1]; at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = a.ncta; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    rt_check(cudaLaunchKernelEx(&cfg, k_ipp_tail, a), "k_ipp_tail");
    rt_timeline_end(tl_, s_); rt_count_launch("k_ipp_tail");
}
#endif
// the shared niels generators as extended points (a tail that starts at round 0 freezes the original generators)
KERNEL void LB(128, 4) k_niels_to_p3(p3_st *Gf, p3_st *Hf, const niels_st *G, const niels_st *H, uint32_t F, uint32_t stride) {
    const int c = blockIdx.y; const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    ge_niels n; ge_p3 p;
    ld_niels(n, G + i); ge_niels_to_p3(p, n); st_p3(Gf + (size_t)c * stride + i, p);
    ld_niels(n, H + i); ge_niels_to_p3(p, n); st_p3(Hf + (size_t)c * stride + i, p);
}
KLAUNCH(k_niels_to_p3, false, (p3_st *Gf, p3_st *Hf, const niels_st *G, const niels_st *H, uint32_t F, uint32_t stride), (Gf, Hf, G, H, F, stride))
#endif
void launch_k_ipp_tail(dim3 g_, dim3 b_, cudaStream_t s_, tail_args a);
void launch_k_niels_to_p3(dim3 g_, dim3 b_, cudaStream_t s_, p3_st *Gf, p3_st *Hf, const niels_st *G, const niels_st *H, uint32_t F, uint32_t stride);

#include "ts_kernels.cuh"
