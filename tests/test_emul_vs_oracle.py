"""Product kernels + host engine + C ABI executed under the CUDA-on-CPU emulation (tests/hostsim/libemul.so, a test
tool) and compared byte for byte with the oracle.  This is the CPU-side rehearsal of tests/test_gpu_parity.py: same
calls, same seeds, tiny sizes.  CPU only."""
import ctypes as C
import importlib.util
import os
import subprocess
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def api():
    d = os.path.join(HERE, "hostsim")
    locked_make(d, "libemul.so", env={"CXX": "g++"})
    spec = importlib.util.spec_from_file_location("rofl_ffi", os.path.join(ROOT, "rofl-project-code_b200", "_ffi.py"))
    ffi = importlib.util.module_from_spec(spec); spec.loader.exec_module(ffi)
    a = ffi.Api(C.CDLL(os.path.join(d, "libemul.so")))
    yield a
    a.close()


def test_commit_and_conversion(api, oracle):
    rng = np.random.default_rng(0)
    v = np.concatenate([rng.uniform(-300, 300, 20), [0.0, -0.0, 0.25, -1.5, 600.0, -600.0]]).astype(np.float32)
    bl = oracle.rnd_scalar_vec(b"\x31" * 32, v.size)
    for nb, fr in [(16, 7), (32, 7), (8, 7)]:
        assert (api.f32_to_scalar_vec(v, nb, fr) == oracle.f32_to_scalar_vec(v, nb, fr)).all()
        L, R = api.commit(v, bl, nb, fr, want_R=True)
        assert (L == oracle.commit_f32(v, bl, nb, fr)).all()
        assert (R == oracle.elgamal_R(bl)).all()
        assert (api.commit(v, None, nb, fr) == oracle.commit_f32(v, None, nb, fr)).all()
    assert (api.rnd_scalar_vec(b"\x31" * 32, 9) == oracle.rnd_scalar_vec(b"\x31" * 32, 9)).all()
    s = oracle.f32_to_scalar_vec(v, 16, 7)
    assert (api.scalar_to_f32_vec(s, 16, 7) == oracle.scalar_to_f32_vec(s, 16, 7)).all()


@pytest.mark.parametrize("D,rngbits,P,nb", [(5, 8, 2, 16), (3, 16, 4, 16), (8, 8, 1, 16), (1, 8, 4, 16), (4, 32, 2, 32)])
def test_range_prove_bytes_and_verify(api, oracle, D, rngbits, P, nb):
    rng = np.random.default_rng(D * 100 + rngbits)
    mn, mx = oracle.clip_bounds(rngbits, nb, 7)
    v = rng.uniform(mn, mx, D).astype(np.float32)
    v[0] = mx; v[-1] = mn          # the extremes (at fp32 / range 32 the reference wraps +2^24 around; reproduced)
    bl = oracle.rnd_scalar_vec(b"\x32" * 32, D)
    seed = bytes([7] * 32)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, rngbits, P, nb, 7, seed)
    rc, p, c = api.range_prove(v, bl, rngbits, P, nb, 7, seed)
    assert rc == rc_o == 0
    assert (c == c_o).all()
    assert p.shape == p_o.shape and (p == p_o).all()
    assert api.range_verify(p, c, rngbits, seed) == 1 and oracle.range_verify(p, c, rngbits, seed) == 1
    bad = c.copy(); bad[0] = np.frombuffer(oracle.basepoint(), np.uint8)
    assert api.range_verify(p, bad, rngbits, seed) == 0
    badp = p.copy(); badp[0, 40] ^= 1
    assert api.range_verify(badp, c, rngbits, seed) == oracle.range_verify(badp, c, rngbits, seed)
    badp = p.copy(); badp[0, 128:160] = 0xff
    assert api.range_verify(badp, c, rngbits, seed) == -1


def test_range_prove_errors(api, oracle):
    z = np.zeros((8, 32), np.uint8)
    assert api.range_prove(np.full(8, 1.5, np.float32), z, 8, 4, 16, 7)[0] == 2
    assert api.range_prove(np.zeros(8, np.float32), z, 8, 3, 16, 7)[0] == -99
    assert api.range_prove(np.zeros(8, np.float32), z, 12, 4, 16, 7)[0] == -7 == oracle.range_prove(np.zeros(8, np.float32), z, 12, 4, 16, 7)[0]


def test_l2_and_square(api, oracle):
    rng = np.random.default_rng(5)
    D = 6
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(b"\x33" * 32, D); r2 = oracle.rnd_scalar_vec(b"\x34" * 32, D)
    seed = bytes([9] * 32)
    rc_o, pf_o, cm_o = oracle.l2_prove(v, r2, 32, 32, 7, seed)
    rc, pf, cm = api.l2_prove(v, r2, 32, 32, 7, seed)
    assert rc == rc_o == 0 and (pf == pf_o).all() and (cm == cm_o).all()
    assert api.l2_verify(pf, cm, 32, seed) == 1
    assert api.l2_verify(pf, oracle.basepoint(), 32, seed) == 0
    assert api.l2_prove(np.array([8.0], np.float32), np.zeros((1, 32), np.uint8), 16, 32, 7)[0] == 4
    cl = oracle.commit_f32(v, r1, 32, 7)
    rc_o, sp_o, sc_o = oracle.square_prove(v, cl, r1, r2, 32, 7, seed)
    rc, sp, sc = api.square_prove(v, cl, r1, r2, 32, 7, seed)
    assert rc == rc_o == 0 and (sp == sp_o).all() and (sc == sc_o).all()
    assert api.square_verify(sp, sc) == 1
    bad = sc.copy(); bad[1, 32:] = sc[2, 32:]
    assert api.square_verify(sp, bad) == 0
    bad = sp.copy(); bad[0, 64:96] = 0xff
    assert api.square_verify(bad, sc) == -1


def test_tail_tables_in_batches_of_chunks(api, oracle):
    """The tail's per-digit tables are built for a bounded number of chunks at a time (tail_batch_mb): one chunk per batch here, same bytes."""
    rng = np.random.default_rng(16)
    D, rb, P = 40, 8, 8
    v = rng.uniform(-0.9, 0.9, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x37" * 32, D); seed = bytes([12] * 32)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, rb, P, 16, 7, seed)
    try:
        api.set_option("tail_batch_mb", 1)
        rc, p, c = api.range_prove(v, bl, rb, P, 16, 7, seed)
        assert rc == rc_o == 0 and (p == p_o).all() and (c == c_o).all()
    finally:
        api.set_option("tail_batch_mb", 2048)


def test_square_proofs_batched_check(api, oracle):
    """All square proofs of a call in ONE random linear combination (k_sigma_rlc_*, kind 0): it holds for honest proofs, fails when any element is tampered with
    (commitment, proof point or response) or malformed, and rofl_square_verify's verdict stays the reference's in every case."""
    rng = np.random.default_rng(15)
    D = 260
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(b"\x35" * 32, D); r2 = oracle.rnd_scalar_vec(b"\x36" * 32, D)
    cl = oracle.commit_f32(v, r1, 32, 7)
    rc, sp, sc = api.square_prove(v, cl, r1, r2, 32, 7, bytes([11] * 32))
    assert rc == 0
    assert api.debug_square_rlc(sp, sc) == 1 and api.square_verify(sp, sc) == 1
    k = D - 3
    bad = sc.copy(); bad[k, 32:] = sc[k - 1, 32:]                       # another element's c_sq
    assert api.debug_square_rlc(sp, bad) == 0 and api.square_verify(sp, bad) == 0
    bad = sp.copy(); bad[k, :32] = sp[k - 1, :32]                       # another element's C'_l
    assert api.debug_square_rlc(bad, sc) == 0 and api.square_verify(bad, sc) == 0
    bad = sp.copy(); bad[k, 64] ^= 1                                    # z_m
    assert api.debug_square_rlc(bad, sc) == 0 and api.square_verify(bad, sc) == 0
    bad = sp.copy(); bad[k, 128] ^= 1                                   # z_r2
    assert api.debug_square_rlc(bad, sc) == 0 and api.square_verify(bad, sc) == 0
    bad = sp.copy(); bad[0, 64:96] = 0xff                               # non-canonical scalar -> FormatError
    assert api.debug_square_rlc(bad, sc) == 0 and api.square_verify(bad, sc) == -1
    bad = sc.copy(); bad[5, :32] = 0xff; bad[5, 31] = 0x7f              # undecodable point -> FormatError
    assert api.debug_square_rlc(sp, bad) == 0 and api.square_verify(sp, bad) == -1
    # two proofs whose errors would cancel under EQUAL weights do not cancel under the Fiat-Shamir weights: swap the responses of two elements
    bad = sp.copy(); bad[[1, 2], 64:] = sp[[2, 1], 64:]
    assert api.debug_square_rlc(bad, sc) == 0 and api.square_verify(bad, sc) == 0


def test_aggregate_and_dlog(api, oracle):
    x = np.array([[0.25, 1.25, -1.5], [-0.75, 1.25, -2.0], [0.5, 1.25, -3.0]], np.float32)
    cs = np.stack([oracle.commit_f32(r, None, 16, 7) for r in x])
    agg = api.aggregate(cs, 0)
    assert (agg == oracle.aggregate(cs, 0)).all()
    assert (api.aggregate(cs, 1) == oracle.aggregate(cs, 1)).all()
    rc, s, f = api.dlog(agg, 1 << 9, 16, 16, 7)        # small table: giant steps
    rc_o, s_o = oracle.dlog(agg, 1 << 9, 16)
    assert rc == rc_o == 0 and (s == s_o).all()
    assert (f == np.array([0.0, 3.75, -6.5], np.float32)).all()
    far = oracle.commit_f32(np.array([400.0], np.float32), None, 16, 7)
    assert api.dlog(far, 1 << 4, 8, 8, 7)[0] == -5 and oracle.dlog(far, 1 << 4, 8)[0] == -5


@pytest.mark.parametrize("c,slices,rt", [(3, 1, 1), (4, 3, 0), (5, 1, 0), (6, 2, 1), (7, 1, 0), (8, 2, 0), (9, 1, 0), (10, 3, 0), (11, 2, 1)])
def test_msm_window_widths(api, oracle, monkeypatch, c, slices, rt):
    """Every window width / slicing of the bucket MSM (k_msm, c <= 8) and of the wide-window sorted Pippenger (k_bm_*, c >= 9; `slices` = parts per
    bucket there) gives the oracle's bytes; rt=0 also exercises the path without generator tables (generic MSM for S and the verifier, folded IPP
    from round 0)."""
    monkeypatch.setenv("ROFL_MSM_C", str(c)); monkeypatch.setenv("ROFL_MSM_SLICES", str(slices))
    api.set_use_rt(rt)
    try:
        rng = np.random.default_rng(c)
        D, rngbits, P, nb = 6, 8, 2, 16
        mn, mx = oracle.clip_bounds(rngbits, nb, 7)
        v = rng.uniform(mn, mx, D).astype(np.float32)
        bl = oracle.rnd_scalar_vec(b"\x35" * 32, D)
        seed = bytes([c] * 32)
        rc_o, p_o, c_o = oracle.range_prove(v, bl, rngbits, P, nb, 7, seed)
        rc, p, cm = api.range_prove(v, bl, rngbits, P, nb, 7, seed)
        assert rc == rc_o == 0 and (cm == c_o).all() and (p == p_o).all()
        assert api.range_verify(p, cm, rngbits, seed) == 1
        badp = p.copy(); badp[1, 230] ^= 4
        assert api.range_verify(badp, cm, rngbits, seed) == 0
    finally:
        api.set_use_rt(1)


@pytest.mark.parametrize("tail_np,rt,unfold", [(0, 1, 3), (0, 0, 3), (4, 1, 3), (4, 0, 3), (2, 1, 1), (1, 1, 2), (32, 1, 3), (8, 0, 0)])
def test_ipp_tail_kernel_handover(api, oracle, tail_np, rt, unfold):
    """The fused on-device tail (k_ipp_tail: transcript, challenge inversion and folds on the device, frozen generators)
    takes over from the host-driven rounds at any round: from round 0, after the table catch-up, after ordinary folds."""
    api.set_option("tail_np", tail_np); api.set_use_rt(rt); api.set_option("rt_unfold", unfold)
    try:
        rng = np.random.default_rng(tail_np * 7 + rt)
        D, rngbits, P, nb = 7, 8, 2, 16            # 2 chunks x (m = 4, n = 8): N = 32, 5 rounds
        mn, mx = oracle.clip_bounds(rngbits, nb, 7)
        v = rng.uniform(mn, mx, D).astype(np.float32)
        bl = oracle.rnd_scalar_vec(b"\x36" * 32, D)
        seed = bytes([tail_np + 1] * 32)
        rc_o, p_o, c_o = oracle.range_prove(v, bl, rngbits, P, nb, 7, seed)
        rc, p, cm = api.range_prove(v, bl, rngbits, P, nb, 7, seed)
        assert rc == rc_o == 0 and (cm == c_o).all() and (p == p_o).all()
        assert api.range_verify(p, cm, rngbits, seed) == 1
    finally:
        api.set_option("tail_np", 32); api.set_use_rt(1); api.set_option("rt_unfold", 3)


@pytest.mark.parametrize("bits", [9, 10])
def test_generator_table_radix(api, oracle, bits):
    """Radix-2^9 / 2^10 generator tables (fewer additions per term than radix 2^8) give the same bytes."""
    api.set_option("rt_bits", bits); api.set_option("tail_np", 2)
    try:
        rng = np.random.default_rng(bits)
        D, rngbits, P, nb = 2, 8, 1, 8             # one chunk, m = 2, n = 8: 16 + 16 generators, fresh (n, fp) so the tables are rebuilt
        mn, mx = oracle.clip_bounds(rngbits, nb, 3)
        v = rng.uniform(mn, mx, D).astype(np.float32)
        bl = oracle.rnd_scalar_vec(b"\x37" * 32, D)
        seed = bytes([bits] * 32)
        rc_o, p_o, c_o = oracle.range_prove(v, bl, rngbits, P, nb, 3, seed)
        api.set_use_rt(0); api.set_use_rt(1)
        rc, p, cm = api.range_prove(v, bl, rngbits, P, nb, 3, seed)
        assert rc == rc_o == 0 and (cm == c_o).all() and (p == p_o).all()
        assert api.range_verify(p, cm, rngbits, seed) == 1
    finally:
        api.set_option("rt_bits", 8); api.set_option("tail_np", 32)


def test_compressed_rand_proof(api, oracle):
    """compressed_rand_proof (one sigma proof over all ElGamal pairs): bytes, R halves, existing-commitment mode, tamper and format rejection."""
    rng = np.random.default_rng(21)
    for D in (1, 9, 300):                      # 300 > 256: the 3-byte pair labels wrap around (generate_unique_u8_triplets.py:9-13)
        v = rng.uniform(-3, 3, D).astype(np.float32)
        bl = oracle.rnd_scalar_vec(b"\x61" * 32, D)
        seed = bytes([D % 251] * 32)
        rc_o, pf_o, pairs_o = oracle.crp_prove(v, None, bl, 16, 7, seed)
        rc, pf, pairs = api.crp_prove(v, None, bl, 16, 7, seed)
        assert rc == rc_o == 0 and (pf == pf_o).all() and (pairs == pairs_o).all()
        assert (pairs[:, 32:] == oracle.elgamal_R(bl)).all()
        assert api.crp_verify(pf, pairs) == 1 and oracle.crp_verify(pf, pairs) == 1
        rc2, pf2, pairs2 = api.crp_prove(v, pairs[:, :32].copy(), bl, 16, 7, seed)            # prove_existing
        assert rc2 == 0 and (pf2 == pf).all() and (pairs2 == pairs).all()
        if D > 1:
            bad = pairs.copy(); bad[D // 2, 32:] = pairs[0, 32:]
            assert api.crp_verify(pf, bad) == 0 and oracle.crp_verify(pf, bad) == 0
    badp = pf.copy(); badp[64:96] = 0xff
    assert api.crp_verify(badp, pairs) == -1 and oracle.crp_verify(badp, pairs) == -1
    badc = pairs.copy(); badc[1, :32] = 0xff
    assert api.crp_verify(pf, badc) == -1 and oracle.crp_verify(pf, badc) == -1
    assert api.crp_prove(v, badc[:, :32].copy(), bl, 16, 7, seed)[0] == -4


@pytest.mark.parametrize("tail_np,rt,unfold", [(2, 1, 1), (2, 0, 0), (1, 1, 2), (0, 1, 1), (0, 0, 0), (4, 1, 1)])
def test_ipp_frozen_level(api, oracle, tail_np, rt, unfold):
    """Middle rounds over FROZEN generators with on-the-fly Straus tables (k_frz_*): entered after the table catch-up or after ordinary
    folds, left through k_frz_exit into the tail kernel, or run to the last round when the tail is off -- always the oracle's bytes."""
    api.set_option("tail_np", tail_np); api.set_use_rt(rt); api.set_option("rt_unfold", unfold); api.set_option("frozen", 1)
    try:
        rng = np.random.default_rng(tail_np * 11 + rt)
        D, rngbits, P, nb = 14, 8, 2, 16            # 2 chunks x (m = 8, n = 8): N = 64, 6 rounds
        mn, mx = oracle.clip_bounds(rngbits, nb, 7)
        v = rng.uniform(mn, mx, D).astype(np.float32)
        bl = oracle.rnd_scalar_vec(b"\x38" * 32, D)
        seed = bytes([tail_np + 40] * 32)
        rc_o, p_o, c_o = oracle.range_prove(v, bl, rngbits, P, nb, 7, seed)
        rc, p, cm = api.range_prove(v, bl, rngbits, P, nb, 7, seed)
        assert rc == rc_o == 0 and (cm == c_o).all() and (p == p_o).all()
        api.set_option("frozen", 0)
        rc, p2, _ = api.range_prove(v, bl, rngbits, P, nb, 7, seed)
        assert (p2 == p).all()
    finally:
        api.set_option("tail_np", 32); api.set_use_rt(1); api.set_option("rt_unfold", 3)


def test_optimised_encodings_end_to_end(api, oracle):
    """EncParamsRangeCompressed / EncParamsL2Compressed (params.rs): encrypt gives exactly the pieces the oracle builds one by one,
    verify accepts them, honours check_percentage, and rejects a tampered field of every kind."""
    rng = np.random.default_rng(33)
    D, P, seed = 6, 2, bytes([11] * 32)
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x65" * 32, D)
    # --- range compressed (fp 16/7, 8-bit)
    rc, msg = api.enc_range_compressed_encrypt(v, bl, 8, P, 16, 7, seed)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 16, 7, seed)
    rc2, rp_o, pairs_o = oracle.crp_prove(v, c_o, bl, 16, 7, seed)
    assert rc == rc_o == rc2 == 0 and (msg["range_proof"] == p_o).all() and (msg["enc_values"] == pairs_o).all() and (msg["rand_proof"] == rp_o).all()
    assert api.enc_range_compressed_verify(msg, 1.0, seed) == 1
    bad = dict(msg); bad["enc_values"] = msg["enc_values"].copy(); bad["enc_values"][1, 32:] = msg["enc_values"][0, 32:]
    assert api.enc_range_compressed_verify(bad, 1.0, seed) == 0
    bad = dict(msg); bad["range_proof"] = msg["range_proof"].copy(); bad["range_proof"][0, 70] ^= 1
    assert api.enc_range_compressed_verify(bad, 1.0, seed) == 0
    # --- L2 compressed (fp 32/7, 8-bit L-inf, 32-bit L2)
    rc, m2 = api.enc_l2_compressed_encrypt(v, bl, 8, P, 32, 32, 7, seed)
    assert rc == 0
    rnd = oracle.rnd_scalar_vec(oracle.derive_key(seed, 7, 1), D)                     # rand_scalars: DOM_RND_VEC stream 1
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 32, 7, seed)
    rc_s, sumproof_o, sumcm_o = oracle.l2_prove(v, rnd, 32, 32, 7, seed)
    rc_c, rp_o, pairs_o = oracle.crp_prove(v, c_o, bl, 32, 7, seed)
    rc_q, sp_o, sc_o = oracle.square_prove(v, c_o, bl, rnd, 32, 7, seed)
    assert rc_o == rc_s == rc_c == rc_q == 0
    assert (m2["range_proof"] == p_o).all() and (m2["square_range_proof"] == sumproof_o).all() and (m2["rand_proof"] == rp_o).all() and (m2["square_proof"] == sp_o).all()
    assert (m2["enc_values"][:, :64] == pairs_o).all() and (m2["enc_values"][:, 64:] == sc_o[:, 32:]).all()
    assert api.enc_l2_compressed_verify(m2, seed) == 1
    for field, (i, j) in [("enc_values", (2, 70)), ("square_proof", (3, 100)), ("range_proof", (1, 40)), ("square_range_proof", (None, 50))]:
        bad = dict(m2); bad[field] = m2[field].copy()
        if i is None: bad[field][j] ^= 1
        else: bad[field][i, j] ^= 1
        assert api.enc_l2_compressed_verify(bad, seed) in (0, -4), field


def test_unoptimised_encodings_end_to_end(api, oracle):
    """EncParamsRange / EncParamsL2 (params.rs:467-510, 607-646, 186-233): encrypt == the oracle's pieces put together the reference's way,
    verify accepts, honours check_percentage, rejects tampering; the reference's quirk that the RandProofs cover the UNCLIPPED plaintext."""
    rng = np.random.default_rng(34)
    D, P, seed = 6, 2, bytes([12] * 32)
    v = (rng.integers(-100, 100, D) / 128).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x6c" * 32, D)
    rc, msg = api.enc_range_encrypt(v, bl, 8, P, 1.0, 16, 7, seed)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 16, 7, seed)
    rc_r, pf_o, pairs_o = oracle.rand_prove(v, c_o, bl, 16, 7, seed)
    assert rc == rc_o == rc_r == 0 and (msg["range_proof"] == p_o).all() and (msg["rand_proof"] == pf_o).all() and (msg["enc_values"] == pairs_o).all()
    assert api.enc_range_verify(msg, 1.0, seed) == 1
    bad = dict(msg); bad["rand_proof"] = msg["rand_proof"].copy(); bad["rand_proof"][2, 70] ^= 1
    assert api.enc_range_verify(bad, 1.0, seed) == 0
    bad = dict(msg); bad["range_proof"] = msg["range_proof"].copy(); bad["range_proof"][1, 40] ^= 1
    assert api.enc_range_verify(bad, 1.0, seed) == 0
    # probabilistic checking: range proofs over the first round(6 * 0.5) = 3 elements only, fresh commitments for the pairs
    rc, half = api.enc_range_encrypt(v, bl, 8, P, 0.5, 16, 7, seed)
    rc_o, p3, c3 = oracle.range_prove(v[:3], bl[:3], 8, P, 16, 7, seed)
    rc_r, pf3, pairs3 = oracle.rand_prove(v, None, bl, 16, 7, seed)
    assert rc == rc_o == rc_r == 0 and half["range_proof"].shape == p3.shape and (half["range_proof"] == p3).all() and (half["rand_proof"] == pf3).all() and (half["enc_values"] == pairs3).all()
    assert api.enc_range_verify(half, 0.5, seed) == 1 and api.enc_range_verify(half, 1.0, seed) == 0
    # quirk: a value outside the range is clipped for the range proof but not for the RandProof -> bytes as the reference would make them, verify fails
    v2 = v.copy(); v2[4] = 5.0
    clipped = oracle.clip_f32_to_range_vec(v2, 8, 16, 7) if hasattr(oracle, "clip_f32_to_range_vec") else np.clip(v2, *oracle.clip_bounds(8, 16, 7)).astype(np.float32)
    rc, m2 = api.enc_range_encrypt(v2, bl, 8, P, 1.0, 16, 7, seed)
    rc_o, p_o, c_o = oracle.range_prove(clipped, bl, 8, P, 16, 7, seed)
    rc_r, pf_o, pairs_o = oracle.rand_prove(v2, c_o, bl, 16, 7, seed)
    assert rc == rc_o == rc_r == 0 and (m2["range_proof"] == p_o).all() and (m2["rand_proof"] == pf_o).all() and (m2["enc_values"] == pairs_o).all()
    assert api.enc_range_verify(m2, 1.0, seed) == 0
    # --- L2 (fp 32/7, 8-bit L-inf, 32-bit L2)
    rc, m3 = api.enc_l2_encrypt(v, bl, 8, P, 32, 32, 7, seed)
    rnd = oracle.rnd_scalar_vec(oracle.derive_key(seed, 7, 1), D)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 32, 7, seed)
    rc_s, sumproof_o, sumcm_o = oracle.l2_prove(v, rnd, 32, 32, 7, seed)
    rc_q, sp_o, sc_o = oracle.square_rand_prove(v, c_o, bl, rnd, 32, 7, seed)
    assert rc == rc_o == rc_s == rc_q == 0
    assert (m3["range_proof"] == p_o).all() and (m3["square_range_proof"] == sumproof_o).all() and (m3["square_proof"] == sp_o).all() and (m3["enc_values"] == sc_o).all()
    assert api.enc_l2_verify(m3, seed) == 1
    for field, (i, j) in [("enc_values", (2, 70)), ("square_proof", (3, 100)), ("range_proof", (1, 40)), ("square_range_proof", (None, 50))]:
        bad = dict(m3); bad[field] = m3[field].copy()
        if i is None: bad[field][j] ^= 1
        else: bad[field][i, j] ^= 1
        assert api.enc_l2_verify(bad, seed) == 0, field


def test_rand_and_square_rand_proofs(api, oracle):
    """RandProof (enc type 2) and SquareRandProof (enc type 3): bytes, existing-commitment mode, tamper and format rejection."""
    rng = np.random.default_rng(55)
    D = 7
    v = (rng.integers(-200, 200, D) / 128).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(b"\x66" * 32, D); r2 = oracle.rnd_scalar_vec(b"\x67" * 32, D); seed = bytes([13] * 32)
    rc_o, pf_o, pr_o = oracle.rand_prove(v, None, r1, 16, 7, seed)
    rc, pf, pr = api.rand_prove(v, None, r1, 16, 7, seed)
    assert rc == rc_o == 0 and (pf == pf_o).all() and (pr == pr_o).all()
    assert (pr[:, :32] == oracle.commit_f32(v, r1, 16, 7)).all() and (pr[:, 32:] == oracle.elgamal_R(r1)).all()
    assert api.rand_verify(pf, pr) == 1 and oracle.rand_verify(pf, pr) == 1
    rc, pf2, pr2 = api.rand_prove(v, pr[:, :32].copy(), r1, 16, 7, seed)
    assert rc == 0 and (pf2 == pf).all() and (pr2 == pr).all()
    bad = pr.copy(); bad[2, 32:] = pr[3, 32:]
    assert api.rand_verify(pf, bad) == 0 and oracle.rand_verify(pf, bad) == 0
    badp = pf.copy(); badp[1, 64:96] = 0xff
    assert api.rand_verify(badp, pr) == -1 and oracle.rand_verify(badp, pr) == -1
    rc_o, sp_o, sc_o = oracle.square_rand_prove(v, None, r1, r2, 32, 7, seed)
    rc, sp, sc = api.square_rand_prove(v, None, r1, r2, 32, 7, seed)
    assert rc == rc_o == 0 and (sp == sp_o).all() and (sc == sc_o).all()
    assert api.square_rand_verify(sp, sc) == 1 and oracle.square_rand_verify(sp, sc) == 1
    rc, sp2, sc2 = api.square_rand_prove(v, sc[:, :32].copy(), r1, r2, 32, 7, seed)
    assert rc == 0 and (sp2 == sp).all() and (sc2 == sc).all()
    bad = sc.copy(); bad[4, 64:] = sc[5, 64:]
    assert api.square_rand_verify(sp, bad) == 0 and oracle.square_rand_verify(sp, bad) == 0
    bad = sc.copy(); bad[0, 32:64] = sc[1, 32:64]
    assert api.square_rand_verify(sp, bad) == 0 and oracle.square_rand_verify(sp, bad) == 0
    badp = sp.copy(); badp[6, 160:] = 0xff
    assert api.square_rand_verify(badp, sc) == -1 and oracle.square_rand_verify(badp, sc) == -1


def test_device_transcript_absorb_matches_sequential(api):
    """ts_kernels.cuh k_ts_absorbV: the warp-cooperative absorb of m commitments (closed-form STROBE framing bytes, one lane per Keccak word)
    against the sequential Merlin code, for every alignment of the 41-byte records against the 166-byte sponge rate."""
    rng = np.random.default_rng(77)
    for m in list(range(1, 48)) + [83, 166, 167, 331]:
        V = rng.integers(0, 256, (m, 32), dtype=np.uint8)
        assert api.debug_ts_absorb(V, 8 if m % 2 else 16, m % 2) == 0, m


def test_verifier_weights_are_bound_to_every_proof_of_the_call(api, oracle):
    """The batched verifier's scalars (c_i, rho_i) are Fiat-Shamir outputs over the seed AND all proofs / commitments of the call: changing any
    chunk changes the weights of ALL chunks, so a prover who knows the seed still cannot craft chunks whose errors cancel (the reference
    verifies chunk by chunk with thread_rng, range_proof_vec/mod.rs:178-190)."""
    rng = np.random.default_rng(78)
    D, P = 16, 4
    v = rng.uniform(-0.9, 0.9, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x71" * 32, D)
    rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, b"\x72" * 32)
    seed = bytes(32)                                               # a seed the attacker knows
    ok, w0 = api.debug_verify_weights(p, c, 8, seed)
    assert ok == 1 and len({w0[k, i].tobytes() for k in range(2) for i in range(P)}) == 2 * P
    ok, w1 = api.debug_verify_weights(p, c, 8, seed)
    assert (w1 == w0).all()                                        # deterministic
    ok, w2 = api.debug_verify_weights(p, c, 8, b"\x01" * 32)
    assert ok == 1 and all((w2[k, i] != w0[k, i]).any() for k in range(2) for i in range(P))
    for what in ("proof_point", "proof_scalar", "commitment"):
        pp, cc = p.copy(), c.copy()
        if what == "proof_point": pp[P - 1, 224 + 3] ^= 1           # L_1 of the last chunk
        elif what == "proof_scalar": pp[P - 1, -32] ^= 1            # b of the last chunk (stays canonical: low byte)
        else: cc[D - 1] = c[0]
        ok, w = api.debug_verify_weights(pp, cc, 8, seed)
        assert ok in (0, 1)
        assert all((w[k, i] != w0[k, i]).any() for k in range(2) for i in range(P)), what      # chunk 0's weights moved although only the last chunk changed


def test_l2_compressed_message_with_undecodable_R_is_refused(api, oracle):
    """decode_l2enc_vec (params.rs:560-571) deserialises c.L, c.R and c_sq of every record; EncL2Compressed::verify never looks at c.R again, so the
    validation has to happen at the boundary (square_rand_proof/pedersen.rs:33-45, rand_proof/el_gamal.rs:112-123)."""
    rng = np.random.default_rng(79)
    D, P, seed = 6, 2, bytes([12] * 32)
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x73" * 32, D)
    rc, m = api.enc_l2_compressed_encrypt(v, bl, 8, P, 32, 32, 7, seed)
    assert rc == 0 and api.enc_l2_compressed_verify(m, seed) == 1
    for col in (0, 32, 64):
        bad = dict(m); bad["enc_values"] = m["enc_values"].copy(); bad["enc_values"][D - 2, col:col + 32] = 0xff
        assert not oracle.point_valid(bad["enc_values"][D - 2, col:col + 32])
        assert api.enc_l2_compressed_verify(bad, seed) == -4, col
    # a VALID but different R is not this arm's business (the reference does not check the rand proof here: params.rs:257-289)
    ok = dict(m); ok["enc_values"] = m["enc_values"].copy(); ok["enc_values"][1, 32:64] = np.frombuffer(oracle.basepoint(), np.uint8)
    assert api.enc_l2_compressed_verify(ok, seed) == 1


def test_concurrent_callers_share_one_context(api, oracle):
    """rofl_service calls verify() for many clients at once from a rayon pool (server.rs:516-522,666) and proves several clients per process
    (bin/basic_client.rs:136-161): concurrent callers of ONE context run on separate lanes (streams) and share the cached tables; every
    caller must get exactly the bytes / verdicts of a lone caller."""
    import threading
    rng = np.random.default_rng(80)
    jobs = []
    for k in range(8):
        D = [5, 8, 3, 16, 7, 4, 12, 9][k]; P = [2, 4, 1, 4, 2, 4, 2, 1][k]
        v = rng.uniform(-0.9, 0.9, D).astype(np.float32); bl = oracle.rnd_scalar_vec(bytes([0x60 + k]) * 32, D)
        jobs.append((v, bl, P, bytes([0x20 + k]) * 32))
    want = [api.range_prove(v, bl, 8, P, 16, 7, seed) for v, bl, P, seed in jobs]
    got, errs = [None] * len(jobs), []
    def run(i):
        try:
            v, bl, P, seed = jobs[i]
            rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, seed)
            ok = api.range_verify(p, c, 8, seed)
            bad = c.copy(); bad[0] = c[-1] if len(c) > 1 else np.frombuffer(oracle.basepoint(), np.uint8)
            got[i] = (rc, p, c, ok, api.range_verify(p, bad, 8, seed))
        except Exception as ex:  # noqa: BLE001
            errs.append(repr(ex))
    th = [threading.Thread(target=run, args=(i,)) for i in range(len(jobs))]
    for x in th: x.start()
    for x in th: x.join()
    assert not errs, errs
    for (rc0, p0, c0), (rc, p, c, ok, okbad) in zip(want, got):
        assert rc == rc0 == 0 and (p == p0).all() and (c == c0).all() and ok == 1 and okbad == 0


def test_host_absorb_fallback_gives_the_same_bytes(api, oracle):
    """Chunks with very many commitments (resnet18-full: 2^18 per chunk) absorb them on the host instead of the device (engine.cuh
    absorb_commitments); forced here at a tiny size: same proof bytes, same verdicts."""
    rng = np.random.default_rng(81)
    D, P = 12, 2
    v = rng.uniform(-0.9, 0.9, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x74" * 32, D); seed = b"\x75" * 32
    rc0, p0, c0 = api.range_prove(v, bl, 8, P, 16, 7, seed)
    api.set_option("ts_host_m", 0)
    try:
        rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, seed)
        assert rc == rc0 == 0 and (p == p0).all() and (c == c0).all()
        assert api.range_verify(p, c, 8, seed) == 1
        bad = c.copy(); bad[3] = c[4]
        assert api.range_verify(p, bad, 8, seed) == 0
    finally:
        api.set_option("ts_host_m", 8192)
    rc_o, p_o, _ = oracle.range_prove(v, bl, 8, P, 16, 7, seed)
    assert (p0 == p_o).all()


def test_server_batch_verification_names_the_offending_client(api, oracle):
    """rofl_range_verify_batch / rofl_enc_l2_compressed_verify_batch: all clients of a round in ONE random linear combination (server.rs:516-522,
    666-667 verifies them one by one); the per-client verdicts must be exactly those of the per-client calls, for honest and tampered clients."""
    rng = np.random.default_rng(82)
    K, D, P = 3, 6, 2
    proofs, commits, msgs, seeds = [], [], [], []
    for k in range(K):
        v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = oracle.rnd_scalar_vec(bytes([0x76 + k]) * 32, D); seed = bytes([0x30 + k]) * 32
        rc, p, c = api.range_prove(v, bl, 8, P, 32, 7, seed); assert rc == 0
        proofs.append(p); commits.append(c)
        rc, m = api.enc_l2_compressed_encrypt(v, bl, 8, P, 32, 32, 7, seed); assert rc == 0
        msgs.append(m)
    vs = b"\x44" * 32
    assert api.range_verify_batch(np.stack(proofs), np.stack(commits), 8, vs).tolist() == [1, 1, 1]
    bad_c = [c.copy() for c in commits]; bad_c[1][2] = commits[1][3]
    assert api.range_verify_batch(np.stack(proofs), np.stack(bad_c), 8, vs).tolist() == [1, 0, 1]
    bad_p = [p.copy() for p in proofs]; bad_p[2][0, 128:160] = 0xff                      # non-canonical t_x: FormatError for that client only
    assert api.range_verify_batch(np.stack(bad_p), np.stack(commits), 8, vs).tolist() == [1, 1, -1]
    bad_c = [c.copy() for c in commits]; bad_c[0][0] = 0xff
    assert api.range_verify_batch(np.stack(proofs), np.stack(bad_c), 8, vs).tolist() == [-4, 1, 1]
    # whole messages
    assert api.enc_l2_compressed_verify_batch(msgs, vs).tolist() == [1, 1, 1]
    for field, idx, want in [("enc_values", (2, 70), (0, -4)), ("square_proof", (3, 100), (0,)), ("range_proof", (1, 40), (0,)), ("square_range_proof", (50,), (0,)), ("enc_values", (1, 33), (0, -4, 1))]:
        tam = [dict(m) for m in msgs]; tam[1][field] = msgs[1][field].copy(); tam[1][field][idx] ^= 1
        got = api.enc_l2_compressed_verify_batch(tam, vs).tolist()
        assert got[0] == 1 and got[2] == 1 and got[1] in want and got[1] == api.enc_l2_compressed_verify(tam[1], vs), (field, got)


@pytest.mark.parametrize("unf,tail_np,frz,D,P", [(1, 0, 0, 8, 2), (2, 2, 1, 16, 2), (3, 0, 1, 16, 1), (4, 4, 0, 32, 2), (4, 1, 1, 64, 1), (2, 32, 1, 6, 4)])
def test_unfolded_rounds_without_generator_tables(api, oracle, unf, tail_np, frz, D, P):
    """Chunks too large for generator tables (resnet18-full: 2^21 bit positions per chunk) run their first IPP rounds UNFOLDED as Pippenger MSMs over the
    original generators (hi / lo halves of the 2np-blocks addressed through the MSM segments) and then catch up with ONE joint double-and-add per folded
    generator (k_catchup_naf) instead of a fold ladder per round; forced here at tiny sizes: same proof bytes for every schedule."""
    rng = np.random.default_rng(100 + unf)
    v = rng.uniform(-0.99, 0.99, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x77" * 32, D); seed = bytes([0x40 + unf]) * 32
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 16, 7, seed); assert rc_o == 0
    api.set_use_rt(0); api.set_option("nt_unfold_min", 2); api.set_option("nt_unfold", unf); api.set_option("tail_np", tail_np); api.set_option("frozen", frz)
    try:
        rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, seed)
        assert rc == 0 and (c == c_o).all() and (p == p_o).all()
        assert api.range_verify(p, c, 8, seed) == 1
    finally:
        api.set_use_rt(1); api.set_option("nt_unfold_min", 1 << 16); api.set_option("nt_unfold", 4); api.set_option("tail_np", 32); api.set_option("frozen", 1)


def test_unfolded_rounds_through_the_wide_window_msm(api, oracle, monkeypatch):
    """The same schedule with the wide-window sorted Pippenger (k_bm_*) forced for every MSM: mapped segments + bucket sort + fat top window."""
    monkeypatch.setenv("ROFL_MSM_C", "9"); monkeypatch.setenv("ROFL_MSM_SLICES", "2")
    rng = np.random.default_rng(111)
    D, P = 32, 2
    v = rng.uniform(-0.99, 0.99, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x78" * 32, D); seed = b"\x79" * 32
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 16, 7, seed); assert rc_o == 0
    api.set_use_rt(0); api.set_option("nt_unfold_min", 2); api.set_option("nt_unfold", 3)
    try:
        rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, seed)
        assert rc == 0 and (c == c_o).all() and (p == p_o).all() and api.range_verify(p, c, 8, seed) == 1
    finally:
        api.set_use_rt(1); api.set_option("nt_unfold_min", 1 << 16); api.set_option("nt_unfold", 4)
