"""GPU parity tests (run on the B200 box with -m gpu): every call goes through the C ABI of librofl_b200.so (CUDA only)
and is compared with the CPU oracle on the same seeded inputs -- bit-exact for commitments, proofs, verdicts and
decrypted values -- plus size-independent properties at BASELINE.json's full sizes (prove -> verify round trips,
homomorphism, tamper rejection)."""
import os
import sys
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = 2**252 + 27742317777372353535851937790883648493


@pytest.fixture(scope="module")
def api():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    pkg = g.load_package()
    return pkg.context(0)          # raises (no CPU fallback) if the CUDA library or the device is missing


def test_library_is_cuda_and_loaded(api):
    with open("/proc/self/maps") as f:
        assert "librofl_b200.so" in f.read()
    assert api.lib.rofl_ctx_stream(api.h) is not None


def test_field_arithmetic_device_paths(api):
    """The inline-PTX field arithmetic (fe25519.cuh: Comba columns with carry predicates) against Python integers, on random
    and extreme 256-bit LOOSE representatives (values >= p, all ones, 2^256-38+-1, p, p+-1 ...)."""
    P = 2**255 - 19
    rng = np.random.default_rng(11)
    edge = [0, 1, 2, 18, 19, 20, 37, 38, 39, P - 1, P, P + 1, 2 * P, 2 * P + 1, 2**255 - 1, 2**255, 2**255 + 18, 2**255 + 19, 2**256 - 39, 2**256 - 38,
            2**256 - 37, 2**256 - 1, 2**256 - 2, 2**224 - 1, 2**32 - 1, 2**32, (2**256 - 1) // 3, 0xFFFFFFFF00000000FFFFFFFF00000000FFFFFFFF00000000FFFFFFFF00000000]
    vals_a = [x for x in edge for _ in edge] + [int.from_bytes(rng.bytes(32), "little") for _ in range(4000)]
    vals_b = [y for _ in edge for y in edge] + [int.from_bytes(rng.bytes(32), "little") for _ in range(4000)]
    a = np.frombuffer(b"".join(x.to_bytes(32, "little") for x in vals_a), np.uint8).reshape(-1, 32)
    b = np.frombuffer(b"".join(x.to_bytes(32, "little") for x in vals_b), np.uint8).reshape(-1, 32)
    out = api.field_selftest(a, b)
    for i, (x, y) in enumerate(zip(vals_a, vals_b)):
        exp = [x * y % P, x * x % P, (x + y) % P, (x - y) % P, (x + y) * (x - y) % P, pow(x, P - 2, P)]
        got = [int.from_bytes(out[i, k].tobytes(), "little") for k in range(6)]
        assert got == exp, (i, hex(x), hex(y), [hex(g) for g in got], [hex(e) for e in exp])


def test_device_scalar_arithmetic_against_python_integers(api):
    """sc_mul's fold reduction (any 256-bit operands) and the division-step inversion, as compiled for the device, against Python integers."""
    L = 2**252 + 27742317777372353535851937790883648493
    rng = np.random.default_rng(11)
    edge = [0, 1, 2, L - 1, L, L + 1, 2 * L - 1, 2 * L, 2**252 - 1, 2**252, 2**253 - 1, 2**255 - 19, 2**256 - 1, 2**256 - 2**224, 2**124, 2**125 - 1, 2**62, 2**186]
    vals_a = [x for x in edge for _ in edge] + [int.from_bytes(rng.bytes(32), "little") for _ in range(6000)] + [int.from_bytes(rng.bytes(32), "little") % L for _ in range(2000)]
    vals_b = [y for _ in edge for y in edge] + [int.from_bytes(rng.bytes(32), "little") for _ in range(6000)] + [int.from_bytes(rng.bytes(32), "little") % L for _ in range(2000)]
    a = np.frombuffer(b"".join(x.to_bytes(32, "little") for x in vals_a), np.uint8).reshape(-1, 32)
    b = np.frombuffer(b"".join(x.to_bytes(32, "little") for x in vals_b), np.uint8).reshape(-1, 32)
    out = api.scalar_selftest(a, b)
    for i, (x, y) in enumerate(zip(vals_a, vals_b)):
        inv = pow(x % L, L - 2, L)
        got = [int.from_bytes(out[i, k].tobytes(), "little") for k in range(3)]
        assert got == [x * y % L, inv, inv], (i, hex(x), hex(y), [hex(g) for g in got])


def test_commit_conversion_parity(api, oracle):
    rng = np.random.default_rng(0)
    v = np.concatenate([rng.uniform(-300, 300, 2000), [0.0, -0.0, 0.25, -1.5, 600.0, -600.0, 0.5 / 128, 1.5 / 128]]).astype(np.float32)
    bl = oracle.rnd_scalar_vec(b"\x31" * 32, v.size)
    for nb, fr in [(16, 7), (32, 7), (8, 7), (64, 7), (16, 0), (32, 12)]:
        assert (api.f32_to_scalar_vec(v, nb, fr) == oracle.f32_to_scalar_vec(v, nb, fr)).all()
        L_, R_ = api.commit(v, bl, nb, fr, want_R=True)
        assert (L_ == oracle.commit_f32(v, bl, nb, fr)).all()
        assert (R_ == oracle.elgamal_R(bl)).all()
    assert (api.commit(v, None, 16, 7) == oracle.commit_f32(v, None, 16, 7)).all()
    s = oracle.f32_to_scalar_vec(v, 16, 7)
    assert (api.scalar_to_f32_vec(s, 16, 7) == oracle.scalar_to_f32_vec(s, 16, 7)).all()
    assert (api.rnd_scalar_vec(b"\x31" * 32, 100) == oracle.rnd_scalar_vec(b"\x31" * 32, 100)).all()


# (D, range bits, n_partition, n_bits): ragged / padded / single element / single chunk / many chunks
CASES = [(5, 8, 2, 16), (3, 16, 4, 16), (8, 8, 1, 16), (1, 8, 4, 16), (100, 8, 4, 16), (300, 16, 64, 16), (64, 32, 8, 32), (17, 64, 2, 64)]


@pytest.mark.parametrize("D,rb,P,nb", CASES)
def test_range_proof_bytes_match_oracle(api, oracle, D, rb, P, nb):
    rng = np.random.default_rng(D * 100 + rb)
    mn, mx = oracle.clip_bounds(rb, nb, 7)
    v = rng.uniform(mn, mx, D).astype(np.float32)
    v[0] = mx; v[-1] = mn
    bl = oracle.rnd_scalar_vec(b"\x32" * 32, D)
    seed = bytes([7] * 32)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, rb, P, nb, 7, seed)
    rc, p, c = api.range_prove(v, bl, rb, P, nb, 7, seed)
    assert rc == rc_o == 0
    assert (c == c_o).all()
    assert p.shape == p_o.shape and (p == p_o).all()
    assert api.range_verify(p, c, rb, seed) == 1
    assert oracle.range_verify(p, c, rb, seed) == 1          # GPU proof accepted by the reference-equivalent verifier
    bad = c.copy(); bad[0] = np.frombuffer(oracle.basepoint(), np.uint8)
    assert api.range_verify(p, bad, rb, seed) == 0
    badp = p.copy(); badp[0, 40] ^= 1
    assert api.range_verify(badp, c, rb, seed) == oracle.range_verify(badp, c, rb, seed)
    badp = p.copy(); badp[-1, 128:160] = 0xff
    assert api.range_verify(badp, c, rb, seed) == -1 == oracle.range_verify(badp, c, rb, seed)
    badp = p.copy(); badp[0, 0:32] = 0
    assert api.range_verify(badp, c, rb, seed) == 0


def test_range_prove_zero_blindings_like_the_service(api, oracle):      # client.rs:70-72 derive_dummy_blindings
    v = np.linspace(-0.9, 0.9, 40).astype(np.float32)
    z = np.zeros((40, 32), np.uint8)
    rc, p, c = api.range_prove(v, z, 8, 4, 16, 7, b"\x05" * 32)
    rc_o, p_o, c_o = oracle.range_prove(v, z, 8, 4, 16, 7, b"\x05" * 32)
    assert rc == 0 and (p == p_o).all() and (c == c_o).all()
    assert (c == oracle.commit_f32(v, None, 16, 7)).all()


def test_range_prove_errors(api, oracle):
    z = np.zeros((8, 32), np.uint8)
    assert api.range_prove(np.full(8, 1.5, np.float32), z, 8, 4, 16, 7)[0] == 2
    assert api.range_prove(np.zeros(8, np.float32), z, 8, 3, 16, 7)[0] == -99
    assert api.range_prove(np.zeros(8, np.float32), z, 12, 4, 16, 7)[0] == -7 == oracle.range_prove(np.zeros(8, np.float32), z, 12, 4, 16, 7)[0]
    assert api.range_prove(np.array([np.nan] + [0] * 7, np.float32), z, 8, 4, 16, 7)[0] == -98


def test_oracle_proofs_verify_on_gpu(api, oracle):
    rng = np.random.default_rng(11)
    v = rng.uniform(-0.99, 0.99, 50).astype(np.float32)
    rc, p, c = oracle.range_prove(v, oracle.rnd_scalar_vec(b"\x40" * 32, 50), 8, 8, 16, 7, b"\x41" * 32)
    assert rc == 0 and api.range_verify(p, c, 8, b"\x42" * 32) == 1


def test_l2_and_square_parity(api, oracle):
    rng = np.random.default_rng(5)
    D = 500
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(b"\x33" * 32, D); r2 = oracle.rnd_scalar_vec(b"\x34" * 32, D)
    seed = bytes([9] * 32)
    rc_o, pf_o, cm_o = oracle.l2_prove(v, r2, 32, 32, 7, seed)
    rc, pf, cm = api.l2_prove(v, r2, 32, 32, 7, seed)
    assert rc == rc_o == 0 and (pf == pf_o).all() and (cm == cm_o).all()
    assert api.l2_verify(pf, cm, 32, seed) == 1 and oracle.l2_verify(pf, cm, 32, seed) == 1
    assert api.l2_verify(pf, oracle.basepoint(), 32, seed) == 0
    assert api.l2_prove(np.array([8.0], np.float32), np.zeros((1, 32), np.uint8), 16, 32, 7)[0] == 4        # l2_range_proof_vec/mod.rs:356-373
    assert api.l2_prove(np.array([6.0, 6.0], np.float32), np.zeros((2, 32), np.uint8), 16, 32, 7)[0] == 4
    cl = oracle.commit_f32(v, r1, 32, 7)
    rc_o, sp_o, sc_o = oracle.square_prove(v, cl, r1, r2, 32, 7, seed)
    rc, sp, sc = api.square_prove(v, cl, r1, r2, 32, 7, seed)
    assert rc == rc_o == 0 and (sp == sp_o).all() and (sc == sc_o).all()
    assert api.square_verify(sp, sc) == 1 and oracle.square_verify(sp, sc) == 1
    # sum of c_sq equals the L2 commitment (l2_range_proof_vec/mod.rs:539-561)
    assert api.aggregate(sc[:, 32:].reshape(D, 1, 32), 0)[0].tobytes() == cm.tobytes()
    bad = sc.copy(); bad[1, 32:] = sc[2, 32:]
    assert api.square_verify(sp, bad) == 0
    bad = sp.copy(); bad[0, 64:96] = 0xff
    assert api.square_verify(bad, sc) == -1


def test_square_proofs_batched_check(api, oracle):
    """All square proofs of a call in ONE random linear combination (k_sigma_rlc_*, kind 0): it holds for honest proofs, fails when any element is tampered with
    (commitment, proof point or response) or malformed, and rofl_square_verify's verdict stays the reference's in every case."""
    rng = np.random.default_rng(15)
    D = 3000
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


def test_aggregate_dlog_parity(api, oracle):
    rng = np.random.default_rng(6)
    n_clients, D = 6, 400
    x = (rng.integers(-2000, 2000, (n_clients, D)) / 128).astype(np.float32)
    cs = np.stack([oracle.commit_f32(r, None, 16, 7) for r in x])
    agg = api.aggregate(cs, 0)
    assert (agg == oracle.aggregate(cs, 0)).all()
    assert (api.aggregate(cs, 1) == oracle.aggregate(cs, 1)).all()
    rc, s, f = api.dlog(agg, 1 << 16, 16, 16, 7)
    rc_o, s_o = oracle.dlog(agg, 1 << 16, 16)
    assert rc == rc_o == 0 and (s == s_o).all()
    assert (f == x.sum(0, dtype=np.float64).astype(np.float32)).all()
    rc, s, f = api.dlog(agg[:50], 1 << 9, 16, 16, 7)           # small table: giant steps
    assert rc == 0 and (s == s_o[:50]).all()
    far = oracle.commit_f32(np.array([400.0], np.float32), None, 16, 7)
    assert api.dlog(far, 1 << 4, 8, 8, 7)[0] == -5
    # accumulator quirk: (B,B) start => +1 LSB (SURVEY.md Appendix B.1)
    rc, _, f1 = api.dlog(api.aggregate(cs, 1), 1 << 16, 16, 16, 7)
    assert (f1 == f_plus(x)).all()


def f_plus(x):
    return (x.sum(0, dtype=np.float64) + 1.0 / 128).astype(np.float32)


def test_cancelling_blindings_homomorphism(api, oracle):      # range_proof_vec/mod.rs:369-399
    vecs = [[0.25, 1.25, -1.5], [-0.75, 1.25, -2.0], [0.5, 1.25, -3.0]]
    b1 = oracle.rnd_scalar_vec(b"\x08" * 32, 3); b2 = oracle.rnd_scalar_vec(b"\x09" * 32, 3)
    b3 = np.stack([np.frombuffer(((-(int.from_bytes(b1[i].tobytes(), "little") + int.from_bytes(b2[i].tobytes(), "little"))) % L).to_bytes(32, "little"), np.uint8) for i in range(3)])
    cs = []
    for v, b in zip(vecs, [b1, b2, b3]):
        rc, p, c = api.range_prove(np.array(v, np.float32), b, 16, 4, 16, 7)
        assert rc == 0 and api.range_verify(p, c, 16) == 1
        cs.append(c)
    rc, _, f = api.dlog(api.aggregate(np.stack(cs), 0), 1 << 16, 16, 16, 7)
    assert rc == 0 and (f == np.array([0.0, 3.75, -6.5], np.float32)).all()


def test_full_size_round_trip_cifar_lenet5(api, oracle):
    """BASELINE.json configs[1]: 62 006 params, 16-bit range, 64 chunks.  Too big for the oracle prover in seconds, so:
    prove on GPU -> verify on GPU; commitments equal the (cheap) oracle commitments; every one of the 64 proofs verified by the oracle."""
    rng = np.random.default_rng(2)
    D = 62006
    mn, mx = oracle.clip_bounds(16, 16, 7)
    v = rng.uniform(mn, mx, D).astype(np.float32)
    bl = api.rnd_scalar_vec(b"\x50" * 32, D)
    rc, p, c = api.range_prove(v, bl, 16, 64, 16, 7, b"\x51" * 32)
    assert rc == 0 and p.shape == (64, 32 * (9 + 2 * 14))
    assert api.range_verify(p, c, 16, b"\x52" * 32) == 1
    assert oracle.range_verify(p, c, 16, b"\x52" * 32) == 1          # ALL 64 GPU proofs accepted by the reference-equivalent verifier (chunk by chunk)
    assert (c[:2000] == oracle.commit_f32(v[:2000], bl[:2000], 16, 7)).all()
    bad = c.copy(); bad[40000] = c[40001]
    assert api.range_verify(p, bad, 16, b"\x52" * 32) == 0
    # determinism: same seed -> same bytes
    rc, p2, c2 = api.range_prove(v, bl, 16, 64, 16, 7, b"\x51" * 32)
    assert (p2 == p).all() and (c2 == c).all()


def test_compressed_rand_proof_parity_and_full_size(api, oracle):
    """compressed_rand_proof: byte parity with the oracle at a size it finishes quickly, then configs[2]'s 50 000 pairs on the
    GPU alone (prove -> verify, tamper rejection) -- the verifier is one 2 x 50 000-term MSM sharing its challenge-power scalars."""
    rng = np.random.default_rng(31)
    D = 700
    v = rng.uniform(-3, 3, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x62" * 32, D); seed = bytes([4] * 32)
    rc_o, pf_o, pairs_o = oracle.crp_prove(v, None, bl, 16, 7, seed)
    rc, pf, pairs = api.crp_prove(v, None, bl, 16, 7, seed)
    assert rc == rc_o == 0 and (pf == pf_o).all() and (pairs == pairs_o).all()
    assert api.crp_verify(pf, pairs) == 1 and oracle.crp_verify(pf, pairs) == 1
    D = 50000
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = api.rnd_scalar_vec(b"\x63" * 32, D)
    L_ = api.commit(v, bl, 32, 7)
    rc, pf, pairs = api.crp_prove(v, L_, bl, 32, 7, seed)                 # prove_existing, as the service does (params.rs:729-735)
    assert rc == 0 and (pairs[:, :32] == L_).all()
    assert api.crp_verify(pf, pairs) == 1
    bad = pairs.copy(); bad[D - 1, 32:] = pairs[0, 32:]
    assert api.crp_verify(pf, bad) == 0
    badp = pf.copy(); badp[97] ^= 1
    assert api.crp_verify(badp, pairs) in (0, -1)
    assert api.crp_prove(np.zeros(900001, np.float32), None, np.zeros((900001, 32), np.uint8), 16, 7, seed)[0] == -6


def test_unoptimised_encodings_whole_messages(api, oracle):
    """EncParamsRange / EncParamsL2 end to end through the C ABI: byte parity with the oracle's pieces at a small size, then configs[0]'s
    5 000 parameters on the GPU alone (encrypt -> verify, probabilistic checking, tamper rejection)."""
    rng = np.random.default_rng(35)
    D, P, seed = 40, 4, bytes([14] * 32)
    v = (rng.integers(-100, 100, D) / 128).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x6d" * 32, D)
    rc, msg = api.enc_range_encrypt(v, bl, 8, P, 1.0, 16, 7, seed)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 16, 7, seed)
    rc_r, pf_o, pairs_o = oracle.rand_prove(v, c_o, bl, 16, 7, seed)
    assert rc == rc_o == rc_r == 0 and (msg["range_proof"] == p_o).all() and (msg["rand_proof"] == pf_o).all() and (msg["enc_values"] == pairs_o).all()
    rc, m3 = api.enc_l2_encrypt(v, bl, 8, P, 32, 32, 7, seed)
    rnd = oracle.rnd_scalar_vec(oracle.derive_key(seed, 7, 1), D)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 32, 7, seed)
    rc_s, sumproof_o, _ = oracle.l2_prove(v, rnd, 32, 32, 7, seed)
    rc_q, sp_o, sc_o = oracle.square_rand_prove(v, c_o, bl, rnd, 32, 7, seed)
    assert rc == rc_o == rc_s == rc_q == 0
    assert (m3["range_proof"] == p_o).all() and (m3["square_range_proof"] == sumproof_o).all() and (m3["square_proof"] == sp_o).all() and (m3["enc_values"] == sc_o).all()
    D = 5000
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = api.rnd_scalar_vec(b"\x6e" * 32, D)
    rc, msg = api.enc_range_encrypt(v, bl, 8, 64, 1.0, 16, 7, seed)
    assert rc == 0 and api.enc_range_verify(msg, 1.0, seed) == 1
    bad = dict(msg); bad["enc_values"] = msg["enc_values"].copy(); bad["enc_values"][D - 1, 32:] = msg["enc_values"][0, 32:]
    assert api.enc_range_verify(bad, 1.0, seed) == 0
    rc, part = api.enc_range_encrypt(v, bl, 8, 64, 0.25, 16, 7, seed)
    assert rc == 0 and api.enc_range_verify(part, 0.25, seed) == 1
    rc, m3 = api.enc_l2_encrypt(v, bl, 8, 64, 32, 32, 7, seed)
    assert rc == 0 and api.enc_l2_verify(m3, seed) == 1
    bad = dict(m3); bad["enc_values"] = m3["enc_values"].copy(); bad["enc_values"][7, 64:] = m3["enc_values"][8, 64:]
    assert api.enc_l2_verify(bad, seed) == 0


def test_every_table_radix_gives_the_same_bytes(api, oracle):
    """The generator-table radix is chosen by free memory (2^11 on an empty B200): force 8, 9, 10 and no tables at all and compare
    proofs with the oracle byte for byte; the verifier accepts them at every radix."""
    rng = np.random.default_rng(77)
    D, rb, P, nb = 700, 16, 8, 16
    mn, mx = oracle.clip_bounds(rb, nb, 7)
    v = rng.uniform(mn, mx, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x70" * 32, D); seed = bytes([21] * 32)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, rb, P, nb, 7, seed)
    assert rc_o == 0
    try:
        for bits, use_rt in [(8, 1), (9, 1), (10, 1), (11, 1), (11, 0)]:
            api.set_option("rt_bits", bits); api.set_option("use_rt", use_rt)
            rc, p, c = api.range_prove(v, bl, rb, P, nb, 7, seed)
            assert rc == 0 and (c == c_o).all() and (p == p_o).all(), (bits, use_rt)
            assert api.range_verify(p, c, rb, seed) == 1
    finally:
        api.set_option("use_rt", 1); api.set_option("rt_bits", 11)


def test_tail_cluster_sizes_and_entry_points_give_the_same_bytes(api, oracle):
    """k_ipp_tail runs as a thread-block cluster (1, 2, 4 or 8 blocks per chunk: the table sums are dealt over the blocks, the leader runs the serial
    part) and may start at half-size 32, 16, 8 ... : every combination must give the oracle's bytes, the chunk-group count as well."""
    rng = np.random.default_rng(79)
    D, rb, P, nb = 900, 16, 8, 16
    mn, mx = oracle.clip_bounds(rb, nb, 7)
    v = rng.uniform(mn, mx, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x73" * 32, D); seed = bytes([23] * 32)
    rc_o, p_o, c_o = oracle.range_prove(v, bl, rb, P, nb, 7, seed)
    assert rc_o == 0
    try:
        for ncta, tail_np, groups in [(1, 32, 3), (2, 32, 3), (4, 32, 1), (8, 32, 2), (2, 16, 3), (4, 4, 1), (2, 1, 2), (2, 0, 3)]:
            api.set_option("tail_ncta", ncta); api.set_option("tail_np", tail_np); api.set_option("groups", groups)
            rc, p, c = api.range_prove(v, bl, rb, P, nb, 7, seed)
            assert rc == 0 and (c == c_o).all() and (p == p_o).all(), (ncta, tail_np, groups)
            assert api.range_verify(p, c, rb, seed) == 1
        api.set_option("tail_ncta", 2); api.set_option("tail_np", 32); api.set_option("groups", 3)
        api.set_option("tail_batch_mb", 10)                                   # the tail's tables for one chunk at a time
        rc, p, c = api.range_prove(v, bl, rb, P, nb, 7, seed)
        assert rc == 0 and (c == c_o).all() and (p == p_o).all()
    finally:
        api.set_option("tail_ncta", 2); api.set_option("tail_np", 32); api.set_option("groups", 3); api.set_option("tail_batch_mb", 2048)


def test_rand_and_square_rand_proof_parity_and_full_size(api, oracle):
    """Per-element proofs of the un-optimised encodings (enc types 2 and 3): byte parity at 3 000 elements, then configs[0]'s 5 000 x 4
    on the GPU alone with existing commitments (as params.rs creates them), tamper and format rejection."""
    rng = np.random.default_rng(41)
    D = 3000
    v = (rng.integers(-300, 300, D) / 128).astype(np.float32); seed = bytes([6] * 32)
    r1 = oracle.rnd_scalar_vec(b"\x68" * 32, D); r2 = oracle.rnd_scalar_vec(b"\x69" * 32, D)
    rc_o, pf_o, pr_o = oracle.rand_prove(v, None, r1, 16, 7, seed)
    rc, pf, pr = api.rand_prove(v, None, r1, 16, 7, seed)
    assert rc == rc_o == 0 and (pf == pf_o).all() and (pr == pr_o).all()
    assert api.rand_verify(pf, pr) == 1 and oracle.rand_verify(pf, pr) == 1
    rc_o, sp_o, sc_o = oracle.square_rand_prove(v, None, r1, r2, 32, 7, seed)
    rc, sp, sc = api.square_rand_prove(v, None, r1, r2, 32, 7, seed)
    assert rc == rc_o == 0 and (sp == sp_o).all() and (sc == sc_o).all()
    assert api.square_rand_verify(sp, sc) == 1 and oracle.square_rand_verify(sp, sc) == 1
    D = 20000
    v = (rng.integers(-100, 100, D) / 128).astype(np.float32)
    r1 = api.rnd_scalar_vec(b"\x6a" * 32, D); r2 = api.rnd_scalar_vec(b"\x6b" * 32, D)
    L_ = api.commit(v, r1, 32, 7)
    rc, pf, pr = api.rand_prove(v, L_, r1, 32, 7, seed)
    assert rc == 0 and (pr[:, :32] == L_).all() and api.rand_verify(pf, pr) == 1
    bad = pr.copy(); bad[D - 1, 32:] = pr[0, 32:]
    assert api.rand_verify(pf, bad) == 0
    badp = pf.copy(); badp[D // 2, 64:96] = 0xff
    assert api.rand_verify(badp, pr) == -1
    rc, sp, sc = api.square_rand_prove(v, L_, r1, r2, 32, 7, seed)
    assert rc == 0 and (sc[:, :32] == L_).all() and api.square_rand_verify(sp, sc) == 1
    sq = api.commit(((v.astype(np.float64) * 128) ** 2).astype(np.float32), r2, 32, 0)                 # c_sq commits to m^2 under r2
    assert (sc[:, 64:] == sq).all()
    bad = sc.copy(); bad[7, 64:] = sc[8, 64:]
    assert api.square_rand_verify(sp, bad) == 0
    badp = sp.copy(); badp[3, :32] = 0xff
    assert api.square_rand_verify(badp, sc) == -1


@pytest.mark.parametrize("P", [64, 4])
def test_config0_mnist_5k_full_size_byte_parity(api, oracle, P):
    """BASELINE.json configs[0] at its real size (5 000 params, 8-bit, 1 client; P = 64 as in mnist_e2e.yml and P = 4 as in the reference's
    own bench): the oracle proves it in seconds, so the comparison is byte for byte on all proofs and commitments."""
    rng = np.random.default_rng(3)
    D = 5000
    mn, mx = oracle.clip_bounds(8, 16, 7)
    v = rng.uniform(mn, mx, D).astype(np.float32)
    bl = oracle.rnd_scalar_vec(b"\x53" * 32, D)
    seed = b"\x54" * 32
    rc_o, p_o, c_o = oracle.range_prove(v, bl, 8, P, 16, 7, seed)
    rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, seed)
    assert rc == rc_o == 0 and (c == c_o).all() and p.shape == p_o.shape and (p == p_o).all()
    assert api.range_verify(p, c, 8, seed) == 1 and oracle.range_verify(p, c, 8, seed) == 1


def test_config2_resnet18_intrinsic_50k_l2_pipeline(api, oracle):
    """BASELINE.json configs[2]: 50 000 params, L2 bound = per-element square proofs + ONE 32-bit range proof on the sum of squares, plus the
    8-bit L-inf range proofs.  Sum proof: byte parity with the oracle (it is O(D) scalar work there).  Square proofs: byte parity on a
    prefix, then full-size verification, homomorphic consistency (sum of the square commitments == the L2 commitment) and tamper rejection."""
    rng = np.random.default_rng(4)
    D = 50000
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32)               # SURVEY 8d: keeps the reference's f32 cross-check exact
    r1 = api.rnd_scalar_vec(b"\x55" * 32, D); r2 = api.rnd_scalar_vec(b"\x56" * 32, D); seed = b"\x57" * 32
    rc, pf, cm = api.l2_prove(v, r2, 32, 32, 7, seed)
    rc_o, pf_o, cm_o = oracle.l2_prove(v, r2, 32, 32, 7, seed)
    assert rc == rc_o == 0 and (pf == pf_o).all() and (np.asarray(cm) == np.asarray(cm_o)).all()
    assert api.l2_verify(pf, cm, 32, seed) == 1 and oracle.l2_verify(pf, cm, 32, seed) == 1
    cl = api.commit(v, r1, 32, 7)
    rc, sp, sc = api.square_prove(v, cl, r1, r2, 32, 7, seed)
    assert rc == 0 and api.square_verify(sp, sc) == 1
    k = 300
    rc_o, sp_o, sc_o = oracle.square_prove(v[:k], cl[:k], r1[:k], r2[:k], 32, 7, seed)
    assert rc_o == 0 and (sp[:k] == sp_o).all() and (sc[:k] == sc_o).all()
    # sum_i c_sq,i == commitment of the sum proof (same value sum x_i^2, same blinding sum r2_i): the link the server relies on (params.rs:81-124)
    agg = api.aggregate(sc[:, 32:].reshape(D, 1, 32).copy(), 0)            # D "clients" x 1 point: sums all square commitments
    assert (agg[0] == np.asarray(cm)).all()
    bad = sp.copy(); bad[D - 7, 64] ^= 1
    assert api.square_verify(bad, sc) in (0, -1)
    mn, mx = oracle.clip_bounds(8, 32, 7)
    assert mn <= v.min() and v.max() <= mx
    rc, p, c = api.range_prove(v, r1, 8, 64, 32, 7, seed)
    assert rc == 0 and api.range_verify(p, c, 8, seed) == 1 and (c == cl).all()


def test_config3_resnet18_full_one_gpu_share_of_eight(api, oracle):
    """BASELINE.json configs[3]: 11 689 512 params, 8-bit, 64 chunks of 2^18 values sharded over 8 GPUs.  This is the work of ONE of the
    eight ranks (8 chunks = 2^21 values, 2^24 bit positions, no generator tables at this size: bucket MSMs and folds), through the
    shard entry points; a spot chunk of the commitments is compared with the oracle and a tampered shard is rejected."""
    from importlib import import_module
    D, P = 11689512, 64
    m = (1 << 24) // P
    rank, world = 5, 8
    c0, n_chunks = rank * (P // world), P // world
    e0, e1 = c0 * m, min(D, (c0 + n_chunks) * m)
    rng = np.random.default_rng(6)
    v = rng.uniform(-0.99, 0.99, e1 - e0).astype(np.float32)
    bl = api.rnd_scalar_vec(b"\x58" * 32, e1 - e0)
    seed = b"\x59" * 32
    rc, p, c = api.range_prove_shard(v, bl, m, c0, n_chunks, 8, 16, 7, seed)
    assert rc == 0 and p.shape == (n_chunks, 32 * (9 + 2 * 21)) and c.shape == (e1 - e0, 32)
    assert api.range_verify_shard(p, c, m, c0, 8, seed) == 1
    assert (c[:1000] == oracle.commit_f32(v[:1000], bl[:1000], 16, 7)).all()
    # one whole chunk (2^18 values, N = 2^21: the no-table path -- bucket MSMs and generator folds) through the oracle's verifier
    assert oracle.range_verify(p[2:3], c[2 * m:3 * m], 8, seed) == 1
    bad = c.copy(); bad[123456] = c[123457]
    assert api.range_verify_shard(p, bad, m, c0, 8, seed) == 0


def test_config4_server_batch_verify_aggregate_decrypt(api, oracle):
    """BASELINE.json configs[4] (server side) with all 48 clients: verify every client's proofs, aggregate the ElGamal halves with
    cancelling blindings, decrypt with the 2^16 table; the decrypted aggregate must equal the exact sum of the quantised inputs."""
    rng = np.random.default_rng(7)
    n_clients, D = 48, 50000
    vs = [(rng.integers(-24, 25, D) / 128).astype(np.float32) for _ in range(n_clients)]
    bls = [np.frombuffer(api.rnd_scalar_vec(bytes([0x40 + k]) * 32, D).tobytes(), np.uint8).reshape(D, 32).copy() for k in range(n_clients - 1)]
    # last client's blindings cancel the others (pedersen_ops.rs:110-122): r_last = -sum r_k mod l
    Lmod = L
    tot = np.zeros(D, dtype=object)
    for b in bls:
        tot = (tot + np.array([int.from_bytes(row.tobytes(), "little") for row in b], dtype=object)) % Lmod
    last = np.frombuffer(b"".join(int((Lmod - t) % Lmod).to_bytes(32, "little") for t in tot), np.uint8).reshape(D, 32).copy()
    bls.append(last)
    Ls, Rs = [], []
    for k in range(n_clients):
        seed = bytes([0x80 + k]) * 32
        rc, p, c = api.range_prove(vs[k], bls[k], 8, 64, 32, 7, seed)
        assert rc == 0 and api.range_verify(p, c, 8, seed) == 1
        rc, pf, pairs = api.crp_prove(vs[k], c, bls[k], 32, 7, seed)
        assert rc == 0 and api.crp_verify(pf, pairs) == 1
        Ls.append(pairs[:, :32].copy()); Rs.append(pairs[:, 32:].copy())
    aggL = api.aggregate(np.stack(Ls), 1); aggR = api.aggregate(np.stack(Rs), 1)            # accumulators start at (B, B) (el_gamal.rs:83-88)
    B = np.frombuffer(oracle.basepoint(), np.uint8)
    assert (aggR == B).all()                                                                   # blindings cancelled: right halves are the unity element
    rc, s, f = api.dlog(api.aggregate(np.stack(Ls), 0), 1 << 16, 16, 32, 7)
    assert rc == 0
    assert (f == np.sum(np.stack(vs), axis=0, dtype=np.float64).astype(np.float32)).all()


def test_optimised_encodings_server_path_full_size(api, oracle):
    """params.rs EncParamsL2Compressed / EncParamsRangeCompressed at configs[2] size (50 000 params): encrypt on the GPU, verify on the GPU from
    the wire fields, tamper rejection; pieces spot-checked against the oracle; several clients aggregated and decrypted (configs[4] in small)."""
    rng = np.random.default_rng(41)
    D, P = 50000, 64
    msgs, vs = [], []
    n_clients = 3
    bls = [np.frombuffer(api.rnd_scalar_vec(bytes([0x90 + k]) * 32, D).tobytes(), np.uint8).reshape(D, 32).copy() for k in range(n_clients - 1)]
    tot = np.zeros(D, dtype=object)
    for b in bls:
        tot = (tot + np.array([int.from_bytes(row.tobytes(), "little") for row in b], dtype=object)) % L
    bls.append(np.frombuffer(b"".join(int((L - t) % L).to_bytes(32, "little") for t in tot), np.uint8).reshape(D, 32).copy())
    for k in range(n_clients):
        v = (rng.integers(-24, 25, D) / 128).astype(np.float32); vs.append(v)
        seed = bytes([0xa0 + k]) * 32
        rc, m = api.enc_l2_compressed_encrypt(v, bls[k], 8, P, 32, 32, 7, seed)
        assert rc == 0 and api.enc_l2_compressed_verify(m, seed) == 1
        assert api.crp_verify(m["rand_proof"], m["enc_values"][:, :64].copy()) == 1
        msgs.append(m)
    m = msgs[0]
    assert (m["enc_values"][:500, :32] == oracle.commit_f32(vs[0][:500], bls[0][:500], 32, 7)).all()
    bad = dict(m); bad["enc_values"] = m["enc_values"].copy(); bad["enc_values"][D - 3, 64:] = m["enc_values"][0, 64:]
    assert api.enc_l2_compressed_verify(bad, bytes([0xa0]) * 32) == 0
    bad = dict(m); bad["square_range_proof"] = m["square_range_proof"].copy(); bad["square_range_proof"][33] ^= 2
    assert api.enc_l2_compressed_verify(bad, bytes([0xa0]) * 32) == 0
    # aggregate the ElGamal halves of all clients and decrypt
    aggL = api.aggregate(np.stack([x["enc_values"][:, :32].copy() for x in msgs]), 0)
    aggR = api.aggregate(np.stack([x["enc_values"][:, 32:64].copy() for x in msgs]), 1)
    assert (aggR == np.frombuffer(oracle.basepoint(), np.uint8)).all()
    rc, s, f = api.dlog(aggL, 1 << 16, 16, 32, 7)
    assert rc == 0 and (f == np.sum(np.stack(vs), axis=0, dtype=np.float64).astype(np.float32)).all()
    # range-compressed encoding with probabilistic checking (check_percentage < 1 verifies a prefix, params.rs:243-249)
    v = rng.uniform(-0.99, 0.99, 5000).astype(np.float32); bl = api.rnd_scalar_vec(b"\x99" * 32, 5000); seed = b"\x9a" * 32
    rc, m = api.enc_range_compressed_encrypt(v, bl, 8, 64, 16, 7, seed)
    assert rc == 0 and api.enc_range_compressed_verify(m, 1.0, seed) == 1
    bad = dict(m); bad["rand_proof"] = m["rand_proof"].copy(); bad["rand_proof"][70] ^= 1
    assert api.enc_range_compressed_verify(bad, 1.0, seed) == 0


def test_clip_bounds_and_clipping_match_oracle(api, oracle):
    """conversion32::get_clip_bounds / get_l2_clip_bounds (conversion32.rs:56-64) and range_proof_vec::clip_f32_to_range_vec
    (range_proof_vec/mod.rs:104-111) through the C ABI, for every fixed-point feature combination the experiments build."""
    rng = np.random.default_rng(12)
    v = np.concatenate([rng.uniform(-70000, 70000, 5000), rng.uniform(-2, 2, 5000), [0.0, -0.0, 0.9921875, -0.9921875, 1.0, -1.0, 255.9921875, 256.0, 3.4e38, -3.4e38]]).astype(np.float32)
    for nb, fr in [(8, 7), (16, 7), (32, 7), (64, 7), (16, 0), (32, 12), (16, 10)]:
        for rb in [1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64]:
            if rb > nb:
                continue
            assert api.clip_bounds(rb, nb, fr) == oracle.clip_bounds(rb, nb, fr), (rb, nb, fr)
            assert api.l2_clip_bound(rb, nb, fr) == oracle.l2_clip_bound(rb, nb, fr), (rb, nb, fr)
            a = api.clip_f32_to_range_vec(v, rb, nb, fr); o = oracle.clip_f32_to_range_vec(v, rb, nb, fr)
            assert a.dtype == np.float32 and (a.view(np.uint32) == o.view(np.uint32)).all(), (rb, nb, fr)
    # the literal values of the reference's own tests: 8 bits at frac 7 -> +-(2^7 - 1)/2^7 (conversion32.rs:56-60)
    assert api.clip_bounds(8, 16, 7) == (-0.9921875, 0.9921875)
    # a clipped vector is always provable, an unclipped one is not (range_proof_vec/mod.rs:22-29)
    z = np.zeros((8, 32), np.uint8); x = np.array([5.0, -5.0, 0.5, 0, 0, 0, 0, 0], np.float32)
    assert api.range_prove(x, z, 8, 4, 16, 7, b"\x01" * 32)[0] == 2
    assert api.range_prove(api.clip_f32_to_range_vec(x, 8, 16, 7), z, 8, 4, 16, 7, b"\x01" * 32)[0] == 0


def test_device_transcript_absorb_matches_sequential(api):
    """ts_kernels.cuh k_ts_absorbV on the GPU (warp-cooperative STROBE absorb + Keccak-f with one lane per word) against the sequential Merlin
    code, for every alignment of the 41-byte records against the 166-byte rate and for the chunk sizes of the BASELINE configs."""
    rng = np.random.default_rng(77)
    for m in list(range(1, 170)) + [331, 1024, 2048, 16384]:
        V = rng.integers(0, 256, (m, 32), dtype=np.uint8)
        assert api.debug_ts_absorb(V, 8 if m % 2 else 16, m % 2) == 0, m


def test_verifier_weights_are_bound_to_every_proof_of_the_call(api, oracle):
    """ADVICE r01 (high): with weights that depended on the seed alone, a prover who knew the seed could make the errors of two chunks cancel.
    Now (c_i, rho_i) are Fiat-Shamir outputs over the seed and ALL proofs / commitments of the call: changing any chunk changes every weight."""
    rng = np.random.default_rng(78)
    D, P = 300, 8
    v = rng.uniform(-0.9, 0.9, D).astype(np.float32); bl = oracle.rnd_scalar_vec(b"\x71" * 32, D)
    rc, p, c = api.range_prove(v, bl, 8, P, 16, 7, b"\x72" * 32)
    seed = bytes(32)
    ok, w0 = api.debug_verify_weights(p, c, 8, seed)
    assert ok == 1 and len({w0[k, i].tobytes() for k in range(2) for i in range(P)}) == 2 * P
    assert (api.debug_verify_weights(p, c, 8, seed)[1] == w0).all()
    w2 = api.debug_verify_weights(p, c, 8, b"\x01" * 32)[1]
    assert all((w2[k, i] != w0[k, i]).any() for k in range(2) for i in range(P))
    for what in ("proof_point", "proof_scalar", "commitment"):
        pp, cc = p.copy(), c.copy()
        if what == "proof_point": pp[P - 1, 224 + 3] ^= 1
        elif what == "proof_scalar": pp[P - 1, -32] ^= 1
        else: cc[D - 1] = c[0]
        ok, w = api.debug_verify_weights(pp, cc, 8, seed)
        assert ok in (0, 1)
        assert all((w[k, i] != w0[k, i]).any() for k in range(2) for i in range(P)), what


def test_l2_compressed_message_with_undecodable_point_is_refused(api, oracle):
    """VERDICT r01 a17 / ADVICE (medium): c.R of every 96-byte record is validated like the reference's from_bytes does
    (square_rand_proof/pedersen.rs:33-45, rand_proof/el_gamal.rs:112-123), at configs[2] size."""
    rng = np.random.default_rng(79)
    D, P, seed = 50000, 64, bytes([12] * 32)
    v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = api.rnd_scalar_vec(b"\x73" * 32, D)
    rc, m = api.enc_l2_compressed_encrypt(v, bl, 8, P, 32, 32, 7, seed)
    assert rc == 0 and api.enc_l2_compressed_verify(m, seed) == 1
    for col, row in ((32, D - 2), (0, 17), (64, 31337)):
        bad = dict(m); bad["enc_values"] = m["enc_values"].copy(); bad["enc_values"][row, col:col + 32] = 0xff
        assert api.enc_l2_compressed_verify(bad, seed) == -4, col
    ok = dict(m); ok["enc_values"] = m["enc_values"].copy(); ok["enc_values"][1, 32:64] = np.frombuffer(oracle.basepoint(), np.uint8)
    assert api.enc_l2_compressed_verify(ok, seed) == 1          # a valid but different R: this arm does not check the rand proof (params.rs:257-289)


def test_concurrent_callers_share_one_context(api, oracle):      # VERDICT r01 item 5: a threaded test with 8 callers on one GPU
    """rofl_service calls verify() for many clients at once from a rayon pool (server.rs:516-522,666) and proves several clients per process
    (bin/basic_client.rs:136-161): concurrent callers of ONE context run on separate lanes (streams) and share the cached tables; every
    caller must get exactly the bytes / verdicts of a lone caller."""
    import threading
    rng = np.random.default_rng(80)
    jobs = []
    for k in range(8):
        D = [5000, 800, 62006, 1600, 70, 4000, 12000, 9][k]; P = [64, 4, 64, 16, 2, 64, 32, 1][k]
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


def test_config4_server_batch_path_48_clients(api, oracle):
    """BASELINE.json configs[4] through the batch entry points: 48 EncL2Compressed messages of 50 000 parameters verified in ONE call
    (rofl_enc_l2_compressed_verify_batch: one random linear combination over 48 x 64 chunks, one generator MSM), then aggregated and decrypted;
    a tampered client is named, the others still pass; the verdicts equal the per-client calls' (server.rs:516-522,666-667, params.rs:81-147,257-290)."""
    rng = np.random.default_rng(83)
    K, D, P = 48, 50000, 64
    vs_, msgs = [], []
    bls = [np.frombuffer(api.rnd_scalar_vec(bytes([0x10 + k]) * 32, D).tobytes(), np.uint8).reshape(D, 32).copy() for k in range(K - 1)]
    tot = np.zeros(D, dtype=object)
    for b in bls:
        tot = (tot + np.array([int.from_bytes(row.tobytes(), "little") for row in b], dtype=object)) % L
    bls.append(np.frombuffer(b"".join(int((L - t) % L).to_bytes(32, "little") for t in tot), np.uint8).reshape(D, 32).copy())
    for k in range(K):
        v = (rng.integers(-24, 25, D) / 128).astype(np.float32); vs_.append(v)
        rc, m = api.enc_l2_compressed_encrypt(v, bls[k], 8, P, 32, 32, 7, bytes([0x50 + k]) * 32)
        assert rc == 0
        msgs.append(m)
    seed = b"\x66" * 32
    assert api.enc_l2_compressed_verify_batch(msgs, seed).tolist() == [1] * K
    proofs = np.stack([m["range_proof"] for m in msgs]); commits = np.stack([m["enc_values"][:, :32] for m in msgs])
    assert api.range_verify_batch(proofs, commits, 8, seed).tolist() == [1] * K
    tam = [dict(m) for m in msgs]; tam[17]["enc_values"] = msgs[17]["enc_values"].copy(); tam[17]["enc_values"][40000, :32] = msgs[17]["enc_values"][40001, :32]
    tam[30]["square_proof"] = msgs[30]["square_proof"].copy(); tam[30]["square_proof"][123, 70] ^= 1
    got = api.enc_l2_compressed_verify_batch(tam, seed).tolist()
    assert got[17] == 0 and got[30] in (0, -1) and all(g == 1 for i, g in enumerate(got) if i not in (17, 30))
    assert api.enc_l2_compressed_verify(tam[17], seed) == 0 and api.enc_l2_compressed_verify(msgs[3], seed) == 1
    aggL = api.aggregate(np.stack([m["enc_values"][:, :32].copy() for m in msgs]), 0)
    aggR = api.aggregate(np.stack([m["enc_values"][:, 32:64].copy() for m in msgs]), 1)
    assert (aggR == np.frombuffer(oracle.basepoint(), np.uint8)).all()
    rc, s, f = api.dlog(aggL, 1 << 16, 16, 32, 7)
    assert rc == 0 and (f == np.sum(np.stack(vs_), axis=0, dtype=np.float64).astype(np.float32)).all()
