"""Server-side batch verification of the L-inf message of rofl_service (EncParamsRangeCompressed, params.rs:236-256) and of its building
block, the compressed rand proof (compressed_rand_proof/mod.rs:149-158): rofl_enc_range_compressed_verify_batch and rofl_crp_verify_batch
check all K clients of a round in one random linear combination and, when it fails, client by client -- every verdict must be exactly that
of the per-client call.  The emulation tests run the product kernels and engine on CPU threads (tiny sizes); the GPU tests run the
B200 library at round sizes."""
import ctypes as C
import importlib.util
import os
import sys
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NB, FR, RB = 16, 7, 8                     # fixed point 16/7, 8-bit range proofs at the tiny sizes
ROFL_ERR_ARGS = -2


@pytest.fixture(scope="module")
def api():
    d = os.path.join(HERE, "hostsim")
    locked_make(d, "libemul.so", env={"CXX": "g++"})
    spec = importlib.util.spec_from_file_location("rofl_ffi", os.path.join(ROOT, "rofl-project-code_b200", "_ffi.py"))
    ffi = importlib.util.module_from_spec(spec); spec.loader.exec_module(ffi)
    a = ffi.Api(C.CDLL(os.path.join(d, "libemul.so")))
    yield a
    a.close()


@pytest.fixture(scope="module")
def gpu_api():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    return g.load_package().context(0)


def llroundf(D, p):
    return int(np.floor(float(np.float32(np.float32(D) * np.float32(p))) + 0.5))


def make_msgs(api, K, D, P, rng_bits, tag, n_bits=NB):
    """K honest messages from rofl_enc_range_compressed_encrypt"""
    rng = np.random.default_rng(tag)
    msgs = []
    for k in range(K):
        v = rng.uniform(-0.99, 0.99, D).astype(np.float32)
        bl = api.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D)
        rc, m = api.enc_range_compressed_encrypt(v, bl, rng_bits, P, n_bits, FR, bytes([(0x80 + tag + k) & 0xff]) * 32)
        assert rc == 0
        msgs.append(m)
    return msgs


def copy_msgs(msgs):
    return [{f: (x.copy() if isinstance(x, np.ndarray) else x) for f, x in m.items()} for m in msgs]


def flipped_point(oracle, pt, want_valid):
    """pt with one bit flipped, chosen so that the result does (want_valid) or does not decode"""
    for byte in range(31):
        for bit in range(8):
            x = pt.copy(); x[byte] ^= 1 << bit
            if oracle.point_valid(x) == want_valid:
                return x
    raise AssertionError("no such flip")


def scalar_plus_one(api, z):
    one = np.zeros(32, np.uint8); one[0] = 1
    return api.scalar_add(z.reshape(1, 32), one.reshape(1, 32))[0]


def tamper_cases(api, oracle, msgs):
    """(name, tampered copy of the round, indices of the tampered clients)"""
    t = 1
    out = []
    for half, lo in (("L", 0), ("R", 32)):
        for valid in (False, True):
            ms = copy_msgs(msgs); i = ms[t]["enc_values"].shape[0] // 2
            ms[t]["enc_values"][i, lo:lo + 32] = flipped_point(oracle, msgs[t]["enc_values"][i, lo:lo + 32], valid)
            out.append((f"{half} half, flipped bit, decodes={valid}", ms, [t]))
    for name, lo in (("C'_L", 0), ("C'_R", 32)):
        ms = copy_msgs(msgs); ms[t]["rand_proof"][lo:lo + 32] = np.frombuffer(oracle.point_add(msgs[t]["rand_proof"][lo:lo + 32], oracle.basepoint()), np.uint8)
        out.append((f"{name} + B", ms, [t]))
        ms = copy_msgs(msgs); ms[t]["rand_proof"][lo:lo + 32] = flipped_point(oracle, msgs[t]["rand_proof"][lo:lo + 32], False)
        out.append((f"{name} undecodable", ms, [t]))
    for name, lo in (("z_m", 64), ("z_r", 96)):
        ms = copy_msgs(msgs); ms[t]["rand_proof"][lo:lo + 32] = scalar_plus_one(api, msgs[t]["rand_proof"][lo:lo + 32])
        out.append((f"wrong {name}", ms, [t]))
        ms = copy_msgs(msgs); ms[t]["rand_proof"][lo:lo + 32] = 0xff
        out.append((f"non-canonical {name}", ms, [t]))
    ms = copy_msgs(msgs); ms[t]["range_proof"][0, 70] ^= 1
    out.append(("range proof byte", ms, [t]))
    ms = copy_msgs(msgs); ms[0]["rand_proof"], ms[t]["rand_proof"] = msgs[t]["rand_proof"].copy(), msgs[0]["rand_proof"].copy()
    out.append(("rand proofs of two clients swapped", ms, [0, t]))
    return out


def check_round(api, msgs, seed, oracle=None, cp=1.0):
    """batch verdicts == single-call verdicts (and the oracle's, when given), for the messages and for their rand proofs alone"""
    got = api.enc_range_compressed_verify_batch(msgs, cp, seed).tolist()
    single = [api.enc_range_compressed_verify(m, cp, seed) for m in msgs]
    assert got == single, (got, single)
    crp = api.crp_verify_batch(np.stack([m["rand_proof"] for m in msgs]), np.stack([m["enc_values"] for m in msgs]), seed).tolist()
    crp_single = [api.crp_verify(m["rand_proof"], m["enc_values"]) for m in msgs]
    assert crp == crp_single, (crp, crp_single)
    # the combined check itself holds exactly when every rand proof is valid (else the verdicts above came from the per-client re-checks)
    if crp and msgs[0]["enc_values"].shape[0]:
        assert api.debug_crp_rlc(np.stack([m["rand_proof"] for m in msgs]), np.stack([m["enc_values"] for m in msgs]), seed) == int(all(x == 1 for x in crp))
    if oracle is not None:
        num = llroundf(msgs[0]["enc_values"].shape[0], cp)
        assert crp == [oracle.crp_verify(m["rand_proof"], m["enc_values"]) for m in msgs]
        want = [int(c == 1 and oracle.range_verify(m["range_proof"], m["enc_values"][:num, :32].copy(), m["range_bits"], seed) == 1) for c, m in zip(crp, msgs)]
        assert got == want, (got, want)
    return got, crp


def run_tamper_matrix(api, oracle, msgs, seed, with_oracle):
    for name, ms, bad in tamper_cases(api, oracle, msgs):
        got, crp = check_round(api, ms, seed, oracle if with_oracle else None)
        assert all(got[k] == 1 for k in range(len(ms)) if k not in bad), (name, got)
        assert all(got[k] == 0 for k in bad), (name, got)
        if name.startswith("non-canonical"):
            assert crp[bad[0]] == -1, (name, crp)
        elif name == "range proof byte":
            assert crp == [1] * len(ms), (name, crp)
        else:
            assert all(crp[k] in (0, -1) for k in bad), (name, crp)
    # the same honest message twice in one batch
    twice = [msgs[0], msgs[1], msgs[1]] + list(msgs[2:])
    got, crp = check_round(api, twice, seed)
    assert got == [1] * len(twice) and crp == [1] * len(twice)


def weights_are_not_uniform(api, oracle, msgs, seed):
    """C'_L + B on one client and C'_L - B on another: equal weights would cancel the two changes"""
    ms = copy_msgs(msgs)
    ms[0]["rand_proof"][:32] = np.frombuffer(oracle.point_add(msgs[0]["rand_proof"][:32], oracle.basepoint()), np.uint8)
    ms[1]["rand_proof"][:32] = np.frombuffer(oracle.point_sub(msgs[1]["rand_proof"][:32], oracle.basepoint()), np.uint8)
    got, crp = check_round(api, ms, seed)
    assert got[:2] == [0, 0] and crp[:2] == [0, 0] and got[2:] == [1] * (len(ms) - 2)


# ---- emulation (CPU) -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,D,P", [(1, 1, 1), (2, 5, 2), (3, 6, 2), (4, 20, 2)])
def test_honest_round_all_accepted(api, oracle, K, D, P):
    msgs = make_msgs(api, K, D, P, RB, 10 * K + D)
    got, crp = check_round(api, msgs, b"\x21" * 32, oracle)
    assert got == [1] * K and crp == [1] * K


def test_tamper_matrix(api, oracle):
    msgs = make_msgs(api, 3, 6, 2, RB, 3)
    run_tamper_matrix(api, oracle, msgs, b"\x22" * 32, with_oracle=True)


def test_weights_are_not_uniform(api, oracle):
    weights_are_not_uniform(api, oracle, make_msgs(api, 3, 5, 1, RB, 4), b"\x23" * 32)


@pytest.mark.parametrize("D,cp", [(20, 0.5), (20, 0.25), (7, 0.5)])
def test_prefix_mode(api, oracle, D, cp):
    """check_percentage < 1: the rand proof covers all D pairs, the range proofs the first round(D * cp) L halves (params.rs:243-249).
    The encrypt call has no prefix mode, so the messages are put together from crp_prove (L = commit) and range_prove over the prefix."""
    num = llroundf(D, cp)
    rng = np.random.default_rng(D)
    mn, mx = oracle.clip_bounds(RB, NB, FR)
    msgs = []
    for k in range(3):
        v = rng.uniform(mn, mx, D).astype(np.float32); bl = oracle.rnd_scalar_vec(bytes([0x50 + k]) * 32, D); seed = bytes([0x60 + k]) * 32
        rc, proof, pairs = api.crp_prove(v, None, bl, NB, FR, seed); assert rc == 0
        rc, rp, commits = api.range_prove(v[:num], bl[:num], RB, 2, NB, FR, seed); assert rc == 0
        assert (commits == pairs[:num, :32]).all()
        msgs.append(dict(enc_values=pairs, rand_proof=proof, range_proof=rp, range_bits=RB))
    vs = b"\x24" * 32
    got, _ = check_round(api, msgs, vs, oracle, cp)
    assert got == [1, 1, 1]
    ms = copy_msgs(msgs); ms[2]["enc_values"][num - 1, :32] = msgs[2]["enc_values"][0, :32]      # inside the prefix: both parts reject
    assert check_round(api, ms, vs, oracle, cp)[0] == [1, 1, 0]
    ms = copy_msgs(msgs); ms[0]["range_proof"][0, 40] ^= 1
    assert check_round(api, ms, vs, oracle, cp)[0] == [0, 1, 1]
    for bad_cp in (0.01, 1.5):                          # num == 0 and num > D: every message is rejected, as by the single call
        assert api.enc_range_compressed_verify_batch(msgs, bad_cp, vs).tolist() == [0, 0, 0] == [api.enc_range_compressed_verify(m, bad_cp, vs) for m in msgs]


def test_argument_edges(api):
    seed = np.frombuffer(b"\x25" * 32, np.uint8)
    ok = np.full(2, 7, np.int32)
    # more than 900 000 pairs: -6 (rand proofs) / 0 (messages) for every client, before anything is copied
    D = 900001
    pairs = np.zeros((2, D, 64), np.uint8); proofs = np.zeros((2, 128), np.uint8)
    assert api.crp_verify_batch(proofs, pairs, seed).tolist() == [-6, -6]
    del pairs
    rp = np.zeros((2, 1, 32 * 13), np.uint8)
    L = api.lib
    assert L.rofl_enc_range_compressed_verify_batch(api.h, 2, proofs.ctypes.data, D, proofs.ctypes.data, rp.ctypes.data, rp.shape[2], 1, 16, 1.0, seed.ctypes.data, ok.ctypes.data) == 0
    assert ok.tolist() == [0, 0]
    # K = 0: nothing is written
    ok[:] = 7
    assert L.rofl_crp_verify_batch(api.h, 0, None, None, 5, seed.ctypes.data, ok.ctypes.data) == 0
    assert L.rofl_enc_range_compressed_verify_batch(api.h, 0, None, 5, None, None, 32 * 13, 1, 16, 1.0, seed.ctypes.data, ok.ctypes.data) == 0
    assert ok.tolist() == [7, 7]
    # null out_ok, D == 0, n_proofs == 0
    assert L.rofl_enc_range_compressed_verify_batch(api.h, 2, proofs.ctypes.data, 5, proofs.ctypes.data, rp.ctypes.data, rp.shape[2], 1, 16, 1.0, seed.ctypes.data, None) == ROFL_ERR_ARGS
    assert L.rofl_enc_range_compressed_verify_batch(api.h, 2, proofs.ctypes.data, 0, proofs.ctypes.data, rp.ctypes.data, rp.shape[2], 1, 16, 1.0, seed.ctypes.data, ok.ctypes.data) == ROFL_ERR_ARGS
    assert L.rofl_enc_range_compressed_verify_batch(api.h, 2, proofs.ctypes.data, 5, proofs.ctypes.data, rp.ctypes.data, rp.shape[2], 0, 16, 1.0, seed.ctypes.data, ok.ctypes.data) == ROFL_ERR_ARGS
    assert L.rofl_crp_verify_batch(api.h, 2, proofs.ctypes.data, None, 5, seed.ctypes.data, None) == ROFL_ERR_ARGS
    assert ok.tolist() == [7, 7]


def test_rand_proofs_without_pairs(api, oracle):
    """D = 0 (the per-client path): C' alone must equal z_m B + z_r H | z_r B"""
    rc, proof, _ = api.crp_prove(np.zeros(0, np.float32), None, np.zeros((0, 32), np.uint8), NB, FR, b"\x26" * 32)
    assert rc == 0
    bad = proof.copy(); bad[64:96] = scalar_plus_one(api, proof[64:96])
    proofs = np.stack([proof, bad, proof])
    got = api.crp_verify_batch(proofs, np.zeros((3, 0, 64), np.uint8), b"\x27" * 32).tolist()
    assert got == [api.crp_verify(p, np.zeros((0, 64), np.uint8)) for p in proofs] == [1, 0, 1]


def test_single_lane(api, oracle):
    """the rand-proof transcripts run on helper threads that never take a lane: with one lane the call still returns"""
    msgs = make_msgs(api, 3, 4, 1, RB, 5)
    api.set_option("max_lanes", 1)
    try:
        got, crp = check_round(api, msgs, b"\x28" * 32)
        assert got == [1, 1, 1] and crp == [1, 1, 1]
    finally:
        api.set_option("max_lanes", 8)


# ---- B200 -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_tamper_matrix(gpu_api, oracle):
    msgs = make_msgs(gpu_api, 3, 2000, 4, RB, 6)
    run_tamper_matrix(gpu_api, oracle, msgs, b"\x31" * 32, with_oracle=False)
    weights_are_not_uniform(gpu_api, oracle, msgs, b"\x32" * 32)


@pytest.mark.gpu
def test_gpu_configs1_round_48_clients(gpu_api, oracle):
    """a configs[1]-shaped round: 48 clients x 62 006 values, 16-bit range proofs in 64 chunks, from rofl_enc_range_compressed_encrypt"""
    api = gpu_api
    msgs = make_msgs(api, 48, 62006, 64, 16, 7)
    seed = b"\x33" * 32
    assert api.enc_range_compressed_verify_batch(msgs, 1.0, seed).tolist() == [1] * 48
    ms = copy_msgs(msgs)
    ms[11]["enc_values"][30000, 32:] = msgs[11]["enc_values"][30001, 32:]          # an R half of another pair: the rand proof fails
    ms[40]["range_proof"][17, 100] ^= 1                                              # a range proof byte
    got = api.enc_range_compressed_verify_batch(ms, 1.0, seed).tolist()
    assert got[11] == 0 and got[40] == 0 and all(g == 1 for i, g in enumerate(got) if i not in (11, 40)), got
    assert [api.enc_range_compressed_verify(ms[k], 1.0, seed) for k in (11, 40, 0)] == [0, 0, 1]


@pytest.mark.gpu
def test_gpu_crp_batch_48_clients(gpu_api, oracle):
    api = gpu_api
    K, D = 48, 50000
    rng = np.random.default_rng(8)
    proofs, pairs = [], []
    for k in range(K):
        v = rng.uniform(-3, 3, D).astype(np.float32); bl = api.rnd_scalar_vec(bytes([k]) * 32, D)
        rc, pf, pr = api.crp_prove(v, None, bl, NB, FR, bytes([0x40 + k]) * 32); assert rc == 0
        proofs.append(pf); pairs.append(pr)
    proofs = np.stack(proofs); pairs = np.stack(pairs)
    seed = b"\x34" * 32
    assert api.crp_verify_batch(proofs, pairs, seed).tolist() == [1] * K
    proofs[5, 64] ^= 1; pairs[20, 123, :32] = pairs[20, 124, :32]; proofs[33, 96:128] = 0xff
    got = api.crp_verify_batch(proofs, pairs, seed).tolist()
    assert got == [api.crp_verify(proofs[k], pairs[k]) for k in range(K)]
    assert got[5] == 0 and got[20] == 0 and got[33] == -1 and got.count(1) == K - 3


@pytest.mark.gpu
def test_gpu_crp_batch_at_the_pair_limit(gpu_api, oracle):
    """K = 2 at D = 900 000, the largest rand proof the reference can label"""
    api = gpu_api
    D = 900000
    rng = np.random.default_rng(9)
    proofs, pairs = [], []
    for k in range(2):
        v = rng.uniform(-3, 3, D).astype(np.float32); bl = api.rnd_scalar_vec(bytes([0x70 + k]) * 32, D)
        rc, pf, pr = api.crp_prove(v, None, bl, NB, FR, bytes([0x72 + k]) * 32); assert rc == 0
        proofs.append(pf); pairs.append(pr)
    proofs = np.stack(proofs); pairs = np.stack(pairs)
    assert api.crp_verify_batch(proofs, pairs, b"\x35" * 32).tolist() == [1, 1]
    pairs[1, D - 1, 32:] = pairs[1, 0, 32:]
    assert api.crp_verify_batch(proofs, pairs, b"\x35" * 32).tolist() == [1, 0] == [api.crp_verify(proofs[k], pairs[k]) for k in range(2)]
