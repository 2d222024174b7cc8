"""Server-side batch verification of the un-optimised messages of rofl_service (EncRange and EncL2, params.rs:186-233) and of their
per-element proofs: rofl_rand_verify_batch / rofl_square_rand_verify_batch check all K x D rand or square-rand proofs of a round in random
linear combinations (one MSM per range of elements) and fall back to the per-element kernel for the clients of a range that fails;
rofl_enc_range_verify_batch / rofl_enc_l2_verify_batch check whole messages.  Every verdict must be exactly that of the per-client call.
The emulation tests run the product kernels and engine on CPU threads (small sizes); the GPU tests run the B200 library at round sizes."""
import ctypes as C
import importlib.util
import os
import sys
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NB, FR, RB = 16, 7, 8                     # fixed point 16/7 and 8-bit range proofs for EncRange; EncL2 uses 32/7 with l2_range 32
ROFL_ERR_ARGS = -2
KIND = {1: dict(pw=128, cw=64, pts=("C'_L", "L", "C'_R", "R"), resp=("z_m", "z_r")),
        2: dict(pw=192, cw=96, pts=("C'_L", "c.L", "C'_R", "c.R", "C'_sq", "c_sq"), resp=("z_m", "z_r1", "z_r2"))}


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


def point_loc(kind, w):
    """(array, byte offset) of point w of an element: even w in the proof, odd w in the commitments (word w // 2)"""
    return ("p" if w % 2 == 0 else "c"), 32 * (w // 2)


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


def make_proofs(api, kind, K, D, tag):
    """K clients' honest rand (kind 1) or square-rand (kind 2) proofs -> (proofs[K, D, pw], commits[K, D, cw])"""
    rng = np.random.default_rng(tag)
    P, Cm = [], []
    for k in range(K):
        v = rng.uniform(-3, 3, D).astype(np.float32); r1 = api.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D)
        if kind == 1:
            rc, p, c = api.rand_prove(v, None, r1, NB, FR, bytes([(0x80 + tag + k) & 0xff]) * 32)
        else:
            r2 = api.rnd_scalar_vec(bytes([(0x40 + tag + k) & 0xff]) * 32, D)
            rc, p, c = api.square_rand_prove(v, None, r1, r2, 32, FR, bytes([(0x80 + tag + k) & 0xff]) * 32)
        assert rc == 0
        P.append(p); Cm.append(c)
    return np.stack(P), np.stack(Cm)


def single(api, kind, p, c):
    return api.rand_verify(p, c) if kind == 1 else api.square_rand_verify(p, c)


def batch(api, kind, P, Cm, seed):
    return (api.rand_verify_batch(P, Cm, seed) if kind == 1 else api.square_rand_verify_batch(P, Cm, seed)).tolist()


def check_proofs(api, kind, P, Cm, seed, oracle=None):
    """batch verdicts == single-call verdicts (and the oracle's); the combined check itself holds exactly when every verdict is 1"""
    got = batch(api, kind, P, Cm, seed)
    want = [single(api, kind, P[k], Cm[k]) for k in range(P.shape[0])]
    assert got == want, (got, want)
    if oracle is not None:
        orc = [(oracle.rand_verify if kind == 1 else oracle.square_rand_verify)(P[k], Cm[k]) for k in range(P.shape[0])]
        assert got == orc, (got, orc)
    if P.shape[1]:
        assert api.debug_sigma_rlc(kind, P, Cm, seed) == int(all(x == 1 for x in got))
    return got


def tamper_cases(api, oracle, kind, P, Cm):
    """(name, tampered copies of (P, Cm), indices of the tampered clients)"""
    t, i = 1, P.shape[1] // 2
    kd = KIND[kind]
    out = []
    for w, name in enumerate(kd["pts"]):
        where, off = point_loc(kind, w)
        for valid in (True, False):
            p, c = P.copy(), Cm.copy(); arr = p if where == "p" else c
            arr[t, i, off:off + 32] = flipped_point(oracle, arr[t, i, off:off + 32], valid)
            out.append((f"{name} flipped bit, decodes={valid}", p, c, [t]))
    for j, name in enumerate(kd["resp"]):
        off = kd["pw"] // 2 + 32 * j
        p = P.copy(); p[t, i, off:off + 32] = scalar_plus_one(api, P[t, i, off:off + 32])
        out.append((f"{name} + 1", p, Cm.copy(), [t]))
        p = P.copy(); p[t, i, off:off + 32] = 0xff
        out.append((f"{name} non-canonical", p, Cm.copy(), [t]))
    p = P.copy(); p[t, i] = P[t, i + 1]
    out.append(("another element's proof", p, Cm.copy(), [t]))
    p = P.copy(); p[0], p[t] = P[t].copy(), P[0].copy()
    out.append(("proofs of two clients swapped", p, Cm.copy(), [0, t]))
    return out


def run_tamper_matrix(api, oracle, kind, P, Cm, seed, with_oracle):
    for name, p, c, bad in tamper_cases(api, oracle, kind, P, Cm):
        got = check_proofs(api, kind, p, c, seed, oracle if with_oracle else None)
        assert all(got[k] == 1 for k in range(P.shape[0]) if k not in bad), (name, got)
        assert all(got[k] in (0, -1) for k in bad), (name, got)
        if "non-canonical" in name or "decodes=False" in name:
            assert got[bad[0]] == -1, (name, got)


def cancelling_errors(api, oracle, kind, P, Cm, seed):
    """errors that cancel under equal weights: C'_L + B on one element and C'_L - B on another; the responses of two elements swapped"""
    a, b = 3, P.shape[1] - 4
    p = P.copy()
    p[1, a, :32] = np.frombuffer(oracle.point_add(P[1, a, :32], oracle.basepoint()), np.uint8)
    p[1, b, :32] = np.frombuffer(oracle.point_sub(P[1, b, :32], oracle.basepoint()), np.uint8)
    assert check_proofs(api, kind, p, Cm, seed) == [1, 0, 1]
    p = P.copy(); lo = KIND[kind]["pw"] // 2
    p[2, a, lo:], p[2, b, lo:] = P[2, b, lo:].copy(), P[2, a, lo:].copy()
    assert check_proofs(api, kind, p, Cm, seed) == [1, 1, 0]


# ---- whole messages ------------------------------------------------------------------------------------------------------------------
def make_range_msgs(api, oracle, K, D, cp, P, tag):
    """EncRange messages: rand proofs over all D pairs (L = commit(v, r)), range proofs over the first round(D cp) L halves"""
    num = llroundf(D, cp)
    rng = np.random.default_rng(tag)
    mn, mx = oracle.clip_bounds(RB, NB, FR)
    msgs = []
    for k in range(K):
        v = rng.uniform(mn, mx, D).astype(np.float32); bl = oracle.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D); seed = bytes([(0x60 + k) & 0xff]) * 32
        rc, proofs, pairs = api.rand_prove(v, None, bl, NB, FR, seed); assert rc == 0
        rc, rp, commits = api.range_prove(v[:num], bl[:num], RB, P, NB, FR, seed); assert rc == 0
        assert (commits == pairs[:num, :32]).all()
        msgs.append(dict(enc_values=pairs, rand_proof=proofs, range_proof=rp, range_bits=RB))
    return msgs


def make_l2_msgs(api, K, D, P, tag, rb=RB, l2=32):
    rng = np.random.default_rng(tag)
    msgs = []
    for k in range(K):
        v = rng.uniform(-0.9, 0.9, D).astype(np.float32); bl = api.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D)
        rc, m = api.enc_l2_encrypt(v, bl, rb, P, l2, 32, FR, bytes([(0x80 + tag + k) & 0xff]) * 32)
        assert rc == 0
        msgs.append(m)
    return msgs


def copy_msgs(msgs):
    return [{f: (x.copy() if isinstance(x, np.ndarray) else x) for f, x in m.items()} for m in msgs]


def check_range_round(api, msgs, seed, cp=1.0):
    got = api.enc_range_verify_batch(msgs, cp, seed).tolist()
    want = [api.enc_range_verify(m, cp, seed) for m in msgs]
    assert got == want, (got, want)
    return got


def check_l2_round(api, msgs, seed):
    got = api.enc_l2_verify_batch(msgs, seed).tolist()
    want = [api.enc_l2_verify(m, seed) for m in msgs]
    assert got == want, (got, want)
    return got


# ---- emulation (CPU) -----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def proofs1(api):
    return make_proofs(api, 1, 3, 100, 11)


@pytest.fixture(scope="module")
def proofs2(api):
    return make_proofs(api, 2, 3, 100, 12)


@pytest.mark.parametrize("kind", [1, 2])
def test_honest_round_all_accepted(api, oracle, proofs1, proofs2, kind):
    P, Cm = proofs1 if kind == 1 else proofs2
    assert check_proofs(api, kind, P, Cm, b"\x41" * 32, oracle) == [1, 1, 1]
    assert api.debug_sigma_rlc(kind, P, Cm, b"\x41" * 32) == 1


@pytest.mark.parametrize("kind", [1, 2])
def test_tamper_matrix(api, oracle, proofs1, proofs2, kind):
    P, Cm = proofs1 if kind == 1 else proofs2
    run_tamper_matrix(api, oracle, kind, P, Cm, b"\x42" * 32, with_oracle=True)


@pytest.mark.parametrize("kind", [1, 2])
def test_cancelling_errors(api, oracle, proofs1, proofs2, kind):
    P, Cm = proofs1 if kind == 1 else proofs2
    cancelling_errors(api, oracle, kind, P, Cm, b"\x43" * 32)


@pytest.mark.parametrize("kind", [1, 2])
def test_ranges_split_mid_client(api, oracle, proofs1, proofs2, kind):
    """ranges of 37 elements (148 / 222 MSM terms): boundaries fall inside clients, one client spans three ranges"""
    P, Cm = proofs1 if kind == 1 else proofs2
    seed = b"\x44" * 32
    api.set_option("sigma_rlc_terms", 37 * (4 if kind == 1 else 6))
    try:
        assert check_proofs(api, kind, P, Cm, seed) == [1, 1, 1]
        for k, i in ((1, 0), (1, 99), (0, 73), (1, 11)):        # first / last element of a client, the last element of a range, the first of one
            p = P.copy(); p[k, i, KIND[kind]["pw"] // 2] ^= 1                                 # z_m
            got = check_proofs(api, kind, p, Cm, seed)
            assert got[k] == 0 and got.count(1) == 2, (k, i, got)
        c = Cm.copy(); c[0, 99, 32:64] = Cm[1, 0, 32:64]                 # R of the last element of client 0, inside the range that starts client 1
        assert check_proofs(api, kind, P, c, seed) == [0, 1, 1]
    finally:
        api.set_option("sigma_rlc_terms", 1 << 24)


@pytest.mark.parametrize("cp", [1.0, 0.5, 0.25])
def test_enc_range_messages(api, oracle, cp):
    msgs = make_range_msgs(api, oracle, 3, 100, cp, 2, 20 + int(4 * cp))
    seed = b"\x45" * 32
    assert check_range_round(api, msgs, seed, cp) == [1, 1, 1]
    num = llroundf(100, cp)
    ms = copy_msgs(msgs); ms[1]["range_proof"][0, 70] ^= 1
    assert check_range_round(api, ms, seed, cp) == [1, 0, 1]
    ms = copy_msgs(msgs); ms[2]["enc_values"][num - 1, 32:] = msgs[2]["enc_values"][0, 32:]        # an R half: only the rand proof fails
    assert check_range_round(api, ms, seed, cp) == [1, 1, 0]
    ms = copy_msgs(msgs); ms[0]["rand_proof"][10, 96:] = 0xff                                        # a rand-proof format error is a reject
    assert check_range_round(api, ms, seed, cp) == [0, 1, 1]
    for bad_cp in (0.001, 1.5):                                                                      # num == 0 and num > D
        assert check_range_round(api, msgs, seed, bad_cp) == [0, 0, 0]


def test_enc_l2_messages(api, oracle):
    msgs = make_l2_msgs(api, 3, 100, 2, 30)
    seed = b"\x46" * 32
    assert check_l2_round(api, msgs, seed) == [1, 1, 1]
    ms = copy_msgs(msgs); ms[1]["range_proof"][0, 70] ^= 1
    assert check_l2_round(api, ms, seed) == [1, 0, 1]
    ms = copy_msgs(msgs); ms[2]["square_range_proof"][70] ^= 1
    assert check_l2_round(api, ms, seed) == [1, 1, 0]
    ms = copy_msgs(msgs); ms[0]["enc_values"][5, 64:] = flipped_point(oracle, msgs[0]["enc_values"][5, 64:], False)   # c_sq undecodable
    assert check_l2_round(api, ms, seed) == [0, 1, 1]
    ms = copy_msgs(msgs); ms[1]["enc_values"][50, 32:64] = flipped_point(oracle, msgs[1]["enc_values"][50, 32:64], False)   # c.R undecodable
    assert check_l2_round(api, ms, seed) == [1, 0, 1]
    ms = copy_msgs(msgs); ms[2]["square_proof"][99, 160:] = scalar_plus_one(api, msgs[2]["square_proof"][99, 160:])
    assert check_l2_round(api, ms, seed) == [1, 1, 0]


def test_argument_edges(api, proofs1):
    L = api.lib
    seed = np.frombuffer(b"\x47" * 32, np.uint8)
    P, Cm = proofs1
    ok = np.full(3, 7, np.int32)
    rp = np.zeros((3, 1, 32 * 13), np.uint8)
    # K = 0: nothing is written
    for f in (L.rofl_rand_verify_batch, L.rofl_square_rand_verify_batch):
        assert f(api.h, 0, None, None, 5, seed.ctypes.data, ok.ctypes.data) == 0
    assert L.rofl_enc_range_verify_batch(api.h, 0, None, 5, None, None, 32 * 13, 1, 8, 1.0, seed.ctypes.data, ok.ctypes.data) == 0
    assert L.rofl_enc_l2_verify_batch(api.h, 0, None, 5, None, None, 32 * 13, 1, None, 32 * 13, 8, 32, seed.ctypes.data, ok.ctypes.data) == 0
    assert ok.tolist() == [7, 7, 7]
    # null out_ok; D == 0 and n_proofs == 0 for the messages
    assert L.rofl_rand_verify_batch(api.h, 3, P.ctypes.data, Cm.ctypes.data, 100, seed.ctypes.data, None) == ROFL_ERR_ARGS
    assert L.rofl_square_rand_verify_batch(api.h, 3, P.ctypes.data, Cm.ctypes.data, 100, seed.ctypes.data, None) == ROFL_ERR_ARGS
    assert L.rofl_enc_range_verify_batch(api.h, 3, Cm.ctypes.data, 100, P.ctypes.data, rp.ctypes.data, rp.shape[2], 1, 8, 1.0, seed.ctypes.data, None) == ROFL_ERR_ARGS
    assert L.rofl_enc_range_verify_batch(api.h, 3, Cm.ctypes.data, 0, P.ctypes.data, rp.ctypes.data, rp.shape[2], 1, 8, 1.0, seed.ctypes.data, ok.ctypes.data) == ROFL_ERR_ARGS
    assert L.rofl_enc_range_verify_batch(api.h, 3, Cm.ctypes.data, 100, P.ctypes.data, rp.ctypes.data, rp.shape[2], 0, 8, 1.0, seed.ctypes.data, ok.ctypes.data) == ROFL_ERR_ARGS
    for D, n in ((100, None), (0, 1), (100, 0)):
        out = None if n is None else ok.ctypes.data
        assert L.rofl_enc_l2_verify_batch(api.h, 3, Cm.ctypes.data, D, P.ctypes.data, rp.ctypes.data, rp.shape[2], 1 if n is None else n, rp.ctypes.data, rp.shape[2], 8, 32,
                                          seed.ctypes.data, out) == ROFL_ERR_ARGS
    assert ok.tolist() == [7, 7, 7]
    # D == 0 in the proof-only calls: every client passes, as in the single calls
    assert api.rand_verify_batch(np.zeros((3, 0, 128), np.uint8), np.zeros((3, 0, 64), np.uint8), seed).tolist() == [1, 1, 1] == [api.rand_verify(np.zeros((0, 128), np.uint8), np.zeros((0, 64), np.uint8))] * 3
    assert api.square_rand_verify_batch(np.zeros((3, 0, 192), np.uint8), np.zeros((3, 0, 96), np.uint8), seed).tolist() == [1, 1, 1]


def test_below_the_size_threshold(api, oracle, proofs1):
    """fewer than 256 elements: the per-element kernel alone, per-client verdicts all the same"""
    P, Cm = proofs1
    p = P[:, :20].copy(); c = Cm[:, :20].copy()
    assert check_proofs(api, 1, p, c, b"\x48" * 32, oracle) == [1, 1, 1]
    p[2, 7, 64] ^= 1; p[0, 3, 96:] = 0xff
    assert check_proofs(api, 1, p, c, b"\x48" * 32, oracle) == [-1, 1, 0]


@pytest.mark.parametrize("kind", [1, 2])
def test_single_lane(api, proofs1, proofs2, kind):
    P, Cm = proofs1 if kind == 1 else proofs2
    api.set_option("max_lanes", 1)
    try:
        assert check_proofs(api, kind, P, Cm, b"\x49" * 32) == [1, 1, 1]
        msgs = make_l2_msgs(api, 2, 20, 1, 31) if kind == 2 else None
        if msgs:
            assert check_l2_round(api, msgs, b"\x49" * 32) == [1, 1]
    finally:
        api.set_option("max_lanes", 8)


# ---- B200 -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", [1, 2])
def test_gpu_tamper_matrix(gpu_api, oracle, kind):
    P, Cm = make_proofs(gpu_api, kind, 3, 2000, 13 + kind)
    assert check_proofs(gpu_api, kind, P, Cm, b"\x51" * 32) == [1, 1, 1]
    run_tamper_matrix(gpu_api, oracle, kind, P, Cm, b"\x52" * 32, with_oracle=False)
    cancelling_errors(gpu_api, oracle, kind, P, Cm, b"\x53" * 32)


def configs4_msgs(api, K, D, tag, l2):
    """configs[4]-shaped messages: 8-bit range proofs in 64 chunks, fixed point 32/7, l2_range 32, check_percentage 1"""
    rng = np.random.default_rng(tag)
    msgs = []
    for k in range(K):
        v = rng.uniform(-0.05, 0.05, D).astype(np.float32); bl = api.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D); seed = bytes([(0x80 + k) & 0xff]) * 32
        rc, m = api.enc_l2_encrypt(v, bl, 8, 64, 32, 32, 7, seed) if l2 else api.enc_range_encrypt(v, bl, 8, 64, 1.0, 32, 7, seed)
        assert rc == 0
        msgs.append(m)
    return msgs


@pytest.mark.gpu
def test_gpu_enc_range_round_48_clients(gpu_api):
    api = gpu_api
    msgs = configs4_msgs(api, 48, 50000, 14, l2=False)
    seed = b"\x54" * 32
    assert api.enc_range_verify_batch(msgs, 1.0, seed).tolist() == [1] * 48
    ms = copy_msgs(msgs)
    ms[9]["enc_values"][25000, 32:] = msgs[9]["enc_values"][25001, 32:]            # an R half of another pair: that rand proof fails
    ms[30]["range_proof"][17, 100] ^= 1                                              # a range-proof byte
    got = api.enc_range_verify_batch(ms, 1.0, seed).tolist()
    assert got == [api.enc_range_verify(m, 1.0, seed) for m in ms]
    assert got[9] == 0 and got[30] == 0 and got.count(1) == 46, got


@pytest.mark.gpu
def test_gpu_enc_l2_round_48_clients(gpu_api):
    api = gpu_api
    msgs = configs4_msgs(api, 48, 50000, 15, l2=True)
    seed = b"\x55" * 32
    assert api.enc_l2_verify_batch(msgs, seed).tolist() == [1] * 48
    ms = copy_msgs(msgs)
    ms[4]["square_proof"][49999, 100] ^= 1                                           # a response of the last element
    ms[41]["square_range_proof"][70] ^= 1
    got = api.enc_l2_verify_batch(ms, seed).tolist()
    assert got == [api.enc_l2_verify(m, seed) for m in ms]
    assert got[4] == 0 and got[41] == 0 and got.count(1) == 46, got


@pytest.mark.gpu
def test_gpu_one_client_over_several_ranges(gpu_api):
    """K = 1 at D = 3 000 000 square-rand proofs: 18 M MSM terms, more than one 2^24-term range"""
    api = gpu_api
    D = 3000000
    P, Cm = make_proofs(api, 2, 1, D, 16)
    seed = b"\x56" * 32
    assert api.debug_sigma_rlc(2, P, Cm, seed) == 1
    assert api.square_rand_verify_batch(P, Cm, seed).tolist() == [1]
    P[0, D - 1, 96] ^= 1
    assert api.debug_sigma_rlc(2, P, Cm, seed) == 0
    assert api.square_rand_verify_batch(P, Cm, seed).tolist() == [0] == [api.square_rand_verify(P[0], Cm[0])]
