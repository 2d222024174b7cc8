"""The random linear combinations of the batch verifiers, term by term, against a plain restatement of their Fiat-Shamir weights (DESIGN.md §2).

A batched check accepts a whole round when ONE weighted sum is the identity, so it is only sound while every weight is an unpredictable function
of every byte it checks.  Verdict tests cannot see that: honest rounds pass under any weights, one tampered element fails under any nonzero
weight.  Here the production code of each check (square_verify_rlc, sigma_verify_rlc, crp_batch_end, through the test hook rofl_debug_rlc_terms,
which copies what those functions computed and derives nothing) is compared with this file's reference -- hashlib SHA3-256, the oracle's ChaCha20
and challenges (its own radix-2^51 transcript code), Python integers mod l -- for the root, every challenge, every MSM scalar, every fixed-base
coefficient and the weight width; then the weights are shown to move with every byte of a record and with the seed, and an adaptive forgery that
cancels under the weights it predicts is shown to be rejected.

Families: 0 square proofs, 1 rand proofs, 2 square-rand proofs, 3 compressed rand proofs (K clients x D pairs).  The "emu" tests run the
product code under the CUDA-on-CPU emulation (tests/hostsim), the gpu ones on the device at round sizes."""
import ctypes as C
import hashlib
import importlib.util
import os
import sys
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
L = 2**252 + 27742317777372353535851937790883648493
TERMS_MAX = 1 << 24                                          # the default and upper bound of sigma_rlc_terms / crp_batch_terms
SEED = bytes(range(32))
# proof / commitment bytes per element, MSM terms per element, key tag, offset of the responses in the proof
FAM = {0: dict(pw=160, cw=64, np=4, tag=b"sqrl", z=64), 1: dict(pw=128, cw=64, np=4, tag=b"rprl", z=64),
       2: dict(pw=192, cw=96, np=6, tag=b"srrl", z=96), 3: dict(pw=128, cw=64)}


# ---- fixtures --------------------------------------------------------------------------------------------------------------
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


def honest(oracle, fam, K, D, tag=1):
    """K updates of D honest proofs from the oracle -> (proofs, commits) shaped for Api.debug_rlc_terms"""
    rng = np.random.default_rng(tag)
    v = rng.uniform(-3, 3, K * D).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(bytes([tag & 0xff]) * 32, K * D); r2 = oracle.rnd_scalar_vec(bytes([(tag + 0x40) & 0xff]) * 32, K * D)
    seed = bytes([(tag + 0x80) & 0xff]) * 32
    if fam == 3:
        P, Cm = [], []
        for k in range(K):
            rc, p, c = oracle.crp_prove(v[k * D:(k + 1) * D], None, r1[k * D:(k + 1) * D], seed=bytes([(tag + k) & 0xff]) * 32)
            assert rc == 0
            P.append(p); Cm.append(c)
        return np.stack(P), np.stack(Cm)
    if fam == 0:
        rc, p, c = oracle.square_prove(v, oracle.commit_f32(v, r1, 32, 7), r1, r2, seed=seed)
    elif fam == 1:
        rc, p, c = oracle.rand_prove(v, None, r1, seed=seed)
    else:
        rc, p, c = oracle.square_rand_prove(v, None, r1, r2, seed=seed)
    assert rc == 0
    return p.reshape(K, D, -1), c.reshape(K, D, -1)


# ---- the reference: DESIGN.md §2 restated -----------------------------------------------------------------------------------
def sha3(b):
    return hashlib.sha3_256(b).digest()


def le(x, n=8):
    return int(x).to_bytes(n, "little")


def sc_int(b):
    return int.from_bytes(bytes(b), "little")


def tree_root(leaves):
    """inner node = SHA3-256(0x01 | up to 64 child digests), level by level; do-while, so a single leaf still gets one node above it"""
    level = leaves
    while True:
        level = [sha3(b"\x01" + b"".join(level[j:j + 64])) for j in range(0, len(level), 64)]
        if len(level) == 1:
            return level[0]


def chacha_blocks(keys, ctr=0):
    """ChaCha20 block `ctr` (zero nonce, RFC 8439 layout with a 64-bit counter as rand_chacha) of many 32-byte keys at once -> uint8 [n, 64].
    Vectorised so that the GPU-sized references stay short; test_reference_chacha_is_the_oracles pins it to oracle.chacha20_block."""
    k = np.frombuffer(b"".join(keys), dtype="<u4").reshape(-1, 8).astype(np.uint32)
    n = k.shape[0]
    st = np.zeros((16, n), np.uint32)
    st[0:4] = np.array([0x61707865, 0x3320646e, 0x79622d32, 0x6b206574], np.uint32)[:, None]
    st[4:12] = k.T
    st[12] = ctr & 0xffffffff; st[13] = ctr >> 32
    x = st.copy()

    def rotl(v, r):
        return (v << np.uint32(r)) | (v >> np.uint32(32 - r))

    def qr(a, b, c, d):
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16)
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12)
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8)
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7)
    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    return np.ascontiguousarray((x + st).T).astype("<u4").view(np.uint8).reshape(n, 64)


def wbits_of(c):
    """the smallest c w - 1 >= 125: a top window of c - 1 bits"""
    return c * ((126 + c - 1) // c) - 1


def records(fam, P, Cm):
    """commitments_i | proof_i of every element, flattened over the updates -> uint8 [N, cw + pw]"""
    f = FAM[fam]
    return np.concatenate([Cm.reshape(-1, f["cw"]), P.reshape(-1, f["pw"])], axis=1)


def ref_sigma(oracle, fam, P, Cm, seed, terms=TERMS_MAX, idx=None):
    """families 0-2: root, challenges and the expected ranges (i0, n, weights per element, scalars of the elements in idx, sB, sH).
    Weights and fixed-base sums are computed for every element, challenges and scalars only at idx (default: all)."""
    f = FAM[fam]
    rec = records(fam, P, Cm); N = rec.shape[0]
    root = tree_root([sha3(b"\x00" + rec[i].tobytes()) for i in range(N)])
    pre = hashlib.sha3_256(root + (b"" if fam == 0 else seed) + f["tag"] + le(N))      # the square-proof key has no seed
    keys = []
    for i in range(N):
        h = pre.copy(); h.update(le(i)); keys.append(h.digest())
    blocks = chacha_blocks(keys)
    cw, z = f["cw"], f["z"]
    zs = [[sc_int(rec[i, cw + z + 32 * q:cw + z + 32 * q + 32]) for q in range(3 if fam != 1 else 2)] for i in range(N)]
    idx = range(N) if idx is None else sorted(set(idx))
    chal = {}
    for i in idx:
        com, pf = rec[i, :cw], rec[i, cw:]
        chal[i] = sc_int((oracle.sq_challenge if fam == 0 else oracle.rp_challenge if fam == 1 else oracle.srp_challenge)(com, pf))
    R = max(1, min(terms, TERMS_MAX) // f["np"]) if fam else N
    out = []
    for i0 in range(0, N, R):
        n = min(R, N - i0)
        out.append(dict(i0=i0, n=n, blocks=blocks[i0:i0 + n], zs=zs[i0:i0 + n]))
    return dict(root=root, chal=chal, ranges=out, N=N)


def weights_of(blocks, wbits):
    m = (1 << wbits) - 1
    return [tuple(sc_int(b[20 * q:20 * q + 20]) & m for q in range(3)) for b in blocks]


def sigma_terms(fam, w, z, c):
    """the MSM scalars of one element and its B / H contributions (before negation), kernels.cuh k_sq_rlc_scalars / k_sigma_rlc_scalars"""
    rho, sig, tau = w
    if fam == 0:
        zm, zr1, zr2 = z
        return [rho, (rho * c - sig * zm) % L, sig, sig * c % L], rho * zm, rho * zr1 + sig * zr2
    if fam == 1:
        zm, zr = z
        return [rho, rho * c % L, sig, sig * c % L], rho * zm + sig * zr, rho * zr
    zm, zr1, zr2 = z
    return [rho, (rho * c - tau * zm) % L, sig, sig * c % L, tau, tau * c % L], rho * zm + sig * zr1, rho * zr1 + tau * zr2


def ref_crp(oracle, proofs, pairs, seed, terms=TERMS_MAX):
    """family 3: challenges c_k from the oracle's transcript, the crpb root, rho_k with the zero-retry rule, the groups"""
    K, D = pairs.shape[0], pairs.shape[1]
    c = [sc_int(oracle.crp_challenge(proofs[k], pairs[k])) for k in range(K)]
    z = [(sc_int(proofs[k, 64:96]), sc_int(proofs[k, 96:128])) for k in range(K)]
    dig = [sha3(le(c[k], 32) + proofs[k, 64:128].tobytes()) for k in range(K)]
    root = sha3(seed + b"crpb" + le(K) + le(D) + b"".join(dig))
    rho = []
    for k in range(K):
        key = sha3(root + le(k))
        for ctr in range(1 << 20):
            r = sc_int(oracle.chacha20_block(key, ctr)[:16])
            if r:
                break
        rho.append(r)
    G = max(1, min(K, min(terms, TERMS_MAX) // (D + 1)))
    groups = [(k0, min(G, K - k0)) for k0 in range(0, K, G)]
    return dict(root=root, c=c, z=z, rho=rho, groups=groups, D=D)


# ---- comparison of the hook with the reference -------------------------------------------------------------------------------
def b32(x):
    return (x % L).to_bytes(32, "little")


def check_sigma(oracle, fam, got, P, Cm, seed, terms=TERMS_MAX, sample=None):
    """every term of a family 0-2 call equals the reference; sample = None compares every scalar, else (edge, count, rng): the first and last
    `edge` elements of each range plus `count` random ones.  Returns the weights (rho, sigma, tau) per element as the hook computed them."""
    f = FAM[fam]; npe = f["np"]
    N = P.shape[0] * P.shape[1]
    idx = None
    if sample is not None:
        edge, count, rng = sample
        R = max(1, min(terms, TERMS_MAX) // npe) if fam else N
        idx = set(int(i) for i in rng.integers(0, N, count))
        for i0 in range(0, N, R):
            n = min(R, N - i0)
            idx |= set(range(i0, i0 + min(edge, n))) | set(range(i0 + max(0, n - edge), i0 + n))
    ref = ref_sigma(oracle, fam, P, Cm, seed, terms, idx)
    assert got["root"] == ref["root"]
    assert got["held"] == 1 and got["verdicts"] == [1] * P.shape[0]
    for i, c in ref["chal"].items():
        assert sc_int(got["chal"][i]) == c, i
    assert [(r["i0"], r["n"]) for r in got["ranges"]] == [(r["i0"], r["n"]) for r in ref["ranges"]]
    allw = []
    for g, r in zip(got["ranges"], ref["ranges"]):
        wb = g["wbits"]
        assert 125 <= wb <= 134 and wb == wbits_of(g["c"]), (wb, g["c"])
        assert g["is_id"] == (1, -1) and not any(g["bad"])
        ws = weights_of(r["blocks"], wb)
        sB = sH = 0
        scal = g["scal"]; assert scal.shape == (npe * r["n"], 32)
        for t in range(r["n"]):
            i = r["i0"] + t
            w = ws[t] if fam == 2 else (ws[t][0], ws[t][1], 0)
            c = ref["chal"].get(i)
            terms_i, b, h = sigma_terms(fam, w, r["zs"][t], c or 0)
            sB += b; sH += h
            if c is not None:
                assert [sc_int(scal[npe * t + q]) for q in range(npe)] == terms_i, (i, wb)
            allw.append(w if fam == 2 else w[:2])
        for q in range(0, npe, 2):                               # the weights sit at the even terms: nothing above wbits
            assert max(sc_int(x) for x in scal[q::npe]) >> wb == 0
        assert g["sB"] == (b32(-sB), bytes(32)) and g["sH"] == (b32(-sH), bytes(32))
    return allw


def check_crp(oracle, got, proofs, pairs, seed, terms=TERMS_MAX, sample=None):
    """every term of a family 3 call equals the reference (scalars at `sample` = (edge, count, rng) positions of each group, or all)"""
    ref = ref_crp(oracle, proofs, pairs, seed, terms)
    D = ref["D"]
    assert got["root"] == ref["root"]
    assert got["held"] == 1 and got["verdicts"] == [1] * len(ref["c"])
    assert [sc_int(x) for x in got["chal"]] == ref["c"]
    assert [(g["i0"], g["n"]) for g in got["ranges"]] == ref["groups"]
    for g in got["ranges"]:
        k0, n = g["i0"], g["n"]
        assert g["is_id"] == (1, 1) and g["bad"] == [0] * n and g["wbits"] == 0
        scal = g["scal"]; assert scal.shape == (n * (D + 1), 32)
        T = n * D
        pos = range(T) if sample is None else sorted(set(range(min(sample[0], T))) | set(range(max(0, T - sample[0]), T)) |
                                                       set(int(x) for x in sample[2].integers(0, T, sample[1])))
        for t in pos:
            k = k0 + t // D
            assert sc_int(scal[t]) == ref["rho"][k] * pow(ref["c"][k], t % D + 1, L) % L, t
        assert [sc_int(x) for x in scal[T:]] == ref["rho"][k0:k0 + n]
        assert max(ref["rho"][k0:k0 + n]) >> 128 == 0
        sB0 = -sum(ref["rho"][k] * ref["z"][k][0] for k in range(k0, k0 + n)); sB1 = -sum(ref["rho"][k] * ref["z"][k][1] for k in range(k0, k0 + n))
        assert g["sB"] == (b32(sB0), b32(sB1)) and g["sH"] == (b32(sB1), bytes(32))
    return ref["rho"]


def hook_weights(fam, got):
    """(rho, sigma[, tau]) of every element (families 0-2) or rho_k of every client (3), read from the hook's MSM scalars"""
    out = []
    for g in got["ranges"]:
        s = g["scal"]
        if fam == 3:
            out += [sc_int(x) for x in s[g["n"] * (len(s) // g["n"] - 1):]]
        else:
            npe = FAM[fam]["np"]
            out += [tuple(sc_int(s[npe * t + q]) for q in range(0, npe, 2)) for t in range(g["n"])]
    return out


# ---- exact equality, emulation ---------------------------------------------------------------------------------------------------
def test_reference_chacha_is_the_oracles(oracle):
    keys = [sha3(bytes([i])) for i in range(64)]
    got = chacha_blocks(keys)
    for i, k in enumerate(keys):
        assert got[i].tobytes() == oracle.chacha20_block(k, 0)
    assert chacha_blocks(keys[:3], 5)[2].tobytes() == oracle.chacha20_block(keys[2], 5)


@pytest.fixture(scope="module")
def pool(oracle):
    """4097 honest elements of families 1 and 2 (prefixes give every N below)"""
    return {fam: honest(oracle, fam, 1, 4097, tag=fam) for fam in (1, 2)}


NS = [1, 2, 63, 64, 65, 127, 128, 129, 256, 4095, 4096, 4097]      # hash-tree fan-in, 128-thread block sums, three tree levels


@pytest.mark.parametrize("fam", [1, 2])
@pytest.mark.parametrize("N", NS)
def test_sigma_terms_exact(api, oracle, pool, fam, N):
    P, Cm = pool[fam][0][:, :N], pool[fam][1][:, :N]
    got = api.debug_rlc_terms(fam, P, Cm, SEED)
    w = check_sigma(oracle, fam, got, P, Cm, SEED)
    assert len(set(x for t in w for x in t)) == len(w) * len(w[0])


@pytest.mark.parametrize("fam", [1, 2])
@pytest.mark.parametrize("per_range,K,D", [(1, 3, 7), (37, 3, 100), (128, 3, 100), (129, 4, 95)])
def test_sigma_ranges_exact(api, oracle, fam, per_range, K, D):
    """ranges of 1, 37, 128, 129 elements that start and end inside updates: keys use the call's index i0 + t, weights never repeat across ranges"""
    P, Cm = honest(oracle, fam, K, D, tag=10 + fam)
    terms = per_range * FAM[fam]["np"]
    api.set_option("sigma_rlc_terms", terms)
    try:
        got = api.debug_rlc_terms(fam, P, Cm, SEED)
    finally:
        api.set_option("sigma_rlc_terms", TERMS_MAX)
    assert len(got["ranges"]) == -(-K * D // per_range)
    w = check_sigma(oracle, fam, got, P, Cm, SEED, terms)
    assert len(set(x for t in w for x in t)) == len(w) * len(w[0])


@pytest.mark.parametrize("D", [1, 64, 65, 300])
def test_square_terms_exact(api, oracle, D):
    """the square-proof batch, also below its 256-element threshold; its key has no seed (DESIGN.md §2)"""
    P, Cm = honest(oracle, 0, 1, D, tag=20)
    got = api.debug_rlc_terms(0, P, Cm, SEED)
    w = check_sigma(oracle, 0, got, P, Cm, SEED)
    assert len(set(x for t in w for x in t)) == 2 * len(w)
    assert api.debug_rlc_terms(0, P, Cm, bytes(32))["ranges"][0]["scal"].tobytes() == got["ranges"][0]["scal"].tobytes()


@pytest.fixture(scope="module")
def crp_pool(oracle):
    return {D: honest(oracle, 3, 5, D, tag=30 + D % 200) for D in (1, 2, 3, 127, 128, 129, 1000)}


@pytest.mark.parametrize("D", [1, 2, 3, 127, 128, 129, 1000])           # split power tables: the index boundaries 2^L of ilog2(D + 2)
@pytest.mark.parametrize("K", [1, 2, 5])
def test_crp_terms_exact(api, oracle, crp_pool, K, D):
    P, Cm = crp_pool[D][0][:K], crp_pool[D][1][:K]
    got = api.debug_rlc_terms(3, P, Cm, SEED)
    rho = check_crp(oracle, got, P, Cm, SEED)
    assert len(set(rho)) == K


@pytest.mark.parametrize("per_group,K,D", [(1, 3, 4), (2, 5, 4), (3, 5, 4), (2, 5, 129), (3, 7, 2)])
def test_crp_groups_exact(api, oracle, per_group, K, D):
    """client groups of 1, 2, 3 (partial last groups included): decompress(k0, g) for k0 > 0, group-local bad flags and scalars"""
    P, Cm = honest(oracle, 3, K, D, tag=40 + K)
    terms = per_group * (D + 1)
    api.set_option("crp_batch_terms", terms)
    try:
        got = api.debug_rlc_terms(3, P, Cm, SEED)
        assert len(got["ranges"]) == -(-K // per_group)
        check_crp(oracle, got, P, Cm, SEED, terms)
        assert api.crp_verify_batch(P, Cm, SEED).tolist() == [1] * K
        bad = Cm.copy(); bad[K - 1, D - 1, 40] ^= 1                     # a wrong R in the last group's last client
        want = [api.crp_verify(P[k], bad[k]) for k in range(K)]
        assert want[K - 1] in (0, -1) and want[:K - 1] == [1] * (K - 1)
        assert api.crp_verify_batch(P, bad, SEED).tolist() == want
    finally:
        api.set_option("crp_batch_terms", TERMS_MAX)


# ---- binding: every byte, the seed, distinctness --------------------------------------------------------------------------------
def flip_canonical(oracle, buf, j, zoff):
    """buf with one bit of byte j flipped; in the responses (from byte zoff on) one that keeps the scalar canonical: the weights are also
    derived for malformed elements, but the compressed-rand-proof batch skips a client whose response is not canonical"""
    for bit in range(8):
        out = buf.copy(); out[j] = buf[j] ^ (1 << bit)
        if j < zoff or oracle.sc_is_canonical(out[zoff + 32 * ((j - zoff) // 32):zoff + 32 * ((j - zoff) // 32) + 32]):
            return out
    raise AssertionError("no canonical flip")


def moved_everywhere(a, b):
    """every weight of a differs from the same weight of b"""
    assert len(a) == len(b)
    return all((x != y) if not isinstance(x, tuple) else all(u != v for u, v in zip(x, y)) for x, y in zip(a, b))


@pytest.mark.parametrize("fam", [0, 1, 2])
def test_every_record_byte_moves_every_weight(api, oracle, fam):
    """flip each byte of element 0's commitments | proof record in turn: both elements' weights change (224 / 192 / 288 bytes)"""
    f = FAM[fam]
    P, Cm = honest(oracle, fam, 1, 2, tag=50 + fam)
    base = hook_weights(fam, api.debug_rlc_terms(fam, P, Cm, SEED))
    for j in range(f["cw"] + f["pw"]):
        p, c = P.copy(), Cm.copy()
        if j < f["cw"]:
            c[0, 0] = flip_canonical(oracle, c[0, 0], j, 1 << 30)
        else:
            p[0, 0] = flip_canonical(oracle, p[0, 0], j - f["cw"], f["z"])
        w = hook_weights(fam, api.debug_rlc_terms(fam, p, c, SEED))
        assert moved_everywhere(w, base), j


def test_every_crp_byte_moves_every_weight(api, oracle):
    """every byte of client 0's 128-byte proof, and one byte of one of its pairs, move rho of both clients"""
    P, Cm = honest(oracle, 3, 2, 1, tag=60)
    base = hook_weights(3, api.debug_rlc_terms(3, P, Cm, SEED))
    for j in range(129):
        p, c = P.copy(), Cm.copy()
        if j < 128:
            p[0] = flip_canonical(oracle, p[0], j, 64)
        else:
            c[0, 0, 7] ^= 0x10
        got = api.debug_rlc_terms(3, p, c, SEED)
        assert len(got["ranges"]) == 1, j
        assert moved_everywhere(hook_weights(3, got), base), j


@pytest.mark.parametrize("fam", [1, 2, 3])
def test_new_seed_moves_every_weight(api, oracle, fam):
    P, Cm = honest(oracle, fam, 2, 40, tag=70 + fam)
    a = hook_weights(fam, api.debug_rlc_terms(fam, P, Cm, SEED))
    b = hook_weights(fam, api.debug_rlc_terms(fam, P, Cm, bytes([0xa5]) + SEED[1:]))
    assert moved_everywhere(a, b)


# ---- adaptive forgery ---------------------------------------------------------------------------------------------------------------
def old_weight_sums(fam, P, Cm, w_of):
    """the fixed-base sums of the reference under fixed weights w_of(i) -> (sB, sH) mod l"""
    f = FAM[fam]
    rec = records(fam, P, Cm); sB = sH = 0
    for i in range(rec.shape[0]):
        z = [sc_int(rec[i, f["cw"] + f["z"] + 32 * q:f["cw"] + f["z"] + 32 * q + 32]) for q in range(2 if fam == 1 else 3)]
        _, b, h = sigma_terms(fam, w_of(i), z, 0)
        sB += b; sH += h
    return sB % L, sH % L


@pytest.mark.parametrize("fam", [0, 1, 2, 3])
def test_adaptive_forgery_is_rejected(api, oracle, fam):
    """a forger who predicts the weights makes two invalid proofs cancel under them (positive control: the reference's fixed-base sums
    under the predicted weights are unchanged); the real weights move and the check, batched and public, rejects both updates"""
    K, D = (3, 4) if fam == 3 else (2, 128)                       # at least 256 elements: the public calls take the batched path
    P, Cm = honest(oracle, fam, K, D, tag=80 + fam)
    delta = 0x1234567890abcdef1234567890abcdef
    pred = api.debug_rlc_terms(fam, P, Cm, SEED)
    if fam == 3:
        rho = check_crp(oracle, pred, P, Cm, SEED)
        i, j = 0, 2
        F = P.copy()
        F[i, 64:96] = np.frombuffer(b32(sc_int(P[i, 64:96]) + rho[j] * delta), np.uint8)
        F[j, 64:96] = np.frombuffer(b32(sc_int(P[j, 64:96]) - rho[i] * delta), np.uint8)
        old = lambda Q: sum(rho[k] * sc_int(Q[k, 64:96]) for k in range(K)) % L
        assert old(F) == old(P)                                   # positive control
        got = api.debug_rlc_terms(3, F, Cm, SEED)
        assert moved_everywhere(hook_weights(3, got), rho)
        assert got["held"] == 0 and got["ranges"][0]["is_id"] != (1, 1)
        single = [api.crp_verify(F[k], Cm[k]) for k in range(K)]
        assert single == [0, 1, 0]
        assert got["verdicts"] == single and api.crp_verify_batch(F, Cm, SEED).tolist() == single
        return
    f = FAM[fam]
    w = check_sigma(oracle, fam, pred, P, Cm, SEED)                # the predicted weights: the reference's, equal to the hook's
    i, j = 5, D + 17                                               # one element in each update
    q = {0: 2, 1: 0, 2: 2}[fam]                                    # the response changed: z_r2, z_m, z_r2
    wi = {0: 1, 1: 0, 2: 2}[fam]                                   # the weight it is multiplied by: sigma, rho, tau
    F = P.copy().reshape(K * D, -1)
    zo = f["z"] + 32 * q
    F[i, zo:zo + 32] = np.frombuffer(b32(sc_int(F[i, zo:zo + 32]) + w[j][wi] * delta), np.uint8)
    F[j, zo:zo + 32] = np.frombuffer(b32(sc_int(F[j, zo:zo + 32]) - w[i][wi] * delta), np.uint8)
    F = F.reshape(P.shape)
    full = lambda t: tuple(t) + (0,) * (3 - len(t))
    assert old_weight_sums(fam, F, Cm, lambda k: full(w[k])) == old_weight_sums(fam, P, Cm, lambda k: full(w[k]))      # positive control
    got = api.debug_rlc_terms(fam, F, Cm, SEED)
    assert moved_everywhere(hook_weights(fam, got), w)
    assert got["held"] == 0 and got["ranges"][0]["is_id"][0] == 0 and not any(got["ranges"][0]["bad"])
    single = [(api.square_verify, api.rand_verify, api.square_rand_verify)[fam](F[k], Cm[k]) for k in range(K)]
    assert single == [0, 0]
    assert got["verdicts"] == single
    if fam == 0:
        assert api.square_verify(F, Cm) == 0
    else:
        assert (api.rand_verify_batch if fam == 1 else api.square_rand_verify_batch)(F, Cm, SEED).tolist() == single


# ---- the device, at round sizes --------------------------------------------------------------------------------------------------
def gpu_proofs(api, fam, K, D, tag):
    rng = np.random.default_rng(tag)
    P, Cm = [], []
    for k in range(K):
        v = rng.uniform(-3, 3, D).astype(np.float32); r1 = api.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D)
        if fam == 1:
            rc, p, c = api.rand_prove(v, None, r1, 16, 7, bytes([(0x80 + k) & 0xff]) * 32)
        else:
            r2 = api.rnd_scalar_vec(bytes([(0x40 + tag + k) & 0xff]) * 32, D)
            rc, p, c = api.square_rand_prove(v, None, r1, r2, 32, 7, bytes([(0x80 + k) & 0xff]) * 32)
        assert rc == 0
        P.append(p); Cm.append(c)
    return np.stack(P), np.stack(Cm)


@pytest.mark.gpu
def test_gpu_rand_proofs_four_tree_levels(gpu_api, oracle):
    """N = 262 145 = 64^3 + 1: leaves -> 4097 -> 65 -> 2 -> root"""
    P, Cm = gpu_proofs(gpu_api, 1, 1, 262145, tag=1)
    got = gpu_api.debug_rlc_terms(1, P, Cm, SEED)
    check_sigma(oracle, 1, got, P, Cm, SEED, sample=(64, 4096, np.random.default_rng(5)))


@pytest.mark.gpu
def test_gpu_square_rand_round_48_clients(gpu_api, oracle):
    P, Cm = gpu_proofs(gpu_api, 2, 48, 50000, tag=2)
    got = gpu_api.debug_rlc_terms(2, P, Cm, SEED)
    check_sigma(oracle, 2, got, P, Cm, SEED, sample=(64, 4096, np.random.default_rng(6)))


@pytest.mark.gpu
def test_gpu_crp_two_groups_at_the_pair_limit(gpu_api, oracle):
    D, K = 900000, 2
    rng = np.random.default_rng(7)
    P, Cm = [], []
    for k in range(K):
        rc, p, c = gpu_api.crp_prove(rng.uniform(-3, 3, D).astype(np.float32), None, gpu_api.rnd_scalar_vec(bytes([k + 1]) * 32, D), 16, 7, bytes([k + 9]) * 32)
        assert rc == 0
        P.append(p); Cm.append(c)
    P, Cm = np.stack(P), np.stack(Cm)
    gpu_api.set_option("crp_batch_terms", D + 1)
    try:
        got = gpu_api.debug_rlc_terms(3, P, Cm, SEED)
    finally:
        gpu_api.set_option("crp_batch_terms", TERMS_MAX)
    assert len(got["ranges"]) == 2
    check_crp(oracle, got, P, Cm, SEED, D + 1, sample=(64, 4096, np.random.default_rng(8)))
