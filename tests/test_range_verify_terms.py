"""The range-proof verifier's batched check (engine.cuh verify_chunks), term by term, against an exact restatement of Bulletproofs' verification
equation and of the weights of DESIGN.md §2.

verify_chunks checks every chunk of a call -- and of a whole round in the batch calls -- with ONE random linear combination.  Honest proofs pass
under any weights, so verdict tests cannot see a root that leaves out a digest, a key that ignores the shard offset or a weight that does not bind
some proof field; each of those lets a prover who knows the seed make errors in two chunks cancel.  Here the records of the test hook
rofl_debug_range_terms (copies of the device buffers verify_chunks filled, nothing derived) are compared with this file's reference: the
oracle's own transcript code for the challenges and digests (oracle.rp_challenges), hashlib SHA3-256 and ChaCha20 for the weights, Python integers
mod l for every scalar, s_k from the bits of k, and oracle.msm over the restated scalars for the equation itself.  The "emu" tests run the product
code under the CUDA-on-CPU emulation (tests/hostsim), the gpu ones on the device at production shapes."""
import ctypes as C
import hashlib
import importlib.util
import multiprocessing
import os
import sys
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
L = 2**252 + 27742317777372353535851937790883648493
SEED = bytes(range(32))
DOM_RANGE, DOM_L2 = 2, 5


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


def values(rng, D, n, n_bits, tag):
    """D values inside the clip bounds of an n-bit range, both bounds included"""
    mn, mx = rng_bounds(n, n_bits)
    v = np.random.default_rng(tag).uniform(mn, mx, D).astype(np.float32)
    v[:min(D, 2)] = [mx, mn][:min(D, 2)]
    return v


def rng_bounds(n, n_bits):
    import oracle
    return oracle.clip_bounds(n, n_bits, 7)


def linf(oracle, D, n, P, tag=1, shifts=None):
    """an honest L-infinity update from the oracle: (proofs [P', plen], commits [D, 32]); shifts: the same proofs with t_x_blinding of
    chunk c shifted by shifts[c] before it is absorbed (a forger who knows the witness)"""
    n_bits = max(16, n)
    v = values(None, D, n, n_bits, tag); bl = oracle.rnd_scalar_vec(bytes([tag & 0xff]) * 32, D); seed = bytes([(tag + 0x40) & 0xff]) * 32
    if shifts is None:
        rc, p, c = oracle.range_prove(v, bl, n, P, n_bits, 7, seed)
    else:
        rc, p, c = oracle.range_prove_tx_bl_shifted(v, bl, n, P, np.concatenate([np.frombuffer(b32(x), np.uint8) for x in shifts]), n_bits, 7, seed)
    assert rc == 0
    return p, c


def l2(oracle, K, n, tag=1):
    """K honest sum-of-squares proofs: (proofs [K, plen], commits [K, 32])"""
    P, Cm = [], []
    for k in range(K):
        v = np.random.default_rng(tag * 1000 + k).uniform(-0.05, 0.05, 4).astype(np.float32)
        rc, p, c = oracle.l2_prove(v, oracle.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, 4), n, 32, 7, bytes([(tag + 2 * k + 1) & 0xff]) * 32)
        assert rc == 0
        P.append(p); Cm.append(c)
    return np.stack(P), np.stack(Cm)


# ---- the reference -------------------------------------------------------------------------------------------------------------
def sha3(b):
    return hashlib.sha3_256(b).digest()


def le(x, n):
    return int(x).to_bytes(n, "little")


def sc_int(b):
    return int.from_bytes(bytes(b), "little")


def b32(x):
    return (x % L).to_bytes(32, "little")


def inv(x):
    return pow(x, L - 2, L)


def shifted(oracle, commits, n, total):
    """what the L-infinity transcript absorbs: commitment + 2^(n-1) B, then identity encodings (32 zero bytes) up to `total` positions"""
    c = np.ascontiguousarray(commits.reshape(-1, 32))
    off = np.frombuffer(oracle.scalarmult_base(b32(1 << (n - 1))), np.uint8)
    out = np.zeros((total, 32), np.uint8)
    out[:c.shape[0]] = oracle.aggregate(np.stack([c, np.broadcast_to(off, c.shape)]))
    return out


def weights_of(oracle, seed, digests, dom, c_off):
    """root = SHA3-256(seed | LE64 C | digest_0 .. digest_(C-1)); key_i = SHA3-256(root | LE32 dom | LE64 (c_off + i));
    c_i, rho_i = ChaCha20 blocks 0 and 1 of key_i, each a 64-byte little-endian integer mod l"""
    root = sha3(seed + le(len(digests), 8) + b"".join(digests))
    cs, rhos = [], []
    for i in range(len(digests)):
        key = sha3(root + le(dom, 4) + le(c_off + i, 8))
        cs.append(sc_int(oracle.chacha20_block(key, 0)) % L); rhos.append(sc_int(oracle.chacha20_block(key, 1)) % L)
    return cs, rhos


def ref_call(oracle, proofs, V, n, m, seed, dom, c_off=0, label=0, weights=None):
    """Everything verify_chunks computes for C chunks (proofs [C, plen], V [C m, 32] as absorbed), except g / h (gh_ref).
    weights = (c, rho) replaces the derived weights (the forger's prediction)."""
    C = proofs.shape[0]; N = n * m; lgN = N.bit_length() - 1; lgm = m.bit_length() - 1
    vch, dig = [], []
    for c in range(C):
        _, ch, d = oracle.rp_challenges(proofs[c], V[c * m:(c + 1) * m], n, m, label)
        vch.append([sc_int(x) for x in ch]); dig.append(d)
    cs, rhos = weights_of(oracle, seed, dig, dom, c_off) if weights is None else weights
    chal, small, var, par = [], [], [], []
    for c in range(C):
        y, z, x, w = vch[c][:4]; u = vch[c][4:]; ui = [inv(t) for t in u]
        pf = proofs[c]; ipp = 224
        t_x, t_xb, e_bl = (sc_int(pf[o:o + 32]) for o in (128, 160, 192))
        a, b = sc_int(pf[ipp + 64 * lgN:ipp + 64 * lgN + 32]), sc_int(pf[ipp + 64 * lgN + 32:ipp + 64 * lgN + 64])
        cc, rho = cs[c], rhos[c]
        delta = (z - z * z) * power_sum(y, N) - z ** 3 * (2 ** n - 1) * power_sum(z, m)
        chal.append([rho * z, rho * z * z, rho * a, rho * b, cc] + u + ui)
        small.append([rho, rho * x, rho * cc * x, rho * cc * x * x] + [rho * t * t for t in u] + [rho * t * t for t in ui]
                     + [-rho * (e_bl + cc * t_xb), rho * (w * (t_x - a * b) + cc * (delta - t_x))])
        e = rho * cc * z * z % L
        for _ in range(m):
            var.append(e); e = e * z % L
        par.append((rho, z, a, b, inv(y), u, ui))
    return dict(C=C, n=n, m=m, lgN=lgN, lgm=lgm, vch=vch, digest=dig, cs=cs, rhos=rhos, chal=chal, small=small, var=var, par=par)


def power_sum(x, count):
    """sum_{i < count} x^i mod l, term by term"""
    s, e = 0, 1
    for _ in range(count):
        s += e; e = e * x % L
    return s % L


def _nibble_tables(pairs):
    """pairs[p] = (factor when bit p of the index is 1, when it is 0) -> per group of 4 bits the 16 products"""
    tabs = []
    for q in range(0, len(pairs), 4):
        grp = pairs[q:q + 4]; t = []
        for e in range(1 << len(grp)):
            v = 1
            for r, (one, zero) in enumerate(grp):
                v = v * (one if (e >> r) & 1 else zero) % L
            t.append(v)
        tabs.append(t)
    return tabs


def _pick(tabs, k):
    v = 1
    for q, t in enumerate(tabs):
        v = v * t[(k >> (4 * q)) & 15]
    return v % L


def _gh_chunks(args):
    """sums over some chunks of g_k = -(rho z + rho a s_k), h_k = rho z + y^-k (rho z^2 z^j 2^i - rho b s_k^-1), k = j n + i, at positions ks.
    s_k = prod_p (bit p of k ? u_(lgN-1-p) : u_(lgN-1-p)^-1) and the powers from the bits of k and j (four bits at a time)"""
    par, ks, n, lgN, lgm = args
    g = [0] * len(ks); h = [0] * len(ks)
    for rho, z, a, b, yi, u, ui in par:
        S = _nibble_tables([(u[lgN - 1 - p], ui[lgN - 1 - p]) for p in range(lgN)])
        Si = _nibble_tables([(ui[lgN - 1 - p], u[lgN - 1 - p]) for p in range(lgN)])
        Y = _nibble_tables([(pow(yi, 1 << p, L), 1) for p in range(lgN)])
        Z = _nibble_tables([(pow(z, 1 << p, L), 1) for p in range(lgm)])
        rz, rzz, ra, rb = rho * z % L, rho * z * z % L, rho * a % L, rho * b % L
        for t, k in enumerate(ks):
            j, i = divmod(k, n)
            g[t] -= rz + ra * _pick(S, k)
            h[t] += rz + _pick(Y, k) * (rzz * _pick(Z, j) * (1 << i) - rb * _pick(Si, k))
    return [x % L for x in g], [x % L for x in h]


def gh_ref(ref, ks):
    """(g_k, h_k) at positions ks, summed over every chunk of the call (worker processes when the call is large)"""
    par, n, lgN, lgm = ref["par"], ref["n"], ref["lgN"], ref["lgm"]
    work = len(par) * len(ks)
    procs = min(os.cpu_count() or 1, 32) if work > 2_000_000 else 1
    if procs == 1:
        return _gh_chunks((par, ks, n, lgN, lgm))
    step = -(-len(par) // procs)
    with multiprocessing.get_context("fork").Pool(procs) as pool:
        parts = pool.map(_gh_chunks, [(par[i:i + step], ks, n, lgN, lgm) for i in range(0, len(par), step)])
    return [sum(p[0][t] for p in parts) % L for t in range(len(ks))], [sum(p[1][t] for p in parts) % L for t in range(len(ks))]


def as_rows(xs):
    return np.frombuffer(b"".join(b32(x) for x in xs), np.uint8).reshape(-1, 32)


def same(got, want, what):
    """byte-for-byte equality of [*, 32] arrays, naming the first differing row"""
    got = np.asarray(got).reshape(-1, 32); want = np.asarray(want).reshape(-1, 32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, f"{what}: first difference at row {bad[0]} of {got.shape[0]}"


def check_rec(rec, ref, seed, dom, c_off=0, ks=None):
    """every tapped value of one verify_chunks record equals the reference; g / h at the positions ks (default: all)"""
    C, lgN, m = ref["C"], ref["lgN"], ref["m"]
    assert (rec["C"], rec["n"], rec["m"], rec["lgN"], rec["c_off"], rec["dom"]) == (C, ref["n"], m, lgN, c_off, dom)
    same(rec["vch"], as_rows([x for r in ref["vch"] for x in r]), "y z x w u")
    assert [bytes(d) for d in rec["digest"]] == ref["digest"], "digest"
    same(rec["cs"], as_rows(ref["cs"]), "c"); same(rec["rho"], as_rows(ref["rhos"]), "rho")
    same(rec["chal"], as_rows([x for r in ref["chal"] for x in r]), "chal block")
    same(rec["small"], as_rows([x for r in ref["small"] for x in r]), "small-point scalars")
    same(rec["var"], as_rows(ref["var"]), "commitment scalars")
    N = 1 << lgN
    ks = list(range(N)) if ks is None else sorted(set(ks))
    g, h = gh_ref(ref, ks)
    same(rec["g"][ks], as_rows(g), "g"); same(rec["h"][ks], as_rows(h), "h")
    assert len(set(bytes(x) for x in rec["cs"]) | set(bytes(x) for x in rec["rho"])) == 2 * C, "a weight repeats"


def equation_points(oracle, proofs, V, n, m):
    """G | H | V | per chunk A S T_1 T_2 L.. R.. H B -- the bases of the restated equation, in the tap's scalar order"""
    C = proofs.shape[0]; lgN = (n * m).bit_length() - 1
    G = np.concatenate([oracle.bp_gens("G", j, n) for j in range(m)]); H = np.concatenate([oracle.bp_gens("H", j, n) for j in range(m)])
    Hb, B = np.frombuffer(oracle.blinding_basepoint(), np.uint8), np.frombuffer(oracle.basepoint(), np.uint8)
    sp = []
    for c in range(C):
        pf = proofs[c].reshape(-1, 32)
        sp += [pf[0], pf[1], pf[2], pf[3]] + [pf[7 + 2 * k] for k in range(lgN)] + [pf[8 + 2 * k] for k in range(lgN)] + [Hb, B]
    return np.concatenate([G, H, V[:C * m], np.stack(sp)])


def equation_holds(oracle, ref, proofs, V):
    """the whole restated equation: sum of g G + h H + commitment and proof-point terms == identity"""
    N = 1 << ref["lgN"]
    g, h = gh_ref(ref, list(range(N)))
    sc = as_rows(g + h + ref["var"] + [x for r in ref["small"] for x in r])
    return oracle.msm(sc, equation_points(oracle, proofs, V, ref["n"], ref["m"])) == bytes(32)


def full_check(oracle, rec, proofs, V, n, m, seed, dom, c_off=0, label=0):
    ref = ref_call(oracle, proofs, V, n, m, seed, dom, c_off, label)
    check_rec(rec, ref, seed, dom, c_off)
    assert equation_holds(oracle, ref, proofs, V) == (rec["id"] == 1)
    return ref


# ---- exact equality, emulation ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m", [(8, 1), (8, 2), (16, 2), (8, 8), (32, 4), (64, 4), (64, 8)])     # lgN 3 .. 9, lgm 0 .. 3, range 64
def test_shapes_exact(api, oracle, n, m):
    p, c = linf(oracle, m * 4 - 1, n, 4, tag=n + m)                 # Dp = 4 m in four chunks: the last position is identity padding
    got = api.debug_range_terms(0, p, c, n, SEED)
    assert got["verdicts"] == [1] == [oracle.range_verify(p, c, n, SEED)]
    assert len(got["recs"]) == 1
    full_check(oracle, got["recs"][0], p, shifted(oracle, c, n, 4 * m), n, m, SEED, DOM_RANGE)


# (D, proofs made, proofs checked): C = 1, 3, 4, 5, 20, 21 chunks of m = 1.  40 + 32 C is a multiple of the SHA3 rate (136) at C = 3 and 20;
# C = 5 is past the four chunk lanes of k_verify_scalars; D = 19 pads positions 19 .. 31 with the identity, and 21 proofs do not divide Dp = 32
@pytest.mark.parametrize("D,P,C", [(1, 1, 1), (4, 4, 3), (4, 4, 4), (8, 8, 5), (32, 32, 20), (19, 32, 21)])
def test_chunk_counts_exact(api, oracle, D, P, C):
    p, c = linf(oracle, D, 8, P, tag=C)
    got = api.debug_range_terms(0, p[:C], c, 8, SEED)
    assert got["verdicts"] == [oracle.range_verify(p[:C], c, 8, SEED)] == [1]
    full_check(oracle, got["recs"][0], p[:C], shifted(oracle, c, 8, max(C, D)), 8, 1, SEED, DOM_RANGE)


def test_shard_exact(api, oracle):
    """chunks [1, 3) of a 4-chunk update as a shard: the keys use c_off + i"""
    p, c = linf(oracle, 14, 8, 4, tag=7)                            # m = 4; the shard holds positions 4 .. 11
    got = api.debug_range_terms(0, p[1:3], c[4:12], 8, SEED, chunk_len=4, chunk_begin=1)
    assert got["verdicts"] == [1]
    full_check(oracle, got["recs"][0], p[1:3], shifted(oracle, c[4:12], 8, 8), 8, 4, SEED, DOM_RANGE, c_off=1)


@pytest.mark.parametrize("K", [1, 2, 5])
def test_batch_exact(api, oracle, K):
    ups = [linf(oracle, 3, 8, 2, tag=20 + k) for k in range(K)]    # D = 3 of Dp = 4: one identity position per client
    P, Cm = np.stack([u[0] for u in ups]), np.stack([u[1] for u in ups])
    got = api.debug_range_terms(1, P, Cm, 8, SEED)
    assert got["verdicts"] == [1] * K and len(got["recs"]) == 1
    V = np.concatenate([shifted(oracle, Cm[k], 8, 4) for k in range(K)])
    full_check(oracle, got["recs"][0], P.reshape(2 * K, -1), V, 8, 2, SEED, DOM_RANGE)


@pytest.mark.parametrize("K", [1, 3, 20, 257])
def test_l2_exact(api, oracle, K):
    """K = 1 the single call, else the L2 batch (K = 257 chunks is past the 256 threads of k_verify_keys); commitments are not shifted"""
    P, Cm = l2(oracle, K, 8 if K > 3 else 32, tag=K)
    n = 8 if K > 3 else 32
    got = api.debug_range_terms(2 if K == 1 else 3, P[0] if K == 1 else P, Cm[0] if K == 1 else Cm, n, SEED)
    assert got["verdicts"] == [oracle.l2_verify(P[k], Cm[k], n, SEED) for k in range(K)] == [1] * K
    assert len(got["recs"]) == 1
    full_check(oracle, got["recs"][0], P, Cm.reshape(-1, 32), n, 1, SEED, DOM_L2, label=1)


@pytest.mark.parametrize("host_ts,use_rt", [(0, 0), (0, 1), (8192, 1)])
def test_transcript_and_generator_paths(api, oracle, host_ts, use_rt):
    """commitments absorbed on the host (ts_host_m = 0) or the device, fixed generators through the tables or the bucket MSM"""
    p, c = linf(oracle, 16, 16, 4, tag=40)
    api.set_option("ts_host_m", host_ts); api.set_use_rt(use_rt)
    try:
        got = api.debug_range_terms(0, p, c, 16, SEED)
    finally:
        api.set_option("ts_host_m", 8192); api.set_use_rt(1)
    rec = got["recs"][0]
    assert got["verdicts"] == [1] and rec["rt"] == use_rt and rec["win"] > 0
    full_check(oracle, rec, p, shifted(oracle, c, 16, 16), 16, 4, SEED, DOM_RANGE)


# ---- binding -----------------------------------------------------------------------------------------------------------------------
def fields(lgN):
    """(name, offset, is_point) of every 32-byte field of a proof"""
    f = [("A", 0, 1), ("S", 32, 1), ("T_1", 64, 1), ("T_2", 96, 1), ("t_x", 128, 0), ("t_x_blinding", 160, 0), ("e_blinding", 192, 0)]
    for k in range(lgN):
        f += [(f"L_{k}", 224 + 64 * k, 1), (f"R_{k}", 256 + 64 * k, 1)]
    return f + [("a", 224 + 64 * lgN, 0), ("b", 256 + 64 * lgN, 0)]


def moved(oracle, p, off, is_point):
    """the field at `off` replaced by a different valid value: point + B, scalar + 1"""
    q = p.copy()
    new = oracle.point_add(bytes(p[off:off + 32]), oracle.basepoint()) if is_point else b32(sc_int(p[off:off + 32]) + 1)
    q[off:off + 32] = np.frombuffer(new, np.uint8)
    return q


def weights(rec):
    return [bytes(x) for x in rec["cs"]], [bytes(x) for x in rec["rho"]]


def all_moved(a, b):
    return all(x != y for x, y in zip(a[0] + a[1], b[0] + b[1]))


@pytest.mark.parametrize("chunk", [0, 1])
def test_every_proof_field_moves_every_weight(api, oracle, chunk):
    p, c = linf(oracle, 4, 8, 2, tag=50)                            # two chunks, lgN = 4
    base = weights(api.debug_range_terms(0, p, c, 8, SEED)["recs"][0])
    for name, off, pt in fields(4):
        q = p.copy(); q[chunk] = moved(oracle, p[chunk], off, pt)
        got = api.debug_range_terms(0, q, c, 8, SEED)
        assert len(got["recs"]) == 1 and got["verdicts"] == [0], name
        assert all_moved(weights(got["recs"][0]), base), name


def test_commitments_seed_and_shard_offset_move_every_weight(api, oracle):
    p, c = linf(oracle, 4, 8, 2, tag=51)
    base = weights(api.debug_range_terms(0, p, c, 8, SEED)["recs"][0])
    for j in range(4):
        d = c.copy(); d[j] = np.frombuffer(oracle.point_add(bytes(c[j]), oracle.basepoint()), np.uint8)
        assert all_moved(weights(api.debug_range_terms(0, p, d, 8, SEED)["recs"][0]), base), j
    assert all_moved(weights(api.debug_range_terms(0, p, c, 8, bytes([0xa5]) + SEED[1:])["recs"][0]), base)
    a = api.debug_range_terms(0, p, c, 8, SEED, chunk_len=2, chunk_begin=0)
    b = api.debug_range_terms(0, p, c, 8, SEED, chunk_len=2, chunk_begin=1)
    assert weights(a["recs"][0]) == base and a["verdicts"] == b["verdicts"] == [1]
    assert all_moved(weights(b["recs"][0]), base)


# ---- tamper matrix ------------------------------------------------------------------------------------------------------------------
UNDECODABLE = bytes([1]) + bytes(31)                               # s = 1 is negative: not an encoding


def tampers(oracle, p, lgN):
    """(label, tampered proof, expected bad flag on the chunk) for one proof: every point as the identity, undecodable and another valid
    point; every scalar + 1 and once non-canonical (l itself)"""
    out = []
    for name, off, pt in fields(lgN):
        if pt:
            for kind, val in (("identity", bytes(32)), ("undecodable", UNDECODABLE)):
                q = p.copy(); q[off:off + 32] = np.frombuffer(val, np.uint8); out.append((f"{name} {kind}", q, 1))
            out.append((f"{name} moved", moved(oracle, p, off, 1), 0))
        else:
            out.append((f"{name} + 1", moved(oracle, p, off, 0), 0))
            q = p.copy(); q[off:off + 32] = np.frombuffer(L.to_bytes(32, "little"), np.uint8); out.append((f"{name} non-canonical", q, None))
    return out


def test_tamper_matrix_single_call(api, oracle):
    p, c = linf(oracle, 3, 8, 4, tag=60)                            # four chunks of m = 1 (lgN = 3), one identity position; chunk 1 tampered
    for label, q, bad in tampers(oracle, p[1], 3):
        P = p.copy(); P[1] = q
        got = api.debug_range_terms(0, P, c, 8, SEED)
        want = oracle.range_verify(P, c, 8, SEED)
        assert got["verdicts"] == [want], label
        if bad is None:
            assert want == -1 and got["recs"] == [], label
            continue
        assert want == 0 and len(got["recs"]) == 1, label
        rec = got["recs"][0]
        assert rec["bad"] == [0, bad, 0, 0], label
        if not bad:                                                # a valid but wrong value: the equation is still restated exactly, and fails
            assert rec["id"] == 0, label
            full_check(oracle, rec, P, shifted(oracle, c, 8, 4), 8, 1, SEED, DOM_RANGE)
    d = c.copy(); d[2] = np.frombuffer(UNDECODABLE, np.uint8)
    got = api.debug_range_terms(0, p, d, 8, SEED)
    assert got["verdicts"] == [oracle.range_verify(p, d, 8, SEED)] == [-4] and len(got["recs"]) == 1


def test_tamper_batch_and_l2(api, oracle):
    """a failing batch is followed by one re-check per client; the verdicts are the oracle's per client"""
    K = 3
    ups = [linf(oracle, 2, 8, 2, tag=70 + k) for k in range(K)]
    P, Cm = np.stack([u[0] for u in ups]), np.stack([u[1] for u in ups])
    picks = {"A identity", "L_0 undecodable", "T_1 moved", "t_x + 1", "b non-canonical"}
    for label, q, bad in tampers(oracle, P[1, 0], 3):
        if label not in picks:
            continue
        T = P.copy(); T[1, 0] = q
        got = api.debug_range_terms(1, T, Cm, 8, SEED)
        want = [oracle.range_verify(T[k], Cm[k], 8, SEED) for k in range(K)]
        assert got["verdicts"] == want and want[1] in (0, -1) and want[0] == want[2] == 1, label
        recs = got["recs"]
        if bad is None:                                            # malformed: no batch, the other clients one by one
            assert [r["C"] for r in recs] == [2, 2], label
        else:
            assert [r["C"] for r in recs] == [2 * K, 2, 2, 2] and [r["id"] for r in recs[1:]] == [1, 0, 1], label
            assert recs[0]["bad"] == [0, 0, bad, 0, 0, 0], label
    d = Cm.copy(); d[2, 1] = np.frombuffer(UNDECODABLE, np.uint8)
    got = api.debug_range_terms(1, P, d, 8, SEED)
    assert got["verdicts"] == [1, 1, -4] == [oracle.range_verify(P[k], d[k], 8, SEED) for k in range(K)]
    assert [r["C"] for r in got["recs"]] == [2 * K, 2, 2, 2]
    LP, LC = l2(oracle, K, 8, tag=80)
    for label, q, bad in tampers(oracle, LP[1], 3):
        if label not in picks:
            continue
        T = LP.copy(); T[1] = q
        want = [oracle.l2_verify(T[k], LC[k], 8, SEED) for k in range(K)]
        assert api.debug_range_terms(3, T, LC, 8, SEED)["verdicts"] == want, label
        assert api.debug_range_terms(2, T[1], LC[1], 8, SEED)["verdicts"] == [want[1]] == [api.l2_verify(T[1], LC[1], 8, SEED)], label
    d = LC.copy(); d[0] = np.frombuffer(UNDECODABLE, np.uint8)
    assert api.debug_range_terms(3, LP, d, 8, SEED)["verdicts"] == [oracle.l2_verify(LP[k], d[k], 8, SEED) for k in range(K)] == [-4, 1, 1]


# ---- adaptive forgery ------------------------------------------------------------------------------------------------------------
DELTA = 0x1234567890abcdef1234567890abcdef


def cancelling(cs, rhos):
    """t_x_blinding shifts d0, d1 of chunks 0 and 1 with rho0 c0 d0 + rho1 c1 d1 = 0: their -c d B_blinding errors cancel under (c, rho)"""
    return [rhos[1] * cs[1] * DELTA % L, -rhos[0] * cs[0] * DELTA % L]


def test_adaptive_forgery_is_rejected(api, oracle):
    """a forger who knows the witness and predicts the weights from the honest proofs re-proves two chunks with shifted t_x_blinding so that
    their errors cancel under those weights (positive control: the restated equation under the predicted weights is the identity).  The real
    weights move with the forged bytes, and the hook, range_verify and the oracle reject."""
    p, c = linf(oracle, 4, 8, 2, tag=90)
    V = shifted(oracle, c, 8, 4)
    pred = ref_call(oracle, p, V, 8, 2, SEED, DOM_RANGE)
    check_rec(api.debug_range_terms(0, p, c, 8, SEED)["recs"][0], pred, SEED, DOM_RANGE)
    F, c2 = linf(oracle, 4, 8, 2, tag=90, shifts=cancelling(pred["cs"], pred["rhos"]))
    assert (c2 == c).all() and (F[:, :160] == p[:, :160]).all() and (F[:, 160:192] != p[:, 160:192]).any(axis=1).all()
    assert equation_holds(oracle, ref_call(oracle, F, V, 8, 2, SEED, DOM_RANGE, weights=(pred["cs"], pred["rhos"])), F, V)   # positive control
    got = api.debug_range_terms(0, F, c, 8, SEED)
    rec = got["recs"][0]
    assert all_moved(weights(rec), (as_list(pred["cs"]), as_list(pred["rhos"]))) and rec["id"] == 0 and rec["bad"] == [0, 0]
    full_check(oracle, rec, F, V, 8, 2, SEED, DOM_RANGE)
    assert got["verdicts"] == [0] == [oracle.range_verify(F, c, 8, SEED)] == [api.range_verify(F, c, 8, SEED)]


def test_adaptive_forgery_across_clients_is_rejected(api, oracle):
    """the same forgery spread over two clients of one round: the batch fails and the per-client re-checks reject both"""
    ups = [linf(oracle, 2, 8, 1, tag=91 + k) for k in range(2)]
    P, Cm = np.stack([u[0] for u in ups]), np.stack([u[1] for u in ups])
    V = np.concatenate([shifted(oracle, Cm[k], 8, 2) for k in range(2)])
    pred = ref_call(oracle, P.reshape(2, -1), V, 8, 2, SEED, DOM_RANGE)
    check_rec(api.debug_range_terms(1, P, Cm, 8, SEED)["recs"][0], pred, SEED, DOM_RANGE)
    d = cancelling(pred["cs"], pred["rhos"])
    F = np.stack([linf(oracle, 2, 8, 1, tag=91 + k, shifts=[d[k]])[0] for k in range(2)])
    assert equation_holds(oracle, ref_call(oracle, F.reshape(2, -1), V, 8, 2, SEED, DOM_RANGE, weights=(pred["cs"], pred["rhos"])), F.reshape(2, -1), V)
    got = api.debug_range_terms(1, F, Cm, 8, SEED)
    assert [r["C"] for r in got["recs"]] == [2, 1, 1] and [r["id"] for r in got["recs"]] == [0, 0, 0]
    assert all_moved(weights(got["recs"][0]), (as_list(pred["cs"]), as_list(pred["rhos"])))
    assert got["verdicts"] == [0, 0] == [oracle.range_verify(F[k], Cm[k], 8, SEED) for k in range(2)] == api.range_verify_batch(F, Cm, 8, SEED).tolist()


def as_list(xs):
    return [b32(x) for x in xs]


# ---- the device-pointer entry points ----------------------------------------------------------------------------------------------
def test_dev_entry_points_match_host_calls(api, oracle):
    """range_prove_dev / range_verify_dev (what bench.py times) against range_prove / range_verify; numpy pointers stand in for device ones"""
    D, n, P = 13, 8, 4
    v = values(None, D, n, 16, 95); bl = oracle.rnd_scalar_vec(b"\x07" * 32, D); seed = b"\x08" * 32
    rc, ph, ch = api.range_prove(v, bl, n, P, 16, 7, seed)
    cd = np.zeros((D, 32), np.uint8)
    rc2, pd = api.range_prove_dev(v.ctypes.data, bl.ctypes.data, D, n, P, 16, 7, seed, cd.ctypes.data)
    assert rc == rc2 == 0 and (pd == ph).all() and (cd == ch).all()
    assert api.range_verify_dev(pd, cd.ctypes.data, D, n, SEED) == api.range_verify(ph, ch, n, SEED) == 1
    full_check(oracle, api.debug_range_terms(0, pd, cd, n, SEED)["recs"][0], pd, shifted(oracle, cd, n, 16), n, 4, SEED, DOM_RANGE)
    bad = pd.copy(); bad[2, 170] ^= 1
    assert api.range_verify_dev(bad, cd.ctypes.data, D, n, SEED) == api.range_verify(bad, ch, n, SEED) == oracle.range_verify(bad, ch, n, SEED) == 0


# ---- the device, at production shapes -----------------------------------------------------------------------------------------------
def seams_and_sample(N, count, seed):
    L2 = (N.bit_length() - 1) // 2
    return sorted(set(np.random.default_rng(seed).integers(0, N, count).tolist()) | {0, (1 << L2) - 1, 1 << L2, N - 1})


@pytest.mark.gpu
@pytest.mark.parametrize("use_rt", [1, 0])
def test_gpu_configs1_shape(gpu_api, oracle, use_rt):
    """configs[1]: 16-bit, 64 chunks of 1024 values, every term and the whole equation"""
    D, n, P = 65536, 16, 64
    v = values(None, D, n, 16, 101); bl = gpu_api.rnd_scalar_vec(b"\x11" * 32, D)
    rc, p, c = gpu_api.range_prove(v, bl, n, P, 16, 7, b"\x12" * 32)
    assert rc == 0
    gpu_api.set_use_rt(use_rt)
    try:
        got = gpu_api.debug_range_terms(0, p, c, n, SEED)
    finally:
        gpu_api.set_use_rt(1)
    rec = got["recs"][0]
    assert got["verdicts"] == [1] and rec["rt"] == use_rt and rec["id"] == 1
    full_check(oracle, rec, p, shifted(oracle, c, n, D), n, 1024, SEED, DOM_RANGE)


@pytest.mark.gpu
def test_gpu_round_48_clients(gpu_api, oracle):
    """the configs[4] round: 48 clients x 50 000 values, range 8, 64 proofs each -> C = 3072 chunks, N = 8192; the public *_dev path on
    torch CUDA tensors for one client"""
    import torch
    K, D, n, P = 48, 50000, 8, 64
    Ps, Cs = [], []
    for k in range(K):
        v = values(None, D, n, 16, 200 + k); bl = gpu_api.rnd_scalar_vec(bytes([k + 1]) * 32, D)
        rc, p, c = gpu_api.range_prove(v, bl, n, P, 16, 7, bytes([k + 100]) * 32)
        assert rc == 0
        Ps.append(p); Cs.append(c)
        if k == 0:
            vd, bd = torch.from_numpy(v).cuda(), torch.from_numpy(bl).cuda(); cd = torch.zeros((D, 32), dtype=torch.uint8, device="cuda")
            rc, pd = gpu_api.range_prove_dev(vd.data_ptr(), bd.data_ptr(), D, n, P, 16, 7, bytes([k + 100]) * 32, cd.data_ptr())
            torch.cuda.synchronize()
            assert rc == 0 and (pd == p).all() and (cd.cpu().numpy() == c).all()
            assert gpu_api.range_verify_dev(pd, cd.data_ptr(), D, n, SEED) == 1
            bad = pd.copy(); bad[5, 170] ^= 1
            assert gpu_api.range_verify_dev(bad, cd.data_ptr(), D, n, SEED) == 0
    P_, C_ = np.stack(Ps), np.stack(Cs)
    got = gpu_api.debug_range_terms(1, P_, C_, n, SEED)
    assert got["verdicts"] == [1] * K and len(got["recs"]) == 1
    rec = got["recs"][0]
    assert rec["C"] == K * P and rec["lgN"] == 13
    V = np.concatenate([shifted(oracle, C_[k], n, 65536) for k in range(K)])
    ref = ref_call(oracle, P_.reshape(K * P, -1), V, n, 1024, SEED, DOM_RANGE)
    check_rec(rec, ref, SEED, DOM_RANGE, ks=seams_and_sample(8192, 4096, 3))


@pytest.mark.gpu
def test_gpu_configs3_chunk(gpu_api, oracle):
    """one configs[3]-sized chunk: m = 2^18 (8-bit, N = 2^21), commitments absorbed on the host"""
    D, n = 1 << 18, 8
    v = values(None, D, n, 16, 300); bl = gpu_api.rnd_scalar_vec(b"\x31" * 32, D)
    rc, p, c = gpu_api.range_prove(v, bl, n, 1, 16, 7, b"\x32" * 32)
    assert rc == 0
    got = gpu_api.debug_range_terms(0, p, c, n, SEED)
    rec = got["recs"][0]
    assert got["verdicts"] == [1] and rec["id"] == 1 and rec["m"] == D
    ref = ref_call(oracle, p, shifted(oracle, c, n, D), n, D, SEED, DOM_RANGE)
    check_rec(rec, ref, SEED, DOM_RANGE, ks=seams_and_sample(n * D, 4096, 4))
