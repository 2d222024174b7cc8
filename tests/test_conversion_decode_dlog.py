"""The three pieces of device code every value passes through on its way into and out of the library, each compared with a plain restatement
of its definition in Python integers / Fraction (not with the oracle) at the edges where such code goes wrong:

  1. f32 -> fixed point -> scalar (devfn.cuh f32_to_fix / f32_to_scalar: k_f32_to_scalar, k_commit) at all 52 formats: ties at every frac,
     the saturation threshold of every width, zeros of both signs, infinities, subnormals, FLT_MAX, NaN.
  2. scalar -> f32 (devfn.cuh scalar_to_f32: k_scalar_to_f32, bsgs_solve_point) at the same formats, including the scalars whose sign rule is
     odd (byte 31 != 0 is negative, so [2^248, l) counts as negative) and the ones that decode to -0.0.
  3. The shifted commitments of the range prover (k_commit in shift mode) at the clip bounds of every range / width pair.
  4. Ristretto decoding (ge25519.cuh ge_decompress, RFC 9496 4.3.1): one verdict per candidate, with the check that rejects it named, so that
     non-canonical, negative-s, non-square, negative-t and y = 0 encodings are each aimed at rather than hit by chance.
  5. BSGS decryption (bsgs_solve_point through k_bsgs_solve and k_acc_extract) at the giant-step boundaries, the last giant step, the sign
     fallback, the truncation to the table's width, tables that are not powers of two, and the table whose giant step is the identity.
  6. rofl_dlog / rofl_acc_extract refuse an unsupported fixed-point format like every other entry point.

The "emu" cases run the product code under the CUDA-on-CPU emulation (tests/hostsim), the "gpu" ones on the device.  Outputs must equal the
restatements exactly: bytes for scalars and points, bit patterns (the sign of zero included) for f32."""
import ctypes as C
import importlib.util
import math
import os
import sys
from collections import Counter
from fractions import Fraction
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
L = 2**252 + 27742317777372353535851937790883648493
P = 2**255 - 19
ERR_ARGS, ERR_POINT, ERR_DLOG, ERR_NAN = -2, -4, -5, -98
VALUE_OUT_OF_RANGE = 2
BUILDS = [pytest.param("emu", id="emu"), pytest.param("gpu", id="gpu", marks=pytest.mark.gpu)]
WIDTHS = (8, 16, 32, 64)
FORMATS = [(nb, fr) for nb in WIDTHS for fr in range(13)]
F32 = np.float32


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(HERE, "hostsim")
    locked_make(d, "libemul.so", env={"CXX": "g++"})
    spec = importlib.util.spec_from_file_location("rofl_ffi", os.path.join(ROOT, "rofl-project-code_b200", "_ffi.py"))
    ffi = importlib.util.module_from_spec(spec); spec.loader.exec_module(ffi)
    a = ffi.Api(C.CDLL(os.path.join(d, "libemul.so")))
    yield a
    a.close()


@pytest.fixture(scope="module")
def gpu():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    return g.load_package().context(0)          # raises (no CPU fallback) if the CUDA library or the device is missing


@pytest.fixture
def api(request, build):
    return request.getfixturevalue(build)


def enc(xs):
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32)


def ints(a):
    return [int.from_bytes(r.tobytes(), "little") for r in np.asarray(a, np.uint8).reshape(-1, 32)]


def bits(f):
    return np.asarray(f, np.float32).view(np.uint32)


def base_mul(oracle, x):
    return oracle.scalarmult_base((x % L).to_bytes(32, "little"))


def rc_of(call):
    """the library's return code of a call the binding raises on"""
    try:
        call()
    except Exception as ex:                                      # RoflError of whichever binding module loaded the library
        if not hasattr(ex, "code"):
            raise
        return ex.code
    return 0


# ---- 1 / 2: the restatements of conversion32.rs ------------------------------------------------------------------------------
def f32_nearest(n):
    """the f32 nearest to the integer n >= 0 (ties to even), as an integer"""
    sh = max(n.bit_length() - 24, 0)
    q, r = divmod(n, 1 << sh)
    if 2 * r > (1 << sh) or (2 * r == (1 << sh) and q & 1):
        q += 1
    return q << sh


def to_scalar(x, nb, fr):
    """conversion32.rs:11-22: raw = Fix::saturating_from_float(|x|).to_bits() -- |x| 2^fr rounded half to even, at most 2^nb - 1 (inf
    saturates) -- negated mod l when x < 0"""
    x = float(x)
    raw = 2**nb - 1 if math.isinf(x) else min(round(Fraction(abs(x)) * 2**fr), 2**nb - 1)
    return (-raw) % L if x < 0 else raw


def to_f32(s, nb, fr):
    """conversion32.rs:24-34: byte 31 != 0 is negative; the magnitude is the low nb bits of s (or of l - s), over 2^fr, correctly rounded"""
    neg = (s >> 248) != 0
    mag = ((L - s) if neg else s) & (2**nb - 1)
    v = F32(f32_nearest(mag) / 2**fr)                            # exact: at most 24 significant bits over a power of two
    return -v if neg else v


def up(x):
    return np.nextafter(F32(x), F32(np.inf))


def down(x):
    return np.nextafter(F32(x), F32(-np.inf))


TIE_K = list(range(40)) + [127, 128, 255, 256, 2**15 - 1, 2**15, 2**16 - 1, 2**23 - 1]


def edge_values(nb, fr, rng, n_random=600):
    """±0, ±inf, the smallest subnormal and normal, ±FLT_MAX; every tie (k + 1/2) / 2^fr of TIE_K with its two f32 neighbours; the f32 values
    around (2^nb - 1/2) / 2^fr and (2^nb - 1) / 2^fr (the saturation threshold); magnitudes spread over the format's range and beyond;
    random finite bit patterns.  Each with both signs."""
    fi = np.finfo(np.float32)
    v = [0.0, np.inf, fi.smallest_subnormal, 2 * fi.smallest_subnormal, fi.tiny, fi.max, 1.0]
    for k in TIE_K:
        t = F32((k + 0.5) / 2**fr)
        v += [t, down(t), up(t)]
    for top in (2**nb - 0.5, 2**nb - 1, 2**nb):
        t = F32(top / 2**fr)
        v += [t, down(t), up(t)]
    mag = np.exp2(rng.uniform(-fr - 3, nb - fr + 3, n_random)).astype(np.float32)
    pat = rng.integers(0, 1 << 31, n_random, dtype=np.uint32).view(np.float32)
    v += list(mag) + list(pat[np.isfinite(pat)])
    v = np.array(v, np.float32)
    return np.concatenate([v, -v])


@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("nb,fr", FORMATS)
def test_f32_to_scalar_and_back(api, build, nb, fr):
    """rofl_f32_to_scalar_vec against to_scalar, then rofl_scalar_to_f32_vec on those scalars and on scalars of every sign / width class
    against to_f32, bit for bit."""
    rng = np.random.default_rng(100 * nb + fr)
    v = edge_values(nb, fr, rng)
    got = api.f32_to_scalar_vec(v, nb, fr)
    want = [to_scalar(x, nb, fr) for x in v]
    bad = [(float(x), g, w) for x, g, w in zip(v, ints(got), want) if g != w]
    assert not bad, (len(bad), bad[:5])

    special = [0, 1, L - 1, L - 2, 2**248 - 1, 2**248, 2**248 + 1, L - 2**248 - 1, L - 2**248, L - 2**248 + 1]
    for k in WIDTHS:
        special += [2**k - 1, 2**k, 2**k + 1, L - 2**k + 1, L - 2**k, L - 2**k - 1]    # L - 2^k: low k bits of l - s are zero -> -0.0
    rand = [int.from_bytes(rng.bytes(32), "little") % L for _ in range(200)]
    rand += [int(x) for x in rng.integers(0, 2**63, 100)] + [L - int(x) for x in rng.integers(1, 2**63, 100)]
    rand += [2**248 + int.from_bytes(rng.bytes(31), "little") % (L - 2**248) for _ in range(100)]     # "negative" with a large l - s
    rand += [int.from_bytes(rng.bytes(31), "little") for _ in range(100)]                             # below 2^248, junk above bit 64
    s = want + special + rand
    back = api.scalar_to_f32_vec(enc(s), nb, fr)
    ref = np.array([to_f32(x, nb, fr) for x in s], np.float32)
    bad = np.nonzero(bits(back) != bits(ref))[0]
    assert bad.size == 0, (bad.size, [(hex(s[i]), float(back[i]), float(ref[i])) for i in bad[:5]])


@pytest.mark.parametrize("build", BUILDS)
def test_nan_is_refused(api, build):
    """Fix::saturating_from_float panics on NaN: ROFL_ERR_NAN from the conversion and from a commitment, whatever the NaN's sign and payload
    and wherever it sits in the vector"""
    nans = np.array([0x7fc00000, 0xffc00000, 0x7f800001, 0xffffffff], np.uint32).view(np.float32)
    for nb, fr in ((8, 0), (16, 7), (64, 12)):
        for n in nans:
            v = np.array([0.5, -3.0, n, 1.0], np.float32)
            assert rc_of(lambda: api.f32_to_scalar_vec(v, nb, fr)) == ERR_NAN
            assert rc_of(lambda: api.commit(v, None, nb, fr)) == ERR_NAN


@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("nb,fr", [(8, 0), (8, 12), (16, 7), (32, 3), (64, 12)])
def test_commit_converts_like_the_restatement(api, oracle, build, nb, fr):
    """k_commit's own conversion: rofl_commit(v, no blinding) = to_scalar(v) B for the edge values of the format"""
    v = edge_values(nb, fr, np.random.default_rng(7 * nb + fr), n_random=40 if build == "emu" else 400)
    got = api.commit(v, None, nb, fr)
    for i, x in enumerate(v):
        assert got[i].tobytes() == base_mul(oracle, to_scalar(x, nb, fr)), (i, float(x))


# ---- 3: the range prover's shifted commitments at the clip bounds -----------------------------------------------------------------
RANGE_GRID = [(nb, r) for nb in WIDTHS for r in WIDTHS if r <= nb]


def clip_max(r, fr):
    """conversion32.rs:56-60: the largest value of range r, (2^(r-1) - 1) / 2^fr, as the f32 nearest to it"""
    return F32(f32_nearest(2**(r - 1) - 1) / 2**fr)


@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("nb,r", RANGE_GRID)
@pytest.mark.parametrize("fr", [0, 7, 12])
def test_range_commitments_at_the_clip_bounds(api, oracle, build, nb, r, fr):
    """rofl_range_prove with zero blindings at mn, mx, their f32 neighbours, ±0 and small values.  The f32 bound check alone decides between
    rc 0 and VALUE_OUT_OF_RANGE (one call per rejected value); the accepted values go into one call whose commitments must be
    ((sh - 2^(r-1)) mod l) B with sh the low nb bits of (to_scalar(x) + 2^(r-1)) mod l -- the wrap to sh = 0 at mx when f32 rounds mx up to
    2^(r-1) / 2^fr included -- and whose proof verifies exactly when every sh is below 2^r."""
    if build == "emu" and (r == 64 or (r == 32 and fr != 7)):
        pytest.skip("64-bit and most 32-bit ranges on the device only: their generator tables are slow to build under the emulation")
    mx = clip_max(r, fr)
    mn = -mx
    assert api.clip_bounds(r, nb, fr) == (float(mn), float(mx))
    small = [F32(k / 2**fr) for k in (0.5, 1, 1.5, 3)]                 # with the bounds: 15 values accepted, one chunk of 16
    cand = [mn, mx, down(mn), up(mn), down(mx), up(mx), F32(0.0), F32(-0.0), F32(mx / 3)] + small + [-x for x in small]
    inside = [x for x in cand if mn <= x <= mx]
    outside = [x for x in cand if not mn <= x <= mx]
    assert len(outside) == 2 and len(inside) == len(cand) - 2
    for x in outside:
        v = np.array([0.0, x], np.float32)
        assert api.range_prove(v, np.zeros((2, 32), np.uint8), r, 1, nb, fr, bytes(32))[0] == VALUE_OUT_OF_RANGE, float(x)
    off = 2**(r - 1)
    sh = [((to_scalar(x, nb, fr) + off) % L) & (2**nb - 1) for x in inside]
    # r - 1 > 24: mx rounds up to 2^(r-1) / 2^fr, so raw + 2^(r-1) = 2^r.  At r = nb that wraps to 0; below nb it stays 2^r, outside the
    # range, and the reference proves it all the same: a proof that does not verify (range_proof_vec/mod.rs:26-43 checks in f32 only)
    assert sum(x > 0 and s == 0 for x, s in zip(inside, sh)) == (r == nb and r > 24)
    assert sum(s >= 2**r for s in sh) == (r < nb and r > 24)
    seed = bytes([r, nb, fr]) * 8 + bytes(8)
    sets = [list(range(len(inside)))]
    if max(sh) >= 2**r:
        sets.append([i for i, s in enumerate(sh) if s < 2**r])
    for idx in sets:
        v = np.array([inside[i] for i in idx], np.float32)
        rc, proofs, commits = api.range_prove(v, np.zeros((v.size, 32), np.uint8), r, 1, nb, fr, seed)
        assert rc == 0
        for j, i in enumerate(idx):
            assert commits[j].tobytes() == base_mul(oracle, sh[i] - off), (i, float(inside[i]))
        assert api.range_verify(proofs, commits, r, seed) == int(max(sh[i] for i in idx) < 2**r)


# ---- 4: Ristretto decoding, RFC 9496 4.3.1 --------------------------------------------------------------------------------------
D_EDW = (-121665 * pow(121666, P - 2, P)) % P
SQRT_M1 = 19681161376707505956807079304988542015446066515923890162744021073123829784752


def is_neg(x):
    return (x % P) & 1


def sqrt_ratio_m1(u, v):
    """RFC 9496 4.2 SQRT_RATIO_M1 -> (was_square, r)"""
    u, v = u % P, v % P
    r = u * pow(v, 3, P) * pow(u * pow(v, 7, P), (P - 5) // 8, P) % P
    check = v * r * r % P
    correct, flipped, flipped_i = check == u, check == (-u) % P, check == (-u * SQRT_M1) % P
    if flipped or flipped_i:
        r = r * SQRT_M1 % P
    if is_neg(r):
        r = P - r
    return correct or flipped, r


def decode_verdict(b):
    """RFC 9496 4.3.1 Decode, returning which check rejects b (in the RFC's order), or "ok" """
    s = int.from_bytes(b, "little")
    if s >= P:
        return "non_canonical"
    if is_neg(s):
        return "negative_s"
    ss = s * s % P
    u1, u2 = (1 - ss) % P, (1 + ss) % P
    u2_sqr = u2 * u2 % P
    v = (-(D_EDW * u1 * u1) - u2_sqr) % P
    was_square, invsqrt = sqrt_ratio_m1(1, v * u2_sqr)
    den_x = invsqrt * u2 % P
    den_y = invsqrt * den_x * v % P
    x = 2 * s * den_x % P
    if is_neg(x):
        x = P - x
    y = u1 * den_y % P
    t = x * y % P
    if not was_square:
        return "not_square"
    if is_neg(t):
        return "negative_t"
    if y == 0:
        return "y_zero"
    return "ok"


REJECTIONS = ("non_canonical", "negative_s", "not_square", "negative_t", "y_zero")


def decode_candidates(oracle, rng):
    """encodings of random points (multiples of B and hash-to-group points) and the identity; s + 2^255 and s + p of some of them; p + k for
    k < 19; p - s; small and random even s (not square / negative t); s = p - 1 (y = 0)"""
    ok = [base_mul(oracle, int(x)) for x in rng.integers(1, 2**62, 24)] + [oracle.from_uniform_bytes(rng.bytes(64)) for _ in range(24)] + [bytes(32)]
    cands = list(ok)
    for b in ok[:16]:
        s = int.from_bytes(b, "little")
        cands += [s + 2**255, (P - s) % P] + ([s + P] if s + P < 2**256 else [])
    cands += [P + k for k in range(19)] + [P - 1, P - 2, 1, 2**255 - 1, 2**256 - 1]
    cands += list(range(0, 300, 2)) + [2 * int(x) % P for x in rng.integers(0, 2**63, 200)] + [int.from_bytes(rng.bytes(32), "little") >> 1 for _ in range(100)]
    return [c if isinstance(c, bytes) else int(c).to_bytes(32, "little") for c in cands]


@pytest.mark.parametrize("build", BUILDS)
def test_decoding_verdicts(api, oracle, build):
    """rofl_acc_add (D = 1, one candidate per client) accepts exactly the encodings RFC 9496 decodes; the accepted ones come back unchanged from
    export and sum to the chain of oracle.point_add; rofl_dlog and rofl_aggregate refuse one candidate of every rejection class"""
    rng = np.random.default_rng(41)
    cands = decode_candidates(oracle, rng)
    verdict = [decode_verdict(b) for b in cands]
    count = Counter(verdict)
    assert all(count[c] for c in REJECTIONS + ("ok",)), count
    recs = np.frombuffer(b"".join(cands), np.uint8).reshape(-1, 1, 32)
    with api.accumulator(1, 32, 0) as acc:
        added = acc.add(recs)
        bad = [(i, verdict[i], int(added[i])) for i in range(len(cands)) if int(added[i]) != (1 if verdict[i] == "ok" else ERR_POINT)]
        assert not bad, (len(bad), bad[:8])
        total = bytes(32)
        for b, vd in zip(cands, verdict):
            if vd == "ok":
                total = oracle.point_add(total, b)
        assert acc.export()[0].tobytes() == total
    good = np.frombuffer(b"".join(b for b, vd in zip(cands, verdict) if vd == "ok"), np.uint8).reshape(-1, 32)
    with api.accumulator(good.shape[0], 32, 0) as acc:
        assert acc.add(good[None]).tolist() == [1]
        assert (acc.export() == good).all()
    for cls in REJECTIONS:
        b = np.frombuffer(cands[verdict.index(cls)], np.uint8).reshape(1, 32)
        assert api.dlog(b, 1 << 4, 8, 8, 0)[0] == ERR_POINT, cls
        pts = np.stack([good[:3], np.concatenate([good[3:5], b])])
        assert rc_of(lambda: api.aggregate(pts, 0)) == ERR_POINT, cls


# ---- 5: BSGS decryption, bsgs32.rs restated on discrete logarithms ----------------------------------------------------------------
def bsgs(x, m, nbits):
    """solve_discrete_log_with_neg for x B: the table maps i B -> i as a u<nbits> for i in 0..=m (size = m), max_it = 2^nbits / m giant
    steps of -(m & vmask) B from M, then from -M; the result (it size + v) & vmask, negated mod l when found from -M; None on a miss"""
    vmask = 2**nbits - 1
    max_it = 2**nbits // m
    for sign in (1, -1):
        cur = sign * x % L
        for it in range(max_it):
            if cur <= m:
                v = (it * m + (cur & vmask)) & vmask
                return v if sign == 1 else (-v) % L
            cur = (cur - (m & vmask)) % L
    return None


BSGS_CONFIGS = [(16, 8), (7, 8), (10, 8), (300, 8), (256, 8), (1 << 9, 16), (1000, 16), (3, 4), (5, 3)]


def bsgs_xs(m, nbits):
    """±(k m + {-1, 0, 1}) for k = 0 .. max_it + 1, 0, 1, ±2^nbits, ±(2^nbits ± 1), l - 1 (and ±65536, ±65537 for the 2^16 table)"""
    xs = {k * m + d for k in range(2**nbits // m + 2) for d in (-1, 0, 1)} | {0, 1, 2**nbits - 1, 2**nbits, 2**nbits + 1, 65536, 65537}
    return sorted({x for x in xs if x >= 0} | {-x for x in xs}) + [L - 1]


@pytest.mark.parametrize("build,m,nbits", [pytest.param(b, m, n, id=f"{m}-{n}-{b}", marks=[pytest.mark.gpu] if b == "gpu" else [])
                                           for b in ("emu", "gpu") for m, n in BSGS_CONFIGS] +
                         [pytest.param("gpu", 1 << 16, 16, id="65536-16-gpu", marks=pytest.mark.gpu)])
def test_bsgs_decryption(api, oracle, build, m, nbits):
    """rofl_dlog on x B and rofl_acc_extract on one client of records (x B, B) (init at the identity: the R check passes and L is a resident,
    non-affine point): the found x give bsgs()'s scalar and to_f32 of it at several formats; every miss is ROFL_ERR_DLOG on its own.
    With m = 2^nbits the giant step m & vmask is zero: 65536 B decrypts to 0 with the server's 2^16 table (SURVEY B.3)."""
    xs = bsgs_xs(m, nbits)
    want = {x: bsgs(x, m, nbits) for x in xs}
    hits = [x for x in xs if want[x] is not None]
    misses = [x for x in xs if want[x] is None]
    assert misses and (hits or m > 2**nbits)
    if m == 1 << 16:
        assert want[65536] == 0 and want[-65536] == 0 and want[65537] is None and want[-65537] is None
    formats = [(16, 7), (8, 0), (64, 12)] if build == "gpu" else [(16, 7), (64, 12)]
    if hits:
        pts = np.stack([np.frombuffer(base_mul(oracle, x), np.uint8) for x in hits])
        ref = enc([want[x] for x in hits])
        for nb, fr in formats:
            rc, s, f = api.dlog(pts, m, nbits, nb, fr)
            assert rc == 0
            bad = [(hits[i], ints(s[i])[0], want[hits[i]]) for i in range(len(hits)) if not (s[i] == ref[i]).all()]
            assert not bad, (len(bad), bad[:5])
            assert (bits(f) == bits([to_f32(want[x], nb, fr) for x in hits])).all()
        recs = np.zeros((1, len(hits), 64), np.uint8)
        recs[0, :, :32] = pts
        recs[0, :, 32:] = np.frombuffer(oracle.basepoint(), np.uint8)
        with api.accumulator(len(hits), 64, 0) as acc:
            assert acc.add(recs).tolist() == [1]
            for nb, fr in formats[:2]:
                rc, s, f = acc.extract(m, nbits, nb, fr)
                assert rc == 0 and (s == ref).all()
                assert (bits(f) == bits([to_f32(want[x], nb, fr) for x in hits])).all()
    for x in misses:
        pt = np.frombuffer(base_mul(oracle, x), np.uint8).reshape(1, 32)
        assert api.dlog(pt, m, nbits, 16, 7)[0] == ERR_DLOG, x
        with api.accumulator(1, 64, 0) as acc:
            acc.add(np.concatenate([pt, np.frombuffer(oracle.basepoint(), np.uint8).reshape(1, 32)], axis=1).reshape(1, 1, 64))
            assert acc.extract(m, nbits, 16, 7)[0] == ERR_DLOG, x


# ---- 6: unsupported fixed-point formats -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("build", BUILDS)
def test_dlog_and_extract_refuse_unsupported_formats(api, oracle, build):
    """n_bits outside {8, 16, 32, 64} or frac outside 0..12 is ROFL_ERR_ARGS from rofl_dlog and rofl_acc_extract, as from every other call
    that takes a format (frac = -1 used to shift 1u by -1 in fix_to_f32); nothing is written to the outputs"""
    pt = np.frombuffer(base_mul(oracle, 300), np.uint8).reshape(1, 32)
    assert api.dlog(pt, 1 << 9, 16, 16, 7)[0] == 0
    with api.accumulator(1, 32, 0) as acc:
        acc.add(pt.reshape(1, 1, 32))
        assert acc.extract(1 << 9, 16, 16, 7)[0] == 0
        for nb, fr in ((12, 7), (0, 7), (16, -1), (16, 13), (16, 40)):
            for rc, s, f in (api.dlog(pt, 1 << 9, 16, nb, fr), acc.extract(1 << 9, 16, nb, fr)):
                assert rc == ERR_ARGS and not s.any() and not f.any(), (nb, fr)
