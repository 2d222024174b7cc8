"""The multiscalar-multiplication front end on its own (rofl_debug_msm: engine.cuh msm_plan_for / msm_plan_forced / run_msm / run_rt_msm and
kernels.cuh k_msm, k_bm_*, k_rt_msm, k_finalize), compared with exact references: the oracle's MSM over hash-to-group points and Bulletproofs
generators for short sums, points of known discrete logarithm (k_i B + u_i H) for sums of up to 2^22 + 1 terms.  Every window width and
path, the plan's switch points, and the inputs where bucket MSMs break: zero, l - 1, signed digits +B and -(B - 1) in every window (the
boundary buckets), one bucket taking every term, short and negated short scalars, duplicate points, P and -P, the identity as a base.
The "emu" cases run the product code under the CUDA-on-CPU emulation (tests/hostsim), the "gpu" ones on the device."""
import ctypes as C
import importlib.util
import os
import sys
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
L = 2**252 + 27742317777372353535851937790883648493
ZERO = bytes(32)
ERR_ARGS, ERR_POINT = -2, -4
BUILDS = [pytest.param("emu", id="emu"), pytest.param("gpu", id="gpu", marks=pytest.mark.gpu)]


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


# ---- scalars -------------------------------------------------------------------------------------------------------------
def nw_of(c):
    return (254 + c - 1) // c


def digits(x, c):
    """the product's signed recoding: digit_w = field_w(x + K) - (B - 1), K = sum_w (B - 1) 2^(cw), B = 2^(c-1)"""
    B, nw = 1 << (c - 1), nw_of(c)
    y = x + sum((B - 1) << (c * w) for w in range(nw))
    return [((y >> (c * w)) & ((1 << c) - 1)) - (B - 1) for w in range(nw)]


def crafted(c, target, rng, keep=1.0):
    """A reduced scalar whose signed digit is `target` (+B or -(B - 1)) in the non-top windows (each with probability `keep`, a random digit
    otherwise).  x = sum_w d_w 2^(cw) with every d_w in [-(B - 1), B] has exactly the digits d_w; the top digit and, where l leaves no room
    (c = 11: 23 windows reach bit 253), the highest windows are then moved just enough to bring x into [0, l)."""
    B, nw = 1 << (c - 1), nw_of(c)
    d = [target if rng.random() < keep else int(rng.integers(-(B - 1), B + 1)) for _ in range(nw - 1)] + [0]
    val = lambda: sum(dw << (c * w) for w, dw in enumerate(d))
    x = val()
    if x < 0:
        d[-1] = -(x >> (c * (nw - 1)))
        if val() >= L:
            d[-1] = 0
    for w in range(nw - 2, -1, -1):
        x = val()
        if 0 <= x < L:
            break
        if x < 0:
            d[w] += min(-(x >> (c * w)), B - d[w])
        else:
            d[w] -= min(-((L - 1 - x) >> (c * w)), d[w] + B - 1)
    x = val()
    assert 0 <= x < L and digits(x, c) == d
    return x


def rand_scalars(rng, n):
    return [int.from_bytes(rng.bytes(64), "little") % L for _ in range(n)]


EXTREMES = [0, 1, L - 1, L - 2, 2**252, 2**252 - 1]


def family(name, T, c, rng):
    if name == "random":
        return rand_scalars(rng, T)
    if name == "zero":
        return [0] * T
    if name == "mostly_zero":
        return [x if i % 7 == 3 else 0 for i, x in enumerate(rand_scalars(rng, T))]
    if name == "extremes":
        return [EXTREMES[i % len(EXTREMES)] for i in range(T)]
    if name == "equal":                     # every term in the same bucket of every window
        return [rand_scalars(rng, 1)[0]] * T
    if name == "short16":
        return [int(x) for x in rng.integers(0, 1 << 16, T)]
    if name == "short125":                  # the verifier's batching weights
        return [int.from_bytes(rng.bytes(16), "little") >> 3 for _ in range(T)]
    if name == "neg_short":
        return [L - 1 - int(x) for x in rng.integers(0, 1 << 16, T)]
    if name in ("plus_B", "minus_B"):       # the boundary buckets B - 1 and B - 2
        return [crafted(c, (1 << (c - 1)) if name == "plus_B" else -((1 << (c - 1)) - 1), rng, 1.0 if i % 4 == 0 else 0.8) for i in range(T)]
    if name == "mix":
        parts = [family(f, T, c, rng) for f in ("random", "extremes", "short16", "short125", "neg_short", "mostly_zero", "plus_B", "minus_B")]
        return [parts[i % len(parts)][i] for i in range(T)]
    raise ValueError(name)


def enc(xs):
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32)


# ---- points and references -----------------------------------------------------------------------------------------------
def neg(oracle, P):
    return oracle.point_sub(ZERO, P)


def hash_points(oracle, rng, T):
    """hash-to-group points, with an exact duplicate, a P / -P pair and the identity among the first terms"""
    P = [oracle.from_uniform_bytes(rng.bytes(64)) for _ in range(T)]
    if T > 3: P[3] = P[1]
    if T > 4: P[4] = neg(oracle, P[2])
    if T > 5: P[5] = ZERO
    if T > 130: P[128] = P[127]; P[129] = neg(oracle, P[126])
    return np.frombuffer(b"".join(P), np.uint8).reshape(T, 32)


def with_fixed(oracle, R, sB, sH):
    if sB is not None: R = oracle.point_add(R, oracle.scalarmult_base(int(sB).to_bytes(32, "little")))
    if sH is not None: R = oracle.point_add(R, oracle.scalarmult(int(sH).to_bytes(32, "little"), oracle.blinding_basepoint()))
    return R


def check(api, oracle, scal, pts, sB=None, sH=None, **kw):
    """run the hook on scal (list of n_msm scalar lists) over pts ([T, 32] shared or [n_msm, T, 32]) and compare with the oracle's MSM"""
    n = len(scal)
    rc, out, info = api.debug_msm(np.stack([enc(s) for s in scal]), pts, sB=None if sB is None else enc(sB), sH=None if sH is None else enc(sH), **kw)
    assert rc == 0, rc
    for k in range(n):
        P = pts if pts.ndim == 2 else pts[k]
        want = with_fixed(oracle, oracle.msm(enc(scal[k]), P), None if sB is None else sB[k], None if sH is None else sH[k])
        assert out[k].tobytes() == want, (k, info)
    return info


# ---- every window width and second knob ------------------------------------------------------------------------------------
SWEEP = [(c, k) for c in range(3, 9) for k in (1, 2, 3)] + [(c, k) for c in range(9, 17) for k in (1, 2, 8)]
T_EMU = [1, 2, 3, 127, 128, 129, 300]
T_GPU = [1, 3, 129, 300, 1025, 2049, 3000]
THIRD = ["equal", "zero", "plus_B", "neg_short", "minus_B", "short125", "extremes"]


@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("c,knob", SWEEP)
def test_every_window_width(api, oracle, build, c, knob):
    """Forced width c = 3 .. 16 with 1 - 3 slices (k_msm) or 1, 2, 8 parts per bucket (k_bm_*), then k_finalize's doubling chain (four lanes on
    the device, one under the emulation).  Three instances per call: a mix of every scalar family, the boundary digits +B / -(B - 1), and one
    family that loads a single bucket or none; shared and per-instance bases, with and without sB B + sH H."""
    i = SWEEP.index((c, knob))
    rng = np.random.default_rng(1000 + i)
    T = (T_EMU if build == "emu" else T_GPU)[i % 7]
    scal = [family("mix", T, c, rng), family("plus_B" if i % 2 else "minus_B", T, c, rng), family(THIRD[i % 7], T, c, rng)]
    if build == "emu":                                        # (the emulation runs every block of a cooperative launch on 128 - 256 OS threads:
        scal = scal[i % 3:] + scal[:i % 3]                    #  fewer instances there, the three kinds take turns at the front)
        scal = scal[:2 if c <= 6 else 1]
    n = len(scal)
    pts = hash_points(oracle, rng, T) if i % 2 else np.stack([hash_points(oracle, rng, T) for _ in range(n)])
    fixed = i % 3 == 0
    sB = rand_scalars(rng, n)[:-1] + [L - 1] if fixed else None
    sH = [0] + rand_scalars(rng, n - 1) if fixed else None
    info = check(api, oracle, scal, pts, sB, sH, path=1, c=c, knob=knob)
    assert info[0] == c and info[2] == int(c > 8) and (info[1] == knob if c > 8 else 1 <= info[1] <= knob)


@pytest.mark.parametrize("build,c", [pytest.param("emu", c, id=f"{c}-emu") for c in (None, 3, 5, 8, 9, 11, 13, 16)] +
                         [pytest.param("gpu", c, id=f"{c}-gpu", marks=pytest.mark.gpu) for c in [None] + list(range(3, 17))])
def test_cancelling_terms_give_the_identity(api, oracle, build, c):
    """(s, s) on (P, -P), (s, l - s) on (P, P), duplicates, the identity as a base and zero scalars: every instance sums to the identity, whose
    encoding is 32 zero bytes -- through the production plan and at every width on the device (a subset under the emulation)."""
    rng = np.random.default_rng(2000 + (c or 0))
    T = 128
    P = [oracle.from_uniform_bytes(rng.bytes(64)) for _ in range(T // 4)]
    pts, scal_a, scal_b = [], [], []
    for j, p in enumerate(P):
        s, t = rand_scalars(rng, 2)
        if j % 8 == 0: s = crafted(c or 9, 1 << ((c or 9) - 1), rng)
        last = j == len(P) - 1                                                              # identity bases: contribute nothing
        pts += [p, neg(oracle, p)] + ([ZERO, ZERO] if last else [p, p])
        scal_a += [s, s, t, L - t if t else 0]
        scal_b += [s if j % 2 else 0, s if j % 2 else 0, L - 1, 1 if not last else L - 2]
    pts = np.frombuffer(b"".join(pts), np.uint8).reshape(T, 32)
    kw = dict(path=0) if c is None else dict(path=1, c=c, knob=2)
    rc, out, info = api.debug_msm(np.stack([enc(scal_a), enc(scal_b), enc([0] * T)]), pts, **kw)
    assert rc == 0 and (out == 0).all(), info


@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("T", T_EMU)
def test_production_plan_small_sums(api, oracle, build, T):
    """msm_plan_for at small T (k_msm, the width msm_pick_c chooses): one and three instances, shared and per-instance bases, sB / sH."""
    rng = np.random.default_rng(3000 + T)
    pts = hash_points(oracle, rng, T)
    info = check(api, oracle, [family("mix", T, 9, rng)], pts, path=0)
    assert info[2] == 0
    scal = [family(f, T, info[0], rng) for f in ("plus_B", "equal", "minus_B")]
    check(api, oracle, scal, np.stack([hash_points(oracle, rng, T) for _ in range(3)]), [L - 1, 2**252, 0], rand_scalars(rng, 3), path=0)


def gens(oracle, n, m):
    """BulletproofGens(n, m) as the hook lays them out: G then H, party-major (j = party * n + i, k_gens_build)"""
    G = np.concatenate([oracle.bp_gens("G", j, n) for j in range(m)])
    H = np.concatenate([oracle.bp_gens("H", j, n) for j in range(m)])
    return np.concatenate([G, H])


@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("path,c,knob", [(0, 0, 1), (1, 4, 2), (1, 9, 2), (1, 12, 8), (2, 0, 1)])
def test_generator_bases(api, oracle, build, path, c, knob):
    """Niels-record generator bases (the verifier's d_gh layout), without tables through the plan / forced widths (several instances: the
    no-table layout of the prover's S), and through the radix-2^c tables (k_rt_msm, whatever radix the context builds)."""
    rng = np.random.default_rng(4000 + 10 * path + c)
    n, m = 8, 4
    T = 2 * n * m
    ref = gens(oracle, n, m)
    scal = [family(f, T, c or 8, rng) for f in ("mix", "plus_B", "equal")]
    sB, sH = rand_scalars(rng, 3), [L - 1, 0, 5]
    rc, out, info = api.debug_msm(np.stack([enc(s) for s in scal]), None, gen_n=n, path=path, c=c, knob=knob, sB=enc(sB), sH=enc(sH))
    assert rc == 0 and info[2] == (2 if path == 2 else int(info[0] > 8)) and (path != 1 or info[:2] == (c, knob))
    for k in range(3):
        assert out[k].tobytes() == with_fixed(oracle, oracle.msm(enc(scal[k]), ref), sB[k], sH[k]), (k, info)


@pytest.mark.parametrize("build", BUILDS)
def test_rejections(api, oracle, build):
    """A scalar >= l (the recoding assumes reduced scalars) is ROFL_ERR_ARGS on every path, an undecodable base ROFL_ERR_POINT."""
    rng = np.random.default_rng(5)
    T = 8
    pts = hash_points(oracle, rng, T)
    good = rand_scalars(rng, T)
    for bad in (L, L + 1, 2**253, 2**256 - 1):
        s = enc(good[:-1] + [bad])[None]
        for kw in (dict(path=0), dict(path=1, c=5), dict(path=1, c=10)):
            assert api.debug_msm(s, pts, **kw)[0] == ERR_ARGS
        assert api.debug_msm(enc(good[:4] + [bad] + good[5:])[None], None, gen_n=4, path=2)[0] == ERR_ARGS
        assert api.debug_msm(enc(good)[None], pts, sB=enc([bad]))[0] == ERR_ARGS
    badp = pts.copy(); badp[6] = 0xff; badp[6, 31] = 0x7f
    assert not oracle.point_valid(badp[6])
    assert api.debug_msm(enc(good)[None], badp, path=1, c=9)[0] == ERR_POINT
    assert api.debug_msm(np.stack([enc(good)] * 2), np.stack([pts, badp]), path=0)[0] == ERR_POINT
    assert api.debug_msm(enc(good)[None], pts, path=2)[0] == ERR_ARGS                   # tables exist for generators only
    assert api.debug_msm(enc(good)[None], None, gen_n=3, path=0)[0] == ERR_ARGS         # T is not 2 n m


# ---- device only: table radixes, tile / plan boundaries, sums of millions of terms ----------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bits,n,m", [(8, 16, 4), (9, 32, 2), (10, 64, 2), (11, 16, 8)])
def test_table_msm_every_radix(gpu, oracle, bits, n, m):
    """k_rt_msm over radix-2^8 .. 2^11 generator tables (all four radixes a B200 builds), several instances, sB / sH, against the oracle."""
    api = gpu
    rng = np.random.default_rng(6000 + bits)
    T = 2 * n * m
    ref = gens(oracle, n, m)
    scal = [family(f, T, bits, rng) for f in ("mix", "plus_B", "minus_B", "equal")]
    sB, sH = rand_scalars(rng, 4), rand_scalars(rng, 4)
    api.set_option("rt_bits", bits)
    try:
        rc, out, info = api.debug_msm(np.stack([enc(s) for s in scal]), None, gen_n=n, path=2, sB=enc(sB), sH=enc(sH))
    finally:
        api.set_option("rt_bits", 11)
    assert rc == 0 and info[0] == bits and info[2] == 2
    for k in range(4):
        assert out[k].tobytes() == with_fixed(oracle, oracle.msm(enc(scal[k]), ref), sB[k], sH[k]), k


class KnownBases:
    """P_i = k_i B + u_i H with small signed k_i, u_i (|k| < 2^15: the values k / 128 of 16-bit fixed point; |u| < 2^23), made by the product's
    commitment kernel and spot-checked against the oracle.  Every sum_i s_i P_i then has the exact value (sum s_i k_i) B + (sum s_i u_i) H,
    computed from 16-bit limbs of the scalars in int64 without overflow at 2^22 terms.  Crafted entries: the identity (k = u = 0), exact
    duplicates and P / -P pairs."""

    def __init__(self, api, oracle, N):
        rng = np.random.default_rng(7)
        k = rng.integers(-(1 << 15) + 1, 1 << 15, N).astype(np.int64); u = rng.integers(-(1 << 23), 1 << 23, N).astype(np.int64)
        i = np.arange(N)
        for r, f in ((5, None), (7, 1), (9, -1)):
            sel = i[(i % 101 == r)]
            if f is None: k[sel] = 0; u[sel] = 0
            else: k[sel] = f * k[sel - 1]; u[sel] = f * u[sel - 1]
        self.k, self.u = k, u
        bl = np.zeros((N, 32), np.uint8)
        lo = np.where(u >= 0, u, (L & (2**64 - 1)) + u).astype(np.uint64)          # l - |u| never borrows past the low 64 bits of l
        bl[:, :8] = lo[:, None].view(np.uint8).reshape(N, 8)
        bl[u < 0, 8:] = np.frombuffer(L.to_bytes(32, "little"), np.uint8)[8:]
        v = (k / 128).astype(np.float32)
        self.P = api.commit(v, bl, 16, 7)
        assert (self.P[:300] == oracle.commit_f32(v[:300], bl[:300], 16, 7)).all()
        assert (oracle.f32_to_scalar_vec(v[:300], 16, 7) == enc([int(x) % L for x in k[:300]])).all()
        assert (self.P[5] == 0).all() and (self.P[7] == self.P[6]).all() and oracle.point_add(self.P[8].tobytes(), self.P[9].tobytes()) == ZERO

    @staticmethod
    def dot(s, y):
        """sum_i s_i y_i mod l, s: [T, 32] scalars, y: int64"""
        acc = [0] * 16
        for a in range(0, s.shape[0], 1 << 18):
            limbs = np.ascontiguousarray(s[a:a + (1 << 18)]).view("<u2").astype(np.int64)
            part = (limbs * y[a:a + (1 << 18), None]).sum(axis=0)
            acc = [x + int(p) for x, p in zip(acc, part)]
        return sum(x << (16 * j) for j, x in enumerate(acc)) % L

    def expected(self, oracle, s, T):
        a, b = self.dot(s, self.k[:T]), self.dot(s, self.u[:T])
        return oracle.point_add(oracle.scalarmult_base(a.to_bytes(32, "little")), oracle.scalarmult(b.to_bytes(32, "little"), oracle.blinding_basepoint()))


N_BIG = (1 << 22) + 2


@pytest.fixture(scope="module")
def known(gpu, oracle):
    return KnownBases(gpu, oracle, N_BIG)


@pytest.fixture(scope="module")
def big_scalars():
    """random scalars below 2^252, with zero, 1, l - 1, l - 2, 2^252, 2^252 - 1, short and negated short scalars every 61 terms"""
    rng = np.random.default_rng(8)
    s = rng.integers(0, 256, (N_BIG, 32), dtype=np.uint8); s[:, 31] &= 0x0f
    edge = enc(EXTREMES + [12345, L - 12345, 1 << 124])
    pos = np.arange(3, N_BIG, 61)
    s[pos] = edge[np.arange(pos.size) % len(edge)]
    return s


def run_known(api, oracle, known, s, **kw):
    T = s.shape[1]
    rc, out, info = api.debug_msm(s, known.P[:T], **kw)
    assert rc == 0, rc
    for k in range(s.shape[0]):
        assert out[k].tobytes() == known.expected(oracle, s[k], T), (k, T, info)
    return info


def filled(T, x):
    return np.broadcast_to(np.frombuffer(int(x).to_bytes(32, "little"), np.uint8), (1, T, 32))


@pytest.mark.gpu
@pytest.mark.parametrize("c", range(3, 9))
def test_k_msm_tile_boundaries(gpu, oracle, known, big_scalars, c):
    """k_msm sorts MSM_SORT / wpb = 64 B terms per shared-memory tile: T = 64 B - 1, 64 B, 64 B + 1 (1 and 2 slices), plus one bucket holding
    every term of the sum (all scalars equal) and the boundary digits at 64 B + 1."""
    rng = np.random.default_rng(9000 + c)
    B = 1 << (c - 1)
    for T in (64 * B - 1, 64 * B, 64 * B + 1):
        for knob in (1, 2):
            assert run_known(gpu, oracle, known, big_scalars[None, :T], path=1, c=c, knob=knob)[:2] == (c, knob)
    T = 64 * B + 1
    run_known(gpu, oracle, known, np.concatenate([filled(T, rand_scalars(rng, 1)[0]), enc(family("plus_B", T, c, rng))[None]]), path=1, c=c, knob=1)


SWITCH = [(2047, 2048, 0), (2048, 2048, 1), (4095, 0, 0), (4096, 0, 0), (32767, 0, 0), (32768, 0, 1)] + \
         [(T, 0, 1) for k in range(16, 23) for T in ((1 << k) - 2, (1 << k) - 1, 1 << k)] + [((1 << 22) + 1, 0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("T,big_min,kernel", SWITCH)
def test_production_plan_switch_points(gpu, oracle, known, big_scalars, T, big_min, kernel):
    """msm_plan_for one term either side of every switch: k_msm <-> k_bm_* at big_min = 2048 (the verifier's threshold) and at the default
    32768, the slicing switch at 4096, and every width change of the wide-window plan, T + 1 = 2^16 .. 2^22 (c = 9 at big_min = 2048, 10 .. 16
    above 32768 terms, with the parts the plan picks: every fat top window).  Up to 2^20 terms the boundary digits +B of the width the plan
    chose are run as well."""
    rc_info = run_known(gpu, oracle, known, big_scalars[None, :T], path=0, big_min=big_min)
    assert rc_info[2] == kernel
    if kernel:
        assert rc_info[0] == max(9, min(16, T.bit_length() - 6))                         # ilog2_sz(T + 1) - 6
    if T == 4096:
        assert rc_info[1] > 1
    if T == 4095:
        assert rc_info[1] == 1
    if T <= (1 << 20):
        rng = np.random.default_rng(T)
        c = rc_info[0]
        fam = np.array(enc(family("plus_B", 512, c, rng)))
        s = fam[np.arange(T) % 512][None]
        assert run_known(gpu, oracle, known, s, path=0, big_min=big_min) == rc_info


@pytest.mark.gpu
@pytest.mark.parametrize("c", range(9, 17))
def test_wide_windows_forced_parts(gpu, oracle, known, big_scalars, c):
    """k_bm_* at every wide width with forced parts 1, 3 and 8 (the fat top windows of c = 9 .. 14 dealt out as parts_top threads; c = 13 takes
    k_bm_reduce's branch for 128 and more top buckets), boundary digits, and one bucket holding all 2^20 terms (8 parts: 2^17 additions)."""
    rng = np.random.default_rng(10000 + c)
    T = 40000
    fams = np.stack([enc(family(f, 256, c, rng)) for f in ("plus_B", "minus_B")])
    s = np.concatenate([big_scalars[None, :T], fams[:, np.arange(T) % 256]])
    for knob in (1, 3, 8):
        assert run_known(gpu, oracle, known, s, path=1, c=c, knob=knob) == (c, knob, 1)
    run_known(gpu, oracle, known, filled(1 << 20, L - 1), path=1, c=c, knob=8)
