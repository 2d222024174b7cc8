"""ORACLE -- test infrastructure only.  ctypes loader for oracle/librofl_oracle.so (CPU restatement of the
rofl_crypto hot path).  Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs; the product package never imports this module."""
import ctypes as C
import os
import subprocess
import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_DIR, "librofl_oracle.so")


def build(force=False):
    srcs = [os.path.join(_DIR, f) for f in os.listdir(_DIR) if f.endswith((".c", ".h"))]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        subprocess.check_call(["make", "-C", _DIR, "-s"], env={**os.environ, "CC": "gcc"})
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.orc_next_pow2.restype = C.c_size_t
        _lib.orc_next_pow2.argtypes = [C.c_size_t]
        _lib.orc_rp_proof_len.restype = C.c_size_t
        _lib.orc_rp_proof_len.argtypes = [C.c_size_t]
        _lib.orc_l2_clip_bound.restype = C.c_float
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _u8(x, n=None):
    a = np.ascontiguousarray(np.frombuffer(bytes(x), dtype=np.uint8) if isinstance(x, (bytes, bytearray)) else x, dtype=np.uint8)
    if n is not None:
        assert a.size == n, (a.size, n)
    return a


def _f32(x):
    return np.ascontiguousarray(x, dtype=np.float32)


SEED0 = bytes(32)

# ---- primitives -------------------------------------------------------------------------------
def _bin32(name):
    def f(a, b):
        o = np.zeros(32, np.uint8); getattr(lib(), name)(_p(o), _p(_u8(a, 32)), _p(_u8(b, 32))); return o.tobytes()
    return f
sc_mul, sc_add, sc_sub, fe_mul = _bin32("orc_sc_mul"), _bin32("orc_sc_add"), _bin32("orc_sc_sub"), _bin32("orc_fe_mul")
def sc_invert(a):
    o = np.zeros(32, np.uint8); lib().orc_sc_invert(_p(o), _p(_u8(a, 32))); return o.tobytes()
def fe_invert(a):
    o = np.zeros(32, np.uint8); lib().orc_fe_invert(_p(o), _p(_u8(a, 32))); return o.tobytes()
def sc_reduce_wide(a):
    o = np.zeros(32, np.uint8); lib().orc_sc_reduce_wide(_p(o), _p(_u8(a, 64))); return o.tobytes()
def sc_is_canonical(a): return bool(lib().orc_sc_is_canonical(_p(_u8(a, 32))))
def basepoint():
    o = np.zeros(32, np.uint8); lib().orc_basepoint(_p(o)); return o.tobytes()
def blinding_basepoint():
    o = np.zeros(32, np.uint8); lib().orc_blinding_basepoint(_p(o)); return o.tobytes()
def scalarmult(s, p):
    o = np.zeros(32, np.uint8); rc = lib().orc_scalarmult(_p(o), _p(_u8(s, 32)), _p(_u8(p, 32))); assert rc == 0; return o.tobytes()
def scalarmult_base(s):
    o = np.zeros(32, np.uint8); lib().orc_scalarmult_base(_p(o), _p(_u8(s, 32))); return o.tobytes()
def point_add(a, b):
    o = np.zeros(32, np.uint8); rc = lib().orc_point_add(_p(o), _p(_u8(a, 32)), _p(_u8(b, 32))); assert rc == 0; return o.tobytes()
def point_sub(a, b):
    o = np.zeros(32, np.uint8); rc = lib().orc_point_sub(_p(o), _p(_u8(a, 32)), _p(_u8(b, 32))); assert rc == 0; return o.tobytes()
def point_valid(a): return bool(lib().orc_point_valid(_p(_u8(a, 32))))
def from_uniform_bytes(b):
    o = np.zeros(32, np.uint8); lib().orc_from_uniform_bytes(_p(o), _p(_u8(b, 64))); return o.tobytes()
def msm(scalars, points):
    s, p = _u8(scalars), _u8(points); n = s.size // 32; assert p.size == s.size
    o = np.zeros(32, np.uint8); rc = lib().orc_msm(_p(o), _p(s), _p(p), C.c_size_t(n)); assert rc == 0; return o.tobytes()
def sha3_512(m):
    o = np.zeros(64, np.uint8); a = _u8(m); lib().orc_sha3_512(_p(o), _p(a), C.c_size_t(a.size)); return o.tobytes()
def sha3_256(m):
    o = np.zeros(32, np.uint8); a = _u8(m); lib().orc_sha3_256(_p(o), _p(a), C.c_size_t(a.size)); return o.tobytes()
def shake256(m, n):
    o = np.zeros(n, np.uint8); a = _u8(m); lib().orc_shake256(_p(o), C.c_size_t(n), _p(a), C.c_size_t(a.size)); return o.tobytes()
def chacha20_block(key, ctr):
    o = np.zeros(64, np.uint8); lib().orc_chacha20_block(_p(o), _p(_u8(key, 32)), C.c_uint64(ctr)); return o.tobytes()
def merlin_simple(proto, label, msg, clabel, n):
    o = np.zeros(n, np.uint8); a = _u8(msg)
    lib().orc_merlin_simple(_p(o), C.c_size_t(n), C.c_char_p(proto), C.c_char_p(label), _p(a), C.c_size_t(a.size), C.c_char_p(clabel)); return o.tobytes()
def bp_gens(which, party, n):
    o = np.zeros(32 * n, np.uint8); lib().orc_bp_gens(_p(o), ord(which), C.c_uint32(party), n); return o.reshape(n, 32)
def derive_key(seed, domain, index):
    o = np.zeros(32, np.uint8); lib().orc_derive_key(_p(o), _p(_u8(seed, 32)), C.c_uint32(domain), C.c_uint64(index)); return o.tobytes()
def rnd_scalar_vec(seed, n):
    o = np.zeros(32 * n, np.uint8); lib().orc_rnd_scalar_vec(_p(o), _p(_u8(seed, 32)), C.c_size_t(n)); return o.reshape(n, 32)

# ---- rofl_crypto vector API ----------------------------------------------------------------------
def next_pow2(v): return lib().orc_next_pow2(v)
def rp_proof_len(N): return lib().orc_rp_proof_len(N)
def f32_to_scalar_vec(v, n_bits=16, frac=7):
    v = _f32(v); o = np.zeros((v.size, 32), np.uint8)
    rc = lib().orc_f32_to_scalar_vec(_p(o), _p(v), C.c_size_t(v.size), n_bits, frac); assert rc == 0, rc; return o
def scalar_to_f32_vec(s, n_bits=16, frac=7):
    s = _u8(s).reshape(-1, 32); o = np.zeros(s.shape[0], np.float32)
    rc = lib().orc_scalar_to_f32_vec(_p(o), _p(s), C.c_size_t(s.shape[0]), n_bits, frac); assert rc == 0; return o
def clip_bounds(rng, n_bits=16, frac=7):
    mn, mx = C.c_float(), C.c_float(); lib().orc_clip_bounds(C.byref(mn), C.byref(mx), rng, n_bits, frac); return mn.value, mx.value
def l2_clip_bound(rng, n_bits=16, frac=7): return lib().orc_l2_clip_bound(rng, n_bits, frac)
def clip_f32_to_range_vec(v, rng, n_bits=16, frac=7):
    v = _f32(v); o = np.zeros_like(v); lib().orc_clip_f32_to_range_vec(_p(o), _p(v), C.c_size_t(v.size), rng, n_bits, frac); return o
def square(s, n_bits=16, frac=7):
    o = np.zeros(32, np.uint8); rc = lib().orc_square(_p(o), _p(_u8(s, 32)), n_bits, frac)
    if rc: raise OverflowError("square overflows")
    return o.tobytes()
def commit_f32(v, blind=None, n_bits=16, frac=7):
    v = _f32(v); o = np.zeros((v.size, 32), np.uint8); b = _u8(blind) if blind is not None else None
    rc = lib().orc_commit_f32(_p(o), _p(v), _p(b), C.c_size_t(v.size), n_bits, frac); assert rc == 0, rc; return o
def commit_scalars(vals, blind=None):
    s = _u8(vals).reshape(-1, 32); o = np.zeros_like(s); b = _u8(blind) if blind is not None else None
    lib().orc_commit_scalars(_p(o), _p(s), _p(b), C.c_size_t(s.shape[0])); return o
def elgamal_R(blind):
    b = _u8(blind).reshape(-1, 32); o = np.zeros_like(b); lib().orc_elgamal_R(_p(o), _p(b), C.c_size_t(b.shape[0])); return o

def range_prove(values, blind, rng, n_partition, n_bits=16, frac=7, seed=SEED0):
    """-> (rc, proofs[n_chunks, plen], commits[D,32])  (range_proof_vec::create_rangeproof)"""
    v = _f32(values); D = v.size; b = _u8(blind, 32 * D)
    Dp = next_pow2(D); nc = min(Dp, n_partition); chunk = Dp // nc
    plen = rp_proof_len(rng * chunk)
    proofs = np.zeros((nc, plen), np.uint8); commits = np.zeros((D, 32), np.uint8)
    rc = lib().orc_range_prove(_p(proofs), _p(commits), _p(v), _p(b), C.c_size_t(D), rng, C.c_size_t(n_partition), n_bits, frac, _p(_u8(seed, 32)))
    return rc, proofs, commits
def range_prove_tx_bl_shifted(values, blind, rng, n_partition, shifts, n_bits=16, frac=7, seed=SEED0):
    """range_prove with t_x_blinding of chunk c shifted by the scalar shifts[c] (32 bytes each) before it is absorbed: otherwise honest proofs
    whose verification equations are off by exactly -c shift B_blinding (adaptive-forgery tests of the batched verifier)"""
    v = _f32(values); D = v.size; b = _u8(blind, 32 * D)
    Dp = next_pow2(D); nc = min(Dp, n_partition); chunk = Dp // nc
    proofs = np.zeros((nc, rp_proof_len(rng * chunk)), np.uint8); commits = np.zeros((D, 32), np.uint8)
    rc = lib().orc_range_prove_tx_bl_shifted(_p(proofs), _p(commits), _p(v), _p(b), C.c_size_t(D), rng, C.c_size_t(n_partition), n_bits, frac,
                                             _p(_u8(seed, 32)), _p(_u8(shifts, 32 * nc)))
    return rc, proofs, commits
def range_verify(proofs, commits, rng, seed=SEED0):
    p = _u8(proofs); c = _u8(commits).reshape(-1, 32)
    p = p.reshape(p.shape[0], -1) if p.ndim > 1 else p
    n_proofs, plen = p.shape
    return lib().orc_range_verify(_p(p), C.c_size_t(plen), C.c_size_t(n_proofs), _p(c), C.c_size_t(c.shape[0]), rng, _p(_u8(seed, 32)))
def l2_prove(values, blind, rng, n_bits=32, frac=7, seed=SEED0):
    v = _f32(values); D = v.size; b = _u8(blind, 32 * D)
    proof = np.zeros(rp_proof_len(rng), np.uint8); commit = np.zeros(32, np.uint8)
    rc = lib().orc_l2_prove(_p(proof), _p(commit), _p(v), _p(b), C.c_size_t(D), rng, n_bits, frac, _p(_u8(seed, 32)))
    return rc, proof, commit
def l2_verify(proof, commit, rng, seed=SEED0):
    p = _u8(proof); return lib().orc_l2_verify(_p(p), C.c_size_t(p.size), _p(_u8(commit, 32)), rng, _p(_u8(seed, 32)))
def square_prove(values, value_com, r1, r2, n_bits=32, frac=7, seed=SEED0):
    v = _f32(values); D = v.size
    proofs = np.zeros((D, 160), np.uint8); commits = np.zeros((D, 64), np.uint8)
    rc = lib().orc_square_prove(_p(proofs), _p(commits), _p(v), _p(_u8(value_com, 32 * D)), _p(_u8(r1, 32 * D)), _p(_u8(r2, 32 * D)), C.c_size_t(D), n_bits, frac, _p(_u8(seed, 32)))
    return rc, proofs, commits
def square_verify(proofs, commits):
    p = _u8(proofs).reshape(-1, 160); c = _u8(commits).reshape(-1, 64)
    return lib().orc_square_verify(_p(p), _p(c), C.c_size_t(p.shape[0]))
def rand_prove(values, value_com, blind, n_bits=16, frac=7, seed=SEED0):
    """rand_proof_vec::create_randproof_vec (value_com None) / _existing -> (rc, proofs[D, 128], pairs[D, 64])"""
    v = _f32(values); D = v.size; proofs = np.zeros((D, 128), np.uint8); pairs = np.zeros((D, 64), np.uint8)
    rc = lib().orc_rand_prove(_p(proofs), _p(pairs), _p(v), None if value_com is None else _p(_u8(value_com, 32 * D)), _p(_u8(blind, 32 * D)), C.c_size_t(D), n_bits, frac, _p(_u8(seed, 32)))
    return rc, proofs, pairs
def rand_verify(proofs, pairs):
    p = _u8(proofs).reshape(-1, 128); c = _u8(pairs).reshape(-1, 64)
    return lib().orc_rand_verify(_p(p), _p(c), C.c_size_t(p.shape[0]))
def square_rand_prove(values, value_com, r1, r2, n_bits=32, frac=7, seed=SEED0):
    """square_rand_proof_vec::create_l2rangeproof_vec(_existing) -> (rc, proofs[D, 192], commits[D, 96])"""
    v = _f32(values); D = v.size; proofs = np.zeros((D, 192), np.uint8); commits = np.zeros((D, 96), np.uint8)
    rc = lib().orc_square_rand_prove(_p(proofs), _p(commits), _p(v), None if value_com is None else _p(_u8(value_com, 32 * D)), _p(_u8(r1, 32 * D)), _p(_u8(r2, 32 * D)), C.c_size_t(D), n_bits, frac, _p(_u8(seed, 32)))
    return rc, proofs, commits
def square_rand_verify(proofs, commits):
    p = _u8(proofs).reshape(-1, 192); c = _u8(commits).reshape(-1, 96)
    return lib().orc_square_rand_verify(_p(p), _p(c), C.c_size_t(p.shape[0]))
def crp_prove(values, value_com, blind, n_bits=16, frac=7, seed=SEED0):
    """CompressedRandProof::helper_prove (value_com None) / helper_prove_existing -> (rc, proof[128], pairs[D, 64])"""
    v = _f32(values); D = v.size
    proof = np.zeros(128, np.uint8); pairs = np.zeros((D, 64), np.uint8)
    rc = lib().orc_crp_prove(_p(proof), _p(pairs), _p(v), None if value_com is None else _p(_u8(value_com, 32 * D)), _p(_u8(blind, 32 * D)), C.c_size_t(D), n_bits, frac, _p(_u8(seed, 32)))
    return rc, proof, pairs
def crp_verify(proof, pairs):
    p = _u8(pairs).reshape(-1, 64)
    return lib().orc_crp_verify(_p(_u8(proof, 128)), _p(p), C.c_size_t(p.shape[0]))
# challenges of the sigma proofs, from the oracle's own transcripts (the batched verifiers' weights are keyed on them)
def _challenge(name, com, cp, *mid):
    o = np.zeros(32, np.uint8); com = _u8(com); cp = _u8(cp).copy()
    getattr(lib(), name)(_p(o), _p(com), *mid, _p(cp)); return o.tobytes()
def sq_challenge(commits64, proof160):
    """square proof: commitments c_l | c_sq, proof C'_l | C'_sq | z_m | z_r1 | z_r2"""
    return _challenge("orc_sq_challenge", _u8(commits64, 64), _u8(proof160, 160)[:64])
def rp_challenge(pair64, proof128):
    return _challenge("orc_rp_challenge", _u8(pair64, 64), _u8(proof128, 128)[:64])
def srp_challenge(commits96, proof192):
    return _challenge("orc_srp_challenge", _u8(commits96, 96), _u8(proof192, 192)[:96])
def crp_challenge(proof128, pairs):
    p = _u8(pairs).reshape(-1, 64); return _challenge("orc_crp_challenge", p, _u8(proof128, 128)[:64], C.c_size_t(p.shape[0]))
def rp_challenges(proof, V32, n, m, label_id=0):
    """the range-proof verifier's transcript replayed by the oracle -> (rc, [y, z, x, w, u_0 .. u_(lgN-1)] as 32-byte scalars, the 32-byte
    "rofl-batch" digest); rc 1, or 0 when a proof point is the identity encoding (the transcript still absorbs it)"""
    p = _u8(proof); v = _u8(V32, 32 * m); lg = (p.size // 32 - 9) // 2
    ch = np.zeros((4 + lg, 32), np.uint8); dg = np.zeros(32, np.uint8)
    rc = lib().orc_rp_challenges(_p(p), C.c_size_t(p.size), _p(v), n, m, label_id, _p(ch), _p(dg))
    return rc, [bytes(x) for x in ch], dg.tobytes()
def aggregate(pts, init=0):
    a = _u8(pts); assert a.ndim == 3 and a.shape[2] == 32
    o = np.zeros((a.shape[1], 32), np.uint8); rc = lib().orc_aggregate(_p(o), _p(a), C.c_size_t(a.shape[0]), C.c_size_t(a.shape[1]), init); assert rc == 0; return o
def dlog(pts, table_size=1 << 16, bsgs_bits=16):
    a = _u8(pts).reshape(-1, 32); o = np.zeros_like(a)
    rc = lib().orc_dlog(_p(o), _p(a), C.c_size_t(a.shape[0]), C.c_size_t(table_size), bsgs_bits); return rc, o
def num_threads(): return lib().orc_num_threads()
def set_num_threads(n): lib().orc_set_num_threads(n)
