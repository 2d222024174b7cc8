"""ctypes binding of include/rofl_b200.h (the C ABI of librofl_b200.so) plus a thin numpy-facing wrapper.

`Api(cdll)` is agnostic of where the handle came from; the package (`__init__.py`) only ever hands it the CUDA
library.  Array arguments are numpy arrays (host-buffer calls) or integer device addresses (`*_dev` calls, e.g.
`tensor.data_ptr()` of a torch CUDA tensor)."""
import ctypes as C
import numpy as np

c_sz, c_u8p, c_f32p, c_vp = C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p

_SIGS = {
    "rofl_ctx_create": (C.c_int, [C.POINTER(c_vp), C.c_int]),
    "rofl_ctx_destroy": (None, [c_vp]),
    "rofl_last_error": (C.c_char_p, []),
    "rofl_set_host_threads": (None, [c_vp, C.c_int]),
    "rofl_set_option": (C.c_int, [c_vp, C.c_char_p, C.c_long]),
    "rofl_next_pow2": (c_sz, [c_sz]),
    "rofl_range_proof_len": (c_sz, [c_sz]),
    "rofl_range_proof_shape": (None, [c_sz, C.c_int, c_sz, C.POINTER(c_sz), C.POINTER(c_sz)]),
    "rofl_field_selftest": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz, c_u8p]),
    "rofl_scalar_selftest": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz, c_u8p]),
    "rofl_debug_square_rlc": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz]),
    "rofl_f32_to_scalar_vec": (C.c_int, [c_vp, c_f32p, c_sz, C.c_int, C.c_int, c_u8p]),
    "rofl_scalar_to_f32_vec": (C.c_int, [c_vp, c_u8p, c_sz, C.c_int, C.c_int, c_f32p]),
    "rofl_clip_bounds": (None, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "rofl_l2_clip_bound": (C.c_float, [C.c_int, C.c_int, C.c_int]),
    "rofl_clip_f32_to_range_vec": (None, [c_f32p, c_sz, C.c_int, C.c_int, C.c_int, c_f32p]),
    "rofl_rnd_scalar_vec": (None, [c_u8p, c_sz, c_u8p]),
    "rofl_scalar_ops": (C.c_int, [C.c_int, c_u8p, c_u8p, c_sz, c_u8p]),
    "rofl_commit": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p]),
    "rofl_commit_dev": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p]),
    "rofl_range_prove": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, C.POINTER(c_sz), C.POINTER(c_sz), c_u8p]),
    "rofl_range_prove_dev": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, C.POINTER(c_sz), C.POINTER(c_sz), c_u8p]),
    "rofl_range_prove_shard": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, c_sz, c_sz, c_sz, C.c_int, C.c_int, C.c_int, c_u8p, c_u8p, C.POINTER(c_sz), c_u8p]),
    "rofl_range_verify_shard": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, c_u8p, c_sz, c_sz, c_sz, C.c_int, c_u8p]),
    "rofl_range_verify": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, c_u8p]),
    "rofl_range_verify_dev": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, c_u8p]),
    "rofl_l2_prove": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, C.c_int, C.c_int, c_u8p, c_u8p, C.POINTER(c_sz), c_u8p]),
    "rofl_l2_verify": (C.c_int, [c_vp, c_u8p, c_sz, c_u8p, C.c_int, c_u8p]),
    "rofl_enc_range_compressed_encrypt": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p, c_u8p, C.POINTER(c_sz), C.POINTER(c_sz)]),
    "rofl_enc_range_compressed_verify": (C.c_int, [c_vp, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, C.c_int, C.c_float, c_u8p]),
    "rofl_enc_l2_compressed_encrypt": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, c_sz, C.c_int, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, C.POINTER(c_sz), C.POINTER(c_sz), c_u8p, C.POINTER(c_sz)]),
    "rofl_enc_range_encrypt": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, c_sz, C.c_float, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p, c_u8p, C.POINTER(c_sz), C.POINTER(c_sz)]),
    "rofl_enc_range_verify": (C.c_int, [c_vp, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, C.c_int, C.c_float, c_u8p]),
    "rofl_enc_l2_encrypt": (C.c_int, [c_vp, c_f32p, c_u8p, c_sz, C.c_int, c_sz, C.c_int, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p, c_u8p, C.POINTER(c_sz), C.POINTER(c_sz), c_u8p, C.POINTER(c_sz)]),
    "rofl_enc_l2_verify": (C.c_int, [c_vp, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, C.c_int, c_u8p]),
    "rofl_enc_l2_compressed_verify": (C.c_int, [c_vp, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, C.c_int, c_u8p]),
    "rofl_rand_prove": (C.c_int, [c_vp, c_f32p, c_u8p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p]),
    "rofl_rand_verify": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz]),
    "rofl_square_rand_prove": (C.c_int, [c_vp, c_f32p, c_u8p, c_u8p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p]),
    "rofl_square_rand_verify": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz]),
    "rofl_crp_prove": (C.c_int, [c_vp, c_f32p, c_u8p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p]),
    "rofl_crp_verify": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz]),
    "rofl_square_prove": (C.c_int, [c_vp, c_f32p, c_u8p, c_u8p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p]),
    "rofl_square_prove_dev": (C.c_int, [c_vp, c_f32p, c_u8p, c_u8p, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_u8p, c_u8p]),
    "rofl_square_verify": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz]),
    "rofl_square_verify_dev": (C.c_int, [c_vp, c_u8p, c_u8p, c_sz]),
    "rofl_aggregate": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, C.c_int, c_u8p]),
    "rofl_aggregate_dev": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, C.c_int, c_u8p]),
    "rofl_dlog": (C.c_int, [c_vp, c_u8p, c_sz, C.c_uint64, C.c_int, C.c_int, C.c_int, c_u8p, c_f32p]),
    "rofl_dlog_dev": (C.c_int, [c_vp, c_u8p, c_sz, C.c_uint64, C.c_int, C.c_int, C.c_int, c_u8p, c_f32p]),
    "rofl_acc_create": (C.c_int, [c_vp, c_sz, C.c_int, C.c_int, C.POINTER(c_vp)]),
    "rofl_acc_destroy": (None, [c_vp]),
    "rofl_acc_reset": (C.c_int, [c_vp]),
    "rofl_acc_add": (C.c_int, [c_vp, c_u8p, c_sz, c_vp, c_vp]),
    "rofl_acc_add_dev": (C.c_int, [c_vp, c_u8p, c_sz, c_vp, c_vp]),
    "rofl_acc_count": (c_sz, [c_vp]),
    "rofl_acc_export": (C.c_int, [c_vp, c_u8p]),
    "rofl_acc_extract": (C.c_int, [c_vp, C.c_uint64, C.c_int, C.c_int, C.c_int, c_u8p, c_f32p]),
    "rofl_prof_enable": (None, [C.c_int]),
    "rofl_prof_reset": (None, []),
    "rofl_prof_ms": (C.c_double, [C.c_int]),
    "rofl_prof_work": (C.c_double, [C.c_int]),
    "rofl_probe_imad_wide": (C.c_double, [c_vp]),
    "rofl_prof_launches": (C.c_long, [C.c_int]),
    "rofl_ctx_stream": (c_vp, [c_vp]),
    "rofl_range_verify_batch": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, c_u8p, c_sz, c_sz, C.c_int, c_u8p, c_vp]),
    "rofl_enc_l2_compressed_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_vp]),
    "rofl_crp_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_u8p, c_sz, c_u8p, c_vp]),
    "rofl_enc_range_compressed_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, C.c_int, C.c_float, c_u8p, c_vp]),
    "rofl_debug_ts_absorb": (C.c_int, [c_vp, c_u8p, c_sz, C.c_int, C.c_int]),
    "rofl_debug_crp_rlc": (C.c_int, [c_vp, c_sz, c_u8p, c_u8p, c_sz, c_u8p]),
    "rofl_rand_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_u8p, c_sz, c_u8p, c_vp]),
    "rofl_square_rand_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_u8p, c_sz, c_u8p, c_vp]),
    "rofl_enc_range_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, C.c_int, C.c_float, c_u8p, c_vp]),
    "rofl_enc_l2_verify_batch": (C.c_int, [c_vp, c_sz, c_u8p, c_sz, c_u8p, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, C.c_int, c_u8p, c_vp]),
    "rofl_debug_sigma_rlc": (C.c_int, [c_vp, C.c_int, c_sz, c_u8p, c_u8p, c_u8p]),
    "rofl_debug_verify_weights": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, c_u8p, c_sz, C.c_int, c_u8p, c_u8p]),
    "rofl_debug_msm": (C.c_int, [c_vp, c_u8p, c_sz, c_sz, c_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_sz, c_u8p, c_u8p, c_u8p, c_vp]),
    "rofl_debug_rlc_terms": (C.c_int, [c_vp, C.c_int, c_sz, c_sz, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_vp, c_u8p, c_u8p, c_vp, c_vp, c_vp, c_vp]),
}
EXPORTED_SYMBOLS = tuple(_SIGS)


def bind(lib):
    for name, (res, args) in _SIGS.items():
        f = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        f.restype, f.argtypes = res, args
    return lib


class RoflError(RuntimeError):
    def __init__(self, code, msg=""):
        super().__init__(f"rofl_b200 error {code}: {msg}")
        self.code = code


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return a
    return a.ctypes.data


def _u8(x, n=None):
    if isinstance(x, (bytes, bytearray)):
        x = np.frombuffer(bytes(x), dtype=np.uint8)
    a = np.ascontiguousarray(x, dtype=np.uint8)
    if n is not None and a.size != n:
        raise ValueError(f"expected {n} bytes, got {a.size}")
    return a


def _f32(x):
    return np.ascontiguousarray(x, dtype=np.float32)


import os as _os


def _seed(seed):
    """Prover nonces and verifier weights are derived from `seed`: None draws 32 fresh bytes from the OS (what every production call must
    use, see the SECURITY note of include/rofl_b200.h); parity tests pass fixed seeds."""
    return _u8(_os.urandom(32) if seed is None else seed, 32)


class Api:
    """One context (= one GPU) of the library."""

    def __init__(self, lib, device=0):
        self.lib = bind(lib)
        h = c_vp()
        rc = self.lib.rofl_ctx_create(C.byref(h), device)
        if rc != 0:
            raise RoflError(rc, (self.lib.rofl_last_error() or b"").decode())
        self.h = h

    def close(self):
        if self.h:
            self.lib.rofl_ctx_destroy(self.h); self.h = None

    def field_selftest(self, a, b):
        a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8); n = a.shape[0]
        out = np.zeros((n, 6, 32), np.uint8)
        rc = self.lib.rofl_field_selftest(self.h, _ptr(a), _ptr(b), n, _ptr(out))
        if rc != 0:
            raise self._err(rc)
        return out

    def debug_square_rlc(self, proofs, commits):
        p = _u8(proofs).reshape(-1, 160); c = _u8(commits).reshape(-1, 64)
        return self.lib.rofl_debug_square_rlc(self.h, _ptr(p), _ptr(c), p.shape[0])

    def scalar_add(self, a, b):
        """element-wise a + b mod l on 32-byte scalars (host; bindings32.rs `add_scalars`)"""
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32); b = np.ascontiguousarray(b, np.uint8).reshape(-1, 32); o = np.zeros_like(a)
        rc = self.lib.rofl_scalar_ops(0, _ptr(a), _ptr(b), a.shape[0], _ptr(o))
        if rc: raise self._err(rc)
        return o

    def scalar_neg(self, a):
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32); o = np.zeros_like(a)
        rc = self.lib.rofl_scalar_ops(1, _ptr(a), None, a.shape[0], _ptr(o))
        if rc: raise self._err(rc)
        return o

    def cancelling_blindings(self, n_clients, D, seed_byte=0x40):
        """n_clients blinding vectors that sum to zero (pedersen_ops.rs:110-122 generate_cancelling_blindings: the last one is minus the sum of the others)"""
        bls = [np.frombuffer(self.rnd_scalar_vec(bytes([(seed_byte + k) & 0xff]) * 32, D).tobytes(), np.uint8).reshape(D, 32).copy() for k in range(n_clients - 1)]
        tot = np.zeros((D, 32), np.uint8)
        for b in bls:
            tot = self.scalar_add(tot, b)
        return bls + [self.scalar_neg(tot)]

    def scalar_selftest(self, a, b):
        a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8); n = a.shape[0]
        out = np.zeros((n, 3, 32), np.uint8)
        rc = self.lib.rofl_scalar_selftest(self.h, _ptr(a), _ptr(b), n, _ptr(out))
        if rc != 0:
            raise self._err(rc)
        return out

    # ---- per-element proofs of the un-optimised encodings
    def rand_prove(self, v, value_com, blind, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D); vc = None if value_com is None else _u8(value_com, 32 * D)
        proofs = np.zeros((D, 128), np.uint8); pairs = np.zeros((D, 64), np.uint8)
        rc = self.lib.rofl_rand_prove(self.h, _ptr(v), _ptr(vc), _ptr(b), D, n_bits, frac, _ptr(_seed(seed)), _ptr(proofs), _ptr(pairs))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proofs, pairs
    def rand_verify(self, proofs, pairs):
        p = _u8(proofs).reshape(-1, 128); c = _u8(pairs).reshape(-1, 64)
        rc = self.lib.rofl_rand_verify(self.h, _ptr(p), _ptr(c), p.shape[0])
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    def square_rand_prove(self, v, value_com, r1, r2, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; vc = None if value_com is None else _u8(value_com, 32 * D)
        proofs = np.zeros((D, 192), np.uint8); commits = np.zeros((D, 96), np.uint8)
        rc = self.lib.rofl_square_rand_prove(self.h, _ptr(v), _ptr(vc), _ptr(_u8(r1, 32 * D)), _ptr(_u8(r2, 32 * D)), D, n_bits, frac, _ptr(_seed(seed)), _ptr(proofs), _ptr(commits))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proofs, commits
    def square_rand_verify(self, proofs, commits):
        p = _u8(proofs).reshape(-1, 192); c = _u8(commits).reshape(-1, 96)
        rc = self.lib.rofl_square_rand_verify(self.h, _ptr(p), _ptr(c), p.shape[0])
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    # ---- compressed randomness proof: (rc, proof[128], pairs[D, 64]) / 1|0|<0
    def crp_prove(self, v, value_com, blind, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        proof = np.zeros(128, np.uint8); pairs = np.zeros((max(D, 1), 64), np.uint8)
        vc = None if value_com is None else _u8(value_com, 32 * D)
        rc = self.lib.rofl_crp_prove(self.h, _ptr(v), _ptr(vc), _ptr(b), D, n_bits, frac, _ptr(_seed(seed)), _ptr(proof), _ptr(pairs))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proof, pairs[:D]
    def crp_verify(self, proof, pairs):
        p = _u8(pairs).reshape(-1, 64)
        rc = self.lib.rofl_crp_verify(self.h, _ptr(_u8(proof, 128)), _ptr(p), p.shape[0])
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc

    # ---- the optimised encodings end to end (params.rs EncParamsRangeCompressed / EncParamsL2Compressed); dicts of wire fields
    def enc_range_compressed_encrypt(self, v, blind, prove_range, n_partition, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        npf, plen = self.range_proof_shape(D, prove_range, n_partition)
        enc = np.zeros((D, 64), np.uint8); rp = np.zeros(128, np.uint8); proofs = np.zeros((npf, max(plen, 1)), np.uint8); a, c = c_sz(), c_sz()
        rc = self.lib.rofl_enc_range_compressed_encrypt(self.h, _ptr(v), _ptr(b), D, prove_range, n_partition, n_bits, frac, _ptr(_seed(seed)), _ptr(enc), _ptr(rp), _ptr(proofs), C.byref(a), C.byref(c))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, dict(enc_values=enc, rand_proof=rp, range_proof=proofs, range_bits=prove_range)
    def enc_range_compressed_verify(self, msg, check_percentage=1.0, seed=None):
        enc = _u8(msg["enc_values"]).reshape(-1, 64); p = _u8(msg["range_proof"]); p = p.reshape(p.shape[0], -1)
        rc = self.lib.rofl_enc_range_compressed_verify(self.h, _ptr(enc), enc.shape[0], _ptr(_u8(msg["rand_proof"], 128)), _ptr(p), p.shape[1], p.shape[0], msg["range_bits"], check_percentage, _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    def enc_l2_compressed_encrypt(self, v, blind, prove_range, n_partition, l2_range, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        npf, plen = self.range_proof_shape(D, prove_range, n_partition)
        enc = np.zeros((D, 96), np.uint8); sp = np.zeros((D, 160), np.uint8); rp = np.zeros(128, np.uint8); proofs = np.zeros((npf, max(plen, 1)), np.uint8)
        sq = np.zeros(self.range_proof_len(max(l2_range, 1)), np.uint8); a, c, q = c_sz(), c_sz(), c_sz()
        rc = self.lib.rofl_enc_l2_compressed_encrypt(self.h, _ptr(v), _ptr(b), D, prove_range, n_partition, l2_range, n_bits, frac, _ptr(_seed(seed)), _ptr(enc), _ptr(sp), _ptr(rp), _ptr(proofs),
                                                     C.byref(a), C.byref(c), _ptr(sq), C.byref(q))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, dict(enc_values=enc, square_proof=sp, rand_proof=rp, range_proof=proofs, square_range_proof=sq, range_bits=prove_range, l2_range_bits=l2_range)
    def enc_l2_compressed_verify(self, msg, seed=None):
        enc = _u8(msg["enc_values"]).reshape(-1, 96); sp = _u8(msg["square_proof"]).reshape(-1, 160); p = _u8(msg["range_proof"]); p = p.reshape(p.shape[0], -1); sq = _u8(msg["square_range_proof"])
        rc = self.lib.rofl_enc_l2_compressed_verify(self.h, _ptr(enc), enc.shape[0], _ptr(sp), _ptr(p), p.shape[1], p.shape[0], _ptr(sq), sq.size, msg["range_bits"], msg["l2_range_bits"], _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc

    # ---- the un-optimised encodings end to end (params.rs EncParamsRange / EncParamsL2)
    def enc_range_encrypt(self, v, blind, prove_range, n_partition, check_percentage, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        num = D if check_percentage >= 1.0 else int(np.floor(float(np.float32(np.float32(D) * np.float32(check_percentage))) + 0.5))      # llroundf
        npf, plen = self.range_proof_shape(max(num, 1), prove_range, n_partition)
        enc = np.zeros((D, 64), np.uint8); rp = np.zeros((D, 128), np.uint8); proofs = np.zeros((npf, max(plen, 1)), np.uint8); a, c = c_sz(), c_sz()
        rc = self.lib.rofl_enc_range_encrypt(self.h, _ptr(v), _ptr(b), D, prove_range, n_partition, check_percentage, n_bits, frac, _ptr(_seed(seed)), _ptr(enc), _ptr(rp), _ptr(proofs), C.byref(a), C.byref(c))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, dict(enc_values=enc, rand_proof=rp, range_proof=proofs[:c.value, :a.value] if rc == 0 else proofs, range_bits=prove_range)
    def enc_range_verify(self, msg, check_percentage=1.0, seed=None):
        enc = _u8(msg["enc_values"]).reshape(-1, 64); rp = _u8(msg["rand_proof"]).reshape(-1, 128); p = _u8(msg["range_proof"]); p = p.reshape(p.shape[0], -1)
        rc = self.lib.rofl_enc_range_verify(self.h, _ptr(enc), enc.shape[0], _ptr(rp), _ptr(p), p.shape[1], p.shape[0], msg["range_bits"], check_percentage, _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    def enc_l2_encrypt(self, v, blind, prove_range, n_partition, l2_range, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        npf, plen = self.range_proof_shape(D, prove_range, n_partition)
        enc = np.zeros((D, 96), np.uint8); sp = np.zeros((D, 192), np.uint8); proofs = np.zeros((npf, max(plen, 1)), np.uint8)
        sq = np.zeros(self.range_proof_len(max(l2_range, 1)), np.uint8); a, c, q = c_sz(), c_sz(), c_sz()
        rc = self.lib.rofl_enc_l2_encrypt(self.h, _ptr(v), _ptr(b), D, prove_range, n_partition, l2_range, n_bits, frac, _ptr(_seed(seed)), _ptr(enc), _ptr(sp), _ptr(proofs),
                                          C.byref(a), C.byref(c), _ptr(sq), C.byref(q))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, dict(enc_values=enc, square_proof=sp, range_proof=proofs, square_range_proof=sq, range_bits=prove_range, l2_range_bits=l2_range)
    def enc_l2_verify(self, msg, seed=None):
        enc = _u8(msg["enc_values"]).reshape(-1, 96); sp = _u8(msg["square_proof"]).reshape(-1, 192); p = _u8(msg["range_proof"]); p = p.reshape(p.shape[0], -1); sq = _u8(msg["square_range_proof"])
        rc = self.lib.rofl_enc_l2_verify(self.h, _ptr(enc), enc.shape[0], _ptr(sp), _ptr(p), p.shape[1], p.shape[0], _ptr(sq), sq.size, msg["range_bits"], msg["l2_range_bits"], _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc

    # ---- server side: all clients of a round in one batched check; returns the per-client verdicts (1 / 0 / < 0)
    def range_verify_batch(self, proofs, commits, rng, seed=None):
        p = _u8(proofs); K = p.shape[0]; p = p.reshape(K, p.shape[1], -1); c = _u8(commits).reshape(K, -1, 32); ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_range_verify_batch(self.h, _ptr(p), p.shape[2], p.shape[1], _ptr(c), c.shape[1], K, rng, _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def enc_l2_compressed_verify_batch(self, msgs, seed=None):
        K = len(msgs); enc = _u8(np.stack([m["enc_values"] for m in msgs])).reshape(K, -1, 96); sp = _u8(np.stack([m["square_proof"] for m in msgs])).reshape(K, -1, 160)
        rp = _u8(np.stack([m["range_proof"] for m in msgs])); rp = rp.reshape(K, rp.shape[1], -1); sq = _u8(np.stack([m["square_range_proof"] for m in msgs])).reshape(K, -1)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_enc_l2_compressed_verify_batch(self.h, K, _ptr(enc), enc.shape[1], _ptr(sp), _ptr(rp), rp.shape[2], rp.shape[1], _ptr(sq), sq.shape[1], msgs[0]["range_bits"], msgs[0]["l2_range_bits"],
                                                          _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def crp_verify_batch(self, proofs, pairs, seed=None):
        """K compressed rand proofs [K, 128] over their pairs [K, D, 64] in one batched check -> int32[K], each exactly crp_verify's verdict"""
        p = _u8(proofs); K = p.shape[0] if p.ndim > 1 else p.size // 128; p = p.reshape(K, 128); c = _u8(pairs).reshape(K, -1, 64)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_crp_verify_batch(self.h, K, _ptr(p), _ptr(c), c.shape[1], _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def enc_range_compressed_verify_batch(self, msgs, check_percentage=1.0, seed=None):
        """K EncRangeCompressed messages of one shape in one call -> int32[K], each exactly enc_range_compressed_verify's verdict"""
        K = len(msgs); enc = _u8(np.stack([m["enc_values"] for m in msgs])).reshape(K, -1, 64); rp = _u8(np.stack([m["rand_proof"] for m in msgs])).reshape(K, 128)
        p = _u8(np.stack([m["range_proof"] for m in msgs])); p = p.reshape(K, p.shape[1], -1)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_enc_range_compressed_verify_batch(self.h, K, _ptr(enc), enc.shape[1], _ptr(rp), _ptr(p), p.shape[2], p.shape[1], msgs[0]["range_bits"], check_percentage,
                                                             _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def rand_verify_batch(self, proofs, pairs, seed=None):
        """K x D rand proofs [K, D, 128] over their pairs [K, D, 64] in one batched check -> int32[K], each exactly rand_verify's verdict"""
        c = _u8(pairs); K = c.shape[0]; c = c.reshape(K, -1, 64); p = _u8(proofs).reshape(K, c.shape[1], 128)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_rand_verify_batch(self.h, K, _ptr(p), _ptr(c), c.shape[1], _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def square_rand_verify_batch(self, proofs, commits, seed=None):
        """K x D square-rand proofs [K, D, 192] over their commitments [K, D, 96] in one batched check -> int32[K], each exactly square_rand_verify's verdict"""
        c = _u8(commits); K = c.shape[0]; c = c.reshape(K, -1, 96); p = _u8(proofs).reshape(K, c.shape[1], 192)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_square_rand_verify_batch(self.h, K, _ptr(p), _ptr(c), c.shape[1], _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def enc_range_verify_batch(self, msgs, check_percentage=1.0, seed=None):
        """K EncRange messages of one shape in one call -> int32[K], each exactly enc_range_verify's verdict"""
        K = len(msgs); enc = _u8(np.stack([m["enc_values"] for m in msgs])).reshape(K, -1, 64); rp = _u8(np.stack([m["rand_proof"] for m in msgs])).reshape(K, -1, 128)
        p = _u8(np.stack([m["range_proof"] for m in msgs])); p = p.reshape(K, p.shape[1], -1)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_enc_range_verify_batch(self.h, K, _ptr(enc), enc.shape[1], _ptr(rp), _ptr(p), p.shape[2], p.shape[1], msgs[0]["range_bits"], check_percentage,
                                                  _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok
    def enc_l2_verify_batch(self, msgs, seed=None):
        """K EncL2 messages of one shape in one call -> int32[K], each exactly enc_l2_verify's verdict"""
        K = len(msgs); enc = _u8(np.stack([m["enc_values"] for m in msgs])).reshape(K, -1, 96); sp = _u8(np.stack([m["square_proof"] for m in msgs])).reshape(K, -1, 192)
        rp = _u8(np.stack([m["range_proof"] for m in msgs])); rp = rp.reshape(K, rp.shape[1], -1); sq = _u8(np.stack([m["square_range_proof"] for m in msgs])).reshape(K, -1)
        ok = np.zeros(K, np.int32)
        rc = self.lib.rofl_enc_l2_verify_batch(self.h, K, _ptr(enc), enc.shape[1], _ptr(sp), _ptr(rp), rp.shape[2], rp.shape[1], _ptr(sq), sq.shape[1], msgs[0]["range_bits"],
                                               msgs[0]["l2_range_bits"], _ptr(_seed(seed)), _ptr(ok))
        if rc < 0: raise self._err(rc)
        return ok

    # ---- test hooks
    def debug_ts_absorb(self, V32, n, label_id=0):
        v = _u8(V32).reshape(-1, 32)
        return self.lib.rofl_debug_ts_absorb(self.h, _ptr(v), v.shape[0], n, label_id)
    def debug_crp_rlc(self, proofs, pairs, seed=None):
        p = _u8(proofs).reshape(-1, 128); K = p.shape[0]; c = _u8(pairs).reshape(K, -1, 64)
        return self.lib.rofl_debug_crp_rlc(self.h, K, _ptr(p), _ptr(c), c.shape[1], _ptr(_seed(seed)))
    def debug_sigma_rlc(self, kind, proofs, commits, seed=None):
        """the batched rand (kind 1) / square-rand (kind 2) proof check alone over all elements as one update: 1 held, 0 did not"""
        pw, cw = (128, 64) if kind == 1 else (192, 96)
        p = _u8(proofs).reshape(-1, pw); c = _u8(commits).reshape(-1, cw)
        return self.lib.rofl_debug_sigma_rlc(self.h, kind, p.shape[0], _ptr(p), _ptr(c), _ptr(_seed(seed)))
    RLC_WIDTHS = {0: (160, 64), 1: (128, 64), 2: (192, 96), 3: (128, 64)}
    def debug_rlc_terms(self, family, proofs, commits, seed, max_ranges=None):
        """The terms of one batched check as its production code computed them (rofl_debug_rlc_terms).  family 0 square, 1 rand, 2 square-rand
        proofs: proofs [K, D, pw], commits [K, D, cw]; 3 compressed rand proofs: proofs [K, 128], commits = pairs [K, D, 64].
        -> dict(held, root (32 bytes), chal [K * D or K, 32], verdicts [K], ranges: list of dicts (i0, n, c, wbits, is_id (2), scal [T, 32],
        sB (2 x 32 bytes), sH (2 x 32 bytes), bad [clients touched]))"""
        pw, cw = self.RLC_WIDTHS[family]
        c = _u8(commits); K = c.shape[0]; c = c.reshape(K, -1, cw); D = c.shape[1]
        p = _u8(proofs).reshape(K, -1) if family == 3 else _u8(proofs).reshape(K, D, pw)
        N = K if family == 3 else K * D
        nsc = K * (D + 1) if family == 3 else (6 if family == 2 else 4) * N
        cap = np.array([max_ranges or min(N, 1 << 16), nsc, (max_ranges or min(N, 1 << 16)) + K], np.uintp)
        for _ in range(2):                                   # a second call only when the first capacities were short
            cnt = np.zeros(3, np.uintp); root = np.zeros(32, np.uint8); chal = np.zeros((N, 32), np.uint8); verd = np.zeros(K, np.int32)
            rng = np.zeros((int(cap[0]), 8), np.int64); sc = np.zeros((int(cap[1]), 32), np.uint8); coef = np.zeros((int(cap[0]), 4, 32), np.uint8); bad = np.zeros(int(cap[2]), np.int32)
            rc = self.lib.rofl_debug_rlc_terms(self.h, family, K, D, _ptr(p), _ptr(c), _ptr(_u8(seed, 32)), _ptr(root), _ptr(chal), _ptr(rng), _ptr(sc), _ptr(coef), _ptr(bad),
                                               _ptr(verd), _ptr(cap), _ptr(cnt))
            if rc == -2 and (cnt > cap).any():
                cap = np.maximum(cap, cnt); continue
            break
        if rc < 0: raise self._err(rc)
        ranges = []
        for j in range(int(cnt[0])):
            i0, n, w, wbits, id0, id1, os_, ob = (int(x) for x in rng[j])
            T = (int(cnt[1]) if j + 1 == cnt[0] else int(rng[j + 1][6])) - os_
            nb = (int(cnt[2]) if j + 1 == cnt[0] else int(rng[j + 1][7])) - ob
            ranges.append(dict(i0=i0, n=n, c=w, wbits=wbits, is_id=(id0, id1), scal=sc[os_:os_ + T], sB=(coef[j, 0].tobytes(), coef[j, 1].tobytes()),
                               sH=(coef[j, 2].tobytes(), coef[j, 3].tobytes()), bad=bad[ob:ob + nb].tolist()))
        return dict(held=rc, root=root.tobytes(), chal=chal, verdicts=verd.tolist(), ranges=ranges)
    def debug_verify_weights(self, proofs, commits, rng, seed):
        p = _u8(proofs); p = p.reshape(p.shape[0], -1); c = _u8(commits).reshape(-1, 32); w = np.zeros((2, p.shape[0], 32), np.uint8)
        rc = self.lib.rofl_debug_verify_weights(self.h, _ptr(p), p.shape[1], p.shape[0], _ptr(c), c.shape[0], rng, _ptr(_seed(seed)), _ptr(w))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, w

    def debug_msm(self, scalars, points=None, gen_n=0, path=0, c=0, knob=1, big_min=0, sB=None, sH=None):
        """The MSM front end alone: scalars [n_msm, T, 32] (canonical); points None (generators BulletproofGens(gen_n, T / (2 gen_n)), G then H),
        [T, 32] shared by every instance or [n_msm, T, 32]; path 0 production plan (big_min as msm_plan_for), 1 window width c with `knob` slices / parts,
        2 generator tables.  -> (rc, out [n_msm, 32] compressed sums, (width, slices | parts | blocks, kernel))"""
        s = _u8(scalars); n_msm, T = s.shape[0], s.shape[1]; s = s.reshape(n_msm, T, 32)
        p = None if points is None else _u8(points)
        per = 0 if p is None or p.ndim == 2 else 1
        if p is not None:
            assert p.shape == ((n_msm, T, 32) if per else (T, 32)), p.shape
        b = None if sB is None else _u8(sB, 32 * n_msm); h = None if sH is None else _u8(sH, 32 * n_msm)
        out = np.zeros((n_msm, 32), np.uint8); info = np.zeros(3, np.int32)
        rc = self.lib.rofl_debug_msm(self.h, _ptr(s), n_msm, T, _ptr(p), per, gen_n, path, c, knob, big_min, _ptr(b), _ptr(h), _ptr(out), _ptr(info))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, out, tuple(int(x) for x in info)

    def set_option(self, name, value):
        rc = self.lib.rofl_set_option(self.h, name.encode(), int(value))
        if rc != 0:
            raise self._err(rc)

    def set_use_rt(self, on):
        self.set_option("use_rt", 1 if on else 0)

    def _err(self, rc):
        return RoflError(rc, (self.lib.rofl_last_error() or b"").decode())

    # ---- sizes / conversions
    def next_pow2(self, v): return self.lib.rofl_next_pow2(v)
    def range_proof_len(self, N): return self.lib.rofl_range_proof_len(N)
    def range_proof_shape(self, D, rng, n_partition):
        a, b = c_sz(), c_sz(); self.lib.rofl_range_proof_shape(D, rng, n_partition, C.byref(a), C.byref(b)); return a.value, b.value
    def clip_bounds(self, rng, n_bits, frac):
        mn, mx = C.c_float(), C.c_float(); self.lib.rofl_clip_bounds(rng, n_bits, frac, C.byref(mn), C.byref(mx)); return mn.value, mx.value
    def l2_clip_bound(self, rng, n_bits, frac): return self.lib.rofl_l2_clip_bound(rng, n_bits, frac)
    def clip_f32_to_range_vec(self, v, rng, n_bits, frac):
        v = _f32(v); o = np.empty_like(v); self.lib.rofl_clip_f32_to_range_vec(_ptr(v), v.size, rng, n_bits, frac, _ptr(o)); return o
    def rnd_scalar_vec(self, seed, D):
        o = np.zeros((D, 32), np.uint8); self.lib.rofl_rnd_scalar_vec(_ptr(_seed(seed)), D, _ptr(o)); return o
    def f32_to_scalar_vec(self, v, n_bits, frac):
        v = _f32(v); o = np.zeros((v.size, 32), np.uint8)
        rc = self.lib.rofl_f32_to_scalar_vec(self.h, _ptr(v), v.size, n_bits, frac, _ptr(o))
        if rc: raise self._err(rc)
        return o
    def scalar_to_f32_vec(self, s, n_bits, frac):
        s = _u8(s).reshape(-1, 32); o = np.zeros(s.shape[0], np.float32)
        rc = self.lib.rofl_scalar_to_f32_vec(self.h, _ptr(s), s.shape[0], n_bits, frac, _ptr(o))
        if rc: raise self._err(rc)
        return o

    # ---- commitments
    def commit(self, v, blind, n_bits, frac, want_R=False):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D) if blind is not None else None
        L = np.zeros((D, 32), np.uint8); R = np.zeros((D, 32), np.uint8) if (want_R and b is not None) else None
        rc = self.lib.rofl_commit(self.h, _ptr(v), _ptr(b), D, n_bits, frac, _ptr(L), _ptr(R))
        if rc: raise self._err(rc)
        return (L, R) if want_R else L

    # ---- range proofs; return (rc, proofs[n_proofs, proof_len], commits[D, 32])
    def range_prove(self, v, blind, rng, n_partition, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        npf, plen = self.range_proof_shape(D, rng, n_partition)
        proofs = np.zeros((npf, max(plen, 1)), np.uint8); commits = np.zeros((D, 32), np.uint8)
        a, c = c_sz(), c_sz()
        rc = self.lib.rofl_range_prove(self.h, _ptr(v), _ptr(b), D, rng, n_partition, n_bits, frac, _ptr(_seed(seed)), _ptr(proofs), C.byref(a), C.byref(c), _ptr(commits))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proofs, commits
    def range_prove_dev(self, v_ptr, blind_ptr, D, rng, n_partition, n_bits, frac, seed, commits_ptr):
        npf, plen = self.range_proof_shape(D, rng, n_partition)
        proofs = np.zeros((npf, max(plen, 1)), np.uint8); a, c = c_sz(), c_sz()
        rc = self.lib.rofl_range_prove_dev(self.h, v_ptr, blind_ptr, D, rng, n_partition, n_bits, frac, _ptr(_seed(seed)), _ptr(proofs), C.byref(a), C.byref(c), commits_ptr)
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proofs
    def range_verify(self, proofs, commits, rng, seed=None):
        p = _u8(proofs); p = p.reshape(p.shape[0], -1); c = _u8(commits).reshape(-1, 32)
        rc = self.lib.rofl_range_verify(self.h, _ptr(p), p.shape[1], p.shape[0], _ptr(c), c.shape[0], rng, _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    def range_prove_shard(self, v, blind, chunk_len, chunk_begin, n_chunks, rng, n_bits, frac, seed=None, out_commits=None):
        """Chunks [chunk_begin, chunk_begin + n_chunks) of a larger update; v / blind hold the real elements of that slice.  out_commits: optional
        caller-owned uint8 [D, 32] buffer (e.g. a view of pinned memory) the commitments are written to."""
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        plen = self.range_proof_len(rng * chunk_len)
        proofs = np.zeros((n_chunks, plen), np.uint8); a = c_sz()
        commits = np.zeros((D, 32), np.uint8) if out_commits is None else out_commits
        assert commits.dtype == np.uint8 and commits.shape == (D, 32) and commits.flags["C_CONTIGUOUS"]
        rc = self.lib.rofl_range_prove_shard(self.h, _ptr(v), _ptr(b), D, chunk_len, chunk_begin, n_chunks, rng, n_bits, frac, _ptr(_seed(seed)), _ptr(proofs), C.byref(a), _ptr(commits))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proofs, commits
    def range_verify_shard(self, proofs, commits, chunk_len, chunk_begin, rng, seed=None):
        p = _u8(proofs); p = p.reshape(p.shape[0], -1); c = _u8(commits).reshape(-1, 32)
        rc = self.lib.rofl_range_verify_shard(self.h, _ptr(p), p.shape[1], p.shape[0], _ptr(c), c.shape[0], chunk_len, chunk_begin, rng, _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    def range_verify_dev(self, proofs, commits_ptr, D, rng, seed=None):
        p = _u8(proofs); p = p.reshape(p.shape[0], -1)
        rc = self.lib.rofl_range_verify_dev(self.h, _ptr(p), p.shape[1], p.shape[0], commits_ptr, D, rng, _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    def l2_prove(self, v, blind, rng, n_bits, frac, seed=None):
        v = _f32(v); D = v.size; b = _u8(blind, 32 * D)
        proof = np.zeros(self.range_proof_len(max(rng, 1)), np.uint8); commit = np.zeros(32, np.uint8); a = c_sz()
        rc = self.lib.rofl_l2_prove(self.h, _ptr(v), _ptr(b), D, rng, n_bits, frac, _ptr(_seed(seed)), _ptr(proof), C.byref(a), _ptr(commit))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proof, commit
    def l2_verify(self, proof, commit, rng, seed=None):
        p = _u8(proof)
        rc = self.lib.rofl_l2_verify(self.h, _ptr(p), p.size, _ptr(_u8(commit, 32)), rng, _ptr(_seed(seed)))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    # ---- square proofs
    def square_prove(self, v, value_com, r1, r2, n_bits, frac, seed=None):
        v = _f32(v); D = v.size
        proofs = np.zeros((D, 160), np.uint8); commits = np.zeros((D, 64), np.uint8)
        rc = self.lib.rofl_square_prove(self.h, _ptr(v), _ptr(_u8(value_com, 32 * D)), _ptr(_u8(r1, 32 * D)), _ptr(_u8(r2, 32 * D)), D, n_bits, frac, _ptr(_seed(seed)), _ptr(proofs), _ptr(commits))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, proofs, commits
    def square_verify(self, proofs, commits):
        p = _u8(proofs).reshape(-1, 160); c = _u8(commits).reshape(-1, 64)
        rc = self.lib.rofl_square_verify(self.h, _ptr(p), _ptr(c), p.shape[0])
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc
    # ---- aggregate / decrypt
    def aggregate(self, pts, init_unity=0):
        a = _u8(pts); assert a.ndim == 3 and a.shape[2] == 32
        o = np.zeros((a.shape[1], 32), np.uint8)
        rc = self.lib.rofl_aggregate(self.h, _ptr(a), a.shape[0], a.shape[1], init_unity, _ptr(o))
        if rc: raise self._err(rc)
        return o
    def dlog(self, pts, table_size=1 << 16, bsgs_bits=16, n_bits=16, frac=7):
        a = _u8(pts).reshape(-1, 32); s = np.zeros_like(a); f = np.zeros(a.shape[0], np.float32)
        rc = self.lib.rofl_dlog(self.h, _ptr(a), a.shape[0], table_size, bsgs_bits, n_bits, frac, _ptr(s), _ptr(f))
        if rc <= ROFL_ERR_CUDA: raise self._err(rc)
        return rc, s, f

    def accumulator(self, D, rec_bytes, init_unity=1):
        """A device-resident round accumulator (EncModelParamsAccumulator) of D elements over rec_bytes-wide records (32, 64 or 96)."""
        return Accumulator(self, D, rec_bytes, init_unity)


class Accumulator:
    """rofl_acc: clients are added as they arrive, the sums stay on the device; extract() checks R == B and decrypts L.
    Keep the Api (its context) alive while the accumulator is in use; close() or a with-block frees the device state."""

    def __init__(self, api, D, rec_bytes, init_unity=1):
        self.api, self.D, self.rec_bytes = api, D, rec_bytes
        h = c_vp()
        rc = api.lib.rofl_acc_create(api.h, D, rec_bytes, init_unity, C.byref(h))
        if rc != 0:
            raise api._err(rc)
        self.h = h

    def close(self):
        if self.h:
            self.api.lib.rofl_acc_destroy(self.h); self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _mask(self, mask, K):
        if mask is None:
            return None
        m = np.ascontiguousarray(mask, np.int32)
        if m.size != K:
            raise ValueError(f"mask has {m.size} entries for {K} clients")
        return m

    def add(self, records, mask=None):
        """records [K, D, rec_bytes] (or [D, rec_bytes] for one client) -> out_added int32[K]: 1 added, 0 masked out, ROFL_ERR_POINT"""
        r = _u8(records).reshape(-1, self.D, self.rec_bytes); K = r.shape[0]
        m = self._mask(mask, K); added = np.zeros(K, np.int32)
        rc = self.api.lib.rofl_acc_add(self.h, _ptr(r), K, _ptr(m), _ptr(added))
        if rc < 0: raise self.api._err(rc)
        return added

    def add_dev(self, ptr, n_clients, mask=None):
        """records already on the device (n_clients x D x rec_bytes at address ptr, e.g. a torch CUDA tensor's data_ptr()) -> out_added"""
        m = self._mask(mask, n_clients); added = np.zeros(n_clients, np.int32)
        rc = self.api.lib.rofl_acc_add_dev(self.h, ptr, n_clients, _ptr(m), _ptr(added))
        if rc < 0: raise self.api._err(rc)
        return added

    @property
    def count(self):
        return self.api.lib.rofl_acc_count(self.h)

    def reset(self):
        """back to the initial state with count 0, the device memory kept (the next round)"""
        rc = self.api.lib.rofl_acc_reset(self.h)
        if rc: raise self.api._err(rc)

    def export(self):
        """-> uint8 [D, 32] (rec_bytes 32) or [D, 64] (L | R): canonical encodings of the accumulated values"""
        o = np.zeros((self.D, 32 if self.rec_bytes == 32 else 64), np.uint8)
        rc = self.api.lib.rofl_acc_export(self.h, _ptr(o))
        if rc: raise self.api._err(rc)
        return o

    def extract(self, table_size=1 << 16, bsgs_bits=16, n_bits=16, frac=7):
        """-> (rc, scalars [D, 32], f32 [D]); rc 0, ROFL_ERR_UNBALANCED (-8, an R is not B: outputs stay zero), ROFL_ERR_DLOG (-5) or ROFL_ERR_ARGS"""
        s = np.zeros((self.D, 32), np.uint8); f = np.zeros(self.D, np.float32)
        rc = self.api.lib.rofl_acc_extract(self.h, table_size, bsgs_bits, n_bits, frac, _ptr(s), _ptr(f))
        if rc <= ROFL_ERR_CUDA: raise self.api._err(rc)
        return rc, s, f


ROFL_ERR_CUDA = -100
