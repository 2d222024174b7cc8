#!/usr/bin/env python3
"""Generate tests/golden/*.json.

Two kinds of fixtures (the reference itself ships no golden vectors and cannot be built here -- no cargo -- see DESIGN.md section 2):
  primitives.json  produced by INDEPENDENT implementations present in this image: libsodium ristretto255 (pyzmq's bundled copy)
                   and hashlib.  They pin the group / scalar / hash layers of the oracle and of the CUDA library.
  protocol.json    produced by the oracle (oracle/, itself pinned by primitives.json and the reference's literal-value unit
                   tests) for fixed seeds: commitments, range / L2 / square proofs, aggregates and decrypted values.  They
                   freeze the byte-level behaviour so that the GPU box (which has neither /root/reference nor a need to
                   re-derive anything) can compare the CUDA path against committed bytes.
  sodium.json      libsodium's outputs for the seeded inputs of tests/test_oracle_primitives.py, which compares the oracle with them.
Usage: python tools/gen_golden.py   (deterministic; re-running must not change the files)
"""
import ctypes as C
import glob
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402

L = 2**252 + 27742317777372353535851937790883648493


def sodium():
    import zmq
    cands = glob.glob(os.path.join(os.path.dirname(os.path.dirname(zmq.__file__)), "pyzmq.libs", "libsodium*.so*"))
    lib = C.CDLL(cands[0]); assert lib.sodium_init() >= 0
    return lib


def sod(lib, name, outlen, *ins):
    o = C.create_string_buffer(outlen)
    fn = getattr(lib, name)
    void = name in ("crypto_core_ristretto255_scalar_mul", "crypto_core_ristretto255_scalar_add", "crypto_core_ristretto255_scalar_reduce")
    fn.restype = None if void else C.c_int
    rc = fn(o, *[C.c_char_p(bytes(i)) for i in ins])
    assert void or rc == 0, name
    return o.raw


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def sodium_vectors(lib):
    """libsodium's answers for the inputs tests/test_oracle_primitives.py draws (same generators, same order), so that the
    oracle is compared with libsodium without loading it at test time."""
    out = {"source": "libsodium crypto_core_ristretto255_* / crypto_scalarmult_ristretto255*", "scalar": [], "group": [], "valid": []}
    rng = np.random.default_rng(1)
    for _ in range(200):
        a = (int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little")
        b = (int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little")
        w = rng.bytes(64)
        out["scalar"].append({"a": a.hex(), "b": b.hex(), "wide": w.hex(), "mul": sod(lib, "crypto_core_ristretto255_scalar_mul", 32, a, b).hex(),
                              "reduce": sod(lib, "crypto_core_ristretto255_scalar_reduce", 32, w).hex()})
    rng = np.random.default_rng(3)
    for _ in range(40):
        h = rng.bytes(64)
        p = sod(lib, "crypto_core_ristretto255_from_hash", 32, h)
        s = (int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little")
        q = sod(lib, "crypto_scalarmult_ristretto255", 32, s, p)
        out["group"].append({"hash": h.hex(), "point": p.hex(), "scalar": s.hex(), "scalarmult": q.hex(), "scalarmult_base": sod(lib, "crypto_scalarmult_ristretto255_base", 32, s).hex(),
                             "add": sod(lib, "crypto_core_ristretto255_add", 32, p, q).hex(), "sub": sod(lib, "crypto_core_ristretto255_sub", 32, p, q).hex()})
    P = 2**255 - 19
    edge = [bytes(32), bytes([1] + [0] * 31), P.to_bytes(32, "little"), (P - 1).to_bytes(32, "little"), bytes([0xff] * 32), bytes([2] + [0] * 30 + [0x80])]
    for e in edge + [rng.bytes(32) for _ in range(300)]:
        out["valid"].append({"bytes": e.hex(), "valid": bool(lib.crypto_core_ristretto255_is_valid_point(C.c_char_p(e)))})
    return out


def main():
    oracle.build()
    lib = sodium()
    rng = np.random.default_rng(20261017)
    prim = {"source": "libsodium crypto_core_ristretto255_* / crypto_scalarmult_ristretto255* and hashlib", "base_multiples": [], "from_hash": [], "scalarmult": [], "add_sub": [],
            "scalar_ops": [], "scalar_reduce": [], "sha3_512": [], "shake256": []}
    for k in list(range(1, 17)) + [160, 2**16, 2**32 - 1, L - 1]:
        s = (k % L).to_bytes(32, "little")
        prim["base_multiples"].append({"k": str(k), "point": sod(lib, "crypto_scalarmult_ristretto255_base", 32, s).hex()})
    for _ in range(12):
        h = rng.bytes(64)
        prim["from_hash"].append({"hash": h.hex(), "point": sod(lib, "crypto_core_ristretto255_from_hash", 32, h).hex()})
    pts = [bytes.fromhex(e["point"]) for e in prim["from_hash"]]
    for i in range(8):
        s = (int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little")
        prim["scalarmult"].append({"scalar": s.hex(), "point": pts[i].hex(), "out": sod(lib, "crypto_scalarmult_ristretto255", 32, s, pts[i]).hex()})
        prim["add_sub"].append({"p": pts[i].hex(), "q": pts[i + 1].hex(), "add": sod(lib, "crypto_core_ristretto255_add", 32, pts[i], pts[i + 1]).hex(),
                                "sub": sod(lib, "crypto_core_ristretto255_sub", 32, pts[i], pts[i + 1]).hex()})
        a = (int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little"); b = (int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little")
        prim["scalar_ops"].append({"a": a.hex(), "b": b.hex(), "mul": sod(lib, "crypto_core_ristretto255_scalar_mul", 32, a, b).hex(),
                                   "add": sod(lib, "crypto_core_ristretto255_scalar_add", 32, a, b).hex(), "inv_a": sod(lib, "crypto_core_ristretto255_scalar_invert", 32, a).hex()})
        w = rng.bytes(64)
        prim["scalar_reduce"].append({"wide": w.hex(), "out": sod(lib, "crypto_core_ristretto255_scalar_reduce", 32, w).hex()})
    for n in [0, 1, 71, 72, 136, 137, 500]:
        m = rng.bytes(n)
        prim["sha3_512"].append({"msg": m.hex(), "out": hashlib.sha3_512(m).hexdigest()})
        prim["shake256"].append({"msg": m.hex(), "out": hashlib.shake_256(m).hexdigest(96)})
    prim["merlin_conformance"] = {"proto": "test protocol", "label": "some label", "msg": "some data", "challenge_label": "challenge",
                                  "out": "d5a21972d0d5fe320c0d263fac7fffb8145aa640af6e9bca177c03c7efcf0615", "source": "merlin 3.0.0 transcript.rs test `equivalence_simple` (published constant)"}

    prot = {"source": "oracle/ (CPU restatement, pinned by primitives.json); seeds and inputs below reproduce every entry", "cases": []}
    # commitments and conversion
    v = np.array([0.0, -0.0, 0.25, -1.5, 3.0078125, -255.9921875, 600.0, -600.0], np.float32)
    bl = oracle.rnd_scalar_vec(b"\x41" * 32, v.size)
    prot["commit"] = {"values": v.tolist(), "blind_seed": "41" * 32, "n_bits": 16, "frac": 7,
                      "scalars": np.asarray(oracle.f32_to_scalar_vec(v, 16, 7)).tobytes().hex(),
                      "L": np.asarray(oracle.commit_f32(v, bl, 16, 7)).tobytes().hex(), "R": np.asarray(oracle.elgamal_R(bl)).tobytes().hex(),
                      "L_no_blinding": np.asarray(oracle.commit_f32(v, None, 16, 7)).tobytes().hex()}
    # range proofs (configs[0]-like shapes at toy size + one 16-bit and one 32-bit case)
    for (D, rb, Pn, nb, seedb) in [(5, 8, 2, 16, 7), (3, 16, 4, 16, 8), (4, 32, 2, 32, 9), (37, 8, 4, 16, 3)]:
        r2 = np.random.default_rng(D * 1000 + rb)
        mn, mx = oracle.clip_bounds(rb, nb, 7)
        vals = r2.uniform(mn, mx, D).astype(np.float32); vals[0] = mx; vals[-1] = mn
        blind = oracle.rnd_scalar_vec(bytes([seedb + 0x40]) * 32, D)
        rc, proofs, commits = oracle.range_prove(vals, blind, rb, Pn, nb, 7, bytes([seedb]) * 32)
        assert rc == 0 and oracle.range_verify(proofs, commits, rb, bytes([seedb]) * 32) == 1
        prot["cases"].append({"kind": "range", "D": D, "range_bits": rb, "n_partition": Pn, "n_bits": nb, "frac": 7, "values": [float(x) for x in vals], "blind_seed": bytes([seedb + 0x40]).hex() * 32,
                              "seed": bytes([seedb]).hex() * 32, "proofs_shape": list(np.asarray(proofs).shape), "proofs": np.asarray(proofs).tobytes().hex(),
                              "commits": np.asarray(commits).tobytes().hex()})
    # L2 (sum of squares, 32-bit) + square proofs
    D = 6
    r2 = np.random.default_rng(5)
    vals = (r2.integers(-24, 25, D) / 128).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(b"\x33" * 32, D); r2s = oracle.rnd_scalar_vec(b"\x34" * 32, D)
    rc, pf, cm = oracle.l2_prove(vals, r2s, 32, 32, 7, bytes([9]) * 32); assert rc == 0
    cl = oracle.commit_f32(vals, r1, 32, 7)
    rc, sp, sc = oracle.square_prove(vals, cl, r1, r2s, 32, 7, bytes([9]) * 32); assert rc == 0 and oracle.square_verify(sp, sc) == 1
    prot["l2"] = {"values": [float(x) for x in vals], "r1_seed": "33" * 32, "r2_seed": "34" * 32, "seed": "09" * 32, "range_bits": 32, "n_bits": 32, "frac": 7,
                  "proof": np.asarray(pf).tobytes().hex(), "commit": bytes(cm).hex() if not isinstance(cm, np.ndarray) else cm.tobytes().hex(),
                  "square_proofs": np.asarray(sp).tobytes().hex(), "square_commits": np.asarray(sc).tobytes().hex()}
    # compressed randomness proof (one sigma proof over all ElGamal pairs)
    D = 10
    r3 = np.random.default_rng(77)
    vals = r3.uniform(-3, 3, D).astype(np.float32); blind = oracle.rnd_scalar_vec(b"\x64" * 32, D)
    rc, pf, pairs = oracle.crp_prove(vals, None, blind, 16, 7, bytes([6]) * 32); assert rc == 0 and oracle.crp_verify(pf, pairs) == 1
    prot["crp"] = {"values": [float(x) for x in vals], "blind_seed": "64" * 32, "seed": "06" * 32, "n_bits": 16, "frac": 7,
                   "proof": np.asarray(pf).tobytes().hex(), "pairs": np.asarray(pairs).tobytes().hex()}
    # per-element proofs of the un-optimised encodings (enc types 2 and 3)
    D = 5
    r4 = np.random.default_rng(78)
    vals = (r4.integers(-300, 300, D) / 128).astype(np.float32)
    r1 = oracle.rnd_scalar_vec(b"\x65" * 32, D); r2s = oracle.rnd_scalar_vec(b"\x66" * 32, D)
    rc, pf, pairs = oracle.rand_prove(vals, None, r1, 16, 7, bytes([11]) * 32); assert rc == 0 and oracle.rand_verify(pf, pairs) == 1
    rc, sp, sc = oracle.square_rand_prove(vals, None, r1, r2s, 32, 7, bytes([11]) * 32); assert rc == 0 and oracle.square_rand_verify(sp, sc) == 1
    prot["rand"] = {"values": [float(x) for x in vals], "r1_seed": "65" * 32, "r2_seed": "66" * 32, "seed": "0b" * 32, "frac": 7,
                    "rand_n_bits": 16, "rand_proofs": np.asarray(pf).tobytes().hex(), "rand_pairs": np.asarray(pairs).tobytes().hex(),
                    "square_rand_n_bits": 32, "square_rand_proofs": np.asarray(sp).tobytes().hex(), "square_rand_commits": np.asarray(sc).tobytes().hex()}
    # aggregate + discrete log
    x = np.array([[0.25, 1.25, -1.5, 100.5], [-0.75, 1.25, -2.0, 27.25], [0.5, 1.25, -3.0, 0.0078125]], np.float32)
    cs = np.stack([oracle.commit_f32(r, None, 16, 7) for r in x])
    agg = oracle.aggregate(cs, 0)
    rc, s = oracle.dlog(agg, 1 << 16, 16); assert rc == 0
    prot["aggregate"] = {"clients": x.tolist(), "n_bits": 16, "frac": 7, "sum_unity_start": np.asarray(oracle.aggregate(cs, 1)).tobytes().hex(), "sum": np.asarray(agg).tobytes().hex(),
                         "dlog_scalars": np.asarray(s).tobytes().hex(), "decoded": [float(t) for t in oracle.scalar_to_f32_vec(s, 16, 7)]}
    # generators
    prot["bp_gens"] = {"G_party0_first4": np.asarray(oracle.bp_gens("G", 0, 4)).tobytes().hex(), "H_party0_first4": np.asarray(oracle.bp_gens("H", 0, 4)).tobytes().hex(),
                       "G_party5_first2": np.asarray(oracle.bp_gens("G", 5, 2)).tobytes().hex()}
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    for name, obj in [("primitives.json", prim), ("protocol.json", prot), ("sodium.json", sodium_vectors(lib))]:
        with open(os.path.join(ROOT, "tests", "golden", name), "w") as f:
            json.dump(obj, f, indent=1, sort_keys=True); f.write("\n")
    print("wrote tests/golden/primitives.json, protocol.json, sodium.json")


if __name__ == "__main__":
    main()
