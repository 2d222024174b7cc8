"""Pin the oracle's arithmetic layers against independent anchors: libsodium ristretto255 (its outputs for seeded
inputs, stored in tests/golden/sodium.json by tools/gen_golden.py), hashlib SHA3/SHAKE, the published Merlin
conformance vector and the KATs of SURVEY.md Appendix A.6.  CPU only."""
import hashlib
import json
import os
import numpy as np
import pytest

L = 2**252 + 27742317777372353535851937790883648493
P = 2**255 - 19


@pytest.fixture(scope="module")
def sodium():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sodium.json")) as f:
        return json.load(f)


def test_kats_appendix_a6(oracle):
    assert oracle.basepoint().hex() == "e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76"
    assert oracle.scalarmult_base((2).to_bytes(32, "little")).hex() == "6a493210f7499cd17fecb510ae0cea23a110e8d5b901f8acadd3095c73a3b919"
    assert oracle.blinding_basepoint().hex() == "8c9240b456a9e6dc65c377a1048d745f94a08cdb7f44cbcd7b46f34048871134"
    assert oracle.scalarmult_base((160).to_bytes(32, "little")).hex() == "124f288e9cde61e6b965a69040d7c60405d94d494a0c5a35d65526cb980d9c01"
    assert oracle.scalarmult_base((L - 160).to_bytes(32, "little")).hex() == "d885fd552a977060d914d0509b646c8868fa3bac0eec8a395db285a83ab0e343"
    assert oracle.point_add(oracle.basepoint(), oracle.blinding_basepoint()).hex() == "b8180a6778aba0f7bd121a403e09146d274edf702241a67c67689dc9bd87dd10"
    # B_blinding = from_uniform_bytes(SHA3-512(compress(B)))  (el_gamal.rs:31-40)
    assert oracle.from_uniform_bytes(hashlib.sha3_512(oracle.basepoint()).digest()) == oracle.blinding_basepoint()


def test_merlin_conformance_vector(oracle):
    out = oracle.merlin_simple(b"test protocol", b"some label", b"some data", b"challenge", 32)
    assert out.hex() == "d5a21972d0d5fe320c0d263fac7fffb8145aa640af6e9bca177c03c7efcf0615"


def test_sha3_shake_vs_hashlib(oracle):
    rng = np.random.default_rng(0)
    for n in [0, 1, 71, 72, 73, 135, 136, 137, 1000]:
        m = rng.bytes(n)
        assert oracle.sha3_512(m) == hashlib.sha3_512(m).digest()
        assert oracle.sha3_256(m) == hashlib.sha3_256(m).digest()
        assert oracle.shake256(m, 700) == hashlib.shake_256(m).digest(700)


def test_chacha20_rfc8439_keystream_shape(oracle):
    # RFC 8439 2.3.2 uses a 32-bit counter + 96-bit nonce; with nonce 0 and counter 1 the block equals
    # our 64-bit-counter layout.  Check the well known all-zero-key block 0 instead (first keystream bytes).
    ks = oracle.chacha20_block(bytes(32), 0)
    assert ks[:16].hex() == "76b8e0ada0f13d90405d6ae55386bd28"
    ks1 = oracle.chacha20_block(bytes(32), 1)
    assert ks1[:16].hex() == "9f07e7be5551387a98ba977c732d080d"


def test_generator_chain_kats(oracle):
    g0 = oracle.bp_gens("G", 0, 2)
    assert g0[0].tobytes().hex() == "fc3b25801422672a6a8d3adb5d8457d4301fe92324b4fc56ae934c8713ddfe2d"
    assert g0[1].tobytes().hex() == "ae817fdef62f713dd169dc8a26406f68be0bd3cd53652614636b0801567c4264"
    assert oracle.bp_gens("H", 0, 1)[0].tobytes().hex() == "ba698f6dd08c501e32b55d2ee7259f6019d629fa2ba4d7039c5de157cba4df73"
    assert oracle.bp_gens("G", 1, 1)[0].tobytes().hex() == "0eeebec183d151ded1e24320cf43c987617b36e77114788e5ae8ace41570b74b"
    # definition: from_uniform_bytes(SHAKE256("GeneratorsChain" || 'G' || u32le(j)) stream)
    xof = hashlib.shake_256(b"GeneratorsChain" + b"G" + (3).to_bytes(4, "little")).digest(64 * 5)
    g3 = oracle.bp_gens("G", 3, 5)
    for i in range(5):
        assert g3[i].tobytes() == oracle.from_uniform_bytes(xof[64 * i:64 * i + 64])


def test_scalar_field_vs_python_and_sodium(oracle, sodium):
    assert len(sodium["scalar"]) == 200
    for e in sodium["scalar"]:
        ab, bb, w = bytes.fromhex(e["a"]), bytes.fromhex(e["b"]), bytes.fromhex(e["wide"])
        a, b = int.from_bytes(ab, "little"), int.from_bytes(bb, "little")
        assert int.from_bytes(oracle.sc_mul(ab, bb), "little") == a * b % L
        assert int.from_bytes(oracle.sc_add(ab, bb), "little") == (a + b) % L
        assert int.from_bytes(oracle.sc_sub(ab, bb), "little") == (a - b) % L
        assert int.from_bytes(oracle.sc_reduce_wide(w), "little") == int.from_bytes(w, "little") % L
        assert oracle.sc_mul(ab, bb).hex() == e["mul"]
        assert oracle.sc_reduce_wide(w).hex() == e["reduce"]
    for a in [1, 2, L - 1, 12345678901234567890]:
        inv = int.from_bytes(oracle.sc_invert(a.to_bytes(32, "little")), "little")
        assert inv * a % L == 1
    edge = bytes([0xff] * 64)
    assert int.from_bytes(oracle.sc_reduce_wide(edge), "little") == int.from_bytes(edge, "little") % L
    assert oracle.sc_is_canonical((L - 1).to_bytes(32, "little")) and not oracle.sc_is_canonical(L.to_bytes(32, "little"))


def test_field_vs_python(oracle):
    rng = np.random.default_rng(2)
    for _ in range(200):
        a = int.from_bytes(rng.bytes(32), "little") % P
        b = int.from_bytes(rng.bytes(32), "little") % P
        assert int.from_bytes(oracle.fe_mul(a.to_bytes(32, "little"), b.to_bytes(32, "little")), "little") == a * b % P
        if a:
            assert int.from_bytes(oracle.fe_invert(a.to_bytes(32, "little")), "little") * a % P == 1
    m1 = (P - 1).to_bytes(32, "little")
    assert int.from_bytes(oracle.fe_mul(m1, m1), "little") == 1


def test_group_vs_sodium(oracle, sodium):
    assert len(sodium["group"]) == 40
    for e in sodium["group"]:
        h, p, s = bytes.fromhex(e["hash"]), bytes.fromhex(e["point"]), bytes.fromhex(e["scalar"])
        q = bytes.fromhex(e["scalarmult"])
        assert oracle.from_uniform_bytes(h) == p
        assert oracle.scalarmult(s, p) == q
        assert oracle.scalarmult_base(s).hex() == e["scalarmult_base"]
        assert oracle.point_add(p, q).hex() == e["add"]
        assert oracle.point_sub(p, q).hex() == e["sub"]
        assert oracle.point_valid(p)
    # decode rejection agrees with libsodium on random / edge encodings
    assert len(sodium["valid"]) == 306
    for e in sodium["valid"]:
        b = bytes.fromhex(e["bytes"])
        assert oracle.point_valid(b) == e["valid"] or b == bytes(32)
    assert oracle.point_valid(bytes(32))        # identity decodes in dalek (libsodium's is_valid_point rejects it)


def test_msm_straus_pippenger_vs_naive(oracle):
    rng = np.random.default_rng(4)
    for n in [1, 3, 50, 189, 190, 600, 900]:
        pts = np.stack([np.frombuffer(oracle.from_uniform_bytes(rng.bytes(64)), np.uint8) for _ in range(n)])
        scs = np.stack([np.frombuffer((int.from_bytes(rng.bytes(32), "little") % L).to_bytes(32, "little"), np.uint8) for _ in range(n)])
        acc = bytes(32)
        for i in range(n):
            acc = oracle.point_add(acc, oracle.scalarmult(scs[i].tobytes(), pts[i].tobytes()))
        assert oracle.msm(scs, pts) == acc
