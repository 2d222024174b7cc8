"""The device-resident round accumulator (rofl_acc_*, EncModelParamsAccumulator params.rs:74-148): clients are added as they arrive, the
sums stay on the device, extract checks that every accumulated R is B and decrypts L.  The emulation tests run the product kernels and
engine on CPU threads at tiny sizes, exact against the oracle; the GPU tests run a configs[4]-sized round on the B200 library."""
import ctypes as C
import importlib.util
import os
import sys
import threading
import numpy as np
import pytest
from conftest import locked_make

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NB, FR = 16, 7
TS, BB = 1 << 9, 16                        # small BSGS table in the emulation: giant steps
ROFL_ERR_ARGS, ROFL_ERR_POINT, ROFL_ERR_DLOG, ROFL_ERR_UNBALANCED = -2, -4, -5, -8


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


def quantised(rng, K, D, lo=-24, hi=25):
    return [(rng.integers(lo, hi, D) / 128).astype(np.float32) for _ in range(K)]


def make_records(oracle, vs, bls, rec_bytes):
    """[K, D, rec_bytes]: L = commit(v, r) | R = r B | c_sq = commit(v, r) + B (any valid point; it is validated, never added)"""
    K, D = len(vs), vs[0].size
    out = np.zeros((K, D, rec_bytes), np.uint8)
    for k in range(K):
        L = oracle.commit_f32(vs[k], bls[k], NB, FR)
        out[k, :, :32] = L
        if rec_bytes >= 64:
            out[k, :, 32:64] = oracle.elgamal_R(bls[k])
        if rec_bytes == 96:
            B = oracle.basepoint()
            out[k, :, 64:] = np.stack([np.frombuffer(oracle.point_add(bytes(x), B), np.uint8) for x in L])
    return out


def random_blindings(api, K, D, tag=0x20):
    return [api.rnd_scalar_vec(bytes([(tag + k) & 0xff]) * 32, D) for k in range(K)]


def oracle_export(oracle, recs, init):
    cols = [oracle.aggregate(np.ascontiguousarray(recs[:, :, 0:32]), init)]
    if recs.shape[2] >= 64:
        cols.append(oracle.aggregate(np.ascontiguousarray(recs[:, :, 32:64]), init))
    return np.concatenate(cols, axis=1)


def undecodable(oracle, pt):
    for byte in range(31):
        for bit in range(8):
            x = pt.copy(); x[byte] ^= 1 << bit
            if not oracle.point_valid(x):
                return x
    raise AssertionError("no such flip")


@pytest.mark.parametrize("rec_bytes", [32, 64, 96])
@pytest.mark.parametrize("init", [0, 1])
def test_export_matches_oracle(api, oracle, rec_bytes, init):
    rng = np.random.default_rng(rec_bytes + init)
    K, D = 5, 7
    recs = make_records(oracle, quantised(rng, K, D), random_blindings(api, K, D), rec_bytes)
    with api.accumulator(D, rec_bytes, init) as acc:
        assert acc.count == 0
        assert acc.add(recs).tolist() == [1] * K and acc.count == K
        got = acc.export()
    assert got.shape == (D, 32 if rec_bytes == 32 else 64)
    assert (got == oracle_export(oracle, recs, init)).all()
    assert (got[:, :32] == api.aggregate(np.ascontiguousarray(recs[:, :, :32]), init)).all()
    if rec_bytes >= 64:
        assert (got[:, 32:] == api.aggregate(np.ascontiguousarray(recs[:, :, 32:64]), init)).all()


def test_initial_state(api, oracle):
    B = np.frombuffer(oracle.basepoint(), np.uint8)
    with api.accumulator(3, 64, 1) as acc:
        assert (acc.export() == np.tile(B, 2)).all()
    with api.accumulator(3, 64, 0) as acc:
        assert (acc.export() == 0).all()                      # the identity encodes as 32 zero bytes


def test_order_independence(api, oracle):
    rng = np.random.default_rng(11)
    K, D = 8, 5
    recs = make_records(oracle, quantised(rng, K, D), random_blindings(api, K, D, 0x31), 96)

    def run(groups, threads=False):
        with api.accumulator(D, 96, 1) as acc:
            if threads:
                errs = []
                def work(g):
                    try:
                        for idx in g:
                            assert acc.add(recs[idx]).tolist() == [1] * len(idx)
                    except Exception as ex:  # noqa: BLE001
                        errs.append(ex)
                th = [threading.Thread(target=work, args=(g,)) for g in groups]
                [t.start() for t in th]; [t.join() for t in th]
                assert not errs, errs
            else:
                for idx in groups:
                    assert acc.add(recs[idx]).tolist() == [1] * len(idx)
            assert acc.count == K
            return acc.export().tobytes()

    ref = run([list(range(K))])
    assert ref == oracle_export(oracle, recs, 1).tobytes()
    assert run([[k] for k in range(K)]) == ref
    assert run([[k] for k in reversed(range(K))]) == ref
    assert run([[5, 1, 7], [0], [6, 2, 3, 4]]) == ref
    # four threads adding disjoint subsets concurrently, each in several calls
    assert run([[[0], [4]], [[1, 5]], [[2], [6]], [[7], [3]]], threads=True) == ref


def test_mask(api, oracle):
    rng = np.random.default_rng(12)
    K, D = 6, 4
    recs = make_records(oracle, quantised(rng, K, D), random_blindings(api, K, D, 0x41), 64)
    mask = np.array([1, 0, 1, -4, 1, 0], np.int32)           # a verifier's out_ok: only 1 means accepted
    with api.accumulator(D, 64, 1) as acc:
        assert acc.add(recs, mask).tolist() == [1, 0, 1, 0, 1, 0]
        assert acc.count == 3
        assert (acc.export() == oracle_export(oracle, recs[[0, 2, 4]], 1)).all()
        assert acc.add(recs[1:2], [1]).tolist() == [1] and acc.count == 4
        assert (acc.export() == oracle_export(oracle, recs[[0, 1, 2, 4]], 1)).all()
        assert acc.add(recs, np.zeros(K, np.int32)).tolist() == [0] * K and acc.count == 4


@pytest.mark.parametrize("col", [0, 1, 2])
def test_malformed_record(api, oracle, col):
    """an undecodable point in any column of client k (c_sq included): nothing of k is added, the other clients are"""
    rng = np.random.default_rng(13 + col)
    K, D = 4, 5
    recs = make_records(oracle, quantised(rng, K, D), random_blindings(api, K, D, 0x51), 96)
    bad = recs.copy(); bad[2, 3, 32 * col:32 * col + 32] = undecodable(oracle, recs[2, 3, 32 * col:32 * col + 32])
    with api.accumulator(D, 96, 1) as acc:
        assert acc.add(bad).tolist() == [1, 1, ROFL_ERR_POINT, 1]
        assert acc.count == 3
        assert (acc.export() == oracle_export(oracle, recs[[0, 1, 3]], 1)).all()
        assert acc.add(bad, [0, 0, 0, 0]).tolist() == [0, 0, 0, 0]          # masked out: not even looked at
    with api.accumulator(D, 96, 1) as acc:
        assert acc.add(bad[2:3]).tolist() == [ROFL_ERR_POINT] and acc.count == 0
        assert (acc.export() == oracle_export(oracle, recs[:0], 1)).all()


def balanced_round(api, oracle, K, D, rec_bytes, seed):
    rng = np.random.default_rng(seed)
    vs = quantised(rng, K, D)
    bls = api.cancelling_blindings(K, D, seed & 0xff)
    return vs, bls, make_records(oracle, vs, bls, rec_bytes)


@pytest.mark.parametrize("rec_bytes", [64, 96])
def test_extract_balanced(api, oracle, rec_bytes):
    K, D = 3, 6
    vs, _, recs = balanced_round(api, oracle, K, D, rec_bytes, 21)
    with api.accumulator(D, rec_bytes, 1) as acc:
        acc.add(recs)
        exp = acc.export()
        assert (exp[:, 32:] == np.frombuffer(oracle.basepoint(), np.uint8)).all()
        rc, s, f = acc.extract(TS, BB, NB, FR)
        assert rc == 0
        assert (f == (np.sum(np.stack(vs), axis=0, dtype=np.float64) + 2.0 ** -FR).astype(np.float32)).all()
        rc_d, s_d, f_d = api.dlog(np.ascontiguousarray(exp[:, :32]), TS, BB, NB, FR)
        assert rc_d == 0 and (s == s_d).all() and (f == f_d).all()
        rc_o, s_o = oracle.dlog(np.ascontiguousarray(exp[:, :32]), TS, BB)
        assert rc_o == 0 and (s == s_o).all()
        assert (acc.export() == exp).all() and acc.count == K            # extract leaves the accumulator as it was
        rc, s2, f2 = acc.extract(TS, BB, NB, FR)
        assert rc == 0 and (s2 == s).all() and (f2 == f).all()


def test_extract_unbalanced(api, oracle):
    K, D = 3, 4
    rng = np.random.default_rng(22)
    vs = quantised(rng, K, D)
    # blindings that do not cancel
    recs = make_records(oracle, vs, random_blindings(api, K, D, 0x61), 64)
    with api.accumulator(D, 64, 1) as acc:
        acc.add(recs)
        rc, s, f = acc.extract(TS, BB, NB, FR)
        assert rc == ROFL_ERR_UNBALANCED and not s.any() and not f.any()       # nothing written
    # cancelling blindings, but one client's blinding off at a single element
    bls = api.cancelling_blindings(K, D, 0x62)
    bls[1] = bls[1].copy(); bls[1][2] = api.rnd_scalar_vec(b"\x77" * 32, 1)[0]
    recs = make_records(oracle, vs, bls, 96)
    with api.accumulator(D, 96, 1) as acc:
        acc.add(recs)
        assert acc.extract(TS, BB, NB, FR)[0] == ROFL_ERR_UNBALANCED
    # an accumulator without clients is balanced at the unity (R = B) and decrypts to one LSB
    with api.accumulator(D, 64, 1) as acc:
        rc, _, f = acc.extract(TS, BB, NB, FR)
        assert rc == 0 and (f == np.float32(2.0 ** -FR)).all()
    # started at the identity, R = identity != B
    with api.accumulator(D, 64, 0) as acc:
        assert acc.extract(TS, BB, NB, FR)[0] == ROFL_ERR_UNBALANCED


def test_extract_out_of_range(api, oracle):
    K, D = 2, 3
    vs = [np.full(D, 200.0, np.float32), np.full(D, 200.0, np.float32)]
    bls = api.cancelling_blindings(K, D, 0x71)
    recs = make_records(oracle, vs, bls, 64)
    with api.accumulator(D, 64, 1) as acc:
        acc.add(recs)
        assert acc.extract(1 << 4, 8, 8, FR)[0] == ROFL_ERR_DLOG


def test_extract_commitments_no_R_check(api, oracle):
    """rec_bytes 32 (Pedersen commitments, add_rp_vec_vec): no R to check; unblinded commitments decrypt to the sum"""
    rng = np.random.default_rng(24)
    K, D = 4, 5
    vs = quantised(rng, K, D)
    recs = np.stack([oracle.commit_f32(v, None, NB, FR) for v in vs]).reshape(K, D, 32)
    for init, extra in ((0, 0.0), (1, 2.0 ** -FR)):
        with api.accumulator(D, 32, init) as acc:
            acc.add(recs)
            rc, s, f = acc.extract(TS, BB, NB, FR)
            assert rc == 0 and (f == (np.sum(np.stack(vs), axis=0, dtype=np.float64) + extra).astype(np.float32)).all()
            assert (s == api.dlog(acc.export(), TS, BB, NB, FR)[1]).all()


def test_reset(api, oracle):
    K, D = 3, 4
    vs, _, recs = balanced_round(api, oracle, K, D, 96, 31)
    with api.accumulator(D, 96, 1) as fresh:
        fresh.add(recs)
        want = fresh.export()
    with api.accumulator(D, 96, 1) as acc:
        init = acc.export()
        acc.add(recs[:2]); acc.add(recs[1:])
        assert acc.count == 4
        acc.reset()
        assert acc.count == 0 and (acc.export() == init).all()
        acc.add(recs)
        assert acc.count == K and (acc.export() == want).all()
        assert acc.extract(TS, BB, NB, FR)[0] == 0


def test_bad_arguments(api):
    lib = api.lib
    h = C.c_void_p()
    assert lib.rofl_acc_create(api.h, 0, 64, 1, C.byref(h)) == ROFL_ERR_ARGS and not h.value
    for rb in (0, 31, 48, 128):
        assert lib.rofl_acc_create(api.h, 4, rb, 1, C.byref(h)) == ROFL_ERR_ARGS and not h.value
    assert lib.rofl_acc_create(api.h, 4, 64, 2, C.byref(h)) == ROFL_ERR_ARGS
    assert lib.rofl_acc_create(None, 4, 64, 1, C.byref(h)) == ROFL_ERR_ARGS
    assert lib.rofl_acc_create(api.h, 4, 64, 1, None) == ROFL_ERR_ARGS
    assert lib.rofl_acc_reset(None) == ROFL_ERR_ARGS
    assert lib.rofl_acc_add(None, b"\0" * 64, 1, None, None) == ROFL_ERR_ARGS
    assert lib.rofl_acc_add_dev(None, b"\0" * 64, 1, None, None) == ROFL_ERR_ARGS
    assert lib.rofl_acc_export(None, b"\0" * 64) == ROFL_ERR_ARGS
    assert lib.rofl_acc_extract(None, TS, BB, NB, FR, None, None) == ROFL_ERR_ARGS
    assert lib.rofl_acc_count(None) == 0
    lib.rofl_acc_destroy(None)
    with api.accumulator(1, 64, 1) as acc:
        assert lib.rofl_acc_add(acc.h, None, 1, None, None) == ROFL_ERR_ARGS
        assert lib.rofl_acc_add_dev(acc.h, None, 1, None, None) == ROFL_ERR_ARGS
        assert lib.rofl_acc_export(acc.h, None) == ROFL_ERR_ARGS
        assert acc.extract(0, BB, NB, FR)[0] == ROFL_ERR_ARGS
        assert acc.extract(TS, 0, NB, FR)[0] == ROFL_ERR_ARGS
        assert acc.add(np.zeros((0, 1, 64), np.uint8)).tolist() == [] and acc.count == 0
        with pytest.raises(ValueError):
            acc.add(np.zeros((2, 1, 64), np.uint8), mask=[1])


# ---------------------------------------------------------------------------------------------------------- GPU (B200 library)
def cancelling(api, K, D, tag):
    """K blinding vectors of D scalars that sum to zero mod l"""
    return api.cancelling_blindings(K, D, tag)


@pytest.mark.gpu
def test_gpu_whole_round(gpu_api, oracle):
    """configs[4]: 48 EncL2Compressed messages of 50 000 parameters, verified in one batch call; the verdicts are the mask.  One client's
    message is tampered so that it is rejected (it still decodes); the blindings of the 47 others cancel."""
    api = gpu_api
    rng = np.random.default_rng(91)
    K, D, P, t = 48, 50000, 64, 29
    bls = cancelling(api, K - 1, D, 0x90)
    bls.insert(t, api.rnd_scalar_vec(b"\x55" * 32, D))
    vs, msgs = [], []
    for k in range(K):
        v = (rng.integers(-24, 25, D) / 128).astype(np.float32); vs.append(v)
        rc, m = api.enc_l2_compressed_encrypt(v, bls[k], 8, P, 32, 32, FR, bytes([0x30 + k]) * 32)
        assert rc == 0
        msgs.append(m)
    msgs[t]["square_range_proof"] = msgs[t]["square_range_proof"].copy(); msgs[t]["square_range_proof"][33] ^= 2
    ok = api.enc_l2_compressed_verify_batch(msgs, b"\x67" * 32)
    assert ok[t] == 0 and all(ok[k] == 1 for k in range(K) if k != t)
    recs = np.stack([m["enc_values"] for m in msgs])
    keep = [k for k in range(K) if k != t]
    with api.accumulator(D, 96, 1) as acc:
        added = []
        for k0 in range(0, K, 5):                                     # clients arrive a few at a time
            added += acc.add(recs[k0:k0 + 5], ok[k0:k0 + 5]).tolist()
        assert added == [0 if k == t else 1 for k in range(K)] and acc.count == K - 1
        exp = acc.export()
        assert (exp[:, :32] == api.aggregate(np.ascontiguousarray(recs[keep, :, :32]), 1)).all()
        assert (exp[:, 32:] == api.aggregate(np.ascontiguousarray(recs[keep, :, 32:64]), 1)).all()
        rc, s, f = acc.extract(1 << 16, 16, 32, FR)
        assert rc == 0
        assert (f == (np.sum(np.stack([vs[k] for k in keep]), axis=0, dtype=np.float64) + 2.0 ** -FR).astype(np.float32)).all()
        rc_d, s_d, _ = api.dlog(np.ascontiguousarray(exp[:, :32]), 1 << 16, 16, 32, FR)
        assert rc_d == 0 and (s == s_d).all()
        # the rejected client added after all: its blinding no longer cancels
        assert acc.add(recs[t]).tolist() == [1]
        assert acc.extract(1 << 16, 16, 32, FR)[0] == ROFL_ERR_UNBALANCED


@pytest.mark.gpu
def test_gpu_add_dev(gpu_api):
    import torch
    api = gpu_api
    rng = np.random.default_rng(92)
    K, D = 6, 4096
    bls = cancelling(api, K, D, 0xa0)
    recs = np.stack([np.concatenate(api.commit((rng.integers(-50, 50, D) / 128).astype(np.float32), bls[k], NB, FR, want_R=True), axis=1) for k in range(K)])
    mask = np.array([1, 1, 0, 1, 1, 1], np.int32)
    with api.accumulator(D, 64, 1) as a, api.accumulator(D, 64, 1) as b:
        assert a.add(recs, mask).tolist() == mask.tolist()
        t = torch.from_numpy(recs).cuda()
        assert b.add_dev(t.data_ptr(), K, mask).tolist() == mask.tolist()
        torch.cuda.synchronize()
        assert a.count == b.count == 5 and (a.export() == b.export()).all()
        ra, sa, fa = a.extract(1 << 16, 16, NB, FR); rb, sb, fb = b.extract(1 << 16, 16, NB, FR)
        assert ra == rb == ROFL_ERR_UNBALANCED                        # client 2 is missing from a set of cancelling blindings
        assert b.add_dev(t[2].data_ptr(), 1).tolist() == [1] and a.add(recs[2]).tolist() == [1]
        assert (a.export() == b.export()).all()
        ra, sa, fa = a.extract(1 << 16, 16, NB, FR); rb, sb, fb = b.extract(1 << 16, 16, NB, FR)
        assert ra == rb == 0 and (sa == sb).all() and (fa == fb).all()


@pytest.mark.gpu
def test_gpu_large_D(gpu_api):
    api = gpu_api
    rng = np.random.default_rng(93)
    K, D = 4, 1 << 20
    bls = cancelling(api, K, D, 0xb0)
    vs = quantised(rng, K, D, -500, 500)
    recs = np.stack([np.concatenate(api.commit(vs[k], bls[k], NB, FR, want_R=True), axis=1) for k in range(K)])
    with api.accumulator(D, 64, 1) as acc:
        assert acc.add(recs[:1]).tolist() == [1] and acc.add(recs[1:]).tolist() == [1] * 3
        exp = acc.export()
        assert (exp[:, :32] == api.aggregate(np.ascontiguousarray(recs[:, :, :32]), 1)).all()
        assert (exp[:, 32:] == api.aggregate(np.ascontiguousarray(recs[:, :, 32:]), 1)).all()
        rc, s, f = acc.extract(1 << 16, 16, NB, FR)
        rc_d, s_d, f_d = api.dlog(np.ascontiguousarray(exp[:, :32]), 1 << 16, 16, NB, FR)
        assert rc == rc_d == 0 and (s == s_d).all() and (f == f_d).all()
        assert (f == (np.sum(np.stack(vs), axis=0, dtype=np.float64) + 2.0 ** -FR).astype(np.float32)).all()


@pytest.mark.gpu
def test_gpu_params_accumulator(gpu_api):
    """params.EncModelParamsAccumulator over EncRangeCompressed messages (fixed point 16/7), as the server uses it"""
    import __graft_entry__ as g
    params = g.load_package().params
    rng = np.random.default_rng(94)
    K, D = 3, 1000
    bls = cancelling(gpu_api, K, D, 0xc0)
    vs = quantised(rng, K, D)
    acc = params.EncModelParamsAccumulator.unity(D, "RangeCompressed")
    for k in range(K):
        acc.accumulate_other(params.EncParamsRangeCompressed.encrypt(vs[k], bls[k], 8, 4, bytes([0xd0 + k]) * 32))
    assert acc.count == K
    assert (acc.extract() == (np.sum(np.stack(vs), axis=0, dtype=np.float64) + 2.0 ** -FR).astype(np.float32)).all()
    acc.close()
    with pytest.raises(ValueError):
        params.EncModelParamsAccumulator.unity(D, "Plain")
