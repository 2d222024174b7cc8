#!/usr/bin/env python3
"""The server's round accumulator on one GPU (rofl_acc_*, EncModelParamsAccumulator params.rs:74-148), in two shapes.

configs4: 48 clients x 50 000 values of EncL2Compressed messages (96-byte records, 8-bit range proofs in 64 chunks, l2_range 32, fixed point
  32/7) with cancelling blindings, verified by rofl_enc_l2_compressed_verify_batch; its out_ok is the mask of every add.  Times, with a host
  clock around calls that end in a device synchronise, after one warm-up round, over --reps rounds (the accumulator reset in between):
    add_host_ms / add_dev_ms     one client per rofl_acc_add (records on the host) / rofl_acc_add_dev (records already in HBM): median over
                                 all adds, and the total of the 48 adds of a round
    extract_ms                   rofl_acc_extract (R == B check fused with BSGS on the resident L, 2^16 table)
    today_*_ms                   the round end without the accumulator: rofl_aggregate of the L and of the R column over all 48 clients
                                 (records on the host), rofl_dlog of the L sum
  and asserts that the decrypted values are the exact sum plus one LSB (the unity start) and that export equals rofl_aggregate.
full_model: D = 11 689 512 with 64-byte records (ElGamal pairs with zero blindings, as the reference's clients send them), added
  --full-per-call clients per rofl_acc_add_dev call; free device memory is read after every call to show that the state stays O(D).
Prints one JSON object (and writes it to --out when given)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return name, power
    except Exception as ex:  # noqa: BLE001
        return f"unknown ({ex})", "unknown"


def timed(f):
    t0 = time.perf_counter(); r = f(); return (time.perf_counter() - t0) * 1e3, r


def stats(xs):
    return dict(median=round(statistics.median(xs), 3), min=round(min(xs), 3), max=round(max(xs), 3), n=len(xs))


def configs4(api, torch, K, D, reps):
    P, RB, L2, NB, FR = 64, 8, 32, 32, 7
    rng = np.random.default_rng(4)
    bls = api.cancelling_blindings(K, D, 0x10)
    vs, msgs = [], []
    for k in range(K):
        v = (rng.integers(-24, 25, D) / 128).astype(np.float32); vs.append(v)
        rc, m = api.enc_l2_compressed_encrypt(v, bls[k], RB, P, L2, NB, FR, bytes([0x50 + k]) * 32); assert rc == 0
        msgs.append(m)
    ok = api.enc_l2_compressed_verify_batch(msgs, b"\x66" * 32)
    assert ok.tolist() == [1] * K
    recs = np.ascontiguousarray(np.stack([m["enc_values"] for m in msgs]))                  # [K, D, 96]
    recs_dev = torch.from_numpy(recs).cuda(); torch.cuda.synchronize()
    Lcol = np.ascontiguousarray(recs[:, :, :32]); Rcol = np.ascontiguousarray(recs[:, :, 32:64])
    want = (np.sum(np.stack(vs), axis=0, dtype=np.float64) + 2.0 ** -FR).astype(np.float32)
    acc = api.accumulator(D, 96, 1)
    t_host, t_dev, tot_host, tot_dev, t_ext, t_aggL, t_aggR, t_dlog = [], [], [], [], [], [], [], []
    for r in range(reps + 1):                                           # round 0 = warm-up (BSGS table, scratch, module load)
        for dev in (False, True):
            acc.reset()
            ts = []
            for k in range(K):
                if dev:
                    t, a = timed(lambda: acc.add_dev(recs_dev[k].data_ptr(), 1, ok[k:k + 1]))
                else:
                    t, a = timed(lambda: acc.add(recs[k], ok[k:k + 1]))
                assert a.tolist() == [1]
                ts.append(t)
            assert acc.count == K
            t, (rc, s, f) = timed(lambda: acc.extract(1 << 16, 16, NB, FR))
            assert rc == 0 and (f == want).all()
            if r:
                (t_dev if dev else t_host).extend(ts); (tot_dev if dev else tot_host).append(sum(ts)); t_ext.append(t)
        t1, aL = timed(lambda: api.aggregate(Lcol, 1))
        t2, aR = timed(lambda: api.aggregate(Rcol, 1))
        t3, (rc, s0, f0) = timed(lambda: api.dlog(aL, 1 << 16, 16, NB, FR))
        assert rc == 0 and (f0 == want).all() and (s0 == s).all()
        if r:
            t_aggL.append(t1); t_aggR.append(t2); t_dlog.append(t3)
    exp = acc.export()
    assert (exp[:, :32] == aL).all() and (exp[:, 32:] == aR).all()
    acc.close()
    return dict(workload=f"{K} clients x EncL2Compressed D={D} (96-byte records), {RB}-bit range proofs, n_partition={P}, l2_range={L2}, fp {NB}/{FR}, cancelling blindings, "
                         "mask = out_ok of rofl_enc_l2_compressed_verify_batch",
                add_host_ms=stats(t_host), add_dev_ms=stats(t_dev), round_adds_host_ms=stats(tot_host), round_adds_dev_ms=stats(tot_dev), extract_ms=stats(t_ext),
                today_aggregate_L_ms=stats(t_aggL), today_aggregate_R_ms=stats(t_aggR), today_dlog_ms=stats(t_dlog),
                decrypted_equals_exact_sum_plus_one_lsb=True, export_equals_rofl_aggregate=True)


def full_model(api, torch, K, D, per_call):
    import ctypes as C
    NB, FR = 16, 7
    rng = np.random.default_rng(5)
    zeros = torch.zeros((D, 32), dtype=torch.uint8, device="cuda")
    recs = torch.empty((K, D, 64), dtype=torch.uint8, device="cuda")
    L = torch.empty((D, 32), dtype=torch.uint8, device="cuda"); R = torch.empty_like(L)
    total = np.zeros(D, np.float64)
    for k in range(K):
        v = (rng.integers(-24, 25, D) / 128).astype(np.float32); total += v
        vd = torch.from_numpy(v).cuda()
        rc = api.lib.rofl_commit_dev(api.h, vd.data_ptr(), zeros.data_ptr(), D, NB, FR, L.data_ptr(), R.data_ptr()); assert rc == 0
        recs[k, :, :32] = L; recs[k, :, 32:] = R
    del L, R, zeros
    torch.cuda.synchronize(); torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    t_create, acc = timed(lambda: api.accumulator(D, 64, 1))
    free1 = torch.cuda.mem_get_info()[0]
    calls, free_after = [], []
    for k0 in range(0, K, per_call):
        n = min(per_call, K - k0)
        t, a = timed(lambda: acc.add_dev(recs[k0].data_ptr(), n))
        assert a.tolist() == [1] * n
        calls.append(t); free_after.append(torch.cuda.mem_get_info()[0])
    t_ext, (rc, s, f) = timed(lambda: acc.extract(1 << 16, 16, NB, FR))
    assert rc == 0 and (f == (total + 2.0 ** -FR).astype(np.float32)).all()
    t_exp, _ = timed(lambda: acc.export())
    acc.close()
    GB = 1e9
    return dict(workload=f"D={D} ElGamal pairs (64-byte records, zero blindings), {K} clients, {per_call} per rofl_acc_add_dev call, fp {NB}/{FR}",
                state_bytes=128 * 2 * D, create_ms=round(t_create, 2), add_call_ms=[round(x, 2) for x in calls], per_client_ms=round(statistics.median(calls) / per_call, 2),
                extract_ms=round(t_ext, 2), export_ms=round(t_exp, 2),
                free_gb_before_create=round(free0 / GB, 3), free_gb_after_create=round(free1 / GB, 3), free_gb_after_each_call=[round(x / GB, 3) for x in free_after],
                decrypted_equals_exact_sum_plus_one_lsb=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clients", type=int, default=48)
    ap.add_argument("--D", type=int, default=50000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--full-D", type=int, default=11689512)
    ap.add_argument("--full-clients", type=int, default=8)
    ap.add_argument("--full-per-call", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as g
    api = g.load_package().context(0)
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, host_cpus=os.cpu_count(),
               timing="host clock around calls that end in a device synchronise (warm); records staged from pageable host memory for rofl_acc_add / rofl_aggregate / rofl_dlog")
    res["configs4"] = configs4(api, torch, a.clients, a.D, a.reps)
    if a.full_D:
        res["full_model"] = full_model(api, torch, a.full_clients, a.full_D, a.full_per_call)
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
