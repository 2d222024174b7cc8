#!/usr/bin/env python3
"""One server round of the un-optimised messages (EncRange and EncL2, params.rs:186-233) on one GPU: 48 clients x 50 000 values in the
configs[4] shape (8-bit range proofs in 64 chunks, l2_range 32, fixed point 32/7, check_percentage = 1).

Times, with a host clock around calls that end in a device synchronise (after one warm-up call of each), as median and spread of --reps
repetitions, the forms alternating within each repetition:
  range_batch_ms / range_one_by_one_ms      rofl_enc_range_verify_batch over the 48 EncRange messages / 48 x rofl_enc_range_verify
  l2_batch_ms / l2_one_by_one_ms            rofl_enc_l2_verify_batch over the 48 EncL2 messages / 48 x rofl_enc_l2_verify
  rand_batch_ms / rand_one_by_one_ms        rofl_rand_verify_batch over the 48 x D rand proofs / 48 x rofl_rand_verify
  srand_batch_ms / srand_one_by_one_ms      rofl_square_rand_verify_batch over the 48 x D square-rand proofs / 48 x rofl_square_rand_verify
and asserts that both forms of each pair give the same verdicts.  Prints one JSON object (and writes it to --out when given)."""
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
    return dict(median=round(statistics.median(xs), 2), min=round(min(xs), 2), max=round(max(xs), 2), n=len(xs))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clients", type=int, default=48)
    ap.add_argument("--D", type=int, default=50000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import __graft_entry__ as g
    api = g.load_package().context(0)
    K, D, P, RB, L2, NB, FR = a.clients, a.D, 64, 8, 32, 32, 7
    rng = np.random.default_rng(1)
    rmsgs, lmsgs = [], []
    for k in range(K):
        v = rng.uniform(-0.05, 0.05, D).astype(np.float32); bl = api.rnd_scalar_vec(bytes([k]) * 32, D)
        rc, m = api.enc_range_encrypt(v, bl, RB, P, 1.0, NB, FR, bytes([0x80 + k]) * 32); assert rc == 0
        rmsgs.append(m)
        rc, m = api.enc_l2_encrypt(v, bl, RB, P, L2, NB, FR, bytes([0xc0 - k]) * 32); assert rc == 0
        lmsgs.append(m)
    seed = b"\x5b" * 32
    rp = np.stack([m["rand_proof"] for m in rmsgs]); pairs = np.stack([m["enc_values"] for m in rmsgs])
    sp = np.stack([m["square_proof"] for m in lmsgs]); coms = np.stack([m["enc_values"] for m in lmsgs])
    forms = {
        "range_batch_ms": lambda: api.enc_range_verify_batch(rmsgs, 1.0, seed).tolist(),
        "range_one_by_one_ms": lambda: [api.enc_range_verify(m, 1.0, seed) for m in rmsgs],
        "l2_batch_ms": lambda: api.enc_l2_verify_batch(lmsgs, seed).tolist(),
        "l2_one_by_one_ms": lambda: [api.enc_l2_verify(m, seed) for m in lmsgs],
        "rand_batch_ms": lambda: api.rand_verify_batch(rp, pairs, seed).tolist(),
        "rand_one_by_one_ms": lambda: [api.rand_verify(rp[k], pairs[k]) for k in range(K)],
        "srand_batch_ms": lambda: api.square_rand_verify_batch(sp, coms, seed).tolist(),
        "srand_one_by_one_ms": lambda: [api.square_rand_verify(sp[k], coms[k]) for k in range(K)],
    }
    verdicts = {n: f() for n, f in forms.items()}                                  # warm-up (generator tables, scratch)
    times = {n: [] for n in forms}
    for _ in range(a.reps):
        for n, f in forms.items():
            t, r = timed(f); times[n].append(t)
            assert r == verdicts[n], n
    for f in ("range", "l2", "rand", "srand"):
        assert verdicts[f + "_batch_ms"] == verdicts[f + "_one_by_one_ms"] == [1] * K, f
    name, power = gpu_info()
    res = dict(workload=f"{K} clients x configs[4]-shaped EncRange and EncL2 messages: D={D}, {RB}-bit range proofs, n_partition={P}, l2_range={L2}, fp {NB}/{FR}, check_percentage=1",
               gpu=name, power_limit=power, host_cpus=os.cpu_count(),
               timing="host clock around calls ending in a device synchronise, after one warm-up call each; the forms alternate within each repetition",
               verdicts_equal=True, all_accepted=True)
    for n in forms:
        res[n] = stats(times[n])
    for f in ("range", "l2", "rand", "srand"):
        res[f + "_speedup"] = round(res[f + "_one_by_one_ms"]["median"] / res[f + "_batch_ms"]["median"], 2)
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
