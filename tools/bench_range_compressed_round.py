#!/usr/bin/env python3
"""One server round of L-inf messages (EncParamsRangeCompressed, params.rs:236-256) on one GPU: 48 clients x BASELINE.json configs[1]
(62 006 values, 16-bit range proofs in 64 chunks, fixed point 16/7, check_percentage = 1).

Times, with a host clock around calls that end in a device synchronise (after one warm-up call of each), as median and spread of --reps
repetitions, the two forms alternating within each repetition:
  verify_batch_ms       rofl_enc_range_compressed_verify_batch over the 48 messages
  verify_one_by_one_ms  48 x rofl_enc_range_compressed_verify
  crp_batch_ms          rofl_crp_verify_batch over the 48 compressed rand proofs
  crp_one_by_one_ms     48 x rofl_crp_verify
  range_batch_ms        rofl_range_verify_batch over the same range proofs and L halves (the part of the message batch that runs on the
                        calling thread while the 48 rand-proof transcripts run on host threads)
and asserts that both forms give the same verdicts.  Prints one JSON object (and writes it to --out when given)."""
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
    ap.add_argument("--D", type=int, default=62006)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import __graft_entry__ as g
    api = g.load_package().context(0)
    K, D, P, RB, NB, FR = a.clients, a.D, 64, 16, 16, 7
    rng = np.random.default_rng(1)
    msgs = []
    for k in range(K):
        v = rng.uniform(-0.99, 0.99, D).astype(np.float32); bl = api.rnd_scalar_vec(bytes([k]) * 32, D)
        rc, m = api.enc_range_compressed_encrypt(v, bl, RB, P, NB, FR, bytes([0x80 + k]) * 32)
        assert rc == 0
        msgs.append(m)
    seed = b"\x5a" * 32
    proofs = np.stack([m["rand_proof"] for m in msgs]); pairs = np.stack([m["enc_values"] for m in msgs])
    rproofs = np.stack([m["range_proof"] for m in msgs]); commits = np.ascontiguousarray(pairs[:, :, :32])
    forms = {
        "verify_batch_ms": lambda: api.enc_range_compressed_verify_batch(msgs, 1.0, seed).tolist(),
        "verify_one_by_one_ms": lambda: [api.enc_range_compressed_verify(m, 1.0, seed) for m in msgs],
        "crp_batch_ms": lambda: api.crp_verify_batch(proofs, pairs, seed).tolist(),
        "crp_one_by_one_ms": lambda: [api.crp_verify(proofs[k], pairs[k]) for k in range(K)],
        "range_batch_ms": lambda: api.range_verify_batch(rproofs, commits, RB, seed).tolist(),
    }
    verdicts = {n: f() for n, f in forms.items()}                                  # warm-up (generator tables, scratch)
    times = {n: [] for n in forms}
    for _ in range(a.reps):
        for n, f in forms.items():
            t, r = timed(f); times[n].append(t)
            assert r == verdicts[n], n
    assert verdicts["verify_batch_ms"] == verdicts["verify_one_by_one_ms"] == [1] * K
    assert verdicts["crp_batch_ms"] == verdicts["crp_one_by_one_ms"] == [1] * K
    name, power = gpu_info()
    res = dict(workload=f"{K} clients x configs[1] EncRangeCompressed messages: D={D}, {RB}-bit range proofs, n_partition={P}, fp {NB}/{FR}, check_percentage=1",
               gpu=name, power_limit=power, host_threads=os.cpu_count() and min(os.cpu_count(), 32), host_cpus=os.cpu_count(),
               timing="host clock around calls ending in a device synchronise, after one warm-up call each; the forms alternate within each repetition",
               verdicts_equal=True, all_accepted=True)
    for n in forms:
        res[n] = stats(times[n])
    res["verify_speedup"] = round(res["verify_one_by_one_ms"]["median"] / res["verify_batch_ms"]["median"], 2)
    res["crp_speedup"] = round(res["crp_one_by_one_ms"]["median"] / res["crp_batch_ms"]["median"], 2)
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
