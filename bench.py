#!/usr/bin/env python3
"""bench.py -- range-proved commitment elements/s (prove & verify) on N B200s (BASELINE.json metric).

A step = one pass of the hot path over one synthetic client update of BASELINE.json configs[1] (cifar_lenet5,
D = 62 006 parameters, L-inf 16-bit range proofs, n_partition 64, fp16/frac7): commit + create_rangeproof, then
verify_rangeproof.  elements/s = D / (t_prove + t_verify).
  value : inputs already resident in HBM (rofl_range_prove_dev / rofl_range_verify_dev), CUDA-event timed
  e2e   : the reference-facing host-buffer calls (rofl_range_prove / rofl_range_verify) from pinned host memory,
          host<->device copies inside the timed region
N > 1 (torchrun): one process per GPU, each rank proves and verifies its own client's update (sharding by client, no
data-path collective) -> `value` is weak scaling; in addition the `strong` block times ONE resnet18-full update
(configs[3], 11 689 512 parameters, 64 chunks of 2^18) sharded by chunk over the N ranks (sharding.py: all_gather of proofs
and commitments over NCCL, all_reduce(MIN) of the verdicts -- the gathers are inside its timed region).
At N = 1 the `configs` block adds prove / verify / end-to-end figures for the other BASELINE configs ([0], [2], [3], [4]),
each with its cold (first call: generators and tables are built) and warm times.
--impl reference : the CPU restatement of the reference (oracle/, OpenMP over chunks, all host cores) on a bounded
sample of the same workload; the real Rust reference cannot be built here (no cargo), see DESIGN.md.
--dump-outputs DIR : after the timed steps, the proofs and commitments of the last resident step (proofs.npy, commitments.npy) and
of the last end-to-end step (e2e_proofs.npy, e2e_commitments.npy), bytes as float32.  Inputs and proof seeds depend only on the
arguments, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(workload="cifar_lenet5 update: commit + L-inf range proofs, prove and verify", D=62006, range_bits=16, n_partition=64, n_bits=16, frac=7)
METRIC = "range-proved commitment elements/s (prove & verify)"
IMAD_PER_FIELD_MUL = 72                        # 8 x 8 limb schoolbook (64) + the 2^256 = 38 fold (8): the algorithmic cost of one field multiplication


def bench_config(world):
    """The `config` object of BOTH arms (the driver compares them key by key)."""
    return dict(WORKLOAD, l2_flush="256 MiB device write between timed iterations (GPU arm; the CPU arm's working set exceeds its caches)", parallelism=f"client x{world}",
                generators="warm (cached per device); cold figures in `cold`")


def synth(D, rng_bits, n_bits, frac, seed):
    rng = np.random.default_rng(seed)
    mx = ((1 << (rng_bits - 1)) - 1) / float(1 << frac)
    v = rng.uniform(-mx, mx, D).astype(np.float32)
    return np.clip(v, -mx, mx)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.lines, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.p.stdout], daemon=True); self.t.start()
            t0 = time.time()                     # nvidia-smi's start-up (NVML attach to every GPU of the box) stalls CUDA calls of running
            while not self.lines and time.time() - t0 < 15 and self.p.poll() is None:      # processes: let it finish before any timing
                time.sleep(0.05)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        print("clock samples (sm MHz):", sm, file=sys.stderr)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_run(steps, warmup, sample_chunks=None):
    """CPU restatement of the reference on a bounded sample: `cores` chunks of the real chunk size (1024 values, 16 bit)."""
    import oracle
    oracle.set_num_threads(os.cpu_count() or 1)          # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses all host threads it can
    cores = oracle.num_threads()
    w = WORKLOAD
    Dp = 1 << (w["D"] - 1).bit_length()
    m = Dp // w["n_partition"]
    chunks = sample_chunks or 1 << (max(1, min(cores, w["n_partition"])).bit_length() - 1)      # a power of two (range_proof_vec/mod.rs:25-28), one chunk per thread
    Ds = m * chunks
    if chunks < cores:                                   # one chunk per thread: the threads actually used
        oracle.set_num_threads(chunks); cores = oracle.num_threads()
    v = synth(Ds, w["range_bits"], w["n_bits"], w["frac"], 1)
    bl = oracle.rnd_scalar_vec(b"\x01" * 32, Ds)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        rc, p, c = oracle.range_prove(v, bl, w["range_bits"], chunks, w["n_bits"], w["frac"], bytes([it % 256] * 32))
        t1 = time.perf_counter()
        ok = oracle.range_verify(p, c, w["range_bits"], bytes(32))
        t2 = time.perf_counter()
        assert rc == 0 and ok == 1
        if it >= warmup:
            times.append((t1 - t0, t2 - t1))
    tp = float(np.mean([a for a, _ in times])); tv = float(np.mean([b for _, b in times]))
    return dict(value=Ds / (tp + tv), prove_eps=Ds / tp, verify_eps=Ds / tv, cores=cores, steps=steps, warmup=warmup,
                sample=f"{chunks} chunks x {m} values ({Ds} elements) of the same workload per step, OpenMP over chunks, {steps} timed steps after {warmup} warm-up", ms=(tp + tv) * 1e3,
                outputs=dict(proofs=p, commitments=c))


def dump_outputs(path, arrays):
    """Write what the timed path returned in its last step as <path>/<name>.npy.  The proof and commitment bytes are stored as
    float32 (exact for 0..255), so that two builds of the project can be compared output for output."""
    arrays = {k: np.asarray(a, dtype=np.float32) for k, a in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def wall(f):
    t0 = time.perf_counter(); r = f(); return (time.perf_counter() - t0) * 1e3, r


def extra_configs(api, torch, steps):
    """BASELINE.json configs [3], [0], [2], [4] on one GPU through the host-buffer C ABI (wall clock around the call: copies included).
    cold = first call on this device (Bulletproofs generators derived, radix tables built), warm = median of the following calls."""
    out = {}
    seed = b"\x02" * 32
    rng = np.random.default_rng(123)
    reps = max(2, min(5, steps))

    def warm(f, n=reps):
        ts = [wall(f)[0] for _ in range(n)]
        return float(np.median(ts))

    # ---- configs[3]: resnet18 full, 11 689 512 parameters, 8-bit, 64 chunks of 2^18 values (N = 2^21 bit positions per chunk: no generator tables
    #      at this size -- bucket MSMs and folds).  Run FIRST: its ~45 GB of scratch must not compete with the generator tables of the other configs.
    D = 11689512
    v = rng.uniform(-0.99, 0.99, D).astype(np.float32); bl = api.rnd_scalar_vec(b"\x05" * 32, D)
    cold_ms, (rc, p, c) = wall(lambda: api.range_prove(v, bl, 8, 64, 16, 7, seed)); assert rc == 0
    vcold_ms, ok = wall(lambda: api.range_verify(p, c, 8, seed)); assert ok == 1
    prove_ms = warm(lambda: api.range_prove(v, bl, 8, 64, 16, 7, seed), 1); verify_ms = warm(lambda: api.range_verify(p, c, 8, seed), 2)
    out["configs[3] resnet18 full (11 689 512 params, 8-bit, 64 chunks of 2^18), 1 GPU"] = dict(D=D, prove_ms=prove_ms, verify_ms=verify_ms, cold_prove_ms=cold_ms, cold_verify_ms=vcold_ms,
                                                                                           prove_eps=D / prove_ms * 1e3, verify_eps=D / verify_ms * 1e3, e2e_eps=D / (prove_ms + verify_ms) * 1e3)
    del v, bl, p, c
    api.set_option("trim", 1)
    # ---- configs[0]: mnist_dev_intrinsic_5k, 8-bit, P = 64, fp16/7 (the reference's own CPU-runnable case)
    D = 5000; v = rng.uniform(-0.99, 0.99, D).astype(np.float32); bl = api.rnd_scalar_vec(b"\x01" * 32, D)
    cold_ms, (rc, p, c) = wall(lambda: api.range_prove(v, bl, 8, 64, 16, 7, seed)); assert rc == 0
    prove_ms = warm(lambda: api.range_prove(v, bl, 8, 64, 16, 7, seed)); verify_ms = warm(lambda: api.range_verify(p, c, 8, seed))
    out["configs[0] mnist_dev_intrinsic_5k (8-bit, P=64)"] = dict(D=D, prove_ms=prove_ms, verify_ms=verify_ms, cold_prove_ms=cold_ms, prove_eps=D / prove_ms * 1e3, verify_eps=D / verify_ms * 1e3,
                                                                  e2e_eps=D / (prove_ms + verify_ms) * 1e3)
    # ---- configs[2]: resnet18_intrinsic_50k, whole EncParamsL2Compressed message (8-bit range proofs + 50 000 square proofs + 32-bit sum proof + compressed rand proof)
    D = 50000; v = (rng.integers(-24, 25, D) / 128).astype(np.float32); bl = api.rnd_scalar_vec(b"\x04" * 32, D)
    cold_ms, (rc, m) = wall(lambda: api.enc_l2_compressed_encrypt(v, bl, 8, 64, 32, 32, 7, seed)); assert rc == 0
    prove_ms = warm(lambda: api.enc_l2_compressed_encrypt(v, bl, 8, 64, 32, 32, 7, seed), 3); verify_ms = warm(lambda: api.enc_l2_compressed_verify(m, seed), 3)
    assert api.enc_l2_compressed_verify(m, seed) == 1
    out["configs[2] resnet18_intrinsic_50k (L2: 8-bit range + square proofs + 32-bit sum proof + compressed rand proof; whole message)"] = dict(
        D=D, prove_ms=prove_ms, verify_ms=verify_ms, cold_prove_ms=cold_ms, prove_eps=D / prove_ms * 1e3, verify_eps=D / verify_ms * 1e3, e2e_eps=D / (prove_ms + verify_ms) * 1e3)
    # ---- configs[4]: server side, 48 clients x configs[2]: batch verification of all 48 messages in one call + homomorphic aggregate + bsgs32 decrypt (table 2^16)
    K = 48
    bls = api.cancelling_blindings(K, D)                  # the clients' blindings sum to zero, so the aggregate decrypts (pedersen_ops.rs:110-122)
    msgs, vsum = [], np.zeros(D, np.float64)
    for k in range(K):
        vk = (rng.integers(-24, 25, D) / 128).astype(np.float32); vsum += vk
        rc, mk = api.enc_l2_compressed_encrypt(vk, bls[k], 8, 64, 32, 32, 7, bytes([k + 1]) * 32); assert rc == 0
        msgs.append(mk)
    ok = api.enc_l2_compressed_verify_batch(msgs, seed); assert (ok == 1).all()
    batch_ms = warm(lambda: api.enc_l2_compressed_verify_batch(msgs, seed), 2)
    one_by_one_ms = wall(lambda: [api.enc_l2_compressed_verify(x, seed) for x in msgs])[0]
    Ls = np.stack([x["enc_values"][:, :32].copy() for x in msgs])
    agg_ms = warm(lambda: api.aggregate(Ls, 1), 3); agg = api.aggregate(Ls, 0)
    dlog_ms = warm(lambda: api.dlog(agg, 1 << 16, 16, 32, 7), 3)
    rc, _, dec = api.dlog(agg, 1 << 16, 16, 32, 7); assert rc == 0 and (dec == vsum.astype(np.float32)).all()      # the decrypted aggregate is the exact sum
    out["configs[4] server: 48 clients x resnet18_intrinsic_50k -- batch verify + aggregate + bsgs32 decrypt"] = dict(
        clients=K, D=D, verify_batch_ms=batch_ms, verify_one_by_one_ms=one_by_one_ms, aggregate_ms=agg_ms, dlog_ms=dlog_ms, round_ms=batch_ms + agg_ms + dlog_ms,
        verified_eps=K * D / batch_ms * 1e3, round_eps=K * D / (batch_ms + agg_ms + dlog_ms) * 1e3)
    del msgs, Ls
    api.set_option("trim", 1)
    # ---- several callers of ONE context (rofl_service proves / verifies several clients per process: bin/basic_client.rs:136-161, server.rs:516-522): every
    #      caller runs on its own lane of streams, the tables are shared; one chunk group per call, the callers overlap each other's Fiat-Shamir chains
    import threading
    w = WORKLOAD; K, R = 3, 4
    def caller(k, res):
        vv = np.random.default_rng(500 + k).uniform(-255.9, 255.9, w["D"]).astype(np.float32); bb = api.rnd_scalar_vec(bytes([40 + k]) * 32, w["D"])
        for it in range(R):
            rc, pp, cc = api.range_prove(vv, bb, w["range_bits"], w["n_partition"], w["n_bits"], w["frac"], bytes([it + 1]) * 32)
            res[k] = rc == 0 and api.range_verify(pp, cc, w["range_bits"], seed) == 1
    res = {}; caller(0, res)                                      # warm-up (generator tables of configs[1] are rebuilt after configs[3] evicted them)
    api.set_option("groups", 1)
    for rep in range(2):                                          # the first pass lets every lane allocate its scratch blocks
        ths = [threading.Thread(target=caller, args=(k, res)) for k in range(K)]
        t0 = time.perf_counter()
        for t in ths: t.start()
        for t in ths: t.join()
        dt = time.perf_counter() - t0
    api.set_option("groups", int(os.environ.get("BENCH_GROUPS", os.environ.get("ROFL_GROUPS", "3"))))
    assert all(res.get(k) for k in range(K))
    out["configs[1] with %d concurrent callers of one context (one lane of streams each, host buffers, Python threads)" % K] = dict(
        callers=K, D=w["D"], ms_per_prove_verify_per_caller=dt / R * 1e3, e2e_eps=K * R * w["D"] / dt)
    return out


def strong_block(api, pkg, torch, dist, rank, world, local):
    """ONE configs[3] update (resnet18 full) sharded by chunk over the ranks: sharding.prove_range_sharded / verify_range_sharded, NCCL gathers
    inside the timed region, max over ranks."""
    sh = pkg.sharding
    D, rb, P, nb, fr = 11689512, 8, 64, 16, 7
    rng = np.random.default_rng(321)                      # every rank generates the same update and uses its slice
    v = rng.uniform(-0.99, 0.99, D).astype(np.float32); bl = api.rnd_scalar_vec(b"\x05" * 32, D)
    dev = torch.device("cuda", local)
    kw = dict(dist=dist if world > 1 else None, device=dev)
    res = {}
    for tag in ("cold", "warm"):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        rc, p, c = sh.prove_range_sharded(api, v, bl, rb, P, nb, fr, b"\x09" * 32, **kw)
        torch.cuda.synchronize(); t1 = time.perf_counter()
        ok = sh.verify_range_sharded(api, p, c, rb, b"\x0a" * 32, **kw)
        torch.cuda.synchronize(); t2 = time.perf_counter()
        assert rc == 0 and ok == 1
        tt = torch.tensor([t1 - t0, t2 - t1], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        res[tag] = tt.tolist()
    tp, tv = res["warm"]
    out = dict(workload="configs[3] resnet18 full: ONE update of 11 689 512 parameters, 8-bit, 64 chunks of 2^18, sharded by chunk over the ranks", scaling="strong", n_gpus=world, D=D,
               prove_s=tp, verify_s=tv, prove_eps=D / tp, verify_eps=D / tv, e2e_eps=D / (tp + tv), cold_prove_s=res["cold"][0], cold_verify_s=res["cold"][1],
               collectives="all_gather(proof bytes, commitments) + all_reduce(MIN) of the verdicts over NCCL, inside the timed region; host buffers in and out")
    del v, bl, p, c
    api.set_option("trim", 1)
    out["server"] = strong_server(api, pkg, torch, dist, rank, world, local)
    return out


def strong_server(api, pkg, torch, dist, rank, world, local):
    """configs[4] over the ranks: ONE server round of 48 clients x resnet18_intrinsic_50k.  Verification is sharded by CLIENT (every rank checks its
    contiguous share in one batched call, verdicts MIN-reduced), aggregate + bsgs32 decrypt by PARAMETER range (sharding.decrypt_sharded, the f32
    slices all-gathered).  Every rank holds all 48 messages, as a server process per GPU fed by the same gRPC stream would."""
    sh = pkg.sharding
    K, D = 48, 50000
    rng = np.random.default_rng(77)
    bls = api.cancelling_blindings(K, D, 0x60)
    msgs, vsum = [], np.zeros(D, np.float64)
    for k in range(K):
        vk = (rng.integers(-24, 25, D) / 128).astype(np.float32); vsum += vk
        rc, mk = api.enc_l2_compressed_encrypt(vk, bls[k], 8, 64, 32, 32, 7, bytes([k + 1]) * 32); assert rc == 0
        msgs.append(mk)
    Ls = np.stack([x["enc_values"][:, :32].copy() for x in msgs])
    b, e = sh.split_range(K, world)[rank]
    dev = torch.device("cuda", local)
    res = {}
    for tag in ("cold", "warm"):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ok = api.enc_l2_compressed_verify_batch(msgs[b:e], b"\x0b" * 32) if e > b else np.ones(0, np.int32)
        good = torch.tensor([int((ok == 1).all())], device=dev, dtype=torch.int32)
        if world > 1:
            dist.all_reduce(good, op=dist.ReduceOp.MIN)
        torch.cuda.synchronize(); t1 = time.perf_counter()
        rc, f = sh.decrypt_sharded(api, Ls, 0, 1 << 16, 16, 32, 7, dist=dist if world > 1 else None, device=dev)
        torch.cuda.synchronize(); t2 = time.perf_counter()
        assert int(good.item()) == 1 and rc == 0 and (f == vsum.astype(np.float32)).all()
        tt = torch.tensor([t1 - t0, t2 - t1], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        res[tag] = tt.tolist()
    tv, td = res["warm"]
    return dict(workload="configs[4] server round: 48 clients x resnet18_intrinsic_50k, verification sharded by client, aggregate + bsgs32 decrypt by parameter range",
                scaling="strong", n_gpus=world, clients=K, D=D, verify_s=tv, aggregate_decrypt_s=td, round_s=tv + td, verified_eps=K * D / tv, round_eps=K * D / (tv + td),
                collectives="all_reduce(MIN) of the verdicts, all_gather of the decrypted f32 slices over NCCL, inside the timed region")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the `configs` / `strong` blocks (only the contract metric on configs[1])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the proofs and commitments of the last timed step as DIR/<name>.npy (float32; rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    w = WORKLOAD
    # stdout carries exactly ONE JSON line: everything any library prints to fd 1 meanwhile (NCCL's version banner at NCCL_DEBUG=VERSION
    # ignores NCCL_DEBUG_FILE) is sent to stderr, and the line is written to the saved descriptor at the end
    sys.stdout.flush(); json_fd = os.dup(1); os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(args.steps, min(args.warmup, 1))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        line = dict(metric=METRIC, value=r["value"], unit="elements/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=r["ms"], higher_is_better=True,
                    scaling="weak", vs_baseline=None, dtype="u32 limbs (GF(2^255-19), mod l) on CPU u64", data="synthetic", impl="reference", config=bench_config(args.gpus),
                    cpu_baseline=dict(value=r["value"], unit="elements/s", cores=r["cores"], kind="port", sample=r["sample"], prove_eps=r["prove_eps"], verify_eps=r["verify_eps"]),
                    e2e=dict(value=r["value"], unit="elements/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        emit(line); return

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep NCCL's own version / debug lines off stdout: stdout carries the one JSON line
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    pkg = g.load_package()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    api = pkg.context(local)                       # raises without the CUDA library / device: no CPU fallback
    lib = api.lib
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 16)
    host_threads = int(os.environ.get("BENCH_HOST_THREADS", "0")) or max(2, min(32, ncpu // max(1, world)))
    lib.rofl_set_host_threads(api.h, host_threads)  # (only the host absorb of very large chunks still uses host threads)
    stream = torch.cuda.ExternalStream(lib.rofl_ctx_stream(api.h), device=torch.device("cuda", local))
    D, rb, P, nb, fr = w["D"], w["range_bits"], w["n_partition"], w["n_bits"], w["frac"]
    extra = not args.no_extra and not os.environ.get("BENCH_NO_EXTRA")
    configs = strong = None
    if extra and world == 1:
        print("== configs block (BASELINE configs [3], [0], [2], [4])", file=sys.stderr, flush=True)
        configs = extra_configs(api, torch, args.steps)
        for k, r in configs.items():
            print("  ", k, {a: (round(b, 2) if isinstance(b, float) else b) for a, b in r.items()}, file=sys.stderr, flush=True)
    if extra and world > 1:
        print("== strong block (configs[3] sharded over %d ranks)" % world, file=sys.stderr, flush=True)
        strong = strong_block(api, pkg, torch, dist, rank, world, local)
        api.set_option("trim", 1)
        if rank == 0:
            print("  ", strong, file=sys.stderr, flush=True)
    v_h = torch.from_numpy(synth(D, rb, nb, fr, 1000 + rank)).pin_memory()
    bl_h = torch.from_numpy(api.rnd_scalar_vec(bytes([rank + 1] * 32), D)).pin_memory()
    v_d, bl_d = v_h.cuda(), bl_h.cuda()
    commits_d = torch.empty((D, 32), dtype=torch.uint8, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")           # > 126 MB L2
    n_proofs, plen = api.range_proof_shape(D, rb, P)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(it):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        flush.fill_(it & 0xff); torch.cuda.synchronize()
        e0.record(stream)
        rc, proofs = api.range_prove_dev(v_d.data_ptr(), bl_d.data_ptr(), D, rb, P, nb, fr, bytes([it % 251 + 1] * 32), commits_d.data_ptr())
        e1.record(stream)
        ok = api.range_verify_dev(proofs, commits_d.data_ptr(), D, rb, bytes([it % 249 + 2] * 32))
        e2.record(stream); e2.synchronize()
        assert rc == 0 and ok == 1
        return e0.elapsed_time(e1), e1.elapsed_time(e2), proofs

    def step_e2e(it):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        flush.fill_(it & 0xff); torch.cuda.synchronize()
        e0.record(stream)
        rc, proofs, commits = api.range_prove(v_h.numpy(), bl_h.numpy(), rb, P, nb, fr, bytes([it % 251 + 1] * 32))
        e1.record(stream)
        ok = api.range_verify(proofs, commits, rb, bytes([it % 249 + 2] * 32))
        e2.record(stream); e2.synchronize()
        assert rc == 0 and ok == 1
        return e0.elapsed_time(e1), e1.elapsed_time(e2), proofs, commits

    # cold: the very first prove / verify of this shape on the device derives the Bulletproofs generators and builds their radix-2^11 tables
    cold_p, cold_v, _ = step_resident(0)
    cold = dict(first_call_prove_ms=cold_p, first_call_verify_ms=cold_v, note="first call on the device for this (range, chunk size): generator derivation (k_gens_build) + radix tables (k_rt_shifts / k_rt_rows)")
    sampler = ClockSampler(local)
    if not os.environ.get("BENCH_NO_CLOCKS"):          # (diagnostic switch: how much does the sampling itself perturb the steps?)
        sampler.start()      # started BEFORE the warm-up: nvidia-smi's own start-up (NVML init) stalls the driver for a moment
    for it in range(args.warmup):
        step_resident(it); step_e2e(it)
    sampler.lines.clear()                               # keep only the samples taken during the timed regions
    imad_peak = lib.rofl_probe_imad_wide(api.h) if rank == 0 else 0.0       # roofline denominator, measured on this GPU before the timed region
    print("== timed region starts", file=sys.stderr, flush=True)
    # ---- timed: resident (no per-kernel events inside the timed region)
    lib.rofl_prof_enable(0); lib.rofl_prof_reset()
    barrier()
    t_p = t_v = 0.0
    per_step = []
    for it in range(args.steps):
        a, b, proofs = step_resident(100 + it); t_p += a; t_v += b; per_step.append((round(a, 2), round(b, 2)))
    barrier()
    outputs = dict(proofs=proofs, commitments=commits_d.cpu().numpy())      # the last timed step's (the profiling pass reuses commits_d)
    if rank == 0:
        print("resident per-step (prove_ms, verify_ms):", per_step, file=sys.stderr)
    launches = lib.rofl_prof_launches(-1)
    # ---- timed: end to end through the host-buffer API
    barrier()
    e_p = e_v = 0.0
    per_step = []
    for it in range(args.steps):
        a, b, outputs["e2e_proofs"], outputs["e2e_commitments"] = step_e2e(200 + it); e_p += a; e_v += b; per_step.append((round(a, 2), round(b, 2)))
    barrier()
    if rank == 0:
        print("e2e per-step (prove_ms, verify_ms):", per_step, file=sys.stderr)
    clocks = sampler.stop()
    print("== profiling pass", file=sys.stderr, flush=True)
    # ---- per-kernel breakdown: the same K resident steps again with CUDA events around every launch of the main kernel families
    # (separate pass: creating / recording the events costs host time that must not leak into `value`)
    groups = int(os.environ.get("BENCH_GROUPS", os.environ.get("ROFL_GROUPS", "3")))
    api.set_option("groups", 1)             # one chunk group: every kernel is timed ALONE on the GPU (several groups overlap kernels of different rounds)
    step_resident(299); torch.cuda.synchronize()      # untimed: the one-group scratch sizes are new to the block cache
    lib.rofl_prof_enable(1); lib.rofl_prof_reset()
    prof_step_ms = 0.0
    prof_steps = []
    for it in range(args.steps):
        k0 = sum(lib.rofl_prof_ms(i) for i in range(7))
        a, b, _ = step_resident(300 + it); prof_step_ms += a + b
        torch.cuda.synchronize()
        prof_steps.append((round(a + b, 2), round(sum(lib.rofl_prof_ms(i) for i in range(7)) - k0, 2)))
    prof_step_ms /= args.steps
    if rank == 0:      # slow steps with an unchanged kernel sum = the GPU was waiting, not computing more slowly
        print("profiling pass per-step (step_ms, event-timed kernel ms of the instrumented families):", prof_steps, file=sys.stderr)
    torch.cuda.synchronize()
    api.set_option("groups", groups)
    prof = dict(fold_ms=lib.rofl_prof_ms(0), msm_ms=lib.rofl_prof_ms(1), commit_ms=lib.rofl_prof_ms(2), rt_ms=lib.rofl_prof_ms(4), tail_ms=lib.rofl_prof_ms(5), frz_ms=lib.rofl_prof_ms(6),
                rt_launches=lib.rofl_prof_launches(4), rt_madds=lib.rofl_prof_work(4))
    lib.rofl_prof_enable(0)
    if world > 1:      # proof pieces are the only thing that crosses NVLink in the replica mode: gather them (outside the timed kernels)
        pt = torch.from_numpy(proofs).cuda(); out = [torch.empty_like(pt) for _ in range(world)]; dist.all_gather(out, pt)
        tt = torch.tensor([t_p, t_v, e_p, e_v], device="cuda", dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); t_p, t_v, e_p, e_v = tt.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    K = args.steps
    ms_step = (t_p + t_v) / K
    value = world * D / (ms_step / 1e3)
    e2e_val = world * D / ((e_p + e_v) / K / 1e3)
    # ---- roofline of the dominant kernel: k_rt_msm (direct table MSM: S, the unfolded IPP rounds, the verifier's generator part).
    # The path is bound by the IMAD.WIDE.U32 pipe (32 lanes/clk/SM), not by HBM or the tensor cores (DESIGN.md section 5).
    #   achieved = algorithmic multiply-adds / measured kernel time;  algorithmic = mixed additions x 7 field multiplications x 72
    #   IMAD.WIDE.U32 (8x8 schoolbook + 8 for the 2^256 = 38 fold);  peak = IMAD.WIDE issue rate measured now by rofl_probe_imad_wide
    madds = prof["rt_madds"]; rt_ms = prof["rt_ms"]
    achieved = madds * 7 * IMAD_PER_FIELD_MUL / (rt_ms / 1e3) / 1e12 if rt_ms > 0 else None
    peak = imad_peak / 1e12 if imad_peak else None
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic, traffic_src = None, None
    for name in ("r02_rt_msm_traffic.json", "r01_rt_msm_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            tj = json.load(open(tpath)); traffic = tj.get("dram_bytes_per_launch")
            traffic_src = f"profiles/{name} (ncu --set full capture of one launch of the same shape, code at {tj.get('commit', 'round-1 head febbf85')}); not measurable inside a timed run"
            break
    launches_rt = max(1, prof["rt_launches"])
    roofline = dict(bound="int-imad-wide (integer multiply pipe; not hbm / tensor: see DESIGN.md section 5)", kernel="k_rt_msm", achieved=achieved, peak=peak, unit="T IMAD.WIDE.U32/s",
                    frac=(achieved / peak) if (achieved and peak) else None, traffic=traffic, traffic_source=traffic_src,
                    algorithmic=dict(mixed_additions_per_launch=madds / launches_rt, field_muls_per_addition=7, imad_wide_per_field_mul=IMAD_PER_FIELD_MUL, launches_per_step=launches_rt / K,
                                     bytes_per_launch=madds / launches_rt * 96),
                    kernel_ms_per_launch=rt_ms / launches_rt, kernel_ms_per_step=rt_ms / K, kernel_share_of_step=rt_ms / K / prof_step_ms,
                    share_note="share of the one-chunk-group step of the profiling pass (%.1f ms): the timed steps overlap %d chunk groups" % (prof_step_ms, groups),
                    peak_source="rofl_probe_imad_wide: best of two mad.wide.u32 patterns (rotating multiplicands; carry-chained as in the field multiply), all SMs, best of 5, run before the timed region",
                    hbm=dict(achieved_gbs=madds * 96 / (rt_ms / 1e3) / 1e9 if rt_ms > 0 else None, peak_gbs=hbm_peak, note="table gathers: 96 B per mixed addition; MEASURED_PEAKS.json copy bandwidth" if peaks else "fallback 6650 GB/s"),
                    other_kernels_ms_per_step=dict(bucket_msm=prof["msm_ms"] / K, catch_up=prof["fold_ms"] / K, frozen_level=prof["frz_ms"] / K, ipp_tail=prof["tail_ms"] / K, commit=prof["commit_ms"] / K))
    line = dict(metric=METRIC, value=value, unit="elements/s", n_gpus=world, steps=K, warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="u32 (8 saturated 32-bit limbs of GF(2^255-19), IMAD.WIDE.U32 with 64-bit accumulate; scalars mod l)", data="synthetic",
                config=bench_config(world),
                prove_eps=world * D / (t_p / K / 1e3), verify_eps=world * D / (t_v / K / 1e3), prove_ms=t_p / K, verify_ms=t_v / K,
                e2e=dict(value=e2e_val, unit="elements/s", h2d_bytes_per_step=int(v_h.numel() * 4 + bl_h.numel() + D * 32 + n_proofs * plen), d2h_bytes_per_step=int(D * 32 + n_proofs * plen),
                         prove_ms=e_p / K, verify_ms=e_v / K),
                gpu_launches=int(launches), clocks=clocks, roofline=roofline, cold=cold)
    if configs is not None:
        line["configs"] = configs
    if strong is not None:
        line["strong"] = strong
    if not args.no_cpu_baseline:
        try:
            r = cpu_reference_run(3, 1)
            line["cpu_baseline"] = dict(value=r["value"], unit="elements/s", cores=r["cores"], kind="port", sample=r["sample"], prove_eps=r["prove_eps"], verify_eps=r["verify_eps"])
        except Exception as ex:  # noqa: BLE001
            line["cpu_baseline"] = dict(value=None, unit="elements/s", cores=0, kind="port", sample=f"failed: {ex}")
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
