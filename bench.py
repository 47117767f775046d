#!/usr/bin/env python3
"""bench.py -- blobs verified / second through verify_blob_kzg_proof_batch (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--blobs B] [--impl b200|reference] [--config batch|tuples]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step = one blocking verify_blob_kzg_proof_batch over B synthetic blobs per GPU (default 16384 = 2 GiB of blob bytes per
GPU, BASELINE.json configs[3]) in the library's DEFAULT mode: exact transcript, r bit-identical to kzg-rs.  With N ranks the
batch is N*B blobs sharded by contiguous ranges through the library's group API (csrc/group.cu: transcript entries to the
leader's host hash, partial sums stored over NVLink into the leader GPU, one pairing check) -- `value`, "scaling": "weak";
the `strong` record beside it runs BASELINE's fixed 16384 blobs TOTAL split over the N GPUs.  `value` times the step with
inputs resident in HBM; `e2e` times the same call from pinned HOST buffers (host->device copies inside the timed region), with
a pageable-memory leg and the PCIe roofline beside it.  Timing: CUDA events on the library's stream, barrier + synchronize
on both sides, max over ranks.

--impl reference times the reference's CPU algorithm (the C oracle port, kind "port": the Rust crate cannot be built here)
with all host threads on the same number of blobs per step; it does not load libkzgb200.so.
--config tuples: BASELINE configs[4], m independent verify_kzg_proof tuples (checks / second).
--dump-outputs DIR writes what the last timed step returned, as DIR/<name>.npy: the batch path's verdict and every blob's z and y
(32-bit words of each 32-byte big-endian field element, most significant first, as float64), the tuple path's verdict per tuple
(1 true, 0 false, 2 Err).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
Above DUMP_ROWS blobs or tuples a fixed seeded sample of them is written, with their positions in index.npy.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # the tree may be read-only: nothing is written into it
BLOB = 131072
DUMP_ROWS = 1 << 18                      # z and y of 2^18 blobs as float64 words: 32 MB
ALGO_BYTES_PER_BLOB = 131072 + 48 + 48   # SURVEY.md 8(d)
PHASES = ["g1_decompress", "challenge_sha256", "evaluate_barycentric", "transcript_r_exposed", "lincomb_terms", "reduce", "final_pairing",
          "g1_subgroup_deferred"]
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
DTYPE = "u32-limb modular integer (Fr 255-bit / Fp 381-bit) + SHA-256"
METRIC = "blobs verified/sec (verify_blob_kzg_proof_batch)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--blobs", type=int, default=16384, help="blobs per GPU (weak record); the strong record splits this many over all GPUs")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="batch", choices=["batch", "tuples"])
    ap.add_argument("--tuples", type=int, default=1000000, help="--config tuples: number of (C, z, y, proof) tuples")
    ap.add_argument("--cpu-sample", type=int, default=4096, help="blobs in the CPU-baseline sample of the b200 arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (transcript modes, pipeline, pageable leg)")
    ap.add_argument("--inflight", type=int, default=2, help="batches in flight in the streaming front-end measurement")
    ap.add_argument("--lowdegree-blobs", action="store_true",
                    help="blobs = evaluations of random degree<8 polynomials (cheap generator) instead of uniformly random "
                         "blobs committed / proved by the GPU commit/prove path")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    return ap.parse_args()


def field_words(raw):
    """32-byte big-endian field elements -> (n, 8) float64 of their 32-bit words, most significant first (exact)."""
    import numpy as np
    return np.frombuffer(raw, dtype=">u4").reshape(-1, 8).astype(np.float64)


def dump_outputs(path, arrays):
    """Writes every array as path/<name>.npy.  Arrays longer than DUMP_ROWS keep a fixed seeded sample of their rows, the same
    rows for all of them, whose positions go to index.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    n = max(len(a) for a in arrays.values())
    if n > DUMP_ROWS:
        idx = np.sort(np.random.default_rng(0x4B5A47).choice(n, DUMP_ROWS, replace=False))
        arrays = {k: a[idx] if len(a) == n else a for k, a in arrays.items()}
        arrays["index"] = idx.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def all_ranks(dist, t):
    """A CUDA tensor of the same shape on every rank -> all ranks' copies concatenated in rank order."""
    import torch
    if dist is None:
        return t
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return torch.cat(parts)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[1]) for r in self.rows if r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def bind_to_gpu_numa_node(index):
    """Pin this rank's host threads (and hence its first-touch pinned allocations) to the CPUs local to its GPU, so that
    the end-to-end leg's host->device copies do not cross the socket interconnect.  Best effort."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        cpus = open("/sys/bus/pci/devices/%s/local_cpulist" % bus).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return cpus
    except Exception:
        pass
    return None


def workload_config(args, n, world, reference=False):
    cfg = {"workload": "verify_blob_kzg_proof_batch on %d synthetic blobs per GPU (%d total, %.2f GiB of blob bytes per GPU), "
                       "BASELINE.json configs[3]" % (n, n * world, n * BLOB / 2**30),
           "blobs_per_gpu": n, "total_blobs": n * world, "parallelism": "blob-sharded x%d" % world,
           "cache": "inputs (>= 2 GiB per step) are larger than the 126 MB L2",
           "transcript": "exact (library default: r bit-identical to kzg-rs compute_r_powers)"}
    if reference:
        cfg["generator"] = ("64 distinct uniformly random blobs, commitments / proofs by the oracle's commit/prove over the mainnet setup, "
                            "repeated to %d blobs (the verifier does identical work for every blob; no result is cached)" % n)
    else:
        cfg["generator"] = ("uniformly random field elements, commitments/proofs by the GPU commit/prove path over the mainnet setup" if not args.lowdegree_blobs
                            else "harness: random degree<8 polynomials in evaluation form, commitments/proofs over the mainnet setup, seed 0x4B5A47")
    return cfg


def oracle_workload(n, distinct=64):
    """Reference arm's inputs without any GPU code: `distinct` uniformly random blobs with oracle-side commitments / proofs, tiled."""
    import random
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    rnd = random.Random(0x4B5A47)
    distinct = min(distinct, n)
    blobs = [b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096)) for _ in range(distinct)]

    def make(blob):
        c = O.blob_to_kzg_commitment(blob)
        return blob, c, O.compute_blob_kzg_proof(blob, c)
    O.lib()
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:      # ctypes releases the GIL
        uniq = list(ex.map(make, blobs))
    seq = [uniq[i % distinct] for i in range(n)]
    return b"".join(x[0] for x in seq), b"".join(x[1] for x in seq), b"".join(x[2] for x in seq)


def run_reference(args, rank, world):
    """The reference's CPU path (oracle port), all host threads, the same number of blobs per step as the b200 arm."""
    if rank != 0:
        return
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    if args.config == "tuples":
        return run_reference_tuples(args, O, cores)
    n = args.blobs
    blobs, cs, ps = oracle_workload(n)
    times = []
    for i in range(args.warmup + args.steps):
        t = time.perf_counter()
        rc, ok, z, y = O.verify_batch_raw(blobs, cs, ps, n, nthreads=cores)
        dt = time.perf_counter() - t
        assert rc == 0 and ok, "reference arm rejected a valid batch"
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        import numpy as np
        dump_outputs(args.dump_outputs, {"verdict": np.ones(1), "z": field_words(z), "y": field_words(y)})
    ms = 1e3 * sum(times) / len(times)
    val = n / (ms / 1e3)
    sample = "%d blobs per step (the b200 arm's size), %d threads (blob-parallel; the reference itself is single-threaded), SHA-NI=%d" % (
        n, cores, O.lib().kzgo_sha256_uses_shani())
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "blobs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": workload_config(args, n, world, reference=True),
        "cpu_baseline": {"value": val, "unit": "blobs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "blobs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------ config 5: tuples
def make_tuples(m, seed=0x7e57):
    """BASELINE configs[4] / SURVEY 8d: m (C, z, y, pi) tuples without per-tuple MSMs: C = aG + bT, y = a + b z, pi = bG with T = [tau]G1
    (then e(C - yG, G2) = e(pi, [tau - z]G2)); ~1 % negatives (y + 1), ~0.1 % malformed (z >= q).  Built from a pool of 256 distinct
    (a, b) pairs with fresh z per tuple -- points are pooled (host-side scalar multiplications in Python are slow), scalars are not.
    Returns (commitments, zs, ys, proofs, expected verdict bytes)."""
    import random
    from oracle import oracle as O
    from oracle import pyref as R
    rnd = random.Random(seed)
    T = R.g1_from_compressed(O.tau_power_g1(1))[1]
    pool = []
    for _ in range(256):
        a, b = rnd.randrange(Q), rnd.randrange(Q)
        pool.append((a, b, R.g1_to_compressed(R.g1_add(R.g1_mul(R.G1_GEN, a), R.g1_mul(T, b))), R.g1_to_compressed(R.g1_mul(R.G1_GEN, b))))
    cs, zs, ys, ps, want = bytearray(), bytearray(), bytearray(), bytearray(), bytearray()
    for i in range(m):
        a, b, c48, p48 = pool[rnd.randrange(256)]
        z = rnd.randrange(Q)
        y = (a + b * z) % Q
        v = 1
        u = rnd.random()
        if u < 0.01:
            y, v = (y + 1) % Q, 0
        elif u < 0.011:
            z, v = Q + rnd.randrange(1000), 2
        cs += c48; ps += p48
        zs += z.to_bytes(32, "big"); ys += y.to_bytes(32, "big")
        want.append(v)
    return bytes(cs), bytes(zs), bytes(ys), bytes(ps), bytes(want)


def run_reference_tuples(args, O, cores):
    from concurrent.futures import ThreadPoolExecutor
    m = min(args.tuples, 2048 * cores // 16 or 128)
    cs, zs, ys, ps, want = make_tuples(m)

    def one(i):
        r = O.verify_kzg_proof(cs[48 * i:48 * i + 48], zs[32 * i:32 * i + 32], ys[32 * i:32 * i + 32], ps[48 * i:48 * i + 48])
        return 2 if r is None else int(r)
    times = []
    O.lib()
    for it in range(args.warmup + args.steps):
        t = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as ex:
            got = bytes(ex.map(one, range(m)))
        dt = time.perf_counter() - t
        assert got == want
        if it >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        import numpy as np
        dump_outputs(args.dump_outputs, {"verdict": np.frombuffer(got, dtype=np.uint8).astype(np.float32)})
    ms = 1e3 * sum(times) / len(times)
    val = m / (ms / 1e3)
    print(json.dumps({"impl": "reference", "metric": "verify_kzg_proof checks/sec (independent tuples)", "value": val, "unit": "checks/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": DTYPE, "data": "synthetic", "config": {"workload": "BASELINE.json configs[4]: independent verify_kzg_proof tuples", "tuples": m},
                      "cpu_baseline": {"value": val, "unit": "checks/s", "cores": cores, "kind": "port", "sample": "%d tuples per step, %d threads" % (m, cores)},
                      "e2e": {"value": val, "unit": "checks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_tuples(args, rank, world, local_rank):
    """m independent verify_kzg_proof tuples per GPU (pure replicas across ranks: no exchange)."""
    import torch
    import kzg_rs_b200 as K
    from kzg_rs_b200.api import Library
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = Library.get().dll
    S = K.KzgSettings.load_trusted_setup_file()
    ctx = S.context(local_rank)
    m = args.tuples
    cs, zs, ys, ps, want = make_tuples(m, seed=0x7e57 + rank)
    pin = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()
    hc, hz, hy, hp = pin(cs), pin(zs), pin(ys), pin(ps)
    out = torch.empty(m, dtype=torch.uint8).pin_memory()
    stream = torch.cuda.ExternalStream(lib.kzgb200_stream(ctx), device=torch.device("cuda", local_rank))
    lib.kzgb200_set_profiling(ctx, 1)
    sampler = ClockSampler(local_rank)
    sampler.start()

    def step():
        rc = lib.kzgb200_verify_kzg_proof_many(ctx, hc.data_ptr(), hz.data_ptr(), hy.data_ptr(), hp.data_ptr(), m, out.data_ptr())
        assert rc == 0
    for _ in range(max(args.warmup, 3)):
        step()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if dist is not None:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    sampler.stop_flag = True
    sampler.join(timeout=2)
    ok = out.numpy().tobytes() == want
    if args.dump_outputs:
        verdicts = all_ranks(dist, out.cuda()).cpu().numpy()
        if rank == 0:
            dump_outputs(args.dump_outputs, {"verdict": verdicts.astype("float32")})
    kernel_ms = (C.c_float * 8)()
    lib.kzgb200_get_phase_ms(ctx, kernel_ms)
    if rank == 0:
        val = m * world / (ms / 1e3)
        # integer roofline: ~25 k Fp multiplications per check (SURVEY 8d) against the measured Fp multiplication rate of the chip
        fp_mul_peak = 2.9e10
        res = {"metric": "verify_kzg_proof checks/sec (independent tuples)", "value": val, "unit": "checks/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
               "data": "synthetic", "config": {"workload": "BASELINE.json configs[4]: %d independent verify_kzg_proof tuples per GPU (160 B each), host buffers" % m,
                                               "tuples_per_gpu": m, "negatives": "1 % wrong y, 0.1 % non-canonical z"},
               "e2e": {"value": val, "unit": "checks/s", "ms_per_step": ms, "h2d_bytes_per_step": 160 * m * world, "d2h_bytes_per_step": m * world},
               "verdicts_match_construction": ok, "clocks": sampler.summary(),
               "phases_ms_last_chunk": {"g1_parse": kernel_ms[0], "lhs_points": kernel_ms[4], "pairings": kernel_ms[6]},
               "roofline": {"bound": "integer (FMA-heavy pipe)", "achieved": val / world * 25000, "peak": fp_mul_peak, "unit": "Fp mul/s", "frac": val / world * 25000 / fp_mul_peak,
                            "note": "~25 k Fp multiplications per check (SURVEY.md 8d) against the measured 2.9e10 Fp mul/s (profiles/intpipe_r01.txt)"}}
        print(json.dumps(res))
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ the batch path
def make_workload_device(lib, ctx, args, n, rank):
    import torch
    import kzg_rs_b200 as K
    tau = open(os.path.join(os.path.dirname(K.__file__), "data", "tau_powers_g1.bin"), "rb").read()
    blobs = torch.empty(n * BLOB, dtype=torch.uint8, device="cuda")
    cs = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    ps = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    if not getattr(args, "lowdegree_blobs", False):
        S = K.KzgSettings.load_trusted_setup_file()
        assert lib.kzgb200_load_g1_lagrange(ctx, S.g1_lagrange_bytes, 4096) == 0
        g = torch.Generator(device="cuda").manual_seed(0x4B5A47 + rank)
        blobs = torch.randint(0, 256, (n * BLOB,), dtype=torch.uint8, device="cuda", generator=g)
        blobs.view(n * 4096, 32)[:, 0] &= 0x3f          # every element < 2^254 < q
        torch.cuda.synchronize()                         # the library works on its own stream
        assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, blobs.data_ptr(), n, cs.data_ptr()) == 0
        assert lib.kzgb200_compute_blob_kzg_proof_batch(ctx, blobs.data_ptr(), cs.data_ptr(), n, ps.data_ptr()) == 0
        return blobs, cs, ps
    rc = lib.kzgb200_harness_generate(ctx, 0x4B5A47 + rank, n, 8, tau, blobs.data_ptr(), cs.data_ptr(), ps.data_ptr())
    assert rc == 0, "harness failed rc=%d" % rc
    return blobs, cs, ps


def resident_chunks(n, mode):
    """mirror of plan_chunks (csrc/kzgb200.cu) for resident inputs"""
    if n < 2048 or mode == "tree":
        return 1
    if mode == "device":
        return math.ceil(n / (math.ceil(math.ceil(n / 8) / 16) * 16))
    k, lo, quarter = 0, 0, n // 4 // 16 * 16
    while lo < n:
        rem = n - lo
        take = quarter if k < 3 else rem // 2 // 16 * 16
        take = max(take, 256)
        if rem - min(take, rem) < 256:
            take = rem
        k += 1
        lo += take
    return k


def count_launches(n, resident, mode, world=1, leader=True):
    """Kernels of libkzgb200.so launched by one batch on one rank (mirrors launch_phase1 / transcript_enqueue_chunk / launch_lincomb)."""
    if resident:
        chunks = resident_chunks(n, mode)
        head = 1 + chunks                      # one challenge launch, evaluation per chunk
    else:
        chunks = math.ceil(n / (math.ceil(max(1024, math.ceil(n / 64)) / 16) * 16))
        head = 2 * chunks
    transcript = {"exact": 1, "tree": 2 * chunks + 1, "device": 2 * chunks}[mode]
    # msm x6 (scalars, sort, bucket, bucket join, window, combine), final check x2 (G1 prelude + pairing engine), flag merge | the
    # leader of a group also launches wait_flags
    tail = 6 + 2 + 1 if world == 1 else (6 + (4 if leader else 1))
    return 2 + head + (1 if resident else 0) + transcript + tail        # 2 = G1 decompression + subgroup checks; export of z / y on resident calls


def load_profiled_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernels, from the committed ncu capture of this round (profiles/traffic_r02.csv)"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_full_r02_traffic.json")))
    except Exception:
        return {}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.config == "tuples":
        return run_tuples(args, rank, world, local_rank)

    import numpy as np
    import torch
    import kzg_rs_b200 as K
    from kzg_rs_b200.api import Library
    from kzg_rs_b200 import sharded
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    numa_cpus = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))     # barrier / max over ranks only: not on the data path
    lib = Library.get().dll
    S = K.KzgSettings.load_trusted_setup_file()
    n = args.blobs
    plan = sharded.ShardedBatch(lib, S, n, rank, world, local_rank, session=sharded.session_name() + "w")
    ctx = plan.ctx
    d_blobs, d_cs, d_ps = make_workload_device(lib, ctx, args, n, rank)
    # pinned host copies for the end-to-end leg
    h_blobs = torch.empty(n * BLOB, dtype=torch.uint8).pin_memory()
    h_cs = torch.empty(n * 48, dtype=torch.uint8).pin_memory()
    h_ps = torch.empty(n * 48, dtype=torch.uint8).pin_memory()
    h_blobs.copy_(d_blobs); h_cs.copy_(d_cs); h_ps.copy_(d_ps)
    torch.cuda.synchronize()
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.ExternalStream(lib.kzgb200_stream(ctx), device=dev)
    lib.kzgb200_set_profiling(ctx, 1)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, st=stream, cx=ctx):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        phase_acc = [0.0] * 8
        for _ in range(steps):
            fn()
            ph = (C.c_float * 8)()
            lib.kzgb200_get_phase_ms(cx, ph)
            phase_acc = [a + b for a, b in zip(phase_acc, ph)]
        e1.record(st)
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if dist is not None:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, [a / steps for a in phase_acc]

    def must(v, what):
        assert v is True, "valid batch rejected (%s)" % what

    W = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- headline: library default (exact transcript), one blocking call at a time ----------------------------------
    plan.set_transcript_mode(0)
    ms, phases = timed(lambda: must(plan.verify_device(d_blobs, d_cs, d_ps), "resident"), args.steps, W)
    if args.dump_outputs:      # the last step's verdict (must() passed: true) and the z, y it wrote; later calls overwrite them
        z, y = (all_ranks(dist, t).cpu().numpy().tobytes() for t in (plan.z_out, plan.y_out))
        if rank == 0:
            dump_outputs(args.dump_outputs, {"verdict": np.ones(1), "z": field_words(z), "y": field_words(y)})
    ms_e2e, _ = timed(lambda: must(plan.verify_host(h_blobs, h_cs, h_ps), "e2e pinned"), args.steps, W)
    launches = args.steps * (count_launches(n, True, "exact", world, rank == 0) + count_launches(n, False, "exact", world, rank == 0))
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # PCIe roofline of the end-to-end leg: pinned host -> device copy of the same blob buffer, same run
    d_tmp = torch.empty(n * BLOB, dtype=torch.uint8, device=dev)
    best = 0.0
    for _ in range(4):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        d_tmp.copy_(h_blobs, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, n * BLOB / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del d_tmp
    pcie_peak = best

    extras = {}
    if not args.no_extras:
        # pageable caller memory (an ordinary Vec<Blob>): the library's pinned staging ring
        p_blobs = torch.from_numpy(np.empty(n * BLOB, dtype=np.uint8))
        p_blobs.copy_(h_blobs)
        ms_pg, _ = timed(lambda: must(plan.verify_host(p_blobs, h_cs, h_ps), "e2e pageable"), args.steps, 2)
        extras["pageable"] = ms_pg
        del p_blobs
        # the other transcript modes, same workload
        for name, mode in (("tree", 1), ("device", 2)):
            if world > 1 and mode == 2:
                continue
            plan.set_transcript_mode(mode)
            m1, ph1 = timed(lambda: must(plan.verify_device(d_blobs, d_cs, d_ps), name), args.steps, 2)
            m2 = timed(lambda: must(plan.verify_host(h_blobs, h_cs, h_ps), name + " e2e"), args.steps, 2)[0] if mode == 1 else None
            extras[name] = (m1, ph1, m2)
        plan.set_transcript_mode(0)

    # Streaming front-end (kzgb200_pipeline_*, SURVEY 8f-3), single GPU, default transcript: several batches in flight
    pipelined = None
    if world == 1 and not args.no_extras:
        pipe_batches = args.steps
        with K.BatchPipeline(S, depth=args.inflight, device=local_rank) as pipe:
            def run(submit, steps):
                tickets = [submit() for _ in range(steps)]
                for t in tickets:
                    assert pipe.wait(t) is True, "valid batch rejected (pipeline)"

            def timed_pipe(submit):
                run(submit, args.inflight * W)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(submit, pipe_batches)
                torch.cuda.synchronize()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / pipe_batches
            ms_p = timed_pipe(lambda: pipe.submit_device(d_blobs, d_cs, d_ps, n))
            ms_pe = timed_pipe(lambda: pipe.submit(h_blobs, n, h_cs, n, h_ps, n))
        pipelined = {"in_flight": args.inflight, "value": n / (ms_p / 1e3), "ms_per_step": ms_p, "e2e": n / (ms_pe / 1e3), "e2e_ms_per_step": ms_pe,
                     "unit": "blobs/s", "transcript": "exact", "batches": pipe_batches,
                     "note": "kzgb200_pipeline_submit / _wait: every ticket is one verify_blob_kzg_proof_batch call; "
                             "`batches` batches, in_flight at a time, wall time of all of them (ramp-up and drain included) / batches"}

    # ---- strong scaling: BASELINE configs[3] as written -- args.blobs blobs TOTAL split over the ranks ------------------
    strong = None
    if world > 1:
        lo, hi = sharded.shard_ranges(n, world)[rank]
        ns = hi - lo
        plan_s = sharded.ShardedBatch(lib, S, ns, rank, world, local_rank, session=sharded.session_name() + "s", cap=sharded.shard_ranges(n, world)[0][1])
        lib.kzgb200_set_profiling(plan_s.ctx, 1)
        st_s = torch.cuda.ExternalStream(lib.kzgb200_stream(plan_s.ctx), device=dev)
        sb, sc, sp = d_blobs[:ns * BLOB], d_cs[:ns * 48], d_ps[:ns * 48]
        hb, hc, hp = h_blobs[:ns * BLOB], h_cs[:ns * 48], h_ps[:ns * 48]
        ms_s, ph_s = timed(lambda: must(plan_s.verify_device(sb, sc, sp), "strong resident"), args.steps, W, st_s, plan_s.ctx)
        ms_se, _ = timed(lambda: must(plan_s.verify_host(hb, hc, hp), "strong e2e"), args.steps, W, st_s, plan_s.ctx)
        strong = {"scaling": "strong", "total_blobs": n, "blobs_per_gpu": ns, "value": n / (ms_s / 1e3), "ms_per_step": ms_s,
                  "e2e": {"value": n / (ms_se / 1e3), "ms_per_step": ms_se, "h2d_bytes_per_step": n * ALGO_BYTES_PER_BLOB, "d2h_bytes_per_step": n * 64 + 16 * world},
                  "unit": "blobs/s", "phases_ms_rank0": dict(zip(PHASES, ph_s)),
                  "peer_stores": bool(plan_s.group.uses_peer_stores(0)),
                  "note": "BASELINE.json configs[3] as written: %d blobs (2 GiB) in total, sharded over %d GPUs; the per-blob SHA-256 chain "
                          "(2050 dependent compressions, ~2.9 ms) does not shrink with the shard" % (n, world)}
        launches += args.steps * (count_launches(ns, True, "exact", world, rank == 0) + count_launches(ns, False, "exact", world, rank == 0))
        plan_s.close()

    must(plan.verify_device(d_blobs, d_cs, d_ps), "parity run")
    m_par = min(n, args.cpu_sample if world == 1 else 512)
    zy_sample = plan.last_zy_host(m_par) if rank == 0 else None
    r_gpu = C.create_string_buffer(32)
    lib.kzgb200_last_r(ctx, r_gpu)
    # negatives on the same workload (verdict only, untimed)
    neg = plan.check_negatives(d_blobs, d_cs, d_ps)

    total = n * world
    value = total / (ms / 1e3)
    e2e = total / (ms_e2e / 1e3)
    out = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # dominant kernel = the longest KERNEL phase of the blocking call (rank 0's phases at N > 1).  Phase 0 (G1 decompression) runs
        # beside the hash and phase 3 is the host's transcript hash, not a kernel: when it is the longest phase of the step (exact
        # transcript at N = 8: one SHA-256 stream over all ranks' entries) the roofline says so in `step_bound`.
        top = max((1, 2, 4, 5, 6), key=lambda i: phases[i])
        traffic = load_profiled_traffic()
        ach = n * ALGO_BYTES_PER_BLOB / (phases[top] / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": PHASES[top], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic.get(PHASES[top]), "traffic_source": "profiles/ncu_full_r02_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum of this launch on the same workload: profiles/traffic_r02.csv)" if traffic.get(PHASES[top]) else None,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s",
                "note": "the path is integer-pipe / latency bound, not HBM bound; see int_pipe and DESIGN.md section 4"}
        if phases[3] > phases[top]:
            roof["step_bound"] = "host transcript hash (%.2f ms exposed): compute_r_powers is one SHA-256 chain over every rank's entries" % phases[3]
        # algorithmic integer work of the two blob-streaming kernels against the MEASURED pipe peaks (tools/microbench/intpipe.cu,
        # profiles/intpipe_r01.txt): ALU 69.2 thread-ops/clk/SM, carry-chained IMAD.WIDE.X 31.0 /clk/SM, 148 SMs
        clk = 1.965e9
        sha_ops = n * 2050 * 1218.0          # ALU-pipe instructions per 64-byte block (SASS count: 672 SHF + 352 LOP3 + 178 IADD3 + 16 PRMT)
        fr_ops = n * 4095 * 192.0            # IMAD.WIDE.X per fused dual Fr product
        int_pipe = {"challenge_sha256": {"achieved_ops_per_s": sha_ops / (phases[1] / 1e3), "peak_ops_per_s": 69.2 * 148 * clk,
                                         "frac": sha_ops / (phases[1] / 1e3) / (69.2 * 148 * clk), "pipe": "ALU (SHF/LOP3/IADD3)"},
                    "evaluate_barycentric": {"achieved_ops_per_s": fr_ops / (phases[2] / 1e3), "peak_ops_per_s": 31.0 * 148 * clk,
                                             "frac": fr_ops / (phases[2] / 1e3) / (31.0 * 148 * clk), "pipe": "FMA-heavy (IMAD.WIDE.U32.X)"}}
        cfg = workload_config(args, n, world)
        cfg["host_affinity"] = numa_cpus
        e2e_gbs = n * ALGO_BYTES_PER_BLOB / (ms_e2e / 1e3) / 1e9       # per GPU (each rank feeds its own GPU over its own link)
        out = {"metric": METRIC, "value": value, "unit": "blobs/s", "n_gpus": world,
               "steps": args.steps, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": cfg,
               "e2e": {"value": e2e, "unit": "blobs/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": (n * ALGO_BYTES_PER_BLOB + 32) * world,
                       "d2h_bytes_per_step": (n * 64 + 16) * world, "host_memory": "pinned",
                       "roofline": {"bound": "pcie", "achieved": e2e_gbs, "peak": pcie_peak, "unit": "GB/s per GPU", "frac": e2e_gbs / pcie_peak,
                                    "peak_source": "pinned host->device copy of the same 2 GiB buffer, timed in this run (best of 4)"}},
               "gpu_launches": launches, "clocks": sampler.summary(),
               "phases_ms": dict(zip(PHASES, phases)), "roofline": roof, "int_pipe": int_pipe, "negatives": neg,
               "pipelined": pipelined, "strong": strong,
               "group": None if world == 1 else {"peer_stores": bool(plan.group.uses_peer_stores(0)), "exchange": "library group API (csrc/group.cu): "
                                                 "transcript entries -> shared host block -> leader's host hash; partials -> NVLink peer stores into the leader GPU"}}
        if "pageable" in extras:
            out["e2e"]["pageable"] = {"value": total / (extras["pageable"] / 1e3), "ms_per_step": extras["pageable"],
                                      "note": "same call from ordinary (unpinned) host memory: pinned staging ring inside the library"}
        modes = {}
        for name in ("tree", "device"):
            if name in extras:
                m1, ph1, m2 = extras[name]
                modes[name] = {"value": total / (m1 / 1e3), "ms_per_step": m1, "e2e": (total / (m2 / 1e3)) if m2 else None, "phases_ms": dict(zip(PHASES, ph1))}
        if modes:
            out["other_transcript_modes"] = {"note": "tree: opt-in KZGB200_TRANSCRIPT_TREE (r differs from kzg-rs's, verdict / z / y do not); device: "
                                                     "the exact chain on one warp of the GPU (round 1's default)", **modes}
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as O
        cores = os.cpu_count() or 1
        m = m_par
        hb = h_blobs[:m * BLOB].numpy().tobytes(); hc = h_cs[:m * 48].numpy().tobytes(); hp = h_ps[:m * 48].numpy().tobytes()
        t = time.perf_counter()
        rc, ok, z, y = O.verify_batch_raw(hb, hc, hp, m, nthreads=cores)
        dt = time.perf_counter() - t
        assert rc == 0 and ok
        # bit-exactness of z, y on the sample against the oracle
        out["parity_sample"] = {"blobs": m, "z_y_bit_exact": zy_sample == (z, y)}
        if world == 1:
            m1 = min(m, 64)
            t = time.perf_counter()
            O.verify_batch_raw(hb[:m1 * BLOB], hc[:m1 * 48], hp[:m1 * 48], m1, nthreads=1)
            dt1 = time.perf_counter() - t
            out["cpu_baseline"] = {"value": m / dt, "unit": "blobs/s", "cores": cores, "kind": "port",
                                   "sample": "first %d of the %d blobs, %d threads (blob-parallel); single thread on %d blobs: %.1f blobs/s; SHA-NI=%d"
                                             % (m, n, cores, m1, m1 / dt1, O.lib().kzgo_sha256_uses_shani())}
            if m == n:      # the whole batch went through the oracle: r too
                rr, _ = O.compute_r_powers([hc[48 * i:48 * i + 48] for i in range(n)], [z[32 * i:32 * i + 32] for i in range(n)],
                                           [y[32 * i:32 * i + 32] for i in range(n)], [hp[48 * i:48 * i + 48] for i in range(n)])
                out["parity_sample"]["r_bit_exact"] = rr == r_gpu.raw
    if rank == 0:
        print(json.dumps(out))
    plan.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
