#!/usr/bin/env python3
"""EIP-4844 publisher calls on one GPU: blob_to_kzg_commitment, compute_kzg_proof and compute_blob_kzg_proof.

    python tools/bench_prove.py [--steps 5] [--warmup 1] [--lib NAME=PATH ...] [--out profiles/bench_prove.json]

Workloads, for every library given with --lib (default: this tree's kzg_rs_b200/libkzgb200.so), run alternately, one call of each
library per step, so that libraries are compared under the same conditions:
  host    one host blob per call: the commitment, compute_kzg_proof at a z in the evaluation domain and at a z outside it, and
          compute_blob_kzg_proof (host clock around the blocking call)
  device  the device batches at 1, 21, 128, 1024 and 4096 blobs: commitments, blob proofs (at the Fiat-Shamir challenge), kzg
          proofs at caller-given z, a third of them in the domain (CUDA events on the library's stream, kzgb200_stream)
Medians, minima and maxima are over the timed steps, after warm-up.  Every timed output is compared with the repository's CPU oracle
on a sample of entries, and the libraries' outputs with each other in full.  Entry points a library does not export are skipped,
so an older build can be measured beside this one.  The one-time table build (kzgb200_load_g1_lagrange) is timed by a host clock.
Blobs are uniformly random canonical field elements.  The GPU name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
OMEGA = pow(7, (Q - 1) // 4096, Q)
SIZES = (1, 21, 128, 1024, 4096)


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not available"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not available"
    return info


class Lib:
    def __init__(self, name, path, settings):
        import torch
        self.name, self.path = name, path
        self.dll = d = C.CDLL(path)
        p, sz = C.c_void_p, C.c_size_t
        d.kzgb200_create.argtypes = [C.POINTER(p), C.c_int, C.c_char_p, sz]
        d.kzgb200_load_g1_lagrange.argtypes = [p, C.c_char_p, sz]
        d.kzgb200_stream.argtypes = [p]
        d.kzgb200_stream.restype = p
        d.kzgb200_blob_to_kzg_commitment_batch.argtypes = [p, p, sz, p]
        d.kzgb200_compute_blob_kzg_proof_batch.argtypes = [p, p, p, sz, p]
        self.has = {k: hasattr(d, "kzgb200_" + k) for k in ("blob_to_kzg_commitment", "compute_kzg_proof", "compute_blob_kzg_proof",
                                                             "compute_kzg_proof_batch_device")}
        if self.has["blob_to_kzg_commitment"]:
            d.kzgb200_blob_to_kzg_commitment.argtypes = [p, C.c_char_p, p]
        if self.has["compute_kzg_proof"]:
            d.kzgb200_compute_kzg_proof.argtypes = [p, C.c_char_p, C.c_char_p, p, p]
        if self.has["compute_blob_kzg_proof"]:
            d.kzgb200_compute_blob_kzg_proof.argtypes = [p, C.c_char_p, C.c_char_p, p]
        if self.has["compute_kzg_proof_batch_device"]:
            d.kzgb200_compute_kzg_proof_batch_device.argtypes = [p, p, p, sz, p, p]
        self.ctx = p()
        assert d.kzgb200_create(C.byref(self.ctx), 0, settings.g2_monomial_bytes[:192], 192) == 0
        t0 = time.perf_counter()
        assert d.kzgb200_load_g1_lagrange(self.ctx, settings.g1_lagrange_bytes, 4096) == 0
        self.setup_s = time.perf_counter() - t0
        self.stream = torch.cuda.ExternalStream(d.kzgb200_stream(self.ctx))


def stats(ts, n=None):
    ts = sorted(ts)
    r = {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "steps": len(ts)}
    if n:
        r["blobs_per_s"] = n / (r["median_ms"] / 1e3)
    return r


def device_call(lib, fn):
    """CUDA events on the library's stream around one blocking call"""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lib.stream)
    assert fn() == 0
    e1.record(lib.stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


def host_call(fn):
    t0 = time.perf_counter()
    assert fn() == 0
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of a libkzgb200.so to measure (repeatable)")
    ap.add_argument("--sizes", default=",".join(map(str, SIZES)))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_prove.json"))
    a = ap.parse_args()
    import torch
    import kzg_rs_b200 as K
    from oracle import oracle as O
    assert torch.cuda.is_available(), "bench_prove needs a GPU"
    O.build(); O.lib()
    S = K.KzgSettings.load_trusted_setup_file()
    specs = [x.split("=", 1) for x in a.lib] or [["this", K.lib_path()]]
    libs = [Lib(name, path, S) for name, path in specs]
    sizes = [int(x) for x in a.sizes.split(",")]
    res = {"info": gpu_info(), "steps": a.steps, "warmup": a.warmup,
           "libs": {lb.name: {"path": os.path.relpath(lb.path, ROOT), "exports": lb.has, "g1_lagrange_setup_s": lb.setup_s} for lb in libs},
           "host": {}, "device": {}}
    rnd = random.Random(1)

    # ---- host calls: one blob each
    blob = b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))
    z_in, z_out = pow(OMEGA, 1234, Q).to_bytes(32, "big"), rnd.randrange(Q).to_bytes(32, "big")
    want_c = O.blob_to_kzg_commitment(blob)
    out48, y32 = C.create_string_buffer(48), C.create_string_buffer(32)
    host = [("blob_to_kzg_commitment", "blob_to_kzg_commitment", lambda d, ctx: d.kzgb200_blob_to_kzg_commitment(ctx, blob, out48),
             lambda: out48.raw == want_c),
            ("compute_kzg_proof_z_in_domain", "compute_kzg_proof", lambda d, ctx: d.kzgb200_compute_kzg_proof(ctx, blob, z_in, out48, y32),
             lambda: (out48.raw, y32.raw) == O.compute_kzg_proof(blob, z_in)),
            ("compute_kzg_proof_z_outside", "compute_kzg_proof", lambda d, ctx: d.kzgb200_compute_kzg_proof(ctx, blob, z_out, out48, y32),
             lambda: (out48.raw, y32.raw) == O.compute_kzg_proof(blob, z_out)),
            ("compute_blob_kzg_proof", "compute_blob_kzg_proof", lambda d, ctx: d.kzgb200_compute_blob_kzg_proof(ctx, blob, want_c, out48),
             lambda: out48.raw == O.compute_blob_kzg_proof(blob, want_c))]
    for key, sym, fn, check in host:
        run = [lb for lb in libs if lb.has[sym]]
        if not run:
            continue
        ts = {lb.name: [] for lb in run}
        for lb in run:
            for _ in range(a.warmup):
                assert fn(lb.dll, lb.ctx) == 0
        for _ in range(a.steps):
            for lb in run:
                ts[lb.name].append(host_call(lambda: fn(lb.dll, lb.ctx)))
        for lb in run:
            assert fn(lb.dll, lb.ctx) == 0 and check(), (lb.name, key)
            res["host"].setdefault(key, {})[lb.name] = dict(stats(ts[lb.name]), outputs_checked=True)
        print(key, {k: round(v["median_ms"], 3) for k, v in res["host"][key].items()}, flush=True)

    # ---- device batches
    for n in sizes:
        g = torch.Generator(device="cuda").manual_seed(n)
        blobs = torch.randint(0, 256, (n * 131072,), dtype=torch.uint8, device="cuda", generator=g)
        blobs.view(n * 4096, 32)[:, 0] &= 0x3f
        zs = [pow(OMEGA, rnd.randrange(4096), Q) if i % 3 == 0 else rnd.randrange(Q) for i in range(n)]
        d_z = torch.frombuffer(bytearray(b"".join(z.to_bytes(32, "big") for z in zs)), dtype=torch.uint8).cuda()
        outs = {lb.name: {k: torch.empty(n * w, dtype=torch.uint8, device="cuda") for k, w in (("c", 48), ("p", 48), ("kp", 48), ("y", 32))}
                for lb in libs}
        torch.cuda.synchronize()
        kinds = [("blob_to_kzg_commitment_batch", None,
                  lambda lb, o: lb.dll.kzgb200_blob_to_kzg_commitment_batch(lb.ctx, blobs.data_ptr(), n, o["c"].data_ptr())),
                 ("compute_blob_kzg_proof_batch", None,
                  lambda lb, o: lb.dll.kzgb200_compute_blob_kzg_proof_batch(lb.ctx, blobs.data_ptr(), o["c"].data_ptr(), n, o["p"].data_ptr())),
                 ("compute_kzg_proof_batch_device", "compute_kzg_proof_batch_device",
                  lambda lb, o: lb.dll.kzgb200_compute_kzg_proof_batch_device(lb.ctx, blobs.data_ptr(), d_z.data_ptr(), n, o["kp"].data_ptr(),
                                                                              o["y"].data_ptr()))]
        for key, sym, fn in kinds:
            run = [lb for lb in libs if sym is None or lb.has[sym]]
            if not run:
                continue
            ts = {lb.name: [] for lb in run}
            for lb in run:
                for _ in range(a.warmup):
                    assert fn(lb, outs[lb.name]) == 0
            for _ in range(a.steps):
                for lb in run:
                    ts[lb.name].append(device_call(lb, lambda: fn(lb, outs[lb.name])))
            for lb in run:
                res["device"].setdefault(key, {}).setdefault(str(n), {})[lb.name] = dict(stats(ts[lb.name], n), outputs_checked=True)
            print(key, n, {lb.name: round(res["device"][key][str(n)][lb.name]["median_ms"], 3) for lb in run}, flush=True)
        # outputs: sampled entries against the oracle, every entry across libraries
        host_out = {lb.name: {k: t.cpu().numpy().tobytes() for k, t in outs[lb.name].items()} for lb in libs}
        ref = host_out[libs[0].name]
        for i in sorted({0, n // 2, n - 1}):
            b = blobs[131072 * i:131072 * (i + 1)].cpu().numpy().tobytes()
            c = O.blob_to_kzg_commitment(b)
            assert ref["c"][48 * i:48 * i + 48] == c, (n, i)
            assert ref["p"][48 * i:48 * i + 48] == O.compute_blob_kzg_proof(b, c), (n, i)
            kp = [lb for lb in libs if lb.has["compute_kzg_proof_batch_device"]]
            if kp:
                o = host_out[kp[0].name]
                assert (o["kp"][48 * i:48 * i + 48], o["y"][32 * i:32 * i + 32]) == O.compute_kzg_proof(b, zs[i].to_bytes(32, "big")), (n, i)
        for lb in libs[1:]:
            assert host_out[lb.name]["c"] == ref["c"] and host_out[lb.name]["p"] == ref["p"], (lb.name, n)
        res["device"].setdefault("libraries_agree_byte_for_byte", {})[str(n)] = True
        del blobs, outs
        torch.cuda.empty_cache()

    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
