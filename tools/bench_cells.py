#!/usr/bin/env python3
"""EIP-7594 cell workloads on one GPU: verify_cell_kzg_proof_batch and compute_cells through the C ABI.

    python tools/bench_cells.py [--steps 10] [--warmup 2] [--out profiles/bench_cells.json]

Workloads (all data from the cell workload generator, kzgb200_harness_generate_cells, valid proofs):
  a  one data column: 21 blobs x 1 cell at the same index, host buffers
  b  128 blobs x 128 cells = 16384 cells, device-resident
  c  512 blobs x 128 cells = 65536 cells, device-resident
  d  mempool: 128 blobs -> compute_cells (device) -> verify their 128 cell proofs each
For each: the call time (host clock around the blocking call), cells/s, and -- on the identical transcript bytes -- the host
SHA-256 time (kzgb200_host_sha256): the exact challenge is one serial hash over 2112 bytes per cell, run by a host thread
beside the GPU's parsing, so a call is bound by whichever of the two is longer; `bound` says which.  Per-phase device times of
one extra profiled call are included.  The single-thread CPU oracle rate at a small n is given for scale, labelled as such.
The GPU name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CELL = 2048


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not available"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not available"
    return info


def transcript(commitments, idx, cells, proofs):
    """the exact challenge input (commitments deduplicated by bytes, first occurrence)"""
    uniq, pos = [], {}
    cidx = []
    for c in commitments:
        if c not in pos:
            pos[c] = len(uniq)
            uniq.append(c)
        cidx.append(pos[c])
    n = len(idx)
    parts = [b"RCKZGCBATCH__V1_", (4096).to_bytes(8, "big"), (64).to_bytes(8, "big"), len(uniq).to_bytes(8, "big"), n.to_bytes(8, "big")] + uniq
    for k in range(n):
        parts += [cidx[k].to_bytes(8, "big"), int(idx[k]).to_bytes(8, "big"), cells[k], proofs[k]]
    return b"".join(parts)


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    ts.sort()
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "steps": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_cells.json"))
    a = ap.parse_args()
    import torch
    import kzg_rs_b200 as K
    from cell_oracle import cells as CO
    assert torch.cuda.is_available(), "bench_cells needs a GPU"
    lib = K.Library.get().dll
    S = K.KzgSettings.load_trusted_setup_file()
    ctx = S.cell_context(0)
    tau = K.api.mainnet_g1_monomial()
    res = {"tool": "tools/bench_cells.py", **gpu_info(), "workloads": {}}

    def gen(nb, seed):
        cells = torch.empty(nb * 128 * CELL, dtype=torch.uint8, device="cuda")
        cs = torch.empty(nb * 48, dtype=torch.uint8, device="cuda")
        ps = torch.empty(nb * 128 * 48, dtype=torch.uint8, device="cuda")
        assert lib.kzgb200_harness_generate_cells(ctx, seed, nb, 192, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
        torch.cuda.synchronize()
        return cells, cs, ps

    def phases():
        lib.kzgb200_set_profiling(ctx, 1)
        yield
        out = (C.c_float * 8)()
        lib.kzgb200_get_phase_ms(ctx, out)
        lib.kzgb200_set_profiling(ctx, 0)
        # the slot layout of a cell verification call (kzgb200.h): slots 1 and 2 are the host hashing's wall ms and thread count
        names = ["parse", "host_hash_wall", "hasher_threads", "weights", "lincomb", "reduce", "final", "fallback"]
        yield {k: round(v, 4) for k, v in zip(names, out) if v}

    def record(name, desc, n, call, host_bytes, extra=None):
        ok = call()
        assert ok == 1, (name, ok)
        t = timed(call, a.steps, a.warmup)
        msg = transcript(*host_bytes)
        h = timed(lambda: K.api.host_sha256(msg), max(3, a.steps // 2), 1)
        g = phases(); next(g); call(); ph = next(g)
        share = h["median_ms"] / t["median_ms"]
        res["workloads"][name] = {
            "what": desc, "cells": n, "call": t, "cells_per_s": n / (t["median_ms"] / 1e3),
            "host_sha256_same_transcript": {**h, "bytes": len(msg), "MB_per_s": len(msg) / (h["median_ms"] / 1e3) / 1e6},
            "hash_share_of_call": share,
            "bound": "host transcript hash (serial SHA-256 over 2112 B per cell)" if share >= 0.5 else "GPU / fixed latency (the hash is the smaller part)",
            "phase_ms_of_one_profiled_call": ph, **(extra or {})}
        print(name, json.dumps(res["workloads"][name]), flush=True)

    def dev_call(d_c, d_idx, d_cells, d_p, n):
        ok = C.c_int(-1)
        rc = lib.kzgb200_verify_cell_kzg_proof_batch_device(ctx, d_c.data_ptr(), d_idx.data_ptr(), d_cells.data_ptr(), d_p.data_ptr(), n, C.byref(ok))
        assert rc == 0, rc
        return ok.value

    def host_split(d_c, d_idx, d_cells, d_p, n):
        hc, hi, hce, hp = (t.cpu().numpy().tobytes() for t in (d_c, d_idx, d_cells, d_p))
        return [hc[48 * k:48 * k + 48] for k in range(n)], [int.from_bytes(hi[8 * k:8 * k + 8], "little") for k in range(n)], \
            [hce[CELL * k:CELL * (k + 1)] for k in range(n)], [hp[48 * k:48 * k + 48] for k in range(n)]

    def full(nb, seed):
        cells, cs, ps = gen(nb, seed)
        d_c = cs.view(nb, 1, 48).expand(nb, 128, 48).contiguous().view(-1)
        d_idx = torch.arange(128, dtype=torch.int64, device="cuda").repeat(nb)
        return cells, d_c, d_idx, ps

    # (a) one data column, host buffers
    nb, col = 21, 37
    cells, cs, ps = gen(nb, 1)
    sel = torch.arange(nb, device="cuda") * 128 + col
    hc = cs.cpu().numpy().tobytes()
    hce = cells.view(-1, CELL)[sel].contiguous().cpu().numpy().tobytes()
    hp = ps.view(-1, 48)[sel].contiguous().cpu().numpy().tobytes()
    idx = (C.c_uint64 * nb)(*([col] * nb))

    def col_call():
        ok = C.c_int(-1)
        assert lib.kzgb200_verify_cell_kzg_proof_batch(ctx, hc, C.cast(idx, C.c_void_p), hce, hp, nb, C.byref(ok)) == 0
        return ok.value
    hb = ([hc[48 * k:48 * k + 48] for k in range(nb)], [col] * nb, [hce[CELL * k:CELL * (k + 1)] for k in range(nb)],
          [hp[48 * k:48 * k + 48] for k in range(nb)])
    record("a_one_column_21_blobs", "21 blobs x 1 cell (index 37), host buffers", nb, col_call, hb)
    # CPU oracle rate at this small n (single thread), for scale only
    CO.verify_cell_kzg_proof_batch(*hb)      # first call derives the oracle's monomial points
    t0 = time.perf_counter()
    assert CO.verify_cell_kzg_proof_batch(*hb) is True
    dt = time.perf_counter() - t0
    res["cpu_oracle_single_thread"] = {"what": "cell_oracle/kzg_cell_oracle.c verify_cell_kzg_proof_batch, one thread, workload a (its setup points derived beforehand)", "cells": nb,
                                       "ms": dt * 1e3, "cells_per_s": nb / dt}
    # (b), (c) device-resident full blobs
    for name, nb in (("b_16384_cells_device", 128), ("c_65536_cells_device", 512)):
        cells, d_c, d_idx, ps = full(nb, nb)
        n = nb * 128
        record(name, "%d blobs x 128 cells, device-resident" % nb, n, lambda: dev_call(d_c, d_idx, cells, ps, n), host_split(d_c, d_idx, cells, ps, n))
        del cells, d_c, d_idx, ps
    # (d) mempool: compute_cells on the blobs, then verify all their cell proofs
    nb = 128
    cells0, d_c, d_idx, ps = full(nb, 7)
    blobs = cells0.view(nb, 128 * CELL)[:, :64 * CELL].contiguous()
    out = torch.empty_like(cells0)
    n = nb * 128

    def mempool():
        assert lib.kzgb200_compute_cells_batch_device(ctx, blobs.data_ptr(), nb, out.data_ptr()) == 0
        return dev_call(d_c, d_idx, out, ps, n)
    cc = timed(lambda: lib.kzgb200_compute_cells_batch_device(ctx, blobs.data_ptr(), nb, out.data_ptr()), a.steps, a.warmup)
    record("d_mempool_128_blobs", "128 blobs -> compute_cells (device) -> verify 16384 cell proofs", n, mempool,
           host_split(d_c, d_idx, cells0, ps, n), {"compute_cells_128_blobs_alone": cc, "blobs_per_s_compute_cells": nb / (cc["median_ms"] / 1e3)})
    assert torch.equal(out, cells0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"out": a.out, **{k: round(v["cells_per_s"]) for k, v in res["workloads"].items()}}))


if __name__ == "__main__":
    main()
