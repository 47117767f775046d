#!/usr/bin/env python3
"""EIP-7594 cell proofs and recovery on one GPU: compute_cells_and_kzg_proofs (FK20) and recover_cells_and_kzg_proofs.

    python tools/bench_cell_proofs.py [--steps 10] [--warmup 2] [--out profiles/bench_cell_proofs.json]

Workloads (blobs from the cell workload generator, kzgb200_harness_generate_cells: degree-192 polynomials whose 128 cells and proofs
the generator computes independently; every timed call's output is compared with them byte for byte):
  a  compute_cells_and_kzg_proofs of one host blob (latency)
  b  the device batch call at 128 and at 1024 blobs (blobs/s)
  c  recovery of a block of 48 device blobs from a random 64 columns (one shared index set)
  d  recovery of one host blob from a random 64 cells
Times are CUDA events on the library's stream around each blocking call, after warm-up.  Also: the one-time proof setup (host clock
around kzgb200_load_cell_proof_setup, which ends in a synchronise) and the device memory it takes, per-phase device times of one
extra profiled call, and the repository's CPU test oracle (direct division, single-threaded C; not an optimised library) for scale.
The GPU name and power limit are read in the same run.
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


def timed(stream, fn, check, steps, warmup):
    """CUDA events on the library's stream around each call; fn returns the C return code; check() validates the last output"""
    import torch
    for _ in range(warmup):
        assert fn() == 0
    ts = []
    with torch.cuda.stream(stream):
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            assert fn() == 0
            e1.record(stream)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
    assert check(), "output differs from the generator's"
    ts.sort()
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "steps": steps, "outputs_checked": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_cell_proofs.json"))
    a = ap.parse_args()
    import torch
    import kzg_rs_b200 as K
    from cell_oracle import cells as CO
    assert torch.cuda.is_available(), "bench_cell_proofs needs a GPU"
    lib = K.Library.get().dll
    S = K.KzgSettings.load_trusted_setup_file()
    ctx = S.cell_context(0)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    t0 = time.perf_counter()
    assert lib.kzgb200_load_cell_proof_setup(ctx, S.g1_lagrange_bytes, 4096) == 0
    setup_s = time.perf_counter() - t0
    free1 = torch.cuda.mem_get_info(0)[0]
    S._proofs.add(0)
    stream = torch.cuda.ExternalStream(lib.kzgb200_stream(ctx))
    res = {"tool": "tools/bench_cell_proofs.py", **gpu_info(),
           "setup": {"load_cell_proof_setup_s": round(setup_s, 3), "device_memory_gb": round((free0 - free1) / 1e9, 3)}}

    nmax = 1024
    tau = K.api.mainnet_g1_monomial()
    g_cells = torch.empty(nmax * 128 * CELL, dtype=torch.uint8, device="cuda")
    g_cs = torch.empty(nmax * 48, dtype=torch.uint8, device="cuda")
    g_ps = torch.empty(nmax * 128 * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_harness_generate_cells(ctx, 0xbe7c, nmax, 192, tau, g_cells.data_ptr(), g_cs.data_ptr(), g_ps.data_ptr()) == 0
    torch.cuda.synchronize()
    blobs = g_cells.view(nmax, 128 * CELL)[:, :64 * CELL].contiguous()
    out_c = torch.empty_like(g_cells)
    out_p = torch.empty_like(g_ps)

    # (a) one host blob
    hblob = blobs[0].cpu().numpy().tobytes()
    hc, hp = C.create_string_buffer(128 * CELL), C.create_string_buffer(128 * 48)
    ref_c, ref_p = g_cells[:128 * CELL].cpu().numpy().tobytes(), g_ps[:128 * 48].cpu().numpy().tobytes()
    res["a_single_host_blob"] = timed(stream, lambda: lib.kzgb200_compute_cells_and_kzg_proofs(ctx, hblob, hc, hp),
                                      lambda: hc.raw == ref_c and hp.raw == ref_p, a.steps, a.warmup)

    # (b) device batches
    for n in (128, 1024):
        r = timed(stream, lambda: lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, blobs.data_ptr(), n, out_c.data_ptr(), out_p.data_ptr()),
                  lambda: torch.equal(out_c[:n * 128 * CELL], g_cells[:n * 128 * CELL]) and torch.equal(out_p[:n * 128 * 48], g_ps[:n * 128 * 48]),
                  a.steps, a.warmup)
        r["blobs_per_s"] = round(n / (r["median_ms"] / 1e3), 1)
        r["cell_proofs_per_s"] = round(128 * n / (r["median_ms"] / 1e3), 1)
        res["b_batch_device_%d" % n] = r

    # (c) a block of 48 blobs from a random 64 columns
    nb = 48
    cols = sorted(random.Random(64).sample(range(128), 64))
    ia = (C.c_uint64 * 64)(*cols)
    given = g_cells[:nb * 128 * CELL].view(nb, 128, CELL)[:, torch.tensor(cols, device="cuda")].contiguous()
    r = timed(stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, 64, given.data_ptr(), nb, out_c.data_ptr(), out_p.data_ptr()),
              lambda: torch.equal(out_c[:nb * 128 * CELL], g_cells[:nb * 128 * CELL]) and torch.equal(out_p[:nb * 128 * 48], g_ps[:nb * 128 * 48]),
              a.steps, a.warmup)
    r["blobs_per_s"] = round(nb / (r["median_ms"] / 1e3), 1)
    r["columns"] = cols
    res["c_recover_block_48_device"] = r

    # (d) one host blob from a random 64 cells
    hgiven = b"".join(ref_c[CELL * k:CELL * (k + 1)] for k in cols)
    res["d_recover_single_host"] = timed(stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs(ctx, ia, hgiven, 64, hc, hp),
                                         lambda: hc.raw == ref_c and hp.raw == ref_p, a.steps, a.warmup)

    # per-phase device times of one profiled call each (profiling adds events; these are not the timed numbers above)
    names = ["coefficients", "fixed_base_products", "g1_transforms", "recovery_transforms"]
    phases = {}
    ms = (C.c_float * 8)()
    lib.kzgb200_set_profiling(ctx, 1)
    for label, fn in (("batch_device_128", lambda: lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, blobs.data_ptr(), 128, out_c.data_ptr(), out_p.data_ptr())),
                      ("recover_block_48", lambda: lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, 64, given.data_ptr(), nb, out_c.data_ptr(), out_p.data_ptr())),
                      ("single_host_blob", lambda: lib.kzgb200_compute_cells_and_kzg_proofs(ctx, hblob, hc, hp))):
        assert fn() == 0
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
        phases[label] = {names[i]: round(ms[i], 3) for i in range(4)}
    lib.kzgb200_set_profiling(ctx, 0)
    res["phases_ms"] = phases

    # the CPU test oracle, for scale
    t0 = time.perf_counter()
    assert CO.compute_cell_kzg_proof(hblob, 5) == ref_p[48 * 5:48 * 6]
    one = time.perf_counter() - t0
    t0 = time.perf_counter()
    assert CO.recover_cells(cols, [ref_c[CELL * k:CELL * (k + 1)] for k in cols]) == [ref_c[CELL * k:CELL * (k + 1)] for k in range(128)]
    rec = time.perf_counter() - t0
    res["cpu_test_oracle"] = {"note": "cell_oracle/kzg_cell_oracle.c, a test oracle (direct division and a 4096-point MSM per proof), not an optimised library",
                              "one_cell_proof_s": round(one, 3), "128_cell_proofs_s_extrapolated": round(128 * one, 1),
                              "recover_cells_s": round(rec, 3)}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
