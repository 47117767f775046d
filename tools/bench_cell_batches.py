#!/usr/bin/env python3
"""Many cell batches in one call (verify_cell_kzg_proof_batch_many) against the same batches as sequential single calls.

    python tools/bench_cell_batches.py [--steps 7] [--warmup 2] [--out profiles/bench_cell_batches.json]

Workloads (data from the cell workload generator, kzgb200_harness_generate_cells; a data column sidecar = cell i of every blob):
  a  the 128 sidecars of a 21-blob block, host buffers: one _many call vs 128 verify_cell_kzg_proof_batch calls on the same bytes
  b  the 128 sidecars of a 48-blob block (6144 cells), device buffers: _many_device vs 128 _device calls
  c  workload a with 1 and with 64 tampered sidecars (proof + G): the cost of the per-group fallback
  d  8 custody columns of a 48-blob block, host buffers: one _many call vs 8 single calls
Each timed call is bracketed by CUDA events on the library's stream (the calls block, so the events span the whole call); median of
--steps calls after --warmup calls.  Every timed call's verdicts are compared with the expected ones.  Reported per workload: time
per call, sidecars/s, cells/s, the host hashing time and hasher thread count of the _many call, and the per-phase device times of
one extra call with profiling on.  The GPU name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CELL = 2048
PHASES = ["parse", "host_hash_wall", "hasher_threads", "weights", "lincomb", "reduce", "combined_pairing", "fallback"]


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not available"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not available"
    return info


class Bench:
    def __init__(self, K, steps, warmup):
        import torch
        self.torch, self.K = torch, K
        self.lib = K.Library.get().dll
        self.S = K.KzgSettings.load_trusted_setup_file()
        self.ctx = self.S.cell_context(0)
        self.stream = torch.cuda.ExternalStream(self.lib.kzgb200_stream(self.ctx))
        self.steps, self.warmup = steps, warmup

    def timed(self, fn, check):
        torch = self.torch
        for _ in range(self.warmup):
            check(fn())
        ts = []
        for _ in range(self.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            out = fn()
            e1.record(self.stream)
            e1.synchronize()
            check(out)
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "steps": self.steps}

    def block(self, n_blobs, seed):
        torch = self.torch
        tau = self.K.api.mainnet_g1_monomial()[:192 * 48]
        cells = torch.empty(n_blobs * 128 * CELL, dtype=torch.uint8, device="cuda")
        cs = torch.empty(n_blobs * 48, dtype=torch.uint8, device="cuda")
        ps = torch.empty(n_blobs * 128 * 48, dtype=torch.uint8, device="cuda")
        assert self.lib.kzgb200_harness_generate_cells(self.ctx, seed, n_blobs, 192, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
        torch.cuda.synchronize()
        return [t.cpu().numpy().tobytes() for t in (cells, cs, ps)]

    @staticmethod
    def sidecars(blk, n_blobs, columns):
        """host bytes of the given columns, column-major: commitments, indices, cells, proofs, offsets"""
        hc, hcs, hps = blk
        cs, idx, ce, ps, offs = [], [], [], [], [0]
        for i in columns:
            for b in range(n_blobs):
                cs.append(hcs[48 * b:48 * b + 48])
                idx.append(i)
                ce.append(hc[CELL * (128 * b + i):CELL * (128 * b + i + 1)])
                ps.append(hps[48 * (128 * b + i):48 * (128 * b + i + 1)])
            offs.append(offs[-1] + n_blobs)
        return cs, idx, ce, ps, offs

    def host_many(self, cs, idx, ce, ps, offs):
        k, n = len(offs) - 1, offs[-1]
        bc, bce, bps = b"".join(cs), b"".join(ce), b"".join(ps)
        ia = (C.c_uint64 * n)(*idx)
        off = (C.c_uint64 * (k + 1))(*offs)
        out = C.create_string_buffer(k)

        def run():
            assert self.lib.kzgb200_verify_cell_kzg_proof_batch_many(self.ctx, bc, C.cast(ia, C.c_void_p), bce, bps, C.cast(off, C.c_void_p), k, out) == 0
            return list(out.raw[:k])
        return run

    def host_loop(self, cs, idx, ce, ps, offs):
        calls = []
        for g in range(len(offs) - 1):
            lo, hi = offs[g], offs[g + 1]
            calls.append((b"".join(cs[lo:hi]), (C.c_uint64 * (hi - lo))(*idx[lo:hi]), b"".join(ce[lo:hi]), b"".join(ps[lo:hi]), hi - lo))

        def run():
            res = []
            for bc, ia, bce, bps, n in calls:
                ok = C.c_int(-1)
                rc = self.lib.kzgb200_verify_cell_kzg_proof_batch(self.ctx, bc, C.cast(ia, C.c_void_p), bce, bps, n, C.byref(ok))
                res.append(2 if rc == 1 else ok.value)
            return res
        return run

    def device_forms(self, cs, idx, ce, ps, offs):
        torch = self.torch
        dev = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        d_c, d_ce, d_p = dev(b"".join(cs)), dev(b"".join(ce)), dev(b"".join(ps))
        d_i = torch.tensor(idx, dtype=torch.int64).cuda()
        k = len(offs) - 1
        off = (C.c_uint64 * (k + 1))(*offs)
        out = C.create_string_buffer(k)

        def many():
            assert self.lib.kzgb200_verify_cell_kzg_proof_batch_many_device(self.ctx, d_c.data_ptr(), d_i.data_ptr(), d_ce.data_ptr(), d_p.data_ptr(),
                                                                            C.cast(off, C.c_void_p), k, out) == 0
            return list(out.raw[:k])

        def loop():
            res = []
            for g in range(k):
                lo, n = offs[g], offs[g + 1] - offs[g]
                ok = C.c_int(-1)
                rc = self.lib.kzgb200_verify_cell_kzg_proof_batch_device(self.ctx, d_c.data_ptr() + 48 * lo, d_i.data_ptr() + 8 * lo,
                                                                         d_ce.data_ptr() + CELL * lo, d_p.data_ptr() + 48 * lo, n, C.byref(ok))
                res.append(2 if rc == 1 else ok.value)
            return res
        return many, loop, (d_c, d_i, d_ce, d_p)

    def phases(self, fn):
        ms = (C.c_float * 8)()
        fn()
        self.lib.kzgb200_get_phase_ms(self.ctx, ms)
        host = {"host_hash_ms": round(ms[1], 3), "hasher_threads": int(ms[2])}
        self.lib.kzgb200_set_profiling(self.ctx, 1)
        fn()
        self.lib.kzgb200_get_phase_ms(self.ctx, ms)
        self.lib.kzgb200_set_profiling(self.ctx, 0)
        prof = {PHASES[i]: round(ms[i], 3) for i in range(8) if i not in (1, 2)}
        return host, prof

    def workload(self, name, many, loop, expected, n_cells):
        check = lambda v: self._check(v, expected, name)
        k = len(expected)
        t_many = self.timed(many, check)
        host, prof = self.phases(many)
        out = {"sidecars": k, "cells": n_cells, "many": t_many,
               "many_sidecars_per_s": round(k / t_many["median_ms"] * 1e3, 1),
               "many_cells_per_s": round(n_cells / t_many["median_ms"] * 1e3, 1),
               **host, "many_phase_ms_profiled": prof}
        if loop is not None:
            t_loop = self.timed(loop, check)
            out.update({"sequential_single_calls": t_loop,
                        "sequential_sidecars_per_s": round(k / t_loop["median_ms"] * 1e3, 1),
                        "sequential_cells_per_s": round(n_cells / t_loop["median_ms"] * 1e3, 1),
                        "speedup": round(t_loop["median_ms"] / t_many["median_ms"], 2)})
        print(name, json.dumps(out), flush=True)
        return out

    @staticmethod
    def _check(v, expected, name):
        assert v == expected, "%s: verdicts differ from the expected ones" % name


def tamper(ps, offs, groups):
    from oracle import pyref as R
    ps = list(ps)
    for g in groups:
        j = offs[g]
        ps[j] = R.g1_to_compressed(R.g1_add(R.g1_from_compressed(ps[j])[1], R.G1_GEN))
    return ps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_cell_batches.json"))
    a = ap.parse_args()
    assert a.steps >= 5, "the median of at least 5 calls"
    import torch
    import kzg_rs_b200 as K
    assert torch.cuda.is_available(), "bench_cell_batches needs a GPU"
    B = Bench(K, a.steps, a.warmup)
    res = {"config": {"steps": a.steps, "warmup": a.warmup, "hardware_concurrency": os.cpu_count()}, **gpu_info(), "workloads": {}}
    W = res["workloads"]

    blk21 = B.block(21, 0x7594)
    cs, idx, ce, ps, offs = B.sidecars(blk21, 21, range(128))
    W["a_21_blobs_128_sidecars_host"] = B.workload("a", B.host_many(cs, idx, ce, ps, offs), B.host_loop(cs, idx, ce, ps, offs), [1] * 128, len(idx))

    blk48 = B.block(48, 0x48)
    cs48, idx48, ce48, ps48, offs48 = B.sidecars(blk48, 48, range(128))
    many, loop, keep = B.device_forms(cs48, idx48, ce48, ps48, offs48)
    W["b_48_blobs_128_sidecars_device"] = B.workload("b", many, loop, [1] * 128, len(idx48))
    del keep

    for bad in (1, 64):
        groups = set(range(0, 128, 128 // bad)) if bad > 1 else {57}
        pst = tamper(ps, offs, groups)
        W["c_21_blobs_%d_tampered_sidecars_host" % bad] = B.workload(
            "c%d" % bad, B.host_many(cs, idx, ce, pst, offs), B.host_loop(cs, idx, ce, pst, offs),
            [0 if g in groups else 1 for g in range(128)], len(idx))

    cols = [3, 19, 35, 51, 67, 83, 99, 115]
    csd, idxd, ced, psd, offsd = B.sidecars(blk48, 48, cols)
    W["d_48_blobs_8_custody_columns_host"] = B.workload("d", B.host_many(csd, idxd, ced, psd, offsd), B.host_loop(csd, idxd, ced, psd, offsd),
                                                        [1] * 8, len(idxd))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"gpu": res["gpu"], "power": res["power_limit_and_max_sm_clock"],
                      "a_speedup": W["a_21_blobs_128_sidecars_host"]["speedup"], "b_speedup": W["b_48_blobs_128_sidecars_device"]["speedup"]}))


if __name__ == "__main__":
    main()
