#!/usr/bin/env python3
"""compute_commitments_and_cell_proofs on one GPU: a publisher's commitment and 128 cell proofs per blob from one FK20 pass, against
the composition it replaces (blob_to_kzg_commitment on the commit path, then compute_cells_and_kzg_proofs).

    python tools/bench_commit_cell_proofs.py [--steps 7] [--warmup 2] [--parent PATH] [--out profiles/bench_commit_cell_proofs.json]

Workloads, all on random full-degree blobs (every element uniform in [0, 2^254), so canonical; the cell generator's degree-192
blobs would leave FK20's new table entry, the coefficients m >= 4032, unused):
  a  one host blob: the host form without cells, against kzgb200_blob_to_kzg_commitment + kzgb200_compute_cells_and_kzg_proofs
  b  one 6-blob transaction from host memory: the host form without cells, against the same composition blob by blob
  c  128 device blobs: the _device form (with and without cells), against kzgb200_blob_to_kzg_commitment_batch +
     kzgb200_compute_cells_and_kzg_proofs_batch_device
  d  1024 device blobs (two passes of 512), as (c)
  e  with --parent PATH (the parent commit's libkzgb200.so): kzgb200_compute_cells_and_kzg_proofs_batch_device on (c)'s 128 blobs,
     this build against the parent build, same bytes
The calls of a workload alternate call by call in one process.  Device forms: CUDA events on the library's stream around each call;
host forms: a host clock around each blocking call.  Medians of --steps calls after --warmup calls, with [min, max]; every timed
output (warm-up included) is compared byte for byte with the composition's bytes, computed once before.  Also recorded: the device
memory the proof setup holds with and without the commit path's table (cudaMemGetInfo, device-wide), and the host time of
kzgb200_load_g1_lagrange, the setup the composition needs and the new call does not.  The GPU name, power limit and clocks are read
in the same run.
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
BLOB, CELL, PROOF = 131072, 2048, 48
BLOB_CELLS, BLOB_PROOFS = 128 * CELL, 128 * PROOF


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["power_limit_max_sm_clock_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not available"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_max_sm_clock_sm_clock"] = "not available"
    return info


class ParentLib:
    """another build of the library with its own context and proof setup"""

    def __init__(self, path, S):
        import torch
        self.dll = d = C.CDLL(path)
        p, sz = C.c_void_p, C.c_size_t
        d.kzgb200_create.argtypes = [C.POINTER(p), C.c_int, C.c_char_p, sz]
        d.kzgb200_load_cell_setup.argtypes = [p, C.c_char_p, sz, C.c_char_p]
        d.kzgb200_load_cell_proof_setup.argtypes = [p, C.c_char_p, sz]
        d.kzgb200_compute_cells_and_kzg_proofs_batch_device.argtypes = [p, p, sz, p, p]
        d.kzgb200_stream.argtypes = [p]
        d.kzgb200_stream.restype = p
        d.kzgb200_destroy.argtypes = [p]
        self.ctx = p()
        assert d.kzgb200_create(C.byref(self.ctx), 0, S.g2_monomial_bytes[:192], 192) == 0
        g1m = S._monomial_points()
        assert d.kzgb200_load_cell_setup(self.ctx, g1m, len(g1m) // 48, S.g2_monomial_bytes[64 * 96:65 * 96]) == 0
        assert d.kzgb200_load_cell_proof_setup(self.ctx, S.g1_lagrange_bytes, 4096) == 0
        self.stream = torch.cuda.ExternalStream(d.kzgb200_stream(self.ctx))


def stats(ts):
    ts = sorted(ts)
    return {"median_ms": round(ts[len(ts) // 2], 3), "min_ms": round(ts[0], 3), "max_ms": round(ts[-1], 3), "steps": len(ts), "outputs_checked": True}


def alternate(calls, steps, warmup):
    """calls: name -> (stream or None, fn returning the C return code, check of the output).  One call of each per step: with a
    stream, CUDA events on it around the call; without, a host clock around the blocking call.  Every output is checked outside the
    timed window."""
    import torch
    ts = {name: [] for name in calls}
    for step in range(warmup + steps):
        for name, (stream, fn, check) in calls.items():
            if stream is None:
                t0 = time.perf_counter()
                assert fn() == 0, name
                dt = (time.perf_counter() - t0) * 1e3
            else:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                assert fn() == 0, name
                e1.record(stream)
                e1.synchronize()
                dt = e0.elapsed_time(e1)
            assert check(), "%s: output differs from the composition's" % name
            if step >= warmup:
                ts[name].append(dt)
    return {name: stats(t) for name, t in ts.items()}


def gain(res, new, old):
    r = res[new]["median_ms"], res[old]["median_ms"]
    res["%s_vs_%s" % (new, old)] = {"saved_ms": round(r[1] - r[0], 3), "ratio": round(r[0] / r[1], 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--parent", default=None, help="path of the parent commit's libkzgb200.so, for workload (e)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_commit_cell_proofs.json"))
    a = ap.parse_args()
    import torch
    import kzg_rs_b200 as K
    assert torch.cuda.is_available(), "bench_commit_cell_proofs needs a GPU"
    lib = K.Library.get().dll
    res = {"tool": "tools/bench_commit_cell_proofs.py", **gpu_info()}

    # device memory: the proof setup alone, then with the commit path's table; and the host time of that table's setup
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    S = K.KzgSettings.load_trusted_setup_file()
    S.context(0)
    free1 = torch.cuda.mem_get_info(0)[0]
    ctx = S.cell_proof_context(0)
    free2 = torch.cuda.mem_get_info(0)[0]
    t0 = time.perf_counter()
    assert S.commit_context(0).value == ctx.value
    t_lag = time.perf_counter() - t0
    free3 = torch.cuda.mem_get_info(0)[0]
    gb = lambda b: round(b / 1e9, 3)
    res["device_memory_gb"] = {"context": gb(free0 - free1), "cell_proof_context": gb(free1 - free2),
                               "cell_proof_context_plus_commit_context": gb(free1 - free3)}
    res["load_g1_lagrange_host_s"] = round(t_lag, 3)
    stream = torch.cuda.ExternalStream(lib.kzgb200_stream(ctx))

    nmax = 1024
    g = torch.Generator(device="cuda").manual_seed(4844)
    d = torch.randint(0, 256, (nmax * 4096, 32), dtype=torch.uint8, device="cuda", generator=g)
    d[:, 0] &= 0x3f
    d_blobs = d.view(-1).contiguous()
    del d
    # the composition's bytes, once: commitments on the commit path, cells and proofs on the FK20 path
    want_cm = torch.empty(nmax * 48, dtype=torch.uint8, device="cuda")
    want_ce = torch.empty(nmax * BLOB_CELLS, dtype=torch.uint8, device="cuda")
    want_p = torch.empty(nmax * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, d_blobs.data_ptr(), nmax, want_cm.data_ptr()) == 0
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, d_blobs.data_ptr(), nmax, want_ce.data_ptr(), want_p.data_ptr()) == 0
    torch.cuda.synchronize()
    h_blobs = d_blobs[:6 * BLOB].cpu().numpy().tobytes()
    h_cm, h_p = want_cm[:6 * 48].cpu().numpy().tobytes(), want_p[:6 * BLOB_PROOFS].cpu().numpy().tobytes()
    h_ce = want_ce[:6 * BLOB_CELLS].cpu().numpy().tobytes()

    # (a) and (b): host forms
    for label, n in (("a_one_host_blob", 1), ("b_6_blob_transaction_host", 6)):
        cm, pr, st = C.create_string_buffer(48 * n), C.create_string_buffer(BLOB_PROOFS * n), C.create_string_buffer(n)
        ccm, cce, cpr = C.create_string_buffer(48 * n), C.create_string_buffer(BLOB_CELLS * n), C.create_string_buffer(BLOB_PROOFS * n)
        blobs = h_blobs[:n * BLOB]

        def composition(n=n, blobs=blobs, ccm=ccm, cce=cce, cpr=cpr):
            for b in range(n):
                blob = blobs[b * BLOB:(b + 1) * BLOB]
                rc = lib.kzgb200_blob_to_kzg_commitment(ctx, blob, C.byref(ccm, 48 * b)) or \
                    lib.kzgb200_compute_cells_and_kzg_proofs(ctx, blob, C.byref(cce, BLOB_CELLS * b), C.byref(cpr, BLOB_PROOFS * b))
                if rc:
                    return rc
            return 0
        res[label] = alternate({
            "new_host_no_cells": (None, lambda n=n, blobs=blobs, cm=cm, pr=pr, st=st: lib.kzgb200_compute_commitments_and_cell_proofs(
                ctx, blobs, n, cm, pr, None, st),
                lambda n=n, cm=cm, pr=pr, st=st: st.raw == bytes(n) and cm.raw == h_cm[:48 * n] and pr.raw == h_p[:BLOB_PROOFS * n]),
            "composition_host": (None, composition,
                                 lambda n=n, ccm=ccm, cce=cce, cpr=cpr: ccm.raw == h_cm[:48 * n] and cce.raw == h_ce[:BLOB_CELLS * n]
                                 and cpr.raw == h_p[:BLOB_PROOFS * n]),
        }, a.steps, a.warmup)
        gain(res[label], "new_host_no_cells", "composition_host")

    # (c) and (d): device forms.  After each check the outputs are cleared (outside the timed window), so that a call that wrote
    # nothing fails its check.
    out_cm = torch.zeros(nmax * 48, dtype=torch.uint8, device="cuda")
    out_ce = torch.zeros(nmax * BLOB_CELLS, dtype=torch.uint8, device="cuda")
    out_p = torch.zeros(nmax * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    st = C.create_string_buffer(nmax)

    def checked(n, cm, ce, status=False):
        def check():
            ok = torch.equal(out_p[:BLOB_PROOFS * n], want_p[:BLOB_PROOFS * n])
            ok = ok and (not cm or torch.equal(out_cm[:48 * n], want_cm[:48 * n]))
            ok = ok and (not ce or torch.equal(out_ce[:BLOB_CELLS * n], want_ce[:BLOB_CELLS * n]))
            ok = ok and (not status or st.raw[:n] == bytes(n))
            for t in (out_cm, out_ce, out_p):
                t.zero_()
            torch.cuda.synchronize()
            return ok
        return check
    for label, n in (("c_128_device_blobs", 128), ("d_1024_device_blobs", 1024)):
        r = alternate({
            "new_device_with_cells": (stream, lambda n=n: lib.kzgb200_compute_commitments_and_cell_proofs_device(
                ctx, d_blobs.data_ptr(), n, out_cm.data_ptr(), out_p.data_ptr(), out_ce.data_ptr(), st), checked(n, True, True, True)),
            "new_device_no_cells": (stream, lambda n=n: lib.kzgb200_compute_commitments_and_cell_proofs_device(
                ctx, d_blobs.data_ptr(), n, out_cm.data_ptr(), out_p.data_ptr(), None, st), checked(n, True, False, True)),
            "composition_device": (stream, lambda n=n: lib.kzgb200_blob_to_kzg_commitment_batch(ctx, d_blobs.data_ptr(), n, out_cm.data_ptr())
                                   or lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, d_blobs.data_ptr(), n, out_ce.data_ptr(),
                                                                                             out_p.data_ptr()), checked(n, True, True)),
        }, a.steps, a.warmup)
        gain(r, "new_device_with_cells", "composition_device")
        gain(r, "new_device_no_cells", "composition_device")
        r["new_device_with_cells"]["blobs_per_s"] = round(n / (r["new_device_with_cells"]["median_ms"] / 1e3), 1)
        res[label] = r

    # (e) this build's FK20 batch against the parent build's, same bytes
    if a.parent:
        parent = ParentLib(a.parent, S)
        n = 128
        res["e_fk20_batch_128_vs_parent"] = alternate({
            "this_build": (stream, lambda: lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(
                ctx, d_blobs.data_ptr(), n, out_ce.data_ptr(), out_p.data_ptr()), checked(n, False, True)),
            "parent_build": (parent.stream, lambda: parent.dll.kzgb200_compute_cells_and_kzg_proofs_batch_device(
                parent.ctx, d_blobs.data_ptr(), n, out_ce.data_ptr(), out_p.data_ptr()), checked(n, False, True)),
        }, a.steps, a.warmup)
        gain(res["e_fk20_batch_128_vs_parent"], "this_build", "parent_build")
        parent.dll.kzgb200_destroy(parent.ctx)

    # per-phase device times of one profiled call each (profiling adds events; these are not the timed numbers above)
    names = ["coefficients", "fixed_base_products", "g1_transforms_and_commitments"]
    ms = (C.c_float * 8)()
    lib.kzgb200_set_profiling(ctx, 1)
    phases = {}
    for label, n in (("new_device_no_cells_128", 128),):      # one pass: a slot spans first start to last end over all passes
        assert lib.kzgb200_compute_commitments_and_cell_proofs_device(ctx, d_blobs.data_ptr(), n, out_cm.data_ptr(), out_p.data_ptr(), None, st) == 0
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
        phases[label] = {names[i]: round(ms[i], 3) for i in range(3)}
    lib.kzgb200_set_profiling(ctx, 0)
    res["phases_ms"] = phases
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
