#!/usr/bin/env python3
"""Batch verifier tail: split (per-window Miller loops on [256^w]-scaled G2 lines) against the Horner + one-pairing tail.

    python tools/bench_final_split.py [--sizes 16384,2048,64] [--steps 30] [--warmup 5] [--out profiles/bench_final_split.json]

One process, one GPU, two contexts of this tree's library: one created with KZGB200_FINAL_SPLIT=1 (the default) and one with
KZGB200_FINAL_SPLIT=0.  Both verify the same seeded resident batch (bench.py's generator: uniformly random blobs committed and
proved on the GPU), calls alternating between the two contexts.  Per call: CUDA events on the context's stream around the blocking
kzgb200_verify_blob_kzg_proof_batch_device.  Reported per context and size: median, min and max per call, the per-phase device times
(kzgb200_get_phase_ms, a separate profiled pass) and the final-check clock stamps (kzgb200_debug_final_ticks).  Verdicts, z and y of
the two contexts are compared on every call, and on a batch with two proofs swapped both must say false with the same GT element.
The GPU name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def make_ctx(lib, g2, split):
    os.environ["KZGB200_FINAL_SPLIT"] = "1" if split else "0"
    h = C.c_void_p()
    assert lib.kzgb200_create(C.byref(h), 0, g2, 192) == 0
    return h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="16384,2048,64")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_final_split.json"))
    args = ap.parse_args()
    import torch
    import kzg_rs_b200 as K
    from kzg_rs_b200.api import Library
    import bench
    from tools.bench_prove import gpu_info
    assert torch.cuda.is_available(), "needs a GPU"
    lib = Library.get().dll
    lib.kzgb200_debug_final_ticks.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
    lib.kzgb200_debug_last_gt.argtypes = [C.c_void_p, C.c_char_p]
    S = K.KzgSettings.load_trusted_setup_file()
    g2 = S.g2_monomial_bytes[:192]
    ctxs = {"split": make_ctx(lib, g2, True), "horner": make_ctx(lib, g2, False)}
    os.environ.pop("KZGB200_FINAL_SPLIT")
    sizes = [int(x) for x in args.sizes.split(",")]
    gen = argparse.Namespace(lowdegree_blobs=False)
    blobs, cs, ps = bench.make_workload_device(lib, ctxs["split"], gen, max(sizes), 0)
    out = {"gpu": gpu_info(), "steps": args.steps, "warmup": args.warmup, "sizes": {}}
    n_max = max(sizes)
    zb = {k: torch.empty(n_max * 32, dtype=torch.uint8, device="cuda") for k in ctxs}
    yb = {k: torch.empty(n_max * 32, dtype=torch.uint8, device="cuda") for k in ctxs}
    streams = {k: torch.cuda.ExternalStream(lib.kzgb200_stream(c)) for k, c in ctxs.items()}

    def call(k, n, proofs=ps):
        okv = C.c_int(-1)
        rc = lib.kzgb200_verify_blob_kzg_proof_batch_device(ctxs[k], blobs.data_ptr(), cs.data_ptr(), proofs.data_ptr(), n, C.byref(okv),
                                                            zb[k].data_ptr(), yb[k].data_ptr())
        assert rc == 0, rc
        return okv.value

    for n in sizes:
        rec = {}
        times = {k: [] for k in ctxs}
        for k, c in ctxs.items():
            lib.kzgb200_set_profiling(c, 0)
        for i in range(args.warmup + args.steps):
            for k in (("split", "horner") if i % 2 == 0 else ("horner", "split")):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(streams[k])
                ok = call(k, n)
                e1.record(streams[k])
                e1.synchronize()
                assert ok == 1, (k, n, ok)
                if i >= args.warmup:
                    times[k].append(e0.elapsed_time(e1))
            assert torch.equal(zb["split"][:n * 32], zb["horner"][:n * 32]) and torch.equal(yb["split"][:n * 32], yb["horner"][:n * 32])
        for k, c in ctxs.items():
            lib.kzgb200_set_profiling(c, 1)
            acc = [0.0] * 8
            for _ in range(5):
                call(k, n)
                ph = (C.c_float * 8)()
                lib.kzgb200_get_phase_ms(c, ph)
                acc = [a + b / 5 for a, b in zip(acc, ph)]
            lib.kzgb200_set_profiling(c, 0)
            tk = (C.c_longlong * 14)()
            lib.kzgb200_debug_final_ticks(c, tk)
            t = list(tk)
            rec[k] = {"ms_per_call_median": statistics.median(times[k]), "ms_per_call_min": min(times[k]), "ms_per_call_max": max(times[k]),
                      "phase_ms": dict(zip(bench.PHASES, [round(x, 4) for x in acc])),
                      "final_ticks_clocks": {"miller": t[2] - t[1], "easy_part": t[3] - t[2], "hard_part": t[4] - t[3], "to_done": t[5] - t[4]}}
        rec["median_saving_ms"] = rec["horner"]["ms_per_call_median"] - rec["split"]["ms_per_call_median"]
        rec["ranges_overlap"] = rec["split"]["ms_per_call_max"] >= rec["horner"]["ms_per_call_min"]
        out["sizes"][str(n)] = rec
        print(n, json.dumps(rec), flush=True)
    # a false batch (two proofs swapped): same verdict and the same GT element on both tails
    bad = ps.clone()
    bad[:48], bad[48:96] = ps[48:96].clone(), ps[:48].clone()
    gts = {}
    for k in ctxs:
        assert call(k, 64, bad) == 0
        g = C.create_string_buffer(576)
        assert lib.kzgb200_debug_last_gt(ctxs[k], g) == 0
        gts[k] = g.raw
    assert gts["split"] == gts["horner"] and gts["split"] != (b"\x01" + b"\x00" * 575)
    out["false_batch_gt_identical"] = True
    for c in ctxs.values():
        lib.kzgb200_destroy(c)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
