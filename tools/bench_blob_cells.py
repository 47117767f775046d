#!/usr/bin/env python3
"""Blob transactions' cell proofs on one GPU: verify_blob_cell_kzg_proof_batch[_many] through the C ABI, against the caller-side
composition it replaces (compute_cells_batch_device, then verify_cell_kzg_proof_batch_many_device on the expanded arrays).

    python tools/bench_blob_cells.py [--steps 9] [--warmup 2] [--out profiles/bench_blob_cells.json]

Workloads (harness blobs, kzgb200_harness_generate_cells, with their commitments and 128 cell proofs each):
  a  one 6-blob transaction, host buffers (the single call)
  b  a burst of 64 transactions x 6 blobs (384 blobs), host buffers: one _many call, against 64 single calls, against the
     composition (upload, compute_cells_batch_device, expand commitments / indices on the device, _many_device)
  c  128 blobs in one group, device-resident: the _many_device call against the same composition (bench_cells.py's workload d)
  d  b with one tampered transaction (a proof swapped): the combined check fails and every group gets its own check
Every call's verdicts are checked.  Beside each: the serial host SHA-256 time of the same transcripts (one thread; the call hashes
them on up to 16 threads), and compute_cells plus a device-to-host copy of the cells of the same blobs, timed alone, so that the
share of the cell read-back in the call is visible.  Host clock around blocking calls, median of --steps calls after --warmup.
The GPU name, power limit and max SM clock are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_cells import gpu_info, timed, transcript  # noqa: E402

CELL = 2048
BLOB = 131072


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_blob_cells.json"))
    a = ap.parse_args()
    assert a.steps >= 7, "the medians need at least 7 calls"
    import torch
    import kzg_rs_b200 as K
    assert torch.cuda.is_available(), "bench_blob_cells needs a GPU"
    lib = K.Library.get().dll
    S = K.KzgSettings.load_trusted_setup_file()
    ctx = S.cell_context(0)
    tau = K.api.mainnet_g1_monomial()
    res = {"tool": "tools/bench_blob_cells.py", **gpu_info(), "timing": "host clock around blocking calls; median of %d after %d warm-up"
           % (a.steps, a.warmup), "workloads": {}}

    def gen(nb, seed):
        """nb harness blobs on the device: (blobs nb x 131072, commitments nb x 48, cell proofs nb x 128 x 48, all cells)"""
        cells = torch.empty(nb * 128 * CELL, dtype=torch.uint8, device="cuda")
        cs = torch.empty(nb * 48, dtype=torch.uint8, device="cuda")
        ps = torch.empty(nb * 128 * 48, dtype=torch.uint8, device="cuda")
        assert lib.kzgb200_harness_generate_cells(ctx, seed, nb, 192, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
        blobs = cells.view(nb, 128 * CELL)[:, :64 * CELL].contiguous().view(-1)
        torch.cuda.synchronize()
        return blobs, cs, ps, cells

    def host(t):
        return t.cpu().numpy().tobytes()

    def many_host(hb, hc, hp, boffs, want):
        k = len(boffs) - 1
        off = (C.c_uint64 * (k + 1))(*boffs)
        out = C.create_string_buffer(k)

        def call():
            assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many(ctx, hb, hc, hp, C.cast(off, C.c_void_p), k, out) == 0
            assert list(out.raw[:k]) == want
        return call

    def many_device(d_b, d_c, d_p, boffs, want):
        k = len(boffs) - 1
        off = (C.c_uint64 * (k + 1))(*boffs)
        out = C.create_string_buffer(k)

        def call():
            assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many_device(ctx, d_b.data_ptr(), d_c.data_ptr(), d_p.data_ptr(),
                                                                            C.cast(off, C.c_void_p), k, out) == 0
            assert list(out.raw[:k]) == want
        return call

    def singles(hb, hc, hp, boffs, want):
        def call():
            for g in range(len(boffs) - 1):
                lo, hi = boffs[g], boffs[g + 1]
                ok = C.c_int(-1)
                assert lib.kzgb200_verify_blob_cell_kzg_proof_batch(ctx, hb[BLOB * lo:BLOB * hi], hi - lo, hc[48 * lo:48 * hi], hi - lo,
                                                                    hp[48 * 128 * lo:48 * 128 * hi], 128 * (hi - lo), C.byref(ok)) == 0
                assert ok.value == want[g]
        return call

    def composition(blobs_src, cs_src, ps_src, boffs, want):
        """what a caller does without the new call: blobs / commitments / proofs to the device (host sources: pageable bytes),
        compute_cells_batch_device, expanded commitments and indices on the device, verify_cell_kzg_proof_batch_many_device"""
        k, nb = len(boffs) - 1, boffs[-1]
        n = 128 * nb
        off = (C.c_uint64 * (k + 1))(*[128 * b for b in boffs])
        out = C.create_string_buffer(k)
        d_cells = torch.empty(n * CELL, dtype=torch.uint8, device="cuda")
        d_idx = torch.arange(128, dtype=torch.int64, device="cuda").repeat(nb)
        if isinstance(blobs_src, bytes):
            srcs = [torch.frombuffer(bytearray(x), dtype=torch.uint8) for x in (blobs_src, cs_src, ps_src)]
            to_dev = lambda t: t.cuda()
        else:
            srcs, to_dev = [blobs_src, cs_src, ps_src], lambda t: t

        def call():
            d_b, d_c, d_p = (to_dev(t) for t in srcs)
            assert lib.kzgb200_compute_cells_batch_device(ctx, d_b.data_ptr(), nb, d_cells.data_ptr()) == 0
            d_cx = d_c.view(nb, 1, 48).expand(nb, 128, 48).contiguous()
            torch.cuda.synchronize()
            assert lib.kzgb200_verify_cell_kzg_proof_batch_many_device(ctx, d_cx.data_ptr(), d_idx.data_ptr(), d_cells.data_ptr(), d_p.data_ptr(),
                                                                       C.cast(off, C.c_void_p), k, out) == 0
            assert list(out.raw[:k]) == want
        return call

    def readback(d_b, nb):
        """compute_cells of the same blobs plus a device->host copy of their cells into pinned memory, alone"""
        d_cells = torch.empty(nb * 128 * CELL, dtype=torch.uint8, device="cuda")
        h_cells = torch.empty(nb * 128 * CELL, dtype=torch.uint8, pin_memory=True)

        def cc():
            assert lib.kzgb200_compute_cells_batch_device(ctx, d_b.data_ptr(), nb, d_cells.data_ptr()) == 0

        def copy():
            h_cells.copy_(d_cells, non_blocking=True)
            torch.cuda.synchronize()
        t_cc, t_copy = timed(cc, a.steps, a.warmup), timed(copy, a.steps, a.warmup)
        return {"compute_cells_ms": t_cc["median_ms"], "d2h_copy_ms": t_copy["median_ms"], "d2h_bytes": nb * 128 * CELL,
                "d2h_GB_per_s": nb * 128 * CELL / (t_copy["median_ms"] / 1e3) / 1e9, "sum_ms": t_cc["median_ms"] + t_copy["median_ms"]}

    def hash_time(cells_dev, hc, hp, boffs):
        """serial host SHA-256 of the groups' exact transcripts (the expanded calls' bytes), one thread"""
        cells = host(cells_dev)
        msgs = []
        for g in range(len(boffs) - 1):
            lo, hi = boffs[g], boffs[g + 1]
            ents = range(128 * lo, 128 * hi)
            msgs.append(transcript([hc[48 * (e // 128):48 * (e // 128) + 48] for e in ents], [e % 128 for e in ents],
                                   [cells[CELL * e:CELL * (e + 1)] for e in ents], [hp[48 * e:48 * e + 48] for e in ents]))
        h = timed(lambda: [K.api.host_sha256(m) for m in msgs], max(3, a.steps // 2), 1)
        return {"ms": h["median_ms"], "bytes": sum(len(m) for m in msgs)}

    def record(name, desc, variants, nb, d_b, cells_dev, hc, hp, boffs):
        r = {"what": desc, "blobs": nb, "groups": len(boffs) - 1}
        for vname, call in variants:
            r[vname] = timed(call, a.steps, a.warmup)
        main_ms = r[variants[0][0]]["median_ms"]
        r["host_sha256_same_transcripts_serial"] = hash_time(cells_dev, hc, hp, boffs)
        rb = readback(d_b, nb)
        r["compute_cells_plus_d2h_alone"] = rb
        r["d2h_share_of_call"] = rb["d2h_copy_ms"] / main_ms
        r["compute_cells_plus_d2h_share_of_call"] = rb["sum_ms"] / main_ms
        res["workloads"][name] = r
        print(name, json.dumps(r), flush=True)

    # (a) one 6-blob transaction, host buffers
    d_b, d_c, d_p, cells = gen(6, 1)
    hb, hc, hp = host(d_b), host(d_c), host(d_p)
    record("a_one_tx_6_blobs_host", "one 6-blob transaction, host buffers, the single call", [("single_call", singles(hb, hc, hp, [0, 6], [1]))],
           6, d_b, cells, hc, hp, [0, 6])
    # (b) 64 x 6 blobs, host buffers
    nb = 384
    boffs = [6 * g for g in range(65)]
    d_b, d_c, d_p, cells = gen(nb, 2)
    hb, hc, hp = host(d_b), host(d_c), host(d_p)
    want = [1] * 64
    record("b_burst_64x6_host", "64 transactions x 6 blobs (384 blobs), host buffers",
           [("many_call", many_host(hb, hc, hp, boffs, want)), ("single_calls_x64", singles(hb, hc, hp, boffs, want)),
            ("composition", composition(hb, hc, hp, boffs, want))], nb, d_b, cells, hc, hp, boffs)
    # (d) the same burst with one tampered transaction
    t = bytearray(hp)
    e0, e1 = 48 * (128 * 6 * 17 + 3), 48 * (128 * 6 * 17 + 4)       # transaction 17: proofs 3 and 4 of its first blob swapped
    t[e0:e0 + 48], t[e1:e1 + 48] = hp[e1:e1 + 48], hp[e0:e0 + 48]
    hpt = bytes(t)
    want_t = [0 if g == 17 else 1 for g in range(64)]
    record("d_burst_64x6_host_one_tampered", "b with transaction 17's proofs 3 and 4 swapped (per-group fallback)",
           [("many_call", many_host(hb, hc, hpt, boffs, want_t)), ("composition", composition(hb, hc, hpt, boffs, want_t))],
           nb, d_b, cells, hc, hpt, boffs)
    del d_b, d_c, d_p, cells
    # (c) 128 blobs, one group, device-resident
    nb = 128
    d_b, d_c, d_p, cells = gen(nb, 7)
    record("c_one_group_128_blobs_device", "128 blobs in one group, device-resident",
           [("many_device_call", many_device(d_b, d_c, d_p, [0, nb], [1])), ("composition", composition(d_b, d_c, d_p, [0, nb], [1]))],
           nb, d_b, cells, host(d_c), host(d_p), [0, nb])
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    summary = {k: {vk: round(vv["median_ms"], 3) for vk, vv in v.items() if isinstance(vv, dict) and "median_ms" in vv}
               for k, v in res["workloads"].items()}
    print(json.dumps({"out": a.out, **summary}))


if __name__ == "__main__":
    main()
