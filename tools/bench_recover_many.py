#!/usr/bin/env python3
"""recover_cells_and_kzg_proofs_many on one GPU: many blobs in one call, each recovered from its own cells and index set.

    python tools/bench_recover_many.py [--steps 7] [--warmup 2] [--parent PATH] [--out profiles/bench_recover_many.json]

Workloads (blobs from the cell workload generator, kzgb200_harness_generate_cells: degree-192 polynomials whose 128 cells and proofs
the generator computes independently; every timed call's output is compared with them byte for byte):
  a  a 48-blob block, every blob with its own random index set (64..127 cells, random order), host form: the _many call against a
     loop of 48 single kzgb200_recover_cells_and_kzg_proofs calls on the same bytes
  b  the same 48 blobs with one shared random 64-column set, device form: the _many_device call and
     kzgb200_recover_cells_and_kzg_proofs_batch_device, alternated call by call
  c  600 device blobs with their own sets (crosses a 512-blob pass)
  d  (a) with three bad blobs (63 cells, a repeated index, a non-canonical element): their status must be 1, the others bit-exact
  e  (a)'s index sets on 48 uniformly random (full-degree) blobs, and the single call on the first of them; the reference is the
     compute batch on the same blobs, one proof spot-checked against the CPU oracle
With --parent PATH (another build of libkzgb200.so), that build's batch_device call on (b) and its single host call on (a)'s first
blob run in the same process, alternated call by call with this build's, so that the shared-set and single paths can be compared.
Times are CUDA events on each library's stream around each blocking call (a loop of single calls: around the whole loop), after
warm-up; medians with [min, max].  The GPU name, power limit and clock are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import random
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CELL, PROOF = 2048, 48
BLOB_CELLS, BLOB_PROOFS = 128 * CELL, 128 * PROOF
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


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
        d.kzgb200_recover_cells_and_kzg_proofs.argtypes = [p, p, p, sz, p, p]
        d.kzgb200_recover_cells_and_kzg_proofs_batch_device.argtypes = [p, p, sz, p, sz, p, p]
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
    """calls: name -> (stream, fn returning the C return code, check of the output).  One call of each per step, CUDA events on the
    call's stream around it; every output (warm-up included) is checked outside the timed window."""
    import torch
    ts = {name: [] for name in calls}
    for step in range(warmup + steps):
        for name, (stream, fn, check) in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            assert fn() == 0, name
            e1.record(stream)
            e1.synchronize()
            assert check(), "%s: output differs from the generator's" % name
            if step >= warmup:
                ts[name].append(e0.elapsed_time(e1))
    return {name: stats(t) for name, t in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--parent", default=None, help="path of another libkzgb200.so to compare the shared-set and single calls with")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_recover_many.json"))
    a = ap.parse_args()
    import torch
    import kzg_rs_b200 as K
    assert torch.cuda.is_available(), "bench_recover_many needs a GPU"
    lib = K.Library.get().dll
    S = K.KzgSettings.load_trusted_setup_file()
    ctx = S.cell_proof_context(0)
    stream = torch.cuda.ExternalStream(lib.kzgb200_stream(ctx))
    res = {"tool": "tools/bench_recover_many.py", **gpu_info()}

    nmax = 600
    tau = K.api.mainnet_g1_monomial()
    g_cells = torch.empty(nmax * BLOB_CELLS, dtype=torch.uint8, device="cuda")
    g_cs = torch.empty(nmax * 48, dtype=torch.uint8, device="cuda")
    g_ps = torch.empty(nmax * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_harness_generate_cells(ctx, 0x5eca, nmax, 192, tau, g_cells.data_ptr(), g_cs.data_ptr(), g_ps.data_ptr()) == 0
    torch.cuda.synchronize()
    rows = g_cells.view(-1, CELL)

    def inputs(sets):
        """one index set per blob (blob b = generator blob b) -> (flat indices, offsets, device cells)"""
        offs = [0]
        for s in sets:
            offs.append(offs[-1] + len(s))
        sel = torch.tensor([b * 128 + k for b, s in enumerate(sets) for k in s], device="cuda")
        return [k for s in sets for k in s], offs, rows[sel].contiguous().view(-1)

    def c_arrays(idx, offs):
        return (C.c_uint64 * len(idx))(*idx), (C.c_uint64 * len(offs))(*offs)

    nb = 48
    rnd = random.Random(48)
    own = [rnd.sample(range(128), rnd.randint(64, 127)) for _ in range(nb)]
    want_c, want_p = g_cells[:nb * BLOB_CELLS].cpu().numpy().tobytes(), g_ps[:nb * BLOB_PROOFS].cpu().numpy().tobytes()

    # (a) per-blob sets, host form: the _many call and a loop of single calls
    idx, offs_a, d_in = inputs(own)
    h_in = d_in.cpu().numpy().tobytes()
    ia, oa = c_arrays(idx, offs_a)
    hc, hp, st = C.create_string_buffer(nb * BLOB_CELLS), C.create_string_buffer(nb * BLOB_PROOFS), C.create_string_buffer(nb)
    sc, sp = C.create_string_buffer(nb * BLOB_CELLS), C.create_string_buffer(nb * BLOB_PROOFS)
    own_cells = [h_in[offs_a[b] * CELL:offs_a[b + 1] * CELL] for b in range(nb)]
    singles = [((C.c_uint64 * len(s))(*s), own_cells[b]) for b, s in enumerate(own)]

    def single_loop():
        for b, (sa, cells) in enumerate(singles):
            rc = lib.kzgb200_recover_cells_and_kzg_proofs(ctx, sa, cells, len(own[b]), C.byref(sc, b * BLOB_CELLS), C.byref(sp, b * BLOB_PROOFS))
            if rc:
                return rc
        return 0
    res["a_own_sets_48_host"] = alternate({
        "many": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, ia, h_in, oa, nb, hc, hp, st),
                 lambda: st.raw == bytes(nb) and hc.raw == want_c and hp.raw == want_p),
        "single_call_loop": (stream, single_loop, lambda: sc.raw == want_c and sp.raw == want_p),
    }, a.steps, a.warmup)
    res["a_own_sets_48_host"]["cells_per_blob"] = [len(s) for s in own]

    # (b) one shared 64-column set, device form: the _many call and the shared-set batch, alternated
    cols = random.Random(64).sample(range(128), 64)
    idx, offs, d_in = inputs([cols] * nb)
    ia_b, oa_b = c_arrays(idx, offs)
    ca = (C.c_uint64 * 64)(*cols)
    out_c, out_p = torch.empty(nb * BLOB_CELLS, dtype=torch.uint8, device="cuda"), torch.empty(nb * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    ok_dev = lambda n: torch.equal(out_c[:n * BLOB_CELLS], g_cells[:n * BLOB_CELLS]) and torch.equal(out_p[:n * BLOB_PROOFS], g_ps[:n * BLOB_PROOFS])
    calls = {
        "many_device": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many_device(ctx, ia_b, d_in.data_ptr(), oa_b, nb, out_c.data_ptr(),
                                                                                             out_p.data_ptr(), st),
                        lambda: st.raw[:nb] == bytes(nb) and ok_dev(nb)),
        "batch_device": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ca, 64, d_in.data_ptr(), nb, out_c.data_ptr(),
                                                                                               out_p.data_ptr()),
                         lambda: ok_dev(nb)),
    }
    parent = ParentLib(a.parent, S) if a.parent else None
    if parent:
        calls["parent_batch_device"] = (parent.stream, lambda: parent.dll.kzgb200_recover_cells_and_kzg_proofs_batch_device(
            parent.ctx, ca, 64, d_in.data_ptr(), nb, out_c.data_ptr(), out_p.data_ptr()), lambda: ok_dev(nb))
    res["b_shared_set_48_device"] = alternate(calls, a.steps, a.warmup)
    res["b_shared_set_48_device"]["columns"] = cols

    # the single host call on (a)'s first blob, this build and the parent alternated
    sa0, cells0 = singles[0]
    c1, p1 = C.create_string_buffer(BLOB_CELLS), C.create_string_buffer(BLOB_PROOFS)
    calls = {"single_host": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs(ctx, sa0, cells0, len(own[0]), c1, p1),
                             lambda: c1.raw == want_c[:BLOB_CELLS] and p1.raw == want_p[:BLOB_PROOFS])}
    if parent:
        calls["parent_single_host"] = (parent.stream, lambda: parent.dll.kzgb200_recover_cells_and_kzg_proofs(parent.ctx, sa0, cells0, len(own[0]), c1, p1),
                                       lambda: c1.raw == want_c[:BLOB_CELLS] and p1.raw == want_p[:BLOB_PROOFS])
    res["single_host_blob"] = alternate(calls, a.steps, a.warmup)

    # (c) 600 device blobs with their own sets
    rnd = random.Random(600)
    big = [rnd.sample(range(128), rnd.randint(64, 127)) for _ in range(nmax)]
    idx, offs, d_big = inputs(big)
    ia_c, oa_c = c_arrays(idx, offs)
    big_c, big_p = torch.empty_like(g_cells), torch.empty_like(g_ps)
    st_c = C.create_string_buffer(nmax)
    res["c_own_sets_600_device"] = alternate({
        "many_device": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many_device(ctx, ia_c, d_big.data_ptr(), oa_c, nmax, big_c.data_ptr(),
                                                                                             big_p.data_ptr(), st_c),
                        lambda: st_c.raw == bytes(nmax) and torch.equal(big_c, g_cells) and torch.equal(big_p, g_ps))}, a.steps, a.warmup)
    r = res["c_own_sets_600_device"]["many_device"]
    r["blobs_per_s"] = round(nmax / (r["median_ms"] / 1e3), 1)

    # (d) (a) with three bad blobs
    bad_sets = [list(s) for s in own]
    cells_d = list(own_cells)
    bad_sets[5], cells_d[5] = bad_sets[5][:63], cells_d[5][:63 * CELL]                                  # 63 cells
    bad_sets[20] = bad_sets[20][:-1] + [bad_sets[20][0]]                                                # a repeated index
    t = bytearray(cells_d[33]); t[32 * 70:32 * 71] = Q.to_bytes(32, "big"); cells_d[33] = bytes(t)     # an element equal to q
    offs_d = [0]
    for s in bad_sets:
        offs_d.append(offs_d[-1] + len(s))
    ia_d, oa_d = c_arrays([k for s in bad_sets for k in s], offs_d)
    h_in_d = b"".join(cells_d)
    is_bad = bytes(int(b in (5, 20, 33)) for b in range(nb))

    def check_d():
        if st.raw != is_bad:
            return False
        return all(hc.raw[b * BLOB_CELLS:(b + 1) * BLOB_CELLS] == want_c[b * BLOB_CELLS:(b + 1) * BLOB_CELLS]
                   and hp.raw[b * BLOB_PROOFS:(b + 1) * BLOB_PROOFS] == want_p[b * BLOB_PROOFS:(b + 1) * BLOB_PROOFS] for b in range(nb) if not is_bad[b])
    res["d_own_sets_48_host_3_bad"] = alternate({
        "many": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, ia_d, h_in_d, oa_d, nb, hc, hp, st), check_d)}, a.steps, a.warmup)

    # (e) (a)'s index sets on 48 uniformly random (full-degree) blobs: the generator's degree-192 blobs leave most of FK20's H_t at
    # the identity, which the G1 transforms skip.  Reference: the compute batch on the same blobs, spot-checked with the CPU oracle.
    from cell_oracle import cells as CO
    rnd = random.Random(4844)
    fblobs = b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(nb * 4096))
    f_cells, f_ps = torch.empty(nb * BLOB_CELLS, dtype=torch.uint8, device="cuda"), torch.empty(nb * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    d_fb = torch.frombuffer(bytearray(fblobs), dtype=torch.uint8).cuda()
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, d_fb.data_ptr(), nb, f_cells.data_ptr(), f_ps.data_ptr()) == 0
    torch.cuda.synchronize()
    fwant_c, fwant_p = f_cells.cpu().numpy().tobytes(), f_ps.cpu().numpy().tobytes()
    assert CO.compute_cell_kzg_proof(fblobs[:131072], 5) == fwant_p[5 * PROOF:6 * PROOF]
    fh_in = f_cells.view(-1, CELL)[torch.tensor([b * 128 + k for b, s in enumerate(own) for k in s], device="cuda")].cpu().numpy().tobytes()
    f0 = fh_in[:len(own[0]) * CELL]
    res["e_full_degree_own_sets_48_host"] = alternate({
        "many": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, ia, fh_in, oa, nb, hc, hp, st),
                 lambda: st.raw == bytes(nb) and hc.raw == fwant_c and hp.raw == fwant_p),
        "single_host_blob0": (stream, lambda: lib.kzgb200_recover_cells_and_kzg_proofs(ctx, sa0, f0, len(own[0]), c1, p1),
                              lambda: c1.raw == fwant_c[:BLOB_CELLS] and p1.raw == fwant_p[:BLOB_PROOFS]),
    }, a.steps, a.warmup)

    # per-phase device times of one profiled call each (profiling adds events; these are not the timed numbers above)
    names = ["coefficients", "fixed_base_products", "g1_transforms", "recovery_transforms"]
    phases = {}
    ms = (C.c_float * 8)()
    lib.kzgb200_set_profiling(ctx, 1)
    for label, fn in (("a_many", lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, ia, h_in, oa, nb, hc, hp, st)),
                      ("b_many_device", lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many_device(ctx, ia_b, d_in.data_ptr(), oa_b, nb,
                                                                                                      out_c.data_ptr(), out_p.data_ptr(), st)),
                      ("e_many", lambda: lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, ia, fh_in, oa, nb, hc, hp, st)),
                      ("b_batch_device", lambda: lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ca, 64, d_in.data_ptr(), nb,
                                                                                                        out_c.data_ptr(), out_p.data_ptr()))):
        assert fn() == 0
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
        phases[label] = {names[i]: round(ms[i], 3) for i in range(4)}
    lib.kzgb200_set_profiling(ctx, 0)
    res["phases_ms"] = phases
    if parent:
        parent.dll.kzgb200_destroy(parent.ctx)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
