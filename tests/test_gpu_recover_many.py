"""recover_cells_and_kzg_proofs_many on the GPU (pytest -m gpu): many blobs in one call, each recovered from its own cells and index
set, one status per blob.  Every good blob's cells and proofs are compared byte for byte with compute_cells_and_kzg_proofs of the
source blob and with the single recover_cells_and_kzg_proofs call; bad blobs among good ones get status 1 and change nothing else."""
import ctypes as C
import random

import pytest

from cell_oracle import cells as CO

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
CELL, PROOF = 2048, 48
BLOB_CELLS, BLOB_PROOFS = 128 * CELL, 128 * PROOF


@pytest.fixture(scope="module")
def K():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import kzg_rs_b200 as K
    return K


@pytest.fixture(scope="module")
def settings(K):
    s = K.KzgSettings.load_trusted_setup_file()
    s.cell_proof_context(0)
    yield s
    s.close()


@pytest.fixture(scope="module")
def lib(K):
    return K.Library.get().dll


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))


def dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


@pytest.fixture(scope="module")
def sources(settings, lib):
    """six random blobs and the zero blob with their 128 cells and proofs (compute_cells_and_kzg_proofs_batch_device), device tensors"""
    import torch
    blobs = [rand_blob(700 + i) for i in range(6)] + [bytes(131072)]
    n = len(blobs)
    d_c = torch.empty(n * BLOB_CELLS, dtype=torch.uint8, device="cuda")
    d_p = torch.empty(n * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(settings.cell_proof_context(0), dev(b"".join(blobs)).data_ptr(), n,
                                                                 d_c.data_ptr(), d_p.data_ptr()) == 0
    torch.cuda.synchronize()
    return blobs, d_c, d_p


def host_cells(d_c, s):
    raw = d_c[s * BLOB_CELLS:(s + 1) * BLOB_CELLS].cpu().numpy().tobytes()
    return [raw[CELL * k:CELL * (k + 1)] for k in range(128)]


def host_ref(d_c, d_p, s):
    return (d_c[s * BLOB_CELLS:(s + 1) * BLOB_CELLS].cpu().numpy().tobytes(), d_p[s * BLOB_PROOFS:(s + 1) * BLOB_PROOFS].cpu().numpy().tobytes())


def call_host(lib, ctx, items):
    """items: (indices, joined cell bytes) per blob -> (rc, cells, proofs, status) of the host form"""
    idx = [i for ids, _ in items for i in ids]
    offs = [0]
    for ids, _ in items:
        offs.append(offs[-1] + len(ids))
    k = len(items)
    ia = (C.c_uint64 * max(len(idx), 1))(*idx)
    off = (C.c_uint64 * (k + 1))(*offs)
    cells, proofs = C.create_string_buffer(max(k, 1) * BLOB_CELLS), C.create_string_buffer(max(k, 1) * BLOB_PROOFS)
    status = C.create_string_buffer(b"\xaa" * max(k, 1), max(k, 1))
    rc = lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, C.cast(ia, C.c_void_p), b"".join(c for _, c in items), C.cast(off, C.c_void_p), k,
                                                       cells, proofs, status)
    return rc, cells.raw, proofs.raw, list(status.raw[:k])


def call_device(lib, ctx, idx, offs, d_in):
    """the device form on device input cells -> (rc, cells tensor, proofs tensor, status)"""
    import torch
    k = len(offs) - 1
    ia = (C.c_uint64 * max(len(idx), 1))(*idx)
    off = (C.c_uint64 * (k + 1))(*offs)
    d_c = torch.empty(max(k, 1) * BLOB_CELLS, dtype=torch.uint8, device="cuda")
    d_p = torch.empty(max(k, 1) * BLOB_PROOFS, dtype=torch.uint8, device="cuda")
    status = C.create_string_buffer(b"\xaa" * max(k, 1), max(k, 1))
    rc = lib.kzgb200_recover_cells_and_kzg_proofs_many_device(ctx, C.cast(ia, C.c_void_p), d_in.data_ptr() if d_in is not None else None,
                                                              C.cast(off, C.c_void_p), k, d_c.data_ptr(), d_p.data_ptr(), status)
    torch.cuda.synchronize()
    return rc, d_c, d_p, list(status.raw[:k])


def gather(d_c, plan):
    """plan: (source, indices) per blob -> (flat indices, offsets, device cells in that order)"""
    import torch
    rows = [s * 128 + i for s, ids in plan for i in ids]
    offs = [0]
    for _, ids in plan:
        offs.append(offs[-1] + len(ids))
    return [i for _, ids in plan for i in ids], offs, d_c.view(-1, CELL)[torch.tensor(rows, device="cuda")].contiguous().view(-1)


def random_sets(seed, sizes):
    rnd = random.Random(seed)
    return [rnd.sample(range(128), n) for n in sizes]


def test_per_blob_index_sets(K, settings, lib, sources):
    """64, 65..127 and 128 cells, unsorted, one set per blob: the source's cells and proofs, and the single call's bytes"""
    import torch
    ctx = settings.cell_proof_context(0)
    blobs, d_c, d_p = sources
    sets = random_sets(11, [64, 65, 97, 127, 128, 64, 80])
    plan = [(s % len(blobs), sets[s]) for s in range(len(sets))]
    idx, offs, d_in = gather(d_c, plan)
    rc, o_c, o_p, st = call_device(lib, ctx, idx, offs, d_in)
    assert rc == 0 and st == [0] * len(plan)
    want_c = torch.cat([d_c[s * BLOB_CELLS:(s + 1) * BLOB_CELLS] for s, _ in plan])
    want_p = torch.cat([d_p[s * BLOB_PROOFS:(s + 1) * BLOB_PROOFS] for s, _ in plan])
    assert torch.equal(o_c, want_c) and torch.equal(o_p, want_p)
    # the host form and the Python API give the same bytes; so does one single call per blob
    items = []
    for s, ids in plan:
        cells = host_cells(d_c, s)
        items.append((ids, b"".join(cells[k] for k in ids)))
    rc, h_c, h_p, st = call_host(lib, ctx, items)
    assert rc == 0 and st == [0] * len(plan)
    assert h_c == o_c.cpu().numpy().tobytes() and h_p == o_p.cpu().numpy().tobytes()
    py = K.recover_cells_and_kzg_proofs_many([(ids, [c[CELL * j:CELL * (j + 1)] for j in range(len(ids))]) for ids, c in items], settings)
    for b, (s, ids) in enumerate(plan):
        cells = host_cells(d_c, s)
        single = K.recover_cells_and_kzg_proofs(ids, [cells[k] for k in ids], settings)
        assert py[b] == single, b
        assert b"".join(single[0]) == h_c[b * BLOB_CELLS:(b + 1) * BLOB_CELLS]
        assert b"".join(single[1]) == h_p[b * BLOB_PROOFS:(b + 1) * BLOB_PROOFS]


def test_shared_set_equals_batch_device(settings, lib, sources):
    import torch
    ctx = settings.cell_proof_context(0)
    blobs, d_c, _ = sources
    ids = random_sets(12, [70])[0]
    plan = [(s, ids) for s in range(len(blobs))]
    idx, offs, d_in = gather(d_c, plan)
    rc, o_c, o_p, st = call_device(lib, ctx, idx, offs, d_in)
    assert rc == 0 and st == [0] * len(plan)
    b_c, b_p = torch.empty_like(o_c), torch.empty_like(o_p)
    ia = (C.c_uint64 * len(ids))(*ids)
    assert lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, len(ids), d_in.data_ptr(), len(plan), b_c.data_ptr(), b_p.data_ptr()) == 0
    torch.cuda.synchronize()
    assert torch.equal(o_c, b_c) and torch.equal(o_p, b_p)
    assert torch.equal(o_c, d_c)


def test_inconsistent_blob(K, settings, lib, sources):
    """an altered element in one blob: that blob gets the spec's bytes (the C oracle's) and the single call's proofs, status 0"""
    ctx = settings.cell_proof_context(0)
    blobs, d_c, d_p = sources
    a_ids, b_ids = random_sets(13, [80, 66])
    a_cells, b_cells = host_cells(d_c, 0), host_cells(d_c, 1)
    given = [b_cells[k] for k in b_ids]
    t = bytearray(given[9]); t[32 * 5 + 31] ^= 1
    given[9] = bytes(t)
    ref = CO.recover_cells(b_ids, given)
    assert ref is not None and ref != b_cells
    items = [(a_ids, b"".join(a_cells[k] for k in a_ids)), (b_ids, b"".join(given))]
    rc, h_c, h_p, st = call_host(lib, ctx, items)
    assert rc == 0 and st == [0, 0]
    assert (h_c[:BLOB_CELLS], h_p[:BLOB_PROOFS]) == host_ref(d_c, d_p, 0)
    assert h_c[BLOB_CELLS:2 * BLOB_CELLS] == b"".join(ref)
    single = K.recover_cells_and_kzg_proofs(b_ids, given, settings)
    assert b"".join(single[0]) == b"".join(ref) and b"".join(single[1]) == h_p[BLOB_PROOFS:2 * BLOB_PROOFS]


def test_bad_blobs_among_good(K, settings, lib, sources):
    """63 cells, 129 cells, index 128, a repeated index and an element equal to q: status 1 exactly there, the good blobs bit-exact"""
    import torch
    ctx = settings.cell_proof_context(0)
    blobs, d_c, d_p = sources
    good = random_sets(14, [64, 100, 128, 77])
    cells = [host_cells(d_c, s) for s in range(4)]
    g = lambda s: (good[s], b"".join(cells[s][k] for k in good[s]))
    r = random_sets(15, [64])[0]
    noncanon = bytearray(b"".join(cells[1][k] for k in r))
    noncanon[20 * CELL + 32 * 7:20 * CELL + 32 * 8] = Q.to_bytes(32, "big")
    bad = [
        (r[:63], b"".join(cells[0][k] for k in r[:63])),                                   # 63 cells
        (list(range(128)) + [5], b"".join(cells[2]) + cells[2][5]),                        # 129 cells
        (r[:63] + [128], b"".join(cells[3][k] for k in r)),                                # index 128
        (r[:64] + [r[10]], b"".join(cells[0][k] for k in r) + cells[0][r[10]]),            # a repeated index
        (r, bytes(noncanon)),                                                              # an element equal to q
    ]
    items = [g(0), bad[0], bad[1], g(1), bad[2], g(2), bad[3], bad[4], g(3)]
    is_bad = [0, 1, 1, 0, 1, 0, 1, 1, 0]
    src = {0: 0, 3: 1, 5: 2, 8: 3}
    rc, h_c, h_p, st = call_host(lib, ctx, items)
    assert rc == 0 and st == is_bad
    for b, s in src.items():
        assert (h_c[b * BLOB_CELLS:(b + 1) * BLOB_CELLS], h_p[b * BLOB_PROOFS:(b + 1) * BLOB_PROOFS]) == host_ref(d_c, d_p, s), b
    # the device form: the same statuses and bytes
    offs = [0]
    for ids, _ in items:
        offs.append(offs[-1] + len(ids))
    rc, o_c, o_p, st2 = call_device(lib, ctx, [i for ids, _ in items for i in ids], offs, dev(b"".join(c for _, c in items)))
    assert rc == 0 and st2 == is_bad
    for b, s in src.items():
        assert torch.equal(o_c[b * BLOB_CELLS:(b + 1) * BLOB_CELLS], d_c[s * BLOB_CELLS:(s + 1) * BLOB_CELLS])
        assert torch.equal(o_p[b * BLOB_PROOFS:(b + 1) * BLOB_PROOFS], d_p[s * BLOB_PROOFS:(s + 1) * BLOB_PROOFS])
    # every bad blob alone is BadArgs for the single call, and None (with an index outside u64 too) through the Python API
    split = lambda c: [c[CELL * j:CELL * (j + 1)] for j in range(len(c) // CELL)]
    for ids, c in bad:
        with pytest.raises(K.KzgError) as e:
            K.recover_cells_and_kzg_proofs(ids, split(c), settings)
        assert e.value.kind == "BadArgs"
    py = K.recover_cells_and_kzg_proofs_many([(ids, split(c)) for ids, c in items] + [([-1] + good[0][1:], split(g(0)[1]))], settings)
    assert [p is None for p in py] == [bool(x) for x in is_bad] + [True]
    assert b"".join(py[3][0]) == host_ref(d_c, d_p, 1)[0]


def test_passes_crossed(settings, lib, sources):
    """600 blobs (the seven sources tiled, each blob with its own random set of 64..128 cells) cross a 512-blob pass; host == device"""
    import torch
    ctx = settings.cell_proof_context(0)
    blobs, d_c, d_p = sources
    rnd = random.Random(16)
    plan = [(b % len(blobs), rnd.sample(range(128), rnd.randint(64, 128))) for b in range(600)]
    idx, offs, d_in = gather(d_c, plan)
    rc, o_c, o_p, st = call_device(lib, ctx, idx, offs, d_in)
    assert rc == 0 and st == [0] * len(plan)
    src = torch.tensor([s for s, _ in plan], device="cuda")
    assert torch.equal(o_c.view(len(plan), -1), d_c.view(len(blobs), -1)[src])
    assert torch.equal(o_p.view(len(plan), -1), d_p.view(len(blobs), -1)[src])
    # the host form on the same bytes, with a bad blob in the second pass
    raw = d_in.cpu().numpy().tobytes()
    items = [(ids, raw[offs[b] * CELL:offs[b + 1] * CELL]) for b, (_, ids) in enumerate(plan)]
    items[555] = (items[555][0][:63], items[555][1][:63 * CELL])
    rc, h_c, h_p, st = call_host(lib, ctx, items)
    assert rc == 0 and st == [int(b == 555) for b in range(len(plan))]
    want_c, want_p = bytearray(o_c.cpu().numpy().tobytes()), bytearray(o_p.cpu().numpy().tobytes())
    want_c[555 * BLOB_CELLS:556 * BLOB_CELLS] = h_c[555 * BLOB_CELLS:556 * BLOB_CELLS]
    want_p[555 * BLOB_PROOFS:556 * BLOB_PROOFS] = h_p[555 * BLOB_PROOFS:556 * BLOB_PROOFS]
    assert h_c == bytes(want_c) and h_p == bytes(want_p)


def test_call_level_errors(K, settings, lib, sources):
    ctx = settings.cell_proof_context(0)
    _, d_c, _ = sources
    assert call_host(lib, ctx, [])[0] == 0
    assert lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, None, None, None, 0, None, None, None) == 0
    assert lib.kzgb200_recover_cells_and_kzg_proofs_many_device(ctx, None, None, None, 0, None, None, None) == 0
    ids = list(range(64))
    cells = b"".join(host_cells(d_c, 0)[:64])
    ia = (C.c_uint64 * 64)(*ids)
    out_c, out_p, status = C.create_string_buffer(2 * BLOB_CELLS), C.create_string_buffer(2 * BLOB_PROOFS), C.create_string_buffer(2)
    call = lambda offs, k=None, st=status, cs=cells: lib.kzgb200_recover_cells_and_kzg_proofs_many(
        ctx, C.cast(ia, C.c_void_p), cs, C.cast((C.c_uint64 * len(offs))(*offs), C.c_void_p), len(offs) - 1 if k is None else k, out_c, out_p, st)
    assert call([0, 64]) == 0 and status.raw[0] == 0
    assert call([1, 64]) == 1                      # offsets[0] != 0
    assert call([0, 64, 32]) == 1                  # decreasing offsets
    assert call([0, 0x7fffffff // 2 + 1]) == 1     # above the cell limit
    assert call([0, 64], st=None) == 1             # no status buffer
    assert call([0, 64], cs=None) == 1             # no cells with cells to read
    assert call([0, 0, 0]) == 0 and status.raw == b"\x01\x01"   # blobs without cells: bad blobs, not a bad call
    assert lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, C.cast(ia, C.c_void_p), cells, None, 1, out_c, out_p, status) == 1
    assert lib.kzgb200_recover_cells_and_kzg_proofs_many(ctx, None, None, None, 0x7fffffff // 2 + 1, out_c, out_p, status) == 1
    # before the proof setup
    fresh = K.KzgSettings(settings.g1_lagrange_bytes, settings.g2_monomial_bytes)
    try:
        fctx = fresh.cell_context(0)
        off = (C.c_uint64 * 2)(0, 64)
        assert lib.kzgb200_recover_cells_and_kzg_proofs_many(fctx, C.cast(ia, C.c_void_p), cells, C.cast(off, C.c_void_p), 1, out_c, out_p, status) == 5
        assert lib.kzgb200_recover_cells_and_kzg_proofs_many_device(fctx, None, None, None, 0, None, None, None) == 5
    finally:
        fresh.close()


def test_profiled_phases(settings, lib, sources):
    ctx = settings.cell_proof_context(0)
    _, d_c, _ = sources
    idx, offs, d_in = gather(d_c, [(s, ids) for s, ids in enumerate(random_sets(17, [64, 90, 128]))])
    ms = (C.c_float * 8)()
    lib.kzgb200_set_profiling(ctx, 1)
    try:
        rc, _, _, st = call_device(lib, ctx, idx, offs, d_in)
        assert rc == 0 and st == [0, 0, 0]
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
    finally:
        lib.kzgb200_set_profiling(ctx, 0)
    assert all(ms[i] > 0 for i in range(4)) and all(ms[i] == 0 for i in range(4, 8))


def test_block_recovery_verifies(settings, lib, sources):
    """a 24-blob block recovered with per-blob index sets: all 3072 recovered cells and proofs verify against the blobs' commitments"""
    import torch
    ctx = settings.cell_proof_context(0)
    blobs, d_c, _ = sources
    nb = 24
    rnd = random.Random(18)
    plan = [(b % len(blobs), rnd.sample(range(128), rnd.randint(64, 127))) for b in range(nb)]
    idx, offs, d_in = gather(d_c, plan)
    rc, o_c, o_p, st = call_device(lib, ctx, idx, offs, d_in)
    assert rc == 0 and st == [0] * nb
    assert lib.kzgb200_load_g1_lagrange(ctx, settings.g1_lagrange_bytes, 4096) == 0
    d_b = dev(b"".join(blobs[s] for s, _ in plan))
    cs = torch.empty(nb * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, d_b.data_ptr(), nb, cs.data_ptr()) == 0
    d_cm = cs.view(nb, 1, 48).expand(nb, 128, 48).contiguous().view(-1)
    d_idx = torch.arange(128, dtype=torch.int64, device="cuda").repeat(nb)
    ok = C.c_int(-1)
    assert lib.kzgb200_verify_cell_kzg_proof_batch_device(ctx, d_cm.data_ptr(), d_idx.data_ptr(), o_c.data_ptr(), o_p.data_ptr(), nb * 128,
                                                          C.byref(ok)) == 0
    assert ok.value == 1
    # one swapped proof fails the batch
    o_p[:48], o_p[48:96] = o_p[48:96].clone(), o_p[:48].clone()
    assert lib.kzgb200_verify_cell_kzg_proof_batch_device(ctx, d_cm.data_ptr(), d_idx.data_ptr(), o_c.data_ptr(), o_p.data_ptr(), nb * 128,
                                                          C.byref(ok)) == 0
    assert ok.value == 0
