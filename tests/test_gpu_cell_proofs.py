"""EIP-7594 cell proofs and recovery on the GPU (pytest -m gpu): the monomial setup derived from the Lagrange points, FK20
compute_cells_and_kzg_proofs and recover_cells_and_kzg_proofs through the C ABI and the Python API -- bit-exact against the cell
workload generator, the CPU oracle's direct-division proofs and its spec recovery, and checked by both verifiers."""
import ctypes as C
import os
import random

import pytest
from conftest import GOLDEN, unhex

from cell_oracle import cells as CO

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
CELL = 2048
IDENTITY = b"\xc0" + bytes(47)


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
    return s


@pytest.fixture(scope="module")
def lib(K):
    return K.Library.get().dll


@pytest.fixture(scope="module")
def fixture_blobs(vectors):
    """full-degree fixture blobs with their fixture commitments (valid verify_blob_kzg_proof cases)"""
    out = []
    for c in vectors["verify_blob_kzg_proof"]:
        b = vectors.blobs[c["blob"]]
        full = len(b) == 131072 and len({b[32 * i:32 * i + 32] for i in range(4096)}) == 4096
        if c["output"] is True and full and (b, unhex(c["commitment"])) not in out:
            out.append((b, unhex(c["commitment"])))
    assert len(out) >= 2
    return out


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))


def bad_args(K, fn):
    with pytest.raises(K.KzgError) as e:
        fn()
    assert e.value.kind == "BadArgs", e.value.kind


def dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


def batch_device(lib, ctx, blobs):
    import torch
    n = len(blobs)
    d_b = dev(b"".join(blobs))
    d_c = torch.empty(n * 128 * CELL, dtype=torch.uint8, device="cuda")
    d_p = torch.empty(n * 128 * 48, dtype=torch.uint8, device="cuda")
    rc = lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, d_b.data_ptr(), n, d_c.data_ptr(), d_p.data_ptr())
    return rc, d_c, d_p


def gpu_verify(lib, ctx, commitments, idx, cells, proofs):
    ok = C.c_int(-1)
    n = len(idx)
    ia = (C.c_uint64 * n)(*idx)
    rc = lib.kzgb200_verify_cell_kzg_proof_batch(ctx, b"".join(commitments), ia, b"".join(cells), b"".join(proofs), n, C.byref(ok))
    assert rc == 0
    return bool(ok.value)


# ---- monomial setup ------------------------------------------------------------------------------------------------------
def test_monomial_points(K, settings, lib, oracle):
    ctx = settings.cell_proof_context(0)
    out = C.create_string_buffer(4096 * 48)
    assert lib.kzgb200_cell_proof_monomial(ctx, out, 4096) == 0
    mono = out.raw
    assert mono[:192 * 48] == K.api.mainnet_g1_monomial()
    pt = lambda j: mono[48 * j:48 * j + 48]
    for j in (191, 1000, 2047, 4030):                              # e([tau^(j+1)], G2) == e([tau^j], [tau]G2)
        assert oracle.pairings_verify(pt(j + 1), 0, pt(j), 1) is True
    assert oracle.pairings_verify(pt(1001), 0, pt(999), 1) is False
    assert pt(4030) == oracle.tau_power_g1(4030)
    assert lib.kzgb200_cell_proof_monomial(ctx, out, 4097) == 1


def test_setup_errors(K, settings, lib):
    # proof setup before the cell setup, and every proof / recovery call before the proof setup
    fresh = K.KzgSettings(settings.g1_lagrange_bytes, settings.g2_monomial_bytes)
    try:
        ctx = fresh.context(0)
        assert lib.kzgb200_load_cell_proof_setup(ctx, settings.g1_lagrange_bytes, 4096) == 5
        fresh.cell_context(0)
        cells, proofs = C.create_string_buffer(128 * CELL), C.create_string_buffer(128 * 48)
        idx = (C.c_uint64 * 64)(*range(64))
        assert lib.kzgb200_compute_cells_and_kzg_proofs(ctx, bytes(131072), cells, proofs) == 5
        assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, None, 0, None, None) == 5
        assert lib.kzgb200_recover_cells_and_kzg_proofs(ctx, idx, bytes(64 * CELL), 64, cells, proofs) == 5
        assert lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, idx, 64, None, 0, None, None) == 5
        assert lib.kzgb200_cell_proof_monomial(ctx, cells, 4) == 5
        assert lib.kzgb200_load_cell_proof_setup(ctx, settings.g1_lagrange_bytes, 4095) == 5
        # the cell verifier still runs on this context
        assert K.KzgProof.verify_cell_kzg_proof_batch([], [], [], [], fresh) is True
    finally:
        fresh.close()
    # Lagrange points of another setup than the loaded cell points
    custom = K.KzgSettings.load_trusted_setup_file(os.path.join(GOLDEN, "custom_setup.bin"), g1_monomial_bytes=K.api.mainnet_g1_monomial())
    try:
        with pytest.raises(K.KzgError) as e:
            custom.cell_proof_context(0)
        assert e.value.kind == "InvalidTrustedSetup"
    finally:
        custom.close()


# ---- compute_cells_and_kzg_proofs ------------------------------------------------------------------------------------------
def test_harness_blobs_bit_exact(K, settings, lib):
    """128 degree-192 harness blobs: the batch call reproduces the generator's 16384 proofs and its cells"""
    import torch
    nb = 128
    ctx = settings.cell_proof_context(0)
    tau = K.api.mainnet_g1_monomial()
    cells = torch.empty(nb * 128 * CELL, dtype=torch.uint8, device="cuda")
    cs = torch.empty(nb * 48, dtype=torch.uint8, device="cuda")
    ps = torch.empty(nb * 128 * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_harness_generate_cells(ctx, 0xf20, nb, 192, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
    blobs = cells.view(nb, 128 * CELL)[:, :64 * CELL].contiguous()
    d_c = torch.empty_like(cells)
    d_p = torch.empty_like(ps)
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, blobs.data_ptr(), nb, d_c.data_ptr(), d_p.data_ptr()) == 0
    torch.cuda.synchronize()
    assert torch.equal(d_p, ps)
    assert torch.equal(d_c, cells)


def test_full_degree_blobs(K, settings, lib, oracle, fixture_blobs):
    ctx = settings.cell_proof_context(0)
    cases = [(b, c) for b, c in fixture_blobs[:2]] + [(rand_blob(s), None) for s in (31, 32)]
    for i, (blob, c) in enumerate(cases):
        if c is None:
            c = oracle.blob_to_kzg_commitment(blob)
        cells, proofs = K.compute_cells_and_kzg_proofs(blob, settings)
        assert cells == K.compute_cells(blob, settings)
        for k in ((0, 1, 63, 64, 100, 127) if i in (0, 2) else (5, 99)):
            assert proofs[k] == CO.compute_cell_kzg_proof(blob, k), k
        idx = list(range(128))
        assert CO.verify_cell_kzg_proof_batch([c] * 128, idx, cells, proofs) is True
        assert K.KzgProof.verify_cell_kzg_proof_batch([c] * 128, idx, cells, proofs, settings) is True
        assert gpu_verify(lib, ctx, [c] * 128, idx, cells, proofs) is True
        bad = list(proofs)
        bad[40], bad[41] = proofs[41], proofs[40]
        assert K.KzgProof.verify_cell_kzg_proof_batch([c] * 128, idx, cells, bad, settings) is False


def test_edge_cases(K, settings, lib):
    ctx = settings.cell_proof_context(0)
    cells, proofs = K.compute_cells_and_kzg_proofs(bytes(131072), settings)
    assert proofs == [IDENTITY] * 128 and cells == [bytes(CELL)] * 128
    blobs = [rand_blob(41), rand_blob(42), bytes(131072), rand_blob(43)]
    rc, d_c, d_p = batch_device(lib, ctx, blobs)
    assert rc == 0
    hc, hp = d_c.cpu().numpy().tobytes(), d_p.cpu().numpy().tobytes()
    for i, b in enumerate(blobs):
        ce, pr = K.compute_cells_and_kzg_proofs(b, settings)
        assert b"".join(ce) == hc[i * 128 * CELL:(i + 1) * 128 * CELL]
        assert b"".join(pr) == hp[i * 128 * 48:(i + 1) * 128 * 48]
    bad = bytearray(blobs[0]); bad[32 * 77:32 * 78] = Q.to_bytes(32, "big")
    bad_args(K, lambda: K.compute_cells_and_kzg_proofs(bytes(bad), settings))
    assert batch_device(lib, ctx, [blobs[1], bytes(bad), blobs[3]])[0] == 1
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, None, 0, None, None) == 0


# ---- recover_cells_and_kzg_proofs -----------------------------------------------------------------------------------------
def index_sets():
    rnd = random.Random(77)
    r64 = rnd.sample(range(128), 64)
    unsorted = rnd.sample(range(128), 90)
    return {"first_half": list(range(64)), "second_half": list(range(64, 128)), "random64": r64, "every_other": list(range(0, 128, 2)),
            "127": [k for k in range(128) if k != 37], "all": list(range(128)), "unsorted": unsorted}


def test_recover_patterns(K, settings):
    blobs = [rand_blob(51), rand_blob(52)]
    for bi, blob in enumerate(blobs):
        cells, proofs = K.compute_cells_and_kzg_proofs(blob, settings)
        for name, idx in index_sets().items():
            rc, rp = K.recover_cells_and_kzg_proofs(idx, [cells[k] for k in idx], settings)
            assert rc == cells, (bi, name)
            assert rp == proofs, (bi, name)


def test_recover_fixture_blob(K, settings, fixture_blobs):
    blob, c = fixture_blobs[0]
    cells, proofs = K.compute_cells_and_kzg_proofs(blob, settings)
    idx = index_sets()["random64"]
    assert K.recover_cells_and_kzg_proofs(idx, [cells[k] for k in idx], settings) == (cells, proofs)


def test_recover_inconsistent(K, settings, lib):
    """an altered element among 80 cells: the spec's bytes (the C oracle's), the proofs of the recovered blob, no error"""
    blob = rand_blob(61)
    cells = CO.compute_cells(blob)
    idx = random.Random(5).sample(range(128), 80)
    given = [cells[k] for k in idx]
    t = bytearray(given[7]); t[32 * 3 + 31] ^= 1
    given[7] = bytes(t)
    ref = CO.recover_cells(idx, given)
    assert ref is not None and ref != cells
    rc, rp = K.recover_cells_and_kzg_proofs(idx, given, settings)
    assert rc == ref
    for k in (0, 64, 127):
        assert rp[k] == CO.compute_cell_kzg_proof(b"".join(ref[:64]), k)


def test_recover_bad_args(K, settings, lib):
    blob = rand_blob(71)
    cells = CO.compute_cells(blob)
    idx = list(range(0, 128, 2))
    R = lambda i, c: K.recover_cells_and_kzg_proofs(i, c, settings)
    bad_args(K, lambda: R(idx[:63], [cells[k] for k in idx[:63]]))                      # 63 cells
    bad_args(K, lambda: R(idx[:64] + [idx[3]], [cells[k] for k in idx[:64]] + [cells[idx[3]]]))   # a duplicate index
    bad_args(K, lambda: R(idx[:63] + [128], [cells[k] for k in idx[:64]]))              # index 128
    t = bytearray(cells[idx[5]]); t[32 * 9:32 * 10] = Q.to_bytes(32, "big")
    bad_args(K, lambda: R(idx, [cells[k] for k in idx[:5]] + [bytes(t)] + [cells[k] for k in idx[6:]]))   # non-canonical
    with pytest.raises(K.KzgError) as e:
        R(idx, [cells[k] for k in idx[:63]])
    assert e.value.kind == "InvalidBytesLength"
    ctx = settings.cell_proof_context(0)
    ia = (C.c_uint64 * 129)(*range(129))
    assert lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, 129, None, 0, None, None) == 1


def test_recover_batch_shared_indices(K, settings, lib):
    import torch
    ctx = settings.cell_proof_context(0)
    nb = 6
    blobs = [rand_blob(80 + i) for i in range(nb)]
    idx = index_sets()["unsorted"]
    full = [CO.compute_cells(b) for b in blobs]
    given = b"".join(b"".join(f[k] for k in idx) for f in full)
    d_in = dev(given)
    d_c = torch.empty(nb * 128 * CELL, dtype=torch.uint8, device="cuda")
    d_p = torch.empty(nb * 128 * 48, dtype=torch.uint8, device="cuda")
    ia = (C.c_uint64 * len(idx))(*idx)
    assert lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, len(idx), d_in.data_ptr(), nb, d_c.data_ptr(), d_p.data_ptr()) == 0
    hc, hp = d_c.cpu().numpy().tobytes(), d_p.cpu().numpy().tobytes()
    for i in range(nb):
        ce, pr = K.recover_cells_and_kzg_proofs(idx, [full[i][k] for k in idx], settings)
        assert b"".join(ce) == hc[i * 128 * CELL:(i + 1) * 128 * CELL] == b"".join(full[i])
        assert b"".join(pr) == hp[i * 128 * 48:(i + 1) * 128 * 48]
    # a non-canonical element in one blob of the batch
    bad = bytearray(given); bad[3 * len(idx) * CELL + 32 * 10:3 * len(idx) * CELL + 32 * 11] = Q.to_bytes(32, "big")
    d_in = dev(bytes(bad))
    assert lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, len(idx), d_in.data_ptr(), nb, d_c.data_ptr(), d_p.data_ptr()) == 1


def test_custom_setup_proofs(K, settings, oracle):
    path = os.path.join(GOLDEN, "custom_setup.bin")
    blob = rand_blob(91)
    oracle.use_setup(path)
    try:
        mono = b"".join(oracle.tau_power_g1(j) for j in range(64))
        c = oracle.blob_to_kzg_commitment(blob)
    finally:
        oracle.use_setup(None)
    custom = K.KzgSettings.load_trusted_setup_file(path, g1_monomial_bytes=mono)
    try:
        cells, proofs = K.compute_cells_and_kzg_proofs(blob, custom)
        idx = list(range(128))
        assert K.KzgProof.verify_cell_kzg_proof_batch([c] * 128, idx, cells, proofs, custom) is True
        assert K.KzgProof.verify_cell_kzg_proof_batch([c] * 128, idx, cells, proofs, settings) is False
        r = random.Random(3).sample(range(128), 64)
        assert K.recover_cells_and_kzg_proofs(r, [cells[k] for k in r], custom) == (cells, proofs)
    finally:
        custom.close()


def test_block_recovery_composition(K, settings, lib):
    """a block of 21 blobs recovered from a random 64 columns; all 2688 recovered cells and proofs verify on the GPU"""
    import torch
    ctx = settings.cell_proof_context(0)
    nb = 21
    blobs = [rand_blob(1000 + i) for i in range(nb)]
    rc, d_c, d_p = batch_device(lib, ctx, blobs)
    assert rc == 0
    cols = sorted(random.Random(21).sample(range(128), 64))
    sel = torch.tensor(cols, device="cuda")
    given = d_c.view(nb, 128, CELL)[:, sel].contiguous()
    out_c = torch.empty_like(d_c)
    out_p = torch.empty_like(d_p)
    ia = (C.c_uint64 * 64)(*cols)
    assert lib.kzgb200_recover_cells_and_kzg_proofs_batch_device(ctx, ia, 64, given.data_ptr(), nb, out_c.data_ptr(), out_p.data_ptr()) == 0
    assert torch.equal(out_c, d_c) and torch.equal(out_p, d_p)
    # commitments of the blobs from the GPU commit path
    assert lib.kzgb200_load_g1_lagrange(ctx, settings.g1_lagrange_bytes, 4096) == 0
    d_b = dev(b"".join(blobs))
    cs = torch.empty(nb * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, d_b.data_ptr(), nb, cs.data_ptr()) == 0
    d_cm = cs.view(nb, 1, 48).expand(nb, 128, 48).contiguous().view(-1)
    d_idx = torch.arange(128, dtype=torch.int64, device="cuda").repeat(nb)
    ok = C.c_int(-1)
    assert lib.kzgb200_verify_cell_kzg_proof_batch_device(ctx, d_cm.data_ptr(), d_idx.data_ptr(), out_c.data_ptr(), out_p.data_ptr(), nb * 128,
                                                          C.byref(ok)) == 0
    assert ok.value == 1
