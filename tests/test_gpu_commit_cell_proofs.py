"""compute_commitments_and_cell_proofs on the GPU (pytest -m gpu): a publisher's commitment and 128 cell proofs per blob from one FK20
pass.  The commitments are compared byte for byte with the commit path (kzgb200_blob_to_kzg_commitment_batch), the c-kzg vectors,
the CPU oracle and the derived monomial points; the proofs and cells with compute_cells_and_kzg_proofs."""
import ctypes as C
import os
import random

import pytest
from conftest import GOLDEN, unhex

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
OMEGA = pow(7, (Q - 1) // 4096, Q)
IDENTITY = b"\xc0" + bytes(47)
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


def monomial_blob(m):
    """the blob of X^m: evaluations at omega^rev12(i), i < 4096"""
    return b"".join(pow(OMEGA, m * int(format(i, "012b")[::-1], 2), Q).to_bytes(32, "big") for i in range(4096))


def dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


def host_call(lib, ctx, blobs, want_cells):
    n = len(blobs)
    cm, pr = C.create_string_buffer(48 * max(n, 1)), C.create_string_buffer(BLOB_PROOFS * max(n, 1))
    ce = C.create_string_buffer(BLOB_CELLS * max(n, 1)) if want_cells else None
    st = C.create_string_buffer(max(n, 1))
    rc = lib.kzgb200_compute_commitments_and_cell_proofs(ctx, b"".join(blobs), n, cm, pr, ce, st)
    return rc, cm.raw[:48 * n], pr.raw[:BLOB_PROOFS * n], ce.raw[:BLOB_CELLS * n] if want_cells else None, st.raw[:n]


def device_call(lib, ctx, d_blobs, n, want_cells):
    import torch
    cm = torch.empty(48 * n, dtype=torch.uint8, device="cuda")
    pr = torch.empty(BLOB_PROOFS * n, dtype=torch.uint8, device="cuda")
    ce = torch.empty(BLOB_CELLS * n, dtype=torch.uint8, device="cuda") if want_cells else None
    st = C.create_string_buffer(n)
    rc = lib.kzgb200_compute_commitments_and_cell_proofs_device(ctx, d_blobs.data_ptr(), n, cm.data_ptr(), pr.data_ptr(),
                                                                 ce.data_ptr() if want_cells else None, st)
    torch.cuda.synchronize()
    return rc, cm, pr, ce, st.raw


def test_600_random_blobs_equal_the_commit_path_and_the_proof_batch(K, settings, lib):
    """600 uniformly random blobs (crossing the 512-blob pass): commitments = kzgb200_blob_to_kzg_commitment_batch, proofs and cells =
    kzgb200_compute_cells_and_kzg_proofs_batch_device, byte for byte, in the device form and the host form"""
    import torch
    n = 600
    g = torch.Generator(device="cuda").manual_seed(600)
    d = torch.randint(0, 256, (n * 4096, 32), dtype=torch.uint8, device="cuda", generator=g)
    d[:, 0] &= 0x3f                                   # every element < 2^254 < q: canonical, full degree
    d_blobs = d.view(-1).contiguous()
    ctx = settings.commit_context(0)
    assert settings.cell_proof_context(0).value == ctx.value
    want_c = torch.empty(48 * n, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, d_blobs.data_ptr(), n, want_c.data_ptr()) == 0
    want_ce = torch.empty(BLOB_CELLS * n, dtype=torch.uint8, device="cuda")
    want_p = torch.empty(BLOB_PROOFS * n, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, d_blobs.data_ptr(), n, want_ce.data_ptr(), want_p.data_ptr()) == 0
    torch.cuda.synchronize()
    rc, cm, pr, ce, st = device_call(lib, ctx, d_blobs, n, True)
    assert rc == 0 and st == bytes(n)
    assert torch.equal(cm, want_c) and torch.equal(pr, want_p) and torch.equal(ce, want_ce)
    rc, cm, pr, _, st = device_call(lib, ctx, d_blobs, n, False)
    assert rc == 0 and st == bytes(n) and torch.equal(cm, want_c) and torch.equal(pr, want_p)
    raw = d_blobs.cpu().numpy().tobytes()
    rc, hcm, hpr, _, st = host_call(lib, ctx, [raw[131072 * b:131072 * (b + 1)] for b in range(n)], False)
    assert rc == 0 and st == bytes(n)
    assert hcm == want_c.cpu().numpy().tobytes() and hpr == want_p.cpu().numpy().tobytes()


def test_commitments_of_the_ckzg_vectors(K, settings, vectors, oracle):
    """every stored blob the oracle accepts: the host form's commitments equal the oracle's and those of the vectors' true cases"""
    good = [(i, b) for i, b in enumerate(vectors.blobs) if len(b) == 131072 and oracle.blob_to_kzg_commitment(b) is not None]
    assert len(good) >= 7
    out = K.compute_commitments_and_cell_proofs([b for _, b in good], settings)
    by_index = {i: r[0] for (i, _), r in zip(good, out)}
    for i, b in good:
        assert by_index[i] == oracle.blob_to_kzg_commitment(b), i
    cases = [c for c in vectors["verify_blob_kzg_proof"] if c["output"] is True]
    assert cases
    for c in cases:
        assert by_index[c["blob"]] == unhex(c["commitment"]), c["name"]


def test_monomial_blobs_hit_the_new_table_entry(K, settings, lib):
    """X^m for m = 4032 (w_b[65] alone), 4095, 4031 and 0: the commitment is the derived monomial point m; the zero blob gives the
    identity for the commitment and all 128 proofs"""
    ctx = settings.cell_proof_context(0)
    mono = C.create_string_buffer(4096 * 48)
    assert lib.kzgb200_cell_proof_monomial(ctx, mono, 4096) == 0
    ms = [4032, 4095, 4031, 0]
    out = K.compute_commitments_and_cell_proofs([monomial_blob(m) for m in ms] + [bytes(131072)], settings, want_cells=True)
    for m, (c, cells, proofs) in zip(ms, out):
        assert c == mono.raw[48 * m:48 * (m + 1)], m
        assert (cells, proofs) == K.compute_cells_and_kzg_proofs(monomial_blob(m), settings), m
    c, cells, proofs = out[-1]
    assert c == IDENTITY and proofs == [IDENTITY] * 128 and cells == [bytes(CELL)] * 128


def test_per_blob_status_and_calls_before_the_proof_setup(K, settings, lib):
    good = [rand_blob(41), rand_blob(42)]
    bad = bytearray(rand_blob(43))
    bad[32 * 1000:32 * 1001] = Q.to_bytes(32, "big")
    blobs = [good[0], bytes(bad), good[1], bytes(131072)]
    ctx = settings.cell_proof_context(0)
    rc, cm, pr, ce, st = host_call(lib, ctx, blobs, True)
    assert rc == 0 and st == b"\x00\x01\x00\x00"
    for b in (0, 2):
        c1 = K.compute_cells_and_kzg_proofs(blobs[b], settings)
        assert ce[BLOB_CELLS * b:BLOB_CELLS * (b + 1)] == b"".join(c1[0]) and pr[BLOB_PROOFS * b:BLOB_PROOFS * (b + 1)] == b"".join(c1[1])
        assert cm[48 * b:48 * (b + 1)] == K.blob_to_kzg_commitment(blobs[b], settings)
    assert cm[144:192] == IDENTITY
    rc, dcm, dpr, dce, dst = device_call(lib, ctx, dev(b"".join(blobs)), 4, True)
    assert rc == 0 and dst == st
    for b in (0, 2, 3):
        assert dcm[48 * b:48 * (b + 1)].cpu().numpy().tobytes() == cm[48 * b:48 * (b + 1)]
        assert dpr[BLOB_PROOFS * b:BLOB_PROOFS * (b + 1)].cpu().numpy().tobytes() == pr[BLOB_PROOFS * b:BLOB_PROOFS * (b + 1)]
    out = K.compute_commitments_and_cell_proofs(blobs, settings)
    assert out[1] is None and [r[0] for r in out if r] == [cm[0:48], cm[96:144], IDENTITY]
    with pytest.raises(K.KzgError) as e:
        K.blob_to_kzg_commitment(blobs[1], settings)
    assert e.value.kind == "BadArgs"
    # a context without the proof setup: INVALID_SETUP (5) in both forms, OK with nothing to do
    fresh = K.KzgSettings(settings.g1_lagrange_bytes, settings.g2_monomial_bytes)      # its own contexts
    try:
        for c in (fresh.context(0), fresh.cell_context(0)):
            assert host_call(lib, c, good[:1], False)[0] == 5
            assert device_call(lib, c, dev(good[0]), 1, False)[0] == 5
            assert lib.kzgb200_compute_commitments_and_cell_proofs(c, None, 0, None, None, None, None) == 0
    finally:
        fresh.close()


def test_round_trip_through_the_blob_cell_verifier(K, settings):
    txs = [[rand_blob(500 + 10 * t + i) for i in range(n)] for t, n in enumerate((1, 6, 3))]
    built = []
    for blobs in txs:
        out = K.compute_commitments_and_cell_proofs(blobs, settings)
        cs, ps = [r[0] for r in out], [p for r in out for p in r[1]]
        assert K.KzgProof.verify_blob_cell_kzg_proof_batch(blobs, cs, ps, settings) is True
        built.append((blobs, cs, ps))
    blobs, cs, ps = built[1]
    swapped = [cs[1], cs[0]] + cs[2:]
    assert K.KzgProof.verify_blob_cell_kzg_proof_batch(blobs, swapped, ps, settings) is False
    assert K.KzgProof.verify_blob_cell_kzg_proof_batch_many(built, settings) == [True, True, True]


def test_custom_setup(K, settings, oracle):
    path = os.path.join(GOLDEN, "custom_setup.bin")
    blobs = [rand_blob(91), rand_blob(92)]
    oracle.use_setup(path)
    try:
        mono = b"".join(oracle.tau_power_g1(j) for j in range(64))
        want = [oracle.blob_to_kzg_commitment(b) for b in blobs]
    finally:
        oracle.use_setup(None)
    custom = K.KzgSettings.load_trusted_setup_file(path, g1_monomial_bytes=mono)
    try:
        out = K.compute_commitments_and_cell_proofs(blobs, custom)
        assert [r[0] for r in out] == want
        assert K.KzgProof.verify_blob_cell_kzg_proof_batch(blobs, want, [p for r in out for p in r[1]], custom) is True
    finally:
        custom.close()
    assert want != [r[0] for r in K.compute_commitments_and_cell_proofs(blobs, settings)]


@pytest.mark.parametrize("n", [1, 6])
def test_host_and_device_forms_agree(K, settings, lib, n):
    blobs = [rand_blob(800 + n + i) for i in range(n)]
    ctx = settings.cell_proof_context(0)
    for want_cells in (False, True):
        rc, cm, pr, ce, st = host_call(lib, ctx, blobs, want_cells)
        assert rc == 0 and st == bytes(n)
        rc, dcm, dpr, dce, dst = device_call(lib, ctx, dev(b"".join(blobs)), n, want_cells)
        assert rc == 0 and dst == bytes(n)
        assert dcm.cpu().numpy().tobytes() == cm and dpr.cpu().numpy().tobytes() == pr
        if want_cells:
            assert dce.cpu().numpy().tobytes() == ce
    cells, proofs = K.compute_cells_and_kzg_proofs(blobs[0], settings)
    commitment = K.blob_to_kzg_commitment(blobs[0], settings)
    assert K.compute_commitments_and_cell_proofs(blobs[:1], settings, want_cells=True) == [(commitment, cells, proofs)]
    assert K.compute_commitments_and_cell_proofs(blobs[:1], settings) == [(commitment, proofs)]
    assert cm[:48] == commitment and pr[:BLOB_PROOFS] == b"".join(proofs) and ce[:BLOB_CELLS] == b"".join(cells)
