"""EIP-7594 cells on the GPU (pytest -m gpu): compute_cells and verify_cell_kzg_proof_batch through the C ABI and the Python
API, against the CPU cell oracle (verdicts, r, cells bit-exact), at scale on the cell workload generator, under a custom setup, and
composed as the mempool path (compute_cells -> verify 128 cell proofs per blob)."""
import ctypes as C
import os
import random

import pytest
from conftest import GOLDEN, ROOT, unhex

from cell_oracle import cells as CO

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
DATA = os.path.join(ROOT, "kzg_rs_b200", "data")
CELL = 2048


@pytest.fixture(scope="module")
def K():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import kzg_rs_b200 as K
    return K


@pytest.fixture(scope="module")
def settings(K):
    s = K.KzgSettings.load_trusted_setup_file()
    s.cell_context(0)
    return s


@pytest.fixture(scope="module")
def lib(K):
    return K.Library.get().dll


@pytest.fixture(scope="module")
def fixture_blobs(vectors):
    """full-degree fixture blobs (4096 distinct elements) with their fixture commitments (the valid verify_blob_kzg_proof cases)"""
    out = []
    for c in vectors["verify_blob_kzg_proof"]:
        b = vectors.blobs[c["blob"]]
        full = len(b) == 131072 and len({b[32 * i:32 * i + 32] for i in range(4096)}) == 4096
        if c["output"] is True and full and (b, unhex(c["commitment"])) not in out:
            out.append((b, unhex(c["commitment"])))
    assert len(out) >= 2
    return out


_PROOFS = {}


def proof(oracle, blob, k):
    if (blob, k) not in _PROOFS:
        _PROOFS[(blob, k)] = CO.compute_cell_kzg_proof(blob, k)
    return _PROOFS[(blob, k)]


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))


def last_r(lib, ctx):
    r = C.create_string_buffer(32)
    assert lib.kzgb200_last_r(ctx, r) == 0
    return r.raw


def tri(K, fn):
    try:
        return fn()
    except K.KzgError as e:
        assert e.kind == "BadArgs", e.kind
        return None


def gen_cells(K, settings, n_blobs, seed, degree=192):
    """cell workload generator: (cells, commitments, proofs) device tensors; cells / proofs blob-major, 128 per blob"""
    import torch
    lib, ctx = K.Library.get().dll, settings.cell_context(0)
    tau = K.api.mainnet_g1_monomial()[:degree * 48]
    cells = torch.empty(n_blobs * 128 * CELL, dtype=torch.uint8, device="cuda")
    cs = torch.empty(n_blobs * 48, dtype=torch.uint8, device="cuda")
    ps = torch.empty(n_blobs * 128 * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_harness_generate_cells(ctx, seed, n_blobs, degree, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
    torch.cuda.synchronize()
    return cells, cs, ps


def verify_device(K, settings, d_c, d_idx, d_cells, d_p, n):
    lib, ctx, ok = K.Library.get().dll, settings.cell_context(0), C.c_int(-1)
    rc = lib.kzgb200_verify_cell_kzg_proof_batch_device(ctx, d_c.data_ptr(), d_idx.data_ptr(), d_cells.data_ptr(), d_p.data_ptr(), n, C.byref(ok))
    return rc, ok.value


def test_compute_cells_matches_oracle(K, settings, lib, oracle, fixture_blobs, vectors):
    import torch
    blobs = [b for b in vectors.blobs if len(b) == 131072 and CO.compute_cells(b) is not None]
    blobs += [rand_blob(s) for s in (1, 2, 3)]
    for b in blobs:
        assert K.compute_cells(b, settings) == CO.compute_cells(b)
    # device batch form, blob-major output
    n = 4
    d_b = torch.frombuffer(bytearray(b"".join(blobs[-n:])), dtype=torch.uint8).cuda()
    d_out = torch.empty(n * 128 * CELL, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_compute_cells_batch_device(settings.cell_context(0), d_b.data_ptr(), n, d_out.data_ptr()) == 0
    assert d_out.cpu().numpy().tobytes() == b"".join(b"".join(CO.compute_cells(b)) for b in blobs[-n:])
    bad = bytearray(blobs[-1]); bad[32 * 4000:32 * 4001] = Q.to_bytes(32, "big")
    assert tri(K, lambda: K.compute_cells(bytes(bad), settings)) is None
    d_b[131072 * 2 + 32 * 7:131072 * 2 + 32 * 8] = torch.tensor(list(Q.to_bytes(32, "big")), dtype=torch.uint8)
    assert lib.kzgb200_compute_cells_batch_device(settings.cell_context(0), d_b.data_ptr(), n, d_out.data_ptr()) == 1


def test_cell_setup_required(K, settings, lib):
    fresh = K.KzgSettings(settings.g1_lagrange_bytes, settings.g2_monomial_bytes)
    try:
        ctx, ok = fresh.context(0), C.c_int()
        out = C.create_string_buffer(128 * CELL)
        assert lib.kzgb200_compute_cells(ctx, bytes(131072), out) == 5
        assert lib.kzgb200_verify_cell_kzg_proof_batch(ctx, None, None, None, None, 0, C.byref(ok)) == 5
    finally:
        fresh.close()


def _cases(oracle, fixture_blobs):
    (b0, c0), (b1, c1) = fixture_blobs[0], fixture_blobs[1]
    cells0, cells1 = CO.compute_cells(b0), CO.compute_cells(b1)
    e = lambda b, c, cells, k: (c, k, cells[k], proof(oracle, b, k))
    cases = {
        "n1": [e(b0, c0, cells0, 77)],
        "whole_blob": [e(b0, c0, cells0, k) for k in range(128)],
        "column": [e(b, c, CO.compute_cells(b), 9) for b, c in fixture_blobs[:4]],
        "dup_commitments_apart": [e(b0, c0, cells0, 3), e(b1, c1, cells1, 100), e(b0, c0, cells0, 64), e(b1, c1, cells1, 1)],
        "repeated_cell": [e(b1, c1, cells1, 50), e(b0, c0, cells0, 2), e(b1, c1, cells1, 50)],
    }
    return cases, (b0, c0, cells0), (b1, c1, cells1)


def test_verify_valid_and_r(K, settings, lib, oracle, fixture_blobs):
    cases, _, _ = _cases(oracle, fixture_blobs)
    ctx = settings.cell_context(0)
    for name, es in cases.items():
        cs, idx, ce, ps = (list(x) for x in zip(*es))
        ok, r = CO.verify_cell_kzg_proof_batch(cs, idx, ce, ps, want_r=True)
        assert ok is True, name
        assert K.KzgProof.verify_cell_kzg_proof_batch(cs, idx, ce, ps, settings) is True, name
        assert last_r(lib, ctx) == r, name
        assert K.KzgProof.verify_cell_kzg_proof_batch(cs, idx, [K.Cell.from_slice(x) for x in ce], [K.Bytes48.from_slice(p) for p in ps], settings) is True


def test_verify_tampered_and_bad_args(K, settings, lib, oracle, fixture_blobs):
    cases, (b0, c0, cells0), (b1, c1, cells1) = _cases(oracle, fixture_blobs)
    cs, idx, ce, ps = (list(x) for x in zip(*cases["dup_commitments_apart"]))
    V = lambda *a: tri(K, lambda: K.KzgProof.verify_cell_kzg_proof_batch(*a, settings))
    ctx = settings.cell_context(0)
    t = bytearray(ce[2]); t[32 * 10 + 31] ^= 1
    false_cases = [
        (cs, idx, ce, [ps[1], ps[0]] + ps[2:]),                    # a proof swapped between two cells
        (cs, idx, ce[:2] + [bytes(t)] + ce[3:], ps),               # one element changed
        (cs, [3, 100, 65, 1], ce, ps),                             # a wrong cell index
        ([c0, c0] + cs[2:], idx, ce, ps),                          # another blob's commitment
    ]
    for args in false_cases:
        ok, r = CO.verify_cell_kzg_proof_batch(*args, want_r=True)
        assert ok is False
        assert V(*args) is False
        assert last_r(lib, ctx) == r
    t = bytearray(ce[1]); t[32 * 63:32 * 64] = Q.to_bytes(32, "big")
    for args in [(cs, idx, [ce[0], bytes(t)] + ce[2:], ps),     # element == q
                 (cs, [3, 100, 64, 128], ce, ps),                # cell index 128
                 (cs[:3] + [bytes(48)], idx, ce, ps),            # invalid commitment bytes
                 (cs, idx, ce, [ps[0], b"\xc0" + bytes(46) + b"\x01"] + ps[2:])]:   # invalid proof bytes
        assert CO.verify_cell_kzg_proof_batch(*args) is None
        assert V(*args) is None
    assert K.KzgProof.verify_cell_kzg_proof_batch([], [], [], [], settings) is True
    with pytest.raises(K.KzgError) as e:
        K.KzgProof.verify_cell_kzg_proof_batch(cs, idx[:3], ce, ps, settings)
    assert e.value.kind == "InvalidBytesLength"
    with pytest.raises(K.KzgError) as e:
        K.KzgProof.verify_cell_kzg_proof_batch(cs, idx, ce, ps[:3], settings)
    assert e.value.kind == "InvalidBytesLength"


def test_harness_cells_agree_with_oracle_and_compute_cells(K, settings, oracle):
    cells, cs, ps = gen_cells(K, settings, 2, 0x7594)
    hc, hcs, hps = (t.cpu().numpy().tobytes() for t in (cells, cs, ps))
    blob = hc[:131072]
    assert CO.compute_cells(blob) == [hc[CELL * k:CELL * (k + 1)] for k in range(128)]
    assert oracle.blob_to_kzg_commitment(blob) == hcs[:48]
    ks = [0, 5, 64, 127]
    assert CO.verify_cell_kzg_proof_batch([hcs[48:96]] * 4, ks, [hc[CELL * (128 + k):CELL * (129 + k)] for k in ks],
                                              [hps[48 * (128 + k):48 * (129 + k)] for k in ks]) is True
    assert CO.compute_cell_kzg_proof(blob, 5) == hps[48 * 5:48 * 6]


def test_scale_16384_cells(K, settings, lib):
    import torch
    from oracle import pyref as R
    nb = 128
    cells, cs, ps = gen_cells(K, settings, nb, 11)
    n = nb * 128
    d_c = cs.view(nb, 1, 48).expand(nb, 128, 48).contiguous().view(-1)
    d_idx = torch.arange(128, dtype=torch.int64, device="cuda").repeat(nb)
    assert verify_device(K, settings, d_c, d_idx, cells, ps, n) == (0, 1)
    # the host entry point on the same batch: same verdict, same r
    r_dev = last_r(lib, settings.cell_context(0))
    hc, hi, hce, hp = (t.cpu().numpy().tobytes() for t in (d_c, d_idx, cells, ps))
    ok = C.c_int(-1)
    assert lib.kzgb200_verify_cell_kzg_proof_batch(settings.cell_context(0), hc, hi, hce, hp, n, C.byref(ok)) == 0 and ok.value == 1
    assert last_r(lib, settings.cell_context(0)) == r_dev
    # one proof replaced by pi + G
    j = 12345
    pi = R.g1_from_compressed(hp[48 * j:48 * j + 48])[1]
    bad = R.g1_to_compressed(R.g1_add(pi, R.G1_GEN))
    ps2 = ps.clone()
    ps2[48 * j:48 * j + 48] = torch.tensor(list(bad), dtype=torch.uint8)
    assert verify_device(K, settings, d_c, d_idx, cells, ps2, n) == (0, 0)


def test_custom_setup_cells(K, settings, oracle):
    path = os.path.join(GOLDEN, "custom_setup.bin")
    blob = rand_blob(21)
    oracle.use_setup(path)
    CO.use_setup(path)
    try:
        mono = b"".join(oracle.tau_power_g1(j) for j in range(64))
        c = oracle.blob_to_kzg_commitment(blob)
        cells = CO.compute_cells(blob)
        ks = [0, 33, 64, 101]
        ps = [CO.compute_cell_kzg_proof(blob, k) for k in ks]
        assert CO.verify_cell_kzg_proof_batch([c] * 4, ks, [cells[k] for k in ks], ps) is True
    finally:
        oracle.use_setup(None)
        CO.use_setup(None)
    custom = K.KzgSettings.load_trusted_setup_file(path, g1_monomial_bytes=mono)
    try:
        args = ([c] * 4, ks, [cells[k] for k in ks], ps)
        assert K.KzgProof.verify_cell_kzg_proof_batch(*args, custom) is True
        assert K.KzgProof.verify_cell_kzg_proof_batch(*args, settings) is False          # the mainnet context says no
        mb = rand_blob(22)
        mc, mcells = oracle.blob_to_kzg_commitment(mb), CO.compute_cells(mb)
        margs = ([mc] * 2, [7, 90], [mcells[7], mcells[90]], [CO.compute_cell_kzg_proof(mb, 7), CO.compute_cell_kzg_proof(mb, 90)])
        assert K.KzgProof.verify_cell_kzg_proof_batch(*margs, settings) is True
        assert K.KzgProof.verify_cell_kzg_proof_batch(*margs, custom) is False           # mainnet data under the custom setup
        with pytest.raises(K.KzgError) as e:
            K.KzgProof.verify_cell_kzg_proof_batch(*args, K.KzgSettings.load_trusted_setup_file(path))
        assert e.value.kind == "InvalidTrustedSetup"                                      # no monomial points for this setup
    finally:
        custom.close()


def test_gpu_commit_reproduces_monomial_points(K, settings, lib):
    """[tau^j]G1 is the commitment to X^j, whose evaluation form is the blob of omega_i^j: the GPU commit path over the
    Lagrange setup reproduces the shipped monomial points 0..63"""
    import torch
    from oracle import pyref as R
    ctx = settings.context(0)
    assert lib.kzgb200_load_g1_lagrange(ctx, settings.g1_lagrange_bytes, 4096) == 0
    roots = R.roots_of_unity()
    n = 64
    blobs = b"".join(b"".join(pow(w, j, Q).to_bytes(32, "big") for w in roots) for j in range(n))
    d_b = torch.frombuffer(bytearray(blobs), dtype=torch.uint8).cuda()
    d_c = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, d_b.data_ptr(), n, d_c.data_ptr()) == 0
    assert d_c.cpu().numpy().tobytes() == K.api.mainnet_g1_monomial()[:n * 48]


def test_mempool_compute_cells_then_verify(K, settings, lib):
    """blobs -> GPU compute_cells -> verify all 128 cell proofs per blob (proofs from the workload generator)"""
    import torch
    nb = 8
    cells, cs, ps = gen_cells(K, settings, nb, 99)
    blobs = cells.view(nb, 128 * CELL)[:, :64 * CELL].contiguous()
    out = torch.empty(nb * 128 * CELL, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_compute_cells_batch_device(settings.cell_context(0), blobs.data_ptr(), nb, out.data_ptr()) == 0
    assert torch.equal(out, cells)
    d_c = cs.view(nb, 1, 48).expand(nb, 128, 48).contiguous().view(-1)
    d_idx = torch.arange(128, dtype=torch.int64, device="cuda").repeat(nb)
    assert verify_device(K, settings, d_c, d_idx, out, ps, nb * 128) == (0, 1)
    # a single column across the blobs (one data column sidecar)
    col = 17
    sel = torch.arange(nb, device="cuda") * 128 + col
    c_col = cs.view(nb, 48).contiguous().view(-1)
    cells_col = out.view(-1, CELL)[sel].contiguous().view(-1)
    ps_col = ps.view(-1, 48)[sel].contiguous().view(-1)
    idx_col = torch.full((nb,), col, dtype=torch.int64, device="cuda")
    assert verify_device(K, settings, c_col, idx_col, cells_col, ps_col, nb) == (0, 1)
