"""The batch verifier's split tail (per-window Miller loops on the [256^w]-scaled G2 lines, KZGB200_FINAL_SPLIT=1, the default)
against the Horner + one-pairing tail (KZGB200_FINAL_SPLIT=0), two contexts in one process: same verdicts, z, y and BadArgs on
valid, false and malformed batches, on all-identity proofs and under a custom setup; the same GT element on false batches; and
the shifted line tables equal the CPU's prepare_g2 of [256^w]Q (tools/hosttest/final_split_host.cu)."""
import ctypes as C
import os
import shutil
import subprocess

import pytest
from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
ONE_GT = b"\x01" + b"\x00" * 575


@pytest.fixture(scope="module")
def K():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import kzg_rs_b200 as K
    return K


def make_pair(K, g2):
    """(split context, Horner context) on cuda:0 for the setup's first two G2 points"""
    lib = K.Library.get().dll
    out = []
    for split in ("1", "0"):
        os.environ["KZGB200_FINAL_SPLIT"] = split
        h = C.c_void_p()
        assert lib.kzgb200_create(C.byref(h), 0, g2[:192], 192) == 0
        out.append(h)
    os.environ.pop("KZGB200_FINAL_SPLIT")
    return out


@pytest.fixture(scope="module")
def ctxs(K):
    S = K.KzgSettings.load_trusted_setup_file()
    pair = make_pair(K, S.g2_monomial_bytes)
    yield pair
    for h in pair:
        K.Library.get().dll.kzgb200_destroy(h)


def harness(K, ctx, n, seed):
    import torch
    lib = K.Library.get().dll
    tau = open(os.path.join(os.path.dirname(K.__file__), "data", "tau_powers_g1.bin"), "rb").read()
    b = torch.empty(n * 131072, dtype=torch.uint8, device="cuda")
    c = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    p = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_harness_generate(ctx, seed, n, 8, tau, b.data_ptr(), c.data_ptr(), p.data_ptr()) == 0
    torch.cuda.synchronize()
    return b, c, p


def run(K, ctx, b, c, p, n):
    """(rc, verdict, z bytes, y bytes, GT bytes) of one resident batch call"""
    import torch
    lib = K.Library.get().dll
    z = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
    y = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
    ok = C.c_int(-1)
    rc = lib.kzgb200_verify_blob_kzg_proof_batch_device(ctx, b.data_ptr(), c.data_ptr(), p.data_ptr(), n, C.byref(ok), z.data_ptr(), y.data_ptr())
    gt = C.create_string_buffer(576)
    assert lib.kzgb200_debug_last_gt(ctx, gt) == 0
    torch.cuda.synchronize()
    return rc, ok.value, z.cpu().numpy().tobytes(), y.cpu().numpy().tobytes(), gt.raw


def both(K, ctxs, b, c, p, n):
    r_split, r_old = (run(K, h, b, c, p, n) for h in ctxs)
    assert r_split[:4] == r_old[:4]
    return r_split, r_old


@pytest.mark.parametrize("n", [2, 64, 2048, 16384])
def test_valid_batches(K, ctxs, n):
    b, c, p = harness(K, ctxs[0], n, 0x5117 + n)
    s, o = both(K, ctxs, b, c, p, n)
    assert s[0] == 0 and s[1] == 1 and s[4] == ONE_GT == o[4]


def test_false_batches_same_gt(K, ctxs):
    n = 64
    b, c, p = harness(K, ctxs[0], n, 0xfa15e)
    swapped = p.clone()
    swapped[:48], swapped[48:96] = p[48:96].clone(), p[:48].clone()
    s, o = both(K, ctxs, b, c, swapped, n)
    assert s[:2] == (0, 0) and s[4] == o[4] != ONE_GT
    tampered = b.clone()                                   # another blob element: y of blob 5 changes, its proof does not
    tampered[5 * 131072 + 31] ^= 1
    s, o = both(K, ctxs, tampered, c, p, n)
    assert s[:2] == (0, 0) and s[4] == o[4] != ONE_GT


def test_bad_args(K, ctxs):
    import torch
    from kzg_rs_b200.sharded import NOT_IN_G1
    n = 64
    b, c, p = harness(K, ctxs[0], n, 0xbad)
    bq = b.clone()
    bq[3 * 131072 + 7 * 32:3 * 131072 + 8 * 32] = torch.tensor(list(Q.to_bytes(32, "big")), dtype=torch.uint8, device="cuda")
    s, _ = both(K, ctxs, bq, c, p, n)
    assert s[0] == 1                                        # KZGB200_BAD_ARGS
    cs = c.clone()
    cs[11 * 48:12 * 48] = torch.tensor(list(NOT_IN_G1), dtype=torch.uint8, device="cuda")
    s, _ = both(K, ctxs, b, cs, p, n)
    assert s[0] == 1


def test_all_identity(K, ctxs):
    """zero blobs, identity commitments and proofs: every window is the identity, every Miller value 1"""
    import torch
    n = 64
    b = torch.zeros(n * 131072, dtype=torch.uint8, device="cuda")
    ident = torch.tensor(list(b"\xc0" + b"\x00" * 47) * n, dtype=torch.uint8, device="cuda")
    s, o = both(K, ctxs, b, ident, ident, n)
    assert s[:2] == (0, 1) and s[4] == o[4] == ONE_GT
    b2, c2, _ = harness(K, ctxs[0], n, 0x1de)             # identity proofs of nonzero blobs: false
    s, o = both(K, ctxs, b2, c2, ident, n)
    assert s[:2] == (0, 0) and s[4] == o[4] != ONE_GT


def test_custom_setup(K):
    import torch
    custom = K.KzgSettings.load_trusted_setup_file(os.path.join(GOLDEN, "custom_setup.bin"))
    pair = make_pair(K, custom.g2_monomial_bytes)
    lib = K.Library.get().dll
    try:
        assert lib.kzgb200_load_g1_lagrange(pair[0], custom.g1_lagrange_bytes, 4096) == 0
        n = 48
        g = torch.Generator(device="cuda").manual_seed(11)
        b = torch.randint(0, 256, (n * 131072,), dtype=torch.uint8, device="cuda", generator=g)
        b.view(n * 4096, 32)[:, 0] &= 0x3f
        c = torch.empty(n * 48, dtype=torch.uint8, device="cuda"); p = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        assert lib.kzgb200_blob_to_kzg_commitment_batch(pair[0], b.data_ptr(), n, c.data_ptr()) == 0
        assert lib.kzgb200_compute_blob_kzg_proof_batch(pair[0], b.data_ptr(), c.data_ptr(), n, p.data_ptr()) == 0
        s, o = both(K, pair, b, c, p, n)
        assert s[:2] == (0, 1)
        p2 = p.clone(); p2[:48], p2[48:96] = p[48:96].clone(), p[:48].clone()
        s, o = both(K, pair, b, c, p2, n)
        assert s[:2] == (0, 0) and s[4] == o[4]
    finally:
        for h in pair:
            lib.kzgb200_destroy(h)


@pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not found")
@pytest.mark.parametrize("setup", ["mainnet", "custom"])
def test_shifted_line_tables_match_cpu(K, ctxs, tmp_path, setup):
    path = os.path.join(ROOT, "kzg_rs_b200", "data", "mainnet_setup.bin") if setup == "mainnet" else os.path.join(GOLDEN, "custom_setup.bin")
    exe = str(tmp_path / "final_split_host")
    subprocess.check_call(["nvcc", "-std=c++17", "-O1", "-x", "cu", "-I", os.path.join(ROOT, "kzg_rs_b200", "csrc"),
                           os.path.join(ROOT, "tools", "hosttest", "final_split_host.cu"), "-o", exe], stderr=subprocess.DEVNULL)
    want = bytes.fromhex(subprocess.run([exe, "lines", path], capture_output=True, text=True, check=True, timeout=1800).stdout.strip())
    lib = K.Library.get().dll
    if setup == "mainnet":
        ctx, pair = ctxs[0], None
    else:
        pair = make_pair(K, K.KzgSettings.load_trusted_setup_file(path).g2_monomial_bytes)
        ctx = pair[0]
    try:
        got = C.create_string_buffer(len(want))
        assert len(want) == 2 * 15 * 68 * 6 * 64
        assert lib.kzgb200_debug_lines29w(ctx, got, len(want)) == 0
        assert got.raw == want
    finally:
        for h in pair or ():
            lib.kzgb200_destroy(h)
