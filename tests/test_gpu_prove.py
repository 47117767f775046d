"""EIP-4844 publisher calls on the GPU (pytest -m gpu): blob_to_kzg_commitment, compute_kzg_proof and compute_blob_kzg_proof,
host and device-batch forms, against the c-kzg vectors and the CPU oracle.  The batch sizes sit on both sides of the slice choice
of the commitment MSM (one blob over every SM ... one CTA per blob) and across the 1024-blob chunk."""
import os
import random
import subprocess

import pytest
from conftest import GOLDEN, ROOT, unhex

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
IDENTITY = b"\xc0" + bytes(47)
OMEGA = pow(7, (Q - 1) // 4096, Q)          # the spec's primitive 4096th root of unity (PRIMITIVE_ROOT_OF_UNITY = 7)


def be32(x):
    return x.to_bytes(32, "big")


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(be32(rnd.randrange(Q)) for _ in range(4096))


@pytest.fixture(scope="module")
def K():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import kzg_rs_b200 as K
    return K


@pytest.fixture(scope="module")
def settings(K):
    s = K.KzgSettings.load_trusted_setup_file()
    s.commit_context(0)
    return s


def bad_args(K, fn):
    with pytest.raises(K.KzgError) as e:
        fn()
    assert e.value.kind == "BadArgs"


def valid_blobs(vectors, oracle):
    """(index, blob, oracle commitment) of every stored 131072-byte blob the oracle accepts."""
    out = []
    for i, b in enumerate(vectors.blobs):
        if len(b) == 131072:
            c = oracle.blob_to_kzg_commitment(b)
            if c is not None:
                out.append((i, b, c))
    return out


def test_compute_kzg_proof_reproduces_every_true_verify_kzg_proof_vector(K, settings, vectors, oracle):
    """The 54 true verify_kzg_proof cases, proof and y byte for byte; each case's blob is the stored blob with its commitment.
    Their z include 0, 1, 2, -1 and a 4096th root of unity."""
    by_c = {c: b for _, b, c in valid_blobs(vectors, oracle)}
    cases = [c for c in vectors["verify_kzg_proof"] if c["output"] is True]
    assert len(cases) == 54
    zs = set()
    for c in cases:
        blob = by_c[unhex(c["commitment"])]
        proof, y = K.compute_kzg_proof(blob, unhex(c["z"]), settings)
        assert proof == unhex(c["proof"]) and y == unhex(c["y"]), c["name"]
        zs.add(int(c["z"], 16))
    assert {0, 1, 2, Q - 1} <= zs and any(z not in (0, 1, 2, Q - 1) and pow(z, 4096, Q) == 1 for z in zs)


def test_blob_to_kzg_commitment_on_every_stored_blob(K, settings, vectors, oracle):
    n_valid = n_bad = 0
    for i, b in enumerate(vectors.blobs):
        if len(b) != 131072:
            with pytest.raises(K.KzgError) as e:
                K.blob_to_kzg_commitment(b, settings)
            assert e.value.kind == "InvalidBytesLength"
            continue
        want = oracle.blob_to_kzg_commitment(b)
        if want is None:
            bad_args(K, lambda: K.blob_to_kzg_commitment(b, settings))
            n_bad += 1
        else:
            assert K.blob_to_kzg_commitment(b, settings) == want, i
            n_valid += 1
    assert n_valid >= 7 and n_bad >= 2
    assert K.blob_to_kzg_commitment(bytes(131072), settings) == IDENTITY


def test_compute_blob_kzg_proof_vectors_and_commitment_checks(K, settings, vectors, oracle):
    cases = [c for c in vectors["verify_blob_kzg_proof"] if c["output"] is True]
    assert cases
    for c in cases:
        blob = vectors.blobs[c["blob"]]
        assert K.compute_blob_kzg_proof(blob, unhex(c["commitment"]), settings) == unhex(c["proof"]), c["name"]
    blob = vectors.blobs[cases[1]["blob"]]
    good_c = unhex(cases[1]["commitment"])
    invalid = [unhex(c["commitment"]) for c in vectors["verify_blob_kzg_proof"] if "invalid_commitment" in c["name"]]
    for c in [c for c in invalid if len(c) != 48]:        # wrong lengths are refused before the GPU
        with pytest.raises(K.KzgError) as e:
            K.compute_blob_kzg_proof(blob, c, settings)
        assert e.value.kind == "InvalidBytesLength"
    invalid = [c for c in invalid if len(c) == 48]
    assert invalid
    # hand-made encodings: infinity flag with nonzero bytes; an x off the curve; a point on the curve outside the subgroup
    inf_nonzero = b"\xc0" + bytes(46) + b"\x01"
    x = 1
    while True:       # compressed-form x that decompresses (x^3 + 4 is a square) but fails the subgroup check
        enc = bytes([0x80 | (x >> 376)]) + (x % (1 << 376)).to_bytes(47, "big")
        chk = oracle.g1_check(enc)         # None: does not decompress; else (in subgroup, in subgroup by the naive check)
        if chk is not None and not chk[0] and not chk[1]:
            break
        x += 1
    off_curve = None
    for x2 in range(1, 64):
        enc2 = bytes([0x80]) + x2.to_bytes(47, "big")
        if oracle.g1_check(enc2) is None:
            off_curve = enc2
            break
    assert off_curve is not None
    for c in invalid + [inf_nonzero, off_curve, enc]:
        assert oracle.compute_blob_kzg_proof(blob, c) is None, c.hex()
        bad_args(K, lambda: K.compute_blob_kzg_proof(blob, c, settings))
    # a non-canonical blob
    nc = [b for b in vectors.blobs if len(b) == 131072 and oracle.blob_to_kzg_commitment(b) is None]
    assert nc
    bad_args(K, lambda: K.compute_blob_kzg_proof(nc[0], good_c, settings))


def test_z_edge_cases(K, settings, vectors, oracle):
    blobs = [b for _, b, _ in valid_blobs(vectors, oracle)][1:4] + [rand_blob(3)]
    rnd = random.Random(11)
    zs = [pow(OMEGA, i, Q) for i in (0, 1, 2048, 4095)] + [rnd.randrange(Q) for _ in range(2)]
    for blob in blobs:
        c = K.blob_to_kzg_commitment(blob, settings)
        assert c == oracle.blob_to_kzg_commitment(blob)
        for z in zs:
            proof, y = K.compute_kzg_proof(blob, be32(z), settings)
            assert (proof, y) == oracle.compute_kzg_proof(blob, be32(z)), z
            assert K.KzgProof.verify_kzg_proof(c, be32(z), y, proof, settings) is True
    for z in (Q, (1 << 256) - 1):
        assert oracle.compute_kzg_proof(blobs[0], be32(z)) is None
        bad_args(K, lambda: K.compute_kzg_proof(blobs[0], be32(z), settings))


def _device_blobs(n, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    blobs = torch.randint(0, 256, (n * 131072,), dtype=torch.uint8, device="cuda", generator=g)
    blobs.view(n * 4096, 32)[:, 0] &= 0x3f
    torch.cuda.synchronize()
    return blobs


@pytest.mark.parametrize("n", [1, 21, 128, 1025])
def test_compute_kzg_proof_batch_device(K, settings, oracle, n):
    """In-domain and random z mixed; sampled entries against the oracle and the single host call."""
    import torch
    lib, ctx = K.Library.get().dll, settings.commit_context(0)
    blobs = _device_blobs(n, 100 + n)
    rnd = random.Random(n)
    zs = [pow(OMEGA, rnd.randrange(4096), Q) if i % 3 == 0 else rnd.randrange(Q) for i in range(n)]
    d_z = torch.frombuffer(bytearray(b"".join(be32(z) for z in zs)), dtype=torch.uint8).cuda()
    d_p = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    d_y = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert lib.kzgb200_compute_kzg_proof_batch_device(ctx, blobs.data_ptr(), d_z.data_ptr(), n, d_p.data_ptr(), d_y.data_ptr()) == 0
    hp, hy = d_p.cpu().numpy().tobytes(), d_y.cpu().numpy().tobytes()
    sample = sorted({0, n - 1, n // 2} | set(rnd.sample(range(n), min(n, 4))))
    if n > 1024:
        sample += [1023, 1024]
    for i in sample:
        blob = blobs[131072 * i:131072 * (i + 1)].cpu().numpy().tobytes()
        want = oracle.compute_kzg_proof(blob, be32(zs[i]))
        assert (hp[48 * i:48 * i + 48], hy[32 * i:32 * i + 32]) == want, i
        assert K.compute_kzg_proof(blob, be32(zs[i]), settings) == want, i
    # one bad z (or blob element) fails the whole call; n == 0 is OK
    bad = bytearray(d_z.cpu().numpy().tobytes()); bad[32 * (n - 1):32 * n] = be32(Q)
    d_bad = torch.frombuffer(bad, dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    assert lib.kzgb200_compute_kzg_proof_batch_device(ctx, blobs.data_ptr(), d_bad.data_ptr(), n, d_p.data_ptr(), d_y.data_ptr()) == 1
    assert lib.kzgb200_compute_kzg_proof_batch_device(ctx, None, None, 0, None, None) == 0


@pytest.mark.parametrize("n", [1, 1025])
def test_existing_device_batches_on_both_sides_of_the_slice_choice(K, settings, oracle, n):
    import torch
    lib, ctx = K.Library.get().dll, settings.commit_context(0)
    blobs = _device_blobs(n, 200 + n)
    d_c = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    d_p = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_blob_to_kzg_commitment_batch(ctx, blobs.data_ptr(), n, d_c.data_ptr()) == 0
    assert lib.kzgb200_compute_blob_kzg_proof_batch(ctx, blobs.data_ptr(), d_c.data_ptr(), n, d_p.data_ptr()) == 0
    hc, hp = d_c.cpu().numpy().tobytes(), d_p.cpu().numpy().tobytes()
    for i in sorted({0, n // 2, n - 1} | ({1023, 1024} if n > 1024 else set())):
        blob = blobs[131072 * i:131072 * (i + 1)].cpu().numpy().tobytes()
        c = oracle.blob_to_kzg_commitment(blob)
        assert hc[48 * i:48 * i + 48] == c, i
        assert hp[48 * i:48 * i + 48] == oracle.compute_blob_kzg_proof(blob, c), i


def test_custom_setup(K, oracle):
    path = os.path.join(GOLDEN, "custom_setup.bin")
    custom = K.KzgSettings.load_trusted_setup_file(path)
    blob, z = rand_blob(77), be32(pow(OMEGA, 5, Q))
    try:
        c = K.blob_to_kzg_commitment(blob, custom)
        pz = K.compute_kzg_proof(blob, z, custom)
        pr = K.compute_kzg_proof(blob, be32(12345), custom)
        pb = K.compute_blob_kzg_proof(blob, c, custom)
    finally:
        custom.close()
    oracle.use_setup(path)
    try:
        assert c == oracle.blob_to_kzg_commitment(blob)
        assert pz == oracle.compute_kzg_proof(blob, z) and pr == oracle.compute_kzg_proof(blob, be32(12345))
        assert pb == oracle.compute_blob_kzg_proof(blob, c)
    finally:
        oracle.use_setup(None)
    assert c != oracle.blob_to_kzg_commitment(blob)          # another tau than the mainnet setup


def test_publisher_flow_blob_and_cells_on_one_context(K, settings):
    blobs = [rand_blob(31), rand_blob(32)]
    ctx = settings.commit_context(0)
    assert settings.cell_proof_context(0).value == ctx.value          # one context holds both setups
    cs = [K.blob_to_kzg_commitment(b, settings) for b in blobs]
    ps = [K.compute_blob_kzg_proof(b, c, settings) for b, c in zip(blobs, cs)]
    assert K.KzgProof.verify_blob_kzg_proof_batch(blobs, cs, ps, settings) is True
    cells, proofs = K.compute_cells_and_kzg_proofs(blobs[0], settings)
    assert K.KzgProof.verify_cell_kzg_proof_batch([cs[0]] * 128, list(range(128)), cells, proofs, settings) is True
    assert K.KzgProof.verify_cell_kzg_proof_batch([cs[1]] * 128, list(range(128)), cells, proofs, settings) is False


def test_cpp_mirror_runs_the_three_calls(tmp_path, vectors):
    case = [c for c in vectors["verify_kzg_proof"] if c["output"] is True and int(c["z"], 16) == Q - 1][0]
    blob_case = [c for c in vectors["verify_blob_kzg_proof"] if c["output"] is True and c["commitment"] == case["commitment"]][0]
    blob = vectors.blobs[blob_case["blob"]]
    (tmp_path / "blob.bin").write_bytes(blob)
    src = tmp_path / "prove.cpp"
    src.write_text(r'''
#include "kzg_rs.hpp"
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iterator>
int main(int argc, char** argv) {
    using namespace kzg_rs;
    std::ifstream f(argv[2], std::ios::binary);
    std::vector<uint8_t> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    auto blob = Blob::from_slice(raw.data(), raw.size()).unwrap();
    auto s = KzgSettings::load_trusted_setup_file(argv[1]);
    if (s.is_err() || s.unwrap().load_commit_setup().is_err()) return 2;
    Bytes32 z{};
    for (int i = 0; i < 32; i++) z.bytes[i] = (uint8_t)strtoul(std::string(argv[3] + 2 * i, 2).c_str(), nullptr, 16);
    auto c = blob_to_kzg_commitment(blob, s.unwrap());
    auto py = compute_kzg_proof(blob, z, s.unwrap());
    if (c.is_err() || py.is_err()) return 3;
    auto pb = compute_blob_kzg_proof(blob, c.unwrap(), s.unwrap());
    if (pb.is_err()) return 4;
    Bytes48 bad{}; bad.bytes[0] = 0x81;
    auto e = compute_blob_kzg_proof(blob, bad, s.unwrap());
    if (!e.is_err() || e.unwrap_err().kind != KzgError::BadArgs) return 5;
    auto hex = [](const uint8_t* p, size_t n) { for (size_t i = 0; i < n; i++) std::printf("%02x", p[i]); std::printf("\n"); };
    hex(c.unwrap().as_slice(), 48); hex(py.unwrap().first.as_slice(), 48); hex(py.unwrap().second.as_slice(), 32); hex(pb.unwrap().as_slice(), 48);
    return 0;
}
''')
    lib = os.path.join(ROOT, "kzg_rs_b200", "libkzgb200.so")
    exe = tmp_path / "prove"
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", os.path.dirname(lib), "-lkzgb200", "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.run([str(exe), os.path.join(ROOT, "kzg_rs_b200", "data", "mainnet_setup.bin"), str(tmp_path / "blob.bin"), case["z"][2:]],
                         capture_output=True, text=True)
    assert out.returncode == 0, (out.returncode, out.stderr)
    c, p, y, pb = out.stdout.split()
    assert (c, p, y, pb) == (case["commitment"][2:], case["proof"][2:], case["y"][2:], blob_case["proof"][2:])
