"""verify_blob_cell_kzg_proof_batch[_many] on the GPU (pytest -m gpu): the cell proofs of whole blob transactions, one verdict per
transaction.  Every verdict is checked against kzgb200_verify_cell_kzg_proof_batch on the transaction's expanded inputs (commitment of
blob b repeated 128 times, indices 0..127 per blob, the cells of compute_cells, the proofs), and every r_g of a group that is not
BadArgs against that call's r: harness blobs, the CPU cell oracle, full-degree blobs with FK20 proofs, a seeded mempool of tampered
and malformed transactions, edge shapes, argument errors, the device forms, a custom setup, the Python API and the C++ mirror."""
import ctypes as C
import os
import random
import subprocess

import pytest
from conftest import GOLDEN, ROOT

from cell_oracle import cells as CO

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
CELL = 2048
BLOB = 131072
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
    s.cell_context(0)
    return s


@pytest.fixture(scope="module")
def lib(K):
    return K.Library.get().dll


@pytest.fixture(scope="module")
def ctx(settings):
    return settings.cell_context(0)


class Harness:
    """harness blobs (degree-192 polynomials, mainnet monomial points): blob b = cells 0..63 of the generator's output, with its
    commitment and its 128 cell proofs"""

    def __init__(self, K, settings, n_blobs, seed):
        import torch
        lib, ctx = K.Library.get().dll, settings.cell_context(0)
        tau = K.api.mainnet_g1_monomial()[:192 * 48]
        cells = torch.empty(n_blobs * 128 * CELL, dtype=torch.uint8, device="cuda")
        cs = torch.empty(n_blobs * 48, dtype=torch.uint8, device="cuda")
        ps = torch.empty(n_blobs * 128 * 48, dtype=torch.uint8, device="cuda")
        assert lib.kzgb200_harness_generate_cells(ctx, seed, n_blobs, 192, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
        torch.cuda.synchronize()
        hc, hcs, hps = (t.cpu().numpy().tobytes() for t in (cells, cs, ps))
        self.blobs = [hc[128 * CELL * b:128 * CELL * b + BLOB] for b in range(n_blobs)]
        self.cs = [hcs[48 * b:48 * b + 48] for b in range(n_blobs)]
        self.ps = [[hps[48 * (128 * b + j):48 * (128 * b + j + 1)] for j in range(128)] for b in range(n_blobs)]

    def tx(self, bs):
        """a transaction of the blobs bs (in that order): [blobs, commitments, cell proofs]"""
        return [[self.blobs[b] for b in bs], [self.cs[b] for b in bs], [p for b in bs for p in self.ps[b]]]


@pytest.fixture(scope="module")
def h64(K, settings):
    return Harness(K, settings, 64, 0x4844)


def dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda() if b else None


def ptr(t):
    return t.data_ptr() if t is not None else None


def joined(txs):
    offs = [0]
    for t in txs:
        offs.append(offs[-1] + len(t[0]))
    return (b"".join(b"".join(t[0]) for t in txs), b"".join(b"".join(t[1]) for t in txs), b"".join(b"".join(t[2]) for t in txs), offs)


def last_many_r(lib, ctx, k):
    r, rho = C.create_string_buffer(32 * max(k, 1)), C.create_string_buffer(32)
    assert lib.kzgb200_last_cell_many_r(ctx, r, k, rho) == 0
    return [r.raw[32 * g:32 * g + 32] for g in range(k)], rho.raw


def many(lib, ctx, txs, device=False):
    """one _many call (host or device form): (verdicts, [r_g], rho)"""
    bl, cs, ps, offs = joined(txs)
    k = len(txs)
    off = (C.c_uint64 * (k + 1))(*offs)
    out = C.create_string_buffer(max(k, 1))
    if device:
        d = [dev(x) for x in (bl, cs, ps)]
        rc = lib.kzgb200_verify_blob_cell_kzg_proof_batch_many_device(ctx, *[ptr(t) for t in d], C.cast(off, C.c_void_p), k, out)
    else:
        rc = lib.kzgb200_verify_blob_cell_kzg_proof_batch_many(ctx, bl, cs, ps, C.cast(off, C.c_void_p), k, out)
    assert rc == 0, rc
    return (list(out.raw[:k]),) + tuple(last_many_r(lib, ctx, k))


def single(lib, ctx, t, device=False):
    """the single call (host or device form): (verdict 1 / 0 / 2, its r or None)"""
    blobs, cs, ps = t
    ok = C.c_int(-1)
    if device:
        d = [dev(b"".join(x)) for x in t]
        rc = lib.kzgb200_verify_blob_cell_kzg_proof_batch_device(ctx, *[ptr(x) for x in d], len(blobs), C.byref(ok))
    else:
        rc = lib.kzgb200_verify_blob_cell_kzg_proof_batch(ctx, b"".join(blobs), len(blobs), b"".join(cs), len(cs), b"".join(ps), len(ps),
                                                          C.byref(ok))
    assert rc in (0, 1), rc
    if rc == 1:
        return 2, None
    if not blobs:
        return ok.value, None
    r = C.create_string_buffer(32)
    assert lib.kzgb200_last_r(ctx, r) == 0
    assert last_many_r(lib, ctx, 1)[0] == [r.raw]
    return ok.value, r.raw


def reference(lib, ctx, t):
    """verify_cell_kzg_proof_batch on the expanded inputs, cells by kzgb200_compute_cells: (verdict, r or None); a blob that
    compute_cells refuses makes the transaction BadArgs"""
    blobs, cs, ps = t
    cells = []
    for b in blobs:
        out = C.create_string_buffer(128 * CELL)
        rc = lib.kzgb200_compute_cells(ctx, b, out)
        assert rc in (0, 1), rc
        if rc == 1:
            return 2, None
        cells.append(out.raw)
    n = 128 * len(blobs)
    idx = (C.c_uint64 * max(n, 1))(*[j for _ in blobs for j in range(128)])
    ok = C.c_int(-1)
    rc = lib.kzgb200_verify_cell_kzg_proof_batch(ctx, b"".join(c * 128 for c in cs), C.cast(idx, C.c_void_p), b"".join(cells),
                                                 b"".join(ps), n, C.byref(ok))
    assert rc in (0, 1), rc
    if rc == 1:
        return 2, None
    if not n:
        return ok.value, None
    r = C.create_string_buffer(32)
    assert lib.kzgb200_last_r(ctx, r) == 0
    return ok.value, r.raw


def check_against_reference(lib, ctx, txs, verdicts, rs):
    for g, t in enumerate(txs):
        v, r = reference(lib, ctx, t)
        assert verdicts[g] == v, (g, verdicts[g], v)
        if v != 2 and r is not None:
            assert rs[g] == r, g


def g1_plus_gen(p48):
    from oracle import pyref as R
    return R.g1_to_compressed(R.g1_add(R.g1_from_compressed(p48)[1], R.G1_GEN))


def off_curve_point():
    from oracle import pyref as R
    x = next(x for x in range(1, 1000) if R.fp_sqrt((x ** 3 + 4) % R.P) is None)
    return bytes([0x80]) + x.to_bytes(48, "big")[1:]


def non_subgroup_point():
    from oracle import pyref as R
    for x in range(0, 1000):
        y = R.fp_sqrt((x ** 3 + 4) % R.P)
        if y is not None and not R.g1_in_subgroup((x, y)):
            return R.g1_to_compressed((x, y))
    raise AssertionError("no point found")


def set_element(blob, i, value):
    return blob[:32 * i] + value.to_bytes(32, "big") + blob[32 * i + 32:]


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))


# ---- valid transactions --------------------------------------------------------------------------------------------------
def test_harness_transaction_and_block(K, settings, lib, ctx, h64):
    tx6, block = h64.tx(range(6)), h64.tx(range(10, 31))
    for t in (tx6, block):
        v, r = single(lib, ctx, t)
        assert (v, r) == reference(lib, ctx, t) and v == 1
    verdicts, rs, _ = many(lib, ctx, [tx6, block])
    assert verdicts == [1, 1]
    check_against_reference(lib, ctx, [tx6, block], verdicts, rs)


def test_cpu_cell_oracle(K, settings, lib, ctx, h64):
    t = h64.tx([7, 8])
    blobs, cs, ps = t
    cells = [c for b in blobs for c in CO.compute_cells(b)]
    expanded = ([c for c in cs for _ in range(128)], [j for _ in blobs for j in range(128)], cells)
    ok, r = CO.verify_cell_kzg_proof_batch(*expanded, ps, want_r=True)
    assert ok is True and single(lib, ctx, t) == (1, r)
    bad = list(ps)
    bad[3], bad[200] = bad[200], bad[3]
    ok, r = CO.verify_cell_kzg_proof_batch(*expanded, bad, want_r=True)
    assert ok is False and single(lib, ctx, [blobs, cs, bad]) == (0, r)


def test_full_degree_blobs(K, settings, lib):
    import torch
    ctx = settings.cell_proof_context(0)
    settings.commit_context(0)
    blobs = [rand_blob(0xb10b + s) for s in range(8)] + [bytes(BLOB), (Q - 1).to_bytes(32, "big") * 4096]
    n = len(blobs)
    d_b = dev(b"".join(blobs))
    d_c = torch.empty(n * 128 * CELL, dtype=torch.uint8, device="cuda")
    d_p = torch.empty(n * 128 * 48, dtype=torch.uint8, device="cuda")
    assert lib.kzgb200_compute_cells_and_kzg_proofs_batch_device(ctx, d_b.data_ptr(), n, d_c.data_ptr(), d_p.data_ptr()) == 0
    torch.cuda.synchronize()
    hp = d_p.cpu().numpy().tobytes()
    ps = [[hp[48 * (128 * b + j):48 * (128 * b + j + 1)] for j in range(128)] for b in range(n)]
    cs = [K.blob_to_kzg_commitment(b, settings) for b in blobs]
    assert cs[8] == IDENTITY and ps[8] == [IDENTITY] * 128
    tx = lambda bs: [[blobs[b] for b in bs], [cs[b] for b in bs], [p for b in bs for p in ps[b]]]
    txs = [tx(range(4)), tx(range(4, 8)), tx([8]), tx([9]), tx([9, 8, 0])]
    verdicts, rs, _ = many(lib, ctx, txs)
    assert verdicts == [1] * 5
    check_against_reference(lib, ctx, txs, verdicts, rs)
    assert single(lib, ctx, tx(range(n)))[0] == 1


# ---- a mempool burst: one verdict per transaction ----------------------------------------------------------------------------
def mempool(h, seed, n_tx=40):
    """seeded transactions of 0..6 harness blobs, each untouched or with one fault; returns (txs, the verdict each fault implies)"""
    rnd = random.Random(seed)
    bad_points = [off_curve_point(), non_subgroup_point(), bytes(48)]
    n = len(h.blobs)
    txs, want = [], []
    for _ in range(n_tx):
        nb = rnd.randrange(7)
        t = h.tx(rnd.sample(range(n), nb))
        kind = rnd.randrange(8) if nb else 0
        blobs, cs, ps = t
        b, j = rnd.randrange(max(nb, 1)), rnd.randrange(128)
        if kind == 1:                                    # two proofs swapped inside a blob
            j2 = (j + 1 + rnd.randrange(127)) % 128
            ps[128 * b + j], ps[128 * b + j2] = ps[128 * b + j2], ps[128 * b + j]
        elif kind == 2:                                  # a proof from another blob
            other = next(o for o in range(n) if h.cs[o] != cs[b])
            ps[128 * b + j] = h.ps[other][j]
        elif kind == 3 and nb >= 2:                      # two commitments swapped
            cs[0], cs[1] = cs[1], cs[0]
        elif kind == 3:                                  # one commitment replaced by another blob's
            cs[0] = next(c for c in h.cs if c != cs[0])
        elif kind == 4:                                  # one blob element changed, still canonical
            i = rnd.randrange(4096)
            v = int.from_bytes(blobs[b][32 * i:32 * i + 32], "big")
            blobs[b] = set_element(blobs[b], i, (v + 1 + rnd.randrange(1000)) % Q)
        elif kind == 5:                                  # a non-canonical element
            blobs[b] = set_element(blobs[b], rnd.randrange(4096), rnd.choice([Q, Q + 1, (1 << 256) - 1]))
        elif kind == 6:                                  # an invalid commitment
            cs[b] = rnd.choice(bad_points)
        elif kind == 7:                                  # an invalid proof
            ps[128 * b + j] = rnd.choice(bad_points)
        txs.append(t)
        want.append(1 if kind == 0 or not nb else (2 if kind >= 5 else 0))
    return txs, want


def test_mempool_burst_takes_the_fallback(K, settings, lib, ctx, h64):
    txs, want = mempool(h64, 0x7594)
    assert 0 in want and 2 in want and 1 in want and any(not t[0] for t in txs)
    ms = (C.c_float * 8)()
    assert lib.kzgb200_set_profiling(ctx, 1) == 0
    try:
        verdicts, rs, _ = many(lib, ctx, txs)
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
        assert ms[7] > 0, list(ms)                       # the combined check failed: every group got its own check
    finally:
        lib.kzgb200_set_profiling(ctx, 0)
    assert verdicts == want
    check_against_reference(lib, ctx, txs, verdicts, rs)
    # the same burst without its false transactions: the combined check passes, BadArgs transactions still get 2
    keep = [t for t, w in zip(txs, want) if w != 0]
    verdicts, rs, _ = many(lib, ctx, keep)
    assert verdicts == [w for w in want if w != 0]
    check_against_reference(lib, ctx, keep, verdicts, rs)


# ---- shapes ------------------------------------------------------------------------------------------------------------
def test_shapes(K, settings, lib, ctx, h64):
    off = (C.c_uint64 * 1)(0)
    assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many(ctx, None, None, None, C.cast(off, C.c_void_p), 0, None) == 0
    assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many(ctx, None, None, None, None, 0, None) == 0
    assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many_device(ctx, None, None, None, None, 0, None) == 0
    empty = h64.tx([])
    verdicts, rs, _ = many(lib, ctx, [empty] * 3)
    assert verdicts == [1, 1, 1] and rs == [bytes(32)] * 3
    assert single(lib, ctx, empty) == (1, None)
    txs = [empty, h64.tx([1, 2]), empty, empty, h64.tx([5]), empty]
    verdicts, rs, _ = many(lib, ctx, txs)
    assert verdicts == [1] * 6 and rs[0] == rs[2] == rs[3] == rs[5] == bytes(32)
    check_against_reference(lib, ctx, txs, verdicts, rs)
    # the same blob twice in a transaction; one commitment (blob 9) in two transactions; a false transaction beside them
    false = h64.tx([20, 21])
    false[2][0], false[2][1] = false[2][1], false[2][0]
    txs = [h64.tx([3, 3]), h64.tx([8, 9]), h64.tx([9, 10, 9]), false]
    verdicts, rs, _ = many(lib, ctx, txs)
    assert verdicts == [1, 1, 1, 0]
    check_against_reference(lib, ctx, txs, verdicts, rs)


def test_one_128_blob_transaction(K, settings, lib, ctx):
    h = Harness(K, settings, 128, 11)
    t = h.tx(range(128))
    verdicts, rs, _ = many(lib, ctx, [t])
    assert verdicts == [1]
    check_against_reference(lib, ctx, [t], verdicts, rs)
    assert single(lib, ctx, t, device=True) == (1, rs[0])
    t[2][12345] = g1_plus_gen(t[2][12345])
    assert single(lib, ctx, t) == reference(lib, ctx, t)
    assert single(lib, ctx, t)[0] == 0


# ---- argument errors ---------------------------------------------------------------------------------------------------
def test_errors(K, settings, lib, ctx, h64):
    ok = C.c_int(-1)
    blobs, cs, ps = (b"".join(x) for x in h64.tx([0, 1]))
    f = lib.kzgb200_verify_blob_cell_kzg_proof_batch
    assert f(ctx, blobs, 2, cs, 1, ps, 256, C.byref(ok)) == 3
    assert f(ctx, blobs, 2, cs, 3, ps, 256, C.byref(ok)) == 3
    assert f(ctx, blobs, 2, cs, 2, ps, 255, C.byref(ok)) == 3
    assert f(ctx, blobs, 2, cs, 2, ps, 128, C.byref(ok)) == 3
    assert f(ctx, None, 0, None, 0, None, 1, C.byref(ok)) == 3
    assert f(ctx, blobs, 2, cs, 2, ps, 256, None) == 1
    assert f(ctx, None, 2, cs, 2, ps, 256, C.byref(ok)) == 1
    assert f(ctx, None, 0, None, 0, None, 0, C.byref(ok)) == 0 and ok.value == 1
    assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_device(ctx, None, None, None, 1, C.byref(ok)) == 1
    assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_device(ctx, None, None, None, 1 << 23, C.byref(ok)) == 1
    out = C.create_string_buffer(2)
    for m in (lib.kzgb200_verify_blob_cell_kzg_proof_batch_many, lib.kzgb200_verify_blob_cell_kzg_proof_batch_many_device):
        for offs in ((1, 2), (0, 2, 1), (0, 1 << 23), (0, 1, 1 << 23)):          # 128 x (1 << 23) cells > 0x7fffffff / 2
            off = (C.c_uint64 * len(offs))(*offs)
            assert m(ctx, blobs, cs, ps, C.cast(off, C.c_void_p), len(offs) - 1, out) == 1, offs
        off = (C.c_uint64 * 2)(0, 2)
        assert m(ctx, blobs, cs, ps, C.cast(off, C.c_void_p), 1, None) == 1
        assert m(ctx, blobs, cs, ps, None, 1, out) == 1
        assert m(ctx, None, cs, ps, C.cast(off, C.c_void_p), 1, out) == 1
        assert m(ctx, blobs, None, ps, C.cast(off, C.c_void_p), 1, out) == 1
        assert m(ctx, blobs, cs, None, C.cast(off, C.c_void_p), 1, out) == 1
    # a context without the cell setup
    fresh = K.KzgSettings(settings.g1_lagrange_bytes, settings.g2_monomial_bytes)
    try:
        fctx = fresh.context(0)
        off = (C.c_uint64 * 2)(0, 2)
        assert f(fctx, blobs, 2, cs, 2, ps, 256, C.byref(ok)) == 5
        assert f(fctx, None, 0, None, 0, None, 0, C.byref(ok)) == 5
        assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_device(fctx, None, None, None, 0, C.byref(ok)) == 5
        assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many(fctx, blobs, cs, ps, C.cast(off, C.c_void_p), 1, out) == 5
        assert lib.kzgb200_verify_blob_cell_kzg_proof_batch_many_device(fctx, None, None, None, None, 0, None) == 5
    finally:
        fresh.close()


# ---- other forms -------------------------------------------------------------------------------------------------------
def test_device_forms(K, settings, lib, ctx, h64):
    txs, want = mempool(h64, 0x4844, n_tx=24)
    for gs in (txs, [h64.tx(range(6))], [h64.tx([]), h64.tx([4, 4])]):
        host = many(lib, ctx, gs)
        assert many(lib, ctx, gs, device=True) == host
    for t in txs[:12] + [h64.tx([])]:
        assert single(lib, ctx, t, device=True) == single(lib, ctx, t)


def test_custom_setup(K, settings, oracle):
    path = os.path.join(GOLDEN, "custom_setup.bin")
    blobs = [rand_blob(41), rand_blob(42)]
    oracle.use_setup(path)
    try:
        mono = b"".join(oracle.tau_power_g1(j) for j in range(64))
        cs = [oracle.blob_to_kzg_commitment(b) for b in blobs]
    finally:
        oracle.use_setup(None)
    custom = K.KzgSettings.load_trusted_setup_file(path, g1_monomial_bytes=mono)
    try:
        lib, ctx = K.Library.get().dll, custom.cell_proof_context(0)
        ps = [p for b in blobs for p in K.compute_cells_and_kzg_proofs(b, custom)[1]]
        good = [blobs, cs, ps]
        swapped = [blobs, cs, ps[:5] + [ps[6], ps[5]] + ps[7:]]
        verdicts, rs, _ = many(lib, ctx, [good, swapped, [blobs[:1], cs[:1], ps[:128]]])
        assert verdicts == [1, 0, 1]
        check_against_reference(lib, ctx, [good, swapped], verdicts, rs)
        assert K.KzgProof.verify_blob_cell_kzg_proof_batch(blobs, cs, ps, custom) is True
        assert K.KzgProof.verify_blob_cell_kzg_proof_batch(blobs, cs, ps, settings) is False
    finally:
        custom.close()


def test_python_api(K, settings, h64):
    P = K.KzgProof
    good = h64.tx([0, 1, 2])
    false = h64.tx([3, 4])
    false[1] = false[1][::-1]
    bad = h64.tx([5])
    bad[0][0] = set_element(bad[0][0], 7, Q)
    typed = [[K.Blob.from_slice(b) for b in good[0]], [K.Bytes48.from_slice(c) for c in good[1]], [K.Bytes48.from_slice(p) for p in good[2]]]
    assert P.verify_blob_cell_kzg_proof_batch(*good, settings) is True
    assert P.verify_blob_cell_kzg_proof_batch(*typed, settings) is True
    assert P.verify_blob_cell_kzg_proof_batch(*false, settings) is False
    assert P.verify_blob_cell_kzg_proof_batch([], [], [], settings) is True
    with pytest.raises(K.KzgError) as e:
        P.verify_blob_cell_kzg_proof_batch(*bad, settings)
    assert e.value.kind == "BadArgs"
    assert P.verify_blob_cell_kzg_proof_batch_many([tuple(good), tuple(false), tuple(bad), ([], [], []), tuple(typed)], settings) == \
        [True, False, None, True, True]
    assert P.verify_blob_cell_kzg_proof_batch_many([], settings) == []
    with pytest.raises(K.KzgError) as e:
        P.verify_blob_cell_kzg_proof_batch_many([tuple(good), (good[0], good[1], good[2][:-1])], settings)
    assert e.value.kind == "InvalidBytesLength"


def test_cpp_mirror(tmp_path, K, settings, h64):
    good = h64.tx([0, 1])
    false = h64.tx([2])
    false[2][0], false[2][1] = false[2][1], false[2][0]
    for name, t in (("good", good), ("false", false)):
        for part, data in zip(("blobs", "cs", "ps"), t):
            (tmp_path / f"{name}_{part}.bin").write_bytes(b"".join(data))
    (tmp_path / "mono.bin").write_bytes(K.api.mainnet_g1_monomial()[:64 * 48])
    src = tmp_path / "blob_cells.cpp"
    src.write_text(r'''
#include "kzg_rs.hpp"
#include <cstdio>
#include <fstream>
#include <iterator>
#include <string>
static std::vector<uint8_t> slurp(const std::string& p) {
    std::ifstream f(p, std::ios::binary);
    return std::vector<uint8_t>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}
template <class T> static std::vector<T> split(const std::vector<uint8_t>& raw) {
    std::vector<T> out;
    for (size_t o = 0; o < raw.size(); o += sizeof(T)) out.push_back(T::from_slice(raw.data() + o, sizeof(T)).unwrap());
    return out;
}
int main(int argc, char** argv) {
    using namespace kzg_rs;
    const std::string d = argv[2];
    auto s = KzgSettings::load_trusted_setup_file(argv[1]);
    if (s.is_err()) return 2;
    auto mono = slurp(d + "/mono.bin");
    if (s.unwrap().load_cell_setup(mono.data(), mono.size() / 48).is_err()) return 3;
    std::vector<Blob> blobs; std::vector<Bytes48> cs, ps; std::vector<uint64_t> offs{0};
    for (const char* name : {"good", "false"}) {
        auto b = split<Blob>(slurp(d + "/" + name + "_blobs.bin"));
        auto c = split<Bytes48>(slurp(d + "/" + name + "_cs.bin"));
        auto p = split<Bytes48>(slurp(d + "/" + name + "_ps.bin"));
        auto v = KzgProof::verify_blob_cell_kzg_proof_batch(b, c, p, s.unwrap());
        if (v.is_err()) return 4;
        std::printf("%d ", (int)v.unwrap());
        blobs.insert(blobs.end(), b.begin(), b.end()); cs.insert(cs.end(), c.begin(), c.end()); ps.insert(ps.end(), p.begin(), p.end());
        offs.push_back(blobs.size());
    }
    auto m = KzgProof::verify_blob_cell_kzg_proof_batch_many(blobs, cs, ps, offs, s.unwrap());
    if (m.is_err()) return 5;
    for (uint8_t v : m.unwrap()) std::printf("%d ", (int)v);
    auto e = KzgProof::verify_blob_cell_kzg_proof_batch(blobs, cs, std::vector<Bytes48>(ps.begin() + 1, ps.end()), s.unwrap());
    if (!e.is_err() || e.unwrap_err().kind != KzgError::InvalidBytesLength) return 6;
    std::printf("\n");
    return 0;
}
''')
    lib = os.path.join(ROOT, "kzg_rs_b200", "libkzgb200.so")
    exe = tmp_path / "blob_cells"
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", os.path.dirname(lib), "-lkzgb200", "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.run([str(exe), os.path.join(ROOT, "kzg_rs_b200", "data", "mainnet_setup.bin"), str(tmp_path)],
                         capture_output=True, text=True)
    assert out.returncode == 0, (out.returncode, out.stderr)
    assert out.stdout.split() == ["1", "0", "1", "0"]
