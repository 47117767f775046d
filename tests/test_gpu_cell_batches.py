"""verify_cell_kzg_proof_batch_many on the GPU (pytest -m gpu): k independent cell batches in one call, one verdict each.  Every
verdict is checked against a single verify_cell_kzg_proof_batch call on the same group (and the CPU cell oracle where it is cheap),
every r_g against the oracle's r and the single call's, for data column sidecars of harness blocks, tampered and malformed groups,
edge shapes, the per-group fallback at scale, seeded random mixes, the device form and a custom setup."""
import ctypes as C
import hashlib
import os
import random

import pytest
from conftest import GOLDEN

from cell_oracle import cells as CO

pytestmark = pytest.mark.gpu
Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
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
def ctx(settings):
    return settings.cell_context(0)


class Block:
    """harness blobs (degree 192, mainnet monomial points) as host bytes: cell(b, i), commitment(b), proof(b, i)"""

    def __init__(self, K, settings, n_blobs, seed):
        import torch
        lib, ctx = K.Library.get().dll, settings.cell_context(0)
        tau = K.api.mainnet_g1_monomial()[:192 * 48]
        cells = torch.empty(n_blobs * 128 * CELL, dtype=torch.uint8, device="cuda")
        cs = torch.empty(n_blobs * 48, dtype=torch.uint8, device="cuda")
        ps = torch.empty(n_blobs * 128 * 48, dtype=torch.uint8, device="cuda")
        assert lib.kzgb200_harness_generate_cells(ctx, seed, n_blobs, 192, tau, cells.data_ptr(), cs.data_ptr(), ps.data_ptr()) == 0
        torch.cuda.synchronize()
        self.n = n_blobs
        self.hc, self.hcs, self.hps = (t.cpu().numpy().tobytes() for t in (cells, cs, ps))

    def cell(self, b, i): return self.hc[CELL * (128 * b + i):CELL * (128 * b + i + 1)]
    def commitment(self, b): return self.hcs[48 * b:48 * b + 48]
    def proof(self, b, i): return self.hps[48 * (128 * b + i):48 * (128 * b + i + 1)]

    def entry(self, b, i): return [self.commitment(b), i, self.cell(b, i), self.proof(b, i)]

    def sidecar(self, i, blobs=None):
        """data column sidecar i: cell i of every blob, with the blobs' commitments -> [commitments, indices, cells, proofs]"""
        return group([self.entry(b, i) for b in (range(self.n) if blobs is None else blobs)])


def group(entries):
    return [list(x) for x in zip(*entries)] if entries else [[], [], [], []]


@pytest.fixture(scope="module")
def block21(K, settings):
    return Block(K, settings, 21, 0x7594)


def many(lib, ctx, groups):
    """the C ABI on host buffers: (verdicts, [r_g], rho)"""
    k = len(groups)
    offs = [0]
    for g in groups:
        offs.append(offs[-1] + len(g[1]))
    n = offs[-1]
    cs = b"".join(b"".join(g[0]) for g in groups)
    idx = (C.c_uint64 * max(n, 1))(*[i for g in groups for i in g[1]])
    ce = b"".join(b"".join(g[2]) for g in groups)
    ps = b"".join(b"".join(g[3]) for g in groups)
    off = (C.c_uint64 * (k + 1))(*offs)
    out = C.create_string_buffer(max(k, 1))
    rc = lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, cs, C.cast(idx, C.c_void_p), ce, ps, C.cast(off, C.c_void_p), k, out)
    assert rc == 0, rc
    r, rho = C.create_string_buffer(32 * max(k, 1)), C.create_string_buffer(32)
    assert lib.kzgb200_last_cell_many_r(ctx, r, k, rho) == 0
    return list(out.raw[:k]), [r.raw[32 * g:32 * g + 32] for g in range(k)], rho.raw


def single(lib, ctx, g):
    """one verify_cell_kzg_proof_batch call: (verdict 1 / 0 / 2, its r or None)"""
    n = len(g[1])
    idx = (C.c_uint64 * max(n, 1))(*g[1])
    ok = C.c_int(-1)
    rc = lib.kzgb200_verify_cell_kzg_proof_batch(ctx, b"".join(g[0]), C.cast(idx, C.c_void_p), b"".join(g[2]), b"".join(g[3]), n, C.byref(ok))
    assert rc in (0, 1), rc
    if rc == 1:
        return 2, None
    r = C.create_string_buffer(32)
    assert lib.kzgb200_last_r(ctx, r) == 0
    return ok.value, r.raw if n else None


def oracle_verdict(g, want_r=False):
    res = CO.verify_cell_kzg_proof_batch(*g, want_r=want_r)
    v = res[0] if want_r else res
    code = 2 if v is None else int(v)
    return (code, res[1]) if want_r else code


def rho_ref(rs, sizes):
    """rho = SHA-256("RCKZGCMANY___V1_" | u64be k | per group: u64be n_g | r_g, or 32 zero bytes when n_g = 0) mod q, 0 -> 1"""
    h = hashlib.sha256(b"RCKZGCMANY___V1_" + len(sizes).to_bytes(8, "big"))
    for r, n in zip(rs, sizes):
        h.update(n.to_bytes(8, "big") + (r if n else bytes(32)))
    v = int.from_bytes(h.digest(), "big") % Q
    return (v or 1).to_bytes(32, "big")


def check_against_single(lib, ctx, groups, verdicts, rs=None):
    for gi, g in enumerate(groups):
        v, r = single(lib, ctx, g)
        assert verdicts[gi] == v, (gi, verdicts[gi], v)
        if rs is not None and v != 2 and r is not None:
            assert rs[gi] == r, gi


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


def test_block_sidecars_all_valid_and_r(K, settings, lib, ctx, block21):
    groups = [block21.sidecar(i) for i in range(128)]
    verdicts, rs, rho = many(lib, ctx, groups)
    assert verdicts == [1] * 128
    assert rho == rho_ref(rs, [21] * 128)
    for i, g in enumerate(groups):
        ok, r = CO.verify_cell_kzg_proof_batch(*g, want_r=True)
        assert ok is True and rs[i] == r, i
        assert single(lib, ctx, g) == (1, r), i


def test_tampered_groups(K, settings, lib, ctx, block21):
    groups = [block21.sidecar(i) for i in range(128)]
    t = bytearray(groups[3][2][5]); t[32 * 17 + 31] ^= 1
    groups[3][2][5] = bytes(t)                                                   # one cell element
    groups[40][3][7], groups[40][3][8] = groups[40][3][8], groups[40][3][7]     # a proof swapped with a neighbour's
    groups[77][0][2] = block21.commitment(3)                                     # the commitment of another blob
    groups[100][3][20] = g1_plus_gen(groups[100][3][20])                         # proof + G
    verdicts, rs, rho = many(lib, ctx, groups)
    bad = {3, 40, 77, 100}
    assert verdicts == [0 if i in bad else 1 for i in range(128)]
    assert rho == rho_ref(rs, [21] * 128)
    for i in sorted(bad) + [0, 64, 127]:
        code, r = oracle_verdict(groups[i], want_r=True)
        assert verdicts[i] == code and rs[i] == r, i
        assert single(lib, ctx, groups[i]) == (code, r), i


def bad_args_groups(block21):
    groups = [block21.sidecar(i) for i in range(24)]
    t = bytearray(groups[2][2][4]); t[32 * 9:32 * 10] = Q.to_bytes(32, "big")
    groups[2][2][4] = bytes(t)                                                   # non-canonical element
    groups[5][3][1] = off_curve_point()                                          # proof not on the curve
    groups[8][3][0] = non_subgroup_point()                                       # proof outside the subgroup
    groups[11][0][6] = bytes(48)                                                 # invalid commitment bytes
    groups[14][1][3] = 128                                                       # cell index 128
    groups[6][3][2], groups[6][3][3] = groups[6][3][3], groups[6][3][2]          # false groups beside them
    groups[15][0][0] = block21.commitment(1)
    return groups, {2, 5, 8, 11, 14}, {6, 15}


def test_bad_args_per_group(K, settings, lib, ctx, block21):
    groups, bad, false = bad_args_groups(block21)
    verdicts, rs, _ = many(lib, ctx, groups)
    assert verdicts == [2 if i in bad else 0 if i in false else 1 for i in range(len(groups))]
    for i in sorted(bad | false) + [0, 23]:
        assert oracle_verdict(groups[i]) == verdicts[i], i
    check_against_single(lib, ctx, groups, verdicts, rs)
    # only BadArgs groups beside valid ones: the combined check passes, the BadArgs groups still get 2
    only_bad = [g if i in bad else block21.sidecar(i) for i, g in enumerate(groups)]
    verdicts, _, _ = many(lib, ctx, only_bad)
    assert verdicts == [2 if i in bad else 1 for i in range(len(groups))]


def test_shapes(K, settings, lib, ctx, block21):
    import torch
    # k = 0: OK, no verdicts
    off = (C.c_uint64 * 1)(0)
    assert lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, None, None, None, None, C.cast(off, C.c_void_p), 0, None) == 0
    assert lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, None, None, None, None, None, 0, None) == 0
    # only empty groups
    verdicts, rs, rho = many(lib, ctx, [group([])] * 3)
    assert verdicts == [1, 1, 1] and rs == [bytes(32)] * 3 and rho == rho_ref(rs, [0, 0, 0])
    # empty groups among others
    e = block21.entry
    groups = [group([]), block21.sidecar(9), group([]), group([]), group([e(0, 1), e(1, 2)]), group([])]
    verdicts, rs, rho = many(lib, ctx, groups)
    assert verdicts == [1] * 6
    assert rs[0] == rs[2] == rs[3] == rs[5] == bytes(32)
    assert rho == rho_ref(rs, [len(g[1]) for g in groups])
    check_against_single(lib, ctx, groups, verdicts, rs)
    # k = 1 against the single call, valid and false
    g = block21.sidecar(33)
    verdicts, rs, _ = many(lib, ctx, [g])
    assert (verdicts[0], rs[0]) == single(lib, ctx, g) == (1, CO.verify_cell_kzg_proof_batch(*g, want_r=True)[1])
    g[3][0] = g1_plus_gen(g[3][0])
    verdicts, rs, _ = many(lib, ctx, [g])
    assert (verdicts[0], rs[0]) == single(lib, ctx, g) and verdicts[0] == 0
    # one-cell group, a repeated cell, mixed indices with non-adjacent duplicate commitments, a whole blob's 128 cells
    groups = [group([e(4, 100)]),
              group([e(2, 50), e(1, 2), e(2, 50)]),
              group([e(0, 3), e(1, 100), e(0, 64), e(1, 1), e(0, 3)]),
              group([e(7, i) for i in range(128)])]
    verdicts, rs, _ = many(lib, ctx, groups)
    assert verdicts == [1, 1, 1, 1]
    for i, g in enumerate(groups):
        assert rs[i] == CO.verify_cell_kzg_proof_batch(*g, want_r=True)[1], i
    check_against_single(lib, ctx, groups, verdicts, rs)
    # malformed calls: offsets that do not start at 0 / decrease, null verdicts
    off = (C.c_uint64 * 3)(0, 2, 1)
    out = C.create_string_buffer(2)
    z = bytes(48 * 2)
    assert lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, z, z, bytes(2 * CELL), z, C.cast(off, C.c_void_p), 2, out) == 1
    off = (C.c_uint64 * 2)(1, 2)
    assert lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, z, z, bytes(2 * CELL), z, C.cast(off, C.c_void_p), 1, out) == 1
    off = (C.c_uint64 * 2)(0, 2)
    assert lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, z, z, bytes(2 * CELL), z, C.cast(off, C.c_void_p), 1, None) == 1
    assert lib.kzgb200_verify_cell_kzg_proof_batch_many(ctx, None, None, None, None, C.cast(off, C.c_void_p), 1, out) == 1


def test_one_false_group_skips_fallback(K, settings, lib, ctx, block21):
    """with one group the combined check is that group's own (rho^0 = 1): a false group gets 0 without the per-group pass"""
    g = block21.sidecar(61)
    g[3][4] = g1_plus_gen(g[3][4])
    ms = (C.c_float * 8)()
    assert lib.kzgb200_set_profiling(ctx, 1) == 0
    try:
        assert many(lib, ctx, [g])[0] == [0]
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
        assert ms[6] > 0 and ms[7] == 0, list(ms)
        assert single(lib, ctx, g)[0] == 0
        assert lib.kzgb200_get_phase_ms(ctx, ms) == 0
        assert ms[6] > 0 and ms[7] == 0, list(ms)
    finally:
        lib.kzgb200_set_profiling(ctx, 0)


def test_large_group_beside_small_ones(K, settings, lib, ctx):
    blk = Block(K, settings, 128, 11)
    whole = group([blk.entry(b, i) for b in range(128) for i in range(128)])
    groups = [blk.sidecar(5, range(3)), whole, group([blk.entry(9, 9)]), blk.sidecar(70, range(10))]
    verdicts, rs, _ = many(lib, ctx, groups)
    assert verdicts == [1, 1, 1, 1]
    check_against_single(lib, ctx, groups, verdicts, rs)
    whole[3][12345] = g1_plus_gen(whole[3][12345])
    verdicts, rs, _ = many(lib, ctx, groups)
    assert verdicts == [1, 0, 1, 1]
    check_against_single(lib, ctx, groups, verdicts, rs)


def test_fallback_at_scale(K, settings, lib, ctx, block21):
    base = [block21.sidecar(i) for i in range(128)]
    for pattern in (lambda i: True, lambda i: i % 2 == 1):
        groups = [[list(x) for x in g] for g in base]
        for i, g in enumerate(groups):
            if pattern(i):
                j = i % 21
                g[3][j] = g1_plus_gen(g[3][j])
        verdicts, rs, _ = many(lib, ctx, groups)
        assert verdicts == [0 if pattern(i) else 1 for i in range(128)]
        check_against_single(lib, ctx, groups, verdicts, rs)


def test_seeded_random_groups(K, settings, lib, ctx, block21):
    rnd = random.Random(0x5eed)
    bad_points = [bytes(48), off_curve_point(), non_subgroup_point()]
    for _ in range(20):
        groups = []
        for _ in range(32):
            n = rnd.choice([0, 1, 2, 3, 5, 8, 21, 40])
            g = group([block21.entry(rnd.randrange(21), rnd.randrange(128)) for _ in range(n)])
            if n:
                kind, j = rnd.randrange(9), rnd.randrange(n)
                if kind == 0: g[3][j] = g1_plus_gen(g[3][j])
                elif kind == 1: g[0][j] = block21.commitment((block21.hcs.index(g[0][j]) // 48 + 1) % 21)
                elif kind == 2:
                    t = bytearray(g[2][j]); t[rnd.randrange(CELL)] ^= 1 << rnd.randrange(8); g[2][j] = bytes(t)
                elif kind == 3: g[3][j] = rnd.choice(bad_points)
                elif kind == 4: g[1][j] = rnd.choice([128, 255, (1 << 64) - 1])
                elif kind == 5:
                    o = 32 * rnd.randrange(64); t = bytearray(g[2][j]); t[o:o + 32] = b"\xff" * 32; g[2][j] = bytes(t)
            groups.append(g)
        verdicts, rs, rho = many(lib, ctx, groups)
        assert rho == rho_ref(rs, [len(g[1]) for g in groups])
        check_against_single(lib, ctx, groups, verdicts, rs)


def test_device_form(K, settings, lib, ctx, block21):
    import torch
    groups, _, _ = bad_args_groups(block21)
    tampered = [block21.sidecar(i) for i in range(8)]
    tampered[3][3][4] = g1_plus_gen(tampered[3][3][4])
    for gs in ([block21.sidecar(i) for i in range(128)], tampered, groups):
        verdicts, rs, rho = many(lib, ctx, gs)
        offs = [0]
        for g in gs:
            offs.append(offs[-1] + len(g[1]))
        dev = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        d_c = dev(b"".join(b"".join(g[0]) for g in gs))
        d_i = torch.tensor([i for g in gs for i in g[1]], dtype=torch.int64).cuda()
        d_ce = dev(b"".join(b"".join(g[2]) for g in gs))
        d_p = dev(b"".join(b"".join(g[3]) for g in gs))
        k = len(gs)
        off = (C.c_uint64 * (k + 1))(*offs)
        out = C.create_string_buffer(k)
        assert lib.kzgb200_verify_cell_kzg_proof_batch_many_device(ctx, d_c.data_ptr(), d_i.data_ptr(), d_ce.data_ptr(), d_p.data_ptr(),
                                                                   C.cast(off, C.c_void_p), k, out) == 0
        assert list(out.raw[:k]) == verdicts
        r, rho2 = C.create_string_buffer(32 * k), C.create_string_buffer(32)
        assert lib.kzgb200_last_cell_many_r(ctx, r, k, rho2) == 0
        assert [r.raw[32 * g:32 * g + 32] for g in range(k)] == rs and rho2.raw == rho


def test_custom_setup(K, settings, oracle):
    path = os.path.join(GOLDEN, "custom_setup.bin")
    rnd = random.Random(23)
    blobs = [b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096)) for _ in range(2)]
    oracle.use_setup(path)
    CO.use_setup(path)
    try:
        mono = b"".join(oracle.tau_power_g1(j) for j in range(64))
        cs = [oracle.blob_to_kzg_commitment(b) for b in blobs]
        cells = [CO.compute_cells(b) for b in blobs]
        ks = [0, 33, 101]
        groups = [group([[cs[b], i, cells[b][i], CO.compute_cell_kzg_proof(blobs[b], i)] for b in range(2)]) for i in ks]
        assert all(CO.verify_cell_kzg_proof_batch(*g) is True for g in groups)
    finally:
        oracle.use_setup(None)
        CO.use_setup(None)
    custom = K.KzgSettings.load_trusted_setup_file(path, g1_monomial_bytes=mono)
    try:
        lib, ctx = K.Library.get().dll, custom.cell_context(0)
        assert many(lib, ctx, groups)[0] == [1, 1, 1]
        groups[1][3][0], groups[1][3][1] = groups[1][3][1], groups[1][3][0]
        assert many(lib, ctx, groups)[0] == [1, 0, 1]
    finally:
        custom.close()


def test_python_api(K, settings, block21):
    P = K.KzgProof.verify_cell_kzg_proof_batch_many
    good = block21.sidecar(1)
    false = block21.sidecar(2)
    false[3][0] = g1_plus_gen(false[3][0])
    bad_idx = block21.sidecar(3)
    bad_idx[1][0] = 1 << 64                      # does not fit in u64: that batch is BadArgs
    neg_idx = block21.sidecar(4)
    neg_idx[1][1] = -1
    bad_pt = block21.sidecar(5)
    bad_pt[3][2] = bytes(48)
    typed = [good[0], good[1], [K.Cell.from_slice(x) for x in good[2]], [K.Bytes48.from_slice(p) for p in good[3]]]
    assert P([tuple(good), tuple(false), tuple(bad_idx), tuple(neg_idx), tuple(bad_pt), ([], [], [], []), tuple(typed)], settings) == \
        [True, False, None, None, None, True, True]
    assert P([], settings) == []
    for broken in ([good[0], good[1][:-1], good[2], good[3]], [good[0], good[1], good[2], good[3][:-1]],
                   [good[0], good[1], good[2][:-1] + [good[2][-1][:-1]], good[3]]):
        with pytest.raises(K.KzgError) as e:
            P([tuple(false), tuple(broken)], settings)
        assert e.value.kind == "InvalidBytesLength"
