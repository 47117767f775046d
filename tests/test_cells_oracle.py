"""EIP-7594 cells on the CPU (no GPU): the C cell oracle's compute_cells / cell proofs / verify_cell_kzg_proof_batch against the
pure-Python restatement and against the polynomial identities they rest on, and the shipped monomial setup points."""
import os
import random

import pytest
from conftest import ROOT

from cell_oracle import cells as CO
from cell_oracle import pyref_cells as PC

Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))


def vals(cell_bytes):
    return [int.from_bytes(cell_bytes[32 * j:32 * j + 32], "big") for j in range(len(cell_bytes) // 32)]


@pytest.fixture(scope="module")
def valid_blob(vectors):
    """a full-degree fixture blob and its commitment (a valid verify_blob_kzg_proof case)"""
    from conftest import unhex
    full = lambda b: len(b) == 131072 and len({b[32 * i:32 * i + 32] for i in range(4096)}) == 4096
    c = [x for x in vectors["verify_blob_kzg_proof"] if x["output"] is True and full(vectors.blobs[x["blob"]])][0]
    return vectors.blobs[c["blob"]], unhex(c["commitment"])


def test_compute_cells_matches_pyref_and_extends_the_blob(oracle, valid_blob):
    from oracle import pyref as R
    for blob in (valid_blob[0], rand_blob(3)):
        cells = CO.compute_cells(blob)
        assert cells == PC.compute_cells(blob)
        assert b"".join(cells[:64]) == blob                          # the blob is the even half of the extended domain
        # all 8192 values lie on one polynomial of degree < 4096: the interpolants of the two halves agree at random points
        ext = vals(b"".join(cells))
        w8192 = pow(7, (Q - 1) // 8192, Q)
        roots = R.roots_of_unity()                                    # omega4096^rev12(i)

        def bary(v, shift, z):                                        # value at z of the interpolant of v on shift * roots
            y = z * pow(shift, Q - 2, Q) % Q
            acc = sum(v[i] * roots[i] % Q * pow(y - roots[i], Q - 2, Q) for i in range(4096)) % Q
            return acc * (pow(y, 4096, Q) - 1) % Q * pow(4096, Q - 2, Q) % Q
        rnd = random.Random(9)
        for _ in range(2):
            z = rnd.randrange(Q)
            assert bary(ext[:4096], 1, z) == bary(ext[4096:], w8192, z)
    bad = bytearray(rand_blob(4))
    bad[32 * 100:32 * 101] = Q.to_bytes(32, "big")
    assert CO.compute_cells(bytes(bad)) is None


def test_cell_batch_challenge_matches_pyref(oracle, valid_blob):
    from oracle import pyref as R
    blob, c = valid_blob
    cells = CO.compute_cells(blob)
    other = rand_blob(5)
    c2 = oracle.blob_to_kzg_commitment(other)
    cells2 = CO.compute_cells(other)
    idx = [3, 70, 3, 127]
    cs = [c, c2, c, c2]
    ce = [cells[3], cells2[70], cells[3], cells2[127]]
    ps = [CO.compute_cell_kzg_proof(blob, 3), CO.compute_cell_kzg_proof(other, 70), CO.compute_cell_kzg_proof(blob, 3),
          CO.compute_cell_kzg_proof(other, 127)]
    ok, r = CO.verify_cell_kzg_proof_batch(cs, idx, ce, ps, want_r=True)
    assert ok is True
    assert r == PC.cell_batch_challenge(cs, idx, ce, ps).to_bytes(32, "big")


def test_oracle_accepts_valid_and_rejects_tampered(oracle, valid_blob):
    blob, c = valid_blob
    other = rand_blob(6)
    c2 = oracle.blob_to_kzg_commitment(other)
    cells, cells2 = CO.compute_cells(blob), CO.compute_cells(other)
    ks = [0, 1, 64, 127]
    pr = {k: CO.compute_cell_kzg_proof(blob, k) for k in ks}
    pr2 = CO.compute_cell_kzg_proof(other, 1)
    V = CO.verify_cell_kzg_proof_batch
    cs, ce, ps = [c] * 4, [cells[k] for k in ks], [pr[k] for k in ks]
    assert V(cs, ks, ce, ps) is True
    assert V([c], [64], [cells[64]], [pr[64]]) is True                               # n = 1
    assert V(cs + [c2], ks + [1], ce + [cells2[1]], ps + [pr2]) is True              # two blobs
    assert V([], [], [], []) is True                                                  # n = 0
    assert V(cs, ks, ce, [ps[1], ps[0]] + ps[2:]) is False                            # proofs swapped between two cells
    t = bytearray(ce[2]); t[31] ^= 1
    assert V(cs, ks, ce[:2] + [bytes(t)] + ce[3:], ps) is False                      # one element changed
    assert V(cs, [0, 2, 64, 127], ce, ps) is False                                    # wrong cell index
    assert V([c, c2, c, c], ks, ce, ps) is False                                      # another blob's commitment
    # BadArgs
    t = bytearray(ce[0]); t[32 * 5:32 * 6] = Q.to_bytes(32, "big")
    assert V(cs, ks, [bytes(t)] + ce[1:], ps) is None                                 # element == q
    assert V(cs, [0, 1, 64, 128], ce, ps) is None                                     # cell index 128
    assert V([bytes(48)] + cs[1:], ks, ce, ps) is None                                # not a compressed point
    assert V(cs, ks, ce, ps[:3] + [bytes(48)]) is None


def test_cell_proof_quotient_identity(oracle):
    """the proof of cell k commits to (p - I_k) / (X^64 - h_k^64): e(pi, [tau^64 - h_k^64]) == e(C - [I_k(tau)], G2) is what the batch
    checks; here through the single-cell batch for every cell class (first / last of each half)"""
    blob = rand_blob(7)
    c = oracle.blob_to_kzg_commitment(blob)
    cells = CO.compute_cells(blob)
    for k in (63, 126):
        assert CO.verify_cell_kzg_proof_batch([c], [k], [cells[k]], [CO.compute_cell_kzg_proof(blob, k)]) is True


def test_g1_monomial_file_extends_tau_powers():
    data = os.path.join(ROOT, "kzg_rs_b200", "data")
    mono = b"".join(bytes.fromhex(x) for x in open(os.path.join(data, "g1_monomial.txt")).read().split())
    assert len(mono) == 192 * 48
    assert mono[:16 * 48] == open(os.path.join(data, "tau_powers_g1.bin"), "rb").read()
