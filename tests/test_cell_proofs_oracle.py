"""EIP-7594 cell proofs and recovery on the CPU (no GPU): the FK20 arrangement the GPU implements, checked "in the exponent" against
the direct quotient for every cell, and the C oracle's spec recovery against its pure-Python restatement and against compute_cells."""
import random

import pytest

from cell_oracle import cells as CO
from cell_oracle import pyref_cells as PC

Q = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def rand_blob(seed):
    rnd = random.Random(seed)
    return b"".join(rnd.randrange(Q).to_bytes(32, "big") for _ in range(4096))


@pytest.mark.parametrize("kind", ["random_a", "random_b", "degree_191", "x4095"])
def test_fk20_in_the_exponent_equals_direct_quotient(kind):
    rnd = random.Random(kind)
    if kind.startswith("random"):
        coeffs = [rnd.randrange(Q) for _ in range(4096)]
    elif kind == "degree_191":
        coeffs = [rnd.randrange(Q) for _ in range(192)] + [0] * (4096 - 192)
    else:
        coeffs = [0] * 4095 + [1]
    tau = rnd.randrange(Q)
    fk = PC.fk20_in_exponent(coeffs, tau)
    assert fk == [PC.cell_quotient_at(coeffs, tau, k) for k in range(128)]


def index_sets():
    rnd = random.Random(77)
    return {"first_half": list(range(64)), "second_half": list(range(64, 128)), "random64": rnd.sample(range(128), 64),
            "every_other": list(range(0, 128, 2)), "127": [k for k in range(128) if k != 37], "all": list(range(128)),
            "unsorted": rnd.sample(range(128), 90)}


@pytest.fixture(scope="module")
def blob_cells():
    blob = rand_blob(12)
    return blob, CO.compute_cells(blob)


@pytest.mark.parametrize("name", sorted(index_sets()))
def test_recovery_c_equals_python_and_compute_cells(name, blob_cells):
    _, cells = blob_cells
    idx = index_sets()[name]
    given = [cells[k] for k in idx]
    rec = CO.recover_cells(idx, given)
    assert rec == cells
    assert PC.recover_cells(idx, given) == rec


def test_recovery_inconsistent_input_c_equals_python(blob_cells):
    _, cells = blob_cells
    idx = random.Random(5).sample(range(128), 80)
    given = [cells[k] for k in idx]
    t = bytearray(given[7]); t[32 * 3 + 31] ^= 1
    given[7] = bytes(t)
    rec = CO.recover_cells(idx, given)
    assert rec is not None and rec != cells
    assert PC.recover_cells(idx, given) == rec
    assert CO.compute_cells(b"".join(rec[:64])) == rec           # the recovered cells are the extension of a blob


def test_recovery_bad_args(blob_cells):
    _, cells = blob_cells
    idx = list(range(0, 128, 2))
    assert CO.recover_cells(idx[:63], [cells[k] for k in idx[:63]]) is None
    assert CO.recover_cells(idx[:64] + [idx[0]], [cells[k] for k in idx[:64]] + [cells[idx[0]]]) is None
    assert CO.recover_cells(idx[:63] + [128], [cells[k] for k in idx[:64]]) is None
    t = bytearray(cells[idx[1]]); t[:32] = Q.to_bytes(32, "big")
    assert CO.recover_cells(idx, [cells[idx[0]], bytes(t)] + [cells[k] for k in idx[2:]]) is None
