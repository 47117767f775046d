"""FK20's inverse G1 DFT also yields the blob's commitment: output 0 is [p(tau)] once the fixed bases carry w_b[65] = [tau^(4032+b)]
(d = 63), and that entry leaves every proof unchanged.  Checked "in the exponent" (every [tau^j]G1 replaced by tau^j for a random tau)
on the arrangement the GPU uses, without a GPU."""
import random

import pytest

from cell_oracle import pyref_cells as PC

Q = PC.Q


def p_at(coeffs, tau):
    v = 0
    for c in reversed(coeffs):
        v = (v * tau + c) % Q
    return v


def polynomial(kind):
    rnd = random.Random(kind)
    if kind.startswith("random"):
        return [rnd.randrange(Q) for _ in range(4096)]
    if kind == "degree_191":
        return [rnd.randrange(Q) for _ in range(192)] + [0] * (4096 - 192)
    m = int(kind[1:])
    return [0] * m + [1] + [0] * (4095 - m)


@pytest.mark.parametrize("kind", ["random_a", "random_b", "x4095", "x4032", "degree_191"])
def test_output_0_is_the_commitment_and_the_proofs_are_the_quotients(kind):
    coeffs = polynomial(kind)
    tau = random.Random("tau " + kind).randrange(Q)
    commitment, proofs = PC.fk20_commitment_and_proofs_in_exponent(coeffs, tau)
    assert commitment == p_at(coeffs, tau)
    assert proofs == [PC.cell_quotient_at(coeffs, tau, k) for k in range(128)]
    assert PC.fk20_in_exponent(coeffs, tau) == proofs


def test_without_the_new_entry_output_0_misses_the_top_terms():
    coeffs = polynomial("x4095")
    tau = random.Random("tau x4095").randrange(Q)
    commitment, proofs = PC.fk20_commitment_and_proofs_in_exponent(coeffs, tau, d_max=62)
    assert commitment != p_at(coeffs, tau)
    assert commitment == 0                 # X^4095 has no term below 4032
    assert proofs == PC.fk20_commitment_and_proofs_in_exponent(coeffs, tau)[1]
