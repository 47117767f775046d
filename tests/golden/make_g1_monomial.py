#!/usr/bin/env python3
"""[tau^j]G1 for j < 192 (the monomial form of the mainnet setup's first 192 G1 points), derived from the Lagrange setup with
the CPU oracle like make_tau_powers.py:
    [tau^j]G1 = sum_i w_i^j * L_i(tau)G      (the commitment to X^j)
Output: kzg_rs_b200/data/g1_monomial.txt (192 compressed points, 48 bytes each, one hex line per point).  Cell proof verification (EIP-7594) needs j < 64 (the
interpolation commitment RLI); the cell workload generator commits to polynomials of degree < 192 with them.
Checks: the first 16 points equal tau_powers_g1.bin; e([tau^(j+1)]G1, G2) == e([tau^j]G1, [tau]G2) along the whole chain; and
e([tau^64]G1, G2) == e(G1, [tau^64]G2) against the setup's G2 point 64.
    python tests/golden/make_g1_monomial.py
"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O
from oracle import pyref as R

N = 192
pts = [O.tau_power_g1(j) for j in range(N)]
with open(os.path.join(ROOT, "kzg_rs_b200", "data", "tau_powers_g1.bin"), "rb") as fh:
    assert b"".join(pts[:16]) == fh.read()
assert pts[0] == R.g1_to_compressed(R.G1_GEN)
for j in range(N - 1):
    assert O.pairings_verify(pts[j + 1], 0, pts[j], 1) is True, j
with open(O.SETUP_BIN, "rb") as fh:
    raw = fh.read()
n1 = int.from_bytes(raw[4:8], "little")
g2_64 = R.g2_from_compressed(raw[12 + 48 * n1 + 64 * 96:12 + 48 * n1 + 65 * 96])[1]
t64 = R.g1_from_compressed(pts[64])[1]
assert R.pairings_verify(t64, R.G2_GEN, R.G1_GEN, g2_64) is True
with open(os.path.join(ROOT, "kzg_rs_b200", "data", "g1_monomial.txt"), "w") as fh:
    fh.write("".join(p.hex() + "\n" for p in pts))
print("wrote", len(pts), "points")
