"""Pure-Python restatement of EIP-7594 compute_cells and of the cell batch challenge (consensus-specs Fulu,
polynomial-commitments-sampling.md): an independent cross-check of the C cell oracle.  TEST INFRASTRUCTURE ONLY."""
import hashlib

from oracle.pyref import Q, ROOT_OF_UNITY_4096, bit_reverse, blob_as_polynomial

FIELD_ELEMENTS_PER_CELL = 64
BYTES_PER_CELL = 2048
CELLS_PER_EXT_BLOB = 128
RANDOM_CHALLENGE_KZG_CELL_BATCH_DOMAIN = b"RCKZGCBATCH__V1_"
PRIMITIVE_ROOT_OF_UNITY = 7


def _fft(vals, w):
    """Plain recursive radix-2 DFT: out[k] = sum_m vals[m] w^(mk)."""
    n = len(vals)
    if n == 1:
        return list(vals)
    even, odd = _fft(vals[0::2], w * w % Q), _fft(vals[1::2], w * w % Q)
    out, x = [0] * n, 1
    for k in range(n // 2):
        t = x * odd[k] % Q
        out[k], out[k + n // 2] = (even[k] + t) % Q, (even[k] - t) % Q
        x = x * w % Q
    return out


def compute_cells(blob):
    """blob bytes -> 128 cells (bytes); KzgError on a non-canonical element."""
    poly = blob_as_polynomial(blob)
    w4096 = pow(PRIMITIVE_ROOT_OF_UNITY, (Q - 1) // 4096, Q)
    assert w4096 == ROOT_OF_UNITY_4096
    inv = pow(4096, Q - 2, Q)
    coeffs = [c * inv % Q for c in _fft([poly[bit_reverse(i)] for i in range(4096)], pow(w4096, Q - 2, Q))]
    w8192 = pow(PRIMITIVE_ROOT_OF_UNITY, (Q - 1) // 8192, Q)
    ext = _fft(coeffs + [0] * 4096, w8192)
    ext = [ext[bit_reverse(i, 13)] for i in range(8192)]
    flat = b"".join(v.to_bytes(32, 'big') for v in ext)
    return [flat[BYTES_PER_CELL * k:BYTES_PER_CELL * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)]


def cell_batch_challenge(commitments, cell_indices, cells, proofs):
    """compute_verify_cell_kzg_proof_batch_challenge with commitments deduplicated by bytes (first occurrence order)."""
    uniq = []
    for c in commitments:
        if c not in uniq:
            uniq.append(c)
    n = len(cell_indices)
    msg = RANDOM_CHALLENGE_KZG_CELL_BATCH_DOMAIN + (4096).to_bytes(8, 'big') + FIELD_ELEMENTS_PER_CELL.to_bytes(8, 'big') \
        + len(uniq).to_bytes(8, 'big') + n.to_bytes(8, 'big') + b"".join(uniq)
    for k in range(n):
        msg += uniq.index(commitments[k]).to_bytes(8, 'big') + cell_indices[k].to_bytes(8, 'big') + cells[k] + proofs[k]
    return int.from_bytes(hashlib.sha256(msg).digest(), 'big') % Q


def _ifft(vals, w):
    n = len(vals)
    inv = pow(n, Q - 2, Q)
    return [v * inv % Q for v in _fft(vals, pow(w, Q - 2, Q))]


def _coset_fft(vals, w, inv=False):
    """coset_fft_field with the shift PRIMITIVE_ROOT_OF_UNITY"""
    factor = pow(PRIMITIVE_ROOT_OF_UNITY, Q - 2, Q) if inv else PRIMITIVE_ROOT_OF_UNITY

    def shift(v):
        out, x = [], 1
        for a in v:
            out.append(a * x % Q)
            x = x * factor % Q
        return out
    return shift(_ifft(vals, w)) if inv else _fft(shift(vals), w)


def recover_cells(cell_indices, cells):
    """recover_cells_and_kzg_proofs' cells, restating recover_polynomialcoeff and compute_cells_and_kzg_proofs_polynomialcoeff;
    raises AssertionError / KzgError where the spec asserts."""
    assert CELLS_PER_EXT_BLOB // 2 <= len(cell_indices) <= CELLS_PER_EXT_BLOB and len(set(cell_indices)) == len(cell_indices)
    assert all(0 <= i < CELLS_PER_EXT_BLOB for i in cell_indices)
    n_ext = 2 * 4096
    w8192 = pow(PRIMITIVE_ROOT_OF_UNITY, (Q - 1) // n_ext, Q)
    rbo = [0] * n_ext
    for k, cell in zip(cell_indices, cells):
        vals = [int.from_bytes(cell[32 * j:32 * j + 32], 'big') for j in range(FIELD_ELEMENTS_PER_CELL)]
        assert all(v < Q for v in vals)
        rbo[k * FIELD_ELEMENTS_PER_CELL:(k + 1) * FIELD_ELEMENTS_PER_CELL] = vals
    ext = [rbo[bit_reverse(i, 13)] for i in range(n_ext)]
    w128 = pow(w8192, FIELD_ELEMENTS_PER_CELL, Q)
    short = [1]
    for k in range(CELLS_PER_EXT_BLOB):
        if k in cell_indices:
            continue
        x = pow(w128, bit_reverse(k, 7), Q)
        short = [((short[i - 1] if i else 0) - x * (short[i] if i < len(short) else 0)) % Q for i in range(len(short) + 1)]
    zcoef = [0] * n_ext
    for i, c in enumerate(short):
        zcoef[i * FIELD_ELEMENTS_PER_CELL] = c
    zev = _fft(zcoef, w8192)
    ez = _ifft([a * b % Q for a, b in zip(ext, zev)], w8192)
    ez_cos, z_cos = _coset_fft(ez, w8192), _coset_fft(zcoef, w8192)
    coeffs = _coset_fft([a * pow(b, Q - 2, Q) % Q for a, b in zip(ez_cos, z_cos)], w8192, inv=True)[:4096]
    out = _fft(coeffs + [0] * 4096, w8192)
    flat = b"".join(out[bit_reverse(i, 13)].to_bytes(32, 'big') for i in range(n_ext))
    return [flat[BYTES_PER_CELL * k:BYTES_PER_CELL * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)]


def fk20_in_exponent(coeffs, tau):
    """FK20 as the GPU computes it, with every [tau^j]G1 replaced by tau^j: the 128 "proofs" q_k(tau) of the polynomial with these
    4096 coefficients, in cell order.  u_b[a] = c_{64a+b} (zero-padded to 128), w_b[0] = tau^b, w_b[128-d] = tau^(64d+b)
    (d = 1..62); V[f] = sum_b DFT(u_b)[f] DFT(w_b)[f]; H_t = IDFT(V)[t+1] (t < 63); pi_k = DFT(H)[rev7(k)]."""
    w128 = pow(PRIMITIVE_ROOT_OF_UNITY, (Q - 1) // 128, Q)
    V = [0] * 128
    for b in range(FIELD_ELEMENTS_PER_CELL):
        u = [coeffs[64 * a + b] for a in range(64)] + [0] * 64
        w = [0] * 128
        w[0] = pow(tau, b, Q)
        for d in range(1, 63):
            w[128 - d] = pow(tau, 64 * d + b, Q)
        U, W = _fft(u, w128), _fft(w, w128)
        V = [(V[f] + U[f] * W[f]) % Q for f in range(128)]
    conv = _ifft(V, w128)
    H = conv[1:64] + [0] * 65
    out = _fft(H, w128)
    return [out[bit_reverse(k, 7)] for k in range(CELLS_PER_EXT_BLOB)]


def cell_quotient_at(coeffs, tau, k):
    """(p(tau) - r_k(tau)) / (tau^64 - s_k), r_k = p mod (X^64 - s_k), s_k = omega128^rev7(k): the direct value of cell k's proof"""
    s = pow(PRIMITIVE_ROOT_OF_UNITY, (Q - 1) // 128 * bit_reverse(k, 7), Q)
    p = r = 0
    for m in reversed(range(len(coeffs))):
        p = (p * tau + coeffs[m]) % Q
    for b in reversed(range(64)):
        rb = 0
        for a in reversed(range(64)):
            rb = (rb * s + coeffs[64 * a + b]) % Q
        r = (r * tau + rb) % Q
    return (p - r) * pow(pow(tau, 64, Q) - s, Q - 2, Q) % Q
