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
