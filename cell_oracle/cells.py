"""ctypes binding of the EIP-7594 cell oracle (cell_oracle/kzg_cell_oracle.c).  TEST INFRASTRUCTURE ONLY.

May be imported by tests/ and tools/bench_cells.py; never by the product package.  Results are True / False / None (None =
the spec's verify_cell_kzg_proof_batch would fail an assertion: BadArgs).
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
SETUP_BIN = os.path.join(os.path.dirname(_HERE), "kzg_rs_b200", "data", "mainnet_setup.bin")
BYTES_PER_CELL, CELLS_PER_EXT_BLOB = 2048, 128


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "libkzg_cell_oracle.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
        _LIB.kzgco_init.argtypes = [C.c_char_p, C.c_size_t]
        _LIB.kzgco_compute_cells.argtypes = [C.c_char_p, C.c_char_p]
        _LIB.kzgco_compute_cell_kzg_proof.argtypes = [C.c_char_p, C.c_int, C.c_char_p]
        _LIB.kzgco_recover_cells.argtypes = [C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t, C.c_char_p]
        _LIB.kzgco_verify_cell_kzg_proof_batch.argtypes = [C.c_char_p, C.POINTER(C.c_uint64), C.c_char_p, C.c_char_p, C.c_size_t,
                                                           C.POINTER(C.c_int), C.c_char_p]
        use_setup(None)
    return _LIB


def use_setup(path=None):
    """(Re-)initialise with a trusted setup ("KZGS" container, >= 65 G2 points); None = the mainnet setup."""
    with open(path or SETUP_BIN, "rb") as fh:
        raw = fh.read()
    rc = lib().kzgco_init(raw, len(raw))
    if rc:
        raise RuntimeError("cell oracle setup load failed rc=%d" % rc)


def compute_cells(blob):
    """compute_cells: the 128 cells (2048 bytes each) of the extended blob, or None (non-canonical element)."""
    out = C.create_string_buffer(BYTES_PER_CELL * CELLS_PER_EXT_BLOB)
    rc = lib().kzgco_compute_cells(bytes(blob), out)
    return None if rc else [out.raw[BYTES_PER_CELL * k:BYTES_PER_CELL * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)]


def compute_cell_kzg_proof(blob, k):
    """The KZG multi-proof of cell k of the blob (48 bytes), or None."""
    out = C.create_string_buffer(48)
    rc = lib().kzgco_compute_cell_kzg_proof(bytes(blob), k, out)
    return None if rc else out.raw


def recover_cells(cell_indices, cells):
    """recover_cells_and_kzg_proofs' cells: the 128 cells (bytes) recovered from the given ones, or None (BadArgs)."""
    n = len(cell_indices)
    assert len(cells) == n
    if any(len(x) != BYTES_PER_CELL for x in cells) or any(not 0 <= i < 1 << 64 for i in cell_indices):
        return None
    out = C.create_string_buffer(BYTES_PER_CELL * CELLS_PER_EXT_BLOB)
    idx = (C.c_uint64 * max(n, 1))(*cell_indices)
    rc = lib().kzgco_recover_cells(idx, b"".join(cells), n, out)
    return None if rc else [out.raw[BYTES_PER_CELL * k:BYTES_PER_CELL * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)]


def verify_cell_kzg_proof_batch(commitments, cell_indices, cells, proofs, want_r=False):
    """verify_cell_kzg_proof_batch over sequences of bytes / ints: True / False / None (BadArgs); with want_r: (verdict, r),
    r = the batch challenge (32 bytes big-endian; None when n = 0 or on error)."""
    n = len(cell_indices)
    assert len(commitments) == len(cells) == len(proofs) == n
    if any(len(c) != 48 for c in commitments) or any(len(p) != 48 for p in proofs) or any(len(x) != BYTES_PER_CELL for x in cells):
        return (None, None) if want_r else None
    ok, r = C.c_int(0), C.create_string_buffer(32)
    idx = (C.c_uint64 * max(n, 1))(*cell_indices)
    rc = lib().kzgco_verify_cell_kzg_proof_batch(b"".join(commitments), idx, b"".join(cells), b"".join(proofs), n, C.byref(ok), r)
    v = None if rc else bool(ok.value)
    return (v, r.raw if v is not None and n else None) if want_r else v
