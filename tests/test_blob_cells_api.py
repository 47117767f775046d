"""CPU-side checks of verify_blob_cell_kzg_proof_batch[_many] (the cell proofs of whole blob transactions): wrong list or byte
lengths raise InvalidBytesLength before any GPU work, and without a GPU the calls fail loudly instead of falling back."""
import ctypes as C
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOB, POINT = bytes(131072), b"\xc0" + bytes(47)


@pytest.fixture(scope="module")
def K():
    import kzg_rs_b200 as K
    return K


class NoContext:
    """Settings whose context must never be reached: a length error has to come first."""

    def __getattr__(self, name):
        raise AssertionError("GPU context requested before the length checks")


def tx(n_blobs, n_commitments=None, n_proofs=None):
    n_commitments = n_blobs if n_commitments is None else n_commitments
    n_proofs = 128 * n_blobs if n_proofs is None else n_proofs
    return [BLOB] * n_blobs, [POINT] * n_commitments, [POINT] * n_proofs


BROKEN = [
    tx(2, n_commitments=1),
    tx(2, n_commitments=3),
    tx(2, n_proofs=255),
    tx(2, n_proofs=257),
    tx(0, n_commitments=1),
    tx(0, n_proofs=128),
    tx(1, n_proofs=0),
    ([BLOB[:-1]], [POINT], [POINT] * 128),
    ([BLOB + b"\0"], [POINT], [POINT] * 128),
    ([BLOB], [POINT[:47]], [POINT] * 128),
    ([BLOB], [POINT], [POINT] * 127 + [POINT + b"\0"]),
]


@pytest.mark.parametrize("case", range(len(BROKEN)))
def test_wrong_lengths_raise_invalid_bytes_length(K, case):
    with pytest.raises(K.KzgError) as e:
        K.KzgProof.verify_blob_cell_kzg_proof_batch(*BROKEN[case], NoContext())
    assert e.value.kind == "InvalidBytesLength"
    # one broken transaction among good ones fails the whole _many call, before any GPU work
    with pytest.raises(K.KzgError) as e:
        K.KzgProof.verify_blob_cell_kzg_proof_batch_many([tx(1), tx(0), BROKEN[case], tx(2)], NoContext())
    assert e.value.kind == "InvalidBytesLength"


def test_no_cpu_fallback_without_gpu(K):
    """Without a device no context exists: the Python calls raise InternalError, and the C entry points refuse a null context."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    settings = K.KzgSettings.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "custom_setup.bin"))
    for call in (lambda: K.KzgProof.verify_blob_cell_kzg_proof_batch(*tx(1), settings),
                 lambda: K.KzgProof.verify_blob_cell_kzg_proof_batch(*tx(0), settings),
                 lambda: K.KzgProof.verify_blob_cell_kzg_proof_batch_many([tx(1)], settings),
                 lambda: K.KzgProof.verify_blob_cell_kzg_proof_batch_many([], settings)):
        with pytest.raises(K.KzgError) as e:
            call()
        assert e.value.kind == "InternalError"
    dll = K.Library.get().dll
    ok = C.c_int(-1)
    off = (C.c_uint64 * 2)(0, 1)
    out = C.create_string_buffer(1)
    proofs = POINT * 128
    assert dll.kzgb200_verify_blob_cell_kzg_proof_batch(None, BLOB, 1, POINT, 1, proofs, 128, C.byref(ok)) == 1
    assert dll.kzgb200_verify_blob_cell_kzg_proof_batch(None, None, 0, None, 0, None, 0, C.byref(ok)) == 1
    assert dll.kzgb200_verify_blob_cell_kzg_proof_batch_device(None, None, None, None, 0, C.byref(ok)) == 1
    assert dll.kzgb200_verify_blob_cell_kzg_proof_batch_many(None, BLOB, POINT, proofs, C.cast(off, C.c_void_p), 1, out) == 1
    assert dll.kzgb200_verify_blob_cell_kzg_proof_batch_many_device(None, None, None, None, None, 0, out) == 1
    assert ok.value == -1
