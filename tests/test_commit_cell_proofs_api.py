"""CPU-side checks of compute_commitments_and_cell_proofs (a publisher's commitments and cell proofs in one call): a wrong blob length
raises InvalidBytesLength before any GPU work, and the C entry points reject malformed calls without touching a context."""
import ctypes as C
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOB = bytes(131072)


@pytest.fixture(scope="module")
def K():
    import kzg_rs_b200 as K
    return K


class NoContext:
    """Settings whose context must never be reached: a length error has to come first."""

    def __getattr__(self, name):
        raise AssertionError("GPU context requested before the length checks")


@pytest.mark.parametrize("length", [0, 131071, 131073, 2 * 131072])
@pytest.mark.parametrize("want_cells", [False, True])
def test_wrong_blob_length_raises_before_any_library_call(K, length, want_cells):
    for blobs in ([bytes(length)], [BLOB, bytes(length)], [BLOB, BLOB[:-1] + b"\1", bytes(length), BLOB]):
        with pytest.raises(K.KzgError) as e:
            K.compute_commitments_and_cell_proofs(blobs, NoContext(), want_cells=want_cells)
        assert e.value.kind == "InvalidBytesLength"


def test_c_abi_argument_checks_without_a_context(K):
    dll = K.Library.get().dll
    out = [C.create_string_buffer(n) for n in (48, 128 * 48, 128 * 2048)]
    status = C.create_string_buffer(b"\x07", 1)
    for fn in (dll.kzgb200_compute_commitments_and_cell_proofs, dll.kzgb200_compute_commitments_and_cell_proofs_device):
        assert fn(None, BLOB, 1, out[0], out[1], out[2], status) == 1                   # null context with a blob to do
        assert fn(None, None, 1, out[0], out[1], None, status) == 1
        assert fn(None, BLOB, 1, None, out[1], None, status) == 1
        assert fn(None, BLOB, 1, out[0], None, None, status) == 1
        assert fn(None, BLOB, 1, out[0], out[1], None, None) == 1
        assert fn(None, None, 0, None, None, None, None) == 0                           # nothing to do
    assert status.raw == b"\x07"


def test_no_cpu_fallback_without_gpu(K):
    """Without a device no context exists: the Python call raises InternalError."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    settings = K.KzgSettings.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "custom_setup.bin"))
    for blobs in ([BLOB], []):
        with pytest.raises(K.KzgError) as e:
            K.compute_commitments_and_cell_proofs(blobs, settings)
        assert e.value.kind == "InternalError"
