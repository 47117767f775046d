"""CPU-side checks of recover_cells_and_kzg_proofs_many (many blobs, each recovered from its own cells): wrong list or byte lengths
raise InvalidBytesLength before any GPU work, and without a GPU the calls fail loudly instead of falling back."""
import ctypes as C
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CELL = bytes(2048)


@pytest.fixture(scope="module")
def K():
    import kzg_rs_b200 as K
    return K


class NoContext:
    """Settings whose context must never be reached: a length error has to come first."""

    def __getattr__(self, name):
        raise AssertionError("GPU context requested before the length checks")


def blob(n_indices, n_cells=None):
    n_cells = n_indices if n_cells is None else n_cells
    return list(range(n_indices)), [CELL] * n_cells


BROKEN = [
    blob(64, n_cells=63),
    blob(64, n_cells=65),
    blob(0, n_cells=1),
    blob(1, n_cells=0),
    (list(range(64)), [CELL] * 63 + [CELL[:-1]]),
    (list(range(64)), [CELL + b"\0"] + [CELL] * 63),
    ([0], [b""]),
]


@pytest.mark.parametrize("case", range(len(BROKEN)))
def test_wrong_lengths_raise_invalid_bytes_length(K, case):
    with pytest.raises(K.KzgError) as e:
        K.recover_cells_and_kzg_proofs_many([BROKEN[case]], NoContext())
    assert e.value.kind == "InvalidBytesLength"
    # one broken blob among good ones and bad-argument ones fails the whole call, before any GPU work
    with pytest.raises(K.KzgError) as e:
        K.recover_cells_and_kzg_proofs_many([blob(64), blob(63), BROKEN[case], blob(128), ([1 << 64] * 64, [CELL] * 64)], NoContext())
    assert e.value.kind == "InvalidBytesLength"


def test_no_cpu_fallback_without_gpu(K):
    """Without a device no context exists: the Python call raises InternalError, and the C entry points refuse a null context."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    settings = K.KzgSettings.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "custom_setup.bin"))
    for blobs in ([blob(64)], [blob(63)], []):
        with pytest.raises(K.KzgError) as e:
            K.recover_cells_and_kzg_proofs_many(blobs, settings)
        assert e.value.kind == "InternalError"
    dll = K.Library.get().dll
    idx = (C.c_uint64 * 64)(*range(64))
    off = (C.c_uint64 * 2)(0, 64)
    cells, proofs = C.create_string_buffer(128 * 2048), C.create_string_buffer(128 * 48)
    status = C.create_string_buffer(b"\x07", 1)
    assert dll.kzgb200_recover_cells_and_kzg_proofs_many(None, idx, CELL * 64, C.cast(off, C.c_void_p), 1, cells, proofs, status) == 1
    assert dll.kzgb200_recover_cells_and_kzg_proofs_many(None, None, None, None, 0, None, None, None) == 1
    assert dll.kzgb200_recover_cells_and_kzg_proofs_many_device(None, idx, None, C.cast(off, C.c_void_p), 1, None, None, status) == 1
    assert dll.kzgb200_recover_cells_and_kzg_proofs_many_device(None, None, None, None, 0, None, None, None) == 1
    assert status.raw == b"\x07"
