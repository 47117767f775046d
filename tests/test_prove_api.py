"""CPU-side checks of the EIP-4844 publisher calls (blob_to_kzg_commitment, compute_kzg_proof, compute_blob_kzg_proof): wrong
byte lengths raise InvalidBytesLength before any GPU work, and without a GPU the calls fail loudly instead of falling back."""
import ctypes as C
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOB, Z, COMMITMENT = bytes(131072), bytes(32), b"\xc0" + bytes(47)


@pytest.fixture(scope="module")
def K():
    import kzg_rs_b200 as K
    return K


class NoContext:
    """Settings whose context must never be reached: a length error has to come first."""

    def __getattr__(self, name):
        raise AssertionError("GPU context requested before the length checks")


@pytest.mark.parametrize("call", [
    lambda K, s: K.blob_to_kzg_commitment(BLOB[:-1], s),
    lambda K, s: K.blob_to_kzg_commitment(BLOB + b"\0", s),
    lambda K, s: K.compute_kzg_proof(BLOB[:-1], Z, s),
    lambda K, s: K.compute_kzg_proof(BLOB, Z[:31], s),
    lambda K, s: K.compute_kzg_proof(BLOB, Z + b"\0", s),
    lambda K, s: K.compute_blob_kzg_proof(BLOB + b"\0", COMMITMENT, s),
    lambda K, s: K.compute_blob_kzg_proof(BLOB, COMMITMENT[:47], s),
    lambda K, s: K.compute_blob_kzg_proof(BLOB, COMMITMENT + b"\0", s),
])
def test_wrong_lengths_raise_invalid_bytes_length(K, call):
    with pytest.raises(K.KzgError) as e:
        call(K, NoContext())
    assert e.value.kind == "InvalidBytesLength"


def test_no_cpu_fallback_without_gpu(K):
    """Without a device no context exists: kzgb200_create returns INTERNAL_ERROR, so every publisher call raises InternalError;
    the C entry points refuse a null context (BAD_ARGS)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    dll = K.Library.get().dll
    ctx = C.c_void_p()
    assert dll.kzgb200_create(C.byref(ctx), 0, bytes(192), 192) == 2      # KZGB200_INTERNAL_ERROR
    assert not ctx.value
    settings = K.KzgSettings.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "custom_setup.bin"))
    for call in (lambda: K.blob_to_kzg_commitment(BLOB, settings), lambda: K.compute_kzg_proof(BLOB, Z, settings),
                 lambda: K.compute_blob_kzg_proof(BLOB, COMMITMENT, settings), lambda: settings.commit_context(0)):
        with pytest.raises(K.KzgError) as e:
            call()
        assert e.value.kind == "InternalError"
    out = C.create_string_buffer(48)
    y = C.create_string_buffer(32)
    assert dll.kzgb200_blob_to_kzg_commitment(None, BLOB, out) == 1
    assert dll.kzgb200_compute_kzg_proof(None, BLOB, Z, out, y) == 1
    assert dll.kzgb200_compute_blob_kzg_proof(None, BLOB, COMMITMENT, out) == 1
    assert dll.kzgb200_compute_kzg_proof_batch_device(None, None, None, 0, None, None) == 1
