"""Python mirror of kzg-rs's public API for the verification path, bound to libkzgb200.so with ctypes.

Same names, argument meaning and error behaviour as the reference:
  KzgProof.verify_kzg_proof / verify_blob_kzg_proof / verify_blob_kzg_proof_batch   src/kzg_proof.rs:353-525
  KzgSettings.load_trusted_setup_file                                               src/trusted_setup.rs:94-98
  Blob / Bytes32 / Bytes48 (.from_slice length check, .as_slice)                    src/dtypes.rs:7-46
  KzgError                                                                          src/enums.rs:6-18
`Result<bool, KzgError>` becomes "return bool or raise KzgError".

There is no CPU path: loading fails loudly when the CUDA library has not been built, and every call
fails with KzgError(InternalError) when no sm_100 GPU is usable.
"""
import ctypes as C
import os
import struct
import threading

BYTES_PER_BLOB = 131072          # src/consts.rs:8
BYTES_PER_COMMITMENT = 48        # src/consts.rs:9
BYTES_PER_PROOF = 48             # src/consts.rs:10
BYTES_PER_FIELD_ELEMENT = 32     # src/consts.rs:3
BYTES_PER_CELL = 2048            # EIP-7594: 64 field elements of the extended blob
CELLS_PER_EXT_BLOB = 128
PARTIAL_BYTES = 352

_HERE = os.path.dirname(os.path.abspath(__file__))
_RC_KIND = {1: "BadArgs", 2: "InternalError", 3: "InvalidBytesLength", 5: "InvalidTrustedSetup"}
_RC_MSG = {1: "Failed to parse G1Affine from bytes", 2: "Internal error", 3: "Invalid commitments length",
           5: "Invalid trusted setup"}


class KzgError(Exception):
    """src/enums.rs:6-18.  .kind is one of BadArgs, InternalError, InvalidBytesLength, InvalidHexFormat,
    InvalidTrustedSetup."""

    def __init__(self, kind, msg=""):
        super().__init__(msg or kind)
        self.kind = kind


def lib_path():
    return os.path.join(_HERE, "libkzgb200.so")


class Library:
    """The C ABI (include/kzgb200.h).  One process-wide instance."""
    _inst = None
    _lock = threading.Lock()

    @classmethod
    def get(cls):
        with cls._lock:
            if cls._inst is None:
                cls._inst = cls()
            return cls._inst

    def __init__(self):
        path = lib_path()
        if not os.path.exists(path):
            raise RuntimeError("libkzgb200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "or `make -C kzg_rs_b200/csrc`); there is no CPU fallback")
        self.dll = d = C.CDLL(path)
        p, sz, ip = C.c_void_p, C.c_size_t, C.POINTER(C.c_int)
        d.kzgb200_create.argtypes = [C.POINTER(p), C.c_int, C.c_char_p, sz]
        d.kzgb200_destroy.argtypes = [p]
        d.kzgb200_last_error.argtypes = [p]
        d.kzgb200_last_error.restype = C.c_char_p
        d.kzgb200_verify_kzg_proof.argtypes = [p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, ip]
        d.kzgb200_verify_blob_kzg_proof.argtypes = [p, p, C.c_char_p, C.c_char_p, ip, p, p]
        d.kzgb200_verify_blob_kzg_proof_batch.argtypes = [p, p, sz, p, sz, p, sz, ip, p, p]
        d.kzgb200_verify_blob_kzg_proof_batch_device.argtypes = [p, p, p, p, sz, ip, p, p]
        d.kzgb200_verify_kzg_proof_many.argtypes = [p, p, p, p, p, sz, p]
        d.kzgb200_verify_kzg_proof_batch.argtypes = [p, p, p, p, p, sz, ip]
        d.kzgb200_verify_blob_kzg_proof_batch_each.argtypes = [p, p, p, p, sz, p, p, p]
        d.kzgb200_compute_challenge.argtypes = [p, p, C.c_char_p, C.c_char_p]
        d.kzgb200_evaluate_polynomial_in_evaluation_form.argtypes = [p, p, C.c_char_p, C.c_char_p]
        d.kzgb200_host_sha256.argtypes = [C.c_char_p, sz, C.c_char_p, C.c_int]
        pp, psz = C.POINTER(p), C.POINTER(sz)
        d.kzgb200_group_create.argtypes = [C.POINTER(p), C.POINTER(C.c_int), C.c_int, C.c_char_p, sz, sz]
        d.kzgb200_group_join.argtypes = [C.POINTER(p), C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_char_p, sz, sz]
        d.kzgb200_group_destroy.argtypes = [p]
        d.kzgb200_group_size.argtypes = [p]
        d.kzgb200_group_local_members.argtypes = [p]
        d.kzgb200_group_context.argtypes = [p, C.c_int]
        d.kzgb200_group_context.restype = p
        d.kzgb200_group_last_error.argtypes = [p]
        d.kzgb200_group_last_error.restype = C.c_char_p
        d.kzgb200_group_uses_peer_stores.argtypes = [p, C.c_int]
        d.kzgb200_group_verify_blob_kzg_proof_batch.argtypes = [p, p, sz, p, sz, p, sz, ip, p, p]
        d.kzgb200_group_verify_shards.argtypes = [p, pp, pp, pp, psz, C.c_int, ip, pp, pp]
        d.kzgb200_group_last_partials.argtypes = [p, C.c_char_p, sz]
        d.kzgb200_group_host_protocol_test.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, sz, sz, C.c_char_p]
        d.kzgb200_harness_generate.argtypes = [p, C.c_uint64, sz, C.c_int, C.c_char_p, p, p, p]
        d.kzgb200_set_profiling.argtypes = [p, C.c_int]
        d.kzgb200_get_phase_ms.argtypes = [p, C.POINTER(C.c_float)]
        d.kzgb200_stream.argtypes = [p]
        d.kzgb200_stream.restype = p
        d.kzgb200_set_transcript_mode.argtypes = [p, C.c_int]
        d.kzgb200_last_r.argtypes = [p, C.c_char_p]
        d.kzgb200_last_partial.argtypes = [p, C.c_char_p]
        d.kzgb200_debug_last_gt.argtypes = [p, C.c_char_p]
        d.kzgb200_debug_lines29w.argtypes = [p, C.c_char_p, sz]
        d.kzgb200_load_g1_lagrange.argtypes = [p, C.c_char_p, sz]
        d.kzgb200_blob_to_kzg_commitment_batch.argtypes = [p, p, sz, p]
        d.kzgb200_compute_blob_kzg_proof_batch.argtypes = [p, p, p, sz, p]
        d.kzgb200_blob_to_kzg_commitment.argtypes = [p, C.c_char_p, p]
        d.kzgb200_compute_kzg_proof.argtypes = [p, C.c_char_p, C.c_char_p, p, p]
        d.kzgb200_compute_blob_kzg_proof.argtypes = [p, C.c_char_p, C.c_char_p, p]
        d.kzgb200_compute_kzg_proof_batch_device.argtypes = [p, p, p, sz, p, p]
        u64 = C.c_uint64
        d.kzgb200_pipeline_create.argtypes = [C.POINTER(p), C.c_int, C.c_char_p, sz, C.c_int]
        d.kzgb200_pipeline_destroy.argtypes = [p]
        d.kzgb200_pipeline_depth.argtypes = [p]
        d.kzgb200_pipeline_context.argtypes = [p, C.c_int]
        d.kzgb200_pipeline_context.restype = p
        d.kzgb200_pipeline_submit.argtypes = [p, p, sz, p, sz, p, sz, p, p, C.POINTER(u64)]
        d.kzgb200_pipeline_submit_device.argtypes = [p, p, p, p, sz, p, p, C.POINTER(u64)]
        d.kzgb200_pipeline_wait.argtypes = [p, u64, ip]
        d.kzgb200_alloc_pinned.argtypes = [sz]
        d.kzgb200_alloc_pinned.restype = p
        d.kzgb200_free_pinned.argtypes = [p]
        d.kzgb200_load_cell_setup.argtypes = [p, C.c_char_p, sz, C.c_char_p]
        d.kzgb200_verify_cell_kzg_proof_batch.argtypes = [p, p, p, p, p, sz, ip]
        d.kzgb200_verify_cell_kzg_proof_batch_device.argtypes = [p, p, p, p, p, sz, ip]
        d.kzgb200_verify_cell_kzg_proof_batch_many.argtypes = [p, p, p, p, p, p, sz, p]
        d.kzgb200_verify_cell_kzg_proof_batch_many_device.argtypes = [p, p, p, p, p, p, sz, p]
        d.kzgb200_last_cell_many_r.argtypes = [p, p, sz, p]
        d.kzgb200_compute_cells.argtypes = [p, C.c_char_p, p]
        d.kzgb200_compute_cells_batch_device.argtypes = [p, p, sz, p]
        d.kzgb200_harness_generate_cells.argtypes = [p, C.c_uint64, sz, C.c_int, C.c_char_p, p, p, p]
        d.kzgb200_load_cell_proof_setup.argtypes = [p, C.c_char_p, sz]
        d.kzgb200_cell_proof_monomial.argtypes = [p, p, sz]
        d.kzgb200_compute_cells_and_kzg_proofs.argtypes = [p, C.c_char_p, p, p]
        d.kzgb200_compute_cells_and_kzg_proofs_batch_device.argtypes = [p, p, sz, p, p]
        d.kzgb200_recover_cells_and_kzg_proofs.argtypes = [p, p, p, sz, p, p]
        d.kzgb200_recover_cells_and_kzg_proofs_batch_device.argtypes = [p, p, sz, p, sz, p, p]


def _raise(rc, ctx=None, msg=None):
    kind = _RC_KIND.get(rc, "InternalError")
    if msg is None:
        msg = _RC_MSG.get(rc, "Internal error")
        if kind == "InternalError" and ctx is not None:
            detail = Library.get().dll.kzgb200_last_error(ctx)
            if detail:
                msg += ": " + detail.decode(errors="replace")
    raise KzgError(kind, msg)


class _BytesN:
    SIZE = 0

    def __init__(self, data):
        self._b = bytes(data)

    @classmethod
    def from_slice(cls, data):
        if len(data) != cls.SIZE:   # src/dtypes.rs:20-24
            raise KzgError("InvalidBytesLength", "Invalid slice length")
        return cls(data)

    @classmethod
    def from_hex(cls, s):
        try:
            raw = bytes.fromhex(s[2:] if s.startswith("0x") else s)
        except ValueError as e:
            raise KzgError("InvalidHexFormat", "Failed to decode hex: %s" % e)
        return cls.from_slice(raw)

    def as_slice(self):
        return self._b

    def __bytes__(self):
        return self._b

    def __len__(self):
        return len(self._b)


class Bytes32(_BytesN):
    SIZE = 32


class Bytes48(_BytesN):
    SIZE = 48


class Blob(_BytesN):
    SIZE = BYTES_PER_BLOB


class Cell(_BytesN):
    """EIP-7594 cell: 64 field elements (32 bytes big-endian each) of the extended blob."""
    SIZE = BYTES_PER_CELL


class KzgSettings:
    """src/trusted_setup.rs:44-50.  Holds the setup and one device context per GPU (created on first use:
    the device-resident tables -- roots of unity, Miller-loop lines of g2_points[0..2] -- are built there)."""
    _default = None
    _dlock = threading.Lock()

    def __init__(self, g1_lagrange_bytes, g2_monomial_bytes, g1_monomial_bytes=None):
        self.g1_lagrange_bytes = g1_lagrange_bytes      # 4096 x 48 (file order); unused by verification
        self.g2_monomial_bytes = g2_monomial_bytes      # 65 x 96; blob verification reads [0] and [1], cell verification [64]
        # [tau^j]G1, j >= 64, compressed: cell verification needs j < 64.  None: the shipped points when this is the mainnet setup
        self.g1_monomial_bytes = g1_monomial_bytes
        self._ctx = {}
        self._cells = set()
        self._proofs = set()
        self._commit = set()
        self._lock = threading.Lock()

    @classmethod
    def load_trusted_setup_file(cls, path=None, g1_monomial_bytes=None):
        """Default: the embedded mainnet setup (the reference embeds it at build time, build.rs:23-87).  g1_monomial_bytes: the
        setup's [tau^j]G1 (j < 64 at least) for cell proofs under a custom setup."""
        if path is None:
            with cls._dlock:
                if cls._default is None:
                    cls._default = cls._load(os.path.join(_HERE, "data", "mainnet_setup.bin"))
                return cls._default
        s = cls._load(path)
        s.g1_monomial_bytes = g1_monomial_bytes
        return s

    @classmethod
    def _load(cls, path):
        with open(path, "rb") as fh:
            raw = fh.read()
        if raw[:4] == b"KZGS":
            n1, n2 = struct.unpack("<II", raw[4:12])
            if len(raw) != 12 + n1 * 48 + n2 * 96 or n2 < 2:
                raise KzgError("InvalidTrustedSetup", "Invalid trusted setup")
            return cls(raw[12:12 + n1 * 48], raw[12 + n1 * 48:])
        # c-kzg text format: n1, n2, then hex lines
        try:
            tok = raw.decode().split()
            n1, n2 = int(tok[0]), int(tok[1])
            g1 = b"".join(bytes.fromhex(x) for x in tok[2:2 + n1])
            g2 = b"".join(bytes.fromhex(x) for x in tok[2 + n1:2 + n1 + n2])
        except (ValueError, IndexError):
            raise KzgError("InvalidTrustedSetup", "Invalid trusted setup")
        if len(g1) != n1 * 48 or len(g2) != n2 * 96 or n2 < 2:
            raise KzgError("InvalidTrustedSetup", "Invalid trusted setup")
        return cls(g1, g2)

    def context(self, device=0):
        with self._lock:
            if device not in self._ctx:
                lib = Library.get().dll
                h = C.c_void_p()
                rc = lib.kzgb200_create(C.byref(h), device, self.g2_monomial_bytes[:192], 192)
                if rc:
                    _raise(rc, msg="kzgb200_create failed (rc=%d): no usable sm_100 GPU or invalid setup" % rc if rc == 2 else None)
                self._ctx[device] = h
            return self._ctx[device]

    def _monomial_points(self):
        if self.g1_monomial_bytes is not None:
            return self.g1_monomial_bytes
        with open(os.path.join(_HERE, "data", "mainnet_setup.bin"), "rb") as fh:
            raw = fh.read()
        n1 = struct.unpack("<I", raw[4:8])[0]
        if self.g1_lagrange_bytes == raw[12:12 + n1 * 48] and self.g2_monomial_bytes[:65 * 96] == raw[12 + n1 * 48:12 + n1 * 48 + 65 * 96]:
            return mainnet_g1_monomial()
        raise KzgError("InvalidTrustedSetup", "cell proofs need the setup's monomial G1 points (g1_monomial_bytes)")

    def cell_context(self, device=0):
        """The device context with the cell tables loaded (EIP-7594: [tau^j]G1, j < 64, and g2_monomial[64])."""
        ctx = self.context(device)
        with self._lock:
            if device not in self._cells:
                if len(self.g2_monomial_bytes) < 65 * 96:
                    raise KzgError("InvalidTrustedSetup", "cell proofs need the setup's G2 point 64")
                g1m = self._monomial_points()
                rc = Library.get().dll.kzgb200_load_cell_setup(ctx, g1m, len(g1m) // 48, self.g2_monomial_bytes[64 * 96:65 * 96])
                if rc:
                    _raise(rc, ctx)
                self._cells.add(device)
        return ctx

    def cell_proof_context(self, device=0):
        """The cell context with the proof setup loaded as well (compute / recover cells and proofs): every [tau^j]G1, j < 4096,
        derived on the GPU from g1_lagrange_bytes, and the FK20 tables (3.3 GB of device memory)."""
        ctx = self.cell_context(device)
        with self._lock:
            if device not in self._proofs:
                if len(self.g1_lagrange_bytes) != 4096 * 48:
                    raise KzgError("InvalidTrustedSetup", "cell proofs need the setup's 4096 Lagrange G1 points")
                rc = Library.get().dll.kzgb200_load_cell_proof_setup(ctx, self.g1_lagrange_bytes, 4096)
                if rc:
                    _raise(rc, ctx)
                self._proofs.add(device)
        return ctx

    def commit_context(self, device=0):
        """The device context with the Lagrange window table loaded (blob_to_kzg_commitment, compute_kzg_proof,
        compute_blob_kzg_proof): 4.8 GB of device memory, built once from g1_lagrange_bytes."""
        ctx = self.context(device)
        with self._lock:
            if device not in self._commit:
                if len(self.g1_lagrange_bytes) != 4096 * 48:
                    raise KzgError("InvalidTrustedSetup", "commitments and proofs need the setup's 4096 Lagrange G1 points")
                rc = Library.get().dll.kzgb200_load_g1_lagrange(ctx, self.g1_lagrange_bytes, 4096)
                if rc:
                    _raise(rc, ctx)
                self._commit.add(device)
        return ctx

    def close(self):
        with self._lock:
            for h in self._ctx.values():
                Library.get().dll.kzgb200_destroy(h)
            self._ctx = {}
            self._cells = set()
            self._proofs = set()
            self._commit = set()


def mainnet_g1_monomial():
    """[tau^j]G1, j < 192, of the mainnet setup: 192 x 48 bytes, compressed (kzg_rs_b200/data/g1_monomial.txt, one hex point per line)."""
    with open(os.path.join(_HERE, "data", "g1_monomial.txt")) as fh:
        return b"".join(bytes.fromhex(line) for line in fh.read().split())


def _b(x, size, what):
    b = x.as_slice() if isinstance(x, _BytesN) else bytes(x)
    if len(b) != size:
        raise KzgError("InvalidBytesLength", "Invalid slice length")
    return b


class KzgProof:
    """src/kzg_proof.rs:350-526."""

    @staticmethod
    def verify_kzg_proof(commitment_bytes, z_bytes, y_bytes, proof_bytes, kzg_settings, device=0):
        c, z = _b(commitment_bytes, 48, "commitment"), _b(z_bytes, 32, "z")
        y, p = _b(y_bytes, 32, "y"), _b(proof_bytes, 48, "proof")
        ctx, ok = kzg_settings.context(device), C.c_int(0)
        rc = Library.get().dll.kzgb200_verify_kzg_proof(ctx, c, z, y, p, C.byref(ok))
        if rc:
            _raise(rc, ctx)
        return bool(ok.value)

    @staticmethod
    def verify_blob_kzg_proof(blob, commitment_bytes, proof_bytes, kzg_settings, device=0, want_zy=False):
        b, c, p = _b(blob, BYTES_PER_BLOB, "blob"), _b(commitment_bytes, 48, "commitment"), _b(proof_bytes, 48, "proof")
        ctx, ok = kzg_settings.context(device), C.c_int(0)
        z, y = C.create_string_buffer(32), C.create_string_buffer(32)
        rc = Library.get().dll.kzgb200_verify_blob_kzg_proof(ctx, b, c, p, C.byref(ok), z, y)
        if rc:
            _raise(rc, ctx)
        return (bool(ok.value), z.raw, y.raw) if want_zy else bool(ok.value)

    @staticmethod
    def verify_blob_kzg_proof_batch(blobs, commitments_bytes, proofs_bytes, kzg_settings, device=0, want_zy=False):
        """blobs / commitments_bytes / proofs_bytes: sequences (the reference's three Vecs)."""
        bl = [_b(x, BYTES_PER_BLOB, "blob") for x in blobs]
        cs = [_b(x, 48, "commitment") for x in commitments_bytes]
        ps = [_b(x, 48, "proof") for x in proofs_bytes]
        return KzgProof.verify_blob_kzg_proof_batch_raw(b"".join(bl), len(bl), b"".join(cs), len(cs), b"".join(ps), len(ps),
                                                        kzg_settings, device, want_zy)

    @staticmethod
    def verify_blob_kzg_proof_batch_raw(blobs, n_blobs, commitments, n_commitments, proofs, n_proofs, kzg_settings,
                                        device=0, want_zy=False):
        """Contiguous host buffers (bytes / ctypes arrays / integer addresses), exactly what the C ABI takes."""
        ctx, ok = kzg_settings.context(device), C.c_int(0)
        z = C.create_string_buffer(32 * max(n_blobs, 1)) if want_zy else None
        y = C.create_string_buffer(32 * max(n_blobs, 1)) if want_zy else None
        rc = Library.get().dll.kzgb200_verify_blob_kzg_proof_batch(ctx, _ptr(blobs), n_blobs, _ptr(commitments), n_commitments,
                                                                   _ptr(proofs), n_proofs, C.byref(ok), z, y)
        if rc:
            _raise(rc, ctx, "Invalid commitments length" if rc == 3 and n_blobs != n_commitments else
                   ("Invalid proofs length" if rc == 3 else None))
        if want_zy:
            zs = [z.raw[32 * i:32 * i + 32] for i in range(n_blobs)]
            ys = [y.raw[32 * i:32 * i + 32] for i in range(n_blobs)]
            return bool(ok.value), zs, ys
        return bool(ok.value)

    @staticmethod
    def verify_kzg_proof_batch(commitments, zs, ys, proofs, n, kzg_settings, device=0):
        """src/kzg_proof.rs:399-444 on already-parsed inputs in the reference's in-memory layout: commitments / proofs =
        n x 104 bytes (G1Affine: x, y as 6 x u64 Montgomery limbs, infinity byte, padding), zs / ys = n x 32 bytes (Scalar:
        4 x u64 Montgomery limbs).  Contiguous host buffers."""
        ctx, ok = kzg_settings.context(device), C.c_int(0)
        rc = Library.get().dll.kzgb200_verify_kzg_proof_batch(ctx, _ptr(commitments), _ptr(zs), _ptr(ys), _ptr(proofs), n, C.byref(ok))
        if rc:
            _raise(rc, ctx)
        return bool(ok.value)

    @staticmethod
    def verify_blob_kzg_proof_batch_each(blobs, commitments, proofs, n, kzg_settings, device=0, want_zy=False):
        """Per-blob verdicts of a batch (contiguous host buffers): list of True / False / None, None = the reference's
        verify_blob_kzg_proof would return Err(BadArgs) for that blob."""
        ctx = kzg_settings.context(device)
        out = C.create_string_buffer(max(n, 1))
        z = C.create_string_buffer(32 * max(n, 1)) if want_zy else None
        y = C.create_string_buffer(32 * max(n, 1)) if want_zy else None
        rc = Library.get().dll.kzgb200_verify_blob_kzg_proof_batch_each(ctx, _ptr(blobs), _ptr(commitments), _ptr(proofs), n, out, z, y)
        if rc:
            _raise(rc, ctx)
        verdicts = [{0: False, 1: True, 2: None}[v] for v in out.raw[:n]]
        return (verdicts, z.raw, y.raw) if want_zy else verdicts

    @staticmethod
    def verify_kzg_proof_many(commitments, zs, ys, proofs, m, kzg_settings, device=0):
        """m independent (C, z, y, proof) tuples in contiguous buffers -> bytes of m verdicts (0/1/2=BadArgs)."""
        ctx = kzg_settings.context(device)
        out = C.create_string_buffer(max(m, 1))
        rc = Library.get().dll.kzgb200_verify_kzg_proof_many(ctx, _ptr(commitments), _ptr(zs), _ptr(ys), _ptr(proofs), m, out)
        if rc:
            _raise(rc, ctx)
        return out.raw[:m]


    @staticmethod
    def verify_cell_kzg_proof_batch(commitments_bytes, cell_indices, cells, proofs_bytes, kzg_settings, device=0):
        """EIP-7594 verify_cell_kzg_proof_batch: commitments_bytes / cell_indices / cells / proofs_bytes are sequences of one
        entry per cell (commitment of the cell's blob, its index < 128, the cell, its proof).  Mismatched lengths ->
        KzgError(InvalidBytesLength); an index >= 128, a non-canonical cell element or an invalid point -> KzgError(BadArgs)."""
        n = len(cell_indices)
        if not (len(commitments_bytes) == len(cells) == len(proofs_bytes) == n):
            raise KzgError("InvalidBytesLength", "Invalid cells / commitments / proofs length")
        cs = b"".join(_b(x, 48, "commitment") for x in commitments_bytes)
        ce = b"".join(_b(x, BYTES_PER_CELL, "cell") for x in cells)
        ps = b"".join(_b(x, 48, "proof") for x in proofs_bytes)
        if any(not 0 <= int(i) < 1 << 64 for i in cell_indices):
            raise KzgError("BadArgs", "Invalid cell index")
        idx = (C.c_uint64 * max(n, 1))(*[int(i) for i in cell_indices])
        ctx, ok = kzg_settings.cell_context(device), C.c_int(0)
        rc = Library.get().dll.kzgb200_verify_cell_kzg_proof_batch(ctx, _ptr(cs), C.cast(idx, C.c_void_p), _ptr(ce), _ptr(ps), n, C.byref(ok))
        if rc:
            _raise(rc, ctx, "Failed to parse cell / G1Affine / cell index" if rc == 1 else None)
        return bool(ok.value)

    @staticmethod
    def verify_cell_kzg_proof_batch_many(batches, kzg_settings, device=0):
        """Many independent verify_cell_kzg_proof_batch calls in one GPU call (e.g. one per data column sidecar): batches is a
        sequence of (commitments_bytes, cell_indices, cells, proofs_bytes), each as for verify_cell_kzg_proof_batch.  Returns one
        verdict per batch: True / False / None, None = that batch alone would raise BadArgs; a bad batch does not change another's
        verdict.  Mismatched lengths inside a batch or wrong byte lengths -> KzgError(InvalidBytesLength) for the whole call."""
        cs, ce, ps, idx, offs = [], [], [], [], [0]
        for commitments_bytes, cell_indices, cells, proofs_bytes in batches:
            n = len(cell_indices)
            if not (len(commitments_bytes) == len(cells) == len(proofs_bytes) == n):
                raise KzgError("InvalidBytesLength", "Invalid cells / commitments / proofs length")
            cs += [_b(x, 48, "commitment") for x in commitments_bytes]
            ce += [_b(x, BYTES_PER_CELL, "cell") for x in cells]
            ps += [_b(x, 48, "proof") for x in proofs_bytes]
            idx += [int(i) if 0 <= int(i) < 1 << 64 else (1 << 64) - 1 for i in cell_indices]   # out of range: that batch gets None
            offs.append(offs[-1] + n)
        k, n = len(offs) - 1, offs[-1]
        ctx = kzg_settings.cell_context(device)
        out = C.create_string_buffer(max(k, 1))
        off = (C.c_uint64 * (k + 1))(*offs)
        ia = (C.c_uint64 * max(n, 1))(*idx)
        rc = Library.get().dll.kzgb200_verify_cell_kzg_proof_batch_many(ctx, _ptr(b"".join(cs)), C.cast(ia, C.c_void_p), _ptr(b"".join(ce)),
                                                                        _ptr(b"".join(ps)), C.cast(off, C.c_void_p), k, out)
        if rc:
            _raise(rc, ctx)
        return [{0: False, 1: True, 2: None}[v] for v in out.raw[:k]]


def compute_cells(blob, kzg_settings, device=0):
    """EIP-7594 compute_cells: the 128 cells (2048 bytes each) of the blob's extension; BadArgs on a non-canonical element."""
    b = _b(blob, BYTES_PER_BLOB, "blob")
    ctx = kzg_settings.cell_context(device)
    out = C.create_string_buffer(BYTES_PER_CELL * CELLS_PER_EXT_BLOB)
    rc = Library.get().dll.kzgb200_compute_cells(ctx, b, out)
    if rc:
        _raise(rc, ctx, "Failed to parse blob" if rc == 1 else None)
    raw = out.raw
    return [raw[BYTES_PER_CELL * k:BYTES_PER_CELL * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)]


def _cells_and_proofs(raw_cells, raw_proofs):
    return ([raw_cells[BYTES_PER_CELL * k:BYTES_PER_CELL * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)],
            [raw_proofs[BYTES_PER_PROOF * k:BYTES_PER_PROOF * (k + 1)] for k in range(CELLS_PER_EXT_BLOB)])


def compute_cells_and_kzg_proofs(blob, kzg_settings, device=0):
    """EIP-7594 compute_cells_and_kzg_proofs: (cells, proofs), 128 of each (2048 / 48 bytes), the proofs by FK20 on the GPU;
    BadArgs on a non-canonical element."""
    b = _b(blob, BYTES_PER_BLOB, "blob")
    ctx = kzg_settings.cell_proof_context(device)
    cells = C.create_string_buffer(BYTES_PER_CELL * CELLS_PER_EXT_BLOB)
    proofs = C.create_string_buffer(BYTES_PER_PROOF * CELLS_PER_EXT_BLOB)
    rc = Library.get().dll.kzgb200_compute_cells_and_kzg_proofs(ctx, b, cells, proofs)
    if rc:
        _raise(rc, ctx, "Failed to parse blob" if rc == 1 else None)
    return _cells_and_proofs(cells.raw, proofs.raw)


def recover_cells_and_kzg_proofs(cell_indices, cells, kzg_settings, device=0):
    """EIP-7594 recover_cells_and_kzg_proofs: all 128 (cells, proofs) of a blob from 64 or more of its cells, in any order.
    Mismatched lengths -> KzgError(InvalidBytesLength); fewer than 64 or more than 128 cells, an index >= 128, a repeated index or a
    non-canonical element -> KzgError(BadArgs)."""
    n = len(cell_indices)
    if len(cells) != n:
        raise KzgError("InvalidBytesLength", "Invalid cells / cell indices length")
    ce = b"".join(_b(x, BYTES_PER_CELL, "cell") for x in cells)
    if any(not 0 <= int(i) < 1 << 64 for i in cell_indices):
        raise KzgError("BadArgs", "Invalid cell index")
    idx = (C.c_uint64 * max(n, 1))(*[int(i) for i in cell_indices])
    ctx = kzg_settings.cell_proof_context(device)
    out_cells = C.create_string_buffer(BYTES_PER_CELL * CELLS_PER_EXT_BLOB)
    out_proofs = C.create_string_buffer(BYTES_PER_PROOF * CELLS_PER_EXT_BLOB)
    rc = Library.get().dll.kzgb200_recover_cells_and_kzg_proofs(ctx, C.cast(idx, C.c_void_p), _ptr(ce), n, out_cells, out_proofs)
    if rc:
        _raise(rc, ctx, "Invalid cell indices / cells" if rc == 1 else None)
    return _cells_and_proofs(out_cells.raw, out_proofs.raw)


def blob_to_kzg_commitment(blob, kzg_settings, device=0):
    """EIP-4844 blob_to_kzg_commitment: the blob's commitment, 48 bytes compressed; BadArgs on a non-canonical element."""
    b = _b(blob, BYTES_PER_BLOB, "blob")
    ctx, out = kzg_settings.commit_context(device), C.create_string_buffer(48)
    rc = Library.get().dll.kzgb200_blob_to_kzg_commitment(ctx, b, out)
    if rc:
        _raise(rc, ctx, "Failed to parse blob" if rc == 1 else None)
    return out.raw


def compute_kzg_proof(blob, z_bytes, kzg_settings, device=0):
    """EIP-4844 compute_kzg_proof: (proof, y) for the blob's polynomial at z, y = p(z) (48 and 32 bytes); z may be a point of
    the evaluation domain.  BadArgs on a non-canonical blob element or z."""
    b, z = _b(blob, BYTES_PER_BLOB, "blob"), _b(z_bytes, 32, "z")
    ctx = kzg_settings.commit_context(device)
    proof, y = C.create_string_buffer(48), C.create_string_buffer(32)
    rc = Library.get().dll.kzgb200_compute_kzg_proof(ctx, b, z, proof, y)
    if rc:
        _raise(rc, ctx, "Failed to parse blob / z" if rc == 1 else None)
    return proof.raw, y.raw


def compute_blob_kzg_proof(blob, commitment_bytes, kzg_settings, device=0):
    """EIP-4844 compute_blob_kzg_proof: the proof at the Fiat-Shamir challenge of (blob, commitment), 48 bytes.  BadArgs on a
    non-canonical blob element or a commitment that is not a valid compressed point of the G1 subgroup."""
    b, c = _b(blob, BYTES_PER_BLOB, "blob"), _b(commitment_bytes, 48, "commitment")
    ctx, out = kzg_settings.commit_context(device), C.create_string_buffer(48)
    rc = Library.get().dll.kzgb200_compute_blob_kzg_proof(ctx, b, c, out)
    if rc:
        _raise(rc, ctx, "Failed to parse blob / commitment" if rc == 1 else None)
    return out.raw


def compute_challenge(blob, commitment_bytes, kzg_settings, device=0):
    """src/kzg_proof.rs:46-72 (re-exported by src/lib.rs:8): the Fiat-Shamir challenge z, 32 bytes big-endian."""
    b, c = _b(blob, BYTES_PER_BLOB, "blob"), _b(commitment_bytes, 48, "commitment")
    ctx, z = kzg_settings.context(device), C.create_string_buffer(32)
    rc = Library.get().dll.kzgb200_compute_challenge(ctx, b, c, z)
    if rc:
        _raise(rc, ctx)
    return z.raw


def evaluate_polynomial_in_evaluation_form(blob, z_bytes, kzg_settings, device=0):
    """src/kzg_proof.rs:94-133 (re-exported by src/lib.rs:8) on the blob's 4096 field elements at z: y, 32 bytes big-endian."""
    b, z = _b(blob, BYTES_PER_BLOB, "blob"), _b(z_bytes, 32, "z")
    ctx, y = kzg_settings.context(device), C.create_string_buffer(32)
    rc = Library.get().dll.kzgb200_evaluate_polynomial_in_evaluation_form(ctx, b, z, y)
    if rc:
        _raise(rc, ctx)
    return y.raw


TRANSCRIPT_EXACT, TRANSCRIPT_TREE, TRANSCRIPT_EXACT_DEVICE = 0, 1, 2


class DeviceGroup:
    """Blob-sharded batches over several GPUs (include/kzgb200.h "multi-GPU").

        DeviceGroup.create(settings, [0, 1, ..., 7], max_blobs_per_device)       one process drives all GPUs
        DeviceGroup.join(settings, session, rank, world, device, max_blobs)      one process per GPU (collective calls)
    """

    def __init__(self, handle):
        self.lib = Library.get().dll
        self.h = handle
        self.world = self.lib.kzgb200_group_size(handle)
        self.local = self.lib.kzgb200_group_local_members(handle)

    @classmethod
    def create(cls, kzg_settings, device_ids, max_blobs_per_device):
        lib, h = Library.get().dll, C.c_void_p()
        ids = (C.c_int * len(device_ids))(*device_ids)
        rc = lib.kzgb200_group_create(C.byref(h), ids, len(device_ids), kzg_settings.g2_monomial_bytes[:192], 192, max_blobs_per_device)
        if rc:
            _raise(rc)
        return cls(h)

    @classmethod
    def join(cls, kzg_settings, session, rank, world, device, max_blobs_per_rank):
        lib, h = Library.get().dll, C.c_void_p()
        rc = lib.kzgb200_group_join(C.byref(h), session.encode(), rank, world, device, kzg_settings.g2_monomial_bytes[:192], 192, max_blobs_per_rank)
        if rc:
            _raise(rc)
        return cls(h)

    def context(self, i=0):
        return C.c_void_p(self.lib.kzgb200_group_context(self.h, i))

    def uses_peer_stores(self, i=0):
        return bool(self.lib.kzgb200_group_uses_peer_stores(self.h, i))

    def set_transcript_mode(self, mode):
        for i in range(self.local):
            self.lib.kzgb200_set_transcript_mode(self.context(i), mode)

    def _fail(self, rc):
        if rc == 2:
            raise KzgError("InternalError", "Internal error: " + self.lib.kzgb200_group_last_error(self.h).decode(errors="replace"))
        _raise(rc)

    def verify_blob_kzg_proof_batch_raw(self, blobs, n_blobs, commitments, n_commitments, proofs, n_proofs, want_zy=False):
        """The whole batch in contiguous host buffers (created group): same semantics as KzgProof.verify_blob_kzg_proof_batch_raw."""
        ok = C.c_int(0)
        z = C.create_string_buffer(32 * max(n_blobs, 1)) if want_zy else None
        y = C.create_string_buffer(32 * max(n_blobs, 1)) if want_zy else None
        rc = self.lib.kzgb200_group_verify_blob_kzg_proof_batch(self.h, _ptr(blobs), n_blobs, _ptr(commitments), n_commitments, _ptr(proofs),
                                                                n_proofs, C.byref(ok), z, y)
        if rc:
            self._fail(rc)
        return (bool(ok.value), z.raw, y.raw) if want_zy else bool(ok.value)

    def verify_shards(self, blobs, commitments, proofs, n_local, device_pointers, z_out=None, y_out=None):
        """One shard per local member (lists); device_pointers: the buffers are device memory on each member's GPU.
        Returns True / False, raises KzgError (BadArgs on any rank raises on every rank)."""
        k = self.local
        assert len(blobs) == len(commitments) == len(proofs) == len(n_local) == k
        arr = lambda xs: (C.c_void_p * k)(*[_ptr(x) for x in xs]) if xs is not None else None
        ok = C.c_int(0)
        rc = self.lib.kzgb200_group_verify_shards(self.h, arr(blobs), arr(commitments), arr(proofs), (C.c_size_t * k)(*n_local),
                                                  int(bool(device_pointers)), C.byref(ok), arr(z_out), arr(y_out))
        if rc:
            self._fail(rc)
        return bool(ok.value)

    def last_partials(self, n_ranks=None):
        n_ranks = n_ranks or self.world
        out = C.create_string_buffer(PARTIAL_BYTES * n_ranks)
        rc = self.lib.kzgb200_group_last_partials(self.h, out, n_ranks)
        if rc:
            self._fail(rc)
        return [out.raw[PARTIAL_BYTES * i:PARTIAL_BYTES * (i + 1)] for i in range(n_ranks)]

    def close(self):
        if self.h:
            self.lib.kzgb200_group_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def host_sha256(msg, portable=False):
    """(digest, used_sha_ni) by the host code that hashes the batch transcript."""
    out = C.create_string_buffer(32)
    used = Library.get().dll.kzgb200_host_sha256(bytes(msg), len(msg), out, int(portable))
    return out.raw, bool(used)


class BatchPipeline:
    """Streaming front-end (SURVEY.md 8f-3): `depth` batches in flight on one GPU, each one exactly a
    KzgProof::verify_blob_kzg_proof_batch call (reference src/kzg_proof.rs:472-525).  The latency-bound tail of one
    batch (transcript, MSM reduction, pairing) runs under the blob-streaming head / the PCIe copy of the next.

        pipe = BatchPipeline(settings, depth=2)
        t = pipe.submit(blobs, n, commitments, n, proofs, n)      # host buffers (bytes / pinned tensors / pointers)
        ...                                                       # submit more; blocks when `depth` are in flight
        ok = pipe.wait(t)                                         # True / False, raises KzgError like the blocking call
    """

    def __init__(self, kzg_settings, depth=2, device=0, transcript_mode=None):
        self.lib = Library.get().dll
        self.h = C.c_void_p()
        rc = self.lib.kzgb200_pipeline_create(C.byref(self.h), device, kzg_settings.g2_monomial_bytes[:192], 192, depth)
        if rc:
            _raise(rc)
        self.depth = depth
        self._keep = {}
        if transcript_mode is not None:
            for i in range(depth):
                self.lib.kzgb200_set_transcript_mode(self.context(i), transcript_mode)

    def context(self, slot):
        return C.c_void_p(self.lib.kzgb200_pipeline_context(self.h, slot))

    def submit(self, blobs, n_blobs, commitments, n_commitments, proofs, n_proofs, z_out=None, y_out=None):
        """Host buffers; they must stay alive and unmodified until wait() (bytes objects are held by the pipeline)."""
        t = C.c_uint64()
        rc = self.lib.kzgb200_pipeline_submit(self.h, _ptr(blobs), n_blobs, _ptr(commitments), n_commitments, _ptr(proofs), n_proofs,
                                              _ptr(z_out), _ptr(y_out), C.byref(t))
        if rc:
            _raise(rc)
        self._keep[t.value] = (blobs, commitments, proofs, z_out, y_out)
        return t.value

    def submit_device(self, d_blobs, d_commitments, d_proofs, n, d_z_out=None, d_y_out=None):
        """Device pointers (ints or objects with data_ptr()) on the pipeline's GPU; pending writes must be complete."""
        t = C.c_uint64()
        rc = self.lib.kzgb200_pipeline_submit_device(self.h, _ptr(d_blobs), _ptr(d_commitments), _ptr(d_proofs), n,
                                                     _ptr(d_z_out), _ptr(d_y_out), C.byref(t))
        if rc:
            _raise(rc)
        self._keep[t.value] = (d_blobs, d_commitments, d_proofs, d_z_out, d_y_out)
        return t.value

    def wait(self, ticket):
        ok = C.c_int(0)
        rc = self.lib.kzgb200_pipeline_wait(self.h, ticket, C.byref(ok))
        self._keep.pop(ticket, None)
        if rc:
            _raise(rc)
        return bool(ok.value)

    def close(self):
        if self.h:
            self.lib.kzgb200_pipeline_destroy(self.h)
            self.h = C.c_void_p()
            self._keep = {}

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def set_transcript_mode(kzg_settings, mode, device=0):
    """EXACT (default, r bit-identical to kzg-rs) or TREE (parallel hash, same verdicts)."""
    rc = Library.get().dll.kzgb200_set_transcript_mode(kzg_settings.context(device), mode)
    if rc:
        _raise(rc)


def last_batch_intermediates(kzg_settings, device=0):
    """(r, proof_lincomb, rhs_g1) of the last n >= 2 batch on this device, as the oracle's trace gives them:
    r 32-byte big-endian; the two sums as affine integer pairs (or None for the identity)."""
    ctx = kzg_settings.context(device) if isinstance(kzg_settings, KzgSettings) else kzg_settings
    r, part = C.create_string_buffer(32), C.create_string_buffer(PARTIAL_BYTES)
    lib = Library.get().dll
    for rc in (lib.kzgb200_last_r(ctx, r), lib.kzgb200_last_partial(ctx, part)):
        if rc:
            _raise(rc, ctx)
    return decode_partial(part.raw, r.raw)


def decode_partial(part, r=None):
    """A 352-byte partial -> affine integer pairs (None = identity), sum r_i y_i and the error flags."""
    P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
    rinv = pow(1 << 384, -1, P)
    fe = lambda off: int.from_bytes(part[off:off + 48], "little") * rinv % P

    def affine(off):
        x, y, z = fe(off), fe(off + 48), fe(off + 96)
        if z == 0:
            return None
        zi = pow(z, -1, P)
        return (x * zi * zi % P, y * zi * zi * zi % P)
    s = int.from_bytes(part[288:320], "little")
    return {"r": r, "A": affine(0), "B_prime": affine(144), "sum_r_y": s, "err": int.from_bytes(part[320:324], "little")}


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, int):
        return C.c_void_p(x)
    if hasattr(x, "data_ptr"):          # torch tensor (pinned host or device memory)
        return C.c_void_p(x.data_ptr())
    if isinstance(x, (bytes, bytearray)):
        return C.cast(C.c_char_p(bytes(x)), C.c_void_p) if isinstance(x, bytes) else C.cast((C.c_char * len(x)).from_buffer(x), C.c_void_p)
    return C.cast(x, C.c_void_p)
