// kzg_rs.hpp -- header-only C++17 mirror of kzg-rs's public verification interface over the C ABI of
// kzgb200.h.  Same names, argument meaning and error behaviour as the reference (the north star asks for a
// Rust host; this image has no Rust toolchain, INTEGRATION.md carries the Rust shim as source):
//   kzg_rs::KzgProof::verify_kzg_proof / verify_blob_kzg_proof / verify_blob_kzg_proof_batch   src/kzg_proof.rs:353-525
//   kzg_rs::KzgSettings::load_trusted_setup_file                                                src/trusted_setup.rs:94-98
//   kzg_rs::Blob / Bytes32 / Bytes48 (from_slice length check, as_slice)                        src/dtypes.rs:7-46
//   kzg_rs::KzgError                                                                            src/enums.rs:6-18
// plus the EIP-4844 publisher calls kzg_rs::blob_to_kzg_commitment / compute_kzg_proof / compute_blob_kzg_proof, and EIP-7594 cells: kzg_rs::Cell, KzgProof::verify_cell_kzg_proof_batch[_many], kzg_rs::compute_cells, kzg_rs::compute_cells_and_kzg_proofs,
// kzg_rs::recover_cells_and_kzg_proofs (c-kzg-4844 / rust-kzg names), and kzg_rs::compute_commitments_and_cell_proofs (a blob publisher's
// commitments and cell proofs in one call).
// Result<bool, KzgError> is kzg_rs::Result<bool>: either a value or an error.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <string>
#include <utility>
#include <vector>
#include "kzgb200.h"

namespace kzg_rs {

constexpr size_t BYTES_PER_BLOB = KZGB200_BYTES_PER_BLOB;
constexpr size_t BYTES_PER_COMMITMENT = KZGB200_BYTES_PER_COMMITMENT;
constexpr size_t BYTES_PER_PROOF = KZGB200_BYTES_PER_PROOF;
constexpr size_t BYTES_PER_FIELD_ELEMENT = KZGB200_BYTES_PER_FIELD_ELEMENT;
constexpr size_t BYTES_PER_CELL = 2048;          // EIP-7594: 64 field elements of the extended blob
constexpr size_t CELLS_PER_EXT_BLOB = 128;

struct KzgError {
    enum Kind { BadArgs, InternalError, InvalidBytesLength, InvalidHexFormat, InvalidTrustedSetup } kind;
    std::string message;
};

template <class T>
class Result {
    bool ok_;
    T value_{};
    KzgError err_{KzgError::InternalError, ""};
public:
    Result(T v) : ok_(true), value_(std::move(v)) {}
    Result(KzgError e) : ok_(false), err_(std::move(e)) {}
    bool is_ok() const { return ok_; }
    bool is_err() const { return !ok_; }
    const T& unwrap() const { return value_; }
    T& unwrap() { return value_; }
    const KzgError& unwrap_err() const { return err_; }
};

template <size_t N>
struct BytesN {
    std::array<uint8_t, N> bytes{};
    static Result<BytesN> from_slice(const uint8_t* p, size_t len) {   // src/dtypes.rs:19-29
        if (len != N) return KzgError{KzgError::InvalidBytesLength, "Invalid slice length"};
        BytesN b;
        std::memcpy(b.bytes.data(), p, N);
        return b;
    }
    const uint8_t* as_slice() const { return bytes.data(); }
};
using Bytes32 = BytesN<32>;
using Bytes48 = BytesN<48>;
using Blob = BytesN<BYTES_PER_BLOB>;
using Cell = BytesN<BYTES_PER_CELL>;
static_assert(sizeof(Blob) == BYTES_PER_BLOB && sizeof(Bytes48) == 48, "vectors of these are contiguous byte arrays");

class KzgSettings {
    struct Deleter { void operator()(kzgb200_ctx* c) const { kzgb200_destroy(c); } };
    std::shared_ptr<kzgb200_ctx> ctx_;
public:
    std::vector<uint8_t> g2_points;   // compressed, 96 bytes each; the verification path reads [0] and [1]
    std::vector<uint8_t> g1_lagrange; // compressed, 48 bytes each, file order; read by load_commit_setup
    // setup file: "KZGS" | u32 n1 | u32 n2 | n1*48 G1 Lagrange | n2*96 G2 monomial (kzg_rs_b200/data/mainnet_setup.bin)
    static Result<KzgSettings> load_trusted_setup_file(const std::string& path, int device = 0) {
        std::ifstream f(path, std::ios::binary);
        std::vector<uint8_t> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        if (raw.size() < 12 || std::memcmp(raw.data(), "KZGS", 4)) return KzgError{KzgError::InvalidTrustedSetup, "Invalid trusted setup"};
        uint32_t n1, n2;
        std::memcpy(&n1, raw.data() + 4, 4); std::memcpy(&n2, raw.data() + 8, 4);
        if (n2 < 2 || raw.size() != 12 + size_t(n1) * 48 + size_t(n2) * 96) return KzgError{KzgError::InvalidTrustedSetup, "Invalid trusted setup"};
        KzgSettings s;
        s.g2_points.assign(raw.begin() + 12 + size_t(n1) * 48, raw.end());
        s.g1_lagrange.assign(raw.begin() + 12, raw.begin() + 12 + size_t(n1) * 48);
        kzgb200_ctx* c = nullptr;
        int rc = kzgb200_create(&c, device, s.g2_points.data(), 192);
        if (rc) return KzgError{rc == KZGB200_INVALID_SETUP ? KzgError::InvalidTrustedSetup : KzgError::InternalError, "kzgb200_create failed"};
        s.ctx_ = std::shared_ptr<kzgb200_ctx>(c, Deleter());
        return s;
    }
    kzgb200_ctx* ctx() const { return ctx_.get(); }
    // cell proofs (EIP-7594): the setup's [tau^j]G1, j < 64 at least (for mainnet: kzg_rs_b200/data/g1_monomial.txt, hex-decoded), and
    // g2_points[64]; once, before the cell calls
    Result<bool> load_cell_setup(const uint8_t* g1_monomial48, size_t n_points) const {
        if (g2_points.size() < 65 * 96) return KzgError{KzgError::InvalidTrustedSetup, "the setup has no G2 point 64"};
        int rc = kzgb200_load_cell_setup(ctx(), g1_monomial48, n_points, g2_points.data() + 64 * 96);
        if (rc) return KzgError{rc == KZGB200_INVALID_SETUP ? KzgError::InvalidTrustedSetup : KzgError::InternalError, "kzgb200_load_cell_setup failed"};
        return true;
    }
    // commitments and proofs (EIP-4844 publisher calls): the window table of the 4096 Lagrange points (4.8 GB of device memory);
    // once, before the calls
    Result<bool> load_commit_setup() const {
        int rc = kzgb200_load_g1_lagrange(ctx(), g1_lagrange.data(), g1_lagrange.size() / 48);
        if (rc) return KzgError{rc == KZGB200_INVALID_SETUP ? KzgError::InvalidTrustedSetup : KzgError::InternalError, "kzgb200_load_g1_lagrange failed"};
        return true;
    }
};

namespace detail {
inline Result<bool> to_result(int rc, int ok, const char* len_msg = "Invalid commitments length") {
    switch (rc) {
        case KZGB200_OK: return ok != 0;
        case KZGB200_BAD_ARGS: return KzgError{KzgError::BadArgs, "Failed to parse G1Affine from bytes"};
        case KZGB200_INVALID_LENGTH: return KzgError{KzgError::InvalidBytesLength, len_msg};
        case KZGB200_INVALID_SETUP: return KzgError{KzgError::InvalidTrustedSetup, "Invalid trusted setup"};
        default: return KzgError{KzgError::InternalError, "Internal error"};
    }
}
}  // namespace detail

struct KzgProof {
    static Result<bool> verify_kzg_proof(const Bytes48& commitment_bytes, const Bytes32& z_bytes, const Bytes32& y_bytes,
                                         const Bytes48& proof_bytes, const KzgSettings& kzg_settings) {
        int ok = 0;
        int rc = kzgb200_verify_kzg_proof(kzg_settings.ctx(), commitment_bytes.as_slice(), z_bytes.as_slice(), y_bytes.as_slice(),
                                          proof_bytes.as_slice(), &ok);
        return detail::to_result(rc, ok);
    }
    static Result<bool> verify_blob_kzg_proof(const Blob& blob, const Bytes48& commitment_bytes, const Bytes48& proof_bytes,
                                              const KzgSettings& kzg_settings) {
        int ok = 0;
        int rc = kzgb200_verify_blob_kzg_proof(kzg_settings.ctx(), blob.as_slice(), commitment_bytes.as_slice(), proof_bytes.as_slice(),
                                               &ok, nullptr, nullptr);
        return detail::to_result(rc, ok);
    }
    static Result<bool> verify_blob_kzg_proof_batch(const std::vector<Blob>& blobs, const std::vector<Bytes48>& commitments_bytes,
                                                    const std::vector<Bytes48>& proofs_bytes, const KzgSettings& kzg_settings) {
        int ok = 0;
        int rc = kzgb200_verify_blob_kzg_proof_batch(kzg_settings.ctx(), reinterpret_cast<const uint8_t*>(blobs.data()), blobs.size(),
                                                     reinterpret_cast<const uint8_t*>(commitments_bytes.data()), commitments_bytes.size(),
                                                     reinterpret_cast<const uint8_t*>(proofs_bytes.data()), proofs_bytes.size(), &ok,
                                                     nullptr, nullptr);
        return detail::to_result(rc, ok, blobs.size() != commitments_bytes.size() ? "Invalid commitments length" : "Invalid proofs length");
    }
    // EIP-7594: one entry per cell (its blob's commitment, its index < 128, the cell, its proof)
    static Result<bool> verify_cell_kzg_proof_batch(const std::vector<Bytes48>& commitments_bytes, const std::vector<uint64_t>& cell_indices,
                                                    const std::vector<Cell>& cells, const std::vector<Bytes48>& proofs_bytes,
                                                    const KzgSettings& kzg_settings) {
        const size_t n = cell_indices.size();
        if (commitments_bytes.size() != n || cells.size() != n || proofs_bytes.size() != n)
            return KzgError{KzgError::InvalidBytesLength, "Invalid cells / commitments / proofs length"};
        int ok = 0;
        int rc = kzgb200_verify_cell_kzg_proof_batch(kzg_settings.ctx(), reinterpret_cast<const uint8_t*>(commitments_bytes.data()),
                                                     cell_indices.data(), reinterpret_cast<const uint8_t*>(cells.data()),
                                                     reinterpret_cast<const uint8_t*>(proofs_bytes.data()), n, &ok);
        return detail::to_result(rc, ok);
    }
    // k independent verify_cell_kzg_proof_batch calls in one: the cells of all groups contiguous, group g = cells
    // [group_offsets[g], group_offsets[g + 1]) (k + 1 offsets, the first 0, the last n).  One verdict per group: 1 = true, 0 = false,
    // 2 = the group alone would give BadArgs.  An error only for the call itself (lengths, offsets, setup).
    static Result<std::vector<uint8_t>> verify_cell_kzg_proof_batch_many(const std::vector<Bytes48>& commitments_bytes,
                                                                         const std::vector<uint64_t>& cell_indices, const std::vector<Cell>& cells,
                                                                         const std::vector<Bytes48>& proofs_bytes,
                                                                         const std::vector<uint64_t>& group_offsets, const KzgSettings& kzg_settings) {
        const size_t n = cell_indices.size();
        if (commitments_bytes.size() != n || cells.size() != n || proofs_bytes.size() != n || group_offsets.empty() || group_offsets.back() != n)
            return KzgError{KzgError::InvalidBytesLength, "Invalid cells / commitments / proofs / group offsets length"};
        std::vector<uint8_t> verdicts(group_offsets.size() - 1);
        int rc = kzgb200_verify_cell_kzg_proof_batch_many(kzg_settings.ctx(), reinterpret_cast<const uint8_t*>(commitments_bytes.data()),
                                                          cell_indices.data(), reinterpret_cast<const uint8_t*>(cells.data()),
                                                          reinterpret_cast<const uint8_t*>(proofs_bytes.data()), group_offsets.data(),
                                                          verdicts.size(), verdicts.data());
        if (rc) return detail::to_result(rc, 0).unwrap_err();
        return verdicts;
    }
    // The cell proofs of a blob transaction: its blobs, one commitment per blob and 128 cell proofs per blob (proof j of blob b at
    // 128 b + j).  The verdict of verify_cell_kzg_proof_batch on the expanded lists; the cells are computed on the GPU.
    static Result<bool> verify_blob_cell_kzg_proof_batch(const std::vector<Blob>& blobs, const std::vector<Bytes48>& commitments_bytes,
                                                         const std::vector<Bytes48>& cell_proofs_bytes, const KzgSettings& kzg_settings) {
        int ok = 0;
        int rc = kzgb200_verify_blob_cell_kzg_proof_batch(kzg_settings.ctx(), reinterpret_cast<const uint8_t*>(blobs.data()), blobs.size(),
                                                          reinterpret_cast<const uint8_t*>(commitments_bytes.data()), commitments_bytes.size(),
                                                          reinterpret_cast<const uint8_t*>(cell_proofs_bytes.data()), cell_proofs_bytes.size(), &ok);
        return detail::to_result(rc, ok, "Invalid blobs / commitments / cell proofs length");
    }
    // Many transactions in one call, contiguous: transaction g = blobs and commitments [blob_offsets[g], blob_offsets[g + 1]) and the
    // 128 cell proofs of each of those blobs (k + 1 offsets, the first 0, the last blobs.size()).  One verdict per transaction: 1 = true,
    // 0 = false, 2 = the transaction alone would give BadArgs.  An error only for the call itself (lengths, offsets, setup).
    static Result<std::vector<uint8_t>> verify_blob_cell_kzg_proof_batch_many(const std::vector<Blob>& blobs, const std::vector<Bytes48>& commitments_bytes,
                                                                              const std::vector<Bytes48>& cell_proofs_bytes,
                                                                              const std::vector<uint64_t>& blob_offsets, const KzgSettings& kzg_settings) {
        const size_t n = blobs.size();
        if (commitments_bytes.size() != n || cell_proofs_bytes.size() != CELLS_PER_EXT_BLOB * n || blob_offsets.empty() || blob_offsets.back() != n)
            return KzgError{KzgError::InvalidBytesLength, "Invalid blobs / commitments / cell proofs / blob offsets length"};
        std::vector<uint8_t> verdicts(blob_offsets.size() - 1);
        int rc = kzgb200_verify_blob_cell_kzg_proof_batch_many(kzg_settings.ctx(), reinterpret_cast<const uint8_t*>(blobs.data()),
                                                               reinterpret_cast<const uint8_t*>(commitments_bytes.data()),
                                                               reinterpret_cast<const uint8_t*>(cell_proofs_bytes.data()), blob_offsets.data(),
                                                               verdicts.size(), verdicts.data());
        if (rc) return detail::to_result(rc, 0).unwrap_err();
        return verdicts;
    }
};

// EIP-4844 publisher calls (need load_commit_setup).  BadArgs for a non-canonical blob element or z, and for a commitment that is not
// a valid compressed point of the G1 subgroup.
inline Result<Bytes48> blob_to_kzg_commitment(const Blob& blob, const KzgSettings& kzg_settings) {
    Bytes48 c;
    int rc = kzgb200_blob_to_kzg_commitment(kzg_settings.ctx(), blob.as_slice(), c.bytes.data());
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return c;
}
// (proof, y) with y = p(z); z may be a point of the evaluation domain
inline Result<std::pair<Bytes48, Bytes32>> compute_kzg_proof(const Blob& blob, const Bytes32& z_bytes, const KzgSettings& kzg_settings) {
    std::pair<Bytes48, Bytes32> out;
    int rc = kzgb200_compute_kzg_proof(kzg_settings.ctx(), blob.as_slice(), z_bytes.as_slice(), out.first.bytes.data(), out.second.bytes.data());
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return out;
}
inline Result<Bytes48> compute_blob_kzg_proof(const Blob& blob, const Bytes48& commitment_bytes, const KzgSettings& kzg_settings) {
    Bytes48 p;
    int rc = kzgb200_compute_blob_kzg_proof(kzg_settings.ctx(), blob.as_slice(), commitment_bytes.as_slice(), p.bytes.data());
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return p;
}

// EIP-7594 compute_cells: the 128 cells of the blob's extension
inline Result<std::vector<Cell>> compute_cells(const Blob& blob, const KzgSettings& kzg_settings) {
    std::vector<Cell> cells(CELLS_PER_EXT_BLOB);
    int rc = kzgb200_compute_cells(kzg_settings.ctx(), blob.as_slice(), reinterpret_cast<uint8_t*>(cells.data()));
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return cells;
}

// EIP-7594 compute_cells_and_kzg_proofs / recover_cells_and_kzg_proofs (FK20 on the GPU).  Both need the proof setup once per
// context: load_cell_proof_setup with the setup's 4096 Lagrange G1 points (file order), after load_cell_setup.
inline Result<bool> load_cell_proof_setup(const KzgSettings& kzg_settings, const uint8_t* g1_lagrange48, size_t n_points) {
    int rc = kzgb200_load_cell_proof_setup(kzg_settings.ctx(), g1_lagrange48, n_points);
    if (rc) return KzgError{rc == KZGB200_INVALID_SETUP ? KzgError::InvalidTrustedSetup : KzgError::InternalError, "kzgb200_load_cell_proof_setup failed"};
    return true;
}
struct CellsAndProofs { std::vector<Cell> cells; std::vector<Bytes48> proofs; };
inline Result<CellsAndProofs> compute_cells_and_kzg_proofs(const Blob& blob, const KzgSettings& kzg_settings) {
    CellsAndProofs out{std::vector<Cell>(CELLS_PER_EXT_BLOB), std::vector<Bytes48>(CELLS_PER_EXT_BLOB)};
    int rc = kzgb200_compute_cells_and_kzg_proofs(kzg_settings.ctx(), blob.as_slice(), reinterpret_cast<uint8_t*>(out.cells.data()),
                                                  reinterpret_cast<uint8_t*>(out.proofs.data()));
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return out;
}
// 64..128 cells of a blob, indices in any order -> all 128 cells and proofs; BadArgs for the spec's failed assertions
inline Result<CellsAndProofs> recover_cells_and_kzg_proofs(const std::vector<uint64_t>& cell_indices, const std::vector<Cell>& cells,
                                                          const KzgSettings& kzg_settings) {
    if (cells.size() != cell_indices.size()) return KzgError{KzgError::InvalidBytesLength, "Invalid cells / cell indices length"};
    CellsAndProofs out{std::vector<Cell>(CELLS_PER_EXT_BLOB), std::vector<Bytes48>(CELLS_PER_EXT_BLOB)};
    int rc = kzgb200_recover_cells_and_kzg_proofs(kzg_settings.ctx(), cell_indices.data(), reinterpret_cast<const uint8_t*>(cells.data()),
                                                  cells.size(), reinterpret_cast<uint8_t*>(out.cells.data()),
                                                  reinterpret_cast<uint8_t*>(out.proofs.data()));
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return out;
}
// A publisher's outputs for many blobs in one FK20 pass per 512 blobs, with only the proof setup: blob b's commitment (commitments[b],
// the bytes of blob_to_kzg_commitment), its 128 cell proofs (proofs[128 b ..], cell order) and, with want_cells, its cells
// (cells[128 b ..]).  status[b] = 0, or 1 where the blob alone would give BadArgs (its slots then unspecified).  An error only for
// the call itself (setup, device).
struct CommitmentsAndCellProofs { std::vector<Bytes48> commitments; std::vector<Cell> cells; std::vector<Bytes48> proofs; std::vector<uint8_t> status; };
inline Result<CommitmentsAndCellProofs> compute_commitments_and_cell_proofs(const std::vector<Blob>& blobs, const KzgSettings& kzg_settings,
                                                                            bool want_cells = false) {
    const size_t n = blobs.size();
    CommitmentsAndCellProofs out{std::vector<Bytes48>(n), std::vector<Cell>(want_cells ? CELLS_PER_EXT_BLOB * n : 0),
                                 std::vector<Bytes48>(CELLS_PER_EXT_BLOB * n), std::vector<uint8_t>(n)};
    int rc = kzgb200_compute_commitments_and_cell_proofs(kzg_settings.ctx(), reinterpret_cast<const uint8_t*>(blobs.data()), n,
                                                         reinterpret_cast<uint8_t*>(out.commitments.data()),
                                                         reinterpret_cast<uint8_t*>(out.proofs.data()),
                                                         want_cells ? reinterpret_cast<uint8_t*>(out.cells.data()) : nullptr, out.status.data());
    if (rc) return detail::to_result(rc, 0).unwrap_err();
    return out;
}

// Streaming front-end (include/kzgb200.h, kzgb200_pipeline_*): `depth` verify_blob_kzg_proof_batch calls in flight on one GPU.
// The pipeline owns the submitted vectors until the ticket has been waited for (the C ABI reads them asynchronously).
class BatchPipeline {
    struct Deleter { void operator()(kzgb200_pipeline* p) const { kzgb200_pipeline_destroy(p); } };
    struct Held { std::vector<Blob> blobs; std::vector<Bytes48> commitments, proofs; };
    std::shared_ptr<kzgb200_pipeline> p_;
    std::map<uint64_t, Held> held_;
public:
    using Ticket = uint64_t;
    static Result<BatchPipeline> create(const KzgSettings& kzg_settings, int depth = 2, int device = 0) {
        kzgb200_pipeline* raw = nullptr;
        int rc = kzgb200_pipeline_create(&raw, device, kzg_settings.g2_points.data(), 192, depth);
        if (rc) return KzgError{rc == KZGB200_INVALID_SETUP ? KzgError::InvalidTrustedSetup : KzgError::InternalError, "kzgb200_pipeline_create failed"};
        BatchPipeline bp;
        bp.p_ = std::shared_ptr<kzgb200_pipeline>(raw, Deleter());
        return bp;
    }
    // same arguments as KzgProof::verify_blob_kzg_proof_batch (reference src/kzg_proof.rs:472-477), taken by value like there
    Result<Ticket> submit(std::vector<Blob> blobs, std::vector<Bytes48> commitments_bytes, std::vector<Bytes48> proofs_bytes) {
        Held h{std::move(blobs), std::move(commitments_bytes), std::move(proofs_bytes)};
        uint64_t t = 0;
        int rc = kzgb200_pipeline_submit(p_.get(), reinterpret_cast<const uint8_t*>(h.blobs.data()), h.blobs.size(),
                                         reinterpret_cast<const uint8_t*>(h.commitments.data()), h.commitments.size(),
                                         reinterpret_cast<const uint8_t*>(h.proofs.data()), h.proofs.size(), nullptr, nullptr, &t);
        if (rc) return KzgError{KzgError::InternalError, "kzgb200_pipeline_submit failed"};
        held_.emplace(t, std::move(h));          // moving a vector keeps its buffer where it is
        return t;
    }
    Result<bool> wait(Ticket t) {
        int ok = 0;
        int rc = kzgb200_pipeline_wait(p_.get(), t, &ok);
        auto it = held_.find(t);
        bool c_len = it != held_.end() && it->second.blobs.size() != it->second.commitments.size();
        if (it != held_.end()) held_.erase(it);
        return detail::to_result(rc, ok, c_len ? "Invalid commitments length" : "Invalid proofs length");
    }
};

}  // namespace kzg_rs
