/* kzgb200 -- C ABI of the B200-native (sm_100a) replacement for the EIP-4844 verification hot path of
 * succinctlabs/kzg-rs v0.2.8.  This is the boundary a Rust (extern "C"), cgo, or ctypes binding binds;
 * INTEGRATION.md shows the Rust shim that keeps kzg-rs's public API unchanged on top of it.
 *
 * Conventions
 *   - plain pointers and sizes only; the library never frees or retains caller memory past return;
 *   - "host" entry points take host memory (pinned: copied straight by the DMA engine; pageable: through a ring of pinned staging
 *     buffers filled by a few memcpy threads -- env KZGB200_PAGEABLE=direct|register selects the driver's staging / in-place pinning);
 *     "_device" entry points take device pointers on the context's GPU (inputs already resident in HBM).  The library
 *     works on its own CUDA streams: device inputs must be complete before the call (synchronise the stream that
 *     produced them); every entry point returns only after its outputs are complete;
 *   - return codes map 1:1 onto kzg-rs's KzgError (reference src/enums.rs:6-18):
 *         KZGB200_OK                 Ok(verdict), verdict in *ok (1 = true, 0 = false)
 *         KZGB200_BAD_ARGS           Err(KzgError::BadArgs)            -- unparsable scalar / G1 point
 *         KZGB200_INTERNAL_ERROR     Err(KzgError::InternalError)      -- CUDA failure
 *         KZGB200_INVALID_LENGTH     Err(KzgError::InvalidBytesLength) -- vector length mismatch
 *         KZGB200_INVALID_SETUP      Err(KzgError::InvalidTrustedSetup)
 *   - a context is bound to one GPU; calls on one context are serialised by an internal lock, use one
 *     context per thread (or per GPU) for concurrency.  There is no CPU fallback: every entry point fails
 *     with KZGB200_INTERNAL_ERROR when no sm_100 device / kernel image is available.
 */
#ifndef KZGB200_H
#define KZGB200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define KZGB200_OK 0
#define KZGB200_BAD_ARGS 1
#define KZGB200_INTERNAL_ERROR 2
#define KZGB200_INVALID_LENGTH 3
#define KZGB200_INVALID_SETUP 5

#define KZGB200_BYTES_PER_BLOB 131072       /* reference src/consts.rs:8 */
#define KZGB200_BYTES_PER_COMMITMENT 48     /* src/consts.rs:9 */
#define KZGB200_BYTES_PER_PROOF 48          /* src/consts.rs:10 */
#define KZGB200_BYTES_PER_FIELD_ELEMENT 32  /* src/consts.rs:3 */
#define KZGB200_PARTIAL_BYTES 352           /* per-rank partial of the sharded batch (see below) */

typedef struct kzgb200_ctx kzgb200_ctx;

/* Replaces KzgSettings::load_trusted_setup_file (reference src/trusted_setup.rs:94-98) + the table building
 * of build.rs:131-170: uploads / derives the device-resident tables (roots of unity in Montgomery form,
 * Miller-loop line coefficients of g2_points[0] and g2_points[1]).  g2_points = the first two G2 points of
 * the trusted setup, ZCash-compressed, 2 x 96 bytes (trusted_setup.txt lines 4099-4100).  The verification
 * path reads nothing else from the setup (SURVEY.md section 0). */
int kzgb200_create(kzgb200_ctx** out, int device, const uint8_t* g2_points, size_t g2_points_len);
void kzgb200_destroy(kzgb200_ctx* ctx);
/* last CUDA error string of the context ("" if none); valid until the next call */
const char* kzgb200_last_error(const kzgb200_ctx* ctx);

/* KzgProof::verify_kzg_proof (reference src/kzg_proof.rs:353-397). */
int kzgb200_verify_kzg_proof(kzgb200_ctx* ctx, const uint8_t* commitment48, const uint8_t* z32, const uint8_t* y32,
                             const uint8_t* proof48, int* ok);

/* KzgProof::verify_blob_kzg_proof (reference src/kzg_proof.rs:446-470).  z_out / y_out (32 bytes, big-endian,
 * nullable) receive the Fiat-Shamir challenge and the evaluation -- intermediates that must be bit-exact. */
int kzgb200_verify_blob_kzg_proof(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* commitment48,
                                  const uint8_t* proof48, int* ok, uint8_t* z_out, uint8_t* y_out);

/* KzgProof::verify_blob_kzg_proof_batch (reference src/kzg_proof.rs:472-525).  The three lengths are the
 * lengths of the three Vec arguments; n == 0 -> Ok(true); n == 1 -> single path; mismatch -> INVALID_LENGTH.
 * blobs = n_blobs x 131072 bytes contiguous (a Vec<Blob> is exactly that), commitments / proofs = n x 48.
 * z_out / y_out: n_blobs x 32 bytes big-endian, nullable. */
int kzgb200_verify_blob_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n_blobs,
                                        const uint8_t* commitments, size_t n_commitments,
                                        const uint8_t* proofs, size_t n_proofs, int* ok,
                                        uint8_t* z_out, uint8_t* y_out);
/* Same, inputs (and z_out / y_out, nullable) are device pointers on the context's GPU; n >= 1. */
int kzgb200_verify_blob_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                               const uint8_t* d_proofs, size_t n, int* ok,
                                               uint8_t* d_z_out, uint8_t* d_y_out);

/* m independent verify_kzg_proof tuples (BASELINE config 5); verdicts[i] = 0 false, 1 true, 2 BadArgs.
 * Host pointers. */
int kzgb200_verify_kzg_proof_many(kzgb200_ctx* ctx, const uint8_t* commitments, const uint8_t* zs, const uint8_t* ys,
                                  const uint8_t* proofs, size_t m, uint8_t* verdicts);

/* KzgProof::verify_kzg_proof_batch on ALREADY-PARSED inputs (reference src/kzg_proof.rs:399-444; SURVEY.md 8f-4).  Inputs in the
 * reference's in-memory layout on a little-endian host (build.rs:185-203): a G1Affine is 104 bytes = x (6 x u64 Montgomery limbs) |
 * y (6 x u64) | infinity flag byte | 7 bytes padding; a Scalar is 4 x u64 Montgomery limbs (32 bytes).  Like the reference it does
 * not validate the points or check the subgroup (the arguments are typed values there).  Host pointers; n == 0 -> Ok(true). */
int kzgb200_verify_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* commitments104, const uint8_t* zs32, const uint8_t* ys32,
                                   const uint8_t* proofs104, size_t n, int* ok);

/* Per-blob verdicts (SURVEY.md 8f-4): verdicts[i] = what KzgProof::verify_blob_kzg_proof(blob_i, commitment_i, proof_i) returns
 * (src/kzg_proof.rs:446-470): 1 = Ok(true), 0 = Ok(false), 2 = Err(BadArgs).  The batch equation is checked first (one MSM, one pairing);
 * only a failing batch is bisected down to the blob, on the GPU, from the already-parsed points and already-computed z_i, y_i.
 * Host pointers; z_out / y_out nullable (n x 32 big-endian). */
int kzgb200_verify_blob_kzg_proof_batch_each(kzgb200_ctx* ctx, const uint8_t* blobs, const uint8_t* commitments, const uint8_t* proofs,
                                             size_t n, uint8_t* verdicts, uint8_t* z_out, uint8_t* y_out);

/* The reference's public helpers (src/lib.rs:8): compute_challenge (src/kzg_proof.rs:46-72) and
 * evaluate_polynomial_in_evaluation_form (:94-133, including z inside the evaluation domain, :109-111), one blob each, host pointers,
 * 32-byte big-endian scalars.  Non-canonical blob elements / z -> KZGB200_BAD_ARGS. */
int kzgb200_compute_challenge(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* commitment48, uint8_t* z_out32);
int kzgb200_evaluate_polynomial_in_evaluation_form(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* z32, uint8_t* y_out32);

/* ---- multi-GPU: blob-sharded batches (SURVEY.md 8e) -----------------------------------------------------------------
 * A group is one context per GPU; rank k owns a contiguous range of the batch's blobs and never sees the others'.  The ranks meet
 * twice per batch: (1) their transcript entries (C_i, z_i, y_i, pi_i: 160 bytes per blob) flow, chunk by chunk behind the evaluation
 * kernels, into a shared host block where the leader (rank 0) hashes them in global order into r (compute_r_powers, reference
 * src/kzg_proof.rs:291-348); (2) every rank's 352-byte partial (sum r_i pi_i, sum r_i C_i + r_i z_i pi_i, sum r_i y_i, flags) is the last
 * store of its reduction kernel, over NVLink straight into the leader GPU's memory, where the single pairing check runs.  No
 * collective library, no host synchronisation between the phases.
 *   kzgb200_group_create: ONE process drives n GPUs (what a Rust caller of verify_blob_kzg_proof_batch uses to reach 8 GPUs).
 *   kzgb200_group_join:   one process PER GPU (torchrun-style); every rank calls it with the same session string, world and
 *                         max_blobs_per_rank; the ranks find each other in a POSIX shared-memory segment named after the session.
 * Every verify call on a joined group is collective: all ranks call it, each with its own shard (>= 1 blob), and all return the
 * same verdict / error.  Waits are bounded (30 s) and fail with KZGB200_INTERNAL_ERROR. */
typedef struct kzgb200_group kzgb200_group;
int kzgb200_group_create(kzgb200_group** out, const int* device_ids, int n_devices, const uint8_t* g2_points, size_t g2_points_len,
                         size_t max_blobs_per_device);
int kzgb200_group_join(kzgb200_group** out, const char* session, int rank, int world, int device, const uint8_t* g2_points,
                       size_t g2_points_len, size_t max_blobs_per_rank);
void kzgb200_group_destroy(kzgb200_group* g);
int kzgb200_group_size(const kzgb200_group* g);               /* ranks in the group */
int kzgb200_group_local_members(const kzgb200_group* g);      /* contexts driven by this process: all of them, or 1 */
kzgb200_ctx* kzgb200_group_context(kzgb200_group* g, int local_index);
const char* kzgb200_group_last_error(const kzgb200_group* g);
int kzgb200_group_uses_peer_stores(const kzgb200_group* g, int local_index);
/* KzgProof::verify_blob_kzg_proof_batch over all GPUs of a created (single-process) group: the whole batch in host memory, same
 * argument checks and return codes as kzgb200_verify_blob_kzg_proof_batch; batches below 32 blobs run on the first GPU. */
int kzgb200_group_verify_blob_kzg_proof_batch(kzgb200_group* g, const uint8_t* blobs, size_t n_blobs, const uint8_t* commitments,
                                              size_t n_commitments, const uint8_t* proofs, size_t n_proofs, int* ok, uint8_t* z_out,
                                              uint8_t* y_out);
/* Per-shard entry: arrays with one element per LOCAL member (n GPUs for a created group, 1 for a joined rank); shard k of the
 * batch = rank k's blobs, in rank order.  device_pointers != 0: inputs (and z_out / y_out) are device pointers on that member's GPU,
 * complete before the call; else host memory.  z_out / y_out arrays (or their elements) may be null. */
int kzgb200_group_verify_shards(kzgb200_group* g, const uint8_t* const* blobs, const uint8_t* const* commitments,
                                const uint8_t* const* proofs, const size_t* n_local, int device_pointers, int* ok,
                                uint8_t* const* z_out, uint8_t* const* y_out);
/* the gathered partials of the last collective call, n_ranks x KZGB200_PARTIAL_BYTES (leader's process only); for parity tests */
int kzgb200_group_last_partials(kzgb200_group* g, uint8_t* out, size_t n_ranks);
/* host-side protocol of a joined group without any GPU (CPU tests of the N > 1 path): the ranks pass the transcript entries of their
 * shards -- commitments (n_local x 48), zy (n_local x 64: z_i, y_i little-endian), proofs (n_local x 48) -- in chunks of `chunk`
 * entries through the shared block; every rank receives the transcript digest the leader hashed over all ranks' entries. */
int kzgb200_group_host_protocol_test(const char* session, int rank, int world, const uint8_t* commitments, const uint8_t* zy,
                                     const uint8_t* proofs, size_t n_local, size_t chunk, uint8_t* digest_out32);

/* ---- transcript mode of the batch challenge r -----------------------------------------------------------------
 * EXACT (default): r = SHA-256 over the serial transcript exactly as compute_r_powers (reference src/kzg_proof.rs:291-348) -- r, its
 *   powers and both MSM sums are bit-identical to kzg-rs.  The hash is ONE serial chain of 2.5 SHA-256 blocks per blob over data of
 *   every blob; it is run by a host thread (SHA-NI when the CPU has it) incrementally behind the evaluation kernels, chunk by chunk
 *   as the (z, y) pairs leave the GPU; only the last small chunk's hash is exposed.
 * EXACT_DEVICE: the same chain on one warp of the GPU (~2.4 us per blob: 40 ms at 16384 blobs; round 1's default).  Same r.
 * TREE (opt-in): the same entries hashed as a two-level tree with domain separation -- leaf j = SHA-256("RCKZGBATCH_LEAF_" | 16
 *   entries) on the GPU in parallel, r = SHA-256("RCKZGBATCH___V1_" | u64be 4096 | u64be n | leaves) mod q.  r differs from kzg-rs's;
 *   verdicts, z, y do not.  For very large multi-GPU batches, where even the host chain (2 GB/s) would limit. */
#define KZGB200_TRANSCRIPT_EXACT 0
#define KZGB200_TRANSCRIPT_TREE 1
#define KZGB200_TRANSCRIPT_EXACT_DEVICE 2
int kzgb200_set_transcript_mode(kzgb200_ctx* ctx, int mode);
/* canonical big-endian r of the last batch verified on this context (blob batches: n >= 2; cell batches: n >= 1) */
int kzgb200_last_r(kzgb200_ctx* ctx, uint8_t* r_out32);
/* test hook: SHA-256 of msg by the host code that hashes the transcript; force_portable = 1 selects the portable compression
 * function; returns 1 if the SHA-NI path was used */
int kzgb200_host_sha256(const uint8_t* msg, size_t len, uint8_t* out32, int force_portable);

/* raw partial of the last single-GPU batch (n >= 2), KZGB200_PARTIAL_BYTES: Jacobian A = sum r_i pi_i and
 * B' = sum r_i C_i + r_i z_i pi_i as 3 x 12 little-endian u32 Montgomery limbs each (R = 2^384), then
 * s = sum r_i y_i (8 limbs, canonical), then the error flags.  For parity tests of the MSM intermediates. */
int kzgb200_last_partial(kzgb200_ctx* ctx, uint8_t* out352);

/* ---- harness (test / bench data; kzg-rs itself has no commit/prove path) ---------------------------------
 * Fills device buffers with n synthetic blobs (evaluation form of seeded random polynomials of degree <
 * `degree`, 2 <= degree <= 16) and their valid commitments and proofs over the trusted setup whose
 * [tau^j]G1, j < degree, are given compressed in tau_powers48 (host, degree x 48 bytes). */
int kzgb200_harness_generate(kzgb200_ctx* ctx, uint64_t seed, size_t n, int degree, const uint8_t* tau_powers48,
                             uint8_t* d_blobs, uint8_t* d_commitments, uint8_t* d_proofs);
/* ---- commit / prove: EIP-4844 blob_to_kzg_commitment, compute_kzg_proof, compute_blob_kzg_proof (c-kzg-4844 semantics) ------
 * The publisher side of EIP-4844 (kzg-rs itself has none).  All outputs are compressed G1 points (48 bytes; the identity is 0xc0
 * then 47 zero bytes) and 32-byte big-endian scalars.
 * kzgb200_load_g1_lagrange: the setup's 4096 Lagrange G1 points, compressed, FILE order (host, 4096 x 48 bytes); builds a 4.8 GB
 *   fixed-base window table on the device (once per context; later calls return OK).  Every call below returns
 *   KZGB200_INVALID_SETUP before it.
 * kzgb200_blob_to_kzg_commitment: one host blob -> its commitment.  A non-canonical blob element -> BAD_ARGS.
 * kzgb200_compute_kzg_proof: one host blob and a host z -> the proof of p(z) = y and y.  z may be any canonical scalar, a point of
 *   the evaluation domain included.  A non-canonical blob element or z -> BAD_ARGS.
 * kzgb200_compute_blob_kzg_proof: one host blob and its commitment -> the proof at the Fiat-Shamir challenge of (blob, commitment).
 *   BAD_ARGS for a non-canonical blob element and for a commitment that is not a valid compressed point of the G1 subgroup
 *   (bad encoding, off the curve, outside the subgroup), as the spec's bytes_to_kzg_commitment.
 * kzgb200_compute_kzg_proof_batch_device: n device blobs and n device z (n x 32) -> n proofs (n x 48) and n y (n x 32), device
 *   pointers; n == 0 -> OK; any bad blob element or z -> BAD_ARGS for the whole call (outputs undefined).
 * kzgb200_blob_to_kzg_commitment_batch / kzgb200_compute_blob_kzg_proof_batch: the device-pointer batch forms (n >= 1); a bad blob
 *   element -> BAD_ARGS for the whole call.  The proof batch takes its commitments as given: it does not decompress or check them
 *   (the single-blob kzgb200_compute_blob_kzg_proof does). */
int kzgb200_load_g1_lagrange(kzgb200_ctx* ctx, const uint8_t* g1_lagrange, size_t n_points);
int kzgb200_blob_to_kzg_commitment(kzgb200_ctx* ctx, const uint8_t* blob, uint8_t* commitment_out48);
int kzgb200_compute_kzg_proof(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* z32, uint8_t* proof_out48, uint8_t* y_out32);
int kzgb200_compute_blob_kzg_proof(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* commitment48, uint8_t* proof_out48);
int kzgb200_compute_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_zs, size_t n,
                                           uint8_t* d_proofs_out, uint8_t* d_ys_out);
int kzgb200_blob_to_kzg_commitment_batch(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_commitments_out);
int kzgb200_compute_blob_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments, size_t n,
                                         uint8_t* d_proofs_out);

/* ---- EIP-7594 cells (PeerDAS; consensus-specs Fulu, polynomial-commitments-sampling.md) ---------------------------------
 * A blob extends to 8192 values (the polynomial on the 8192 roots of unity, bit-reversed order), split into 128 cells of 64 field
 * elements (2048 bytes, 32 big-endian bytes each).  Cells 0..63 are the blob itself.  Each cell has its own KZG multi-proof.
 * kzgb200_load_cell_setup: [tau^j]G1 for j < 64 at least (host, n_points x 48, compressed; for mainnet the
 *   points of kzg_rs_b200/data/g1_monomial.txt, one hex line each) and g2_monomial[64] = [tau^64]G2 (96 bytes).  Once per context; every cell entry point returns
 *   KZGB200_INVALID_SETUP before it.
 * kzgb200_verify_cell_kzg_proof_batch: one entry per cell -- the commitment of its blob, its index (< 128), the cell, its proof;
 *   n == 0 -> Ok(true); an index >= 128, a non-canonical cell element, or a commitment / proof that is not a valid compressed
 *   point of the G1 subgroup -> KZGB200_BAD_ARGS.  The batch challenge r is the spec's (commitments deduplicated by their bytes),
 *   hashed by a host thread over the caller's buffers while the GPU parses the inputs; kzgb200_last_r returns it afterwards.
 *   The call is the one-group case of kzgb200_verify_cell_kzg_proof_batch_many below.  The _device form takes device pointers; the inputs are copied back to pinned host memory once for the hash.
 * kzgb200_compute_cells: the 128 cells of one host blob (cells_out: 128 x 2048 bytes, host);
 * kzgb200_compute_cells_batch_device: n device blobs -> n x 128 cells (device, blob-major).  Non-canonical element -> BAD_ARGS. */
int kzgb200_load_cell_setup(kzgb200_ctx* ctx, const uint8_t* g1_monomial48, size_t n_points, const uint8_t* g2_tau64_96);
int kzgb200_verify_cell_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* commitments, const uint64_t* cell_indices, const uint8_t* cells,
                                        const uint8_t* proofs, size_t n, int* ok);
int kzgb200_verify_cell_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_commitments, const uint64_t* d_cell_indices,
                                               const uint8_t* d_cells, const uint8_t* d_proofs, size_t n, int* ok);
int kzgb200_compute_cells(kzgb200_ctx* ctx, const uint8_t* blob, uint8_t* cells_out);
int kzgb200_compute_cells_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_cells);
/* cell workload (test / bench data): n_blobs seeded polynomials of degree < `degree` (128 < degree <= 192) built from their
 * coefficients, their cells (n_blobs x 128 x 2048, device), commitments (n_blobs x 48) and the proofs of all their cells
 * (n_blobs x 128 x 48, same order as the cells); tau_powers48 = [tau^j]G1, j < degree (host).  Needs the cell setup. */
int kzgb200_harness_generate_cells(kzgb200_ctx* ctx, uint64_t seed, size_t n_blobs, int degree, const uint8_t* tau_powers48,
                                   uint8_t* d_cells, uint8_t* d_commitments, uint8_t* d_proofs);

/* ---- many cell batches in one call, one verdict each (PeerDAS data column sidecars) ----------------------------------------
 * kzgb200_verify_cell_kzg_proof_batch_many: n cells in the per-cell layout of kzgb200_verify_cell_kzg_proof_batch, split into
 *   n_groups groups by group_offsets[0..n_groups] (host: offsets[0] = 0, never decreasing, offsets[n_groups] = n; group g = cells
 *   [offsets[g], offsets[g + 1])).  verdicts[g] (host, n_groups bytes) = 1 / 0 / 2: verify_cell_kzg_proof_batch on group g alone
 *   returns true / false / fails an assertion (an index >= 128, a non-canonical element, a commitment or proof that is not a valid
 *   compressed subgroup point).  An empty group gets 1; a bad group never changes another group's verdict.  Each group's challenge
 *   r_g is the spec's, hashed over that group's bytes alone (its own deduplication of commitments) by up to 16 host threads while
 *   the GPU parses.  All groups are checked together first (weights rho^g r_g^j, one MSM and one pairing; a false group passes it
 *   with probability <= n_groups / q); only if that fails does every group get its own check (one extra pass for any number of bad
 *   groups; with one group the combined check is that group's own, and there is no second pass).  Returns BAD_ARGS only for a malformed call (a null pointer with n > 0 or n_groups > 0, bad offsets, n or n_groups
 *   above 0x7fffffff / 2), INVALID_SETUP without the cell setup; n_groups == 0 -> OK.
 *   The _device form takes device pointers for the four data arrays (group_offsets and verdicts stay host memory); the inputs are
 *   copied back to pinned host memory once for the transcripts.
 *   kzgb200_get_phase_ms after any cell verification call (single or _many, either form): {parse, host hashing (wall ms, every
 *   call), hasher threads (every call), r_g upload and weights, lincomb, reduce, combined pairing, per-group fallback}; the device
 *   slots with kzgb200_set_profiling on.
 * kzgb200_last_cell_many_r: r_g of the last cell verification call (a single call is one group; r_out: n_groups x 32, zeros for
 *   empty groups) and rho (rho_out32), canonical big-endian; n_groups must be that call's (else BAD_ARGS).  A call with one group
 *   sets what kzgb200_last_r reports to r_0, as the single call does; a call with more groups leaves it untouched.  No cell call
 *   changes what kzgb200_last_partial reports. */
int kzgb200_verify_cell_kzg_proof_batch_many(kzgb200_ctx* ctx, const uint8_t* commitments, const uint64_t* cell_indices, const uint8_t* cells,
                                             const uint8_t* proofs, const uint64_t* group_offsets, size_t n_groups, uint8_t* verdicts);
int kzgb200_verify_cell_kzg_proof_batch_many_device(kzgb200_ctx* ctx, const uint8_t* d_commitments, const uint64_t* d_cell_indices,
                                                    const uint8_t* d_cells, const uint8_t* d_proofs, const uint64_t* group_offsets,
                                                    size_t n_groups, uint8_t* verdicts);
int kzgb200_last_cell_many_r(kzgb200_ctx* ctx, uint8_t* r_out, size_t n_groups, uint8_t* rho_out32);

/* ---- cell proofs of whole blobs, one verdict per blob transaction (EIP-7594 network form of a blob transaction) ---------------
 * A blob transaction carries its blobs, their commitments and 128 cell proofs per blob.  An execution-layer node checks it as
 * verify_cell_kzg_proof_batch on the expanded lists: per blob b in order and j < 128, (commitment b, index j, cell j of
 * compute_cells(blob b), proof 128 b + j).  These calls run that composition on the GPU: the cells are computed on the device and
 * never handed to the caller.  Only the cell setup is needed (kzgb200_load_cell_setup), else INVALID_SETUP.
 * kzgb200_verify_blob_cell_kzg_proof_batch: blobs n_blobs x 131072, commitments n_commitments x 48, cell_proofs n_cell_proofs x 48
 *   (blob-major: proof j of blob b at 128 b + j), host.  n_commitments != n_blobs or n_cell_proofs != 128 n_blobs -> INVALID_LENGTH;
 *   n_blobs == 0 -> Ok(true); a non-canonical blob element (compute_cells fails) or a commitment / proof that is not a valid
 *   compressed point of the G1 subgroup -> BAD_ARGS.  The _device form takes the three arrays in device memory (n_blobs each).
 * kzgb200_verify_blob_cell_kzg_proof_batch_many: n_groups transactions in one call; blob_offsets[0..n_groups] (host, blobs: offsets[0]
 *   = 0, never decreasing) split the blobs, commitments (one per blob) and cell proofs (128 per blob) into groups.  verdicts[g] (host)
 *   = 1 / 0 / 2 for true / false / BadArgs of group g alone, exactly as the single call on that group; an empty group gets 1; a bad
 *   group never changes another group's verdict.  BAD_ARGS only for a malformed call (a null pointer with work to do, bad offsets,
 *   128 x blobs or n_groups above 0x7fffffff / 2).  The _device form takes the three data arrays in device memory.
 *   The single calls are its one-group case.  It is kzgb200_verify_cell_kzg_proof_batch_many on the expanded groups (cell offsets =
 *   128 x blob offsets): r_g is the spec's r of group g's expanded call, bit for bit (kzgb200_last_cell_many_r reports it; a one-group
 *   call also sets kzgb200_last_r), and kzgb200_get_phase_ms reports the same slots.  The computed cells (256 KiB per blob) are read
 *   back to pinned host memory once, for the exact transcripts. */
int kzgb200_verify_blob_cell_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n_blobs, const uint8_t* commitments,
                                             size_t n_commitments, const uint8_t* cell_proofs, size_t n_cell_proofs, int* ok);
int kzgb200_verify_blob_cell_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                                    const uint8_t* d_cell_proofs, size_t n_blobs, int* ok);
int kzgb200_verify_blob_cell_kzg_proof_batch_many(kzgb200_ctx* ctx, const uint8_t* blobs, const uint8_t* commitments,
                                                  const uint8_t* cell_proofs, const uint64_t* blob_offsets, size_t n_groups,
                                                  uint8_t* verdicts);
int kzgb200_verify_blob_cell_kzg_proof_batch_many_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                                         const uint8_t* d_cell_proofs, const uint64_t* blob_offsets, size_t n_groups,
                                                         uint8_t* verdicts);

/* ---- EIP-7594 cell proofs and recovery (FK20; consensus-specs Fulu compute_cells_and_kzg_proofs / recover_cells_and_kzg_proofs) --
 * kzgb200_load_cell_proof_setup: the setup's 4096 Lagrange G1 points (host, 4096 x 48 compressed, file order: point j pairs with
 *   omega4096^j; KzgSettings.g1_lagrange_bytes).  n_points must be 4096 and the cell setup must be loaded, else INVALID_SETUP.  Derives
 *   every [tau^m]G1 (m < 4096) on the device (a 4096-point DFT over G1), checks that the first 64 are the points given to
 *   kzgb200_load_cell_setup (INVALID_SETUP otherwise), and builds the FK20 tables.  Device memory: 3.34 GB of window tables
 *   (8192 bases x 16 windows x 255 affine points), 0.4 MB of monomial points, 0.4 MB of scalar tables; a workspace of ~0.9 MB per
 *   blob (at most 512 blobs at a time) is allocated by the first call that needs it.  Once per context (later calls return OK);
 *   the blob and cell verification paths keep working.  Every entry point below returns INVALID_SETUP before it.
 * kzgb200_cell_proof_monomial: the derived [tau^m]G1, m < n_points (<= 4096; else BAD_ARGS), compressed, to out48 (host).
 * kzgb200_compute_cells_and_kzg_proofs: one host blob -> its 128 cells (cells_out, 128 x 2048) and their proofs (proofs_out,
 *   128 x 48, compressed; the identity is 0xc0 then 47 zero bytes), host pointers, none nullable.
 * kzgb200_compute_cells_and_kzg_proofs_batch_device: n device blobs -> n x 128 cells and n x 128 proofs (device, blob-major, proofs
 *   in the order of the cells); n == 0 -> OK.  A non-canonical blob element -> BAD_ARGS for the whole call (outputs undefined).
 * kzgb200_recover_cells_and_kzg_proofs: all 128 cells and proofs of a blob from n_cells of its cells (host: cell_indices n_cells x u64,
 *   cells n_cells x 2048 in the same order, any order of indices).  BAD_ARGS unless 64 <= n_cells <= 128, every index < 128, no index
 *   twice and every element canonical.  Inconsistent cells are not detected (as in the spec): the result is the spec's bytes.
 * kzgb200_recover_cells_and_kzg_proofs_batch_device: n_blobs blobs that share one index set (host cell_indices, n_cells); d_cells =
 *   n_blobs x n_cells x 2048 (device, blob-major, each blob's cells in index-set order); outputs as the batch compute call.
 * kzgb200_recover_cells_and_kzg_proofs_many[_device]: n_blobs blobs in one call, each recovered from its own cells and index set.
 *   cell_offsets (host, n_blobs + 1 entries, [0] = 0, never decreasing): blob b owns cells [off[b], off[b + 1]), one u64 index per cell
 *   in cell_indices (host in both forms) and 2048 bytes per cell in cells (host; _device: device), any order of indices within a blob.
 *   Outputs are blob-major, n_blobs x 128 x 2048 cells and n_blobs x 128 x 48 proofs (host; _device: device).  status (host, one
 *   byte per blob) = the return code kzgb200_recover_cells_and_kzg_proofs gives for that blob alone: 0 = its outputs are that call's
 *   bytes; 1 (BAD_ARGS) = fewer than 64 or more than 128 cells, an index >= 128, a repeated index or a non-canonical element, its
 *   output slot unspecified.  A bad blob changes no other blob's output, and no blob's cells are read outside its own range.  The call
 *   returns BAD_ARGS only when malformed (a null pointer with blobs to recover, bad offsets, n_blobs or off[n_blobs] above
 *   0x7fffffff / 2), INVALID_SETUP before the proof setup, and OK for n_blobs == 0 (cell_offsets then unread).  Blobs that share one
 *   index set cost about what the _batch_device call costs for them.
 * kzgb200_compute_commitments_and_cell_proofs[_device]: what a blob publisher needs, in one FK20 pass per 512 blobs: for blob b its
 *   commitment (commitments_out + 48 b, the bytes of kzgb200_blob_to_kzg_commitment), its 128 cell proofs (proofs_out + 128 x 48 b, in
 *   cell order) and, when cells_out is not null, its cells (cells_out + 128 x 2048 b).  The commitment is output 0 of FK20's inverse
 *   G1 DFT, so only the proof setup is needed (not kzgb200_load_g1_lagrange).  blobs n_blobs x 131072 bytes; host pointers, _device:
 *   device pointers except status.  status (host, one byte per blob) = what kzgb200_blob_to_kzg_commitment /
 *   kzgb200_compute_cells_and_kzg_proofs return for that blob alone: 0, or 1 (BAD_ARGS: a non-canonical element), its output slots
 *   unspecified; a bad blob changes no other blob's output.  The call returns OK for n_blobs == 0 (nothing read, ctx may be null),
 *   BAD_ARGS for a null pointer other than cells_out or n_blobs above 0x7fffffff / 2, INVALID_SETUP before the proof setup.
 * With kzgb200_set_profiling on, kzgb200_get_phase_ms reports for these calls {coefficients (with compute_cells), fixed-base products
 * (with the scalar DFTs), G1 transforms (with compression), recovery transforms, 0, 0, 0, 0}, first start to last end. */
int kzgb200_load_cell_proof_setup(kzgb200_ctx* ctx, const uint8_t* g1_lagrange48, size_t n_points);
int kzgb200_cell_proof_monomial(kzgb200_ctx* ctx, uint8_t* out48, size_t n_points);
int kzgb200_compute_cells_and_kzg_proofs(kzgb200_ctx* ctx, const uint8_t* blob, uint8_t* cells_out, uint8_t* proofs_out);
int kzgb200_compute_cells_and_kzg_proofs_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_cells, uint8_t* d_proofs);
int kzgb200_recover_cells_and_kzg_proofs(kzgb200_ctx* ctx, const uint64_t* cell_indices, const uint8_t* cells, size_t n_cells,
                                         uint8_t* cells_out, uint8_t* proofs_out);
int kzgb200_recover_cells_and_kzg_proofs_batch_device(kzgb200_ctx* ctx, const uint64_t* cell_indices, size_t n_cells, const uint8_t* d_cells,
                                                      size_t n_blobs, uint8_t* d_cells_out, uint8_t* d_proofs_out);
int kzgb200_recover_cells_and_kzg_proofs_many(kzgb200_ctx* ctx, const uint64_t* cell_indices, const uint8_t* cells, const uint64_t* cell_offsets,
                                              size_t n_blobs, uint8_t* cells_out, uint8_t* proofs_out, uint8_t* status);
int kzgb200_recover_cells_and_kzg_proofs_many_device(kzgb200_ctx* ctx, const uint64_t* cell_indices, const uint8_t* d_cells,
                                                     const uint64_t* cell_offsets, size_t n_blobs, uint8_t* d_cells_out, uint8_t* d_proofs_out,
                                                     uint8_t* status);
int kzgb200_compute_commitments_and_cell_proofs(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n_blobs, uint8_t* commitments_out,
                                                uint8_t* proofs_out, uint8_t* cells_out, uint8_t* status);
int kzgb200_compute_commitments_and_cell_proofs_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n_blobs, uint8_t* d_commitments_out,
                                                       uint8_t* d_proofs_out, uint8_t* d_cells_out, uint8_t* status);

/* per-phase device timing of batch calls (CUDA event pairs on the stream each phase runs on).  out8 = milliseconds of
 * {G1 decompression, challenge, evaluate, transcript r (exposed part: last chunk copy + host hash + upload), lincomb terms, reduce,
 * final pairing, deferred subgroup checks (run beside the last three)} of the last call. */
int kzgb200_set_profiling(kzgb200_ctx* ctx, int on);
/* Host-memory batches copy their last chunk slab-wise, with the challenge-hash kernel started behind the first slab (on by default:
 * it shortens a blocking call by ~2 ms).  The streaming front-end turns it off for its contexts: with several calls in flight the
 * tail of one call already runs under the copies of the next, and the strided copies would only interleave badly. */
int kzgb200_set_slab_tail(kzgb200_ctx* ctx, int on);
int kzgb200_get_phase_ms(kzgb200_ctx* ctx, float* out8);
/* profiling aid: SM clock stamps of the sections of the last single-GPU final pairing kernel */
int kzgb200_debug_final_ticks(kzgb200_ctx* ctx, long long* out14);
/* f^(3(p^12-1)/r) of the last single-GPU batch check, 12 canonical Fp coefficients of 48 little-endian bytes (the verdict is true iff
 * it is 1), and the split tail's shifted line tables ([256^w]G2, [256^w tau]G2, w = 1..15; len = 783360).  Test aids. */
int kzgb200_debug_last_gt(kzgb200_ctx* ctx, uint8_t* out576);
int kzgb200_debug_lines29w(kzgb200_ctx* ctx, uint8_t* out, size_t len);
/* Self-test of the pairing engine's 16-lane instructions (csrc/vliw29.cuh): every engine program is run `rounds` times on the
 * cooperative executors and on the sequential reference executors from the same seeded register files; mismatches[i] receives
 * the number of registers of program i whose canonical values differ (all zero = pass).  n_programs receives their count. */
int kzgb200_debug_engine_selftest(kzgb200_ctx* ctx, uint32_t seed, int rounds, uint32_t* mismatches32, int* n_programs);
/* the cudaStream_t all work of this context is issued on (for CUDA-event timing by the caller) */
void* kzgb200_stream(kzgb200_ctx* ctx);

/* ---- streaming front-end (SURVEY.md 8f-3): several batches in flight on one GPU --------------------------------
 * A batch is a blob-streaming head (challenges, evaluations, G1 parsing: all SMs busy) followed by a latency-bound tail
 * (transcript hash, MSM reduction, ONE pairing: a handful of CTAs).  A pipeline owns `depth` (1..8; 2 is enough)
 * independent contexts with one host worker thread each, so that the tail of one batch runs under the head -- and,
 * for host buffers, under the PCIe copy -- of the next.  Each ticket is exactly one kzgb200_verify_blob_kzg_proof_batch
 * (host pointers) or ..._batch_device (device pointers) call: same verdicts, same return codes, same z / y.
 * submit returns once the batch is queued (it blocks while `depth` batches are already in flight); the buffers must
 * stay valid and unmodified until the ticket has been waited for.  wait returns that batch's return code and verdict;
 * a ticket can be waited for once (KZGB200_BAD_ARGS otherwise).  Tickets complete in any order; wait in any order.
 * kzgb200_pipeline_context(p, slot) exposes the contexts for the tuning calls (e.g. kzgb200_set_transcript_mode). */
typedef struct kzgb200_pipeline kzgb200_pipeline;
int kzgb200_pipeline_create(kzgb200_pipeline** out, int device, const uint8_t* g2_points, size_t g2_points_len, int depth);
void kzgb200_pipeline_destroy(kzgb200_pipeline* p);   /* finishes what was submitted, then frees */
int kzgb200_pipeline_depth(const kzgb200_pipeline* p);
kzgb200_ctx* kzgb200_pipeline_context(kzgb200_pipeline* p, int slot);
int kzgb200_pipeline_submit(kzgb200_pipeline* p, const uint8_t* blobs, size_t n_blobs, const uint8_t* commitments,
                            size_t n_commitments, const uint8_t* proofs, size_t n_proofs, uint8_t* z_out, uint8_t* y_out,
                            uint64_t* ticket);
int kzgb200_pipeline_submit_device(kzgb200_pipeline* p, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                   const uint8_t* d_proofs, size_t n, uint8_t* d_z_out, uint8_t* d_y_out, uint64_t* ticket);
int kzgb200_pipeline_wait(kzgb200_pipeline* p, uint64_t ticket, int* ok);

/* pinned host memory helpers for callers that want full-rate host->device copies */
void* kzgb200_alloc_pinned(size_t bytes);
void kzgb200_free_pinned(void* p);

#ifdef __cplusplus
}
#endif
#endif
