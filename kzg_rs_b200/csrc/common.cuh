// Shared declarations of the sm_100a kernels of the kzg-rs verification hot path (K1..K8 of SURVEY.md section 2.1):
// constants, device-resident structures, small load helpers and the prototypes of every kernel.  The kernels live in
// k_*.cu (one translation unit per group so that they compile in parallel); kzgb200.cu is the host runtime.
#pragma once
#include <cuda_runtime.h>
#include "sha256.cuh"
#include "verify.cuh"
#include "vliw.cuh"
#include "vliw29.cuh"
#include "glv.cuh"

namespace kzgb200 {

constexpr int kFieldElementsPerBlob = 4096;       // reference src/consts.rs:7
constexpr int kBytesPerBlob = 4096 * 32;          // src/consts.rs:8
constexpr uint32_t kErrBlob = 1, kErrCommitment = 2, kErrProof = 4, kErrScalar = 8;
// canonical (non-Montgomery) z_i, y_i; the memory image is 2 x 32 little-endian bytes, which is exactly what
// the batch transcript hashes (reference src/kzg_proof.rs:320-328) and what ranks exchange
struct ZY { Fr z, y; };

// Device-resident trusted-setup tables (K8; replaces KzgSettings::load_trusted_setup_file,
// reference src/trusted_setup.rs:94-98 and build.rs:131-170).
struct DeviceTables {
    // twiddle[g] = roots_of_unity[2g] = omega^bitrev12(2g), Montgomery form.  In the bit-reversed domain the
    // group of 2^(k+1) consecutive points starting at index a has prod (z - w_i) = z^(2^(k+1)) - w_a^(2^(k+1)),
    // and w_a^(2^k) = roots_of_unity[2g] for g = a >> (k+1), independent of the level k.
    Fr twiddle[2048];
    // the same twiddles in the order thread t of eval_kernel consumes them (post-order over its 32-leaf subtree): 31 per
    // thread + 1 pad, so the stream is sequential and the next one can be fetched while the current merge runs
    Fr twiddle_po[128][32];
    PairingTables pairing;
    // the same line triples in the representation of the cooperative pairing engine (vliw29.cuh): [0] = G2 generator, [1] = [tau]G2
    vliw29::LineCoeffs29 lines29[2][kMillerSteps];
    // ... and of their multiples by 256^w, w = 1..15 ([0] = [256^w]G2, [1] = [256^w tau]G2): the batch verifier's split tail pairs MSM
    // window w with them (window_miller_kernel), so the window weights need no Horner chain on the G1 side
    vliw29::LineCoeffs29 lines29w[2][15][kMillerSteps];
    // fixed-base table of the G1 generator: gen_table[w][d-1] = [d * 16^w] G, d = 1..15, w < 64
    G1Affine gen_table[64][15];
    uint32_t setup_ok;
};

// ---- launch shapes shared by kernels and host ---------------------------------------------------------------
#ifndef KSHA_THREADS
#define KSHA_THREADS 32
#endif
constexpr int kShaThreads = KSHA_THREADS;     // blobs (threads) per CTA of K2
constexpr int kEvalThreads = 128;
constexpr int kLeavesPerThread = kFieldElementsPerBlob / kEvalThreads;  // 32
constexpr int kTreeGroup = 16;      // transcript entries (160 B each) per leaf hash: 40 compressions
constexpr int kTreeMid = 32;        // leaf digests per middle-level hash: 17 compressions
constexpr int kWindows = 16, kBuckets = 256, kMsmSets = 3, kDigitRows = 4 * kWindows;   // rows: (kind r|rz) x (half lo|hi) x window
static_assert(kWindows - 1 == sizeof(DeviceTables::lines29w[0]) / sizeof(DeviceTables::lines29w[0][0]), "one shifted line table per window > 0");
constexpr int kMinSlice = 8, kMsmRows = kMsmSets * 2 * kWindows;   // bucket accumulation: fewest entries per thread (msm_slice_len); rows = (set, GLV half, window)
constexpr int kWinLanes = kBuckets;                                 // window sums: one thread per bucket (suffix scan + tree in shared memory)
constexpr int kWinSmemBytes = kWinLanes * 144;                      // one Jacobian point per thread
constexpr int kCombineThreads = 544;    // msm_combine_kernel: 384 engine threads (three Horner chains in lockstep) + 160 helpers
constexpr int kCombHelpers = 160;       // ... of which helpers ([s]G, flags; alone: msm_sg_kernel)
constexpr int kCombineSmemBytes = 48 * 1024;
constexpr int kFinalThreads = 64;       // G1 prelude of the final check (sums, [s]G, affine conversion)
constexpr int kPairThreads = 768;       // pairing engine: 24 warps = 24 products (one per warp) or 48 sums (16 lanes each) at a time
constexpr int kManyThreads = 512, kManyGroups = 28;   // many_pairing_kernel: checks run in lockstep by one CTA (28 x 36 products = 1.97 x 512; 128 registers)
constexpr int kManyCtasPerSm = 1;                     // (two CTAs of 14 checks per SM, not in lockstep with each other: 491 k instead of 555 k checks/s)
constexpr int kManyWarps = 4;         // many_pairing_warp_kernel (identity inputs): one check per warp
constexpr int kHarnessMaxDegree = 16;
constexpr int kLagWindows = 32, kLagEntries = 255;
constexpr int kLagTerms = kFieldElementsPerBlob * kLagWindows;   // (point, window) terms of a blob's commitment MSM
constexpr int kLagMsmThreads = 256, kLagMaxSlices = kLagTerms / kLagMsmThreads / 2;   // lag_msm_slice_kernel: >= 2 terms per thread
constexpr int kLagFinishThreads = 64;                             // lag_msm_finish_kernel
// EIP-7594 cells (k_cells.cu)
constexpr int kCellsPerExtBlob = 128, kFieldElementsPerCell = 64, kBytesPerCell = 2048;
constexpr int kCellNttThreads = 512;                              // compute_cells_kernel: one CTA per blob, 4096 values in shared memory
constexpr int kCellNttSmemBytes = kFieldElementsPerBlob * 32;     // 128 KiB
constexpr int kCellAggSlices = 16;                                // CTAs per cell index of the r-weighted value sums
constexpr int kCellHarnessMaxDegree = 192;

__device__ __forceinline__ Fr load_fe_be(const uint4* p) {
    uint4 hi = __ldg(p), lo = __ldg(p + 1);   // 32 big-endian bytes: hi holds the most significant 16
    Fr f;
    f.l[7] = sha_bswap(hi.x); f.l[6] = sha_bswap(hi.y); f.l[5] = sha_bswap(hi.z); f.l[4] = sha_bswap(hi.w);
    f.l[3] = sha_bswap(lo.x); f.l[2] = sha_bswap(lo.y); f.l[1] = sha_bswap(lo.z); f.l[0] = sha_bswap(lo.w);
    return f;
}
__device__ __forceinline__ Fr ldg_fr(const Fr* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    Fr f;
    f.l[0] = a.x; f.l[1] = a.y; f.l[2] = a.z; f.l[3] = a.w; f.l[4] = b.x; f.l[5] = b.y; f.l[6] = b.z; f.l[7] = b.w;
    return f;
}

// per-rank partial result exchanged between ranks (the payload of the allgather)
struct Partial {
    G1 a, b;          // sum r_i pi_i ; sum (r_i C_i + r_i z_i pi_i) - [sum r_i y_i]G (the fixed-base term is folded in by msm_combine_kernel)
    Fr ry;            // a scalar s still to be applied as - [s]G by the final check (normal form); zero since the term is folded into b
    uint32_t err;     // OR of the per-blob error flags of this rank
    uint32_t pad[7];
};

// dynamic shared memory of the final kernels: engine register file, program tables, G1 tree scratch (> 48 KB: opt-in)
struct FinalSmem {                       // prelude kernels (padded: see kTailPadSmem in runtime.cuh)
    G1 sm[kFinalThreads];
    unsigned char pad[20 * 1024];
};
struct PairSmem {                        // pairing_check_kernel
    f29::F29 regs[vliw29::kTotalRegs];
    vliw29::SharedTables stab;
};
// hand-over from the prelude kernel to the pairing kernel (device memory, 256 bytes into the context's 512-byte scratch)
struct FinalPts { G1Affine pts[2]; uint32_t go; };

// hand-over buffer of the split tail of a batch (kzgb200_ctx::d_split; see window_miller_kernel)
struct SplitTail {
    G1 sg;                                  // [s]G, s = sum r_i y_i (msm_sg_kernel)
    uint32_t err;                           // OR of the per-blob error flags (msm_sg_kernel)
    uint32_t pad[3];
    G1Affine pts[kWindows][2];              // per window: -W0_w, B_w (window_prelude_kernel)
    alignas(16) f29::F29 f[kWindows][12];   // per-window Miller values (window_miller_kernel)
    Fp gt[12];                              // f^(3(p^12-1)/r) of the last batch check, canonical integers (kzgb200_debug_last_gt)
};

constexpr int kManyStride = vliw::kTotalRegsThr * 12 + 1;     // words between the register files of consecutive groups (odd: bank skew)
constexpr int kManySmemBytes = kManyGroups * kManyStride * 4 + (int)sizeof(vliw::SharedTables) + vliw::kNumSharedRegs * (int)sizeof(Fp) +
                               kManyGroups * (2 * (int)sizeof(G1Affine) + 2) + 64;
// Device tables of the cell path (kzgb200_load_cell_setup): roots of unity of the extended domain, the fixed bases of the RLI
// MSM, and the Miller-loop lines of [tau^64]G2.
struct CellTables {
    Fr w4096[2048], w4096_inv[2048];   // omega4096^(+-k), natural order, Montgomery
    Fr coset[4096];                    // omega8192^m / 4096
    Fr shift64[kCellsPerExtBlob];      // h_k^64 = omega128^rev7(k)
    Fr shift_inv[kCellsPerExtBlob];    // h_k^-1
    Fr w64_inv[kFieldElementsPerCell / 2];
    Fr omega8192, inv64;
    G1Affine tau_tab[kFieldElementsPerCell][4];   // [2^(64q) tau^m]G1
    LineCoeffs tau64_lines[kMillerSteps];
    vliw29::LineCoeffs29 lines29[kMillerSteps];    // [tau^64]G2 for pairing_check_kernel
    uint32_t ok;
};
// Cell proofs (kzgb200_load_cell_proof_setup, k_cell_proofs.cu): FK20 over the fixed bases W_b[f] = DFT_128(w_b)[f] (b < 64,
// f < 128), each with a GLV window table tab[f * 64 + b][w][d - 1] = [d * 256^w] W_b[f] (w < 16, d = 1..255), and the scalar tables
// of the 8192-point recovery transforms.
constexpr int kFk20Bases = kFieldElementsPerCell * kCellsPerExtBlob;   // 8192
constexpr int kFk20Windows = 16, kFk20Entries = 255;
constexpr size_t kFk20TablePoints = (size_t)kFk20Bases * kFk20Windows * kFk20Entries;
constexpr int kExtElements = 2 * kFieldElementsPerBlob;                  // 8192
struct ProofTables {
    Fr w8192[kFieldElementsPerBlob], w8192_inv[kFieldElementsPerBlob];   // omega8192^(+-i)
    Fr pow7[kExtElements];                  // 7^i / 8192: the spec's coset shift (PRIMITIVE_ROOT_OF_UNITY) with the inverse 1/n
    Fr pow7_inv[kFieldElementsPerBlob];     // 7^-i / 8192
    Fr s7_64;                               // 7^64
};
// ---- kernels (k_*.cu) ----------------------------------------------------------------------------------------
__global__ void setup_tables_kernel(DeviceTables* T, const uint8_t* g2_points);
__global__ void setup_lines29_kernel(DeviceTables* T);
__global__ void setup_lines29w_kernel(DeviceTables* T, const uint8_t* g2_points, LineCoeffs* scratch);
constexpr int kChallengeSlabs = 8;   // slab-wise arrival of the last host chunk (k_challenge.cu)
void launch_challenge(int stages, cudaStream_t st, const uint8_t* blobs, const uint8_t* commitments, int n, Fr* z_mont, ZY* zy, Fr* zpow,
                      const uint8_t* slab_flags = nullptr);   // K2
__global__ void eval_kernel(const uint8_t* __restrict__ blobs, int n, const Fr* __restrict__ zpow, const DeviceTables* __restrict__ T,
                            ZY* __restrict__ zy, uint32_t* __restrict__ status);
__global__ void g1_decompress_kernel(const uint8_t* __restrict__ commitments, const uint8_t* __restrict__ proofs, int n, G1Affine* __restrict__ C,
                                     G1Affine* __restrict__ P, uint32_t* __restrict__ status, bool with_subgroup_check);
__global__ void g1_subgroup_kernel(const G1Affine* __restrict__ C, const G1Affine* __restrict__ P, int n, uint32_t* __restrict__ status);
__global__ void transcript_schedule_kernel(const uint8_t* __restrict__ commitments, const ZY* __restrict__ zy, const uint8_t* __restrict__ proofs,
                                           uint64_t n, uint32_t* __restrict__ wk, uint64_t first_blk, uint64_t blk_count);
__global__ void transcript_chain_kernel(const uint32_t* __restrict__ wk_all, uint64_t n, Fr* __restrict__ r_mont, uint32_t* __restrict__ state,
                                        uint64_t first_blk, uint64_t blk_count);
__global__ void transcript_words_kernel(const uint8_t* __restrict__ commitments, const ZY* __restrict__ zy, const uint8_t* __restrict__ proofs,
                                        uint64_t first_entry, uint64_t entry_count, uint32_t* __restrict__ words);
__global__ void transcript_tree_leaf_words_kernel(const uint32_t* __restrict__ words, uint64_t n, uint32_t* __restrict__ digests,
                                                  uint64_t first_group, uint64_t group_count);
__global__ void r_from_digest_kernel(const uint32_t* __restrict__ digest, Fr* __restrict__ r_mont);
__global__ void z_setup_kernel(const uint8_t* __restrict__ z_be32, int n, Fr* __restrict__ z_mont, ZY* __restrict__ zy, Fr* __restrict__ zpow,
                               uint32_t* __restrict__ status);
__global__ void import_parsed_kernel(const uint8_t* __restrict__ c104, const uint8_t* __restrict__ p104, const uint8_t* __restrict__ z32,
                                     const uint8_t* __restrict__ y32, int n, G1Affine* __restrict__ C, G1Affine* __restrict__ P,
                                     uint8_t* __restrict__ c48, uint8_t* __restrict__ p48, Fr* __restrict__ z_mont, ZY* __restrict__ zy);
// weights: per-entry scalars (Montgomery) in place of r^(offset + i); nullptr = the powers of r
__global__ void msm_scalars_kernel(const Fr* __restrict__ z_mont, const ZY* __restrict__ zy, const Fr* __restrict__ r_mont, uint64_t offset, int n,
                                   uint8_t* __restrict__ digits, Fr* __restrict__ ry, const Fr* __restrict__ weights);
__global__ void msm_sort_kernel(const uint8_t* __restrict__ digits, int n, uint32_t* __restrict__ order, uint32_t* __restrict__ start);
void launch_msm_bucket(int ctas_per_sm, int n, int slice, cudaStream_t st, const G1Affine* C, const G1Affine* P, const uint32_t* order,
                       const uint32_t* start, G1* halfsum, G1* part);
void launch_msm_bucket_join(int lanes, int n, int slice, cudaStream_t st, const uint32_t* start, const G1* halfsum, const G1* part, G1* buckets);
__global__ void msm_window_kernel(const G1* __restrict__ buckets, G1* __restrict__ windows);
__global__ void msm_combine_kernel(const G1* __restrict__ windows, const Fr* __restrict__ ry, const uint32_t* __restrict__ status, int n,
                                   const DeviceTables* __restrict__ T, Partial* __restrict__ out, uint32_t* flag, uint32_t epoch);
__global__ void msm_sg_kernel(const Fr* __restrict__ ry, const uint32_t* __restrict__ status, int n, const DeviceTables* __restrict__ T,
                              SplitTail* __restrict__ out);
__global__ void window_prelude_kernel(const G1* __restrict__ windows, SplitTail* __restrict__ io);
__global__ void window_miller_kernel(const DeviceTables* __restrict__ T, SplitTail* __restrict__ io, long long* __restrict__ ticks);
__global__ void split_final_kernel(const SplitTail* __restrict__ io, uint32_t* __restrict__ result, Fp* __restrict__ gt, long long* __restrict__ ticks);
__global__ void wait_flags_kernel(const uint32_t* flags, int count, uint32_t epoch, uint32_t* __restrict__ timed_out);
__global__ void batch_final_kernel(const Partial* __restrict__ parts, int nparts, const DeviceTables* __restrict__ T, uint32_t* __restrict__ result,
                                   FinalPts* __restrict__ out);
__global__ void single_final_kernel(const G1Affine* __restrict__ C, const G1Affine* __restrict__ P, const ZY* __restrict__ zy,
                                    const uint32_t* __restrict__ status, const DeviceTables* __restrict__ T, uint32_t* __restrict__ result,
                                    FinalPts* __restrict__ out);
// lines_b: line table of the G2 point paired with pts[0]; nullptr = [tau]G2 (T->lines29[1], the blob checks)
// gt (nullable): receives f^(3(p^12-1)/r) as 12 canonical integers
__global__ void pairing_check_kernel(const FinalPts* __restrict__ in, const DeviceTables* __restrict__ T, const vliw29::LineCoeffs29* __restrict__ lines_b,
                                     uint32_t* __restrict__ result, long long* __restrict__ ticks, Fp* __restrict__ gt);
__global__ void engine_selftest_kernel(uint32_t seed, int rounds, f29::F29* __restrict__ ref, uint32_t* __restrict__ mismatches);
// final check of a batch = G1 prelude + pairing engine, back to back on `st`; scratch512 = the context's 512-byte device scratch
// (ticks at +128 when profiling, the hand-over points at +256); lines_b: see pairing_check_kernel (cells: [tau^64]G2)
inline void launch_batch_final(cudaStream_t st, const Partial* parts, int nparts, const DeviceTables* T, uint32_t* result, unsigned char* scratch512,
                               bool ticks, const vliw29::LineCoeffs29* lines_b = nullptr, Fp* gt = nullptr) {
    FinalPts* fp = reinterpret_cast<FinalPts*>(scratch512 + 256);
    batch_final_kernel<<<1, kFinalThreads, sizeof(FinalSmem), st>>>(parts, nparts, T, result, fp);
    pairing_check_kernel<<<1, kPairThreads, sizeof(PairSmem), st>>>(fp, T, lines_b, result, ticks ? reinterpret_cast<long long*>(scratch512 + 128) : nullptr, gt);
}
__global__ void many_lhs_kernel(const uint8_t* __restrict__ z32, const uint8_t* __restrict__ y32, const G1Affine* __restrict__ C,
                                const G1Affine* __restrict__ P, size_t m, const DeviceTables* __restrict__ T, G1Affine* __restrict__ X,
                                uint32_t* __restrict__ status);
__global__ void many_lhs_zy_kernel(const ZY* __restrict__ zy, const G1Affine* __restrict__ C, const G1Affine* __restrict__ P, size_t m,
                                   const DeviceTables* __restrict__ T, G1Affine* __restrict__ X, const uint32_t* __restrict__ status);
// e(X_i, G2) e(-P_i, Q) == 1; lines_b: line table of Q, nullptr = [tau]G2 (T->pairing.tau_g2)
__global__ void many_pairing_kernel(const G1Affine* __restrict__ X, const G1Affine* __restrict__ P, const uint32_t* __restrict__ status, size_t m,
                                    const DeviceTables* __restrict__ T, const LineCoeffs* __restrict__ lines_b, uint8_t* __restrict__ verdicts);
__global__ void many_pairing_warp_kernel(const G1Affine* __restrict__ X, const G1Affine* __restrict__ P, size_t m, const DeviceTables* __restrict__ T,
                                         const LineCoeffs* __restrict__ lines_b, uint8_t* __restrict__ verdicts);
__global__ void export_scalars_kernel(const ZY* __restrict__ zy, int n, uint8_t* __restrict__ z_out, uint8_t* __restrict__ y_out);
__global__ void r_to_raw_kernel(const Fr* __restrict__ r_mont, ZY* __restrict__ out);
__global__ void status_or_kernel(const uint32_t* __restrict__ status, int n, uint32_t* __restrict__ out);
__global__ void harness_parse_points_kernel(const uint8_t* bytes, int n, G1Affine* out, uint32_t* bad);
__global__ void harness_blob_kernel(uint64_t seed, int n, int D, const DeviceTables* __restrict__ T, uint8_t* __restrict__ blobs);
__global__ void harness_commit_kernel(uint64_t seed, int n, int D, const G1Affine* __restrict__ M, const Fr* __restrict__ z_mont,
                                      uint8_t* __restrict__ out, int want_proof);
__global__ void lag_parse_kernel(const uint8_t* __restrict__ bytes, G1Affine* __restrict__ out, uint32_t* __restrict__ bad);
__global__ void lag_table_kernel(const G1Affine* __restrict__ L, G1* __restrict__ table);
__global__ void blob_scalars_kernel(const uint8_t* __restrict__ blobs, int n, Fr* __restrict__ scalars, uint32_t* __restrict__ status);
__global__ void quotient_kernel(const uint8_t* __restrict__ blobs, int n, const Fr* __restrict__ z_mont, const ZY* __restrict__ zy,
                                const DeviceTables* __restrict__ T, Fr* __restrict__ scalars);
__global__ void lag_msm_slice_kernel(const Fr* __restrict__ scalars, int n, int slices, const G1* __restrict__ table, G1* __restrict__ partials,
                                     uint8_t* __restrict__ out48);
__global__ void lag_msm_finish_kernel(const G1* __restrict__ partials, int n, int slices, uint8_t* __restrict__ out48);
__global__ void cell_setup_kernel(CellTables* T, const uint8_t* __restrict__ g2_tau64);
__global__ void cell_setup_points_kernel(CellTables* T, const uint8_t* __restrict__ g1_monomial48);
__global__ void cell_setup_lines29_kernel(CellTables* T);
__global__ void compute_cells_kernel(const uint8_t* __restrict__ blobs, int n, const CellTables* __restrict__ T, uint8_t* __restrict__ cells,
                                     uint32_t* __restrict__ status);
__global__ void compute_cells_coeffs_kernel(const uint8_t* __restrict__ blobs, int n, const CellTables* __restrict__ T, uint8_t* __restrict__ cells,
                                            uint32_t* __restrict__ status, Fr* __restrict__ coeffs);
// cell proofs / recovery (k_cell_proofs.cu)
__global__ void proof_setup_kernel(ProofTables* P);
__global__ void mono_load_kernel(const uint8_t* __restrict__ lag48, G1* __restrict__ a, uint32_t* __restrict__ bad);
__global__ void mono_level_kernel(G1* __restrict__ a, int len, const CellTables* __restrict__ T);
__global__ void mono_finish_kernel(const G1* __restrict__ a, const CellTables* __restrict__ T, G1Affine* __restrict__ mono, uint32_t* __restrict__ bad);
__global__ void mono_compress_kernel(const G1Affine* __restrict__ mono, int n, uint8_t* __restrict__ out48);
__global__ void fk20_w_kernel(const G1Affine* __restrict__ mono, const CellTables* __restrict__ T, G1Affine* __restrict__ W);
__global__ void fk20_table_kernel(const G1Affine* __restrict__ W, G1Affine* __restrict__ tab);
__global__ void fk20_scalars_kernel(const Fr* __restrict__ coeffs, const CellTables* __restrict__ T, Fr* __restrict__ U);
__global__ void fk20_products_kernel(const Fr* __restrict__ U, const G1Affine* __restrict__ tab, G1* __restrict__ V);
__global__ void fk20_proofs_kernel(const G1* __restrict__ V, const CellTables* __restrict__ T, uint8_t* __restrict__ proofs);
__global__ void recover_z_kernel(const uint32_t* __restrict__ missing, int n_missing, const CellTables* __restrict__ T, const ProofTables* __restrict__ P,
                                 Fr* __restrict__ zvals);
__global__ void recover_load_kernel(const uint8_t* __restrict__ cells, int n_cells, const int* __restrict__ pos, const Fr* __restrict__ zvals, int nb,
                                    Fr* __restrict__ A, uint32_t* __restrict__ status);
__global__ void recover_ntt_inv_kernel(Fr* __restrict__ A, const CellTables* __restrict__ T);
__global__ void recover_ntt_div_kernel(Fr* __restrict__ A, const CellTables* __restrict__ T, const Fr* __restrict__ zvals);
__global__ void recover_mid_kernel(Fr* __restrict__ A, const ProofTables* __restrict__ P, int nb);
__global__ void recover_final_kernel(const Fr* __restrict__ A, const ProofTables* __restrict__ P, int nb, Fr* __restrict__ coeffs);
__global__ void recover_blob_kernel(const Fr* __restrict__ coeffs, const CellTables* __restrict__ T, uint8_t* __restrict__ blobs);
__global__ void cell_points_kernel(const uint8_t* __restrict__ bytes, int count, G1Affine* __restrict__ out, uint32_t* __restrict__ status, uint32_t flag);
__global__ void cell_check_kernel(const uint8_t* __restrict__ cells, int n, uint32_t* __restrict__ status);
// meta = [cell index (n) | unique-commitment index (n) | cells ordered by cell index (n) | start of each index in that order (129)]
__global__ void cell_scalars_kernel(const uint32_t* __restrict__ meta, int n, const G1Affine* __restrict__ U, const uint32_t* __restrict__ ustatus,
                                    const CellTables* __restrict__ T, Fr* __restrict__ z_mont, ZY* __restrict__ zy, G1Affine* __restrict__ C,
                                    uint32_t* __restrict__ status);
__global__ void cell_agg_kernel(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ meta, int n, const Fr* __restrict__ rk, Fr* __restrict__ agg);
__global__ void cell_interp_kernel(const Fr* __restrict__ agg, const uint32_t* __restrict__ meta, int n, const CellTables* __restrict__ T,
                                   Fr* __restrict__ coeffs);
__global__ void cell_rli_kernel(const Fr* __restrict__ coeffs, const CellTables* __restrict__ T, Partial* __restrict__ out);
// verify_cell_kzg_proof_batch_many (k_cells.cu): goff = the k + 1 group offsets, gbad = per-group BadArgs flags
__global__ void many_group_status_kernel(const uint32_t* __restrict__ status, int n, const uint32_t* __restrict__ goff, int k, uint32_t* __restrict__ gbad);
__global__ void many_weights_kernel(int n, const uint32_t* __restrict__ goff, int k, const uint8_t* __restrict__ rg, const uint32_t* __restrict__ gbad,
                                    Fr* __restrict__ w, uint32_t* __restrict__ status);
__global__ void many_terms_kernel(int n, const Fr* __restrict__ w, const Fr* __restrict__ z_mont, const G1Affine* __restrict__ C, const G1Affine* __restrict__ P,
                                  G1* __restrict__ terms);
__global__ void many_group_sums_kernel(const uint32_t* __restrict__ goff, const G1* __restrict__ terms, G1* __restrict__ AB);
__global__ void many_run_interp_kernel(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ fmeta, int n, int runs, const Fr* __restrict__ w,
                                       const CellTables* __restrict__ T, Fr* __restrict__ rcoef);
__global__ void many_group_rli_kernel(const Fr* __restrict__ rcoef, const uint32_t* __restrict__ grun, const G1* __restrict__ AB, const CellTables* __restrict__ T,
                                      G1Affine* __restrict__ X, G1Affine* __restrict__ A);
__global__ void cell_harness_terms_kernel(uint64_t seed, int n, int D, const G1Affine* __restrict__ M, G1* __restrict__ terms);
__global__ void cell_harness_sums_kernel(int n, const G1* __restrict__ terms, G1* __restrict__ sums);
__global__ void cell_harness_points_kernel(int n, const G1* __restrict__ sums, const CellTables* __restrict__ T, uint8_t* __restrict__ commitments,
                                           uint8_t* __restrict__ proofs);
__global__ void cell_harness_eval_kernel(uint64_t seed, int n, int D, const CellTables* __restrict__ T, uint8_t* __restrict__ cells);

}  // namespace kzgb200
