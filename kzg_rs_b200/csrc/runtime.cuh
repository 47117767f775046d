// Internal header of the host runtime: the per-GPU context and the phase launchers shared by kzgb200.cu (single-GPU C ABI)
// and group.cu (blob-sharded multi-GPU batches).  Not part of the public boundary (that is include/kzgb200.h).
#pragma once
#include <cuda_runtime.h>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>
#include "../../include/kzgb200.h"
#include "common.cuh"
#include "host_sha256.h"

namespace kzgb200 {

constexpr int kTailSms = 8;                    // SMs kept free of deferred subgroup checks for the latency-bound tail kernels
constexpr int kTailSmsSplit = 20;              // ... with the split tail: 16 window Miller CTAs, msm_combine_kernel, the product CTA
constexpr int kTailHogSmem = 200 * 1024;       // dynamic shared memory of a subgroup-check CTA in deferred mode (never touched)
constexpr int kTailPadSmem = 28 * 1024;        // ... and of the tail kernels: 200 KB + 28 KB do not fit one SM
static_assert(sizeof(FinalSmem) >= (size_t)kTailPadSmem && sizeof(PairSmem) >= (size_t)kTailPadSmem, "the final-check kernels must not fit beside a subgroup-check CTA");
static_assert(sizeof(Partial) == KZGB200_PARTIAL_BYTES, "Partial layout is part of the ABI");
static_assert(sizeof(ZY) == 64, "ZY layout is part of the ABI");

enum Phase { kPhParse = 0, kPhChallenge, kPhEval, kPhTranscript, kPhLincomb, kPhReduce, kPhFinal, kPhCount };
constexpr int kMaxChunks = 64, kWorkStreams = 4;
constexpr size_t kMinChunk = 1024;             // blobs per host->device chunk (128 MiB)
struct Chunk { size_t lo, cnt; };

// Multi-threaded memcpy for the pinned staging ring (pageable caller memory -> pinned buffers the DMA engine reads at full rate).
struct CopyPool {
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cv, cv_done;
    const uint8_t* src = nullptr;
    uint8_t* dst = nullptr;
    size_t bytes = 0, piece = 1 << 20, next = 0, pieces = 0, done = 0;
    uint64_t gen = 0;
    bool stop = false;
    explicit CopyPool(int nthreads);
    ~CopyPool();
    void copy(uint8_t* d, const uint8_t* s, size_t n);   // blocking; the caller takes part
    void work(uint64_t seen);
    bool grab(size_t* off, size_t* len);
};

// State of the cell path (EIP-7594), created by kzgb200_load_cell_setup.  Workspace sized for `cap` cells / `blob_cap` blobs.
struct CellCtx {
    CellTables* tables = nullptr;
    size_t cap = 0, blob_cap = 0;
    uint8_t *d_cells = nullptr, *d_p = nullptr, *d_uc = nullptr;   // staging of host cells / proofs, unique commitment bytes
    uint32_t *d_meta = nullptr, *d_ustatus = nullptr;              // see cell_scalars_kernel
    G1Affine* d_U = nullptr;                                       // unique commitments
    Fr *d_rk = nullptr, *d_agg = nullptr, *d_coeffs = nullptr;
    Partial* d_part = nullptr;                                     // [0] = LL / RLC + RLP (launch_lincomb), [1] = (O, -RLI)
    uint8_t* d_ext = nullptr;                                      // compute_cells output of a host blob (128 cells)
    // pinned host side: metadata, unique commitments, and (device-resident inputs) the copies the transcript is hashed from
    size_t host_cap = 0;
    uint32_t* h_meta = nullptr;
    uint8_t *h_uc = nullptr, *h_c = nullptr, *h_cells = nullptr, *h_p = nullptr;
    uint64_t* h_idx = nullptr;
    std::vector<uint32_t> slot;                                    // open-addressing table of the commitment deduplication
    cudaEvent_t ev_r = nullptr, ev_rli = nullptr;
    // cell proofs and recovery (kzgb200_load_cell_proof_setup): tables, and a workspace for up to proof_cap blobs at a time
    ProofTables* ptables = nullptr;
    G1Affine *d_mono = nullptr, *d_fk_tab = nullptr;               // [tau^m]G1 (m < 4096), FK20 window tables (kFk20TablePoints)
    size_t proof_cap = 0;
    Fr *d_pcoef = nullptr, *d_fkU = nullptr, *d_A = nullptr;        // coefficients x 4096 / recovered coefficients, U_b[f], 8192-point work
    G1* d_V = nullptr;                                             // V[f] = sum_b U_b[f] W_b[f]
    G1* d_pcommit = nullptr;                                       // IDFT(V)[0] per blob: the commitments of a pass (Jacobian)
    uint8_t* d_rblobs = nullptr;                                   // recovered blobs
    uint8_t *d_rin = nullptr, *d_pout = nullptr;                   // staging of one host call: input cells, 128 proofs
    RecoverPlan* d_plans = nullptr;                                // recovery: the index sets of a pass (proof_cap), see recover_plan
    Fr* d_z = nullptr;                                             // their Z rows (2 x 128 per plan), see recover_z_kernel
    size_t mstage_cells = 0, mout_cap = 0;                         // recover_cells_and_kzg_proofs_many, host form: staging of one pass's
    uint8_t *d_mstage = nullptr, *d_mcells = nullptr, *d_mproofs = nullptr;   // input cells, output cells and proofs (grow on demand)
    // verify_cell_kzg_proof_batch_many: per-group buffers for gcap groups, the fallback's workspace (per cell, per (group, index)
    // run), and the last call's r_g (32 bytes each, canonical big-endian) followed by rho
    size_t gcap = 0, fmeta_cap = 0, terms_cap = 0, rcoef_cap = 0;
    uint32_t *d_goff = nullptr, *d_gbad = nullptr, *d_fmeta = nullptr;   // group offsets (k + 1), BadArgs flags (k), see many_run_interp_kernel
    uint8_t *d_rg = nullptr, *d_gv = nullptr;                      // r_g and rho (k + 1 x 32 bytes), fallback verdicts (k)
    G1 *d_terms = nullptr, *d_AB = nullptr;                        // fallback: per-cell terms (2 per cell), per-group A_g, B'_g
    G1Affine* d_gX = nullptr;                                      // fallback: X_g (k), then A_g (k)
    Fr* d_rcoef = nullptr;                                         // fallback: interpolated coefficients per run (64 each)
    std::vector<uint8_t> many_rg;
    size_t many_k = 0;
    bool many_done = false;
};

}  // namespace kzgb200

struct kzgb200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    kzgb200::DeviceTables* tables = nullptr;
    // workspace, sized for `cap` blobs
    size_t cap = 0, blob_cap = 0, many_cap = 0, host_cap = 0;
    uint8_t *d_blobs = nullptr, *d_c = nullptr, *d_p = nullptr;     // staging of host inputs
    kzgb200::Fr* d_z_mont = nullptr;
    kzgb200::Fr* d_zpow = nullptr;           // z^(2^k), k = 0..12, per blob (K2 -> K1/K3)
    kzgb200::ZY* d_zy = nullptr;
    kzgb200::G1Affine *d_C = nullptr, *d_P = nullptr;
    uint32_t* d_status = nullptr;
    kzgb200::Fr *d_ry = nullptr, *d_r = nullptr;
    uint8_t* d_digits = nullptr;            // [4*16][cap]
    uint32_t *d_order = nullptr, *d_start = nullptr;
    kzgb200::G1 *d_buckets = nullptr, *d_windows = nullptr;
    kzgb200::G1 *d_halfsum = nullptr, *d_part = nullptr;   // bucket accumulation: finished half-buckets [96][256], slice partials [96][slices][2]
    kzgb200::Partial* d_partial = nullptr;
    uint32_t* d_result = nullptr;
    uint8_t *d_zout = nullptr, *d_yout = nullptr;
    uint8_t* d_many = nullptr;
    kzgb200::G1* d_lag_table = nullptr;      // [4096][32][255] window table of the Lagrange G1 points (commit / prove only)
    kzgb200::Fr* d_scalars = nullptr;
    kzgb200::G1* d_lag_part = nullptr;      // slice partials of the commitment MSM (lag_msm_slice_kernel)
    uint32_t* d_wk = nullptr;       // device transcript scratch: W+K words (exact-device) / entry words + leaf digests (tree)
    size_t wk_cap = 0;
    uint32_t* h_result = nullptr;   // pinned
    // host side of the transcript: pinned copies of (z, y) [or leaf digests], of the commitments / proofs when the inputs are
    // device-resident, and of the 32-byte digest
    uint8_t *h_zy = nullptr, *h_c = nullptr, *h_p = nullptr, *h_digest = nullptr, *h_partial = nullptr;
    uint32_t* d_digest = nullptr;
    const uint8_t *tr_c = nullptr, *tr_p = nullptr;    // host commitments / proofs the transcript reads (caller's or h_c / h_p)
    kzgb200::HostSha256 tr_sha;
    size_t tr_n = 0, tr_done = 0;     // entries of the current transcript / entries (exact), blocks (exact-device), groups (tree) hashed
    int tr_next_chunk = 0;            // next chunk whose host payload has not been consumed yet
    int tr_enqueued = 0;              // chunks whose payload copy has been queued by the current call
    bool tr_active = false;
    void (*chunk_sink)(void*, int) = nullptr;   // set by a group: consumes chunk payloads instead of the local transcript hash
    void* chunk_sink_arg = nullptr;
    // inputs of the current shard (device pointers owned by the caller or by the staging buffers)
    const uint8_t *cur_c = nullptr, *cur_p = nullptr;
    size_t cur_n = 0;
    kzgb200::Chunk chunks[kzgb200::kMaxChunks];
    int nchunks = 0;
    int transcript_mode = KZGB200_TRANSCRIPT_EXACT;
    int num_sms = 148;
    int msm_occ = 3;                   // CTAs per SM of the bucket kernel variant in use (KZGB200_MSM_OCC: 2, 3, 4)
    int msm_join = 2;                  // threads per bucket of the join kernel (KZGB200_MSM_JOIN: 2, 4, 8; measured 1.08 / 1.18 / 1.15 ms lincomb phase)
    int msm_slice = 0;                 // > 0: fixed slice length of the bucket kernel (KZGB200_MSM_SLICE), else msm_slice_len()
    int parse_fused = 0;            // tuning: decompression + subgroup check in one kernel (env KZGB200_PARSE_FUSED; measured slower)
    int defer_subgroup = 1;         // subgroup checks run beside the latency-bound tail on their own SMs (env KZGB200_DEFER_SUBGROUP)
    bool slab_tail = true;          // last host chunk copied slab-wise with the hash kernel waiting on arrival flags (env KZGB200_SLAB_TAIL=0: off)
    int sha_stages = 8;             // cp.async ring depth of the challenge hash (env KZGB200_SHA_STAGES: 4 or 8)
    int pageable_mode = 0;          // 0 = pinned staging ring, 1 = plain cudaMemcpyAsync (driver staging), 2 = cudaHostRegister in place
    bool subgroup_pending = false;
    int parse_first = 0;            // tuning: launch G1 parsing before the first hash launch (env KZGB200_PARSE_FIRST)
    int final_split = 1;            // batch check against [tau]G2: per-window Miller loops on the [256^w]-scaled G2 lines (env KZGB200_FINAL_SPLIT=0: Horner + one pairing)
    kzgb200::SplitTail* d_split = nullptr;
    cudaStream_t s_tail = nullptr;  // split tail: msm_sg_kernel, then msm_combine_kernel
    cudaEvent_t ev_sg = nullptr, ev_comb = nullptr;
    cudaStream_t s_aux = nullptr, s_copy = nullptr, s_d2h = nullptr, s_work[kzgb200::kWorkStreams] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_begin = nullptr, ev_parse = nullptr, ev_decomp = nullptr, ev_bucket = nullptr, ev_sha_all = nullptr, ev_leaf = nullptr;
    cudaEvent_t ev_h2d[kzgb200::kMaxChunks] = {nullptr}, ev_zy[kzgb200::kMaxChunks] = {nullptr}, ev_zyh[kzgb200::kMaxChunks] = {nullptr};
    uint32_t* d_chain_state = nullptr;
    uint8_t* h_flags = nullptr;     // pinned: 8 zeros, 8 ones (arrival flags of the slab-wise last chunk)
    uint8_t* d_scratch = nullptr;   // 512 bytes for small exports
    // pinned staging ring for pageable caller memory
    static constexpr int kStageBufs = 4;
    static constexpr size_t kStageBytes = 32u << 20;
    uint8_t* h_stage[kStageBufs] = {nullptr};
    cudaEvent_t ev_stage[kStageBufs] = {nullptr};
    int stage_next = 0;
    kzgb200::CopyPool* pool = nullptr;
    // optional per-phase timing (CUDA event pairs on the stream each phase runs on)
    bool profile = false;
    cudaEvent_t ev_s[8] = {nullptr}, ev_e[8] = {nullptr};
    bool ph_started[8] = {false};
    float phase_ms[8] = {0};
    kzgb200::CellCtx* cells = nullptr;   // EIP-7594 cell path (kzgb200_load_cell_setup)
    std::mutex lock;
    char err[256] = {0};
};

#define CK(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            snprintf(ctx->err, sizeof(ctx->err), "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return KZGB200_INTERNAL_ERROR;                                                         \
        }                                                                                          \
    } while (0)

namespace kzgb200 {

// Every entry point runs on its context's GPU and leaves the calling thread's current CUDA device as it found it (callers
// such as PyTorch cache the current device and would otherwise allocate on the wrong GPU afterwards).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int device) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; cudaSetDevice(device); }
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

template <class T>
inline cudaError_t regrow(T*& p, size_t count) {
    if (p) cudaFree(p);
    p = nullptr;
    return cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T));
}

// ---- phases (kzgb200.cu) --------------------------------------------------------------------------------------
int ensure_capacity(kzgb200_ctx* ctx, size_t n, bool need_blob_staging);
// phase 1 for blobs [0, n): G1 parsing, per-chunk challenge -> evaluation; the chunk plan is left in ctx->chunks.  With
// `transcript` the per-chunk transcript payloads ((z, y) pairs, or leaf digests in tree mode) are copied to pinned host memory
// behind the chunks (ctx->ev_zyh[c]); hc / hp = host copies of the commitments / proofs (nullptr: fetched from d_c / d_p).
int launch_phase1(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* h_blobs, const uint8_t* d_c, const uint8_t* d_p, size_t n,
                  bool transcript, bool defer_subgroup, const uint8_t* hc, const uint8_t* hp);
// host side of the transcript: consume the chunk payloads that have arrived (block = false: only those already complete)
int transcript_progress(kzgb200_ctx* ctx, bool block);
// after every chunk has been consumed: digest -> device -> r (Montgomery) on the main stream
int transcript_finish(kzgb200_ctx* ctx);
// upload a 32-byte transcript digest computed elsewhere (multi-GPU: the group leader) and derive r from it
int upload_r_digest(kzgb200_ctx* ctx, const uint8_t digest[32]);
// d_weights: per-entry scalars in place of r^(offset + i) (cell groups), nullptr = the powers of r
// split: the split tail follows (kzgb200_ctx::final_split): [s]G and the flags go to d_split beside the bucket phase (ev_sg), and
// msm_combine_kernel runs on s_tail beside the window Miller CTAs (ev_comb)
int launch_lincomb(kzgb200_ctx* ctx, size_t offset, Partial* d_out, bool wait_subgroup, uint32_t* d_flag = nullptr, uint32_t epoch = 0,
                   const Fr* d_weights = nullptr, bool split = false);
int read_result(kzgb200_ctx* ctx, int* ok);
int export_zy(kzgb200_ctx* ctx, size_t n, uint8_t* d_z, uint8_t* d_y);
void phase_begin(kzgb200_ctx* ctx, int ph, cudaStream_t st);
void phase_end(kzgb200_ctx* ctx, int ph, cudaStream_t st);
void collect_phase_times(kzgb200_ctx* ctx);
// transcript bytes of entries [lo, lo + cnt): C_i | z_i LE | y_i LE | pi_i from the three host arrays (indexed from 0)
void hash_entries(HostSha256* s, const uint8_t* c, const uint8_t* zy, const uint8_t* p, size_t lo, size_t cnt);
void hash_transcript_header(HostSha256* s, uint64_t n);

}  // namespace kzgb200
