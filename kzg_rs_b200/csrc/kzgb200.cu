// libkzgb200.so -- host runtime + C ABI (include/kzgb200.h) over the sm_100a kernels.
// Mirrors the orchestration of KzgProof::{verify_kzg_proof, verify_blob_kzg_proof,
// verify_blob_kzg_proof_batch, verify_kzg_proof_batch} (reference src/kzg_proof.rs:353-525): argument checks and phase
// ordering on the host, every field / curve / pairing operation and every per-blob hash in a kernel.  The one serial hash of
// the path -- the batch transcript of compute_r_powers (:291-348) -- is hashed by the host behind the kernels (host_sha256.cpp).
// No CPU fallback: CUDA failures surface as KZGB200_INTERNAL_ERROR.
#include <algorithm>
#include <chrono>
#include <new>
#include "runtime.cuh"

using namespace kzgb200;

// ---- pinned staging for pageable caller memory -------------------------------------------------------------------
namespace kzgb200 {
CopyPool::CopyPool(int nthreads) {
    for (int i = 0; i < nthreads; i++) threads.emplace_back([this] {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return stop || gen != seen; });
                if (stop) return;
                seen = gen;
            }
            work(seen);
        }
    });
}
CopyPool::~CopyPool() {
    { std::lock_guard<std::mutex> lk(m); stop = true; }
    cv.notify_all();
    for (auto& t : threads) t.join();
}
bool CopyPool::grab(size_t* off, size_t* len) {
    std::lock_guard<std::mutex> lk(m);
    if (next >= pieces) return false;
    *off = next++ * piece;
    *len = bytes - *off < piece ? bytes - *off : piece;
    return true;
}
void CopyPool::work(uint64_t) {
    size_t off, len, mine = 0;
    while (grab(&off, &len)) { memcpy(dst + off, src + off, len); mine++; }
    if (mine) {
        std::lock_guard<std::mutex> lk(m);
        done += mine;
        if (done == pieces) cv_done.notify_all();
    }
}
void CopyPool::copy(uint8_t* d, const uint8_t* s, size_t n) {
    if (!n) return;
    {
        std::lock_guard<std::mutex> lk(m);
        dst = d; src = s; bytes = n; pieces = (n + piece - 1) / piece; next = 0; done = 0; gen++;
    }
    cv.notify_all();
    work(0);
    std::unique_lock<std::mutex> lk(m);
    cv_done.wait(lk, [&] { return done == pieces; });
}

void phase_begin(kzgb200_ctx* ctx, int ph, cudaStream_t st) { if (ctx->profile && !ctx->ph_started[ph]) { cudaEventRecord(ctx->ev_s[ph], st); ctx->ph_started[ph] = true; } }
void phase_end(kzgb200_ctx* ctx, int ph, cudaStream_t st) { if (ctx->profile) cudaEventRecord(ctx->ev_e[ph], st); }
void collect_phase_times(kzgb200_ctx* ctx) {
    if (!ctx->profile) return;
    cudaDeviceSynchronize();
    for (int i = 0; i < 8; i++) { ctx->phase_ms[i] = 0; if (ctx->ph_started[i]) cudaEventElapsedTime(&ctx->phase_ms[i], ctx->ev_s[i], ctx->ev_e[i]); }
}

int ensure_capacity(kzgb200_ctx* ctx, size_t n, bool need_blob_staging) {
    if (n > ctx->cap) {
        size_t c = n;
        CK(regrow(ctx->d_c, c * 48)); CK(regrow(ctx->d_p, c * 48));
        CK(regrow(ctx->d_z_mont, c)); CK(regrow(ctx->d_zy, c)); CK(regrow(ctx->d_zpow, c * 13));
        CK(regrow(ctx->d_C, c)); CK(regrow(ctx->d_P, c));
        CK(regrow(ctx->d_status, c)); CK(regrow(ctx->d_ry, c));
        CK(regrow(ctx->d_digits, c * kDigitRows)); CK(regrow(ctx->d_order, c * kDigitRows));
        CK(regrow(ctx->d_zout, c * 32)); CK(regrow(ctx->d_yout, c * 32));
        CK(regrow(ctx->d_part, (size_t)kMsmRows * ((c + kMinSlice - 1) / kMinSlice) * 2));
        ctx->cap = c;
    }
    if (n > ctx->host_cap) {
        for (uint8_t** p : {&ctx->h_zy, &ctx->h_c, &ctx->h_p}) { if (*p) cudaFreeHost(*p); *p = nullptr; }
        CK(cudaMallocHost(&ctx->h_zy, n * 64)); CK(cudaMallocHost(&ctx->h_c, n * 48)); CK(cudaMallocHost(&ctx->h_p, n * 48));
        ctx->host_cap = n;
    }
    if (need_blob_staging && n > ctx->blob_cap) {
        CK(regrow(ctx->d_blobs, n * (size_t)kBytesPerBlob));
        ctx->blob_cap = n;
    }
    return KZGB200_OK;
}

// ---- transcript ---------------------------------------------------------------------------------------------------
// compute_r_powers (reference src/kzg_proof.rs:291-348): r = SHA-256("RCKZGBATCH___V1_" | u64be 4096 | u64be n | entries) mod q.
void hash_transcript_header(HostSha256* s, uint64_t n) {
    uint8_t hdr[32] = {'R', 'C', 'K', 'Z', 'G', 'B', 'A', 'T', 'C', 'H', '_', '_', '_', 'V', '1', '_', 0, 0, 0, 0, 0, 0, 0x10, 0x00};
    for (int i = 0; i < 8; i++) hdr[24 + i] = (uint8_t)(n >> (56 - 8 * i));
    host_sha256_init(s);
    host_sha256_update(s, hdr, 32);
}
void hash_entries(HostSha256* s, const uint8_t* c, const uint8_t* zy, const uint8_t* p, size_t lo, size_t cnt) {
    uint8_t buf[64 * 160];      // 64 entries = exactly 160 SHA-256 blocks
    for (size_t i = lo; i < lo + cnt;) {
        size_t m = lo + cnt - i < 64 ? lo + cnt - i : 64;
        for (size_t k = 0; k < m; k++, i++) {
            uint8_t* e = buf + 160 * k;
            memcpy(e, c + 48 * i, 48);            // to_compressed(C_i): the caller's bytes (canonical for every accepted encoding)
            memcpy(e + 48, zy + 64 * i, 64);      // z_i, y_i: 32 little-endian bytes each = the device's canonical limb image
            memcpy(e + 112, p + 48 * i, 48);
        }
        host_sha256_update(s, buf, 160 * m);
    }
}
static size_t tree_groups(size_t n) { return (n + kTreeGroup - 1) / kTreeGroup; }
// start the transcript of an n-entry batch; hc / hp: host commitments / proofs, or nullptr (fetched from the device arrays)
static int transcript_begin(kzgb200_ctx* ctx, size_t n, const uint8_t* d_c, const uint8_t* d_p, const uint8_t* hc, const uint8_t* hp) {
    ctx->tr_n = n; ctx->tr_done = 0; ctx->tr_next_chunk = 0; ctx->tr_enqueued = 0; ctx->tr_active = true;
    ctx->tr_c = hc; ctx->tr_p = hp;
    const int mode = ctx->transcript_mode;
    size_t words = 0;
    if (mode == KZGB200_TRANSCRIPT_TREE) words = n * 40 + tree_groups(n) * 8;
    else if (mode == KZGB200_TRANSCRIPT_EXACT_DEVICE) words = ((32 + n * 160 + 9 + 63) / 64) * 64;
    if (words > ctx->wk_cap) { CK(regrow(ctx->d_wk, words)); ctx->wk_cap = words; }
    if (mode == KZGB200_TRANSCRIPT_EXACT_DEVICE) return KZGB200_OK;
    hash_transcript_header(&ctx->tr_sha, n);
    if (mode == KZGB200_TRANSCRIPT_EXACT && !hc) {
        // device-resident inputs: the 96 bytes per blob the transcript hashes beside (z, y) come back once, at the start
        CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_begin, 0));
        CK(cudaMemcpyAsync(ctx->h_c, d_c, n * 48, cudaMemcpyDeviceToHost, ctx->s_d2h));
        CK(cudaMemcpyAsync(ctx->h_p, d_p, n * 48, cudaMemcpyDeviceToHost, ctx->s_d2h));
        ctx->tr_c = ctx->h_c; ctx->tr_p = ctx->h_p;
    }
    return KZGB200_OK;
}
// chunk c's (z, y) exist once ev_zy[c] has fired (the main stream already waits for it): queue what the transcript needs of it
static int transcript_enqueue_chunk(kzgb200_ctx* ctx, int c, const uint8_t* d_c, const uint8_t* d_p) {
    const size_t n = ctx->tr_n, lo = ctx->chunks[c].lo, cnt = ctx->chunks[c].cnt, end = lo + cnt;
    switch (ctx->transcript_mode) {
    case KZGB200_TRANSCRIPT_EXACT:
        CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_zy[c], 0));
        CK(cudaMemcpyAsync(ctx->h_zy + lo * 64, ctx->d_zy + lo, cnt * 64, cudaMemcpyDeviceToHost, ctx->s_d2h));
        CK(cudaEventRecord(ctx->ev_zyh[c], ctx->s_d2h));
        break;
    case KZGB200_TRANSCRIPT_TREE: {
        // chunk boundaries are multiples of kTreeGroup (plan_chunks), so the chunk owns whole leaves
        size_t g0 = lo / kTreeGroup, g1 = end >= n ? tree_groups(n) : end / kTreeGroup;
        uint32_t *words = ctx->d_wk, *digests = ctx->d_wk + n * 40;
        transcript_words_kernel<<<(unsigned)((cnt * 40 + 255) / 256), 256, 0, ctx->stream>>>(d_c, ctx->d_zy, d_p, lo, cnt, words);
        if (g1 > g0) transcript_tree_leaf_words_kernel<<<(unsigned)((g1 - g0 + 63) / 64), 64, 0, ctx->stream>>>(words, (uint64_t)n, digests, g0, g1 - g0);
        CK(cudaEventRecord(ctx->ev_leaf, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_leaf, 0));
        if (g1 > g0) CK(cudaMemcpyAsync(ctx->h_zy + g0 * 32, digests + g0 * 8, (g1 - g0) * 32, cudaMemcpyDeviceToHost, ctx->s_d2h));
        CK(cudaEventRecord(ctx->ev_zyh[c], ctx->s_d2h));
        break;
    }
    default: {   // KZGB200_TRANSCRIPT_EXACT_DEVICE: the serial chain on one warp of the GPU (round 1's path; ~2.4 us per blob)
        size_t nblk = (32 + n * 160 + 9 + 63) / 64;
        size_t ready = end >= n ? nblk : (32 + end * 160) / 64;
        if (ready > ctx->tr_done) {
            size_t k = ready - ctx->tr_done;
            transcript_schedule_kernel<<<(unsigned)((k + 127) / 128), 128, 0, ctx->stream>>>(d_c, ctx->d_zy, d_p, (uint64_t)n, ctx->d_wk, ctx->tr_done, k);
            transcript_chain_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_wk, (uint64_t)n, ctx->d_r, ctx->d_chain_state, ctx->tr_done, k);
            ctx->tr_done = ready;
        }
    }
    }
    CK(cudaGetLastError());
    ctx->tr_enqueued = c + 1;
    return KZGB200_OK;
}
int transcript_progress(kzgb200_ctx* ctx, bool block) {
    if (!ctx->tr_active) return KZGB200_OK;
    if (ctx->transcript_mode == KZGB200_TRANSCRIPT_EXACT_DEVICE) { ctx->tr_next_chunk = ctx->tr_enqueued; return KZGB200_OK; }
    while (ctx->tr_next_chunk < ctx->tr_enqueued) {      // only payloads queued by THIS call (the events are reused across calls)
        int c = ctx->tr_next_chunk;
        if (block) CK(cudaEventSynchronize(ctx->ev_zyh[c]));
        else {
            cudaError_t e = cudaEventQuery(ctx->ev_zyh[c]);
            if (e == cudaErrorNotReady) break;
            CK(e);
        }
        size_t lo = ctx->chunks[c].lo, cnt = ctx->chunks[c].cnt, end = lo + cnt;
        if (ctx->chunk_sink) ctx->chunk_sink(ctx->chunk_sink_arg, c);        // multi-GPU: the payload goes to the group's shared block
        else if (ctx->transcript_mode == KZGB200_TRANSCRIPT_EXACT) hash_entries(&ctx->tr_sha, ctx->tr_c, ctx->h_zy, ctx->tr_p, lo, cnt);
        else {
            size_t g0 = lo / kTreeGroup, g1 = end >= ctx->tr_n ? tree_groups(ctx->tr_n) : end / kTreeGroup;
            host_sha256_update(&ctx->tr_sha, ctx->h_zy + g0 * 32, (g1 - g0) * 32);
        }
        ctx->tr_next_chunk++;
    }
    return KZGB200_OK;
}
int upload_r_digest(kzgb200_ctx* ctx, const uint8_t digest[32]) {
    memcpy(ctx->h_digest, digest, 32);
    CK(cudaMemcpyAsync(ctx->d_digest, ctx->h_digest, 32, cudaMemcpyHostToDevice, ctx->stream));
    r_from_digest_kernel<<<1, 1, 0, ctx->stream>>>(ctx->d_digest, ctx->d_r);
    CK(cudaGetLastError());
    return KZGB200_OK;
}
int transcript_finish(kzgb200_ctx* ctx) {
    if (ctx->transcript_mode != KZGB200_TRANSCRIPT_EXACT_DEVICE) {
        uint8_t digest[32];
        host_sha256_final(&ctx->tr_sha, digest);
        int rc = upload_r_digest(ctx, digest);
        if (rc) return rc;
    }
    phase_end(ctx, kPhTranscript, ctx->stream);
    ctx->tr_active = false;
    return KZGB200_OK;
}

// ---- phase 1 --------------------------------------------------------------------------------------------------------
// Streams: `stream` (main: transcript, MSM, pairing, result), `s_aux` (G1 decompression beside the hashing; the subgroup checks
// beside the tail, see launch_lincomb), `s_work[k]` (challenge / evaluation), `s_copy` (host->device blob chunks), `s_d2h`
// (transcript payloads back to the host).
// Chunk plans.  Host blobs: equal chunks of >= 128 MiB so that hashing / evaluation of chunk c overlap the PCIe copy of chunk
// c+1.  Resident blobs: ONE challenge launch (the per-blob SHA-256 chain is latency-bound: 16384 chains are 512 warps on 592 SM
// sub-partitions, splitting it would idle half the machine), then the evaluation in a few chunks that shrink towards the end,
// so that the host hashes the transcript behind the evaluation and only the last, small chunk's hash is exposed.
static int plan_chunks(kzgb200_ctx* ctx, size_t n, bool host_blobs, bool transcript) {
    int k = 0;
    if (host_blobs) {
        size_t chunk = (n + kMaxChunks - 1) / kMaxChunks;
        if (chunk < kMinChunk) chunk = kMinChunk;
        chunk = (chunk + kTreeGroup - 1) / kTreeGroup * kTreeGroup;
        for (size_t lo = 0; lo < n; lo += chunk) ctx->chunks[k++] = {lo, n - lo < chunk ? n - lo : chunk};
    } else if (!transcript || n < 2048 || ctx->transcript_mode == KZGB200_TRANSCRIPT_TREE) {
        ctx->chunks[k++] = {0, n};
    } else if (ctx->transcript_mode == KZGB200_TRANSCRIPT_EXACT_DEVICE) {
        size_t chunk = ((n + 7) / 8 + kTreeGroup - 1) / kTreeGroup * kTreeGroup;
        for (size_t lo = 0; lo < n; lo += chunk) ctx->chunks[k++] = {lo, n - lo < chunk ? n - lo : chunk};
    } else {
        size_t lo = 0, quarter = n / 4 / kTreeGroup * kTreeGroup;
        while (lo < n) {
            size_t rem = n - lo, take = k < 3 ? quarter : rem / 2 / kTreeGroup * kTreeGroup;
            if (take < 256) take = 256;
            if (rem - (take < rem ? take : rem) < 256 || k == kMaxChunks - 1) take = rem;
            ctx->chunks[k++] = {lo, take};
            lo += take;
        }
    }
    ctx->nchunks = k;
    return k;
}
static bool host_pointer_is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
// host->device copy of a blob range on s_copy.  Pinned (or registered) caller memory goes straight to the DMA engine; pageable
// memory goes through a ring of pinned staging buffers filled by a few memcpy threads (a cudaMemcpyAsync from pageable memory is
// staged by the driver on ONE thread and blocks the caller); the host hashes transcript chunks that have arrived in between.
static int h2d_blobs(kzgb200_ctx* ctx, uint8_t* d_dst, const uint8_t* h_src, size_t bytes, bool direct) {
    if (direct) { CK(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->s_copy)); return KZGB200_OK; }
    if (!ctx->pool) {
        unsigned hw = std::thread::hardware_concurrency();
        int t = hw >= 16 ? 7 : (hw >= 8 ? 3 : 1);
        if (const char* v = getenv("KZGB200_COPY_THREADS")) t = atoi(v) > 0 ? atoi(v) - 1 : 0;
        ctx->pool = new CopyPool(t);
        for (int b = 0; b < kzgb200_ctx::kStageBufs; b++) {
            CK(cudaMallocHost(&ctx->h_stage[b], kzgb200_ctx::kStageBytes));
            CK(cudaEventCreateWithFlags(&ctx->ev_stage[b], cudaEventDisableTiming));
        }
    }
    for (size_t off = 0; off < bytes; off += kzgb200_ctx::kStageBytes) {
        size_t len = bytes - off < kzgb200_ctx::kStageBytes ? bytes - off : kzgb200_ctx::kStageBytes;
        int b = ctx->stage_next;
        ctx->stage_next = (b + 1) % kzgb200_ctx::kStageBufs;
        CK(cudaEventSynchronize(ctx->ev_stage[b]));          // the DMA that last read this buffer is done
        ctx->pool->copy(ctx->h_stage[b], h_src + off, len);
        CK(cudaMemcpyAsync(d_dst + off, ctx->h_stage[b], len, cudaMemcpyHostToDevice, ctx->s_copy));
        CK(cudaEventRecord(ctx->ev_stage[b], ctx->s_copy));
        int rc = transcript_progress(ctx, false);
        if (rc) return rc;
    }
    return KZGB200_OK;
}
int launch_phase1(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* h_blobs, const uint8_t* d_c, const uint8_t* d_p, size_t n,
                  bool transcript, bool defer_subgroup, const uint8_t* hc, const uint8_t* hp) {
    for (int i = 0; i < 8; i++) ctx->ph_started[i] = false;
    const int nchunks = plan_chunks(ctx, n, h_blobs != nullptr, transcript);
    ctx->tr_next_chunk = 0; ctx->tr_enqueued = 0; ctx->tr_active = false;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));    // a previous call's deferred subgroup checks still write status
    CK(cudaMemsetAsync(ctx->d_status, 0, n * sizeof(uint32_t), ctx->stream));
    CK(cudaEventRecord(ctx->ev_begin, ctx->stream));
    if (transcript) { int rc = transcript_begin(ctx, n, d_c, d_p, hc, hp); if (rc) return rc; }
    bool direct = true, registered = false;
    if (h_blobs) {
        CK(cudaStreamWaitEvent(ctx->s_copy, ctx->ev_begin, 0));
        if (!host_pointer_is_pinned(h_blobs)) {
            direct = ctx->pageable_mode != 0;
            if (ctx->pageable_mode == 2) registered = cudaHostRegister(const_cast<uint8_t*>(h_blobs), n * (size_t)kBytesPerBlob, cudaHostRegisterDefault) == cudaSuccess;
            if (ctx->pageable_mode == 2 && !registered) cudaGetLastError();
        }
    }
    auto launch_parse = [&]() -> int {
        CK(cudaStreamWaitEvent(ctx->s_aux, ctx->ev_begin, 0));
        phase_begin(ctx, kPhParse, ctx->s_aux);
        g1_decompress_kernel<<<(2 * (int)n + 127) / 128, 128, 0, ctx->s_aux>>>(d_c, d_p, (int)n, ctx->d_C, ctx->d_P, ctx->d_status, ctx->parse_fused != 0);
        CK(cudaEventRecord(ctx->ev_decomp, ctx->s_aux));
        if (defer_subgroup && !ctx->parse_fused) { ctx->subgroup_pending = true; phase_end(ctx, kPhParse, ctx->s_aux); return KZGB200_OK; }   // checks: launched by launch_lincomb
        if (!ctx->parse_fused) g1_subgroup_kernel<<<(2 * (int)n + 255) / 256, 256, 0, ctx->s_aux>>>(ctx->d_C, ctx->d_P, (int)n, ctx->d_status);
        phase_end(ctx, kPhParse, ctx->s_aux);
        CK(cudaEventRecord(ctx->ev_parse, ctx->s_aux));
        return KZGB200_OK;
    };
    if (ctx->parse_first) { int rc = launch_parse(); if (rc) return rc; }
    if (!h_blobs) {
        // resident: one challenge launch over the whole batch, evaluation per chunk on two alternating streams
        cudaStream_t s0 = ctx->s_work[0];
        CK(cudaStreamWaitEvent(s0, ctx->ev_begin, 0));
        phase_begin(ctx, kPhChallenge, s0);
        launch_challenge(ctx->sha_stages, s0, d_blobs, d_c, (int)n, ctx->d_z_mont, ctx->d_zy, ctx->d_zpow);
        phase_end(ctx, kPhChallenge, s0);
        CK(cudaEventRecord(ctx->ev_sha_all, s0));
        if (!ctx->parse_first) { int rc = launch_parse(); if (rc) return rc; }   // G1 decompression queued behind the hash launch
        for (int c = 0; c < nchunks; c++) {
            size_t lo = ctx->chunks[c].lo, cnt = ctx->chunks[c].cnt;
            cudaStream_t sw = ctx->s_work[c & 1];
            if (c & 1) CK(cudaStreamWaitEvent(sw, ctx->ev_sha_all, 0));
            phase_begin(ctx, kPhEval, sw);
            eval_kernel<<<(int)cnt, kEvalThreads, 0, sw>>>(d_blobs + lo * kBytesPerBlob, (int)cnt, ctx->d_zpow + lo * 13, ctx->tables, ctx->d_zy + lo, ctx->d_status + lo);
            if (c == nchunks - 1) phase_end(ctx, kPhEval, sw);
            CK(cudaEventRecord(ctx->ev_zy[c], sw));
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_zy[c], 0));
            if (transcript && c == nchunks - 1) phase_begin(ctx, kPhTranscript, ctx->stream);
            if (transcript) { int rc = transcript_enqueue_chunk(ctx, c, d_c, d_p); if (rc) return rc; }
        }
    } else {
        for (int c = 0; c < nchunks; c++) {
            size_t lo = ctx->chunks[c].lo, cnt = ctx->chunks[c].cnt;
            cudaStream_t sw = ctx->s_work[c % kWorkStreams];
            int rc = KZGB200_OK;
            // The last chunk of a multi-chunk copy arrives slab-wise (bytes [16 KiB q, 16 KiB (q+1)) of all its blobs, q = 0..7) and
            // its hash kernel starts behind slab 0: the per-blob chain (2.7 ms whatever the blob count) then ends ~0.5 ms after the
            // last byte instead of a whole chain after it.
            const bool slabs = direct && ctx->slab_tail && nchunks > 1 && c == nchunks - 1 && cnt >= 64;
            uint8_t* slab_flags = ctx->d_scratch + 480;
            if (slabs) {
                const size_t sb = kBytesPerBlob / kChallengeSlabs;
                CK(cudaMemcpyAsync(slab_flags, ctx->h_flags, kChallengeSlabs, cudaMemcpyHostToDevice, ctx->s_copy));     // zeros; by the copy engine, in order with the slabs
                for (int q = 0; q < kChallengeSlabs; q++) {
                    CK(cudaMemcpy2DAsync(const_cast<uint8_t*>(d_blobs) + lo * kBytesPerBlob + q * sb, kBytesPerBlob, h_blobs + lo * kBytesPerBlob + q * sb,
                                         kBytesPerBlob, sb, cnt, cudaMemcpyHostToDevice, ctx->s_copy));
                    CK(cudaMemcpyAsync(slab_flags + q, ctx->h_flags + 8, 1, cudaMemcpyHostToDevice, ctx->s_copy));        // a one
                    if (q == 0) CK(cudaEventRecord(ctx->ev_h2d[c], ctx->s_copy));
                }
            } else {
                rc = h2d_blobs(ctx, const_cast<uint8_t*>(d_blobs) + lo * kBytesPerBlob, h_blobs + lo * kBytesPerBlob, cnt * (size_t)kBytesPerBlob, direct);
                if (rc) return rc;
                CK(cudaEventRecord(ctx->ev_h2d[c], ctx->s_copy));
            }
            CK(cudaStreamWaitEvent(sw, ctx->ev_h2d[c], 0));
            CK(cudaStreamWaitEvent(sw, ctx->ev_begin, 0));
            phase_begin(ctx, kPhChallenge, sw);
            launch_challenge(ctx->sha_stages, sw, d_blobs + lo * kBytesPerBlob, d_c + lo * 48, (int)cnt, ctx->d_z_mont + lo,
                             ctx->d_zy + lo, ctx->d_zpow + lo * 13, slabs ? slab_flags : nullptr);
            phase_end(ctx, kPhChallenge, sw);
            phase_begin(ctx, kPhEval, sw);
            eval_kernel<<<(int)cnt, kEvalThreads, 0, sw>>>(d_blobs + lo * kBytesPerBlob, (int)cnt, ctx->d_zpow + lo * 13, ctx->tables, ctx->d_zy + lo, ctx->d_status + lo);
            phase_end(ctx, kPhEval, sw);
            CK(cudaEventRecord(ctx->ev_zy[c], sw));
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_zy[c], 0));
            if (c == 0 && !ctx->parse_first) { rc = launch_parse(); if (rc) return rc; }   // G1 parsing queued behind the first hash launch
            if (transcript && c == nchunks - 1) phase_begin(ctx, kPhTranscript, ctx->stream);
            if (transcript) { rc = transcript_enqueue_chunk(ctx, c, d_c, d_p); if (rc) return rc; }
        }
    }
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_decomp, 0));   // the points exist; the subgroup verdicts (ev_parse) are awaited
    CK(cudaGetLastError());                                     // only where the error flags are consumed
    if (registered) {   // in-place pinning: the copies must be done before the pages are released
        CK(cudaStreamSynchronize(ctx->s_copy));
        cudaHostUnregister(const_cast<uint8_t*>(h_blobs));
    }
    ctx->cur_c = d_c; ctx->cur_p = d_p; ctx->cur_n = n;
    return KZGB200_OK;
}
// Entries per thread of the bucket kernel.  Its kMsmRows * ceil(n / slice) threads run as 128-thread CTAs, two per SM (216
// registers), and every thread is one chain of mixed additions: the slice length is chosen so that the CTAs fill whole waves of
// the machine, about 16 entries each (16384 blobs on 148 SMs: 14 entries, 878 CTAs = 2.97 waves; 16 entries were 2.6 waves).
static int msm_slice_len(const kzgb200_ctx* ctx, int n) {
    if (ctx->msm_slice > 0) return ctx->msm_slice < kMinSlice ? kMinSlice : ctx->msm_slice;      // KZGB200_MSM_SLICE (experiments)
    const double wave = (double)ctx->msm_occ * ctx->num_sms * 128, work = (double)kMsmRows * n;
    int waves = (int)(work / 16.0 / wave + 0.5);
    if (waves < 1) waves = 1;
    int slice = (int)((work + waves * wave - 1) / (waves * wave));
    return slice < kMinSlice ? kMinSlice : slice;
}
// K6: digits, counting sort, buckets, window sums, Horner -> partial (optionally stored into a peer's exchange buffer + flag)
int launch_lincomb(kzgb200_ctx* ctx, size_t offset, Partial* d_out, bool wait_subgroup, uint32_t* d_flag, uint32_t epoch, const Fr* d_weights,
                   bool split) {
    int n = (int)ctx->cur_n;
    phase_begin(ctx, kPhLincomb, ctx->stream);
    msm_scalars_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_z_mont, ctx->d_zy, ctx->d_r, (uint64_t)offset, n, ctx->d_digits, ctx->d_ry, d_weights);
    if (split) {        // s = sum r_i y_i, [s]G and the flags on one CTA beside the bucket phase
        CK(cudaEventRecord(ctx->ev_sg, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->s_tail, ctx->ev_sg, 0));
        if (wait_subgroup) CK(cudaStreamWaitEvent(ctx->s_tail, ctx->ev_parse, 0));
        msm_sg_kernel<<<1, kCombHelpers, 0, ctx->s_tail>>>(ctx->d_ry, ctx->d_status, n, ctx->tables, ctx->d_split);
        CK(cudaEventRecord(ctx->ev_sg, ctx->s_tail));
    }
    msm_sort_kernel<<<kDigitRows, 256, 0, ctx->stream>>>(ctx->d_digits, n, ctx->d_order, ctx->d_start);
    {
        const int slice = msm_slice_len(ctx, n);
        launch_msm_bucket(ctx->msm_occ, n, slice, ctx->stream, ctx->d_C, ctx->d_P, ctx->d_order, ctx->d_start, ctx->d_halfsum, ctx->d_part);
        launch_msm_bucket_join(ctx->msm_join, n, slice, ctx->stream, ctx->d_start, ctx->d_halfsum, ctx->d_part, ctx->d_buckets);
    }
    phase_end(ctx, kPhLincomb, ctx->stream);
    phase_begin(ctx, kPhReduce, ctx->stream);
    // window sums: 48 CTAs of one thread per bucket, still with the whole machine (the deferred checks start behind them)
    msm_window_kernel<<<kMsmSets * kWindows, kWinLanes, kWinSmemBytes, ctx->stream>>>(ctx->d_buckets, ctx->d_windows);
    if (ctx->subgroup_pending) {
        // Deferred subgroup checks: from here on the batch is latency-bound (Horner combination, one pairing: single
        // CTAs), so the checks get the rest of the machine.  They run one CTA per SM on all but kTailSms SMs -- each CTA
        // asks for kTailHogSmem of shared memory it never touches, and the tail kernels ask for kTailPadSmem, so that the two
        // cannot share an SM: the tail keeps SMs of its own and is not slowed down (sharing SMs cost more than the deferral saved).
        CK(cudaEventRecord(ctx->ev_bucket, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->s_aux, ctx->ev_bucket, 0));
        if (ctx->profile) cudaEventRecord(ctx->ev_s[7], ctx->s_aux);
        g1_subgroup_kernel<<<ctx->num_sms - (split ? kTailSmsSplit : kTailSms), 256, kTailHogSmem, ctx->s_aux>>>(ctx->d_C, ctx->d_P, n, ctx->d_status);
        if (ctx->profile) { cudaEventRecord(ctx->ev_e[7], ctx->s_aux); ctx->ph_started[7] = true; }
        CK(cudaEventRecord(ctx->ev_parse, ctx->s_aux));
        ctx->subgroup_pending = false;
    }
    if (split) {        // the combined partial (kzgb200_last_partial) beside the window Miller CTAs: off the critical path
        phase_end(ctx, kPhReduce, ctx->stream);
        CK(cudaEventRecord(ctx->ev_comb, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->s_tail, ctx->ev_comb, 0));
        msm_combine_kernel<<<1, kCombineThreads, kCombineSmemBytes, ctx->s_tail>>>(ctx->d_windows, ctx->d_ry, ctx->d_status, n, ctx->tables, d_out, d_flag, epoch);
        CK(cudaEventRecord(ctx->ev_comb, ctx->s_tail));
        CK(cudaGetLastError());
        return KZGB200_OK;
    }
    if (wait_subgroup) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));    // combine ORs the per-blob error flags
    msm_combine_kernel<<<1, kCombineThreads, kCombineSmemBytes, ctx->stream>>>(ctx->d_windows, ctx->d_ry, ctx->d_status, n, ctx->tables, d_out, d_flag, epoch);
    phase_end(ctx, kPhReduce, ctx->stream);
    CK(cudaGetLastError());
    return KZGB200_OK;
}
// K6 + K7 of a single-GPU batch against [tau]G2 (batch verdict in d_result, f^(3(p^12-1)/r) in d_split->gt): the split tail
// (window_miller_kernel) or, with final_split = 0, the Horner combination + one pairing check.  phase_final: open the final phase
// (closed by the caller); ticks: kzgb200_debug_final_ticks stamps.
int launch_batch_check(kzgb200_ctx* ctx, bool wait_subgroup, bool phase_final, bool ticks) {
    int rc;
    const bool split = ctx->final_split != 0;
    if ((rc = launch_lincomb(ctx, 0, ctx->d_partial, wait_subgroup, nullptr, 0, nullptr, split))) return rc;
    if (phase_final) phase_begin(ctx, kPhFinal, ctx->stream);
    if (!split) {
        launch_batch_final(ctx->stream, ctx->d_partial, 1, ctx->tables, ctx->d_result, ctx->d_scratch, ticks, nullptr, ctx->d_split->gt);
    } else {
        long long* tk = ticks ? reinterpret_cast<long long*>(ctx->d_scratch + 128) : nullptr;
        if (tk) CK(cudaMemsetAsync(tk, 0, 14 * sizeof(long long), ctx->stream));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_sg, 0));
        window_prelude_kernel<<<kWindows, kFinalThreads, sizeof(FinalSmem), ctx->stream>>>(ctx->d_windows, ctx->d_split);
        window_miller_kernel<<<kWindows, kPairThreads, sizeof(PairSmem), ctx->stream>>>(ctx->tables, ctx->d_split, tk);
        split_final_kernel<<<1, kPairThreads, sizeof(PairSmem), ctx->stream>>>(ctx->d_split, ctx->d_result, ctx->d_split->gt, tk);
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_comb, 0));     // the combined partial is in place when the call returns
    }
    CK(cudaGetLastError());
    return KZGB200_OK;
}
int read_result(kzgb200_ctx* ctx, int* ok) {
    CK(cudaMemcpyAsync(ctx->h_result, ctx->d_result, 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_result[0] == kBadArgs || ctx->h_result[2]) return KZGB200_BAD_ARGS;
    *ok = ctx->h_result[0] == kTrue ? 1 : 0;
    return KZGB200_OK;
}
int export_zy(kzgb200_ctx* ctx, size_t n, uint8_t* d_z, uint8_t* d_y) {
    if (!d_z && !d_y) return KZGB200_OK;
    export_scalars_kernel<<<((int)n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_zy, (int)n, d_z, d_y);
    CK(cudaGetLastError());
    return KZGB200_OK;
}
}  // namespace kzgb200

extern "C" int kzgb200_create(kzgb200_ctx** out, int device, const uint8_t* g2_points, size_t g2_points_len) {
    if (!out) return KZGB200_BAD_ARGS;
    *out = nullptr;
    if (!g2_points || g2_points_len != 192) return KZGB200_INVALID_SETUP;
    kzgb200_ctx* ctx = new (std::nothrow) kzgb200_ctx();
    if (!ctx) return KZGB200_INTERNAL_ERROR;
    ctx->device = device;
    DeviceGuard dev;
    auto fail = [&](int rc) { fprintf(stderr, "kzgb200_create: %s\n", ctx->err); kzgb200_destroy(ctx); return rc; };
    int rc = [&]() -> int {
        CK(cudaSetDevice(device));      // (restored by the guard below)
        CK(cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device));
        int prio_lo = 0, prio_hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CK(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi));
        // the hash chains are the long pole of phase 1: their CTAs go first, G1 parsing fills the rest of the machine
        { const char* v = getenv("KZGB200_PARSE_PRIO"); CK(cudaStreamCreateWithPriority(&ctx->s_aux, cudaStreamNonBlocking, v && atoi(v) ? prio_hi : prio_lo)); }
        if (const char* v = getenv("KZGB200_PARSE_FIRST")) ctx->parse_first = atoi(v);
        if (const char* v = getenv("KZGB200_PARSE_FUSED")) ctx->parse_fused = atoi(v);
        if (const char* v = getenv("KZGB200_DEFER_SUBGROUP")) ctx->defer_subgroup = atoi(v);
        if (const char* v = getenv("KZGB200_SHA_STAGES")) ctx->sha_stages = atoi(v);
        if (const char* v = getenv("KZGB200_SLAB_TAIL")) ctx->slab_tail = atoi(v) != 0;
        if (const char* v = getenv("KZGB200_PAGEABLE")) ctx->pageable_mode = !strcmp(v, "direct") ? 1 : (!strcmp(v, "register") ? 2 : 0);
        if (const char* v = getenv("KZGB200_MSM_SLICE")) ctx->msm_slice = atoi(v);
        if (const char* v = getenv("KZGB200_MSM_JOIN")) ctx->msm_join = atoi(v);
        if (const char* v = getenv("KZGB200_MSM_OCC")) { int o = atoi(v); if (o >= 2 && o <= 4) ctx->msm_occ = o; }
        if (const char* v = getenv("KZGB200_FINAL_SPLIT")) ctx->final_split = atoi(v) != 0;
        if (const char* v = getenv("KZGB200_TRANSCRIPT")) ctx->transcript_mode = !strcmp(v, "tree") ? KZGB200_TRANSCRIPT_TREE : (!strcmp(v, "device") ? KZGB200_TRANSCRIPT_EXACT_DEVICE : KZGB200_TRANSCRIPT_EXACT);
        CK(cudaFuncSetAttribute(g1_subgroup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailHogSmem));
        CK(cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithPriority(&ctx->s_d2h, cudaStreamNonBlocking, prio_hi));
        for (auto& w : ctx->s_work) CK(cudaStreamCreateWithPriority(&w, cudaStreamNonBlocking, prio_hi));
        CK(cudaStreamCreateWithPriority(&ctx->s_tail, cudaStreamNonBlocking, prio_hi));
        for (cudaEvent_t* e : {&ctx->ev_begin, &ctx->ev_parse, &ctx->ev_decomp, &ctx->ev_bucket, &ctx->ev_sha_all, &ctx->ev_leaf, &ctx->ev_sg, &ctx->ev_comb})
            CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        for (auto& e : ctx->ev_h2d) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : ctx->ev_zy) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : ctx->ev_zyh) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaMalloc(&ctx->d_chain_state, 32));
        CK(cudaMalloc(&ctx->d_scratch, 512));
        CK(cudaMalloc(&ctx->d_digest, 32));
        CK(cudaFuncSetAttribute(batch_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FinalSmem)));
        CK(cudaFuncSetAttribute(single_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FinalSmem)));
        CK(cudaFuncSetAttribute(pairing_check_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PairSmem)));
        CK(cudaFuncSetAttribute(window_prelude_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FinalSmem)));
        CK(cudaFuncSetAttribute(window_miller_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PairSmem)));
        CK(cudaFuncSetAttribute(split_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PairSmem)));
        CK(cudaFuncSetAttribute(msm_combine_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCombineSmemBytes));
        CK(cudaFuncSetAttribute(many_pairing_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kManySmemBytes));
        CK(cudaFuncSetAttribute(many_pairing_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kManySmemBytes));
        CK(cudaMalloc(&ctx->tables, sizeof(DeviceTables)));
        CK(cudaMalloc(&ctx->d_r, sizeof(Fr)));
        CK(cudaMalloc(&ctx->d_partial, sizeof(Partial)));
        CK(cudaMalloc(&ctx->d_split, sizeof(SplitTail)));
        CK(cudaMemsetAsync(ctx->d_split, 0, sizeof(SplitTail), ctx->stream));
        CK(cudaMalloc(&ctx->d_result, 16));
        CK(cudaMalloc(&ctx->d_start, kDigitRows * (kBuckets + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&ctx->d_buckets, kMsmSets * kWindows * kBuckets * sizeof(G1)));
        CK(cudaMalloc(&ctx->d_halfsum, kMsmRows * kBuckets * sizeof(G1)));
        CK(cudaMalloc(&ctx->d_windows, kMsmSets * kWindows * sizeof(G1)));
        CK(cudaMallocHost(&ctx->h_result, 16));
        CK(cudaMallocHost(&ctx->h_flags, 16));
        memset(ctx->h_flags, 0, 8); memset(ctx->h_flags + 8, 1, 8);
        CK(cudaMallocHost(&ctx->h_digest, 32));
        CK(cudaMallocHost(&ctx->h_partial, sizeof(Partial)));
        uint8_t* d_g2 = nullptr;
        CK(cudaMalloc(&d_g2, 192));
        CK(cudaMemcpyAsync(d_g2, g2_points, 192, cudaMemcpyHostToDevice, ctx->stream));
        setup_tables_kernel<<<(8192 + 4096) / 128, 128, 0, ctx->stream>>>(ctx->tables, d_g2);
        setup_lines29_kernel<<<(2 * kMillerSteps * 6 + 127) / 128, 128, 0, ctx->stream>>>(ctx->tables);
        LineCoeffs* d_lines_tmp = nullptr;
        CK(cudaMalloc(&d_lines_tmp, 2 * (kWindows - 1) * kMillerSteps * sizeof(LineCoeffs)));
        setup_lines29w_kernel<<<1, 32, 0, ctx->stream>>>(ctx->tables, d_g2, d_lines_tmp);
        CK(cudaGetLastError());
        uint32_t ok = 0;
        CK(cudaMemcpyAsync(&ok, &ctx->tables->setup_ok, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        cudaFree(d_g2);
        cudaFree(d_lines_tmp);
        return ok ? KZGB200_OK : KZGB200_INVALID_SETUP;
    }();
    if (rc != KZGB200_OK) return fail(rc);
    *out = ctx;
    return KZGB200_OK;
}

static void cell_destroy(kzgb200_ctx* ctx);
extern "C" void kzgb200_destroy(kzgb200_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard dev(ctx->device);
    cudaDeviceSynchronize();
    cell_destroy(ctx);
    delete ctx->pool;
    for (cudaStream_t st : {ctx->s_tail, ctx->s_aux, ctx->s_copy, ctx->s_d2h, ctx->s_work[0], ctx->s_work[1], ctx->s_work[2], ctx->s_work[3]}) if (st) cudaStreamDestroy(st);
    for (cudaEvent_t e : {ctx->ev_begin, ctx->ev_parse, ctx->ev_decomp, ctx->ev_bucket, ctx->ev_sha_all, ctx->ev_leaf, ctx->ev_sg, ctx->ev_comb}) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_h2d) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_zy) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_zyh) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_s) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_e) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_stage) if (e) cudaEventDestroy(e);
    void* ptrs[] = {ctx->tables, ctx->d_blobs, ctx->d_c, ctx->d_p, ctx->d_z_mont, ctx->d_zy, ctx->d_C, ctx->d_P, ctx->d_status,
                    ctx->d_ry, ctx->d_r, ctx->d_partial, ctx->d_result, ctx->d_zout, ctx->d_yout, ctx->d_many, ctx->d_wk,
                    ctx->d_digits, ctx->d_order, ctx->d_start, ctx->d_buckets, ctx->d_halfsum, ctx->d_part, ctx->d_windows, ctx->d_lag_table, ctx->d_scalars, ctx->d_lag_part, ctx->d_zpow,
                    ctx->d_chain_state, ctx->d_scratch, ctx->d_digest, ctx->d_split};
    for (void* p : ptrs) if (p) cudaFree(p);
    void* hptrs[] = {ctx->h_flags, ctx->h_result, ctx->h_digest, ctx->h_partial, ctx->h_zy, ctx->h_c, ctx->h_p, ctx->h_stage[0], ctx->h_stage[1], ctx->h_stage[2], ctx->h_stage[3]};
    for (void* p : hptrs) if (p) cudaFreeHost(p);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* kzgb200_last_error(const kzgb200_ctx* ctx) { return ctx ? ctx->err : "null context"; }

// per tuple of the many-tuple path: 3 affine points, a status word, 160 input bytes, a verdict byte (rounded up)
constexpr size_t kManyBytesPerTuple = 3 * sizeof(G1Affine) + 4 + 160 + 4;
// the pairing checks of m parsed tuples: kManyGroups per CTA in lockstep (kManyCtasPerSm persistent CTAs per SM), then the rare identity inputs
// (lines_b: the second G2 point's line table, nullptr = [tau]G2)
static int launch_many_pairings(kzgb200_ctx* ctx, const G1Affine* X, const G1Affine* P, const uint32_t* status, size_t m, uint8_t* dv,
                                const LineCoeffs* lines_b = nullptr) {
    size_t nbatch = (m + kManyGroups - 1) / kManyGroups;
    const size_t slots = (size_t)ctx->num_sms * kManyCtasPerSm;
    unsigned grid = (unsigned)(nbatch < slots ? nbatch : slots);
    many_pairing_kernel<<<grid, kManyThreads, kManySmemBytes, ctx->stream>>>(X, P, status, m, ctx->tables, lines_b, dv);
    size_t nw = (m + kManyWarps - 1) / kManyWarps;
    many_pairing_warp_kernel<<<(unsigned)(nw < (size_t)ctx->num_sms ? nw : (size_t)ctx->num_sms), 32 * kManyWarps, kManySmemBytes, ctx->stream>>>(X, P, m, ctx->tables, lines_b, dv);
    CK(cudaGetLastError());
    return KZGB200_OK;
}
// whole batch on one GPU, n >= 1; blobs either resident (h_blobs == nullptr) or streamed from the host (then hc / hp = the
// caller's host commitments / proofs, which the transcript reads in place)
static int batch_locked(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* h_blobs, const uint8_t* d_c, const uint8_t* d_p, size_t n, int* ok,
                        uint8_t* d_z_out, uint8_t* d_y_out, const uint8_t* hc, const uint8_t* hp) {
    const bool defer = n >= 2 && ctx->defer_subgroup;
    int rc = launch_phase1(ctx, d_blobs, h_blobs, d_c, d_p, n, n >= 2, defer, hc, hp);
    if (rc) return rc;
    if ((rc = export_zy(ctx, n, d_z_out, d_y_out))) return rc;
    if (n == 1) {   // single path (reference src/kzg_proof.rs:482-489)
        phase_begin(ctx, kPhFinal, ctx->stream);
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
        FinalPts* fp = reinterpret_cast<FinalPts*>(ctx->d_scratch + 256);
        single_final_kernel<<<1, kFinalThreads, sizeof(FinalSmem), ctx->stream>>>(ctx->d_C, ctx->d_P, ctx->d_zy, ctx->d_status, ctx->tables, ctx->d_result, fp);
        pairing_check_kernel<<<1, kPairThreads, sizeof(PairSmem), ctx->stream>>>(fp, ctx->tables, nullptr, ctx->d_result, nullptr, nullptr);
    } else {
        if ((rc = transcript_progress(ctx, true))) return rc;     // the host hashes the transcript behind the evaluation chunks
        if ((rc = transcript_finish(ctx))) return rc;
        if ((rc = launch_batch_check(ctx, !defer, true, true))) return rc;   // deferred: the flags are merged by status_or below
    }
    phase_end(ctx, kPhFinal, ctx->stream);
    // the deferred subgroup checks may still be running beside the pairing: their flags are merged last
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    status_or_kernel<<<1, 256, 0, ctx->stream>>>(ctx->d_status, (int)n, ctx->d_result + 2);
    CK(cudaGetLastError());
    rc = read_result(ctx, ok);
    collect_phase_times(ctx);
    return rc;
}

extern "C" int kzgb200_verify_blob_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                                          const uint8_t* d_proofs, size_t n, int* ok, uint8_t* d_z_out, uint8_t* d_y_out) {
    if (!ctx || !ok || n == 0 || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, n, false);
    if (rc) return rc;
    return batch_locked(ctx, d_blobs, nullptr, d_commitments, d_proofs, n, ok, d_z_out, d_y_out, nullptr, nullptr);
}

extern "C" int kzgb200_verify_blob_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n_blobs, const uint8_t* commitments,
                                                   size_t n_commitments, const uint8_t* proofs, size_t n_proofs, int* ok,
                                                   uint8_t* z_out, uint8_t* y_out) {
    if (!ctx || !ok) return KZGB200_BAD_ARGS;
    if (n_blobs == 0) { *ok = 1; return KZGB200_OK; }                 // reference src/kzg_proof.rs:478-480
    if (n_blobs == 1) {                                                // :482-489, before the length checks
        if (n_commitments < 1 || n_proofs < 1) return KZGB200_BAD_ARGS;   // the reference would index out of bounds (panic)
    } else {
        if (n_blobs != n_commitments) return KZGB200_INVALID_LENGTH;   // :491-495
        if (n_blobs != n_proofs) return KZGB200_INVALID_LENGTH;        // :497-501
    }
    if (n_blobs > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    size_t n = n_blobs;
    int rc = ensure_capacity(ctx, n, true);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_c, commitments, n * 48, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_p, proofs, n * 48, cudaMemcpyHostToDevice, ctx->stream));
    rc = batch_locked(ctx, ctx->d_blobs, blobs, ctx->d_c, ctx->d_p, n, ok, z_out ? ctx->d_zout : nullptr, y_out ? ctx->d_yout : nullptr, commitments, proofs);
    if (rc == KZGB200_OK) {
        if (z_out) CK(cudaMemcpyAsync(z_out, ctx->d_zout, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
        if (y_out) CK(cudaMemcpyAsync(y_out, ctx->d_yout, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return rc;
}

extern "C" int kzgb200_verify_blob_kzg_proof(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* commitment48, const uint8_t* proof48,
                                             int* ok, uint8_t* z_out, uint8_t* y_out) {
    return kzgb200_verify_blob_kzg_proof_batch(ctx, blob, 1, commitment48, 1, proof48, 1, ok, z_out, y_out);
}

// per-blob verdicts (SURVEY 8f-4): the batch check first -- one MSM + one pairing for all blobs; only when it fails (or some input
// did not parse) every blob is checked on its own from the already-parsed points and the already-computed z_i, y_i.
extern "C" int kzgb200_verify_blob_kzg_proof_batch_each(kzgb200_ctx* ctx, const uint8_t* blobs, const uint8_t* commitments, const uint8_t* proofs,
                                                        size_t n, uint8_t* verdicts, uint8_t* z_out, uint8_t* y_out) {
    if (!ctx || (n && (!blobs || !commitments || !proofs || !verdicts)) || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (n == 0) return KZGB200_OK;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, n, true);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_c, commitments, n * 48, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_p, proofs, n * 48, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = launch_phase1(ctx, ctx->d_blobs, blobs, ctx->d_c, ctx->d_p, n, n >= 2, false, commitments, proofs))) return rc;
    if ((rc = export_zy(ctx, n, z_out ? ctx->d_zout : nullptr, y_out ? ctx->d_yout : nullptr))) return rc;
    int ok = 0;
    bool all_true = false;
    if (n >= 2) {
        if ((rc = transcript_progress(ctx, true))) return rc;
        if ((rc = transcript_finish(ctx))) return rc;
        if ((rc = launch_batch_check(ctx, true, false, false))) return rc;
        status_or_kernel<<<1, 256, 0, ctx->stream>>>(ctx->d_status, (int)n, ctx->d_result + 2);
        CK(cudaGetLastError());
        rc = read_result(ctx, &ok);
        if (rc != KZGB200_OK && rc != KZGB200_BAD_ARGS) return rc;
        all_true = rc == KZGB200_OK && ok == 1;
    }
    if (all_true) memset(verdicts, 1, n);
    else {
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
        if (n > ctx->many_cap) { CK(regrow(ctx->d_many, n * kManyBytesPerTuple)); ctx->many_cap = n; }
        G1Affine* X = reinterpret_cast<G1Affine*>(ctx->d_many);
        uint8_t* dv = ctx->d_many + n * sizeof(G1Affine);
        many_lhs_zy_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_zy, ctx->d_C, ctx->d_P, n, ctx->tables, X, ctx->d_status);
        if ((rc = launch_many_pairings(ctx, X, ctx->d_P, ctx->d_status, n, dv))) return rc;
        CK(cudaMemcpyAsync(verdicts, dv, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (z_out) CK(cudaMemcpyAsync(z_out, ctx->d_zout, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    if (y_out) CK(cudaMemcpyAsync(y_out, ctx->d_yout, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}

// KzgProof::verify_kzg_proof_batch on already-parsed inputs (reference src/kzg_proof.rs:399-444; SURVEY 8f-4).  Like the
// reference it neither validates the points nor checks the subgroup (its arguments are typed G1Affine / Scalar values).
extern "C" int kzgb200_verify_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* commitments104, const uint8_t* zs32, const uint8_t* ys32,
                                              const uint8_t* proofs104, size_t n, int* ok) {
    if (!ctx || !ok || (n && (!commitments104 || !zs32 || !ys32 || !proofs104)) || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (n == 0) { *ok = 1; return KZGB200_OK; }     // empty sums: both pairing arguments are the identity
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, n, false);
    if (rc) return rc;
    if (n > ctx->many_cap) { CK(regrow(ctx->d_many, n * kManyBytesPerTuple)); ctx->many_cap = n; }
    uint8_t *dc = ctx->d_many, *dp = dc + n * 104, *dz = dp + n * 104, *dy = dz + n * 32;
    for (int i = 0; i < 8; i++) ctx->ph_started[i] = false;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    CK(cudaMemcpyAsync(dc, commitments104, n * 104, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dp, proofs104, n * 104, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dz, zs32, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dy, ys32, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_status, 0, n * sizeof(uint32_t), ctx->stream));
    import_parsed_kernel<<<(unsigned)((2 * n + 127) / 128), 128, 0, ctx->stream>>>(dc, dp, dz, dy, (int)n, ctx->d_C, ctx->d_P, ctx->d_c, ctx->d_p, ctx->d_z_mont, ctx->d_zy);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev_begin, ctx->stream));
    ctx->chunks[0] = {0, n}; ctx->nchunks = 1;
    ctx->cur_c = ctx->d_c; ctx->cur_p = ctx->d_p; ctx->cur_n = n; ctx->subgroup_pending = false;
    if ((rc = transcript_begin(ctx, n, ctx->d_c, ctx->d_p, nullptr, nullptr))) return rc;
    CK(cudaEventRecord(ctx->ev_zy[0], ctx->stream));
    if ((rc = transcript_enqueue_chunk(ctx, 0, ctx->d_c, ctx->d_p))) return rc;
    if ((rc = transcript_progress(ctx, true))) return rc;
    if ((rc = transcript_finish(ctx))) return rc;
    if ((rc = launch_batch_check(ctx, false, false, false))) return rc;
    CK(cudaMemsetAsync(ctx->d_result + 2, 0, 4, ctx->stream));
    CK(cudaGetLastError());
    return read_result(ctx, ok);
}

// compute_challenge (reference src/kzg_proof.rs:46-72) for one blob: z as 32 big-endian bytes
extern "C" int kzgb200_compute_challenge(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* commitment48, uint8_t* z_out32) {
    if (!ctx || !blob || !commitment48 || !z_out32) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, 1, true);
    if (rc) return rc;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    CK(cudaMemcpyAsync(ctx->d_blobs, blob, kBytesPerBlob, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_c, commitment48, 48, cudaMemcpyHostToDevice, ctx->stream));
    launch_challenge(ctx->sha_stages, ctx->stream, ctx->d_blobs, ctx->d_c, 1, ctx->d_z_mont, ctx->d_zy, ctx->d_zpow);
    export_scalars_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_zy, 1, ctx->d_zout, nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(z_out32, ctx->d_zout, 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
// evaluate_polynomial_in_evaluation_form (reference src/kzg_proof.rs:94-133) of one blob at a caller-supplied z, including
// z in the evaluation domain (:109-111).  Non-canonical blob elements (Blob::as_polynomial) or z -> KZGB200_BAD_ARGS.
extern "C" int kzgb200_evaluate_polynomial_in_evaluation_form(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* z32, uint8_t* y_out32) {
    if (!ctx || !blob || !z32 || !y_out32) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, 1, true);
    if (rc) return rc;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    CK(cudaMemcpyAsync(ctx->d_blobs, blob, kBytesPerBlob, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_zout, z32, 32, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_status, 0, 4, ctx->stream));
    z_setup_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_zout, 1, ctx->d_z_mont, ctx->d_zy, ctx->d_zpow, ctx->d_status);
    eval_kernel<<<1, kEvalThreads, 0, ctx->stream>>>(ctx->d_blobs, 1, ctx->d_zpow, ctx->tables, ctx->d_zy, ctx->d_status);
    export_scalars_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_zy, 1, nullptr, ctx->d_yout);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(y_out32, ctx->d_yout, 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_result, ctx->d_status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return ctx->h_result[0] ? KZGB200_BAD_ARGS : KZGB200_OK;
}

// m independent verify_kzg_proof tuples (BASELINE config 5): parse kernels (one thread per point), X_i = C_i - [y_i]G + [z_i]pi_i (one
// thread per tuple), then one warp per pairing check on the cooperative engine (k_many.cu); chunks of 2^20 tuples.
extern "C" int kzgb200_verify_kzg_proof_many(kzgb200_ctx* ctx, const uint8_t* commitments, const uint8_t* zs, const uint8_t* ys,
                                             const uint8_t* proofs, size_t m, uint8_t* verdicts) {
    if (!ctx || (m && (!commitments || !zs || !ys || !proofs || !verdicts))) return KZGB200_BAD_ARGS;
    if (m == 0) return KZGB200_OK;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    const size_t kChunk = (size_t)1 << 20, c = m < kChunk ? m : kChunk;
    if (c > ctx->many_cap) { CK(regrow(ctx->d_many, c * kManyBytesPerTuple)); ctx->many_cap = c; }
    G1Affine *dC = reinterpret_cast<G1Affine*>(ctx->d_many), *dP = dC + c, *dX = dP + c;
    uint32_t* dst = reinterpret_cast<uint32_t*>(dX + c);
    uint8_t *dc = reinterpret_cast<uint8_t*>(dst + c), *dp = dc + c * 48, *dz = dp + c * 48, *dy = dz + c * 32, *dv = dy + c * 32;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    for (int i = 0; i < 8; i++) ctx->ph_started[i] = false;
    for (size_t lo = 0; lo < m; lo += c) {
        size_t cnt = m - lo < c ? m - lo : c;
        CK(cudaMemcpyAsync(dc, commitments + lo * 48, cnt * 48, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dz, zs + lo * 32, cnt * 32, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dy, ys + lo * 32, cnt * 32, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dp, proofs + lo * 48, cnt * 48, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemsetAsync(dst, 0, cnt * 4, ctx->stream));
        phase_begin(ctx, kPhParse, ctx->stream);
        g1_decompress_kernel<<<(unsigned)((2 * cnt + 127) / 128), 128, 0, ctx->stream>>>(dc, dp, (int)cnt, dC, dP, dst, false);
        g1_subgroup_kernel<<<(unsigned)((2 * cnt + 255) / 256), 256, 0, ctx->stream>>>(dC, dP, (int)cnt, dst);
        phase_end(ctx, kPhParse, ctx->stream);
        phase_begin(ctx, kPhLincomb, ctx->stream);
        many_lhs_kernel<<<(unsigned)((cnt + 127) / 128), 128, 0, ctx->stream>>>(dz, dy, dC, dP, cnt, ctx->tables, dX, dst);
        phase_end(ctx, kPhLincomb, ctx->stream);
        phase_begin(ctx, kPhFinal, ctx->stream);
        { int rc = launch_many_pairings(ctx, dX, dP, dst, cnt, dv); if (rc) return rc; }
        phase_end(ctx, kPhFinal, ctx->stream);
        CK(cudaMemcpyAsync(verdicts + lo, dv, cnt, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    collect_phase_times(ctx);
    return KZGB200_OK;
}

extern "C" int kzgb200_verify_kzg_proof(kzgb200_ctx* ctx, const uint8_t* commitment48, const uint8_t* z32, const uint8_t* y32,
                                        const uint8_t* proof48, int* ok) {
    if (!ok) return KZGB200_BAD_ARGS;
    uint8_t v = 0;
    int rc = kzgb200_verify_kzg_proof_many(ctx, commitment48, z32, y32, proof48, 1, &v);
    if (rc) return rc;
    if (v == kBadArgs) return KZGB200_BAD_ARGS;
    *ok = v == kTrue;
    return KZGB200_OK;
}

// test hook: the host SHA-256 of the batch transcript (both code paths); returns 1 if SHA-NI was used
extern "C" int kzgb200_host_sha256(const uint8_t* msg, size_t len, uint8_t* out32, int force_portable) {
    host_sha256_force_portable(force_portable);
    HostSha256 s;
    host_sha256_init(&s);
    host_sha256_update(&s, msg, len);
    host_sha256_final(&s, out32);
    int used = host_sha256_uses_shani();
    host_sha256_force_portable(0);
    return used;
}

// ---- harness: synthetic workload with valid commitments / proofs (device outputs) ---------------------------
extern "C" int kzgb200_harness_generate(kzgb200_ctx* ctx, uint64_t seed, size_t n, int degree, const uint8_t* tau_powers48,
                                        uint8_t* d_blobs, uint8_t* d_commitments, uint8_t* d_proofs) {
    if (!ctx || n == 0 || degree < 2 || degree > kHarnessMaxDegree || !tau_powers48) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, n, false);
    if (rc) return rc;
    uint8_t* d_bytes = nullptr; G1Affine* d_M = nullptr; uint32_t* d_bad = nullptr; uint32_t bad = 0;
    CK(cudaMalloc(&d_bytes, degree * 48)); CK(cudaMalloc(&d_M, degree * sizeof(G1Affine))); CK(cudaMalloc(&d_bad, 4));
    CK(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
    CK(cudaMemcpyAsync(d_bytes, tau_powers48, degree * 48, cudaMemcpyHostToDevice, ctx->stream));
    harness_parse_points_kernel<<<1, 32, 0, ctx->stream>>>(d_bytes, degree, d_M, d_bad);
    int ni = (int)n;
    harness_blob_kernel<<<ni, 128, 0, ctx->stream>>>(seed, ni, degree, ctx->tables, d_blobs);
    harness_commit_kernel<<<(ni + 63) / 64, 64, 0, ctx->stream>>>(seed, ni, degree, d_M, nullptr, d_commitments, 0);
    launch_challenge(ctx->sha_stages, ctx->stream, d_blobs, d_commitments, ni, ctx->d_z_mont, ctx->d_zy, ctx->d_zpow);
    harness_commit_kernel<<<(ni + 63) / 64, 64, 0, ctx->stream>>>(seed, ni, degree, d_M, ctx->d_z_mont, d_proofs, 1);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_bytes); cudaFree(d_M); cudaFree(d_bad);
    return bad ? KZGB200_BAD_ARGS : KZGB200_OK;
}
extern "C" int kzgb200_set_transcript_mode(kzgb200_ctx* ctx, int mode) {
    if (!ctx || (mode != KZGB200_TRANSCRIPT_EXACT && mode != KZGB200_TRANSCRIPT_TREE && mode != KZGB200_TRANSCRIPT_EXACT_DEVICE)) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    ctx->transcript_mode = mode;
    return KZGB200_OK;
}
// the canonical big-endian r of the last batch (exact mode: bit-identical to compute_r_powers' r)
extern "C" int kzgb200_last_r(kzgb200_ctx* ctx, uint8_t* r_out32) {
    if (!ctx || !r_out32) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    // scratch: the first ZY slot of the (idle) z/y export buffers
    ZY* tmp = reinterpret_cast<ZY*>(ctx->d_scratch);
    uint8_t* d_out = ctx->d_scratch + sizeof(ZY);
    r_to_raw_kernel<<<1, 1, 0, ctx->stream>>>(ctx->d_r, tmp);
    export_scalars_kernel<<<1, 1, 0, ctx->stream>>>(tmp, 1, d_out, nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(r_out32, d_out, 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
// raw per-rank partial of the last single-GPU batch (Partial struct: Jacobian A, B in Montgomery limbs, sum r_i y_i, flags)
extern "C" int kzgb200_last_partial(kzgb200_ctx* ctx, uint8_t* out352) {
    if (!ctx || !out352) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    CK(cudaMemcpyAsync(out352, ctx->d_partial, sizeof(Partial), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
// per-phase device times of the last single-GPU batch call: parse, challenge, eval, transcript, lincomb, reduce, final
extern "C" int kzgb200_set_profiling(kzgb200_ctx* ctx, int on) {
    if (!ctx) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    if (on) { for (auto& e : ctx->ev_s) if (!e) CK(cudaEventCreate(&e)); for (auto& e : ctx->ev_e) if (!e) CK(cudaEventCreate(&e)); }
    ctx->profile = on != 0;
    return KZGB200_OK;
}
extern "C" int kzgb200_get_phase_ms(kzgb200_ctx* ctx, float* out7) {
    if (!ctx || !out7) return KZGB200_BAD_ARGS;
    for (int i = 0; i < 8; i++) out7[i] = ctx->phase_ms[i];
    return KZGB200_OK;
}
// ---- commit / prove (SURVEY 8f-1) ------------------------------------------------------------------------------
extern "C" int kzgb200_load_g1_lagrange(kzgb200_ctx* ctx, const uint8_t* g1_lagrange, size_t n_points) {
    if (!ctx || !g1_lagrange || n_points != (size_t)kFieldElementsPerBlob) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    if (ctx->d_lag_table) return KZGB200_OK;
    uint8_t* d_bytes = nullptr; G1Affine* d_L = nullptr; uint32_t* d_bad = nullptr; uint32_t bad = 0;
    CK(cudaMalloc(&d_bytes, n_points * 48)); CK(cudaMalloc(&d_L, n_points * sizeof(G1Affine))); CK(cudaMalloc(&d_bad, 4));
    CK(cudaMalloc(&ctx->d_lag_table, (size_t)kFieldElementsPerBlob * kLagWindows * kLagEntries * sizeof(G1)));
    CK(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
    CK(cudaMemcpyAsync(d_bytes, g1_lagrange, n_points * 48, cudaMemcpyHostToDevice, ctx->stream));
    lag_parse_kernel<<<(kFieldElementsPerBlob + 127) / 128, 128, 0, ctx->stream>>>(d_bytes, d_L, d_bad);
    lag_table_kernel<<<(kFieldElementsPerBlob * kLagWindows + 127) / 128, 128, 0, ctx->stream>>>(d_L, ctx->d_lag_table);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_bytes); cudaFree(d_L); cudaFree(d_bad);
    if (bad) { cudaFree(ctx->d_lag_table); ctx->d_lag_table = nullptr; return KZGB200_INVALID_SETUP; }
    return KZGB200_OK;
}
// Slices per blob of the commitment MSM for a chunk of cnt blobs: as many as keep the grid within one wave of one CTA per SM
// (lag_msm_slice_kernel uses 180 registers: two 256-thread CTAs do not fit one SM).  One blob then spreads over every SM; from
// num_sms / 2 + 1 blobs on it is one CTA per blob, the batch throughput form.
static int lag_slices(const kzgb200_ctx* ctx, int cnt) {
    int s = ctx->num_sms / cnt;
    return s < 1 ? 1 : (s > kLagMaxSlices ? kLagMaxSlices : s);
}
enum ProveMode { kProveCommit, kProveBlob, kProveAtZ };
// Shared driver of every commit / prove entry point, in chunks of 1024 blobs:
//   kProveCommit  commitments of the blobs (d_in unused);
//   kProveBlob    proofs at the Fiat-Shamir challenge of (blob, commitment), d_in = the commitments (n x 48); check_commitments also
//                 decompresses them and checks the subgroup (the spec's bytes_to_kzg_commitment);
//   kProveAtZ     proofs at caller-given points, d_in = z (n x 32 big-endian); d_y_out (nullable) receives y = p(z) (n x 32).
// BAD_ARGS when any blob element, z or checked commitment is invalid; the outputs are then undefined.
static int commit_or_prove(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_in, size_t n, uint8_t* d_out, ProveMode mode,
                           bool check_commitments = false, uint8_t* d_y_out = nullptr) {
    if (!ctx->d_lag_table) return KZGB200_INVALID_SETUP;
    const size_t kChunk = 1024;
    int rc = ensure_capacity(ctx, n < kChunk ? n : kChunk, false);
    if (rc) return rc;
    if (!ctx->d_scalars) CK(cudaMalloc(&ctx->d_scalars, kChunk * (size_t)kFieldElementsPerBlob * sizeof(Fr)));
    if (!ctx->d_lag_part) CK(cudaMalloc(&ctx->d_lag_part, (kChunk > (size_t)ctx->num_sms ? kChunk : (size_t)ctx->num_sms) * sizeof(G1)));
    uint32_t any_bad = 0;
    for (size_t lo = 0; lo < n; lo += kChunk) {
        int cnt = (int)(n - lo < kChunk ? n - lo : kChunk);
        const uint8_t* blobs = d_blobs + lo * kBytesPerBlob;
        CK(cudaMemsetAsync(ctx->d_status, 0, cnt * sizeof(uint32_t), ctx->stream));
        if (mode == kProveCommit) {
            blob_scalars_kernel<<<(unsigned)(((size_t)cnt * kFieldElementsPerBlob + 127) / 128), 128, 0, ctx->stream>>>(blobs, cnt, ctx->d_scalars, ctx->d_status);
        } else {
            if (mode == kProveBlob) {
                const uint8_t* cs = d_in + lo * 48;
                launch_challenge(ctx->sha_stages, ctx->stream, blobs, cs, cnt, ctx->d_z_mont, ctx->d_zy, ctx->d_zpow);
                if (check_commitments)   // each commitment as both point arguments: one kernel, flags in d_status
                    g1_decompress_kernel<<<(2 * cnt + 127) / 128, 128, 0, ctx->stream>>>(cs, cs, cnt, ctx->d_C, ctx->d_P, ctx->d_status, true);
            } else {
                z_setup_kernel<<<(cnt + 127) / 128, 128, 0, ctx->stream>>>(d_in + lo * 32, cnt, ctx->d_z_mont, ctx->d_zy, ctx->d_zpow, ctx->d_status);
            }
            eval_kernel<<<cnt, kEvalThreads, 0, ctx->stream>>>(blobs, cnt, ctx->d_zpow, ctx->tables, ctx->d_zy, ctx->d_status);
            quotient_kernel<<<cnt, kEvalThreads, 0, ctx->stream>>>(blobs, cnt, ctx->d_z_mont, ctx->d_zy, ctx->tables, ctx->d_scalars);
            if (d_y_out) export_scalars_kernel<<<(cnt + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_zy, cnt, nullptr, d_y_out + lo * 32);
        }
        const int slices = lag_slices(ctx, cnt);
        lag_msm_slice_kernel<<<dim3(slices, cnt), kLagMsmThreads, 0, ctx->stream>>>(ctx->d_scalars, cnt, slices, ctx->d_lag_table, ctx->d_lag_part,
                                                                                     d_out + lo * 48);
        if (slices > 1) lag_msm_finish_kernel<<<cnt, kLagFinishThreads, 0, ctx->stream>>>(ctx->d_lag_part, cnt, slices, d_out + lo * 48);
        status_or_kernel<<<1, 256, 0, ctx->stream>>>(ctx->d_status, cnt, ctx->d_result);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ctx->h_result, ctx->d_result, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        any_bad |= ctx->h_result[0];
    }
    return any_bad ? KZGB200_BAD_ARGS : KZGB200_OK;
}
extern "C" int kzgb200_blob_to_kzg_commitment_batch(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_commitments_out) {
    if (!ctx || !d_blobs || !d_commitments_out || n == 0) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    return commit_or_prove(ctx, d_blobs, nullptr, n, d_commitments_out, kProveCommit);
}
extern "C" int kzgb200_compute_blob_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments, size_t n,
                                                    uint8_t* d_proofs_out) {
    if (!ctx || !d_blobs || !d_commitments || !d_proofs_out || n == 0) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    return commit_or_prove(ctx, d_blobs, d_commitments, n, d_proofs_out, kProveBlob);
}
extern "C" int kzgb200_compute_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_zs, size_t n,
                                                      uint8_t* d_proofs_out, uint8_t* d_ys_out) {
    if (!ctx || (n && (!d_blobs || !d_zs || !d_proofs_out || !d_ys_out)) || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (!ctx->d_lag_table) return KZGB200_INVALID_SETUP;
    if (n == 0) return KZGB200_OK;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    return commit_or_prove(ctx, d_blobs, d_zs, n, d_proofs_out, kProveAtZ, false, d_ys_out);
}
// one host blob through commit_or_prove on the context's staging buffers: the blob in d_blobs, the 48-byte commitment or the
// 32-byte z in d_c, the point out of d_p and y out of d_yout
static int prove_host(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* in, size_t in_bytes, ProveMode mode, uint8_t* out48, uint8_t* y_out32) {
    if (!ctx->d_lag_table) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, 1, true);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_blobs, blob, kBytesPerBlob, cudaMemcpyHostToDevice, ctx->stream));
    if (in) CK(cudaMemcpyAsync(ctx->d_c, in, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = commit_or_prove(ctx, ctx->d_blobs, ctx->d_c, 1, ctx->d_p, mode, mode == kProveBlob, y_out32 ? ctx->d_yout : nullptr))) return rc;
    CK(cudaMemcpyAsync(out48, ctx->d_p, 48, cudaMemcpyDeviceToHost, ctx->stream));
    if (y_out32) CK(cudaMemcpyAsync(y_out32, ctx->d_yout, 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
extern "C" int kzgb200_blob_to_kzg_commitment(kzgb200_ctx* ctx, const uint8_t* blob, uint8_t* commitment_out48) {
    if (!ctx || !blob || !commitment_out48) return KZGB200_BAD_ARGS;
    return prove_host(ctx, blob, nullptr, 0, kProveCommit, commitment_out48, nullptr);
}
extern "C" int kzgb200_compute_kzg_proof(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* z32, uint8_t* proof_out48, uint8_t* y_out32) {
    if (!ctx || !blob || !z32 || !proof_out48 || !y_out32) return KZGB200_BAD_ARGS;
    return prove_host(ctx, blob, z32, 32, kProveAtZ, proof_out48, y_out32);
}
extern "C" int kzgb200_compute_blob_kzg_proof(kzgb200_ctx* ctx, const uint8_t* blob, const uint8_t* commitment48, uint8_t* proof_out48) {
    if (!ctx || !blob || !commitment48 || !proof_out48) return KZGB200_BAD_ARGS;
    return prove_host(ctx, blob, commitment48, 48, kProveBlob, proof_out48, nullptr);
}
// f^(3(p^12-1)/r) of the last single-GPU batch check (either tail): 12 canonical Fp values, 48 little-endian bytes each, in the
// order c0.c0.c0, c0.c0.c1, c0.c1.c0, ... of the engine's F slot
extern "C" int kzgb200_debug_last_gt(kzgb200_ctx* ctx, uint8_t* out576) {
    if (!ctx || !out576) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    CK(cudaMemcpyAsync(out576, ctx->d_split->gt, 12 * sizeof(Fp), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
// the shifted line tables of the split tail (DeviceTables::lines29w: [2][15][68][6] values of 16 little-endian 32-bit words)
extern "C" int kzgb200_debug_lines29w(kzgb200_ctx* ctx, uint8_t* out, size_t len) {
    if (!ctx || !out || len != sizeof(DeviceTables::lines29w)) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    CK(cudaMemcpyAsync(out, ctx->tables->lines29w, len, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
// clock64() stamps of the last single-GPU batch check: start, prelude end, Miller loop end, easy part end, hard part end, done.  With the
// split tail the first three are rebased onto the product CTA's clock from the longest window CTA, and the product of the 16
// Miller values counts into the easy part.
extern "C" int kzgb200_debug_final_ticks(kzgb200_ctx* ctx, long long* out14) {
    if (!ctx || !out14) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    CK(cudaMemcpy(out14, ctx->d_scratch + 128, 112, cudaMemcpyDeviceToHost));
    return KZGB200_OK;
}
extern "C" int kzgb200_set_slab_tail(kzgb200_ctx* ctx, int on) {
    if (!ctx) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    ctx->slab_tail = on != 0;
    return KZGB200_OK;
}
extern "C" int kzgb200_debug_engine_selftest(kzgb200_ctx* ctx, uint32_t seed, int rounds, uint32_t* mismatches32, int* n_programs) {
    if (!ctx || !mismatches32 || !n_programs || rounds < 1) return KZGB200_BAD_ARGS;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    f29::F29* d_ref = nullptr; uint32_t* d_mis = nullptr;
    CK(cudaMalloc(&d_ref, sizeof(f29::F29) * vliw29::kTotalRegs));
    CK(cudaMalloc(&d_mis, 32 * sizeof(uint32_t)));
    CK(cudaMemsetAsync(d_mis, 0, 32 * sizeof(uint32_t), ctx->stream));
    CK(cudaFuncSetAttribute(engine_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PairSmem)));
    engine_selftest_kernel<<<1, kPairThreads, sizeof(PairSmem), ctx->stream>>>(seed, rounds, d_ref, d_mis);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(mismatches32, d_mis, 32 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_ref); cudaFree(d_mis);
    *n_programs = vliw29::kNumPrograms;
    static_assert(vliw29::kNumPrograms <= 32, "mismatch array");
    return KZGB200_OK;
}
// the stream every call of this context is issued on (cudaStream_t), for event timing by the caller
extern "C" void* kzgb200_stream(kzgb200_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

extern "C" void* kzgb200_alloc_pinned(size_t bytes) {
    void* p = nullptr;
    return cudaMallocHost(&p, bytes) == cudaSuccess ? p : nullptr;
}
extern "C" void kzgb200_free_pinned(void* p) { if (p) cudaFreeHost(p); }

// ---- EIP-7594 cells (k_cells.cu; consensus-specs Fulu polynomial-commitments-sampling.md) ---------------------------------
static void proof_destroy(CellCtx* c) {
    void* d[] = {c->ptables, c->d_mono, c->d_fk_tab, c->d_pcoef, c->d_fkU, c->d_A, c->d_V, c->d_pcommit, c->d_rblobs, c->d_rin, c->d_pout, c->d_plans, c->d_z,
                 c->d_mstage, c->d_mcells, c->d_mproofs};
    for (void* p : d) if (p) cudaFree(p);
    c->ptables = nullptr; c->d_mono = c->d_fk_tab = nullptr; c->d_pcoef = c->d_fkU = c->d_A = c->d_z = nullptr; c->d_V = c->d_pcommit = nullptr;
    c->d_rblobs = c->d_rin = c->d_pout = nullptr; c->d_plans = nullptr; c->proof_cap = 0;
    c->d_mstage = c->d_mcells = c->d_mproofs = nullptr; c->mstage_cells = c->mout_cap = 0;
}
static void cell_destroy(kzgb200_ctx* ctx) {
    CellCtx* c = ctx->cells;
    if (!c) return;
    void* d[] = {c->tables, c->d_cells, c->d_p, c->d_uc, c->d_meta, c->d_ustatus, c->d_U, c->d_rk, c->d_agg, c->d_coeffs, c->d_part, c->d_ext,
                 c->d_goff, c->d_gbad, c->d_fmeta, c->d_rg, c->d_gv, c->d_terms, c->d_AB, c->d_gX, c->d_rcoef};
    for (void* p : d) if (p) cudaFree(p);
    void* h[] = {c->h_meta, c->h_uc, c->h_c, c->h_cells, c->h_p, c->h_idx};
    for (void* p : h) if (p) cudaFreeHost(p);
    for (cudaEvent_t e : {c->ev_r, c->ev_rli}) if (e) cudaEventDestroy(e);
    proof_destroy(c);
    delete c;
    ctx->cells = nullptr;
}

extern "C" int kzgb200_load_cell_setup(kzgb200_ctx* ctx, const uint8_t* g1_monomial48, size_t n_points, const uint8_t* g2_tau64_96) {
    if (!ctx) return KZGB200_BAD_ARGS;
    if (!g1_monomial48 || n_points < (size_t)kFieldElementsPerCell || !g2_tau64_96) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    if (ctx->cells) return KZGB200_OK;
    CellCtx* c = new (std::nothrow) CellCtx();
    if (!c) return KZGB200_INTERNAL_ERROR;
    ctx->cells = c;
    uint8_t* d_bytes = nullptr;
    uint32_t ok = 0;
    int rc = [&]() -> int {
        CK(cudaMalloc(&c->tables, sizeof(CellTables)));
        CK(cudaMalloc(&d_bytes, kFieldElementsPerCell * 48 + 96));
        CK(cudaMemcpyAsync(d_bytes, g1_monomial48, kFieldElementsPerCell * 48, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(d_bytes + kFieldElementsPerCell * 48, g2_tau64_96, 96, cudaMemcpyHostToDevice, ctx->stream));
        cell_setup_kernel<<<4096 / 128, 128, 0, ctx->stream>>>(c->tables, d_bytes + kFieldElementsPerCell * 48);
        cell_setup_points_kernel<<<kFieldElementsPerCell * 4 / 64, 64, 0, ctx->stream>>>(c->tables, d_bytes);
        cell_setup_lines29_kernel<<<(kMillerSteps * 6 + 127) / 128, 128, 0, ctx->stream>>>(c->tables);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&ok, &c->tables->ok, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaFuncSetAttribute(compute_cells_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCellNttSmemBytes));
        CK(cudaMalloc(&c->d_agg, (size_t)kCellsPerExtBlob * kCellAggSlices * kFieldElementsPerCell * sizeof(Fr)));
        CK(cudaMalloc(&c->d_coeffs, (size_t)kCellsPerExtBlob * kFieldElementsPerCell * sizeof(Fr)));
        CK(cudaMalloc(&c->d_part, 2 * sizeof(Partial)));
        CK(cudaEventCreateWithFlags(&c->ev_r, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&c->ev_rli, cudaEventDisableTiming));
        return KZGB200_OK;
    }();
    if (d_bytes) cudaFree(d_bytes);
    if (rc == KZGB200_OK && !ok) rc = KZGB200_INVALID_SETUP;
    if (rc != KZGB200_OK) cell_destroy(ctx);
    return rc;
}

static int cell_capacity(kzgb200_ctx* ctx, size_t n, bool host_inputs, bool device_inputs) {
    CellCtx* c = ctx->cells;
    int rc = ensure_capacity(ctx, n, false);
    if (rc) return rc;
    if (n > c->cap) {
        CK(regrow(c->d_meta, 3 * n + kCellsPerExtBlob + 1)); CK(regrow(c->d_ustatus, n)); CK(regrow(c->d_uc, n * 48));
        CK(regrow(c->d_U, n)); CK(regrow(c->d_rk, n));
        if (c->d_cells) { cudaFree(c->d_cells); c->d_cells = nullptr; }
        if (c->d_p) { cudaFree(c->d_p); c->d_p = nullptr; }
        c->cap = n;
        c->slot.assign(1, 0);
    }
    if (host_inputs && !c->d_cells) { CK(cudaMalloc(&c->d_cells, c->cap * kBytesPerCell)); CK(cudaMalloc(&c->d_p, c->cap * 48)); }
    if (n > c->host_cap) {
        for (void* p : {(void*)c->h_meta, (void*)c->h_uc, (void*)c->h_c, (void*)c->h_cells, (void*)c->h_p, (void*)c->h_idx}) if (p) cudaFreeHost(p);
        c->h_meta = nullptr; c->h_uc = c->h_c = c->h_cells = c->h_p = nullptr; c->h_idx = nullptr;
        CK(cudaMallocHost(&c->h_meta, (3 * n + kCellsPerExtBlob + 1) * 4)); CK(cudaMallocHost(&c->h_uc, n * 48));
        c->host_cap = n;
    }
    if (device_inputs && !c->h_cells) {
        CK(cudaMallocHost(&c->h_c, c->host_cap * 48)); CK(cudaMallocHost(&c->h_cells, c->host_cap * kBytesPerCell));
        CK(cudaMallocHost(&c->h_p, c->host_cap * 48)); CK(cudaMallocHost(&c->h_idx, c->host_cap * 8));
    }
    return KZGB200_OK;
}

// Host side of a cell batch: commitments deduplicated by their bytes (first-occurrence order), the cells grouped by cell index,
// both into h_meta (see cell_scalars_kernel); returns the number of unique commitments.
static size_t cell_plan(CellCtx* c, const uint8_t* commitments, const uint64_t* idx, size_t n) {
    uint32_t* meta = c->h_meta;
    uint32_t *cidx = meta + n, *order = meta + 2 * n, *start = meta + 3 * n;
    size_t tsize = 1;
    while (tsize < 2 * n) tsize <<= 1;
    if (c->slot.size() < tsize) c->slot.resize(tsize);
    std::fill(c->slot.begin(), c->slot.begin() + tsize, 0u);
    size_t m = 0;
    for (size_t k = 0; k < n; k++) {
        const uint8_t* key = commitments + 48 * k;
        uint64_t h;
        memcpy(&h, key + 8, 8);                         // x-coordinate bytes: uniform for valid points
        size_t s = (size_t)(h * 0x9e3779b97f4a7c15ull) & (tsize - 1);
        for (;; s = (s + 1) & (tsize - 1)) {
            const uint32_t u = c->slot[s];
            if (!u) { c->slot[s] = (uint32_t)(m + 1); memcpy(c->h_uc + 48 * m, key, 48); cidx[k] = (uint32_t)m++; break; }
            if (!memcmp(c->h_uc + 48 * (u - 1), key, 48)) { cidx[k] = u - 1; break; }
        }
        meta[k] = (uint32_t)idx[k];
    }
    for (int i = 0; i <= kCellsPerExtBlob; i++) start[i] = 0;
    for (size_t k = 0; k < n; k++) start[meta[k] + 1]++;
    for (int i = 0; i < kCellsPerExtBlob; i++) start[i + 1] += start[i];
    std::vector<uint32_t> cur(start, start + kCellsPerExtBlob);
    for (size_t k = 0; k < n; k++) order[cur[meta[k]]++] = (uint32_t)k;
    return m;
}
// r = SHA-256("RCKZGCBATCH__V1_" | u64be 4096 | u64be 64 | u64be m | u64be n | unique commitments |
//             per cell: u64be commitment index | u64be cell index | cell | proof) mod q; every byte is caller input
static void cell_transcript(uint8_t digest[32], const uint8_t* uc, size_t m, const uint32_t* cidx, const uint64_t* idx, const uint8_t* cells,
                            const uint8_t* proofs, size_t n) {
    HostSha256 s;
    host_sha256_init(&s);
    uint8_t hdr[48] = {'R', 'C', 'K', 'Z', 'G', 'C', 'B', 'A', 'T', 'C', 'H', '_', '_', 'V', '1', '_'};
    const uint64_t v[4] = {(uint64_t)kFieldElementsPerBlob, (uint64_t)kFieldElementsPerCell, (uint64_t)m, (uint64_t)n};
    for (int w = 0; w < 4; w++) for (int i = 0; i < 8; i++) hdr[16 + 8 * w + i] = (uint8_t)(v[w] >> (56 - 8 * i));
    host_sha256_update(&s, hdr, 48);
    host_sha256_update(&s, uc, m * 48);
    constexpr size_t kEntry = 16 + kBytesPerCell + 48, kBatch = 16;   // 2112 bytes = 33 SHA-256 blocks per cell
    std::vector<uint8_t> buf(kEntry * kBatch);
    for (size_t k = 0; k < n;) {
        size_t cnt = n - k < kBatch ? n - k : kBatch;
        for (size_t e = 0; e < cnt; e++, k++) {
            uint8_t* p = buf.data() + kEntry * e;
            for (int i = 0; i < 8; i++) { p[i] = (uint8_t)((uint64_t)cidx[k] >> (56 - 8 * i)); p[8 + i] = (uint8_t)(idx[k] >> (56 - 8 * i)); }
            memcpy(p + 16, cells + k * kBytesPerCell, kBytesPerCell);
            memcpy(p + 16 + kBytesPerCell, proofs + 48 * k, 48);
        }
        host_sha256_update(&s, buf.data(), kEntry * cnt);
    }
    host_sha256_final(&s, digest);
}

// ---- verify_cell_kzg_proof_batch[_many]: k independent cell batches (groups), one verdict each -------------------------------
// The spec's check of a group is linear in its per-cell weights r^j.  With w = rho^g r_g^j on the cells of group g, all groups are
// checked at once (one MSM, one pairing); only if that fails is every group checked on its own (many_*_kernel, k_cells.cu, and one
// pairing check per group on the many-check engine).  Each r_g is the spec's challenge of group g alone: its own transcript with its
// own deduplication of commitments, hashed by a small pool of host threads.  verify_cell_kzg_proof_batch is the case k = 1.

// x mod q for a 32-byte big-endian x (hash_to_bls_field): x < 2^256 < 3q, at most two subtractions
static void fr_reduce_be(uint8_t v[32]) {
    static const uint8_t q[32] = {0x73, 0xed, 0xa7, 0x53, 0x29, 0x9d, 0x7d, 0x48, 0x33, 0x39, 0xd8, 0x08, 0x09, 0xa1, 0xd8, 0x05,
                                  0x53, 0xbd, 0xa4, 0x02, 0xff, 0xfe, 0x5b, 0xfe, 0xff, 0xff, 0xff, 0xff, 0x00, 0x00, 0x00, 0x01};
    while (memcmp(v, q, 32) >= 0) {
        int borrow = 0;
        for (int i = 31; i >= 0; i--) {
            const int d = (int)v[i] - (int)q[i] - borrow;
            borrow = d < 0;
            v[i] = (uint8_t)(d + (borrow ? 256 : 0));
        }
    }
}
static void put_be64(uint8_t* p, uint64_t v) { for (int i = 0; i < 8; i++) p[i] = (uint8_t)(v >> (56 - 8 * i)); }
// what the hasher threads read: the globally deduplicated commitments (uc, cidx: see cell_plan) and the caller's host inputs
struct ManyHashJob {
    const uint8_t *uc, *cells, *proofs;
    const uint32_t* cidx;
    const uint64_t *idx, *off;
    size_t m;
};
// r_g of groups [g0, g1) -> rg + 32 g: the group's commitments deduplicated in first-occurrence order within the group (the global
// indices mapped to local ones), then cell_transcript as for a single call; an empty group gets 32 zero bytes
static void many_hash_range(const ManyHashJob* J, size_t g0, size_t g1, uint8_t* rg) {
    std::vector<size_t> seen(J->m, SIZE_MAX);
    std::vector<uint32_t> local(J->m), lcidx;
    std::vector<uint8_t> luc;
    for (size_t g = g0; g < g1; g++) {
        const size_t lo = J->off[g], cnt = J->off[g + 1] - lo;
        if (!cnt) { memset(rg + 32 * g, 0, 32); continue; }
        luc.clear();
        lcidx.resize(cnt);
        uint32_t lm = 0;
        for (size_t e = 0; e < cnt; e++) {
            const uint32_t u = J->cidx[lo + e];
            if (seen[u] != g) { seen[u] = g; local[u] = lm++; luc.insert(luc.end(), J->uc + 48 * (size_t)u, J->uc + 48 * (size_t)u + 48); }
            lcidx[e] = local[u];
        }
        cell_transcript(rg + 32 * g, luc.data(), lm, lcidx.data(), J->idx + lo, J->cells + lo * kBytesPerCell, J->proofs + 48 * lo, cnt);
        fr_reduce_be(rg + 32 * g);
    }
}
// rho = SHA-256("RCKZGCMANY___V1_" | u64be k | per group: u64be n_g | r_g (32 zero bytes if n_g = 0)) mod q; 0 -> 1
static void many_rho(const uint8_t* rg, const uint64_t* off, size_t k, uint8_t rho[32]) {
    HostSha256 s;
    host_sha256_init(&s);
    uint8_t hdr[24] = {'R', 'C', 'K', 'Z', 'G', 'C', 'M', 'A', 'N', 'Y', '_', '_', '_', 'V', '1', '_'};
    put_be64(hdr + 16, k);
    host_sha256_update(&s, hdr, 24);
    for (size_t g = 0; g < k; g++) {
        uint8_t e[40];
        put_be64(e, off[g + 1] - off[g]);
        memcpy(e + 8, rg + 32 * g, 32);
        host_sha256_update(&s, e, 40);
    }
    host_sha256_final(&s, rho);
    fr_reduce_be(rho);
    uint8_t o = 0;
    for (int i = 0; i < 32; i++) o |= rho[i];
    if (!o) rho[31] = 1;
}
template <class T>
static cudaError_t grow(T*& p, size_t& cap, size_t count) {
    if (count <= cap) return cudaSuccess;
    cap = 0;
    cudaError_t e = regrow(p, count);
    if (e == cudaSuccess) cap = count;
    return e;
}
// the per-group checks (only when the combined check fails): verdicts for every group from the parsed points, the weights and
// gbad of the combined check (all still on the device)
static int cell_many_fallback(kzgb200_ctx* ctx, const uint8_t* d_cells, size_t n, const uint64_t* off, const std::vector<uint32_t>& goff,
                              const std::vector<uint32_t>& gbad, size_t k, uint8_t* verdicts) {
    CellCtx* c = ctx->cells;
    const uint32_t* meta = c->h_meta;                 // [cell index | unique commitment | cells ordered by index | start]
    // the cells of every group ordered by index (a stable pass over the global order), and its runs of one index
    std::vector<uint32_t> cgroup(n), cur(goff.begin(), goff.end() - 1), ord(n), rstart, ridx, grun(k + 1);
    for (size_t g = 0; g < k; g++) for (size_t i = off[g]; i < off[g + 1]; i++) cgroup[i] = (uint32_t)g;
    for (size_t p = 0; p < n; p++) { const uint32_t i = meta[2 * n + p]; ord[cur[cgroup[i]]++] = i; }
    for (size_t g = 0; g < k; g++) {
        grun[g] = (uint32_t)ridx.size();
        if (gbad[g]) continue;                        // weights 0: no runs
        for (uint32_t p = goff[g]; p < goff[g + 1]; p++)
            if (p == goff[g] || meta[ord[p]] != meta[ord[p - 1]]) { rstart.push_back(p); ridx.push_back(meta[ord[p]]); }
    }
    const size_t runs = ridx.size();
    grun[k] = (uint32_t)runs;
    std::vector<uint32_t> fmeta;
    fmeta.reserve(n + 2 * runs + k + 2);
    fmeta.insert(fmeta.end(), ord.begin(), ord.end());
    fmeta.insert(fmeta.end(), rstart.begin(), rstart.end());
    fmeta.push_back((uint32_t)n);
    fmeta.insert(fmeta.end(), ridx.begin(), ridx.end());
    fmeta.insert(fmeta.end(), grun.begin(), grun.end());
    CK(grow(c->d_fmeta, c->fmeta_cap, fmeta.size()));
    CK(grow(c->d_terms, c->terms_cap, 2 * n));
    CK(grow(c->d_rcoef, c->rcoef_cap, (runs ? runs : 1) * kFieldElementsPerCell));
    const int ni = (int)n, ri = (int)runs;
    const unsigned kg = (unsigned)k;
    phase_begin(ctx, 7, ctx->stream);
    CK(cudaMemcpyAsync(c->d_fmeta, fmeta.data(), fmeta.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    many_terms_kernel<<<(ni + 127) / 128, 128, 0, ctx->stream>>>(ni, c->d_rk, ctx->d_z_mont, ctx->d_C, ctx->d_P, c->d_terms);
    many_group_sums_kernel<<<kg, 128, 0, ctx->stream>>>(c->d_goff, c->d_terms, c->d_AB);
    if (ri) many_run_interp_kernel<<<ri, kFieldElementsPerCell, 0, ctx->stream>>>(d_cells, c->d_fmeta, ni, ri, c->d_rk, c->tables, c->d_rcoef);
    many_group_rli_kernel<<<kg, 256, 0, ctx->stream>>>(c->d_rcoef, c->d_fmeta + n + 2 * runs + 1, c->d_AB, c->tables, c->d_gX, c->d_gX + k);
    CK(cudaGetLastError());
    int rc = launch_many_pairings(ctx, c->d_gX, c->d_gX + k, c->d_gbad, k, c->d_gv, c->tables->tau64_lines);
    if (rc) return rc;
    phase_end(ctx, 7, ctx->stream);
    CK(cudaMemcpyAsync(verdicts, c->d_gv, k, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t g = 0; g < k; g++) if (off[g] == off[g + 1]) verdicts[g] = kTrue;
    return KZGB200_OK;
}

// n = off[k] >= 1 cells in k groups.  hc / hidx / hcells / hp: host copies (the caller's, or the pinned read-back of device inputs);
// d_cells / d_p: the cells / proofs on the device, or (copy_inputs) copied there from the host copies.
static int cell_verify_groups(kzgb200_ctx* ctx, const uint8_t* hc, const uint64_t* hidx, const uint8_t* hcells, const uint8_t* hp,
                              const uint8_t* d_cells, const uint8_t* d_p, const uint64_t* off, size_t k, uint8_t* verdicts, bool copy_inputs) {
    CellCtx* c = ctx->cells;
    const size_t n = off[k];
    // an index >= 128 fails its group's first assertion; the plan sees index 0 in its place (the group's weights are 0)
    std::vector<uint32_t> goff(k + 1), gbad(k, 0);
    std::vector<uint64_t> sidx;
    for (size_t g = 0; g < k; g++) {
        goff[g] = (uint32_t)off[g];
        for (size_t i = off[g]; i < off[g + 1]; i++) if (hidx[i] >= (uint64_t)kCellsPerExtBlob) { gbad[g] = kErrScalar; break; }
        if (gbad[g]) {
            if (sidx.empty()) sidx.assign(hidx, hidx + n);
            for (size_t i = off[g]; i < off[g + 1]; i++) sidx[i] = 0;
        }
    }
    goff[k] = (uint32_t)n;
    const size_t m = cell_plan(c, hc, sidx.empty() ? hidx : sidx.data(), n);
    if (k > c->gcap) {
        CK(regrow(c->d_goff, k + 1)); CK(regrow(c->d_gbad, k)); CK(regrow(c->d_rg, 32 * (k + 1))); CK(regrow(c->d_gv, k));
        CK(regrow(c->d_AB, 2 * k)); CK(regrow(c->d_gX, 2 * k));
        c->gcap = k;
    }
    c->many_done = false;
    c->many_rg.assign(32 * (k + 1), 0);
    uint8_t* rg = c->many_rg.data();
    // the k transcripts on up to 16 host threads, each a contiguous range of groups of about n / threads cells, while the GPU parses
    const ManyHashJob job{c->h_uc, hcells, hp, c->h_meta + n, hidx, off, m};
    const size_t hw = std::max<size_t>(1, std::thread::hardware_concurrency()), nt = std::min<size_t>({k, hw, 16});
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> pool;
    for (size_t t = 0, g = 0; t < nt && g < k; t++) {
        size_t g1 = g + 1;
        const uint64_t target = (uint64_t)((unsigned __int128)n * (t + 1) / nt);
        while (g1 < k && off[g1 + 1] <= target) g1++;
        if (t + 1 == nt) g1 = k;
        pool.emplace_back(many_hash_range, &job, g, g1, rg);
        g = g1;
    }
    const int ni = (int)n, mi = (int)m, ki = (int)k;
    int rc = [&]() -> int {
        for (int i = 0; i < 8; i++) ctx->ph_started[i] = false;
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
        CK(cudaMemsetAsync(ctx->d_status, 0, n * sizeof(uint32_t), ctx->stream));
        CK(cudaMemsetAsync(c->d_ustatus, 0, m * sizeof(uint32_t), ctx->stream));
        CK(cudaMemcpyAsync(c->d_meta, c->h_meta, (3 * n + kCellsPerExtBlob + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(c->d_uc, c->h_uc, m * 48, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(c->d_goff, goff.data(), (k + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(c->d_gbad, gbad.data(), k * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (copy_inputs) {
            CK(cudaMemcpyAsync(c->d_p, hp, n * 48, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaMemcpyAsync(c->d_cells, hcells, n * kBytesPerCell, cudaMemcpyHostToDevice, ctx->stream));
            d_cells = c->d_cells; d_p = c->d_p;
        }
        phase_begin(ctx, kPhParse, ctx->stream);
        cell_points_kernel<<<(mi + 127) / 128, 128, 0, ctx->stream>>>(c->d_uc, mi, c->d_U, c->d_ustatus, kErrCommitment);
        cell_points_kernel<<<(ni + 127) / 128, 128, 0, ctx->stream>>>(d_p, ni, ctx->d_P, ctx->d_status, kErrProof);
        cell_check_kernel<<<(unsigned)(((size_t)n * kFieldElementsPerCell + 255) / 256), 256, 0, ctx->stream>>>(d_cells, ni, ctx->d_status);
        cell_scalars_kernel<<<(ni + 127) / 128, 128, 0, ctx->stream>>>(c->d_meta, ni, c->d_U, c->d_ustatus, c->tables, ctx->d_z_mont, ctx->d_zy,
                                                                        ctx->d_C, ctx->d_status);
        many_group_status_kernel<<<(ni + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_status, ni, c->d_goff, ki, c->d_gbad);
        phase_end(ctx, kPhParse, ctx->stream);
        CK(cudaGetLastError());
        return KZGB200_OK;
    }();
    for (auto& t : pool) t.join();
    const float hash_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (rc) return rc;
    many_rho(rg, off, k, rg + 32 * k);
    c->many_k = k;
    c->many_done = true;
    // the combined check: the weights (in d_rk), then RLI on the aux stream beside the big MSM
    phase_begin(ctx, kPhTranscript, ctx->stream);
    CK(cudaMemcpyAsync(c->d_rg, rg, 32 * (k + 1), cudaMemcpyHostToDevice, ctx->stream));
    many_weights_kernel<<<(ni + 127) / 128, 128, 0, ctx->stream>>>(ni, c->d_goff, ki, c->d_rg, c->d_gbad, c->d_rk, ctx->d_status);
    if (k == 1) r_from_digest_kernel<<<1, 1, 0, ctx->stream>>>(reinterpret_cast<const uint32_t*>(c->d_rg), ctx->d_r);   // for kzgb200_last_r
    phase_end(ctx, kPhTranscript, ctx->stream);
    CK(cudaEventRecord(c->ev_r, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->s_aux, c->ev_r, 0));
    cell_agg_kernel<<<dim3(kCellsPerExtBlob, kCellAggSlices), kFieldElementsPerCell, 0, ctx->s_aux>>>(d_cells, c->d_meta, ni, c->d_rk, c->d_agg);
    cell_interp_kernel<<<kCellsPerExtBlob, kFieldElementsPerCell, 0, ctx->s_aux>>>(c->d_agg, c->d_meta, ni, c->tables, c->d_coeffs);
    cell_rli_kernel<<<1, 256, 0, ctx->s_aux>>>(c->d_coeffs, c->tables, c->d_part + 1);
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->ev_rli, ctx->s_aux));
    // LL and RLC + RLP: the blob batch's MSM with z_k = h_k^64, y_k = 0
    ctx->cur_c = nullptr; ctx->cur_p = d_p; ctx->cur_n = n; ctx->subgroup_pending = false;
    if ((rc = launch_lincomb(ctx, 0, c->d_part, false, nullptr, 0, c->d_rk))) return rc;
    CK(cudaStreamWaitEvent(ctx->stream, c->ev_rli, 0));
    phase_begin(ctx, kPhFinal, ctx->stream);
    launch_batch_final(ctx->stream, c->d_part, 2, ctx->tables, ctx->d_result, ctx->d_scratch, false, c->tables->lines29);
    phase_end(ctx, kPhFinal, ctx->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(gbad.data(), c->d_gbad, k * 4, cudaMemcpyDeviceToHost, ctx->stream));
    int ok = 0;
    rc = read_result(ctx, &ok);
    if (rc != KZGB200_OK && rc != KZGB200_BAD_ARGS) return rc;
    if (rc == KZGB200_OK && ok) for (size_t g = 0; g < k; g++) verdicts[g] = gbad[g] ? kBadArgs : kTrue;
    else if (k == 1) verdicts[0] = gbad[0] || rc ? kBadArgs : kFalse;      // rho^0 = 1: the combined check is the group's own
    else if ((rc = cell_many_fallback(ctx, d_cells, n, off, goff, gbad, k, verdicts))) return rc;
    collect_phase_times(ctx);
    ctx->phase_ms[1] = hash_ms;
    ctx->phase_ms[2] = (float)pool.size();
    return KZGB200_OK;
}
// The four entry points: the argument checks, then the k groups of n = off[k] cells, from host or (device_inputs) device pointers.
static int cell_verify(kzgb200_ctx* ctx, const uint8_t* cm, const uint64_t* idx, const uint8_t* cells, const uint8_t* p, const uint64_t* off,
                       size_t k, uint8_t* verdicts, bool device_inputs) {
    if (!ctx || (k && (!off || !verdicts)) || k > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    size_t n = 0;
    if (k) {
        if (off[0] != 0) return KZGB200_BAD_ARGS;
        for (size_t g = 0; g < k; g++) if (off[g + 1] < off[g] || off[g + 1] > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
        n = off[k];
    }
    if (n && (!cm || !idx || !cells || !p)) return KZGB200_BAD_ARGS;
    if (!ctx->cells) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    CellCtx* c = ctx->cells;
    if (n == 0) {                                     // every group is empty (true); r_g = 0 and rho as for any call
        c->many_rg.assign(32 * (k + 1), 0);
        many_rho(c->many_rg.data(), off, k, c->many_rg.data() + 32 * k);
        c->many_k = k;
        c->many_done = true;
        if (k) memset(verdicts, kTrue, k);
        return KZGB200_OK;
    }
    DeviceGuard dev(ctx->device);
    int rc = cell_capacity(ctx, n, !device_inputs, device_inputs);
    if (rc) return rc;
    if (!device_inputs) return cell_verify_groups(ctx, cm, idx, cells, p, nullptr, nullptr, off, k, verdicts, true);
    // the exact transcripts are host chains over every input byte: the inputs come back to pinned memory once
    CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_parse, 0));
    CK(cudaMemcpyAsync(c->h_idx, idx, n * 8, cudaMemcpyDeviceToHost, ctx->s_d2h));
    CK(cudaMemcpyAsync(c->h_c, cm, n * 48, cudaMemcpyDeviceToHost, ctx->s_d2h));
    CK(cudaMemcpyAsync(c->h_p, p, n * 48, cudaMemcpyDeviceToHost, ctx->s_d2h));
    CK(cudaMemcpyAsync(c->h_cells, cells, n * kBytesPerCell, cudaMemcpyDeviceToHost, ctx->s_d2h));
    CK(cudaStreamSynchronize(ctx->s_d2h));
    return cell_verify_groups(ctx, c->h_c, c->h_idx, c->h_cells, c->h_p, cells, p, off, k, verdicts, false);
}
// one group: its verdict 2 (an assertion of the spec fails) is the call's BAD_ARGS
static int cell_verify_one(kzgb200_ctx* ctx, const uint8_t* cm, const uint64_t* idx, const uint8_t* cells, const uint8_t* p, size_t n, int* ok,
                           bool device_inputs) {
    if (!ok) return KZGB200_BAD_ARGS;
    const uint64_t off[2] = {0, n};
    uint8_t v = kFalse;
    int rc = cell_verify(ctx, cm, idx, cells, p, off, 1, &v, device_inputs);
    if (rc) return rc;
    if (v == kBadArgs) return KZGB200_BAD_ARGS;
    *ok = v == kTrue;
    return KZGB200_OK;
}

extern "C" int kzgb200_verify_cell_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* commitments, const uint64_t* cell_indices, const uint8_t* cells,
                                                   const uint8_t* proofs, size_t n, int* ok) {
    return cell_verify_one(ctx, commitments, cell_indices, cells, proofs, n, ok, false);
}
extern "C" int kzgb200_verify_cell_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_commitments, const uint64_t* d_cell_indices,
                                                          const uint8_t* d_cells, const uint8_t* d_proofs, size_t n, int* ok) {
    return cell_verify_one(ctx, d_commitments, d_cell_indices, d_cells, d_proofs, n, ok, true);
}
extern "C" int kzgb200_verify_cell_kzg_proof_batch_many(kzgb200_ctx* ctx, const uint8_t* commitments, const uint64_t* cell_indices, const uint8_t* cells,
                                                        const uint8_t* proofs, const uint64_t* group_offsets, size_t n_groups, uint8_t* verdicts) {
    return cell_verify(ctx, commitments, cell_indices, cells, proofs, group_offsets, n_groups, verdicts, false);
}
extern "C" int kzgb200_verify_cell_kzg_proof_batch_many_device(kzgb200_ctx* ctx, const uint8_t* d_commitments, const uint64_t* d_cell_indices,
                                                               const uint8_t* d_cells, const uint8_t* d_proofs, const uint64_t* group_offsets,
                                                               size_t n_groups, uint8_t* verdicts) {
    return cell_verify(ctx, d_commitments, d_cell_indices, d_cells, d_proofs, group_offsets, n_groups, verdicts, true);
}

// ---- verify_blob_cell_kzg_proof_batch[_many]: the cell proofs of whole blobs (EIP-7594 blob transactions), one verdict per group ---
// Group g = blobs [boff[g], boff[g + 1]) with their commitments and 128 cell proofs each.  Its verdict and r_g are those of
// verify_cell_kzg_proof_batch on the expanded call: per blob b in order and j < 128, (C_b, j, cell j of compute_cells(blob_b),
// proof 128 b + j).  The cells are computed on the device straight into d_cells, whose blob-major layout is already that per-cell
// order, and read back once to pinned memory: the exact transcripts are host chains over every cell byte.  The expanded commitments
// and indices are built on the host; then the cell pipeline (cell_verify_groups) runs unchanged with cell offsets = 128 x blob offsets.
static int blob_cell_verify(kzgb200_ctx* ctx, const uint8_t* blobs, const uint8_t* cm, const uint8_t* p, const uint64_t* boff, size_t k,
                            uint8_t* verdicts, bool device_inputs) {
    constexpr uint64_t kMaxBlobs = 0x7fffffff / 2 / kCellsPerExtBlob;       // 128 x blobs within the cell path's limit
    if (!ctx || (k && (!boff || !verdicts)) || k > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    size_t nb = 0;
    if (k) {
        if (boff[0] != 0) return KZGB200_BAD_ARGS;
        for (size_t g = 0; g < k; g++) if (boff[g + 1] < boff[g] || boff[g + 1] > kMaxBlobs) return KZGB200_BAD_ARGS;
        nb = boff[k];
    }
    if (nb && (!blobs || !cm || !p)) return KZGB200_BAD_ARGS;
    if (!ctx->cells) return KZGB200_INVALID_SETUP;
    std::vector<uint64_t> off(k + 1, 0);
    for (size_t g = 1; g <= k; g++) off[g] = boff[g] * kCellsPerExtBlob;
    if (nb == 0) return cell_verify(ctx, nullptr, nullptr, nullptr, nullptr, off.data(), k, verdicts, false);   // every group empty
    const size_t n = nb * kCellsPerExtBlob;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    CellCtx* c = ctx->cells;
    int rc = cell_capacity(ctx, n, true, true);                       // d_cells for the computed cells, the pinned h_* for the transcripts
    if (!rc && !device_inputs) rc = ensure_capacity(ctx, nb, true);   // the blob staging buffer
    if (rc) return rc;
    const uint8_t *d_blobs = blobs, *d_p = p, *hc = cm, *hp = p;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    if (device_inputs) {                              // as the cell _device form: commitments and proofs back to pinned memory once
        CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_parse, 0));
        CK(cudaMemcpyAsync(ctx->h_c, cm, nb * 48, cudaMemcpyDeviceToHost, ctx->s_d2h));
        CK(cudaMemcpyAsync(c->h_p, p, n * 48, cudaMemcpyDeviceToHost, ctx->s_d2h));
        hc = ctx->h_c; hp = c->h_p;
    } else {
        CK(cudaMemcpyAsync(ctx->d_blobs, blobs, nb * kBytesPerBlob, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(c->d_p, p, n * 48, cudaMemcpyHostToDevice, ctx->stream));
        d_blobs = ctx->d_blobs; d_p = c->d_p;
    }
    // No canonicity check here: compute_cells_kernel copies the raw blob bytes into cells 0..63, where cell_check_kernel flags any
    // element >= q and makes the group BadArgs -- the spec's compute_cells failing.  (The flags this kernel sets in d_status are cleared
    // by cell_verify_groups before its parse.)
    compute_cells_kernel<<<(unsigned)nb, kCellNttThreads, kCellNttSmemBytes, ctx->stream>>>(d_blobs, (int)nb, c->tables, c->d_cells, ctx->d_status);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(c->h_cells, c->d_cells, n * kBytesPerCell, cudaMemcpyDeviceToHost, ctx->stream));
    if (device_inputs) CK(cudaStreamSynchronize(ctx->s_d2h));
    for (size_t b = 0; b < nb; b++)
        for (int j = 0; j < kCellsPerExtBlob; j++) {
            const size_t e = b * kCellsPerExtBlob + j;
            memcpy(c->h_c + 48 * e, hc + 48 * b, 48);
            c->h_idx[e] = (uint64_t)j;
        }
    CK(cudaStreamSynchronize(ctx->stream));
    return cell_verify_groups(ctx, c->h_c, c->h_idx, c->h_cells, hp, c->d_cells, d_p, off.data(), k, verdicts, false);
}
// one group: its verdict 2 is the call's BAD_ARGS
static int blob_cell_verify_one(kzgb200_ctx* ctx, const uint8_t* blobs, const uint8_t* cm, const uint8_t* p, size_t n_blobs, int* ok,
                                bool device_inputs) {
    if (!ok) return KZGB200_BAD_ARGS;
    const uint64_t boff[2] = {0, n_blobs};
    uint8_t v = kFalse;
    int rc = blob_cell_verify(ctx, blobs, cm, p, boff, 1, &v, device_inputs);
    if (rc) return rc;
    if (v == kBadArgs) return KZGB200_BAD_ARGS;
    *ok = v == kTrue;
    return KZGB200_OK;
}

extern "C" int kzgb200_verify_blob_cell_kzg_proof_batch(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n_blobs, const uint8_t* commitments,
                                                        size_t n_commitments, const uint8_t* cell_proofs, size_t n_cell_proofs, int* ok) {
    if (!ctx || !ok) return KZGB200_BAD_ARGS;
    if (n_commitments != n_blobs || n_cell_proofs % kCellsPerExtBlob || n_cell_proofs / kCellsPerExtBlob != n_blobs) return KZGB200_INVALID_LENGTH;
    return blob_cell_verify_one(ctx, blobs, commitments, cell_proofs, n_blobs, ok, false);
}
extern "C" int kzgb200_verify_blob_cell_kzg_proof_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                                               const uint8_t* d_cell_proofs, size_t n_blobs, int* ok) {
    return blob_cell_verify_one(ctx, d_blobs, d_commitments, d_cell_proofs, n_blobs, ok, true);
}
extern "C" int kzgb200_verify_blob_cell_kzg_proof_batch_many(kzgb200_ctx* ctx, const uint8_t* blobs, const uint8_t* commitments,
                                                             const uint8_t* cell_proofs, const uint64_t* blob_offsets, size_t n_groups,
                                                             uint8_t* verdicts) {
    return blob_cell_verify(ctx, blobs, commitments, cell_proofs, blob_offsets, n_groups, verdicts, false);
}
extern "C" int kzgb200_verify_blob_cell_kzg_proof_batch_many_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, const uint8_t* d_commitments,
                                                                    const uint8_t* d_cell_proofs, const uint64_t* blob_offsets, size_t n_groups,
                                                                    uint8_t* verdicts) {
    return blob_cell_verify(ctx, d_blobs, d_commitments, d_cell_proofs, blob_offsets, n_groups, verdicts, true);
}

// test hook: r_g of every group of the last cell verification call (zeros for empty groups) and rho, canonical big-endian
extern "C" int kzgb200_last_cell_many_r(kzgb200_ctx* ctx, uint8_t* r_out, size_t n_groups, uint8_t* rho_out32) {
    if (!ctx || !rho_out32 || (n_groups && !r_out)) return KZGB200_BAD_ARGS;
    if (!ctx->cells) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    CellCtx* c = ctx->cells;
    if (!c->many_done || n_groups != c->many_k) return KZGB200_BAD_ARGS;
    if (n_groups) memcpy(r_out, c->many_rg.data(), 32 * n_groups);
    memcpy(rho_out32, c->many_rg.data() + 32 * n_groups, 32);
    return KZGB200_OK;
}

static int compute_cells_locked(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_out) {
    int rc = ensure_capacity(ctx, n, false);
    if (rc) return rc;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    CK(cudaMemsetAsync(ctx->d_status, 0, n * sizeof(uint32_t), ctx->stream));
    compute_cells_kernel<<<(unsigned)n, kCellNttThreads, kCellNttSmemBytes, ctx->stream>>>(d_blobs, (int)n, ctx->cells->tables, d_out, ctx->d_status);
    status_or_kernel<<<1, 256, 0, ctx->stream>>>(ctx->d_status, (int)n, ctx->d_result);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(ctx->h_result, ctx->d_result, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return ctx->h_result[0] ? KZGB200_BAD_ARGS : KZGB200_OK;
}
extern "C" int kzgb200_compute_cells(kzgb200_ctx* ctx, const uint8_t* blob, uint8_t* cells_out) {
    if (!ctx || !blob || !cells_out) return KZGB200_BAD_ARGS;
    if (!ctx->cells) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, 1, true);
    if (rc) return rc;
    CellCtx* c = ctx->cells;
    if (!c->d_ext) CK(cudaMalloc(&c->d_ext, (size_t)kCellsPerExtBlob * kBytesPerCell));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    CK(cudaMemcpyAsync(ctx->d_blobs, blob, kBytesPerBlob, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = compute_cells_locked(ctx, ctx->d_blobs, 1, c->d_ext))) return rc;
    CK(cudaMemcpyAsync(cells_out, c->d_ext, (size_t)kCellsPerExtBlob * kBytesPerCell, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
extern "C" int kzgb200_compute_cells_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_cells) {
    if (!ctx || (n && (!d_blobs || !d_cells)) || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (!ctx->cells) return KZGB200_INVALID_SETUP;
    if (n == 0) return KZGB200_OK;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    return compute_cells_locked(ctx, d_blobs, n, d_cells);
}

// cell workload: n_blobs polynomials of degree < `degree` (128 < degree <= 192), their 128 cells each (n_blobs x 128 x 2048
// bytes, blob-major), commitments (n_blobs x 48) and cell proofs (n_blobs x 128 x 48); tau_powers48 = [tau^j]G1, j < degree
extern "C" int kzgb200_harness_generate_cells(kzgb200_ctx* ctx, uint64_t seed, size_t n_blobs, int degree, const uint8_t* tau_powers48,
                                              uint8_t* d_cells, uint8_t* d_commitments, uint8_t* d_proofs) {
    if (!ctx || n_blobs == 0 || n_blobs > (1u << 20) || degree <= 2 * kFieldElementsPerCell || degree > kCellHarnessMaxDegree || !tau_powers48 ||
        !d_cells || !d_commitments || !d_proofs)
        return KZGB200_BAD_ARGS;
    if (!ctx->cells) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    const int n = (int)n_blobs;
    uint8_t* d_bytes = nullptr; G1Affine* d_M = nullptr; uint32_t* d_bad = nullptr; G1 *d_terms = nullptr, *d_sums = nullptr;
    uint32_t bad = 0;
    int rc = [&]() -> int {
        CK(cudaMalloc(&d_bytes, degree * 48)); CK(cudaMalloc(&d_M, degree * sizeof(G1Affine))); CK(cudaMalloc(&d_bad, 4));
        CK(cudaMalloc(&d_terms, (size_t)n * 6 * 64 * sizeof(G1))); CK(cudaMalloc(&d_sums, (size_t)n * 6 * sizeof(G1)));
        CK(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
        CK(cudaMemcpyAsync(d_bytes, tau_powers48, degree * 48, cudaMemcpyHostToDevice, ctx->stream));
        harness_parse_points_kernel<<<(degree + 31) / 32, 32, 0, ctx->stream>>>(d_bytes, degree, d_M, d_bad);
        cell_harness_eval_kernel<<<dim3(kCellsPerExtBlob * kFieldElementsPerCell / 128, n), 128, 0, ctx->stream>>>(seed, n, degree, ctx->cells->tables, d_cells);
        cell_harness_terms_kernel<<<(n * 6 * 64 + 127) / 128, 128, 0, ctx->stream>>>(seed, n, degree, d_M, d_terms);
        cell_harness_sums_kernel<<<(n * 6 + 127) / 128, 128, 0, ctx->stream>>>(n, d_terms, d_sums);
        cell_harness_points_kernel<<<(n * (kCellsPerExtBlob + 1) + 127) / 128, 128, 0, ctx->stream>>>(n, d_sums, ctx->cells->tables, d_commitments, d_proofs);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return KZGB200_OK;
    }();
    for (void* p : {(void*)d_bytes, (void*)d_M, (void*)d_bad, (void*)d_terms, (void*)d_sums}) if (p) cudaFree(p);
    if (rc) return rc;
    return bad ? KZGB200_BAD_ARGS : KZGB200_OK;
}

// ---- EIP-7594 cell proofs and recovery (k_cell_proofs.cu) ---------------------------------------------------------------
// FK20 tables: 8192 bases x 16 windows x 255 affine points (3.34 GB); monomial points 4096 x 100 bytes; scalar tables 416 KiB.
constexpr size_t kProofChunk = 512;          // blobs per pass through the proof / recovery workspace (~0.4 GB at 512)

extern "C" int kzgb200_load_cell_proof_setup(kzgb200_ctx* ctx, const uint8_t* g1_lagrange48, size_t n_points) {
    if (!ctx) return KZGB200_BAD_ARGS;
    if (!g1_lagrange48 || n_points != (size_t)kFieldElementsPerBlob) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    CellCtx* c = ctx->cells;
    if (!c) return KZGB200_INVALID_SETUP;
    if (c->d_fk_tab) return KZGB200_OK;
    uint8_t* d_bytes = nullptr; G1* d_a = nullptr; G1Affine* d_W = nullptr; uint32_t* d_bad = nullptr;
    uint32_t bad = 0;
    int rc = [&]() -> int {
        CK(cudaMalloc(&c->ptables, sizeof(ProofTables)));
        CK(cudaMalloc(&c->d_mono, kFieldElementsPerBlob * sizeof(G1Affine)));
        CK(cudaMalloc(&d_bytes, kFieldElementsPerBlob * 48)); CK(cudaMalloc(&d_a, kFieldElementsPerBlob * sizeof(G1)));
        CK(cudaMalloc(&d_W, kFk20Bases * sizeof(G1Affine))); CK(cudaMalloc(&d_bad, 4));
        CK(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
        CK(cudaMemcpyAsync(d_bytes, g1_lagrange48, kFieldElementsPerBlob * 48, cudaMemcpyHostToDevice, ctx->stream));
        proof_setup_kernel<<<kExtElements / 128, 128, 0, ctx->stream>>>(c->ptables);
        mono_load_kernel<<<kFieldElementsPerBlob / 128, 128, 0, ctx->stream>>>(d_bytes, d_a, d_bad);
        for (int len = 2; len <= kFieldElementsPerBlob; len <<= 1)
            mono_level_kernel<<<kFieldElementsPerBlob / 2 / 128, 128, 0, ctx->stream>>>(d_a, len, c->tables);
        mono_finish_kernel<<<kFieldElementsPerBlob / 128, 128, 0, ctx->stream>>>(d_a, c->tables, c->d_mono, d_bad);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (bad) return KZGB200_INVALID_SETUP;      // not the setup of the loaded cell points (or a point that does not parse)
        CK(cudaMalloc(&c->d_fk_tab, kFk20TablePoints * sizeof(G1Affine)));
        fk20_w_kernel<<<kFieldElementsPerCell, 64, 0, ctx->stream>>>(c->d_mono, c->tables, d_W);
        fk20_table_kernel<<<kFk20Bases * kFk20Windows / 128, 128, 0, ctx->stream>>>(d_W, c->d_fk_tab);
        CK(cudaGetLastError());
        CK(cudaFuncSetAttribute(compute_cells_coeffs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCellNttSmemBytes));
        CK(cudaFuncSetAttribute(recover_ntt_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCellNttSmemBytes));
        CK(cudaFuncSetAttribute(recover_ntt_div_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCellNttSmemBytes));
        CK(cudaFuncSetAttribute(recover_blob_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCellNttSmemBytes));
        CK(cudaMalloc(&c->d_rin, (size_t)kCellsPerExtBlob * kBytesPerCell)); CK(cudaMalloc(&c->d_pout, (size_t)kCellsPerExtBlob * 48));
        CK(cudaStreamSynchronize(ctx->stream));
        return KZGB200_OK;
    }();
    for (void* p : {(void*)d_bytes, (void*)d_a, (void*)d_W, (void*)d_bad}) if (p) cudaFree(p);
    if (rc != KZGB200_OK) proof_destroy(c);
    return rc;
}

extern "C" int kzgb200_cell_proof_monomial(kzgb200_ctx* ctx, uint8_t* out48, size_t n_points) {
    if (!ctx || !out48 || n_points > (size_t)kFieldElementsPerBlob) return KZGB200_BAD_ARGS;
    if (!ctx->cells || !ctx->cells->d_fk_tab) return KZGB200_INVALID_SETUP;
    if (n_points == 0) return KZGB200_OK;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    uint8_t* d_out = nullptr;
    int rc = [&]() -> int {
        CK(cudaMalloc(&d_out, n_points * 48));
        mono_compress_kernel<<<(unsigned)((n_points + 127) / 128), 128, 0, ctx->stream>>>(ctx->cells->d_mono, (int)n_points, d_out);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out48, d_out, n_points * 48, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return KZGB200_OK;
    }();
    if (d_out) cudaFree(d_out);
    return rc;
}

static int proof_workspace(kzgb200_ctx* ctx, size_t n) {
    CellCtx* c = ctx->cells;
    const size_t nb = n < kProofChunk ? n : kProofChunk;
    if (nb <= c->proof_cap) return KZGB200_OK;
    c->proof_cap = 0;
    CK(regrow(c->d_pcoef, nb * kFieldElementsPerBlob)); CK(regrow(c->d_fkU, nb * kFk20Bases)); CK(regrow(c->d_A, nb * kExtElements));
    CK(regrow(c->d_V, nb * kCellsPerExtBlob)); CK(regrow(c->d_pcommit, nb)); CK(regrow(c->d_rblobs, nb * kBytesPerBlob));
    CK(regrow(c->d_plans, nb)); CK(regrow(c->d_z, nb * 2 * kCellsPerExtBlob));
    c->proof_cap = nb;
    return KZGB200_OK;
}
// cells and proofs of n device blobs (the caller has checked n <= proof_cap or chunks; status: n flags, zeroed by the caller), and
// with d_commitments (nullable) their commitments, output 0 of FK20's inverse G1 DFT.
// Profiling slots: 0 = coefficients (with the cells), 1 = fixed-base products (with the scalar DFTs), 2 = G1 transforms (with the
// commitments' compression).
static int fk20_launch(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_cells, uint8_t* d_proofs, uint32_t* status,
                       uint8_t* d_commitments = nullptr) {
    CellCtx* c = ctx->cells;
    cudaStream_t st = ctx->stream;
    for (size_t lo = 0; lo < n; lo += kProofChunk) {
        const int cnt = (int)(n - lo < kProofChunk ? n - lo : kProofChunk);
        phase_begin(ctx, 0, st);
        compute_cells_coeffs_kernel<<<cnt, kCellNttThreads, kCellNttSmemBytes, st>>>(d_blobs + lo * kBytesPerBlob, cnt, c->tables,
                                                                                    d_cells + lo * kCellsPerExtBlob * kBytesPerCell, status + lo, c->d_pcoef);
        phase_end(ctx, 0, st);
        phase_begin(ctx, 1, st);
        fk20_scalars_kernel<<<dim3(kFieldElementsPerCell, cnt), 64, 0, st>>>(c->d_pcoef, c->tables, c->d_fkU);
        fk20_products_kernel<<<dim3(kCellsPerExtBlob, cnt), 64, 0, st>>>(c->d_fkU, c->d_fk_tab, c->d_V);
        phase_end(ctx, 1, st);
        phase_begin(ctx, 2, st);
        if (d_commitments) {
            fk20_proofs_commit_kernel<<<cnt, 64, 0, st>>>(c->d_V, c->tables, d_proofs + lo * kCellsPerExtBlob * 48, c->d_pcommit);
            fk20_commit_kernel<<<(cnt + 127) / 128, 128, 0, st>>>(c->d_pcommit, cnt, d_commitments + lo * 48);
        } else {
            fk20_proofs_kernel<<<cnt, 64, 0, st>>>(c->d_V, c->tables, d_proofs + lo * kCellsPerExtBlob * 48);
        }
        phase_end(ctx, 2, st);
    }
    CK(cudaGetLastError());
    return KZGB200_OK;
}
static int proof_begin(kzgb200_ctx* ctx, size_t n) {
    for (int i = 0; i < 8; i++) ctx->ph_started[i] = false;
    int rc = ensure_capacity(ctx, n, false);
    if (!rc) rc = proof_workspace(ctx, n);
    if (rc) return rc;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_parse, 0));
    CK(cudaMemsetAsync(ctx->d_status, 0, n * sizeof(uint32_t), ctx->stream));
    return KZGB200_OK;
}
// BAD_ARGS if any of the n blobs had a non-canonical element
static int proof_result(kzgb200_ctx* ctx, size_t n) {
    status_or_kernel<<<1, 256, 0, ctx->stream>>>(ctx->d_status, (int)n, ctx->d_result);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(ctx->h_result, ctx->d_result, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    collect_phase_times(ctx);
    return ctx->h_result[0] ? KZGB200_BAD_ARGS : KZGB200_OK;
}
// per-blob form of proof_result: status[b] = BAD_ARGS if blob b had a non-canonical element or host_bad[b], else OK
static int proof_result_each(kzgb200_ctx* ctx, size_t n, const uint8_t* host_bad, uint8_t* status) {
    std::vector<uint32_t> flags(n);
    CK(cudaMemcpyAsync(flags.data(), ctx->d_status, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    collect_phase_times(ctx);
    for (size_t b = 0; b < n; b++) status[b] = (host_bad[b] || flags[b]) ? KZGB200_BAD_ARGS : KZGB200_OK;
    return KZGB200_OK;
}
static bool proof_ready(kzgb200_ctx* ctx) { return ctx->cells && ctx->cells->d_fk_tab; }

extern "C" int kzgb200_compute_cells_and_kzg_proofs(kzgb200_ctx* ctx, const uint8_t* blob, uint8_t* cells_out, uint8_t* proofs_out) {
    if (!ctx || !blob || !cells_out || !proofs_out) return KZGB200_BAD_ARGS;
    if (!proof_ready(ctx)) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = ensure_capacity(ctx, 1, true);
    if (!rc) rc = proof_begin(ctx, 1);
    if (rc) return rc;
    CellCtx* c = ctx->cells;
    if (!c->d_ext) CK(cudaMalloc(&c->d_ext, (size_t)kCellsPerExtBlob * kBytesPerCell));
    CK(cudaMemcpyAsync(ctx->d_blobs, blob, kBytesPerBlob, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = fk20_launch(ctx, ctx->d_blobs, 1, c->d_ext, c->d_pout, ctx->d_status))) return rc;
    if ((rc = proof_result(ctx, 1))) return rc;
    CK(cudaMemcpyAsync(cells_out, c->d_ext, (size_t)kCellsPerExtBlob * kBytesPerCell, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(proofs_out, c->d_pout, (size_t)kCellsPerExtBlob * 48, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
extern "C" int kzgb200_compute_cells_and_kzg_proofs_batch_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n, uint8_t* d_cells, uint8_t* d_proofs) {
    if (!ctx || (n && (!d_blobs || !d_cells || !d_proofs)) || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (!proof_ready(ctx)) return KZGB200_INVALID_SETUP;
    if (n == 0) return KZGB200_OK;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = proof_begin(ctx, n);
    if (!rc) rc = fk20_launch(ctx, d_blobs, n, d_cells, d_proofs, ctx->d_status);
    return rc ? rc : proof_result(ctx, n);
}
// the commitment and the cell proofs (and, with cells_out, the cells) of n blobs, one FK20 pass per kProofChunk blobs, the commitment from the same
// inverse G1 DFT (fk20_launch with commitments): blob-major outputs, status[b] = what blob_to_kzg_commitment /
// compute_cells_and_kzg_proofs would return for blob b alone.  Host form (host = true): each pass of kProofChunk blobs is staged in
// the context's blob buffer and its outputs are copied back.  Without cells_out the cells go to the _many workspace (d_mcells).
static int commit_cells_proofs(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n, uint8_t* commitments_out, uint8_t* proofs_out,
                               uint8_t* cells_out, uint8_t* status, bool host) {
    if (n == 0) return KZGB200_OK;
    if (!ctx || !blobs || !commitments_out || !proofs_out || !status || n > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (!proof_ready(ctx)) return KZGB200_INVALID_SETUP;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = proof_begin(ctx, n);
    const size_t chunk = std::min(n, kProofChunk);
    if (!rc && host) rc = ensure_capacity(ctx, chunk, true);
    if (rc) return rc;
    CellCtx* c = ctx->cells;
    cudaStream_t st = ctx->stream;
    if ((host || !cells_out) && chunk > c->mout_cap) {
        c->mout_cap = 0;
        CK(regrow(c->d_mcells, chunk * kCellsPerExtBlob * kBytesPerCell)); CK(regrow(c->d_mproofs, chunk * kCellsPerExtBlob * 48));
        c->mout_cap = chunk;
    }
    for (size_t lo = 0; lo < n; lo += kProofChunk) {
        const size_t cnt = std::min(n - lo, kProofChunk);
        const uint8_t* d_in = blobs + lo * kBytesPerBlob;
        uint8_t* d_cm = commitments_out + lo * 48;
        uint8_t* d_c = cells_out && !host ? cells_out + lo * kCellsPerExtBlob * kBytesPerCell : c->d_mcells;
        uint8_t* d_p = host ? c->d_mproofs : proofs_out + lo * kCellsPerExtBlob * 48;
        if (host) {
            CK(cudaMemcpyAsync(ctx->d_blobs, d_in, cnt * kBytesPerBlob, cudaMemcpyHostToDevice, st));
            d_in = ctx->d_blobs;
            d_cm = ctx->d_c;
        }
        if ((rc = fk20_launch(ctx, d_in, cnt, d_c, d_p, ctx->d_status + lo, d_cm))) return rc;
        if (host) {
            CK(cudaMemcpyAsync(commitments_out + lo * 48, d_cm, cnt * 48, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(proofs_out + lo * kCellsPerExtBlob * 48, d_p, cnt * kCellsPerExtBlob * 48, cudaMemcpyDeviceToHost, st));
            if (cells_out)
                CK(cudaMemcpyAsync(cells_out + lo * kCellsPerExtBlob * kBytesPerCell, d_c, cnt * kCellsPerExtBlob * kBytesPerCell, cudaMemcpyDeviceToHost, st));
        }
    }
    const std::vector<uint8_t> no_host_checks(n);
    return proof_result_each(ctx, n, no_host_checks.data(), status);
}
extern "C" int kzgb200_compute_commitments_and_cell_proofs(kzgb200_ctx* ctx, const uint8_t* blobs, size_t n_blobs, uint8_t* commitments_out,
                                                           uint8_t* proofs_out, uint8_t* cells_out, uint8_t* status) {
    return commit_cells_proofs(ctx, blobs, n_blobs, commitments_out, proofs_out, cells_out, status, true);
}
extern "C" int kzgb200_compute_commitments_and_cell_proofs_device(kzgb200_ctx* ctx, const uint8_t* d_blobs, size_t n_blobs, uint8_t* d_commitments_out,
                                                                  uint8_t* d_proofs_out, uint8_t* d_cells_out, uint8_t* status) {
    return commit_cells_proofs(ctx, d_blobs, n_blobs, d_commitments_out, d_proofs_out, d_cells_out, status, false);
}

// The spec's argument checks on one index set: 64 <= n_cells <= 128, every index < 128, no index twice.  plan: pos[k] = the input
// position of cell index k or -1, missing = the absent indices, first = 0.  On failure the plan is the empty plan (reads nothing).
static int recover_plan(const uint64_t* idx, size_t n_cells, RecoverPlan* plan) {
    memset(plan->pos, 0xff, sizeof(plan->pos));
    plan->n_missing = 0;
    plan->first = 0;
    if (!idx || n_cells < (size_t)kCellsPerExtBlob / 2 || n_cells > (size_t)kCellsPerExtBlob) return KZGB200_BAD_ARGS;
    for (size_t j = 0; j < n_cells; j++) {
        if (idx[j] >= (uint64_t)kCellsPerExtBlob || plan->pos[idx[j]] >= 0) {
            memset(plan->pos, 0xff, sizeof(plan->pos));
            return KZGB200_BAD_ARGS;
        }
        plan->pos[idx[j]] = (int8_t)j;
    }
    for (int k = 0; k < kCellsPerExtBlob; k++) if (plan->pos[k] < 0) plan->missing[plan->n_missing++] = (uint8_t)k;
    return KZGB200_OK;
}
// n plans (n <= proof_cap) to the workspace, and their Z rows
static int recover_upload(kzgb200_ctx* ctx, const RecoverPlan* plans, size_t n) {
    CellCtx* c = ctx->cells;
    CK(cudaMemcpyAsync(c->d_plans, plans, n * sizeof(RecoverPlan), cudaMemcpyHostToDevice, ctx->stream));
    recover_z_kernel<<<(unsigned)n, 2 * kCellsPerExtBlob, 0, ctx->stream>>>(c->d_plans, c->tables, c->ptables, c->d_z);
    return KZGB200_OK;
}
// one pass of cnt <= kProofChunk blobs through the workspace: blob i uses uploaded plan i * plan_stride and reads its cells from
// d_in + (first + i * cell_stride + pos) x 2048; outputs as compute_cells_and_kzg_proofs; status: cnt flags.
// Profiling slot 3 = the recovery transforms (E Z, the three 8192-point transforms, the 4096-point transform back to the blob).
static int recover_pass(kzgb200_ctx* ctx, int plan_stride, const uint8_t* d_in, size_t cell_stride, int cnt, uint8_t* d_cells_out,
                        uint8_t* d_proofs_out, uint32_t* status) {
    CellCtx* c = ctx->cells;
    cudaStream_t st = ctx->stream;
    phase_begin(ctx, 3, st);
    recover_load_kernel<<<(unsigned)((size_t)cnt * kExtElements / 256), 256, 0, st>>>(d_in, (int)cell_stride, c->d_plans, plan_stride, c->d_z, cnt,
                                                                                     c->d_A, status);
    recover_ntt_inv_kernel<<<dim3(2, cnt), kCellNttThreads, kCellNttSmemBytes, st>>>(c->d_A, c->tables);
    recover_mid_kernel<<<(unsigned)((size_t)cnt * kFieldElementsPerBlob / 256), 256, 0, st>>>(c->d_A, c->ptables, cnt);
    recover_ntt_div_kernel<<<dim3(2, cnt), kCellNttThreads, kCellNttSmemBytes, st>>>(c->d_A, c->tables, c->d_z, plan_stride);
    recover_final_kernel<<<(unsigned)((size_t)cnt * kFieldElementsPerBlob / 256), 256, 0, st>>>(c->d_A, c->ptables, cnt, c->d_pcoef);
    recover_blob_kernel<<<cnt, kCellNttThreads, kCellNttSmemBytes, st>>>(c->d_pcoef, c->tables, c->d_rblobs);
    phase_end(ctx, 3, st);
    CK(cudaGetLastError());
    return fk20_launch(ctx, c->d_rblobs, cnt, d_cells_out, d_proofs_out, status);
}
// recovery of nb blobs that share one index set: d_in = nb x n_cells cells (blob-major).  One plan, one Z, for every pass.
static int recover_launch(kzgb200_ctx* ctx, const RecoverPlan& plan, const uint8_t* d_in, size_t n_cells, size_t nb, uint8_t* d_cells_out,
                          uint8_t* d_proofs_out) {
    int rc = recover_upload(ctx, &plan, 1);
    for (size_t lo = 0; !rc && lo < nb; lo += kProofChunk) {
        const int cnt = (int)(nb - lo < kProofChunk ? nb - lo : kProofChunk);
        rc = recover_pass(ctx, 0, d_in + lo * n_cells * kBytesPerCell, n_cells, cnt, d_cells_out + lo * kCellsPerExtBlob * kBytesPerCell,
                          d_proofs_out + lo * kCellsPerExtBlob * 48, ctx->d_status + lo);
    }
    return rc;
}
extern "C" int kzgb200_recover_cells_and_kzg_proofs(kzgb200_ctx* ctx, const uint64_t* cell_indices, const uint8_t* cells, size_t n_cells,
                                                    uint8_t* cells_out, uint8_t* proofs_out) {
    if (!ctx || !cells || !cells_out || !proofs_out) return KZGB200_BAD_ARGS;
    if (!proof_ready(ctx)) return KZGB200_INVALID_SETUP;
    RecoverPlan plan;
    int rc = recover_plan(cell_indices, n_cells, &plan);
    if (rc) return rc;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    if ((rc = proof_begin(ctx, 1))) return rc;
    CellCtx* c = ctx->cells;
    if (!c->d_ext) CK(cudaMalloc(&c->d_ext, (size_t)kCellsPerExtBlob * kBytesPerCell));
    CK(cudaMemcpyAsync(c->d_rin, cells, n_cells * kBytesPerCell, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = recover_launch(ctx, plan, c->d_rin, n_cells, 1, c->d_ext, c->d_pout))) return rc;
    if ((rc = proof_result(ctx, 1))) return rc;
    CK(cudaMemcpyAsync(cells_out, c->d_ext, (size_t)kCellsPerExtBlob * kBytesPerCell, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(proofs_out, c->d_pout, (size_t)kCellsPerExtBlob * 48, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KZGB200_OK;
}
extern "C" int kzgb200_recover_cells_and_kzg_proofs_batch_device(kzgb200_ctx* ctx, const uint64_t* cell_indices, size_t n_cells, const uint8_t* d_cells,
                                                                 size_t n_blobs, uint8_t* d_cells_out, uint8_t* d_proofs_out) {
    if (!ctx || (n_blobs && (!d_cells || !d_cells_out || !d_proofs_out)) || n_blobs > 0x7fffffff / 2) return KZGB200_BAD_ARGS;
    if (!proof_ready(ctx)) return KZGB200_INVALID_SETUP;
    RecoverPlan plan;
    int rc = recover_plan(cell_indices, n_cells, &plan);
    if (rc || n_blobs == 0) return rc;
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    if ((rc = proof_begin(ctx, n_blobs))) return rc;
    if ((rc = recover_launch(ctx, plan, d_cells, n_cells, n_blobs, d_cells_out, d_proofs_out))) return rc;
    return proof_result(ctx, n_blobs);
}
// recover_cells_and_kzg_proofs of n_blobs blobs, each from its own cells and index set: blob b owns cells and indices [off[b], off[b + 1]).
// The plans are built on the host; a blob that fails the argument checks keeps the empty plan (its kernels read nothing) and gets
// status BAD_ARGS.  Passes of kProofChunk blobs: the pass's plans and Z rows, then the recovery and FK20 kernels with one plan per
// blob.  Host form (host = true): the cells of a pass's good blobs are staged packed (one copy per run of consecutive good blobs),
// and the pass's outputs are copied back.
static int recover_many(kzgb200_ctx* ctx, const uint64_t* idx, const uint8_t* cells, const uint64_t* off, size_t n_blobs, uint8_t* cells_out,
                        uint8_t* proofs_out, uint8_t* status, bool host) {
    const size_t limit = 0x7fffffff / 2;
    if (!ctx || n_blobs > limit || (n_blobs && (!off || !cells_out || !proofs_out || !status))) return KZGB200_BAD_ARGS;
    if (n_blobs) {
        if (off[0] != 0) return KZGB200_BAD_ARGS;
        for (size_t b = 0; b < n_blobs; b++) if (off[b + 1] < off[b]) return KZGB200_BAD_ARGS;
        if (off[n_blobs] > limit || (off[n_blobs] && (!idx || !cells))) return KZGB200_BAD_ARGS;
    }
    if (!proof_ready(ctx)) return KZGB200_INVALID_SETUP;
    if (n_blobs == 0) return KZGB200_OK;
    std::vector<RecoverPlan> plans(n_blobs);
    std::vector<uint8_t> bad(n_blobs);
    size_t stage_cells = 0, pass_cells = 0;      // host form: the largest pass's cells of good blobs
    for (size_t b = 0; b < n_blobs; b++) {
        if (b % kProofChunk == 0) pass_cells = 0;
        bad[b] = recover_plan(idx + off[b], off[b + 1] - off[b], &plans[b]) != KZGB200_OK;
        if (!bad[b]) pass_cells += off[b + 1] - off[b];
        stage_cells = std::max(stage_cells, pass_cells);
    }
    std::lock_guard<std::mutex> g(ctx->lock);
    DeviceGuard dev(ctx->device);
    int rc = proof_begin(ctx, n_blobs);
    if (rc) return rc;
    CellCtx* c = ctx->cells;
    cudaStream_t st = ctx->stream;
    const size_t chunk = std::min(n_blobs, kProofChunk);
    if (host && stage_cells > c->mstage_cells) {
        c->mstage_cells = 0;
        CK(regrow(c->d_mstage, stage_cells * kBytesPerCell));
        c->mstage_cells = stage_cells;
    }
    if (host && chunk > c->mout_cap) {
        c->mout_cap = 0;
        CK(regrow(c->d_mcells, chunk * kCellsPerExtBlob * kBytesPerCell)); CK(regrow(c->d_mproofs, chunk * kCellsPerExtBlob * 48));
        c->mout_cap = chunk;
    }
    for (size_t lo = 0; lo < n_blobs; lo += kProofChunk) {
        const size_t cnt = std::min(n_blobs - lo, kProofChunk), hi = lo + cnt;
        const uint8_t* d_in = nullptr;
        if (host) {
            size_t packed = 0;
            for (size_t b = lo; b < hi;) {
                if (bad[b]) { b++; continue; }
                size_t e = b;
                for (; e < hi && !bad[e]; e++) plans[e].first = (uint32_t)(packed + off[e] - off[b]);
                const size_t n = off[e] - off[b];
                CK(cudaMemcpyAsync(c->d_mstage + packed * kBytesPerCell, cells + off[b] * kBytesPerCell, n * kBytesPerCell, cudaMemcpyHostToDevice, st));
                packed += n;
                b = e;
            }
            d_in = c->d_mstage;
        } else {
            for (size_t b = lo; b < hi; b++) plans[b].first = (uint32_t)(off[b] - off[lo]);
            d_in = cells + off[lo] * kBytesPerCell;
        }
        if ((rc = recover_upload(ctx, plans.data() + lo, cnt))) return rc;
        uint8_t* d_c = host ? c->d_mcells : cells_out + lo * kCellsPerExtBlob * kBytesPerCell;
        uint8_t* d_p = host ? c->d_mproofs : proofs_out + lo * kCellsPerExtBlob * 48;
        if ((rc = recover_pass(ctx, 1, d_in, 0, (int)cnt, d_c, d_p, ctx->d_status + lo))) return rc;
        if (host) {
            CK(cudaMemcpyAsync(cells_out + lo * kCellsPerExtBlob * kBytesPerCell, d_c, cnt * kCellsPerExtBlob * kBytesPerCell, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(proofs_out + lo * kCellsPerExtBlob * 48, d_p, cnt * kCellsPerExtBlob * 48, cudaMemcpyDeviceToHost, st));
        }
    }
    return proof_result_each(ctx, n_blobs, bad.data(), status);
}
extern "C" int kzgb200_recover_cells_and_kzg_proofs_many(kzgb200_ctx* ctx, const uint64_t* cell_indices, const uint8_t* cells,
                                                         const uint64_t* cell_offsets, size_t n_blobs, uint8_t* cells_out, uint8_t* proofs_out,
                                                         uint8_t* status) {
    return recover_many(ctx, cell_indices, cells, cell_offsets, n_blobs, cells_out, proofs_out, status, true);
}
extern "C" int kzgb200_recover_cells_and_kzg_proofs_many_device(kzgb200_ctx* ctx, const uint64_t* cell_indices, const uint8_t* d_cells,
                                                                const uint64_t* cell_offsets, size_t n_blobs, uint8_t* d_cells_out,
                                                                uint8_t* d_proofs_out, uint8_t* status) {
    return recover_many(ctx, cell_indices, d_cells, cell_offsets, n_blobs, d_cells_out, d_proofs_out, status, false);
}
