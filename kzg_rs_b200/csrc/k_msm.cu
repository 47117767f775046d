// K6: random linear combination (Pippenger MSM with GLV).
#include "common.cuh"
#include "coop.cuh"

namespace kzgb200 {

// ------------------------------------------------------------------------------------------------ K6
// Random linear combination (reference src/kzg_proof.rs:399-433), regrouped so that it needs no per-blob
// [y_i]G:   A = sum r_i pi_i ,  B = sum (r_i C_i + (r_i z_i) pi_i) - [sum r_i y_i] G ,  r_i = r^(offset+i).
// v1: one thread per blob does its scalar multiplications (Shamir's trick for the pair), results are then
// tree-summed by pair_sum_kernel.
// Pippenger bucket method with the GLV split: every scalar k = k1 + k2 x^2 (glv.cuh), so a point P contributes
// [k1]P + [k2](-phi(P)) with two 128-bit halves -> 16 windows of 8 bits x 255 buckets.  Three point/scalar sets per rank:
//   set 0: pi_i with r_i  (-> A),   set 1: C_i with r_i,   set 2: pi_i with r_i z_i   (sets 1+2 -> B').
// No sorting network and no atomics on points: a counting sort of the digits per (scalar kind, half, window) gives
// every bucket two contiguous index lists (low halves -> P_i, high halves -> -phi(P_i)); threads own buckets.
__global__ void __launch_bounds__(128) msm_scalars_kernel(const Fr* __restrict__ z_mont, const ZY* __restrict__ zy, const Fr* __restrict__ r_mont,
                                                          uint64_t offset, int n, uint8_t* __restrict__ digits /* [4*16][n] */,
                                                          Fr* __restrict__ ry, const Fr* __restrict__ weights) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t e = offset + (uint64_t)i;
    uint32_t ee[2] = {(uint32_t)e, (uint32_t)(e >> 32)};
    Fr ri = weights ? weights[i] : r_mont->pow(ee, 64);   // r^(offset+i), Montgomery (compute_powers, kzg_proof.rs:279-289), or the caller's weight
    Fr ri_raw = ri.to_raw();
    Fr rz_raw = (ri * z_mont[i]).to_raw();    // r_i z_i   (kzg_proof.rs:425)
    ry[i] = ri * zy[i].y;                     // r_i y_i in normal form
    uint32_t h[2][2][4];
    glv_split(ri_raw.l, h[0][0], h[0][1]);
    glv_split(rz_raw.l, h[1][0], h[1][1]);
    for (int kind = 0; kind < 2; kind++)
        for (int half = 0; half < 2; half++)
            for (int w = 0; w < kWindows; w++)
                digits[((size_t)(kind * 2 + half) * kWindows + w) * n + i] = (uint8_t)(h[kind][half][w >> 2] >> (8 * (w & 3)));
}
// counting sort of one digit row: grid = kDigitRows; order[row][*] = blob indices grouped by digit,
// start[row][b] = first position of digit b (start[row][256] = n)
__global__ void __launch_bounds__(256) msm_sort_kernel(const uint8_t* __restrict__ digits, int n, uint32_t* __restrict__ order,
                                                       uint32_t* __restrict__ start) {
    __shared__ uint32_t hist[kBuckets], cursor[kBuckets];
    int row_id = blockIdx.x, t = threadIdx.x;
    const uint8_t* row = digits + (size_t)row_id * n;
    uint32_t* ord = order + (size_t)row_id * n;
    uint32_t* st = start + (size_t)row_id * (kBuckets + 1);
    hist[t] = 0;
    __syncthreads();
    for (int i = t; i < n; i += blockDim.x) atomicAdd(&hist[row[i]], 1u);
    __syncthreads();
    if (t == 0) {
        uint32_t acc = 0;
        for (int b = 0; b < kBuckets; b++) { cursor[b] = acc; st[b] = acc; acc += hist[b]; }
        st[kBuckets] = acc;
    }
    __syncthreads();
    for (int i = t; i < n; i += blockDim.x) ord[atomicAdd(&cursor[row[i]], 1u)] = (uint32_t)i;
}
// Bucket accumulation, balanced.  A "row" = (point set, GLV half, window): its sorted index list (n entries, grouped by digit) is
// cut into slices of `slice` consecutive entries (msm_slice_len) and every thread sums exactly one slice -- round 1 gave whole bucket lists to
// threads (Poisson-sized: a warp ran at the pace of its longest lane, +40 %).  A slice spans one or a few digit runs: a run that
// lies entirely inside the slice is a finished half-bucket and goes to `halfsum`; the slice's first / last run may continue in
// the neighbouring slices and goes to `part` slot 0 / 1 (a slice that is one single run: slot 0).  msm_bucket_join_kernel adds
// up the few partials per bucket and the two GLV halves.  The next entry's index and point are fetched one addition ahead.
__device__ __forceinline__ G1Affine ldg_point(const G1Affine* p) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    G1Affine a;
#pragma unroll
    for (int k = 0; k < 12; k++) { a.x.l[k] = __ldg(w + k); a.y.l[k] = __ldg(w + 12 + k); }
    a.inf = __ldg(w + 24);
    return a;
}
template <int kCtasPerSm>
__global__ void __launch_bounds__(128, kCtasPerSm) msm_bucket_kernel(const G1Affine* __restrict__ C, const G1Affine* __restrict__ P, int n,
                                                         const uint32_t* __restrict__ order, const uint32_t* __restrict__ start,
                                                         G1* __restrict__ halfsum /* [96][256] */, G1* __restrict__ part /* [96][slices][2] */, int slice) {
    const int slices = (n + slice - 1) / slice;
    int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= kMsmRows * slices) return;
    int row = tid / slices, s = tid % slices;                 // row = (set * 2 + half) * kWindows + w
    int w = row % kWindows, half = (row / kWindows) & 1, set = row / (2 * kWindows);
    const G1Affine* pts = set == 1 ? C : P;
    int digit_row = ((set == 2 ? 1 : 0) * 2 + half) * kWindows + w;
    const uint32_t* ord = order + (size_t)digit_row * n;
    const uint32_t* st = start + (size_t)digit_row * (kBuckets + 1);
    const uint32_t pos0 = (uint32_t)s * slice, end0 = pos0 + slice < (uint32_t)n ? pos0 + slice : (uint32_t)n;
    // digit of the first entry: the largest b with st[b] <= pos0
    int b = 0;
#pragma unroll
    for (int step = 128; step >= 1; step >>= 1) if (b + step <= 255 && __ldg(st + b + step) <= pos0) b += step;
    uint32_t next_boundary = __ldg(st + b + 1);
    G1 acc = G1::identity();
    bool first = true;
    auto flush = [&](int bb) {
        uint32_t lo = __ldg(st + bb), hi = __ldg(st + bb + 1);
        if (bb != 0 && hi > lo) {
            if (lo >= pos0 && hi <= end0) halfsum[(size_t)row * kBuckets + bb] = acc;
            else part[((size_t)row * slices + s) * 2 + (first ? 0 : 1)] = acc;
        }
        first = false;
        acc = G1::identity();
    };
    const uint32_t beta_l[12] = KZG_FP_BETA_M;
    const Fp beta = fp_const(beta_l);
    G1Affine nxt = ldg_point(pts + __ldg(ord + pos0));
    for (uint32_t k = pos0; k < end0; k++) {
        G1Affine q = nxt;
        if (k + 1 < end0) nxt = ldg_point(pts + __ldg(ord + k + 1));
        while (k >= next_boundary) { flush(b); b++; next_boundary = __ldg(st + b + 1); }
        if (b != 0) {
            if (half && !q.inf) { q.x = q.x * beta; q.y = q.y.neg(); }     // -phi(P) = (beta x, -y)
            acc = acc.add_mixed(q);
        }
    }
    flush(b);
}
// occupancy variants: 2 CTAs per SM keep everything in registers (216), 3 / 4 trade a few spilled words for more chains in flight
void launch_msm_bucket(int ctas_per_sm, int n, int slice, cudaStream_t st, const G1Affine* C, const G1Affine* P, const uint32_t* order,
                       const uint32_t* start, G1* halfsum, G1* part) {
    const int slices = (n + slice - 1) / slice, grid = (kMsmRows * slices + 127) / 128;
    if (ctas_per_sm >= 4) msm_bucket_kernel<4><<<grid, 128, 0, st>>>(C, P, n, order, start, halfsum, part, slice);
    else if (ctas_per_sm == 3) msm_bucket_kernel<3><<<grid, 128, 0, st>>>(C, P, n, order, start, halfsum, part, slice);
    else msm_bucket_kernel<2><<<grid, 128, 0, st>>>(C, P, n, order, start, halfsum, part, slice);
}
// kJoinLanes (2, 4 or 8; kzgb200_ctx::msm_join) threads per (set, window, bucket): the bucket's partial sums of both GLV halves ->
// buckets[set][window][bucket].  A bucket of ~n/256 entries spans several slices per half (about 10 partial sums at n = 16384).
// The list is dealt round-robin to the lanes -- ONE call site of the addition, so lanes with different list shapes do not run
// divergent copies of it (round 2's first form, one thread per bucket with a branch per half, took 0.40 ms) -- and the lane sums
// are folded by a shuffle tree.  Two lanes measured best (0.20 ms): more lanes shorten the chain but every tree step costs a
// whole warp an addition for a few active lanes.
__device__ __forceinline__ G1 shfl_xor_point(const G1& p, int m) {
    G1 r;
#pragma unroll
    for (int k = 0; k < 12; k++) {
        r.x.l[k] = __shfl_xor_sync(0xffffffffu, p.x.l[k], m);
        r.y.l[k] = __shfl_xor_sync(0xffffffffu, p.y.l[k], m);
        r.z.l[k] = __shfl_xor_sync(0xffffffffu, p.z.l[k], m);
    }
    return r;
}
template <int kJoinLanes>
__global__ void __launch_bounds__(128) msm_bucket_join_kernel(int n, const uint32_t* __restrict__ start, const G1* __restrict__ halfsum,
                                                              const G1* __restrict__ part, G1* __restrict__ buckets /* [3][16][256] */, int slice) {
    const int slices = (n + slice - 1) / slice;
    const uint32_t usl = (uint32_t)slice;
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;       // the grid is exactly kMsmSets * kWindows * kBuckets * kJoinLanes threads
    const int tid = gt / kJoinLanes, j = gt % kJoinLanes;
    int b = tid % kBuckets, w = (tid / kBuckets) % kWindows, set = tid / (kBuckets * kWindows);
    G1 acc = G1::identity();
    if (b != 0) {
        uint32_t lo[2], s0[2], cnt[2];
        int row[2];
#pragma unroll
        for (int half = 0; half < 2; half++) {
            row[half] = (set * 2 + half) * kWindows + w;
            const int digit_row = ((set == 2 ? 1 : 0) * 2 + half) * kWindows + w;
            const uint32_t* st = start + (size_t)digit_row * (kBuckets + 1);
            const uint32_t l = __ldg(st + b), h = __ldg(st + b + 1);
            lo[half] = l; s0[half] = l / usl;
            cnt[half] = h > l ? (h - 1) / usl - l / usl + 1 : 0u;
        }
        const uint32_t total = cnt[0] + cnt[1];
        for (uint32_t i = (uint32_t)j; i < total; i += kJoinLanes) {
            const int half = i >= cnt[0] ? 1 : 0;
            const uint32_t k = half ? i - cnt[0] : i;
            const G1* src;
            if (cnt[half] == 1) src = halfsum + (size_t)row[half] * kBuckets + b;          // the run lies inside one slice
            else {
                const uint32_t s = s0[half] + k;
                const int slot = (k == 0 && lo[half] != s0[half] * usl) ? 1 : 0;        // the bucket opens inside slice s0: that slice's last run
                src = part + ((size_t)row[half] * slices + s) * 2 + slot;
            }
            acc = acc.add(*src);
        }
    }
#pragma unroll 1
    for (int m = 1; m < kJoinLanes; m <<= 1) {
        const G1 o = shfl_xor_point(acc, m);
        if ((j & (2 * m - 1)) == 0) acc = acc.add(o);
    }
    if (j == 0) buckets[tid] = acc;
}
void launch_msm_bucket_join(int lanes, int n, int slice, cudaStream_t st, const uint32_t* start, const G1* halfsum, const G1* part, G1* buckets) {
    const int items = kMsmSets * kWindows * kBuckets;
    if (lanes >= 8) msm_bucket_join_kernel<8><<<items * 8 / 128, 128, 0, st>>>(n, start, halfsum, part, buckets, slice);
    else if (lanes >= 4) msm_bucket_join_kernel<4><<<items * 4 / 128, 128, 0, st>>>(n, start, halfsum, part, buckets, slice);
    else msm_bucket_join_kernel<2><<<items * 2 / 128, 128, 0, st>>>(n, start, halfsum, part, buckets, slice);
}
// one CTA per (set, window), one thread per bucket: W = sum_b b * bucket[b] = sum_{b >= 1} T_b with the suffix sums
// T_b = sum_{c >= b} bucket[c].  Suffix scan (8 steps) + tree (8 steps) through shared memory: 16 additions deep, no doublings
// (round 2 first ran 4 buckets per lane with the running-sum trick and a double-and-add for the segment offset: ~26 deep).
static_assert(sizeof(G1) * kWinLanes == kWinSmemBytes, "keep kWinSmemBytes (common.cuh) in step with G1");
__global__ void __launch_bounds__(kWinLanes) msm_window_kernel(const G1* __restrict__ buckets, G1* __restrict__ windows /* [3][16] */) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    G1* sm = reinterpret_cast<G1*>(dyn_smem);      // [kWinLanes]
    const int l = threadIdx.x, sw = blockIdx.x;   // sw = set * kWindows + window
    G1 mine = buckets[(size_t)sw * kBuckets + l];  // bucket 0 holds the identity
#pragma unroll 1
    for (int d = 1; d < kWinLanes; d <<= 1) {
        sm[l] = mine;
        __syncthreads();
        if (l + d < kWinLanes) mine = mine.add(sm[l + d]);
        __syncthreads();
    }
    sm[l] = l ? mine : G1::identity();
    __syncthreads();
#pragma unroll 1
    for (int span = kWinLanes / 2; span >= 1; span >>= 1) {
        if (l < span) sm[l] = sm[l].add(sm[l + span]);
        __syncthreads();
    }
    if (l == 0) windows[sw] = sm[0];
}
// window sums -> A = sum_w 256^w W[0][w], B' = sum_w 256^w (W[1][w] + W[2][w]) (Horner, 8 doublings per window): the serial part
// of the MSM, 120 doublings + 16 additions per point set.
//
// Round 2: the three chains run in LOCKSTEP on the cooperative engine of the pairing check (vliw29.cuh: programs g1_dbl / g1_add over
// three register files, one warp per Fp product, 16 lanes per sum) on 384 threads -- a doubling is 6 short levels (~2 us) instead of
// three lone-thread Fp products in a row (~4.9 us).  The generic addition formula is only valid for distinct non-identity points;
// identities are tracked exactly (flags from the window sums), and the astronomically unlikely equal-x case (H = 0, checked after
// every addition) switches the whole kernel back to round 1's warp-cooperative chains (coop.cuh), which handle every case.
// Beside the chains, 160 helper threads OR the per-blob error flags, tree-sum s = sum r_i y_i and form [s]G from the fixed-base
// table (64 lookups, a 6-level tree); the partial carries B' - [s]G and ry = 0, so the final check has no fixed-base work left.
// `out` may be a peer-mapped pointer into the group leader's exchange buffer (multi-GPU: the partial-sum gather is this kernel's
// last store, over NVLink); then `flag` (same buffer) receives `epoch` after the partial, with a system-scope fence in between.
constexpr int kCombEngine = 384;                              // kCombineThreads = 544, kCombHelpers = 160 (common.cuh)
constexpr int kCombRegs = 96;                                  // registers per chain: g1_add needs 83; 90..92 = saved accumulator
static_assert(kCombEngine + kCombHelpers == kCombineThreads, "thread split of msm_combine_kernel");
// kCombHelpers threads (h = 0..kCombHelpers-1, meeting at `bar`): OR of the per-blob error flags into *err (shared), s = sum r_i y_i
// tree-summed in sry[kCombHelpers], [s]G from the fixed-base table (64 lookups, a 6-level tree) into sg[0] (sg: 64 shared points)
template <class Bar>
__device__ __forceinline__ void sum_s_sg(int h, const Fr* __restrict__ ry, const uint32_t* __restrict__ status, int n, const DeviceTables* __restrict__ T,
                                         uint32_t* err, Fr* sry, G1* sg, Bar bar) {
    uint32_t e = 0;
    Fr acc_ry = Fr::zero();
    for (int i = h; i < n; i += kCombHelpers) { e |= status[i]; acc_ry = acc_ry.add_inl(ry[i]); }
    if (e) atomicOr(err, e);
    sry[h] = acc_ry;
    bar();
    for (int span = 128; span >= 1; span >>= 1) {
        if (h < span && h + span < kCombHelpers) sry[h] = sry[h].add_inl(sry[h + span]);
        bar();
    }
    // [s]G: helper h < 64 takes the h-th 4-bit digit of s (normal form), then a tree over the 64 table points
    if (h < 64) {
        const Fr sv = sry[0];
        const uint32_t d = (sv.l[h / 8] >> (4 * (h % 8))) & 15u;
        sg[h] = d ? G1::from_affine(T->gen_table[h][d - 1]) : G1::identity();
    }
    bar();
    for (int span = 32; span >= 1; span >>= 1) {
        if (h < span) sg[h] = sg[h].add(sg[h + span]);
        bar();
    }
}
struct CombineSmem {
    f29::F29 regs[kMsmSets][kCombRegs];
    f29::F29 win[kMsmSets][kWindows][3];
    vliw29::SharedTables stab;
};
static_assert(sizeof(CombineSmem) <= kCombineSmemBytes, "keep kCombineSmemBytes (common.cuh) in step with CombineSmem");
__global__ void __launch_bounds__(kCombineThreads) msm_combine_kernel(const G1* __restrict__ windows, const Fr* __restrict__ ry, const uint32_t* __restrict__ status,
                                                                      int n, const DeviceTables* __restrict__ T, Partial* __restrict__ out, uint32_t* flag, uint32_t epoch) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    CombineSmem& S = *reinterpret_cast<CombineSmem*>(dyn_smem);
    __shared__ uint32_t s_err, s_fallback;
    __shared__ uint8_t s_wid[kMsmSets][kWindows];
    __shared__ Fr s_ry[kCombHelpers];
    __shared__ CoopPoint cp[3];
    __shared__ G1 s_sg[64];
    const int t = threadIdx.x;
    if (t == 0) { s_err = 0; s_fallback = 0; }
    __syncthreads();
    if (t < kCombEngine) {
        auto ebar = [] { asm volatile("bar.sync 2, %0;" ::"n"(kCombEngine) : "memory"); };
        // program tables + the window sums in the engine's representation
        {
            const vliw29::Tables src = vliw29::default_tables();
            for (int i = t; i < vliw29::kNumMul * 4; i += kCombEngine) (&S.stab.mul[0][0])[i] = (&src.mul[0][0])[i];
            for (int i = t; i < vliw29::kNumLin * 4; i += kCombEngine) (&S.stab.lin[0][0])[i] = (&src.lin[0][0])[i];
            for (int i = t; i < vliw29::kNumTerm; i += kCombEngine) S.stab.term[i] = src.term[i];
            for (int i = t; i < vliw29::kNumLevel; i += kCombEngine) S.stab.level[i] = src.level[i];
            for (int i = t; i < vliw29::kNumPrograms; i += kCombEngine) S.stab.prog[i] = src.prog[i];
            if (t < 16) S.stab.p29[t] = t < 14 ? (int32_t)f29::p29_rt(t) : 0;
        }
        for (int i = t; i < kMsmSets * kWindows * 3; i += kCombEngine) {
            const int sw = i / 3, c = i % 3;
            const G1& w = windows[sw];
            S.win[sw / kWindows][sw % kWindows][c] = f29::from_fp(c == 0 ? w.x : (c == 1 ? w.y : w.z));
            if (c == 2) s_wid[sw / kWindows][sw % kWindows] = w.z.is_zero() ? 1 : 0;
        }
        for (int i = t; i < kMsmSets * kCombRegs; i += kCombEngine) S.regs[i / kCombRegs][i % kCombRegs] = f29::f29_zero();
        ebar();
        vliw29::Lanes L{t, kCombEngine, vliw29::Tables{S.stab.mul, S.stab.lin, S.stab.term, S.stab.level, S.stab.prog}, nullptr, S.stab.p29};
        L.groups = kMsmSets; L.gstride = kCombRegs; L.bar_id = 2; L.bar_threads = kCombEngine;
        f29::F29* regs = &S.regs[0][0];
        bool acc_id[kMsmSets] = {true, true, true};       // the accumulator of chain g is the identity (same value in every thread)
        for (int w = kWindows - 1; w >= 0; w--) {
            if (w != kWindows - 1) for (int k = 0; k < 8; k++) vliw29::run(vliw29::kProg_g1_dbl, regs, L);
            // (X, Y, Z) += window sum w of every chain: addend into registers 3..5, accumulator saved in 90..92
            for (int i = t; i < kMsmSets * 3 * 4; i += kCombEngine) {
                const int g = i / 12, c = (i / 4) % 3, q = i % 4;
                reinterpret_cast<uint4*>(&S.regs[g][3 + c])[q] = reinterpret_cast<const uint4*>(&S.win[g][w][c])[q];
                reinterpret_cast<uint4*>(&S.regs[g][90 + c])[q] = reinterpret_cast<const uint4*>(&S.regs[g][c])[q];
            }
            ebar();
            vliw29::run(vliw29::kProg_g1_add, regs, L);
            // the cases the generic formula does not cover
            for (int i = t; i < kMsmSets * 3 * 4; i += kCombEngine) {
                const int g = i / 12, c = (i / 4) % 3, q = i % 4;
                if (s_wid[g][w]) reinterpret_cast<uint4*>(&S.regs[g][c])[q] = reinterpret_cast<const uint4*>(&S.regs[g][90 + c])[q];     // + identity
                else if (acc_id[g]) reinterpret_cast<uint4*>(&S.regs[g][c])[q] = reinterpret_cast<const uint4*>(&S.regs[g][3 + c])[q];    // identity + W
            }
            if (t < kMsmSets && !s_wid[t][w] && !acc_id[t]) {          // equal x (P = +-Q): not handled here
                if (vliw29::canonical_signed(S.regs[t][6]).is_zero()) s_fallback = 1;
            }
#pragma unroll
            for (int g = 0; g < kMsmSets; g++) acc_id[g] = acc_id[g] && s_wid[g][w];
            ebar();
        }
        // back to the 12 x 32 Montgomery form for the last two additions (coop.cuh handles every case)
        if (t < kMsmSets * 3) {
            const int g = t / 3, c = t % 3;
            Fp v = Fp::from_raw(vliw29::canonical_signed(S.regs[g][c]));
            if (acc_id[g]) v = c == 2 ? Fp::zero() : Fp::one();
            cp[g].v[c] = v;
        }
        ebar();
        if (s_fallback && t < 32 * kMsmSets) {        // round 1's chains
            const int warp = t >> 5, lane = t & 31;
            CoopPoint* s = &cp[warp];
            __syncwarp();
            if (lane == 0) { s->v[0] = Fp::one(); s->v[1] = Fp::one(); s->v[2] = Fp::zero(); }
            __syncwarp();
            for (int w = kWindows - 1; w >= 0; w--) {
                if (w != kWindows - 1) for (int k = 0; k < 8; k++) coop_dbl(s, lane);
                coop_add(s, windows[warp * kWindows + w], lane);
            }
        }
    } else {
        // helpers, beside the chains: OR of the per-blob error flags, s = sum r_i y_i, [s]G
        sum_s_sg(t - kCombEngine, ry, status, n, T, &s_err, s_ry, s_sg, [] { asm volatile("bar.sync 1, %0;" ::"n"(kCombHelpers) : "memory"); });
    }
    __syncthreads();
    const int warp = t >> 5, lane = t & 31;
    if (warp == 1) {          // B' = set 1 + set 2 - [s]G
        G1 q = {cp[2].v[0], cp[2].v[1], cp[2].v[2]};
        coop_add(&cp[1], q, lane);
        coop_add(&cp[1], s_sg[0].neg(), lane);
    }
    if (warp < 2 && lane == 0) { G1 r = {cp[warp].v[0], cp[warp].v[1], cp[warp].v[2]}; if (warp == 1) out->b = r; else out->a = r; }
    if (t == 0) { out->ry = Fr::zero(); out->err = s_err; }
    if (flag) {
        __threadfence_system();
        __syncthreads();
        if (t == 0) { *reinterpret_cast<volatile uint32_t*>(flag) = epoch; __threadfence_system(); }
    }
}

// the helpers' work of msm_combine_kernel on their own CTA (kCombHelpers threads), for the split tail: launched beside the bucket
// phase, it hands [s]G and the flags to window_miller_kernel off the critical path
__global__ void __launch_bounds__(kCombHelpers) msm_sg_kernel(const Fr* __restrict__ ry, const uint32_t* __restrict__ status, int n,
                                                              const DeviceTables* __restrict__ T, SplitTail* __restrict__ out) {
    __shared__ uint32_t s_err;
    __shared__ Fr s_ry[kCombHelpers];
    __shared__ G1 s_sg[64];
    const int t = threadIdx.x;
    if (t == 0) s_err = 0;
    __syncthreads();
    sum_s_sg(t, ry, status, n, T, &s_err, s_ry, s_sg, [] { __syncthreads(); });
    if (t == 0) { out->sg = s_sg[0]; out->err = s_err; }
}

}  // namespace kzgb200
