// Cooperative pairing engine, second generation: the level-scheduled programs of vliw29_programs.cuh over a shared-memory
// register file of 29-bit-limb values (fp29.cuh).  Same idea as vliw.cuh (a level = independent instructions, a barrier per
// level; reference src/pairings.rs:5-9 via src/kzg_proof.rs:436-441), different arithmetic and a different execution shape:
//
//   * values are SIGNED 14-limb numbers (limbs 0..12 in [-1, 2^29 + 1], limb 13 signed, |v| < 2^405) and ANY representative of
//     their residue: 2^406 = 2^25.3 p of headroom replaces the modular reduction after every sum; the bounds that make this
//     sound are tracked statically by tools/gen_vliw.py;
//   * ONE INSTRUCTION RUNS ON MANY LANES, not on one thread.  Measured on B200 (tools/microbench/lonewarp.cu): a lone warp issues
//     an IMAD.WIDE only every ~7 clocks however many lanes are active, so a one-thread Montgomery product (620 wide
//     multiplications) costs ~4200 clocks and a level of 36 of them leaves 32 lanes busy on two sub-partitions.
//       MUL  dst = (a b +- c d) / 2^406 : ONE WARP, lane k owns column k of the 28-column product: T_k = sum_s b_s a_(k-s) with b_s
//            broadcast and a_(k-s) a shuffle-rotation of the lane-resident limbs (lanes 14..31 hold zeros: the wrap-around is the
//            zero fill); two carry rounds; m = T_lo * (-p^-1) mod 2^406 and m * p the same way with the constants as immediates;
//            the low half of T + m p is an exact multiple of 2^406, so its carry into the high half is read off its top limb
//            without a ripple loop.  56 wide multiplications per lane and dual product, no shared-memory traffic but the operands;
//       LIN  dst = sum +-(1|2) src      : 16 lanes, lane j adds limb j of every term (32-bit multiply-adds on 16-bit halves: no wide
//            multiplication), two carry rounds; with the `reduce` flag round(v / p) p is subtracted first (float estimate from
//            the two top columns), leaving |v| < 4 p.
//   A 768-thread CTA runs 24 products or 48 sums at a time.
//
// The sequential executors (exec_*_ref, host + device) are the specification of the two instructions: the CPU unit test runs the
// pairing with them (tools/hosttest/vliw29_host.cu), the GPU unit test compares the 16-lane forms with them limb for limb.
#pragma once
#include "vliw.cuh"
#include "fp29.cuh"
#include "vliw29_programs.cuh"

namespace kzgb200 {
namespace vliw29 {
using f29::F29;
constexpr int32_t kM = (int32_t)f29::kMask;

struct Tables {
    const uint32_t (*mul)[4];
    const uint32_t (*lin)[4];
    const uint32_t* term;
    const Level* level;
    const Program* prog;
};
constexpr int kGroupLanes = 16;
struct Lanes {
    int tid, n;                   // this thread's index and the number of cooperating threads (host: 0, 1)
    Tables tab;
    long long* ticks = nullptr;   // optional: per-section clock64() stamps (profiling aid)
    const int32_t* p29s = nullptr;   // device: limbs of p, one per lane, in shared memory
    int groups = 1, gstride = 0;     // independent register files run in lockstep through the same program, gstride registers apart
    int bar_id = 0, bar_threads = 0; // != 0: the cooperating threads are a subset of the CTA and meet at this named barrier
    KZG_HD void tick(int i) const {
#ifdef __CUDA_ARCH__
        if (ticks && tid == 0) ticks[i] = clock64();
#endif
    }
    KZG_HD void sync() const {
#ifdef __CUDA_ARCH__
        if (bar_threads) asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
        else __syncthreads();
#endif
    }
};
KZG_HD Tables default_tables() {
#ifdef __CUDA_ARCH__
    return Tables{d_mul, d_lin, d_term, d_level, d_prog};
#else
    return Tables{h_mul, h_lin, h_term, h_level, h_prog};
#endif
}
struct SharedTables {
    uint32_t mul[kNumMul][4];
    uint32_t lin[kNumLin][4];
    uint32_t term[kNumTerm];
    Level level[kNumLevel];
    Program prog[kNumPrograms];
    int32_t p29[16];              // limbs of p, one per lane (lanes 14, 15: 0)
};
#ifdef __CUDACC__
__device__ __forceinline__ Tables load_tables(SharedTables* st, int tid, int n) {
    const Tables src = default_tables();
    for (int i = tid; i < kNumMul * 4; i += n) (&st->mul[0][0])[i] = (&src.mul[0][0])[i];
    for (int i = tid; i < kNumLin * 4; i += n) (&st->lin[0][0])[i] = (&src.lin[0][0])[i];
    for (int i = tid; i < kNumTerm; i += n) st->term[i] = src.term[i];
    for (int i = tid; i < kNumLevel; i += n) st->level[i] = src.level[i];
    for (int i = tid; i < kNumPrograms; i += n) st->prog[i] = src.prog[i];
    if (tid < 16) st->p29[tid] = tid < 14 ? (int32_t)f29::p29_rt(tid) : 0;
    __syncthreads();
    return Tables{st->mul, st->lin, st->term, st->level, st->prog};
}
#endif

// Frobenius coefficients xi^(k(p-1)/6), k = 1..5, (c0, c1) each, in the engine's representation
#define KZG29_FROB_TABLE {KZG29_FROB6_1_C0, KZG29_FROB6_1_C1, KZG29_FROB6_2_C0, KZG29_FROB6_2_C1, KZG29_FROB6_3_C0, KZG29_FROB6_3_C1, \
                          KZG29_FROB6_4_C0, KZG29_FROB6_4_C1, KZG29_FROB6_5_C0, KZG29_FROB6_5_C1}
#ifdef __CUDACC__
static __device__ const uint32_t d_frob29[10][14] = KZG29_FROB_TABLE;
#endif
KZG_HD F29 frob_const(int i) {
    F29 r;
#ifdef __CUDA_ARCH__
    for (int k = 0; k < 14; k++) r.l[k] = d_frob29[i][k];
#else
    static const uint32_t h[10][14] = KZG29_FROB_TABLE;
    for (int k = 0; k < 14; k++) r.l[k] = h[i][k];
#endif
    r.l[14] = r.l[15] = 0;
    return r;
}

// ------------------------------------------------------------------------------------------ sequential reference executors
// t[] = signed 64-bit column sums of a 14-limb number -> limbs 0..12 in [0, 2^29), limb 13 = the (signed) rest
KZG_HD void normalize_ref(F29& r, int64_t* t) {
    for (int i = 0; i < 13; i++) { r.l[i] = (uint32_t)t[i] & f29::kMask; t[i + 1] += t[i] >> 29; }
    r.l[13] = (uint32_t)t[13]; r.l[14] = 0; r.l[15] = 0;
}
KZG_HD int32_t limb(const F29& v, int i) { return (int32_t)v.l[i]; }
// MUL row: {dst | a << 16, b | c << 16, d | flags << 16, 0}; flags bit 0 = dual product, bit 1 = the second product is subtracted
KZG_NI void exec_mul_ref(F29* regs, const uint32_t* ins) {
    const uint32_t w0 = ins[0], w1 = ins[1], w2 = ins[2];
    const bool dual = (w2 >> 16) & 1u, neg = (w2 >> 17) & 1u;
    const F29 a = regs[w0 >> 16], b = regs[w1 & 0xffffu];
    int64_t t[29];
    for (int k = 0; k < 29; k++) t[k] = 0;
    for (int i = 0; i < 14; i++) for (int j = 0; j < 14; j++) t[i + j] += (int64_t)limb(a, i) * limb(b, j);
    if (dual) {
        const F29 c = regs[w1 >> 16], d = regs[w2 & 0xffffu];
        for (int i = 0; i < 14; i++) for (int j = 0; j < 14; j++) t[i + j] += (int64_t)(neg ? -limb(c, i) : limb(c, i)) * limb(d, j);
    }
    for (int k = 0; k < 28; k++) { int64_t c = t[k] >> 29; t[k] &= f29::kMask; t[k + 1] += c; }    // exact 29-limb form (t[28] = signed rest)
    for (int i = 0; i < 14; i++) {
        int64_t m = (int64_t)(((uint32_t)t[i] * KZG29_PINV) & f29::kMask);
        for (int j = 0; j < 14; j++) t[i + j] += m * (int64_t)f29::p29_rt(j);
        t[i + 1] += t[i] >> 29;            // t[i] is now a multiple of 2^29
    }
    t[27] += t[28] << 29;
    F29 r;
    normalize_ref(r, t + 14);
    regs[w0 & 0xffffu] = r;
}
// LIN row: {dst, first term, term count, reduce}; a term = byte offset of the source register (reg * 64) | coefficient << 16
KZG_NI void exec_lin_ref(F29* regs, const uint32_t* ins, const uint32_t* terms) {
    int64_t t[14];
    for (int i = 0; i < 14; i++) t[i] = 0;
    for (uint32_t k = 0; k < ins[2]; k++) {
        const uint32_t e = terms[ins[1] + k];
        const F29& v = regs[(e & 0xffffu) >> 6];
        const int32_t coef = (int32_t)e >> 16;
        for (int i = 0; i < 14; i++) t[i] += (int64_t)limb(v, i) * coef;
    }
    if (ins[3] & 1u) {
        // |v| < 2^20 p: quotient estimate from the two top columns in float (relative error ~2^-22: off by less than 1)
        const float vf = (float)t[13] * 536870912.0f + (float)t[12];
        const float pinv = 1.0f / ((float)f29::p29_rt(13) * 536870912.0f + (float)f29::p29_rt(12));
        const int32_t q = (int32_t)rintf(vf * pinv);
        for (int i = 0; i < 14; i++) t[i] -= (int64_t)f29::p29_rt(i) * q;
    }
    F29 r;
    normalize_ref(r, t);
    regs[ins[0]] = r;
}

// ------------------------------------------------------------------------------------------ 16-lane executors (device)
#ifdef __CUDACC__
constexpr unsigned kFull = 0xffffffffu;
__device__ __forceinline__ int32_t up(int32_t v, int d, int lane) { int32_t r = __shfl_up_sync(kFull, v, d, kGroupLanes); return lane < d ? 0 : r; }
__device__ __forceinline__ int32_t from(int32_t v, int src) { return __shfl_sync(kFull, v, src, kGroupLanes); }
// Two carry rounds over a 14-limb number given as signed 64-bit column sums (lane j: column j; lanes 14, 15: zero), lane 13
// holding everything above bit 377 (the value's true top limb fits 32 bits).  Result limbs 0..12 in [-1, 2^29 + 1].
__device__ __forceinline__ int32_t carry_top(int64_t t, int lane) {
    const bool top = lane >= 13;
    const int64_t c64 = t >> 29;
    int32_t low = top ? (int32_t)t : ((int32_t)t & kM);
    int32_t cmid = top ? 0 : (lane == 12 ? (int32_t)c64 : ((int32_t)c64 & kM));     // lane 12 hands its whole carry to the top limb
    int32_t chi = (top || lane == 12) ? 0 : (int32_t)(t >> 58);
    int32_t l = low + up(cmid, 1, lane) + up(chi, 2, lane);
    int32_t c = top ? 0 : (l >> 29);
    l = top ? l : (l & kM);
    return l + up(c, 1, lane);
}
// ---- MUL on one warp: lane k owns column k of the 28-column product (lanes 28..31 idle) -----------------------------------
// T_k = sum_s b_s a_(k-s): b_s is the same for every lane (broadcast load), a_(k-s) is lane k-s's limb -- a rotation of the lane-
// resident operand by s, one shuffle, with lanes 14..31 holding zeros so that the wrap-around brings the zero fill.  No shared-
// memory traffic beyond the operand loads, no lo/hi bookkeeping; m = T_lo (-p^-1) mod 2^406 and m p use the same rotation with the
// constants as immediates.  (Round 2 first ran a MUL on 16 lanes with the rows summed by columns through a shared-memory
// scratch: 12.5 KB of traffic per product made a 36-product level wait ~3500 clocks for the SM's shared-memory port.)
__device__ __forceinline__ int64_t mulw(int32_t a, int32_t b) { uint64_t r = 0; f29::madw_s(r, a, b); return (int64_t)r; }
__device__ __forceinline__ int32_t up32(int32_t v, int d, int k) { int32_t r = __shfl_up_sync(kFull, v, d); return k < d ? 0 : r; }
__device__ __forceinline__ int32_t rot(int32_t v, int k, int s) { return __shfl_sync(kFull, v, (k - s) & 31); }
// two carry rounds over lanes 0..nlow-1 (all of them carry out); the lanes above receive the outgoing carries into their 64-bit
// column t.  Returns the limb (lanes < nlow; 0 above).
__device__ __forceinline__ int32_t carry_split(int64_t& t, int k, int nlow) {
    const bool lowlane = k < nlow;
    const int32_t low = lowlane ? ((int32_t)t & kM) : 0, cmid = lowlane ? ((int32_t)(t >> 29) & kM) : 0, chi = lowlane ? (int32_t)(t >> 58) : 0;
    const int32_t u1 = up32(cmid, 1, k), u2 = up32(chi, 2, k);
    int32_t l = low + u1 + u2;
    if (!lowlane) t += (int64_t)u1 + (int64_t)u2;
    const int32_t c = lowlane ? (l >> 29) : 0;
    const int32_t u = up32(c, 1, k);
    l = lowlane ? ((l & kM) + u) : 0;
    if (!lowlane) t += (int64_t)u;
    return l;
}
// two carry rounds over the 28 columns of lanes 0..27, lane 27 keeping everything above (the true top limb fits 32 bits)
__device__ __forceinline__ int32_t carry_full(int64_t t, int k) {
    const bool top = k >= 27;
    const int64_t c64 = t >> 29;
    const int32_t low = top ? (int32_t)t : ((int32_t)t & kM);
    const int32_t cmid = top ? 0 : (k == 26 ? (int32_t)c64 : ((int32_t)c64 & kM));
    const int32_t chi = (top || k == 26) ? 0 : (int32_t)(t >> 58);
    int32_t l = low + up32(cmid, 1, k) + up32(chi, 2, k);
    const int32_t c = top ? 0 : (l >> 29);
    l = top ? l : (l & kM);
    return l + up32(c, 1, k);
}
__device__ __forceinline__ void exec_mul32(F29* regs, const uint32_t* ins, int k) {
    const uint32_t w0 = ins[0], w1 = ins[1], w2 = ins[2];
    const bool dual = (w2 >> 16) & 1u, neg = (w2 >> 17) & 1u;
    uint64_t acc = 0, acc1 = 0;           // two accumulators: the wide multiply-adds of a column do not form one dependency chain
    {
        const int32_t av = k < 16 ? reinterpret_cast<const int32_t*>(regs[w0 >> 16].l)[k] : 0;      // limbs 14, 15 are zero padding
        const int4* B = reinterpret_cast<const int4*>(regs[w1 & 0xffffu].l);
        const int4 b0 = B[0], b1 = B[1], b2 = B[2], b3 = B[3];
        const int32_t bb[14] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w, b2.x, b2.y, b2.z, b2.w, b3.x, b3.y};
#pragma unroll
        for (int s = 0; s < 14; s++) f29::madw_s((s & 1) ? acc1 : acc, rot(av, k, s), bb[s]);
    }
    if (dual) {
        int32_t cv = k < 16 ? reinterpret_cast<const int32_t*>(regs[w1 >> 16].l)[k] : 0;
        if (neg) cv = -cv;
        const int4* D = reinterpret_cast<const int4*>(regs[w2 & 0xffffu].l);
        const int4 d0 = D[0], d1 = D[1], d2 = D[2], d3 = D[3];
        const int32_t dd[14] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w, d2.x, d2.y, d2.z, d2.w, d3.x, d3.y};
#pragma unroll
        for (int s = 0; s < 14; s++) f29::madw_s((s & 1) ? acc1 : acc, rot(cv, k, s), dd[s]);
    }
    // low half: limbs for m; its carries move into columns 14, 15
    int64_t hi = (int64_t)(acc + acc1);
    const int32_t tl = carry_split(hi, k, 14);
    // m = T_lo * (-p^-1) mod 2^406
    uint64_t mc = 0, mc1 = 0;
    {
        constexpr uint32_t pinv[14] = KZG29_PINV_FULL;
#pragma unroll
        for (int s = 0; s < 14; s++) f29::madw_s((s & 1) ? mc1 : mc, rot(tl, k, s), (int32_t)pinv[s]);
    }
    int64_t mcol = k < 14 ? (int64_t)(mc + mc1) : 0;         // columns beyond 13 are multiples of 2^406: dropped
    int32_t m = carry_split(mcol, k, 14);
    if (k == 13) m &= kM;
    // T + m p: the low half becomes an exact multiple of 2^406 (-2^406, 0 or 2^406 after the carry rounds, told apart by limb 13)
    uint64_t mp = 0, mp1 = 0;
    {
        constexpr uint32_t pp[14] = KZG29_P;
#pragma unroll
        for (int s = 0; s < 14; s++) f29::madw_s((s & 1) ? mp1 : mp, rot(m, k, s), (int32_t)pp[s]);
    }
    const int64_t tot = (k < 14 ? (int64_t)tl : hi) + (int64_t)(mp + mp1);
    int32_t r = carry_full(tot, k);
    const int32_t z13 = __shfl_sync(kFull, r, 13);
    if (k == 14) r += (z13 + (1 << 28)) >> 29;
    if (k >= 14 && k < 30) reinterpret_cast<int32_t*>(regs[w0 & 0xffffu].l)[k - 14] = k < 28 ? r : 0;   // lanes 28, 29: the zero padding
}
__device__ __forceinline__ void exec_lin16(F29* regs, const uint32_t* ins, const uint32_t* terms, bool active, const int32_t* p29s, int lane) {
    // limb sums on 16-bit halves (48 units of 2^29 overflow 32 bits): two 32-bit multiply-adds per term, no wide multiplication
    int32_t sl = 0, sh = 0;
    const uint32_t* tt = terms + ins[1];
    const uint32_t count = ins[2];
    const unsigned char* base = reinterpret_cast<const unsigned char*>(regs) + 4 * lane;
#pragma unroll 4
    for (uint32_t k = 0; k < count; k++) {
        const uint32_t e = tt[k];
        const int32_t v = *reinterpret_cast<const int32_t*>(base + (e & 0xffffu));
        const int32_t coef = (int32_t)e >> 16;
        sl += (v & 0xffff) * coef;
        sh += (v >> 16) * coef;
    }
    int64_t t = (int64_t)sl + ((int64_t)sh << 16);
    if (__any_sync(kFull, ins[3] & 1u)) {   // warp-uniform test: the two groups of a warp may run instructions with different flags
        const float f = lane == 13 ? (float)t * 536870912.0f : (lane == 12 ? (float)t : 0.0f);
        const float vf = __shfl_sync(kFull, f, 13, kGroupLanes) + __shfl_sync(kFull, f, 12, kGroupLanes);
        if (ins[3] & 1u) {
            const float pinv = 1.0f / ((float)f29::p29_rt(13) * 536870912.0f + (float)f29::p29_rt(12));
            const int32_t q = (int32_t)rintf(vf * pinv);
            t -= mulw(p29s[lane], q);
        }
    }
    const int32_t r = carry_top(t, lane);
    if (active) reinterpret_cast<int32_t*>(regs[ins[0]].l)[lane] = r;
}
#endif

// run one program; every cooperating thread must call it (barriers inside).  Force-inlined: the pairing is driven by ONE interpreter
// loop (run_script), so the executors exist once in the kernel and see the shared-memory address space of their operands.
KZG_HD void run(int prog, F29* regs, const Lanes& L) {
    const Program p = L.tab.prog[prog];
    for (int lv = p.first_level; lv < p.first_level + p.n_levels; lv++) {
        const Level lev = L.tab.level[lv];
#ifdef __CUDA_ARCH__
        long long c0 = L.ticks ? clock64() : 0;
        const int total = lev.count * L.groups;                   // instruction instances: (instruction k, register file g)
        if (lev.kind == 1) {
            // one product per warp; a level of more products than warps runs in balanced passes (36 on 24 warps: 18 + 18)
            const int w = L.tid >> 5, nw = L.n >> 5;
            const int passes = (total + nw - 1) / nw, per = (total + passes - 1) / passes;
            if (w < per)
                for (int i = w; i < total; i += per) {
                    const int k = L.groups == 1 ? i : i / L.groups, g = i - k * L.groups;
                    exec_mul32(regs + g * L.gstride, L.tab.mul[lev.first + k], L.tid & 31);
                }
        } else {
            const int slot = L.tid >> 4, nslots = L.n >> 4, lane = L.tid & 15;
            for (int base = 0; base < total; base += nslots) {
                const int i = base + slot;
                if (base + (slot & ~1) >= total) break;               // neither group of this warp has an instruction left (warp-uniform)
                const bool active = i < total;                        // an idle second group runs along: the shuffles need every lane
                const int ii = active ? i : base, k = L.groups == 1 ? ii : ii / L.groups, g = ii - k * L.groups;
                exec_lin16(regs + g * L.gstride, L.tab.lin[lev.first + k], L.tab.term, active, L.p29s, lane);
            }
        }
        long long c1 = L.ticks ? clock64() : 0;
#else
        for (int g = 0; g < L.groups; g++) {
            if (lev.kind == 1) { for (int k = 0; k < lev.count; k++) exec_mul_ref(regs + g * L.gstride, L.tab.mul[lev.first + k]); }
            else { for (int k = 0; k < lev.count; k++) exec_lin_ref(regs + g * L.gstride, L.tab.lin[lev.first + k], L.tab.term); }
        }
#endif
        L.sync();
#ifdef __CUDA_ARCH__
        if (L.ticks && L.tid == 0) {   // profiling aid: body / barrier-wait cycles of thread 0 per level kind
            long long c2 = clock64();
            int b = lev.kind == 1 ? 10 : 8;
            L.ticks[b] += c1 - c0; L.ticks[b + 1] += c2 - c1; L.ticks[b == 10 ? 13 : 12] += 1;
        }
#endif
    }
}
// the same program on the sequential executors, one thread (GPU unit test of the 16-lane forms)
KZG_NI void run_ref(int prog, F29* regs, const Tables& tab) {
    const Program p = tab.prog[prog];
    for (int lv = p.first_level; lv < p.first_level + p.n_levels; lv++) {
        const Level lev = tab.level[lv];
        if (lev.kind == 1) { for (int k = 0; k < lev.count; k++) exec_mul_ref(regs, tab.mul[lev.first + k]); }
        else { for (int k = 0; k < lev.count; k++) exec_lin_ref(regs, tab.lin[lev.first + k], tab.term); }
    }
}
// regs[dst .. dst+count) = regs[src ..)   (16-byte words)
KZG_HD void copy_regs(F29* regs, int dst, int src, int count, const Lanes& L) {
    uint4* d = reinterpret_cast<uint4*>(regs + dst);
    const uint4* s = reinterpret_cast<const uint4*>(regs + src);
    for (int j = L.tid; j < count * 4; j += L.n) d[j] = s[j];
    L.sync();
}

// Line tables in the engine's representation: per fixed G2 point, per Miller step, (A, B, C) as 6 values (setup: k_setup.cu)
struct LineCoeffs29 { F29 v[6]; };
KZG_HD void load_lines(F29* regs, const LineCoeffs29* c1, const LineCoeffs29* c2, int k, const Lanes& L) {
    uint4* d = reinterpret_cast<uint4*>(regs + kRegLines);
    for (int q = L.tid; q < 2 * 6 * 4; q += L.n) {
        const LineCoeffs29* src = q < 24 ? c1 : c2;
        if (!src) continue;
        d[q] = reinterpret_cast<const uint4*>(src[k].v)[q < 24 ? q : q - 24];
    }
    L.sync();
}

// any register value (signed, |v| < bound p) -> the canonical integer of the field element it stands for
KZG_NI Fp canonical_signed(const F29& v, int bound = kIoBound) {
    int64_t t[14];
    for (int i = 0; i < 14; i++) t[i] = (int64_t)limb(v, i) + (int64_t)bound * (int64_t)f29::p29_rt(i);
    F29 u;
    normalize_ref(u, t);                        // now non-negative, limbs in [0, 2^29)
    return f29::canonical(u);
}
// v^-1 (both in the engine's representation); v != 0 mod p
KZG_NI F29 inv29(const F29& v) {
    Fp x = canonical_signed(v), y;
    vliw::fp_inv_raw(y.l, x.l);
    return f29::from_raw(y);
}

constexpr int kSave0 = kMaxRegs;            // each save slot = 12 registers (the scripts of tools/gen_vliw.py use the same layout)
constexpr int kNumSaves = 5;
constexpr int kTotalRegs = kMaxRegs + 12 * kNumSaves;

// The engine steps of a generated script (vliw29_programs.cuh): run a program, copy an Fp12 slot, load the lines of Miller step a
// (ca: slot-0 pair, cb: slot-1 pair, nullptr = none), invert one register, stamp a profiling tick.
KZG_HD void run_script(F29* regs, const uint32_t* script, int n_steps, const LineCoeffs29* ca, const LineCoeffs29* cb, const Lanes& L) {
    for (int s = 0; s < n_steps; s++) {
        const uint32_t w = script[s];
        const int op = (int)(w & 0xffu), a = (int)((w >> 8) & 0xfffu), b = (int)(w >> 20);
#ifdef __CUDA_ARCH__
        const long long s0 = L.ticks ? clock64() : 0;
#endif
        if (op == kOpRun) run(a, regs, L);
        else if (op == kOpCopy) copy_regs(regs, a, b, 12, L);
        else if (op == kOpLines) load_lines(regs, ca, cb, a, L);
        else if (op == kOpInv) { if (L.tid == 0) regs[kRegH + 8] = inv29(regs[kRegH + 8]); L.sync(); }
        else L.tick(a);
#ifdef __CUDA_ARCH__
        if (L.ticks && L.tid == 0 && (op == kOpCopy || op == kOpLines)) L.ticks[op == kOpCopy ? 6 : 7] += clock64() - s0;   // profiling aid
#endif
    }
}
// Miller loop of e(P1, Q1) e(P2, Q2) with the lines of Q1, Q2 precomputed (c1, c2): leaves prod f_{|x|,Q_i}(P_i), conjugated, in
// the F slot (registers kRegF..+11) and the Frobenius constants in kRegConst.  Pairs whose P is the identity contribute 1.
KZG_HD void coop_miller(F29* regs, const G1Affine& P1, const LineCoeffs29* c1, const G1Affine& P2, const LineCoeffs29* c2, const Lanes& L) {
    const bool live1 = !P1.inf, live2 = !P2.inf;
    const G1Affine& Pa = live1 ? P1 : P2;       // with a single live pair it takes slot 0
    const LineCoeffs29* ca = live1 ? c1 : c2;
    const LineCoeffs29* cb = (live1 && live2) ? c2 : nullptr;
    for (int i = L.tid; i < 26; i += L.n) {
        if (i < 10) regs[kRegConst + i] = frob_const(i);
        else if (i < 14) {
            const int j = i - 10;
            if (j < 2) regs[kRegP + j] = f29::from_fp(j == 0 ? Pa.x : Pa.y);
            else regs[kRegP + j] = cb ? f29::from_fp(j == 2 ? P2.x : P2.y) : f29::f29_zero();
        } else regs[kRegF + (i - 14)] = i == 14 ? f29::f29_one() : f29::f29_zero();
    }
    L.sync();
    if (!live1 && !live2) return;
#ifdef __CUDA_ARCH__
    run_script(regs, cb ? d_miller2 : d_miller1, cb ? kLen_miller2 : kLen_miller1, ca, cb, L);
#else
    run_script(regs, cb ? h_miller2 : h_miller1, cb ? kLen_miller2 : kLen_miller1, ca, cb, L);
#endif
}
// F slot == 1 ?  (each coefficient canonicalised by its own thread; the verdict words land in the padding of the G slot).
// gt (nullable): the 12 coefficients as canonical integers (c0.c0.c0, c0.c0.c1, ...: the register order of the F slot).
KZG_HD bool f_is_one(F29* regs, const Lanes& L, Fp* gt = nullptr) {
    for (int i = L.tid; i < 12; i += L.n) {
        Fp x = canonical_signed(regs[kRegF + i]);
        if (gt) gt[i] = x;
        bool good = i == 0 ? (x.l[0] == 1u) : (x.l[0] == 0u);
        for (int w = 1; w < 12; w++) good = good && x.l[w] == 0u;
        regs[kRegG + i].l[15] = good ? 1u : 0u;
    }
    L.sync();
    bool ok = true;
    for (int i = 0; i < 12; i++) ok = ok && regs[kRegG + i].l[15] == 1u;
    L.sync();
    for (int i = L.tid; i < 12; i += L.n) regs[kRegG + i].l[15] = 0;
    L.sync();
    return ok;
}
// final exponentiation f^(3(p^12-1)/r) of the F slot (Frobenius constants in kRegConst), then == 1 ?  Same verdict to all threads.
KZG_HD bool coop_final_exp_is_one(F29* regs, const Lanes& L, Fp* gt = nullptr) {
#ifdef __CUDA_ARCH__
    run_script(regs, d_final_exp, kLen_final_exp, nullptr, nullptr, L);
#else
    run_script(regs, h_final_exp, kLen_final_exp, nullptr, nullptr, L);
#endif
    return f_is_one(regs, L, gt);
}

// e(P1, Q1) e(P2, Q2) == 1 with the lines of Q1, Q2 precomputed (c1, c2).  All cooperating threads call it with the same
// arguments; returns the same verdict to all.  regs: kTotalRegs values shared by the threads.  The sequence of engine steps
// (Miller loop, final exponentiation) is the generated script (vliw29_programs.cuh: script2 = both pairs live, script1 = one).
KZG_HD bool coop_pairing_product_is_one(F29* regs, const G1Affine& P1, const LineCoeffs29* c1, const G1Affine& P2, const LineCoeffs29* c2,
                                        const Lanes& L, Fp* gt = nullptr) {
    const bool live1 = !P1.inf, live2 = !P2.inf;
    if (!live1 && !live2) {
        if (gt) for (int i = L.tid; i < 12; i += L.n) { Fp x = Fp::zero(); x.l[0] = i == 0 ? 1u : 0u; gt[i] = x; }
        return true;
    }
    const G1Affine& Pa = live1 ? P1 : P2;       // with a single live pair it takes slot 0
    const LineCoeffs29* ca = live1 ? c1 : c2;
    const LineCoeffs29* cb = (live1 && live2) ? c2 : nullptr;
    for (int i = L.tid; i < 26; i += L.n) {
        if (i < 10) regs[kRegConst + i] = frob_const(i);
        else if (i < 14) {
            const int j = i - 10;
            if (j < 2) regs[kRegP + j] = f29::from_fp(j == 0 ? Pa.x : Pa.y);
            else regs[kRegP + j] = cb ? f29::from_fp(j == 2 ? P2.x : P2.y) : f29::f29_zero();
        } else regs[kRegF + (i - 14)] = i == 14 ? f29::f29_one() : f29::f29_zero();
    }
    L.sync();
#ifdef __CUDA_ARCH__
    run_script(regs, cb ? d_script2 : d_script1, cb ? kLen_script2 : kLen_script1, ca, cb, L);
#else
    run_script(regs, cb ? h_script2 : h_script1, cb ? kLen_script2 : kLen_script1, ca, cb, L);
#endif
    return f_is_one(regs, L, gt);
}

}  // namespace vliw29
}  // namespace kzgb200
