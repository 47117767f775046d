// K7: final pairing check of a batch: G1 prelude kernel + the cooperative pairing engine kernel.
#include "common.cuh"
#include "coop.cuh"

namespace kzgb200 {

// Prelude of the final check over the gathered per-rank partials (reference src/kzg_proof.rs:436-441):
//   e(sum_k A_k, [tau]G2) == e(sum_k B_k - [sum_k s_k]G, G2)
// one CTA of kFinalThreads threads forms the two affine G1 arguments (-A, B - [s]G) and hands them to pairing_check_kernel.
// result: 0 = false, 1 = true, 2 = BadArgs (some rank flagged an unparsable input)
__global__ void __launch_bounds__(kFinalThreads) batch_final_kernel(const Partial* __restrict__ parts, int nparts, const DeviceTables* __restrict__ T,
                                                                    uint32_t* __restrict__ result, FinalPts* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    FinalSmem& S = *reinterpret_cast<FinalSmem*>(dyn_smem);
    G1* sm = S.sm;
    __shared__ Fr s_sum;
    __shared__ uint32_t s_err;
    int t = threadIdx.x;
    if (t == 0) result[2] = 0;
    if (t == 0) {
        Fr s = Fr::zero(); uint32_t err = 0;
        for (int k = 0; k < nparts; k++) { s = s.add_inl(parts[k].ry); err |= parts[k].err; }
        s_sum = s; s_err = err;
    }
    __syncthreads();
    if (s_err) { if (t == 0) { result[0] = kBadArgs; result[1] = s_err; out->go = 0; } return; }
    G1 sg = G1::identity();
    if (!s_sum.is_zero()) sg = coop_fixed_base_mul(s_sum, T, sm);      // zero on the batch path: msm_combine_kernel folded - [s]G into b
    if ((t & 31) == 0) {     // lane 0 of warp 0 and of warp 1: the two data-dependent inversion loops run side by side, not serialised
        int w = t >> 5;
        G1 acc = G1::identity();
        for (int k = 0; k < nparts; k++) acc = acc.add(w == 0 ? parts[k].a : parts[k].b);
        if (w == 1) acc = acc.add(sg.neg());
        Fp zi = vliw::fp_inv_bingcd(acc.z), zi2 = zi.sqr();
        G1Affine a = acc.is_identity() ? G1Affine{Fp::zero(), Fp::zero(), 1} : G1Affine{acc.x * zi2, acc.y * zi2 * zi, 0};
        if (w == 0 && !a.inf) a.y = a.y.neg();     // -A
        out->pts[w] = a;
        if (w == 0) out->go = 1;
    }
}

// e(pts[1], G2) e(pts[0], Q) == 1 on the cooperative engine (vliw29.cuh): kPairThreads threads = 24 warps.  Q = [tau]G2, or the
// point whose line table lines_b is (cell proofs: [tau^64]G2).
__global__ void __launch_bounds__(kPairThreads) pairing_check_kernel(const FinalPts* __restrict__ in, const DeviceTables* __restrict__ T,
                                                                     const vliw29::LineCoeffs29* __restrict__ lines_b, uint32_t* __restrict__ result,
                                                                     long long* __restrict__ ticks, Fp* __restrict__ gt) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    PairSmem& S = *reinterpret_cast<PairSmem*>(dyn_smem);
    const int t = threadIdx.x;
    if (in->go == 0) return;            // the prelude already wrote the result
    if (ticks && t == 0) { ticks[0] = clock64(); for (int i = 6; i < 14; i++) ticks[i] = 0; }
    vliw29::Tables tab = vliw29::load_tables(&S.stab, t, kPairThreads);
    vliw29::Lanes L{t, kPairThreads, tab, ticks, S.stab.p29};
    const G1Affine p0 = in->pts[0], p1 = in->pts[1];
    bool ok = vliw29::coop_pairing_product_is_one(S.regs, p1, T->lines29[0], p0, lines_b ? lines_b : T->lines29[1], L, gt);
    L.tick(5);
    if (t == 0) { result[0] = ok ? kTrue : kFalse; result[1] = 0; }
}

// Split tail of a single-GPU batch (kzgb200_ctx::final_split).  With A = sum_w 256^w W0_w and B = sum_w 256^w B_w (W*_w: the
// MSM window sums of the three point sets, B_w = W1_w + W2_w, B_0 also - [s]G), bilinearity gives
//   e(-A, [tau]G2) e(B, G2) = prod_w e(-W0_w, [256^w tau]G2) e(B_w, [256^w]G2),
// and the final exponentiation is a homomorphism, so FE(prod_w Miller_w) is the very GT element of the combined check.  The G2
// multiples are setup constants (lines29w), so the Horner chain of msm_combine_kernel (120 doublings + 16 additions) leaves the
// critical path: window_prelude_kernel forms every window's two affine points, CTA w of window_miller_kernel runs its Miller loop,
// split_final_kernel multiplies the 16 values and runs the final exponentiation.
// Prelude: one CTA of kFinalThreads threads per window (a kernel of its own, as batch_final_kernel: the G1 sums and the inversion
// inside the 768-thread engine kernel would spill); lane 0 of warps 0 and 1 run the two inversions side by side.
__global__ void __launch_bounds__(kFinalThreads) window_prelude_kernel(const G1* __restrict__ windows, SplitTail* __restrict__ io) {
    const int t = threadIdx.x, w = blockIdx.x;
    if (io->err || (t & 31) != 0) return;         // BadArgs: split_final_kernel writes the result
    const int k = t >> 5;
    G1 acc;
    if (k == 0) acc = windows[w].neg();                                       // -W0_w
    else {
        acc = windows[kWindows + w].add(windows[2 * kWindows + w]);           // B_w
        if (w == 0) acc = acc.add(io->sg.neg());
    }
    Fp zi = vliw::fp_inv_bingcd(acc.z), zi2 = zi.sqr();
    io->pts[w][k] = acc.is_identity() ? G1Affine{Fp::zero(), Fp::zero(), 1} : G1Affine{acc.x * zi2, acc.y * zi2 * zi, 0};
}
// Miller loop of window w = blockIdx.x on the lines of [256^w]G2 and [256^w tau]G2 (one-pair script for an identity point, f = 1
// for two).  ticks (profiling, nullable): ticks[2] receives the longest Miller time over the CTAs (split_final_kernel rebases it).
__global__ void __launch_bounds__(kPairThreads) window_miller_kernel(const DeviceTables* __restrict__ T, SplitTail* __restrict__ io,
                                                                     long long* __restrict__ ticks) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    PairSmem& S = *reinterpret_cast<PairSmem*>(dyn_smem);
    const int t = threadIdx.x, w = blockIdx.x;
    if (io->err) return;
    const long long c0 = clock64();
    vliw29::Tables tab = vliw29::load_tables(&S.stab, t, kPairThreads);
    vliw29::Lanes L{t, kPairThreads, tab, nullptr, S.stab.p29};
    const vliw29::LineCoeffs29* lg = w ? T->lines29w[0][w - 1] : T->lines29[0];
    const vliw29::LineCoeffs29* lt = w ? T->lines29w[1][w - 1] : T->lines29[1];
    vliw29::coop_miller(S.regs, io->pts[w][1], lg, io->pts[w][0], lt, L);
    uint4* dst = reinterpret_cast<uint4*>(io->f[w]);
    const uint4* src = reinterpret_cast<const uint4*>(S.regs + vliw29::kRegF);
    for (int i = t; i < 12 * 4; i += kPairThreads) dst[i] = src[i];
    if (ticks && t == 0) atomicMax(&ticks[2], clock64() - c0);
}
// product of the 16 window Miller values (15 f12_mul in a row: the program has 3 levels, a 4-level tree over 8 register files
// would run more passes of its wider levels than it saves), final exponentiation, == 1.  Same result words as pairing_check_kernel.
__global__ void __launch_bounds__(kPairThreads) split_final_kernel(const SplitTail* __restrict__ io, uint32_t* __restrict__ result, Fp* __restrict__ gt,
                                                                   long long* __restrict__ ticks) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    PairSmem& S = *reinterpret_cast<PairSmem*>(dyn_smem);
    const int t = threadIdx.x;
    if (io->err) { if (t == 0) { result[0] = kBadArgs; result[1] = io->err; } return; }
    if (ticks && t == 0) {              // stamps on this SM's clock: the longest window Miller loop ends at this start
        const long long c0 = clock64(), mil = ticks[2];
        ticks[0] = c0 - mil; ticks[1] = c0 - mil; ticks[2] = c0;
        for (int i = 6; i < 14; i++) ticks[i] = 0;
    }
    vliw29::Tables tab = vliw29::load_tables(&S.stab, t, kPairThreads);
    vliw29::Lanes L{t, kPairThreads, tab, ticks, S.stab.p29};
    {
        uint4* dst = reinterpret_cast<uint4*>(S.regs + vliw29::kRegF);
        const uint4* src = reinterpret_cast<const uint4*>(io->f[0]);
        for (int i = t; i < 12 * 4; i += kPairThreads) dst[i] = src[i];
        for (int i = t; i < 10; i += kPairThreads) S.regs[vliw29::kRegConst + i] = vliw29::frob_const(i);
    }
    for (int w = 1; w < kWindows; w++) {
        uint4* dst = reinterpret_cast<uint4*>(S.regs + vliw29::kRegG);
        const uint4* src = reinterpret_cast<const uint4*>(io->f[w]);
        for (int i = t; i < 12 * 4; i += kPairThreads) dst[i] = src[i];
        L.sync();
        vliw29::run(vliw29::kProg_f12_mul, S.regs, L);      // F <- F * G
    }
    L.sync();
    const bool ok = vliw29::coop_final_exp_is_one(S.regs, L, gt);
    L.tick(5);
    if (t == 0) { result[0] = ok ? kTrue : kFalse; result[1] = 0; }
}

// Self-test of the 16-lane executors against the sequential reference executors (kzgb200_debug_engine_selftest): the same
// programs on two register files seeded alike; after every program all registers are compared as canonical field elements
// (the two forms may leave different representatives of the same residue).
__global__ void __launch_bounds__(kPairThreads) engine_selftest_kernel(uint32_t seed, int rounds, f29::F29* __restrict__ ref, uint32_t* __restrict__ mismatches) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    PairSmem& S = *reinterpret_cast<PairSmem*>(dyn_smem);
    const int t = threadIdx.x;
    vliw29::Tables tab = vliw29::load_tables(&S.stab, t, kPairThreads);
    vliw29::Lanes L{t, kPairThreads, tab, nullptr, S.stab.p29};
    for (int i = t; i < vliw29::kTotalRegs; i += kPairThreads) {
        Fp x;
        uint32_t s = seed * 2654435761u + (uint32_t)i * 40503u + 1u;
        for (int k = 0; k < 12; k++) { s = s * 1664525u + 1013904223u; x.l[k] = s; }
        x.l[11] &= 0x0fffffffu;                        // < p
        f29::F29 v = f29::from_fp(x);
        if (i >= vliw29::kRegConst && i < vliw29::kRegConst + 10) v = vliw29::frob_const(i - vliw29::kRegConst);
        S.regs[i] = v; ref[i] = v;
    }
    __syncthreads();
    for (int r = 0; r < rounds; r++)
        for (int prog = 0; prog < vliw29::kNumPrograms; prog++) {
            vliw29::run(prog, S.regs, L);
            if (t == 32) vliw29::run_ref(prog, ref, vliw29::default_tables());
            __syncthreads();
            for (int i = t; i < vliw29::kTotalRegs; i += kPairThreads)
                if (!(vliw29::canonical_signed(S.regs[i], 2048) == vliw29::canonical_signed(ref[i], 2048))) atomicAdd(&mismatches[prog], 1u);
            __syncthreads();
        }
}

}  // namespace kzgb200
