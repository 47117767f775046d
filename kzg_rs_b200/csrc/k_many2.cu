// K7 (config 5), the rare path: pairing checks whose X_i or pi_i is the identity (the pair is skipped, reference
// multi_miller_loop semantics) run one per warp on the single-check form of the engine; many_pairing_kernel marks them kPending.
#include "common.cuh"

namespace kzgb200 {

struct ManyWarpSmem {
    Fp regs[kManyWarps][vliw::kTotalRegs];
    vliw::SharedTables stab;
};
static_assert(sizeof(ManyWarpSmem) <= kManySmemBytes, "shared-memory budget of the many-tuple kernels");
__global__ void __launch_bounds__(32 * kManyWarps, 1) many_pairing_warp_kernel(const G1Affine* __restrict__ X, const G1Affine* __restrict__ P, size_t m,
                                                                               const DeviceTables* __restrict__ T, const LineCoeffs* __restrict__ lines_b,
                                                                               uint8_t* __restrict__ verdicts) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    ManyWarpSmem& S = *reinterpret_cast<ManyWarpSmem*>(dyn_smem);
    vliw::Tables tab = vliw::load_tables(&S.stab, threadIdx.x, blockDim.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Fp* regs = S.regs[warp];
    vliw::Lanes L{lane, 32, tab, nullptr, true};
    for (size_t i = (size_t)blockIdx.x * kManyWarps + warp; i < m; i += (size_t)gridDim.x * kManyWarps) {
        if (verdicts[i] != kPending) continue;                            // warp-uniform
        G1Affine x = X[i], np = P[i];
        if (!np.inf) np.y = np.y.neg();
        bool ok = vliw::coop_pairing_product_is_one(regs, x, T->pairing.g2_gen, np, lines_b ? lines_b : T->pairing.tau_g2, L);
        __syncwarp();
        if (lane == 0) verdicts[i] = ok ? kTrue : kFalse;
    }
}

}  // namespace kzgb200
