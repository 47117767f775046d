// K7 (BASELINE config 5): many independent verify_kzg_proof tuples (reference src/kzg_proof.rs:353-397, src/pairings.rs:5-9) --
// also the per-blob verdicts of a failing batch (kzgb200_verify_blob_kzg_proof_batch_each).
//
// Round 1 ran one thread per tuple through the whole check: 255 registers and a 19.7 KB stack frame per thread (an Fp12 is 144
// words), 0.24 of the chip's multiplication rate.  Now the check is a pipeline of kernels with a working set that fits:
//   g1_decompress_kernel / g1_subgroup_kernel (k_g1.cu)   one thread per POINT: parse C_i, pi_i
//   many_lhs_kernel                                        one thread per tuple: z, y canonical?  X_i = C_i - [y_i]G + [z_i]pi_i, affine
//   many_pairing_kernel                                    kManyGroups tuples per CTA in lockstep: e(X_i, G2) e(-pi_i, [tau]G2) == 1 on the
//                                                          cooperative engine (vliw.cuh), the Fp12 values in shared memory
// Both G2 arguments are setup constants, so all tuples share the 2 x 68 precomputed line triples.  The second one is [tau]G2, or
// the point of the line table lines_b when it is given (the per-group cell checks: [tau^64]G2).
#include "common.cuh"

namespace kzgb200 {

// z, y: 32 big-endian bytes each (safe_scalar_affine_from_bytes, kzg_proof.rs:27-43, in the reference's order z, y, C, pi).
// status bits set by the parsing kernels are kept; X is written for every tuple (garbage for flagged ones, never read).
__global__ void __launch_bounds__(128) many_lhs_kernel(const uint8_t* __restrict__ z32, const uint8_t* __restrict__ y32, const G1Affine* __restrict__ C,
                                                       const G1Affine* __restrict__ P, size_t m, const DeviceTables* __restrict__ T,
                                                       G1Affine* __restrict__ X, uint32_t* __restrict__ status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    Fr z, y;
    const uint32_t* zw = reinterpret_cast<const uint32_t*>(z32 + i * 32);
    const uint32_t* yw = reinterpret_cast<const uint32_t*>(y32 + i * 32);
#pragma unroll
    for (int k = 0; k < 8; k++) { z.l[7 - k] = sha_bswap(__ldg(zw + k)); y.l[7 - k] = sha_bswap(__ldg(yw + k)); }
    uint32_t bad = (z.geq_modulus() || y.geq_modulus()) ? kErrScalar : 0u;
    if (bad) status[i] |= bad;
    if (bad || status[i]) return;
    G1 acc = kzg_lhs_point_fast(C[i], z, y, P[i], T->gen_table);
    X[i] = g1_to_affine(acc);
}
// the same from parsed / evaluated batch data (z, y canonical limbs in zy): per-blob verdicts
__global__ void __launch_bounds__(128) many_lhs_zy_kernel(const ZY* __restrict__ zy, const G1Affine* __restrict__ C, const G1Affine* __restrict__ P, size_t m,
                                                          const DeviceTables* __restrict__ T, G1Affine* __restrict__ X, const uint32_t* __restrict__ status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m || status[i]) return;
    ZY s = zy[i];
    X[i] = g1_to_affine(kzg_lhs_point_fast(C[i], s.z, s.y, P[i], T->gen_table));
}

// One CTA runs kManyGroups checks in LOCKSTEP through the engine: every level's instructions of all groups are spread over the
// CTA's threads (a level of 18..50 instructions per check becomes 250..700 independent ones: ~95 % of the lanes busy instead of
// ~55 % for one check per warp), one barrier per level for the whole CTA, and -- since all warps of the SM are at the same place
// of the same code -- the instruction cache holds (one check per warp, 12 unsynchronised warps per SM: `no_instruction` was
// 12 stalls per issue, profiles/ncu_many_r02.txt).  Register files: kManyGroups x 10 KB of shared memory.
// Checks whose X or pi is the identity take a different program path; they are left to many_pairing_warp_kernel (k_many2.cu).
struct ManySmem {
    uint32_t regs[kManyGroups * kManyStride];     // kManyGroups register files, an odd number of words apart
    vliw::SharedTables stab;
    Fp shared[vliw::kNumSharedRegs];               // line coefficients of the current Miller step + Frobenius constants: the same for every check
    G1Affine x[kManyGroups], np[kManyGroups];
    uint8_t ok[kManyGroups], use[kManyGroups];
};
static_assert(sizeof(ManySmem) <= kManySmemBytes, "keep kManySmemBytes (common.cuh) in step with ManySmem");
__global__ void __launch_bounds__(kManyThreads, kManyCtasPerSm) many_pairing_kernel(const G1Affine* __restrict__ X, const G1Affine* __restrict__ P,
                                                                       const uint32_t* __restrict__ status, size_t m,
                                                                       const DeviceTables* __restrict__ T, const LineCoeffs* __restrict__ lines_b,
                                                                       uint8_t* __restrict__ verdicts) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    ManySmem& S = *reinterpret_cast<ManySmem*>(dyn_smem);
    vliw::Tables tab = vliw::load_tables(&S.stab, threadIdx.x, blockDim.x, true);
    vliw::remap_tables_multi(&S.stab, threadIdx.x, blockDim.x);
    __syncthreads();
    const int t = threadIdx.x;
    vliw::Lanes L{t, kManyThreads, tab, nullptr, false};
    L.groups = kManyGroups; L.stride = kManyStride; L.shared = S.shared;
    const size_t nbatch = (m + kManyGroups - 1) / kManyGroups;
    for (size_t batch = blockIdx.x; batch < nbatch; batch += gridDim.x) {      // uniform trip count for the whole CTA
        if (t < kManyGroups) {
            size_t i = batch * kManyGroups + t;
            G1Affine x = g1_generator(), np = g1_generator();                  // filler for slots without a live check
            uint8_t use = 0;
            if (i < m) {
                uint32_t st = __ldg(status + i);
                if (st) verdicts[i] = kBadArgs;
                else {
                    G1Affine xi = X[i], pi = P[i];
                    if (xi.inf || pi.inf) verdicts[i] = kPending;              // identity input: single-check kernel
                    else { x = xi; np = pi; np.y = np.y.neg(); use = 1; }
                }
            }
            S.x[t] = x; S.np[t] = np; S.use[t] = use;
        }
        __syncthreads();
        vliw::coop_pairing_multi(reinterpret_cast<Fp*>(S.regs), S.x, T->pairing.g2_gen, S.np, lines_b ? lines_b : T->pairing.tau_g2, L, S.ok);
        if (t < kManyGroups && S.use[t]) verdicts[batch * kManyGroups + t] = S.ok[t] ? kTrue : kFalse;
        __syncthreads();
    }
}

}  // namespace kzgb200
