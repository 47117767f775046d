// K8: device-resident trusted-setup tables.
#include "common.cuh"

namespace kzgb200 {

// ------------------------------------------------------------------------------------------------ K8
__global__ void setup_tables_kernel(DeviceTables* T, const uint8_t* g2_points /* 2 x 96 B: g2[0], g2[1] */) {
    int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid < 2048) {
        // bitrev12(2g)
        uint32_t i = 2u * tid, e = 0;
        for (int b = 0; b < 12; b++) e |= ((i >> b) & 1u) << (11 - b);
        const uint32_t om[8] = KZG_FR_OMEGA_M;
        uint32_t ee[1] = {e};
        T->twiddle[tid] = fr_const(om).pow(ee, 12);
    }
    if (tid >= 8192 && tid < 8192 + 4096) {
        int t = (tid - 8192) >> 5, m = (tid - 8192) & 31, cnt = 0;
        uint32_t g = 0;                                   // pad entry (m == 31): any valid element
        for (int j = 0; j < 32; j++)
            for (int k = 0; (j >> k) & 1; k++, cnt++)
                if (cnt == m) g = (uint32_t)(t * 32 + j) >> (k + 1);
        uint32_t i = 2u * g, e = 0;
        for (int b = 0; b < 12; b++) e |= ((i >> b) & 1u) << (11 - b);
        const uint32_t om[8] = KZG_FR_OMEGA_M;
        uint32_t ee[1] = {e};
        T->twiddle_po[t][m] = fr_const(om).pow(ee, 12);
    }
    if (tid >= 4096 && tid < 4096 + 960) {
        int w = (tid - 4096) / 15, d = (tid - 4096) % 15 + 1;
        uint32_t k[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        k[w / 8] = (uint32_t)d << (4 * (w % 8));
        T->gen_table[w][d - 1] = g1_to_affine(scalar_mul_affine(g1_generator(), k, 256));
    }
    if (tid == 2048) {
        G2Affine gen, tau;
        bool ok = g2_from_compressed_unchecked(gen, g2_points) && g2_from_compressed_unchecked(tau, g2_points + 96);
        ok = ok && !gen.inf && !tau.inf;
        if (ok) {
            prepare_g2(T->pairing.g2_gen, gen);
            prepare_g2(T->pairing.tau_g2, tau);
        }
        T->setup_ok = ok ? 1u : 0u;
    }
}

// line tables of the two fixed G2 points in the pairing engine's 29-bit-limb representation (one value per thread)
__global__ void setup_lines29_kernel(DeviceTables* T) {
    int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= 2 * kMillerSteps * 6) return;
    int q = tid / (kMillerSteps * 6), k = (tid / 6) % kMillerSteps, e = tid % 6;
    const LineCoeffs& l = q == 0 ? T->pairing.g2_gen[k] : T->pairing.tau_g2[k];
    const Fp2& f2 = e < 2 ? l.A : (e < 4 ? l.B : l.C);
    T->lines29[q][k].v[e] = f29::from_fp((e & 1) ? f2.c1 : f2.c0);
}

// line tables of [256^w]Q, Q in {G2, [tau]G2}, w = 1..15, for the split tail of the batch check (one thread per table: 8w doublings,
// affine conversion, the 68 line triples into `scratch` (30 x kMillerSteps), then the engine's representation).  Built from the
// context's own G2 points, so a custom setup gets its own tables.
__global__ void setup_lines29w_kernel(DeviceTables* T, const uint8_t* g2_points /* 2 x 96 B */, LineCoeffs* scratch) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= 2 * (kWindows - 1)) return;
    const int q = tid / (kWindows - 1), w = tid % (kWindows - 1) + 1;
    G2Affine base;
    if (!g2_from_compressed_unchecked(base, g2_points + 96 * q) || base.inf) return;    // setup_tables_kernel reports the failure
    G2 acc = G2::from_affine(base);
    for (int k = 0; k < 8 * w; k++) acc = acc.dbl();
    LineCoeffs* lc = scratch + (size_t)tid * kMillerSteps;
    prepare_g2(lc, g2_to_affine(acc));
    for (int k = 0; k < kMillerSteps; k++)
        for (int e = 0; e < 6; e++) {
            const Fp2& f2 = e < 2 ? lc[k].A : (e < 4 ? lc[k].B : lc[k].C);
            T->lines29w[q][w - 1][k].v[e] = f29::from_fp((e & 1) ? f2.c1 : f2.c0);
        }
}

}  // namespace kzgb200
