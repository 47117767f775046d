// EIP-7594 (PeerDAS) cells: compute_cells and verify_cell_kzg_proof_batch (consensus-specs Fulu,
// polynomial-commitments-sampling.md), plus the cell workload generator.
//
// Extended domain: the 8192 roots of unity in bit-reversed order; cell k = elements [64k, 64k + 64), element j of cell k at
// h_k * omega64^rev6(j) with coset shift h_k = omega8192^rev7(k), so h_k^64 = omega128^rev7(k).  Cells 0..63 are the blob.
//
// Verification reuses the blob batch's MSM and final check (kzgb200.cu): with C_k = the commitment of cell k, z_k = h_k^64 and
// y_k = 0, launch_lincomb's A = sum r^k pi_k is the spec's LL and B' = sum r^k C_k + r^k z_k pi_k is RLC + RLP.  This file adds
// the parts the blob batch has no counterpart for: cell parsing, the per-cell scalars, and RLI = sum_m c_m [tau^m]G1 with
// c = sum_k r^k coeffs(I_k), computed as r-weighted sums of the cell values per distinct cell index, one 64-point inverse DFT
// per index, and a 64-point fixed-base MSM -- handed to the final check as a second partial (a = O, b = -RLI).
#include "common.cuh"

namespace kzgb200 {

// omega8192 = 7^((q-1)/8192), canonical; omega8192^2 = omega4096 (KZG_FR_OMEGA_M) is checked at setup
#define KZG_FR_OMEGA8192 {0xc78c8967u, 0x6fdd00bfu, 0x434906acu, 0x146b58bcu, 0x972e89edu, 0x2ccddea2u, 0x37b1da3du, 0x485d5127u}

__device__ __forceinline__ uint32_t rev_bits(uint32_t i, int bits) { return __brev(i) >> (32 - bits); }
__device__ __forceinline__ Fr fr_pow_u32(const Fr& b, uint32_t e, int nbits) { return b.pow(&e, nbits); }
__device__ __forceinline__ void store_fe_be(uint8_t* dst, const Fr& mont) {
    Fr raw = mont.to_raw();
    uint4 hi, lo;
    hi.x = sha_bswap(raw.l[7]); hi.y = sha_bswap(raw.l[6]); hi.z = sha_bswap(raw.l[5]); hi.w = sha_bswap(raw.l[4]);
    lo.x = sha_bswap(raw.l[3]); lo.y = sha_bswap(raw.l[2]); lo.z = sha_bswap(raw.l[1]); lo.w = sha_bswap(raw.l[0]);
    reinterpret_cast<uint4*>(dst)[0] = hi; reinterpret_cast<uint4*>(dst)[1] = lo;
}

// ---- setup (kzgb200_load_cell_setup) ------------------------------------------------------------------------------------
__global__ void cell_setup_kernel(CellTables* T, const uint8_t* __restrict__ g2_tau64) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t w8l[8] = KZG_FR_OMEGA8192;
    const Fr w8 = Fr::from_raw(fr_const(w8l));
    if (tid < 2048) {
        const uint32_t om[8] = KZG_FR_OMEGA_M;
        const Fr w = fr_const(om);
        T->w4096[tid] = fr_pow_u32(w, (uint32_t)tid, 12);
        T->w4096_inv[tid] = fr_pow_u32(w, (4096u - (uint32_t)tid) & 4095u, 12);
    }
    if (tid < 4096) { const uint32_t inv[8] = KZG_FR_INV4096_M; T->coset[tid] = fr_pow_u32(w8, (uint32_t)tid, 13) * fr_const(inv); }
    if (tid < kCellsPerExtBlob) {
        const uint32_t e = rev_bits((uint32_t)tid, 7);
        T->shift64[tid] = fr_pow_u32(w8, 64u * e, 14);
        T->shift_inv[tid] = fr_pow_u32(w8, (8192u - e) & 8191u, 14);
    }
    if (tid < kFieldElementsPerCell / 2) T->w64_inv[tid] = fr_pow_u32(w8, (8192u - 128u * (uint32_t)tid) & 8191u, 14);
    if (tid == 0) {
        const uint32_t om[8] = KZG_FR_OMEGA_M;
        T->omega8192 = w8;
        T->inv64 = fr_inv(Fr::from_u32(64));
        G2Affine q;
        bool ok = g2_from_compressed_unchecked(q, g2_tau64) && !q.inf && w8.sqr() == fr_const(om);
        if (ok) prepare_g2(T->tau64_lines, q);
        T->ok = ok ? 1u : 0u;
    }
}
// [tau^m]G1 (m < 64) from the compressed monomial points; tau_tab[m][q] = [2^(64q) tau^m]G1 for the 4 x 64-bit split of RLI
__global__ void cell_setup_points_kernel(CellTables* T, const uint8_t* __restrict__ g1_monomial48) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= kFieldElementsPerCell * 4) return;
    const int m = tid / 4, q = tid % 4;
    uint8_t b[48];
    for (int k = 0; k < 48; k++) b[k] = g1_monomial48[m * 48 + k];
    G1Affine p;
    if (!g1_from_compressed(p, b, true)) { atomicAnd(&T->ok, 0u); p = {Fp::zero(), Fp::zero(), 1}; }
    G1 acc = G1::from_affine(p);
    for (int i = 0; i < 64 * q; i++) acc = acc.dbl();
    T->tau_tab[m][q] = g1_to_affine(acc);
}
// line table of [tau^64]G2 in the pairing engine's representation (as setup_lines29_kernel does for G2 and [tau]G2)
__global__ void cell_setup_lines29_kernel(CellTables* T) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= kMillerSteps * 6) return;
    const int k = tid / 6, e = tid % 6;
    const LineCoeffs& l = T->tau64_lines[k];
    const Fp2& f2 = e < 2 ? l.A : (e < 4 ? l.B : l.C);
    T->lines29[k].v[e] = f29::from_fp((e & 1) ? f2.c1 : f2.c0);
}

// ---- compute_cells ----------------------------------------------------------------------------------------------------
// One CTA per blob, the 4096 values in shared memory (128 KiB).  Only the odd half of the extended domain is new: the blob is
// in bit-reversed order, so a decimation-in-time inverse transform gives the coefficients in natural order; coefficient m is
// scaled by omega8192^m / 4096 (the odd coset, and the inverse transform's 1/n); a decimation-in-frequency forward transform
// then leaves p(omega8192 * omega4096^rev12(i)) at position i -- extended element 4096 + i -- with no explicit permutation.
// kCoeffs: also write the inverse transform's output -- 4096 x the blob's coefficients, natural order, Montgomery -- to coeffs
// (the FK20 proof path, k_cell_proofs.cu).
template <bool kCoeffs>
__device__ __forceinline__ void compute_cells_body(const uint8_t* __restrict__ blobs, int n, const CellTables* __restrict__ T,
                                                   uint8_t* __restrict__ cells, uint32_t* __restrict__ status, Fr* __restrict__ coeffs) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    Fr* a = reinterpret_cast<Fr*>(dyn_smem);
    const int blob = blockIdx.x, t = threadIdx.x;
    if (blob >= n) return;
    const uint4* src = reinterpret_cast<const uint4*>(blobs + (size_t)blob * kBytesPerBlob);
    uint4* out = reinterpret_cast<uint4*>(cells + (size_t)blob * kCellsPerExtBlob * kBytesPerCell);
    bool bad = false;
    for (int i = t; i < kFieldElementsPerBlob; i += kCellNttThreads) {
        const Fr f = load_fe_be(src + 2 * i);
        bad |= f.geq_modulus();
        a[i] = Fr::from_raw(f);
        out[2 * i] = __ldg(src + 2 * i); out[2 * i + 1] = __ldg(src + 2 * i + 1);      // cells 0..63: the blob
    }
    if (bad) atomicOr(&status[blob], kErrBlob);
    __syncthreads();
    for (int len = 2; len <= kFieldElementsPerBlob; len <<= 1) {           // inverse DIT, bit-reversed in, natural out
        const int half = len >> 1, stride = kFieldElementsPerBlob / len;
        for (int b = t; b < kFieldElementsPerBlob / 2; b += kCellNttThreads) {
            const int j = b % half, i0 = (b / half) * len + j;
            const Fr u = a[i0], v = a[i0 + half].mul_inl(T->w4096_inv[j * stride]);
            a[i0] = u.add_inl(v); a[i0 + half] = u.sub_inl(v);
        }
        __syncthreads();
    }
    if (kCoeffs) for (int i = t; i < kFieldElementsPerBlob; i += kCellNttThreads) coeffs[(size_t)blob * kFieldElementsPerBlob + i] = a[i];
    for (int i = t; i < kFieldElementsPerBlob; i += kCellNttThreads) a[i] = a[i].mul_inl(T->coset[i]);
    __syncthreads();
    for (int len = kFieldElementsPerBlob; len >= 2; len >>= 1) {           // forward DIF, natural in, bit-reversed out
        const int half = len >> 1, stride = kFieldElementsPerBlob / len;
        for (int b = t; b < kFieldElementsPerBlob / 2; b += kCellNttThreads) {
            const int j = b % half, i0 = (b / half) * len + j;
            const Fr u = a[i0], v = a[i0 + half];
            a[i0] = u.add_inl(v); a[i0 + half] = u.sub_inl(v).mul_inl(T->w4096[j * stride]);
        }
        __syncthreads();
    }
    uint8_t* odd = cells + ((size_t)blob * kCellsPerExtBlob + kCellsPerExtBlob / 2) * kBytesPerCell;
    for (int i = t; i < kFieldElementsPerBlob; i += kCellNttThreads) store_fe_be(odd + 32 * (size_t)i, a[i]);
}
__global__ void __launch_bounds__(kCellNttThreads) compute_cells_kernel(const uint8_t* __restrict__ blobs, int n, const CellTables* __restrict__ T,
                                                                     uint8_t* __restrict__ cells, uint32_t* __restrict__ status) {
    compute_cells_body<false>(blobs, n, T, cells, status, nullptr);
}
__global__ void __launch_bounds__(kCellNttThreads) compute_cells_coeffs_kernel(const uint8_t* __restrict__ blobs, int n, const CellTables* __restrict__ T,
                                                                            uint8_t* __restrict__ cells, uint32_t* __restrict__ status, Fr* __restrict__ coeffs) {
    compute_cells_body<true>(blobs, n, T, cells, status, coeffs);
}

// ---- verify_cell_kzg_proof_batch --------------------------------------------------------------------------------------
// decompression + subgroup check of `count` compressed points (the unique commitments, or the proofs); failures OR `flag`
// into status[i]
__global__ void __launch_bounds__(128) cell_points_kernel(const uint8_t* __restrict__ bytes, int count, G1Affine* __restrict__ out,
                                                          uint32_t* __restrict__ status, uint32_t flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    uint8_t b[48];
    const uint32_t* src = reinterpret_cast<const uint32_t*>(bytes + (size_t)i * 48);
    for (int k = 0; k < 12; k++) {
        uint32_t v = __ldg(src + k);
        b[4 * k] = (uint8_t)v; b[4 * k + 1] = (uint8_t)(v >> 8); b[4 * k + 2] = (uint8_t)(v >> 16); b[4 * k + 3] = (uint8_t)(v >> 24);
    }
    G1Affine pt;
    if (!g1_from_compressed(pt, b, true)) atomicOr(&status[i], flag);
    out[i] = pt;
}
// canonicity of every cell element (one thread per element)
__global__ void __launch_bounds__(256) cell_check_kernel(const uint8_t* __restrict__ cells, int n, uint32_t* __restrict__ status) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * kFieldElementsPerCell) return;
    if (load_fe_be(reinterpret_cast<const uint4*>(cells) + 2 * i).geq_modulus()) atomicOr(&status[i / kFieldElementsPerCell], kErrBlob);
}
// the blob batch's per-entry inputs for cell k: z_k = h_k^64 (Montgomery; canonical in zy), y_k = 0, C_k = the unique commitment
// it refers to (and that commitment's parse verdict)
__global__ void __launch_bounds__(128) cell_scalars_kernel(const uint32_t* __restrict__ meta, int n, const G1Affine* __restrict__ U,
                                                           const uint32_t* __restrict__ ustatus, const CellTables* __restrict__ T,
                                                           Fr* __restrict__ z_mont, ZY* __restrict__ zy, G1Affine* __restrict__ C,
                                                           uint32_t* __restrict__ status) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t idx = meta[k], u = meta[n + k];
    const Fr z = T->shift64[idx];
    z_mont[k] = z;
    zy[k].z = z.to_raw();
    zy[k].y = Fr::zero();
    C[k] = U[u];
    if (ustatus[u]) atomicOr(&status[k], kErrCommitment);
}
// weighted sums (rk: the per-cell weights) of the cell values per cell index: CTA (index i, slice s) sums its share of the cells with that index
// (order / start: the cells grouped by index, built by the host); thread j = element j
__global__ void __launch_bounds__(kFieldElementsPerCell) cell_agg_kernel(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ meta, int n,
                                                                        const Fr* __restrict__ rk, Fr* __restrict__ agg) {
    const int i = blockIdx.x, s = blockIdx.y, j = threadIdx.x;
    const uint32_t* order = meta + 2 * (size_t)n;
    const uint32_t* start = order + n;
    const uint32_t lo = start[i], hi = start[i + 1], per = (hi - lo + kCellAggSlices - 1) / kCellAggSlices;
    const uint32_t a = lo + s * per, b = a + per < hi ? a + per : hi;
    Fr acc = Fr::zero();
    for (uint32_t p = a; p < b; p++) {
        const uint32_t k = __ldg(order + p);
        const Fr v = Fr::from_raw(load_fe_be(reinterpret_cast<const uint4*>(cells + (size_t)k * kBytesPerCell) + 2 * j));
        acc = acc.add_inl(v.mul_inl(ldg_fr(rk + k)));
    }
    agg[((size_t)i * kCellAggSlices + s) * kFieldElementsPerCell + j] = acc;
}
// 64-point inverse DFT of the 64 values v[] of one cell index i (shared memory, bit-reversed in, natural out), coefficient m scaled
// by h_i^-m / 64: thread j (of 64) gets coefficient j of the interpolant.  Shared by cell_interp_kernel and the per-group checks.
__device__ __forceinline__ Fr cell_interp_body(Fr* v, int i, const CellTables* __restrict__ T) {
    const int j = threadIdx.x;
    __syncthreads();
    for (int len = 2; len <= kFieldElementsPerCell; len <<= 1) {
        const int half = len >> 1, stride = kFieldElementsPerCell / len;
        if (j < kFieldElementsPerCell / 2) {
            const int jj = j % half, i0 = (j / half) * len + jj;
            const Fr u = v[i0], w = v[i0 + half].mul_inl(T->w64_inv[jj * stride]);
            v[i0] = u.add_inl(w); v[i0 + half] = u.sub_inl(w);
        }
        __syncthreads();
    }
    const Fr scale = fr_pow_u32(T->shift_inv[i], (uint32_t)j, 6).mul_inl(T->inv64);
    return v[j].mul_inl(scale);
}
// per distinct index i: the slices' sums, interpolated (cell_interp_body) -> coeffs[i][m]; an index without cells contributes zeros
__global__ void __launch_bounds__(kFieldElementsPerCell) cell_interp_kernel(const Fr* __restrict__ agg, const uint32_t* __restrict__ meta, int n,
                                                                           const CellTables* __restrict__ T, Fr* __restrict__ coeffs) {
    __shared__ Fr v[kFieldElementsPerCell];
    const int i = blockIdx.x, j = threadIdx.x;
    const uint32_t* start = meta + 3 * (size_t)n;
    if (start[i] == start[i + 1]) { coeffs[i * kFieldElementsPerCell + j] = Fr::zero(); return; }
    Fr acc = Fr::zero();
    for (int s = 0; s < kCellAggSlices; s++) acc = acc.add_inl(agg[((size_t)i * kCellAggSlices + s) * kFieldElementsPerCell + j]);
    v[j] = acc;
    coeffs[i * kFieldElementsPerCell + j] = cell_interp_body(v, i, T);
}
// sum_m c_m [tau^m]G1 over 256 threads: thread t = (m, q) = (t / 4, t % 4) holds c_m and multiplies [2^(64q) tau^m]G1 by the q-th
// 64-bit word of c_m, then a tree over the 256 products in sm; the sum is returned to thread 0.  Shared by cell_rli_kernel and the
// per-group checks.
__device__ __forceinline__ G1 cell_rli_body(const Fr& c, const CellTables* __restrict__ T, G1* sm) {
    const int t = threadIdx.x, m = t / 4, q = t % 4;
    const Fr raw = c.to_raw();
    sm[t] = scalar_mul_affine(T->tau_tab[m][q], raw.l + 2 * q, 64);
    __syncthreads();
    for (int span = 128; span >= 1; span >>= 1) {
        if (t < span) sm[t] = sm[t].add(sm[t + span]);
        __syncthreads();
    }
    return sm[0];
}
// RLI = sum_m c_m [tau^m]G1, c_m = sum_i coeffs[i][m] (cell_rli_body).  Written as the second partial of the final check: a = O, b = -RLI.
__global__ void __launch_bounds__(256) cell_rli_kernel(const Fr* __restrict__ coeffs, const CellTables* __restrict__ T, Partial* __restrict__ out) {
    __shared__ G1 sm[256];
    const int t = threadIdx.x, m = t / 4;
    Fr c = Fr::zero();
    for (int i = 0; i < kCellsPerExtBlob; i++) c = c.add_inl(coeffs[i * kFieldElementsPerCell + m]);
    const G1 rli = cell_rli_body(c, T, sm);
    if (t == 0) {
        out->a = G1::identity();
        out->b = rli.neg();
        out->ry = Fr::zero();
        out->err = 0;
    }
}

// ---- verify_cell_kzg_proof_batch[_many]: k independent groups of cells, one verdict each ----------------------------------
// Group g = cells [goff[g], goff[g + 1]).  Every cell gets the weight w_k = rho^g r_g^j (j = its position in the group; with one
// group, r^j); the groups are first checked together by the pipeline above with these weights, and only if that fails (and k > 1),
// each group on its own (the fallback below).  gbad[g] != 0: group g fails an assertion of the spec (BadArgs).
__device__ __forceinline__ uint32_t group_of(const uint32_t* __restrict__ goff, int k, uint32_t cell) {
    int lo = 0, hi = k - 1;                        // the last g with goff[g] <= cell (empty groups before it are skipped)
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (__ldg(goff + mid) <= cell) lo = mid; else hi = mid - 1; }
    return (uint32_t)lo;
}
// the parse flags of every cell, ORed into its group's flag (gbad starts with the host's index checks)
__global__ void __launch_bounds__(128) many_group_status_kernel(const uint32_t* __restrict__ status, int n, const uint32_t* __restrict__ goff, int k,
                                                                uint32_t* __restrict__ gbad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = status[i];
    if (s) atomicOr(&gbad[group_of(goff, k, (uint32_t)i)], s);
}
// w_i = rho^g r_g^j, or 0 in a BadArgs group; rg = k + 1 canonical big-endian values (r_0 .. r_(k-1), rho).  The cell's parse flags are
// cleared: they have been moved to gbad, and a BadArgs group must not fail the combined check.
__global__ void __launch_bounds__(128) many_weights_kernel(int n, const uint32_t* __restrict__ goff, int k, const uint8_t* __restrict__ rg,
                                                           const uint32_t* __restrict__ gbad, Fr* __restrict__ w, uint32_t* __restrict__ status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t g = group_of(goff, k, (uint32_t)i), j = (uint32_t)i - __ldg(goff + g);
    status[i] = 0;
    if (gbad[g]) { w[i] = Fr::zero(); return; }
    const Fr r = Fr::from_raw(load_fe_be(reinterpret_cast<const uint4*>(rg + 32 * (size_t)g)));
    const Fr rho = Fr::from_raw(load_fe_be(reinterpret_cast<const uint4*>(rg + 32 * (size_t)k)));
    w[i] = rho.pow(&g, 32).mul_inl(r.pow(&j, 32));
}
// fallback, per cell: terms[2i] = [w_i]pi_i, terms[2i + 1] = [w_i]C_i + [w_i z_i]pi_i (GLV multiplications); identity for w_i = 0
__global__ void __launch_bounds__(128) many_terms_kernel(int n, const Fr* __restrict__ w, const Fr* __restrict__ z_mont, const G1Affine* __restrict__ C,
                                                         const G1Affine* __restrict__ P, G1* __restrict__ terms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Fr wi = w[i];
    G1 a = G1::identity(), b = G1::identity();
    if (!wi.is_zero()) {
        const G1Affine pi = P[i];
        a = glv_mul(pi, wi.to_raw());
        b = glv_mul(C[i], wi.to_raw()).add(glv_mul(pi, wi.mul_inl(z_mont[i]).to_raw()));
    }
    terms[2 * (size_t)i] = a;
    terms[2 * (size_t)i + 1] = b;
}
// fallback, per group (one CTA each): A_g = sum of the group's [w]pi terms, B'_g = sum of its [w]C + [wz]pi terms
__global__ void __launch_bounds__(128) many_group_sums_kernel(const uint32_t* __restrict__ goff, const G1* __restrict__ terms, G1* __restrict__ AB) {
    __shared__ G1 sm[128];
    const int g = blockIdx.x, t = threadIdx.x;
    const uint32_t lo = goff[g], hi = goff[g + 1];
    for (int part = 0; part < 2; part++) {
        G1 acc = G1::identity();
        for (uint32_t p = lo + t; p < hi; p += blockDim.x) acc = acc.add(terms[2 * (size_t)p + part]);
        sm[t] = acc;
        __syncthreads();
        for (int span = 64; span >= 1; span >>= 1) {
            if (t < span) sm[t] = sm[t].add(sm[t + span]);
            __syncthreads();
        }
        if (t == 0) AB[2 * (size_t)g + part] = sm[0];
        __syncthreads();
    }
}
// fallback, per (group, cell index) run (one CTA of 64 threads each): the w-weighted sum of the run's cells, interpolated ->
// rcoef[run][m].  fmeta = [cells of each group ordered by index (n) | start of each run in that order (runs + 1) | index of each run].
__global__ void __launch_bounds__(kFieldElementsPerCell) many_run_interp_kernel(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ fmeta,
                                                                               int n, int runs, const Fr* __restrict__ w,
                                                                               const CellTables* __restrict__ T, Fr* __restrict__ rcoef) {
    __shared__ Fr v[kFieldElementsPerCell];
    const int r = blockIdx.x, j = threadIdx.x;
    const uint32_t* order = fmeta;
    const uint32_t* rstart = fmeta + n;
    const uint32_t idx = fmeta[n + runs + 1 + r];
    Fr acc = Fr::zero();
    for (uint32_t p = rstart[r]; p < rstart[r + 1]; p++) {
        const uint32_t k = __ldg(order + p);
        const Fr x = Fr::from_raw(load_fe_be(reinterpret_cast<const uint4*>(cells + (size_t)k * kBytesPerCell) + 2 * j));
        acc = acc.add_inl(x.mul_inl(ldg_fr(w + k)));
    }
    v[j] = acc;
    rcoef[(size_t)r * kFieldElementsPerCell + j] = cell_interp_body(v, (int)idx, T);
}
// fallback, per group (one CTA of 256 threads each): RLI_g from the coefficients of its runs (grun[g] .. grun[g + 1]), then the
// two pairing arguments X_g = B'_g - RLI_g and A_g, affine, for e(X_g, G2) e(-A_g, [tau^64]G2) == 1 on the many-check engine
__global__ void __launch_bounds__(256) many_group_rli_kernel(const Fr* __restrict__ rcoef, const uint32_t* __restrict__ grun, const G1* __restrict__ AB,
                                                             const CellTables* __restrict__ T, G1Affine* __restrict__ X, G1Affine* __restrict__ A) {
    __shared__ G1 sm[256];
    const int g = blockIdx.x, t = threadIdx.x, m = t / 4;
    Fr c = Fr::zero();
    for (uint32_t r = grun[g]; r < grun[g + 1]; r++) c = c.add_inl(rcoef[(size_t)r * kFieldElementsPerCell + m]);
    const G1 rli = cell_rli_body(c, T, sm);
    if (t == 0) {
        X[g] = g1_to_affine(AB[2 * (size_t)g + 1].add(rli.neg()));
        A[g] = g1_to_affine(AB[2 * (size_t)g]);
    }
}

// ---- workload generator (kzgb200_harness_generate_cells) ---------------------------------------------------------------
// Blob b is the polynomial p = A + X^64 B + X^128 Cc of degree < D (128 < D <= 192) with seeded coefficients; its 128 cells are
// its values on the extended domain.  Modulo X^64 - s (s = h_k^64) it is A + s B + s^2 Cc, so the quotient of cell k is
// B + s Cc + X^64 Cc and the proof is [B(tau)] + [tau^64 Cc(tau)] + s [Cc(tau)]: three 64-term commitments per blob, then
// one scalar multiplication per cell.
__device__ __noinline__ Fr cell_harness_coeff(uint64_t seed, uint64_t blob, int j) {
    uint64_t s = seed ^ ((blob * kCellHarnessMaxDegree + (uint64_t)j) * 0xd1342543de82ef95ull) ^ 0x7594u;
    Fr raw;
    for (int k = 0; k < 4; k++) {
        uint64_t z = (s += 0x9e3779b97f4a7c15ull);
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        z ^= z >> 31;
        raw.l[2 * k] = (uint32_t)z; raw.l[2 * k + 1] = (uint32_t)(z >> 32);
    }
    return Fr::from_raw(raw);
}
// terms[b][part][m]: part 0..2 = A_m [tau^m], B_m [tau^(64+m)], Cc_m [tau^(128+m)] (the commitment); 3 = B_m [tau^m];
// 4 = Cc_m [tau^m]; 5 = Cc_m [tau^(64+m)]
__global__ void __launch_bounds__(128) cell_harness_terms_kernel(uint64_t seed, int n, int D, const G1Affine* __restrict__ M, G1* __restrict__ terms) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= n * 6 * 64) return;
    const int b = tid / 384, part = (tid / 64) % 6, m = tid % 64;
    const int seg[6] = {0, 1, 2, 1, 2, 2}, pw[6] = {0, 64, 128, 0, 0, 64};
    const int j = 64 * seg[part] + m, e = pw[part] + m;
    G1 r = G1::identity();
    if (j < D) {
        const Fr raw = cell_harness_coeff(seed, (uint64_t)b, j).to_raw();
        r = scalar_mul_affine(M[e], raw.l, 255);
    }
    terms[tid] = r;
}
__global__ void __launch_bounds__(128) cell_harness_sums_kernel(int n, const G1* __restrict__ terms, G1* __restrict__ sums) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= n * 6) return;
    G1 acc = G1::identity();
    for (int m = 0; m < 64; m++) acc = acc.add(terms[(size_t)tid * 64 + m]);
    sums[tid] = acc;
}
// thread (b, k): k < 128 -> proof of cell k; k == 128 -> the commitment
__global__ void __launch_bounds__(128) cell_harness_points_kernel(int n, const G1* __restrict__ sums, const CellTables* __restrict__ T,
                                                                  uint8_t* __restrict__ commitments, uint8_t* __restrict__ proofs) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= n * (kCellsPerExtBlob + 1)) return;
    const int b = tid / (kCellsPerExtBlob + 1), k = tid % (kCellsPerExtBlob + 1);
    const G1* s = sums + (size_t)b * 6;
    G1 acc;
    uint8_t* dst;
    if (k == kCellsPerExtBlob) {
        acc = s[0].add(s[1]).add(s[2]);
        dst = commitments + (size_t)b * 48;
    } else {
        const Fr sr = T->shift64[k].to_raw();
        acc = s[3].add(s[5]).add(scalar_mul(s[4], sr.l, 255));
        dst = proofs + ((size_t)b * kCellsPerExtBlob + k) * 48;
    }
    uint8_t enc[48];
    g1_to_compressed(enc, g1_to_affine(acc));
    for (int i = 0; i < 48; i++) dst[i] = enc[i];
}
// extended element e of blob b: p(omega8192^rev13(e)) by Horner
__global__ void __launch_bounds__(128) cell_harness_eval_kernel(uint64_t seed, int n, int D, const CellTables* __restrict__ T, uint8_t* __restrict__ cells) {
    __shared__ Fr coef[kCellHarnessMaxDegree];
    const int b = blockIdx.y, t = threadIdx.x;
    if (b >= n) return;
    for (int j = t; j < D; j += blockDim.x) coef[j] = cell_harness_coeff(seed, (uint64_t)b, j);
    __syncthreads();
    const int e = blockIdx.x * blockDim.x + t;
    const Fr x = fr_pow_u32(T->omega8192, rev_bits((uint32_t)e, 13), 13);
    Fr f = coef[D - 1];
    for (int k = D - 2; k >= 0; k--) f = f.mul_inl(x).add_inl(coef[k]);
    store_fe_be(cells + ((size_t)b * kCellsPerExtBlob * kFieldElementsPerCell + e) * 32, f);
}

}  // namespace kzgb200
