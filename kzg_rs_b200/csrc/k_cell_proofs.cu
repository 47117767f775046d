// EIP-7594 (PeerDAS) cell proofs and recovery (consensus-specs Fulu, polynomial-commitments-sampling.md):
// compute_cells_and_kzg_proofs by FK20 and recover_cells_and_kzg_proofs, plus the setup both need.  DESIGN.md section 5b.
//
// FK20.  p = sum_{m<4096} c_m X^m, m = 64a + b, s_k = h_k^64 = omega128^rev7(k).  The proof of cell k is [q_k(tau)]G1 with
// q_k = p div (X^64 - s_k) = sum_{t<63} s_k^t Q_t, so pi_k = sum_t s_k^t H_t, H_t = [Q_t(tau)]G1 -- a 128-point G1 DFT of
// (H_0..H_62, 0, ..): pi_k is output rev7(k).  H_t = sum_b (u_b (*) w_b)[t + 1] (cyclic length-128 convolutions) with
// u_b[a] = c_{64a+b} (a < 64, zero above) and w_b[0] = [tau^b], w_b[128 - d] = [tau^(64d+b)] (d = 1..62), zero elsewhere; by the
// convolution theorem H = IDFT(V)[1..63], V[f] = sum_b U_b[f] W_b[f], U_b = DFT(u_b), W_b = DFT_G1(w_b) fixed at setup.
//
// Recovery follows recover_polynomialcoeff literally: E (zeros at the missing cells) times Z on the 8192-point domain, inverse
// transform, coset (shift 7) transform, division by Z on the coset, inverse coset transform, first 4096 coefficients.  Z(X) = z(X^64)
// with z(Y) = prod_{missing k} (Y - s_k), so Z is constant on each cell: z at s_k on the domain and at 7^64 s_k on the coset.  The
// 8192-point transforms are one radix-2 stage through global memory and two 4096-point halves in shared memory (one CTA each).
#include "common.cuh"

namespace kzgb200 {

#define KZG_FR_INV2_19_M {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0x00002000u}     // 2^-19, Montgomery (2^237)
#define KZG_FR_OMEGA8192 {0xc78c8967u, 0x6fdd00bfu, 0x434906acu, 0x146b58bcu, 0x972e89edu, 0x2ccddea2u, 0x37b1da3du, 0x485d5127u}

__device__ __forceinline__ uint32_t rev_bits_p(uint32_t i, int bits) { return __brev(i) >> (32 - bits); }
__device__ __forceinline__ Fr fr_pow_small(const Fr& b, uint32_t e, int nbits) { return b.pow(&e, nbits); }
__device__ __forceinline__ void store_fe_be_p(uint8_t* dst, const Fr& mont) {
    Fr raw = mont.to_raw();
    uint4 hi, lo;
    hi.x = sha_bswap(raw.l[7]); hi.y = sha_bswap(raw.l[6]); hi.z = sha_bswap(raw.l[5]); hi.w = sha_bswap(raw.l[4]);
    lo.x = sha_bswap(raw.l[3]); lo.y = sha_bswap(raw.l[2]); lo.z = sha_bswap(raw.l[1]); lo.w = sha_bswap(raw.l[0]);
    reinterpret_cast<uint4*>(dst)[0] = hi; reinterpret_cast<uint4*>(dst)[1] = lo;
}

// [k]P for a prime-order-subgroup point P, k canonical (raw limbs): GLV split k = k1 + k2 x^2, then a joint 128-bit double-and-add
// over P, -phi(P) = (beta X, -Y, Z) and their sum
__device__ __noinline__ G1 g1_mul_glv(const G1 p, const Fr raw) {
    uint32_t k1[4], k2[4];
    glv_split(raw.l, k1, k2);
    const uint32_t beta[12] = KZG_FP_BETA_M;
    const G1 q = {p.x * fp_const(beta), p.y.neg(), p.z};
    const G1 pq = p.add(q);
    G1 acc = G1::identity();
    for (int i = 127; i >= 0; i--) {
        acc = acc.dbl();
        const uint32_t b1 = (k1[i >> 5] >> (i & 31)) & 1u, b2 = (k2[i >> 5] >> (i & 31)) & 1u;
        if (b1 & b2) acc = acc.add(pq);
        else if (b1) acc = acc.add(p);
        else if (b2) acc = acc.add(q);
    }
    return acc;
}

// 128-point DFT over G1 in shared memory by 64 threads (one butterfly each per level): s in bit-reversed order on entry, natural
// on exit; out[f] = sum_n omega128^(+-fn) in[n]
__device__ void g1_dft128(G1* s, const CellTables* __restrict__ T, bool inverse) {
    const int t = threadIdx.x;
    const Fr* w = inverse ? T->w4096_inv : T->w4096;     // omega128^j = omega4096^(32j)
    for (int len = 2; len <= 128; len <<= 1) {
        const int half = len >> 1, j = t % half, i0 = (t / half) * len + j;
        G1 v = s[i0 + half];
        if (j) v = g1_mul_glv(v, w[32 * j * (128 / len)].to_raw());
        const G1 u = s[i0];
        s[i0] = u.add(v);
        s[i0 + half] = u.add(v.neg());
        __syncthreads();
    }
}

// ---- setup (kzgb200_load_cell_proof_setup) ---------------------------------------------------------------------------
__global__ void proof_setup_kernel(ProofTables* P) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kExtElements) return;
    const uint32_t w8l[8] = KZG_FR_OMEGA8192;
    const Fr w8 = Fr::from_raw(fr_const(w8l)), seven = Fr::from_u32(7);
    const Fr inv8192 = fr_inv(Fr::from_u32(kExtElements));
    P->pow7[i] = fr_pow_small(seven, (uint32_t)i, 13).mul_inl(inv8192);
    if (i < kFieldElementsPerBlob) {
        P->w8192[i] = fr_pow_small(w8, (uint32_t)i, 13);
        P->w8192_inv[i] = fr_pow_small(w8, (uint32_t)(kExtElements - i) & (kExtElements - 1), 13);
        P->pow7_inv[i] = fr_pow_small(fr_inv(seven), (uint32_t)i, 12).mul_inl(inv8192);
    }
    if (i == 0) P->s7_64 = fr_pow_small(seven, 64u, 7);
}
// monomial points [tau^m]G1 = sum_j omega4096^(jm) L_j, L_j = the Lagrange points in file order: a forward 4096-point DFT over G1.
// Radix-2 decimation in time: the points in bit-reversed order, then 12 levels of 2048 butterflies (mono_level_kernel).
__global__ void __launch_bounds__(128) mono_load_kernel(const uint8_t* __restrict__ lag48, G1* __restrict__ a, uint32_t* __restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kFieldElementsPerBlob) return;
    const uint32_t src = rev_bits_p((uint32_t)i, 12);
    uint8_t b[48];
    for (int k = 0; k < 48; k++) b[k] = lag48[(size_t)src * 48 + k];
    G1Affine p;
    if (!g1_from_compressed(p, b, true)) atomicOr(bad, 1u);   // subgroup-checked: the butterflies use the GLV endomorphism
    a[i] = G1::from_affine(p);
}
__global__ void __launch_bounds__(128) mono_level_kernel(G1* __restrict__ a, int len, const CellTables* __restrict__ T) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= kFieldElementsPerBlob / 2) return;
    const int half = len >> 1, j = b % half, i0 = (b / half) * len + j;
    G1 v = a[i0 + half];
    if (j) v = g1_mul_glv(v, T->w4096[j * (kFieldElementsPerBlob / len)].to_raw());
    const G1 u = a[i0];
    a[i0] = u.add(v);
    a[i0 + half] = u.add(v.neg());
}
// affine monomial points; the first 64 must be the points the cell setup was loaded with
__global__ void __launch_bounds__(128) mono_finish_kernel(const G1* __restrict__ a, const CellTables* __restrict__ T, G1Affine* __restrict__ mono,
                                                          uint32_t* __restrict__ bad) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= kFieldElementsPerBlob) return;
    mono[m] = g1_to_affine(a[m]);
    if (m < kFieldElementsPerCell && !a[m].equals(G1::from_affine(T->tau_tab[m][0]))) atomicOr(bad, 2u);
}
__global__ void __launch_bounds__(128) mono_compress_kernel(const G1Affine* __restrict__ mono, int n, uint8_t* __restrict__ out48) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    uint8_t enc[48];
    g1_to_compressed(enc, mono[m]);
    for (int k = 0; k < 48; k++) out48[(size_t)m * 48 + k] = enc[k];
}
// W_b = DFT_G1(w_b): CTA b, 64 threads; W[f * 64 + b] (affine)
__global__ void __launch_bounds__(64) fk20_w_kernel(const G1Affine* __restrict__ mono, const CellTables* __restrict__ T, G1Affine* __restrict__ W) {
    __shared__ G1 s[kCellsPerExtBlob];
    const int b = blockIdx.x, t = threadIdx.x;
    for (int n = t; n < kCellsPerExtBlob; n += 64) {
        G1 v = G1::identity();
        if (n == 0) v = G1::from_affine(mono[b]);
        else if (n >= 66) v = G1::from_affine(mono[64 * (128 - n) + b]);      // d = 128 - n = 1..62
        s[rev_bits_p((uint32_t)n, 7)] = v;
    }
    __syncthreads();
    g1_dft128(s, T, false);
    for (int f = t; f < kCellsPerExtBlob; f += 64) W[f * kFieldElementsPerCell + b] = g1_to_affine(s[f]);
}
// window tables: thread (base, w) writes [d * 256^w] W[base], d = 1..255
__global__ void __launch_bounds__(128) fk20_table_kernel(const G1Affine* __restrict__ W, G1Affine* __restrict__ tab) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= kFk20Bases * kFk20Windows) return;
    const int base = tid / kFk20Windows, w = tid % kFk20Windows;
    G1 p = G1::from_affine(W[base]);
    for (int k = 0; k < 8 * w; k++) p = p.dbl();
    G1Affine* row = tab + (size_t)tid * kFk20Entries;
    G1 acc = p;
    for (int d = 1; d <= kFk20Entries; d++) {
        row[d - 1] = g1_to_affine(acc);
        acc = acc.add(p);
    }
}

// ---- compute_cells_and_kzg_proofs ------------------------------------------------------------------------------------
// U[blob][f][b] = DFT_128(u_b)[f] / 2^19, canonical limbs.  coeffs = 4096 x the coefficients (compute_cells_coeffs_kernel), so
// the scale 1 / (4096 * 128) also takes the inverse DFT's 1/128.  CTA (b, blob), 64 threads.
__global__ void __launch_bounds__(64) fk20_scalars_kernel(const Fr* __restrict__ coeffs, const CellTables* __restrict__ T, Fr* __restrict__ U) {
    __shared__ Fr s[kCellsPerExtBlob];
    const int b = blockIdx.x, blob = blockIdx.y, t = threadIdx.x;
    const Fr* c = coeffs + (size_t)blob * kFieldElementsPerBlob;
    s[rev_bits_p((uint32_t)t, 7)] = c[64 * t + b];
    s[rev_bits_p((uint32_t)t + 64, 7)] = Fr::zero();
    __syncthreads();
    for (int len = 2; len <= 128; len <<= 1) {
        const int half = len >> 1, j = t % half, i0 = (t / half) * len + j;
        const Fr u = s[i0], v = s[i0 + half].mul_inl(T->w4096[32 * j * (128 / len)]);
        s[i0] = u.add_inl(v); s[i0 + half] = u.sub_inl(v);
        __syncthreads();
    }
    const uint32_t inv19[8] = KZG_FR_INV2_19_M;
    const Fr scale = fr_const(inv19);
    for (int f = t; f < kCellsPerExtBlob; f += 64)
        U[((size_t)blob * kCellsPerExtBlob + f) * kFieldElementsPerCell + b] = s[f].mul_inl(scale).to_raw();
}
// V[blob][f] = sum_b U_b[f] W_b[f] through the window tables: CTA (f, blob), thread b does 16 + 16 table additions (GLV halves,
// the second through -phi), then a tree over the 64 threads
__global__ void __launch_bounds__(64) fk20_products_kernel(const Fr* __restrict__ U, const G1Affine* __restrict__ tab, G1* __restrict__ V) {
    __shared__ G1 sm[kFieldElementsPerCell];
    const int f = blockIdx.x, blob = blockIdx.y, b = threadIdx.x;
    const size_t row = (size_t)blob * kCellsPerExtBlob + f;
    const Fr k = ldg_fr(U + row * kFieldElementsPerCell + b);
    uint32_t k1[4], k2[4];
    glv_split(k.l, k1, k2);
    const G1Affine* tb = tab + (size_t)(f * kFieldElementsPerCell + b) * kFk20Windows * kFk20Entries;
    G1 acc = G1::identity();
    for (int w = 0; w < kFk20Windows; w++) {
        const uint32_t d1 = (k1[w >> 2] >> (8 * (w & 3))) & 0xffu, d2 = (k2[w >> 2] >> (8 * (w & 3))) & 0xffu;
        if (d1) acc = acc.add_mixed(tb[w * kFk20Entries + d1 - 1]);
        if (d2) acc = acc.add_mixed(glv_endo_neg(tb[w * kFk20Entries + d2 - 1]));
    }
    sm[b] = acc;
    __syncthreads();
    for (int span = 32; span >= 1; span >>= 1) {
        if (b < span) sm[b] = sm[b].add(sm[b + span]);
        __syncthreads();
    }
    if (b == 0) V[row] = sm[0];
}
// per blob (64 threads): H = IDFT(V)[1..63], then the proofs pi_k = DFT(H)[rev7(k)], compressed (blob-major, cell order)
__global__ void __launch_bounds__(64) fk20_proofs_kernel(const G1* __restrict__ V, const CellTables* __restrict__ T, uint8_t* __restrict__ proofs) {
    __shared__ G1 s[kCellsPerExtBlob];
    const int blob = blockIdx.x, t = threadIdx.x;
    for (int f = t; f < kCellsPerExtBlob; f += 64) s[rev_bits_p((uint32_t)f, 7)] = V[(size_t)blob * kCellsPerExtBlob + f];
    __syncthreads();
    g1_dft128(s, T, true);
    const G1 h = t < 63 ? s[t + 1] : G1::identity();     // H_t
    __syncthreads();
    s[rev_bits_p((uint32_t)t, 7)] = h;
    s[rev_bits_p((uint32_t)t + 64, 7)] = G1::identity();
    __syncthreads();
    g1_dft128(s, T, false);
    for (int k = t; k < kCellsPerExtBlob; k += 64) {
        uint8_t enc[48];
        g1_to_compressed(enc, g1_to_affine(s[rev_bits_p((uint32_t)k, 7)]));
        uint8_t* dst = proofs + ((size_t)blob * kCellsPerExtBlob + k) * 48;
        for (int i = 0; i < 48; i++) dst[i] = enc[i];
    }
}

// ---- recover_cells_and_kzg_proofs ------------------------------------------------------------------------------------
// zvals[k] = z(s_k) (Z on cell k of the domain), zvals[128 + k] = 1 / z(7^64 s_k) (1 / Z on cell k of the coset transform's
// bit-reversed output); missing = the absent cell indices
__global__ void __launch_bounds__(256) recover_z_kernel(const uint32_t* __restrict__ missing, int n_missing, const CellTables* __restrict__ T,
                                                        const ProofTables* __restrict__ P, Fr* __restrict__ zvals) {
    const int t = threadIdx.x;
    const int k = t & (kCellsPerExtBlob - 1);
    const Fr x = t < kCellsPerExtBlob ? T->shift64[k] : T->shift64[k].mul_inl(P->s7_64);
    Fr z = Fr::one();
    for (int i = 0; i < n_missing; i++) z = z.mul_inl(x.sub_inl(T->shift64[missing[i]]));
    zvals[t] = t < kCellsPerExtBlob ? z : fr_inv(z);
}
// E times Z in bit-reversed order (the spec's extended_evaluation_rbo, which is what the inverse DIT transform reads): element p of
// blob `blob` comes from input cell pos[p / 64] (-1: missing, zero); non-canonical elements flag the blob
__global__ void __launch_bounds__(256) recover_load_kernel(const uint8_t* __restrict__ cells, int n_cells, const int* __restrict__ pos,
                                                           const Fr* __restrict__ zvals, int nb, Fr* __restrict__ A, uint32_t* __restrict__ status) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)nb * kExtElements) return;
    const int blob = (int)(i / kExtElements), p = (int)(i % kExtElements), k = p / kFieldElementsPerCell, src = pos[k];
    Fr v = Fr::zero();
    if (src >= 0) {
        const Fr raw = load_fe_be(reinterpret_cast<const uint4*>(cells + ((size_t)blob * n_cells + src) * kBytesPerCell) + 2 * (p % kFieldElementsPerCell));
        if (raw.geq_modulus()) atomicOr(&status[blob], kErrBlob);
        v = Fr::from_raw(raw).mul_inl(zvals[k]);
    }
    A[i] = v;
}
// 4096-point halves of the 8192-point transforms, one CTA per (half, blob), the half in shared memory
__device__ __forceinline__ void ntt4096_dit_inv(Fr* a, const CellTables* __restrict__ T) {     // bit-reversed in, natural out, no 1/n
    const int t = threadIdx.x;
    for (int len = 2; len <= kFieldElementsPerBlob; len <<= 1) {
        const int half = len >> 1, stride = kFieldElementsPerBlob / len;
        for (int b = t; b < kFieldElementsPerBlob / 2; b += kCellNttThreads) {
            const int j = b % half, i0 = (b / half) * len + j;
            const Fr u = a[i0], v = a[i0 + half].mul_inl(T->w4096_inv[j * stride]);
            a[i0] = u.add_inl(v); a[i0 + half] = u.sub_inl(v);
        }
        __syncthreads();
    }
}
__device__ __forceinline__ void ntt4096_dif_fwd(Fr* a, const CellTables* __restrict__ T) {     // natural in, bit-reversed out
    const int t = threadIdx.x;
    for (int len = kFieldElementsPerBlob; len >= 2; len >>= 1) {
        const int half = len >> 1, stride = kFieldElementsPerBlob / len;
        for (int b = t; b < kFieldElementsPerBlob / 2; b += kCellNttThreads) {
            const int j = b % half, i0 = (b / half) * len + j;
            const Fr u = a[i0], v = a[i0 + half];
            a[i0] = u.add_inl(v); a[i0 + half] = u.sub_inl(v).mul_inl(T->w4096[j * stride]);
        }
        __syncthreads();
    }
}
__device__ __forceinline__ Fr* ntt_half_load(Fr* A, Fr* a) {
    Fr* g = A + ((size_t)blockIdx.y * 2 + blockIdx.x) * kFieldElementsPerBlob;
    for (int i = threadIdx.x; i < kFieldElementsPerBlob; i += kCellNttThreads) a[i] = g[i];
    __syncthreads();
    return g;
}
// inverse transform of (E Z), first part: the 4096-point levels of each half
__global__ void __launch_bounds__(kCellNttThreads) recover_ntt_inv_kernel(Fr* __restrict__ A, const CellTables* __restrict__ T) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    Fr* a = reinterpret_cast<Fr*>(dyn_smem);
    Fr* g = ntt_half_load(A, a);
    ntt4096_dit_inv(a, T);
    for (int i = threadIdx.x; i < kFieldElementsPerBlob; i += kCellNttThreads) g[i] = a[i];
}
// coset transform, second part (the 4096-point levels), division by Z on the coset, and the inverse transform's 4096-point levels
__global__ void __launch_bounds__(kCellNttThreads) recover_ntt_div_kernel(Fr* __restrict__ A, const CellTables* __restrict__ T, const Fr* __restrict__ zvals) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    Fr* a = reinterpret_cast<Fr*>(dyn_smem);
    Fr* g = ntt_half_load(A, a);
    ntt4096_dif_fwd(a, T);
    const int base = blockIdx.x * kFieldElementsPerBlob;
    for (int i = threadIdx.x; i < kFieldElementsPerBlob; i += kCellNttThreads)
        a[i] = a[i].mul_inl(zvals[kCellsPerExtBlob + (base + i) / kFieldElementsPerCell]);
    __syncthreads();
    ntt4096_dit_inv(a, T);
    for (int i = threadIdx.x; i < kFieldElementsPerBlob; i += kCellNttThreads) g[i] = a[i];
}
// the global stages: the inverse transform's last level (twiddle omega8192^-i), the coefficients times 7^m / 8192, and the coset
// transform's first level (twiddle omega8192^i); thread (blob, i) owns elements i and i + 4096
__global__ void __launch_bounds__(256) recover_mid_kernel(Fr* __restrict__ A, const ProofTables* __restrict__ P, int nb) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (size_t)nb * kFieldElementsPerBlob) return;
    const int i = (int)(tid % kFieldElementsPerBlob);
    Fr* a = A + (tid / kFieldElementsPerBlob) * kExtElements;
    const Fr u = a[i], v = a[i + kFieldElementsPerBlob].mul_inl(P->w8192_inv[i]);
    const Fr c0 = u.add_inl(v).mul_inl(P->pow7[i]), c1 = u.sub_inl(v).mul_inl(P->pow7[i + kFieldElementsPerBlob]);
    a[i] = c0.add_inl(c1);
    a[i + kFieldElementsPerBlob] = c0.sub_inl(c1).mul_inl(P->w8192[i]);
}
// the inverse coset transform's last level, only the first 4096 outputs, times 7^-m / 8192: the recovered coefficients
__global__ void __launch_bounds__(256) recover_final_kernel(const Fr* __restrict__ A, const ProofTables* __restrict__ P, int nb, Fr* __restrict__ coeffs) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (size_t)nb * kFieldElementsPerBlob) return;
    const int i = (int)(tid % kFieldElementsPerBlob);
    const Fr* a = A + (tid / kFieldElementsPerBlob) * kExtElements;
    coeffs[tid] = a[i].add_inl(a[i + kFieldElementsPerBlob].mul_inl(P->w8192_inv[i])).mul_inl(P->pow7_inv[i]);
}
// the recovered coefficients -> the blob (evaluations in bit-reversed order), one CTA per blob
__global__ void __launch_bounds__(kCellNttThreads) recover_blob_kernel(const Fr* __restrict__ coeffs, const CellTables* __restrict__ T, uint8_t* __restrict__ blobs) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    Fr* a = reinterpret_cast<Fr*>(dyn_smem);
    const int blob = blockIdx.x;
    for (int i = threadIdx.x; i < kFieldElementsPerBlob; i += kCellNttThreads) a[i] = coeffs[(size_t)blob * kFieldElementsPerBlob + i];
    __syncthreads();
    ntt4096_dif_fwd(a, T);
    uint8_t* out = blobs + (size_t)blob * kBytesPerBlob;
    for (int i = threadIdx.x; i < kFieldElementsPerBlob; i += kCellNttThreads) store_fe_be_p(out + 32 * (size_t)i, a[i]);
}

}  // namespace kzgb200
