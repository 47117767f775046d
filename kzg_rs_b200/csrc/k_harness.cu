// Harness workload generator and commit / prove (SURVEY 8f-1).
#include "common.cuh"

namespace kzgb200 {

// ================================================================================================ harness
// Workload generator (harness side; kzg-rs has no commit/prove path).  Blob b is the evaluation form of a
// random polynomial p_b of degree < D over the bit-reversed 4096-point domain; its commitment and proof are
// C = sum_j c_j [tau^j]G1 and pi = sum_j q_j [tau^j]G1 with q = (p - p(z)) / (X - z) by synthetic division,
// over the mainnet setup's [tau^j]G1 (kzg_rs_b200/data/tau_powers_g1.bin).  The verifier never sees the
// structure: it does the same work as for any blob.
__device__ __forceinline__ uint64_t splitmix64(uint64_t& s) {
    uint64_t z = (s += 0x9e3779b97f4a7c15ull);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
// coefficient j of blob b, Montgomery form of a uniform 256-bit value mod q
__device__ __noinline__ Fr harness_coeff(uint64_t seed, uint64_t blob, int j) {
    uint64_t s = seed ^ ((blob * kHarnessMaxDegree + (uint64_t)j) * 0xd1342543de82ef95ull);
    Fr raw;
    for (int k = 0; k < 4; k++) { uint64_t v = splitmix64(s); raw.l[2 * k] = (uint32_t)v; raw.l[2 * k + 1] = (uint32_t)(v >> 32); }
    return Fr::from_raw(raw);
}
__global__ void harness_parse_points_kernel(const uint8_t* bytes, int n, G1Affine* out, uint32_t* bad) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t b[48];
    for (int k = 0; k < 48; k++) b[k] = bytes[i * 48 + k];
    if (!g1_from_compressed(out[i], b, true)) atomicOr(bad, 1u);
}
__global__ void __launch_bounds__(128) harness_blob_kernel(uint64_t seed, int n, int D, const DeviceTables* __restrict__ T, uint8_t* __restrict__ blobs) {
    __shared__ Fr coef[kHarnessMaxDegree];
    int blob = blockIdx.x, t = threadIdx.x;
    if (blob >= n) return;
    if (t < D) coef[t] = harness_coeff(seed, blob, t);
    __syncthreads();
    for (int j = 0; j < 32; j++) {
        int i = t * 32 + j;
        Fr w = T->twiddle[i >> 1];
        if (i & 1) w = w.neg();
        Fr f = coef[D - 1];
        for (int k = D - 2; k >= 0; k--) f = f * w + coef[k];
        Fr raw = f.to_raw();
        uint4 hi, lo;
        hi.x = sha_bswap(raw.l[7]); hi.y = sha_bswap(raw.l[6]); hi.z = sha_bswap(raw.l[5]); hi.w = sha_bswap(raw.l[4]);
        lo.x = sha_bswap(raw.l[3]); lo.y = sha_bswap(raw.l[2]); lo.z = sha_bswap(raw.l[1]); lo.w = sha_bswap(raw.l[0]);
        uint4* dst = reinterpret_cast<uint4*>(blobs + (size_t)blob * kBytesPerBlob) + 2 * i;
        dst[0] = hi; dst[1] = lo;
    }
}
// proofs == nullptr: commitments C = sum c_j M_j ; else proofs pi = sum q_j M_j using z_mont
__global__ void __launch_bounds__(64) harness_commit_kernel(uint64_t seed, int n, int D, const G1Affine* __restrict__ M, const Fr* __restrict__ z_mont,
                                                            uint8_t* __restrict__ out, int want_proof) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    Fr c[kHarnessMaxDegree];
    for (int j = 0; j < D; j++) c[j] = harness_coeff(seed, b, j);
    int terms = D;
    if (want_proof) {   // synthetic division by (X - z): q_{D-2} = c_{D-1}, q_{j-1} = c_j + z q_j
        Fr z = z_mont[b], q[kHarnessMaxDegree];
        q[D - 2] = c[D - 1];
        for (int j = D - 2; j >= 1; j--) q[j - 1] = c[j] + z * q[j];
        for (int j = 0; j < D - 1; j++) c[j] = q[j];
        terms = D - 1;
    }
    G1 acc = G1::identity();
    for (int j = 0; j < terms; j++) {
        Fr raw = c[j].to_raw();
        acc = acc.add(scalar_mul_affine(M[j], raw.l, 255));
    }
    uint8_t enc[48];
    g1_to_compressed(enc, g1_to_affine(acc));
    for (int k = 0; k < 48; k++) out[(size_t)b * 48 + k] = enc[k];
}

// ================================================================================================ commit / prove
// SURVEY.md 8(f)-1: blob_to_kzg_commitment / compute_blob_kzg_proof as GPU operations (EIP-4844 semantics; kzg-rs
// itself has no commit/prove path -- these produce test data for arbitrary blobs and are pinned by the commitment /
// proof bytes of the reference's valid vectors).  Fixed-base MSM over the 4096 bit-reversed Lagrange points with a
// precomputed window table table[j][w][d-1] = [d * 256^w] L_j (Jacobian), so a blob costs 4096 x 32 table additions
// spread over a CTA.
__global__ void lag_parse_kernel(const uint8_t* __restrict__ bytes /* 4096 x 48, file order */, G1Affine* __restrict__ out /* bit-reversed */,
                                 uint32_t* __restrict__ bad) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kFieldElementsPerBlob) return;
    uint32_t src = 0;
    for (int b = 0; b < 12; b++) src |= (((uint32_t)i >> b) & 1u) << (11 - b);
    uint8_t buf[48];
    for (int k = 0; k < 48; k++) buf[k] = bytes[(size_t)src * 48 + k];
    if (!g1_from_compressed(out[i], buf, false)) atomicOr(bad, 1u);   // unchecked, as build.rs:68
}
__global__ void __launch_bounds__(128) lag_table_kernel(const G1Affine* __restrict__ L, G1* __restrict__ table) {
    int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= kFieldElementsPerBlob * kLagWindows) return;
    int j = tid / kLagWindows, w = tid % kLagWindows;
    G1 base = G1::from_affine(L[j]);
    for (int k = 0; k < 8 * w; k++) base = base.dbl();
    G1* row = table + (size_t)tid * kLagEntries;
    G1 acc = base;
    row[0] = acc;
    for (int d = 2; d <= kLagEntries; d++) { acc = acc.add(base); row[d - 1] = acc; }
}
// scalars of the commitment MSM = the blob's field elements (canonical limbs); flags non-canonical elements
__global__ void __launch_bounds__(128) blob_scalars_kernel(const uint8_t* __restrict__ blobs, int n, Fr* __restrict__ scalars, uint32_t* __restrict__ status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * kFieldElementsPerBlob) return;
    Fr f = load_fe_be(reinterpret_cast<const uint4*>(blobs) + 2 * i);
    if (f.geq_modulus()) atomicOr(&status[i / kFieldElementsPerBlob], kErrBlob);
    scalars[i] = f;
}
// quotient q_i = (f_i - y) / (w_i - z) in evaluation form (one CTA of 128 threads per blob, Montgomery batch inversion
// across the CTA); if z = w_m the m-th entry is sum_{i != m} (f_i - y) w_i / (z (z - w_i)) = -(1/z) sum_{i != m} q_i w_i, summed
// by every thread over its own 32 entries, then tree-summed in shared memory
__global__ void __launch_bounds__(kEvalThreads, 5) quotient_kernel(const uint8_t* __restrict__ blobs, int n, const Fr* __restrict__ z_mont,
                                                                const ZY* __restrict__ zy, const DeviceTables* __restrict__ T,
                                                                Fr* __restrict__ scalars) {
    __shared__ Fr s_tot[kEvalThreads], s_pre[kEvalThreads], s_inv;
    __shared__ int s_special;
    int blob = blockIdx.x, t = threadIdx.x;
    if (blob >= n) return;
    if (t == 0) s_special = -1;
    __syncthreads();
    Fr z = z_mont[blob], y_m = Fr::from_raw(zy[blob].y), one = Fr::one();
    const uint4* base = reinterpret_cast<const uint4*>(blobs + (size_t)blob * kBytesPerBlob) + (size_t)t * kLeavesPerThread * 2;
    Fr den[kLeavesPerThread], pre[kLeavesPerThread];
    Fr acc = one;
    for (int j = 0; j < kLeavesPerThread; j++) {
        int i = t * kLeavesPerThread + j;
        Fr w = T->twiddle[i >> 1];
        if (i & 1) w = w.neg();
        Fr d = w - z;
        if (d.is_zero()) { s_special = i; d = one; }
        den[j] = d; pre[j] = acc; acc = acc.mul_inl(d);
    }
    s_tot[t] = acc;
    __syncthreads();
    if (t == 0) {
        Fr run = one;
        for (int k = 0; k < kEvalThreads; k++) { s_pre[k] = run; run = run * s_tot[k]; }
        s_inv = fr_inv(run);
        // s_pre[k] becomes the inverse of (product of the totals of threads 0..k)
        Fr inv = s_inv;
        for (int k = kEvalThreads - 1; k >= 0; k--) { Fr tk = s_tot[k]; s_tot[k] = inv; inv = inv * tk; }
    }
    __syncthreads();
    // inverse of this thread's full product = s_tot[t] * (product of earlier threads' totals) = s_tot[t] * s_pre[t]
    Fr inv_run = s_tot[t] * s_pre[t];
    Fr* out = scalars + (size_t)blob * kFieldElementsPerBlob + (size_t)t * kLeavesPerThread;
    for (int j = kLeavesPerThread - 1; j >= 0; j--) {
        Fr inv_d = inv_run.mul_inl(pre[j]);          // 1 / den[j]
        inv_run = inv_run.mul_inl(den[j]);
        Fr f = Fr::from_raw(load_fe_be(base + 2 * j));
        out[j] = ((f - y_m).mul_inl(inv_d)).to_raw();
    }
    const int special = s_special;      // z in the domain (probability 2^-243 for hashed z; a real input of compute_kzg_proof)
    if (special < 0) return;            // uniform across the CTA
    Fr qw = Fr::zero();                 // sum of q_i w_i over this thread's entries i != special (its own stores, read back)
    for (int j = 0; j < kLeavesPerThread; j++)
        if (t * kLeavesPerThread + j != special) qw = qw + Fr::from_raw(out[j]).mul_inl(den[j] + z);   // den[j] + z = w_i
    __syncthreads();                    // every thread has read s_tot / s_pre
    s_tot[t] = qw;
    __syncthreads();
    for (int span = kEvalThreads / 2; span >= 1; span >>= 1) {
        if (t < span) s_tot[t] = s_tot[t] + s_tot[t + span];
        __syncthreads();
    }
    if (t == 0) scalars[(size_t)blob * kFieldElementsPerBlob + special] = (s_tot[0] * fr_inv(z)).neg().to_raw();
}
// Sliced fixed-base MSM sum_j [s_j] L_j through the window table.  Term i = 32 j + w of a blob (point j, window w) is row i of the
// table, so a blob is 131072 terms in table order; CTA (s, blob) of a (slices x blobs) grid sums the s-th of `slices` equal ranges (thread t takes
// every kLagMsmThreads-th term from t), tree-sums its threads' partials in shared memory and stores one Jacobian partial, which
// lag_msm_finish_kernel sums.  Many slices spread a small batch over the whole GPU (kzgb200.cu, lag_slices); with one slice per blob
// the CTA compresses its sum itself (out48), so that each blob's affine conversion overlaps the MSM of later CTAs.
__global__ void __launch_bounds__(kLagMsmThreads) lag_msm_slice_kernel(const Fr* __restrict__ scalars, int n, int slices, const G1* __restrict__ table,
                                                                       G1* __restrict__ partials, uint8_t* __restrict__ out48) {
    __shared__ G1 sm[kLagMsmThreads];
    int s = blockIdx.x, blob = blockIdx.y, t = threadIdx.x;
    if (blob >= n) return;
    const uint32_t* row = reinterpret_cast<const uint32_t*>(scalars + (size_t)blob * kFieldElementsPerBlob);
    const int lo = (int)((int64_t)s * kLagTerms / slices), hi = (int)((int64_t)(s + 1) * kLagTerms / slices);
    G1 acc = G1::identity();
    for (int i = lo + t; i < hi; i += kLagMsmThreads) {
        uint32_t d = (__ldg(row + 8 * (i >> 5) + ((i & 31) >> 2)) >> (8 * (i & 3))) & 0xffu;   // byte w of s_j
        if (d) acc = acc.add(table[(size_t)i * kLagEntries + d - 1]);
    }
    sm[t] = acc;
    __syncthreads();
    for (int span = kLagMsmThreads / 2; span >= 1; span >>= 1) {
        if (t < span) sm[t] = sm[t].add(sm[t + span]);
        __syncthreads();
    }
    if (t != 0) return;
    if (slices > 1) { partials[(size_t)blob * slices + s] = sm[0]; return; }
    uint8_t enc[48];
    g1_to_compressed(enc, g1_to_affine(sm[0]));
    for (int k = 0; k < 48; k++) out48[(size_t)blob * 48 + k] = enc[k];
}
// slices > 1: one CTA per blob, the sum of its slice partials (thread t takes every kLagFinishThreads-th, then a tree in shared memory), compressed.
// Affine compression is canonical: the bytes do not depend on how the sum was split.
__global__ void __launch_bounds__(kLagFinishThreads) lag_msm_finish_kernel(const G1* __restrict__ partials, int n, int slices, uint8_t* __restrict__ out48) {
    __shared__ G1 sm[kLagFinishThreads];
    int blob = blockIdx.x, t = threadIdx.x;
    if (blob >= n) return;
    G1 acc = G1::identity();
    for (int s = t; s < slices; s += kLagFinishThreads) acc = acc.add(partials[(size_t)blob * slices + s]);
    sm[t] = acc;
    __syncthreads();
    for (int span = kLagFinishThreads / 2; span >= 1; span >>= 1) {
        if (t < span && t + span < slices) sm[t] = sm[t].add(sm[t + span]);
        __syncthreads();
    }
    if (t == 0) {
        uint8_t enc[48];
        g1_to_compressed(enc, g1_to_affine(sm[0]));
        for (int k = 0; k < 48; k++) out48[(size_t)blob * 48 + k] = enc[k];
    }
}

}  // namespace kzgb200
