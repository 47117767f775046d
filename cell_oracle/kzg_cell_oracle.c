/* CPU ORACLE OF THE EIP-7594 CELL PATH -- TEST INFRASTRUCTURE ONLY.
 *
 * A C restatement of compute_cells and verify_cell_kzg_proof_batch (consensus-specs Fulu, polynomial-commitments-sampling.md),
 * plus a cell-proof maker for test data, over the field / curve / pairing arithmetic of the blob oracle (the headers under oracle/).  Only
 * tests/ and tools/bench_cells.py load it; the product (kzg_rs_b200/, libkzgb200.so) never does.
 *
 * Setup: the "KZGS" container (kzg_rs_b200/data/mainnet_setup.bin, tests/golden/custom_setup.bin): 4096 Lagrange G1 points
 * (bit-reversal permuted on load, as the blob oracle does) and at least 65 G2 points (g2[0] = G2, g2[64] = [tau^64]G2).
 * [tau^j]G1 for j < 64 (the interpolation commitment RLI) are derived from the Lagrange points on first use.
 * kzgco_recover_cells restates recover_polynomialcoeff step by step, so that inconsistent cells give the spec's bytes too.
 */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include "../oracle/pairing.h"
#include "../oracle/sha256.h"

#define N_FE 4096
enum { KZG_OK = 0, KZG_BADARGS = 1, KZG_INTERNAL = 2, KZG_BADLEN = 3, KZG_BADSETUP = 5 };

static struct {
    int ready, g1_ready;
    fr roots[N_FE];              /* omega4096^bitrev12(i), Montgomery */
    g1_aff g1_lagrange[N_FE];    /* bit-reversal permuted */
    uint8_t g1_bytes[N_FE][48];
    g2_aff g2_gen, tau64_g2;     /* g2_points[0], g2_points[64] */
    int mono_ready;
    g1_aff g1_monomial[64];      /* [tau^j]G1, j < 64 */
    fr omega8192;                /* primitive 8192-th root of unity, omega8192^2 = omega4096 */
    pthread_mutex_t lock;
} S = {.lock = PTHREAD_MUTEX_INITIALIZER};

static uint32_t bitrev(uint32_t i, int bits) {
    uint32_t r = 0; for (int b = 0; b < bits; b++) r |= ((i >> b) & 1) << (bits - 1 - b); return r;
}

/* setup_bin = "KZGS" | u32 n1 | u32 n2 | n1*48 | n2*96 */
int kzgco_init(const uint8_t *setup_bin, size_t len) {
    if (len < 12 || memcmp(setup_bin, "KZGS", 4)) return KZG_BADSETUP;
    uint32_t n1, n2; memcpy(&n1, setup_bin + 4, 4); memcpy(&n2, setup_bin + 8, 4);
    if (n1 != N_FE || n2 < 65 || len != 12 + (size_t)n1 * 48 + (size_t)n2 * 96) return KZG_BADSETUP;
    fr w, acc; memcpy(w.l, FR_OMEGA_M, 32); fr_set_one(&acc);
    for (uint32_t i = 0; i < N_FE; i++) { S.roots[bitrev(i, 12)] = acc; fr_mul(&acc, &acc, &w); }
    for (uint32_t i = 0; i < N_FE; i++) memcpy(S.g1_bytes[i], setup_bin + 12 + 48 * (size_t)bitrev(i, 12), 48);
    const uint8_t *g2 = setup_bin + 12 + (size_t)n1 * 48;
    if (!g2_from_compressed_unchecked(&S.g2_gen, g2) || !g2_from_compressed_unchecked(&S.tau64_g2, g2 + 64 * 96)) return KZG_BADSETUP;
    /* omega8192 = 7^((q-1)/8192) (the spec's PRIMITIVE_ROOT_OF_UNITY); its square must be the blob domain's omega */
    uint64_t e[4]; fr seven, sq; fr_from_u64(&seven, 7);
    for (int i = 0; i < 4; i++) e[i] = (FR_Q[i] >> 13) | (i < 3 ? FR_Q[i + 1] << 51 : 0);
    fr_pow(&S.omega8192, &seven, e, 4); fr_sqr(&sq, &S.omega8192);
    if (!fr_eq(&sq, &w)) return KZG_INTERNAL;
    S.ready = 1; S.g1_ready = 0; S.mono_ready = 0;
    return KZG_OK;
}
static int ensure_g1(void) {
    int rc = KZG_OK;
    pthread_mutex_lock(&S.lock);
    if (!S.g1_ready) {
        for (int i = 0; i < N_FE && !rc; i++) if (!g1_from_compressed(&S.g1_lagrange[i], S.g1_bytes[i], 0)) rc = KZG_BADSETUP;
        S.g1_ready = !rc;
    }
    pthread_mutex_unlock(&S.lock);
    return rc;
}
/* safe_scalar_affine_from_bytes / safe_g1_affine_from_bytes / hash_to_bls_field */
static int safe_scalar_from_bytes(fr *out, const uint8_t b[32]) {
    uint64_t raw[4]; be32_to_limbs(raw, b);
    if (bn_geq(raw, FR_Q, 4)) return KZG_BADARGS;
    fr_from_raw(out, raw); return KZG_OK;
}
static int safe_g1_from_bytes(g1_aff *out, const uint8_t b[48]) { return g1_from_compressed(out, b, 1) ? KZG_OK : KZG_BADARGS; }
static void scalar_from_bytes_unchecked(fr *out, const uint8_t b[32]) { uint64_t raw[4]; be32_to_limbs(raw, b); fr_from_raw(out, raw); }
static int blob_as_polynomial(fr *poly, const uint8_t *blob) {
    for (int i = 0; i < N_FE; i++) if (safe_scalar_from_bytes(&poly[i], blob + 32 * i)) return KZG_BADARGS;
    return KZG_OK;
}
/* commitment of a polynomial in evaluation form (bit-reversed order) with the Lagrange points */
static int lagrange_msm(uint8_t *out48, const fr *evals) {
    int rc = ensure_g1(); if (rc) return rc;
    uint64_t (*sc)[4] = (uint64_t (*)[4])malloc(32 * N_FE);
    for (int i = 0; i < N_FE; i++) fr_to_raw(sc[i], &evals[i]);
    g1 acc; g1_msm(&acc, S.g1_lagrange, (const uint64_t (*)[4])sc, N_FE); free(sc);
    g1_aff a; g1_to_aff(&a, &acc); g1_to_compressed(out48, &a); return KZG_OK;
}
typedef struct { void (*fn)(size_t); size_t n, next; pthread_mutex_t m; } job_t;
static void *job_worker(void *p) {
    job_t *j = (job_t *)p;
    for (;;) {
        pthread_mutex_lock(&j->m); size_t i = j->next++; pthread_mutex_unlock(&j->m);
        if (i >= j->n) return NULL;
        j->fn(i);
    }
}
static void parallel_for(size_t n, void (*fn)(size_t)) {
    enum { T = 8 };
    pthread_t th[T];
    job_t j = {fn, n, 0, PTHREAD_MUTEX_INITIALIZER};
    for (int t = 0; t < T; t++) pthread_create(&th[t], NULL, job_worker, &j);
    for (int t = 0; t < T; t++) pthread_join(th[t], NULL);
}

/* The extended blob is the blob polynomial evaluated on the 8192 roots of unity in bit-reversed order; cell k holds elements
 * [64k, 64k + 64) of it.  Element j of cell k is the value at h_k * omega64^rev6(j), h_k = omega8192^rev7(k), so h_k^64 =
 * omega128^rev7(k).  Cells 0..63 are the blob itself. */
#define CELLS_PER_EXT_BLOB 128
#define FE_PER_CELL 64
#define BYTES_PER_CELL 2048
#define N_EXT 8192

/* in-place radix-2 transform, natural order in and out: a[k] <- sum_m a[m] w^(mk), w a primitive n-th root */
static void fr_dft(fr *a, int n, const fr *w) {
    int bits = 0; while ((1 << bits) < n) bits++;
    for (int i = 0; i < n; i++) { int j = (int)bitrev((uint32_t)i, bits); if (j > i) { fr t = a[i]; a[i] = a[j]; a[j] = t; } }
    for (int len = 2; len <= n; len <<= 1) {
        fr wl; uint64_t e[1] = {(uint64_t)(n / len)}; fr_pow(&wl, w, e, 1);
        for (int i = 0; i < n; i += len) {
            fr x; fr_set_one(&x);
            for (int j = 0; j < len / 2; j++) {
                fr u = a[i + j], v; fr_mul(&v, &a[i + j + len / 2], &x);
                fr_add(&a[i + j], &u, &v); fr_sub(&a[i + j + len / 2], &u, &v); fr_mul(&x, &x, &wl);
            }
        }
    }
}
static void fr_idft(fr *a, int n, const fr *w) {
    fr wi, ni; fr_inv(&wi, w); fr_dft(a, n, &wi);
    fr_from_u64(&ni, (uint64_t)n); fr_inv(&ni, &ni);
    for (int i = 0; i < n; i++) fr_mul(&a[i], &a[i], &ni);
}
static void omega_pow(fr *r, const fr *w, uint64_t e) { uint64_t ee[1] = {e}; fr_pow(r, w, ee, 1); }
/* coset shift of cell k: h_k = omega8192^rev7(k) */
static void cell_shift(fr *h, int k) { omega_pow(h, &S.omega8192, bitrev((uint32_t)k, 7)); }
/* polynomial_eval_to_coeff: the blob (evaluation form, bit-reversed order) -> 4096 coefficients */
static int blob_to_coeffs(fr *coeffs, const uint8_t *blob) {
    fr *poly = (fr *)malloc(N_FE * sizeof(fr));
    int rc = blob_as_polynomial(poly, blob);
    if (!rc) {
        fr w; memcpy(w.l, FR_OMEGA_M, 32);
        for (int i = 0; i < N_FE; i++) coeffs[i] = poly[bitrev((uint32_t)i, 12)];
        fr_idft(coeffs, N_FE, &w);
    }
    free(poly); return rc;
}

/* compute_cells: coefficients, zero-extended to 8192, evaluated on the 8192 roots, bit-reversal permuted, split into 128 cells */
int kzgco_compute_cells(const uint8_t *blob, uint8_t *cells_out /* 128 x 2048 */) {
    fr *ext = (fr *)calloc(N_EXT, sizeof(fr));
    int rc = blob_to_coeffs(ext, blob);
    if (!rc) {
        fr_dft(ext, N_EXT, &S.omega8192);
        for (int i = 0; i < N_EXT; i++) fr_to_bytes_be(cells_out + 32 * (size_t)i, &ext[bitrev((uint32_t)i, 13)]);
    }
    free(ext); return rc;
}

/* coefficients of cell k's interpolation polynomial from its 64 values (already Montgomery): the values are those of
 * J(Y) = I(h_k Y) at omega64^rev6(j), so an inverse DFT gives J's coefficients a_m h_k^m, then a_m = b_m h_k^-m */
static void cell_interpolate(fr *coeffs, const fr *vals, int k) {
    fr w64, h, hinv, x;
    omega_pow(&w64, &S.omega8192, N_EXT / FE_PER_CELL);
    for (int j = 0; j < FE_PER_CELL; j++) coeffs[bitrev((uint32_t)j, 6)] = vals[j];
    fr_idft(coeffs, FE_PER_CELL, &w64);
    cell_shift(&h, k); fr_inv(&hinv, &h); fr_set_one(&x);
    for (int m = 0; m < FE_PER_CELL; m++) { fr_mul(&coeffs[m], &coeffs[m], &x); fr_mul(&x, &x, &hinv); }
}
static int cell_values(fr *vals, const uint8_t *cell) {
    for (int j = 0; j < FE_PER_CELL; j++) if (safe_scalar_from_bytes(&vals[j], cell + 32 * j)) return KZG_BADARGS;
    return KZG_OK;
}

/* the KZG multi-proof of cell k: quotient of (p - I_k) by X^64 - h_k^64 (synthetic division; the remainder must be I_k),
 * back to evaluation form, committed with the Lagrange points.  A test-data maker (the spec computes all 128 with FK20). */
int kzgco_compute_cell_kzg_proof(const uint8_t *blob, int k, uint8_t *p48) {
    if (k < 0 || k >= CELLS_PER_EXT_BLOB) return KZG_BADARGS;
    fr *c = (fr *)malloc(2 * N_FE * sizeof(fr)), *q = c + N_FE;
    uint8_t *cells = (uint8_t *)malloc((size_t)CELLS_PER_EXT_BLOB * BYTES_PER_CELL);
    int rc = blob_to_coeffs(c, blob);
    if (!rc) rc = kzgco_compute_cells(blob, cells);
    if (!rc) {
        fr h, s, t, vals[FE_PER_CELL], interp[FE_PER_CELL];
        cell_shift(&h, k); omega_pow(&s, &h, FE_PER_CELL);
        memset(q, 0, N_FE * sizeof(fr));
        for (int m = N_FE - 1; m >= FE_PER_CELL; m--) {        /* X^m = X^(m-64) (X^64 - s) + s X^(m-64) */
            q[m - FE_PER_CELL] = c[m];
            fr_mul(&t, &c[m], &s); fr_add(&c[m - FE_PER_CELL], &c[m - FE_PER_CELL], &t);
        }
        cell_values(vals, cells + (size_t)k * BYTES_PER_CELL);
        cell_interpolate(interp, vals, k);
        for (int m = 0; m < FE_PER_CELL; m++) if (!fr_eq(&interp[m], &c[m])) rc = KZG_INTERNAL;   /* (p - I_k) mod (X^64 - s) != 0 */
        if (!rc) {
            fr w, *ev = c; memcpy(w.l, FR_OMEGA_M, 32);
            fr_dft(q, N_FE, &w);
            for (int i = 0; i < N_FE; i++) ev[i] = q[bitrev((uint32_t)i, 12)];
            rc = lagrange_msm(p48, ev);
        }
    }
    free(c); free(cells); return rc;
}

/* [tau^j]G1 = sum_i w_i^j [L_i(tau)]G1 (the commitment to X^j) */
static void job_monomial(size_t j) {
    fr c; uint64_t (*sc)[4] = (uint64_t (*)[4])malloc(32 * N_FE);
    for (int i = 0; i < N_FE; i++) { omega_pow(&c, &S.roots[i], (uint64_t)j); fr_to_raw(sc[i], &c); }
    g1 acc; g1_msm(&acc, S.g1_lagrange, (const uint64_t (*)[4])sc, N_FE); g1_to_aff(&S.g1_monomial[j], &acc);
    free(sc);
}
static int ensure_monomial(void) {
    int rc = ensure_g1(); if (rc) return rc;
    pthread_mutex_lock(&S.lock);
    if (!S.mono_ready) { parallel_for(FE_PER_CELL, job_monomial); S.mono_ready = 1; }
    pthread_mutex_unlock(&S.lock);
    return KZG_OK;
}

static void put_u64be(uint8_t *p, uint64_t v) { for (int i = 0; i < 8; i++) p[i] = (uint8_t)(v >> (56 - 8 * i)); }

/* verify_cell_kzg_proof_batch.  r_out (nullable): the batch challenge r, 32 bytes big-endian (n >= 1). */
int kzgco_verify_cell_kzg_proof_batch(const uint8_t *cb, const uint64_t *cell_indices, const uint8_t *cells, const uint8_t *pb, size_t n,
                                     int *ok, uint8_t *r_out) {
    if (n == 0) { *ok = 1; return KZG_OK; }
    if (!S.ready) return KZG_BADSETUP;
    for (size_t k = 0; k < n; k++) if (cell_indices[k] >= CELLS_PER_EXT_BLOB) return KZG_BADARGS;
    fr *vals = (fr *)malloc(n * FE_PER_CELL * sizeof(fr));
    g1_aff *P = (g1_aff *)malloc(n * sizeof(g1_aff)), *U = (g1_aff *)malloc(n * sizeof(g1_aff));
    size_t *ci = (size_t *)malloc(n * sizeof(size_t)), *first = (size_t *)malloc(n * sizeof(size_t)), m = 0;
    int rc = KZG_OK;
    for (size_t k = 0; k < n && !rc; k++) rc = cell_values(vals + k * FE_PER_CELL, cells + k * BYTES_PER_CELL);
    for (size_t k = 0; k < n && !rc; k++) rc = safe_g1_from_bytes(&P[k], pb + 48 * k);
    /* deduplicate the commitments by their bytes, first-occurrence order */
    for (size_t k = 0; k < n && !rc; k++) {
        size_t u = 0;
        while (u < m && memcmp(cb + 48 * first[u], cb + 48 * k, 48)) u++;
        if (u == m) { rc = safe_g1_from_bytes(&U[m], cb + 48 * k); first[m++] = k; }
        ci[k] = u;
    }
    if (!rc) rc = ensure_monomial();
    if (!rc) {
        /* r = hash_to_bls_field(transcript) */
        size_t len = 48 + 48 * m + n * (16 + BYTES_PER_CELL + 48);
        uint8_t *buf = (uint8_t *)malloc(len), *p = buf, dig[32];
        memcpy(p, "RCKZGCBATCH__V1_", 16); put_u64be(p + 16, N_FE); put_u64be(p + 24, FE_PER_CELL);
        put_u64be(p + 32, m); put_u64be(p + 40, n); p += 48;
        for (size_t u = 0; u < m; u++, p += 48) memcpy(p, cb + 48 * first[u], 48);
        for (size_t k = 0; k < n; k++) {
            put_u64be(p, ci[k]); put_u64be(p + 8, cell_indices[k]); p += 16;
            memcpy(p, cells + k * BYTES_PER_CELL, BYTES_PER_CELL); p += BYTES_PER_CELL;
            memcpy(p, pb + 48 * k, 48); p += 48;
        }
        sha256(dig, buf, len); free(buf);
        fr r, rk; scalar_from_bytes_unchecked(&r, dig);
        if (r_out) fr_to_bytes_be(r_out, &r);
        /* scalars: r^k for LL, r^k h_k^64 for RLP, sum of r^k per commitment for RLC; per-index sums of r^k * cell values */
        uint64_t (*s_ll)[4] = (uint64_t (*)[4])malloc(32 * n), (*s_rlp)[4] = (uint64_t (*)[4])malloc(32 * n);
        uint64_t (*s_rlc)[4] = (uint64_t (*)[4])malloc(32 * m);
        fr *w_c = (fr *)calloc(m, sizeof(fr)), *agg = (fr *)calloc(CELLS_PER_EXT_BLOB * FE_PER_CELL, sizeof(fr));
        int used[CELLS_PER_EXT_BLOB] = {0};
        fr_set_one(&rk);
        for (size_t k = 0; k < n; k++) {
            fr h, s, t; int idx = (int)cell_indices[k];
            cell_shift(&h, idx); omega_pow(&s, &h, FE_PER_CELL);
            fr_to_raw(s_ll[k], &rk);
            fr_mul(&t, &rk, &s); fr_to_raw(s_rlp[k], &t);
            fr_add(&w_c[ci[k]], &w_c[ci[k]], &rk);
            used[idx] = 1;
            for (int j = 0; j < FE_PER_CELL; j++) { fr_mul(&t, &rk, &vals[k * FE_PER_CELL + j]); fr_add(&agg[idx * FE_PER_CELL + j], &agg[idx * FE_PER_CELL + j], &t); }
            fr_mul(&rk, &rk, &r);
        }
        for (size_t u = 0; u < m; u++) fr_to_raw(s_rlc[u], &w_c[u]);
        /* RLI = sum_m c_m [tau^m]G1, c = sum over the distinct indices of the interpolation coefficients of the aggregated values */
        fr c[FE_PER_CELL], ic[FE_PER_CELL];
        for (int j = 0; j < FE_PER_CELL; j++) fr_set_zero(&c[j]);
        for (int idx = 0; idx < CELLS_PER_EXT_BLOB; idx++) {
            if (!used[idx]) continue;
            cell_interpolate(ic, agg + idx * FE_PER_CELL, idx);
            for (int j = 0; j < FE_PER_CELL; j++) fr_add(&c[j], &c[j], &ic[j]);
        }
        uint64_t s_rli[FE_PER_CELL][4];
        for (int j = 0; j < FE_PER_CELL; j++) fr_to_raw(s_rli[j], &c[j]);
        g1 ll, rlc, rlp, rli, rhs;
        g1_msm(&ll, P, (const uint64_t (*)[4])s_ll, n);
        g1_msm(&rlc, U, (const uint64_t (*)[4])s_rlc, m);
        g1_msm(&rlp, P, (const uint64_t (*)[4])s_rlp, n);
        g1_msm(&rli, S.g1_monomial, (const uint64_t (*)[4])s_rli, FE_PER_CELL);
        g1_neg(&rli, &rli); g1_add(&rhs, &rlc, &rli); g1_add(&rhs, &rhs, &rlp);
        g1_aff ll_a, rhs_a; g1_to_aff(&ll_a, &ll); g1_to_aff(&rhs_a, &rhs);
        *ok = pairings_verify(&ll_a, &S.tau64_g2, &rhs_a, &S.g2_gen);       /* e(LL, [tau^64]G2) == e(RLC - RLI + RLP, G2) */
        free(s_ll); free(s_rlp); free(s_rlc); free(w_c); free(agg);
    }
    free(vals); free(P); free(U); free(ci); free(first);
    return rc;
}

/* recover_cells_and_kzg_proofs, cells only: the spec's argument checks, recover_polynomialcoeff literally (zeros at the missing
 * cells, the vanishing polynomial Z(X) = z(X^64), (E Z) on the 8192-point domain, inverse transform, coset transforms with the shift
 * PRIMITIVE_ROOT_OF_UNITY = 7, division by Z on the coset, first 4096 coefficients), then the cells of the recovered polynomial.
 * (Its proofs are those of the blob formed by the recovered cells 0..63: kzgco_compute_cell_kzg_proof.) */
static void coset_shift(fr *a, int n, const fr *factor) {
    fr x; fr_set_one(&x);
    for (int i = 0; i < n; i++) { fr_mul(&a[i], &a[i], &x); fr_mul(&x, &x, factor); }
}
int kzgco_recover_cells(const uint64_t *indices, const uint8_t *cells, size_t n, uint8_t *cells_out /* 128 x 2048 */) {
    if (!S.ready) return KZG_BADSETUP;
    if (n < CELLS_PER_EXT_BLOB / 2 || n > CELLS_PER_EXT_BLOB) return KZG_BADARGS;
    int present[CELLS_PER_EXT_BLOB] = {0};
    for (size_t j = 0; j < n; j++) {
        if (indices[j] >= CELLS_PER_EXT_BLOB || present[indices[j]]) return KZG_BADARGS;
        present[indices[j]] = 1;
    }
    fr *rbo = (fr *)calloc(N_EXT, sizeof(fr)), *E = (fr *)malloc(N_EXT * sizeof(fr)), *Z = (fr *)calloc(N_EXT, sizeof(fr));
    fr *Zev = (fr *)malloc(N_EXT * sizeof(fr)), *Zcos = (fr *)malloc(N_EXT * sizeof(fr));
    int rc = KZG_OK;
    /* extended_evaluation_rbo, then bit_reversal_permutation */
    for (size_t j = 0; j < n && !rc; j++)
        for (int i = 0; i < FE_PER_CELL && !rc; i++) rc = safe_scalar_from_bytes(&rbo[indices[j] * FE_PER_CELL + i], cells + j * BYTES_PER_CELL + 32 * i);
    if (!rc) {
        for (int i = 0; i < N_EXT; i++) E[i] = rbo[bitrev((uint32_t)i, 13)];
        /* construct_vanishing_polynomial: prod over the missing k of (Y - omega128^rev7(k)), spread to X^(64 i) */
        fr w128, shortz[CELLS_PER_EXT_BLOB + 1], root, t;
        int deg = 0;
        omega_pow(&w128, &S.omega8192, FE_PER_CELL);
        fr_set_one(&shortz[0]);
        for (int k = 0; k < CELLS_PER_EXT_BLOB; k++) {
            if (present[k]) continue;
            omega_pow(&root, &w128, bitrev((uint32_t)k, 7));
            fr_set_zero(&shortz[deg + 1]);
            for (int i = deg + 1; i >= 1; i--) { fr_mul(&t, &shortz[i], &root); fr_sub(&shortz[i], &shortz[i - 1], &t); }   /* p * (X - root) */
            fr_mul(&t, &shortz[0], &root); fr_set_zero(&shortz[0]); fr_sub(&shortz[0], &shortz[0], &t);
            deg++;
        }
        for (int i = 0; i <= deg; i++) Z[i * FE_PER_CELL] = shortz[i];
        memcpy(Zev, Z, N_EXT * sizeof(fr));
        fr_dft(Zev, N_EXT, &S.omega8192);
        for (int i = 0; i < N_EXT; i++) fr_mul(&E[i], &E[i], &Zev[i]);          /* (E Z) on the domain */
        fr_idft(E, N_EXT, &S.omega8192);                                        /* (P Z) coefficients */
        fr seven, seven_inv;
        fr_from_u64(&seven, 7); fr_inv(&seven_inv, &seven);
        coset_shift(E, N_EXT, &seven); fr_dft(E, N_EXT, &S.omega8192);        /* (P Z) on the coset */
        memcpy(Zcos, Z, N_EXT * sizeof(fr));
        coset_shift(Zcos, N_EXT, &seven); fr_dft(Zcos, N_EXT, &S.omega8192);  /* Z on the coset */
        for (int i = 0; i < N_EXT; i++) { fr_inv(&t, &Zcos[i]); fr_mul(&E[i], &E[i], &t); }
        fr_idft(E, N_EXT, &S.omega8192); coset_shift(E, N_EXT, &seven_inv);   /* P coefficients */
        /* compute_cells of the first 4096 coefficients */
        for (int i = N_FE; i < N_EXT; i++) fr_set_zero(&E[i]);
        fr_dft(E, N_EXT, &S.omega8192);
        for (int i = 0; i < N_EXT; i++) fr_to_bytes_be(cells_out + 32 * (size_t)i, &E[bitrev((uint32_t)i, 13)]);
    }
    free(rbo); free(E); free(Z); free(Zev); free(Zcos);
    return rc;
}
