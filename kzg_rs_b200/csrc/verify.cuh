// Per-proof verification logic shared by the kernels (and unit-tested on the host).
// Mirrors KzgProof::verify_kzg_proof (reference src/kzg_proof.rs:353-397) with the pairing equation moved
// to the G1 side so both G2 arguments are setup constants:
//   e(C - [y]G, G2) == e(pi, [tau]G2 - [z]G2)   <=>   e(C - [y]G + [z]pi, G2) * e(-pi, [tau]G2) == 1
// (G1, G2 have prime order and e is non-degenerate; identity points contribute 1 on both sides).
#pragma once
#include "pairing.cuh"
#include "glv.cuh"

namespace kzgb200 {

enum Verdict : uint8_t { kFalse = 0, kTrue = 1, kBadArgs = 2, kPending = 3 /* internal: many-tuple path, not yet decided */ };

// 32 big-endian bytes -> raw little-endian limbs
KZG_HD void be32_to_limbs(uint32_t* l, const uint8_t* b) {
    for (int i = 0; i < 8; i++) {
        const uint8_t* p = b + 4 * (7 - i);
        l[i] = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
    }
}
KZG_HD void limbs_to_be32(uint8_t* b, const uint32_t* l) {
    for (int i = 0; i < 8; i++) {
        uint8_t* p = b + 4 * (7 - i);
        p[0] = (uint8_t)(l[i] >> 24); p[1] = (uint8_t)(l[i] >> 16); p[2] = (uint8_t)(l[i] >> 8); p[3] = (uint8_t)l[i];
    }
}
// safe_scalar_affine_from_bytes (kzg_proof.rs:27-43): canonical raw limbs, false if >= q
KZG_HD bool scalar_from_be32_checked(Fr& raw, const uint8_t* b) {
    be32_to_limbs(raw.l, b);
    return !raw.geq_modulus();
}

struct PairingTables {
    LineCoeffs g2_gen[kMillerSteps];   // lines of g2_points[0] (the G2 generator)
    LineCoeffs tau_g2[kMillerSteps];   // lines of g2_points[1] = [tau]G2
};

// e(X, G2) * e(-Pi, [tau]G2) == 1 for already-parsed points
KZG_NI bool kzg_pairing_check(const G1Affine& X, const G1Affine& pi, const PairingTables* T) {
    G1Affine npi = pi;
    if (!npi.inf) npi.y = npi.y.neg();
    return pairing_product_is_one(X, T->g2_gen, npi, T->tau_g2);
}
// C - [y]G + [z]pi for parsed inputs; z, y canonical raw limbs
KZG_NI G1Affine kzg_lhs_point(const G1Affine& C, const Fr& z_raw, const Fr& y_raw, const G1Affine& pi) {
    G1 acc = scalar_mul_affine(g1_generator(), y_raw.l, 255).neg();
    acc = acc.add_mixed(C);
    acc = acc.add(scalar_mul_affine(pi, z_raw.l, 255));
    return g1_to_affine(acc);
}
// [k]P by the GLV split k = k1 + k2 x^2 (glv.cuh) with Shamir's trick over {P, -phi(P), P - phi(P)}: 128 doublings and ~96
// additions instead of 2 x (255 + 128).  k: canonical raw limbs.
KZG_HD G1 glv_mul(const G1Affine& p, const Fr& k_raw) {
    uint32_t k1[4], k2[4];
    glv_split(k_raw.l, k1, k2);
    G1Affine q = glv_endo_neg(p);
    G1 both = G1::from_affine(p).add_mixed(q), acc = G1::identity();
    for (int i = 127; i >= 0; i--) {
        acc = acc.dbl();
        uint32_t b1 = (k1[i >> 5] >> (i & 31)) & 1u, b2 = (k2[i >> 5] >> (i & 31)) & 1u;
        if (b1 & b2) acc = acc.add(both);
        else if (b1) acc = acc.add_mixed(p);
        else if (b2) acc = acc.add_mixed(q);
    }
    return acc;
}
// The same point for the batched per-tuple path (BASELINE config 5): [y]G from the fixed-base table of the generator
// (gen_table[w][d-1] = [d 16^w]G: 64 mixed additions, no doublings) and [z]pi by glv_mul.
KZG_NI G1 kzg_lhs_point_fast(const G1Affine& C, const Fr& z_raw, const Fr& y_raw, const G1Affine& pi, const G1Affine (*gen_table)[15]) {
    G1 acc = G1::from_affine(C);
    for (int w = 0; w < 64; w++) {
        uint32_t d = (y_raw.l[w >> 3] >> (4 * (w & 7))) & 15u;
        if (d) { G1Affine t = gen_table[w][d - 1]; t.y = t.y.neg(); acc = acc.add_mixed(t); }
    }
    if (!pi.inf) acc = acc.add(glv_mul(pi, z_raw));
    return acc;
}
// parse order z, y, commitment, proof as kzg_proof.rs:360-383
KZG_NI Verdict verify_kzg_proof_one(const uint8_t* c48, const uint8_t* z32, const uint8_t* y32, const uint8_t* p48,
                                    const PairingTables* T) {
    Fr z, y;
    G1Affine C, pi;
    if (!scalar_from_be32_checked(z, z32)) return kBadArgs;
    if (!scalar_from_be32_checked(y, y32)) return kBadArgs;
    if (!g1_from_compressed(C, c48, true)) return kBadArgs;
    if (!g1_from_compressed(pi, p48, true)) return kBadArgs;
    return kzg_pairing_check(kzg_lhs_point(C, z, y, pi), pi, T) ? kTrue : kFalse;
}

}  // namespace kzgb200
