// CPU unit test of the batch verifier's split tail (k_final.cu window_miller_kernel / split_final_kernel) on the pairing engine's
// sequential reference executors: for MSM window points A_w, B_w (w < 16), FE(prod_w Miller_w) against the check of the combined
// points A = sum 256^w A_w, B = sum 256^w B_w,
//   e(B, Q1) e(-A, Q2)  ==  FE( prod_w f_{[256^w]Q1}(B_w) f_{[256^w]Q2}(-A_w) ),
// compared as canonical Fp12 coefficients, with identity windows (one pair or both pairs dropped) and the [s]G fold of window 0.
// Q1 = G2, Q2 = [t]G2 with a random t; B_w = [t]A_w makes the relation true, a perturbed window makes it false.
//   final_split_host split <seed>          one line per case: "case <name> verdict <0|1> split <0|1> gt_equal <0|1>"
//   final_split_host lines <setup.bin>     the shifted line tables of the setup's G2 points, hex, in DeviceTables::lines29w layout
// Built and run by tests/test_final_split_host.py and tests/test_gpu_final_split.py.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "verify.cuh"
#include "vliw29.cuh"
using namespace kzgb200;

static void lines29(vliw29::LineCoeffs29* out, const G2Affine& Q) {
  static LineCoeffs lc[kMillerSteps];
  prepare_g2(lc, Q);
  for (int k = 0; k < kMillerSteps; k++)
    for (int e = 0; e < 6; e++) {
      const Fp2& f2 = e < 2 ? lc[k].A : (e < 4 ? lc[k].B : lc[k].C);
      out[k].v[e] = f29::from_fp((e & 1) ? f2.c1 : f2.c0);
    }
}
static G2Affine shifted(const G2Affine& Q, int w) {   // [256^w]Q
  G2 a = G2::from_affine(Q);
  for (int k = 0; k < 8 * w; k++) a = a.dbl();
  return g2_to_affine(a);
}
static uint64_t rng_state = 1;
static uint64_t rnd64() { rng_state = rng_state * 6364136223846793005ull + 1442695040888963407ull; return rng_state ^ (rng_state >> 29); }
static G1 mul_g(uint64_t k) { uint32_t kk[2] = {(uint32_t)k, (uint32_t)(k >> 32)}; return scalar_mul_affine(g1_generator(), kk, 64); }
static G1 mul(const G1& p, uint64_t k) { uint32_t kk[2] = {(uint32_t)k, (uint32_t)(k >> 32)}; return scalar_mul(p, kk, 64); }

int main(int argc, char** argv) {
  if (argc < 3) return 2;
  if (!strcmp(argv[1], "lines")) {
    FILE* f = fopen(argv[2], "rb");
    std::vector<uint8_t> s(12 + 4096 * 48 + 65 * 96);
    if (!f || fread(s.data(), 1, s.size(), f) != s.size()) return 2;
    fclose(f);
    static vliw29::LineCoeffs29 tab[kMillerSteps];
    for (int q = 0; q < 2; q++) {
      G2Affine Q;
      if (!g2_from_compressed_unchecked(Q, s.data() + 12 + 4096 * 48 + 96 * q)) return 3;
      for (int w = 1; w < 16; w++) {
        lines29(tab, shifted(Q, w));
        const uint8_t* b = reinterpret_cast<const uint8_t*>(tab);
        for (size_t i = 0; i < sizeof(tab); i++) printf("%02x", b[i]);
      }
    }
    printf("\n");
    return 0;
  }
  rng_state = strtoull(argv[2], nullptr, 0);
  const uint64_t t = rnd64() | 1;
  const G2Affine Q1 = g2_generator();
  uint32_t tk[2] = {(uint32_t)t, (uint32_t)(t >> 32)};
  const G2Affine Q2 = g2_to_affine(scalar_mul_affine(Q1, tk, 64));
  static vliw29::LineCoeffs29 L[2][16][kMillerSteps];
  for (int w = 0; w < 16; w++) { lines29(L[0][w], shifted(Q1, w)); lines29(L[1][w], shifted(Q2, w)); }
  std::vector<f29::F29> regs(vliw29::kTotalRegs);
  vliw29::Lanes lanes{0, 1, vliw29::default_tables()};
  const char* names[4] = {"true", "true_dense", "false_single_pair", "false_b_identity"};
  for (int c = 0; c < 4; c++) {
    G1 A[16], W1[16], W2[16];
    const G1 sg = mul_g(rnd64());
    for (int w = 0; w < 16; w++) {
      A[w] = (c != 1 && w % 5 == 2) ? G1::identity() : mul_g(rnd64());     // identity windows: both pairs dropped
      W1[w] = mul_g(rnd64());
      W2[w] = mul(A[w], t).add(W1[w].neg());                                 // W1 + W2 = [t]A_w
      if (w == 0) W2[w] = W2[w].add(sg);                                     // ... + [s]G, folded out of window 0 below
    }
    if (c == 2) W2[7] = W2[7].add(mul_g(1));      // A_7 = identity, B_7 = G: the one-pair script
    if (c == 3) W2[9] = W1[9].neg();              // B_9 = identity, A_9 live: the pair in slot 1 alone
    G1 B[16];
    for (int w = 0; w < 16; w++) { B[w] = W1[w].add(W2[w]); if (w == 0) B[w] = B[w].add(sg.neg()); }
    // combined points (Horner) and the single check
    G1 Acc = G1::identity(), Bcc = G1::identity();
    for (int w = 15; w >= 0; w--) {
      for (int k = 0; k < 8; k++) { Acc = Acc.dbl(); Bcc = Bcc.dbl(); }
      Acc = Acc.add(A[w]); Bcc = Bcc.add(B[w]);
    }
    Fp gt_old[12], gt_new[12];
    const bool v_old = vliw29::coop_pairing_product_is_one(regs.data(), g1_to_affine(Bcc), L[0][0], g1_to_affine(Acc.neg()), L[1][0], lanes, gt_old);
    // split: per-window Miller values, their product, one final exponentiation
    static f29::F29 fw[16][12];
    for (int w = 0; w < 16; w++) {
      vliw29::coop_miller(regs.data(), g1_to_affine(B[w]), L[0][w], g1_to_affine(A[w].neg()), L[1][w], lanes);
      for (int i = 0; i < 12; i++) fw[w][i] = regs[vliw29::kRegF + i];
    }
    for (int i = 0; i < 12; i++) regs[vliw29::kRegF + i] = fw[0][i];
    for (int w = 1; w < 16; w++) {
      for (int i = 0; i < 12; i++) regs[vliw29::kRegG + i] = fw[w][i];
      vliw29::run(vliw29::kProg_f12_mul, regs.data(), lanes);
    }
    const bool v_new = vliw29::coop_final_exp_is_one(regs.data(), lanes, gt_new);
    bool eq = true;
    for (int i = 0; i < 12; i++) eq = eq && gt_old[i] == gt_new[i];
    printf("case %s verdict %d split %d gt_equal %d\n", names[c], v_old ? 1 : 0, v_new ? 1 : 0, eq ? 1 : 0);
  }
  return 0;
}
