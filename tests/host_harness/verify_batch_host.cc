// Test harness (NOT part of libb200g16): compiles gnark_whir_b200/csrc/verify_batch.cuh for the host with g++ so
// the CPU test-suite can pin the scalar multiplication the batch verifier's kernels run (rho_i * Ar_i with 128-bit
// coefficients in k_batch_proofs, S * alpha with a 254-bit S in k_fixed_pairs) against the oracle's.
#include <cstring>

#include "verify_batch.cuh"

using namespace b200;

extern "C" {

// out = c * p, c a 128-bit coefficient as two little-endian words (the layout b200g16_verify_batch takes)
void host_g1_mul_coeff(const uint64_t* p, const uint64_t* c, uint64_t* out) {
  Affine<Fp> a;
  memcpy(&a, p, sizeof(a));
  uint32_t k[4];
  coeff_limbs(c, k);
  Affine<Fp> r = scalar_mul_bits(a, k, 128).to_affine();
  memcpy(out, &r, sizeof(r));
}

// out = k * p, k < 2^nbits given as four little-endian words
void host_g1_mul_bits(const uint64_t* p, const uint64_t* k, int nbits, uint64_t* out) {
  Affine<Fp> a;
  memcpy(&a, p, sizeof(a));
  uint32_t w[8];
  for (int i = 0; i < 4; i++) {
    w[2 * i] = (uint32_t)k[i];
    w[2 * i + 1] = (uint32_t)(k[i] >> 32);
  }
  Affine<Fp> r = scalar_mul_bits(a, w, nbits).to_affine();
  memcpy(out, &r, sizeof(r));
}
}
