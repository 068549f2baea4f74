// Group arithmetic of the batch verifier (verify_batch.cu) that the CPU test-suite also compiles for the host
// (tests/host_harness/verify_batch_host.cc pins it against the oracle).
#pragma once
#include "ec.cuh"

namespace b200 {

// k * p for an nbits-bit integer k given as little-endian 32-bit words: double-and-add, MSB first.  The batch
// verifier runs it with the 128-bit coefficients (rho_i * Ar_i) and with S = sum_i rho_i mod r (S * alpha).
template <class F>
B200_HD XYZZ<F> scalar_mul_bits(const Affine<F>& p, const uint32_t* k, int nbits) {
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int i = nbits - 1; i >= 0; i--) {
    acc.dbl();
    if ((k[i >> 5] >> (i & 31)) & 1) acc.madd(p);
  }
  return acc;
}

// the 128-bit coefficient stored as two little-endian 64-bit words, as 32-bit limbs
B200_HD void coeff_limbs(const uint64_t* c, uint32_t out[4]) {
  out[0] = (uint32_t)c[0];
  out[1] = (uint32_t)(c[0] >> 32);
  out[2] = (uint32_t)c[1];
  out[3] = (uint32_t)(c[1] >> 32);
}

}  // namespace b200
