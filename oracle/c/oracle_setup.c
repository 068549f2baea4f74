/* The C restatement of gnark's setupABC (TEST INFRASTRUCTURE ONLY, see oracle.c's header), built on the field
 * arithmetic of oracle.c into its own library (oracle/setup.mk -> _build/liboracle_setup.so):
 * gnark v0.11.0 backend/groth16/bn254/setup.go setupABC, reached from the reference at mt.go:448.
 *
 * Literally gnark's algorithm, deliberately NOT the GPU's (which takes the Lagrange values from one inverse NTT of
 * the tau powers): t_j = tau - w^j for the m constraints, one batch inversion (Montgomery's trick), the recurrence
 *   L_0 = (tau^N - 1) / N / (tau - 1),   L_{j+1} = w L_j t_j / t_{j+1},
 * and a constraint-major accumulation A[wire] += coeff * L_j over the terms of L (B over R, C over O).
 * Single-threaded, like gnark's.  Matrices as b200g16_r1cs_desc holds them (CSR by constraint, Term{CID, VID}).
 * Returns -1 when tau^N = 1 (a t_j is zero: gnark's batch inversion would divide by zero) or memory runs out. */
#include "oracle.c"

int oracle_setup_abc(size_t m, size_t n_wires, const u64* coeffs, const u64* const rows[3], const uint32_t* const wires[3],
                     const uint32_t* const cids[3], const u64* tau_mont, u64* a_out, u64* b_out, u64* c_out) {
  int L = 0;
  while (((size_t)1 << L) < m) L++;
  const size_t n = (size_t)1 << L;
  const fe tau = *(const fe*)tau_mont;
  fe w;
  domain_gen(L, 0, &w);
  fe* t = (fe*)malloc(m * sizeof(fe));
  fe* ti = (fe*)malloc(m * sizeof(fe));
  if (!t || !ti) { free(t); free(ti); return -1; }
  fe wj = FR_ONE;
  for (size_t j = 0; j < m; j++) {            /* t_j = tau - w^j */
    fr_sub(&t[j], &tau, &wj);
    if (fe_is_zero(&t[j])) { free(t); free(ti); return -1; }
    fr_mul(&wj, &wj, &w);
  }
  /* batch inversion: prefix products, one inverse, walk back */
  fe acc = FR_ONE;
  for (size_t j = 0; j < m; j++) { ti[j] = acc; fr_mul(&acc, &acc, &t[j]); }
  fe inv;
  fr_inv(&inv, &acc);
  for (size_t j = m; j-- > 0;) { fr_mul(&ti[j], &ti[j], &inv); fr_mul(&inv, &inv, &t[j]); }
  /* L_0 = (tau^N - 1) / N * 1 / (tau - 1) */
  fe tn = tau, nn, ninv, lag;
  for (int i = 0; i < L; i++) fr_mul(&tn, &tn, &tn);
  fr_sub(&tn, &tn, &FR_ONE);
  fr_from_u64(&nn, (u64)n);
  fr_inv(&ninv, &nn);
  fr_mul(&lag, &tn, &ninv);
  fr_mul(&lag, &lag, &ti[0]);
  u64* outs[3] = {a_out, b_out, c_out};
  for (int k = 0; k < 3; k++) memset(outs[k], 0, n_wires * sizeof(fe));
  const fe* cf = (const fe*)coeffs;
  for (size_t j = 0; j < m; j++) {
    for (int k = 0; k < 3; k++) {
      fe* o = (fe*)outs[k];
      for (u64 e = rows[k][j]; e < rows[k][j + 1]; e++) {
        fe p;
        fr_mul(&p, &cf[cids[k][e]], &lag);
        fr_add(&o[wires[k][e]], &o[wires[k][e]], &p);
      }
    }
    if (j + 1 < m) {                          /* L_{j+1} = w L_j t_j / t_{j+1} */
      fr_mul(&lag, &lag, &w);
      fr_mul(&lag, &lag, &t[j]);
      fr_mul(&lag, &lag, &ti[j + 1]);
    }
  }
  free(t);
  free(ti);
  return 0;
}
