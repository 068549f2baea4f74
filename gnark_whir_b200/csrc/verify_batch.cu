// Batch groth16.Verify: k proofs against one verifying key in one call, by the small-exponent batch test
// (Bellare, Garay, Rabin).  With nonzero 128-bit coefficients rho_i, and tau_i for the BSB22 proofs of knowledge,
// the batch is accepted iff every proof point is valid and
//
//   prod_i e(rho_i Ar_i, Bs_i) * e(-S alpha, beta) * e(-(S K_0 + sum_j y_j K_j + sum_i rho_i D_i), gamma)
//     * e(-sum_i rho_i Krs_i, delta) * e(sum_i tau_i D_i, GSigmaNeg) * e(sum_i tau_i P_i, G) == 1,
//   S = sum_i rho_i,  y_j = sum_i rho_i x_ij  (mod r)
//
// k + 3 (k + 5 with a commitment) Miller loops and ONE final exponentiation instead of 4k (6k) Miller loops and k
// (2k) final exponentiations.  The main equation and the proof-of-knowledge equation take independent coefficients:
// with shared ones an error in one can cancel an error in the other.
//   k_batch_proofs    one thread per proof: point checks, rho_i Ar_i (128-bit double-and-add), Miller loop -> f_i
//   k_fold (+ final)  S and y_j: a partial sum per CTA and column over the k dimension, then one reduction per column
//   msm_device<Fp>    sum rho_i Krs_i;  [K_0..K_{n_k-1}, D_1..D_k] . [S, y, rho];  sum tau_i D_i;  sum tau_i P_i
//   k_fixed_pairs     the 3 (5) Miller loops against the vk's G2 points; forms -S alpha itself
//   k_f12_product     shared-memory product tree per CTA, relaunched until one value is left
//   k_final_exp       final exponentiation, == 1, and no invalid point anywhere in the batch
// A failing batch with ok_each requested falls back to the per-proof check: k_batch_lsum forms each proof's
// L_i = K_0 + sum_j x_ij K_j + D_i and pairing_products (verify.cu) evaluates the very products b200g16_verify
// evaluates for that proof, one CTA per product.
#include "common.cuh"
#include "host_copy.cuh"
#include "pairing.cuh"
#include "verify_batch.cuh"

namespace b200 {
template <class F>
int msm_device(b200g16_ctx* ctx, const Affine<F>* d_bases, const MsmTable* tab, const Fr* d_scalars, size_t n,
               Affine<F>* out);
int pairing_products(b200g16_ctx* ctx, const G1Affine* P, const G2Affine* Q, const uint32_t* flags,
                     const uint32_t* first, int n_prod, bool with_cofactor, Fp12* gt, int* is_one, int* valid);

constexpr int BV_PROOF_THREADS = 64;   // per-proof kernels: long serial chains, ~few hundred registers of state
constexpr int BV_FOLD_THREADS = 256;
constexpr int BV_TREE_THREADS = 64;    // 64 Fp12 = 24 KiB of shared memory per CTA
constexpr size_t BV_MAX_K = (size_t)1 << 20;
constexpr uint32_t BV_MAX_GRID_Y = 65535;

__global__ void __launch_bounds__(BV_PROOF_THREADS) k_batch_proofs(const G1Affine* __restrict__ ar,
                                                                   const G2Affine* __restrict__ bs,
                                                                   const G1Affine* __restrict__ krs,
                                                                   const G1Affine* __restrict__ com,
                                                                   const G1Affine* __restrict__ pok,
                                                                   const uint64_t* __restrict__ coeffs, uint32_t k,
                                                                   Fp12* __restrict__ f, int* __restrict__ valid,
                                                                   int* __restrict__ any_bad) {
  const uint32_t i = blockIdx.x * BV_PROOF_THREADS + threadIdx.x;
  if (i >= k) return;
  const G1Affine a = ar[i];
  const G2Affine b = bs[i];
  bool ok = g1_on_curve(a) && g1_on_curve(krs[i]) && g2_in_subgroup(b);
  if (com) ok = ok && g1_on_curve(com[i]) && g1_on_curve(pok[i]);
  uint32_t rho[4];
  coeff_limbs(coeffs + 2 * (size_t)i, rho);
  f[i] = miller_loop(scalar_mul_bits(a, rho, 128).to_affine(), b);
  valid[i] = ok ? 1 : 0;
  if (!ok) atomicOr(any_bad, 1);
}

template <int T>
__device__ void fr_block_sum(Fr* sh, Fr v) {
  sh[threadIdx.x] = v;
  __syncthreads();
  for (int s = T / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] = Fr::add(sh[threadIdx.x], sh[threadIdx.x + s]);
    __syncthreads();
  }
}

// Column j of the fold (j = 0: rho_i, giving S; j >= 1: rho_i x_{i,j-1}, giving y_j): one partial sum per CTA in
// partial[j * gridDim.x + blockIdx.x].  Column 0 also writes rho_i and tau_i in Montgomery form, the MSM scalars.
__global__ void __launch_bounds__(BV_FOLD_THREADS) k_fold(const uint64_t* __restrict__ coeffs, const Fr* __restrict__ pub,
                                                          uint32_t k, uint32_t n_pub, int with_tau,
                                                          Fr* __restrict__ rho_mont, Fr* __restrict__ tau_mont,
                                                          Fr* __restrict__ partial) {
  __shared__ Fr sh[BV_FOLD_THREADS];
  const uint32_t i = blockIdx.x * BV_FOLD_THREADS + threadIdx.x;
  for (uint32_t j = blockIdx.y; j <= n_pub; j += gridDim.y) {
    Fr v = Fr::zero();
    if (i < k) {
      uint32_t c[4];
      coeff_limbs(coeffs + 2 * (size_t)i, c);
      Fr rho = Fr::zero();
      for (int w = 0; w < 4; w++) rho.l[w] = c[w];
      rho = Fr::to_mont(rho);
      if (j == 0) {
        v = rho;
        rho_mont[i] = rho;
        if (with_tau) {
          coeff_limbs(coeffs + 2 * ((size_t)k + i), c);
          Fr tau = Fr::zero();
          for (int w = 0; w < 4; w++) tau.l[w] = c[w];
          tau_mont[i] = Fr::to_mont(tau);
        }
      } else {
        v = Fr::mul(rho, pub[(size_t)i * n_pub + j - 1]);
      }
    }
    fr_block_sum<BV_FOLD_THREADS>(sh, v);
    if (threadIdx.x == 0) partial[(size_t)j * gridDim.x + blockIdx.x] = sh[0];
    __syncthreads();
  }
}

// out[j] = sum of the nblk partial sums of column j
__global__ void __launch_bounds__(BV_FOLD_THREADS) k_fold_final(const Fr* __restrict__ partial, uint32_t nblk,
                                                                uint32_t n_cols, Fr* __restrict__ out) {
  __shared__ Fr sh[BV_FOLD_THREADS];
  for (uint32_t j = blockIdx.x; j < n_cols; j += gridDim.x) {
    Fr v = Fr::zero();
    for (uint32_t b = threadIdx.x; b < nblk; b += BV_FOLD_THREADS) v = Fr::add(v, partial[(size_t)j * nblk + b]);
    fr_block_sum<BV_FOLD_THREADS>(sh, v);
    if (threadIdx.x == 0) out[j] = sh[0];
    __syncthreads();
  }
}

// Miller loops of the n fixed pairs; pair 0 arrives as (alpha, beta) and is evaluated as (-S alpha, beta)
__global__ void __launch_bounds__(32) k_fixed_pairs(const G1Affine* __restrict__ P, const G2Affine* __restrict__ Q,
                                                    int n, const Fr* __restrict__ S, Fp12* __restrict__ f) {
  const int t = threadIdx.x;
  if (t >= n) return;
  G1Affine p = P[t];
  if (t == 0) {
    const Fr s = Fr::from_mont(*S);
    p = scalar_mul_bits(p, s.l, 254).to_affine();
    p.y = Fp::neg(p.y);
  }
  f[t] = miller_loop(p, Q[t]);
}

// out[b] = in[b T] * ... * in[b T + T - 1] (indexes >= n count as one)
__global__ void __launch_bounds__(BV_TREE_THREADS) k_f12_product(const Fp12* __restrict__ in, uint32_t n,
                                                                 Fp12* __restrict__ out) {
  __shared__ Fp12 sh[BV_TREE_THREADS];
  const uint32_t i = blockIdx.x * BV_TREE_THREADS + threadIdx.x;
  sh[threadIdx.x] = i < n ? in[i] : f12_one();
  __syncthreads();
  for (int s = BV_TREE_THREADS / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] = f12_mul(sh[threadIdx.x], sh[threadIdx.x + s]);
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

// flags[0]: some proof point was invalid; flags[1] <- the batch is accepted
__global__ void __launch_bounds__(32) k_final_exp(const Fp12* __restrict__ f, int* __restrict__ flags) {
  if (threadIdx.x) return;
  flags[1] = (!flags[0] && f12_is_one(final_exponentiation(*f, false))) ? 1 : 0;
}

// L_i = K_0 + sum_j x_ij K_j + D_i, the point b200g16_verify pairs with gamma for proof i: one thread per proof,
// one doubling chain shared by all j (Straus).  pub is turned into canonical form in place.
__global__ void __launch_bounds__(BV_PROOF_THREADS) k_batch_lsum(const G1Affine* __restrict__ K, Fr* __restrict__ pub,
                                                                 uint32_t k, uint32_t n_pub,
                                                                 const G1Affine* __restrict__ com,
                                                                 G1Affine* __restrict__ L) {
  const uint32_t i = blockIdx.x * BV_PROOF_THREADS + threadIdx.x;
  if (i >= k) return;
  Fr* x = pub + (size_t)i * n_pub;
  for (uint32_t j = 0; j < n_pub; j++) x[j] = Fr::from_mont(x[j]);
  G1XYZZ acc = G1XYZZ::inf();
  for (int b = 253; b >= 0; b--) {
    acc.dbl();
    for (uint32_t j = 0; j < n_pub; j++)
      if ((x[j].l[b >> 5] >> (b & 31)) & 1) acc.madd(K[j + 1]);
  }
  acc.madd(K[0]);
  if (com) acc.madd(com[i]);
  L[i] = acc.to_affine();
}

static G1Affine g1_negate(G1Affine p) {
  p.y = Fp::neg(p.y);
  return p;
}

static unsigned bv_cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

struct BvEvents {
  cudaEvent_t e[7] = {};
  ~BvEvents() {
    for (cudaEvent_t x : e)
      if (x) cudaEventDestroy(x);
  }
};

// ok_each for a failing batch: every proof's own products, as b200g16_verify forms them
static int batch_per_proof(b200g16_ctx* ctx, const b200g16_vk_desc* vk, size_t k, const uint64_t* ar,
                           const uint64_t* bs, const uint64_t* krs, const uint64_t* commitments, const uint64_t* poks,
                           const G1Affine* d_L, uint8_t* ok_each) {
  const bool has_com = commitments != nullptr;
  std::vector<G1Affine> L(k);
  B200_CUDA(cudaMemcpyAsync(L.data(), d_L, k * sizeof(G1Affine), cudaMemcpyDeviceToHost, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  const int per = has_com ? 6 : 4, nprod_per = has_com ? 2 : 1;
  const size_t n_pairs = k * per, n_prod = k * nprod_per;
  std::vector<G1Affine> P(n_pairs);
  std::vector<G2Affine> Q(n_pairs);
  std::vector<uint32_t> flags(n_pairs), first(n_prod + 1);
  G1Affine alpha;
  G2Affine beta, gamma, delta, gsn, g;
  memcpy(&alpha, vk->g1_alpha, 64);
  memcpy(&beta, vk->g2_beta, 128);
  memcpy(&gamma, vk->g2_gamma, 128);
  memcpy(&delta, vk->g2_delta, 128);
  if (has_com) { memcpy(&gsn, vk->ped_g_sigma_neg, 128); memcpy(&g, vk->ped_g, 128); }
  const G1Affine nalpha = g1_negate(alpha);
  const uint32_t fl[6] = {3u, 0u, 1u, 0u, 1u, 1u};  // proof points are checked, vk points are trusted
  for (size_t i = 0; i < k; i++) {
    G1Affine* p = &P[i * per];
    G2Affine* q = &Q[i * per];
    G1Affine t;
    memcpy(&p[0], ar + 8 * i, 64);  memcpy(&q[0], bs + 16 * i, 128);
    p[1] = g1_negate(L[i]);         q[1] = gamma;
    memcpy(&t, krs + 8 * i, 64);
    p[2] = g1_negate(t);            q[2] = delta;
    p[3] = nalpha;                  q[3] = beta;
    if (has_com) {
      memcpy(&p[4], commitments + 8 * i, 64);  q[4] = gsn;
      memcpy(&p[5], poks + 8 * i, 64);         q[5] = g;
      first[2 * i] = (uint32_t)(i * per);
      first[2 * i + 1] = (uint32_t)(i * per + 4);
    } else {
      first[i] = (uint32_t)(i * per);
    }
    for (int j = 0; j < per; j++) flags[i * per + j] = fl[j];
  }
  first[n_prod] = (uint32_t)n_pairs;
  std::vector<int> is_one(n_prod), valid(n_prod);
  B200_TRY(pairing_products(ctx, P.data(), Q.data(), flags.data(), first.data(), (int)n_prod, false, nullptr,
                            is_one.data(), valid.data()));
  for (size_t i = 0; i < k; i++) {
    bool ok = true;
    for (int b = 0; b < nprod_per; b++) ok = ok && is_one[i * nprod_per + b] && valid[i * nprod_per + b];
    ok_each[i] = ok ? 1 : 0;
  }
  return 0;
}

}  // namespace b200

using namespace b200;

extern "C" int b200g16_verify_batch(b200g16_ctx* ctx, const b200g16_vk_desc* vk, size_t k, const uint64_t* ar,
                                    const uint64_t* bs, const uint64_t* krs, const uint64_t* commitments,
                                    const uint64_t* poks, const uint64_t* public_inputs, size_t n_public,
                                    const uint64_t* coeffs, int* ok_out, uint8_t* ok_each) {
  if (!ctx || !vk || !ok_out || (k && (!ar || !bs || !krs || !coeffs || (n_public && !public_inputs))))
    return fail(B200G16_ERR_ARG, "verify_batch: null");
  if (!vk->g1_alpha || !vk->g2_beta || !vk->g2_gamma || !vk->g2_delta || !vk->g1_k || vk->n_k == 0)
    return fail(B200G16_ERR_ARG, "verify_batch: verifying key incomplete");
  const bool has_com = commitments != nullptr;
  if (has_com != (poks != nullptr) || (has_com && (!vk->ped_g || !vk->ped_g_sigma_neg)) ||
      (!has_com && (vk->ped_g || vk->ped_g_sigma_neg)))
    return fail(B200G16_ERR_ARG, "verify_batch: commitments, poks and the pedersen verifying key go together");
  if (k > BV_MAX_K) return fail(B200G16_ERR_ARG, "verify_batch: k=%zu proofs, at most %zu", k, BV_MAX_K);
  *ok_out = 0;
  if (n_public + 1 != vk->n_k)
    return fail(B200G16_ERR_ARG, "verify_batch: %zu public inputs, vk.G1.K expects %zu", n_public, vk->n_k - 1);
  const size_t n_coef = has_com ? 2 * k : k;
  for (size_t i = 0; i < n_coef; i++)
    if (!coeffs[2 * i] && !coeffs[2 * i + 1]) return fail(B200G16_ERR_ARG, "verify_batch: coefficient %zu is zero", i);
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active)
    return fail(B200G16_ERR_STATE, "verify_batch: a prove is open on this ctx (prove_begin_dev without _end_dev)");
  if (k == 0) {
    *ok_out = 1;
    return 0;
  }
  B200_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  BvEvents ev;
  for (cudaEvent_t& e : ev.e) B200_CUDA(cudaEventCreate(&e));

  // device layout (one scratch allocation): [K | D] bases, Krs, PoKs, Ar, Bs, publics, coefficients,
  // MSM scalars [S, y, rho | tau], fold partials, f_i, two tree levels, flags, fixed pairs, L_i
  const size_t n_k = vk->n_k, npair = has_com ? 5 : 3, nf = k + npair;
  const uint32_t nblk = bv_cdiv(k, BV_FOLD_THREADS), n_cols = (uint32_t)(n_public + 1);
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += up(bytes); return o; };
  const size_t o_kd = take((n_k + (has_com ? k : 0)) * sizeof(G1Affine)), o_krs = take(k * sizeof(G1Affine)),
               o_pok = take(has_com ? k * sizeof(G1Affine) : 0), o_ar = take(k * sizeof(G1Affine)),
               o_bs = take(k * sizeof(G2Affine)), o_pub = take(k * n_public * sizeof(Fr)), o_coef = take(n_coef * 16),
               o_sc = take((n_k + k + (has_com ? k : 0)) * sizeof(Fr)), o_part = take((size_t)n_cols * nblk * sizeof(Fr)),
               o_f = take(nf * sizeof(Fp12)), o_t0 = take(bv_cdiv(nf, BV_TREE_THREADS) * sizeof(Fp12)),
               o_t1 = take(bv_cdiv(nf, BV_TREE_THREADS) * sizeof(Fp12)), o_valid = take(k * 4), o_flags = take(8),
               o_fp = take(npair * sizeof(G1Affine)), o_fq = take(npair * sizeof(G2Affine)),
               o_L = take(k * sizeof(G1Affine));
  B200_TRY(ctx->io_a.ensure(off));
  char* d = ctx->io_a.as<char>();
  G1Affine* d_kd = (G1Affine*)(d + o_kd);
  G1Affine* d_com = has_com ? d_kd + n_k : nullptr;
  G1Affine* d_pok = has_com ? (G1Affine*)(d + o_pok) : nullptr;
  Fr* d_sc = (Fr*)(d + o_sc);
  Fr* d_rho = d_sc + n_k;
  Fr* d_tau = d_rho + k;
  Fp12* d_f = (Fp12*)(d + o_f);
  int* d_flags = (int*)(d + o_flags);

  B200_CUDA(cudaEventRecord(ev.e[0], st));
  B200_TRY(h2d_copy(ctx, d_kd, vk->g1_k, n_k * sizeof(G1Affine), st));
  if (has_com) {
    B200_TRY(h2d_copy(ctx, d_com, commitments, k * sizeof(G1Affine), st));
    B200_TRY(h2d_copy(ctx, d_pok, poks, k * sizeof(G1Affine), st));
  }
  B200_TRY(h2d_copy(ctx, d + o_krs, krs, k * sizeof(G1Affine), st));
  B200_TRY(h2d_copy(ctx, d + o_ar, ar, k * sizeof(G1Affine), st));
  B200_TRY(h2d_copy(ctx, d + o_bs, bs, k * sizeof(G2Affine), st));
  if (n_public) B200_TRY(h2d_copy(ctx, d + o_pub, public_inputs, k * n_public * sizeof(Fr), st));
  B200_TRY(h2d_copy(ctx, d + o_coef, coeffs, n_coef * 16, st));
  B200_CUDA(cudaMemsetAsync(d_flags, 0, 8, st));
  B200_CUDA(cudaEventRecord(ev.e[1], st));

  // 1. per proof: checks, rho_i Ar_i, Miller loop
  k_batch_proofs<<<bv_cdiv(k, BV_PROOF_THREADS), BV_PROOF_THREADS, 0, st>>>(
      (const G1Affine*)(d + o_ar), (const G2Affine*)(d + o_bs), (const G1Affine*)(d + o_krs), d_com, d_pok,
      (const uint64_t*)(d + o_coef), (uint32_t)k, d_f, (int*)(d + o_valid), d_flags);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaEventRecord(ev.e[2], st));

  // 2. S, y_j and the coefficients as MSM scalars;  3. the MSMs
  k_fold<<<dim3(nblk, n_cols < BV_MAX_GRID_Y ? n_cols : BV_MAX_GRID_Y), BV_FOLD_THREADS, 0, st>>>(
      (const uint64_t*)(d + o_coef), (const Fr*)(d + o_pub), (uint32_t)k, (uint32_t)n_public, has_com ? 1 : 0, d_rho,
      d_tau, (Fr*)(d + o_part));
  k_fold_final<<<n_cols < BV_MAX_GRID_Y ? n_cols : BV_MAX_GRID_Y, BV_FOLD_THREADS, 0, st>>>((const Fr*)(d + o_part),
                                                                                           nblk, n_cols, d_sc);
  B200_CUDA(cudaGetLastError());
  ctx->launches += 3;
  G1Affine m_krs, m_l, m_d = G1Affine::inf(), m_p = G1Affine::inf();
  B200_TRY(msm_device<Fp>(ctx, (const G1Affine*)(d + o_krs), nullptr, d_rho, k, &m_krs));
  B200_TRY(msm_device<Fp>(ctx, d_kd, nullptr, d_sc, n_k + (has_com ? k : 0), &m_l));
  if (has_com) {
    B200_TRY(msm_device<Fp>(ctx, d_com, nullptr, d_tau, k, &m_d));
    B200_TRY(msm_device<Fp>(ctx, d_pok, nullptr, d_tau, k, &m_p));
  }
  G1Affine fp[5];
  G2Affine fq[5];
  memcpy(&fp[0], vk->g1_alpha, 64);  memcpy(&fq[0], vk->g2_beta, 128);
  fp[1] = g1_negate(m_l);            memcpy(&fq[1], vk->g2_gamma, 128);
  fp[2] = g1_negate(m_krs);          memcpy(&fq[2], vk->g2_delta, 128);
  if (has_com) {
    fp[3] = m_d;                     memcpy(&fq[3], vk->ped_g_sigma_neg, 128);
    fp[4] = m_p;                     memcpy(&fq[4], vk->ped_g, 128);
  }
  B200_CUDA(cudaMemcpyAsync(d + o_fp, fp, npair * sizeof(G1Affine), cudaMemcpyHostToDevice, st));
  B200_CUDA(cudaMemcpyAsync(d + o_fq, fq, npair * sizeof(G2Affine), cudaMemcpyHostToDevice, st));
  B200_CUDA(cudaEventRecord(ev.e[3], st));

  // 4. fixed pairs, then the product tree over all k + npair Miller-loop values
  k_fixed_pairs<<<1, 32, 0, st>>>((const G1Affine*)(d + o_fp), (const G2Affine*)(d + o_fq), (int)npair, d_sc, d_f + k);
  const Fp12* in = d_f;
  Fp12* lvl[2] = {(Fp12*)(d + o_t0), (Fp12*)(d + o_t1)};
  int launches = 1;
  for (size_t n = nf, t = 0; n > 1; n = bv_cdiv(n, BV_TREE_THREADS), t ^= 1, launches++) {
    k_f12_product<<<bv_cdiv(n, BV_TREE_THREADS), BV_TREE_THREADS, 0, st>>>(in, (uint32_t)n, lvl[t]);
    in = lvl[t];
  }
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaEventRecord(ev.e[4], st));
  k_final_exp<<<1, 32, 0, st>>>(in, d_flags);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaEventRecord(ev.e[5], st));
  ctx->launches += launches + 1;
  int flags[2] = {0, 0};
  B200_CUDA(cudaMemcpyAsync(flags, d_flags, 8, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  const bool ok = flags[1] != 0;
  *ok_out = ok ? 1 : 0;

  int n_phase = 5;
  if (ok_each && ok) {
    memset(ok_each, 1, k);
  } else if (ok_each) {
    k_batch_lsum<<<bv_cdiv(k, BV_PROOF_THREADS), BV_PROOF_THREADS, 0, st>>>(
        d_kd, (Fr*)(d + o_pub), (uint32_t)k, (uint32_t)n_public, d_com, (G1Affine*)(d + o_L));
    B200_CUDA(cudaGetLastError());
    ctx->launches++;
    B200_TRY(batch_per_proof(ctx, vk, k, ar, bs, krs, commitments, poks, (const G1Affine*)(d + o_L), ok_each));
    B200_CUDA(cudaEventRecord(ev.e[6], st));
    B200_CUDA(cudaStreamSynchronize(st));
    n_phase = 6;
  }
  // phases: upload, per-proof kernel, fold + MSMs, fixed pairs + product tree, final exponentiation[, per-proof fallback]
  for (int i = 0; i < n_phase; i++) cudaEventElapsedTime(&ctx->timings.ms[i], ev.e[i], ev.e[i + 1]);
  ctx->timings.n = n_phase;
  return 0;
}
