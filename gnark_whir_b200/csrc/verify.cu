// groth16.Verify and the pairing entry points (reference call site /root/reference/mt.go:497).
//
// Replaces gnark v0.11.0 backend/groth16/bn254/verify.go Verify():
//   1. proof.isValid(): Ar, Krs on G1, Bs in the r-torsion of the twist
//   2. with a BSB22 commitment: the challenge (hash_to_field, computed by the caller — it is a
//      SHA-256 over ~100 bytes) is one more public input, the commitment is added to the
//      public-input sum, and the Pedersen proof of knowledge is checked:
//           e(commitment, [-sigma]G2) * e(pok, G2) == 1
//   3. kSum = K[0] + MultiExp(K[1:], public inputs) (+ commitment)     — the ordinary G1 MSM
//   4. e(Ar, Bs) * e(-kSum, gamma2) * e(-Krs, delta2) * e(-alpha, beta2) == 1
//      (gnark precomputes e(alpha, beta) into the vk; the product is the same GT element)
// and gnark-crypto's bn254.PairingCheck / bn254.Pair for direct use.
#include "common.cuh"
#include "pairing.cuh"

namespace b200 {
template <class F>
int msm_device(b200g16_ctx* ctx, const Affine<F>* d_bases, const MsmTable* tab, const Fr* d_scalars, size_t n,
               Affine<F>* out);

constexpr int PAIR_THREADS = 32;

// One CTA per product: thread t runs the Miller loops of pairs t, t+32, ...; thread 0 multiplies them,
// does the final exponentiation and compares with 1.  first[b] .. first[b+1] delimit product b.
// flags[i] bit0: check P on curve, bit1: check Q in the r-torsion subgroup.
__global__ void __launch_bounds__(PAIR_THREADS) k_pairing_products(const G1Affine* __restrict__ P,
                                                                    const G2Affine* __restrict__ Q,
                                                                    const uint32_t* __restrict__ flags,
                                                                    const uint32_t* __restrict__ first,
                                                                    int with_cofactor, Fp12* __restrict__ gt_out,
                                                                    int* __restrict__ is_one, int* __restrict__ valid) {
  __shared__ Fp12 part[PAIR_THREADS];
  __shared__ int bad;
  const uint32_t lo = first[blockIdx.x], hi = first[blockIdx.x + 1];
  if (threadIdx.x == 0) bad = 0;
  __syncthreads();
  Fp12 f = f12_one();
  for (uint32_t i = lo + threadIdx.x; i < hi; i += PAIR_THREADS) {
    const G1Affine p = P[i];
    const G2Affine q = Q[i];
    if ((flags[i] & 1u) && !g1_on_curve(p)) atomicOr(&bad, 1);
    if ((flags[i] & 2u) && !g2_in_subgroup(q)) atomicOr(&bad, 1);
    f = f12_mul(f, miller_loop(p, q));
  }
  part[threadIdx.x] = f;
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t used = hi - lo < PAIR_THREADS ? hi - lo : PAIR_THREADS;
    for (uint32_t t = 1; t < used; t++) f = f12_mul(f, part[t]);
    Fp12 g = final_exponentiation(f, with_cofactor != 0);
    gt_out[blockIdx.x] = g;
    is_one[blockIdx.x] = f12_is_one(g) ? 1 : 0;
    valid[blockIdx.x] = bad ? 0 : 1;
  }
}

// n_prod products over pairs laid out back to back; host arrays, device scratch in ctx->io_c
// (also the per-proof fallback of b200g16_verify_batch, verify_batch.cu)
int pairing_products(b200g16_ctx* ctx, const G1Affine* P, const G2Affine* Q, const uint32_t* flags,
                     const uint32_t* first, int n_prod, bool with_cofactor, Fp12* gt, int* is_one, int* valid) {
  const size_t n = first[n_prod];
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t o_q = up(n * sizeof(G1Affine)), o_fl = o_q + up(n * sizeof(G2Affine)), o_first = o_fl + up(n * 4),
               o_gt = o_first + up((n_prod + 1) * 4), o_one = o_gt + up(n_prod * sizeof(Fp12)),
               o_valid = o_one + up(n_prod * 4), total = o_valid + up(n_prod * 4);
  B200_TRY(ctx->io_c.ensure(total));
  char* d = ctx->io_c.as<char>();
  cudaStream_t st = ctx->stream;
  if (n) {
    B200_CUDA(cudaMemcpyAsync(d, P, n * sizeof(G1Affine), cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(d + o_q, Q, n * sizeof(G2Affine), cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(d + o_fl, flags, n * 4, cudaMemcpyHostToDevice, st));
  }
  B200_CUDA(cudaMemcpyAsync(d + o_first, first, (n_prod + 1) * 4, cudaMemcpyHostToDevice, st));
  k_pairing_products<<<n_prod, PAIR_THREADS, 0, st>>>((const G1Affine*)d, (const G2Affine*)(d + o_q),
                                                      (const uint32_t*)(d + o_fl), (const uint32_t*)(d + o_first),
                                                      with_cofactor ? 1 : 0, (Fp12*)(d + o_gt), (int*)(d + o_one),
                                                      (int*)(d + o_valid));
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  if (gt) B200_CUDA(cudaMemcpyAsync(gt, d + o_gt, n_prod * sizeof(Fp12), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaMemcpyAsync(is_one, d + o_one, n_prod * 4, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaMemcpyAsync(valid, d + o_valid, n_prod * 4, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  return 0;
}

static G1Affine g1_neg(const G1Affine& p) {
  G1Affine r = p;
  r.y = Fp::neg(p.y);
  return r;
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200g16_pairing_check(b200g16_ctx* ctx, const uint64_t* g1_points, const uint64_t* g2_points, size_t n,
                          int* ok_out) {
  if (!ctx || !ok_out || (n && (!g1_points || !g2_points))) return fail(B200G16_ERR_ARG, "pairing_check: null");
  if (n > (1u << 20)) return fail(B200G16_ERR_ARG, "pairing_check: too many pairs");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  std::vector<uint32_t> flags(n, 3u);
  uint32_t first[2] = {0, (uint32_t)n};
  int is_one = 0, valid = 0;
  B200_TRY(pairing_products(ctx, (const G1Affine*)g1_points, (const G2Affine*)g2_points, flags.data(), first, 1, false,
                            nullptr, &is_one, &valid));
  if (!valid) return fail(B200G16_ERR_ARG, "pairing_check: a point is not on the curve / not in the r-torsion subgroup");
  *ok_out = is_one;
  return 0;
}

int b200g16_pair(b200g16_ctx* ctx, const uint64_t* g1_points, const uint64_t* g2_points, size_t n, uint64_t out_gt[48]) {
  if (!ctx || !out_gt || (n && (!g1_points || !g2_points))) return fail(B200G16_ERR_ARG, "pair: null");
  if (n > (1u << 20)) return fail(B200G16_ERR_ARG, "pair: too many pairs");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  std::vector<uint32_t> flags(n, 3u);
  uint32_t first[2] = {0, (uint32_t)n};
  int is_one = 0, valid = 0;
  Fp12 gt;
  B200_TRY(pairing_products(ctx, (const G1Affine*)g1_points, (const G2Affine*)g2_points, flags.data(), first, 1, true,
                            &gt, &is_one, &valid));
  if (!valid) return fail(B200G16_ERR_ARG, "pair: a point is not on the curve / not in the r-torsion subgroup");
  to_gnark_layout(gt, out_gt);
  return 0;
}

int b200g16_verify(b200g16_ctx* ctx, const b200g16_vk_desc* vk, const uint64_t ar[8], const uint64_t bs[16],
                   const uint64_t krs[8], const uint64_t* commitment, const uint64_t* commitment_pok,
                   const uint64_t* public_inputs, size_t n_public, int* ok_out) {
  if (!ctx || !vk || !ar || !bs || !krs || !ok_out || (n_public && !public_inputs))
    return fail(B200G16_ERR_ARG, "verify: null");
  if (!vk->g1_alpha || !vk->g2_beta || !vk->g2_gamma || !vk->g2_delta || !vk->g1_k || vk->n_k == 0)
    return fail(B200G16_ERR_ARG, "verify: verifying key incomplete");
  const bool has_com = commitment != nullptr;
  if (has_com && (!commitment_pok || !vk->ped_g || !vk->ped_g_sigma_neg))
    return fail(B200G16_ERR_ARG, "verify: commitment given without pok / pedersen verifying key");
  *ok_out = 0;
  // gnark: "invalid witness size" is an error, not a failed proof
  if (n_public + 1 != vk->n_k)
    return fail(B200G16_ERR_ARG, "verify: %zu public inputs, vk.G1.K expects %zu", n_public, vk->n_k - 1);
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "verify: a prove is open on this ctx (prove_begin_dev without _end_dev)");
  B200_CUDA(cudaSetDevice(ctx->device));

  // kSum = K[0] + sum_i pub_i K[i+1] (+ commitment): the library's own MSM on a scratch upload
  G1Affine msm = G1Affine::inf();
  if (n_public) {
    B200_TRY(ctx->io_a.ensure(n_public * sizeof(G1Affine)));
    B200_TRY(ctx->io_b.ensure(n_public * sizeof(Fr)));
    B200_CUDA(cudaMemcpyAsync(ctx->io_a.p, vk->g1_k + 8, n_public * sizeof(G1Affine), cudaMemcpyHostToDevice, ctx->stream));
    B200_CUDA(cudaMemcpyAsync(ctx->io_b.p, public_inputs, n_public * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
    B200_TRY(msm_device<Fp>(ctx, ctx->io_a.as<G1Affine>(), nullptr, ctx->io_b.as<Fr>(), n_public, &msm));
  }
  G1Affine k0, com = G1Affine::inf(), pok = G1Affine::inf();
  memcpy(&k0, vk->g1_k, sizeof(k0));
  if (has_com) { memcpy(&com, commitment, sizeof(com)); memcpy(&pok, commitment_pok, sizeof(pok)); }
  G1XYZZ acc = G1XYZZ::from_affine(msm);
  acc.madd(k0);
  acc.madd(com);
  const G1Affine ksum = acc.to_affine();

  G1Affine P[6];
  G2Affine Q[6];
  uint32_t flags[6] = {3u, 0u, 1u, 0u, 1u, 1u};  // proof points are checked, vk points are trusted
  G1Affine p_ar, p_krs, alpha;
  memcpy(&p_ar, ar, 64); memcpy(&p_krs, krs, 64); memcpy(&alpha, vk->g1_alpha, 64);
  P[0] = p_ar;            memcpy(&Q[0], bs, 128);
  P[1] = g1_neg(ksum);    memcpy(&Q[1], vk->g2_gamma, 128);
  P[2] = g1_neg(p_krs);   memcpy(&Q[2], vk->g2_delta, 128);
  P[3] = g1_neg(alpha);   memcpy(&Q[3], vk->g2_beta, 128);
  uint32_t first[3] = {0, 4, 4};
  int n_prod = 1;
  if (has_com) {
    P[4] = com;  memcpy(&Q[4], vk->ped_g_sigma_neg, 128);
    P[5] = pok;  memcpy(&Q[5], vk->ped_g, 128);
    first[2] = 6;
    n_prod = 2;
  }
  int is_one[2] = {0, 1}, valid[2] = {0, 1};
  B200_TRY(pairing_products(ctx, P, Q, flags, first, n_prod, false, nullptr, is_one, valid));
  *ok_out = (is_one[0] && valid[0] && is_one[1] && valid[1]) ? 1 : 0;
  return 0;
}

}  // extern "C"
