// Groth16 Prove, everything after the constraint solver, for one GPU.
//
// Replaces gnark v0.11.0 backend/groth16/bn254/prove.go Prove() from "go computeH" to
// "return proof" (steps 4-9 of SURVEY §3.2), as called by the reference at
// /root/reference/mt.go:496.  The BSB22 Pedersen commitment / proof of knowledge, which
// gnark computes inside and right after Solve, go through b200g16_msm_g1 on resident
// pedersen bases (they are ordinary G1 MSMs).
//
// Device timeline (main stream; copies of a,b,c on the copy stream): H2D(wires) -> gather wire values into the A / B / K
// scalar vectors (gnark's filter by pk.InfinityA / pk.InfinityB and by public+committed wires)
// -> MSM B2, B1 (on B2's sorted lists: same scalars), A, K -> computeH (a, b, c arrive on the copy stream meanwhile) -> MSM Z (scalars = h,
// straight from computeH's device buffer), enqueued back to back (each MSM's bucket reduction runs on
// a second stream under its successor; r*delta, s*delta, -rs*delta, s*delta2 are computed on the host meanwhile)
// -> one synchronisation -> host: Horner per MSM, then
//   Ar  = A + alpha + r*delta
//   Bs1 = B1 + beta + s*delta           Bs = B2 + beta2 + s*delta2
//   Krs = K + Z + (-rs)*delta + s*Ar + r*Bs1
#include <algorithm>
#include <thread>

#include "prove.cuh"
#include "host_copy.cuh"

namespace b200 {

__global__ void __launch_bounds__(256) k_gather_fr(const Fr* __restrict__ src, const uint32_t* __restrict__ idx,
                                                    uint32_t n, Fr* __restrict__ dst) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4* s = reinterpret_cast<const uint4*>(src + idx[i]);
  uint4* d = reinterpret_cast<uint4*>(dst + i);
  d[0] = __ldg(s);
  d[1] = __ldg(s + 1);
}

// Batch prove: row y of the (proof) grid gathers proof y's scalar vector from its witness row.
__global__ void __launch_bounds__(256) k_gather_fr_rows(const Fr* __restrict__ src, size_t src_stride,
                                                         const uint32_t* __restrict__ idx, uint32_t n, Fr* __restrict__ dst) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4* s = reinterpret_cast<const uint4*>(src + blockIdx.y * src_stride + idx[i]);
  uint4* d = reinterpret_cast<uint4*>(dst + (size_t)blockIdx.y * n + i);
  d[0] = __ldg(s);
  d[1] = __ldg(s + 1);
}

template <class F>
static Affine<F> host_scalar_mul_aff(const Affine<F>& p, const Fr& k_mont) {
  Fr s = Fr::from_mont(k_mont);
  XYZZ<F> acc = XYZZ<F>::inf();
  int top = 255;
  while (top >= 0 && !((s.l[top >> 5] >> (top & 31)) & 1)) top--;
  for (int i = top; i >= 0; i--) {
    acc.dbl();
    if ((s.l[i >> 5] >> (i & 31)) & 1) acc.madd(p);
  }
  return acc.to_affine();
}

template <class F>
Affine<F> host_sum_points(const Affine<F>* pts, int n) {
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int i = 0; i < n; i++) acc.madd(pts[i]);
  return acc.to_affine();
}
template Affine<Fp> host_sum_points<Fp>(const Affine<Fp>*, int);
template Affine<Fp2> host_sum_points<Fp2>(const Affine<Fp2>*, int);

template <class F>
static Affine<F> host_sum(std::initializer_list<Affine<F>> pts) {
  XYZZ<F> acc = XYZZ<F>::inf();
  for (const auto& p : pts) acc.madd(p);
  return acc.to_affine();
}

// wires kept by `skip` flags, restricted to entries [off, off + expect) of that list (a shard of the key)
static int build_index(const uint8_t* skip, size_t n_wires, size_t off, size_t expect, bool partial, uint32_t** d_out,
                       const char* what) {
  std::vector<uint32_t> idx;
  for (size_t i = 0; i < n_wires; i++)
    if (!skip[i]) idx.push_back((uint32_t)i);
  if (partial ? (off + expect > idx.size()) : (off != 0 || idx.size() != expect))
    return fail(B200G16_ERR_ARG, "pk_upload: %s flags keep %zu wires; the point vector covers [%zu, %zu)", what,
                idx.size(), off, off + expect);
  B200_CUDA(cudaMalloc(d_out, (expect ? expect : 1) * sizeof(uint32_t)));
  if (expect)
    B200_CUDA(cudaMemcpy(*d_out, idx.data() + off, expect * sizeof(uint32_t), cudaMemcpyHostToDevice));
  return 0;
}

void pk_release(b200g16_pk* pk) {
  if (!pk) return;
  cudaSetDevice(pk->device);
  for (int i = 0; i < 5; i++)
    if (pk->owned[i] && pk->vec[i]) b200g16_bases_free(pk->vec[i]);
  for (int i = 0; i < 3; i++)
    if (pk->d_idx[i]) cudaFree(pk->d_idx[i]);
  delete pk;
}

int pk_build(b200g16_ctx* ctx, const b200g16_pk_desc* d, b200g16_pk** out) {
  if (!ctx || !d || !out) return fail(B200G16_ERR_ARG, "pk_upload: null");
  if (!d->g1_alpha || !d->g1_beta || !d->g1_delta || !d->g2_beta || !d->g2_delta)
    return fail(B200G16_ERR_ARG, "pk_upload: alpha/beta/delta missing");
  if (!d->infinity_a || !d->infinity_b || !d->k_skip) return fail(B200G16_ERR_ARG, "pk_upload: wire flags missing");
  if (d->log2_domain > 28) return fail(B200G16_ERR_ARG, "pk_upload: domain 2^%u exceeds two-adicity", d->log2_domain);
  if (d->n_wires >= (1ull << 32)) return fail(B200G16_ERR_ARG, "pk_upload: too many wires");
  b200g16_pk* pk = new b200g16_pk();
  pk->device = ctx->device;
  pk->log2n = d->log2_domain;
  pk->n_wires = d->n_wires;
  const uint64_t* host[5] = {d->g1_a, d->g1_b, d->g1_k, d->g1_z, d->g2_b};
  const b200g16_bases* res[5] = {d->res_a, d->res_b, d->res_k, d->res_z, d->res_b2};
  const size_t n[5] = {d->n_a, d->n_b, d->n_k, d->n_z, d->n_b};
  for (int i = 0; i < 5; i++) {
    if (res[i]) {
      if (res[i]->n != n[i] || res[i]->group != (i == 4 ? 2 : 1) || res[i]->device != ctx->device) {
        pk_release(pk);
        return fail(B200G16_ERR_ARG, "pk_upload: resident vector %d has the wrong size/group/device", i);
      }
      pk->vec[i] = const_cast<b200g16_bases*>(res[i]);
    } else {
      if (n[i] && !host[i]) { pk_release(pk); return fail(B200G16_ERR_ARG, "pk_upload: vector %d missing", i); }
      int st = (i == 4) ? b200g16_bases_upload_g2(ctx, host[i], n[i], &pk->vec[i])
                        : b200g16_bases_upload_g1(ctx, host[i], n[i], &pk->vec[i]);
      if (st) { pk_release(pk); return st; }
      pk->owned[i] = true;
      if (d->precompute && n[i]) {
        st = b200g16_bases_precompute(ctx, pk->vec[i], 0);
        if (st) { pk_release(pk); return st; }
      }
    }
  }
  size_t N = (size_t)1 << d->log2_domain;
  pk->partial = d->partial != 0;
  pk->off_z = d->off_z;
  pk->n_z = d->n_z;
  if (pk->partial ? (d->off_z + d->n_z + 1 > N) : (d->off_z != 0 || d->n_z + 1 != N)) {
    pk_release(pk);
    return fail(B200G16_ERR_ARG, "pk_upload: Z covers [%zu, %zu), domain has N-1=%zu", d->off_z, d->off_z + d->n_z, N - 1);
  }
  memcpy(&pk->alpha, d->g1_alpha, sizeof(G1Affine));
  memcpy(&pk->beta, d->g1_beta, sizeof(G1Affine));
  memcpy(&pk->delta, d->g1_delta, sizeof(G1Affine));
  memcpy(&pk->beta2, d->g2_beta, sizeof(G2Affine));
  memcpy(&pk->delta2, d->g2_delta, sizeof(G2Affine));
  std::lock_guard<std::mutex> lock(ctx->mu);
  cudaSetDevice(ctx->device);
  const uint8_t* flags[3] = {d->infinity_a, d->infinity_b, d->k_skip};
  const size_t expect[3] = {d->n_a, d->n_b, d->n_k};
  const size_t offs[3] = {d->off_a, d->off_b, d->off_k};
  const char* names[3] = {"InfinityA", "InfinityB", "k_skip"};
  for (int i = 0; i < 3; i++) {
    int st = build_index(flags[i], d->n_wires, offs[i], expect[i], pk->partial, &pk->d_idx[i], names[i]);
    if (st) { pk_release(pk); return st; }
    pk->n_idx[i] = expect[i];
  }
  *out = pk;
  return 0;
}

// The multiples of delta do not depend on any MSM result: the prove computes them on the host while the GPU
// is still working.
DeltaMultiples delta_multiples(const b200g16_pk* pk, const Fr& r, const Fr& s) {
  DeltaMultiples m;
  m.r_delta = host_scalar_mul_aff<Fp>(pk->delta, r);
  m.s_delta = host_scalar_mul_aff<Fp>(pk->delta, s);
  m.kr_delta = host_scalar_mul_aff<Fp>(pk->delta, Fr::neg(Fr::mul(r, s)));
  m.s_delta2 = host_scalar_mul_aff<Fp2>(pk->delta2, s);
  return m;
}

// Ar, Bs, Krs (and bs1) from the five complete MSM results.
void prove_finish_host(const b200g16_pk* pk, const DeltaMultiples& dm, const G1Affine& A, const G1Affine& B1,
                       const G1Affine& K, const G1Affine& Z, const G2Affine& B2, const Fr& r, const Fr& s,
                       b200g16_proof* out) {
  G1Affine ar = host_sum<Fp>({A, pk->alpha, dm.r_delta});
  G1Affine bs1 = host_sum<Fp>({B1, pk->beta, dm.s_delta});
  G1Affine krs = host_sum<Fp>({K, Z, dm.kr_delta, host_scalar_mul_aff<Fp>(ar, s), host_scalar_mul_aff<Fp>(bs1, r)});
  G2Affine bs = host_sum<Fp2>({B2, pk->beta2, dm.s_delta2});
  memcpy(out->ar, &ar, 64);
  memcpy(out->bs, &bs, 128);
  memcpy(out->krs, &krs, 64);
  memcpy(out->bs1, &bs1, 64);
}

// A prove runs in two halves — prove_front: the four MSMs that only need the witness; prove_back: the Z MSM
// over h, the join and the host assembly — with its state (ctx->prove_cfg, prove_pk) kept on the ctx.
static int prove_enqueue_one(b200g16_ctx* ctx, const b200g16_pk* pk, int i, const Fr* scalars, size_t count, MsmCfg* cfg) {
  MsmTable tab;
  const MsmTable* tp = nullptr;
  if (i < 4) {
    const G1Affine* pts = msm_operand<Fp>(pk->vec[i], 0, &tab, &tp);
    // Bs1 runs over the same scalar vector as Bs2 (wireValuesB): it reuses Bs2's sorted lists
    return msm_enqueue<Fp>(ctx, pts, tp, scalars, count, 1, count, i, cfg, false, /*share_sort=*/i == 1);
  }
  const G2Affine* pts = msm_operand<Fp2>(pk->vec[i], 0, &tab, &tp);
  return msm_enqueue<Fp2>(ctx, pts, tp, scalars, count, 1, count, i, cfg, false);
}

// Gathers + the four MSMs over witness values — G2 leading: its bucket reduction is the longest tail and
// hides behind the G1 MSMs that follow.  Enqueues only; no synchronisation.
int prove_front(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_wires, int* ev_io) {
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove: another prove is already open on this ctx");
  cudaStream_t st = ctx->stream;
  int ev = *ev_io;
  auto mark = [&]() { if (ev < 18) cudaEventRecord(ctx->ev[ev++], st); };
  size_t tot = pk->n_idx[0] + pk->n_idx[1] + pk->n_idx[2];
  B200_TRY(ctx->io_b.ensure((tot ? tot : 1) * sizeof(Fr)));
  Fr* sv[3];
  sv[0] = ctx->io_b.as<Fr>();
  sv[1] = sv[0] + pk->n_idx[0];
  sv[2] = sv[1] + pk->n_idx[1];
  for (int i = 0; i < 3; i++)
    if (pk->n_idx[i]) {
      k_gather_fr<<<cdiv(pk->n_idx[i], 256), 256, 0, st>>>(d_wires, pk->d_idx[i], (uint32_t)pk->n_idx[i], sv[i]);
      ctx->launches++;
    }
  mark();
  const Fr* scal[5] = {sv[0], sv[1], sv[2], nullptr, sv[1]};
  const size_t cnt[5] = {pk->n_idx[0], pk->n_idx[1], pk->n_idx[2], 0, pk->n_idx[1]};
  for (int i : {4, 1, 0, 2}) {
    B200_TRY(prove_enqueue_one(ctx, pk, i, scal[i], cnt[i], &ctx->prove_cfg[i]));
    mark();
  }
  ctx->prove_pk = pk;
  ctx->prove_active = true;
  *ev_io = ev;
  return 0;
}

// d_h: h (N elements, bit-reversed).  Z MSM, join, host assembly.
int prove_back(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_h, const Fr& r, const Fr& s,
               b200g16_proof* out, int* ev_io) {
  if (!ctx->prove_active || ctx->prove_pk != pk) return fail(B200G16_ERR_STATE, "prove: no matching prove_begin on this ctx");
  ctx->prove_active = false;
  cudaStream_t st = ctx->stream;
  int ev = *ev_io;
  B200_TRY(prove_enqueue_one(ctx, pk, 3, d_h + pk->off_z, pk->n_z, &ctx->prove_cfg[3]));
  if (ev < 18) cudaEventRecord(ctx->ev[ev++], st);
  B200_TRY(msm_join(ctx));
  const MsmCfg* cfg = ctx->prove_cfg;
  G1Affine A, B1, K, Z;
  G2Affine B2;
  memset(out, 0, sizeof(*out));
  if (!pk->partial) {
    // Host work under the GPU's: the delta multiples first, then every result is taken the moment ITS window sums have
    // landed (ev_slot) — Ar, s*Ar, Bs1, r*Bs1 and Bs (0.5 ms of host scalar multiplications and inversions) are done
    // while K, computeH and Z still run; after the last synchronisation only two normalisations and one sum are left.
    DeltaMultiples dm = delta_multiples(pk, r, s);
    B200_CUDA(cudaEventSynchronize(ctx->ev_slot[4]));   // the tails finish in enqueue order: B2, B1, A, K, Z
    B200_TRY(msm_collect<Fp2>(ctx, 4, cfg[4], &B2));
    const G2Affine bs = host_sum<Fp2>({B2, pk->beta2, dm.s_delta2});
    B200_CUDA(cudaEventSynchronize(ctx->ev_slot[1]));
    B200_TRY(msm_collect<Fp>(ctx, 1, cfg[1], &B1));
    const G1Affine bs1 = host_sum<Fp>({B1, pk->beta, dm.s_delta});
    const G1Affine r_bs1 = host_scalar_mul_aff<Fp>(bs1, r);
    B200_CUDA(cudaEventSynchronize(ctx->ev_slot[0]));
    B200_TRY(msm_collect<Fp>(ctx, 0, cfg[0], &A));
    const G1Affine ar = host_sum<Fp>({A, pk->alpha, dm.r_delta});
    const G1Affine s_ar = host_scalar_mul_aff<Fp>(ar, s);
    B200_CUDA(cudaStreamSynchronize(st));
    B200_TRY(msm_collect<Fp>(ctx, 2, cfg[2], &K));
    B200_TRY(msm_collect<Fp>(ctx, 3, cfg[3], &Z));
    const G1Affine krs = host_sum<Fp>({K, Z, dm.kr_delta, s_ar, r_bs1});
    memcpy(out->ar, &ar, 64);
    memcpy(out->bs, &bs, 128);
    memcpy(out->krs, &krs, 64);
    memcpy(out->bs1, &bs1, 64);
  } else {
    B200_CUDA(cudaStreamSynchronize(st));
    B200_TRY(msm_collect<Fp>(ctx, 0, cfg[0], &A));
    B200_TRY(msm_collect<Fp>(ctx, 1, cfg[1], &B1));
    B200_TRY(msm_collect<Fp>(ctx, 2, cfg[2], &K));
    B200_TRY(msm_collect<Fp>(ctx, 3, cfg[3], &Z));
    B200_TRY(msm_collect<Fp2>(ctx, 4, cfg[4], &B2));
  }
  *ev_io = ev;
  memcpy(out->msm_a, &A, 64);
  memcpy(out->msm_b1, &B1, 64);
  memcpy(out->msm_k, &K, 64);
  memcpy(out->msm_z, &Z, 64);
  memcpy(out->msm_b2, &B2, 128);
  return 0;
}

// abc_ready: event after which d_a, d_b, d_c are valid (the host path uploads them on the copy stream while
// the four MSMs that only need the witness already run), or nullptr.
// d_wires: n_wires Fr; d_a/b/c: N Fr each, zero padded. h is left in d_a.
// d_b == nullptr: d_a already holds h (computeH was done elsewhere, e.g. spread over several GPUs).
static int prove_device(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_wires, Fr* d_a, Fr* d_b, Fr* d_c,
                        const Fr& r, const Fr& s, b200g16_proof* out, int* ev_io, cudaEvent_t abc_ready = nullptr) {
  B200_TRY(prove_front(ctx, pk, d_wires, ev_io));
  if (abc_ready) B200_CUDA(cudaStreamWaitEvent(ctx->stream, abc_ready, 0));
  if (d_b) B200_TRY(compute_h_device(ctx, d_a, d_b, d_c, (int)pk->log2n, false));
  if (*ev_io < 18) cudaEventRecord(ctx->ev[(*ev_io)++], ctx->stream);
  return prove_back(ctx, pk, d_a, r, s, out, ev_io);
}

// ---- batch prove: k proofs of one circuit against one resident pk, in sub-batches of m proofs.  Per sub-batch:
// gathers of the m x (A, B, K) scalar rows, the four witness MSMs as batch MSMs (k = m, B1 on B2's sorted lists),
// computeH per proof on rows j * N of m x N buffers, one batch Z MSM over the m h rows (ld = N), one synchronisation,
// then the host assembly spread over threads.  The delta multiples of all k proofs start on those threads before any
// GPU work is enqueued.

// fn(i) for i < count on min(count, hardware threads, 16) threads (the caller's thread included); false when a thread
// could not be started (the started ones are joined, and the work is not complete).
template <class Fn>
static bool host_parallel(size_t count, Fn fn) {
  const size_t hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t T = std::min<size_t>({count, hw, 16});
  if (T <= 1) { for (size_t i = 0; i < count; i++) fn(i); return true; }
  std::vector<std::thread> th;
  bool ok = true;
  try {
    for (size_t t = 1; t < T; t++)
      th.emplace_back([&, t]() { for (size_t i = t; i < count; i += T) fn(i); });
  } catch (...) {
    ok = false;
  }
  if (ok)
    for (size_t i = 0; i < count; i += T) fn(i);
  for (auto& x : th) x.join();
  return ok;
}

// proofs per sub-batch: every one of the five MSMs fits one batch call (msm_batch_max); 1 = the single-prove path.
// *slot_bytes: the batch staging one of those MSMs needs per proof at most.
static size_t prove_batch_max(const b200g16_ctx* ctx, const b200g16_pk* pk, size_t* slot_bytes) {
  const size_t n[5] = {pk->n_idx[0], pk->n_idx[1], pk->n_idx[2], pk->n_z, pk->n_idx[1]};
  size_t m = SIZE_MAX;
  *slot_bytes = 0;
  for (int i = 0; i < 5; i++) {
    MsmTable tab;
    const MsmTable* tp = nullptr;
    if (i < 4) msm_operand<Fp>(pk->vec[i], 0, &tab, &tp);
    else msm_operand<Fp2>(pk->vec[i], 0, &tab, &tp);
    const int c = msm_window_for(ctx, tp, n[i]);
    m = std::min(m, msm_batch_max(c, tp != nullptr, n[i]));
    const size_t wr = tp ? 1 : (size_t)msm_num_windows(c);
    *slot_bytes = std::max(*slot_bytes, wr * (i < 4 ? sizeof(XYZZ<Fp>) : sizeof(XYZZ<Fp2>)));
  }
  return m;
}

// One sub-batch of m >= 2 proofs on device rows: d_wires m x n_wires, d_a/b/c m x N (h is left in the d_a rows).
// abc(&ready) runs once the witness MSMs are enqueued: the host path starts the a, b, c uploads there, under those
// MSMs, and returns the event after which the rows are in place (nullptr: already there).  dm: the proofs' delta
// multiples (threads still filling them are joined by `dm_wait` before the assembly).  ms[4] accumulates the phase times.
template <class Abc, class Wait>
static int prove_batch_sub(b200g16_ctx* ctx, const b200g16_pk* pk, size_t m, const Fr* d_wires, Fr* d_a, Fr* d_b,
                           Fr* d_c, Abc&& abc, const Fr* r, const Fr* s, const DeltaMultiples* dm,
                           Wait&& dm_wait, b200g16_proof* out, float* ms) {
  cudaStream_t st = ctx->stream;
  const size_t N = (size_t)1 << pk->log2n;
  cudaEventRecord(ctx->ev[0], st);
  const size_t tot = pk->n_idx[0] + pk->n_idx[1] + pk->n_idx[2];
  B200_TRY(ctx->io_b.ensure((tot ? tot * m : 1) * sizeof(Fr)));
  Fr* sv[3];
  sv[0] = ctx->io_b.as<Fr>();
  sv[1] = sv[0] + m * pk->n_idx[0];
  sv[2] = sv[1] + m * pk->n_idx[1];
  for (int i = 0; i < 3; i++)
    if (pk->n_idx[i]) {
      k_gather_fr_rows<<<dim3(cdiv(pk->n_idx[i], 256), (unsigned)m), 256, 0, st>>>(d_wires, pk->n_wires, pk->d_idx[i],
                                                                                   (uint32_t)pk->n_idx[i], sv[i]);
      ctx->launches++;
    }
  cudaEventRecord(ctx->ev[1], st);
  MsmCfg cfg[5];
  const size_t cnt[5] = {pk->n_idx[0], pk->n_idx[1], pk->n_idx[2], 0, pk->n_idx[1]};
  const Fr* scal[5] = {sv[0], sv[1], sv[2], nullptr, sv[1]};
  for (int i : {4, 1, 0, 2}) {
    MsmTable tab;
    const MsmTable* tp = nullptr;
    if (i < 4) {
      const G1Affine* pts = msm_operand<Fp>(pk->vec[i], 0, &tab, &tp);
      B200_TRY(msm_enqueue<Fp>(ctx, pts, tp, scal[i], cnt[i], m, cnt[i], i, &cfg[i], false, /*share_sort=*/i == 1));
    } else {
      const G2Affine* pts = msm_operand<Fp2>(pk->vec[i], 0, &tab, &tp);
      B200_TRY(msm_enqueue<Fp2>(ctx, pts, tp, scal[i], cnt[i], m, cnt[i], i, &cfg[i], false));
    }
  }
  cudaEventRecord(ctx->ev[2], st);
  cudaEvent_t abc_ready = nullptr;
  B200_TRY(abc(&abc_ready));
  if (abc_ready) B200_CUDA(cudaStreamWaitEvent(st, abc_ready, 0));
  for (size_t j = 0; j < m; j++) B200_TRY(compute_h_device(ctx, d_a + j * N, d_b + j * N, d_c + j * N, (int)pk->log2n, false));
  cudaEventRecord(ctx->ev[3], st);
  {
    MsmTable tab;
    const MsmTable* tp = nullptr;
    const G1Affine* pts = msm_operand<Fp>(pk->vec[3], 0, &tab, &tp);
    B200_TRY(msm_enqueue<Fp>(ctx, pts, tp, d_a + pk->off_z, pk->n_z, m, N, 3, &cfg[3], false));
  }
  B200_TRY(msm_join(ctx));
  cudaEventRecord(ctx->ev[4], st);
  B200_CUDA(cudaStreamSynchronize(st));
  for (int i = 0; i < 4; i++) {
    float t = 0;
    cudaEventElapsedTime(&t, ctx->ev[i], ctx->ev[i + 1]);
    ms[i] += t;
  }
  dm_wait();
  const bool ok = host_parallel(m, [&](size_t j) {
    G1Affine A, B1, K, Z;
    G2Affine B2;
    msm_collect<Fp>(ctx, 0, cfg[0], &A, j);
    msm_collect<Fp>(ctx, 1, cfg[1], &B1, j);
    msm_collect<Fp>(ctx, 2, cfg[2], &K, j);
    msm_collect<Fp>(ctx, 3, cfg[3], &Z, j);
    msm_collect<Fp2>(ctx, 4, cfg[4], &B2, j);
    b200g16_proof* o = out + j;
    memset(o, 0, sizeof(*o));
    prove_finish_host(pk, dm[j], A, B1, K, Z, B2, r[j], s[j], o);
    memcpy(o->msm_a, &A, 64);
    memcpy(o->msm_b1, &B1, 64);
    memcpy(o->msm_k, &K, 64);
    memcpy(o->msm_z, &Z, 64);
    memcpy(o->msm_b2, &B2, 128);
  });
  if (!ok) return fail(B200G16_ERR_STATE, "prove_batch: could not start the host assembly threads");
  return 0;
}

// The shared body of both entry points.  rows(j0, m, &wires, &a, &b, &c) gives the device rows of proofs [j0, j0 + m)
// (the host path uploads the wires there); abc(j0, m, &ready) is prove_batch_sub's abc for that sub-batch.
template <class Rows, class Abc>
static int prove_batch_run(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, size_t m_max, size_t slot_bytes,
                           const uint64_t* r, const uint64_t* s, b200g16_proof* out, Rows&& rows, Abc&& abc) {
  B200_TRY(msm_batch_stage(ctx, m_max * slot_bytes));
  std::vector<Fr> fr_r(k), fr_s(k);
  memcpy(fr_r.data(), r, k * sizeof(Fr));
  memcpy(fr_s.data(), s, k * sizeof(Fr));
  std::vector<DeltaMultiples> dm(k);
  // the delta multiples of all k proofs, on host threads under the GPU's work
  const size_t T = std::max<size_t>(1, std::min<size_t>({k, (size_t)std::max(1u, std::thread::hardware_concurrency()), 16}));
  std::vector<std::thread> th;
  bool started = true;
  try {
    for (size_t t = 0; t < T; t++)
      th.emplace_back([&, t]() { for (size_t i = t; i < k; i += T) dm[i] = delta_multiples(pk, fr_r[i], fr_s[i]); });
  } catch (...) {
    started = false;
  }
  bool joined = false;
  auto dm_wait = [&]() { if (!joined) { for (auto& x : th) x.join(); joined = true; } };
  if (!started) { dm_wait(); return fail(B200G16_ERR_STATE, "prove_batch: could not start the host threads"); }
  float ms[4] = {0, 0, 0, 0};
  auto body = [&]() -> int {
    for (size_t j0 = 0; j0 < k;) {
      const size_t m = std::min(m_max, k - j0);
      const Fr *w = nullptr;
      Fr *a = nullptr, *b = nullptr, *c = nullptr;
      B200_TRY(rows(j0, m, &w, &a, &b, &c));
      B200_TRY(prove_batch_sub(ctx, pk, m, w, a, b, c, [&](cudaEvent_t* ready) { return abc(j0, m, ready); },
                               fr_r.data() + j0, fr_s.data() + j0, dm.data() + j0, dm_wait, out + j0, ms));
      j0 += m;
    }
    return 0;
  };
  const int status = body();
  dm_wait();
  if (status) {   // leave the ctx usable: whatever is in flight is drained and forgotten
    msm_join(ctx);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->tail_stream);
    cudaStreamSynchronize(ctx->copy_stream);
    ctx->last_sort.valid = false;
    return status;
  }
  for (int i = 0; i < 4; i++) ctx->timings.ms[i] = ms[i];
  ctx->timings.n = 4;
  return 0;
}

static int prove_batch_check(b200g16_ctx* ctx, const b200g16_pk* pk, const char* what) {
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "%s: pk lives on another device", what);
  if (pk->partial) return fail(B200G16_ERR_ARG, "%s: a partial (sharded) pk cannot be batch-proved", what);
  return 0;
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200g16_pk_upload(b200g16_ctx* ctx, const b200g16_pk_desc* desc, b200g16_pk** out) { return pk_build(ctx, desc, out); }

void b200g16_pk_free(b200g16_pk* pk) { pk_release(pk); }

int b200g16_prove(b200g16_ctx* ctx, const b200g16_pk* pk, const uint64_t* wires, size_t n_wires, const uint64_t* a,
                  const uint64_t* b, const uint64_t* c, size_t n_constraints, const uint64_t r[4], const uint64_t s[4],
                  b200g16_proof* proof_out, uint64_t* h_out) {
  if (!ctx || !pk || !wires || !a || !b || !c || !r || !s || !proof_out) return fail(B200G16_ERR_ARG, "prove: null");
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "prove: pk lives on another device");
  if (n_wires != pk->n_wires) return fail(B200G16_ERR_ARG, "prove: %zu wires, pk expects %zu", n_wires, pk->n_wires);
  const size_t N = (size_t)1 << pk->log2n;
  if (n_constraints > N) return fail(B200G16_ERR_ARG, "prove: %zu constraints > domain %zu", n_constraints, N);
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int ev = 0;
  cudaEventRecord(ctx->ev[ev++], st);
  B200_TRY(ctx->io_a.ensure((n_wires ? n_wires : 1) * sizeof(Fr)));
  B200_TRY(h2d_copy(ctx, ctx->io_a.p, wires, n_wires * sizeof(Fr), st));
  // The witness goes first: it gates the four MSMs, which are enqueued BEFORE a, b, c are touched — a copy from
  // pageable memory (a Go slice) occupies the calling thread while it is staged, and the GPU should already be busy.
  // a, b, c then cross PCIe on the copy stream under those MSMs.
  DevBuf* bufs[3] = {&ctx->ntt.a, &ctx->ntt.b, &ctx->ntt.c};
  const uint64_t* src[3] = {a, b, c};
  cudaStream_t cs = ctx->copy_stream;
  for (int i = 0; i < 3; i++) B200_TRY(bufs[i]->ensure(N * sizeof(Fr)));   // (no allocation once the MSMs are in flight)
  B200_CUDA(cudaEventRecord(ctx->ev_copy[1], st));
  cudaEventRecord(ctx->ev[ev++], st);
  Fr fr_r, fr_s;
  memcpy(&fr_r, r, 32);
  memcpy(&fr_s, s, 32);
  B200_TRY(prove_front(ctx, pk, ctx->io_a.as<Fr>(), &ev));
  auto middle = [&]() -> int {
    B200_CUDA(cudaStreamWaitEvent(cs, ctx->ev_copy[1], 0));   // the buffers' previous readers (an earlier prove) are done
    for (int i = 0; i < 3; i++) {
      B200_TRY(h2d_copy(ctx, bufs[i]->p, src[i], n_constraints * sizeof(Fr), cs));
      if (N > n_constraints)
        B200_CUDA(cudaMemsetAsync((char*)bufs[i]->p + n_constraints * sizeof(Fr), 0, (N - n_constraints) * sizeof(Fr), cs));
    }
    B200_CUDA(cudaEventRecord(ctx->ev_copy[0], cs));
    B200_CUDA(cudaStreamWaitEvent(st, ctx->ev_copy[0], 0));
    return compute_h_device(ctx, ctx->ntt.a.as<Fr>(), ctx->ntt.b.as<Fr>(), ctx->ntt.c.as<Fr>(), (int)pk->log2n, false);
  };
  if (int status = middle()) {       // leave the ctx usable: the four MSMs in flight are drained and forgotten
    msm_join(ctx);
    cudaStreamSynchronize(st);
    ctx->prove_active = false;
    return status;
  }
  if (ev < 18) cudaEventRecord(ctx->ev[ev++], st);
  B200_TRY(prove_back(ctx, pk, ctx->ntt.a.as<Fr>(), fr_r, fr_s, proof_out, &ev));
  ctx->timings.n = ev - 1;
  for (int i = 0; i + 1 < ev; i++) cudaEventElapsedTime(&ctx->timings.ms[i], ctx->ev[i], ctx->ev[i + 1]);
  if (h_out) B200_TRY(d2h_copy(ctx, h_out, ctx->ntt.a.p, N * sizeof(Fr), ctx->stream));
  return 0;
}

int b200g16_prove_batch(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const uint64_t* wires, size_t n_wires,
                        const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints, const uint64_t* r,
                        const uint64_t* s, b200g16_proof* proofs_out) {
  if (!ctx || !pk) return fail(B200G16_ERR_ARG, "prove_batch: null");
  if (k && (!wires || !a || !b || !c || !r || !s || !proofs_out)) return fail(B200G16_ERR_ARG, "prove_batch: null");
  B200_TRY(prove_batch_check(ctx, pk, "prove_batch"));
  if (n_wires != pk->n_wires) return fail(B200G16_ERR_ARG, "prove_batch: %zu wires, pk expects %zu", n_wires, pk->n_wires);
  const size_t N = (size_t)1 << pk->log2n;
  if (n_constraints > N) return fail(B200G16_ERR_ARG, "prove_batch: %zu constraints > domain %zu", n_constraints, N);
  if (k && (n_wires > SIZE_MAX / sizeof(Fr) / k || N > SIZE_MAX / sizeof(Fr) / k))
    return fail(B200G16_ERR_ARG, "prove_batch: k x n_wires or k x N overflows");
  if (k == 0) return 0;
  size_t m_max, slot_bytes;
  {
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove_batch: a prove is open on this ctx");
    m_max = std::min(k, prove_batch_max(ctx, pk, &slot_bytes));
  }
  if (m_max <= 1) {   // one proof per sub-batch: the single prove, proof by proof
    for (size_t j = 0; j < k; j++)
      B200_TRY(b200g16_prove(ctx, pk, wires + j * n_wires * 4, n_wires, a + j * n_constraints * 4, b + j * n_constraints * 4,
                             c + j * n_constraints * 4, n_constraints, r + 4 * j, s + 4 * j, proofs_out + j, nullptr));
    return 0;
  }
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove_batch: a prove is open on this ctx");
  B200_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream, cs = ctx->copy_stream;
  B200_TRY(ctx->io_a.ensure((n_wires ? m_max * n_wires : 1) * sizeof(Fr)));
  DevBuf* bufs[3] = {&ctx->ntt.a, &ctx->ntt.b, &ctx->ntt.c};
  for (int i = 0; i < 3; i++) B200_TRY(bufs[i]->ensure(m_max * N * sizeof(Fr)));
  const uint64_t* src[3] = {a, b, c};
  // As b200g16_prove: the wires first on the main stream (they gate the witness MSMs), and a, b, c on the copy stream
  // only once those MSMs are enqueued — a copy from pageable memory occupies this thread while it is staged.
  auto rows = [&](size_t j0, size_t m, const Fr** w, Fr** da, Fr** db, Fr** dc) -> int {
    if (n_wires) B200_TRY(h2d_copy(ctx, ctx->io_a.p, wires + j0 * n_wires * 4, m * n_wires * sizeof(Fr), st));
    B200_CUDA(cudaEventRecord(ctx->ev_copy[1], st));
    *w = ctx->io_a.as<Fr>();
    *da = ctx->ntt.a.as<Fr>();
    *db = ctx->ntt.b.as<Fr>();
    *dc = ctx->ntt.c.as<Fr>();
    return 0;
  };
  auto abc = [&](size_t j0, size_t m, cudaEvent_t* ready) -> int {
    B200_CUDA(cudaStreamWaitEvent(cs, ctx->ev_copy[1], 0));   // the rows' previous readers (the sub-batch before) are done
    for (int i = 0; i < 3; i++)
      for (size_t j = 0; j < m; j++) {
        char* row = (char*)bufs[i]->p + j * N * sizeof(Fr);
        if (n_constraints)
          B200_TRY(h2d_copy(ctx, row, src[i] + (j0 + j) * n_constraints * 4, n_constraints * sizeof(Fr), cs));
        if (N > n_constraints)
          B200_CUDA(cudaMemsetAsync(row + n_constraints * sizeof(Fr), 0, (N - n_constraints) * sizeof(Fr), cs));
      }
    B200_CUDA(cudaEventRecord(ctx->ev_copy[0], cs));
    *ready = ctx->ev_copy[0];
    return 0;
  };
  return prove_batch_run(ctx, pk, k, m_max, slot_bytes, r, s, proofs_out, rows, abc);
}

int b200g16_prove_batch_dev(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const void* d_wires, void* d_a, void* d_b,
                            void* d_c, const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out) {
  if (!ctx || !pk) return fail(B200G16_ERR_ARG, "prove_batch_dev: null");
  if (k && (!d_wires || !d_a || !d_b || !d_c || !r || !s || !proofs_out)) return fail(B200G16_ERR_ARG, "prove_batch_dev: null");
  B200_TRY(prove_batch_check(ctx, pk, "prove_batch_dev"));
  const size_t N = (size_t)1 << pk->log2n;
  if (k && (pk->n_wires > SIZE_MAX / sizeof(Fr) / k || N > SIZE_MAX / sizeof(Fr) / k))
    return fail(B200G16_ERR_ARG, "prove_batch_dev: k x n_wires or k x N overflows");
  if (k == 0) return 0;
  size_t m_max, slot_bytes;
  {
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove_batch_dev: a prove is open on this ctx");
    m_max = std::min(k, prove_batch_max(ctx, pk, &slot_bytes));
  }
  const Fr* W = (const Fr*)d_wires;
  Fr *A = (Fr*)d_a, *B = (Fr*)d_b, *C = (Fr*)d_c;
  if (m_max <= 1) {
    for (size_t j = 0; j < k; j++)
      B200_TRY(b200g16_prove_dev(ctx, pk, W + j * pk->n_wires, A + j * N, B + j * N, C + j * N, r + 4 * j, s + 4 * j,
                                 proofs_out + j));
    return 0;
  }
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove_batch_dev: a prove is open on this ctx");
  B200_CUDA(cudaSetDevice(ctx->device));
  auto rows = [&](size_t j0, size_t, const Fr** w, Fr** da, Fr** db, Fr** dc) -> int {
    *w = W + j0 * pk->n_wires;
    *da = A + j0 * N;
    *db = B + j0 * N;
    *dc = C + j0 * N;
    return 0;
  };
  auto abc = [](size_t, size_t, cudaEvent_t* ready) -> int { *ready = nullptr; return 0; };
  return prove_batch_run(ctx, pk, k, m_max, slot_bytes, r, s, proofs_out, rows, abc);
}

int b200g16_prove_finish(const b200g16_pk* pk, const uint64_t msm_a[8], const uint64_t msm_b1[8],
                         const uint64_t msm_k[8], const uint64_t msm_z[8], const uint64_t msm_b2[16],
                         const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out) {
  if (!pk || !msm_a || !msm_b1 || !msm_k || !msm_z || !msm_b2 || !r || !s || !proof_out)
    return fail(B200G16_ERR_ARG, "prove_finish: null");
  G1Affine A, B1, K, Z;
  G2Affine B2;
  Fr fr_r, fr_s;
  memcpy(&A, msm_a, 64); memcpy(&B1, msm_b1, 64); memcpy(&K, msm_k, 64); memcpy(&Z, msm_z, 64);
  memcpy(&B2, msm_b2, 128); memcpy(&fr_r, r, 32); memcpy(&fr_s, s, 32);
  memset(proof_out, 0, sizeof(*proof_out));
  prove_finish_host(pk, delta_multiples(pk, fr_r, fr_s), A, B1, K, Z, B2, fr_r, fr_s, proof_out);
  memcpy(proof_out->msm_a, msm_a, 64); memcpy(proof_out->msm_b1, msm_b1, 64); memcpy(proof_out->msm_k, msm_k, 64);
  memcpy(proof_out->msm_z, msm_z, 64); memcpy(proof_out->msm_b2, msm_b2, 128);
  return 0;
}

int b200g16_prove_h_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires, void* d_h, const uint64_t r[4],
                        const uint64_t s[4], b200g16_proof* proof_out) {
  if (!ctx || !pk || !d_wires || !d_h || !r || !s || !proof_out) return fail(B200G16_ERR_ARG, "prove_h_dev: null");
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "prove_h_dev: pk lives on another device");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  int ev = 0;
  cudaEventRecord(ctx->ev[ev++], ctx->stream);
  cudaEventRecord(ctx->ev[ev++], ctx->stream);
  Fr fr_r, fr_s;
  memcpy(&fr_r, r, 32);
  memcpy(&fr_s, s, 32);
  B200_TRY(prove_device(ctx, pk, (const Fr*)d_wires, (Fr*)d_h, nullptr, nullptr, fr_r, fr_s, proof_out, &ev));
  ctx->timings.n = ev - 1;
  for (int i = 0; i + 1 < ev; i++) cudaEventElapsedTime(&ctx->timings.ms[i], ctx->ev[i], ctx->ev[i + 1]);
  return 0;
}

int b200g16_prove_begin_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires) {
  if (!ctx || !pk || !d_wires) return fail(B200G16_ERR_ARG, "prove_begin_dev: null");
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "prove_begin_dev: pk lives on another device");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  int ev = 0;
  cudaEventRecord(ctx->ev[ev++], ctx->stream);
  cudaEventRecord(ctx->ev[ev++], ctx->stream);
  B200_TRY(prove_front(ctx, pk, (const Fr*)d_wires, &ev));
  ctx->timings.n = -(ev - 1);   // resolved by prove_end_dev
  return 0;
}

int b200g16_prove_end_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_h, const uint64_t r[4],
                          const uint64_t s[4], b200g16_proof* proof_out) {
  if (!ctx || !pk || !d_h || !r || !s || !proof_out) return fail(B200G16_ERR_ARG, "prove_end_dev: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  int ev = ctx->timings.n < 0 ? 1 - ctx->timings.n : 0;
  if (ev < 18) cudaEventRecord(ctx->ev[ev++], ctx->stream);   // everything the caller ran in between (computeH stages)
  Fr fr_r, fr_s;
  memcpy(&fr_r, r, 32);
  memcpy(&fr_s, s, 32);
  B200_TRY(prove_back(ctx, pk, (const Fr*)d_h, fr_r, fr_s, proof_out, &ev));
  ctx->timings.n = ev - 1;
  for (int i = 0; i + 1 < ev; i++) cudaEventElapsedTime(&ctx->timings.ms[i], ctx->ev[i], ctx->ev[i + 1]);
  return 0;
}

int b200g16_prove_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires, void* d_a, void* d_b, void* d_c,
                      const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out) {
  if (!ctx || !pk || !d_wires || !d_a || !d_b || !d_c || !r || !s || !proof_out)
    return fail(B200G16_ERR_ARG, "prove_dev: null");
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "prove_dev: pk lives on another device");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  int ev = 0;
  cudaEventRecord(ctx->ev[ev++], ctx->stream);
  cudaEventRecord(ctx->ev[ev++], ctx->stream);
  Fr fr_r, fr_s;
  memcpy(&fr_r, r, 32);
  memcpy(&fr_s, s, 32);
  B200_TRY(prove_device(ctx, pk, (const Fr*)d_wires, (Fr*)d_a, (Fr*)d_b, (Fr*)d_c, fr_r, fr_s, proof_out, &ev));
  ctx->timings.n = ev - 1;
  for (int i = 0; i + 1 < ev; i++) cudaEventElapsedTime(&ctx->timings.ms[i], ctx->ev[i], ctx->ev[i + 1]);
  return 0;
}

}  // extern "C"
