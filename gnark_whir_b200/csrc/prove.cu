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
// -> host: Horner per MSM as its window sums land, then
//   Ar  = A + alpha + r*delta
//   Bs1 = B1 + beta + s*delta           Bs = B2 + beta2 + s*delta2
//   Krs = K + Z + (-rs)*delta + s*Ar + r*Bs1
// A batch of m proofs of one circuit runs the same timeline once: the five MSMs as batch MSMs (k = m), computeH once
// per proof, and the host work of the m proofs spread over threads.  A single proof is a batch of one.
#include <algorithm>
#include <thread>

#include "prove.cuh"
#include "host_copy.cuh"

namespace b200 {

// Row y of the (proof) grid gathers proof y's scalar vector from its witness row.
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

// fn(i) for i < count on min(count, hardware threads, 16) threads (the caller's thread included; count = 1 runs inline);
// false when a thread could not be started (the started ones are joined, and the work is not complete).
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

// A prove runs in two halves — prove_front: the four MSMs that only need the witness; prove_back: the Z MSM
// over h, the join and the host assembly — with its state (ctx->prove_cfg, prove_pk) kept on the ctx.
// MSM i of the key (A, B1, K, Z, B2) over k scalar vectors, ld apart, into result slot i.
static int prove_enqueue_one(b200g16_ctx* ctx, const b200g16_pk* pk, int i, const Fr* scalars, size_t count, size_t k,
                             size_t ld, MsmCfg* cfg) {
  MsmTable tab;
  const MsmTable* tp = nullptr;
  if (i < 4) {
    const G1Affine* pts = msm_operand<Fp>(pk->vec[i], 0, &tab, &tp);
    // Bs1 runs over the same scalar vector as Bs2 (wireValuesB): it reuses Bs2's sorted lists
    return msm_enqueue<Fp>(ctx, pts, tp, scalars, count, k, ld, i, cfg, false, /*share_sort=*/i == 1);
  }
  const G2Affine* pts = msm_operand<Fp2>(pk->vec[i], 0, &tab, &tp);
  return msm_enqueue<Fp2>(ctx, pts, tp, scalars, count, k, ld, i, cfg, false);
}

// Gathers + the four MSMs over witness values — G2 leading: its bucket reduction is the longest tail and
// hides behind the G1 MSMs that follow.  Enqueues only; no synchronisation.
int prove_front(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_wires, size_t wire_stride, size_t m, int* ev_io) {
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove: another prove is already open on this ctx");
  cudaStream_t st = ctx->stream;
  int ev = *ev_io;
  auto mark = [&]() { if (ev < 18) cudaEventRecord(ctx->ev[ev++], st); };
  size_t tot = pk->n_idx[0] + pk->n_idx[1] + pk->n_idx[2];
  B200_TRY(ctx->io_b.ensure((tot ? m * tot : 1) * sizeof(Fr)));
  Fr* sv[3];   // m rows each
  sv[0] = ctx->io_b.as<Fr>();
  sv[1] = sv[0] + m * pk->n_idx[0];
  sv[2] = sv[1] + m * pk->n_idx[1];
  for (int i = 0; i < 3; i++)
    if (pk->n_idx[i]) {
      k_gather_fr_rows<<<dim3(cdiv(pk->n_idx[i], 256), (unsigned)m), 256, 0, st>>>(d_wires, wire_stride, pk->d_idx[i],
                                                                                   (uint32_t)pk->n_idx[i], sv[i]);
      ctx->launches++;
    }
  mark();
  const Fr* scal[5] = {sv[0], sv[1], sv[2], nullptr, sv[1]};
  const size_t cnt[5] = {pk->n_idx[0], pk->n_idx[1], pk->n_idx[2], 0, pk->n_idx[1]};
  for (int i : {4, 1, 0, 2}) {
    B200_TRY(prove_enqueue_one(ctx, pk, i, scal[i], cnt[i], m, cnt[i], &ctx->prove_cfg[i]));
    mark();
  }
  ctx->prove_pk = pk;
  ctx->prove_active = true;
  *ev_io = ev;
  return 0;
}

// d_h: m rows of h (N elements each, bit-reversed), h_stride apart.  Z MSM, join, host assembly of out[0 .. m).
int prove_back(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_h, size_t h_stride, size_t m, const Fr* r,
               const Fr* s, b200g16_proof* out, int* ev_io) {
  if (!ctx->prove_active || ctx->prove_pk != pk) return fail(B200G16_ERR_STATE, "prove: no matching prove_begin on this ctx");
  ctx->prove_active = false;
  cudaStream_t st = ctx->stream;
  int ev = *ev_io;
  B200_TRY(prove_enqueue_one(ctx, pk, 3, d_h + pk->off_z, pk->n_z, m, h_stride, &ctx->prove_cfg[3]));
  if (ev < 18) cudaEventRecord(ctx->ev[ev++], st);
  B200_TRY(msm_join(ctx));
  const MsmCfg* cfg = ctx->prove_cfg;
  if (pk->partial) {   // a shard of a key (m = 1: the batch entry points refuse one): the five partial sums only
    G1Affine A, B1, K, Z;
    G2Affine B2;
    B200_CUDA(cudaStreamSynchronize(st));
    B200_TRY(msm_collect<Fp>(ctx, 0, cfg[0], &A));
    B200_TRY(msm_collect<Fp>(ctx, 1, cfg[1], &B1));
    B200_TRY(msm_collect<Fp>(ctx, 2, cfg[2], &K));
    B200_TRY(msm_collect<Fp>(ctx, 3, cfg[3], &Z));
    B200_TRY(msm_collect<Fp2>(ctx, 4, cfg[4], &B2));
    memset(out, 0, sizeof(*out));
    memcpy(out->msm_a, &A, 64);
    memcpy(out->msm_b1, &B1, 64);
    memcpy(out->msm_k, &K, 64);
    memcpy(out->msm_z, &Z, 64);
    memcpy(out->msm_b2, &B2, 128);
    *ev_io = ev;
    return 0;
  }
  // Host work under the GPU's: the delta multiples first, then every result is taken the moment ITS window sums have
  // landed (ev_slot) — Ar, s*Ar, Bs1, r*Bs1 and Bs (0.5 ms of host scalar multiplications and inversions per proof) are
  // done while K, computeH and Z still run; after the last synchronisation only two normalisations and one sum per proof
  // are left.  Each step runs over the m proofs on host threads.
  struct Parts {
    DeltaMultiples dm;
    G1Affine A, B1, K, Z, ar, s_ar, bs1, r_bs1;
    G2Affine B2, bs;
  };
  std::vector<Parts> p(m);
  auto each = [&](auto fn) -> int {
    return host_parallel(m, fn) ? 0 : fail(B200G16_ERR_STATE, "prove: could not start the host assembly threads");
  };
  B200_TRY(each([&](size_t j) { p[j].dm = delta_multiples(pk, r[j], s[j]); }));
  B200_CUDA(cudaEventSynchronize(ctx->ev_slot[4]));   // the tails finish in enqueue order: B2, B1, A, K, Z
  B200_TRY(each([&](size_t j) {
    msm_collect<Fp2>(ctx, 4, cfg[4], &p[j].B2, j);
    p[j].bs = host_sum<Fp2>({p[j].B2, pk->beta2, p[j].dm.s_delta2});
  }));
  B200_CUDA(cudaEventSynchronize(ctx->ev_slot[1]));
  B200_TRY(each([&](size_t j) {
    msm_collect<Fp>(ctx, 1, cfg[1], &p[j].B1, j);
    p[j].bs1 = host_sum<Fp>({p[j].B1, pk->beta, p[j].dm.s_delta});
    p[j].r_bs1 = host_scalar_mul_aff<Fp>(p[j].bs1, r[j]);
  }));
  B200_CUDA(cudaEventSynchronize(ctx->ev_slot[0]));
  B200_TRY(each([&](size_t j) {
    msm_collect<Fp>(ctx, 0, cfg[0], &p[j].A, j);
    p[j].ar = host_sum<Fp>({p[j].A, pk->alpha, p[j].dm.r_delta});
    p[j].s_ar = host_scalar_mul_aff<Fp>(p[j].ar, s[j]);
  }));
  B200_CUDA(cudaStreamSynchronize(st));
  B200_TRY(each([&](size_t j) {
    Parts& q = p[j];
    msm_collect<Fp>(ctx, 2, cfg[2], &q.K, j);
    msm_collect<Fp>(ctx, 3, cfg[3], &q.Z, j);
    const G1Affine krs = host_sum<Fp>({q.K, q.Z, q.dm.kr_delta, q.s_ar, q.r_bs1});
    b200g16_proof* o = out + j;
    memset(o, 0, sizeof(*o));
    memcpy(o->ar, &q.ar, 64);
    memcpy(o->bs, &q.bs, 128);
    memcpy(o->krs, &krs, 64);
    memcpy(o->bs1, &q.bs1, 64);
    memcpy(o->msm_a, &q.A, 64);
    memcpy(o->msm_b1, &q.B1, 64);
    memcpy(o->msm_k, &q.K, 64);
    memcpy(o->msm_z, &q.Z, 64);
    memcpy(o->msm_b2, &q.B2, 128);
  }));
  *ev_io = ev;
  return 0;
}

// proofs per sub-batch: every one of the five MSMs fits one batch call (msm_batch_max).
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

// The body of b200g16_prove(_dev) (k = 1) and b200g16_prove_batch(_dev), called under ctx->mu: k proofs of one circuit
// in sub-batches of as many proofs as every MSM allows in one batch call.  Per sub-batch of m proofs:
// rows(j0, m, &wires, &a, &b, &c) gives the device rows of proofs [j0, j0 + m) — m x n_wires and m x N, h is left in the
// a rows — (the host path uploads the wires there); abc(j0, m) runs once the witness MSMs are enqueued and makes the
// main stream wait for the a, b, c rows (the host path uploads them there, under those MSMs); then computeH per proof
// and prove_back.  ctx->timings: the 8 intervals of a single prove (upload, gather, B2, B1, A, K, computeH, Z), summed
// over the sub-batches.  Any error drains the streams and leaves the ctx usable.
template <class Rows, class Abc>
static int prove_batch_run(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const uint64_t* r, const uint64_t* s,
                           b200g16_proof* out, Rows&& rows, Abc&& abc) {
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "prove: another prove is already open on this ctx");
  size_t slot_bytes = 0;
  const size_t m_max = k > 1 ? std::min(k, prove_batch_max(ctx, pk, &slot_bytes)) : 1;
  // (k = 1 MSMs stage their window sums in the small ws.pinned: a caller that never batches allocates no batch staging)
  if (m_max > 1) B200_TRY(msm_batch_stage(ctx, m_max * slot_bytes));
  std::vector<Fr> fr_r(k), fr_s(k);
  memcpy(fr_r.data(), r, k * sizeof(Fr));
  memcpy(fr_s.data(), s, k * sizeof(Fr));
  const size_t N = (size_t)1 << pk->log2n;
  cudaStream_t st = ctx->stream;
  auto body = [&]() -> int {
    for (size_t j0 = 0; j0 < k;) {
      const size_t m = std::min(m_max, k - j0);
      int ev = 0;
      cudaEventRecord(ctx->ev[ev++], st);
      const Fr* w = nullptr;
      Fr *a = nullptr, *b = nullptr, *c = nullptr;
      B200_TRY(rows(j0, m, &w, &a, &b, &c));
      cudaEventRecord(ctx->ev[ev++], st);
      B200_TRY(prove_front(ctx, pk, w, pk->n_wires, m, &ev));
      B200_TRY(abc(j0, m));
      for (size_t j = 0; j < m; j++) B200_TRY(compute_h_device(ctx, a + j * N, b + j * N, c + j * N, (int)pk->log2n, false));
      cudaEventRecord(ctx->ev[ev++], st);
      B200_TRY(prove_back(ctx, pk, a, N, m, fr_r.data() + j0, fr_s.data() + j0, out + j0, &ev));
      events_to_timings(ctx, ev, /*add=*/j0 > 0);
      j0 += m;
    }
    return 0;
  };
  const int status = body();
  if (status) msm_drain(ctx);
  return status;
}

static int prove_batch_check(b200g16_ctx* ctx, const b200g16_pk* pk, const char* what) {
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "%s: pk lives on another device", what);
  if (pk->partial) return fail(B200G16_ERR_ARG, "%s: a partial (sharded) pk cannot be batch-proved", what);
  return 0;
}

// The host path of b200g16_prove and b200g16_prove_batch: wires (k x n_wires), a, b, c (k x n_constraints each) in host
// memory, staged through ctx->io_a and the computeH buffers ctx->ntt.a/b/c (h is left in ntt.a).  The witness goes
// first: it gates the four MSMs, which are enqueued BEFORE a, b, c are touched — a copy from pageable memory (a Go
// slice) occupies the calling thread while it is staged, and the GPU should already be busy.  a, b, c then cross PCIe
// on the copy stream under those MSMs.
int prove_from_host(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const uint64_t* wires, size_t n_wires,
                           const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints,
                           const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out) {
  const size_t N = (size_t)1 << pk->log2n;
  cudaStream_t st = ctx->stream, cs = ctx->copy_stream;
  DevBuf* bufs[3] = {&ctx->ntt.a, &ctx->ntt.b, &ctx->ntt.c};
  const uint64_t* src[3] = {a, b, c};
  auto rows = [&](size_t j0, size_t m, const Fr** w, Fr** da, Fr** db, Fr** dc) -> int {
    B200_TRY(ctx->io_a.ensure((n_wires ? m * n_wires : 1) * sizeof(Fr)));
    B200_TRY(h2d_copy(ctx, ctx->io_a.p, wires + j0 * n_wires * 4, m * n_wires * sizeof(Fr), st));
    for (int i = 0; i < 3; i++) B200_TRY(bufs[i]->ensure(m * N * sizeof(Fr)));   // (no allocation once the MSMs are in flight)
    B200_CUDA(cudaEventRecord(ctx->ev_copy[1], st));
    *w = ctx->io_a.as<Fr>();
    *da = ctx->ntt.a.as<Fr>();
    *db = ctx->ntt.b.as<Fr>();
    *dc = ctx->ntt.c.as<Fr>();
    return 0;
  };
  auto abc = [&](size_t j0, size_t m) -> int {
    B200_CUDA(cudaStreamWaitEvent(cs, ctx->ev_copy[1], 0));   // the rows' previous readers (an earlier prove or sub-batch) are done
    for (int i = 0; i < 3; i++)
      for (size_t j = 0; j < m; j++) {
        char* row = (char*)bufs[i]->p + j * N * sizeof(Fr);
        B200_TRY(h2d_copy(ctx, row, src[i] + (j0 + j) * n_constraints * 4, n_constraints * sizeof(Fr), cs));
        if (N > n_constraints)
          B200_CUDA(cudaMemsetAsync(row + n_constraints * sizeof(Fr), 0, (N - n_constraints) * sizeof(Fr), cs));
      }
    B200_CUDA(cudaEventRecord(ctx->ev_copy[0], cs));
    B200_CUDA(cudaStreamWaitEvent(st, ctx->ev_copy[0], 0));
    return 0;
  };
  return prove_batch_run(ctx, pk, k, r, s, proofs_out, rows, abc);
}

// The device path of b200g16_prove_dev and b200g16_prove_batch_dev: the caller's rows, n_wires and N apart.
static int prove_on_device(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const void* d_wires, void* d_a, void* d_b,
                           void* d_c, const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out) {
  const size_t N = (size_t)1 << pk->log2n;
  auto rows = [&](size_t j0, size_t, const Fr** w, Fr** da, Fr** db, Fr** dc) -> int {
    *w = (const Fr*)d_wires + j0 * pk->n_wires;
    *da = (Fr*)d_a + j0 * N;
    *db = (Fr*)d_b + j0 * N;
    *dc = (Fr*)d_c + j0 * N;
    return 0;
  };
  auto abc = [](size_t, size_t) -> int { return 0; };
  return prove_batch_run(ctx, pk, k, r, s, proofs_out, rows, abc);
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
  B200_TRY(prove_from_host(ctx, pk, 1, wires, n_wires, a, b, c, n_constraints, r, s, proof_out));
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
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return prove_from_host(ctx, pk, k, wires, n_wires, a, b, c, n_constraints, r, s, proofs_out);
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
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return prove_on_device(ctx, pk, k, d_wires, d_a, d_b, d_c, r, s, proofs_out);
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
  B200_TRY(prove_front(ctx, pk, (const Fr*)d_wires, pk->n_wires, 1, &ev));
  cudaEventRecord(ctx->ev[ev++], ctx->stream);   // (computeH was done elsewhere: an empty interval)
  Fr fr_r, fr_s;
  memcpy(&fr_r, r, 32);
  memcpy(&fr_s, s, 32);
  B200_TRY(prove_back(ctx, pk, (const Fr*)d_h, (size_t)1 << pk->log2n, 1, &fr_r, &fr_s, proof_out, &ev));
  events_to_timings(ctx, ev);
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
  B200_TRY(prove_front(ctx, pk, (const Fr*)d_wires, pk->n_wires, 1, &ev));
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
  B200_TRY(prove_back(ctx, pk, (const Fr*)d_h, (size_t)1 << pk->log2n, 1, &fr_r, &fr_s, proof_out, &ev));
  events_to_timings(ctx, ev);
  return 0;
}

int b200g16_prove_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires, void* d_a, void* d_b, void* d_c,
                      const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out) {
  if (!ctx || !pk || !d_wires || !d_a || !d_b || !d_c || !r || !s || !proof_out)
    return fail(B200G16_ERR_ARG, "prove_dev: null");
  if (pk->device != ctx->device) return fail(B200G16_ERR_STATE, "prove_dev: pk lives on another device");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return prove_on_device(ctx, pk, 1, d_wires, d_a, d_b, d_c, r, s, proof_out);
}

}  // extern "C"
