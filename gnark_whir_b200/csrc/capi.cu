// extern "C" surface of libb200g16 (see include/b200g16.h for the contract and the
// gnark / gnark-crypto routines each entry point replaces).
#include "msm_impl.cuh"
#include "host_copy.cuh"

namespace b200 {
// instantiated in msm_g1.cu / msm_g2.cu
extern template int msm_enqueue<Fp>(b200g16_ctx*, const Affine<Fp>*, const MsmTable*, const Fr*, size_t, size_t, size_t, int, MsmCfg*,
                                   bool, bool);
extern template int msm_collect<Fp>(b200g16_ctx*, int, const MsmCfg&, Affine<Fp>*, size_t);
extern template int msm_device<Fp>(b200g16_ctx*, const Affine<Fp>*, const MsmTable*, const Fr*, size_t, Affine<Fp>*);
extern template int msm_build_table<Fp>(b200g16_ctx*, Affine<Fp>*, size_t, int, int);
extern template int msm_enqueue<Fp2>(b200g16_ctx*, const Affine<Fp2>*, const MsmTable*, const Fr*, size_t, size_t, size_t, int, MsmCfg*,
                                   bool, bool);
extern template int msm_collect<Fp2>(b200g16_ctx*, int, const MsmCfg&, Affine<Fp2>*, size_t);
extern template int msm_device<Fp2>(b200g16_ctx*, const Affine<Fp2>*, const MsmTable*, const Fr*, size_t, Affine<Fp2>*);
extern template int msm_build_table<Fp2>(b200g16_ctx*, Affine<Fp2>*, size_t, int, int);

template <class F>
int fixed_base_mul_device(b200g16_ctx* ctx, const Affine<F>& base, const Fr* d_scalars, size_t n, Affine<F>* d_out);
int modmul_probe(b200g16_ctx* ctx, int blocks_per_sm, int chains, int iters, double* modmul_per_s, float* ms_out);
int pipe_probe(b200g16_ctx* ctx, int mode, int blocks_per_sm, int iters, double* ops_per_s, float* ms_out);
int fp52_probe(b200g16_ctx* ctx, int variant, int blocks_per_sm, int iters, double* modmul_per_s, float* ms_out);
int ntt_device(b200g16_ctx* ctx, Fr* d_data, int L, int batch, bool inverse, bool coset, int decimation);
int compute_h_device(b200g16_ctx* ctx, Fr* a, Fr* b, Fr* c, int L, bool sync_and_time);
int h_pointwise_device(b200g16_ctx* ctx, Fr* a, const Fr* b, const Fr* c, int L);
int keccak_f_batch_device(b200g16_ctx* ctx, uint64_t* d_states, size_t n);
int sponge_batch_device(b200g16_ctx* ctx, const uint8_t* d_in, size_t in_len, size_t n, uint8_t* d_out, size_t out_len);
int merkle_paths_device(b200g16_ctx* ctx, const uint8_t* d_leaves, size_t leaf_len, const uint64_t* d_sib,
                        const uint64_t* d_auth, const uint64_t* d_idx, unsigned height, size_t n,
                        const uint64_t* d_expected_root, uint64_t* d_roots, uint8_t* d_ok);
int keccak_duplex_device(b200g16_ctx* ctx, uint64_t* d_digests, size_t n, const uint8_t* tag, size_t tag_len,
                         const b200g16_duplex_op* d_ops, size_t n_ops, const uint8_t* d_in, size_t in_stride,
                         uint8_t* d_out, size_t out_stride);
int keccak_duplex_check_device(b200g16_ctx* ctx, const uint64_t* d_digests, size_t n, uint32_t* d_flag, bool* bad);

// out[i] = k_i * base; result either copied to the host (out_host) or kept as a new bases handle
template <class F>
static int fixed_base_entry(b200g16_ctx* ctx, const uint64_t* base, const uint64_t* scalars, size_t n, int group,
                            uint64_t* out_host, b200g16_bases** out_bases) {
  if (!ctx || !base || (n && !scalars) || (!out_host && !out_bases)) return fail(B200G16_ERR_ARG, "fixed_base: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  Affine<F> b;
  memcpy(&b, base, sizeof(b));
  B200_TRY(ctx->io_a.ensure((n ? n : 1) * sizeof(Fr)));
  if (n) B200_CUDA(cudaMemcpyAsync(ctx->io_a.p, scalars, n * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
  Affine<F>* d_out = nullptr;
  b200g16_bases* h = nullptr;
  if (out_bases) {
    h = new b200g16_bases();
    h->group = group;
    h->n = n;
    h->device = ctx->device;
    cudaError_t e = cudaMalloc(&h->d_points, (n ? n : 1) * sizeof(Affine<F>));
    if (e != cudaSuccess) { delete h; return fail(B200G16_ERR_CUDA, "fixed_base: %s", cudaGetErrorString(e)); }
    d_out = reinterpret_cast<Affine<F>*>(h->d_points);
  } else {
    B200_TRY(ctx->io_b.ensure((n ? n : 1) * sizeof(Affine<F>)));
    d_out = ctx->io_b.as<Affine<F>>();
  }
  int st = fixed_base_mul_device<F>(ctx, b, ctx->io_a.as<Fr>(), n, d_out);
  if (st == 0 && out_host && n) {
    cudaError_t e = cudaMemcpy(out_host, d_out, n * sizeof(Affine<F>), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) st = fail(B200G16_ERR_CUDA, "fixed_base: %s", cudaGetErrorString(e));
  }
  if (st != 0 && h) { cudaFree(h->d_points); delete h; h = nullptr; }
  if (out_bases) *out_bases = h;
  return st;
}

// Host scalars of a large MSM are uploaded in MSM_PIPE_CHUNKS pieces of growing size on a copy stream; piece j's
// sub-MSM (its own point sub-range, its own result slot) runs while piece j+1 is still crossing PCIe,
// and the host adds the partial results.  Below MSM_PIPE_MIN points one copy + one MSM is faster.
constexpr size_t MSM_PIPE_MIN = (size_t)1 << 20;
constexpr int MSM_PIPE_CHUNKS = 4;   // at n >= 2^22; two pieces below (every sub-MSM pays its own sort and tail)

template <class F>
static int msm_entry(b200g16_ctx* ctx, const b200g16_bases* bases, int group, size_t offset, const void* scalars,
                     bool scalars_on_device, size_t n, uint64_t* out) {
  if (!ctx || !bases || !out || (n && !scalars)) return fail(B200G16_ERR_ARG, "msm: null argument");
  if (bases->group != group) return fail(B200G16_ERR_ARG, "msm: bases are G%d, call is G%d", bases->group, group);
  if (bases->device != ctx->device) return fail(B200G16_ERR_STATE, "msm: bases live on another device");
  if (offset > bases->n || n > bases->n - offset)
    return fail(B200G16_ERR_ARG, "msm: range [%zu,%zu) exceeds %zu bases", offset, offset + n, bases->n);
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active)   // the split prove's four pending MSMs own the result slots and the rotating buffer sets
    return fail(B200G16_ERR_STATE, "msm: a prove is open on this ctx (b200g16_prove_begin_dev without _end_dev)");
  B200_CUDA(cudaSetDevice(ctx->device));
  MsmTable tab;
  const MsmTable* tp = nullptr;
  Affine<F> res;
  if (!scalars_on_device && n >= MSM_PIPE_MIN) {
    B200_TRY(ctx->msm.scalars.ensure(n * sizeof(Fr)));
    const Fr* h = reinterpret_cast<const Fr*>(scalars);
    Fr* d = ctx->msm.scalars.as<Fr>();
    MsmCfg cfg[MSM_PIPE_CHUNKS];
    size_t lo[MSM_PIPE_CHUNKS + 1];
    const int pieces = n >= ((size_t)1 << 22) ? MSM_PIPE_CHUNKS : 2;
    // Geometric pieces (1 : 2 : 4 : 8): only the FIRST piece's copy is exposed, so it is the smallest, and each later
    // piece's copy hides behind the sub-MSM of the piece before it (a sub-MSM takes 2-4x as long as its own copy).
    // 2^24 end to end from pinned memory 41.1 -> 39.6 ms, 2^22 12.2 -> 11.9 ms (3, 5 or 6 pieces: no better); from
    // pageable memory, staged by h2d_copy's host threads, 43.2 -> 41.0 ms.  (With the DRIVER staging pageable memory
    // at ~10 GB/s the pipeline was copy-bound and equal pieces won: 57.8 ms.)
    const bool geometric = n >= ((size_t)1 << 21);   // (2^20: two equal pieces are 2% faster)
    for (int j = 0; j <= pieces; j++)
      lo[j] = geometric ? (size_t)(((unsigned __int128)n * (((size_t)1 << j) - 1)) / (((size_t)1 << pieces) - 1))
                        : n * (size_t)j / pieces;
    ctx->timings.n = 0;
    for (int j = 0; j < pieces; j++) {
      const size_t m = lo[j + 1] - lo[j];
      B200_TRY(h2d_copy(ctx, d + lo[j], h + lo[j], m * sizeof(Fr), ctx->copy_stream));
      B200_CUDA(cudaEventRecord(ctx->ev_copy[j], ctx->copy_stream));
      B200_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy[j], 0));
      const Affine<F>* pts = msm_operand<F>(bases, offset + lo[j], &tab, &tp);
      B200_TRY(msm_enqueue<F>(ctx, pts, tp, d + lo[j], m, 1, m, j, &cfg[j], false));
    }
    B200_TRY(msm_join(ctx));
    B200_CUDA(cudaStreamSynchronize(ctx->stream));
    XYZZ<F> acc = XYZZ<F>::inf();
    for (int j = 0; j < pieces; j++) {
      Affine<F> part;
      B200_TRY(msm_collect<F>(ctx, j, cfg[j], &part));
      acc.madd(part);
    }
    res = acc.to_affine();
  } else {
    const Fr* d_scalars = reinterpret_cast<const Fr*>(scalars);
    if (!scalars_on_device && n) {
      B200_TRY(ctx->msm.scalars.ensure(n * sizeof(Fr)));
      B200_TRY(h2d_copy(ctx, ctx->msm.scalars.p, scalars, n * sizeof(Fr), ctx->stream));
      d_scalars = ctx->msm.scalars.as<Fr>();
    }
    const Affine<F>* pts = msm_operand<F>(bases, offset, &tab, &tp);
    B200_TRY(msm_device<F>(ctx, pts, tp, d_scalars, n, &res));
  }
  memcpy(out, &res, sizeof(res));
  return 0;
}

// k MSMs of n scalars each over the same resident bases: out[j] = sum_i scalars[j * n + i] * bases[offset + i].
// Sub-batches of msm_batch_max vectors, up to MSM_BATCH_SLOTS of them enqueued back to back (each sub-batch's bucket
// reduction runs under the next one's sort and accumulate), then one synchronisation and the host's Horner per vector.
// k == 1, and a shape whose sub-batches hold one vector, take the single-MSM path.
constexpr int MSM_BATCH_SLOTS = 5;   // result slots 0..4: 5..7 belong to open b200g16_msm_g1_begin tickets

template <class F>
static int msm_batch_entry(b200g16_ctx* ctx, const b200g16_bases* bases, int group, size_t offset, const void* scalars,
                           bool scalars_on_device, size_t n, size_t k, uint64_t* out) {
  if (!ctx || !bases || (k && (!out || (n && !scalars)))) return fail(B200G16_ERR_ARG, "msm_batch: null argument");
  if (bases->group != group) return fail(B200G16_ERR_ARG, "msm_batch: bases are G%d, call is G%d", bases->group, group);
  if (bases->device != ctx->device) return fail(B200G16_ERR_STATE, "msm_batch: bases live on another device");
  if (offset > bases->n || n > bases->n - offset)
    return fail(B200G16_ERR_ARG, "msm_batch: range [%zu,%zu) exceeds %zu bases", offset, offset + n, bases->n);
  if (n >= (1ull << 31)) return fail(B200G16_ERR_ARG, "msm_batch: n=%zu too large", n);
  if (n && k > SIZE_MAX / sizeof(Fr) / n) return fail(B200G16_ERR_ARG, "msm_batch: k x n overflows");
  if (k == 0) return 0;
  constexpr size_t words = sizeof(Affine<F>) / sizeof(uint64_t);
  if (k == 1) return msm_entry<F>(ctx, bases, group, offset, scalars, scalars_on_device, n, out);
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active)
    return fail(B200G16_ERR_STATE, "msm_batch: a prove is open on this ctx (b200g16_prove_begin_dev without _end_dev)");
  B200_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  ctx->timings.n = 0;
  B200_CUDA(cudaEventRecord(ctx->ev[0], st));
  const Fr* d = reinterpret_cast<const Fr*>(scalars);
  if (!scalars_on_device && n) {
    B200_TRY(ctx->msm.scalars.ensure(k * n * sizeof(Fr)));
    B200_TRY(h2d_copy(ctx, ctx->msm.scalars.p, scalars, k * n * sizeof(Fr), st));
    d = ctx->msm.scalars.as<Fr>();
  }
  MsmTable tab;
  const MsmTable* tp = nullptr;
  const Affine<F>* pts = msm_operand<F>(bases, offset, &tab, &tp);
  const int c = msm_window_for(ctx, tp, n);
  const size_t ksub = std::min(k, msm_batch_max(c, tp != nullptr, n));
  if (ksub > 1) B200_TRY(msm_batch_stage(ctx, ksub * (tp ? 1 : msm_num_windows(c)) * sizeof(XYZZ<F>)));
  MsmCfg cfg[MSM_BATCH_SLOTS];
  size_t first[MSM_BATCH_SLOTS];
  int pending = 0;
  auto run = [&]() -> int {
    for (size_t j0 = 0; j0 < k;) {
      pending = 0;
      for (; pending < MSM_BATCH_SLOTS && j0 < k; pending++) {
        const size_t m = std::min(ksub, k - j0);
        first[pending] = j0;
        B200_TRY(msm_enqueue<F>(ctx, pts, tp, d + j0 * n, n, m, n, pending, &cfg[pending], false));
        j0 += m;
      }
      B200_TRY(msm_join(ctx));
      B200_CUDA(cudaStreamSynchronize(st));
      for (int q = 0; q < pending; q++)
        for (size_t j = 0; j < std::max<size_t>(cfg[q].k, 1); j++) {
          Affine<F> res;
          B200_TRY(msm_collect<F>(ctx, q, cfg[q], &res, j));
          memcpy(out + (first[q] + j) * words, &res, sizeof(res));
        }
      pending = 0;
    }
    return 0;
  };
  if (int status = run()) {
    msm_drain(ctx);
    return status;
  }
  B200_CUDA(cudaEventRecord(ctx->ev[1], st));
  B200_CUDA(cudaEventSynchronize(ctx->ev[1]));
  cudaEventElapsedTime(&ctx->timings.ms[0], ctx->ev[0], ctx->ev[1]);
  ctx->timings.n = 1;
  return 0;
}

template <class F>
static int upload(b200g16_ctx* ctx, const uint64_t* points, size_t n, int group, b200g16_bases** out) {
  if (!ctx || !out || (n && !points)) return fail(B200G16_ERR_ARG, "bases_upload: null argument");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  b200g16_bases* b = new b200g16_bases();
  b->group = group;
  b->n = n;
  b->device = ctx->device;
  size_t bytes = (n ? n : 1) * sizeof(Affine<F>);
  cudaError_t e = cudaMalloc(&b->d_points, bytes);
  if (e == cudaSuccess && n) e = cudaMemcpy(b->d_points, points, n * sizeof(Affine<F>), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (b->d_points) cudaFree(b->d_points);
    delete b;
    return fail(B200G16_ERR_CUDA, "bases_upload: %s", cudaGetErrorString(e));
  }
  *out = b;
  return 0;
}

// grow a resident vector into a window table: W rows of n points, row k = 2^(c k) * row 0
template <class F>
static int precompute(b200g16_ctx* ctx, b200g16_bases* b, int c) {
  const size_t n = b->n;
  if (n == 0) return 0;
  if (c == 0) c = msm_pick_table_window(n);
  if (c < 8 || c > 22) return fail(B200G16_ERR_ARG, "bases_precompute: window %d outside [8, 22]", c);
  const int W = msm_num_windows(c);
  if ((double)n * W >= 2.0e9) return fail(B200G16_ERR_ARG, "bases_precompute: %zu x %d points exceed the entry index", n, W);
  Affine<F>* table = nullptr;
  cudaError_t e = cudaMalloc(&table, (size_t)W * n * sizeof(Affine<F>));
  if (e != cudaSuccess)
    return fail(B200G16_ERR_CUDA, "bases_precompute: %d rows of %zu points: %s", W, n, cudaGetErrorString(e));
  e = cudaMemcpyAsync(table, b->d_points, n * sizeof(Affine<F>), cudaMemcpyDeviceToDevice, ctx->stream);
  int st = e == cudaSuccess ? msm_build_table<F>(ctx, table, n, c, W)
                            : fail(B200G16_ERR_CUDA, "bases_precompute: %s", cudaGetErrorString(e));
  if (st) { cudaFree(table); return st; }
  cudaFree(b->d_points);
  b->d_points = table;
  b->tab_c = c;
  b->tab_W = W;
  return 0;
}

template <class F>
static void host_add(const uint64_t* a, const uint64_t* b, uint64_t* out) {
  Affine<F> pa, pb;
  memcpy(&pa, a, sizeof(pa));
  memcpy(&pb, b, sizeof(pb));
  XYZZ<F> acc = XYZZ<F>::from_affine(pa);
  acc.madd(pb);
  Affine<F> r = acc.to_affine();
  memcpy(out, &r, sizeof(r));
}

template <class F>
static void host_scalar_mul(const uint64_t* p, const uint64_t* k, uint64_t* out) {
  Affine<F> pa;
  Fr s;
  memcpy(&pa, p, sizeof(pa));
  memcpy(&s, k, sizeof(s));
  s = Fr::from_mont(s);
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int i = 255; i >= 0; i--) {
    acc.dbl();
    if ((s.l[i >> 5] >> (i & 31)) & 1) acc.madd(pa);
  }
  Affine<F> r = acc.to_affine();
  memcpy(out, &r, sizeof(r));
}

// A new vector on `device` with src's points (its window table included), the copy enqueued on `st` (a stream of
// that device, which must be current) and not waited for.  A resident vector is complete once the call that made it
// returned (upload, precompute, setup and fixed-base calls all synchronise), so the copy needs no wait on src.
int bases_copy_enqueue(int device, cudaStream_t st, const b200g16_bases* src, b200g16_bases** out) {
  const size_t sz = src->group == 1 ? sizeof(G1Affine) : sizeof(G2Affine);
  const size_t rows = src->tab_c ? (size_t)src->tab_W : 1;
  const size_t bytes = src->n * rows * sz;
  b200g16_bases* b = new b200g16_bases();
  b->group = src->group;
  b->n = src->n;
  b->device = device;
  b->tab_c = src->tab_c;
  b->tab_W = src->tab_W;
  cudaError_t e = cudaMalloc(&b->d_points, bytes ? bytes : sz);
  if (e == cudaSuccess && bytes) e = cudaMemcpyPeerAsync(b->d_points, device, src->d_points, src->device, bytes, st);
  if (e != cudaSuccess) {
    cudaGetLastError();
    if (b->d_points) cudaFree(b->d_points);
    delete b;
    return fail(B200G16_ERR_CUDA, "bases_copy: %zu bytes from device %d to %d: %s", bytes, src->device, device,
                cudaGetErrorString(e));
  }
  *out = b;
  return 0;
}
}  // namespace b200

using namespace b200;

extern "C" {

int b200g16_version(void) { return 120; }  // 1.2: window tables, verify / pairing, wire formats, staged computeH

const char* b200g16_last_error(void) { return last_error_buf(); }

int b200g16_init(int device, b200g16_ctx** out) {
  if (!out) return fail(B200G16_ERR_ARG, "init: out is null");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(B200G16_ERR_NO_DEVICE, "init: no CUDA device (%s); this library has no CPU fallback",
                e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(B200G16_ERR_ARG, "init: device %d of %d", device, count);
  cudaDeviceProp prop;
  B200_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(B200G16_ERR_NO_DEVICE, "init: device %d is sm_%d%d; kernels are built for sm_100a only", device,
                prop.major, prop.minor);
  B200_CUDA(cudaSetDevice(device));
  b200g16_ctx* ctx = new b200g16_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  B200_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  {  // the tails are short, latency-bound kernels: let them run ahead of the next MSM's bulk work
    int prio_lo = 0, prio_hi = 0;
    B200_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    B200_CUDA(cudaStreamCreateWithPriority(&ctx->tail_stream, cudaStreamNonBlocking, prio_hi));
  }
  B200_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (auto& ev : ctx->ev_copy) B200_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto& ev : ctx->ev_slot) B200_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto& ev : ctx->ev) B200_CUDA(cudaEventCreate(&ev));
  for (int i = 0; i < MSM_SETS; i++) {
    B200_CUDA(cudaEventCreateWithFlags(&ctx->ev_front[i], cudaEventDisableTiming));
    B200_CUDA(cudaEventCreateWithFlags(&ctx->ev_tail[i], cudaEventDisableTiming));
  }
  *out = ctx;
  return 0;
}

void b200g16_destroy(b200g16_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->tail_stream);
  std::vector<DevBuf*> bufs = {&ctx->msm.scalars, &ctx->msm.part, &ctx->msm.bins, &ctx->msm.entries, &ctx->ntt.a, &ctx->ntt.b,
                               &ctx->ntt.c,       &ctx->ntt.tw,     &ctx->ntt.coset,   &ctx->ntt.fused, &ctx->ntt.dist, &ctx->io_a,  &ctx->io_b,
                               &ctx->io_c};
  for (int i = 0; i < MSM_SETS; i++)
    for (DevBuf* b : {&ctx->msm.counts[i], &ctx->msm.partials[i], &ctx->msm.chunks[i], &ctx->msm.misc[i], &ctx->msm.tasks[i]})
      bufs.push_back(b);
  for (auto& b : ctx->async_scalars) bufs.push_back(&b);
  for (DevBuf* b : bufs) b->release();
  for (int v = 0; v < 3; v++) {
    for (int d = 0; d < 8; d++)
      if (ctx->dist_h.ipc_opened[v][d]) cudaIpcCloseMemHandle(ctx->dist_h.peers[v][d]);
    ctx->dist_h.slice[v].release();
  }
  if (ctx->msm.pinned) cudaFreeHost(ctx->msm.pinned);
  if (ctx->msm.batch_pinned) cudaFreeHost(ctx->msm.batch_pinned);
  for (auto& ev : ctx->ev) cudaEventDestroy(ev);
  for (int i = 0; i < MSM_SETS; i++) { cudaEventDestroy(ctx->ev_front[i]); cudaEventDestroy(ctx->ev_tail[i]); }
  for (auto& ev : ctx->ev_copy) cudaEventDestroy(ev);
  for (auto& ev : ctx->ev_slot) cudaEventDestroy(ev);
  h2d_stager_release(ctx);
  cudaStreamDestroy(ctx->copy_stream);
  cudaStreamDestroy(ctx->tail_stream);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

uint64_t b200g16_launch_count(const b200g16_ctx* ctx) { return ctx ? ctx->launches : 0; }

int b200g16_last_timings(const b200g16_ctx* ctx, float* out_ms, int cap) {
  if (!ctx || !out_ms) return 0;
  int n = ctx->timings.n < cap ? ctx->timings.n : cap;
  for (int i = 0; i < n; i++) out_ms[i] = ctx->timings.ms[i];
  return n;
}

int b200g16_set_msm_window(b200g16_ctx* ctx, int c) {
  if (!ctx || c < 0 || c > 24 || c == 1) return fail(B200G16_ERR_ARG, "set_msm_window: bad argument");
  ctx->msm_window_override = c;
  return 0;
}

int b200g16_set_msm_batch_affine(b200g16_ctx* ctx, int mode, int levels, unsigned min_pairs) {
  if (!ctx || mode < 0 || mode > 2 || levels < 0 || levels > AFF_LEVELS_MAX)
    return fail(B200G16_ERR_ARG, "set_msm_batch_affine: bad argument");
  std::lock_guard<std::mutex> lock(ctx->mu);
  ctx->msm_affine_mode = mode;
  if (levels) ctx->msm_affine_levels = levels;
  if (min_pairs) ctx->msm_affine_min_pairs = min_pairs;
  return 0;
}

int b200g16_bases_upload_g1(b200g16_ctx* ctx, const uint64_t* points, size_t n, b200g16_bases** out) {
  return upload<Fp>(ctx, points, n, 1, out);
}
int b200g16_bases_upload_g2(b200g16_ctx* ctx, const uint64_t* points, size_t n, b200g16_bases** out) {
  return upload<Fp2>(ctx, points, n, 2, out);
}
void b200g16_bases_free(b200g16_bases* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  if (b->d_points) cudaFree(b->d_points);
  delete b;
}
size_t b200g16_bases_len(const b200g16_bases* b) { return b ? b->n : 0; }

int b200g16_bases_precompute(b200g16_ctx* ctx, b200g16_bases* b, int window_bits) {
  if (!ctx || !b) return fail(B200G16_ERR_ARG, "bases_precompute: null");
  if (b->device != ctx->device) return fail(B200G16_ERR_STATE, "bases_precompute: bases live on another device");
  if (b->tab_c) return fail(B200G16_ERR_STATE, "bases_precompute: vector already carries a c=%d table", b->tab_c);
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return b->group == 1 ? precompute<Fp>(ctx, b, window_bits) : precompute<Fp2>(ctx, b, window_bits);
}
int b200g16_bases_window(const b200g16_bases* b) { return b ? b->tab_c : 0; }

int b200g16_msm_plan(const b200g16_ctx* ctx, const b200g16_bases* b, size_t n, int* window_bits, int* windows) {
  if (!ctx || !b || !window_bits || !windows) return fail(B200G16_ERR_ARG, "msm_plan: null");
  int c = b->tab_c ? b->tab_c : (ctx->msm_window_override ? ctx->msm_window_override : msm_pick_window(n));
  *window_bits = c;
  *windows = msm_num_windows(c);
  return 0;
}

int b200g16_bases_download(const b200g16_bases* b, size_t offset, size_t n, uint64_t* out) {
  if (!b || !out) return fail(B200G16_ERR_ARG, "bases_download: null");
  if (offset > b->n || n > b->n - offset) return fail(B200G16_ERR_ARG, "bases_download: range");
  size_t sz = b->group == 1 ? sizeof(G1Affine) : sizeof(G2Affine);
  B200_CUDA(cudaSetDevice(b->device));
  B200_CUDA(cudaMemcpy(out, (const char*)b->d_points + offset * sz, n * sz, cudaMemcpyDeviceToHost));
  return 0;
}

int b200g16_bases_copy(b200g16_ctx* ctx, const b200g16_bases* src, b200g16_bases** out) {
  if (!ctx || !src || !out) return fail(B200G16_ERR_ARG, "bases_copy: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  b200g16_bases* b = nullptr;
  B200_TRY(bases_copy_enqueue(ctx->device, ctx->stream, src, &b));
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    b200g16_bases_free(b);
    return fail(B200G16_ERR_CUDA, "bases_copy: %s", cudaGetErrorString(e));
  }
  *out = b;
  return 0;
}

int b200g16_fixed_base_mul_g1(b200g16_ctx* ctx, const uint64_t base[8], const uint64_t* scalars, size_t n,
                              uint64_t* out_points) {
  return fixed_base_entry<Fp>(ctx, base, scalars, n, 1, out_points, nullptr);
}
int b200g16_fixed_base_mul_g2(b200g16_ctx* ctx, const uint64_t base[16], const uint64_t* scalars, size_t n,
                              uint64_t* out_points) {
  return fixed_base_entry<Fp2>(ctx, base, scalars, n, 2, out_points, nullptr);
}
int b200g16_bases_from_scalars_g1(b200g16_ctx* ctx, const uint64_t base[8], const uint64_t* scalars, size_t n,
                                  b200g16_bases** out) {
  return fixed_base_entry<Fp>(ctx, base, scalars, n, 1, nullptr, out);
}
int b200g16_bases_from_scalars_g2(b200g16_ctx* ctx, const uint64_t base[16], const uint64_t* scalars, size_t n,
                                  b200g16_bases** out) {
  return fixed_base_entry<Fp2>(ctx, base, scalars, n, 2, nullptr, out);
}

int b200g16_modmul_probe(b200g16_ctx* ctx, int blocks_per_sm, int chains, int iters, double* modmul_per_s,
                         float* ms) {
  if (!ctx || !modmul_per_s || !ms || blocks_per_sm < 1 || iters < 1) return fail(B200G16_ERR_ARG, "probe: bad arg");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return modmul_probe(ctx, blocks_per_sm, chains, iters, modmul_per_s, ms);
}

int b200g16_pipe_probe(b200g16_ctx* ctx, int mode, int blocks_per_sm, int iters, double* ops_per_s, float* ms) {
  if (!ctx || !ops_per_s || !ms || mode < 0 || mode > 9 || blocks_per_sm < 1 || iters < 1)
    return fail(B200G16_ERR_ARG, "pipe_probe: bad arg");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return pipe_probe(ctx, mode, blocks_per_sm, iters, ops_per_s, ms);
}

int b200g16_fp52_probe(b200g16_ctx* ctx, int variant, int blocks_per_sm, int iters, double* modmul_per_s, float* ms) {
  if (!ctx || !modmul_per_s || !ms || variant < 0 || variant > 5 || blocks_per_sm < 1 || iters < 1)
    return fail(B200G16_ERR_ARG, "fp52_probe: bad arg");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return fp52_probe(ctx, variant, blocks_per_sm, iters, modmul_per_s, ms);
}

int b200g16_msm_g1(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars, size_t n,
                   uint64_t out[8]) {
  return msm_entry<Fp>(ctx, bases, 1, offset, scalars, false, n, out);
}
int b200g16_msm_g2(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars, size_t n,
                   uint64_t out[16]) {
  return msm_entry<Fp2>(ctx, bases, 2, offset, scalars, false, n, out);
}
int b200g16_msm_g1_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars, size_t n,
                       uint64_t out[8]) {
  return msm_entry<Fp>(ctx, bases, 1, offset, d_scalars, true, n, out);
}
int b200g16_msm_g2_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars, size_t n,
                       uint64_t out[16]) {
  return msm_entry<Fp2>(ctx, bases, 2, offset, d_scalars, true, n, out);
}

int b200g16_msm_g1_batch(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars, size_t n,
                         size_t k, uint64_t* out) {
  return msm_batch_entry<Fp>(ctx, bases, 1, offset, scalars, false, n, k, out);
}
int b200g16_msm_g2_batch(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars, size_t n,
                         size_t k, uint64_t* out) {
  return msm_batch_entry<Fp2>(ctx, bases, 2, offset, scalars, false, n, k, out);
}
int b200g16_msm_g1_batch_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars, size_t n,
                             size_t k, uint64_t* out) {
  return msm_batch_entry<Fp>(ctx, bases, 1, offset, d_scalars, true, n, k, out);
}
int b200g16_msm_g2_batch_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars, size_t n,
                             size_t k, uint64_t* out) {
  return msm_batch_entry<Fp2>(ctx, bases, 2, offset, d_scalars, true, n, k, out);
}

// ---- asynchronous G1 MSM: enqueue now, take the result later.  gnark runs pedersen.ProveKnowledge after Solve and
// before the five MSMs of Prove; nothing in between depends on its result, so a host can enqueue it, call
// b200g16_prove, and collect it afterwards — its sort and accumulate run first, its bucket reduction hides under the
// prove's first MSM, and no synchronisation of its own is paid.
constexpr int ASYNC_FIRST_SLOT = 5;   // a prove owns slots 0..4, a pipelined host-scalar MSM 0..3
static int msm_begin(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* scalars, bool on_device,
                     size_t n, int* ticket) {
  if (!ctx || !bases || !ticket || (n && !scalars)) return fail(B200G16_ERR_ARG, "msm_begin: null argument");
  if (bases->group != 1) return fail(B200G16_ERR_ARG, "msm_begin: G1 bases expected");
  if (bases->device != ctx->device) return fail(B200G16_ERR_STATE, "msm_begin: bases live on another device");
  if (offset > bases->n || n > bases->n - offset)
    return fail(B200G16_ERR_ARG, "msm_begin: range [%zu,%zu) exceeds %zu bases", offset, offset + n, bases->n);
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active) return fail(B200G16_ERR_STATE, "msm_begin: a prove is open on this ctx");
  int t = 0;
  while (t < 3 && ctx->async_open[t]) t++;
  if (t == 3) return fail(B200G16_ERR_STATE, "msm_begin: all three tickets are open (b200g16_msm_g1_end releases one)");
  B200_CUDA(cudaSetDevice(ctx->device));
  const Fr* d_scalars = reinterpret_cast<const Fr*>(scalars);
  if (!on_device && n) {
    B200_TRY(ctx->async_scalars[t].ensure(n * sizeof(Fr)));
    B200_TRY(h2d_copy(ctx, ctx->async_scalars[t].p, scalars, n * sizeof(Fr), ctx->stream));
    d_scalars = ctx->async_scalars[t].as<Fr>();
  }
  MsmTable tab;
  const MsmTable* tp = nullptr;
  const Affine<Fp>* pts = msm_operand<Fp>(bases, offset, &tab, &tp);
  B200_TRY(msm_enqueue<Fp>(ctx, pts, tp, d_scalars, n, 1, n, ASYNC_FIRST_SLOT + t, &ctx->async_cfg[t], false));
  ctx->async_open[t] = true;
  *ticket = t;
  return 0;
}

int b200g16_msm_g1_begin(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars, size_t n,
                         int* ticket) {
  return msm_begin(ctx, bases, offset, scalars, false, n, ticket);
}
int b200g16_msm_g1_begin_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars, size_t n,
                             int* ticket) {
  return msm_begin(ctx, bases, offset, d_scalars, true, n, ticket);
}
int b200g16_msm_g1_end(b200g16_ctx* ctx, int ticket, uint64_t out[8]) {
  if (!ctx || !out || ticket < 0 || ticket >= 3) return fail(B200G16_ERR_ARG, "msm_end: bad argument");
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (!ctx->async_open[ticket]) return fail(B200G16_ERR_STATE, "msm_end: ticket %d is not open", ticket);
  B200_CUDA(cudaSetDevice(ctx->device));
  ctx->async_open[ticket] = false;
  if (ctx->async_cfg[ticket].W) B200_CUDA(cudaEventSynchronize(ctx->ev_slot[ASYNC_FIRST_SLOT + ticket]));
  Affine<Fp> res;
  B200_TRY(msm_collect<Fp>(ctx, ASYNC_FIRST_SLOT + ticket, ctx->async_cfg[ticket], &res));
  memcpy(out, &res, sizeof(res));
  return 0;
}

int b200g16_ntt_dev(b200g16_ctx* ctx, void* d_data, unsigned log2n, unsigned batch, int inverse, int coset,
                    int decimation) {
  if (!ctx || !d_data) return fail(B200G16_ERR_ARG, "ntt: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  B200_TRY(ntt_device(ctx, reinterpret_cast<Fr*>(d_data), (int)log2n, (int)batch, inverse != 0, coset != 0, decimation));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b200g16_ntt(b200g16_ctx* ctx, uint64_t* data, unsigned log2n, int inverse, int coset, int decimation) {
  if (!ctx || !data) return fail(B200G16_ERR_ARG, "ntt: null");
  if (log2n > 28) return fail(B200G16_ERR_ARG, "ntt: log2n=%u exceeds the field's two-adicity (28)", log2n);
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  size_t bytes = ((size_t)1 << log2n) * sizeof(Fr);
  B200_TRY(ctx->ntt.a.ensure(bytes));
  B200_TRY(h2d_copy(ctx, ctx->ntt.a.p, data, bytes, ctx->stream));
  B200_TRY(ntt_device(ctx, ctx->ntt.a.as<Fr>(), (int)log2n, 1, inverse != 0, coset != 0, decimation));
  B200_TRY(d2h_copy(ctx, data, ctx->ntt.a.p, bytes, ctx->stream));
  return 0;
}

int b200g16_compute_h_dev(b200g16_ctx* ctx, void* d_a, void* d_b, void* d_c, unsigned log2n) {
  if (!ctx || !d_a || !d_b || !d_c) return fail(B200G16_ERR_ARG, "compute_h: null");
  if (log2n > 28) return fail(B200G16_ERR_ARG, "compute_h: log2n=%u exceeds two-adicity 28", log2n);
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  return compute_h_device(ctx, reinterpret_cast<Fr*>(d_a), reinterpret_cast<Fr*>(d_b), reinterpret_cast<Fr*>(d_c),
                          (int)log2n, true);
}

int b200g16_h_pointwise_dev(b200g16_ctx* ctx, void* d_a, const void* d_b, const void* d_c, unsigned log2n) {
  if (!ctx || !d_a || !d_b || !d_c) return fail(B200G16_ERR_ARG, "h_pointwise: null");
  if (log2n > 28) return fail(B200G16_ERR_ARG, "h_pointwise: log2n=%u exceeds two-adicity 28", log2n);
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  B200_TRY(h_pointwise_device(ctx, reinterpret_cast<Fr*>(d_a), reinterpret_cast<const Fr*>(d_b),
                              reinterpret_cast<const Fr*>(d_c), (int)log2n));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b200g16_compute_h(b200g16_ctx* ctx, const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints,
                      unsigned log2n, uint64_t* h_out) {
  if (!ctx || !a || !b || !c || !h_out) return fail(B200G16_ERR_ARG, "compute_h: null");
  if (log2n > 28) return fail(B200G16_ERR_ARG, "compute_h: log2n=%u exceeds two-adicity 28", log2n);
  size_t n = (size_t)1 << log2n;
  if (n_constraints > n) return fail(B200G16_ERR_ARG, "compute_h: %zu constraints > domain %zu", n_constraints, n);
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  DevBuf* bufs[3] = {&ctx->ntt.a, &ctx->ntt.b, &ctx->ntt.c};
  const uint64_t* src[3] = {a, b, c};
  for (int i = 0; i < 3; i++) {
    B200_TRY(bufs[i]->ensure(n * sizeof(Fr)));
    B200_TRY(h2d_copy(ctx, bufs[i]->p, src[i], n_constraints * sizeof(Fr), ctx->stream));
    if (n > n_constraints)  // computeH pads a, b, c with zeros up to the domain cardinality
      B200_CUDA(cudaMemsetAsync((char*)bufs[i]->p + n_constraints * sizeof(Fr), 0, (n - n_constraints) * sizeof(Fr),
                                ctx->stream));
  }
  B200_TRY(compute_h_device(ctx, ctx->ntt.a.as<Fr>(), ctx->ntt.b.as<Fr>(), ctx->ntt.c.as<Fr>(), (int)log2n, true));
  B200_TRY(d2h_copy(ctx, h_out, ctx->ntt.a.p, n * sizeof(Fr), ctx->stream));
  return 0;
}

int b200g16_keccak_f_batch_dev(b200g16_ctx* ctx, void* d_states, size_t n) {
  if (!ctx || (n && !d_states)) return fail(B200G16_ERR_ARG, "keccak_f_batch: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  B200_TRY(keccak_f_batch_device(ctx, reinterpret_cast<uint64_t*>(d_states), n));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b200g16_keccak_f_batch(b200g16_ctx* ctx, uint64_t* states, size_t n) {
  if (!ctx || (n && !states)) return fail(B200G16_ERR_ARG, "keccak_f_batch: null");
  if (n == 0) return 0;
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  size_t bytes = n * 200;
  B200_TRY(ctx->io_a.ensure(bytes));
  B200_TRY(h2d_copy(ctx, ctx->io_a.p, states, bytes, ctx->stream));
  B200_TRY(keccak_f_batch_device(ctx, ctx->io_a.as<uint64_t>(), n));
  B200_TRY(d2h_copy(ctx, states, ctx->io_a.p, bytes, ctx->stream));
  return 0;
}

int b200g16_keccak_sponge_batch(b200g16_ctx* ctx, const uint8_t* inputs, size_t in_len, size_t n, uint8_t* outputs,
                                size_t out_len) {
  if (!ctx || (n && in_len && !inputs) || (n && out_len && !outputs)) return fail(B200G16_ERR_ARG, "sponge: null");
  if (n == 0 || out_len == 0) return 0;
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  B200_TRY(ctx->io_a.ensure(n * in_len + 8));
  B200_TRY(ctx->io_b.ensure(n * out_len));
  if (in_len) B200_TRY(h2d_copy(ctx, ctx->io_a.p, inputs, n * in_len, ctx->stream));
  B200_TRY(sponge_batch_device(ctx, ctx->io_a.as<uint8_t>(), in_len, n, ctx->io_b.as<uint8_t>(), out_len));
  B200_TRY(d2h_copy(ctx, outputs, ctx->io_b.p, n * out_len, ctx->stream));
  return 0;
}

// Argument checks shared by both duplex entry points: fills the script's absorbed (*in_len) and squeezed (*out_len)
// bytes per sponge.  Returns 0 or B200G16_ERR_ARG (with the message set).
static int duplex_args(b200g16_ctx* ctx, const void* digests, size_t n, const uint8_t* tag, size_t tag_len,
                       const b200g16_duplex_op* ops, size_t n_ops, const void* inputs, const void* outputs,
                       size_t* in_len, size_t* out_len) {
  if (!ctx || (n && !digests) || (n_ops && !ops)) return fail(B200G16_ERR_ARG, "keccak_duplex: null");
  if (tag_len > 64) return fail(B200G16_ERR_ARG, "keccak_duplex: tag_len %zu > 64", tag_len);
  size_t a = 0, s = 0;
  for (size_t k = 0; k < n_ops; k++) {
    if (ops[k].squeeze > 1) return fail(B200G16_ERR_ARG, "keccak_duplex: op %zu has kind %u", k, ops[k].squeeze);
    size_t& acc = ops[k].squeeze ? s : a;
    if (acc > SIZE_MAX - ops[k].len) return fail(B200G16_ERR_ARG, "keccak_duplex: script length overflows");
    acc += ops[k].len;
  }
  if (n && (a > SIZE_MAX / n || s > SIZE_MAX / n)) return fail(B200G16_ERR_ARG, "keccak_duplex: n x row overflows");
  if (n && a && !inputs) return fail(B200G16_ERR_ARG, "keccak_duplex: null inputs");
  if (n && s && !outputs) return fail(B200G16_ERR_ARG, "keccak_duplex: null outputs");
  *in_len = a;
  *out_len = s;
  return 0;
}

int b200g16_keccak_duplex_batch(b200g16_ctx* ctx, b200g16_keccak_digest* digests, size_t n, const uint8_t* tag,
                                size_t tag_len, const b200g16_duplex_op* ops, size_t n_ops, const uint8_t* inputs,
                                uint8_t* outputs) {
  size_t A, S;
  B200_TRY(duplex_args(ctx, digests, n, tag, tag_len, ops, n_ops, inputs, outputs, &A, &S));
  if (!tag)
    for (size_t i = 0; i < n; i++)
      if (digests[i].absorb_pos > 136 || digests[i].squeeze_pos > 136)
        return fail(B200G16_ERR_ARG, "keccak_duplex: digest %zu has a position above 136", i);
  if (n == 0 || (n_ops == 0 && !tag)) return 0;
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  auto up16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
  const size_t sz_dg = n * sizeof(b200g16_keccak_digest), sz_ops = n_ops * sizeof(b200g16_duplex_op);
  const size_t o_ops = up16(sz_dg), o_in = o_ops + up16(sz_ops);
  B200_TRY(ctx->io_a.ensure(o_in + n * A));
  B200_TRY(ctx->io_b.ensure(n * S ? n * S : 1));
  char* d = ctx->io_a.as<char>();
  cudaStream_t st = ctx->stream;
  if (!tag) B200_TRY(h2d_copy(ctx, d, digests, sz_dg, st));
  if (sz_ops) B200_CUDA(cudaMemcpyAsync(d + o_ops, ops, sz_ops, cudaMemcpyHostToDevice, st));
  if (A) B200_TRY(h2d_copy(ctx, d + o_in, inputs, n * A, st));
  B200_TRY(keccak_duplex_device(ctx, (uint64_t*)d, n, tag, tag_len, (const b200g16_duplex_op*)(d + o_ops), n_ops,
                                (const uint8_t*)(d + o_in), A, ctx->io_b.as<uint8_t>(), S));
  if (S) B200_TRY(d2h_copy(ctx, outputs, ctx->io_b.p, n * S, st));
  B200_TRY(d2h_copy(ctx, digests, d, sz_dg, st));
  return 0;
}

int b200g16_keccak_duplex_batch_dev(b200g16_ctx* ctx, void* d_digests, size_t n, const uint8_t* tag, size_t tag_len,
                                    const b200g16_duplex_op* ops, size_t n_ops, const void* d_inputs, void* d_outputs) {
  size_t A, S;
  B200_TRY(duplex_args(ctx, d_digests, n, tag, tag_len, ops, n_ops, d_inputs, d_outputs, &A, &S));
  if (n == 0 || (n_ops == 0 && !tag)) return 0;
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  const size_t sz_ops = n_ops * sizeof(b200g16_duplex_op), o_flag = (sz_ops + 15) & ~(size_t)15;
  B200_TRY(ctx->io_a.ensure(o_flag + 16));
  char* d = ctx->io_a.as<char>();
  if (!tag) {   // every position is checked before any digest changes
    bool bad = false;
    B200_TRY(keccak_duplex_check_device(ctx, (const uint64_t*)d_digests, n, (uint32_t*)(d + o_flag), &bad));
    if (bad) return fail(B200G16_ERR_ARG, "keccak_duplex: a digest has a position above 136");
  }
  if (sz_ops) B200_CUDA(cudaMemcpyAsync(d, ops, sz_ops, cudaMemcpyHostToDevice, ctx->stream));
  B200_TRY(keccak_duplex_device(ctx, (uint64_t*)d_digests, n, tag, tag_len, (const b200g16_duplex_op*)d, n_ops,
                                (const uint8_t*)d_inputs, A, (uint8_t*)d_outputs, S));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b200g16_keccak_merkle_paths_dev(b200g16_ctx* ctx, const void* d_leaves, size_t leaf_len, const void* d_siblings,
                                    const void* d_auth_paths, const void* d_indexes, unsigned height, size_t n_paths,
                                    const void* d_expected_root, void* d_roots_out, void* d_ok_out) {
  if (!ctx) return fail(B200G16_ERR_ARG, "merkle: null ctx");
  if (height < 1 || height > 64) return fail(B200G16_ERR_ARG, "merkle: height %u", height);
  if (leaf_len == 0 || leaf_len % 8) return fail(B200G16_ERR_ARG, "merkle: leaf_len must be a positive multiple of 8");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  B200_TRY(merkle_paths_device(ctx, (const uint8_t*)d_leaves, leaf_len, (const uint64_t*)d_siblings,
                               (const uint64_t*)d_auth_paths, (const uint64_t*)d_indexes, height, n_paths,
                               (const uint64_t*)d_expected_root, (uint64_t*)d_roots_out, (uint8_t*)d_ok_out));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b200g16_keccak_merkle_paths(b200g16_ctx* ctx, const uint8_t* leaves, size_t leaf_len, const uint8_t* siblings,
                                const uint8_t* auth_paths, const uint64_t* indexes, unsigned height, size_t n_paths,
                                const uint8_t* expected_root, uint8_t* roots_out, uint8_t* ok_out) {
  if (!ctx || !leaves || !siblings || !indexes || (height > 1 && !auth_paths) || (!roots_out && !ok_out))
    return fail(B200G16_ERR_ARG, "merkle: null");
  if (height < 1 || height > 64) return fail(B200G16_ERR_ARG, "merkle: height %u", height);
  if (leaf_len == 0 || leaf_len % 8) return fail(B200G16_ERR_ARG, "merkle: leaf_len must be a positive multiple of 8");
  if (ok_out && !expected_root) return fail(B200G16_ERR_ARG, "merkle: ok_out needs expected_root");
  if (n_paths == 0) return 0;
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  const size_t n = n_paths;
  const size_t sz_leaves = n * leaf_len, sz_sib = n * 32, sz_auth = n * (size_t)(height - 1) * 32, sz_idx = n * 8;
  auto up8 = [](size_t v) { return (v + 15) & ~(size_t)15; };
  size_t o_sib = up8(sz_leaves), o_auth = o_sib + up8(sz_sib), o_idx = o_auth + up8(sz_auth),
         o_root = o_idx + up8(sz_idx), o_roots = o_root + 32, o_ok = o_roots + up8(n * 32), total = o_ok + up8(n);
  B200_TRY(ctx->io_a.ensure(total));
  char* d = ctx->io_a.as<char>();
  cudaStream_t st = ctx->stream;
  B200_TRY(h2d_copy(ctx, d, leaves, sz_leaves, st));
  B200_CUDA(cudaMemcpyAsync(d + o_sib, siblings, sz_sib, cudaMemcpyHostToDevice, st));
  if (sz_auth) B200_TRY(h2d_copy(ctx, d + o_auth, auth_paths, sz_auth, st));
  B200_CUDA(cudaMemcpyAsync(d + o_idx, indexes, sz_idx, cudaMemcpyHostToDevice, st));
  if (expected_root) B200_CUDA(cudaMemcpyAsync(d + o_root, expected_root, 32, cudaMemcpyHostToDevice, st));
  B200_TRY(merkle_paths_device(ctx, (const uint8_t*)d, leaf_len, (const uint64_t*)(d + o_sib),
                               (const uint64_t*)(d + o_auth), (const uint64_t*)(d + o_idx), height, n,
                               expected_root ? (const uint64_t*)(d + o_root) : nullptr, (uint64_t*)(d + o_roots),
                               ok_out ? (uint8_t*)(d + o_ok) : nullptr));
  if (roots_out) B200_CUDA(cudaMemcpyAsync(roots_out, d + o_roots, n * 32, cudaMemcpyDeviceToHost, st));
  if (ok_out) B200_CUDA(cudaMemcpyAsync(ok_out, d + o_ok, n, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int b200g16_g1_add(const uint64_t a[8], const uint64_t b[8], uint64_t out[8]) {
  if (!a || !b || !out) return fail(B200G16_ERR_ARG, "g1_add: null");
  host_add<Fp>(a, b, out);
  return 0;
}
int b200g16_g2_add(const uint64_t a[16], const uint64_t b[16], uint64_t out[16]) {
  if (!a || !b || !out) return fail(B200G16_ERR_ARG, "g2_add: null");
  host_add<Fp2>(a, b, out);
  return 0;
}
int b200g16_g1_scalar_mul(const uint64_t p[8], const uint64_t k[4], uint64_t out[8]) {
  if (!p || !k || !out) return fail(B200G16_ERR_ARG, "g1_scalar_mul: null");
  host_scalar_mul<Fp>(p, k, out);
  return 0;
}
int b200g16_g2_scalar_mul(const uint64_t p[16], const uint64_t k[4], uint64_t out[16]) {
  if (!p || !k || !out) return fail(B200G16_ERR_ARG, "g2_scalar_mul: null");
  host_scalar_mul<Fp2>(p, k, out);
  return 0;
}

}  // extern "C"
