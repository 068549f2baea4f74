// One process, several GPUs: the C-ABI a single-process host (gnark's Go prover calls groth16.Prove once,
// /root/reference/mt.go:496) uses to spread one prove / one MSM over the GPUs of a box.
//
// A group is one b200g16_ctx per device, driven by one host thread per device (kernel launches of the
// devices proceed in parallel; a single enqueueing thread would serialise ~1 ms of launches per device).
// Sharding is by point range (BASELINE.json north_star): device i holds entries [lo_i, hi_i) of every
// proving-key vector; a prove runs
//     owners of a, b, c (devices v mod min(n, 3)):  H2D of the vector -> iNTT -> coset NTT
//     root (device 0): coset evaluations of b and c arrive by peer copies (cudaMemcpyPeerAsync over NVLink),
//                      pointwise (a b - c) / (g^N - 1), last inverse coset transform -> h
//     every device: the four witness MSMs on its shard (front), its slice of h by one peer copy, the Z MSM
//     host: the n x 5 partial points are added (n - 1 additions each) and the proof is assembled
// No NCCL, no collective library: the only data crossing devices are two vectors into the root, one slice of h
// out to each device, and 5 points per device back to the host.
#include <algorithm>
#include <array>
#include <condition_variable>
#include <thread>

#include "prove.cuh"
#include "host_copy.cuh"

using namespace b200;

struct b200g16_group {
  int n = 0;
  std::vector<b200g16_ctx*> ctx;
  std::vector<int> devices;
  cudaEvent_t ev_vec[3] = {nullptr, nullptr, nullptr};  // coset evaluations of a / b / c ready on their owner
  cudaEvent_t ev_h = nullptr;                           // h ready on the root
  std::vector<cudaEvent_t> ev_stage[4];                 // distributed computeH: stage s enqueued on device i
  std::mutex mu;                                        // one group call at a time
};

struct b200g16_group_bases {
  int group = 1;
  size_t n = 0;
  std::vector<b200g16_bases*> shard;
  std::vector<size_t> lo;
};

// sharded (b200g16_group_pk_upload): shard[i] holds a point range of every vector; replicated
// (b200g16_group_pk_replicate): shard[i] is the whole key on member i's device, its vectors borrowed from the source
// or from `copies` (one set per distinct device other than the source's, shared by the members on that device)
struct b200g16_group_pk {
  unsigned log2n = 0;
  size_t n_wires = 0;
  std::vector<b200g16_pk*> shard;
  bool replicated = false;
  const b200g16_group* group = nullptr;   // the group that built it
  std::vector<b200g16_bases*> copies;
};

namespace {

void shard_range(size_t n, int i, int world, size_t* lo, size_t* hi) {
  size_t base = n / world, rem = n % world;
  *lo = (size_t)i * base + ((size_t)i < rem ? (size_t)i : rem);
  *hi = *lo + base + ((size_t)i < rem ? 1 : 0);
}

int vector_owner(int v, int n) { return v % (n < 3 ? n : 3); }

// host-side rendezvous between the device threads: "the work that produces X has been ENQUEUED and its event recorded"
struct Flag {
  std::mutex m;
  std::condition_variable cv;
  bool set = false;
  int status = 0;
  void signal(int st) {
    { std::lock_guard<std::mutex> l(m); if (!set || st) { set = true; status = st; } }
    cv.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> l(m);
    cv.wait(l, [&] { return set; });
    return status;
  }
};

// all device threads meet here between the stages of a distributed computeH; a failing thread keeps arriving (with
// its status) so nobody waits forever, and everybody learns that somebody failed
struct Barrier {
  std::mutex m;
  std::condition_variable cv;
  int n, count = 0, gen = 0, status = 0;
  explicit Barrier(int n_) : n(n_) {}
  int arrive(int st) {
    std::unique_lock<std::mutex> l(m);
    if (st && !status) status = st;
    const int my = gen;
    if (++count == n) { count = 0; gen++; cv.notify_all(); }
    else cv.wait(l, [&] { return gen != my; });
    return status;
  }
};

int log2_of(int n) {
  for (int g = 0; g < 6; g++)
    if ((1 << g) == n) return g;
  return -1;
}

// fn(i) on one thread per device; the first failing device's status and message become the caller's
template <class Fn>
int run_on_all(b200g16_group* g, Fn fn) {
  std::vector<int> st(g->n, 0);
  std::vector<std::string> msg(g->n);
  std::vector<std::thread> th;
  for (int i = 0; i < g->n; i++)
    th.emplace_back([&, i] {
      last_error_buf()[0] = 0;
      st[i] = fn(i);
      if (st[i]) msg[i] = last_error_buf();
    });
  for (auto& t : th) t.join();
  for (int i = 0; i < g->n; i++)
    if (st[i]) return fail(st[i], "device %d: %s", g->devices[i], msg[i].c_str());
  return 0;
}

}  // namespace

extern "C" {

int b200g16_group_init(const int* devices, int n, b200g16_group** out) {
  if (!devices || !out || n < 1 || n > 64) return fail(B200G16_ERR_ARG, "group_init: bad argument");
  b200g16_group* g = new b200g16_group();
  g->n = n;
  for (int i = 0; i < n; i++) {
    b200g16_ctx* c = nullptr;
    int st = b200g16_init(devices[i], &c);
    if (st) {
      for (auto* x : g->ctx) b200g16_destroy(x);
      delete g;
      return st;
    }
    g->ctx.push_back(c);
    g->devices.push_back(devices[i]);
  }
  // direct peer access where the hardware offers it (NVLink / NVSwitch); copies fall back to staging otherwise
  for (int i = 0; i < n; i++) {
    cudaSetDevice(devices[i]);
    for (int j = 0; j < n; j++) {
      if (devices[i] == devices[j]) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) == cudaSuccess && can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
        if (e != cudaSuccess) cudaGetLastError();  // already enabled: not an error for us
      }
    }
  }
  for (int v = 0; v < 3; v++) {
    cudaSetDevice(devices[vector_owner(v, n)]);
    B200_CUDA(cudaEventCreateWithFlags(&g->ev_vec[v], cudaEventDisableTiming));
  }
  cudaSetDevice(devices[0]);
  B200_CUDA(cudaEventCreateWithFlags(&g->ev_h, cudaEventDisableTiming));
  for (auto& evs : g->ev_stage) {
    evs.assign(n, nullptr);
    for (int i = 0; i < n; i++) {
      cudaSetDevice(devices[i]);
      B200_CUDA(cudaEventCreateWithFlags(&evs[i], cudaEventDisableTiming));
    }
  }
  *out = g;
  return 0;
}

void b200g16_group_destroy(b200g16_group* g) {
  if (!g) return;
  for (int v = 0; v < 3; v++)
    if (g->ev_vec[v]) cudaEventDestroy(g->ev_vec[v]);
  if (g->ev_h) cudaEventDestroy(g->ev_h);
  for (auto& evs : g->ev_stage)
    for (auto e : evs)
      if (e) cudaEventDestroy(e);
  for (auto* c : g->ctx) b200g16_destroy(c);
  delete g;
}

int b200g16_group_size(const b200g16_group* g) { return g ? g->n : 0; }

b200g16_ctx* b200g16_group_ctx(b200g16_group* g, int i) { return (g && i >= 0 && i < g->n) ? g->ctx[i] : nullptr; }

// ---- page-locking of caller memory (Go slices are pageable: H2D from them runs at a fraction of PCIe speed)
int b200g16_host_register(void* p, size_t bytes) {
  if (!p || !bytes) return fail(B200G16_ERR_ARG, "host_register: null");
  cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(B200G16_ERR_CUDA, "host_register: %s", cudaGetErrorString(e)); }
  return 0;
}
int b200g16_host_unregister(void* p) {
  if (!p) return fail(B200G16_ERR_ARG, "host_unregister: null");
  cudaError_t e = cudaHostUnregister(p);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(B200G16_ERR_CUDA, "host_unregister: %s", cudaGetErrorString(e)); }
  return 0;
}

// ---- sharded resident bases + MSM
static int group_bases_upload(b200g16_group* g, const uint64_t* points, size_t n, int group, b200g16_group_bases** out) {
  if (!g || !out || (n && !points)) return fail(B200G16_ERR_ARG, "group_bases_upload: null");
  std::lock_guard<std::mutex> lock(g->mu);
  b200g16_group_bases* b = new b200g16_group_bases();
  b->group = group;
  b->n = n;
  b->shard.assign(g->n, nullptr);
  b->lo.assign(g->n + 1, 0);
  const size_t words = group == 1 ? 8 : 16;
  int st = run_on_all(g, [&](int i) {
    size_t lo, hi;
    shard_range(n, i, g->n, &lo, &hi);
    b->lo[i] = lo;
    if (i == g->n - 1) b->lo[g->n] = hi;
    return group == 1 ? b200g16_bases_upload_g1(g->ctx[i], points + lo * words, hi - lo, &b->shard[i])
                      : b200g16_bases_upload_g2(g->ctx[i], points + lo * words, hi - lo, &b->shard[i]);
  });
  if (st) {
    for (auto* s : b->shard) b200g16_bases_free(s);
    delete b;
    return st;
  }
  *out = b;
  return 0;
}

int b200g16_group_bases_upload_g1(b200g16_group* g, const uint64_t* points, size_t n, b200g16_group_bases** out) {
  return group_bases_upload(g, points, n, 1, out);
}
int b200g16_group_bases_upload_g2(b200g16_group* g, const uint64_t* points, size_t n, b200g16_group_bases** out) {
  return group_bases_upload(g, points, n, 2, out);
}

void b200g16_group_bases_free(b200g16_group_bases* b) {
  if (!b) return;
  for (auto* s : b->shard) b200g16_bases_free(s);
  delete b;
}

int b200g16_group_bases_precompute(b200g16_group* g, b200g16_group_bases* b, int window_bits) {
  if (!g || !b || (int)b->shard.size() != g->n) return fail(B200G16_ERR_ARG, "group_bases_precompute: bad argument");
  std::lock_guard<std::mutex> lock(g->mu);
  return run_on_all(g, [&](int i) {
    return b200g16_bases_len(b->shard[i]) ? b200g16_bases_precompute(g->ctx[i], b->shard[i], window_bits) : 0;
  });
}

static int group_msm(b200g16_group* g, const b200g16_group_bases* b, int group, const uint64_t* scalars, size_t n,
                     uint64_t* out) {
  if (!g || !b || !out || (n && !scalars)) return fail(B200G16_ERR_ARG, "group_msm: null");
  if (b->group != group || (int)b->shard.size() != g->n) return fail(B200G16_ERR_ARG, "group_msm: bases do not match");
  if (n != b->n) return fail(B200G16_ERR_ARG, "group_msm: %zu scalars for %zu sharded bases", n, b->n);
  std::lock_guard<std::mutex> lock(g->mu);
  const size_t words = group == 1 ? 8 : 16;
  std::vector<uint64_t> part((size_t)g->n * words, 0);
  B200_TRY(run_on_all(g, [&](int i) {
    const size_t lo = b->lo[i], m = b->lo[i + 1] - b->lo[i];
    return group == 1 ? b200g16_msm_g1(g->ctx[i], b->shard[i], 0, scalars + lo * 4, m, part.data() + (size_t)i * words)
                      : b200g16_msm_g2(g->ctx[i], b->shard[i], 0, scalars + lo * 4, m, part.data() + (size_t)i * words);
  }));
  if (group == 1) {
    G1Affine r = host_sum_points<Fp>(reinterpret_cast<const G1Affine*>(part.data()), g->n);
    memcpy(out, &r, sizeof(r));
  } else {
    G2Affine r = host_sum_points<Fp2>(reinterpret_cast<const G2Affine*>(part.data()), g->n);
    memcpy(out, &r, sizeof(r));
  }
  return 0;
}

int b200g16_group_msm_g1(b200g16_group* g, const b200g16_group_bases* b, const uint64_t* scalars, size_t n, uint64_t out[8]) {
  return group_msm(g, b, 1, scalars, n, out);
}
int b200g16_group_msm_g2(b200g16_group* g, const b200g16_group_bases* b, const uint64_t* scalars, size_t n, uint64_t out[16]) {
  return group_msm(g, b, 2, scalars, n, out);
}

// ---- sharded proving key
int b200g16_group_pk_upload(b200g16_group* g, const b200g16_pk_desc* d, b200g16_group_pk** out) {
  if (!g || !d || !out) return fail(B200G16_ERR_ARG, "group_pk_upload: null");
  if (d->res_a || d->res_b || d->res_k || d->res_z || d->res_b2 || d->partial)
    return fail(B200G16_ERR_ARG, "group_pk_upload: takes the whole key as host arrays (no resident vectors, partial = 0)");
  std::lock_guard<std::mutex> lock(g->mu);
  b200g16_group_pk* pk = new b200g16_group_pk();
  pk->log2n = d->log2_domain;
  pk->n_wires = d->n_wires;
  pk->group = g;
  pk->shard.assign(g->n, nullptr);
  int st = run_on_all(g, [&](int i) {
    b200g16_pk_desc s = *d;
    size_t lo, hi;
    shard_range(d->n_a, i, g->n, &lo, &hi);
    s.g1_a = d->g1_a ? d->g1_a + lo * 8 : nullptr; s.n_a = hi - lo; s.off_a = lo;
    shard_range(d->n_b, i, g->n, &lo, &hi);
    s.g1_b = d->g1_b ? d->g1_b + lo * 8 : nullptr; s.g2_b = d->g2_b ? d->g2_b + lo * 16 : nullptr; s.n_b = hi - lo; s.off_b = lo;
    shard_range(d->n_k, i, g->n, &lo, &hi);
    s.g1_k = d->g1_k ? d->g1_k + lo * 8 : nullptr; s.n_k = hi - lo; s.off_k = lo;
    shard_range(d->n_z, i, g->n, &lo, &hi);
    s.g1_z = d->g1_z ? d->g1_z + lo * 8 : nullptr; s.n_z = hi - lo; s.off_z = lo;
    s.partial = 1;
    return pk_build(g->ctx[i], &s, &pk->shard[i]);
  });
  if (st) {
    for (auto* s : pk->shard) pk_release(s);
    delete pk;
    return st;
  }
  *out = pk;
  return 0;
}

void b200g16_group_pk_free(b200g16_group_pk* pk) {
  if (!pk) return;
  for (auto* s : pk->shard) pk_release(s);
  for (auto* b : pk->copies) b200g16_bases_free(b);
  delete pk;
}

// ---- replicated proving key: the whole key on every device, for whole proofs per device
int b200g16_group_pk_replicate(b200g16_group* g, const b200g16_pk* src, b200g16_group_pk** out) {
  if (!g || !src || !out) return fail(B200G16_ERR_ARG, "group_pk_replicate: null");
  if (src->partial) return fail(B200G16_ERR_ARG, "group_pk_replicate: a partial (sharded) key cannot be replicated");
  std::lock_guard<std::mutex> glock(g->mu);
  const int n = g->n;
  // the distinct devices in group order; the first member on each lends its ctx (stream, lock) to the copies
  std::vector<int> dev, lead, slot(n);
  for (int i = 0; i < n; i++) {
    const auto it = std::find(dev.begin(), dev.end(), g->devices[i]);
    slot[i] = (int)(it - dev.begin());
    if (it == dev.end()) { dev.push_back(g->devices[i]); lead.push_back(i); }
  }
  const int D = (int)dev.size();
  std::vector<std::unique_lock<std::mutex>> locks;
  for (int d = 0; d < D; d++) locks.emplace_back(g->ctx[lead[d]]->mu);
  b200g16_group_pk* gpk = new b200g16_group_pk();
  gpk->log2n = src->log2n;
  gpk->n_wires = src->n_wires;
  gpk->replicated = true;
  gpk->group = g;
  gpk->shard.assign(n, nullptr);
  std::vector<std::array<b200g16_bases*, 5>> vecs(D);
  std::vector<cudaEvent_t> ready(D, nullptr);   // ready[d]: the copies onto dev[d] are complete
  std::vector<int> holders, todo;               // holders: devices that can serve a copy (-1: src, off the group)
  for (int d = 0; d < D; d++) {
    if (dev[d] == src->device) {
      for (int v = 0; v < 5; v++) vecs[d][v] = src->vec[v];
      holders.push_back(d);
    } else {
      todo.push_back(d);
    }
  }
  if (holders.empty()) holders.push_back(-1);
  auto body = [&]() -> int {
    // doubling broadcast: each round, every holder serves one device that has no copy yet
    for (size_t next = 0; next < todo.size();) {
      std::vector<int> fresh;
      for (int h : holders) {
        if (next == todo.size()) break;
        const int d = todo[next++];
        b200g16_ctx* c = g->ctx[lead[d]];
        B200_CUDA(cudaSetDevice(c->device));
        if (h >= 0 && ready[h]) B200_CUDA(cudaStreamWaitEvent(c->stream, ready[h], 0));
        for (int v = 0; v < 5; v++) {
          B200_TRY(bases_copy_enqueue(c->device, c->stream, h >= 0 ? vecs[h][v] : src->vec[v], &vecs[d][v]));
          gpk->copies.push_back(vecs[d][v]);
        }
        B200_CUDA(cudaEventCreateWithFlags(&ready[d], cudaEventDisableTiming));
        B200_CUDA(cudaEventRecord(ready[d], c->stream));
        fresh.push_back(d);
      }
      holders.insert(holders.end(), fresh.begin(), fresh.end());
    }
    // every member: the key's small points and sizes, the vectors of its device, its own gather lists
    for (int i = 0; i < n; i++) {
      const int d = slot[i];
      b200g16_ctx* c = g->ctx[lead[d]];
      B200_CUDA(cudaSetDevice(c->device));
      b200g16_pk* pk = new b200g16_pk(*src);
      for (int t = 0; t < 3; t++) pk->d_idx[t] = nullptr;
      for (int v = 0; v < 5; v++) { pk->vec[v] = vecs[d][v]; pk->owned[v] = false; }
      pk->device = c->device;
      gpk->shard[i] = pk;
      for (int t = 0; t < 3; t++) {
        B200_CUDA(cudaMalloc(&pk->d_idx[t], (pk->n_idx[t] ? pk->n_idx[t] : 1) * sizeof(uint32_t)));
        if (pk->n_idx[t])
          B200_CUDA(cudaMemcpyPeerAsync(pk->d_idx[t], c->device, src->d_idx[t], src->device, pk->n_idx[t] * sizeof(uint32_t),
                                        c->stream));
      }
    }
    return 0;
  };
  int st = body();
  for (int d = 0; d < D; d++) {   // every copy complete (or, after a failure, nothing in flight any more)
    b200g16_ctx* c = g->ctx[lead[d]];
    cudaSetDevice(c->device);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess && !st) st = fail(B200G16_ERR_CUDA, "group_pk_replicate: device %d: %s", c->device, cudaGetErrorString(e));
    if (ready[d]) cudaEventDestroy(ready[d]);
  }
  if (st) {
    b200g16_group_pk_free(gpk);
    return st;
  }
  *out = gpk;
  return 0;
}

static int dist_h_alloc(b200g16_ctx* ctx, unsigned log2n, int n_peers, int me);

// computeH split over all 2 / 4 / 8 devices of the group (ntt.cu: cross-GPU levels over peer memory), then the five
// MSMs on every device's shard.  Stages are separated by a host barrier + cross-device event waits.
static int group_prove_dist(b200g16_group* g, const b200g16_group_pk* gpk, const uint64_t* wires, size_t n_wires,
                            const uint64_t* const* src, size_t n_constraints, const Fr& fr_r, const Fr& fr_s,
                            std::vector<b200g16_proof>& parts) {
  const int n = g->n, L = (int)gpk->log2n, gl = log2_of(n);
  const size_t M = ((size_t)1 << L) >> gl;
  Barrier bar(n);
  return run_on_all(g, [&](int i) -> int {
    b200g16_ctx* ctx = g->ctx[i];
    const b200g16_pk* pk = gpk->shard[i];
    std::lock_guard<std::mutex> lock(ctx->mu);
    cudaStream_t stm = ctx->stream;
    int ev = 0;
    auto wait_all = [&](int stage) -> int {
      for (int j = 0; j < n; j++) B200_CUDA(cudaStreamWaitEvent(stm, g->ev_stage[stage][j], 0));
      return 0;
    };
    // ---- allocate / publish slices
    int st = [&]() -> int {
      B200_CUDA(cudaSetDevice(ctx->device));
      DistH& D = ctx->dist_h;
      bool mapped = false;
      for (int v = 0; v < 3; v++)
        for (int d = 0; d < 8; d++) mapped = mapped || D.ipc_opened[v][d];
      if (D.g && !mapped && (D.L != L || D.g != gl || D.me != i)) {
        // a key of another size: the previous prove ended with a stream sync and a barrier, and the peer pointers
        // are taken again after the next barrier, so nobody reads these slices any more
        for (int v = 0; v < 3; v++) D.slice[v].release();
        D = DistH();
      }
      return dist_h_alloc(ctx, (unsigned)L, n, i);
    }();
    st = bar.arrive(st);
    if (!st) st = [&]() -> int {
      DistH& D = ctx->dist_h;
      for (int d = 0; d < n; d++)
        for (int v = 0; v < 3; v++) D.peers[v][d] = g->ctx[d]->dist_h.slice[v].p;
      D.ready = true;
      cudaEventRecord(ctx->ev[ev++], stm);
      // witness on the copy stream, this device's slices of a, b, c (zero padded) on the main stream
      B200_TRY(ctx->io_a.ensure((n_wires ? n_wires : 1) * sizeof(Fr)));
      B200_TRY(h2d_copy(ctx, ctx->io_a.p, wires, n_wires * sizeof(Fr), ctx->copy_stream));
      B200_CUDA(cudaEventRecord(ctx->ev_copy[1], ctx->copy_stream));
      const size_t lo = (size_t)i * M;
      const size_t have = n_constraints > lo ? (n_constraints - lo < M ? n_constraints - lo : M) : 0;
      for (int v = 0; v < 3; v++) {
        char* dst = (char*)D.slice[v].p;
        if (have) B200_TRY(h2d_copy(ctx, dst, src[v] + lo * 4, have * sizeof(Fr), stm));
        if (have < M) B200_CUDA(cudaMemsetAsync(dst + have * sizeof(Fr), 0, (M - have) * sizeof(Fr), stm));
      }
      B200_CUDA(cudaEventRecord(g->ev_stage[0][i], stm));
      return 0;
    }();
    // ---- the four phases of the distributed computeH
    for (int phase = 0; phase < 4; phase++) {
      st = bar.arrive(st);
      if (!st) st = [&]() -> int {
        B200_TRY(wait_all(phase));   // every device has enqueued (and will have finished) the previous stage
        DistH& D = ctx->dist_h;
        B200_TRY(compute_h_dist_phase(ctx, reinterpret_cast<Fr* const (*)[8]>(D.peers), D.g, D.me, D.L, phase));
        if (phase < 3) B200_CUDA(cudaEventRecord(g->ev_stage[phase + 1][i], stm));
        return 0;
      }();
    }
    // ---- the MSMs on this device's shard; h slice = this device's a slice
    if (!st) st = [&]() -> int {
      B200_CUDA(cudaStreamWaitEvent(stm, ctx->ev_copy[1], 0));
      cudaEventRecord(ctx->ev[ev++], stm);
      B200_TRY(prove_front(ctx, pk, ctx->io_a.as<Fr>(), n_wires, 1, &ev));
      if (ev < 18) cudaEventRecord(ctx->ev[ev++], stm);
      const Fr* d_h = reinterpret_cast<const Fr*>(ctx->dist_h.slice[0].p) - pk->off_z;  // prove_back reads d_h[off_z, off_z + n_z)
      B200_TRY(prove_back(ctx, pk, d_h, (size_t)1 << L, 1, &fr_r, &fr_s, &parts[i], &ev));
      events_to_timings(ctx, ev);
      return 0;
    }();
    if (st) ctx->prove_active = false;
    // nobody may reuse (or free) its slices while a peer's cross kernel could still read them
    cudaStreamSynchronize(stm);
    st = bar.arrive(st);
    return st;
  });
}

// ---- the prove
int b200g16_group_prove(b200g16_group* g, const b200g16_group_pk* gpk, const uint64_t* wires, size_t n_wires,
                        const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints, const uint64_t r[4],
                        const uint64_t s[4], b200g16_proof* proof_out, uint64_t* h_out) {
  if (!g || !gpk || !wires || !a || !b || !c || !r || !s || !proof_out) return fail(B200G16_ERR_ARG, "group_prove: null");
  if (gpk->replicated)
    return fail(B200G16_ERR_ARG, "group_prove: a replicated key proves whole proofs per device (b200g16_group_prove_batch)");
  if ((int)gpk->shard.size() != g->n) return fail(B200G16_ERR_STATE, "group_prove: pk belongs to another group");
  if (n_wires != gpk->n_wires) return fail(B200G16_ERR_ARG, "group_prove: %zu wires, pk expects %zu", n_wires, gpk->n_wires);
  const int L = (int)gpk->log2n;
  const size_t N = (size_t)1 << L;
  if (n_constraints > N) return fail(B200G16_ERR_ARG, "group_prove: %zu constraints > domain %zu", n_constraints, N);
  std::lock_guard<std::mutex> glock(g->mu);
  const int n = g->n, root = 0;
  Fr fr_r, fr_s;
  memcpy(&fr_r, r, 32);
  memcpy(&fr_s, s, 32);
  const uint64_t* src[3] = {a, b, c};
  Flag vec_ready[3], h_ready;
  std::vector<b200g16_proof> parts(n);
  const int gl = log2_of(n);
  const bool dist = gl >= 1 && gl <= 3 && L >= 2 * gl + 1;
  for (int i = 0; dist && i < n; i++) {   // the h slices must coincide with the Z shards (true for whole keys: n_z = N - 1)
    const b200g16_pk* pk = gpk->shard[i];
    if (pk->off_z != (size_t)i * (N >> gl) || pk->n_z > (N >> gl)) return fail(B200G16_ERR_STATE, "group_prove: Z shard %d does not match its h slice", i);
  }
  int st = 0;
  if (dist) {
    st = group_prove_dist(g, gpk, wires, n_wires, src, n_constraints, fr_r, fr_s, parts);
  } else {
  auto abort_all = [&](int st) {
    for (auto& f : vec_ready) f.signal(st);
    h_ready.signal(st);
  };
  st = run_on_all(g, [&](int i) -> int {
    auto body = [&]() -> int {
      b200g16_ctx* ctx = g->ctx[i];
      const b200g16_pk* pk = gpk->shard[i];
      std::lock_guard<std::mutex> lock(ctx->mu);
      B200_CUDA(cudaSetDevice(ctx->device));
      cudaStream_t stm = ctx->stream;
      int ev = 0;
      cudaEventRecord(ctx->ev[ev++], stm);
      // the witness crosses PCIe on the copy stream while this device's share of computeH runs
      B200_TRY(ctx->io_a.ensure((n_wires ? n_wires : 1) * sizeof(Fr)));
      B200_TRY(h2d_copy(ctx, ctx->io_a.p, wires, n_wires * sizeof(Fr), ctx->copy_stream));
      B200_CUDA(cudaEventRecord(ctx->ev_copy[1], ctx->copy_stream));
      DevBuf* bufs[3] = {&ctx->ntt.a, &ctx->ntt.b, &ctx->ntt.c};
      for (int v = 0; v < 3; v++) {
        if (vector_owner(v, n) != i) continue;
        B200_TRY(bufs[v]->ensure(N * sizeof(Fr)));
        B200_TRY(h2d_copy(ctx, bufs[v]->p, src[v], n_constraints * sizeof(Fr), stm));
        if (N > n_constraints)
          B200_CUDA(cudaMemsetAsync((char*)bufs[v]->p + n_constraints * sizeof(Fr), 0, (N - n_constraints) * sizeof(Fr), stm));
        Fr* one[1] = {bufs[v]->as<Fr>()};
        const bool den[1] = {v != 1};   // (a b - c) / (g^N - 1) = (a / d) b - c / d: a and c carry the denominator
        B200_TRY(ntt_coset_pair_device(ctx, one, 1, L, den));
        B200_CUDA(cudaEventRecord(g->ev_vec[v], stm));
        vec_ready[v].signal(0);
      }
      const Fr* d_h = nullptr;
      if (i == root) {
        for (int v = 1; v < 3; v++) {
          const int o = vector_owner(v, n);
          if (o == root) continue;
          B200_TRY(bufs[v]->ensure(N * sizeof(Fr)));
          if (int ws = vec_ready[v].wait()) return fail(ws, "group_prove: the owner of vector %d failed", v);
          B200_CUDA(cudaStreamWaitEvent(stm, g->ev_vec[v], 0));
          DevBuf* rb[3] = {&g->ctx[o]->ntt.a, &g->ctx[o]->ntt.b, &g->ctx[o]->ntt.c};
          B200_CUDA(cudaMemcpyPeerAsync(bufs[v]->p, ctx->device, rb[v]->p, g->ctx[o]->device, N * sizeof(Fr), stm));
        }
        B200_TRY(h_pointwise_plain_device(ctx, ctx->ntt.a.as<Fr>(), ctx->ntt.b.as<Fr>(), ctx->ntt.c.as<Fr>(), L));
        B200_TRY(ntt_device(ctx, ctx->ntt.a.as<Fr>(), L, 1, true, true, B200G16_DIF));
        B200_CUDA(cudaEventRecord(g->ev_h, stm));
        h_ready.signal(0);
        d_h = ctx->ntt.a.as<Fr>();
      }
      B200_CUDA(cudaStreamWaitEvent(stm, ctx->ev_copy[1], 0));
      cudaEventRecord(ctx->ev[ev++], stm);
      B200_TRY(prove_front(ctx, pk, ctx->io_a.as<Fr>(), n_wires, 1, &ev));
      if (i != root) {
        B200_TRY(ctx->io_c.ensure((pk->n_z ? pk->n_z : 1) * sizeof(Fr)));
        if (int ws = h_ready.wait()) { ctx->prove_active = false; return fail(ws, "group_prove: the root device failed"); }
        B200_CUDA(cudaStreamWaitEvent(stm, g->ev_h, 0));
        if (pk->n_z)
          B200_CUDA(cudaMemcpyPeerAsync(ctx->io_c.p, ctx->device, g->ctx[root]->ntt.a.as<Fr>() + pk->off_z,
                                        g->ctx[root]->device, pk->n_z * sizeof(Fr), stm));
        d_h = ctx->io_c.as<Fr>() - pk->off_z;  // prove_back reads d_h[off_z, off_z + n_z)
      }
      if (ev < 18) cudaEventRecord(ctx->ev[ev++], stm);
      B200_TRY(prove_back(ctx, pk, d_h, N, 1, &fr_r, &fr_s, &parts[i], &ev));
      events_to_timings(ctx, ev);
      return 0;
    };
    int rc = body();
    if (rc) {
      g->ctx[i]->prove_active = false;
      abort_all(rc);
    }
    return rc;
  });
  }
  if (st) {
    for (int i = 0; i < n; i++) { cudaSetDevice(g->ctx[i]->device); cudaStreamSynchronize(g->ctx[i]->stream); }
    return st;
  }
  // n x 5 partial sums -> the five MultiExp results -> the proof
  std::vector<G1Affine> p1(n);
  std::vector<G2Affine> p2(n);
  G1Affine sums[4];
  const size_t offs[4] = {offsetof(b200g16_proof, msm_a), offsetof(b200g16_proof, msm_b1), offsetof(b200g16_proof, msm_k),
                          offsetof(b200g16_proof, msm_z)};
  for (int k = 0; k < 4; k++) {
    for (int i = 0; i < n; i++) memcpy(&p1[i], (const char*)&parts[i] + offs[k], 64);
    sums[k] = host_sum_points<Fp>(p1.data(), n);
  }
  for (int i = 0; i < n; i++) memcpy(&p2[i], parts[i].msm_b2, 128);
  G2Affine b2 = host_sum_points<Fp2>(p2.data(), n);
  B200_TRY(b200g16_prove_finish(gpk->shard[0], (const uint64_t*)&sums[0], (const uint64_t*)&sums[1], (const uint64_t*)&sums[2],
                                (const uint64_t*)&sums[3], (const uint64_t*)&b2, r, s, proof_out));
  if (h_out && dist) {
    const size_t M = N >> gl;
    for (int i = 0; i < n; i++) {
      B200_CUDA(cudaSetDevice(g->ctx[i]->device));
      B200_CUDA(cudaMemcpy(h_out + (size_t)i * M * 4, g->ctx[i]->dist_h.slice[0].p, M * sizeof(Fr), cudaMemcpyDeviceToHost));
    }
  } else if (h_out) {
    B200_CUDA(cudaSetDevice(g->ctx[root]->device));
    B200_CUDA(cudaMemcpy(h_out, g->ctx[root]->ntt.a.p, N * sizeof(Fr), cudaMemcpyDeviceToHost));
  }
  return 0;
}

// ---- k proofs over the group with a replicated key: contiguous ranges of proofs, b200g16_prove_batch's pipeline on
// every member from its own host thread, no data across devices
int b200g16_group_prove_batch(b200g16_group* g, const b200g16_group_pk* gpk, size_t k, const uint64_t* wires,
                              size_t n_wires, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                              size_t n_constraints, const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out) {
  if (!g || !gpk) return fail(B200G16_ERR_ARG, "group_prove_batch: null");
  if (k && (!wires || !a || !b || !c || !r || !s || !proofs_out)) return fail(B200G16_ERR_ARG, "group_prove_batch: null");
  if (gpk->group != g || (int)gpk->shard.size() != g->n)
    return fail(B200G16_ERR_STATE, "group_prove_batch: pk belongs to another group");
  if (!gpk->replicated)
    return fail(B200G16_ERR_ARG, "group_prove_batch: a sharded key proves one proof over the group (b200g16_group_prove)");
  if (n_wires != gpk->n_wires)
    return fail(B200G16_ERR_ARG, "group_prove_batch: %zu wires, pk expects %zu", n_wires, gpk->n_wires);
  const size_t N = (size_t)1 << gpk->log2n;
  if (n_constraints > N) return fail(B200G16_ERR_ARG, "group_prove_batch: %zu constraints > domain %zu", n_constraints, N);
  if (k && (n_wires > SIZE_MAX / sizeof(Fr) / k || N > SIZE_MAX / sizeof(Fr) / k))
    return fail(B200G16_ERR_ARG, "group_prove_batch: k x n_wires or k x N overflows");
  if (k == 0) return 0;
  std::lock_guard<std::mutex> glock(g->mu);
  const int st = run_on_all(g, [&](int i) -> int {
    size_t lo, hi;
    shard_range(k, i, g->n, &lo, &hi);
    if (lo == hi) return 0;
    b200g16_ctx* ctx = g->ctx[i];
    std::lock_guard<std::mutex> lock(ctx->mu);
    B200_CUDA(cudaSetDevice(ctx->device));
    return prove_from_host(ctx, gpk->shard[i], hi - lo, wires + lo * n_wires * 4, n_wires, a + lo * n_constraints * 4,
                           b + lo * n_constraints * 4, c + lo * n_constraints * 4, n_constraints, r + lo * 4, s + lo * 4,
                           proofs_out + lo);
  });
  if (st)   // (the failing member has drained its own streams; nothing of the others may still run either)
    for (int i = 0; i < g->n; i++) { cudaSetDevice(g->ctx[i]->device); cudaStreamSynchronize(g->ctx[i]->stream); }
  return st;
}

// ---- computeH split over 2 / 4 / 8 GPUs, one PROCESS per GPU (torch.distributed ranks): CUDA IPC maps every
// rank's slices into every other rank, the cross-GPU butterfly levels run as kernels over that peer memory
// (ntt.cu k_ntt_cross / k_ntt_cross_h), and the caller separates the four phases by barriers.
static int dist_h_alloc(b200g16_ctx* ctx, unsigned log2n, int n_peers, int me) {
  const int g = log2_of(n_peers);
  if (g < 1 || g > 3) return fail(B200G16_ERR_ARG, "dist_h: %d peers (2, 4 or 8)", n_peers);
  if (log2n > 28 || (int)log2n < 2 * g + 1) return fail(B200G16_ERR_ARG, "dist_h: 2^%u elements over %d devices", log2n, n_peers);
  if (me < 0 || me >= n_peers) return fail(B200G16_ERR_ARG, "dist_h: rank %d of %d", me, n_peers);
  DistH& D = ctx->dist_h;
  if (D.g && (D.L != (int)log2n || D.g != g || D.me != me)) return fail(B200G16_ERR_STATE, "dist_h: already set up for another shape; close first");
  const size_t M = (size_t)1 << (log2n - g);
  for (int v = 0; v < 3; v++) {
    B200_TRY(D.slice[v].ensure(M * sizeof(Fr)));
    D.peers[v][me] = D.slice[v].p;
  }
  D.g = g; D.me = me; D.L = (int)log2n;
  D.ready = false;
  return 0;
}

int b200g16_dist_h_init(b200g16_ctx* ctx, unsigned log2n, int n_peers, int me, uint8_t* handles_out) {
  if (!ctx || !handles_out) return fail(B200G16_ERR_ARG, "dist_h_init: null");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  B200_TRY(dist_h_alloc(ctx, log2n, n_peers, me));
  for (int v = 0; v < 3; v++) {
    cudaIpcMemHandle_t h;
    B200_CUDA(cudaIpcGetMemHandle(&h, ctx->dist_h.slice[v].p));
    memcpy(handles_out + 64 * v, &h, 64);
  }
  return 0;
}

int b200g16_dist_h_open(b200g16_ctx* ctx, const uint8_t* all_handles) {
  if (!ctx || !all_handles) return fail(B200G16_ERR_ARG, "dist_h_open: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  DistH& D = ctx->dist_h;
  if (!D.g) return fail(B200G16_ERR_STATE, "dist_h_open: call b200g16_dist_h_init first");
  const int G = 1 << D.g;
  for (int d = 0; d < G; d++) {
    if (d == D.me) continue;
    for (int v = 0; v < 3; v++) {
      if (D.ipc_opened[v][d]) continue;
      cudaIpcMemHandle_t h;
      memcpy(&h, all_handles + ((size_t)d * 3 + v) * 64, 64);
      void* p = nullptr;
      B200_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      D.peers[v][d] = p;
      D.ipc_opened[v][d] = true;
    }
  }
  D.ready = true;
  return 0;
}

void* b200g16_dist_h_slice(b200g16_ctx* ctx, int which) {
  if (!ctx || which < 0 || which > 2 || !ctx->dist_h.g) return nullptr;
  return ctx->dist_h.slice[which].p;
}

int b200g16_dist_h_load(b200g16_ctx* ctx, const void* d_a, const void* d_b, const void* d_c) {
  if (!ctx || !d_a || !d_b || !d_c) return fail(B200G16_ERR_ARG, "dist_h_load: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  DistH& D = ctx->dist_h;
  if (!D.g) return fail(B200G16_ERR_STATE, "dist_h_load: call b200g16_dist_h_init first");
  const size_t bytes = (((size_t)1 << D.L) >> D.g) * sizeof(Fr);
  const void* src[3] = {d_a, d_b, d_c};
  for (int v = 0; v < 3; v++)
    B200_CUDA(cudaMemcpyAsync(D.slice[v].p, src[v], bytes, cudaMemcpyDeviceToDevice, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b200g16_dist_h_phase(b200g16_ctx* ctx, int phase) {
  if (!ctx) return fail(B200G16_ERR_ARG, "dist_h_phase: null");
  std::lock_guard<std::mutex> lock(ctx->mu);
  B200_CUDA(cudaSetDevice(ctx->device));
  DistH& D = ctx->dist_h;
  if (!D.ready) return fail(B200G16_ERR_STATE, "dist_h_phase: peers not opened");
  B200_TRY(compute_h_dist_phase(ctx, reinterpret_cast<Fr* const (*)[8]>(D.peers), D.g, D.me, D.L, phase));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

void b200g16_dist_h_close(b200g16_ctx* ctx) {
  if (!ctx) return;
  std::lock_guard<std::mutex> lock(ctx->mu);
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DistH& D = ctx->dist_h;
  for (int v = 0; v < 3; v++)
    for (int d = 0; d < 8; d++) {
      if (D.ipc_opened[v][d]) cudaIpcCloseMemHandle(D.peers[v][d]);
      D.ipc_opened[v][d] = false;
      D.peers[v][d] = nullptr;
    }
  for (int v = 0; v < 3; v++) D.slice[v].release();
  D.g = 0;
  D.ready = false;
}

}  // extern "C"
