// Library context, error plumbing and device workspace shared by every .cu of libb200g16.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200g16.h"

namespace b200 {

// thread-local last error (SURVEY §8b: errors cross the C-ABI as int + string)
inline char* last_error_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

#define B200_CUDA(expr)                                                                     \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return ::b200::fail(B200G16_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,    \
                          cudaGetErrorString(_e));                                          \
  } while (0)

#define B200_TRY(expr)          \
  do {                          \
    int _s = (expr);            \
    if (_s != 0) return _s;     \
  } while (0)

// grow-only device buffer
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) B200_CUDA(cudaFree(p));
    p = nullptr;
    cap = 0;
    size_t want = bytes + (bytes >> 3) + 256;
    B200_CUDA(cudaMalloc(&p, want));
    cap = want;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr int MSM_SETS = 3;  // rotating buffer sets: an MSM only waits for the tail of the MSM three calls back

constexpr int AFF_WS_LEVELS = 4;  // = AFF_LEVELS_MAX of msm_affine.cuh (checked where both are visible)

struct MsmWorkspace {
  // everything the "tail" of an MSM reads (merge of split buckets + bucket reduction) exists MSM_SETS times: the
  // tail runs on a second stream while the next MSMs' sort + accumulate ("front") fill the other sets
  // part: the (bucket, entry) pairs in coarse-bin order, bins: bin counters and tiles (msm_sort.cuh)
  DevBuf scalars, part, bins, entries, counts[MSM_SETS], partials[MSM_SETS], chunks[MSM_SETS], misc[MSM_SETS], tasks[MSM_SETS];
  // batched-affine accumulation: level buffers of the pair tree (aff_lvl[l - 1] = inputs of level l), one spill slot per
  // thread.  One set: accumulate kernels of consecutive MSMs are serialised on the main stream.
  DevBuf aff_lvl[AFF_WS_LEVELS], aff_desc, aff_spill, aff_spill_task;
  void* pinned = nullptr;  // small host staging for window sums
  size_t pinned_cap = 0;
  // window sums of batch MSMs (k vectors: k * Wr items per slot), MSM_SLOTS slots of batch_slot bytes.  Its own buffer:
  // `pinned` is never reallocated while an asynchronous ticket (slots 5..7) may still be landing in it.
  void* batch_pinned = nullptr;
  size_t batch_slot = 0;
};

struct NttWorkspace {
  DevBuf a, b, c, tw, coset, fused, dist;
  int tw_log = -1;     // twiddle table covers 2^tw_log
  int coset_log = -1;  // coset tables built for exactly 2^coset_log
  int fused_log = -1;  // computeH's fused scaling tables (g^i / N with and without 1 / (g^N - 1))
  int dist_log = -1, dist_g = 0, dist_me = -1;  // compact scaling tables of the multi-GPU computeH (this device's slice)
};

// descriptor of a window table attached to a bases vector (b200g16_bases_precompute)
struct MsmTable {
  int c, W;
  uint32_t stride;  // points per row (= length of the bases vector)
  uint32_t off;     // first point of the sub-range this MSM uses
};

struct MsmCfg {
  int c;          // window bits
  int W;          // windows
  uint32_t nbw;   // buckets per window = 2^(c-1)
  uint32_t nb;    // buckets in total: k * (W * nbw, or nbw when the bases carry a window table)
  int Wr;         // window sums per vector produced by the reduction: W, or 1 with a window table
  uint32_t bstride;     // bucket-index stride between windows: nbw, or 0 with a window table
  uint32_t ent_stride;  // entry = w * ent_stride + ent_off + i  (index into the bases / the table)
  uint32_t ent_off;
  uint32_t target_tasks;  // accumulate tasks wanted even for skewed inputs (device picks the task size)
  uint32_t ch;    // buckets per reduce chunk
  uint32_t nch;   // chunks per window
  uint32_t k;     // scalar vectors (1: one MSM); vector j's buckets are [j * nb / k, (j + 1) * nb / k)
};

// The sorted state (entries, counts, offsets, tasks) the last MSM left behind.  A following MSM over
// the SAME scalar vector and the same decomposition — groth16's Bs1 (G1) right after Bs2 (G2), both over
// wireValuesB — skips its sort phase and accumulates over these lists with its own bases.
struct MsmSorted {
  const void* scalars = nullptr;
  size_t n = 0, k = 0, ld = 0;
  int c = 0;
  uint32_t bstride = 0, ent_stride = 0, ent_off = 0;
  int par = 0;
  bool valid = false;
};

// computeH split over 2 / 4 / 8 devices: this device's slices of a, b, c (their own allocations: exported to the other
// processes / devices and never reallocated while open) and the peers' slices as seen from this device
struct DistH {
  int g = 0, me = 0, L = 0;
  DevBuf slice[3];
  void* peers[3][8] = {};    // peers[v][d]; peers[v][me] == slice[v].p
  bool ipc_opened[3][8] = {};
  bool ready = false;        // every peer pointer set
};

// pinned bounce buffers + per-worker streams of h2d_copy (host_copy.cuh): large pageable host buffers -> device
constexpr int H2D_MAX_WORKERS = 8;
struct H2DStager {
  void* pinned = nullptr;            // workers x 2 slots
  int workers = 0;
  cudaStream_t stream[H2D_MAX_WORKERS] = {};
  cudaEvent_t done[H2D_MAX_WORKERS] = {}, slot_free[H2D_MAX_WORKERS][2] = {}, start = nullptr;
};

struct Timings {
  // last-call device timings in ms (CUDA events on ctx stream); index = phase
  float ms[16];
  int n;
};

}  // namespace b200

struct b200g16_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t tail_stream = nullptr;   // bucket reductions (latency-bound, few threads) overlap the next MSM
  cudaStream_t copy_stream = nullptr;   // H2D of host scalars, pipelined against the MSM of the previous piece
  cudaEvent_t ev_copy[8] = {};
  cudaEvent_t ev_front[b200::MSM_SETS] = {}, ev_tail[b200::MSM_SETS] = {};
  cudaEvent_t ev_slot[8] = {};      // ev_slot[s]: the window sums of the MSM enqueued into result slot s have reached pinned memory
  bool tail_pending[b200::MSM_SETS] = {};
  int msm_parity = 0;               // next rotating buffer set (0 .. MSM_SETS-1)
  b200::MsmSorted last_sort;
  // a prove between its two halves (b200g16_prove_begin_dev / _end_dev): decompositions of the five MSMs
  b200::MsmCfg prove_cfg[5] = {};
  // b200g16_msm_g1_begin*/_end: result slots 5..7 (a prove owns 0..4), one cfg and one scalar buffer per ticket
  b200::MsmCfg async_cfg[3] = {};
  bool async_open[3] = {};
  b200::DevBuf async_scalars[3];
  const struct b200g16_pk* prove_pk = nullptr;
  bool prove_active = false;
  int sort_reader[b200::MSM_SETS] = {-1, -1, -1};  // sort_reader[p] = set of an MSM whose tail still reads sorted set p (shared)
  cudaEvent_t ev[18] = {};
  std::mutex mu;  // one call at a time per ctx (gnark calls MSMs from several goroutines)
  b200::MsmWorkspace msm;
  b200::NttWorkspace ntt;
  b200::DistH dist_h;
  b200::DevBuf io_a, io_b, io_c;  // staging for host-pointer entry points
  b200::H2DStager stager;
  b200::Timings timings = {};
  int msm_window_override = 0;  // 0 = auto
  int msm_affine_mode = 0;      // batched-affine accumulation: 0 = never, 1 = by size, 2 = always
  int msm_affine_levels = 3;    // pair-tree levels at most (1 .. 4)
  uint32_t msm_affine_min_pairs = 192;  // additions per inversion below which a level is not worth running
  uint64_t launches = 0;        // kernels launched by this ctx (bench's gpu_launches)
  bool sort_smem_set = false;   // k_sort_coarse_part's dynamic shared-memory limit raised on this device
};

namespace b200 {
// ctx->timings from the events ctx->ev[0 .. ev) a call recorded, all complete: interval i = ev[i] -> ev[i + 1].
// add: sum onto the intervals already there (the sub-batches of one call).
inline void events_to_timings(b200g16_ctx* ctx, int ev, bool add = false) {
  for (int i = 0; i + 1 < ev; i++) {
    float t = 0;
    cudaEventElapsedTime(&t, ctx->ev[i], ctx->ev[i + 1]);
    ctx->timings.ms[i] = add ? ctx->timings.ms[i] + t : t;
  }
  ctx->timings.n = ev - 1;
}
}  // namespace b200

struct b200g16_bases {
  int group = 1;  // 1 = G1, 2 = G2
  size_t n = 0;
  void* d_points = nullptr;  // n points; after b200g16_bases_precompute: tab_W rows of n points,
                             // row k = 2^(tab_c * k) * P_i
  int device = 0;
  int tab_c = 0;             // 0 = no window table
  int tab_W = 0;
};
