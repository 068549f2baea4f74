// Group-independent front half of the MSM: scalar recoding and the two-level counting sort (msm_sort.cuh), task table.
// See msm_impl.cuh for the pipeline overview.
#include <cstdlib>
#include "msm_impl.cuh"

namespace b200 {


// r - 1 as 4 x u64 (for the top-window overflow check)
static const uint64_t kRm1[4] = {0x43e1f593f0000000ull, 0x2833e84879b97091ull, 0xb85045b68181585dull,
                                 0x30644e72e131a029ull};

static uint64_t shr256(const uint64_t v[4], int s) {  // low 64 bits of v >> s
  if (s >= 256) return 0;
  int q = s >> 6, r = s & 63;
  uint64_t lo = v[q] >> r;
  if (r && q + 1 < 4) lo |= v[q + 1] << (64 - r);
  return lo;
}

int msm_num_windows(int c) {
  int W = (254 + c - 1) / c;
  // the top window must absorb the carry of the signed recoding without overflowing
  uint64_t top = shr256(kRm1, (W - 1) * c) + 1;
  if (top >= (1ull << (c - 1))) W += 1;
  return W;
}

int msm_pick_window(size_t n) {
  // minimise W(c) * (n + k * 2^(c-1)): k models the running-sum cost of the bucket reduction
  // relative to one mixed add in a full-occupancy accumulate.  k = 8 and c <= 17 reproduce the
  // measured optimum on B200 (profiles/r01_probe4_window_sweep.log: c = 15 @2^20, 17 @2^22..2^24;
  // c = 18..20 lose more in the reduction than they save in the accumulation).
  int best = 4;
  double best_cost = 1e300;
  for (int c = 4; c <= 17; c++) {
    double cost = (double)msm_num_windows(c) * ((double)n + 8.0 * (double)(1u << (c - 1)));
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

int msm_pick_table_window(size_t n) {
  // Measured on B200 (1000 W, 1965 MHz) with the tree reduction and the two-level sort
  // (profiles/r03a_window_sweep.jsonl: whole-MSM device time, uniform scalars): 2^20: c = 20 (2.81 ms against 2.95 at 19
  // and 3.15 at 21);  2^22: 20 (9.36 / 9.60 at 21);  2^24: 22 (33.17 against 35.68 at 20 and 35.35 at 21: 2.4 ms fewer
  // additions, 0.7 ms more reduction; the sort costs the same at both widths).  Older figures with the one-atomic-per-entry
  // scatter (profiles/r02f_window_sweep.jsonl): 2^18: c = 17 (1.35 ms);  2^19: c = 19 / 20 tie (2.14);  2^21: 20 (5.41 /
  // 6.17).  Widths whose TOP window holds only a few scalar bits (c = 18, 19, 21: 2 / 7 / 2 bits) pile every point's top
  // digit into a handful of low buckets of the shared bucket set and pay for it in the merge of their split buckets
  // (0.2 - 0.4 ms against 0.05) — c = 22 (12 top bits), 20 (14) and 17 (16) do not.
  auto fits = [&](int c) { return (double)n * msm_num_windows(c) < 2.0e9; };
  if (n >= ((size_t)1 << 24) && fits(22)) return 22;
  if (n >= ((size_t)3 << 17) && fits(20)) return 20;
  int best = 8;
  double best_cost = 1e300;
  for (int c = 8; c <= 17; c++) {
    const int W = msm_num_windows(c);
    if (!fits(c)) continue;
    double cost = (double)W * (double)n + 4.0 * (double)(1u << (c - 1));
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

// ------------------------------------------------------------------------------ kernels
// The two-level counting sort (msm_sort.cuh): each kernel runs the header's steps thread by thread between barriers.

// Passes 1 and 3 come in two instances: BATCH = false (one scalar vector) and true (k vectors, msm_sort.cuh).
// pass 1: coarse count.  s[SORT_BINS] counts the CTA's entries (-> totals[3], which drives the task size)
template <bool BATCH>
__global__ void __launch_bounds__(SORT_CTA) k_sort_coarse_count(const SortArgs A) {
  __shared__ uint32_t s[SORT_BINS + 1];
  sort_coarse_init(A, threadIdx.x, s);
  __syncthreads();
  sort_coarse_count<BATCH>(A, blockIdx.x, threadIdx.x, s);
  __syncthreads();
  sort_coarse_flush(A, threadIdx.x, s);
}

// in-place exclusive scan of s[0, N) by SORT_CTA threads (N / SORT_CTA words each); the total goes to s[N]
template <uint32_t N>
__device__ void sort_block_scan(uint32_t* s) {
  constexpr uint32_t PER = N / SORT_CTA;
  __shared__ uint32_t wsum[SORT_CTA / 32];
  const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
  uint32_t a = 0;
#pragma unroll
  for (uint32_t j = 0; j < PER; j++) a += s[t * PER + j];
  uint32_t ia = a;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t x = __shfl_up_sync(0xffffffffu, ia, off);
    if (lane >= (uint32_t)off) ia += x;
  }
  if (lane == 31) wsum[warp] = ia;
  __syncthreads();
  uint32_t e = ia - a;
  for (uint32_t w = 0; w < warp; w++) e += wsum[w];
#pragma unroll
  for (uint32_t j = 0; j < PER; j++) {
    const uint32_t k = t * PER + j, v = s[k];
    s[k] = e;
    e += v;
  }
  if (t == SORT_CTA - 1) s[N] = e;
  __syncthreads();
}

// pass 2, one CTA: exclusive scans of the bins' entries and tiles, then bin offsets and the tile list
__global__ void __launch_bounds__(SORT_CTA) k_sort_bins(const SortArgs A) {
  __shared__ uint32_t sa[SORT_BINS + 1], sb[SORT_BINS + 1];
  sort_bins_load(A, threadIdx.x, sa, sb);
  __syncthreads();
  sort_block_scan<SORT_BINS>(sa);
  sort_block_scan<SORT_BINS>(sb);
  sort_bins_write(A, threadIdx.x, sa, sb);
}

// pass 3: coarse partition into part[] (bin order), staged in dynamic shared memory (sort_part_smem bytes)
template <bool BATCH>
__global__ void __launch_bounds__(SORT_CTA) k_sort_coarse_part(const SortArgs A) {
  extern __shared__ __align__(8) unsigned char sort_smem[];
  SortItem* stage = reinterpret_cast<SortItem*>(sort_smem);
  uint32_t* s = reinterpret_cast<uint32_t*>(stage + SORT_STAGE);
  uint32_t* loc = s + SORT_BINS + 1;
  uint32_t* glob = loc + SORT_BINS;
  for (uint32_t b = threadIdx.x; b < SORT_BINS; b += SORT_CTA) s[b] = 0;
  __syncthreads();
  sort_part_count<BATCH>(A, blockIdx.x, threadIdx.x, s);
  __syncthreads();
  sort_block_scan<SORT_BINS>(s);
  sort_part_reserve(A, threadIdx.x, s, loc, glob);
  __syncthreads();
  sort_part_stage<BATCH>(A, blockIdx.x, threadIdx.x, s, stage);
  __syncthreads();
  sort_part_write(A, threadIdx.x, s[SORT_BINS], loc, glob, stage);
}

// pass 4: fine count, one CTA per tile (the grid is an upper bound on the tiles)
__global__ void __launch_bounds__(SORT_CTA) k_sort_fine_count(const SortArgs A) {
  __shared__ uint32_t s[1u << SORT_FINE_MAX_BITS];
  if (blockIdx.x >= *A.ntiles) return;   // whole CTA past the last tile
  const SortSpan sp = sort_tile_span(A, blockIdx.x);
  sort_fine_init(A, threadIdx.x, s);
  __syncthreads();
  sort_fine_count(A, sp, threadIdx.x, s, true);
  __syncthreads();
  sort_fine_flush(A, sp, threadIdx.x, s);
}

// pass 6: fine place into entries[] (bucket order)
__global__ void __launch_bounds__(SORT_CTA) k_sort_fine_place(const SortArgs A) {
  __shared__ uint32_t s[1u << SORT_FINE_MAX_BITS];
  if (blockIdx.x >= *A.ntiles) return;
  const SortSpan sp = sort_tile_span(A, blockIdx.x);
  sort_fine_init(A, threadIdx.x, s);
  __syncthreads();
  sort_fine_count(A, sp, threadIdx.x, s, false);
  __syncthreads();
  sort_fine_reserve(A, sp, threadIdx.x, s);
  __syncthreads();
  sort_fine_place(A, sp, threadIdx.x, s);
}

// task size.  Many buckets (nb >= target / 2): evenly loaded buckets stay one task each (seg = 2 x mean),
// and a skewed input (few huge buckets) still yields >= target tasks.  Few buckets (window tables with
// a narrow window, small windows): the buckets are cut so that ~target tasks exist at all — otherwise
// the accumulate kernel would run with a fraction of the SMs' threads.  totals[4] = seg.
__global__ void k_pick_seg(uint32_t* __restrict__ totals, uint32_t nb, uint32_t target) {
  uint32_t total = totals[3];
  uint32_t a = 2u * (total / nb) + 2u, b = total / target + 1u;
  uint32_t seg = (nb >= target / 2 && a > b) ? a : b;
  totals[4] = seg < 32u ? 32u : seg;
}

// ---- exclusive scan of (count, #tasks) per bucket: tile sums -> scan of tile sums -> apply
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_sums(const uint32_t* __restrict__ counts, uint32_t nb,
                                                             const uint32_t* __restrict__ totals,
                                                             uint2* __restrict__ tile_sums) {
  __shared__ uint32_t wa[SCAN_THREADS / 32], wb[SCAN_THREADS / 32];
  const uint32_t seg = totals[4];
  uint32_t base = blockIdx.x * SCAN_TILE, a = 0, b = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; j++) {
    uint32_t i = base + threadIdx.x + SCAN_THREADS * j;
    if (i < nb) { uint32_t cnt = counts[i]; a += cnt; b += (cnt + seg - 1) / seg; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    a += __shfl_down_sync(0xffffffffu, a, off);
    b += __shfl_down_sync(0xffffffffu, b, off);
  }
  if ((threadIdx.x & 31) == 0) { wa[threadIdx.x >> 5] = a; wb[threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t ta = 0, tb = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; w++) { ta += wa[w]; tb += wb[w]; }
    tile_sums[blockIdx.x] = make_uint2(ta, tb);
  }
}

// single CTA: in-place exclusive scan of the tile sums (chunks of 1024 with a running carry)
__global__ void __launch_bounds__(1024) k_scan_top(uint2* __restrict__ tile_sums, uint32_t ntiles,
                                                    uint32_t* __restrict__ totals) {
  __shared__ uint32_t s1[1024], s2[1024];
  uint32_t t = threadIdx.x, ca = 0, cb = 0;
  for (uint32_t base = 0; base < ntiles; base += 1024) {
    uint32_t i = base + t;
    uint2 v = i < ntiles ? tile_sums[i] : make_uint2(0, 0);
    s1[t] = v.x;
    s2[t] = v.y;
    __syncthreads();
    for (uint32_t off = 1; off < 1024; off <<= 1) {
      uint32_t x = 0, y = 0;
      if (t >= off) { x = s1[t - off]; y = s2[t - off]; }
      __syncthreads();
      s1[t] += x;
      s2[t] += y;
      __syncthreads();
    }
    if (i < ntiles) tile_sums[i] = make_uint2(ca + s1[t] - v.x, cb + s2[t] - v.y);
    ca += s1[1023];
    cb += s2[1023];
    __syncthreads();
  }
  if (t == 0) {
    totals[0] = ca;  // entries
    totals[1] = cb;  // tasks
    totals[2] = 0;   // split-bucket counters (k_tasks)
    totals[6] = 0;
  }
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(const uint32_t* __restrict__ counts, uint32_t nb,
                                                              const uint32_t* __restrict__ totals,
                                                              const uint2* __restrict__ tile_sums,
                                                              uint32_t* __restrict__ offsets,
                                                              uint32_t* __restrict__ cursor,
                                                              uint32_t* __restrict__ task_off) {
  __shared__ uint32_t wa[SCAN_THREADS / 32], wb[SCAN_THREADS / 32];
  const uint32_t seg = totals[4];
  const uint32_t first = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t cnt[SCAN_ITEMS], a = 0, b = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; j++) {
    cnt[j] = first + j < nb ? counts[first + j] : 0;
    a += cnt[j];
    b += (cnt[j] + seg - 1) / seg;
  }
  // inclusive scan of the per-thread sums across the CTA
  uint32_t ia = a, ib = b;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    uint32_t x = __shfl_up_sync(0xffffffffu, ia, off), y = __shfl_up_sync(0xffffffffu, ib, off);
    if (lane >= (uint32_t)off) { ia += x; ib += y; }
  }
  if (lane == 31) { wa[warp] = ia; wb[warp] = ib; }
  __syncthreads();
  uint32_t pa = 0, pb = 0;
  for (uint32_t w = 0; w < warp; w++) { pa += wa[w]; pb += wb[w]; }
  const uint2 tile = tile_sums[blockIdx.x];
  uint32_t ea = tile.x + pa + ia - a, eb = tile.y + pb + ib - b;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; j++) {
    if (first + j < nb) {
      offsets[first + j] = ea;
      cursor[first + j] = ea;
      task_off[first + j] = eb;
    }
    ea += cnt[j];
    eb += (cnt[j] + seg - 1) / seg;
  }
}

__global__ void __launch_bounds__(256) k_tasks(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ task_off,
                                                uint32_t nb, uint32_t* __restrict__ totals,
                                                uint32_t* __restrict__ task_bucket) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const uint32_t seg = totals[4];
  uint32_t nt = (counts[b] + seg - 1) / seg;
  uint32_t o = task_off[b];
  for (uint32_t t = 0; t < nt; t++) task_bucket[o + t] = b;
  if (nt > 1) atomicMax(&totals[5], nt);  // deepest merge tree needed (k_merge_pass)
  // more than one first-level sum after k_merge_pass: up to MERGE_FANIN of them are summed by one thread
  // (k_merge_mid, list at totals + 16), more by one CTA (k_merge_heavy, list at totals + 16 + nb)
  if (nt > 16) totals[16 + nb + atomicAdd(&totals[6], 1u)] = b;
  else if (nt > 4) totals[16 + atomicAdd(&totals[2], 1u)] = b;
}


// ---- order tasks by length, longest first, so the 32 lanes of a warp run equal trip counts in
// k_accumulate (bucket loads are Poisson distributed: without this the warp waits for its longest lane)
constexpr uint32_t TASK_BINS = 4096;

__device__ __forceinline__ uint32_t task_len(uint32_t cnt, uint32_t j, uint32_t seg) {
  uint32_t rem = cnt - j * seg;
  return rem < seg ? rem : seg;
}

// Task lengths cluster on a few values (evenly loaded buckets: ~30 distinct lengths; a 0/1-heavy witness: most tasks are
// exactly `seg` long), so one global atomic per task serialises on a handful of addresses (2^19 tasks: 119 us for the
// histogram and 121 us for the ordering, profiles/r02j_ncu_launches_bench_2p24.csv).  Both kernels therefore count
// inside the CTA first (shared-memory histogram, the atomic's return value is the task's rank within the CTA) and touch
// global memory once per CTA and occupied bin.
constexpr int TASK_CTA = 1024;

__global__ void __launch_bounds__(TASK_CTA) k_task_hist(const uint32_t* __restrict__ task_bucket,
                                                         const uint32_t* __restrict__ counts,
                                                         const uint32_t* __restrict__ task_off,
                                                         const uint32_t* __restrict__ totals, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[TASK_BINS];
  if (blockIdx.x * TASK_CTA >= totals[1]) return;   // whole CTA past the last task
  for (uint32_t b = threadIdx.x; b < TASK_BINS; b += TASK_CTA) h[b] = 0;
  __syncthreads();
  const uint32_t t = blockIdx.x * TASK_CTA + threadIdx.x;
  if (t < totals[1]) {
    const uint32_t b = task_bucket[t];
    const uint32_t len = task_len(counts[b], t - task_off[b], totals[4]);
    atomicAdd(&h[len < TASK_BINS ? len : TASK_BINS - 1], 1u);
  }
  __syncthreads();
  for (uint32_t b = threadIdx.x; b < TASK_BINS; b += TASK_CTA)
    if (h[b]) atomicAdd(&hist[b], h[b]);
}

// single CTA, 1024 threads x 4 bins: exclusive scan in DESCENDING length order -> cursor[bin]
__global__ void __launch_bounds__(1024) k_task_scan(const uint32_t* __restrict__ hist, uint32_t* __restrict__ cursor) {
  __shared__ uint32_t s[1024];
  uint32_t t = threadIdx.x, v[4], a = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) { v[k] = hist[TASK_BINS - 1 - (4 * t + k)]; a += v[k]; }
  s[t] = a;
  __syncthreads();
  for (uint32_t off = 1; off < 1024; off <<= 1) {
    uint32_t x = t >= off ? s[t - off] : 0;
    __syncthreads();
    s[t] += x;
    __syncthreads();
  }
  uint32_t e = s[t] - a;
#pragma unroll
  for (int k = 0; k < 4; k++) { cursor[TASK_BINS - 1 - (4 * t + k)] = e; e += v[k]; }
}

__global__ void __launch_bounds__(TASK_CTA) k_task_order(const uint32_t* __restrict__ task_bucket,
                                                          const uint32_t* __restrict__ counts,
                                                          const uint32_t* __restrict__ task_off,
                                                          const uint32_t* __restrict__ totals, uint32_t* __restrict__ cursor,
                                                          uint32_t* __restrict__ task_order) {
  __shared__ uint32_t h[TASK_BINS];   // per bin: this CTA's count, then the base of its range in task_order
  if (blockIdx.x * TASK_CTA >= totals[1]) return;
  for (uint32_t b = threadIdx.x; b < TASK_BINS; b += TASK_CTA) h[b] = 0;
  __syncthreads();
  const uint32_t t = blockIdx.x * TASK_CTA + threadIdx.x;
  uint32_t bin = 0, rank = 0;
  const bool valid = t < totals[1];
  if (valid) {
    const uint32_t b = task_bucket[t];
    const uint32_t len = task_len(counts[b], t - task_off[b], totals[4]);
    bin = len < TASK_BINS ? len : TASK_BINS - 1;
    rank = atomicAdd(&h[bin], 1u);
  }
  __syncthreads();
  for (uint32_t b = threadIdx.x; b < TASK_BINS; b += TASK_CTA)
    if (h[b]) h[b] = atomicAdd(&cursor[b], h[b]);
  __syncthreads();
  if (valid) task_order[h[bin] + rank] = t;
}

int msm_sort_phase(b200g16_ctx* ctx, const MsmCfg& cfg, const Fr* d_scalars, uint32_t n, uint32_t ld, SortItem* part,
                   uint32_t* bins, uint32_t* counts, uint32_t* offsets, uint32_t* cursor, uint32_t* task_off,
                   uint32_t* totals, uint32_t* entries, uint32_t* task_bucket, uint32_t* task_order, uint32_t max_tasks,
                   uint32_t* scan_scratch, int* ev) {
  const bool batch = cfg.k > 1;
  cudaStream_t st = ctx->stream;
  auto mark = [&]() { if (ev && *ev < 18) cudaEventRecord(ctx->ev[(*ev)++], st); };
  // B200G16_SORT_TRACE=1: an event after every operation of this phase, printed (and the stream drained) at its end —
  // where the phase's time goes inside a real call, launch gaps included (tools/sweep.py --reduce-ab).  One set of
  // events per process: a single-device debugging aid, not for b200g16_group_* runs.
  static const bool trace = getenv("B200G16_SORT_TRACE") != nullptr;
  static cudaEvent_t tev[16];
  static bool tev_made = false;
  int nt = 0;
  if (trace && !tev_made) { for (auto& e : tev) cudaEventCreate(&e); tev_made = true; }
  auto tr = [&]() { if (trace && nt < 16) cudaEventRecord(tev[nt++], st); };
  SortArgs A;
  A.scalars = d_scalars;
  A.n = n * cfg.k;   // points of all vectors (msm_enqueue keeps n * k * W below 2^32)
  A.vn = batch ? n : 0u;
  A.ld = ld;
  A.vstride = cfg.nb / cfg.k;
  A.c = cfg.c;
  A.W = cfg.W;
  A.bstride = cfg.bstride;
  A.ent_stride = cfg.ent_stride;
  A.ent_off = cfg.ent_off;
  A.F = sort_fine_bits(cfg.nb);
  A.nbins = sort_num_bins(cfg.nb, A.F);
  A.part_points = sort_part_points(cfg.W);
  A.bin_count = bins;
  A.bin_cursor = bins + SORT_BINS;
  A.bin_off = bins + 2 * SORT_BINS;
  A.ntiles = bins + 3 * SORT_BINS + 1;
  A.tiles = reinterpret_cast<SortTile*>(bins + SORT_BIN_WORDS);
  A.part = part;
  // canonical scalars between passes 1 and 3: entries (4 W bytes per point, W >= 11 at every width) is not written
  // before pass 6
  static_assert(sizeof(Fr) == 32, "canonical scalar scratch: 32 bytes per point");
  if (cfg.W < 8) return fail(B200G16_ERR_ARG, "msm sort: W = %d leaves no room for the canonical scalars", cfg.W);
  A.canon = reinterpret_cast<Fr*>(entries);
  A.counts = counts;
  A.cursor = cursor;
  A.entries = entries;
  A.totals = totals;
  const unsigned max_tiles = (unsigned)sort_max_tiles(A.nbins, (size_t)A.n * cfg.W);
  mark();
  tr();
  B200_CUDA(cudaMemsetAsync(counts, 0, (size_t)cfg.nb * sizeof(uint32_t), st));
  B200_CUDA(cudaMemsetAsync(totals, 0, 16 * sizeof(uint32_t), st));
  B200_CUDA(cudaMemsetAsync(A.bin_count, 0, SORT_BINS * sizeof(uint32_t), st));
  if (batch) k_sort_coarse_count<true><<<cdiv(A.n, SORT_POINTS), SORT_CTA, 0, st>>>(A);
  else k_sort_coarse_count<false><<<cdiv(A.n, SORT_POINTS), SORT_CTA, 0, st>>>(A);
  tr();
  k_pick_seg<<<1, 1, 0, st>>>(totals, cfg.nb, cfg.target_tasks);
  tr();
  mark();
  k_sort_bins<<<1, SORT_CTA, 0, st>>>(A);
  tr();
  if (!ctx->sort_smem_set) {   // once per context (= device)
    B200_CUDA(cudaFuncSetAttribute(k_sort_coarse_part<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_part_smem()));
    B200_CUDA(cudaFuncSetAttribute(k_sort_coarse_part<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_part_smem()));
    ctx->sort_smem_set = true;
  }
  if (batch) k_sort_coarse_part<true><<<cdiv(A.n, A.part_points), SORT_CTA, sort_part_smem(), st>>>(A);
  else k_sort_coarse_part<false><<<cdiv(A.n, A.part_points), SORT_CTA, sort_part_smem(), st>>>(A);
  tr();
  k_sort_fine_count<<<max_tiles, SORT_CTA, 0, st>>>(A);
  tr();
  const uint32_t ntiles = cdiv(cfg.nb, SCAN_TILE);
  uint2* tile_sums = reinterpret_cast<uint2*>(scan_scratch);
  uint32_t* hist = scan_scratch + 2 * (size_t)(ntiles + 1);   // 2 x TASK_BINS words after the tile sums
  uint32_t* hist_cursor = hist + TASK_BINS;
  k_scan_sums<<<ntiles, SCAN_THREADS, 0, st>>>(counts, cfg.nb, totals, tile_sums);
  k_scan_top<<<1, 1024, 0, st>>>(tile_sums, ntiles, totals);
  k_scan_apply<<<ntiles, SCAN_THREADS, 0, st>>>(counts, cfg.nb, totals, tile_sums, offsets, cursor, task_off);
  tr();
  k_sort_fine_place<<<max_tiles, SORT_CTA, 0, st>>>(A);
  tr();
  k_tasks<<<cdiv(cfg.nb, 256), 256, 0, st>>>(counts, task_off, cfg.nb, totals, task_bucket);
  tr();
  B200_CUDA(cudaMemsetAsync(hist, 0, TASK_BINS * sizeof(uint32_t), st));
  k_task_hist<<<cdiv(max_tasks, TASK_CTA), TASK_CTA, 0, st>>>(task_bucket, counts, task_off, totals, hist);
  tr();
  k_task_scan<<<1, 1024, 0, st>>>(hist, hist_cursor);
  k_task_order<<<cdiv(max_tasks, TASK_CTA), TASK_CTA, 0, st>>>(task_bucket, counts, task_off, totals, hist_cursor, task_order);
  tr();
  mark();
  if (trace) {
    cudaStreamSynchronize(st);
    static const char* what[] = {"memsets + coarse count", "k_pick_seg", "bin scan", "coarse partition", "fine count",
                                 "scan x3", "fine place", "k_tasks", "memset + k_task_hist", "k_task_scan + k_task_order"};
    fprintf(stderr, "[sort trace n=%u c=%d F=%d]", A.n, cfg.c, A.F);
    for (int i = 0; i + 1 < nt; i++) {
      float ms = 0;
      cudaEventElapsedTime(&ms, tev[i], tev[i + 1]);
      fprintf(stderr, "  %s %.1f us", what[i], ms * 1e3f);
    }
    fprintf(stderr, "\n");
  }
  ctx->launches += 13;
  B200_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace b200
