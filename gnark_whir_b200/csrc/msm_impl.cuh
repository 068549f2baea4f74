// Pippenger multi-scalar multiplication over BN254 G1 / G2 for sm_100a.
//
// Replaces gnark-crypto ecc/bn254/multiexp.go (*G1Affine).MultiExp / (*G2Affine).MultiExp,
// which gnark's groth16 prover (backend/groth16/bn254/prove.go) calls for Ar, Bs1, Krs,
// Krs2 (the H/Z term), Bs2 and the BSB22 Pedersen commitment; reached from the reference at
// /root/reference/mt.go:496.  Only the result (the group element, in affine normal form) is
// observable at that boundary, so the decomposition below is B200-first, not gnark's:
//
//   k_sort_*      scalar Montgomery->canonical, signed c-bit digits (partitionScalars' job), and a two-level
//                 counting sort of the (window, point) entries into bucket order: coarse bins (bucket >> F), then
//                 the buckets inside each bin, one atomic per CTA and bin or bucket (msm_sort.cuh)
//   k_scan_*      exclusive scan of the histogram -> entry offsets; buckets larger than `seg`
//                 are split into several tasks (0/1-heavy witnesses put millions of points in
//                 bucket "1" of window 0) -> task offsets
//   k_tasks, k_task_*  task -> bucket table; tasks ordered by length so a warp's lanes finish together
//   k_accumulate  one thread per task: gathers its affine points with 128-bit loads, mixed
//                 XYZZ adds (10 modmul) on the integer pipe; next point prefetched during the add
//   ---- "tail", on a second stream under the next MSM's work above ----
//   k_merge_pass  fan-in-4 tree over the partials of split buckets
//   k_reduce_first / _level / _tail  log-depth tree for sum_b (b+1) B_b (bit decomposition of the
//                 weights: 2 additions per bucket in total, dependency depth c instead of a running-sum chain)
//   host          Horner over the window sums + one inversion -> affine
//
// With a window table over the bases (b200g16_bases_precompute: row k = 2^(ck) P_i) all digits address
// ONE bucket set, entries index the table, and the host has no Horner to do.  A following MSM over the
// same scalars and decomposition can reuse the sorted lists (share_sort: groth16's Bs1 after Bs2).
#pragma once
#include <cstdlib>

#include "common.cuh"
#include "ec.cuh"
#include "msm_sort.cuh"

namespace b200 {

// (struct MsmCfg lives in common.cuh)

// msm_common.cu
int msm_num_windows(int c);
int msm_pick_window(size_t n);
// two-level counting sort into bucket order + task table on ctx->stream (13 kernels + 4 memsets), for cfg.k vectors of
// n scalars, vector j at d_scalars + j * ld.  part: k * n * W items; bins: sort_bin_bytes(bins, k * n * W) bytes
int msm_sort_phase(b200g16_ctx* ctx, const MsmCfg& cfg, const Fr* d_scalars, uint32_t n, uint32_t ld, SortItem* part,
                   uint32_t* bins, uint32_t* counts, uint32_t* offsets, uint32_t* cursor, uint32_t* task_off,
                   uint32_t* totals, uint32_t* entries, uint32_t* task_bucket, uint32_t* task_order, uint32_t max_tasks,
                   uint32_t* scan_scratch, int* ev);

static inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// 128-bit read-only loads with a 64-byte L2 fetch granule: a G1 point is one 64 B granule, and its
// neighbours in the bases / table are never wanted (random gather), so the default 128 B promotion
// would double the DRAM traffic (ncu: 29 GB/launch at n = 2^24 against 14.8 GB of gathers).
__device__ __forceinline__ uint4 ldg_nc_64(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L2::64B.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

template <class F>
__device__ __forceinline__ Affine<F> load_affine(const Affine<F>* __restrict__ p) {
  constexpr int NV = sizeof(Affine<F>) / 16;
  Affine<F> r;
  const uint4* src = reinterpret_cast<const uint4*>(p);
  uint4* dst = reinterpret_cast<uint4*>(&r);
#pragma unroll
  for (int k = 0; k < NV; k++) dst[k] = ldg_nc_64(src + k);
  return r;
}

// G1: 128 registers -> 4 CTAs/SM.  G2 (Fp2 coordinates): 220 registers, 2 CTAs/SM (capping it at 168
// for 3 CTAs/SM spills and measures the same, profiles/r01 notes).
template <class F>
__global__ void __launch_bounds__(128, (sizeof(F) > 32) ? 2 : 4) k_accumulate(const Affine<F>* __restrict__ bases,
                                                     const uint32_t* __restrict__ entries,
                                                     const uint32_t* __restrict__ task_order,
                                                     const uint32_t* __restrict__ task_bucket,
                                                     const uint32_t* __restrict__ offsets,
                                                     const uint32_t* __restrict__ counts,
                                                     const uint32_t* __restrict__ task_off,
                                                     const uint32_t* __restrict__ totals,
                                                     XYZZ<F>* __restrict__ partials) {
  const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= totals[1]) return;
  const uint32_t t = task_order[gid];  // tasks sorted by length: the lanes of a warp finish together
  const uint32_t seg = totals[4];
  uint32_t b = task_bucket[t];
  uint32_t start = offsets[b] + (t - task_off[b]) * seg;
  uint32_t bend = offsets[b] + counts[b];
  uint32_t end = start + seg < bend ? start + seg : bend;
  XYZZ<F> acc = XYZZ<F>::inf();
  uint32_t e = entries[start];
  Affine<F> p = load_affine(bases + (e >> 1));
  for (uint32_t i = start; i < end; i++) {
    Affine<F> cur = p;
    uint32_t ce = e;
    if (i + 1 < end) {
      e = entries[i + 1];
      p = load_affine(bases + (e >> 1));
    }
    if (ce & 1) cur.y = F::neg(cur.y);
    acc.madd(cur);
  }
  partials[t] = acc;
}

// Merge the partials of buckets that were split into several tasks: a fan-in-4 tree over the
// (contiguous) partials of each bucket, one launch per level (stride = 4^level: 3 dependent additions
// per level, a quarter of the lanes busy).  Thread t owns task
// t; at a level only local indices that are multiples of 4*stride do work, reading slots no other
// thread writes in the same launch.  After the last level the bucket's sum sits in its first partial.
// totals[5] = largest #tasks of any bucket (written by k_tasks), so idle levels exit immediately.
constexpr uint32_t MERGE_FANIN = 4;

template <class F>
__global__ void __launch_bounds__(128) k_merge_pass(XYZZ<F>* __restrict__ partials,
                                                     const uint32_t* __restrict__ task_bucket,
                                                     const uint32_t* __restrict__ counts,
                                                     const uint32_t* __restrict__ task_off,
                                                     const uint32_t* __restrict__ totals, uint32_t stride) {
  if (stride >= totals[5]) return;
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= totals[1]) return;
  const uint32_t seg = totals[4];
  uint32_t b = task_bucket[t];
  uint32_t nt = (counts[b] + seg - 1) / seg;
  uint32_t j = t - task_off[b];
  if (stride >= nt || (j % (MERGE_FANIN * stride)) != 0) return;
  XYZZ<F> acc = partials[t];
  for (uint32_t q = 1; q < MERGE_FANIN; q++) {
    uint32_t idx = j + q * stride;
    if (idx >= nt) break;
    acc.add(partials[t + q * stride]);
  }
  partials[t] = acc;
}

// ---- bucket reduction  S_w = sum_b (b + 1) B_b  as a log-depth tree (no running sums, no serial chains).
// With n = log2(#buckets):  S = G + sum_m 2^m U_m,  G = sum_b B_b,  U_m = sum of the buckets whose index has bit m
// set.  All n + 1 sums come out of ONE in-place halving schedule over a dense array A of the bucket values:
// level l (1..n) folds the main region A[0, 2^(n-l+1)) onto its lower half — the intact upper half is exactly the
// set "bit n-l set" of the folded index and becomes region j = l at offset 2^(n-l) — and halves every older
// region in place.  Before level l all l regions have 2^(n-l+1) items, so a level is l * 2^(n-l) independent
// additions, 2 * 2^n in total (the running sum's count), and the dependency depth is n additions instead of
// ~2 * chunk + 1.5 c.  Afterwards A[0] = G and A[2^m] = U_m; the tail kernel (k_reduce_tail) scales them by 2^m
// (m doublings, one thread each) and adds the n + 1 terms by a halving tree.
//
// INL: the addition is expanded in place with both operands in registers (like k_accumulate's mixed addition: no stack
// copy of the accumulator, every load issued up front) instead of the out-of-line routine.  G1 only — two Fp2 points
// (128 registers) plus the addition's temporaries do not fit a thread.  Experiment knob: B200G16_REDUCE_INLINE (read once).
inline int reduce_inline_default() {   // 0: out of line, 1: the grid-wide levels, 2: also the one-CTA tail
  static const int v = [] { const char* e = getenv("B200G16_REDUCE_INLINE"); return e ? atoi(e) : 2; }();
  return v;
}

template <class F, bool INL>
__global__ void __launch_bounds__(128, INL ? 4 : 0) k_reduce_first(const XYZZ<F>* __restrict__ partials,
                                                       const uint32_t* __restrict__ counts,
                                                       const uint32_t* __restrict__ task_off, uint32_t Wr, uint32_t nbw,
                                                       XYZZ<F>* __restrict__ A) {
  const uint32_t half = nbw >> 1;
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= Wr * half) return;
  const uint32_t w = g / half, i = g % half;
  const uint32_t first = w * nbw;  // bucket b's value = first partial of the bucket (after k_merge_pass)
  XYZZ<F> lo = counts[first + i] ? partials[task_off[first + i]] : XYZZ<F>::inf();
  const XYZZ<F> hi = counts[first + i + half] ? partials[task_off[first + i + half]] : XYZZ<F>::inf();
  A[first + i + half] = hi;
  if constexpr (INL) lo.add_inline(hi);
  else lo.add(hi);
  A[first + i] = lo;
}

template <class F, bool INL>
__global__ void __launch_bounds__(128, INL ? 4 : 0) k_reduce_level(XYZZ<F>* __restrict__ A, uint32_t Wr, uint32_t nbw, uint32_t l) {
  const uint32_t s = nbw >> l, per_w = l * s;
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= Wr * per_w) return;
  const uint32_t w = g / per_w, r = g % per_w, j = r / s, i = r % s;
  XYZZ<F>* p = A + (size_t)w * nbw + (j ? (nbw >> j) : 0u) + i;
  XYZZ<F> a = p[0];
  if constexpr (INL) {
    const XYZZ<F> b = p[s];
    a.add_inline(b);
  } else {
    a.add(p[s]);
  }
  p[0] = a;
}

// The END of the tree in one CTA per window: once a level fits 512 threads (l * 2^(n-l) <= 512) the remaining
// levels, the 2^m weights and the final sum of the n + 1 terms run back to back inside one kernel, separated by
// __syncthreads instead of launches (12 launches of ~12 us each for one dependent addition, the weights and three
// sum passes before: profiles/r02f_ncu_launches_bench_2p24.csv).
constexpr uint32_t REDUCE_TAIL_THREADS = 512;   // <= 128 registers per thread: the XYZZ addition keeps ~95 live

template <class F, bool INL>
__global__ void __launch_bounds__(REDUCE_TAIL_THREADS) k_reduce_tail(XYZZ<F>* __restrict__ A, uint32_t nbw, uint32_t n,
                                                                       uint32_t l0, XYZZ<F>* __restrict__ out) {
  XYZZ<F>* base = A + (size_t)blockIdx.x * nbw;
  const uint32_t t = threadIdx.x;
  for (uint32_t l = l0; l <= n; l++) {
    const uint32_t s = nbw >> l;
    if (t < l * s) {
      const uint32_t j = t / s, i = t % s;
      XYZZ<F>* p = base + (j ? (nbw >> j) : 0u) + i;
      XYZZ<F> a = p[0];
      if constexpr (INL) {
        const XYZZ<F> b = p[s];
        a.add_inline(b);
      } else {
        a.add(p[s]);
      }
      p[0] = a;
    }
    __syncthreads();
  }
  // base[0] = G, base[2^m] = U_m.  Scale in place (2^m positions are distinct; position 1 = U_0 needs no doubling),
  // then sum the n + 1 terms {base[0], base[1], base[2], base[4], ...} by a halving tree over their list index.
  if (t >= 1 && t < n) {
    XYZZ<F> v = base[1u << t];
    for (uint32_t k = 0; k < t; k++) v.dbl();
    base[1u << t] = v;
  }
  __syncthreads();
  auto slot = [&](uint32_t idx) -> XYZZ<F>* { return base + (idx == 0 ? 0u : (1u << (idx - 1))); };  // term idx of n + 1
  for (uint32_t len = n + 1; len > 1;) {
    const uint32_t half = (len + 1) >> 1;
    if (t < len - half) {
      XYZZ<F> a = *slot(t);
      if constexpr (INL) {
        const XYZZ<F> b = *slot(t + half);
        a.add_inline(b);
      } else {
        a.add(*slot(t + half));
      }
      *slot(t) = a;
    }
    __syncthreads();
    len = half;
  }
  if (t == 0) out[blockIdx.x] = base[0];
}

// Buckets split into MORE than MERGE_FANIN tasks have several first-level sums (every MERGE_FANIN-th partial) after
// k_merge_pass; k_tasks lists them in two classes.
//   5..16 tasks (a narrow table window at a small size cuts EVERY bucket into ~5 tasks so that the accumulate kernel
//   has enough threads): one THREAD per listed bucket adds its <= MERGE_FANIN first-level sums;  totals[2] = list length.
template <class F>
__global__ void __launch_bounds__(128) k_merge_mid(XYZZ<F>* __restrict__ partials, const uint32_t* __restrict__ mid,
                                                    const uint32_t* __restrict__ counts,
                                                    const uint32_t* __restrict__ task_off,
                                                    const uint32_t* __restrict__ totals) {
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= totals[2]) return;
  const uint32_t b = mid[h], seg = totals[4];
  XYZZ<F>* p = partials + task_off[b];
  const uint32_t nt = (counts[b] + seg - 1) / seg;
  XYZZ<F> acc = p[0];
  for (uint32_t i = MERGE_FANIN; i < nt; i += MERGE_FANIN) acc.add(p[i]);
  p[0] = acc;
}

//   more than 16 tasks (0/1-heavy witnesses, the low buckets a narrow top window piles its digits into): one CTA per
//   listed bucket finishes the merge as a halving tree over the first-level sums, instead of log4(#tasks) grid-wide
//   launches that find nothing to do for every other bucket.  Grid-stride over the list; totals[6] = list length.
template <class F>
__global__ void __launch_bounds__(256) k_merge_heavy(XYZZ<F>* __restrict__ partials, const uint32_t* __restrict__ heavy,
                                                      const uint32_t* __restrict__ counts,
                                                      const uint32_t* __restrict__ task_off,
                                                      const uint32_t* __restrict__ totals) {
  const uint32_t nheavy = totals[6], seg = totals[4];
  for (uint32_t h = blockIdx.x; h < nheavy; h += gridDim.x) {
    const uint32_t b = heavy[h];
    XYZZ<F>* p = partials + task_off[b];
    const uint32_t nt = (counts[b] + seg - 1) / seg;
    uint32_t m = (nt + MERGE_FANIN - 1) / MERGE_FANIN;   // first-level sums sit at p[MERGE_FANIN * i], i < m
    while (m > 1) {
      const uint32_t half = (m + 1) >> 1;
      for (uint32_t i = threadIdx.x; i < m - half; i += blockDim.x) {
        XYZZ<F> a = p[(size_t)MERGE_FANIN * i];
        a.add(p[(size_t)MERGE_FANIN * (i + half)]);
        p[(size_t)MERGE_FANIN * i] = a;
      }
      __syncthreads();
      m = half;
    }
    __syncthreads();
  }
}

}  // namespace b200
#include "msm_affine.cuh"
namespace b200 {
static_assert(AFF_WS_LEVELS == AFF_LEVELS_MAX, "workspace holds one buffer per pair-tree level");

// ------------------------------------------------------------------------------ host driver
// entries (= n * W at most) from which the batched-affine accumulation is used in mode 1
constexpr size_t AFF_AUTO_MIN_ENTRIES = (size_t)40 << 20;

// Window table attached to a bases vector (b200g16_bases_precompute): row k holds 2^(c k) * P_i, so
// digit k of scalar i addresses entry k * stride + i and ALL windows accumulate into one bucket set.
// (struct MsmTable lives in common.cuh)
constexpr int MSM_SLOTS = 8;           // independent result slots (a prove enqueues 5 MSMs back to back); ctx->ev_slot has as many
constexpr int MSM_MAX_WINDOWS = 130;

// Batch MSMs (k scalar vectors over one bases vector, msm_enqueue with k > 1).  One call holds at most 2^23 buckets
// (k * nb: sort_fine_bits <= 12, so the fine passes count in shared memory) and fewer than 2^32 entries (k * n * W:
// offsets, cursors and tasks are 32-bit).  A larger k is split into sub-batches of msm_batch_max vectors.
constexpr uint64_t MSM_BATCH_MAX_BUCKETS = 1ull << 23;
constexpr uint64_t MSM_BATCH_MAX_ENTRIES = (1ull << 32) - 1;

// window width and windows the library uses for an n-point MSM (with a table: the table's)
inline int msm_window_for(const b200g16_ctx* ctx, const MsmTable* tab, size_t n) {
  return tab ? tab->c : (ctx->msm_window_override ? ctx->msm_window_override : msm_pick_window(n));
}

// vectors of n points one batch enqueue may hold (>= 1; 1 means the single-MSM path)
inline size_t msm_batch_max(int c, bool table, size_t n) {
  if (c < 2 || c > 24) return 1;
  const int W = msm_num_windows(c);
  const uint64_t nb = (uint64_t)(table ? 1 : W) << (c - 1);
  uint64_t k = MSM_BATCH_MAX_BUCKETS / nb;
  if (n) k = std::min<uint64_t>(k, MSM_BATCH_MAX_ENTRIES / ((uint64_t)n * W));
  return k < 1 ? 1 : (size_t)k;
}

// Grow-only pinned staging of batch window sums: MSM_SLOTS slots of `slot_bytes`.  Called by a batch entry point before
// its first enqueue, when none of its slots is pending (every batch call drains its streams before it returns).
inline int msm_batch_stage(b200g16_ctx* ctx, size_t slot_bytes) {
  MsmWorkspace& ws = ctx->msm;
  if (ws.batch_slot >= slot_bytes) return 0;
  if (ws.batch_pinned) B200_CUDA(cudaFreeHost(ws.batch_pinned));
  ws.batch_pinned = nullptr;
  ws.batch_slot = 0;
  B200_CUDA(cudaMallocHost(&ws.batch_pinned, MSM_SLOTS * slot_bytes));
  ws.batch_slot = slot_bytes;
  return 0;
}

// Enqueue one MSM on ctx->stream; its W window sums land in pinned slot `slot` once the stream
// drains.  No host synchronisation.  record_events: fill ctx->ev for b200g16_last_timings.
// share_sort: the caller guarantees that d_scalars still holds what the previous enqueue saw under the
// same pointer; if that MSM used the same decomposition its sorted lists are reused (no sort phase).
// k > 1: k MSMs of n scalars each over the same bases, vector j at d_scalars + j * ld, in one pass of every kernel:
// vector j owns the bucket sets [j * Wr, (j + 1) * Wr) and its window sums land at items [j * Wr, (j + 1) * Wr) of slot
// `slot` of the batch staging (msm_batch_stage: k * Wr items per slot).  k must not exceed msm_batch_max.
template <class F>
int msm_enqueue(b200g16_ctx* ctx, const Affine<F>* d_bases, const MsmTable* tab, const Fr* d_scalars, size_t n, size_t k,
                size_t ld, int slot, MsmCfg* cfg_out, bool record_events, bool share_sort = false) {
  MsmCfg cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.k = (uint32_t)k;
  *cfg_out = cfg;
  if (slot < 0 || slot >= MSM_SLOTS) return fail(B200G16_ERR_ARG, "msm: bad slot");
  if (k == 0 || k >= (1ull << 32) || ld < n || ld >= (1ull << 32)) return fail(B200G16_ERR_ARG, "msm: bad batch shape");
  if (n == 0) return 0;  // cfg.W == 0 marks "infinity"
  if (n >= (1ull << 31)) return fail(B200G16_ERR_ARG, "msm: n=%zu too large", n);
  cfg.c = msm_window_for(ctx, tab, n);
  if (cfg.c < 2 || cfg.c > 24) return fail(B200G16_ERR_ARG, "msm: window %d out of range", cfg.c);
  cfg.W = msm_num_windows(cfg.c);
  if (tab && tab->W != cfg.W) return fail(B200G16_ERR_STATE, "msm: window table has %d rows, want %d", tab->W, cfg.W);
  cfg.nbw = 1u << (cfg.c - 1);
  cfg.Wr = tab ? 1 : cfg.W;
  if (k > 1 && k > msm_batch_max(cfg.c, tab != nullptr, n))
    return fail(B200G16_ERR_ARG, "msm: %zu vectors of %zu points exceed one batch call", k, n);
  cfg.nb = cfg.nbw * (uint32_t)cfg.Wr * (uint32_t)k;
  cfg.bstride = tab ? 0u : cfg.nbw;
  cfg.ent_stride = tab ? tab->stride : 0u;
  cfg.ent_off = tab ? tab->off : 0u;
  if (tab && (double)tab->stride * cfg.W >= 2.0e9) return fail(B200G16_ERR_ARG, "msm: window table too large to index");
  if ((double)n * cfg.W >= 4.0e9) return fail(B200G16_ERR_ARG, "msm: n*W overflows 32-bit entry index");
  size_t m_max = n * k * (size_t)cfg.W;
  const uint32_t R = (uint32_t)(k * cfg.Wr);   // bucket sets (window sums) of all vectors
  cfg.target_tasks = (uint32_t)ctx->sm_count * 2048u;  // ~4 waves of 512 resident threads per SM
  cfg.ch = 1;   // (unused since the tree reduction: one bucket per leaf)
  cfg.nch = cfg.nbw;
  // #tasks = sum ceil(cnt/seg) <= nb + total/seg <= nb + target (k_pick_seg keeps seg >= total/target)
  size_t max_tasks = (size_t)cfg.nb + cfg.target_tasks + 64;

  MsmWorkspace& ws = ctx->msm;
  const int par = ctx->msm_parity;  // own set: partials, chunks
  ctx->msm_parity = (par + 1) % MSM_SETS;
  const MsmSorted& ls = ctx->last_sort;
  const bool reuse = share_sort && ls.valid && ls.par != par && ls.scalars == (const void*)d_scalars && ls.n == n &&
                     ls.k == k && ls.ld == ld && ls.c == cfg.c && ls.bstride == cfg.bstride && ls.ent_stride == cfg.ent_stride &&
                     ls.ent_off == cfg.ent_off;
  const int spar = reuse ? ls.par : par;  // set holding the sorted state: counts, offsets, tasks, totals
  const int sort_F = sort_fine_bits(cfg.nb);
  B200_TRY(ws.part.ensure(m_max * sizeof(SortItem)));
  B200_TRY(ws.bins.ensure(sort_bin_bytes(sort_num_bins(cfg.nb, sort_F), m_max)));
  B200_TRY(ws.entries.ensure(m_max * sizeof(uint32_t)));
  // totals[16] + two lists of split buckets [nb each] + scan tile sums (uint2 per 2048 buckets, 8-byte aligned)
  const size_t scan_off = (64 + 2 * (size_t)cfg.nb * sizeof(uint32_t) + 7) & ~(size_t)7;
  // every rotating set is sized for this call at once: a prove alternates G1 and G2 MSMs over the sets, and
  // growing a set later would cost a cudaFree (device-wide synchronisation) in the middle of a prove
  for (int q = 0; q < MSM_SETS; q++) {
    B200_TRY(ws.counts[q].ensure((size_t)cfg.nb * 4 * sizeof(uint32_t)));  // counts, offsets, cursor, task_off
    B200_TRY(ws.misc[q].ensure(scan_off + ((size_t)cfg.nb / 2048 + 4) * sizeof(uint2) + 2 * 4096 * sizeof(uint32_t)));
    B200_TRY(ws.tasks[q].ensure(2 * max_tasks * sizeof(uint32_t)));  // task_bucket, task_order
    B200_TRY(ws.partials[q].ensure(max_tasks * sizeof(XYZZ<F>)));
    // dense bucket array of the reduction tree + two ping-pong rows of c terms per window for the sum passes
    B200_TRY(ws.chunks[q].ensure(((size_t)R * cfg.nbw + 2 * (size_t)R * (cfg.c + 1)) * sizeof(XYZZ<F>)));
  }
  const size_t slot_bytes = MSM_MAX_WINDOWS * sizeof(XYZZ<Fp2>);
  if (ws.pinned_cap < MSM_SLOTS * slot_bytes) {
    if (ws.pinned) cudaFreeHost(ws.pinned);
    B200_CUDA(cudaMallocHost(&ws.pinned, MSM_SLOTS * slot_bytes));
    ws.pinned_cap = MSM_SLOTS * slot_bytes;
  }
  if (cfg.W > MSM_MAX_WINDOWS - 2) return fail(B200G16_ERR_ARG, "msm: too many windows");
  if (k > 1 && ws.batch_slot < (size_t)R * sizeof(XYZZ<F>)) return fail(B200G16_ERR_STATE, "msm: batch staging too small");
  char* stage = k > 1 ? (char*)ws.batch_pinned + (size_t)slot * ws.batch_slot : (char*)ws.pinned + (size_t)slot * slot_bytes;

  uint32_t* counts = ws.counts[spar].as<uint32_t>();
  uint32_t* offsets = counts + cfg.nb;
  uint32_t* cursor = offsets + cfg.nb;
  uint32_t* task_off = cursor + cfg.nb;
  uint32_t* totals = ws.misc[spar].as<uint32_t>();
  SortItem* part = ws.part.as<SortItem>();
  uint32_t* entries = ws.entries.as<uint32_t>();
  uint32_t* task_bucket = ws.tasks[spar].as<uint32_t>();
  uint32_t* task_order = task_bucket + max_tasks;
  uint32_t* mid = totals + 16;     // buckets split into 5..16 tasks (k_tasks), nb entries reserved
  uint32_t* heavy = mid + cfg.nb;  // buckets split into more than 16 tasks, nb entries reserved
  XYZZ<F>* partials = ws.partials[par].as<XYZZ<F>>();
  XYZZ<F>* chunks = ws.chunks[par].as<XYZZ<F>>();
  XYZZ<F>* windows = nullptr;
  cudaStream_t st = ctx->stream, tail = ctx->tail_stream;
  uint32_t n32 = (uint32_t)n;
  int ev = 0;
  auto mark = [&]() { if (record_events && ev < 18) cudaEventRecord(ctx->ev[ev++], st); };
  // buffer set `par` may still be read by the tail of the MSM before last
  if (ctx->tail_pending[par]) B200_CUDA(cudaStreamWaitEvent(st, ctx->ev_tail[par], 0));
  if (!reuse) {
    // ... and its sorted state by the tail of an MSM that shared it
    const int rd = ctx->sort_reader[par];
    if (rd >= 0 && ctx->tail_pending[rd]) B200_CUDA(cudaStreamWaitEvent(st, ctx->ev_tail[rd], 0));
    ctx->sort_reader[par] = -1;
    ctx->last_sort.valid = false;
    B200_TRY(msm_sort_phase(ctx, cfg, d_scalars, n32, (uint32_t)ld, part, ws.bins.as<uint32_t>(), counts, offsets, cursor, task_off, totals, entries,
                            task_bucket, task_order, (uint32_t)max_tasks,
                            reinterpret_cast<uint32_t*>(ws.misc[par].as<char>() + scan_off),
                            record_events ? &ev : nullptr));
    ctx->last_sort.scalars = d_scalars;
    ctx->last_sort.n = n;
    ctx->last_sort.k = k;
    ctx->last_sort.ld = ld;
    ctx->last_sort.c = cfg.c;
    ctx->last_sort.bstride = cfg.bstride;
    ctx->last_sort.ent_stride = cfg.ent_stride;
    ctx->last_sort.ent_off = cfg.ent_off;
    ctx->last_sort.par = par;
    ctx->last_sort.valid = true;
  } else {
    ctx->sort_reader[spar] = par;   // this MSM's tail reads set spar: its next writer must wait for it
    ctx->last_sort.valid = false;   // one sharer per sort
    if (record_events) { mark(); mark(); mark(); }
  }
  const bool use_aff = ctx->msm_affine_mode == 2 || (ctx->msm_affine_mode == 1 && m_max >= AFF_AUTO_MIN_ENTRIES);
  if (use_aff) {
    const unsigned grid = (unsigned)ctx->sm_count * ((sizeof(F) > 32) ? 2u : 4u);   // one wave: equal shares per thread
    const uint32_t T = grid * (uint32_t)AFF_THREADS;
    AffArgs<F> A;
    A.bases = d_bases; A.entries = entries; A.task_bucket = task_bucket; A.offsets = offsets; A.counts = counts;
    A.task_off = task_off; A.totals = totals; A.partials = partials;
    A.max_levels = ctx->msm_affine_levels < 1 ? 1 : (ctx->msm_affine_levels > AFF_LEVELS_MAX ? AFF_LEVELS_MAX : ctx->msm_affine_levels);
    A.min_pairs = ctx->msm_affine_min_pairs;
    A.lvl[0] = nullptr;
    for (int l = 1; l <= AFF_LEVELS_MAX; l++) {
      A.lvl[l] = nullptr;
      if (l > A.max_levels) continue;
      B200_TRY(ws.aff_lvl[l - 1].ensure(((m_max >> l) + max_tasks + T + 16) * sizeof(Affine<F>)));
      A.lvl[l] = ws.aff_lvl[l - 1].as<Affine<F>>();
    }
    B200_TRY(ws.aff_desc.ensure((max_tasks + T + 16) * sizeof(AffDesc)));
    A.desc = ws.aff_desc.as<AffDesc>();
    B200_TRY(ws.aff_spill.ensure((size_t)T * sizeof(XYZZ<F>)));
    B200_TRY(ws.aff_spill_task.ensure((size_t)T * sizeof(uint32_t)));
    A.spill = ws.aff_spill.as<XYZZ<F>>();
    A.spill_task = ws.aff_spill_task.as<uint32_t>();
    k_accumulate_affine<F><<<grid, AFF_THREADS, 0, st>>>(A);
    k_aff_fixup<F><<<cdiv(T, 128), 128, 0, st>>>(partials, A.spill, A.spill_task, T);
    ctx->launches += 1;
  } else {
    k_accumulate<F><<<cdiv(max_tasks, 128), 128, 0, st>>>(d_bases, entries, task_order, task_bucket, offsets, counts, task_off,
                                                           totals, partials);
  }
  mark();
  // ---- tail: merge of split buckets + bucket reduction on the second stream (few active threads, long
  // dependency chains), so that the next MSM's sort + accumulate on `st` overlap it
  B200_CUDA(cudaEventRecord(ctx->ev_front[par], st));
  B200_CUDA(cudaStreamWaitEvent(tail, ctx->ev_front[par], 0));
  // split buckets: one grid-wide fan-in-4 pass, then one thread (<= 16 tasks) or one CTA per bucket that still has more
  // than one first-level sum
  k_merge_pass<F><<<cdiv(max_tasks, 128), 128, 0, tail>>>(partials, task_bucket, counts, task_off, totals, 1u);
  k_merge_mid<F><<<cdiv(std::min<size_t>(cfg.nb, max_tasks / (MERGE_FANIN + 1) + 1), 128), 128, 0, tail>>>(partials, mid, counts,
                                                                                                        task_off, totals);
  k_merge_heavy<F><<<(unsigned)ctx->sm_count * 2, 256, 0, tail>>>(partials, heavy, counts, task_off, totals);
  if (record_events && ev < 18) cudaEventRecord(ctx->ev[ev++], tail);
  const uint32_t nlev = (uint32_t)cfg.c - 1;  // log2(buckets per window)
  uint32_t l0 = 1;                            // first level the one-CTA tail kernel can take
  while (l0 <= nlev && (uint64_t)l0 * (cfg.nbw >> l0) > REDUCE_TAIL_THREADS) l0++;
  if (l0 < 2) l0 = 2;                         // level 1 (reads the partials through the task table) is always its own kernel
  constexpr bool CAN_INL = sizeof(F) <= 32;
  const bool inl = CAN_INL && reduce_inline_default() >= 1, inl_tail = CAN_INL && reduce_inline_default() >= 2;
  // CTA size of the grid-wide levels.  (G2, ~180 registers per thread with the out-of-line addition: 32 / 64 / 96 / 128
  // threads per CTA measure 1.75 / 1.77 / 2.07 / 1.78 ms for the whole reduction at c = 20, profiles/r02w_g2_reduce_block.jsonl
  // — occupancy is not its lever.)
  constexpr unsigned rb = 128u;
  // R = k * Wr bucket sets, nbw apart: vector j's set w is set j * Wr + w (key j * vstride + w * bstride + |d| - 1)
  const unsigned g1 = cdiv((size_t)R * (cfg.nbw >> 1), rb);
  if (inl) k_reduce_first<F, CAN_INL><<<g1, rb, 0, tail>>>(partials, counts, task_off, R, cfg.nbw, chunks);
  else k_reduce_first<F, false><<<g1, rb, 0, tail>>>(partials, counts, task_off, R, cfg.nbw, chunks);
  int sum_levels = 2;
  for (uint32_t l = 2; l < l0 && l <= nlev; l++, sum_levels++) {
    const unsigned gl = cdiv((size_t)R * l * (cfg.nbw >> l), rb);
    if (inl) k_reduce_level<F, CAN_INL><<<gl, rb, 0, tail>>>(chunks, R, cfg.nbw, l);
    else k_reduce_level<F, false><<<gl, rb, 0, tail>>>(chunks, R, cfg.nbw, l);
  }
  XYZZ<F>* cur = chunks + (size_t)R * cfg.nbw;   // R window sums behind the tree
  if (inl_tail) k_reduce_tail<F, CAN_INL><<<R, REDUCE_TAIL_THREADS, 0, tail>>>(chunks, cfg.nbw, nlev, l0 > nlev ? nlev + 1 : l0, cur);
  else k_reduce_tail<F, false><<<R, REDUCE_TAIL_THREADS, 0, tail>>>(chunks, cfg.nbw, nlev, l0 > nlev ? nlev + 1 : l0, cur);
  const int merge_levels = 3;
  windows = cur;  // R items
  if (record_events && ev < 18) cudaEventRecord(ctx->ev[ev++], tail);
  ctx->launches += merge_levels + sum_levels;
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaMemcpyAsync(stage, windows, (size_t)R * sizeof(XYZZ<F>), cudaMemcpyDeviceToHost, tail));
  B200_CUDA(cudaEventRecord(ctx->ev_tail[par], tail));
  B200_CUDA(cudaEventRecord(ctx->ev_slot[slot], tail));
  ctx->tail_pending[par] = true;
  if (record_events) ctx->timings.n = -(ev - 1);  // negative: events recorded, not yet resolved
  *cfg_out = cfg;
  return 0;
}

// Make ctx->stream wait for every outstanding bucket reduction: after this, synchronising ctx->stream
// guarantees all enqueued MSM results are in their pinned slots.
inline int msm_join(b200g16_ctx* ctx) {
  for (int p = 0; p < MSM_SETS; p++)
    if (ctx->tail_pending[p]) {
      B200_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_tail[p], 0));
      ctx->tail_pending[p] = false;
    }
  return 0;
}

// After a failed call: wait for everything in flight on the ctx's streams and forget it (no open prove, no sorted lists
// to share), so that the ctx is usable again.
inline void msm_drain(b200g16_ctx* ctx) {
  msm_join(ctx);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->tail_stream);
  cudaStreamSynchronize(ctx->copy_stream);
  ctx->prove_active = false;
  ctx->last_sort.valid = false;
}

// After the stream has drained: Horner over the window sums of `slot` (vector j of a batch) on the host,
// acc = sum_w 2^(c w) * S_w, then one inversion to the affine normal form.
template <class F>
int msm_collect(b200g16_ctx* ctx, int slot, const MsmCfg& cfg, Affine<F>* out, size_t j = 0) {
  if (cfg.W == 0) { *out = Affine<F>::inf(); return 0; }
  const size_t slot_bytes = MSM_MAX_WINDOWS * sizeof(XYZZ<Fp2>);
  const XYZZ<F>* hw = cfg.k > 1 ? reinterpret_cast<const XYZZ<F>*>((const char*)ctx->msm.batch_pinned + (size_t)slot * ctx->msm.batch_slot) +
                                      j * cfg.Wr
                                : reinterpret_cast<const XYZZ<F>*>((const char*)ctx->msm.pinned + (size_t)slot * slot_bytes);
  XYZZ<F> acc = hw[cfg.Wr - 1];
  for (int w = cfg.Wr - 2; w >= 0; w--) {
    for (int k = 0; k < cfg.c; k++) acc.dbl();
    acc.add(hw[w]);
  }
  *out = acc.to_affine();
  return 0;
}

inline void msm_resolve_timings(b200g16_ctx* ctx) {
  if (ctx->timings.n < 0) events_to_timings(ctx, 1 - ctx->timings.n);
}

template <class F>
int msm_device(b200g16_ctx* ctx, const Affine<F>* d_bases, const MsmTable* tab, const Fr* d_scalars, size_t n,
               Affine<F>* out) {
  MsmCfg cfg;
  ctx->timings.n = 0;
  B200_TRY(msm_enqueue<F>(ctx, d_bases, tab, d_scalars, n, 1, n, 0, &cfg, true));
  B200_TRY(msm_join(ctx));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  msm_resolve_timings(ctx);
  return msm_collect<F>(ctx, 0, cfg, out);
}

// ------------------------------------------------------------------------------ window tables
// row[i] = 2^c * prev[i] in affine form.  Each thread owns TABLE_BATCH points (strided, so loads and
// stores coalesce): c doublings each in XYZZ, then ONE field inversion shared by the batch
// (Montgomery's trick) for the affine normal forms.
constexpr int TABLE_BATCH = 4;

template <class F>
__global__ void __launch_bounds__(128) k_table_row(const Affine<F>* __restrict__ prev, Affine<F>* __restrict__ next,
                                                    uint32_t n, int c) {
  const uint32_t T = gridDim.x * blockDim.x, t = blockIdx.x * blockDim.x + threadIdx.x;
  XYZZ<F> p[TABLE_BATCH];
  F pref[TABLE_BATCH];
  F acc = F::one();
#pragma unroll 1
  for (int k = 0; k < TABLE_BATCH; k++) {
    const uint32_t i = t + (uint32_t)k * T;
    XYZZ<F> q = XYZZ<F>::inf();
    if (i < n) {
      q = XYZZ<F>::from_affine(load_affine(prev + i));
      for (int j = 0; j < c; j++) q.dbl();
    }
    pref[k] = acc;
    if (!q.is_inf()) acc = F::mul(acc, q.zzz);
    p[k] = q;
  }
  F inv = F::inv(acc);
#pragma unroll 1
  for (int k = TABLE_BATCH - 1; k >= 0; k--) {
    const uint32_t i = t + (uint32_t)k * T;
    if (i >= n) continue;
    Affine<F> o = Affine<F>::inf();
    if (!p[k].is_inf()) {
      F zi = F::mul(inv, pref[k]);  // 1 / zzz_k
      inv = F::mul(inv, p[k].zzz);
      F izz = F::sqr(F::mul(p[k].zz, zi));  // 1 / zz_k = (zz/zzz)^2
      o.x = F::mul(p[k].x, izz);
      o.y = F::mul(p[k].y, zi);
    }
    next[i] = o;
  }
}

// Window width for a table over n bases: minimise W(c) * n (accumulate adds) + 8 * 2^(c-1) (ONE
// bucket set to reduce, same cost model as msm_pick_window), subject to the 31-bit entry index.
int msm_pick_table_window(size_t n);

// table: W rows of n points, row 0 already holds the bases.
template <class F>
int msm_build_table(b200g16_ctx* ctx, Affine<F>* table, size_t n, int c, int W) {
  if (n == 0) return 0;
  const unsigned grid = cdiv(cdiv(n, TABLE_BATCH), 128);
  for (int k = 1; k < W; k++) {
    k_table_row<F><<<grid, 128, 0, ctx->stream>>>(table + (size_t)(k - 1) * n, table + (size_t)k * n, (uint32_t)n, c);
    ctx->launches++;
  }
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// (bases pointer, table descriptor) for points [offset, offset + n) of a resident vector
template <class F>
inline const Affine<F>* msm_operand(const b200g16_bases* b, size_t offset, MsmTable* tab, const MsmTable** tab_out) {
  const Affine<F>* p = reinterpret_cast<const Affine<F>*>(b->d_points);
  if (b->tab_c) {
    tab->c = b->tab_c; tab->W = b->tab_W; tab->stride = (uint32_t)b->n; tab->off = (uint32_t)offset;
    *tab_out = tab;
    return p;
  }
  *tab_out = nullptr;
  return p + offset;
}

}  // namespace b200
