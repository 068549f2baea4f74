// Two-level counting sort of the MSM's (window, point) entries into bucket order (msm_sort_phase, msm_common.cu).
//
// An entry is a nonzero signed digit d of scalar i in window w: key = w * bstride + |d| - 1 (its bucket) and
// value (w * ent_stride + ent_off + i) << 1 | (d < 0).  A bucket's coarse bin is key >> F, with F picked so that
// there are at most SORT_BINS bins (sort_fine_bits).  Every global atomic and every run of stores covers a CTA's
// share of one bin or one bucket, never a single entry:
//
//   1  coarse count      one thread per point converts its scalar to canonical form (kept in canon[] for pass 3)
//                        and recodes it; shared-memory histogram over the bins, one global atomic per (CTA,
//                        occupied bin) -> bin_count;  entries -> totals[3]
//   2  bin scan          one CTA: bin offsets, and tiles of at most SORT_TILE entries; a tile never straddles
//                        two bins, so a skewed input (0/1 witness scalars in bin 0, a narrow top window in the
//                        lowest bins) becomes many tiles of one bin
//   3  coarse partition  recodes canon[] again, stages the CTA's entries in bin order in shared memory, reserves one run
//                        per (CTA, occupied bin) with one global atomic and copies the runs out as (key, value)
//                        pairs into part[] with consecutive threads on consecutive words
//   4  fine count        one CTA per tile: shared histogram over the 2^F buckets of the tile's bin, one global
//                        atomic per occupied bucket -> counts
//      (scan of counts -> offsets / cursor / task_off: k_scan_*)
//   6  fine place        one CTA per tile: count again, reserve one run per occupied bucket from cursor, write
//                        the values into entries[] (staging them as pass 3 does measured slower: the tile's
//                        runs already land in the bin's own few-KB range of entries[])
//
// Passes 3 and 6 hold no per-entry state across a barrier: the count step only counts, the reserve step turns the
// counts into run starts, and the place step takes each entry's slot with a second shared atomic (recoding canon[]
// again / re-reading the tile from L2).  Pass 3 stages its entries in shared memory and copies the runs out: stores issued
// entry by entry leave partly written lines all over part[] for as long as a CTA runs (every CTA writes into every
// bin), a frontier the L2 cannot hold (4.1 ms instead of 1.9 at 2^24).  Order inside a bucket is free.
// With F > SORT_FINE_MAX_BITS (plain windows forced to c >= 20: tens of millions of buckets) passes 4 and 6 count
// and place with one global atomic per entry; no width the library picks for itself goes there.
//
// Batch (BATCH = true, msm_enqueue with k > 1 scalar vectors over one bases vector): the point index q of passes 1 and
// 3 runs over [0, k * vn) and splits as j = q / vn (vector) and i = q - j * vn (point); the scalar is scalars[j * ld + i]
// and canon[q] its canonical form.  Every key gains j * vstride (vector j's own bucket sets, vstride = Wr * nbw), the
// value is that of point i alone, so every vector gathers the same bases / table rows and passes 2, 4 and 6 (and
// everything after the sort) see nothing but more buckets.  The single-vector kernels are the BATCH = false instances,
// which read none of the batch fields (vn == 0 there means one vector).
//
// Everything below is plain C++ over field.cuh, run by the kernels thread by thread between barriers, so
// tests/host_harness/sort_host.cc and sort_batch_host.cc run the same steps CTA by CTA on the CPU against a direct
// counting sort.
#pragma once
#include "field.cuh"

namespace b200 {

constexpr uint32_t SORT_BINS = 2048;       // coarse bins at most
constexpr int SORT_FINE_MAX_BITS = 12;     // fine keys per bin counted in shared memory at most: 2^12
constexpr int SORT_CTA = 512;              // threads of every sort pass
constexpr int SORT_PPT = 4;                // points per thread, pass 1
constexpr uint32_t SORT_POINTS = (uint32_t)SORT_CTA * SORT_PPT;   // points per CTA, pass 1
constexpr int SORT_IPT = 16;               // entries per thread, passes 4 and 6
constexpr uint32_t SORT_TILE = (uint32_t)SORT_CTA * SORT_IPT;     // entries per tile at most

struct alignas(8) SortItem {
  uint32_t key;  // bucket
  uint32_t val;  // (w * ent_stride + ent_off + i) << 1 | neg
};

struct alignas(8) SortTile {
  uint32_t start;  // first entry of the tile in part[]
  uint32_t bin;
};

struct SortArgs {
  const Fr* scalars;     // Montgomery form
  Fr* canon;             // [n]: the scalars in canonical form, written by pass 1 and read by pass 3
  uint32_t n;
  int c, W;
  uint32_t bstride, ent_stride, ent_off;
  int F;                 // fine bits: bin = key >> F
  uint32_t nbins;        // coarse bins (<= SORT_BINS)
  uint32_t part_points;  // points per CTA of pass 3 (sort_part_points)
  uint32_t* bin_count;   // [SORT_BINS]
  uint32_t* bin_cursor;  // [SORT_BINS]
  uint32_t* bin_off;     // [SORT_BINS + 1]
  uint32_t* ntiles;      // [1]
  SortTile* tiles;       // [sort_max_tiles]
  SortItem* part;        // [n * W]: entries in bin order
  uint32_t* counts;      // per bucket
  uint32_t* cursor;      // per bucket: offsets, advanced by pass 6
  uint32_t* entries;     // [n * W]: values in bucket order
  uint32_t* totals;
  // batch fields (read by the BATCH instances only; appended so the single-vector kernels' parameters keep their offsets)
  uint32_t vn;       // points per vector (0: one vector, n points)
  uint32_t ld;       // scalar row stride in elements (>= vn)
  uint32_t vstride;  // buckets per vector
};

// smallest F with at most SORT_BINS bins
inline int sort_fine_bits(uint32_t nb) {
  int F = 0;
  while ((((uint64_t)nb + (1ull << F) - 1) >> F) > SORT_BINS) F++;
  return F;
}
inline uint32_t sort_num_bins(uint32_t nb, int F) { return (uint32_t)(((uint64_t)nb + (1ull << F) - 1) >> F); }
// tiles: sum over bins of ceil(count / SORT_TILE) <= bins + entries / SORT_TILE
inline size_t sort_max_tiles(uint32_t nbins, size_t m) { return nbins + m / SORT_TILE + 1; }
// bin buffer: bin_count, bin_cursor [SORT_BINS] each, bin_off [SORT_BINS + 1], ntiles, then the tiles (8-byte aligned)
constexpr size_t SORT_BIN_WORDS = 3 * (size_t)SORT_BINS + 2;
inline size_t sort_bin_bytes(uint32_t nbins, size_t m) { return SORT_BIN_WORDS * 4 + sort_max_tiles(nbins, m) * sizeof(SortTile); }

B200_HD uint32_t sort_add(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, v);
#else
  const uint32_t o = *p;
  *p = o + v;
  return o;
#endif
}

// Signed c-bit recoding of canonical limbs (limbs[8] = 0): fn(w, d) for every window, d in [-2^(c-1), 2^(c-1)).
// tests/test_msm_digits_cpu.py restates this loop line for line.
template <class Fn>
B200_HD void sort_recode(const uint32_t limbs[9], int c, int W, Fn&& fn) {
  const uint32_t mask = (c == 32) ? 0xffffffffu : ((1u << c) - 1u);
  const uint32_t half = 1u << (c - 1);
  uint32_t carry = 0;
  for (int w = 0; w < W; w++) {
    int bit = w * c;
    int q = bit >> 5, r = bit & 31;
    uint32_t raw = 0;
    if (q < 8) {
      uint64_t two = (uint64_t)limbs[q] | ((uint64_t)limbs[q + 1] << 32);
      raw = (uint32_t)(two >> r) & mask;
    }
    raw += carry;
    int32_t d;
    if (raw >= half) { d = (int32_t)raw - (int32_t)(1u << c); carry = 1; }
    else { d = (int32_t)raw; carry = 0; }
    fn(w, d);
  }
}

// point q -> (vector j, point i of that vector) and the scalar's index in A.scalars
template <bool BATCH>
B200_HD size_t sort_point(const SortArgs& A, uint32_t q, uint32_t& i, uint32_t& j) {
  if constexpr (BATCH) {
    j = q / A.vn;
    i = q - j * A.vn;
    return (size_t)j * A.ld + i;
  } else {
    j = 0;
    i = q;
    return q;
  }
}

// fn(key, val) for every nonzero digit of scalar i of vector j, given in canonical form
template <bool BATCH = false, class Fn>
B200_HD void sort_entries(const SortArgs& A, const Fr& s, uint32_t i, uint32_t j, Fn&& fn) {
  uint32_t limbs[9];
#pragma unroll
  for (int k = 0; k < 8; k++) limbs[k] = s.l[k];
  limbs[8] = 0;
  sort_recode(limbs, A.c, A.W, [&](int w, int32_t d) {
    if (d == 0) return;
    const uint32_t neg = d < 0;
    const uint32_t mag = neg ? (uint32_t)(-d) : (uint32_t)d;
    const uint32_t key = (uint32_t)w * A.bstride + mag - 1;
    fn(BATCH ? j * A.vstride + key : key, (((uint32_t)w * A.ent_stride + A.ent_off + i) << 1) | neg);
  });
}
template <class Fn>
B200_HD void sort_entries(const SortArgs& A, const Fr& s, uint32_t i, Fn&& fn) {
  sort_entries<false>(A, s, i, 0u, fn);
}

// ---- pass 1: CTA `blk` owns points [blk * SORT_POINTS, +SORT_POINTS); s[SORT_BINS + 1] in shared memory
B200_HD void sort_coarse_init(const SortArgs& A, uint32_t tid, uint32_t* s) {
  for (uint32_t b = tid; b < A.nbins; b += SORT_CTA) s[b] = 0;
  if (tid == 0) s[SORT_BINS] = 0;
}

// s[bin] += entries;  s[SORT_BINS] += all entries
template <bool BATCH = false>
B200_HD void sort_coarse_count(const SortArgs& A, uint32_t blk, uint32_t tid, uint32_t* s) {
  uint32_t nz = 0;
  for (int k = 0; k < SORT_PPT; k++) {
    const uint32_t q = blk * SORT_POINTS + (uint32_t)k * SORT_CTA + tid;
    if (q >= A.n) break;
    uint32_t i, j;
    const Fr sc = Fr::from_mont(A.scalars[sort_point<BATCH>(A, q, i, j)]);
    A.canon[q] = sc;
    sort_entries<BATCH>(A, sc, i, j, [&](uint32_t key, uint32_t) { sort_add(&s[key >> A.F], 1u); nz++; });
  }
  if (nz) sort_add(&s[SORT_BINS], nz);
}

B200_HD void sort_coarse_flush(const SortArgs& A, uint32_t tid, const uint32_t* s) {
  for (uint32_t b = tid; b < A.nbins; b += SORT_CTA)
    if (s[b]) sort_add(&A.bin_count[b], s[b]);
  if (tid == 0 && s[SORT_BINS]) sort_add(&A.totals[3], s[SORT_BINS]);
}

// ---- pass 3: CTA `blk` owns points [blk * P, +P), P = A.part_points, so that its P * W entries fit the staging
// area.  Shared memory: s[SORT_BINS + 1] (counts, then their exclusive scan: the bins' runs in the staging area, then
// the staging cursors), loc[SORT_BINS] (run starts), glob[SORT_BINS] (run starts in part[]), stage[SORT_STAGE].
// The entries are staged in bin order first and then copied out run by run: consecutive threads store consecutive
// words, so a run's lines are written in one go instead of entry by entry over the whole pass.
constexpr uint32_t SORT_STAGE = 10240;   // staged entries per CTA: 80 KB, two CTAs per SM

inline uint32_t sort_part_points(int W) { return SORT_STAGE / (uint32_t)W; }
inline size_t sort_part_smem() { return (3 * (size_t)SORT_BINS + 1) * 4 + SORT_STAGE * sizeof(SortItem); }

template <bool BATCH = false>
B200_HD void sort_part_count(const SortArgs& A, uint32_t blk, uint32_t tid, uint32_t* s) {
  for (uint32_t k = tid; k < A.part_points; k += SORT_CTA) {
    const uint32_t q = blk * A.part_points + k;
    if (q >= A.n) break;
    uint32_t i, j;
    sort_point<BATCH>(A, q, i, j);
    sort_entries<BATCH>(A, A.canon[q], i, j, [&](uint32_t key, uint32_t) { sort_add(&s[key >> A.F], 1u); });
  }
}

// after the exclusive scan of s (total in s[SORT_BINS]): one run per occupied bin in part[]
B200_HD void sort_part_reserve(const SortArgs& A, uint32_t tid, const uint32_t* s, uint32_t* loc, uint32_t* glob) {
  for (uint32_t b = tid; b < A.nbins; b += SORT_CTA) {
    const uint32_t cnt = s[b + 1] - s[b];
    loc[b] = s[b];
    if (cnt) glob[b] = sort_add(&A.bin_cursor[b], cnt);
  }
}

template <bool BATCH = false>
B200_HD void sort_part_stage(const SortArgs& A, uint32_t blk, uint32_t tid, uint32_t* s, SortItem* stage) {
  for (uint32_t k = tid; k < A.part_points; k += SORT_CTA) {
    const uint32_t q = blk * A.part_points + k;
    if (q >= A.n) break;
    uint32_t i, j;
    sort_point<BATCH>(A, q, i, j);
    sort_entries<BATCH>(A, A.canon[q], i, j,
                        [&](uint32_t key, uint32_t val) { stage[sort_add(&s[key >> A.F], 1u)] = SortItem{key, val}; });
  }
}

B200_HD void sort_part_write(const SortArgs& A, uint32_t tid, uint32_t total, const uint32_t* loc, const uint32_t* glob,
                             const SortItem* stage) {
  for (uint32_t k = tid; k < total; k += SORT_CTA) {
    const SortItem it = stage[k];
    const uint32_t b = it.key >> A.F;
    A.part[glob[b] + k - loc[b]] = it;
  }
}

// ---- pass 2 (one CTA, SORT_BINS / SORT_CTA bins per thread): sa[b] = entries of bin b, sb[b] = its tiles;
// the kernel turns both (SORT_BINS + 1 words each) into exclusive scans between load and write
constexpr int SORT_BPT = SORT_BINS / SORT_CTA;

B200_HD void sort_bins_load(const SortArgs& A, uint32_t tid, uint32_t* sa, uint32_t* sb) {
  for (int j = 0; j < SORT_BPT; j++) {
    const uint32_t b = tid * SORT_BPT + j;
    const uint32_t cnt = b < A.nbins ? A.bin_count[b] : 0u;
    sa[b] = cnt;
    sb[b] = (cnt + SORT_TILE - 1) / SORT_TILE;
  }
}

B200_HD void sort_bins_write(const SortArgs& A, uint32_t tid, const uint32_t* sa, const uint32_t* sb) {
  for (int j = 0; j < SORT_BPT; j++) {
    const uint32_t b = tid * SORT_BPT + j;
    if (b < A.nbins) { A.bin_off[b] = sa[b]; A.bin_cursor[b] = sa[b]; }
  }
  const uint32_t nt = sb[SORT_BINS];
  if (tid == 0) { A.bin_off[A.nbins] = sa[SORT_BINS]; *A.ntiles = nt; }
  for (uint32_t t = tid; t < nt; t += SORT_CTA) {
    uint32_t lo = 0, hi = A.nbins;   // sb[lo] <= t < sb[hi]
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (sb[mid] <= t) lo = mid; else hi = mid;
    }
    A.tiles[t] = SortTile{sa[lo] + (t - sb[lo]) * SORT_TILE, lo};
  }
}

// ---- passes 4 and 6: one CTA per tile;  s[2^F] in shared memory when F <= SORT_FINE_MAX_BITS
struct SortSpan {
  uint32_t start, end, bin;
};

B200_HD SortSpan sort_tile_span(const SortArgs& A, uint32_t t) {
  const SortTile tl = A.tiles[t];
  const uint32_t bend = A.bin_off[tl.bin + 1];
  return SortSpan{tl.start, tl.start + SORT_TILE < bend ? tl.start + SORT_TILE : bend, tl.bin};
}

B200_HD bool sort_fine_local(const SortArgs& A) { return A.F <= SORT_FINE_MAX_BITS; }

B200_HD void sort_fine_init(const SortArgs& A, uint32_t tid, uint32_t* s) {
  if (!sort_fine_local(A)) return;
  for (uint32_t f = tid; f < (1u << A.F); f += SORT_CTA) s[f] = 0;
}

// pass 4 (global: counts += entries) and the count step of pass 6 (shared only).  Every load of the tile is issued
// before the first atomic.
B200_HD void sort_fine_count(const SortArgs& A, const SortSpan& sp, uint32_t tid, uint32_t* s, bool global) {
  const bool local = sort_fine_local(A);
  if (!local && !global) return;
  const uint32_t fmask = (1u << (local ? A.F : 0)) - 1u;
  uint32_t key[SORT_IPT];
#pragma unroll
  for (int j = 0; j < SORT_IPT; j++) {
    const uint32_t e = sp.start + (uint32_t)j * SORT_CTA + tid;
    key[j] = e < sp.end ? A.part[e].key : 0u;
  }
#pragma unroll
  for (int j = 0; j < SORT_IPT; j++) {
    if (sp.start + (uint32_t)j * SORT_CTA + tid >= sp.end) break;
    if (local) sort_add(&s[key[j] & fmask], 1u);
    else sort_add(&A.counts[key[j]], 1u);
  }
}

B200_HD void sort_fine_flush(const SortArgs& A, const SortSpan& sp, uint32_t tid, const uint32_t* s) {
  if (!sort_fine_local(A)) return;
  for (uint32_t f = tid; f < (1u << A.F); f += SORT_CTA)
    if (s[f]) sort_add(&A.counts[(sp.bin << A.F) | f], s[f]);
}

// pass 6: one run per occupied bucket; s[f] becomes the run's next free slot
B200_HD void sort_fine_reserve(const SortArgs& A, const SortSpan& sp, uint32_t tid, uint32_t* s) {
  if (!sort_fine_local(A)) return;
  for (uint32_t f = tid; f < (1u << A.F); f += SORT_CTA)
    if (s[f]) s[f] = sort_add(&A.cursor[(sp.bin << A.F) | f], s[f]);
}

B200_HD void sort_fine_place(const SortArgs& A, const SortSpan& sp, uint32_t tid, uint32_t* s) {
  const bool local = sort_fine_local(A);
  const uint32_t fmask = (1u << (local ? A.F : 0)) - 1u;
  SortItem it[SORT_IPT];
#pragma unroll
  for (int j = 0; j < SORT_IPT; j++) {
    const uint32_t e = sp.start + (uint32_t)j * SORT_CTA + tid;
    it[j] = e < sp.end ? A.part[e] : SortItem{0u, 0u};
  }
#pragma unroll
  for (int j = 0; j < SORT_IPT; j++) {
    if (sp.start + (uint32_t)j * SORT_CTA + tid >= sp.end) break;
    const uint32_t pos = local ? sort_add(&s[it[j].key & fmask], 1u) : sort_add(&A.cursor[it[j].key], 1u);
    A.entries[pos] = it[j].val;
  }
}

}  // namespace b200
