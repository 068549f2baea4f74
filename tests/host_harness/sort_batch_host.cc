// Test harness (NOT part of libb200g16): the batch form (BATCH = true) of the MSM's two-level counting sort
// (gnark_whir_b200/csrc/msm_sort.cuh), compiled for the host with g++ and run CTA by CTA in a shuffled order as
// sort_host.cc runs the single-vector form: k scalar vectors of n points, row j at scalars + j * ld.  The sorted state
// is compared with a direct counting sort of the vector-major keys j * vstride + (single-vector key of point i of row
// j): counts, offsets, task_off and the multiset of entries of every bucket.  Every slot of the canonical scratch, the
// intermediate array and the entry array must be written exactly once, and nothing past their ends.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "msm_sort.cuh"

using namespace b200;

namespace {
struct Lcg {
  uint64_t s;
  uint32_t next() { s = s * 6364136223846793005ull + 1442695040888963407ull; return (uint32_t)(s >> 33); }
};

constexpr uint32_t GUARD = 64;          // words past the end of part / entries that must stay untouched
constexpr uint32_t JUNK = 0xdeadbeefu;  // shared memory starts out as junk: a missing init shows up

std::vector<uint32_t> shuffled(uint32_t n, Lcg& rng) {
  std::vector<uint32_t> v(n);
  for (uint32_t i = 0; i < n; i++) v[i] = i;
  for (uint32_t i = n; i > 1; i--) std::swap(v[i - 1], v[rng.next() % i]);
  return v;
}
}  // namespace

extern "C" {
// scalars: k rows of ld x 8 words (the first n of each row are the vector), Montgomery form.  Table mode (table != 0):
// one bucket set per vector, entries index rows of ent_stride points from ent_off.  stats[0..4] = F, bins, tiles,
// entries, largest bin.  Returns 0 when everything matches.
int sort_batch_host(const uint32_t* scalars, uint32_t n, uint32_t k, uint32_t ld, int c, int W, int table,
                    uint32_t ent_stride, uint32_t ent_off, uint64_t seed, uint32_t* stats) {
  Lcg rng{seed * 2 + 1};
  const uint32_t nbw = 1u << (c - 1), vstride = table ? nbw : nbw * (uint32_t)W, nb = vstride * k;
  const uint32_t np = n * k;   // points of all vectors
  const size_t m = (size_t)np * W;
  SortArgs A;
  memset(&A, 0, sizeof(A));
  A.scalars = reinterpret_cast<const Fr*>(scalars);
  A.n = np; A.c = c; A.W = W;
  A.vn = n; A.ld = ld; A.vstride = vstride;
  A.bstride = table ? 0u : nbw;
  A.ent_stride = table ? ent_stride : 0u;
  A.ent_off = table ? ent_off : 0u;
  A.F = sort_fine_bits(nb);
  A.nbins = sort_num_bins(nb, A.F);
  A.part_points = sort_part_points(W);
  if (A.nbins > SORT_BINS || A.nbins << A.F < nb) return 1;
  const size_t max_tiles = sort_max_tiles(A.nbins, m);
  std::vector<uint32_t> bins((sort_bin_bytes(A.nbins, m) + 3) / 4, JUNK);
  std::vector<SortItem> part(m + GUARD, SortItem{JUNK, JUNK});
  std::vector<Fr> canon(np + GUARD);
  for (auto& f : canon) for (auto& l : f.l) l = JUNK;
  A.canon = canon.data();
  std::vector<uint32_t> counts(nb, JUNK), cursor(nb, JUNK), entries(m + GUARD, JUNK), totals(16, 0);
  A.bin_count = bins.data();
  A.bin_cursor = bins.data() + SORT_BINS;
  A.bin_off = bins.data() + 2 * SORT_BINS;
  A.ntiles = bins.data() + 3 * SORT_BINS + 1;
  A.tiles = reinterpret_cast<SortTile*>(bins.data() + SORT_BIN_WORDS);
  A.part = part.data(); A.counts = counts.data(); A.cursor = cursor.data(); A.entries = entries.data();
  A.totals = totals.data();
  std::vector<uint32_t> s(std::max<uint32_t>(SORT_BINS + 1, 1u << SORT_FINE_MAX_BITS));
  const uint32_t ctas = (np + SORT_POINTS - 1) / SORT_POINTS;

  // pass 1 (the library zeroes bin_count first)
  std::fill(A.bin_count, A.bin_count + SORT_BINS, 0u);
  for (uint32_t blk : shuffled(ctas, rng)) {
    std::fill(s.begin(), s.end(), JUNK);
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_coarse_init(A, t, s.data());
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_coarse_count<true>(A, blk, t, s.data());
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_coarse_flush(A, t, s.data());
  }
  for (uint32_t q = np; q < np + GUARD; q++)   // the canonical scratch ends at the last point
    for (auto l : canon[q].l) if (l != JUNK) return 18;
  const uint32_t E = totals[3];
  // pass 2: the kernel's exclusive scan between load and write, done directly
  std::vector<uint32_t> sa(SORT_BINS + 1, JUNK), sb(SORT_BINS + 1, JUNK);
  for (uint32_t t = 0; t < SORT_CTA; t++) sort_bins_load(A, t, sa.data(), sb.data());
  uint32_t ea = 0, eb = 0;
  for (uint32_t b = 0; b <= SORT_BINS; b++) {
    const uint32_t va = b < SORT_BINS ? sa[b] : 0, vb = b < SORT_BINS ? sb[b] : 0;
    sa[b] = ea; sb[b] = eb; ea += va; eb += vb;
  }
  for (uint32_t t = 0; t < SORT_CTA; t++) sort_bins_write(A, t, sa.data(), sb.data());
  const uint32_t ntiles = *A.ntiles;
  if (ntiles > max_tiles) return 2;
  if (A.bin_off[A.nbins] != E || E > m) return 3;
  // tiles: consecutive, inside one bin each, at most SORT_TILE entries, covering [0, E)
  uint32_t next = 0, largest = 0;
  for (uint32_t b = 0; b < A.nbins; b++) largest = std::max(largest, A.bin_off[b + 1] - A.bin_off[b]);
  for (uint32_t t = 0; t < ntiles; t++) {
    const SortSpan sp = sort_tile_span(A, t);
    if (sp.bin >= A.nbins || sp.start != next || sp.end <= sp.start || sp.end - sp.start > SORT_TILE) return 4;
    if (sp.start < A.bin_off[sp.bin] || sp.end > A.bin_off[sp.bin + 1]) return 5;
    next = sp.end;
  }
  if (next != E) return 6;
  // pass 3: the kernel's exclusive scan after the count step, done directly
  std::vector<uint32_t> loc(SORT_BINS), glob(SORT_BINS);
  std::vector<SortItem> stage(SORT_STAGE);
  for (uint32_t blk : shuffled((np + A.part_points - 1) / A.part_points, rng)) {
    std::fill(s.begin(), s.end(), JUNK);
    std::fill(loc.begin(), loc.end(), JUNK);
    std::fill(glob.begin(), glob.end(), JUNK);
    std::fill(stage.begin(), stage.end(), SortItem{JUNK, JUNK});
    std::fill(s.begin(), s.begin() + SORT_BINS, 0u);
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_part_count<true>(A, blk, t, s.data());
    uint32_t e = 0;
    for (uint32_t b = 0; b <= SORT_BINS; b++) {
      const uint32_t v = b < SORT_BINS ? s[b] : 0;
      s[b] = e;
      e += v;
    }
    if (e > SORT_STAGE) return 17;
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_part_reserve(A, t, s.data(), loc.data(), glob.data());
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_part_stage<true>(A, blk, t, s.data(), stage.data());
    for (uint32_t t = 0; t < SORT_CTA; t++) sort_part_write(A, t, s[SORT_BINS], loc.data(), glob.data(), stage.data());
  }
  for (uint32_t b = 0; b < A.nbins; b++)
    if (A.bin_cursor[b] != A.bin_off[b + 1]) return 7;
  for (size_t k = 0; k < m + GUARD; k++) {
    const bool written = part[k].key != JUNK || part[k].val != JUNK;
    if (written != (k < E)) return 8;
    if (k < E && (part[k].key >> A.F) >= A.nbins) return 9;
  }
  for (uint32_t b = 0; b < A.nbins; b++)   // every item sits in its own bin's range
    for (uint32_t k = A.bin_off[b]; k < A.bin_off[b + 1]; k++)
      if ((part[k].key >> A.F) != b) return 10;
  // pass 4 (the library zeroes counts first)
  std::fill(counts.begin(), counts.end(), 0u);
  for (uint32_t t : shuffled(ntiles, rng)) {
    const SortSpan sp = sort_tile_span(A, t);
    std::fill(s.begin(), s.end(), JUNK);
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_init(A, tid, s.data());
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_count(A, sp, tid, s.data(), true);
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_flush(A, sp, tid, s.data());
  }
  // k_pick_seg / k_scan_* (unchanged kernels), restated: offsets, cursor, task_off
  const uint32_t target = 148u * 2048u;
  const uint32_t sa_ = 2u * (E / nb) + 2u, sb_ = E / target + 1u;
  uint32_t seg = (nb >= target / 2 && sa_ > sb_) ? sa_ : sb_;
  seg = seg < 32u ? 32u : seg;
  std::vector<uint32_t> offsets(nb), task_off(nb);
  uint32_t o = 0, to = 0;
  for (uint32_t b = 0; b < nb; b++) {
    offsets[b] = o; cursor[b] = o; task_off[b] = to;
    o += counts[b]; to += (counts[b] + seg - 1) / seg;
  }
  if (o != E) return 11;
  // pass 6
  for (uint32_t t : shuffled(ntiles, rng)) {
    const SortSpan sp = sort_tile_span(A, t);
    std::fill(s.begin(), s.end(), JUNK);
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_init(A, tid, s.data());
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_count(A, sp, tid, s.data(), false);
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_reserve(A, sp, tid, s.data());
    for (uint32_t tid = 0; tid < SORT_CTA; tid++) sort_fine_place(A, sp, tid, s.data());
  }
  for (size_t k = E; k < m + GUARD; k++)
    if (entries[k] != JUNK) return 12;

  // direct counting sort of the same entries: the single-vector keys of row j, shifted into vector j's bucket sets
  std::vector<uint32_t> want_counts(nb, 0);
  std::vector<uint64_t> keyed;   // bucket << 32 | value
  keyed.reserve(E);
  for (uint32_t j = 0; j < k; j++)
    for (uint32_t i = 0; i < n; i++)
      sort_entries(A, Fr::from_mont(A.scalars[(size_t)j * ld + i]), i, [&](uint32_t key, uint32_t val) {
        const uint32_t vk = j * vstride + key;
        want_counts[vk]++;
        keyed.push_back((uint64_t)vk << 32 | val);
      });
  if (keyed.size() != E) return 13;
  std::sort(keyed.begin(), keyed.end());
  uint32_t wo = 0, wto = 0;
  for (uint32_t b = 0; b < nb; b++) {
    if (counts[b] != want_counts[b] || offsets[b] != wo || task_off[b] != wto) return 14;
    if (cursor[b] != offsets[b] + counts[b]) return 15;
    std::vector<uint32_t> got(entries.begin() + offsets[b], entries.begin() + offsets[b] + counts[b]);
    std::sort(got.begin(), got.end());
    for (uint32_t k = 0; k < counts[b]; k++)
      if (got[k] != (uint32_t)keyed[wo + k] || (keyed[wo + k] >> 32) != b) return 16;
    wo += want_counts[b];
    wto += (want_counts[b] + seg - 1) / seg;
  }
  stats[0] = (uint32_t)A.F; stats[1] = A.nbins; stats[2] = ntiles; stats[3] = E; stats[4] = largest;
  return 0;
}
}
