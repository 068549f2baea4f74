// Groth16 Setup on the GPU: constraint matrices + toxic waste -> the resident proving key.
//
// Replaces gnark v0.11.0 backend/groth16/bn254/setup.go Setup (reached from the reference at mt.go:448): setupABC,
// the K and Z scalar vectors, the infinity filtering and the BatchScalarMultiplicationG1 / G2 calls.  Everything
// runs on ctx->stream:
//   1. p_k = tau^k for k < N (build_geometric)
//   2. Lagrange values L_j(tau) = (1/N) sum_k tau^k w^-jk, i.e. FFTInverse(p): one inverse DIF NTT of a copy of p,
//      which leaves L_j(tau) at position bitrev(j).  These are the same field elements gnark's recurrence with its N
//      batch-inverted denominators produces.
//   3. Z scalars (tau^N - 1) / delta * p[bitrev(i)]
//   4. per matrix L, R, O: count terms per wire (warp-aggregated atomics: wire 0 sits in a large share of the rows),
//      scan, scatter c * L_row(tau) into wire order, segmented reduction (segments longer than SEG_CHUNK are cut
//      into chunks whose partial sums are reduced again, level after level, so one hot wire never runs on one
//      thread).  The scatter order inside a segment depends on atomics, but field addition is exact and
//      commutative: every A_i(tau), B_i(tau), C_i(tau) is the same field element whatever the order, so the
//      output is deterministic.
//   5. K values, per-wire classes and flags, compaction by prefix sums into the scalar vectors
//   6. fixed-base multiples (fixed_base.cu) into new bases handles, one window table per group
// The scratch is the call's own and is released on return.
#include <algorithm>

#include "prove.cuh"
#include "host_copy.cuh"

namespace b200 {
namespace {

constexpr int ST = 256;                  // threads per CTA of the element-wise kernels
constexpr uint32_t SEG_CHUNK = 64;       // terms one thread adds in the segmented reduction
constexpr int SCAN_T = 512, SCAN_ITEMS = 4;
constexpr size_t SCAN_TILE = (size_t)SCAN_T * SCAN_ITEMS;
constexpr uint32_t NONE = 0xffffffffu;
constexpr uint64_t NNZ_MAX = 0xf0000000ull;   // chunk counts of the reduction stay below 2^32

inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }
__device__ __forceinline__ size_t gtid() { return (size_t)blockIdx.x * blockDim.x + threadIdx.x; }
__device__ __forceinline__ uint32_t brev(uint32_t i, int L) { return L ? __brev(i) >> (32 - L) : 0; }

// Every lane of the warp calls this.  Lanes with the same key share one atomicAdd of their count on ctr[key]; each
// gets the old value plus its rank among them.  Invalid lanes take no part.
__device__ __forceinline__ uint32_t warp_agg_inc(uint32_t* ctr, uint32_t key, bool valid) {
  const uint32_t peers = __match_any_sync(0xffffffffu, valid ? key : NONE);
  const int leader = __ffs(peers) - 1;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t base = 0;
  if (valid && (int)lane == leader) base = atomicAdd(ctr + key, (uint32_t)__popc(peers));
  base = __shfl_sync(0xffffffffu, base, leader);
  return base + __popc(peers & ((1u << lane) - 1));
}

// ---- checks of the index arrays (flag bit 0: a row array decreases, bit 1: a wire or coefficient id out of range)
__global__ void __launch_bounds__(ST) k_setup_check_rows(const uint64_t* __restrict__ row, uint32_t m,
                                                         uint32_t* flag) {
  const size_t j = gtid();
  if (j < m && row[j] > row[j + 1]) atomicOr(flag, 1u);
}

__global__ void __launch_bounds__(ST) k_setup_check_terms(const uint32_t* __restrict__ wire,
                                                          const uint32_t* __restrict__ cid, uint32_t nnz, uint32_t nw,
                                                          uint32_t nc, uint32_t* flag) {
  const size_t e = gtid();
  if (e < nnz && (wire[e] >= nw || cid[e] >= nc)) atomicOr(flag, 2u);
}

// ---- exclusive scan of uint32 (in place): tiles of SCAN_TILE, tile totals scanned recursively
__global__ void __launch_bounds__(SCAN_T) k_setup_scan_tile(uint32_t* __restrict__ x, size_t n,
                                                            uint32_t* __restrict__ sums) {
  constexpr int NW = SCAN_T / 32;
  __shared__ uint32_t warp_off[NW];
  const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    v[k] = base + k < n ? x[base + k] : 0;
    s += v[k];
  }
  uint32_t inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += t;
  }
  if (lane == 31) warp_off[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const uint32_t t0 = lane < NW ? warp_off[lane] : 0;
    uint32_t w = t0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= (uint32_t)o) w += t;
    }
    if (lane < NW) warp_off[lane] = w - t0;
    if (lane == 31) sums[blockIdx.x] = w;
  }
  __syncthreads();
  uint32_t run = warp_off[warp] + inc - s;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    if (base + k < n) x[base + k] = run;
    run += v[k];
  }
}

__global__ void __launch_bounds__(SCAN_T) k_setup_scan_add(uint32_t* __restrict__ x, size_t n,
                                                           const uint32_t* __restrict__ sums) {
  if (blockIdx.x == 0) return;
  const uint32_t add = sums[blockIdx.x];
  const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++)
    if (base + k < n) x[base + k] += add;
}

// ---- per-wire accumulation of one matrix
__global__ void __launch_bounds__(ST) k_setup_count(const uint32_t* __restrict__ wire, uint32_t nnz,
                                                    uint32_t* __restrict__ cnt) {
  const size_t e = gtid();
  const bool v = e < nnz;
  warp_agg_inc(cnt, v ? wire[e] : 0, v);
}

// longest segment of offs (n segments)
__global__ void __launch_bounds__(ST) k_setup_max_len(const uint32_t* __restrict__ offs, uint32_t n,
                                                      uint32_t* out) {
  const size_t w = gtid();
  uint32_t len = w < n ? offs[w + 1] - offs[w] : 0;
#pragma unroll
  for (int o = 16; o; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
  if ((threadIdx.x & 31) == 0 && len) atomicMax(out, len);
}

// vals[offs[w] + slot] = coeff * L_row(tau) for every term of wire w.  The row of entry e is found by binary search
// over the row array, so the cost does not depend on row lengths (one row may hold 2^16 terms, many rows none).
__global__ void __launch_bounds__(ST) k_setup_scatter(const uint64_t* __restrict__ row, uint32_t m,
                                                      const uint32_t* __restrict__ wire,
                                                      const uint32_t* __restrict__ cid, uint32_t nnz,
                                                      const Fr* __restrict__ coeffs, const Fr* __restrict__ lag,
                                                      int L, const uint32_t* __restrict__ offs,
                                                      uint32_t* __restrict__ cursor, Fr* __restrict__ vals) {
  const size_t e = gtid();
  const bool v = e < nnz;
  const uint32_t w = v ? wire[e] : 0;
  const uint32_t slot = warp_agg_inc(cursor, w, v);
  if (!v) return;
  uint32_t lo = 0, hi = m;   // row[lo] <= e < row[hi]  (row[0] = 0, row[m] = nnz)
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (row[mid] <= e) lo = mid;
    else hi = mid;
  }
  vals[offs[w] + slot] = Fr::mul(coeffs[cid[e]], lag[brev(lo, L)]);
}

// nch[w] = chunks of segment w (nch[n] = 0: the scan leaves the total there)
__global__ void __launch_bounds__(ST) k_setup_chunk_count(const uint32_t* __restrict__ offs, uint32_t n,
                                                          uint32_t* __restrict__ nch) {
  const size_t w = gtid();
  if (w < n) nch[w] = (offs[w + 1] - offs[w] + SEG_CHUNK - 1) / SEG_CHUNK;
  else if (w == n) nch[n] = 0;
}

// part[t] = sum of chunk t (chunk j of segment w covers vals[offs[w] + j SEG_CHUNK, ...) inside the segment)
__global__ void __launch_bounds__(ST) k_setup_chunk_sum(const Fr* __restrict__ vals, const uint32_t* __restrict__ offs,
                                                        const uint32_t* __restrict__ choffs, uint32_t n,
                                                        Fr* __restrict__ part) {
  const size_t t = gtid();
  if (t >= choffs[n]) return;
  uint32_t lo = 0, hi = n;   // choffs[lo] <= t < choffs[hi]
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (choffs[mid] <= t) lo = mid;
    else hi = mid;
  }
  const uint32_t b = offs[lo] + ((uint32_t)t - choffs[lo]) * SEG_CHUNK;
  const uint32_t e = min(b + SEG_CHUNK, offs[lo + 1]);
  Fr acc = Fr::zero();
  for (uint32_t i = b; i < e; i++) acc = Fr::add(acc, vals[i]);
  part[t] = acc;
}

// out[w] = sum of segment w (at most SEG_CHUNK terms by now)
__global__ void __launch_bounds__(ST) k_setup_seg_sum(const Fr* __restrict__ vals, const uint32_t* __restrict__ offs,
                                                      uint32_t n, Fr* __restrict__ out) {
  const size_t w = gtid();
  if (w >= n) return;
  Fr acc = Fr::zero();
  for (uint32_t i = offs[w], e = offs[w + 1]; i < e; i++) acc = Fr::add(acc, vals[i]);
  out[w] = acc;
}

// ---- classes, K values, compaction
struct WireClass {
  uint32_t nw, n_pub;
  int64_t cw;                 // commitment wire or -1
  const uint32_t* ped_pos;    // ped_pos[w] = position in the committed list, NONE otherwise
};

__global__ void __launch_bounds__(ST) k_setup_ped_pos(const uint32_t* __restrict__ list, uint32_t n,
                                                      uint32_t* __restrict__ ped_pos) {
  const size_t i = gtid();
  if (i < n) ped_pos[list[i]] = (uint32_t)i;
}

__device__ __forceinline__ bool in_k(const WireClass& c, uint32_t w) {
  return w >= c.n_pub && (int64_t)w != c.cw && c.ped_pos[w] == NONE;
}

// flags (host layout: 1 = dropped / skipped) and the 0/1 keep indicators the compaction scans (entry nw = 0)
__global__ void __launch_bounds__(ST) k_setup_flags(const Fr* __restrict__ A, const Fr* __restrict__ B, WireClass c,
                                                    uint8_t* __restrict__ inf_a, uint8_t* __restrict__ inf_b,
                                                    uint8_t* __restrict__ k_skip, uint32_t* __restrict__ fa,
                                                    uint32_t* __restrict__ fb, uint32_t* __restrict__ fk) {
  const size_t w = gtid();
  if (w > c.nw) return;
  if (w == c.nw) {
    fa[w] = fb[w] = fk[w] = 0;
    return;
  }
  const bool za = A[w].is_zero(), zb = B[w].is_zero(), k = in_k(c, (uint32_t)w);
  inf_a[w] = za;
  inf_b[w] = zb;
  k_skip[w] = !k;
  fa[w] = !za;
  fb[w] = !zb;
  fk[w] = k;
}

struct ToxicFr {
  Fr alpha, beta, gamma_inv, delta_inv, sigma;
};

// Scalar vectors in gnark's orders: A, B (nonzero entries), pk.K (K_i / delta), vk.K (public wires, then the
// commitment wire; K_i / gamma), Pedersen basis (committed list order; K_i / gamma) and sigma times it.
__global__ void __launch_bounds__(ST) k_setup_compact(const Fr* __restrict__ A, const Fr* __restrict__ B,
                                                      const Fr* __restrict__ C, WireClass c, ToxicFr t,
                                                      const uint32_t* __restrict__ fa, const uint32_t* __restrict__ fb,
                                                      const uint32_t* __restrict__ fk, Fr* __restrict__ sa,
                                                      Fr* __restrict__ sb, Fr* __restrict__ sk, Fr* __restrict__ svk,
                                                      Fr* __restrict__ sped, Fr* __restrict__ sped_sigma) {
  const size_t i = gtid();
  if (i >= c.nw) return;
  const uint32_t w = (uint32_t)i;
  const Fr a = A[w], b = B[w];
  if (!a.is_zero()) sa[fa[w]] = a;
  if (!b.is_zero()) sb[fb[w]] = b;
  const Fr k = Fr::add(Fr::add(Fr::mul(t.beta, a), Fr::mul(t.alpha, b)), C[w]);
  if (w < c.n_pub) {
    svk[w] = Fr::mul(k, t.gamma_inv);
  } else if ((int64_t)w == c.cw) {
    svk[c.n_pub] = Fr::mul(k, t.gamma_inv);
  } else if (c.ped_pos[w] != NONE) {
    const Fr p = Fr::mul(k, t.gamma_inv);
    sped[c.ped_pos[w]] = p;
    sped_sigma[c.ped_pos[w]] = Fr::mul(p, t.sigma);
  } else {
    sk[fk[w]] = Fr::mul(k, t.delta_inv);
  }
}

// z[i] = (tau^N - 1) / delta * tau^bitrev(i), i < N - 1
__global__ void __launch_bounds__(ST) k_setup_z(const Fr* __restrict__ p, uint32_t n, int L, Fr zc,
                                                Fr* __restrict__ z) {
  const size_t i = gtid();
  if (i < n) z[i] = Fr::mul(zc, p[brev((uint32_t)i, L)]);
}

// ------------------------------------------------------------------------------------------------ host side
// The call's own device scratch, released when it goes out of scope (every return path).
struct Scratch {
  enum {
    COEFFS, ROW0, WIRE0 = ROW0 + 3, CID0 = WIRE0 + 3, FLAG = CID0 + 3, P, LAG, CNT, CUR, VALS, PART0, PART1, CHO0, CHO1,
    SCAN, ABC, PED_POS, FA, FB, FK, FLAGS8, SCAL, TAB1, TAB2, SMALL, COUNT
  };
  DevBuf b[COUNT];
  ~Scratch() {
    for (auto& x : b) x.release();
  }
  template <class T>
  T* get(int i) const { return b[i].as<T>(); }
};

int scan_exclusive(b200g16_ctx* ctx, uint32_t* x, size_t n, uint32_t* scratch) {
  if (n == 0) return 0;
  const unsigned nb = cdiv(n, SCAN_TILE);
  k_setup_scan_tile<<<nb, SCAN_T, 0, ctx->stream>>>(x, n, scratch);
  ctx->launches++;
  if (nb > 1) {
    B200_TRY(scan_exclusive(ctx, scratch, nb, scratch + nb));
    k_setup_scan_add<<<nb, SCAN_T, 0, ctx->stream>>>(x, n, scratch);
    ctx->launches++;
  }
  B200_CUDA(cudaGetLastError());
  return 0;
}

size_t scan_scratch_words(size_t n) { return 2 * (n / SCAN_TILE) + 64; }

struct Shape {
  uint32_t m, nw, n_pub, nc;
  int L;
  uint64_t nnz[3];
  const uint64_t* row[3];
  const uint32_t* wire[3];
  const uint32_t* cid[3];
};

int check_desc(const b200g16_r1cs_desc* r, Shape* s) {
  if (!r) return fail(B200G16_ERR_ARG, "setup: null r1cs");
  if (r->n_constraints == 0) return fail(B200G16_ERR_ARG, "setup: no constraints");
  if (r->n_constraints > ((size_t)1 << 28))
    return fail(B200G16_ERR_ARG, "setup: %zu constraints exceed the 2^28 domain", r->n_constraints);
  if (r->n_wires >= ((size_t)1 << 32)) return fail(B200G16_ERR_ARG, "setup: n_wires=%zu >= 2^32", r->n_wires);
  if (r->n_public == 0 || r->n_public > r->n_wires)
    return fail(B200G16_ERR_ARG, "setup: n_public=%zu outside [1, n_wires=%zu]", r->n_public, r->n_wires);
  if (r->n_coeffs >= ((size_t)1 << 32)) return fail(B200G16_ERR_ARG, "setup: n_coeffs >= 2^32");
  if (r->n_coeffs && !r->coeffs) return fail(B200G16_ERR_ARG, "setup: null coefficient table");
  s->m = (uint32_t)r->n_constraints;
  s->nw = (uint32_t)r->n_wires;
  s->n_pub = (uint32_t)r->n_public;
  s->nc = (uint32_t)r->n_coeffs;
  s->L = 0;
  while (((size_t)1 << s->L) < r->n_constraints) s->L++;
  const uint64_t* rows[3] = {r->l_row, r->r_row, r->o_row};
  const uint32_t* wires[3] = {r->l_wire, r->r_wire, r->o_wire};
  const uint32_t* cids[3] = {r->l_coeff, r->r_coeff, r->o_coeff};
  for (int k = 0; k < 3; k++) {
    const char* nm = "LRO" + k;
    if (!rows[k]) return fail(B200G16_ERR_ARG, "setup: null %.1s row array", nm);
    if (rows[k][0] != 0) return fail(B200G16_ERR_ARG, "setup: %.1s row[0] = %llu, not 0", nm, (unsigned long long)rows[k][0]);
    const uint64_t nnz = rows[k][s->m];
    if (nnz > NNZ_MAX) return fail(B200G16_ERR_ARG, "setup: %.1s has %llu terms (at most 15 * 2^28)", nm, (unsigned long long)nnz);
    if (nnz && (!wires[k] || !cids[k])) return fail(B200G16_ERR_ARG, "setup: null %.1s term arrays", nm);
    s->nnz[k] = nnz;
    s->row[k] = rows[k];
    s->wire[k] = wires[k];
    s->cid[k] = cids[k];
  }
  // the BSB22 commitment: one at most
  const int64_t cw = r->commitment_wire;
  if (cw < 0) {
    if (cw != -1 || r->n_private_committed)
      return fail(B200G16_ERR_ARG, "setup: committed wires without a commitment wire (or commitment_wire < -1)");
  } else {
    if ((uint64_t)cw < r->n_public || (uint64_t)cw >= r->n_wires)
      return fail(B200G16_ERR_ARG, "setup: commitment wire %lld outside [n_public, n_wires)", (long long)cw);
    if (r->n_private_committed && !r->private_committed) return fail(B200G16_ERR_ARG, "setup: null committed list");
    if (r->n_private_committed > r->n_wires) return fail(B200G16_ERR_ARG, "setup: committed list too long");
    for (size_t i = 0; i < r->n_private_committed; i++) {
      const uint32_t w = r->private_committed[i];
      if (w < r->n_public || w >= r->n_wires || (int64_t)w == cw || (i && w <= r->private_committed[i - 1]))
        return fail(B200G16_ERR_ARG,
                    "setup: committed wire %u (entry %zu) is public, out of range, the commitment wire or out of order",
                    w, i);
    }
  }
  return 0;
}

// Steps 1, 2 and 4: uploads, checks, tau powers (left in P), Lagrange values, A / B / C (n_wires each, in ABC).
// ev_io: next ctx->ev slot; records one event per phase.
int setup_front(b200g16_ctx* ctx, const b200g16_r1cs_desc* r, const Shape& s, const Fr& tau, Scratch& S, int* ev_io) {
  cudaStream_t st = ctx->stream;
  int ev = *ev_io;
  const size_t N = (size_t)1 << s.L;
  uint64_t nnz_max = 0;
  for (int k = 0; k < 3; k++) nnz_max = std::max(nnz_max, s.nnz[k]);
  // ---- uploads + checks
  B200_TRY(S.b[Scratch::COEFFS].ensure(std::max<size_t>(s.nc, 1) * sizeof(Fr)));
  B200_TRY(h2d_copy(ctx, S.b[Scratch::COEFFS].p, r->coeffs, (size_t)s.nc * sizeof(Fr), st));
  B200_TRY(S.b[Scratch::FLAG].ensure(16));
  B200_CUDA(cudaMemsetAsync(S.b[Scratch::FLAG].p, 0, 16, st));
  uint32_t* flag = S.get<uint32_t>(Scratch::FLAG);
  for (int k = 0; k < 3; k++) {
    DevBuf &row = S.b[Scratch::ROW0 + k], &wire = S.b[Scratch::WIRE0 + k], &cid = S.b[Scratch::CID0 + k];
    B200_TRY(row.ensure(((size_t)s.m + 1) * sizeof(uint64_t)));
    B200_TRY(wire.ensure(std::max<uint64_t>(s.nnz[k], 1) * sizeof(uint32_t)));
    B200_TRY(cid.ensure(std::max<uint64_t>(s.nnz[k], 1) * sizeof(uint32_t)));
    B200_TRY(h2d_copy(ctx, row.p, s.row[k], ((size_t)s.m + 1) * sizeof(uint64_t), st));
    B200_TRY(h2d_copy(ctx, wire.p, s.wire[k], s.nnz[k] * sizeof(uint32_t), st));
    B200_TRY(h2d_copy(ctx, cid.p, s.cid[k], s.nnz[k] * sizeof(uint32_t), st));
    k_setup_check_rows<<<cdiv(s.m, ST), ST, 0, st>>>(row.as<uint64_t>(), s.m, flag);
    if (s.nnz[k])
      k_setup_check_terms<<<cdiv(s.nnz[k], ST), ST, 0, st>>>(wire.as<uint32_t>(), cid.as<uint32_t>(), (uint32_t)s.nnz[k],
                                                             s.nw, s.nc, flag);
    ctx->launches += s.nnz[k] ? 2 : 1;
  }
  B200_CUDA(cudaGetLastError());
  uint32_t hflag = 0;
  B200_CUDA(cudaMemcpyAsync(&hflag, flag, sizeof(hflag), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  if (hflag & 1) return fail(B200G16_ERR_ARG, "setup: a row array decreases");
  if (hflag & 2) return fail(B200G16_ERR_ARG, "setup: a wire >= n_wires or a coefficient id >= n_coeffs");
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  // ---- tau powers and Lagrange values
  B200_TRY(S.b[Scratch::P].ensure(N * sizeof(Fr)));
  B200_TRY(S.b[Scratch::LAG].ensure(N * sizeof(Fr)));
  B200_TRY(build_geometric(ctx, S.get<Fr>(Scratch::P), N, Fr::one(), tau));
  B200_CUDA(cudaMemcpyAsync(S.b[Scratch::LAG].p, S.b[Scratch::P].p, N * sizeof(Fr), cudaMemcpyDeviceToDevice, st));
  B200_TRY(ntt_device(ctx, S.get<Fr>(Scratch::LAG), s.L, 1, true, false, B200G16_DIF));
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  // ---- per-wire accumulation of L, R, O
  const size_t nw = s.nw;
  const size_t part_cap = nnz_max / SEG_CHUNK + nw + 1;
  B200_TRY(S.b[Scratch::CNT].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::CUR].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::CHO0].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::CHO1].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::VALS].ensure(std::max<uint64_t>(nnz_max, 1) * sizeof(Fr)));
  B200_TRY(S.b[Scratch::PART0].ensure(part_cap * sizeof(Fr)));
  B200_TRY(S.b[Scratch::PART1].ensure(part_cap * sizeof(Fr)));
  B200_TRY(S.b[Scratch::SCAN].ensure(scan_scratch_words(nw + 1) * sizeof(uint32_t) + 16));
  B200_TRY(S.b[Scratch::ABC].ensure(3 * std::max<size_t>(nw, 1) * sizeof(Fr)));
  uint32_t* scan_tmp = S.get<uint32_t>(Scratch::SCAN);
  uint32_t* d_maxlen = flag + 1;
  const unsigned gw = cdiv(nw + 1, ST);
  for (int k = 0; k < 3; k++) {
    Fr* out = S.get<Fr>(Scratch::ABC) + (size_t)k * nw;
    uint32_t* offs = S.get<uint32_t>(Scratch::CNT);
    uint32_t* cur = S.get<uint32_t>(Scratch::CUR);
    const uint32_t nnz = (uint32_t)s.nnz[k];
    B200_CUDA(cudaMemsetAsync(offs, 0, (nw + 1) * sizeof(uint32_t), st));
    B200_CUDA(cudaMemsetAsync(cur, 0, (nw + 1) * sizeof(uint32_t), st));
    B200_CUDA(cudaMemsetAsync(d_maxlen, 0, sizeof(uint32_t), st));
    if (nnz) {
      k_setup_count<<<cdiv(nnz, ST), ST, 0, st>>>(S.get<uint32_t>(Scratch::WIRE0 + k), nnz, offs);
      ctx->launches++;
    }
    B200_TRY(scan_exclusive(ctx, offs, nw + 1, scan_tmp));
    if (nnz) {
      k_setup_scatter<<<cdiv(nnz, ST), ST, 0, st>>>(S.get<uint64_t>(Scratch::ROW0 + k), s.m,
                                                    S.get<uint32_t>(Scratch::WIRE0 + k),
                                                    S.get<uint32_t>(Scratch::CID0 + k), nnz, S.get<Fr>(Scratch::COEFFS),
                                                    S.get<Fr>(Scratch::LAG), s.L, offs, cur, S.get<Fr>(Scratch::VALS));
      k_setup_max_len<<<gw, ST, 0, st>>>(offs, (uint32_t)nw, d_maxlen);
      ctx->launches += 2;
    }
    B200_CUDA(cudaGetLastError());
    uint32_t maxlen = 0;
    B200_CUDA(cudaMemcpyAsync(&maxlen, d_maxlen, sizeof(maxlen), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    // reduce chunks of SEG_CHUNK terms until every segment fits one thread
    const Fr* vals = S.get<Fr>(Scratch::VALS);
    const uint32_t* seg = offs;
    size_t bound = nnz;   // entries of the current level, at most
    for (int lvl = 0; maxlen > SEG_CHUNK; lvl++) {
      uint32_t* cho = S.get<uint32_t>(lvl & 1 ? Scratch::CHO1 : Scratch::CHO0);
      Fr* part = S.get<Fr>(lvl & 1 ? Scratch::PART1 : Scratch::PART0);
      k_setup_chunk_count<<<gw, ST, 0, st>>>(seg, (uint32_t)nw, cho);
      ctx->launches++;
      B200_TRY(scan_exclusive(ctx, cho, nw + 1, scan_tmp));
      bound = bound / SEG_CHUNK + nw;
      k_setup_chunk_sum<<<cdiv(bound, ST), ST, 0, st>>>(vals, seg, cho, (uint32_t)nw, part);
      ctx->launches++;
      B200_CUDA(cudaGetLastError());
      vals = part;
      seg = cho;
      maxlen = (maxlen + SEG_CHUNK - 1) / SEG_CHUNK;
    }
    k_setup_seg_sum<<<cdiv(nw, ST), ST, 0, st>>>(vals, seg, (uint32_t)nw, out);
    ctx->launches++;
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  }
  *ev_io = ev;
  return 0;
}

Fr fr_of(const uint64_t* v) {
  Fr r;
  memcpy(&r, v, sizeof(r));
  return r;
}

int new_bases(int group, size_t n, int device, b200g16_bases** out) {
  b200g16_bases* h = new b200g16_bases();
  h->group = group;
  h->n = n;
  h->device = device;
  cudaError_t e = cudaMalloc(&h->d_points, (n ? n : 1) * (group == 1 ? sizeof(G1Affine) : sizeof(G2Affine)));
  if (e != cudaSuccess) {
    delete h;
    return fail(B200G16_ERR_CUDA, "setup: %zu points: %s", n, cudaGetErrorString(e));
  }
  *out = h;
  return 0;
}

// G1 / G2 generators, Montgomery limbs
constexpr uint64_t G1_GEN_LIMBS[8] = {0xd35d438dc58f0d9dull, 0x0a78eb28f5c70b3dull, 0x666ea36f7879462cull,
                                      0x0e0a77c19a07df2full, 0xa6ba871b8b1e1b3aull, 0x14f1d651eb8e167bull,
                                      0xccdd46def0f28c58ull, 0x1c14ef83340fbe5eull};
constexpr uint64_t G2_GEN_LIMBS[16] = {
    0x8e83b5d102bc2026ull, 0xdceb1935497b0172ull, 0xfbb8264797811adfull, 0x19573841af96503bull,
    0xafb4737da84c6140ull, 0x6043dd5a5802d8c4ull, 0x09e950fc52a02f86ull, 0x14fef0833aea7b6bull,
    0x619dfa9d886be9f6ull, 0xfe7fd297f59e9b78ull, 0xff9e1a62231b7dfeull, 0x28fd7eebae9e4206ull,
    0x64095b56c71856eeull, 0xdc57f922327d3cbbull, 0x55f935be33351076ull, 0x0da4a0e693fd6482ull};

int setup_run(b200g16_ctx* ctx, const b200g16_r1cs_desc* r, const Shape& s, const b200g16_toxic* tw, uint8_t* inf_a,
              uint8_t* inf_b, uint8_t* k_skip, b200g16_setup_out* out, b200g16_bases** made) {
  cudaStream_t st = ctx->stream;
  const Fr tau = fr_of(tw->tau), gamma = fr_of(tw->gamma), delta = fr_of(tw->delta), sigma = fr_of(tw->sigma);
  if (gamma.is_zero() || delta.is_zero()) return fail(B200G16_ERR_ARG, "setup: gamma or delta is zero");
  Fr tau_n = tau;
  for (int i = 0; i < s.L; i++) tau_n = Fr::sqr(tau_n);
  if (tau_n == Fr::one()) return fail(B200G16_ERR_ARG, "setup: tau^N = 1 (tau lies in the evaluation domain)");
  ToxicFr t{fr_of(tw->alpha), fr_of(tw->beta), Fr::inv(gamma), Fr::inv(delta), sigma};
  const Fr zc = Fr::mul(Fr::sub(tau_n, Fr::one()), t.delta_inv);
  const size_t N = (size_t)1 << s.L, nw = s.nw;
  Scratch S;
  ctx->timings.n = 0;
  int ev = 0;
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  B200_TRY(setup_front(ctx, r, s, tau, S, &ev));
  // ---- K values, flags, compaction
  const size_t n_ped = r->commitment_wire >= 0 ? r->n_private_committed : 0;
  const size_t n_vk = s.n_pub + (r->commitment_wire >= 0 ? 1 : 0);
  B200_TRY(S.b[Scratch::PED_POS].ensure(std::max<size_t>(nw, 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::FA].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::FB].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::FK].ensure((nw + 1) * sizeof(uint32_t)));
  B200_TRY(S.b[Scratch::FLAGS8].ensure(3 * std::max<size_t>(nw, 1)));
  // scalar vectors: A, B, K (n_wires each at most), vk.K, Pedersen x 2, Z (N - 1), small G1 (3), small G2 (4)
  const size_t o_b = nw, o_k = 2 * nw, o_vk = 3 * nw, o_ped = o_vk + n_vk, o_peds = o_ped + n_ped, o_z = o_peds + n_ped,
               o_s1 = o_z + N, o_s2 = o_s1 + 3, n_scal = o_s2 + 4;
  B200_TRY(S.b[Scratch::SCAL].ensure(n_scal * sizeof(Fr)));
  Fr* sc = S.get<Fr>(Scratch::SCAL);
  uint32_t* ped_pos = S.get<uint32_t>(Scratch::PED_POS);
  B200_CUDA(cudaMemsetAsync(ped_pos, 0xff, std::max<size_t>(nw, 1) * sizeof(uint32_t), st));
  if (n_ped) {   // the committed list goes through the (now unused) CUR buffer
    B200_CUDA(cudaMemcpyAsync(S.b[Scratch::CUR].p, r->private_committed, n_ped * sizeof(uint32_t),
                              cudaMemcpyHostToDevice, st));
    k_setup_ped_pos<<<cdiv(n_ped, ST), ST, 0, st>>>(S.get<uint32_t>(Scratch::CUR), (uint32_t)n_ped, ped_pos);
    ctx->launches++;
  }
  WireClass wc{s.nw, s.n_pub, r->commitment_wire, ped_pos};
  const Fr* A = S.get<Fr>(Scratch::ABC);
  uint8_t* f8 = S.get<uint8_t>(Scratch::FLAGS8);
  uint32_t *fa = S.get<uint32_t>(Scratch::FA), *fb = S.get<uint32_t>(Scratch::FB), *fk = S.get<uint32_t>(Scratch::FK);
  k_setup_flags<<<cdiv(nw + 1, ST), ST, 0, st>>>(A, A + nw, wc, f8, f8 + nw, f8 + 2 * nw, fa, fb, fk);
  ctx->launches++;
  uint32_t* scan_tmp = S.get<uint32_t>(Scratch::SCAN);
  for (uint32_t* f : {fa, fb, fk}) B200_TRY(scan_exclusive(ctx, f, nw + 1, scan_tmp));
  if (nw) {
    k_setup_compact<<<cdiv(nw, ST), ST, 0, st>>>(A, A + nw, A + 2 * nw, wc, t, fa, fb, fk, sc, sc + o_b, sc + o_k,
                                                 sc + o_vk, sc + o_ped, sc + o_peds);
    ctx->launches++;
  }
  if (N > 1) {
    k_setup_z<<<cdiv(N - 1, ST), ST, 0, st>>>(S.get<Fr>(Scratch::P), (uint32_t)(N - 1), s.L, zc, sc + o_z);
    ctx->launches++;
  }
  const Fr small[7] = {t.alpha, t.beta, delta, t.beta, delta, gamma, Fr::neg(sigma)};
  B200_CUDA(cudaMemcpyAsync(sc + o_s1, small, sizeof(small), cudaMemcpyHostToDevice, st));
  B200_CUDA(cudaGetLastError());
  uint32_t counts[3];
  B200_CUDA(cudaMemcpyAsync(&counts[0], fa + nw, 4, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaMemcpyAsync(&counts[1], fb + nw, 4, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaMemcpyAsync(&counts[2], fk + nw, 4, cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));   // also: `small` is a host temporary
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  // ---- points
  const size_t n_a = counts[0], n_b = counts[1], n_k = counts[2];
  enum { A_, B_, K_, Z_, B2_, VK_, PED_, PEDS_ };
  const size_t len[8] = {n_a, n_b, n_k, N - 1, n_b, n_vk, n_ped, n_ped};
  const size_t off[8] = {0, o_b, o_k, o_z, o_b, o_vk, o_ped, o_peds};
  const bool ped = r->commitment_wire >= 0;
  for (int i = 0; i < 8; i++)
    if (i < PED_ || ped) B200_TRY(new_bases(i == B2_ ? 2 : 1, len[i], ctx->device, &made[i]));
  B200_TRY(S.b[Scratch::TAB1].ensure(fixed_base_table_points() * sizeof(G1Affine)));
  B200_TRY(S.b[Scratch::TAB2].ensure(fixed_base_table_points() * sizeof(G2Affine)));
  B200_TRY(S.b[Scratch::SMALL].ensure(3 * sizeof(G1Affine) + 4 * sizeof(G2Affine)));
  G1Affine g1, *small1 = S.get<G1Affine>(Scratch::SMALL);
  G2Affine g2, *small2 = reinterpret_cast<G2Affine*>(small1 + 3);
  memcpy(&g1, G1_GEN_LIMBS, sizeof(g1));
  memcpy(&g2, G2_GEN_LIMBS, sizeof(g2));
  const G1Affine* tab1 = S.get<G1Affine>(Scratch::TAB1);
  const G2Affine* tab2 = S.get<G2Affine>(Scratch::TAB2);
  B200_TRY(fixed_base_table_device<Fp>(ctx, g1, S.get<G1Affine>(Scratch::TAB1)));
  for (int i = 0; i < 8; i++)
    if (i != B2_ && made[i])
      B200_TRY(fixed_base_mul_table_device<Fp>(ctx, tab1, sc + off[i], len[i],
                                               reinterpret_cast<G1Affine*>(made[i]->d_points)));
  B200_TRY(fixed_base_mul_table_device<Fp>(ctx, tab1, sc + o_s1, 3, small1));
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  B200_TRY(fixed_base_table_device<Fp2>(ctx, g2, S.get<G2Affine>(Scratch::TAB2)));
  B200_TRY(fixed_base_mul_table_device<Fp2>(ctx, tab2, sc + o_b, n_b, reinterpret_cast<G2Affine*>(made[B2_]->d_points)));
  B200_TRY(fixed_base_mul_table_device<Fp2>(ctx, tab2, sc + o_s2, 4, small2));
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  // ---- results to the host
  if (nw) {
    B200_TRY(d2h_copy(ctx, inf_a, f8, nw, st));
    B200_TRY(d2h_copy(ctx, inf_b, f8 + nw, nw, st));
    B200_TRY(d2h_copy(ctx, k_skip, f8 + 2 * nw, nw, st));
  }
  G1Affine h1[3];
  G2Affine h2[4];
  B200_CUDA(cudaMemcpyAsync(h1, small1, sizeof(h1), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaMemcpyAsync(h2, small2, sizeof(h2), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], st));
  B200_CUDA(cudaStreamSynchronize(st));
  events_to_timings(ctx, ev);
  out->log2_domain = (unsigned)s.L;
  b200g16_bases** dst[8] = {&out->a, &out->b, &out->k, &out->z, &out->b2, &out->vk_k, &out->ped_basis,
                            &out->ped_basis_exp_sigma};
  for (int i = 0; i < 8; i++) *dst[i] = made[i];
  memcpy(out->g1_alpha, &h1[0], sizeof(out->g1_alpha));
  memcpy(out->g1_beta, &h1[1], sizeof(out->g1_beta));
  memcpy(out->g1_delta, &h1[2], sizeof(out->g1_delta));
  memcpy(out->g2_beta, &h2[0], sizeof(out->g2_beta));
  memcpy(out->g2_delta, &h2[1], sizeof(out->g2_delta));
  memcpy(out->g2_gamma, &h2[2], sizeof(out->g2_gamma));
  if (ped) {
    memcpy(out->ped_g, G2_GEN_LIMBS, sizeof(out->ped_g));
    memcpy(out->ped_g_sigma_neg, &h2[3], sizeof(out->ped_g_sigma_neg));
  } else {
    memset(out->ped_g, 0, sizeof(out->ped_g));
    memset(out->ped_g_sigma_neg, 0, sizeof(out->ped_g_sigma_neg));
  }
  return 0;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int b200g16_setup(b200g16_ctx* ctx, const b200g16_r1cs_desc* r1cs, const b200g16_toxic* toxic, uint8_t* infinity_a,
                  uint8_t* infinity_b, uint8_t* k_skip, b200g16_setup_out* out) {
  if (!ctx || !toxic || !infinity_a || !infinity_b || !k_skip || !out) return fail(B200G16_ERR_ARG, "setup: null argument");
  Shape s;
  B200_TRY(check_desc(r1cs, &s));
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active)
    return fail(B200G16_ERR_STATE, "setup: a prove is open on this ctx (b200g16_prove_begin_dev without _end_dev)");
  B200_CUDA(cudaSetDevice(ctx->device));
  b200g16_bases* made[8] = {};
  const int st = setup_run(ctx, r1cs, s, toxic, infinity_a, infinity_b, k_skip, out, made);
  if (st) {
    cudaStreamSynchronize(ctx->stream);
    for (b200g16_bases* b : made) b200g16_bases_free(b);
  }
  return st;
}

int b200g16_setup_wire_polys(b200g16_ctx* ctx, const b200g16_r1cs_desc* r1cs, const uint64_t tau[4], uint64_t* a_out,
                             uint64_t* b_out, uint64_t* c_out) {
  if (!ctx || !tau) return fail(B200G16_ERR_ARG, "setup_wire_polys: null argument");
  Shape s;
  B200_TRY(check_desc(r1cs, &s));
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (ctx->prove_active)
    return fail(B200G16_ERR_STATE, "setup_wire_polys: a prove is open on this ctx (b200g16_prove_begin_dev without _end_dev)");
  B200_CUDA(cudaSetDevice(ctx->device));
  Scratch S;
  ctx->timings.n = 0;
  int ev = 0;
  B200_CUDA(cudaEventRecord(ctx->ev[ev++], ctx->stream));
  int status = setup_front(ctx, r1cs, s, fr_of(tau), S, &ev);
  uint64_t* outs[3] = {a_out, b_out, c_out};
  for (int k = 0; k < 3 && status == 0; k++)
    if (outs[k] && s.nw)
      status = d2h_copy(ctx, outs[k], S.get<Fr>(Scratch::ABC) + (size_t)k * s.nw, (size_t)s.nw * sizeof(Fr), ctx->stream);
  if (status) {
    cudaStreamSynchronize(ctx->stream);
    return status;
  }
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  events_to_timings(ctx, ev);
  return 0;
}

}  // extern "C"
