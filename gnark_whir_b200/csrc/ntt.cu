// Fr number-theoretic transforms with gnark-crypto's fft.Domain conventions, and groth16's
// computeH, for sm_100a.
//
// Replaces gnark-crypto ecc/bn254/fr/fft (Domain.FFT / Domain.FFTInverse with fft.DIF /
// fft.DIT / fft.OnCoset()) and gnark backend/groth16/bn254/prove.go computeH, reached from
// the reference at /root/reference/mt.go:496 (the Domain itself is built by Setup, mt.go:448).
//
//   DIF: natural-order input -> bit-reversed output (Gentleman-Sande butterflies)
//   DIT: bit-reversed input -> natural-order output (Cooley-Tukey butterflies)
//   OnCoset: forward multiplies a[i] by g^i first (index bit-reversed when DIT); inverse
//            multiplies by g^-i/N last (index bit-reversed when DIF); g = 5.
//
// Kernel structure: log2 N levels are split into passes of <= 8 levels.  A pass owns the index
// bits [b0, b0+k): a CTA of 64 threads loads a tile of 2^k "rows" x 2 contiguous "columns" (16 KB)
// into shared memory, runs the k radix-2 levels there (split lo/hi uint4 layout so
// consecutive lanes hit consecutive banks), and stores the tile back: 64 B of HBM traffic per
// element per pass; ~14 such CTAs share an SM and overlap each other's load / butterfly / store phases.
// Coset / 1/N scaling rides on the first pass's load or the last pass's
// store.  Twiddles come from one table w^e (e <= N/2): the pass over the top bits streams it
// once, later passes reuse a few KB of it out of L1/L2; inverse transforms read the same table
// through w^-e = -w^(N/2-e) with the sign folded into the butterfly.
#include "common.cuh"
#include "field.cuh"

namespace b200 {

constexpr int NTT_MAX_K = 8;
constexpr int NTT_LOGC = 3;
constexpr int NTT_THREADS = 64;    // 2 warps per CTA, ~14 CTAs per SM (profiles/r02j_ntt_config_sweep.txt)
constexpr int NTT_CTAS = 14;

static inline unsigned cdiv_u(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

__device__ __forceinline__ uint32_t bitrev_dev(uint32_t i, int L) { return __brev(i) >> (32 - L); }

__device__ __forceinline__ Fr ld_fr(const Fr* p) {
  Fr r;
  const uint4* s = reinterpret_cast<const uint4*>(p);
  uint4 a = s[0], b = s[1];
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}
__device__ __forceinline__ Fr ldg_fr(const Fr* p) {
  Fr r;
  const uint4* s = reinterpret_cast<const uint4*>(p);
  uint4 a = __ldg(s), b = __ldg(s + 1);
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}
__device__ __forceinline__ void st_fr(Fr* p, const Fr& v) {
  uint4* d = reinterpret_cast<uint4*>(p);
  d[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  d[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

struct SmemTile {
  uint4* lo;
  uint4* hi;
  __device__ __forceinline__ Fr get(uint32_t s) const {
    uint4 a = lo[s], b = hi[s];
    Fr r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
    r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
  }
  __device__ __forceinline__ void put(uint32_t s, const Fr& v) const {
    lo[s] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    hi[s] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
  }
};

// w^e (or w^-e) from the forward table; `half` = N_table/2, sh = log2(N_table/N)
__device__ __forceinline__ Fr twiddle(const Fr* __restrict__ tw, uint32_t e, int sh, uint32_t half, bool inverse) {
  uint32_t idx = e << sh;
  if (!inverse || idx == 0) return ldg_fr(tw + idx);
  return Fr::neg(ldg_fr(tw + (half - idx)));
}

struct NttPassArgs {
  Fr* data;         // blockIdx.y-th vector = vecs[y] when nvecs > 0, else data + y * 2^L
  Fr* vecs[3];
  int nvecs;
  const Fr* tw;
  const Fr* pre;    // multiply on load by pre[idx]  (nullptr = none)
  const Fr* post;   // multiply on store by post[idx] (nullptr = none)
  const Fr* post_vec[3];  // post_mode == 2 with nvecs > 0: per-vector tables (computeH's fused scalings)
  Fr post_const;    // used when post_mode == 1
  uint32_t tw_half;
  int tw_sh;
  int L, b0, k, logc;
  int post_mode;    // 0 none, 1 const, 2 table
  int pre_bitrev, post_bitrev;
  int inverse;
};

// (Measured and not kept, profiles/r02c_sweep_ntt_fused_loadstore.jsonl: reading the first level's operands straight
// from global memory and storing the last level's results straight to it — two shared-memory round trips and two
// barriers fewer per pass — is 1.4% SLOWER at 2^24 (3.906 vs 3.853 ms): the separate load loop keeps four independent
// 32-byte loads per thread in flight, the fused form exposes the latency of two.)
// TFAST: rows contiguous in memory (b0 == 0) -> row index fastest in shared memory.
// INV: inverse transform (twiddles w^-e), a template parameter so that the forward kernels carry none of its selects.
template <bool DIT, bool TFAST, bool INV>
__global__ void __launch_bounds__(NTT_THREADS, NTT_CTAS) k_ntt_pass(NttPassArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int k = A.k, L = A.L, b0 = A.b0, logc = A.logc;
  const uint32_t rows = 1u << k;
  const uint32_t T = rows << logc;  // elements per tile
  SmemTile sm{reinterpret_cast<uint4*>(smem_raw), reinterpret_cast<uint4*>(smem_raw) + T};
  const uint32_t lowmask = (1u << b0) - 1u;
  const uint32_t tile = blockIdx.x;
  Fr* data = A.nvecs ? A.vecs[blockIdx.y] : A.data + (size_t)blockIdx.y * ((size_t)1 << L);  // batched transforms
  const Fr* post = (A.post_mode == 2 && A.nvecs) ? A.post_vec[blockIdx.y] : A.post;

  // ---- load
  for (uint32_t x = threadIdx.x; x < T; x += blockDim.x) {
    uint32_t t, c;
    if (TFAST) { t = x & (rows - 1); c = x >> k; }
    else { c = x & ((1u << logc) - 1); t = x >> logc; }
    uint32_t u = (tile << logc) + c;
    uint32_t i = ((u >> b0) << (b0 + k)) | (t << b0) | (u & lowmask);
    Fr v = ld_fr(data + i);
    if (A.pre) v = Fr::mul(v, ldg_fr(A.pre + (A.pre_bitrev ? bitrev_dev(i, L) : i)));
    sm.put(x, v);  // x is exactly the shared-memory slot for this layout
  }
  __syncthreads();

  // ---- k radix-2 levels
  const uint32_t nbf = T >> 1;
  for (int step = 0; step < k; step++) {
    const int lb = DIT ? step : (k - 1 - step);  // local partner bit
    const int pb = b0 + lb;                      // global partner bit
    const uint32_t lbmask = (1u << lb) - 1u;
    for (uint32_t q = threadIdx.x; q < nbf; q += blockDim.x) {
      uint32_t r, c;
      if (TFAST) { r = q & ((rows >> 1) - 1); c = q >> (k - 1); }
      else { c = q & ((1u << logc) - 1); r = q >> logc; }
      uint32_t t0 = ((r >> lb) << (lb + 1)) | (r & lbmask);
      uint32_t t1 = t0 | (1u << lb);
      uint32_t s0 = TFAST ? ((c << k) | t0) : ((t0 << logc) | c);
      uint32_t s1 = TFAST ? ((c << k) | t1) : ((t1 << logc) | c);
      Fr xv = sm.get(s0), yv = sm.get(s1);
      if (pb == 0) {  // the level whose twiddles are all w^0 = 1: no products (warp-uniform branch)
        sm.put(s0, Fr::add(xv, yv));
        sm.put(s1, Fr::sub(xv, yv));
        continue;
      }
      uint32_t u = (tile << logc) + c;
      uint32_t j = ((t0 & lbmask) << b0) | (u & lowmask);
      uint32_t e = j << (L - 1 - pb);
      // Inverse transforms need w^-e = -w^(N/2 - e).  The table carries one entry more than N/2 (w^(N/2) = -1), so
      // the lookup is branch-free for every e, and the sign goes into the butterfly instead of a field negation per
      // twiddle: (x - y) * (-w') = (y - x) * w', and x +- y * (-w') = x -+ y * w'.
      const uint32_t idx = e << A.tw_sh;
      const Fr w = ldg_fr(A.tw + (INV ? A.tw_half - idx : idx));
      if (DIT) {
        yv = Fr::mul(yv, w);
        if (!INV) {
          sm.put(s0, Fr::add(xv, yv));
          sm.put(s1, Fr::sub(xv, yv));
        } else {
          sm.put(s0, Fr::sub(xv, yv));
          sm.put(s1, Fr::add(xv, yv));
        }
      } else {
        sm.put(s0, Fr::add(xv, yv));
        sm.put(s1, Fr::mul(INV ? Fr::sub(yv, xv) : Fr::sub(xv, yv), w));
      }
    }
    __syncthreads();
  }

  // ---- store
  for (uint32_t x = threadIdx.x; x < T; x += blockDim.x) {
    uint32_t t, c;
    if (TFAST) { t = x & (rows - 1); c = x >> k; }
    else { c = x & ((1u << logc) - 1); t = x >> logc; }
    uint32_t u = (tile << logc) + c;
    uint32_t i = ((u >> b0) << (b0 + k)) | (t << b0) | (u & lowmask);
    Fr v = sm.get(x);
    if (A.post_mode == 1) v = Fr::mul(v, A.post_const);
    else if (A.post_mode == 2) v = Fr::mul(v, ldg_fr(post + (A.post_bitrev ? bitrev_dev(i, L) : i)));
    st_fr(data + i, v);
  }
}

// ------------------------------------------------------------------------------ transforms split over G = 2^g GPUs
// Device d holds positions [d M, (d + 1) M) of a vector of N = 2^L elements (M = N / G).  The g levels whose partner
// bit lies among the top g position bits pair elements at the SAME local offset on different devices; every other
// level is local and — because w_N^(e G) = w_M^e — is exactly a level of the ordinary size-M transform of the
// slice.  So a DIF transform is [cross levels] + [local size-M DIF], a DIT transform [local size-M DIT] +
// [cross levels], with unchanged global orderings (natural <-> bit-reversed, sliced by position).
// The cross levels run as ONE kernel per device over peer memory: device `me` takes the offsets
// [me M / G, (me + 1) M / G), loads the G elements of each offset from the G devices' buffers (NVLink peer loads,
// coalesced), runs the g butterfly levels in registers and stores the results back to their owners.  Every
// element is read and written by exactly one device, so the only synchronisation is "all slices ready" before and
// "all cross kernels done" after (events in one process, a barrier between processes).
struct CrossArgs {
  Fr* buf[3][8];    // [vector][device] slice base pointers, valid on this device
  const Fr* tw;
  uint32_t tw_half;
  int tw_sh;
  int L, me;
  int inverse;      // twiddles w^-e
};

template <int GLOG, bool DIT>
__device__ __forceinline__ void cross_levels(Fr (&x)[1 << GLOG], uint32_t o, const Fr* __restrict__ tw, int tw_sh,
                                             uint32_t tw_half, int L, bool inverse) {
  constexpr int G = 1 << GLOG;
  const uint32_t M = 1u << (L - GLOG);
#pragma unroll
  for (int step = 0; step < GLOG; step++) {
    const int q = DIT ? (GLOG - 1 - step) : step;   // level q pairs device indices that differ in bit GLOG-1-q
    const int bit = GLOG - 1 - q;
#pragma unroll
    for (int d0 = 0; d0 < G; d0++) {
      if (d0 & (1 << bit)) continue;
      const int d1 = d0 | (1 << bit);
      const uint32_t j = (uint32_t)(d0 & ((1 << bit) - 1)) * M + o;   // position bits below the partner bit
      const uint32_t e = j << q;
      Fr a = x[d0], b = x[d1];
      if (e == 0 && !inverse) {
        x[d0] = Fr::add(a, b);
        x[d1] = Fr::sub(a, b);
        continue;
      }
      const Fr w = twiddle(tw, e, tw_sh, tw_half, inverse);
      if (DIT) {
        b = Fr::mul(b, w);
        x[d0] = Fr::add(a, b);
        x[d1] = Fr::sub(a, b);
      } else {
        x[d0] = Fr::add(a, b);
        x[d1] = Fr::mul(Fr::sub(a, b), w);
      }
    }
  }
}

template <int GLOG, bool DIT>
__global__ void __launch_bounds__(128) k_ntt_cross(CrossArgs A) {
  constexpr int G = 1 << GLOG;
  const uint32_t share = (1u << (A.L - GLOG)) >> GLOG;           // offsets per device
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= share) return;
  const uint32_t o = (uint32_t)A.me * share + t;
  Fr x[G];
#pragma unroll
  for (int d = 0; d < G; d++) x[d] = ld_fr(A.buf[blockIdx.y][d] + o);
  cross_levels<GLOG, DIT>(x, o, A.tw, A.tw_sh, A.tw_half, A.L, A.inverse != 0);
#pragma unroll
  for (int d = 0; d < G; d++) st_fr(A.buf[blockIdx.y][d] + o, x[d]);
}

// computeH's middle, fused over peer memory: last (cross) levels of the coset FFTs of a, b, c, the pointwise
// a b - c (a and c already carry 1 / (g^N - 1)), and the first (cross) levels of the final inverse transform;
// reads 3 vectors, writes 1 (into the a slices).
template <int GLOG>
__global__ void __launch_bounds__(128) k_ntt_cross_h(CrossArgs A) {
  constexpr int G = 1 << GLOG;
  const uint32_t share = (1u << (A.L - GLOG)) >> GLOG;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= share) return;
  const uint32_t o = (uint32_t)A.me * share + t;
  Fr acc[G], x[G];
#pragma unroll
  for (int d = 0; d < G; d++) acc[d] = ld_fr(A.buf[0][d] + o);
  cross_levels<GLOG, true>(acc, o, A.tw, A.tw_sh, A.tw_half, A.L, false);
#pragma unroll
  for (int d = 0; d < G; d++) x[d] = ld_fr(A.buf[1][d] + o);
  cross_levels<GLOG, true>(x, o, A.tw, A.tw_sh, A.tw_half, A.L, false);
#pragma unroll
  for (int d = 0; d < G; d++) acc[d] = Fr::mul(acc[d], x[d]);
#pragma unroll
  for (int d = 0; d < G; d++) x[d] = ld_fr(A.buf[2][d] + o);
  cross_levels<GLOG, true>(x, o, A.tw, A.tw_sh, A.tw_half, A.L, false);
#pragma unroll
  for (int d = 0; d < G; d++) acc[d] = Fr::sub(acc[d], x[d]);
  cross_levels<GLOG, false>(acc, o, A.tw, A.tw_sh, A.tw_half, A.L, true);
#pragma unroll
  for (int d = 0; d < G; d++) st_fr(A.buf[0][d] + o, acc[d]);
}

// t[s + i] = t[i] * step  for i < s   (doubling construction of geometric tables)
__global__ void __launch_bounds__(256) k_geom_expand(Fr* __restrict__ t, uint32_t s, uint32_t limit, Fr step) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= s || s + i >= limit) return;
  st_fr(t + s + i, Fr::mul(ld_fr(t + i), step));
}

// a[i] = a[i] * b[i] - c[i]   (computeH with the 1 / (g^N - 1) factor folded into the transforms' scaling tables)
__global__ void __launch_bounds__(256) k_h_pointwise_plain(Fr* __restrict__ a, const Fr* __restrict__ b,
                                                            const Fr* __restrict__ c, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  st_fr(a + i, Fr::sub(Fr::mul(ld_fr(a + i), ld_fr(b + i)), ld_fr(c + i)));
}

// a[i] = (a[i] * b[i] - c[i]) * den
__global__ void __launch_bounds__(256) k_h_pointwise(Fr* __restrict__ a, const Fr* __restrict__ b,
                                                      const Fr* __restrict__ c, uint32_t n, Fr den) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr v = Fr::sub(Fr::mul(ld_fr(a + i), ld_fr(b + i)), ld_fr(c + i));
  st_fr(a + i, Fr::mul(v, den));
}

// ------------------------------------------------------------------------------ host side
static Fr fr_from_limbs(const uint32_t (&l)[8]) {
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = l[i];
  return r;
}
static Fr fr_pow_u64(Fr a, uint64_t e) {
  Fr r = Fr::one();
  while (e) {
    if (e & 1) r = Fr::mul(r, a);
    a = Fr::sqr(a);
    e >>= 1;
  }
  return r;
}
static Fr fr_from_u64(uint64_t v) {
  Fr r = Fr::zero();
  r.l[0] = (uint32_t)v;
  r.l[1] = (uint32_t)(v >> 32);
  return Fr::to_mont(r);
}

static Fr coset_denominator_inv(size_t n);

// Build t[0..count) = first * ratio^i on the device.
int build_geometric(b200g16_ctx* ctx, Fr* d_t, size_t count, const Fr& first, Fr ratio) {
  B200_CUDA(cudaMemcpyAsync(d_t, &first, sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));  // `first` is a host temporary
  Fr step = ratio;                                // ratio^s
  for (size_t s = 1; s < count; s <<= 1) {
    k_geom_expand<<<cdiv_u(s, 256), 256, 0, ctx->stream>>>(d_t, (uint32_t)s, (uint32_t)count, step);
    ctx->launches++;
    step = Fr::sqr(step);
  }
  B200_CUDA(cudaGetLastError());
  return 0;
}

struct NttDomain {
  int L = -1;
  Fr w, w_inv, n_inv;
};

static void domain_params(int L, NttDomain* d) {
  const uint32_t root[8] = B200_FR_ROOT28;
  const uint32_t root_inv[8] = B200_FR_ROOT28_INV;
  Fr w = fr_from_limbs(root), wi = fr_from_limbs(root_inv);
  for (int i = L; i < 28; i++) { w = Fr::sqr(w); wi = Fr::sqr(wi); }
  d->L = L;
  d->w = w;
  d->w_inv = wi;
  d->n_inv = Fr::inv(fr_from_u64(1ull << L));
}

// twiddle table w^e, e <= N/2, for the largest N seen so far
static int ensure_twiddles(b200g16_ctx* ctx, int L) {
  NttWorkspace& ws = ctx->ntt;
  if (ws.tw_log >= L) return 0;
  size_t half = (size_t)1 << (L > 0 ? L - 1 : 0);
  B200_TRY(ws.tw.ensure((half + 1) * sizeof(Fr)));   // + w^(N/2) = -1: k_ntt_pass reads w^(N/2 - e) for inverse transforms
  NttDomain d;
  domain_params(L, &d);
  B200_TRY(build_geometric(ctx, ws.tw.as<Fr>(), half + 1, Fr::one(), d.w));
  ws.tw_log = L;
  return 0;
}

// coset tables for size 2^L: fwd[i] = g^i, inv[i] = g^-i / N
static int ensure_coset(b200g16_ctx* ctx, int L) {
  NttWorkspace& ws = ctx->ntt;
  if (ws.coset_log == L) return 0;
  size_t n = (size_t)1 << L;
  B200_TRY(ws.coset.ensure(2 * n * sizeof(Fr)));
  const uint32_t g[8] = B200_FR_GEN;
  const uint32_t gi[8] = B200_FR_GEN_INV;
  NttDomain d;
  domain_params(L, &d);
  B200_TRY(build_geometric(ctx, ws.coset.as<Fr>(), n, Fr::one(), fr_from_limbs(g)));
  B200_TRY(build_geometric(ctx, ws.coset.as<Fr>() + n, n, d.n_inv, fr_from_limbs(gi)));
  ws.coset_log = L;
  return 0;
}

// In-place transform of `batch` vectors of 2^L elements: consecutive at d_data, or (vecs != nullptr,
// batch <= 3) at vecs[0..batch) — computeH transforms a, b, c in one launch per pass.
// fused_post: per-vector tables multiplied in on the last store INSTEAD of the transform's own 1/N (plain inverse
// transforms only); skip_pre: a forward coset transform whose g^i scaling the previous transform already applied.
static int ntt_device_impl(b200g16_ctx* ctx, Fr* d_data, Fr* const* vecs, int L, int batch, bool inverse, bool coset,
                           int decimation, const Fr* const* fused_post = nullptr, bool skip_pre = false) {
  if (L < 0 || L > 28) return fail(B200G16_ERR_ARG, "ntt: log2n=%d out of range (two-adicity 28)", L);
  if (decimation != B200G16_DIF && decimation != B200G16_DIT) return fail(B200G16_ERR_ARG, "ntt: bad decimation");
  if (batch < 1) return fail(B200G16_ERR_ARG, "ntt: batch");
  B200_TRY(ensure_twiddles(ctx, L));
  if (coset) B200_TRY(ensure_coset(ctx, L));
  NttWorkspace& ws = ctx->ntt;
  const size_t n = (size_t)1 << L;
  const bool dit = decimation == B200G16_DIT;
  NttDomain dom;
  domain_params(L, &dom);

  NttPassArgs A;
  A.data = d_data;
  A.nvecs = vecs ? batch : 0;
  for (int i = 0; i < 3; i++) A.vecs[i] = (vecs && i < batch) ? vecs[i] : nullptr;
  A.tw = ws.tw.as<Fr>();
  A.tw_sh = ws.tw_log - L;
  A.tw_half = (uint32_t)(((size_t)1 << ws.tw_log) >> 1);
  A.L = L;
  A.inverse = inverse ? 1 : 0;
  A.post_const = dom.n_inv;

  // forward-coset scaling on the first load, inverse scaling on the last store
  const Fr* pre = (coset && !inverse && !skip_pre) ? ws.coset.as<Fr>() : nullptr;
  const int pre_bitrev = dit ? 1 : 0;        // DIT input is bit-reversed
  int post_mode = 0;
  const Fr* post = nullptr;
  if (inverse) {
    if (coset) { post_mode = 2; post = ws.coset.as<Fr>() + n; }
    else post_mode = 1;
  }
  for (int i = 0; i < 3; i++) A.post_vec[i] = nullptr;
  if (fused_post) {
    if (!inverse || coset || !vecs) return fail(B200G16_ERR_ARG, "ntt: fused scaling needs a plain inverse transform over a vector list");
    post_mode = 2;
    for (int i = 0; i < batch && i < 3; i++) A.post_vec[i] = fused_post[i];
  }
  const int post_bitrev = dit ? 0 : 1;       // DIF output is bit-reversed

  if (L == 0) {  // single element: only scaling applies (n_inv = 1, g^0 = 1) -> nothing to do
    return 0;
  }
  // split L levels into passes of <= NTT_MAX_K, as evenly as possible
  int npass = (L + NTT_MAX_K - 1) / NTT_MAX_K;
  int ks[8];
  for (int p = 0; p < npass; p++) ks[p] = L / npass + (p < L % npass ? 1 : 0);
  // DIF walks partner bits from the top down, DIT from the bottom up
  int b0s[8];
  if (dit) { int b = 0; for (int p = 0; p < npass; p++) { b0s[p] = b; b += ks[p]; } }
  else { int b = L; for (int p = 0; p < npass; p++) { b -= ks[p]; b0s[p] = b; } }

  for (int p = 0; p < npass; p++) {
    A.k = ks[p];
    A.b0 = b0s[p];
    A.pre = (p == 0) ? pre : nullptr;
    A.pre_bitrev = pre_bitrev;
    A.post_mode = (p == npass - 1) ? post_mode : 0;
    A.post = post;
    A.post_bitrev = post_bitrev;
    // tile = 2^k rows x 2^logc columns.  Measured (profiles/r02j_ntt_config_sweep.txt, 2^20 .. 2^24): what matters is
    // ~8 elements per thread per tile in SMALL CTAs — 64 threads x 2 columns (16 KB tiles, 14 CTAs/SM): barriers span 2
    // warps instead of 8 and many CTAs interleave their load / butterfly / store phases.  2^24: 3.78 -> 3.54 ms against
    // 256 threads x 4 columns, computeH 27.6 -> 25.9 ms; 8 columns x 256 threads (round 1): 3.86 ms.
    const int logc_pref = 1;
    int logc = L - A.k < logc_pref ? L - A.k : logc_pref;
    A.logc = logc;
    size_t tiles = n >> (A.k + logc);
    size_t smem = ((size_t)1 << (A.k + logc)) * sizeof(Fr);
    dim3 grid((unsigned)tiles, (unsigned)batch);
    bool tfast = (A.b0 == 0);
    const unsigned ntt_threads = NTT_THREADS;
#define B200_LAUNCH_PASS(DITV, TF, IV)                                                                      \
    do {                                                                                                     \
      B200_CUDA(cudaFuncSetAttribute(k_ntt_pass<DITV, TF, IV>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                     (int)(((size_t)1 << (NTT_MAX_K + NTT_LOGC)) * sizeof(Fr))));            \
      k_ntt_pass<DITV, TF, IV><<<grid, ntt_threads, smem, ctx->stream>>>(A);                                 \
    } while (0)
#define B200_LAUNCH_PASS2(DITV, TF) do { if (A.inverse) B200_LAUNCH_PASS(DITV, TF, true); else B200_LAUNCH_PASS(DITV, TF, false); } while (0)
    if (dit) { if (tfast) B200_LAUNCH_PASS2(true, true); else B200_LAUNCH_PASS2(true, false); }
    else { if (tfast) B200_LAUNCH_PASS2(false, true); else B200_LAUNCH_PASS2(false, false); }
#undef B200_LAUNCH_PASS2
#undef B200_LAUNCH_PASS
    ctx->launches++;
  }
  B200_CUDA(cudaGetLastError());
  return 0;
}

int ntt_device(b200g16_ctx* ctx, Fr* d_data, int L, int batch, bool inverse, bool coset, int decimation) {
  return ntt_device_impl(ctx, d_data, nullptr, L, batch, inverse, coset, decimation);
}

static Fr coset_denominator_inv(size_t n) {  // 1 / (g^N - 1)
  const uint32_t g[8] = B200_FR_GEN;
  return Fr::inv(Fr::sub(fr_pow_u64(fr_from_limbs(g), (uint64_t)n), Fr::one()));
}

// computeH's pointwise step on coset evaluations: a = (a * b - c) / (g^N - 1)
int h_pointwise_device(b200g16_ctx* ctx, Fr* a, const Fr* b, const Fr* c, int L) {
  const size_t n = (size_t)1 << L;
  k_h_pointwise<<<cdiv_u(n, 256), 256, 0, ctx->stream>>>(a, b, c, (uint32_t)n, coset_denominator_inv(n));
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

// fused scaling tables for computeH at size 2^L: t1[i] = g^i / N, t2[i] = g^i / (N (g^N - 1))
static int ensure_fused(b200g16_ctx* ctx, int L) {
  NttWorkspace& ws = ctx->ntt;
  if (ws.fused_log == L) return 0;
  size_t n = (size_t)1 << L;
  B200_TRY(ws.fused.ensure(2 * n * sizeof(Fr)));
  const uint32_t g[8] = B200_FR_GEN;
  NttDomain d;
  domain_params(L, &d);
  B200_TRY(build_geometric(ctx, ws.fused.as<Fr>(), n, d.n_inv, fr_from_limbs(g)));
  B200_TRY(build_geometric(ctx, ws.fused.as<Fr>() + n, n, Fr::mul(d.n_inv, coset_denominator_inv(n)), fr_from_limbs(g)));
  ws.fused_log = L;
  return 0;
}

// The first two transforms of computeH for `batch` vectors (<= 3), fused: FFTInverse (DIF) stores x / N * g^i
// [* 1/(g^N - 1) when with_den[v]] in one product, so the coset FFT (DIT) that follows loads without scaling.
// Same values as ntt(inverse) ; ntt(coset) [; * den], one Fr product per element less (two with the denominator).
int ntt_coset_pair_device(b200g16_ctx* ctx, Fr* const* vecs, int batch, int L, const bool* with_den) {
  if (L == 0) {  // one element: iNTT and coset NTT are the identity; only the denominator remains
    for (int v = 0; v < batch; v++)
      if (with_den[v]) {
        Fr x;
        B200_CUDA(cudaMemcpyAsync(&x, vecs[v], sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
        B200_CUDA(cudaStreamSynchronize(ctx->stream));
        x = Fr::mul(x, coset_denominator_inv(1));
        B200_CUDA(cudaMemcpyAsync(vecs[v], &x, sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
        B200_CUDA(cudaStreamSynchronize(ctx->stream));
      }
    return 0;
  }
  B200_TRY(ensure_twiddles(ctx, L));
  B200_TRY(ensure_coset(ctx, L));
  B200_TRY(ensure_fused(ctx, L));
  const size_t n = (size_t)1 << L;
  const Fr* post[3] = {nullptr, nullptr, nullptr};
  for (int v = 0; v < batch; v++) post[v] = ctx->ntt.fused.as<Fr>() + (with_den[v] ? n : 0);
  B200_TRY(ntt_device_impl(ctx, nullptr, vecs, L, batch, true, false, B200G16_DIF, post, false));
  return ntt_device_impl(ctx, nullptr, vecs, L, batch, false, true, B200G16_DIT, nullptr, true);
}

// a = a * b - c on coset evaluations whose a and c already carry 1 / (g^N - 1)
int h_pointwise_plain_device(b200g16_ctx* ctx, Fr* a, const Fr* b, const Fr* c, int L) {
  const size_t n = (size_t)1 << L;
  k_h_pointwise_plain<<<cdiv_u(n, 256), 256, 0, ctx->stream>>>(a, b, c, (uint32_t)n);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

// computeH on device buffers a,b,c (each 2^L elements, already zero-padded); result in a.
// (a b - c) / (g^N - 1) = (a / d) b - (c / d): the denominator rides on the fused scaling of a and c.
int compute_h_device(b200g16_ctx* ctx, Fr* a, Fr* b, Fr* c, int L, bool sync_and_time) {
  int ev = 0;
  auto mark = [&]() { if (sync_and_time && ev < 18) cudaEventRecord(ctx->ev[ev++], ctx->stream); };
  // warm the tables outside the timed phases
  B200_TRY(ensure_twiddles(ctx, L));
  B200_TRY(ensure_coset(ctx, L));
  if (L > 0) B200_TRY(ensure_fused(ctx, L));
  mark();
  Fr* v[3] = {a, b, c};
  const bool den[3] = {true, false, true};
  B200_TRY(ntt_coset_pair_device(ctx, v, 3, L, den));
  mark();
  mark();
  B200_TRY(h_pointwise_plain_device(ctx, a, b, c, L));
  mark();
  B200_TRY(ntt_device(ctx, a, L, 1, true, true, B200G16_DIF));
  mark();
  B200_CUDA(cudaGetLastError());
  if (!sync_and_time) return 0;
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  events_to_timings(ctx, ev);
  return 0;
}

// ---- computeH over G = 2^g devices (see the kernels above) ------------------------------------------------------
static uint32_t bitrev_host(uint32_t v, int bits) {
  uint32_t r = 0;
  for (int i = 0; i < bits; i++) { r = (r << 1) | (v & 1); v >>= 1; }
  return r;
}

// Compact scaling tables of device `me`: position d M + o (bit-reversed order) has natural index
// bitrev_{L-g}(o) G + bitrev_g(me), so the size-M tables  t1[k] = g^(k G + br) / N,  t2 = t1 / (g^N - 1),
// ti[k] = g^-(k G + br) / N  are read at k = bitrev(o) by the ordinary size-M passes.
static int ensure_dist_tables(b200g16_ctx* ctx, int L, int g, int me) {
  NttWorkspace& ws = ctx->ntt;
  if (ws.dist_log == L && ws.dist_g == g && ws.dist_me == me) return 0;
  const size_t M = (size_t)1 << (L - g);
  B200_TRY(ws.dist.ensure(3 * M * sizeof(Fr)));
  const uint32_t gen[8] = B200_FR_GEN;
  const uint32_t gen_inv[8] = B200_FR_GEN_INV;
  NttDomain d;
  domain_params(L, &d);
  const uint64_t br = bitrev_host((uint32_t)me, g), G = (uint64_t)1 << g;
  const Fr gf = fr_from_limbs(gen), gi = fr_from_limbs(gen_inv);
  const Fr first = Fr::mul(d.n_inv, fr_pow_u64(gf, br));
  B200_TRY(build_geometric(ctx, ws.dist.as<Fr>(), M, first, fr_pow_u64(gf, G)));
  B200_TRY(build_geometric(ctx, ws.dist.as<Fr>() + M, M, Fr::mul(first, coset_denominator_inv((size_t)1 << L)), fr_pow_u64(gf, G)));
  B200_TRY(build_geometric(ctx, ws.dist.as<Fr>() + 2 * M, M, Fr::mul(d.n_inv, fr_pow_u64(gi, br)), fr_pow_u64(gi, G)));
  ws.dist_log = L; ws.dist_g = g; ws.dist_me = me;
  return 0;
}

static int fill_cross_args(b200g16_ctx* ctx, CrossArgs* A, Fr* const (*peers)[8], int nvec, int g, int me, int L, bool inverse) {
  B200_TRY(ensure_twiddles(ctx, L));
  memset(A, 0, sizeof(*A));
  for (int v = 0; v < nvec; v++)
    for (int d = 0; d < (1 << g); d++) A->buf[v][d] = peers[v][d];
  A->tw = ctx->ntt.tw.as<Fr>();
  A->tw_sh = ctx->ntt.tw_log - L;
  A->tw_half = (uint32_t)(((size_t)1 << ctx->ntt.tw_log) >> 1);
  A->L = L;
  A->me = me;
  A->inverse = inverse ? 1 : 0;
  return 0;
}

// One phase of the distributed computeH on this device (enqueued on ctx->stream, no synchronisation):
//   0  cross levels of FFTInverse(a, b, c)                       (needs: every device's slices loaded)
//   1  local: rest of FFTInverse with the fused scaling, then the local levels of the coset FFT
//   2  cross levels of the coset FFTs + pointwise + cross levels of the last FFTInverse -> a slices
//   3  local: rest of the last FFTInverse with g^-i / N  -> this device's slice of h in its a buffer
// peers[v][d]: slice of vector v (0 = a, 1 = b, 2 = c) on device d, addressable from this device.
int compute_h_dist_phase(b200g16_ctx* ctx, Fr* const (*peers)[8], int g, int me, int L, int phase) {
  if (g < 1 || g > 3 || L - 2 * g < 0 || L > 28) return fail(B200G16_ERR_ARG, "compute_h_dist: 2^%d over 2^%d devices", L, g);
  if (me < 0 || me >= (1 << g) || phase < 0 || phase > 3) return fail(B200G16_ERR_ARG, "compute_h_dist: bad rank / phase");
  const int Lm = L - g;
  const size_t M = (size_t)1 << Lm;
  const uint32_t share = (uint32_t)(M >> g);
  CrossArgs A;
  if (phase == 0 || phase == 2) {
    B200_TRY(fill_cross_args(ctx, &A, peers, 3, g, me, L, phase == 0));
    dim3 grid(cdiv_u(share, 128), phase == 0 ? 3 : 1);
    if (phase == 0) {
      if (g == 1) k_ntt_cross<1, false><<<grid, 128, 0, ctx->stream>>>(A);
      else if (g == 2) k_ntt_cross<2, false><<<grid, 128, 0, ctx->stream>>>(A);
      else k_ntt_cross<3, false><<<grid, 128, 0, ctx->stream>>>(A);
    } else {
      if (g == 1) k_ntt_cross_h<1><<<grid, 128, 0, ctx->stream>>>(A);
      else if (g == 2) k_ntt_cross_h<2><<<grid, 128, 0, ctx->stream>>>(A);
      else k_ntt_cross_h<3><<<grid, 128, 0, ctx->stream>>>(A);
    }
    ctx->launches++;
    B200_CUDA(cudaGetLastError());
    return 0;
  }
  B200_TRY(ensure_twiddles(ctx, L));   // the size-N table also serves the size-M passes (stride 2^g)
  B200_TRY(ensure_dist_tables(ctx, L, g, me));
  const Fr* t = ctx->ntt.dist.as<Fr>();
  if (phase == 1) {
    Fr* v[3] = {peers[0][me], peers[1][me], peers[2][me]};
    const Fr* post[3] = {t + M, t, t + M};   // a and c carry 1 / (g^N - 1)
    if (Lm == 0) return fail(B200G16_ERR_ARG, "compute_h_dist: slices of one element");
    B200_TRY(ntt_device_impl(ctx, nullptr, v, Lm, 3, true, false, B200G16_DIF, post, false));
    return ntt_device_impl(ctx, nullptr, v, Lm, 3, false, true, B200G16_DIT, nullptr, true);
  }
  Fr* v[1] = {peers[0][me]};
  const Fr* post[1] = {t + 2 * M};
  return ntt_device_impl(ctx, nullptr, v, Lm, 1, true, false, B200G16_DIF, post, false);
}

}  // namespace b200
