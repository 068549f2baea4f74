// Batch fixed-base scalar multiplication  out[i] = k_i * B  (G1 and G2), and the
// integer-pipe throughput probe.
//
// Replaces gnark-crypto ecc/bn254 BatchScalarMultiplicationG1 / G2, the hot loop of
// gnark backend/groth16/bn254/setup.go (Setup is called by the reference at
// /root/reference/mt.go:448 on every run: ~4N G1 + N G2 multiples of the generators).
// It is also how the tests and bench.py manufacture 2^24-point base sets with known
// discrete logs without shipping gigabytes through PCIe.
//
// Kernel: a per-call table T[w][d] = d * 2^(8w) * B (32 windows x 255 affine entries,
// built on the device by k_fb_table), then one thread per scalar: 32 mixed adds + one
// Fermat inversion for the affine result.
#include "common.cuh"
#include "ec.cuh"

namespace b200 {

constexpr int FB_C = 8;
constexpr int FB_W = 32;
constexpr int FB_ROW = 255;

// thread (w, d): T[w][d-1] = d * 2^(8w) * B, affine
template <class F>
__global__ void __launch_bounds__(256) k_fb_table(Affine<F> base, Affine<F>* __restrict__ table) {
  int w = blockIdx.x;
  uint32_t d = threadIdx.x + 1;
  if (d > FB_ROW) return;
  XYZZ<F> b = XYZZ<F>::from_affine(base);
  for (int i = 0; i < w * FB_C; i++) b.dbl();
  b.mul_small(d, FB_C);
  table[w * FB_ROW + d - 1] = b.to_affine();
}

template <class F>
__global__ void __launch_bounds__(128) k_fb_mul(const Affine<F>* __restrict__ table, const Fr* __restrict__ scalars,
                                                 uint32_t n, Affine<F>* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr s = Fr::from_mont(scalars[i]);
  XYZZ<F> acc = XYZZ<F>::inf();
#pragma unroll 1
  for (int w = 0; w < FB_W; w++) {
    uint32_t d = (s.l[w >> 2] >> ((w & 3) * 8)) & 0xffu;
    if (d) acc.madd(table[w * FB_ROW + d - 1]);
  }
  out[i] = acc.to_affine();
}

// Enqueue the window table of `base` (fixed_base_table_points() points) on ctx->stream.
template <class F>
int fixed_base_table_device(b200g16_ctx* ctx, const Affine<F>& base, Affine<F>* d_table) {
  k_fb_table<F><<<FB_W, 256, 0, ctx->stream>>>(base, d_table);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

// Enqueue out[i] = scalars[i] * base over a table built by fixed_base_table_device (no synchronisation).
template <class F>
int fixed_base_mul_table_device(b200g16_ctx* ctx, const Affine<F>* d_table, const Fr* d_scalars, size_t n,
                                Affine<F>* d_out) {
  if (n == 0) return 0;
  if (n >= (1ull << 32)) return fail(B200G16_ERR_ARG, "fixed_base: n too large");
  k_fb_mul<F><<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(d_table, d_scalars, (uint32_t)n, d_out);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

size_t fixed_base_table_points() { return (size_t)FB_W * FB_ROW; }

template <class F>
int fixed_base_mul_device(b200g16_ctx* ctx, const Affine<F>& base, const Fr* d_scalars, size_t n, Affine<F>* d_out) {
  if (n == 0) return 0;
  if (n >= (1ull << 32)) return fail(B200G16_ERR_ARG, "fixed_base: n too large");
  B200_TRY(ctx->io_c.ensure(fixed_base_table_points() * sizeof(Affine<F>)));
  Affine<F>* table = ctx->io_c.as<Affine<F>>();
  B200_TRY(fixed_base_table_device<F>(ctx, base, table));
  B200_TRY(fixed_base_mul_table_device<F>(ctx, table, d_scalars, n, d_out));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

template int fixed_base_mul_device<Fp>(b200g16_ctx*, const Affine<Fp>&, const Fr*, size_t, Affine<Fp>*);
template int fixed_base_mul_device<Fp2>(b200g16_ctx*, const Affine<Fp2>&, const Fr*, size_t, Affine<Fp2>*);
template int fixed_base_table_device<Fp>(b200g16_ctx*, const Affine<Fp>&, Affine<Fp>*);
template int fixed_base_table_device<Fp2>(b200g16_ctx*, const Affine<Fp2>&, Affine<Fp2>*);
template int fixed_base_mul_table_device<Fp>(b200g16_ctx*, const Affine<Fp>*, const Fr*, size_t, Affine<Fp>*);
template int fixed_base_mul_table_device<Fp2>(b200g16_ctx*, const Affine<Fp2>*, const Fr*, size_t, Affine<Fp2>*);

// ---- integer-pipe probe: `chains` independent dependent-multiply chains per thread ----------
template <int CHAINS>
__global__ void __launch_bounds__(128) k_modmul_probe(Fp* __restrict__ data, int iters) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  Fp x[CHAINS];
  Fp y = data[i];
#pragma unroll
  for (int k = 0; k < CHAINS; k++) { x[k] = y; x[k].l[0] ^= (uint32_t)k; }
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int k = 0; k < CHAINS; k++) x[k] = Fp::mul(x[k], y);
  }
  Fp r = x[0];
#pragma unroll
  for (int k = 1; k < CHAINS; k++) r = Fp::add(r, x[k]);
  data[i] = r;
}

int modmul_probe(b200g16_ctx* ctx, int blocks_per_sm, int chains, int iters, double* modmul_per_s, float* ms_out) {
  size_t threads = (size_t)ctx->sm_count * blocks_per_sm * 128;
  B200_TRY(ctx->io_a.ensure(threads * sizeof(Fp)));
  B200_CUDA(cudaMemsetAsync(ctx->io_a.p, 0x1a, threads * sizeof(Fp), ctx->stream));
  Fp* d = ctx->io_a.as<Fp>();
  unsigned grid = (unsigned)(threads / 128);
  auto launch = [&]() {
    switch (chains) {
      case 1: k_modmul_probe<1><<<grid, 128, 0, ctx->stream>>>(d, iters); break;
      case 2: k_modmul_probe<2><<<grid, 128, 0, ctx->stream>>>(d, iters); break;
      default: k_modmul_probe<4><<<grid, 128, 0, ctx->stream>>>(d, iters); chains = 4; break;
    }
  };
  launch();  // warm-up
  cudaEventRecord(ctx->ev[0], ctx->stream);
  launch();
  cudaEventRecord(ctx->ev[1], ctx->stream);
  ctx->launches += 2;
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  *ms_out = ms;
  *modmul_per_s = (double)threads * chains * iters / (ms * 1e-3);
  return 0;
}

}  // namespace b200
