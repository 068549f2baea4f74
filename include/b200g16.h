/* libb200g16 — C-ABI of the B200-native Groth16/BN254 prover hot path.
 *
 * This is the drop-in boundary behind the three calls the reference makes at
 * /root/reference/mt.go:448 (groth16.Setup), mt.go:496 (groth16.Prove) and mt.go:497
 * (groth16.Verify): a Go package with gnark's Prove signature runs the solver in Go and
 * reaches everything after it through cgo into these entry points (INTEGRATION.md shows
 * the cgo stub).  Each function names the gnark / gnark-crypto routine it replaces
 * (gnark v0.11.0, gnark-crypto v0.14.1-0.20241217131346-b998989abdbe; go.mod:6-7 — the
 * sources are not vendored in the reference, so citations are package/func names).
 *
 * Data layout (identical to gnark-crypto's in-memory layout, so Go passes
 * unsafe.Pointer(&slice[0]) without repacking; the reference shows the same 4 x u64
 * little-endian limb convention at main.go:19-21 and typeConverters.go:26-44):
 *   fr.Element / fp.Element : uint64_t[4], little-endian limbs, MONTGOMERY form (R = 2^256)
 *   G1Affine                : uint64_t[8]  = X, Y            ; infinity = all zero
 *   G2Affine                : uint64_t[16] = X.A0, X.A1, Y.A0, Y.A1 ; infinity = all zero
 * All outputs are affine and in Montgomery form.
 *
 * Conventions
 *   - every function returns 0 on success, a negative B200G16_ERR_* otherwise;
 *     b200g16_last_error() returns a thread-local message for the last failure.
 *   - host pointers are only read/written during the call and never retained
 *     (cgo pointer rules; the one exception, b200g16_msm_g1_begin, says so); device memory is
 *     owned by the ctx / bases handles.
 *   - *_dev entry points take caller-owned DEVICE pointers.  The library works on its own
 *     non-blocking streams: the memory behind such a pointer must be READY when the call is made
 *     (work the caller has in flight on its own streams is not waited for), and every *_dev call
 *     except the _begin forms has finished with it on return.
 *   - a ctx is bound to one GPU; calls on one ctx are serialised internally, so it may
 *     be used from any OS thread (goroutines).  One process per GPU for multi-GPU.
 *   - there is NO CPU fallback: without a usable CUDA device b200g16_init fails.
 */
#ifndef B200G16_H
#define B200G16_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200G16_OK 0
#define B200G16_ERR_CUDA (-1)     /* a CUDA runtime call failed                       */
#define B200G16_ERR_ARG (-2)      /* invalid argument                                 */
#define B200G16_ERR_NO_DEVICE (-3)/* no CUDA device / wrong architecture (no fallback) */
#define B200G16_ERR_STATE (-4)    /* handle used on the wrong ctx / after free        */

#define B200G16_DIF 0 /* fft.DIF : natural-order input -> bit-reversed output */
#define B200G16_DIT 1 /* fft.DIT : bit-reversed input -> natural-order output */

typedef struct b200g16_ctx b200g16_ctx;
typedef struct b200g16_bases b200g16_bases;
typedef struct b200g16_pk b200g16_pk;

/* groth16_bn254.ProvingKey as the prover needs it (gnark backend/groth16/bn254/setup.go).
 * Each point vector is given EITHER as a host pointer (copied to the GPU once, owned by
 * the pk handle) OR as an already-resident b200g16_bases (res_*, borrowed, must outlive
 * the pk).  Lengths follow gnark: len(G1.A) = nbWires - NbInfinityA, len(G1.B) = len(G2.B)
 * = nbWires - NbInfinityB, len(G1.K) = private non-committed wires, len(G1.Z) = N - 1
 * (already bit-reversed by Setup). */
typedef struct b200g16_pk_desc {
  unsigned log2_domain;            /* pk.Domain.Cardinality = 2^log2_domain            */
  size_t n_wires;                  /* len(witness vector) = len(pk.InfinityA)           */
  const uint64_t* g1_a;            /* pk.G1.A   n_a x G1Affine                          */
  const uint64_t* g1_b;            /* pk.G1.B   n_b x G1Affine                          */
  const uint64_t* g1_k;            /* pk.G1.K   n_k x G1Affine                          */
  const uint64_t* g1_z;            /* pk.G1.Z   n_z x G1Affine                          */
  const uint64_t* g2_b;            /* pk.G2.B   n_b x G2Affine                          */
  const b200g16_bases* res_a;      /* resident alternatives (NULL = use host pointer)   */
  const b200g16_bases* res_b;
  const b200g16_bases* res_k;
  const b200g16_bases* res_z;
  const b200g16_bases* res_b2;
  size_t n_a, n_b, n_k, n_z;
  const uint64_t* g1_alpha;        /* pk.G1.Alpha, Beta, Delta : G1Affine               */
  const uint64_t* g1_beta;
  const uint64_t* g1_delta;
  const uint64_t* g2_beta;         /* pk.G2.Beta, Delta : G2Affine                      */
  const uint64_t* g2_delta;
  const uint8_t* infinity_a;       /* pk.InfinityA[n_wires] (1 = wire dropped from A)   */
  const uint8_t* infinity_b;       /* pk.InfinityB[n_wires]                             */
  const uint8_t* k_skip;           /* [n_wires] 1 = wire not in the K MSM: public wires,
                                      BSB22-committed wires and commitment wires        */
  /* Sharding across GPUs (point-range shards, one ctx per GPU).  partial = 0: the vectors are
   * the whole key and the offsets must be 0.  partial = 1: the A/B(=B2)/K/Z vectors given above
   * hold entries [off_x, off_x + n_x) of the full key vectors; b200g16_prove then returns only
   * the partial MSM sums (msm_*), to be added across GPUs and passed to b200g16_prove_finish. */
  int partial;
  size_t off_a, off_b, off_k, off_z;
  /* != 0: b200g16_pk_upload attaches window tables (b200g16_bases_precompute, automatic width)
   * to the point vectors it uploads itself; borrowed res_* vectors keep whatever they carry. */
  int precompute;
} b200g16_pk_desc;

/* Proof{Ar, Bs, Krs} plus every intermediate MSM output, for parity checks against the
 * CPU prover ("every intermediate MSM output ... must match", BASELINE.json north_star). */
typedef struct b200g16_proof {
  uint64_t ar[8];      /* proof.Ar                                  */
  uint64_t bs[16];     /* proof.Bs  (G2)                            */
  uint64_t krs[8];     /* proof.Krs                                 */
  uint64_t msm_a[8];   /* MultiExp(pk.G1.A, wireValuesA)            */
  uint64_t msm_b1[8];  /* MultiExp(pk.G1.B, wireValuesB)            */
  uint64_t msm_k[8];   /* MultiExp(pk.G1.K, private wires)          */
  uint64_t msm_z[8];   /* MultiExp(pk.G1.Z, h[:N-1])   (krs2)       */
  uint64_t msm_b2[16]; /* MultiExp(pk.G2.B, wireValuesB)            */
  uint64_t bs1[8];     /* bs1 = msm_b1 + beta + s*delta             */
} b200g16_proof;

/* ---- lifecycle ------------------------------------------------------------------ */
int b200g16_version(void);
const char* b200g16_last_error(void);
/* Bind a context to CUDA device `device` (one per process per GPU). */
int b200g16_init(int device, b200g16_ctx** out);
void b200g16_destroy(b200g16_ctx* ctx);
/* Number of CUDA kernels this ctx has launched so far (bench.py's gpu_launches). */
uint64_t b200g16_launch_count(const b200g16_ctx* ctx);
/* Device time (ms, CUDA events on the ctx stream) of the phases of the last MSM /
 * computeH / prove / setup call: writes up to `cap` floats, returns how many. */
int b200g16_last_timings(const b200g16_ctx* ctx, float* out_ms, int cap);
/* Force the Pippenger window width (0 = automatic). Testing / tuning only. */
int b200g16_set_msm_window(b200g16_ctx* ctx, int c);
/* Bucket accumulation by BATCHED-AFFINE additions (gnark-crypto's processChunkG1BatchAffine counterpart,
 * ecc/bn254/multiexp_affine.go; csrc/msm_affine.cuh): mode 0 = never (mixed XYZZ additions), 1 = for large inputs,
 * 2 = always.  levels = pair-tree levels at most (1..4, 0 keeps the current value), min_pairs = additions per
 * inversion below which a level is not run (0 keeps the current value).  The MSM result is bit-identical.  Costs
 * scratch memory (64 B x n x windows x (1 - 2^-levels) for G1: 12 GiB at n = 2^24) and is SLOWER than the default on
 * B200 for G1 (38.0 against 31.4 ms at 2^24), on par for G2: off unless set (DESIGN.md section 2). */
int b200g16_set_msm_batch_affine(b200g16_ctx* ctx, int mode, int levels, unsigned min_pairs);

/* ---- resident bases (the proving key's point vectors) ---------------------------- */
/* Copies n affine points to the GPU once; replaces the lazy device copy gnark's icicle
 * backend keeps beside groth16_bn254.ProvingKey.{G1.A,G1.B,G1.K,G1.Z,G2.B} and
 * pedersen.ProvingKey.{Basis,BasisExpSigma}. */
int b200g16_bases_upload_g1(b200g16_ctx* ctx, const uint64_t* points, size_t n, b200g16_bases** out);
int b200g16_bases_upload_g2(b200g16_ctx* ctx, const uint64_t* points, size_t n, b200g16_bases** out);
void b200g16_bases_free(b200g16_bases* bases);
size_t b200g16_bases_len(const b200g16_bases* bases);

/* Attach a WINDOW TABLE to a resident vector: the vector grows from n points to W rows of n
 * points, row k = 2^(c*k) * P_i (built on the GPU, c doublings + a shared inversion per
 * point and row).  Every later MSM on it then needs no per-window bucket sets: digit k of
 * scalar i addresses table entry (k, i), all digits accumulate into ONE set of 2^(c-1)
 * buckets, and c can be wide (20-22 at n = 2^24: 12-13 adds per point instead of 15-16)
 * because only one bucket set has to be reduced.  Costs W x the memory (n = 2^24, G1, c = 22:
 * 12 GiB of the 180 GB) and one pass at upload time — the proving key is uploaded once and
 * proved with many times.  window_bits = 0 picks c from n; otherwise 8 <= c <= 22.
 * Results are bit-identical with and without a table (tests/test_gpu_msm.py). */
int b200g16_bases_precompute(b200g16_ctx* ctx, b200g16_bases* bases, int window_bits);
/* Window width of the attached table (0 = none). */
int b200g16_bases_window(const b200g16_bases* bases);

/* The Pippenger decomposition an n-point MSM on `bases` would use: c-bit signed digits,
 * `windows` digits per scalar (= mixed additions per point).  Reporting only (bench.py). */
int b200g16_msm_plan(const b200g16_ctx* ctx, const b200g16_bases* bases, size_t n, int* window_bits, int* windows);

/* Copy points [offset, offset+n) of a resident vector back to the host (tests / sampling). */
int b200g16_bases_download(const b200g16_bases* bases, size_t offset, size_t n, uint64_t* out_points);

/* A new resident vector on ctx's device with the points of `src` (which may live on any device), including its
 * window table (the tab_W rows of a b200g16_bases_precompute'd vector) when it has one, so the copy needs no
 * precompute of its own.  The copy is device to device (cudaMemcpyPeerAsync on ctx's stream): over NVLink where the
 * devices are peers, staged by the driver otherwise; the call returns once it is complete.  The copy is independent
 * of src: either may be freed first.  A vector from setup or from a multi-device key can so reach another device
 * without a round trip through the host. */
int b200g16_bases_copy(b200g16_ctx* ctx, const b200g16_bases* src, b200g16_bases** out);

/* ---- batch fixed-base scalar multiplication (Setup's hot loop) --------------------- */
/* out_points[i] = scalars[i] * base.  Replaces gnark-crypto ecc/bn254
 * BatchScalarMultiplicationG1 / BatchScalarMultiplicationG2 as used by gnark
 * backend/groth16/bn254/setup.go (groth16.Setup, reference mt.go:448).
 * scalars: n fr.Element (Montgomery), host.  out_points: n affine points, host. */
int b200g16_fixed_base_mul_g1(b200g16_ctx* ctx, const uint64_t base[8], const uint64_t* scalars, size_t n,
                              uint64_t* out_points);
int b200g16_fixed_base_mul_g2(b200g16_ctx* ctx, const uint64_t base[16], const uint64_t* scalars, size_t n,
                              uint64_t* out_points);
/* Same, but the n results stay on the GPU as a new resident bases vector (Setup feeding
 * Prove without a round trip through the host; synthetic 2^24-point workloads). */
int b200g16_bases_from_scalars_g1(b200g16_ctx* ctx, const uint64_t base[8], const uint64_t* scalars, size_t n,
                                  b200g16_bases** out);
int b200g16_bases_from_scalars_g2(b200g16_ctx* ctx, const uint64_t base[16], const uint64_t* scalars, size_t n,
                                  b200g16_bases** out);

/* ---- integer-pipe probe -------------------------------------------------------------- */
/* Runs `chains` independent Montgomery-multiply dependency chains of length `iters` in
 * each of 128 x blocks_per_sm x #SM threads and reports modmul/s: the measured
 * integer-pipe roofline denominator for MSM / NTT (136 multiply-adds per modmul). */
int b200g16_modmul_probe(b200g16_ctx* ctx, int blocks_per_sm, int chains, int iters, double* modmul_per_s,
                         float* ms);

/* Instruction-level probe: ops/s of one integer instruction class with 8 independent chains
 * per thread.  mode 0 IMAD (mad.lo.u32), 1 IMAD.WIDE (mad.wide.u32), 2 IMAD.WIDE.X carry
 * chains (mad.lo.cc/madc.hi.cc pairs, what the Montgomery multiplier issues), 3 IMAD.HI,
 * 4 IADD3.X carry chains, 5 modes 2 and 4 interleaved (reports the wide-MAD rate),
 * 6 DFMA (fma.rz.f64), 7 DFMA + three-input 64-bit integer adds interleaved (reports the
 * DFMA rate), 8 DFMA + IMAD.WIDE.X interleaved 1:1 (reports the rate of each), 9 DADD. */
int b200g16_pipe_probe(b200g16_ctx* ctx, int mode, int blocks_per_sm, int iters, double* ops_per_s, float* ms);

/* Whole Montgomery products per second of the FP64-pipe multiplier (csrc/fp52.cuh: 5 x 52-bit
 * limbs in doubles, DFMA.RZ splitting) alone and next to the integer multiplier in the same
 * thread.  variant 0/1/2: 1/2/4 DFMA chains; 3: 1 integer + 1 DFMA chain; 4: 1 integer + 2 DFMA
 * chains; 5: 2 integer chains (same harness, for reference). */
int b200g16_fp52_probe(b200g16_ctx* ctx, int variant, int blocks_per_sm, int iters, double* modmul_per_s,
                       float* ms);

/* ---- multi-scalar multiplication -------------------------------------------------- */
/* out = sum_i scalars[i] * bases[offset + i], i < n.  Replaces gnark-crypto
 * ecc/bn254 (*G1Affine).MultiExp / (*G2Affine).MultiExp as called by gnark
 * backend/groth16/bn254/prove.go (Ar, Bs1, Krs, Krs2/Z, Bs2) and by
 * fr/pedersen ProvingKey.Commit / ProveKnowledge (the BSB22 commitment, inside Solve).
 * scalars: n fr.Element (Montgomery) in HOST memory. */
int b200g16_msm_g1(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset,
                   const uint64_t* scalars, size_t n, uint64_t out_affine[8]);
int b200g16_msm_g2(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset,
                   const uint64_t* scalars, size_t n, uint64_t out_affine[16]);
/* Same, scalars already resident in DEVICE memory (the prover feeds h straight from
 * computeH; bench.py's device-resident throughput leg). */
int b200g16_msm_g1_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset,
                       const void* d_scalars, size_t n, uint64_t out_affine[8]);
int b200g16_msm_g2_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset,
                       const void* d_scalars, size_t n, uint64_t out_affine[16]);
/* k MultiExps over ONE resident bases vector: out[j] = sum_i scalars[j*n + i] * bases[offset + i], j < k.
 * scalars: k x n fr.Elements (Montgomery), row j contiguous; out: k affine points (k x 8 words for G1, k x 16 for
 * G2).  Each out[j] equals the b200g16_msm_g1 / _g2 result on row j.  The k rows run through one pass of every MSM
 * kernel (vector j has its own bucket sets), so the sort, accumulate and bucket-reduction launches are paid once per
 * batch instead of once per vector.  One pass holds at most 2^23 buckets (k x buckets per vector) and fewer than 2^32
 * digit entries (k x n x windows); a larger k is split into sub-batches of that many vectors, run back to back in
 * one call.  k = 1, and a shape where a sub-batch would hold one vector, run the single-MSM path.
 * B200G16_ERR_ARG: NULL buffers with k > 0, k x n overflowing size_t, n >= 2^31, and the checks of b200g16_msm_g1.
 * B200G16_ERR_STATE between b200g16_prove_begin_dev and _end_dev.  k = 0 returns 0 and writes nothing.
 * b200g16_last_timings (k > 1): one value, the device time of the whole call.  Open b200g16_msm_g1_begin tickets
 * are unaffected. */
int b200g16_msm_g1_batch(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars,
                         size_t n, size_t k, uint64_t* out);
int b200g16_msm_g2_batch(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const uint64_t* scalars,
                         size_t n, size_t k, uint64_t* out);
/* Same with the k x n scalars in DEVICE memory. */
int b200g16_msm_g1_batch_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars,
                             size_t n, size_t k, uint64_t* out);
int b200g16_msm_g2_batch_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset, const void* d_scalars,
                             size_t n, size_t k, uint64_t* out);

/* Asynchronous G1 MSM: _begin enqueues it and returns a ticket (0..2; three can be open per ctx), _end waits for that
 * MSM alone and returns its result.  Calls made in between on the same ctx (b200g16_prove*, b200g16_msm_*, NTTs) run
 * behind it on the GPU while its bucket reduction overlaps them.  For gnark's prover: pedersen ProveKnowledge
 * (backend/groth16/bn254/prove.go, after Solve) can be begun before b200g16_prove and ended after it.
 * The scalars (host or device) must stay valid and unchanged until _end returns — the one place where the library
 * keeps a host pointer beyond a call (from Go: runtime.Pinner around _begin .. _end).
 * Not allowed between b200g16_prove_begin_dev and _end_dev (B200G16_ERR_STATE). */
int b200g16_msm_g1_begin(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset,
                         const uint64_t* scalars, size_t n, int* ticket);
int b200g16_msm_g1_begin_dev(b200g16_ctx* ctx, const b200g16_bases* bases, size_t offset,
                             const void* d_scalars, size_t n, int* ticket);
int b200g16_msm_g1_end(b200g16_ctx* ctx, int ticket, uint64_t out_affine[8]);

/* ---- Fr NTT / computeH -------------------------------------------------------------- */
/* In-place transform of 2^log2n fr.Elements (HOST memory) with gnark-crypto's conventions.
 * Replaces ecc/bn254/fr/fft (*Domain).FFT (inverse=0) / (*Domain).FFTInverse (inverse=1)
 * with decimation fft.DIF / fft.DIT and, when coset != 0, the fft.OnCoset() option
 * (coset shift = fr multiplicative generator 5, as fft.NewDomain defaults).
 * The domain (generator w = w28^(2^(28-log2n)), 1/N, coset tables) is derived from
 * log2n and cached on the ctx, like pk.Domain. */
int b200g16_ntt(b200g16_ctx* ctx, uint64_t* data, unsigned log2n, int inverse, int coset, int decimation);
/* Same on `batch` consecutive vectors already resident in DEVICE memory. */
int b200g16_ntt_dev(b200g16_ctx* ctx, void* d_data, unsigned log2n, unsigned batch, int inverse, int coset,
                    int decimation);
/* h = computeH(a, b, c, domain): replaces gnark backend/groth16/bn254/prove.go computeH.
 * a, b, c: n_constraints fr.Elements each (the solver's L.w, R.w, O.w; host); they are
 * zero-padded to N = 2^log2n.  h_out receives N elements in BIT-REVERSED order, exactly
 * what gnark feeds to the Z MSM (first N-1 entries). */
int b200g16_compute_h(b200g16_ctx* ctx, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                      size_t n_constraints, unsigned log2n, uint64_t* h_out);
/* Same on zero-padded DEVICE vectors of N elements; h overwrites d_a (b, c are clobbered). */
int b200g16_compute_h_dev(b200g16_ctx* ctx, void* d_a, void* d_b, void* d_c, unsigned log2n);

/* computeH split into its stages, for spreading it over several GPUs (gnark runs the three
 * FFTInverse / coset-FFT pairs of a, b, c in three goroutines; here three ranks each take one
 * vector through b200g16_ntt_dev(inverse, DIF) + b200g16_ntt_dev(coset, DIT), broadcast it, and
 * every rank finishes with this pointwise step + b200g16_ntt_dev(inverse, coset, DIF)):
 * d_a[i] = (d_a[i] * d_b[i] - d_c[i]) / (g^N - 1) on N = 2^log2n coset evaluations. */
int b200g16_h_pointwise_dev(b200g16_ctx* ctx, void* d_a, const void* d_b, const void* d_c, unsigned log2n);

/* ---- batched Keccak-f[1600] / duplex sponge / Merkle paths ---------------------------- */
/* Permute n independent 200-byte states (25 little-endian u64 lanes, lane = x + 5y) in
 * place.  Replaces gnark std/permutation/keccakf.Permute as called from the reference's
 * keccakSponge/keccakSponge.go:48,69. */
int b200g16_keccak_f_batch(b200g16_ctx* ctx, uint64_t* states, size_t n);
int b200g16_keccak_f_batch_dev(b200g16_ctx* ctx, void* d_states, size_t n);
/* n independent sponges: NewKeccak(); Absorb(inputs[i*in_len : (i+1)*in_len]);
 * Squeeze(out_len) -> outputs[i*out_len ...].  Exactly keccakSponge.Digest
 * (keccakSponge.go:17-75): rate 136, overwrite-mode absorb, no padding. */
int b200g16_keccak_sponge_batch(b200g16_ctx* ctx, const uint8_t* inputs, size_t in_len, size_t n,
                                uint8_t* outputs, size_t out_len);
/* keccakSponge.Digest between calls (keccakSponge.go:9-15): the 200-byte state as 25 little-endian lanes
 * (lane x + 5y), then the two byte positions, each in 0..136.  NewKeccak = state all zero, absorb_pos 0,
 * squeeze_pos 136.  NewKeccakWithTag(tag) is the same with tag[j] in state byte 136 + j (tag_len <= 64). */
typedef struct b200g16_keccak_digest {
  uint64_t state[25];
  uint32_t absorb_pos;
  uint32_t squeeze_pos;
} b200g16_keccak_digest; /* 208 B */
typedef struct b200g16_duplex_op {
  uint32_t squeeze; /* 0: Absorb(len bytes), 1: Squeeze(len) */
  uint32_t len;
} b200g16_duplex_op;
/* The whole Digest (keccakSponge.go:17-75: NewKeccak, NewKeccakWithTag, Absorb and Squeeze in any order) for n
 * sponges that run the same script of n_ops ops, in order, with the state carried across calls:
 *   inputs   n x A bytes, A = the sum of the absorb lengths; row i is sponge i's absorbed bytes in script order
 *   outputs  n x S bytes, S = the sum of the squeeze lengths; row i receives sponge i's squeezed bytes
 *   tag      non-NULL: every sponge starts from NewKeccakWithTag(tag[:tag_len]) (tag_len 0 = NewKeccak) and the
 *            incoming digests are not read; NULL: every sponge continues from its digest (per-sponge tags: write
 *            the bytes into fresh digests and pass tag = NULL)
 *   digests  receive the final states either way.
 * Byte rules exactly as the Digest: Absorb overwrites state byte absorb_pos (permuting first when it is 136) and
 * sets squeeze_pos = 136 when it ends, also for len 0; Squeeze permutes first when squeeze_pos is 136 (both
 * positions to 0) and emits byte squeeze_pos.  An absorbed full block stays unpermuted (absorb_pos 136) until the
 * next byte or squeeze, across calls too.  ops and tag are host memory in both calls.
 * B200G16_ERR_ARG, with nothing written: tag_len > 64, a digest position above 136 (tag == NULL), an op kind
 * other than 0 / 1, NULL inputs with A > 0 or NULL outputs with S > 0, n x A or n x S overflowing size_t.
 * n = 0 or n_ops = 0 returns 0. */
int b200g16_keccak_duplex_batch(b200g16_ctx* ctx, b200g16_keccak_digest* digests, size_t n,
                                const uint8_t* tag, size_t tag_len, const b200g16_duplex_op* ops, size_t n_ops,
                                const uint8_t* inputs, uint8_t* outputs);
/* Same with digests, inputs and outputs in DEVICE memory (d_digests 8-byte aligned; d_inputs and d_outputs
 * may have any alignment). */
int b200g16_keccak_duplex_batch_dev(b200g16_ctx* ctx, void* d_digests, size_t n,
                                    const uint8_t* tag, size_t tag_len, const b200g16_duplex_op* ops, size_t n_ops,
                                    const void* d_inputs, void* d_outputs);
/* Recompute n_paths Merkle roots.  Mirrors VerifyMerkleTreeProofs
 * (/root/reference/mtUtilities.go:109-141) with the 2-to-1 hash instantiated by the Keccak
 * duplex above (leaf hash = sponge over the leaf's bytes, node = sponge over left||right,
 * 32-byte digests):
 *   leaves      n_paths x leaf_len bytes  (leaf_len a multiple of 8; field elements are 32 B)
 *   siblings    n_paths x 32 bytes        LeafSiblingHashes (level 0)
 *   auth_paths  n_paths x (height-1) x 32 AuthPaths, leaf-side first (level k uses entry k-1)
 *   indexes     n_paths u64               leaf indexes; bit k set => node at level k is the
 *                                         RIGHT child
 *   height      tree height (= len(authPath)+1, mtUtilities.go:113)
 * roots_out (n_paths x 32, may be NULL) receives the recomputed roots; ok_out (n_paths
 * bytes, may be NULL) receives 1 where the root equals expected_root (32 bytes) — the
 * AssertIsEqual at mtUtilities.go:138. */
int b200g16_keccak_merkle_paths(b200g16_ctx* ctx, const uint8_t* leaves, size_t leaf_len,
                                const uint8_t* siblings, const uint8_t* auth_paths,
                                const uint64_t* indexes, unsigned height, size_t n_paths,
                                const uint8_t* expected_root, uint8_t* roots_out, uint8_t* ok_out);
/* Same with every buffer already in DEVICE memory (8-byte aligned). */
int b200g16_keccak_merkle_paths_dev(b200g16_ctx* ctx, const void* d_leaves, size_t leaf_len,
                                    const void* d_siblings, const void* d_auth_paths,
                                    const void* d_indexes, unsigned height, size_t n_paths,
                                    const void* d_expected_root, void* d_roots_out, void* d_ok_out);

/* ---- Groth16 prove ------------------------------------------------------------------- */
/* Upload a proving key (once; stays resident like the icicle backend's device pk). */
int b200g16_pk_upload(b200g16_ctx* ctx, const b200g16_pk_desc* desc, b200g16_pk** out);
void b200g16_pk_free(b200g16_pk* pk);
/* Everything gnark's groth16_bn254.Prove does after r1cs.Solve (backend/groth16/bn254/
 * prove.go; reference call site mt.go:496):
 *   wires  : the full solved witness vector, n_wires fr.Elements (Montgomery), host
 *   a,b,c  : solution.A/B/C = L.w, R.w, O.w per constraint, n_constraints each, host
 *   r, s   : the two blinding scalars (fr.Element, Montgomery).  gnark samples them
 *            internally; they are parameters here so proofs are reproducible bit for bit.
 * proof_out receives Ar, Bs, Krs and the intermediate MSM results; h_out (may be NULL)
 * receives computeH's output: 2^log2_domain fr.Elements, bit-reversed order. */
int b200g16_prove(b200g16_ctx* ctx, const b200g16_pk* pk, const uint64_t* wires, size_t n_wires,
                  const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints,
                  const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out, uint64_t* h_out);
/* Final assembly from the five COMPLETE MSM results (the sums over all shards):
 * Ar = A + alpha + r*delta, Bs1 = B1 + beta + s*delta, Bs = B2 + beta2 + s*delta2,
 * Krs = K + Z - rs*delta + s*Ar + r*Bs1.  Host only; any shard's pk handle supplies alpha..delta2. */
int b200g16_prove_finish(const b200g16_pk* pk, const uint64_t msm_a[8], const uint64_t msm_b1[8],
                         const uint64_t msm_k[8], const uint64_t msm_z[8], const uint64_t msm_b2[16],
                         const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out);
/* Same with wires / a / b / c already in DEVICE memory (a, b, c zero-padded to N and
 * clobbered; h is left in d_a). */
int b200g16_prove_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires, void* d_a, void* d_b,
                      void* d_c, const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out);
/* k proves of one circuit against one resident pk: proof j from wires[j] (k x n_wires), a/b/c[j] (k x n_constraints
 * each), r[j], s[j] (k x 4 each), into proofs_out[j]; every field is bit-identical to b200g16_prove on those inputs.
 * The proofs run in sub-batches: the five MSMs of a sub-batch are batch MSMs (see b200g16_msm_g1_batch; a
 * sub-batch holds as many proofs as the most constrained of the five allows), computeH runs once per proof, and
 * the host assembly runs on up to 16 threads, each step as soon as the MSM results it needs have landed.  A
 * sub-batch of one proof runs exactly as b200g16_prove.
 * B200G16_ERR_ARG: NULL buffers with k > 0, n_wires != the pk's, n_constraints > N, k x n_wires or k x N
 * overflowing, a partial (sharded) pk.  B200G16_ERR_STATE: pk on another device, between
 * b200g16_prove_begin_dev and _end_dev, or host threads that could not be started.  Any error leaves the ctx
 * usable.  k = 0 returns 0 and writes nothing.
 * b200g16_last_timings: the 8 device phases of b200g16_prove, summed over the sub-batches: upload of the witness
 * rows, gathers, MSM B2, B1, A, K, computeH (with the wait for a, b, c), and the Z MSM. */
int b200g16_prove_batch(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const uint64_t* wires, size_t n_wires,
                        const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints,
                        const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out);
/* Same with wires (k x n_wires) and a, b, c (k x N each, zero padded, clobbered; h is left in the d_a rows) in DEVICE
 * memory. */
int b200g16_prove_batch_dev(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const void* d_wires, void* d_a,
                            void* d_b, void* d_c, const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out);

/* ---- Groth16 setup ----------------------------------------------------------------------- */
/* A rank-1 constraint system as gnark's R1CS stores it (constraint/r1cs.go: a Coefficients table and, per
 * constraint, the terms Term{CID, VID} of L, R and O).  Each matrix is CSR by constraint: constraint j has the
 * entries [row[j], row[j+1]) of wire[] / coeff[]; row has n_constraints + 1 entries, row[0] = 0, and
 * nnz = row[n_constraints] is that matrix's number of terms.  A wire may appear more than once in a row (the terms
 * add up); zero coefficients and empty rows are allowed.  At most one BSB22 commitment. */
typedef struct b200g16_r1cs_desc {
  size_t n_constraints, n_wires, n_public;   /* n_public counts wire 0 (the constant one)             */
  const uint64_t* coeffs;                    /* coefficient table: n_coeffs fr.Elements (Montgomery)  */
  size_t n_coeffs;
  const uint64_t* l_row; const uint32_t* l_wire; const uint32_t* l_coeff;
  const uint64_t* r_row; const uint32_t* r_wire; const uint32_t* r_coeff;
  const uint64_t* o_row; const uint32_t* o_wire; const uint32_t* o_coeff;
  const uint32_t* private_committed;         /* committed private wires, strictly increasing          */
  size_t n_private_committed;
  int64_t commitment_wire;                   /* wire receiving the BSB22 challenge; -1: no commitment */
} b200g16_r1cs_desc;
/* The toxic waste, fr.Elements (Montgomery). */
typedef struct b200g16_toxic {
  uint64_t tau[4], alpha[4], beta[4], gamma[4], delta[4], sigma[4];
} b200g16_toxic;
/* The key b200g16_setup produces.  Point vectors are new resident bases handles the caller frees with
 * b200g16_bases_free (an empty vector is a valid n = 0 handle); they go straight into b200g16_pk_desc.res_*. */
typedef struct b200g16_setup_out {
  unsigned log2_domain;                      /* N = 2^log2_domain                                     */
  b200g16_bases* a;                          /* pk.G1.A  (G1)                                         */
  b200g16_bases* b;                          /* pk.G1.B  (G1)                                         */
  b200g16_bases* k;                          /* pk.G1.K  (G1)                                         */
  b200g16_bases* z;                          /* pk.G1.Z  (G1, N - 1 points)                           */
  b200g16_bases* b2;                         /* pk.G2.B  (G2)                                         */
  b200g16_bases* vk_k;                       /* vk.G1.K  (G1): public wires, then the commitment wire  */
  b200g16_bases* ped_basis;                  /* pedersen Basis, BasisExpSigma (G1); NULL without a     */
  b200g16_bases* ped_basis_exp_sigma;        /*   commitment                                          */
  uint64_t g1_alpha[8], g1_beta[8], g1_delta[8];
  uint64_t g2_beta[16], g2_delta[16], g2_gamma[16];
  uint64_t ped_g[16], ped_g_sigma_neg[16];   /* pedersen G = the G2 generator, GSigmaNeg = [-sigma] G  */
} b200g16_setup_out;
/* groth16.Setup (gnark backend/groth16/bn254/setup.go; reference mt.go:448) with explicit toxic waste, on the GPU
 * from the constraint matrices to the resident proving key.  The key is bit-identical to gnark's for the same toxic
 * waste:
 *   N = 2^ceil(log2 n_constraints); A_i, B_i, C_i = sum of coeff * L_j(tau) over wire i's terms of L, R, O
 *   K_i = beta A_i + alpha B_i + C_i:  public wires and then the commitment wire: K_i / gamma -> vk.G1.K;
 *     committed private wires: K_i / gamma -> pedersen Basis (committed-list order), sigma times that -> BasisExpSigma;
 *     every other wire: K_i / delta -> pk.G1.K (wire order)
 *   pk.G1.A, pk.G1.B, pk.G2.B: the wires with A_i != 0 (B_i != 0), in wire order
 *   pk.G1.Z[i] = (tau^N - 1) / delta * tau^bitrev(i), i < N - 1
 * infinity_a[i] = (A_i == 0), infinity_b[i] = (B_i == 0), k_skip[i] = 1 for public, committed and commitment wires
 * (as b200g16_pk_desc takes it): n_wires bytes each, host, written on success.
 * B200G16_ERR_ARG, with nothing left allocated: NULL arguments, n_constraints = 0 or N > 2^28, n_wires >= 2^32,
 * n_public = 0 or > n_wires, a row array that does not start at 0 or decreases, more than 15 * 2^28 terms in one matrix, a wire
 * >= n_wires, a coefficient id >= n_coeffs, a committed list that is not strictly increasing inside
 * [n_public, n_wires), a commitment wire < n_public, >= n_wires or in that list (or committed wires without one),
 * gamma = 0, delta = 0, and tau^N = 1.  The last is a deliberate deviation: gnark divides by tau - w^j and
 * would fail or produce a degenerate key; a sampled tau never hits it.  The index arrays are checked on the
 * GPU (one flag read back).  B200G16_ERR_STATE between b200g16_prove_begin_dev and _end_dev.  Any error leaves
 * the ctx usable.  The setup's scratch is its own and is released on return.
 * b200g16_last_timings: upload + checks, tau powers + Lagrange values, accumulation of L, R, O, K values +
 * compaction + Z scalars, G1 points, G2 points, flags and small points to the host. */
int b200g16_setup(b200g16_ctx* ctx, const b200g16_r1cs_desc* r1cs, const b200g16_toxic* toxic,
                  uint8_t* infinity_a, uint8_t* infinity_b, uint8_t* k_skip, b200g16_setup_out* out);
/* gnark's setupABC alone: A_i(tau), B_i(tau), C_i(tau) for every wire, n_wires fr.Elements each (host; any of the
 * three may be NULL).  The same checks as b200g16_setup on the system, except that tau^N = 1 is accepted (the
 * Lagrange values are then 0 / 1). */
int b200g16_setup_wire_polys(b200g16_ctx* ctx, const b200g16_r1cs_desc* r1cs, const uint64_t tau[4],
                             uint64_t* a_out, uint64_t* b_out, uint64_t* c_out);

/* ---- pairing / Groth16 verify ----------------------------------------------------------- */
/* groth16_bn254.VerifyingKey as Verify needs it (gnark backend/groth16/bn254/verify.go). */
typedef struct b200g16_vk_desc {
  const uint64_t* g1_alpha;         /* vk.G1.Alpha                    G1Affine              */
  const uint64_t* g2_beta;          /* vk.G2.Beta, Gamma, Delta       G2Affine              */
  const uint64_t* g2_gamma;
  const uint64_t* g2_delta;
  const uint64_t* g1_k;             /* vk.G1.K   n_k x G1Affine: K[0] is the constant-one wire,
                                       then the public inputs, then (with a commitment) its wire */
  size_t n_k;
  const uint64_t* ped_g;            /* vk.CommitmentKeys[0].G          G2Affine, NULL if none */
  const uint64_t* ped_g_sigma_neg;  /* vk.CommitmentKeys[0].GSigmaNeg  G2Affine, NULL if none */
} b200g16_vk_desc;

/* *ok_out = 1 iff prod_i e(g1_points[i], g2_points[i]) == 1.  Replaces gnark-crypto
 * ecc/bn254 PairingCheck (optimal ate: Miller loop over 6u+2 + Frobenius lines, final
 * exponentiation).  Points are checked (G1 on curve, G2 in the r-torsion subgroup); a failed
 * check is an error (B200G16_ERR_ARG), like gnark-crypto's.  Host pointers; runs on the GPU,
 * one thread per Miller loop — constant work per proof, not a throughput path. */
int b200g16_pairing_check(b200g16_ctx* ctx, const uint64_t* g1_points, const uint64_t* g2_points, size_t n,
                          int* ok_out);
/* out_gt = prod_i e(g1_points[i], g2_points[i]) as gnark-crypto's GT = E12 in memory order
 * C0.B0, C0.B1, C0.B2, C1.B0, C1.B1, C1.B2 (each E2 = A0, A1; Montgomery).  Replaces
 * ecc/bn254 Pair, including the cofactor 2u(6u^2+3u+1) its FinalExponentiation carries. */
int b200g16_pair(b200g16_ctx* ctx, const uint64_t* g1_points, const uint64_t* g2_points, size_t n,
                 uint64_t out_gt[48]);
/* groth16.Verify (reference mt.go:497; gnark backend/groth16/bn254/verify.go):
 *   public_inputs : n_public fr.Elements (Montgomery) = the public witness WITHOUT the constant
 *                   one wire, followed — when the circuit has a BSB22 commitment — by the
 *                   commitment challenge hash_to_field(commitment || committed publics), which
 *                   the caller computes (gnark_whir_b200/groth16.py commitment_challenge);
 *                   n_public + 1 must equal vk.n_k (else an error, gnark's "invalid witness size")
 *   commitment, commitment_pok : proof.Commitments[0], proof.CommitmentPok (NULL, NULL if none)
 * Checks: proof points valid (Ar, Krs on G1; Bs in the G2 subgroup), the Pedersen proof of
 * knowledge e(commitment, GSigmaNeg) e(pok, G) == 1, and
 * e(Ar, Bs) e(-kSum, gamma) e(-Krs, delta) e(-alpha, beta) == 1 with kSum = K[0] +
 * MultiExp(K[1:], public_inputs) + commitment (the MSM runs through b200g16's Pippenger).
 * *ok_out = 1 for a valid proof, 0 for an invalid one (gnark returns an error value there). */
int b200g16_verify(b200g16_ctx* ctx, const b200g16_vk_desc* vk, const uint64_t ar[8], const uint64_t bs[16],
                   const uint64_t krs[8], const uint64_t* commitment, const uint64_t* commitment_pok,
                   const uint64_t* public_inputs, size_t n_public, int* ok_out);
/* k proofs against one verifying key in one call: the small-exponent batch test (Bellare-Garay-Rabin).  With
 * coefficients rho_i (and, with commitments, independent tau_i for the proofs of knowledge) the batch is accepted iff
 * every proof point is valid (as b200g16_verify checks them) and
 *   prod_i e(rho_i Ar_i, Bs_i) e(-S alpha, beta) e(-(S K_0 + sum_j y_j K_j + sum_i rho_i D_i), gamma)
 *     e(-sum_i rho_i Krs_i, delta) e(sum_i tau_i D_i, GSigmaNeg) e(sum_i tau_i P_i, G) == 1,
 *   S = sum_i rho_i, y_j = sum_i rho_i x_ij (mod r):
 * k + 3 (k + 5) Miller loops, one per proof on its own GPU thread, and one final exponentiation.
 *   ar, bs, krs   : k x 8 / 16 / 8 words (Proof.Ar, Bs, Krs), back to back
 *   commitments, poks : k x 8 words each (Proof.Commitments[0], CommitmentPok), or both NULL; given exactly when
 *                   the vk carries the Pedersen keys
 *   public_inputs : k x n_public fr.Elements, proof i's laid out as b200g16_verify takes them (n_public + 1 == n_k)
 *   coeffs        : 128-bit little-endian integers, 2 words each: k rho_i, then (with commitments) k tau_i; nonzero
 *   ok_each       : k bytes or NULL.  All 1 when the batch passes; otherwise ok_each[i] is exactly b200g16_verify's
 *                   answer for proof i, from a per-proof pass on the GPU (costs about one b200g16_verify call, more
 *                   for large k: DESIGN.md section 6)
 * SOUNDNESS: the coefficients must be unpredictable to whoever produced the proofs (draw them from a CSPRNG after
 * the proofs are fixed).  Then a batch holding an invalid proof passes with probability about 2^-128; with
 * predictable coefficients a forger can make invalid proofs cancel each other.
 * Errors (B200G16_ERR_ARG) as b200g16_verify, plus: a zero coefficient, k > 2^20, commitments without poks or
 * Pedersen keys or the reverse.  k = 0 accepts.  B200G16_ERR_STATE while a split prove is open.  Uses the ctx's MSM
 * scratch; the ctx stays fully usable.  b200g16_last_timings: upload, per-proof kernel, fold + MSMs, fixed pairs +
 * product tree, final exponentiation[, per-proof pass]. */
int b200g16_verify_batch(b200g16_ctx* ctx, const b200g16_vk_desc* vk, size_t k, const uint64_t* ar,
                         const uint64_t* bs, const uint64_t* krs, const uint64_t* commitments, const uint64_t* poks,
                         const uint64_t* public_inputs, size_t n_public, const uint64_t* coeffs, int* ok_out,
                         uint8_t* ok_each);

/* b200g16_prove_dev with computeH already done: d_h holds h (N elements, bit-reversed order, as
 * b200g16_compute_h_dev leaves it in d_a). */
int b200g16_prove_h_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires, void* d_h,
                        const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out);

/* ---- gnark wire formats: point encodings, batched ---------------------------------------- */
/* gnark-crypto ecc/bn254/marshal.go, applied element by element by the curve Encoder / Decoder to the
 * point slices of groth16_bn254.ProvingKey / VerifyingKey / Proof (gnark backend/groth16/bn254/
 * marshal.go WriteTo / WriteRawTo / ReadFrom).  Big-endian field elements, two flag bits on top of the
 * first byte: 0b00 uncompressed, 0b01 COMPRESSED infinity, 0b10 / 0b11 compressed with the
 * lexicographically smallest / largest Y; G2 writes X.A1 before X.A0.  bn254 has two spare bits only, so
 * the uncompressed point at infinity is flag 0b00 followed by zeros (an all-zero record).  Fixed-size
 * records: raw = 0 -> compressed (G1 32 B, G2 64 B: G1Affine.Bytes / SetBytes; infinity = 0x40 then zeros),
 * raw = 1 -> uncompressed (64 / 128 B: RawBytes; infinity = all zero; a 0x40 flag is invalid here because
 * gnark's decoder would consume a compressed-size record for it — walk mixed streams record by record,
 * as gnark_whir_b200/groth16.py _PointReader does).
 * decode: ok_out[i] = 1 for a valid encoding of a curve point (and, for G2 with subgroup_check, a
 * point of the r-torsion subgroup, as the Decoder checks by default); invalid records decode to
 * infinity with ok_out[i] = 0.  Reading a compressed key costs one square root per point, which is
 * why this runs on the GPU.  Host pointers. */
int b200g16_g1_decode(b200g16_ctx* ctx, const uint8_t* in, size_t n, int raw, uint64_t* out_points, uint8_t* ok_out);
int b200g16_g2_decode(b200g16_ctx* ctx, const uint8_t* in, size_t n, int raw, int subgroup_check,
                      uint64_t* out_points, uint8_t* ok_out);
int b200g16_g1_encode(b200g16_ctx* ctx, const uint64_t* points, size_t n, int raw, uint8_t* out);
int b200g16_g2_encode(b200g16_ctx* ctx, const uint64_t* points, size_t n, int raw, uint8_t* out);

/* A prove in two halves, for callers that compute h elsewhere while the witness MSMs already run (the
 * multi-GPU prove: sharded.prove_distributed).  begin: gathers + MSM B2, B1, A, K enqueued on the ctx's
 * streams, returns WITHOUT waiting.  end: MSM Z over d_h (N elements, bit-reversed), waits, assembles
 * the proof (or, for a partial pk, the five partial sums).  One prove in flight per ctx; d_wires must
 * stay valid until end returns.  Between begin and end the ctx accepts b200g16_ntt_dev,
 * b200g16_h_pointwise_dev and b200g16_compute_h_dev (they queue behind the MSMs); every MSM, prove and
 * verify entry point returns B200G16_ERR_STATE, because the pending MSMs own the result slots. */
int b200g16_prove_begin_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_wires);
int b200g16_prove_end_dev(b200g16_ctx* ctx, const b200g16_pk* pk, const void* d_h, const uint64_t r[4],
                          const uint64_t s[4], b200g16_proof* proof_out);

/* ---- one process, several GPUs -------------------------------------------------------------------
 * gnark's prover is ONE process calling groth16.Prove once (/root/reference/mt.go:496); a group lets that
 * process spread the prove over the GPUs of a box without NCCL or helper processes.  A group owns one ctx per
 * device (peer access enabled where the hardware offers it) and drives them with one host thread per device.
 * Sharding is by point range (BASELINE.json north_star): device i holds entries [lo_i, hi_i) of every
 * proving-key vector, lo/hi balanced to within one point.  devices[] may name a device more than once
 * (several shards on one GPU: how the sharding logic is tested on a single-GPU box). */
typedef struct b200g16_group b200g16_group;
typedef struct b200g16_group_bases b200g16_group_bases;
typedef struct b200g16_group_pk b200g16_group_pk;
int b200g16_group_init(const int* devices, int n, b200g16_group** out);
void b200g16_group_destroy(b200g16_group* g);
int b200g16_group_size(const b200g16_group* g);
/* The i-th device's context (owned by the group), for single-device calls in between. */
b200g16_ctx* b200g16_group_ctx(b200g16_group* g, int i);

/* Page-lock caller memory in place (cudaHostRegister, portable): Go slices are pageable, and H2D copies from
 * pageable memory run at a fraction of PCIe speed (bench.py e2e_pageable).  Register the witness / a / b / c
 * buffers once, reuse them across proves, unregister before the slice is freed or moved. */
int b200g16_host_register(void* p, size_t bytes);
int b200g16_host_unregister(void* p);

/* Point vectors sharded over the group's devices, and MultiExp over them: each device receives its slice of
 * the scalars and runs a local Pippenger; the n partial points are added on the host (n - 1 additions).
 * n must equal the length the bases were uploaded with. */
int b200g16_group_bases_upload_g1(b200g16_group* g, const uint64_t* points, size_t n, b200g16_group_bases** out);
int b200g16_group_bases_upload_g2(b200g16_group* g, const uint64_t* points, size_t n, b200g16_group_bases** out);
int b200g16_group_bases_precompute(b200g16_group* g, b200g16_group_bases* b, int window_bits);
void b200g16_group_bases_free(b200g16_group_bases* b);
int b200g16_group_msm_g1(b200g16_group* g, const b200g16_group_bases* b, const uint64_t* scalars, size_t n, uint64_t out[8]);
int b200g16_group_msm_g2(b200g16_group* g, const b200g16_group_bases* b, const uint64_t* scalars, size_t n, uint64_t out[16]);

/* The whole proving key (host arrays, desc->partial = 0, no res_* vectors) cut into point-range shards, one
 * per device, uploaded (and given window tables when desc->precompute) in parallel. */
int b200g16_group_pk_upload(b200g16_group* g, const b200g16_pk_desc* desc, b200g16_group_pk** out);
void b200g16_group_pk_free(b200g16_group_pk* pk);
/* b200g16_prove over the group: same arguments, same result (bit-identical to the single-GPU prove).
 * a, b, c are uploaded to up to three devices (one vector each: iNTT + coset NTT there), the root device
 * receives the other two by peer copies, finishes h and every device fetches its slice of h by one peer copy
 * (cudaMemcpyPeerAsync over NVLink); the five MSMs run on every device's shard and the n x 5 partial points
 * are added on the host.  With 2, 4 or 8 devices and log2 N >= 2 log2(n) + 1, computeH is split over all the
 * devices instead (as b200g16_dist_h_* below, over peer pointers).  A group may prove keys of different sizes one
 * after another: the split computeH's slices are set up again when the domain size changes. */
int b200g16_group_prove(b200g16_group* g, const b200g16_group_pk* pk, const uint64_t* wires, size_t n_wires,
                        const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints,
                        const uint64_t r[4], const uint64_t s[4], b200g16_proof* proof_out, uint64_t* h_out);

/* ---- batch prove over a group: a whole key on every device, whole proofs per device ----------------------
 * A replicated key: the whole (non-partial) resident key `src` (b200g16_pk_upload, with or without precompute, or
 * b200g16_setup's vectors through res_*), on any device, made available on every device of the group.  Members on
 * src's device use src's point vectors without copying (src must then outlive the group key, as res_* vectors must
 * outlive a pk); every other distinct device receives one owned copy of the five vectors, window tables included,
 * shared by the members that name that device.  The copies run as a doubling broadcast: in each round every device
 * that already holds the key serves one that does not, one cudaMemcpyPeerAsync per vector on the receiver's stream
 * after a cross-device event from its source.  Every member gets its own gather lists.  Returns once every copy has
 * completed.  B200G16_ERR_ARG: NULL, a partial src.  A failed copy releases everything created so far.
 * b200g16_group_pk_free releases either kind of group key (never src). */
int b200g16_group_pk_replicate(b200g16_group* g, const b200g16_pk* src, b200g16_group_pk** out);
/* k proves of one circuit over the group, with a replicated key: the arguments, the layout (wires k x n_wires,
 * a / b / c k x n_constraints, r / s k x 4) and the per-proof results of b200g16_prove_batch, every proof
 * bit-identical to it.  Proofs are split into contiguous ranges, one per member, sizes differing by at most one; each
 * member runs b200g16_prove_batch's pipeline (with its sub-batching) on its range from its own host thread, and the
 * proofs land at their own indexes.  No data crosses devices.  Errors: those of b200g16_prove_batch (k = 0 returns 0
 * and writes nothing); a sharded key is B200G16_ERR_ARG (b200g16_group_prove likewise refuses a replicated key:
 * summing the replicas' partial proofs would give a wrong proof); a key built by another group is
 * B200G16_ERR_STATE.  A failure on one device drains every device and names that device; every ctx stays usable.
 * b200g16_last_timings on each member ctx that proved: its 8 phases, as b200g16_prove_batch reports them. */
int b200g16_group_prove_batch(b200g16_group* g, const b200g16_group_pk* pk, size_t k, const uint64_t* wires,
                              size_t n_wires, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                              size_t n_constraints, const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out);

/* ---- computeH split over 2 / 4 / 8 GPUs, one PROCESS per GPU ---------------------------------------
 * (b200g16_group_prove does the same inside one process.)  Rank `me` of n_peers holds positions
 * [me M, (me + 1) M), M = 2^log2n / n_peers, of a, b, c (zero padded) in three slice buffers owned by the library.
 * The levels of every transform whose partner lies on another GPU run as kernels over CUDA-IPC mapped peer
 * memory (NVLink loads / stores, no collective library); all other levels are ordinary size-M passes.
 *   init   allocates the slices, returns their 3 x 64-byte IPC handles (exchange them: e.g. all_gather); on a
 *          context already set up for another shape it fails with B200G16_ERR_STATE (peers may hold mapped
 *          handles of the old slices): close first
 *   open   maps every peer's slices (all_handles = n_peers x 3 x 64 bytes, rank-major)
 *   load   copies this rank's slices of a, b, c (device pointers, M elements each) into the slice buffers
 *   slice  device pointer of the local slice of a (0), b (1), c (2) (to write the inputs in place instead)
 *   phase  runs phase 0..3 on this rank and waits for it; ALL ranks must pass a barrier between consecutive
 *          phases (and between writing the inputs and phase 0).  After phase 3 slice(0) holds this rank's
 *          positions of h (bit-reversed order), which is exactly the Z shard of a point-range sharded key:
 *          pass (char*)slice(0) - 32 * off_z as d_h to b200g16_prove_h_dev / _prove_end_dev.
 *   close  unmaps and frees. */
int b200g16_dist_h_init(b200g16_ctx* ctx, unsigned log2n, int n_peers, int me, uint8_t* handles_out);
int b200g16_dist_h_open(b200g16_ctx* ctx, const uint8_t* all_handles);
int b200g16_dist_h_load(b200g16_ctx* ctx, const void* d_a, const void* d_b, const void* d_c);
void* b200g16_dist_h_slice(b200g16_ctx* ctx, int which);
int b200g16_dist_h_phase(b200g16_ctx* ctx, int phase);
void b200g16_dist_h_close(b200g16_ctx* ctx);

/* ---- small host-side group helpers (final 8-point reduction of sharded MSMs) ------ */
/* out = a + b on affine Montgomery points (handles infinity / doubling). Host only. */
int b200g16_g1_add(const uint64_t a[8], const uint64_t b[8], uint64_t out[8]);
int b200g16_g2_add(const uint64_t a[16], const uint64_t b[16], uint64_t out[16]);
/* out = k * p, k an fr.Element in Montgomery form (gnark ScalarMultiplication). Host only. */
int b200g16_g1_scalar_mul(const uint64_t p[8], const uint64_t k[4], uint64_t out[8]);
int b200g16_g2_scalar_mul(const uint64_t p[16], const uint64_t k[4], uint64_t out[16]);

#ifdef __cplusplus
}
#endif
#endif /* B200G16_H */
