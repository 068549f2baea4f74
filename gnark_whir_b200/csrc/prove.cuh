// Internals of the single-GPU prove shared with the multi-GPU group driver (group.cu).
#pragma once
#include "msm_impl.cuh"

namespace b200 {
int compute_h_device(b200g16_ctx* ctx, Fr* a, Fr* b, Fr* c, int L, bool sync_and_time);
int ntt_device(b200g16_ctx* ctx, Fr* d_data, int L, int batch, bool inverse, bool coset, int decimation);
int h_pointwise_device(b200g16_ctx* ctx, Fr* a, const Fr* b, const Fr* c, int L);
int ntt_coset_pair_device(b200g16_ctx* ctx, Fr* const* vecs, int batch, int L, const bool* with_den);
int h_pointwise_plain_device(b200g16_ctx* ctx, Fr* a, const Fr* b, const Fr* c, int L);
int compute_h_dist_phase(b200g16_ctx* ctx, Fr* const (*peers)[8], int g, int me, int L, int phase);
// t[0 .. count) = first * ratio^i on the device (ntt.cu)
int build_geometric(b200g16_ctx* ctx, Fr* d_t, size_t count, const Fr& first, Fr ratio);
// fixed-base multiples (fixed_base.cu): one window table per base, then any number of vectors over it, enqueued on
// ctx->stream without synchronisation
size_t fixed_base_table_points();
template <class F>
int fixed_base_table_device(b200g16_ctx* ctx, const Affine<F>& base, Affine<F>* d_table);
template <class F>
int fixed_base_mul_table_device(b200g16_ctx* ctx, const Affine<F>* d_table, const Fr* d_scalars, size_t n,
                                Affine<F>* d_out);
// instantiated in msm_g1.cu / msm_g2.cu
extern template int msm_enqueue<Fp>(b200g16_ctx*, const Affine<Fp>*, const MsmTable*, const Fr*, size_t, size_t, size_t, int, MsmCfg*,
                                   bool, bool);
extern template int msm_collect<Fp>(b200g16_ctx*, int, const MsmCfg&, Affine<Fp>*, size_t);
extern template int msm_enqueue<Fp2>(b200g16_ctx*, const Affine<Fp2>*, const MsmTable*, const Fr*, size_t, size_t, size_t, int, MsmCfg*,
                                   bool, bool);
extern template int msm_collect<Fp2>(b200g16_ctx*, int, const MsmCfg&, Affine<Fp2>*, size_t);
}  // namespace b200

struct b200g16_pk {
  int device = 0;
  unsigned log2n = 0;
  size_t n_wires = 0;
  // resident point vectors; owned[i] tells whether pk_free releases them
  b200g16_bases* vec[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // A, B1, K, Z, B2
  bool owned[5] = {false, false, false, false, false};
  b200::G1Affine alpha, beta, delta;
  b200::G2Affine beta2, delta2;
  // wire -> scalar-vector gather lists (device): A, B, K
  uint32_t* d_idx[3] = {nullptr, nullptr, nullptr};
  size_t n_idx[3] = {0, 0, 0};
  size_t off_z = 0;     // this ctx holds Z[off_z, off_z + n_z)
  size_t n_z = 0;
  bool partial = false; // shard of a key: prove returns partial MSM sums only
};

namespace b200 {
// Multiples of delta that do not depend on any MSM result (computed on the host under the GPU's work).
struct DeltaMultiples {
  G1Affine r_delta, s_delta, kr_delta;  // r*delta, s*delta, (-rs)*delta
  G2Affine s_delta2;                    // s*delta2
};
DeltaMultiples delta_multiples(const b200g16_pk* pk, const Fr& r, const Fr& s);
void prove_finish_host(const b200g16_pk* pk, const DeltaMultiples& dm, const G1Affine& A, const G1Affine& B1,
                       const G1Affine& K, const G1Affine& Z, const G2Affine& B2, const Fr& r, const Fr& s,
                       b200g16_proof* out);
int pk_build(b200g16_ctx* ctx, const b200g16_pk_desc* d, b200g16_pk** out);
void pk_release(b200g16_pk* pk);
// m proofs (a single prove: m = 1).  Gathers from the m witness rows d_wires[j * wire_stride ..) + the four witness MSMs
// enqueued on ctx->stream (no synchronisation); ev_io: next free ctx->ev slot
int prove_front(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_wires, size_t wire_stride, size_t m, int* ev_io);
// Z MSM over the m rows d_h[j * h_stride + off_z, + n_z), join, host assembly of out[0 .. m) with r[j], s[j] (or the
// five partial sums for a partial pk, m = 1)
int prove_back(b200g16_ctx* ctx, const b200g16_pk* pk, const Fr* d_h, size_t h_stride, size_t m, const Fr* r,
               const Fr* s, b200g16_proof* out, int* ev_io);
template <class F>
Affine<F> host_sum_points(const Affine<F>* pts, int n);
// The host path of b200g16_prove_batch, called under ctx->mu on ctx's device: k proofs of a whole pk from host rows
int prove_from_host(b200g16_ctx* ctx, const b200g16_pk* pk, size_t k, const uint64_t* wires, size_t n_wires,
                    const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n_constraints,
                    const uint64_t* r, const uint64_t* s, b200g16_proof* proofs_out);
// a copy of src on `device` enqueued on st (capi.cu); complete once st has passed it
int bases_copy_enqueue(int device, cudaStream_t st, const b200g16_bases* src, b200g16_bases** out);
}  // namespace b200
