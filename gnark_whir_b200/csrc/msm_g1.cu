// G1 instantiation of the MSM back half (see msm_impl.cuh).
#include "msm_impl.cuh"
namespace b200 {
template int msm_enqueue<Fp>(b200g16_ctx*, const Affine<Fp>*, const MsmTable*, const Fr*, size_t, size_t, size_t, int, MsmCfg*,
                                   bool, bool);
template int msm_collect<Fp>(b200g16_ctx*, int, const MsmCfg&, Affine<Fp>*, size_t);
template int msm_device<Fp>(b200g16_ctx*, const Affine<Fp>*, const MsmTable*, const Fr*, size_t, Affine<Fp>*);
template int msm_build_table<Fp>(b200g16_ctx*, Affine<Fp>*, size_t, int, int);
}  // namespace b200
