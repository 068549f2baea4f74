// G2 instantiation of the MSM back half (see msm_impl.cuh).
#include "msm_impl.cuh"
namespace b200 {
template int msm_enqueue<Fp2>(b200g16_ctx*, const Affine<Fp2>*, const MsmTable*, const Fr*, size_t, size_t, size_t, int, MsmCfg*,
                                   bool, bool);
template int msm_collect<Fp2>(b200g16_ctx*, int, const MsmCfg&, Affine<Fp2>*, size_t);
template int msm_device<Fp2>(b200g16_ctx*, const Affine<Fp2>*, const MsmTable*, const Fr*, size_t, Affine<Fp2>*);
template int msm_build_table<Fp2>(b200g16_ctx*, Affine<Fp2>*, size_t, int, int);
}  // namespace b200
