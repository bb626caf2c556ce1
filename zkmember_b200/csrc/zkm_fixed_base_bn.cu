// zkm_fixed_base_bn.cu -- fixed-base batch scalar multiplication (zkm_fixed_base.cuh) for BN254 G1 / G2.
#include "zkm_fixed_base.cuh"

namespace zkm {

void fixed_base_run_bn(Context* c, int group, const uint64_t* base_xy, bool base_inf, const uint64_t* d_scalars, size_t n,
                       uint64_t* d_out_xy, uint8_t* d_out_inf, uint32_t* d_flag, cudaStream_t s) {
    if (group == 1) FixedBaseImpl<G1Bn>::run(c, base_xy, base_inf, d_scalars, n, d_out_xy, d_out_inf, d_flag, s);
    else FixedBaseImpl<G2Bn>::run(c, base_xy, base_inf, d_scalars, n, d_out_xy, d_out_inf, d_flag, s);
}

}  // namespace zkm
