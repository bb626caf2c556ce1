// zkm_fixed_base_bls.cu -- fixed-base batch scalar multiplication (zkm_fixed_base.cuh) for BLS12-381 G1 / G2, and the
// curve dispatch of all three curves.
#include "zkm_fixed_base.cuh"

namespace zkm {

void fixed_base_run_bn(Context* c, int group, const uint64_t* base_xy, bool base_inf, const uint64_t* d_scalars, size_t n,
                       uint64_t* d_out_xy, uint8_t* d_out_inf, uint32_t* d_flag, cudaStream_t s);
void fixed_base_run_bw6(Context* c, int group, const uint64_t* base_xy, bool base_inf, const uint64_t* d_scalars, size_t n,
                        uint64_t* d_out_xy, uint8_t* d_out_inf, uint32_t* d_flag, cudaStream_t s);

void fixed_base_run(Context* c, int curve, int group, const uint64_t* base_xy, bool base_inf, const uint64_t* d_scalars, size_t n,
                    uint64_t* d_out_xy, uint8_t* d_out_inf, uint32_t* d_flag, cudaStream_t s) {
    if (curve == ZKM_CURVE_BLS12_381) {
        if (group == 1) FixedBaseImpl<G1Bls>::run(c, base_xy, base_inf, d_scalars, n, d_out_xy, d_out_inf, d_flag, s);
        else FixedBaseImpl<G2Bls>::run(c, base_xy, base_inf, d_scalars, n, d_out_xy, d_out_inf, d_flag, s);
    } else if (curve == ZKM_CURVE_BN254) {
        fixed_base_run_bn(c, group, base_xy, base_inf, d_scalars, n, d_out_xy, d_out_inf, d_flag, s);
    } else if (curve == ZKM_CURVE_BW6_761) {
        fixed_base_run_bw6(c, group, base_xy, base_inf, d_scalars, n, d_out_xy, d_out_inf, d_flag, s);
    } else {
        ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
    }
}

}  // namespace zkm
