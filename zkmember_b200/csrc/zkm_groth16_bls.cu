// zkm_groth16_bls.cu -- Groth16 proof assembly (zkm_groth16.cuh) for BLS12-381, and the curve dispatch of all three curves.
#include "zkm_groth16.cuh"

namespace zkm {

G16Ops groth16_ops_bn();
G16Ops groth16_ops_bw6();

G16Ops groth16_ops(int curve) {
    if (curve == ZKM_CURVE_BLS12_381) return Groth16Impl<G1Bls, G2Bls>::ops();
    if (curve == ZKM_CURVE_BN254) return groth16_ops_bn();
    if (curve == ZKM_CURVE_BW6_761) return groth16_ops_bw6();
    ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
}

}  // namespace zkm
