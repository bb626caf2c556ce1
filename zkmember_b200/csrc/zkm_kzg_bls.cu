// zkm_kzg_bls.cu -- batch-opening kernels (zkm_kzg.cuh) for BLS12-381 Fr, and the field dispatch of all three curves.
#include "zkm_kzg.cuh"

namespace zkm {

KzgOps kzg_ops_bn();
KzgOps kzg_ops_bw6();

KzgOps kzg_ops(int curve) {
    if (curve == ZKM_CURVE_BLS12_381) return KzgImpl<Bls12_381_FrP>::ops();
    if (curve == ZKM_CURVE_BN254) return kzg_ops_bn();
    if (curve == ZKM_CURVE_BW6_761) return kzg_ops_bw6();
    ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
}

}  // namespace zkm
