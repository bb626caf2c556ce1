// zkm_groth16_bn.cu -- Groth16 proof assembly (zkm_groth16.cuh) for BN254.
#include "zkm_groth16.cuh"

namespace zkm {

G16Ops groth16_ops_bn() { return Groth16Impl<G1Bn, G2Bn>::ops(); }

}  // namespace zkm
