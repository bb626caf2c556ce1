// zkm_groth16_bw6.cu -- Groth16 proof assembly (zkm_groth16.cuh) for BW6-761.
#include "zkm_groth16.cuh"

namespace zkm {

G16Ops groth16_ops_bw6() { return Groth16Impl<G1Bw6, G2Bw6>::ops(); }

}  // namespace zkm
