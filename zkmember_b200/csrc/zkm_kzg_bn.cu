// zkm_kzg_bn.cu -- batch-opening kernels (zkm_kzg.cuh) for BN254 Fr.
#include "zkm_kzg.cuh"

namespace zkm {

KzgOps kzg_ops_bn() { return KzgImpl<Bn254_FrP>::ops(); }

}  // namespace zkm
