// zkm_kzg_bw6.cu -- batch-opening kernels (zkm_kzg.cuh) for BW6-761 Fr.
#include "zkm_kzg.cuh"

namespace zkm {

KzgOps kzg_ops_bw6() { return KzgImpl<Bw6_761_FrP>::ops(); }

}  // namespace zkm
