// Compiles and links against include/zkm_b200.hpp + libzkm_b200.so: a Groth16 proving key on the device and one proof.
// Without a GPU every call fails with zkm::Error (no CPU fallback): exit code 0 when the error is NOT_INIT / CUDA.
#include <cstdio>

#include "zkm_b200.hpp"

int main() {
    typedef zkm::Bls12_381 C;
    try {
        zkm::init(0);
        zkm::G1Affine<C> p1{};
        zkm::G2Affine<C> p2{};
        p1.infinity = p2.infinity = true;
        std::vector<zkm::G1Affine<C>> q1(4, p1);
        std::vector<zkm::G2Affine<C>> q2(4, p2);
        zkm::Groth16ProvingKey<C> pk(p1, p1, p2, p1, p2, q1, q1, q2, std::vector<zkm::G1Affine<C>>(3, p1),
                                     std::vector<zkm::G1Affine<C>>(2, p1));
        std::vector<C::Fr> a(4), b(4), c(4);
        std::vector<C::BigInt> inputs(1), aux(2);
        C::BigInt r{}, s{};
        zkm::Proof<C> proof = zkm::create_proof(pk, r, s, a, b, c, inputs, aux);
        std::printf("proof: %zu bytes, a at infinity: %d\n", proof.serialize().size(), (int)proof.a.infinity);
        return proof.a.infinity && proof.b.infinity && proof.c.infinity ? 0 : 1;
    } catch (const zkm::Error& e) {
        std::printf("zkm::Error %d: %s\n", e.code, e.what());
        return e.code == ZKM_ERR_NOT_INIT || e.code == ZKM_ERR_CUDA ? 0 : 2;
    }
}
