// Compiles and links against include/zkm_b200.hpp + libzkm_b200.so: MarlinKZG10 commitments with a shifted item and a
// batch opening at two points.  Without a GPU every call fails with zkm::Error (no CPU fallback): exit code 0 when the
// error is NOT_INIT / CUDA.
#include <cstdio>

#include "zkm_b200.hpp"

int main() {
    typedef zkm::Bls12_381 C;
    try {
        zkm::init(0);
        zkm::G1Affine<C> p1{};
        p1.infinity = true;
        zkm::RegisteredBases<C, 1> g(std::vector<zkm::G1Affine<C>>(9, p1)), gg(std::vector<zkm::G1Affine<C>>(10, p1));
        std::vector<C::Fr> p(5), b(2);
        std::vector<zkm::MarlinCommitItem<C>> items{{&p, 0, &b}, {&p, 4, &b}};
        std::vector<zkm::G1Affine<C>> comms = zkm::MarlinKZG10::commit(g, &gg, items);
        std::vector<C::Fr> points(2);
        std::vector<zkm::MarlinTerm<C>> terms{{0, 0, 0, 0, C::Fr{}}, {1, 0, -1, 4, C::Fr{}}};
        zkm::MarlinBatchProof<C> pr = zkm::MarlinKZG10::batch_open(g, &gg, {&p}, {&b}, points, terms);
        std::printf("%zu commitments, %zu proofs, %zu evaluations\n", comms.size(), pr.proofs.size(), pr.evals.size());
        return comms[0].infinity && pr.proofs[0].w.infinity ? 0 : 1;
    } catch (const zkm::Error& e) {
        std::printf("zkm::Error %d: %s\n", e.code, e.what());
        return e.code == ZKM_ERR_NOT_INIT || e.code == ZKM_ERR_CUDA ? 0 : 2;
    }
}
