// zkm_kzg_ops.cuh -- what zkm_api.cu needs of the batch-opening kernels (zkm_kzg.cuh): the term records the kernels read
// and the per-field launchers.
#pragma once
#include "zkm_common.cuh"

namespace zkm {
// One term of a linear combination: `n` Montgomery coefficients at device address `ptr`, scaled by `coeff` (Montgomery,
// fr_words used).  Records are 64 bytes, so `coeff` is 16-byte aligned in a 16-byte aligned array.
struct KzgLcTerm {
    uint64_t ptr, n;
    uint64_t coeff[6];
};
// One evaluation: the polynomial of `n` coefficients at `ptr`, at points[point].
struct KzgEvalTerm {
    uint64_t ptr, n, point, pad;
};
struct KzgOps {
    // d_out[i] = sum_t terms[t].coeff * p_t[i] for i < len (p_t[i] = 0 beyond its n)
    void (*lincomb)(Context* c, const KzgLcTerm* d_terms, uint32_t nterms, uint64_t len, uint64_t* d_out, cudaStream_t s);
    // d_w[i] += d_q[i] for i < n
    void (*shift_add)(Context* c, const uint64_t* d_q, uint64_t n, uint64_t* d_w, cudaStream_t s);
    // d_out[t] = p_t(points[t.point]); d_partial: nterms * blocks elements, d_tickets: nterms zeroed words (left zeroed)
    void (*eval_many)(Context* c, const KzgEvalTerm* d_terms, uint32_t nterms, unsigned blocks, const uint64_t* d_points,
                      uint64_t* d_partial, uint32_t* d_tickets, uint64_t* d_out, cudaStream_t s);
};
KzgOps kzg_ops(int curve);

// CTAs per term of k_kzg_eval_many: at most one chunk of 32 coefficients per thread for the longest term, and about two
// CTAs per SM over all terms
inline unsigned kzg_eval_blocks(int sm_count, uint32_t nterms, uint64_t max_n) {
    uint64_t b = (max_n + 32 * 256 - 1) / (32 * 256);
    const uint64_t cap = ((uint64_t)sm_count * 2 + nterms - 1) / (nterms ? nterms : 1);
    if (b > cap) b = cap;
    return (unsigned)(b ? b : 1);
}

}  // namespace zkm
