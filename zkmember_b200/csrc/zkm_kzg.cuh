// zkm_kzg.cuh -- the O(n) scalar-field kernels of a batch KZG opening (ark-poly-commit 0.3.0 MarlinKZG10
// open_combinations / batch_open; see DESIGN.md §13).  The division by (X - z) is linear, so a batch opening never
// divides one polynomial per term: for each point and each distinct shift s the terms' polynomials are first combined,
//   k_kzg_lincomb     P(X) = sum_t c_t p_t(X)                  one thread per output coefficient, one coalesced pass
// P is divided once (kzg_quotient_t of zkm_ntt.cuh), and
//   k_kzg_shift_add   w[s + i] += q[i]                         X^s q(X) accumulated into the point's witness vector
// The evaluations p_t(z_t) of every term come from one launch,
//   k_kzg_eval_many   blocked Horner per chunk of ZKM_EVAL_L coefficients, chunk c weighted by z^(c L), a CTA sum,
//                     and the last CTA of a term adds the CTAs' partial sums (ticket counter, reset for the next call)
// All values are Montgomery Fr elements; the results are exact, so the bytes equal any other evaluation order.
#pragma once
#include "zkm_kzg_ops.cuh"

namespace zkm {

constexpr int ZKM_EVAL_L = 32;      // coefficients per Horner chunk
constexpr int ZKM_EVAL_T = 256;     // threads per CTA

template <class P>
__global__ void __launch_bounds__(256) k_kzg_lincomb(const KzgLcTerm* __restrict__ terms, uint32_t nterms, uint64_t len,
                                                     uint32_t* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (uint64_t)gridDim.x * blockDim.x) {
        Fp<P> acc = Fp<P>::zero();
        for (uint32_t t = 0; t < nterms; t++) {
            if (i >= terms[t].n) continue;
            const Fp<P> c = ld_fp<P>(terms[t].coeff);
            acc = fp_add(acc, fp_mul(c, ld_fp<P>((const uint32_t*)terms[t].ptr + i * P::N)));
        }
        st_fp<P>(out + i * P::N, acc);
    }
}

template <class P>
__global__ void __launch_bounds__(256) k_kzg_shift_add(const uint32_t* __restrict__ q, uint64_t n, uint32_t* __restrict__ w) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        st_fp<P>(w + i * P::N, fp_add(ld_fp_plain<P>(w + i * P::N), ld_fp<P>(q + i * P::N)));
}

// grid (blocks per term, terms); partial: terms x gridDim.x elements; tickets: terms words, zero on entry and on exit
template <class P>
__global__ void __launch_bounds__(ZKM_EVAL_T) k_kzg_eval_many(const KzgEvalTerm* __restrict__ terms, const uint32_t* __restrict__ points,
                                                              uint32_t* __restrict__ partial, uint32_t* __restrict__ tickets,
                                                              uint32_t* __restrict__ out) {
    __shared__ uint4 red_smem[ZKM_EVAL_T * P::N / 4];
    __shared__ bool last;
    uint32_t* red = reinterpret_cast<uint32_t*>(red_smem);
    const KzgEvalTerm tm = terms[blockIdx.y];
    const uint32_t* p = (const uint32_t*)tm.ptr;
    const Fp<P> z = ld_fp<P>(points + tm.point * P::N);
    Fp<P> zL = z;
    for (int i = 1; i < ZKM_EVAL_L; i <<= 1) zL = fp_sqr(zL);            // z^L, L a power of two
    const uint64_t nchunks = (tm.n + ZKM_EVAL_L - 1) / ZKM_EVAL_L;
    const uint64_t c0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (uint64_t)gridDim.x * blockDim.x;
    Fp<P> acc = Fp<P>::zero();
    if (c0 < nchunks) {
        Fp<P> wc = fp_pow_u64(zL, c0);                                    // z^(c L) for the thread's current chunk c
        const Fp<P> step = fp_pow_u64(zL, stride);
        for (uint64_t c = c0; c < nchunks; c += stride) {
            const uint64_t lo = c * ZKM_EVAL_L;
            Fp<P> h = Fp<P>::zero();
            for (int j = ZKM_EVAL_L - 1; j >= 0; j--) {
                h = fp_mul(h, z);
                if (lo + j < tm.n) h = fp_add(h, ld_fp<P>(p + (lo + j) * P::N));
            }
            acc = fp_add(acc, fp_mul(h, wc));
            wc = fp_mul(wc, step);
        }
    }
    st_fp<P>(red + threadIdx.x * P::N, acc);
    __syncthreads();
    for (uint32_t d = ZKM_EVAL_T / 2; d > 0; d >>= 1) {
        if (threadIdx.x < d) {
            acc = fp_add(acc, ld_fp_plain<P>(red + (threadIdx.x + d) * P::N));
            st_fp<P>(red + threadIdx.x * P::N, acc);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        st_fp<P>(partial + ((uint64_t)blockIdx.y * gridDim.x + blockIdx.x) * P::N, acc);
        __threadfence();
        last = atomicAdd(tickets + blockIdx.y, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last || threadIdx.x != 0) return;
    __threadfence();
    Fp<P> sum = Fp<P>::zero();
    for (uint32_t b = 0; b < gridDim.x; b++) {
        Fp<P> v;
        const uint32_t* src = partial + ((uint64_t)blockIdx.y * gridDim.x + b) * P::N;
        for (int k = 0; k < P::N; k++) v.l[k] = __ldcg(src + k);         // written by other CTAs: read through L2
        sum = fp_add(sum, v);
    }
    for (int k = 0; k < P::N; k++) out[(uint64_t)blockIdx.y * P::N + k] = sum.l[k];   // the caller's buffer: 4-byte aligned
    tickets[blockIdx.y] = 0;
}

inline unsigned kzg_grid(const Context* c, uint64_t n) {
    const uint64_t blocks = (n + 255) / 256, cap = (uint64_t)c->sm_count * 8;
    return (unsigned)(blocks < cap ? (blocks ? blocks : 1) : cap);
}

template <class P>
struct KzgImpl {
    static void lincomb(Context* c, const KzgLcTerm* d_terms, uint32_t nterms, uint64_t len, uint64_t* d_out, cudaStream_t s) {
        if (len == 0) return;
        ZKM_LAUNCH(k_kzg_lincomb<P>, kzg_grid(c, len), 256, 0, s, d_terms, nterms, len, (uint32_t*)d_out);
    }
    static void shift_add(Context* c, const uint64_t* d_q, uint64_t n, uint64_t* d_w, cudaStream_t s) {
        if (n == 0) return;
        ZKM_LAUNCH(k_kzg_shift_add<P>, kzg_grid(c, n), 256, 0, s, (const uint32_t*)d_q, n, (uint32_t*)d_w);
    }
    static void eval_many(Context* c, const KzgEvalTerm* d_terms, uint32_t nterms, unsigned blocks, const uint64_t* d_points,
                          uint64_t* d_partial, uint32_t* d_tickets, uint64_t* d_out, cudaStream_t s) {
        (void)c;
        if (nterms == 0) return;
        ZKM_LAUNCH(k_kzg_eval_many<P>, dim3(blocks, nterms), ZKM_EVAL_T, 0, s, d_terms, (const uint32_t*)d_points,
                   (uint32_t*)d_partial, d_tickets, (uint32_t*)d_out);
    }
    static KzgOps ops() { return KzgOps{lincomb, shift_add, eval_many}; }
};

}  // namespace zkm
