// zkm_groth16.cuh -- the last step of ark-groth16 0.3.0 create_proof (src/prover.rs) on the device: the five MSM
// records of a proof plus the proving key's points in, Proof { a, b, c } out as normalised affine records.
//
//   A = r delta_1 + alpha_1 + a_0 + MSM(a_query[1..], z)
//   B = s delta_2 + beta_2  + b_0 + MSM(b_g2_query[1..], z)
//   C = s X + r Y + rs delta_1 + MSM(l_query, aux) + MSM(h_query, h)
//       with X = alpha_1 + a_0 + MSM(a_query[1..], z), Y = beta_1 + b_0 + MSM(b_g1_query[1..], z)
//
// C is upstream's s A + r B_1 - rs delta_1 regrouped: the two variable-base products need only the G1 MSMs, so they run
// while the G2 MSM is still going.  Normalised affine points are unique, so the bytes equal upstream's.
//
//   k_g16_range        assignment elements >= r -> flag word (the MSMs only see bits at or above the modulus width)
//   k_g16_assemble_g1  one CTA: warp 0 / warp 1 run s X / r Y (a quad each, ~SCALAR_BITS doublings), warp 2 the
//                      delta_1 multiples r delta_1 and rs delta_1 from the key's window table (no doublings); then A, C
//   k_g16_assemble_g2  one thread: s delta_2 from the table, B
// Each per-curve unit zkm_groth16_{bls,bn,bw6}.cu instantiates Groth16Impl for its G1 / G2 pair.
#pragma once
#include "zkm_fixed_base.cuh"
#include "zkm_groth16_ops.cuh"

namespace zkm {

// window width of the delta tables: W = ceil((bits + 1) / 8) rows of 128 entries (393 KB for BLS12-381 G1)
constexpr int G16_C = 8;

// one record of 2 CB / 8 + 1 words (8-byte aligned: read limb by limb); returns its flag word
template <class F>
__device__ __forceinline__ uint64_t g16_ld_rec(const uint64_t* r, F& x, F& y) {
    constexpr int CB = CoordIO<F>::BYTES;
    const uint32_t* r32 = reinterpret_cast<const uint32_t*>(r);
    uint32_t* xw = reinterpret_cast<uint32_t*>(&x);
    uint32_t* yw = reinterpret_cast<uint32_t*>(&y);
    for (int j = 0; j < CB / 4; j++) {
        xw[j] = r32[j];
        yw[j] = r32[CB / 4 + j];
    }
    return r[2 * CB / 8];
}

// p += record (a record at infinity adds nothing)
template <class F>
__device__ __forceinline__ void g16_add_rec(XYZZ<F>& p, const uint64_t* rec) {
    F x, y;
    if (g16_ld_rec(rec, x, y) == 0) xyzz_madd_ni(p, x, y);
}

// normalised record, limb by limb; identity -> arkworks' zero (x = 0, y = 1, flag 1); invalid -> (0, 1, flag 2)
template <class F>
__device__ void g16_st_rec(uint64_t* out, const XYZZ<F>& p, bool invalid) {
    constexpr int CB = CoordIO<F>::BYTES;
    F x, y;
    const bool ok = !invalid && xyzz_to_affine_ni(p, x, y);
    if (!ok) {
        x = F::zero();
        y = F::one();
    }
    const uint32_t* xw = reinterpret_cast<const uint32_t*>(&x);
    const uint32_t* yw = reinterpret_cast<const uint32_t*>(&y);
    uint32_t* o32 = reinterpret_cast<uint32_t*>(out);
    for (int j = 0; j < CB / 4; j++) {
        o32[j] = xw[j];
        o32[CB / 4 + j] = yw[j];
    }
    out[2 * CB / 8] = invalid ? 2ull : (ok ? 0ull : 1ull);
}

template <class SP>
__device__ __forceinline__ bool g16_canonical(const uint32_t* k) {
    for (int i = SP::N - 1; i >= 0; i--)
        if (k[i] != SP::mod(i)) return k[i] < SP::mod(i);
    return false;
}

template <class SP>
__global__ void __launch_bounds__(256) k_g16_range(const uint32_t* __restrict__ sc, uint64_t n, uint32_t* __restrict__ flag) {
    bool bad = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        bad |= !g16_canonical<SP>(sc + i * SP::N);
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}

template <class SP>
__device__ __forceinline__ bool g16_invalid(const G16Args& a, int nrec) {
    bool bad = *a.range_flag != 0 || !g16_canonical<SP>(a.r) || !g16_canonical<SP>(a.s);
    for (int i = 0; i < nrec; i++) bad |= a.rec[i][a.rec_words[i] - 1] == 2;
    return bad;
}

template <class G1, class G2>
__global__ void __launch_bounds__(96) k_g16_assemble_g1(G16Args a, const char* __restrict__ tab1) {
    typedef typename G1::F F;
    typedef typename FbScalar<G1>::P SP;
    constexpr int W = (G1::SCALAR_BITS + G16_C) / G16_C;
    __shared__ XYZZ<F> part[4];   // s X | r Y | r delta_1 | rs delta_1
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < 2 && lane < 4) {
        const int q = lane;
        const uint32_t mask = 0xfu;
        // warp 0: X = alpha + a_0 + MSM_a, times s;  warp 1: Y = beta + b_0 + MSM_b1, times r
        XYZZ<F> X = XYZZ<F>::identity();
        g16_add_rec(X, a.key1 + (warp == 0 ? G16_ALPHA : G16_BETA) * a.rec_words[G16_A]);
        g16_add_rec(X, a.key1 + (warp == 0 ? G16_A0 : G16_B0) * a.rec_words[G16_A]);
        g16_add_rec(X, a.rec[warp == 0 ? G16_A : G16_B1]);
        const uint32_t* k = warp == 0 ? a.s : a.r;
        XYZZ<F> acc = XYZZ<F>::identity();
        for (int b = G1::SCALAR_BITS - 1; b >= 0; b--) {
            xyzz_dbl_quad_inl(acc, q, mask);
            if ((k[b >> 5] >> (b & 31)) & 1) xyzz_add_quad(acc, X, q, mask);
        }
        if (q == 0) part[warp] = acc;
    } else if (warp == 2 && lane < 2) {
        Fp<SP> k;
        for (int i = 0; i < SP::N; i++) k.l[i] = a.r[i];
        if (lane == 1) {
            Fp<SP> s;
            for (int i = 0; i < SP::N; i++) s.l[i] = a.s[i];
            k = fp_mul(fp_mul(k, Fp<SP>::r2()), s);   // (r R) s R^-1 = r s mod the scalar modulus
        }
        part[2 + lane] = tab1 ? fb_table_mul<F, SP::N>(k.l, tab1, G16_C, W, 1u << (G16_C - 1)) : XYZZ<F>::identity();
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const bool invalid = g16_invalid<SP>(a, 4);
    XYZZ<F> A = part[2];
    g16_add_rec(A, a.key1 + G16_ALPHA * a.rec_words[G16_A]);
    g16_add_rec(A, a.key1 + G16_A0 * a.rec_words[G16_A]);
    g16_add_rec(A, a.rec[G16_A]);
    g16_st_rec(a.out, A, invalid);
    XYZZ<F> C = part[0];
    xyzz_add_ni(C, part[1]);
    xyzz_add_ni(C, part[3]);
    g16_add_rec(C, a.rec[G16_L]);
    g16_add_rec(C, a.rec[G16_H]);
    g16_st_rec(a.out + a.rec_words[G16_A] + a.rec_words[G16_B2], C, invalid);
}

template <class G1, class G2>
__global__ void __launch_bounds__(32) k_g16_assemble_g2(G16Args a, const char* __restrict__ tab2) {
    typedef typename G2::F F;
    typedef typename FbScalar<G2>::P SP;
    constexpr int W = (G2::SCALAR_BITS + G16_C) / G16_C;
    if (threadIdx.x != 0) return;
    const bool invalid = g16_invalid<SP>(a, 5);
    XYZZ<F> B = tab2 ? fb_table_mul<F, SP::N>(a.s, tab2, G16_C, W, 1u << (G16_C - 1)) : XYZZ<F>::identity();
    const int rw = a.rec_words[G16_B2];
    g16_add_rec(B, a.key2 + G16_BETA2 * rw);
    g16_add_rec(B, a.key2 + G16_B2_0 * rw);
    g16_add_rec(B, a.rec[G16_B2]);
    g16_st_rec(a.out + a.rec_words[G16_A], B, invalid);
}

template <class G1, class G2>
struct Groth16Impl {
    template <class G>
    static size_t table_bytes_g() {
        return (size_t)((G::SCALAR_BITS + G16_C) / G16_C) * (1u << (G16_C - 1)) * 2 * CoordIO<typename G::F>::BYTES;
    }
    static size_t table_bytes(int group) { return group == 1 ? table_bytes_g<G1>() : table_bytes_g<G2>(); }
    static void table(Context* c, int group, const uint64_t* base_xy, char* d_table, cudaStream_t s) {
        const uint32_t H = 1u << (G16_C - 1);
        if (group == 1) FixedBaseImpl<G1>::build_table(c, base_xy, G16_C, (G1::SCALAR_BITS + G16_C) / G16_C, H, d_table, s);
        else FixedBaseImpl<G2>::build_table(c, base_xy, G16_C, (G2::SCALAR_BITS + G16_C) / G16_C, H, d_table, s);
    }
    static void range(Context* c, const uint64_t* d_sc, size_t n, uint32_t* d_flag, cudaStream_t s) {
        if (n == 0) return;
        const uint64_t blocks = (n + 255) / 256, cap = (uint64_t)c->sm_count * 4;
        ZKM_LAUNCH(k_g16_range<typename FbScalar<G1>::P>, (unsigned)(blocks < cap ? blocks : cap), 256, 0, s, (const uint32_t*)d_sc,
                   (uint64_t)n, d_flag);
    }
    static void assemble(Context*, int group, const G16Args& a, const char* d_table, cudaStream_t s) {
        if (group == 1) ZKM_LAUNCH((k_g16_assemble_g1<G1, G2>), 1, 96, 0, s, a, d_table);
        else ZKM_LAUNCH((k_g16_assemble_g2<G1, G2>), 1, 32, 0, s, a, d_table);
    }
    static G16Ops ops() { return G16Ops{table_bytes, table, range, assemble}; }
};

}  // namespace zkm
