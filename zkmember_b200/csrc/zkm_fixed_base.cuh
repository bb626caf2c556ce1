// zkm_fixed_base.cuh -- fixed-base batch scalar multiplication: out_i = s_i * B for ONE affine base B and n scalars,
// normalised to affine.  Replaces ark-ec 0.3.0 FixedBaseMSM::{get_mul_window_size, get_window_table,
// multi_scalar_mul} (src/msm/fixed_base.rs) + batch_normalization_into_affine, the bulk of
// Groth16::circuit_specific_setup (ark-groth16 0.3.0 src/generator.rs) and of KZG10::setup (ark-poly-commit 0.3.0
// src/kzg10/mod.rs).  Normalised affine points are unique, so the bytes equal upstream's whatever the algorithm.
//
// Pipeline (fixed launch sequence, nothing read back by the host):
//   k_fb_window_bases  one quad: P_w = 2^(c w) B for the W signed windows (c (W - 1) doublings in one chain)
//   k_fb_normalize     the W window bases to affine
//   k_fb_columns       T[w][j] = (j + 1) P_w, j < H = 2^(c - 1): one thread per run of FB_RUN entries of a column,
//                      its first entry by double-and-add (<= 2 c operations), the rest by one mixed addition each
//   k_fb_normalize     the table to affine: one inversion per FB_RUN points (Montgomery's trick)
//   k_fb_scalars       one thread per scalar: range check, into_repr, signed c-bit digits, W mixed additions of
//                      table entries (a negative digit negates y) -- no doublings, no Horner chain
//   k_fb_normalize     the outputs to affine records + infinity bytes in the caller's buffers
// Each per-curve unit zkm_fixed_base_{bls,bn,bw6}.cu instantiates FixedBaseImpl<G> for its groups.
#pragma once
#include <string.h>

#include "zkm_msm_curve.cuh"

namespace zkm {

template <class G> struct FbScalar;
template <> struct FbScalar<G1Bls> { typedef Bls12_381_FrP P; };
template <> struct FbScalar<G2Bls> { typedef Bls12_381_FrP P; };
template <> struct FbScalar<G1Bn> { typedef Bn254_FrP P; };
template <> struct FbScalar<G2Bn> { typedef Bn254_FrP P; };
template <> struct FbScalar<G1Bw6> { typedef Bw6_761_FrP P; };
template <> struct FbScalar<G2Bw6> { typedef Bw6_761_FrP P; };

// points per thread of the batched normalisation and entries per thread of a table column
constexpr uint32_t FB_RUN = 32;
// the base record travels as a kernel parameter: no host copy, so the device entry point never waits for the host
struct FbBase {
    uint64_t w[24];
};
// Context::ws slots of the fixed-base pipeline (the MSM's slots end below 32)
enum FbSlot { FB_WS_WB = 32, FB_WS_TAB, FB_WS_XYZZ, FB_WS_PRE, FB_WS_FLAG };

template <class F>
__device__ __forceinline__ F fb_ld_coord(const uint64_t* w) {
    F r;
    const uint32_t* s = reinterpret_cast<const uint32_t*>(w);
    uint32_t* d = reinterpret_cast<uint32_t*>(&r);
    for (int i = 0; i < (int)(sizeof(F) / 4); i++) d[i] = s[i];
    return r;
}

// wb[w] = 2^(c w) B, w < W; four lanes of one warp share the chain
template <class F>
__global__ void __launch_bounds__(32) k_fb_window_bases(FbBase base, int c, int W, XYZZ<F>* __restrict__ wb) {
    if (threadIdx.x >= 4 || blockIdx.x != 0) return;
    const int q = threadIdx.x;
    const uint32_t mask = 0xfu;
    constexpr int CW = CoordIO<F>::BYTES / 8;
    XYZZ<F> v = xyzz_from_affine(fb_ld_coord<F>(base.w), fb_ld_coord<F>(base.w + CW));
    for (int w = 0; w < W; w++) {
        if (w > 0)
            for (int k = 0; k < c; k++) xyzz_dbl_quad(v, q, mask);
        if (q == 0) st_xyzz(wb + w, v);
    }
}

// Batched normalisation of n XYZZ points: thread t takes points t, t + T, t + 2T, ... (T threads: coalesced), keeps the
// prefix products of d_i = ZZ_i ZZZ_i in pre[], inverts the product once and unwinds: x = X ZZZ / d, y = Y ZZ / d.
// Identities are skipped and written as arkworks' zero (x = 0, y = 1, infinity byte 1); out_inf may be null (table).
template <class F>
__global__ void __launch_bounds__(128) k_fb_normalize(const XYZZ<F>* __restrict__ in, uint64_t n, uint64_t T, F* __restrict__ pre,
                                                      char* __restrict__ out_xy, uint8_t* __restrict__ out_inf) {
    constexpr int CB = CoordIO<F>::BYTES;
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    F acc = F::one();
    for (uint64_t i = t; i < n; i += T) {
        const XYZZ<F> p = ld_xyzz(in + i);
        if (p.is_identity()) continue;
        CoordIO<F>::st(pre + i, acc);
        acc = acc * (p.ZZ * p.ZZZ);
    }
    F ia = inv(acc);
    for (uint64_t k = (n - 1 - t) / T + 1; k-- > 0;) {
        const uint64_t i = t + k * T;
        const XYZZ<F> p = ld_xyzz(in + i);
        F x = F::zero(), y = F::one();
        const bool id = p.is_identity();
        if (!id) {
            const F d_inv = ia * CoordIO<F>::ld_plain(pre + i);
            ia = ia * (p.ZZ * p.ZZZ);
            x = (p.X * p.ZZZ) * d_inv;
            y = (p.Y * p.ZZ) * d_inv;
        }
        CoordIO<F>::st(out_xy + i * 2 * CB, x);
        CoordIO<F>::st(out_xy + i * 2 * CB + CB, y);
        if (out_inf) out_inf[i] = id ? 1 : 0;
    }
}

// tab[w H + j] = (j + 1) P_w for the run j in [r m, (r + 1) m) of thread (w, r), m = min(FB_RUN, H)
template <class F>
__global__ void __launch_bounds__(128) k_fb_columns(const char* __restrict__ wb_aff, int W, uint32_t H, uint32_t m,
                                                    XYZZ<F>* __restrict__ tab) {
    constexpr int CB = CoordIO<F>::BYTES;
    const uint32_t runs = H / m;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (uint64_t)W * runs) return;
    const uint32_t w = (uint32_t)(g / runs), r = (uint32_t)(g % runs);
    const F px = CoordIO<F>::ld(wb_aff + (size_t)w * 2 * CB), py = CoordIO<F>::ld(wb_aff + (size_t)w * 2 * CB + CB);
    const uint32_t k0 = r * m + 1;
    XYZZ<F> acc = XYZZ<F>::identity();
    for (int b = 31 - __clz(k0); b >= 0; b--) {
        xyzz_dbl_ni(acc);
        if ((k0 >> b) & 1) xyzz_madd_ni(acc, px, py);
    }
    XYZZ<F>* dst = tab + (size_t)w * H + (size_t)r * m;
    st_xyzz(dst, acc);
    for (uint32_t k = 1; k < m; k++) {
        xyzz_madd_ni(acc, px, py);
        st_xyzz(dst + k, acc);
    }
}

// sv B for a canonical scalar sv (SL 32-bit limbs) from the affine table of B (W rows of H entries, window c): signed
// c-bit digits, one mixed addition per non-zero digit (a negative digit negates y), no doublings
template <class F, int SL>
__device__ __forceinline__ XYZZ<F> fb_table_mul(const uint32_t* sv, const char* __restrict__ table, int c, int W, uint32_t H) {
    constexpr int CB = CoordIO<F>::BYTES;
    const uint32_t mask = (1u << c) - 1u;
    XYZZ<F> acc = XYZZ<F>::identity();
    uint32_t s[SL + 2];   // indexed by window: kept in local memory, two loads per window
    for (int k = 0; k < SL; k++) s[k] = sv[k];
    s[SL] = 0;
    s[SL + 1] = 0;
    uint32_t carry = 0;
    for (int w = 0; w < W; w++) {
        const int lo = c * w;
        const int li = lo >> 5, sh = lo & 31;
        const uint64_t two = li < SL ? ((uint64_t)s[li] | ((uint64_t)s[li + 1] << 32)) : 0ull;
        uint32_t d = (uint32_t)(two >> sh) & mask;
        d += carry;
        carry = 0;
        uint32_t neg_d = 0;
        if (d > H) {            // signed digit in [-H, H]: d - 2^c, carry one into the next window
            d = (1u << c) - d;
            neg_d = 1;
            carry = 1;
        }
        if (d == 0) continue;
        const char* p = table + ((size_t)w * H + (d - 1)) * 2 * CB;
        const F x = CoordIO<F>::ld_gather(p);
        F y = CoordIO<F>::ld_gather(p + CB);
        if (neg_d) y = neg(y);
        xyzz_madd(acc, x, y);
    }
    return acc;
}

// out[i] = s_i B from the affine table (W rows of H entries).  Scalars arrive in Montgomery form (upstream's
// &[G::ScalarField]); `flag` (may be null) gets bit 0 when one is not < r.  base_inf: every output is the identity.
template <class G>
__global__ void __launch_bounds__(128, AccumMinBlocks<typename G::F>::value)
k_fb_scalars(const uint32_t* __restrict__ scalars, uint64_t n, const char* __restrict__ table, int c, int W, uint32_t H,
             int base_inf, XYZZ<typename G::F>* __restrict__ out, uint32_t* __restrict__ flag) {
    typedef typename G::F F;
    typedef typename FbScalar<G>::P SP;
    constexpr int SL = SP::N;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        Fp<SP> m = ld_fp<SP>(scalars + i * SL);
        if (flag) {   // canonical: m < r (top limb first)
            int cmp = 0;
            for (int k = SL - 1; k >= 0 && cmp == 0; k--) cmp = m.l[k] > SP::mod(k) ? 1 : (m.l[k] < SP::mod(k) ? -1 : 0);
            if (cmp >= 0) atomicOr(flag, 1u);
        }
        XYZZ<F> acc = XYZZ<F>::identity();
        if (!base_inf) {
            Fp<SP> one_raw = Fp<SP>::zero();
            one_raw.l[0] = 1;   // a * 1 * R^-1 = into_repr(a)
            const Fp<SP> sv = fp_mul(m, one_raw);
            acc = fb_table_mul<F, SL>(sv.l, table, c, W, H);
        }
        st_xyzz(out + i, acc);
    }
}

// Window width for n scalars: minimise n W mixed additions + the table (W H entries at ~3 additions' worth each:
// the column addition, its share of the normalisation, the XYZZ round trip), with the affine table inside 64 MB --
// half of the B200's L2, so that the random gathers of k_fb_scalars are served from there.
inline int fixed_base_window_bits(int scalar_bits, size_t rec_bytes, size_t n) {
    double best = 1e300;
    int best_c = 2;
    for (int c = 2; c <= 20; c++) {
        const int W = (scalar_bits + 1 + c - 1) / c;
        const double H = (double)(1u << (c - 1));
        if (c > 2 && (double)W * H * (double)rec_bytes > 64.0 * (1 << 20)) break;
        const double cost = (double)n * W + 3.0 * W * H;
        if (cost < best) {
            best = cost;
            best_c = c;
        }
    }
    return best_c;
}

template <class G>
struct FixedBaseImpl {
    typedef typename G::F F;
    static void normalize(Context* c, const XYZZ<F>* in, uint64_t m, char* out_xy, uint8_t* out_inf, cudaStream_t s) {
        const uint64_t T = (m + FB_RUN - 1) / FB_RUN;
        F* pre = (F*)c->ws[FB_WS_PRE].get(m * CoordIO<F>::BYTES);
        ZKM_LAUNCH(k_fb_normalize<F>, (unsigned)((T + 127) / 128), 128, 0, s, in, m, T, pre, out_xy, out_inf);
    }
    // the affine table of a finite base (host record base_xy) for window cw: W rows of H entries, written to `table`
    static void build_table(Context* c, const uint64_t* base_xy, int cw, int W, uint32_t H, char* table, cudaStream_t s) {
        constexpr int CB = CoordIO<F>::BYTES;
        constexpr size_t XB = sizeof(XYZZ<F>);
        const size_t entries = (size_t)W * H;
        FbBase b;
        memcpy(b.w, base_xy, 2 * CB);
        XYZZ<F>* wb = (XYZZ<F>*)c->ws[FB_WS_WB].get((size_t)W * (XB + 2 * CB));
        char* wb_aff = (char*)(wb + W);
        ZKM_LAUNCH(k_fb_window_bases<F>, 1, 32, 0, s, b, cw, W, wb);
        normalize(c, wb, (uint64_t)W, wb_aff, nullptr, s);
        const uint32_t m = H < FB_RUN ? H : FB_RUN;
        const uint64_t threads = (uint64_t)W * (H / m);
        XYZZ<F>* xyzz = (XYZZ<F>*)c->ws[FB_WS_XYZZ].get(entries * XB);
        ZKM_LAUNCH(k_fb_columns<F>, (unsigned)((threads + 127) / 128), 128, 0, s, (const char*)wb_aff, W, H, m, xyzz);
        normalize(c, xyzz, (uint64_t)entries, table, nullptr, s);
    }
    // base: one affine record (host memory, 2 * CB bytes); d_flag: null, or a zeroed device word for the range check
    static void run(Context* c, const uint64_t* base_xy, bool base_inf, const uint64_t* d_scalars, size_t n, uint64_t* d_out_xy,
                    uint8_t* d_out_inf, uint32_t* d_flag, cudaStream_t s) {
        constexpr int CB = CoordIO<F>::BYTES;
        constexpr size_t XB = sizeof(XYZZ<F>);
        if (n == 0) return;
        const int cw = fixed_base_window_bits(G::SCALAR_BITS, 2 * CB, n);
        const int W = (G::SCALAR_BITS + 1 + cw - 1) / cw;
        const uint32_t H = 1u << (cw - 1);
        const size_t entries = (size_t)W * H;
        char* table = (char*)c->ws[FB_WS_TAB].get(entries * 2 * CB);
        XYZZ<F>* xyzz = (XYZZ<F>*)c->ws[FB_WS_XYZZ].get((entries > n ? entries : n) * XB);
        c->ws[FB_WS_PRE].get((entries > n ? entries : n) * CB);   // sized once for the table and the outputs
        if (!base_inf) build_table(c, base_xy, cw, W, H, table, s);
        {
            const uint64_t blocks = (n + 127) / 128, cap = (uint64_t)c->sm_count * AccumMinBlocks<F>::value * 16;
            ZKM_LAUNCH(k_fb_scalars<G>, (unsigned)(blocks < cap ? blocks : cap), 128, 0, s, (const uint32_t*)d_scalars, (uint64_t)n,
                       (const char*)table, cw, W, H, base_inf ? 1 : 0, xyzz, d_flag);
        }
        normalize(c, xyzz, (uint64_t)n, (char*)d_out_xy, d_out_inf, s);
    }
};

}  // namespace zkm
