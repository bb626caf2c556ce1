// zkm_b200.hpp -- header-only C++ host layer above the C ABI (include/zkm_b200.h).
//
// zkMember is compiled Rust and no Rust toolchain exists in this build environment, so the compiled-language
// host side of the drop-in is this C++ mirror of the two arkworks interfaces the hot path sits behind
// (same names, argument meaning and error behaviour); INTEGRATION.md shows the equivalent Rust shim.
//
//   zkm::VariableBaseMSM::multi_scalar_mul(bases, scalars)      ark-ec 0.3.0 src/msm/variable_base.rs
//   zkm::FixedBaseMSM::multi_scalar_mul(base, scalars)          ark-ec 0.3.0 src/msm/fixed_base.rs
//   zkm::Radix2EvaluationDomain<Curve>::new_(n) / fft / ifft / coset_fft / coset_ifft (+ _in_place)
//                                                               ark-poly 0.3.0 src/domain/radix2/mod.rs
//   zkm::witness_map(domain, a, b, c)                           ark-groth16 0.3.0 src/r1cs_to_qap.rs
//   zkm::ProvingKeyBases / KZG10::commit                        registered bases (pk / SRS reuse)
//   zkm::serialize(point) / zkm::Proof<Curve>::serialize()      arkworks' compressed CanonicalSerialize (host code)
//   zkm::Groth16ProvingKey<Curve> / zkm::create_proof            ark-groth16 0.3.0 src/prover.rs (after synthesis)
//   zkm::MarlinKZG10::{commit, batch_open}                      ark-poly-commit 0.3.0 src/marlin/marlin_pc (group side)
//
// Types are plain structs with arkworks' memory layout: Fp256 = 4 x u64 Montgomery limbs, Fp384 = 6,
// BigInteger256 = 4 x u64 canonical limbs (BigInteger384 = 6 for BW6-761), GroupAffine{x, y, infinity}.  Errors of the C ABI become
// zkm::Error exceptions (upstream's functions are infallible; there is no CPU fallback to hide behind).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <optional>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "zkm_b200.h"

namespace zkm {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int32_t rc, const char* what) {
    if (rc != ZKM_OK) throw Error(rc, std::string(what) + ": " + zkm_last_error());
}
inline void init(int device = 0) { check(zkm_init(device), "zkm_init"); }
// one process, several GPUs (bit i = CUDA device i, lowest set bit = primary): see zkm_init_mask in zkm_b200.h
inline void init_mask(uint32_t device_mask) { check(zkm_init_mask(device_mask), "zkm_init_mask"); }

template <int L64>
struct Fp {
    uint64_t limbs[L64];  // Montgomery form, little-endian limbs (ark-ff Fp256 / Fp384)
    bool operator==(const Fp& o) const { return std::memcmp(limbs, o.limbs, sizeof(limbs)) == 0; }
};
template <int L64>
struct BigInteger {
    uint64_t limbs[L64];  // canonical integer (Fr::into_repr())
};
typedef BigInteger<4> BigInteger256;
typedef BigInteger<6> BigInteger384;   // scalars of BW6-761 (377-bit Fr)
template <int L64>
struct Fp2 {
    Fp<L64> c0, c1;
};

struct Bls12_381 {
    static constexpr int ID = ZKM_CURVE_BLS12_381;
    static constexpr int TWO_ADICITY = 32;
    typedef Fp<4> Fr;
    typedef Fp<6> Fq;
    typedef Fp2<6> G2Coord;
    typedef BigInteger256 BigInt;
    static constexpr int FQ_BITS = 381;
    static const uint64_t* fq_modulus() {
        static const uint64_t m[6] = {0xb9feffffffffaaabULL, 0x1eabfffeb153ffffULL, 0x6730d2a0f6b0f624ULL, 0x64774b84f38512bfULL, 0x4b1ba7b6434bacd7ULL, 0x1a0111ea397fe69aULL};
        return m;
    }
};
struct Bn254 {
    static constexpr int ID = ZKM_CURVE_BN254;
    static constexpr int TWO_ADICITY = 28;
    typedef Fp<4> Fr;
    typedef Fp<4> Fq;
    typedef Fp2<4> G2Coord;
    typedef BigInteger256 BigInt;
    static constexpr int FQ_BITS = 254;
    static const uint64_t* fq_modulus() {
        static const uint64_t m[4] = {0x3c208c16d87cfd47ULL, 0x97816a916871ca8dULL, 0xb85045b68181585dULL, 0x30644e72e131a029ULL};
        return m;
    }
};
// The second curve zkMember instantiates (/root/reference/benches/groth16.rs:24-29): 761-bit Fq, 377-bit Fr
// (= the base field of BLS12-377), and a G2 that is a curve over Fq itself.
struct Bw6_761 {
    static constexpr int ID = ZKM_CURVE_BW6_761;
    static constexpr int TWO_ADICITY = 46;
    typedef Fp<6> Fr;
    typedef Fp<12> Fq;
    typedef Fp<12> G2Coord;
    typedef BigInteger384 BigInt;
    static constexpr int FQ_BITS = 761;
    static const uint64_t* fq_modulus() {
        static const uint64_t m[12] = {0xf49d00000000008bULL, 0xe6913e6870000082ULL, 0x160cf8aeeaf0a437ULL, 0x98a116c25667a8f8ULL, 0x71dcd3dc73ebff2eULL, 0x8689c8ed12f9fd90ULL, 0x03cebaff25b42304ULL, 0x707ba638e584e919ULL, 0x528275ef8087be41ULL, 0xb926186a81d14688ULL, 0xd187c94004faff3eULL, 0x0122e824fb83ce0aULL};
        return m;
    }
};

// GroupAffine<P>: x, y, infinity.  G1: Coord = Fq; G2: Coord = Fp2<Fq limbs> (BW6-761: Fq).
template <class Curve, int GROUP>
struct GroupAffine {
    typedef typename std::conditional<GROUP == 1, typename Curve::Fq, typename Curve::G2Coord>::type Coord;
    Coord x, y;
    bool infinity = false;
    bool operator==(const GroupAffine& o) const {
        return infinity == o.infinity && std::memcmp(&x, &o.x, sizeof(Coord)) == 0 && std::memcmp(&y, &o.y, sizeof(Coord)) == 0;
    }
};
template <class Curve> using G1Affine = GroupAffine<Curve, 1>;
template <class Curve> using G2Affine = GroupAffine<Curve, 2>;

namespace detail {
template <class Curve, int GROUP>
inline void pack(const std::vector<GroupAffine<Curve, GROUP>>& bases, size_t n, std::vector<uint64_t>& xy, std::vector<uint8_t>& inf) {
    typedef typename GroupAffine<Curve, GROUP>::Coord Coord;
    constexpr size_t W = sizeof(Coord) / 8;
    xy.resize(n * 2 * W);
    inf.resize(n);
    for (size_t i = 0; i < n; i++) {   // GroupAffine is not guaranteed packed: copy field by field
        std::memcpy(&xy[i * 2 * W], &bases[i].x, sizeof(Coord));
        std::memcpy(&xy[i * 2 * W + W], &bases[i].y, sizeof(Coord));
        inf[i] = bases[i].infinity ? 1 : 0;
    }
}
template <class Curve, int GROUP>
inline GroupAffine<Curve, GROUP> unpack(const std::vector<uint64_t>& out, uint8_t out_inf) {
    typedef typename GroupAffine<Curve, GROUP>::Coord Coord;
    constexpr size_t W = sizeof(Coord) / 8;
    GroupAffine<Curve, GROUP> r;
    std::memcpy(&r.x, &out[0], sizeof(Coord));
    std::memcpy(&r.y, &out[W], sizeof(Coord));
    r.infinity = out_inf != 0;
    return r;
}
}  // namespace detail

// Bases uploaded once (proving-key query vectors, KZG powers); `precompute` stores the window multiples.
template <class Curve, int GROUP>
class RegisteredBases {
public:
    // flags: ZKM_REG_PRECOMPUTE | ZKM_REG_SHARD | ZKM_REG_DEVICE(i) -- passed explicitly, never through a process-wide option
    RegisteredBases(const std::vector<GroupAffine<Curve, GROUP>>& bases, bool precompute = false, uint32_t flags = 0) : n_(bases.size()) {
        std::vector<uint64_t> xy;
        std::vector<uint8_t> inf;
        detail::pack<Curve, GROUP>(bases, n_, xy, inf);
        int32_t rc = zkm_bases_register_ex(Curve::ID, GROUP, xy.data(), inf.data(), n_,
                                           flags | (precompute ? ZKM_REG_PRECOMPUTE : 0u), &handle_);
        check(rc, "zkm_bases_register_ex");
    }
    ~RegisteredBases() { if (handle_) zkm_bases_release(handle_); }
    RegisteredBases(const RegisteredBases&) = delete;
    RegisteredBases& operator=(const RegisteredBases&) = delete;
    size_t size() const { return n_; }
    uint64_t handle() const { return handle_; }
    // sum over min(size() - offset, scalars.size()) pairs starting at bases[offset]
    GroupAffine<Curve, GROUP> msm(const std::vector<typename Curve::BigInt>& scalars, size_t offset = 0) const {
        size_t n = std::min(scalars.size(), n_ - std::min(offset, n_));
        typedef typename GroupAffine<Curve, GROUP>::Coord Coord;
        std::vector<uint64_t> out(2 * sizeof(Coord) / 8);
        uint8_t out_inf = 0;
        check(zkm_msm_registered(handle_, offset, reinterpret_cast<const uint64_t*>(scalars.data()), n, out.data(), &out_inf),
              "zkm_msm_registered");
        return detail::unpack<Curve, GROUP>(out, out_inf);
    }

private:
    size_t n_;
    uint64_t handle_ = 0;
};

struct VariableBaseMSM {
    // ark_ec::msm::VariableBaseMSM::multi_scalar_mul followed by into_affine()
    template <class Curve, int GROUP>
    static GroupAffine<Curve, GROUP> multi_scalar_mul(const std::vector<GroupAffine<Curve, GROUP>>& bases,
                                                      const std::vector<typename Curve::BigInt>& scalars) {
        typedef typename GroupAffine<Curve, GROUP>::Coord Coord;
        const size_t size = std::min(bases.size(), scalars.size());   // upstream: min(bases.len(), scalars.len())
        std::vector<uint64_t> xy;
        std::vector<uint8_t> inf;
        detail::pack<Curve, GROUP>(bases, size, xy, inf);
        std::vector<uint64_t> out(2 * sizeof(Coord) / 8);
        uint8_t out_inf = 0;
        const uint64_t* sc = reinterpret_cast<const uint64_t*>(scalars.data());
        int32_t rc = GROUP == 1 ? zkm_msm_g1(Curve::ID, xy.data(), inf.data(), sc, size, out.data(), &out_inf)
                                : zkm_msm_g2(Curve::ID, xy.data(), inf.data(), sc, size, out.data(), &out_inf);
        check(rc, "zkm_msm");
        return detail::unpack<Curve, GROUP>(out, out_inf);
    }
};

struct FixedBaseMSM {
    // ark_ec::msm::FixedBaseMSM::{get_window_table, multi_scalar_mul} + batch_normalization_into_affine: scalars[i] * base
    // for every Montgomery Fr element (the window width is the library's choice)
    template <class Curve, int GROUP>
    static std::vector<GroupAffine<Curve, GROUP>> multi_scalar_mul(const GroupAffine<Curve, GROUP>& base,
                                                                   const std::vector<typename Curve::Fr>& scalars) {
        typedef typename GroupAffine<Curve, GROUP>::Coord Coord;
        constexpr size_t W = sizeof(Coord) / 8;
        std::vector<uint64_t> b, xy(scalars.size() * 2 * W);
        std::vector<uint8_t> binf, inf(scalars.size());
        detail::pack<Curve, GROUP>(std::vector<GroupAffine<Curve, GROUP>>{base}, 1, b, binf);
        check(zkm_fixed_base_msm(Curve::ID, GROUP, b.data(), binf[0], reinterpret_cast<const uint64_t*>(scalars.data()),
                                 scalars.size(), xy.data(), inf.data()),
              "zkm_fixed_base_msm");
        std::vector<GroupAffine<Curve, GROUP>> out(scalars.size());
        for (size_t i = 0; i < scalars.size(); i++) {
            std::memcpy(&out[i].x, &xy[i * 2 * W], sizeof(Coord));
            std::memcpy(&out[i].y, &xy[i * 2 * W + W], sizeof(Coord));
            out[i].infinity = inf[i] != 0;
        }
        return out;
    }
};

template <class Curve>
class Radix2EvaluationDomain {
public:
    typedef typename Curve::Fr F;
    uint64_t size;
    uint32_t log_size_of_group;
    F size_inv, group_gen, group_gen_inv, generator_inv;

    // Radix2EvaluationDomain::new: None when the field has no subgroup of that order
    static std::optional<Radix2EvaluationDomain> new_(size_t num_coeffs) {
        size_t n = num_coeffs ? num_coeffs : 1;
        uint32_t log_n = 0;
        while ((size_t(1) << log_n) < n) log_n++;
        if ((int)log_n > Curve::TWO_ADICITY) return std::nullopt;
        Radix2EvaluationDomain d;
        d.size = uint64_t(1) << log_n;
        d.log_size_of_group = log_n;
        constexpr size_t S = sizeof(F) / 8;
        uint64_t c[5 * S];
        check(zkm_domain_constants(Curve::ID, log_n, c), "zkm_domain_constants");
        std::memcpy(&d.group_gen, c, sizeof(F));
        std::memcpy(&d.group_gen_inv, c + S, sizeof(F));
        std::memcpy(&d.size_inv, c + 2 * S, sizeof(F));
        std::memcpy(&d.generator_inv, c + 4 * S, sizeof(F));
        return d;
    }
    void fft_in_place(std::vector<F>& coeffs) const { run(coeffs, 0, 0); }
    void ifft_in_place(std::vector<F>& evals) const { run(evals, 1, 0); }
    void coset_fft_in_place(std::vector<F>& coeffs) const { run(coeffs, 0, 1); }
    void coset_ifft_in_place(std::vector<F>& evals) const { run(evals, 1, 1); }
    std::vector<F> fft(std::vector<F> v) const { fft_in_place(v); return v; }
    std::vector<F> ifft(std::vector<F> v) const { ifft_in_place(v); return v; }
    std::vector<F> coset_fft(std::vector<F> v) const { coset_fft_in_place(v); return v; }
    std::vector<F> coset_ifft(std::vector<F> v) const { coset_ifft_in_place(v); return v; }

private:
    void run(std::vector<F>& v, int inverse, int coset) const {
        if (v.size() > size) throw Error(ZKM_ERR_ARG, "input longer than the domain");
        F zero;
        std::memset(&zero, 0, sizeof(zero));
        v.resize(size, zero);   // upstream: coeffs.resize(self.size(), T::zero())
        check(zkm_ntt(Curve::ID, reinterpret_cast<uint64_t*>(v.data()), log_size_of_group, inverse, coset), "zkm_ntt");
    }
};

// ark_groth16::R1CStoQAP::witness_map, the part after the matrix-vector products
template <class Curve>
inline std::vector<typename Curve::Fr> witness_map(const Radix2EvaluationDomain<Curve>& d, const std::vector<typename Curve::Fr>& a,
                                                   const std::vector<typename Curve::Fr>& b, const std::vector<typename Curve::Fr>& c) {
    if (a.size() != d.size || b.size() != d.size || c.size() != d.size) throw Error(ZKM_ERR_ARG, "a, b, c must have the domain size");
    std::vector<typename Curve::Fr> h(d.size);
    check(zkm_witness_map(Curve::ID, reinterpret_cast<const uint64_t*>(a.data()), reinterpret_cast<const uint64_t*>(b.data()),
                          reinterpret_cast<const uint64_t*>(c.data()), d.log_size_of_group, reinterpret_cast<uint64_t*>(h.data())),
          "zkm_witness_map");
    return h;
}

// ark_poly_commit::kzg10 (0.3.0 src/kzg10/mod.rs): commit (with or without the hiding term), the commitments of one
// prover round in one call, and open (witness polynomial on the device).  Blinding polynomials are the caller's.
template <class Curve>
struct KZGProof {              // kzg10::Proof { w, random_v }
    G1Affine<Curve> w;
    bool hiding;
    typename Curve::Fr random_v;
};
struct KZG10 {
    template <class Curve>
    static G1Affine<Curve> commit(const RegisteredBases<Curve, 1>& powers_of_g, const std::vector<typename Curve::Fr>& coeffs) {
        std::vector<uint64_t> out(2 * sizeof(typename Curve::Fq) / 8);
        uint8_t out_inf = 0;
        check(zkm_kzg_commit(powers_of_g.handle(), reinterpret_cast<const uint64_t*>(coeffs.data()), coeffs.size(), out.data(), &out_inf),
              "zkm_kzg_commit");
        return detail::unpack<Curve, 1>(out, out_inf);
    }
    template <class Curve>
    static G1Affine<Curve> commit(const RegisteredBases<Curve, 1>& powers_of_g, const RegisteredBases<Curve, 1>& powers_of_gamma_g,
                                  const std::vector<typename Curve::Fr>& coeffs, const std::vector<typename Curve::Fr>& blinding) {
        std::vector<uint64_t> out(2 * sizeof(typename Curve::Fq) / 8);
        uint8_t out_inf = 0;
        check(zkm_kzg_commit_hiding(powers_of_g.handle(), powers_of_gamma_g.handle(), reinterpret_cast<const uint64_t*>(coeffs.data()),
                                    coeffs.size(), reinterpret_cast<const uint64_t*>(blinding.data()), blinding.size(), out.data(), &out_inf),
              "zkm_kzg_commit_hiding");
        return detail::unpack<Curve, 1>(out, out_inf);
    }
    template <class Curve>
    static std::vector<G1Affine<Curve>> commit_batch(const RegisteredBases<Curve, 1>& powers_of_g,
                                                     const std::vector<std::vector<typename Curve::Fr>>& polys) {
        const size_t W2 = 2 * sizeof(typename Curve::Fq) / 8, k = polys.size();
        std::vector<const uint64_t*> ptrs(k ? k : 1);
        std::vector<size_t> ns(k ? k : 1);
        for (size_t i = 0; i < k; i++) {
            ptrs[i] = reinterpret_cast<const uint64_t*>(polys[i].data());
            ns[i] = polys[i].size();
        }
        std::vector<uint64_t> out((k ? k : 1) * W2);
        std::vector<uint8_t> inf(k ? k : 1);
        check(zkm_kzg_commit_batch(powers_of_g.handle(), (int32_t)k, ptrs.data(), ns.data(), out.data(), inf.data()), "zkm_kzg_commit_batch");
        std::vector<G1Affine<Curve>> res;
        for (size_t i = 0; i < k; i++)
            res.push_back(detail::unpack<Curve, 1>(std::vector<uint64_t>(out.begin() + i * W2, out.begin() + (i + 1) * W2), inf[i]));
        return res;
    }
    // `powers_of_gamma_g` / `blinding` may be null / empty: non-hiding opening
    template <class Curve>
    static KZGProof<Curve> open(const RegisteredBases<Curve, 1>& powers_of_g, const std::vector<typename Curve::Fr>& coeffs,
                                const typename Curve::Fr& point, const RegisteredBases<Curve, 1>* powers_of_gamma_g = nullptr,
                                const std::vector<typename Curve::Fr>* blinding = nullptr) {
        std::vector<uint64_t> out(2 * sizeof(typename Curve::Fq) / 8);
        uint8_t out_inf = 0;
        KZGProof<Curve> pr;
        pr.hiding = powers_of_gamma_g && blinding && !blinding->empty();
        std::memset(&pr.random_v, 0, sizeof(pr.random_v));
        check(zkm_kzg_open(powers_of_g.handle(), pr.hiding ? powers_of_gamma_g->handle() : 0,
                           reinterpret_cast<const uint64_t*>(coeffs.data()), coeffs.size(),
                           pr.hiding ? reinterpret_cast<const uint64_t*>(blinding->data()) : nullptr, pr.hiding ? blinding->size() : 0,
                           reinterpret_cast<const uint64_t*>(&point), out.data(), &out_inf, reinterpret_cast<uint64_t*>(&pr.random_v)),
              "zkm_kzg_open");
        pr.w = detail::unpack<Curve, 1>(out, out_inf);
        return pr;
    }
};

// ark_poly_commit::marlin_pc (0.3.0 src/marlin/marlin_pc/mod.rs), the group side: commitments with degree-bound shifts
// and batch openings over flat lists (zkm_kzg_commit_many / zkm_kzg_open_batch).  The MarlinKZG10 bookkeeping (opening
// challenge powers, shifts D - d, linear combinations) is the caller's, as in the Python layer.
template <class Curve>
struct MarlinCommitItem {      // MSM(powers_of_g[shift + zeros ..], coeffs) + MSM(powers_of_gamma_g, blind)
    const std::vector<typename Curve::Fr>* coeffs;
    size_t shift;
    const std::vector<typename Curve::Fr>* blind;   // null or empty: no hiding term
};
template <class Curve>
struct MarlinTerm {            // c X^shift q_(polys[poly], points[point]) [+ c q_(blinds[blind], z)]
    int32_t point, poly, blind;   // blind = -1: none
    size_t shift;
    typename Curve::Fr coeff;
};
template <class Curve>
struct MarlinBatchProof {      // one kzg10::Proof per point, and poly_t(z_t) per term
    std::vector<KZGProof<Curve>> proofs;
    std::vector<typename Curve::Fr> evals;
};
struct MarlinKZG10 {
    // coefficients up to the top non-zero one (DensePolynomial drops trailing zeros; the C ABI's bound checks count
    // every coefficient it is given)
    template <class F>
    static size_t trimmed_size(const std::vector<F>& p) {
        size_t n = p.size();
        F zero;
        std::memset(&zero, 0, sizeof(zero));
        while (n && p[n - 1] == zero) n--;
        return n;
    }
    template <class Curve>
    static std::vector<G1Affine<Curve>> commit(const RegisteredBases<Curve, 1>& powers_of_g, const RegisteredBases<Curve, 1>* powers_of_gamma_g,
                                               const std::vector<MarlinCommitItem<Curve>>& items) {
        const size_t k = items.size(), W2 = 2 * sizeof(typename Curve::Fq) / 8;
        std::vector<const uint64_t*> cp(k), bp(k);
        std::vector<size_t> n(k), sh(k), nb(k);
        for (size_t i = 0; i < k; i++) {
            cp[i] = reinterpret_cast<const uint64_t*>(items[i].coeffs->data());
            n[i] = trimmed_size(*items[i].coeffs);
            sh[i] = items[i].shift;
            bp[i] = items[i].blind ? reinterpret_cast<const uint64_t*>(items[i].blind->data()) : nullptr;
            nb[i] = items[i].blind ? items[i].blind->size() : 0;
        }
        std::vector<uint64_t> out(std::max<size_t>(k, 1) * W2);
        std::vector<uint8_t> inf(std::max<size_t>(k, 1));
        check(zkm_kzg_commit_many(powers_of_g.handle(), powers_of_gamma_g ? powers_of_gamma_g->handle() : 0, (int32_t)k, cp.data(), n.data(),
                                  sh.data(), bp.data(), nb.data(), out.data(), inf.data()),
              "zkm_kzg_commit_many");
        std::vector<G1Affine<Curve>> res;
        for (size_t i = 0; i < k; i++)
            res.push_back(detail::unpack<Curve, 1>(std::vector<uint64_t>(out.begin() + i * W2, out.begin() + (i + 1) * W2), inf[i]));
        return res;
    }
    template <class Curve>
    static MarlinBatchProof<Curve> batch_open(const RegisteredBases<Curve, 1>& powers_of_g, const RegisteredBases<Curve, 1>* powers_of_gamma_g,
                                              const std::vector<const std::vector<typename Curve::Fr>*>& polys,
                                              const std::vector<const std::vector<typename Curve::Fr>*>& blinds,
                                              const std::vector<typename Curve::Fr>& points, const std::vector<MarlinTerm<Curve>>& terms) {
        typedef typename Curve::Fr F;
        const size_t W2 = 2 * sizeof(typename Curve::Fq) / 8, np = points.size(), nt = terms.size();
        std::vector<const uint64_t*> cp, bp;
        std::vector<size_t> n, nb, ts;
        for (auto* p : polys) { cp.push_back(reinterpret_cast<const uint64_t*>(p->data())); n.push_back(trimmed_size(*p)); }
        for (auto* b : blinds) { bp.push_back(reinterpret_cast<const uint64_t*>(b->data())); nb.push_back(b->size()); }
        std::vector<int32_t> tp, tq, tb;
        std::vector<F> tc;
        for (const auto& t : terms) {
            tp.push_back(t.point);
            tq.push_back(t.poly);
            tb.push_back(t.blind);
            ts.push_back(t.shift);
            tc.push_back(t.coeff);
        }
        std::vector<uint64_t> w(std::max<size_t>(np, 1) * W2);
        std::vector<uint8_t> winf(std::max<size_t>(np, 1));
        MarlinBatchProof<Curve> res;
        std::vector<F> rv(std::max<size_t>(np, 1));
        res.evals.resize(nt);
        check(zkm_kzg_open_batch(powers_of_g.handle(), powers_of_gamma_g ? powers_of_gamma_g->handle() : 0, (int32_t)polys.size(), cp.data(),
                                 n.data(), (int32_t)blinds.size(), bp.data(), nb.data(), (int32_t)np,
                                 reinterpret_cast<const uint64_t*>(points.data()), (int32_t)nt, tp.data(), tq.data(), tb.data(), ts.data(),
                                 reinterpret_cast<const uint64_t*>(tc.data()), w.data(), winf.data(), reinterpret_cast<uint64_t*>(rv.data()),
                                 reinterpret_cast<uint64_t*>(res.evals.data())),
              "zkm_kzg_open_batch");
        for (size_t i = 0; i < np; i++) {
            KZGProof<Curve> pr;
            pr.w = detail::unpack<Curve, 1>(std::vector<uint64_t>(w.begin() + i * W2, w.begin() + (i + 1) * W2), winf[i]);
            pr.hiding = false;
            for (const auto& t : terms) pr.hiding = pr.hiding || (t.point == (int32_t)i && t.blind >= 0);
            pr.random_v = rv[i];
            res.proofs.push_back(pr);
        }
        return res;
    }
};

// ---- arkworks CanonicalSerialize (compressed) for affine points and Groth16 proofs -------------------------------
// ark-ec 0.3.0 GroupAffine::serialize (src/models/short_weierstrass_jacobian.rs) + ark-ff 0.3.0
// Fp::serialize_with_flags / QuadExtField::serialize_with_flags + ark-serialize 0.3.0 SWFlags: x canonical
// little-endian in ceil((MODULUS_BITS + 2) / 8) bytes, bit 7 of the last byte = "y > -y", bit 6 = infinity; an Fp2
// writes c0 without flags and c1 with them and is ordered by c1 first.  The wire format of zkMember's proofs
// (/root/reference/src/main.rs:164-169).  Host-side glue on a handful of elements -- plain C++, no GPU involved.
namespace detail {
// out = a * R^-1 mod p (Montgomery reduction of a single element: into_repr), L limbs
template <int L>
inline void from_mont(const uint64_t* a, const uint64_t* p, uint64_t* out) {
    uint64_t inv = 1;                                   // p^-1 mod 2^64 by Newton, then negated
    for (int i = 0; i < 6; i++) inv *= 2 - p[0] * inv;
    inv = 0 - inv;
    uint64_t t[L + 1];
    for (int i = 0; i < L; i++) t[i] = a[i];
    t[L] = 0;
    for (int i = 0; i < L; i++) {
        const uint64_t m = t[0] * inv;
        unsigned __int128 carry = ((unsigned __int128)m * p[0] + t[0]) >> 64;
        for (int j = 1; j < L; j++) {
            unsigned __int128 v = (unsigned __int128)m * p[j] + t[j] + (uint64_t)carry;
            t[j - 1] = (uint64_t)v;
            carry = v >> 64;
        }
        unsigned __int128 v = (unsigned __int128)t[L] + (uint64_t)carry;
        t[L - 1] = (uint64_t)v;
        t[L] = (uint64_t)(v >> 64);
    }
    bool ge = t[L] != 0;                                // t < 2p: one conditional subtraction
    if (!ge) {
        ge = true;
        for (int i = L - 1; i >= 0; i--) {
            if (t[i] != p[i]) { ge = t[i] > p[i]; break; }
        }
    }
    uint64_t borrow = 0;
    for (int i = 0; i < L; i++) {
        if (ge) {
            unsigned __int128 d = (unsigned __int128)t[i] - p[i] - borrow;
            out[i] = (uint64_t)d;
            borrow = (uint64_t)(d >> 64) & 1;
        } else {
            out[i] = t[i];
        }
    }
}
template <int L>
inline void neg_canonical(const uint64_t* a, const uint64_t* p, uint64_t* out) {     // (p - a) mod p
    bool zero = true;
    for (int i = 0; i < L; i++) zero = zero && a[i] == 0;
    uint64_t borrow = 0;
    for (int i = 0; i < L; i++) {
        unsigned __int128 d = (unsigned __int128)p[i] - a[i] - borrow;
        out[i] = zero ? 0 : (uint64_t)d;
        borrow = (uint64_t)(d >> 64) & 1;
    }
}
template <int L>
inline int cmp_limbs(const uint64_t* a, const uint64_t* b) {
    for (int i = L - 1; i >= 0; i--)
        if (a[i] != b[i]) return a[i] > b[i] ? 1 : -1;
    return 0;
}
inline void put_le(std::vector<uint8_t>& out, const uint64_t* v, int limbs, size_t bytes) {
    for (size_t i = 0; i < bytes; i++) out.push_back((size_t)(i / 8) < (size_t)limbs ? (uint8_t)(v[i / 8] >> (8 * (i % 8))) : 0);
}
// canonical limbs of the DEG Fq elements of a coordinate (Fp: 1, Fp2: 2)
template <int L>
inline void coord_canonical(const Fp<L>& c, const uint64_t* p, uint64_t (*out)[12]) { from_mont<L>(c.limbs, p, out[0]); }
template <int L>
inline void coord_canonical(const Fp2<L>& c, const uint64_t* p, uint64_t (*out)[12]) {
    from_mont<L>(c.c0.limbs, p, out[0]);
    from_mont<L>(c.c1.limbs, p, out[1]);
}
template <int L> constexpr int coord_degree(const Fp<L>*) { return 1; }
template <int L> constexpr int coord_degree(const Fp2<L>*) { return 2; }
}  // namespace detail

template <class Curve, int GROUP>
inline std::vector<uint8_t> serialize(const GroupAffine<Curve, GROUP>& pt) {
    typedef typename GroupAffine<Curve, GROUP>::Coord Coord;
    constexpr int L = sizeof(typename Curve::Fq) / 8;
    constexpr int DEG = detail::coord_degree((const Coord*)nullptr);
    const uint64_t* p = Curve::fq_modulus();
    const size_t plain = (Curve::FQ_BITS + 7) / 8, flagged = (Curve::FQ_BITS + 2 + 7) / 8;
    uint64_t x[2][12] = {}, y[2][12] = {}, ny[2][12] = {};
    uint8_t flag;
    if (pt.infinity) {
        flag = 1u << 6;                                  // SWFlags::Infinity, x = 0
    } else {
        detail::coord_canonical(pt.x, p, x);
        detail::coord_canonical(pt.y, p, y);
        for (int d = 0; d < DEG; d++) detail::neg_canonical<L>(y[d], p, ny[d]);
        int c = 0;                                       // y > -y; Fp2: c1 first, then c0
        for (int d = DEG - 1; d >= 0 && c == 0; d--) c = detail::cmp_limbs<L>(y[d], ny[d]);
        flag = c > 0 ? (1u << 7) : 0;                    // PositiveY | NegativeY
    }
    std::vector<uint8_t> out;
    for (int d = 0; d + 1 < DEG; d++) detail::put_le(out, x[d], L, plain);
    detail::put_le(out, x[DEG - 1], L, flagged);
    out.back() |= flag;
    return out;
}

// ark_groth16::Proof { a: G1Affine, b: G2Affine, c: G1Affine }: a || b || c
template <class Curve>
struct Proof {
    G1Affine<Curve> a;
    G2Affine<Curve> b;
    G1Affine<Curve> c;
    std::vector<uint8_t> serialize() const {
        std::vector<uint8_t> out = zkm::serialize(a), sb = zkm::serialize(b), sc = zkm::serialize(c);
        out.insert(out.end(), sb.begin(), sb.end());
        out.insert(out.end(), sc.begin(), sc.end());
        return out;
    }
};

// ark_groth16::ProvingKey on the device (zkm_groth16_pk_create).  a_query, b_g1_query, b_g2_query are the FULL vectors:
// entry 0 (the constant-one variable) goes to the key as a point, entries 1.. are registered; the key keeps the
// registrations alive, the RAII members below only drop this object's own references.
template <class Curve>
class Groth16ProvingKey {
public:
    Groth16ProvingKey(const G1Affine<Curve>& alpha_g1, const G1Affine<Curve>& beta_g1, const G2Affine<Curve>& beta_g2,
                      const G1Affine<Curve>& delta_g1, const G2Affine<Curve>& delta_g2, const std::vector<G1Affine<Curve>>& a_query,
                      const std::vector<G1Affine<Curve>>& b_g1_query, const std::vector<G2Affine<Curve>>& b_g2_query,
                      const std::vector<G1Affine<Curve>>& h_query, const std::vector<G1Affine<Curve>>& l_query, bool precompute = true)
        : h_(h_query, precompute), l_(l_query, precompute), a_(tail(a_query), precompute), b1_(tail(b_g1_query), precompute),
          b2_(tail(b_g2_query), precompute) {
        const uint64_t handles[5] = {h_.handle(), l_.handle(), a_.handle(), b1_.handle(), b2_.handle()};
        std::vector<uint64_t> g1, g2;
        std::vector<uint8_t> g1_inf, g2_inf;
        detail::pack<Curve, 1>({alpha_g1, beta_g1, delta_g1, first(a_query), first(b_g1_query)}, 5, g1, g1_inf);
        detail::pack<Curve, 2>({beta_g2, delta_g2, first(b_g2_query)}, 3, g2, g2_inf);
        check(zkm_groth16_pk_create(Curve::ID, handles, g1.data(), g1_inf.data(), g2.data(), g2_inf.data(), &handle_),
              "zkm_groth16_pk_create");
    }
    ~Groth16ProvingKey() { if (handle_) zkm_groth16_pk_release(handle_); }
    Groth16ProvingKey(const Groth16ProvingKey&) = delete;
    Groth16ProvingKey& operator=(const Groth16ProvingKey&) = delete;
    uint64_t handle() const { return handle_; }

private:
    template <class T>
    static std::vector<T> tail(const std::vector<T>& v) { return v.empty() ? v : std::vector<T>(v.begin() + 1, v.end()); }
    template <class T>
    static T first(const std::vector<T>& v) {
        if (v.empty()) throw Error(ZKM_ERR_ARG, "Groth16ProvingKey: empty query vector");
        return v[0];
    }
    RegisteredBases<Curve, 1> h_, l_, a_, b1_;
    RegisteredBases<Curve, 2> b2_;
    uint64_t handle_ = 0;
};

// create_proof_with_reduction_and_matrices after synthesis: a, b, c are the evaluation vectors of the witness map
// (Montgomery Fr, 2^k elements), inputs = input_assignment[1..] and aux the canonical assignments, r and s canonical.
template <class Curve>
Proof<Curve> create_proof(const Groth16ProvingKey<Curve>& pk, const typename Curve::BigInt& r, const typename Curve::BigInt& s,
                          const std::vector<typename Curve::Fr>& a, const std::vector<typename Curve::Fr>& b,
                          const std::vector<typename Curve::Fr>& c, const std::vector<typename Curve::BigInt>& inputs,
                          const std::vector<typename Curve::BigInt>& aux) {
    uint32_t log_n = 0;
    while (((size_t)1 << log_n) < a.size()) log_n++;
    if (a.empty() || ((size_t)1 << log_n) != a.size() || b.size() != a.size() || c.size() != a.size())
        throw Error(ZKM_ERR_ARG, "create_proof: a, b, c must have the same power-of-two length");
    std::vector<typename Curve::BigInt> z(inputs);
    z.insert(z.end(), aux.begin(), aux.end());
    typedef typename G1Affine<Curve>::Coord C1;
    typedef typename G2Affine<Curve>::Coord C2;
    std::vector<uint64_t> oa(2 * sizeof(C1) / 8), ob(2 * sizeof(C2) / 8), oc(2 * sizeof(C1) / 8);
    uint8_t ia = 0, ib = 0, ic = 0;
    check(zkm_groth16_prove(pk.handle(), reinterpret_cast<const uint64_t*>(a.data()), reinterpret_cast<const uint64_t*>(b.data()),
                            reinterpret_cast<const uint64_t*>(c.data()), log_n, reinterpret_cast<const uint64_t*>(z.data()),
                            inputs.size(), aux.size(), reinterpret_cast<const uint64_t*>(&r), reinterpret_cast<const uint64_t*>(&s),
                            oa.data(), &ia, ob.data(), &ib, oc.data(), &ic),
          "zkm_groth16_prove");
    return Proof<Curve>{detail::unpack<Curve, 1>(oa, ia), detail::unpack<Curve, 2>(ob, ib), detail::unpack<Curve, 1>(oc, ic)};
}

}  // namespace zkm
