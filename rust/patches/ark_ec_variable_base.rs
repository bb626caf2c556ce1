// Replacement for ark-ec 0.3.0 `src/msm/variable_base.rs` (pin /root/reference/Cargo.lock:179-180) plus two hidden
// methods on `AffineCurve`, to be applied in a fork selected with [patch.crates-io] (INTEGRATION.md section 4).
// UNCOMPILED here (no Rust toolchain in this repository's build environment); complete source, written against the
// 0.3.0 public API and the `zkm_write_raw` / `zkm_read_raw` accessors of rust/patches/ark_ff_raw_limbs.rs.
//
// ---------------------------------------------------------------------------------------------------------------
// A. src/lib.rs -- inside `pub trait AffineCurve: ... {`     (0.3.0 exposes no coordinate accessor on the trait)
// ---------------------------------------------------------------------------------------------------------------
//
//     /// zkmember-gpu: write x then y as Montgomery limbs (see ark_ff::Field::zkm_write_raw); 0 = unsupported model.
//     #[doc(hidden)]
//     fn zkm_write_xy(&self, _out: &mut [u64]) -> usize { 0 }
//     /// zkmember-gpu: the affine point with these coordinates (the library returns points ON the curve).
//     #[doc(hidden)]
//     fn zkm_from_xy(_limbs: &[u64]) -> Option<Self> { None }
//
// B. src/models/short_weierstrass_jacobian.rs -- in `impl<P: Parameters> AffineCurve for GroupAffine<P> {`
//
//     fn zkm_write_xy(&self, out: &mut [u64]) -> usize {
//         let a = self.x.zkm_write_raw(out);
//         if a == 0 { return 0; }
//         let b = self.y.zkm_write_raw(&mut out[a..]);
//         if b == 0 { 0 } else { a + b }
//     }
//     fn zkm_from_xy(limbs: &[u64]) -> Option<Self> {
//         let h = limbs.len() / 2;
//         Some(GroupAffine::new(P::BaseField::zkm_read_raw(&limbs[..h])?, P::BaseField::zkm_read_raw(&limbs[h..])?, false))
//     }
//
// C. Cargo.toml of the fork:  zkmember-gpu-sys = { path = "<repo>/rust/zkmember-gpu-sys" }
// ---------------------------------------------------------------------------------------------------------------
// D. src/msm/variable_base.rs -- the whole file:
use crate::{AffineCurve, ProjectiveCurve};
use ark_ff::{BigInteger, Field, FpParameters, PrimeField, Zero};
use ark_std::{collections::BTreeMap, sync::Mutex, vec::Vec};
use zkmember_gpu_sys as sys;

pub struct VariableBaseMSM;

impl VariableBaseMSM {
    /// Same signature and meaning as upstream: sum over min(bases.len(), scalars.len()) pairs.
    pub fn multi_scalar_mul<G: AffineCurve>(
        bases: &[G],
        scalars: &[<G::ScalarField as PrimeField>::BigInt],
    ) -> G::Projective {
        let size = ark_std::cmp::min(bases.len(), scalars.len());
        match gpu_group::<G>() {
            Some(id) => gpu_msm::<G>(id, &bases[..size], &scalars[..size]),
            None => upstream::multi_scalar_mul(bases, scalars), // the original 0.3.0 body, moved verbatim into `mod upstream`
        }
    }
}

/// (curve id, group, u64 words per coordinate, u64 words per scalar) of include/zkm_b200.h.
/// Public (hidden): the fixed-base patch (ark_ec_fixed_base.rs) and the ark-groth16 prover fork
/// (ark_groth16_prover.rs) route with the same table.
#[derive(Clone, Copy)]
#[doc(hidden)]
pub struct GroupId { pub curve: i32, pub group: i32, pub coord_words: usize, pub scalar_words: usize }

// Moduli of the base PRIME fields the library implements (little-endian u64 limbs; the published curve parameters,
// the same numbers as oracle/py/params.py).  Routing compares the type's own `FpParameters::MODULUS` with these, so it
// is exact and needs neither the curve crates (ark-ec cannot depend on them) nor type-name strings.
const BLS12_381_FQ: [u64; 6] = [0xb9feffffffffaaab, 0x1eabfffeb153ffff, 0x6730d2a0f6b0f624, 0x64774b84f38512bf, 0x4b1ba7b6434bacd7, 0x1a0111ea397fe69a];
const BLS12_381_FR: [u64; 4] = [0xffffffff00000001, 0x53bda402fffe5bfe, 0x3339d80809a1d805, 0x73eda753299d7d48];
const BN254_FQ: [u64; 4] = [0x3c208c16d87cfd47, 0x97816a916871ca8d, 0xb85045b68181585d, 0x30644e72e131a029];
const BN254_FR: [u64; 4] = [0x43e1f593f0000001, 0x2833e84879b97091, 0xb85045b68181585d, 0x30644e72e131a029];
const BW6_761_FQ: [u64; 12] = [
    0xf49d00000000008b, 0xe6913e6870000082, 0x160cf8aeeaf0a437, 0x98a116c25667a8f8, 0x71dcd3dc73ebff2e, 0x8689c8ed12f9fd90,
    0x03cebaff25b42304, 0x707ba638e584e919, 0x528275ef8087be41, 0xb926186a81d14688, 0xd187c94004faff3e, 0x0122e824fb83ce0a,
];
const BW6_761_FR: [u64; 6] = [0x8508c00000000001, 0x170b5d4430000000, 0x1ef3622fba094800, 0x1a22d9f300f5138f, 0xc63b05c06ca1493b, 0x01ae3a4617c510ea];

#[doc(hidden)]
pub fn gpu_group<G: AffineCurve>() -> Option<GroupId> {
    type BasePrime<G> = <<G as AffineCurve>::BaseField as Field>::BasePrimeField;
    let q = <<BasePrime<G> as PrimeField>::Params as FpParameters>::MODULUS;
    let r = <<G::ScalarField as PrimeField>::Params as FpParameters>::MODULUS;
    let (q, r) = (q.as_ref(), r.as_ref());
    let deg = <G::BaseField as Field>::extension_degree() as usize;      // 1: curve over Fq, 2: over Fq2
    if q == &BLS12_381_FQ[..] && r == &BLS12_381_FR[..] && deg <= 2 {
        return Some(GroupId { curve: sys::ZKM_CURVE_BLS12_381, group: deg as i32, coord_words: 6 * deg, scalar_words: 4 });
    }
    if q == &BN254_FQ[..] && r == &BN254_FR[..] && deg <= 2 {
        return Some(GroupId { curve: sys::ZKM_CURVE_BN254, group: deg as i32, coord_words: 4 * deg, scalar_words: 4 });
    }
    // BW6-761 (/root/reference/benches/groth16.rs:24-29): G1 and G2 are BOTH curves over the 761-bit Fq; an MSM never
    // reads the curve coefficient b, so either group id selects the same kernels.
    if q == &BW6_761_FQ[..] && r == &BW6_761_FR[..] && deg == 1 {
        return Some(GroupId { curve: sys::ZKM_CURVE_BW6_761, group: 1, coord_words: 12, scalar_words: 6 });
    }
    None
}

/// Proving-key query vectors and SRS powers are the SAME slices for every proof
/// (/root/reference/benches/groth16.rs:107-115 creates `pk` once): they are packed and registered on the device once
/// and found again by (address, length) + a fingerprint of 64 sampled points -- so a proof uploads scalars only.
struct Cached { handle: u64, fingerprint: u64 }
static CACHE: Mutex<BTreeMap<(usize, usize, i32, i32), Cached>> = Mutex::new(BTreeMap::new());

fn fingerprint<G: AffineCurve>(bases: &[G], words: usize) -> u64 {
    let mut h = 0xcbf29ce484222325u64 ^ bases.len() as u64;
    let mut buf = ark_std::vec![0u64; 2 * words];
    let n = bases.len();
    for k in 0..ark_std::cmp::min(64, n) {
        let i = if n <= 64 { k } else { ((k as u128) * ((n - 1) as u128) / 63) as usize };
        for w in buf.iter_mut() { *w = 0; }
        if !bases[i].is_zero() { bases[i].zkm_write_xy(&mut buf); } else { buf[0] = u64::MAX; }
        for w in buf.iter() { h ^= *w; h = h.wrapping_mul(0x100000001b3); }
    }
    h
}

#[doc(hidden)]
pub fn registered<G: AffineCurve>(id: GroupId, bases: &[G]) -> u64 {
    let key = (bases.as_ptr() as usize, bases.len(), id.curve, id.group);
    let fp = fingerprint(bases, id.coord_words);
    let mut cache = CACHE.lock().unwrap();
    if let Some(c) = cache.get(&key) {
        if c.fingerprint == fp { return c.handle; }
        sys::check(unsafe { sys::zkm_bases_release(c.handle) }, "zkm_bases_release");
    }
    // GroupAffine / Fp are not #[repr(C)]: copy into the packed layout of the C ABI (x, y limbs + infinity byte)
    let w2 = 2 * id.coord_words;
    let mut xy = ark_std::vec![0u64; bases.len() * w2];
    let mut inf = ark_std::vec![0u8; bases.len()];
    for (i, b) in bases.iter().enumerate() {
        if b.is_zero() {
            inf[i] = 1;
        } else {
            let n = b.zkm_write_xy(&mut xy[i * w2..(i + 1) * w2]);
            assert_eq!(n, w2, "zkmember-gpu: unexpected coordinate width");
        }
    }
    let mut handle = 0u64;
    // small proving keys: also store the window multiples (no Horner tail in every later MSM)
    let flags = if bases.len() <= 1 << 20 { sys::ZKM_REG_PRECOMPUTE } else { 0 };
    sys::check(unsafe { sys::zkm_bases_register_ex(id.curve, id.group, xy.as_ptr(), inf.as_ptr(), bases.len(), flags, &mut handle) },
               "zkm_bases_register_ex");
    cache.insert(key, Cached { handle, fingerprint: fp });
    handle
}

fn gpu_msm<G: AffineCurve>(id: GroupId, bases: &[G], scalars: &[<G::ScalarField as PrimeField>::BigInt]) -> G::Projective {
    sys::ensure_init();
    let n = bases.len();
    if n == 0 { return G::Projective::zero(); }
    let handle = registered(id, bases);
    // BigInteger256 / BigInteger384: `as_ref()` is the canonical little-endian limb array the C ABI expects
    let mut sc = ark_std::vec![0u64; n * id.scalar_words];
    for (i, s) in scalars.iter().enumerate() {
        sc[i * id.scalar_words..(i + 1) * id.scalar_words].copy_from_slice(s.as_ref());
    }
    let mut out = ark_std::vec![0u64; 2 * id.coord_words];
    let mut out_inf = 0u8;
    sys::check(unsafe { sys::zkm_msm_registered(handle, 0, sc.as_ptr(), n, out.as_mut_ptr(), &mut out_inf) }, "zkm_msm_registered");
    if out_inf != 0 { return G::Projective::zero(); }
    G::zkm_from_xy(&out).expect("zkmember-gpu: affine model without raw-limb access").into_projective() // (x, y, z = 1)
}

mod upstream {
    // The original body of ark-ec 0.3.0 src/msm/variable_base.rs goes here unchanged (`pub fn multi_scalar_mul`):
    // every curve the GPU library does not implement keeps upstream's Pippenger.
    include!("variable_base_upstream.rs");
}
