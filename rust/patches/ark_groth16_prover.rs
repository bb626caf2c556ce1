// Replacement for ark-groth16 0.3.0 `src/prover.rs` plus the split of `R1CStoQAP::witness_map`, applied in a
// [patch.crates-io] fork of ark-groth16 (INTEGRATION.md section 4).  UNCOMPILED here (no Rust toolchain in this
// repository's build environment); written against the 0.3.0 public API, the `zkm_write_raw` accessor of
// rust/patches/ark_ff_raw_limbs.rs and the `zkm_write_xy` / `zkm_from_xy` methods, `gpu_group` and `registered` of
// rust/patches/ark_ec_variable_base.rs (public, hidden; re-exported by ark-ec's `pub use variable_base::*`).
//
// Synthesis, `finalize` and the sparse products a[i] = <A_i, z>, b[i] = <B_i, z>, c[i] = a[i] b[i] stay upstream's code:
// `R1CStoQAP::witness_map` is split at that point (section A: `evaluation_vectors` is its first half, unchanged).  The
// rest -- the seven FFTs, into_repr(h), the five MSMs and the assembly of Proof { a, b, c } -- is ONE zkm_groth16_prove
// call.  The device key is built once per &ProvingKey and found again by (address, lengths) + a fingerprint of sampled
// query points and every single point of the key.  Curves the library does not serve keep upstream's body.
//
// ---------------------------------------------------------------------------------------------------------------
// A. src/r1cs_to_qap.rs -- `witness_map` split in two; the body of `evaluation_vectors` is upstream's `witness_map`
//    from its first line down to (and including) the loop that sets c[i] = a[i] * b[i], moved verbatim; `witness_map`
//    keeps its signature and calls it:
// ---------------------------------------------------------------------------------------------------------------
//
//     /// zkmember-gpu: the evaluation domain and the domain-sized evaluation vectors a, b, c of the QAP (Montgomery
//     /// Fr) -- upstream's witness_map before its first FFT.
//     #[doc(hidden)]
//     pub fn evaluation_vectors<F: PrimeField, D: EvaluationDomain<F>>(
//         prover: ConstraintSystemRef<F>,
//     ) -> Result<(D, Vec<F>, Vec<F>, Vec<F>), SynthesisError> {
//         let matrices = prover.to_matrices().unwrap();
//         let zero = F::zero();
//         let num_inputs = prover.num_instance_variables();
//         let num_constraints = prover.num_constraints();
//         let cs = prover.borrow().unwrap();
//         let full_assignment = [cs.instance_assignment.as_slice(), cs.witness_assignment.as_slice()].concat();
//         let domain = D::new(num_constraints + num_inputs).ok_or(SynthesisError::PolynomialDegreeTooLarge)?;
//         let domain_size = domain.size();
//         let mut a = vec![zero; domain_size];
//         let mut b = vec![zero; domain_size];
//         cfg_iter_mut!(a[..num_constraints]).zip(&mut b[..num_constraints]).zip(&matrices.a).zip(&matrices.b)
//             .for_each(|(((a, b), at_i), bt_i)| {
//                 *a = evaluate_constraint(&at_i, &full_assignment);
//                 *b = evaluate_constraint(&bt_i, &full_assignment);
//             });
//         a[num_constraints..num_constraints + num_inputs].clone_from_slice(&full_assignment[..num_inputs]);
//         let mut c = vec![zero; domain_size];
//         cfg_iter_mut!(c[..num_constraints]).enumerate().for_each(|(i, c)| { *c = a[i] * &b[i]; });
//         Ok((domain, a, b, c))
//     }
//
//     pub(crate) fn witness_map<F: PrimeField, D: EvaluationDomain<F>>(prover: ConstraintSystemRef<F>)
//         -> Result<Vec<F>, SynthesisError> {
//         let (domain, mut a, mut b, mut c) = Self::evaluation_vectors::<F, D>(prover)?;
//         // ... upstream's witness_map from `domain.ifft_in_place(&mut a);` to its end, unchanged
//     }
//
// B. Cargo.toml of the fork:  zkmember-gpu-sys = { path = "<repo>/rust/zkmember-gpu-sys" }
//    (ark-ec resolves to the patched fork through the same [patch.crates-io] table)
// ---------------------------------------------------------------------------------------------------------------
// C. src/prover.rs -- the whole file:
use crate::{r1cs_to_qap::R1CStoQAP, Proof, ProvingKey};
use ark_ec::msm::{gpu_group, registered, GroupId};
use ark_ec::{AffineCurve, PairingEngine};
use ark_ff::{PrimeField, UniformRand, Zero};
use ark_poly::{EvaluationDomain, GeneralEvaluationDomain};
use ark_relations::r1cs::{ConstraintSynthesizer, ConstraintSystem, OptimizationGoal, Result as R1CSResult, SynthesisError};
use ark_std::rand::Rng;
use ark_std::{collections::BTreeMap, sync::Mutex, vec::Vec};
use zkmember_gpu_sys as sys;

pub fn create_random_proof<E, C, R>(circuit: C, pk: &ProvingKey<E>, rng: &mut R) -> R1CSResult<Proof<E>>
where E: PairingEngine, C: ConstraintSynthesizer<E::Fr>, R: Rng {
    let r = E::Fr::rand(rng);
    let s = E::Fr::rand(rng);
    create_proof::<E, C>(circuit, pk, r, s)
}

pub fn create_proof<E, C>(circuit: C, pk: &ProvingKey<E>, r: E::Fr, s: E::Fr) -> R1CSResult<Proof<E>>
where E: PairingEngine, C: ConstraintSynthesizer<E::Fr> {
    let (g1, g2) = match (gpu_group::<E::G1Affine>(), gpu_group::<E::G2Affine>()) {
        (Some(g1), Some(g2)) => (g1, g2),
        _ => return upstream::create_proof::<E, C>(circuit, pk, r, s),
    };
    // upstream: synthesis, inlining, matrices
    let cs = ConstraintSystem::new_ref();
    cs.set_optimization_goal(OptimizationGoal::Constraints);
    circuit.generate_constraints(cs.clone())?;
    debug_assert!(cs.is_satisfied().unwrap());
    cs.finalize();
    // upstream's witness_map up to the FFTs (section A): the domain-sized evaluation vectors (Montgomery Fr)
    let (domain, a, b, c) = R1CStoQAP::evaluation_vectors::<E::Fr, GeneralEvaluationDomain<E::Fr>>(cs.clone())?;
    let log_n = domain.size().trailing_zeros();   // radix-2 for the three scalar fields at every size they support
    let prover = cs.borrow().unwrap();
    let num_inputs = prover.instance_assignment.len() - 1;   // without the constant one
    let num_aux = prover.witness_assignment.len();
    let assignment: Vec<_> = prover.instance_assignment[1..].iter().chain(prover.witness_assignment.iter()).map(|v| v.into_repr()).collect();
    let key = device_key(g1, g2, pk);
    let limbs = |v: &[E::Fr]| {
        let mut out = ark_std::vec![0u64; v.len() * g1.scalar_words];
        for (i, e) in v.iter().enumerate() { e.zkm_write_raw(&mut out[i * g1.scalar_words..(i + 1) * g1.scalar_words]); }
        out
    };
    let (a, b, c) = (limbs(&a), limbs(&b), limbs(&c));
    let mut z = ark_std::vec![0u64; assignment.len() * g1.scalar_words];
    for (i, v) in assignment.iter().enumerate() { z[i * g1.scalar_words..(i + 1) * g1.scalar_words].copy_from_slice(v.as_ref()); }
    let (w1, w2) = (2 * g1.coord_words, 2 * g2.coord_words);
    let (mut oa, mut ob, mut oc) = (ark_std::vec![0u64; w1], ark_std::vec![0u64; w2], ark_std::vec![0u64; w1]);
    let (mut ia, mut ib, mut ic) = (0u8, 0u8, 0u8);
    let (r, s) = (r.into_repr(), s.into_repr());
    sys::check(unsafe {
        sys::zkm_groth16_prove(key, a.as_ptr(), b.as_ptr(), c.as_ptr(), log_n, z.as_ptr(), num_inputs, num_aux, r.as_ref().as_ptr(),
                               s.as_ref().as_ptr(), oa.as_mut_ptr(), &mut ia, ob.as_mut_ptr(), &mut ib, oc.as_mut_ptr(), &mut ic)
    }, "zkm_groth16_prove");
    let g1pt = |xy: &[u64], inf: u8| if inf != 0 { E::G1Affine::zero() } else {
        E::G1Affine::zkm_from_xy(xy).expect("zkmember-gpu: affine model without raw-limb access")
    };
    let b = if ib != 0 { E::G2Affine::zero() } else { E::G2Affine::zkm_from_xy(&ob).expect("zkmember-gpu: affine model without raw-limb access") };
    Ok(Proof { a: g1pt(&oa, ia), b, c: g1pt(&oc, ic) })
}

/// The device key of `pk` (zkm_groth16_pk_create): the five query vectors go through the registration cache of the
/// variable-base patch, the eight points are packed here.  Cached by (address, lengths) + fingerprint; a key found at
/// the same address with a different fingerprint is released and rebuilt.  Like the registration cache, the keys live
/// until the process ends (a prover keeps its ProvingKey for every proof, benches/groth16.rs:107-115).
struct CachedKey { handle: u64, fingerprint: u64 }
static KEYS: Mutex<BTreeMap<(usize, usize, usize), CachedKey>> = Mutex::new(BTreeMap::new());

fn xy_of<G: AffineCurve>(p: &G, words: usize, xy: &mut Vec<u64>, inf: &mut Vec<u8>) {
    let at = xy.len();
    xy.resize(at + 2 * words, 0);
    if p.is_zero() { inf.push(1); } else { p.zkm_write_xy(&mut xy[at..]); inf.push(0); }
}

fn fingerprint<E: PairingEngine>(pk: &ProvingKey<E>, g1: GroupId, g2: GroupId) -> u64 {
    let (mut buf, mut inf) = (Vec::new(), Vec::new());
    fn sample<G: AffineCurve>(q: &[G], words: usize, buf: &mut Vec<u64>, inf: &mut Vec<u8>) {
        let n = q.len();
        for k in 0..ark_std::cmp::min(16, n) {
            xy_of(&q[if n <= 16 { k } else { k * (n - 1) / 15 }], words, buf, inf);
        }
    }
    for q in [&pk.a_query, &pk.b_g1_query, &pk.h_query, &pk.l_query] { sample(q, g1.coord_words, &mut buf, &mut inf); }
    sample(&pk.b_g2_query, g2.coord_words, &mut buf, &mut inf);
    for p in [&pk.vk.alpha_g1, &pk.beta_g1, &pk.delta_g1] { xy_of(p, g1.coord_words, &mut buf, &mut inf); }
    for p in [&pk.vk.beta_g2, &pk.vk.delta_g2] { xy_of(p, g2.coord_words, &mut buf, &mut inf); }
    let mut h = 0xcbf29ce484222325u64;
    for w in buf.iter().copied().chain(inf.iter().map(|b| *b as u64)) { h ^= w; h = h.wrapping_mul(0x100000001b3); }
    h
}

fn device_key<E: PairingEngine>(g1: GroupId, g2: GroupId, pk: &ProvingKey<E>) -> u64 {
    sys::ensure_init();
    let key = (pk as *const _ as usize, pk.a_query.len(), pk.h_query.len());
    let fp = fingerprint(pk, g1, g2);
    let mut keys = KEYS.lock().unwrap();
    if let Some(k) = keys.get(&key) {
        if k.fingerprint == fp { return k.handle; }
        sys::check(unsafe { sys::zkm_groth16_pk_release(k.handle) }, "zkm_groth16_pk_release");
    }
    let handles = [registered(g1, &pk.h_query), registered(g1, &pk.l_query), registered(g1, &pk.a_query[1..]),
                   registered(g1, &pk.b_g1_query[1..]), registered(g2, &pk.b_g2_query[1..])];
    let (mut p1, mut i1, mut p2, mut i2) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    for p in [&pk.vk.alpha_g1, &pk.beta_g1, &pk.delta_g1, &pk.a_query[0], &pk.b_g1_query[0]] { xy_of(p, g1.coord_words, &mut p1, &mut i1); }
    for p in [&pk.vk.beta_g2, &pk.vk.delta_g2, &pk.b_g2_query[0]] { xy_of(p, g2.coord_words, &mut p2, &mut i2); }
    let mut handle = 0u64;
    sys::check(unsafe {
        sys::zkm_groth16_pk_create(g1.curve, handles.as_ptr(), p1.as_ptr(), i1.as_ptr(), p2.as_ptr(), i2.as_ptr(), &mut handle)
    }, "zkm_groth16_pk_create");
    keys.insert(key, CachedKey { handle, fingerprint: fp });
    handle
}

mod upstream {
    // The original body of ark-groth16 0.3.0 src/prover.rs goes here unchanged (create_random_proof, create_proof,
    // create_proof_with_reduction_and_matrices, ...): curves the GPU library does not implement keep it.
    include!("prover_upstream.rs");
}
