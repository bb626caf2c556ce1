// Replacement for the group side of ark-poly-commit 0.3.0 `src/marlin/marlin_pc/mod.rs`, applied in a
// [patch.crates-io] fork of ark-poly-commit (INTEGRATION.md section 4).  UNCOMPILED here (no Rust toolchain in this
// repository's build environment); written against the 0.3.0 public API, the `zkm_write_raw` / `zkm_read_raw` accessors
// of rust/patches/ark_ff_raw_limbs.rs and the `zkm_write_xy` / `zkm_from_xy` methods and `gpu_group` of
// rust/patches/ark_ec_variable_base.rs (public, hidden; re-exported at ark_ec::msm).
//
// `commit` sends every labelled polynomial as one item (two with a degree bound: shift D - d) to ONE
// zkm_kzg_commit_many call; `open_combinations_individual_opening_challenges` expands the linear combinations into flat
// terms (point, polynomial, blinding polynomial, shift, coefficient = challenge(k) * LC coefficient) and makes ONE
// zkm_kzg_open_batch call for all points.  The random draws stay upstream's (the same RNG calls in the same order), so
// the bytes equal upstream's.  Curves the library does not serve keep upstream's bodies.
//
// The committer key of a trimmed SRS holds powers_of_g in two pieces: `ck.powers` = powers_of_g[..=supported_degree]
// and `ck.shifted_powers` = powers_of_g[max_degree - max_bound ..] (both cut from the same universal powers_of_g).
// The library takes absolute shifts D - d into ONE registration, so the two pieces are registered as one vector of
// max_degree + 1 points: ck.powers, points at infinity over the gap between the pieces (never multiplied by a non-zero
// scalar: every bounded term lies inside the shifted piece), then the rest of ck.shifted_powers.  It is registered once
// per committer key and found again by the pieces' addresses and lengths plus a fingerprint of sampled points.
//
// Cargo.toml of the fork:  zkmember-gpu-sys = { path = "<repo>/rust/zkmember-gpu-sys" }
// (ark-ec / ark-ff resolve to the patched forks through the same [patch.crates-io] table)
// ---------------------------------------------------------------------------------------------------------------
// src/marlin/marlin_pc/mod.rs -- added to `impl<E, P> PolynomialCommitment<E::Fr, P> for MarlinKZG10<E, P>`:
use ark_ec::msm::{gpu_group, registered, GroupId};
use ark_ec::AffineCurve;
use ark_ff::{Field, PrimeField, Zero};
use ark_std::{collections::BTreeMap, sync::Mutex, vec::Vec};
use zkmember_gpu_sys as sys;

fn limbs<F: Field>(v: &[F], s: usize) -> Vec<u64> {
    let mut out = ark_std::vec![0u64; v.len() * s];
    for (i, e) in v.iter().enumerate() { e.zkm_write_raw(&mut out[i * s..(i + 1) * s]); }
    out
}

struct CachedSrs { handle: u64, fingerprint: u64 }
static SRS: Mutex<BTreeMap<(usize, usize, usize, usize), CachedSrs>> = Mutex::new(BTreeMap::new());

/// powers_of_g[0..=max_degree] of `ck` as one registration (see the header): handle of the cached one when the key's
/// pieces are unchanged, else a new registration (the stale one is released).
fn powers_of_g_handle<E: PairingEngine>(g1: GroupId, ck: &CommitterKey<E>) -> u64 {
    let shifted: &[E::G1Affine] = ck.shifted_powers.as_deref().unwrap_or(&[]);
    let start = if shifted.is_empty() { ck.powers.len() } else { ck.max_degree + 1 - shifted.len() };
    let total = if shifted.is_empty() { ck.powers.len() } else { ck.max_degree + 1 };
    let at = |i: usize| -> Option<&E::G1Affine> {
        if i < ck.powers.len() { Some(&ck.powers[i]) } else if i >= start { Some(&shifted[i - start]) } else { None }
    };
    let w2 = 2 * g1.coord_words;
    let mut fp = 0xcbf29ce484222325u64 ^ total as u64;
    let mut buf = ark_std::vec![0u64; w2];
    for k in 0..ark_std::cmp::min(64, total) {
        let i = if total <= 64 { k } else { ((k as u128) * ((total - 1) as u128) / 63) as usize };
        for w in buf.iter_mut() { *w = 0; }
        match at(i) { Some(p) if !p.is_zero() => { p.zkm_write_xy(&mut buf); } _ => buf[0] = u64::MAX }
        for w in buf.iter() { fp ^= *w; fp = fp.wrapping_mul(0x100000001b3); }
    }
    let key = (ck.powers.as_ptr() as usize, ck.powers.len(), shifted.as_ptr() as usize, shifted.len());
    let mut cache = SRS.lock().unwrap();
    if let Some(c) = cache.get(&key) {
        if c.fingerprint == fp { return c.handle; }
        sys::check(unsafe { sys::zkm_bases_release(c.handle) }, "zkm_bases_release");
    }
    let mut xy = ark_std::vec![0u64; total * w2];
    let mut inf = ark_std::vec![0u8; total];
    for i in 0..total {
        match at(i) {
            Some(p) if !p.is_zero() => { p.zkm_write_xy(&mut xy[i * w2..(i + 1) * w2]); }
            _ => inf[i] = 1,
        }
    }
    let mut handle = 0u64;
    sys::check(unsafe { sys::zkm_bases_register_ex(g1.curve, 1, xy.as_ptr(), inf.as_ptr(), total, 0, &mut handle) },
               "zkm_bases_register_ex");
    cache.insert(key, CachedSrs { handle, fingerprint: fp });
    handle
}

fn g1_point<G: AffineCurve>(xy: &[u64], inf: u8) -> G {
    if inf != 0 { G::zero() } else { G::zkm_from_xy(xy).expect("zkmember-gpu: affine model without raw-limb access") }
}

fn commit<'a>(ck: &Self::CommitterKey, polynomials: impl IntoIterator<Item = &'a LabeledPolynomial<E::Fr, P>>,
              rng: Option<&mut dyn RngCore>) -> Result<(Vec<LabeledCommitment<Self::Commitment>>, Vec<Self::Randomness>), Self::Error> {
    let g1 = match gpu_group::<E::G1Affine>() { Some(g) => g, None => return upstream::commit(ck, polynomials, rng) };
    let s = g1.scalar_words;
    let rng = &mut crate::optional_rng::OptionalRng(rng);
    let (g, gg) = (powers_of_g_handle::<E>(g1, ck), registered(g1, &ck.powers_of_gamma_g));
    let max_degree = ck.max_degree;
    let mut labels = Vec::new();
    let (mut coeffs, mut shifts, mut blinds, mut rands) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    for p in polynomials {
        kzg10::KZG10::<E, P>::check_degrees_and_bounds(ck.supported_degree(), max_degree, ck.enforced_degree_bounds.as_deref(), &p)?;
        // upstream's draws, in upstream's order: rand, then shifted_rand
        let rand = p.hiding_bound().map(|h| kzg10::Randomness::rand(h, false, None, rng)).unwrap_or_else(kzg10::Randomness::empty);
        coeffs.push(limbs(p.coeffs(), s));
        shifts.push(0usize);
        blinds.push(limbs(&rand.blinding_polynomial.coeffs, s));
        let shifted = p.degree_bound().map(|d| {
            let r = p.hiding_bound().map(|h| kzg10::Randomness::rand(h, false, None, rng)).unwrap_or_else(kzg10::Randomness::empty);
            coeffs.push(limbs(p.coeffs(), s));
            shifts.push(max_degree - d);
            blinds.push(limbs(&r.blinding_polynomial.coeffs, s));
            r
        });
        labels.push((p.label().clone(), p.degree_bound()));
        rands.push(Randomness { rand, shifted_rand: shifted });
    }
    let k = coeffs.len();
    let w2 = 2 * g1.coord_words;
    let (mut xy, mut inf) = (ark_std::vec![0u64; k * w2], ark_std::vec![0u8; k]);
    let cp: Vec<*const u64> = coeffs.iter().map(|c| c.as_ptr()).collect();
    let n: Vec<usize> = coeffs.iter().map(|c| c.len() / s).collect();
    let bp: Vec<*const u64> = blinds.iter().map(|c| c.as_ptr()).collect();
    let nb: Vec<usize> = blinds.iter().map(|c| c.len() / s).collect();
    for start in (0..k).step_by(23) {     // at most 23 items per call
        let e = (start + 23).min(k);
        sys::check(unsafe {
            sys::zkm_kzg_commit_many(g, gg, (e - start) as i32, cp[start..].as_ptr(), n[start..].as_ptr(), shifts[start..].as_ptr(),
                                     bp[start..].as_ptr(), nb[start..].as_ptr(), xy[start * w2..].as_mut_ptr(), inf[start..].as_mut_ptr())
        }, "zkm_kzg_commit_many");
    }
    let pt = |i: usize| kzg10::Commitment(g1_point::<E::G1Affine>(&xy[i * w2..(i + 1) * w2], inf[i]));
    let mut out = Vec::new();
    let mut i = 0;
    for (label, bound) in labels {
        let comm = pt(i);
        i += 1;
        let shifted_comm = bound.map(|_| { i += 1; pt(i - 1) });
        out.push(LabeledCommitment::new(label, Commitment { comm, shifted_comm }, bound));
    }
    Ok((out, rands))
}

fn open_combinations_individual_opening_challenges<'a>(ck: &Self::CommitterKey, lc_s: impl IntoIterator<Item = &'a LinearCombination<E::Fr>>,
        polynomials: impl IntoIterator<Item = &'a LabeledPolynomial<E::Fr, P>>, commitments: impl IntoIterator<Item = &'a LabeledCommitment<Self::Commitment>>,
        query_set: &QuerySet<E::Fr>, opening_challenges: &dyn Fn(u64) -> E::Fr, rands: impl IntoIterator<Item = &'a Self::Randomness>,
        rng: Option<&mut dyn RngCore>) -> Result<BatchLCProof<E::Fr, P, Self>, Self::Error> {
    let g1 = match gpu_group::<E::G1Affine>() {
        Some(g) => g,
        None => return upstream::open_combinations_individual_opening_challenges(ck, lc_s, polynomials, commitments, query_set,
                                                                                  opening_challenges, rands, rng),
    };
    let s = g1.scalar_words;
    let (g, gg) = (powers_of_g_handle::<E>(g1, ck), registered(g1, &ck.powers_of_gamma_g));
    let polys: BTreeMap<_, _> = polynomials.into_iter().zip(rands).map(|(p, r)| (p.label(), (p, r))).collect();
    let lcs: BTreeMap<_, _> = lc_s.into_iter().map(|lc| (lc.label(), lc)).collect();
    // every polynomial and blinding polynomial once; terms refer to them by index
    let (mut idx, mut coeffs, mut blinds) = (BTreeMap::new(), Vec::new(), Vec::new());
    for (label, (p, r)) in polys.iter() {
        idx.insert(*label, coeffs.len() as i32);
        coeffs.push(limbs(p.coeffs(), s));
        blinds.push(limbs(&r.rand.blinding_polynomial.coeffs, s));
        blinds.push(r.shifted_rand.as_ref().map(|sr| limbs(&sr.blinding_polynomial.coeffs, s)).unwrap_or_default());
    }
    // upstream's batch_open order: points by label (BTreeMap), the point's LC labels sorted (BTreeSet)
    let mut by_point: BTreeMap<_, (E::Fr, Vec<&String>)> = BTreeMap::new();
    for (label, (point_label, point)) in query_set.iter() { by_point.entry(point_label).or_insert((*point, Vec::new())).1.push(label); }
    let (mut points, mut tp, mut tq, mut tb, mut ts, mut tc) = (Vec::new(), Vec::new(), Vec::new(), Vec::new(), Vec::new(), Vec::new());
    let mut hiding = Vec::new();        // kzg10::Proof::random_v is Some only where a blinding polynomial was opened
    for (i, (_, (z, mut labels))) in by_point.into_iter().enumerate() {
        labels.sort();
        labels.dedup();
        points.push(z);
        hiding.push(false);
        let mut k = 0u64;
        for lc_label in labels {
            let lc = lcs[lc_label];
            let num_polys = lc.len();          // upstream counts LCTerm::One too
            let mut bound = None;
            for (coeff, term) in lc.iter().filter(|(_, t)| !t.is_one()) {
                let label: &String = term.try_into().expect("cannot be one!");
                let (p, r) = polys[label];
                if let Some(d) = p.degree_bound() {
                    if num_polys != 1 { return Err(Error::EquationHasDegreeBounds(lc_label.clone())); }
                    assert!(coeff.is_one(), "Coefficient must be one for degree-bounded equations");
                    bound = Some((idx[label], d, r.shifted_rand.is_some()));
                }
                tp.push(i as i32); tq.push(idx[label]); ts.push(0usize);
                tb.push(if p.hiding_bound().is_some() { 2 * idx[label] } else { -1 });
                hiding[i] |= p.hiding_bound().is_some();
                tc.push(opening_challenges(k) * coeff);
            }
            k += 1;
            if let Some((pi, d, hiding)) = bound {
                tp.push(i as i32); tq.push(pi); ts.push(ck.max_degree - d);
                tb.push(if hiding { 2 * pi + 1 } else { -1 });
                tc.push(opening_challenges(k));
                k += 1;
            }
        }
    }
    let np = points.len();
    let w2 = 2 * g1.coord_words;
    let (mut w, mut winf, mut rv) = (ark_std::vec![0u64; np * w2], ark_std::vec![0u8; np], ark_std::vec![0u64; np * s]);
    let cp: Vec<*const u64> = coeffs.iter().map(|c| c.as_ptr()).collect();
    let n: Vec<usize> = coeffs.iter().map(|c| c.len() / s).collect();
    let bp: Vec<*const u64> = blinds.iter().map(|c| c.as_ptr()).collect();
    let nb: Vec<usize> = blinds.iter().map(|c| c.len() / s).collect();
    let (zs, cs) = (limbs(&points, s), limbs(&tc, s));
    sys::check(unsafe {
        sys::zkm_kzg_open_batch(g, gg, cp.len() as i32, cp.as_ptr(), n.as_ptr(), bp.len() as i32, bp.as_ptr(), nb.as_ptr(), np as i32,
                                zs.as_ptr(), tc.len() as i32, tp.as_ptr(), tq.as_ptr(), tb.as_ptr(), ts.as_ptr(), cs.as_ptr(),
                                w.as_mut_ptr(), winf.as_mut_ptr(), rv.as_mut_ptr(), core::ptr::null_mut())   // evaluations: the AHP's own
    }, "zkm_kzg_open_batch");
    let proof = (0..np).map(|i| kzg10::Proof {
        w: g1_point::<E::G1Affine>(&w[i * w2..(i + 1) * w2], winf[i]),
        random_v: if hiding[i] {
            Some(E::Fr::zkm_read_raw(&rv[i * s..(i + 1) * s]).expect("zkmember-gpu: field without raw-limb access"))
        } else {
            None
        },
    }).collect();
    Ok(BatchLCProof { proof, evals: None })
}
