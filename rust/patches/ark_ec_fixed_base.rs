// Replacement for ark-ec 0.3.0 `src/msm/fixed_base.rs`, applied in the same [patch.crates-io] fork as
// ark_ec_variable_base.rs (INTEGRATION.md section 4).  UNCOMPILED here (no Rust toolchain in this repository's build
// environment); written against the 0.3.0 public API, the `zkm_write_raw` accessor of rust/patches/ark_ff_raw_limbs.rs
// and the `zkm_write_xy` / `zkm_from_xy` methods of ark_ec_variable_base.rs.
//
// Groth16::circuit_specific_setup (ark-groth16 0.3.0 src/generator.rs) and KZG10::setup (ark-poly-commit 0.3.0
// src/kzg10/mod.rs) call get_mul_window_size + get_window_table + multi_scalar_mul + batch_normalization.  Only
// multi_scalar_mul is routed: for the fields of the library it reads the base back out of the window table
// (table[0][1] = g, built by upstream's get_window_table) and calls zkm_fixed_base_msm, which builds its own table on
// the GPU.  Routing reuses gpu_group() of the variable-base patch (no modulus constants here).  The points come back
// normalised and are returned as projective points with z = 1, so the caller's batch_normalization is a no-op.
use crate::msm::variable_base::gpu_group;
use crate::{AffineCurve, ProjectiveCurve};
use ark_ff::{Field, PrimeField, Zero};
use ark_std::vec::Vec;
use zkmember_gpu_sys as sys;

pub struct FixedBaseMSM;

impl FixedBaseMSM {
    pub fn get_mul_window_size(num_scalars: usize) -> usize {
        upstream::FixedBaseMSM::get_mul_window_size(num_scalars)
    }

    pub fn get_window_table<T: ProjectiveCurve>(scalar_size: usize, window: usize, g: T) -> Vec<Vec<T::Affine>> {
        upstream::FixedBaseMSM::get_window_table(scalar_size, window, g)
    }

    pub fn windowed_mul<T: ProjectiveCurve>(outerc: usize, window: usize, multiples_of_g: &[Vec<T::Affine>], scalar: &T::ScalarField) -> T {
        upstream::FixedBaseMSM::windowed_mul(outerc, window, multiples_of_g, scalar)
    }

    /// Same signature and meaning as upstream: v[i] * g for the g whose window table is `table`.
    pub fn multi_scalar_mul<T: ProjectiveCurve>(scalar_size: usize, window: usize, table: &[Vec<T::Affine>], v: &[T::ScalarField]) -> Vec<T> {
        let full_width = scalar_size >= <T::ScalarField as PrimeField>::size_in_bits();   // a narrower width truncates upstream
        match gpu_group::<T::Affine>() {
            Some(id) if full_width && window >= 1 && !table.is_empty() && table[0].len() >= 2 => gpu_fixed_base::<T>(id, &table[0][1], v),
            _ => upstream::FixedBaseMSM::multi_scalar_mul(scalar_size, window, table, v),
        }
    }
}

fn gpu_fixed_base<T: ProjectiveCurve>(id: crate::msm::variable_base::GroupId, g: &T::Affine, v: &[T::ScalarField]) -> Vec<T> {
    sys::ensure_init();
    let n = v.len();
    let w2 = 2 * id.coord_words;
    let mut base = ark_std::vec![0u64; w2];
    let base_inf = if g.is_zero() { 1u8 } else { assert_eq!(g.zkm_write_xy(&mut base), w2, "zkmember-gpu: unexpected coordinate width"); 0u8 };
    // upstream takes &[G::ScalarField]: the Montgomery limbs go to the device as they are (into_repr happens there)
    let mut sc = ark_std::vec![0u64; n * id.scalar_words];
    for (i, e) in v.iter().enumerate() {
        assert_eq!(e.zkm_write_raw(&mut sc[i * id.scalar_words..(i + 1) * id.scalar_words]), id.scalar_words);
    }
    let mut xy = ark_std::vec![0u64; n * w2];
    let mut inf = ark_std::vec![0u8; n];
    sys::check(unsafe { sys::zkm_fixed_base_msm(id.curve, id.group, base.as_ptr(), base_inf, sc.as_ptr(), n, xy.as_mut_ptr(), inf.as_mut_ptr()) },
               "zkm_fixed_base_msm");
    (0..n)
        .map(|i| {
            if inf[i] != 0 { T::zero() } else {
                T::Affine::zkm_from_xy(&xy[i * w2..(i + 1) * w2]).expect("zkmember-gpu: affine model without raw-limb access").into_projective()
            }
        })
        .collect()
}

mod upstream {
    // The original body of ark-ec 0.3.0 src/msm/fixed_base.rs goes here unchanged (`pub struct FixedBaseMSM` and its
    // four functions): every field the GPU library does not implement keeps upstream's windowed multiplication.
    include!("fixed_base_upstream.rs");
}
