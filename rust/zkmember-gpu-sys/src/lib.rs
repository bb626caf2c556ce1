//! Raw bindings to the C ABI declared in `include/zkm_b200.h`.
//! UNTESTED in this repository's build environment (no cargo/rustc there); written against the header.
//! Raw pointers only, no ark-* types: ark-ec and ark-poly (patched) depend on this crate.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub const ZKM_CURVE_BLS12_381: i32 = 0;
pub const ZKM_CURVE_BN254: i32 = 1;
pub const ZKM_CURVE_BW6_761: i32 = 2; // 12-word coordinates (G1 and G2 both over Fq), 6-word scalars / Fr elements
pub const ZKM_OK: i32 = 0;
pub const ZKM_REG_PRECOMPUTE: u32 = 1;
pub const ZKM_REG_SHARD: u32 = 2;
pub const fn zkm_reg_device(i: u32) -> u32 { (i + 1) << 8 }
pub const ZKM_ERR_DOMAIN: i32 = -4;

extern "C" {
    pub fn zkm_init(device: i32) -> i32;
    pub fn zkm_init_mask(device_mask: u32) -> i32;
    pub fn zkm_bases_register_ex(curve: i32, group: i32, bases_xy: *const u64, infinity: *const u8, n: usize, flags: u32,
                                 handle_out: *mut u64) -> i32;
    pub fn zkm_kzg_commit_batch(handle: u64, count: i32, coeffs: *const *const u64, n: *const usize, out_xy: *mut u64,
                                out_inf: *mut u8) -> i32;
    pub fn zkm_kzg_commit_hiding(handle_g: u64, handle_gamma_g: u64, coeffs: *const u64, n: usize, blinding: *const u64,
                                 nb: usize, out_xy: *mut u64, out_inf: *mut u8) -> i32;
    pub fn zkm_kzg_open(handle_g: u64, handle_gamma_g: u64, coeffs: *const u64, n: usize, blinding: *const u64, nb: usize,
                        point: *const u64, out_w_xy: *mut u64, out_w_inf: *mut u8, out_random_v: *mut u64) -> i32;
    pub fn zkm_shutdown();
    pub fn zkm_last_error() -> *const c_char;
    pub fn zkm_device_count() -> i32;
    pub fn zkm_msm_g1(curve: i32, bases_xy: *const u64, infinity: *const u8, scalars: *const u64, n: usize,
                      out_xy: *mut u64, out_inf: *mut u8) -> i32;
    pub fn zkm_msm_g2(curve: i32, bases_xy: *const u64, infinity: *const u8, scalars: *const u64, n: usize,
                      out_xy: *mut u64, out_inf: *mut u8) -> i32;
    pub fn zkm_fixed_base_msm(curve: i32, group: i32, base_xy: *const u64, base_inf: u8, scalars: *const u64, n: usize,
                              out_xy: *mut u64, out_inf: *mut u8) -> i32;
    pub fn zkm_fixed_base_msm_device(curve: i32, group: i32, base_xy: *const u64, base_inf: u8, d_scalars: *const u64, n: usize,
                                     d_out_xy: *mut u64, d_out_inf: *mut u8, stream: *mut c_void) -> i32;
    pub fn zkm_bases_register(curve: i32, group: i32, bases_xy: *const u64, infinity: *const u8, n: usize,
                              handle_out: *mut u64) -> i32;
    pub fn zkm_bases_release(handle: u64) -> i32;
    pub fn zkm_msm_registered(handle: u64, offset: usize, scalars: *const u64, n: usize, out_xy: *mut u64,
                              out_inf: *mut u8) -> i32;
    pub fn zkm_ntt(curve: i32, data: *mut u64, log_n: u32, inverse: i32, coset: i32) -> i32;
    pub fn zkm_domain_constants(curve: i32, log_n: u32, out5x_s64: *mut u64) -> i32;
    pub fn zkm_witness_map(curve: i32, a: *const u64, b: *const u64, c: *const u64, log_n: u32, h_out: *mut u64) -> i32;
    pub fn zkm_kzg_commit(handle: u64, coeffs: *const u64, n: usize, out_xy: *mut u64, out_inf: *mut u8) -> i32;
    pub fn zkm_set_option(key: *const c_char, value: i64) -> i32;
    pub fn zkm_ntt_device(curve: i32, d_in: *const u64, d_out: *mut u64, log_n: u32, inverse: i32, coset: i32,
                          stream: *mut c_void) -> i32;
    pub fn zkm_msm_registered_device(handle: u64, offset: usize, d_scalars: *const u64, n: usize, d_out: *mut u64,
                                     stream: *mut c_void) -> i32;
    pub fn zkm_groth16_pk_create(curve: i32, handles: *const u64, g1_xy: *const u64, g1_inf: *const u8, g2_xy: *const u64,
                                 g2_inf: *const u8, pk_out: *mut u64) -> i32;
    pub fn zkm_groth16_pk_release(pk: u64) -> i32;
    pub fn zkm_groth16_prove(pk: u64, a: *const u64, b: *const u64, c: *const u64, log_n: u32, assignment: *const u64,
                             num_inputs: usize, num_aux: usize, r: *const u64, s: *const u64, out_a_xy: *mut u64,
                             out_a_inf: *mut u8, out_b_xy: *mut u64, out_b_inf: *mut u8, out_c_xy: *mut u64,
                             out_c_inf: *mut u8) -> i32;
    pub fn zkm_groth16_prove_device(pk: u64, d_a: *mut u64, d_b: *mut u64, d_c: *mut u64, log_n: u32,
                                    d_assignment: *const u64, num_inputs: usize, num_aux: usize, r: *const u64,
                                    s: *const u64, d_out: *mut u64, stream: *mut c_void) -> i32;
    pub fn zkm_kzg_commit_many(handle_g: u64, handle_gamma_g: u64, count: i32, coeffs: *const *const u64, n: *const usize,
                               shift: *const usize, blind: *const *const u64, nb: *const usize, out_xy: *mut u64,
                               out_inf: *mut u8) -> i32;
    pub fn zkm_kzg_open_batch(handle_g: u64, handle_gamma_g: u64, npolys: i32, coeffs: *const *const u64, n: *const usize,
                              nblind: i32, blind: *const *const u64, nb: *const usize, npoints: i32, points: *const u64,
                              nterms: i32, term_point: *const i32, term_poly: *const i32, term_blind: *const i32,
                              term_shift: *const usize, term_coeff: *const u64, out_w_xy: *mut u64, out_w_inf: *mut u8,
                              out_random_v: *mut u64, out_evals: *mut u64) -> i32;
    pub fn zkm_kzg_open_batch_device(handle_g: u64, handle_gamma_g: u64, npolys: i32, d_coeffs: *const *const u64,
                                     n: *const usize, nblind: i32, d_blind: *const *const u64, nb: *const usize, npoints: i32,
                                     points: *const u64, nterms: i32, term_point: *const i32, term_poly: *const i32,
                                     term_blind: *const i32, term_shift: *const usize, term_coeff: *const u64,
                                     d_out_w: *mut u64, d_out_random_v: *mut u64, d_out_evals: *mut u64,
                                     stream: *mut c_void) -> i32;
}

/// Panics with the library's message: the upstream functions are infallible and there is deliberately
/// no CPU fallback.
pub fn check(rc: i32, what: &str) {
    if rc != ZKM_OK {
        let msg = unsafe { std::ffi::CStr::from_ptr(zkm_last_error()) }.to_string_lossy().into_owned();
        panic!("zkm_b200: {} failed ({}): {}", what, rc, msg);
    }
}

/// One-time process initialisation: `ZKM_DEVICE_MASK` (bit i = CUDA device i; one process driving several GPUs, the
/// G2 query / sharded registrations use the others) or `ZKM_DEVICE` (one GPU, default 0).
pub fn ensure_init() {
    use std::sync::Once;
    static INIT: Once = Once::new();
    INIT.call_once(|| {
        if let Some(mask) = std::env::var("ZKM_DEVICE_MASK").ok().and_then(|s| u32::from_str_radix(s.trim_start_matches("0x"), 16).ok()) {
            check(unsafe { zkm_init_mask(mask) }, "zkm_init_mask");
        } else {
            let dev = std::env::var("ZKM_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
            check(unsafe { zkm_init(dev) }, "zkm_init");
        }
    });
}
