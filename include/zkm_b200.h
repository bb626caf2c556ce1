/* zkm_b200.h -- C ABI of the B200-native proving backend for zkMember's hot paths.
 *
 * The boundary does not exist in the reference: zkMember (/root/reference) calls MSM and FFT
 * statically through un-vendored arkworks 0.3.0 crates (pins: /root/reference/Cargo.lock:179-180
 * ark-ec, :338-339 ark-poly, :229-230 ark-ff), reached from /root/reference/benches/groth16.rs:115
 * (Groth16::prove) and /root/reference/benches/marlin.rs:202,311 (Marlin::prove).  Each entry
 * point below names the upstream function it replaces; INTEGRATION.md shows the Rust `-sys`
 * binding and the [patch.crates-io] forks that route the generic arkworks code here.
 *
 * Data formats are arkworks' own, byte for byte:
 *   field element : little-endian u64 limbs, Montgomery form, R = 2^(64*limbs)  (ark-ff Fp256/Fp384)
 *   scalar        : S64 x u64 little-endian, canonical (Fr::into_repr() -> BigInteger256 / BigInteger384)
 *   G1 affine     : x, y                      (2 * L64 words)  + a separate infinity byte per point
 *   G2 affine     : x.c0, x.c1, y.c0, y.c1    (4 * L64 words)  + infinity byte
 *   L64 = 6 for BLS12-381 Fq, 4 for BN254 Fq; Fr is S64 = 4 words for both.
 *   BW6-761: L64 = 12 (761-bit Fq), S64 = 6 (377-bit Fr = BLS12-377's Fq); its G2 is a curve over Fq as well,
 *   so a G2 affine point is x, y (2 * 12 words) exactly like a G1 point.
 *   Wherever a comment below says "4 words" for an Fr element or scalar, read S64.
 *
 * Every function returns 0 on success or a negative ZKM_ERR_* code; the message of the last
 * failure on the calling thread is available from zkm_last_error().  Nothing throws, aborts or
 * calls back.  There is NO CPU fallback: without a usable CUDA device every compute entry point
 * fails with ZKM_ERR_CUDA.
 *
 * Devices and threading.  zkm_init(device) binds the process to one GPU (the torchrun-style deployment: one process
 * per GPU); zkm_init_mask(mask) initialises several GPUs of the box for ONE process (the Rust prover is a single
 * process: /root/reference/benches/groth16.rs:115): bases can then be registered on a chosen device
 * (ZKM_REG_DEVICE(i), e.g. the G2 query on its own GPU) or sharded over all of them (ZKM_REG_SHARD), and MSMs over
 * such registrations run on every owning GPU at once, partial sums reduced on the caller's device over NVLink P2P.
 * Any host thread may call any entry point concurrently.  Every compute call borrows a LANE of the device it runs on
 * (48 per device: a stream plus grow-only workspaces) for its duration; calls on different lanes overlap on the GPU.
 * A lane keeps its workspaces until zkm_shutdown(): after a 2^24-point MSM that is ~20 GB on that lane, so a few
 * concurrent LARGE MSMs can exhaust HBM (they then fail with ZKM_ERR_OOM, nothing is corrupted).
 * Options (zkm_set_option) are snapshotted when a call starts: changing them never affects a call in flight.
 *
 * Device-pointer entry points (`*_device`): pointers must be 16-byte aligned (128-bit vector accesses) and must
 * belong to an initialised device -- the call runs on the device that owns the OUTPUT pointer.  `stream` is a
 * cudaStream_t of that device; NULL means the library's own NON-BLOCKING stream of that device (one per device: NULL-stream
 * calls are ordered among themselves), which does NOT synchronise with the legacy default stream or with the caller's
 * streams: producers of the inputs that ran elsewhere must have completed (or pass the stream they run on).
 *
 * Ownership: the caller owns every buffer it passes; the library reads inputs / writes outputs
 * during the call only and retains nothing except bases registered with zkm_bases_register* (and, for
 * zkm_msm_g1/g2, the internal registration cache described there).  zkm_bases_release() may be called while other
 * threads still use the handle: the memory is freed when the last such call has finished.
 */
#ifndef ZKM_B200_H
#define ZKM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZKM_CURVE_BLS12_381 0
#define ZKM_CURVE_BN254 1
#define ZKM_CURVE_BW6_761 2   /* the second curve zkMember benches (/root/reference/benches/groth16.rs:24-29, marlin.rs:40-73) */

#define ZKM_OK 0
#define ZKM_ERR_ARG (-1)          /* bad curve / group / size / null pointer */
#define ZKM_ERR_CUDA (-2)         /* CUDA runtime failure or no device */
#define ZKM_ERR_NOT_INIT (-3)     /* zkm_init() has not succeeded */
#define ZKM_ERR_DOMAIN (-4)       /* log_n exceeds the field's two-adicity (upstream: Domain::new -> None) */
#define ZKM_ERR_SCALAR_RANGE (-5) /* a scalar has bits at or above the modulus width (not canonical) */
#define ZKM_ERR_HANDLE (-6)       /* unknown / released bases handle, or range outside the registration */
#define ZKM_ERR_OOM (-7)          /* device or pinned-host allocation failed */

/* ---- lifecycle ----------------------------------------------------------------------------- */
int32_t zkm_init(int32_t device);   /* bind this process to CUDA device `device`; idempotent */
/* One process, several GPUs: initialise every device whose bit is set (bit i = CUDA device i); the lowest set bit is
 * the PRIMARY device (index 0), where host-pointer calls run unless a registration says otherwise.  Idempotent for the
 * same mask; zkm_init(d) == zkm_init_mask(1u << d).  (SURVEY.md 8b: `zkm_init(device_mask)`.) */
int32_t zkm_init_mask(uint32_t device_mask);
/* Explicit device list (devices[0] = primary).  A CUDA ordinal may be repeated: the entries then act as separate
 * "devices" with their own lanes on the same GPU -- how the multi-GPU paths are exercised on a one-GPU test box. */
int32_t zkm_init_devices(const int32_t* devices, int32_t count);
int32_t zkm_initialised_devices(void);   /* number of entries zkm_init* initialised (0 before) */
void zkm_shutdown(void);            /* release every device allocation and registered bases */
const char* zkm_last_error(void);   /* thread-local, never NULL */
int32_t zkm_device_count(void);     /* visible CUDA devices (0 when none / no driver) */
const char* zkm_version(void);

/* ---- variable-base MSM ----------------------------------------------------------------------
 * Replaces ark_ec::msm::VariableBaseMSM::multi_scalar_mul (ark-ec 0.3.0 src/msm/variable_base.rs)
 * followed by into_affine() (src/models/short_weierstrass_jacobian.rs): computes
 * sum_{i<n} scalars[i] * bases[i] and returns the unique normalised affine point.  The caller has
 * already taken n = min(len(bases), len(scalars)) as upstream does.  Zero scalars and infinity
 * bases are legal; n = 0 gives the identity (out_inf = 1, out_xy = arkworks' zero: x = 0, y = 1).
 * `infinity` may be NULL (no point at infinity among the bases).  All pointers are HOST pointers.
 *
 * Registration cache (option "msm_cache", default 1): the reference calls multi_scalar_mul(bases, scalars) with the
 * SAME proving-key vectors for every proof (`pk` is created once, /root/reference/benches/groth16.rs:107-115), so for
 * n >= 1024 the uploaded bases are kept as an internal registration keyed by (curve, group, bases pointer, infinity
 * pointer, n) and validated by a content fingerprint on every call: 1 = FNV-1a over 512 evenly spaced records (cheap;
 * assumes the vector is not partially rewritten in place between calls), 2 = over every byte, 0 = no cache (upload
 * every time).  A fingerprint mismatch re-uploads.  Least-recently-used entries are dropped above
 * "msm_cache_max_mb" (default 32768).  A cached vector of at most 2^18 bases that comes back a second time is
 * re-registered with its window multiples (ZKM_REG_PRECOMPUTE; option "msm_cache_precompute", default 1): from the third
 * call on the small MSMs of a real proving key run without the final doubling chain. */
int32_t zkm_msm_g1(int32_t curve, const uint64_t* bases_xy, const uint8_t* infinity,
                   const uint64_t* scalars, size_t n, uint64_t* out_xy, uint8_t* out_inf);
int32_t zkm_msm_g2(int32_t curve, const uint64_t* bases_xy, const uint8_t* infinity,
                   const uint64_t* scalars, size_t n, uint64_t* out_xy, uint8_t* out_inf);

/* Proving-key / SRS vectors are static across proofs (pk reuse at
 * /root/reference/benches/groth16.rs:107-115): upload them once and refer to them by handle. */
int32_t zkm_bases_register(int32_t curve, int32_t group /* 1 | 2 */, const uint64_t* bases_xy,
                           const uint8_t* infinity, size_t n, uint64_t* handle_out);
/* Registration with flags: */
#define ZKM_REG_PRECOMPUTE 1u      /* also store the window multiples 2^(c w) P_i (W x the memory): all windows of later
                                      MSMs share one bucket set, no final doubling chain -- for proving keys / SRS */
#define ZKM_REG_SHARD 2u           /* split the bases evenly over ALL initialised devices (range sharding) */
#define ZKM_REG_DEVICE(i) ((uint32_t)((i) + 1) << 8)   /* place the bases on initialised device index i (default 0) */
/* `bases_xy` / `infinity` may be host pointers or device pointers (of any device). */
int32_t zkm_bases_register_ex(int32_t curve, int32_t group, const uint64_t* bases_xy, const uint8_t* infinity, size_t n,
                              uint32_t flags, uint64_t* handle_out);
int32_t zkm_bases_release(uint64_t handle);
/* MSM over bases[offset .. offset + n) of a registration (KZG10::commit's powers_of_g[z..] slice,
 * ark-poly-commit 0.3.0 src/kzg10/mod.rs); scalars and outputs are HOST pointers. */
int32_t zkm_msm_registered(uint64_t handle, size_t offset, const uint64_t* scalars, size_t n,
                           uint64_t* out_xy, uint8_t* out_inf);

/* Replaces the non-hiding part of ark_poly_commit::kzg10::KZG10::commit (ark-poly-commit 0.3.0
 * src/kzg10/mod.rs; reached from /root/reference/benches/marlin.rs:202,311 through MarlinKZG10::commit):
 * skip_leading_zeros_and_convert_to_bigints + multi_scalar_mul(powers_of_g[z..], coeffs).  `handle` is a
 * registration of powers_of_g, `coeffs` are the n polynomial coefficients as Montgomery Fr (HOST pointer,
 * low degree first); the zero-skip, into_repr() and the MSM run on the device.  Returns the affine
 * commitment.  The hiding term (a second, small MSM over powers_of_gamma_g) is a second call + one add. */
int32_t zkm_kzg_commit(uint64_t handle, const uint64_t* coeffs, size_t n, uint64_t* out_xy, uint8_t* out_inf);
/* All commitments of one prover round in one call (Marlin commits 4 + 3 + 2 polynomials per proof:
 * /root/reference/benches/marlin.rs:311 -> ark-marlin AHP rounds -> MarlinKZG10::commit): `count` polynomials over the
 * same powers, committed concurrently on separate lanes.  out_xy: count x 2 W words, out_inf: count flags. */
int32_t zkm_kzg_commit_batch(uint64_t handle, int32_t count, const uint64_t* const* coeffs, const size_t* n,
                             uint64_t* out_xy, uint8_t* out_inf);
/* KZG10::commit WITH its hiding term (ark-poly-commit 0.3.0 src/kzg10/mod.rs: `random_commitment =
 * multi_scalar_mul(powers_of_gamma_g, random_ints).into_affine(); commitment.add_assign_mixed(&random_commitment)`).
 * `blinding_coeffs`: the nb coefficients of the caller's blinding polynomial (Montgomery Fr; sampling them is the
 * caller's RNG, unchanged host code).  Both MSMs run concurrently; returns the affine sum. */
int32_t zkm_kzg_commit_hiding(uint64_t handle_g, uint64_t handle_gamma_g, const uint64_t* coeffs, size_t n,
                              const uint64_t* blinding_coeffs, size_t nb, uint64_t* out_xy, uint8_t* out_inf);
/* KZG10::open (src/kzg10/mod.rs compute_witness_polynomial + open_with_witness_polynomial): the witness polynomial
 * (p(X) - p(z)) / (X - z) is computed ON THE DEVICE (blocked synthetic division), converted with into_repr and
 * committed over powers_of_g; with a blinding polynomial (handle_gamma_g != 0, nb > 0) the hiding witness is added and
 * out_random_v receives blinding_polynomial.evaluate(z) (Montgomery Fr).  `point`: z, one Montgomery Fr element.
 * Returns Proof.w as an affine point.  out_random_v may be NULL. */
int32_t zkm_kzg_open(uint64_t handle_g, uint64_t handle_gamma_g, const uint64_t* coeffs, size_t n,
                     const uint64_t* blinding_coeffs, size_t nb, const uint64_t* point, uint64_t* out_w_xy,
                     uint8_t* out_w_inf, uint64_t* out_random_v);

/* ---- batch commitments and openings (MarlinKZG10) --------------------------------------------------
 * The group side of ark-poly-commit 0.3.0 MarlinKZG10::{commit, batch_open, open_combinations} (src/marlin/marlin_pc).
 * The MarlinKZG10 bookkeeping (opening-challenge counter, degree-bound shifts, linear combinations) stays with the
 * caller; these calls take flat lists.  Polynomials are Montgomery Fr coefficients, low degree first.
 *
 * zkm_kzg_commit_many: item i = MSM(powers_of_g[shift_i + z_i ..], coeffs_i[z_i ..]) with z_i its leading zero
 * coefficients, plus MSM(powers_of_gamma_g, blind_i) when nb_i > 0 (blind / nb may be NULL: no hiding).  A Marlin
 * polynomial with a degree bound d is two items, the second with shift D - d.  All MSMs run concurrently, the sums are
 * formed on the device, one read-back.  At most 23 items.  out_xy: count x 2 W words, out_inf: count flags.
 * n_i counts every coefficient given, trailing zeros included: pass the polynomial without them (as DensePolynomial
 * keeps it) so that a bounded polynomial of degree d fits shift D - d.
 * Errors: ZKM_ERR_HANDLE when shift_i + n_i exceeds powers_of_g or nb_i exceeds powers_of_gamma_g. */
int32_t zkm_kzg_commit_many(uint64_t handle_g, uint64_t handle_gamma_g, int32_t count, const uint64_t* const* coeffs,
                            const size_t* n, const size_t* shift, const uint64_t* const* blind, const size_t* nb,
                            uint64_t* out_xy, uint8_t* out_inf);
/* zkm_kzg_open_batch: opening proofs at npoints points (at most 23).  Term t names a point, a polynomial, a blinding
 * polynomial (-1: none), a shift s_t and a Montgomery Fr coefficient c_t (term_coeff: nterms x S words).  Per point i:
 *   W_i        = commit_g(sum_t c_t X^(s_t) q_(poly_t, z_i)) + commit_gamma_g(sum_t c_t q_(blind_t, z_i))
 *   random_v_i = sum_t c_t blind_t(z_i)                 q_(p, z) = (p(X) - p(z)) / (X - z)
 * and out_evals[t] = poly_t(z_(point_t)) (Montgomery; out_evals may be NULL).  out_w_xy: npoints x 2 W words,
 * out_w_inf: npoints flags, out_random_v: npoints x S words.  At most 65535 terms.  One pinned upload and one read-back.
 * Errors: ZKM_ERR_ARG for an index out of range, null arrays, a G2 or other-curve registration; ZKM_ERR_HANDLE when
 * s_t + n - 1 exceeds powers_of_g or nb - 1 exceeds powers_of_gamma_g, or for a released handle. */
int32_t zkm_kzg_open_batch(uint64_t handle_g, uint64_t handle_gamma_g, int32_t npolys, const uint64_t* const* coeffs,
                           const size_t* n, int32_t nblind, const uint64_t* const* blind, const size_t* nb, int32_t npoints,
                           const uint64_t* points, int32_t nterms, const int32_t* term_point, const int32_t* term_poly,
                           const int32_t* term_blind, const size_t* term_shift, const uint64_t* term_coeff,
                           uint64_t* out_w_xy, uint8_t* out_w_inf, uint64_t* out_random_v, uint64_t* out_evals);
/* The same with the polynomials (d_coeffs[i], d_blind[i]: 16-byte aligned, ZKM_ERR_ARG otherwise) and the outputs in
 * device memory of one device (the device of d_out_w; a polynomial elsewhere is ZKM_ERR_ARG): d_out_w receives npoints records of 2 W + 1 words (flag word 0 finite, 1 infinity), d_out_random_v npoints x S
 * words, d_out_evals (may be NULL) nterms x S words.  The index arrays, points and term coefficients stay HOST arrays.
 * A fixed launch sequence on `stream` (NULL: the library's stream of that device); no read-back, no host wait. */
int32_t zkm_kzg_open_batch_device(uint64_t handle_g, uint64_t handle_gamma_g, int32_t npolys, const uint64_t* const* d_coeffs,
                                  const size_t* n, int32_t nblind, const uint64_t* const* d_blind, const size_t* nb,
                                  int32_t npoints, const uint64_t* points, int32_t nterms, const int32_t* term_point,
                                  const int32_t* term_poly, const int32_t* term_blind, const size_t* term_shift,
                                  const uint64_t* term_coeff, uint64_t* d_out_w, uint64_t* d_out_random_v,
                                  uint64_t* d_out_evals, void* stream);

/* ---- fixed-base batch scalar multiplication -------------------------------------------------------
 * Replaces ark_ec::msm::FixedBaseMSM::{get_window_table, multi_scalar_mul} (ark-ec 0.3.0 src/msm/fixed_base.rs)
 * + batch_normalization_into_affine: the queries of Groth16::circuit_specific_setup (ark-groth16 0.3.0
 * src/generator.rs) and the powers of KZG10::setup (ark-poly-commit 0.3.0 src/kzg10/mod.rs).
 * out[i] = scalars[i] * base for i < n, as n normalised affine records (2 * W words, Montgomery) in out_xy plus one
 * infinity byte each in out_inf; a zero product is arkworks' zero (x = 0, y = 1, flag 1).
 * scalars: n Montgomery Fr elements (S64 words each), as upstream takes &[G::ScalarField]; base: ONE affine record
 * (HOST pointer, 2 * W words) and its infinity flag.  A base at infinity gives every output at infinity.
 * The window width is chosen from n inside the library.  n = 0 succeeds and writes nothing; a null pointer where
 * n > 0, or an unknown curve or group, gives ZKM_ERR_ARG.
 * zkm_fixed_base_msm: scalars and outputs are HOST pointers; returns when the outputs are written.  An element
 * >= r fails with ZKM_ERR_SCALAR_RANGE (checked on the device, read back with the outputs). */
int32_t zkm_fixed_base_msm(int32_t curve, int32_t group, const uint64_t* base_xy, uint8_t base_inf,
                           const uint64_t* scalars, size_t n, uint64_t* out_xy, uint8_t* out_inf);
/* Device-resident form: d_scalars, d_out_xy and d_out_inf are DEVICE pointers (16-byte aligned, see above; the call
 * runs on the device that owns d_out_xy), base_xy stays a HOST pointer (passed to the kernels by value: nothing is
 * copied, the call never waits for the host).  A fixed sequence of kernel launches on `stream`, no device read-back.
 * Elements >= r are NOT checked (like zkm_fr_into_repr_device).  The outputs are in the format of
 * zkm_bases_register_device: a proving key or SRS built here can be registered without a host round trip. */
int32_t zkm_fixed_base_msm_device(int32_t curve, int32_t group, const uint64_t* base_xy, uint8_t base_inf,
                                  const uint64_t* d_scalars, size_t n, uint64_t* d_out_xy, uint8_t* d_out_inf,
                                  void* stream);

/* ---- Groth16 prover -------------------------------------------------------------------------------
 * Replaces ark-groth16 0.3.0 create_proof_with_reduction_and_matrices (src/prover.rs) after synthesis: the witness
 * map's FFTs, the five MSMs and the final assembly of Proof { a, b, c } in one call.
 *
 * zkm_groth16_pk_create: ark_groth16::ProvingKey on the device.  handles[5] are registrations (any flags) of h_query,
 * l_query, a_query[1..], b_g1_query[1..], b_g2_query[1..] -- groups 1, 1, 1, 1, 2 of one curve, the last three of equal
 * length.  The key holds references to them: the caller may release the handles afterwards.  g1_xy: 5 affine records
 * (2 W1 words each) alpha_g1, beta_g1, delta_g1, a_query[0], b_g1_query[0] with g1_inf[5]; g2_xy: 3 records (2 W2
 * words) beta_g2, delta_g2, b_g2_query[0] with g2_inf[3].  Builds a window table of delta_g1 and delta_g2 on every
 * initialised device, so that the delta multiples of a proof need no doublings.  Unknown curve, wrong group or curve
 * of a handle, or unequal query lengths give ZKM_ERR_ARG; an unknown handle ZKM_ERR_HANDLE. */
int32_t zkm_groth16_pk_create(int32_t curve, const uint64_t* handles, const uint64_t* g1_xy, const uint8_t* g1_inf,
                              const uint64_t* g2_xy, const uint8_t* g2_inf, uint64_t* pk_out);
/* Releases the key (a call still using it keeps it alive until it returns); an unknown key gives ZKM_ERR_HANDLE. */
int32_t zkm_groth16_pk_release(uint64_t pk);
/* a, b, c: the 2^log_n evaluation vectors handed to R1CStoQAP::witness_map (Montgomery Fr, as zkm_witness_map).
 * assignment = input_assignment[1..] || aux_assignment, canonical (into_repr), num_inputs + num_aux elements.
 * r, s: canonical Fr (S64 words); 0 is legal.  All HOST pointers.  Writes Proof { a: G1, b: G2, c: G1 } as normalised
 * affine records (zero = x 0, y 1, infinity byte 1).  Requires len(a_query) - 1 = num_inputs + num_aux,
 * len(l_query) = num_aux and len(h_query) <= 2^log_n, else ZKM_ERR_ARG; a released key gives ZKM_ERR_HANDLE; an
 * assignment element, r or s >= the scalar modulus gives ZKM_ERR_SCALAR_RANGE.  One pinned upload, the device form,
 * one read-back. */
int32_t zkm_groth16_prove(uint64_t pk, const uint64_t* a, const uint64_t* b, const uint64_t* c, uint32_t log_n,
                          const uint64_t* assignment, size_t num_inputs, size_t num_aux, const uint64_t* r, const uint64_t* s,
                          uint64_t* out_a_xy, uint8_t* out_a_inf, uint64_t* out_b_xy, uint8_t* out_b_inf,
                          uint64_t* out_c_xy, uint8_t* out_c_inf);
/* Device form: d_a, d_b, d_c (consumed: overwritten) and d_assignment are DEVICE pointers; d_out receives three packed
 * records A (2 W1 + 1 words), B (2 W2 + 1), C (2 W1 + 1) whose last word is the flag of zkm_msm_registered_device:
 * 0 finite, 1 infinity, 2 invalid (an assignment element, r or s >= the scalar modulus; all three records then carry
 * 2).  r and s stay HOST pointers (passed to the kernels by value).  A fixed launch sequence on `stream`: witness map,
 * into_repr of h, the five MSMs (concurrently, the b_g2 one on the device of its registration), the assembly; no
 * device read-back, no host wait.  Concurrent calls from several host threads overlap on the GPU. */
int32_t zkm_groth16_prove_device(uint64_t pk, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c, uint32_t log_n,
                                 const uint64_t* d_assignment, size_t num_inputs, size_t num_aux, const uint64_t* r,
                                 const uint64_t* s, uint64_t* d_out, void* stream);

/* ---- radix-2 NTT ------------------------------------------------------------------------------
 * Replaces ark_poly::Radix2EvaluationDomain::{fft_in_place, ifft_in_place, coset_fft_in_place,
 * coset_ifft_in_place} (ark-poly 0.3.0 src/domain/radix2/{mod,fft}.rs, src/domain/mod.rs) on the
 * scalar field Fr of `curve`.  `data` holds 2^log_n Montgomery elements, natural order in and out,
 * transformed in place (the caller has already resized to the domain size as upstream does).
 *   inverse = 0, coset = 0 : fft           X[k] = sum_j x[j] w^(jk)
 *   inverse = 0, coset = 1 : coset_fft     x[j] *= g^j first, g = Fr::multiplicative_generator()
 *   inverse = 1, coset = 0 : ifft          includes the multiplication by size_inv
 *   inverse = 1, coset = 1 : coset_ifft    ifft, then x[j] *= g^-j
 * log_n > TWO_ADICITY (32 for BLS12-381 Fr, 28 for BN254 Fr, 46 for BW6-761 Fr) fails with ZKM_ERR_DOMAIN. */
int32_t zkm_ntt(int32_t curve, uint64_t* data, uint32_t log_n, int32_t inverse, int32_t coset);

/* Replaces the FFT section of ark_groth16::R1CStoQAP::witness_map (ark-groth16 0.3.0 src/r1cs_to_qap.rs,
 * reached from /root/reference/benches/groth16.rs:115): given the evaluation vectors a, b, c over the
 * domain (2^log_n Montgomery elements each, already built and zero-padded by the caller as upstream does),
 * returns h = coset_ifft((coset_fft(ifft a) * coset_fft(ifft b) - coset_fft(ifft c)) / (g^n - 1)) --
 * seven NTTs and the pointwise step chained in HBM (one upload of a, b, c and one download of h instead
 * of fourteen PCIe crossings).  HOST pointers; inputs are not modified. */
int32_t zkm_witness_map(int32_t curve, const uint64_t* a, const uint64_t* b, const uint64_t* c, uint32_t log_n,
                        uint64_t* h_out);
/* Device-resident form: d_a, d_b, d_c are consumed (overwritten), d_h receives the 2^log_n coefficients. */
int32_t zkm_witness_map_device(int32_t curve, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c, uint32_t log_n,
                               uint64_t* d_h, void* stream);

/* Fr::into_repr() on n device-resident elements (Montgomery -> canonical BigInteger256): the conversion
 * create_proof applies to h before the h-query MSM (ark-groth16 0.3.0 src/prover.rs).  In place allowed. */
int32_t zkm_fr_into_repr_device(int32_t curve, const uint64_t* d_in, uint64_t* d_out, size_t n, void* stream);

/* Radix2EvaluationDomain::new: the five domain constants, Montgomery, S64 words each:
 * group_gen, group_gen_inv, size_inv, generator (= GENERATOR), generator_inv. */
int32_t zkm_domain_constants(int32_t curve, uint32_t log_n, uint64_t* out5xS64);

/* ---- device-resident variants ---------------------------------------------------------------
 * Same operations with DEVICE pointers, enqueued on `stream` (a cudaStream_t; NULL = the
 * library's own stream) without host synchronisation unless stated.  They are what a
 * device-resident prover (witness map feeding the h-query MSM) chains together, and what
 * bench.py times as the kernel-only figure. */
int32_t zkm_ntt_device(int32_t curve, const uint64_t* d_in, uint64_t* d_out, uint32_t log_n,
                       int32_t inverse, int32_t coset, void* stream);
/* d_out: 2 * W words (affine, Montgomery) followed by one u64 flag word: 0 = finite point, 1 = point at infinity,
 * 2 = INVALID -- a scalar had bits at or above the modulus width (what the host entry points report as
 * ZKM_ERR_SCALAR_RANGE; here the check happens on the device and the call has long returned).
 * Fully asynchronous: a fixed sequence of kernel launches on `stream`, no device read-back, no host wait.  (Do not call it
 * on a stream that is being CAPTURED into a CUDA graph: the library records its lane-completion events on `stream`.)  If the
 * registration lives
 * on other devices (ZKM_REG_DEVICE / ZKM_REG_SHARD) the scalar slices and the result records cross NVLink with
 * peer copies and sharded partial sums are added on the caller's device. */
int32_t zkm_msm_registered_device(uint64_t handle, size_t offset, const uint64_t* d_scalars, size_t n,
                                  uint64_t* d_out, void* stream);
/* `count` independent MSMs over registered bases issued concurrently (one internal host thread, lane and
 * stream per item), ordered after the current point of `stream` and joined back into it: the five MSMs of
 * ark_groth16::create_proof (src/prover.rs) in one call, with the G2 MSM overlapping the G1 ones.
 * Arrays of `count` entries; d_scalars[i] / d_outs[i] are DEVICE pointers as in zkm_msm_registered_device. */
int32_t zkm_msm_batch_registered_device(int32_t count, const uint64_t* handles, const size_t* offsets,
                                        const uint64_t* const* d_scalars, const size_t* n, uint64_t* const* d_outs,
                                        void* stream);
/* Adopt (copy) bases that already live in device memory. */
int32_t zkm_bases_register_device(int32_t curve, int32_t group, const uint64_t* d_bases_xy,
                                  const uint8_t* d_infinity, size_t n, uint64_t* handle_out);
/* Sum of m affine points given as m records of (2 * W words + 1 flag word), e.g. the per-GPU
 * partial results of a range-sharded MSM gathered on one device.  d_out has the same record
 * format.  Replaces the final GroupProjective additions of the sharded caller. */
int32_t zkm_points_sum_device(int32_t curve, int32_t group, const uint64_t* d_points, size_t m,
                              uint64_t* d_out, void* stream);

/* ---- tuning / introspection ------------------------------------------------------------------ */
/* key: "msm_window_bits" (0 = automatic), "msm_chunk" (points per accumulation task, 0 = auto),
 * "ntt_max_radix_log" (6..12), "profile" (0 | 1), "msm_precompute" (0 | 1: bases registered while it is
 * set also store their window multiples 2^(c w) P -- W times the memory, one-time cost -- so that all
 * windows of later MSMs share one bucket set and the final doubling chain disappears; meant for proving
 * keys / SRS that are reused across many proofs), "msm_xarr" (0 | 1: level-0 x-coordinate array, default 1),
 * "msm_prefetch_fwd" / "msm_prefetch_bwd", "msm_fold" (round-1 knobs, accepted and ignored),
 * "msm_cache" (0 | 1 | 2) and "msm_cache_max_mb" (registration cache of zkm_msm_g1/g2, see there),
 * "spread_host_calls" (0 | 1: host-pointer zkm_ntt / zkm_witness_map calls rotate over the initialised devices),
 * "host_wait" (accepted and ignored: since round 2 an MSM has no device read-back to wait for).
 * "msm_precompute" is the legacy form of ZKM_REG_PRECOMPUTE (a process-wide switch: prefer the flag).
 * Unknown keys fail with ZKM_ERR_ARG. */
int32_t zkm_set_option(const char* key, int64_t value);
/* With option "profile" = 1: device time (ms, CUDA events on the launching stream) of the six stages of
 * the last MSM: bucket sort | batched-affine pair levels | task lists | XYZZ bucket accumulation | folds |
 * window reduction. */
int32_t zkm_profile_last_msm(double* ms_out6);
/* Work counters of the same MSM, read back from the device (exact, not estimated): [0] points, [1] windows, [2] window
 * bits, [3] bucket-list entries (non-zero digits of non-infinity bases), [4..4+L) outputs of each batched-affine level
 * (pairs added at level l = inputs - outputs), [12] L, [13] XYZZ tasks of the accumulation kernel, [14] buckets,
 * [15] buckets whose partial sums were folded.  bench.py derives the executed field products of the bucket accumulation from these. */
int32_t zkm_profile_last_msm_counts(uint64_t* out16);
/* registration cache of zkm_msm_g1/g2: drop every entry / {hits, misses, entries, device bytes} */
int32_t zkm_msm_cache_clear(void);
int32_t zkm_msm_cache_stats(uint64_t* out4);
/* Kernel launches issued by this library since the last call with reset != 0. */
uint64_t zkm_launch_count(int32_t reset);
/* Window bits the automatic choice uses for an n-point MSM (for reports). */
int32_t zkm_msm_window_bits(int32_t curve, int32_t group, size_t n);

/* ---- synthetic inputs (bench / tests; SURVEY.md 8d) ------------------------------------------
 * Bases with known discrete logs P_i = (a0 + i * d) * G written to device memory as n affine
 * records of 2 * W words (no infinity among them when a0 + i*d != 0 mod r). */
int32_t zkm_testgen_progression_device(int32_t curve, int32_t group, uint64_t a0, uint64_t d,
                                       size_t n, uint64_t* d_bases_xy, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ZKM_B200_H */
