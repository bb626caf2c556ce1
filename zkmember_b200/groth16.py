"""Host-side mirror of the hot part of ark-groth16 0.3.0's prover (SURVEY.md 8f rows 1-2).

`witness_map` replaces the FFT section of `R1CStoQAP::witness_map` (src/r1cs_to_qap.rs; reached from
/root/reference/benches/groth16.rs:115): the caller (unchanged Rust/host code) evaluates the R1CS
matrices on the assignment -- a[i] = <A_i, z>, b[i] = <B_i, z>, c[i] = <C_i, z>, a[nc + j] = z_j --
and this runs the seven NTTs and the pointwise step on the GPU without leaving HBM.

`ProvingKeyMSMs` holds the five query vectors of a Groth16 proving key registered once on the device
(`pk` is reused for every proof, benches/groth16.rs:107-115) and runs the five MSMs of `create_proof`
(src/prover.rs: h_query, l_query, a_query, b_g1_query on G1, b_g2_query on G2).

`ProvingKey` + `create_proof` mirror `create_proof_with_reduction_and_matrices` from the witness map to the
`Proof { a, b, c }` (final assembly included: `calculate_coeff`, g_c = s g_a + r g1_b - rs delta + l_aux + h_acc) as ONE
library call (`zkm_groth16_prove`): witness map, the five MSMs and the assembly stay on the device.
`serialize.Proof.serialize()` gives the 192-byte (BLS12-381) arkworks wire format.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib
from .msm import RegisteredBases, AffinePoint, FR_WORDS, coord_words, _curve_id, _ptr
from .serialize import Proof, FR_MODULUS


def witness_map(a, b, c, curve="bls12_381") -> np.ndarray:
    """h = coset_ifft((coset_fft(ifft a) * coset_fft(ifft b) - coset_fft(ifft c)) / (g^n - 1)).
    a, b, c: (n, 4) uint64 Montgomery evaluations over the domain, n a power of two."""
    cid = _curve_id(curve)
    S = _lib.FR_WORDS[cid]
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, S)
    b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, S)
    c = np.ascontiguousarray(c, dtype=np.uint64).reshape(-1, S)
    n = len(a)
    log_n = n.bit_length() - 1
    if n == 0 or (1 << log_n) != n or len(b) != n or len(c) != n:
        raise ValueError("a, b, c must have the same power-of-two length")
    h = np.zeros_like(a)
    p = lambda x: ctypes.c_void_p(x.ctypes.data)
    _lib.check(_lib.lib().zkm_witness_map(cid, p(a), p(b), p(c), log_n, p(h)))
    return h


class ProvingKeyMSMs:
    """The five MSM bases of a Groth16 proving key, resident in HBM."""

    def __init__(self, curve, h_query, l_query, a_query, b_g1_query, b_g2_query, infinity=None, precompute=True,
                 g2_device: int | None = None):
        """g2_device: index of the initialised GPU that holds the b_g2 query (SURVEY 8e: the G2 MSM runs on its own GPU
        next to the G1 ones); default: device 1 when the process initialised more than one GPU, else the primary."""
        cid = _curve_id(curve)
        infinity = infinity or {}
        if g2_device is None and _lib.initialised_devices() > 1:
            g2_device = 1
        kw = {"precompute": bool(precompute)}
        self.h = RegisteredBases(cid, 1, h_query, infinity.get("h"), **kw)
        self.l = RegisteredBases(cid, 1, l_query, infinity.get("l"), **kw)
        self.a = RegisteredBases(cid, 1, a_query, infinity.get("a"), **kw)
        self.b_g1 = RegisteredBases(cid, 1, b_g1_query, infinity.get("b_g1"), **kw)
        self.b_g2 = RegisteredBases(cid, 2, b_g2_query, infinity.get("b_g2"), device=g2_device, **kw)

    def prove_msms(self, h_scalars, aux_scalars, full_scalars) -> dict:
        """h_acc, l_acc and the MSM parts of g_a, g1_b, g2_b (calculate_coeff's `acc`).  Upstream runs the
        five MSMs one after another; here they are issued from five host threads, each borrowing its own
        library lane, so the G2 MSM and the serial tails of the G1 ones overlap on the GPU."""
        from concurrent.futures import ThreadPoolExecutor
        jobs = {
            "h_acc": (self.h, h_scalars), "l_acc": (self.l, aux_scalars), "a_acc": (self.a, full_scalars),
            "b_g1_acc": (self.b_g1, full_scalars), "b_g2_acc": (self.b_g2, full_scalars),
        }
        with ThreadPoolExecutor(max_workers=5) as ex:
            futs = {k: ex.submit(reg.msm, sc) for k, (reg, sc) in jobs.items()}
            return {k: f.result() for k, f in futs.items()}

    def release(self):
        for r in (self.h, self.l, self.a, self.b_g1, self.b_g2):
            r.release()


def _scalar_limbs(curve: int, v: int) -> np.ndarray:
    S = FR_WORDS[curve]
    return np.array([(v >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(S)], dtype=np.uint64)


class ProvingKey:
    """ark_groth16::ProvingKey: the verifying-key elements the prover touches plus the five query vectors.
    `a_query`, `b_g1_query`, `b_g2_query` are the FULL vectors (entry 0 belongs to the constant-one variable and is
    added outside the MSM, as `calculate_coeff` does); the remaining entries are registered on the device once, and
    the device key (`handle`, zkm_groth16_pk_create) refers to those registrations and the key's eight points."""

    def __init__(self, curve, alpha_g1, beta_g1, beta_g2, delta_g1, delta_g2, a_query, b_g1_query, b_g2_query,
                 h_query, l_query, infinity=None, precompute=True):
        self.curve = _curve_id(curve)
        W1, W2 = coord_words(self.curve, 1), coord_words(self.curve, 2)
        as1 = lambda a: np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 2 * W1)
        as2 = lambda a: np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 2 * W2)
        self.alpha_g1, self.beta_g1, self.delta_g1 = as1(alpha_g1)[0], as1(beta_g1)[0], as1(delta_g1)[0]
        self.beta_g2, self.delta_g2 = as2(beta_g2)[0], as2(delta_g2)[0]
        a_query, b_g1_query, b_g2_query = as1(a_query), as1(b_g1_query), as2(b_g2_query)
        infinity = dict(infinity or {})
        flags = {k: np.ascontiguousarray(infinity[k], dtype=np.uint8) if infinity.get(k) is not None else None
                 for k in ("a", "b_g1", "b_g2", "h", "l")}
        self.first = {"a": (a_query[0], bool(flags["a"][0]) if flags["a"] is not None else False),
                      "b_g1": (b_g1_query[0], bool(flags["b_g1"][0]) if flags["b_g1"] is not None else False),
                      "b_g2": (b_g2_query[0], bool(flags["b_g2"][0]) if flags["b_g2"] is not None else False)}
        tail = {k: (flags[k][1:] if flags[k] is not None else None) for k in ("a", "b_g1", "b_g2")}
        self.msms = ProvingKeyMSMs(self.curve, h_query, l_query, a_query[1:], b_g1_query[1:], b_g2_query[1:],
                                   infinity={"h": flags["h"], "l": flags["l"], "a": tail["a"], "b_g1": tail["b_g1"],
                                             "b_g2": tail["b_g2"]}, precompute=precompute)
        self.num_vars = len(a_query) - 1
        self.num_aux = self.msms.l.n
        ms = self.msms
        handles = np.array([ms.h.handle, ms.l.handle, ms.a.handle, ms.b_g1.handle, ms.b_g2.handle], dtype=np.uint64)
        g1 = np.ascontiguousarray(np.stack([self.alpha_g1, self.beta_g1, self.delta_g1, self.first["a"][0],
                                            self.first["b_g1"][0]]))
        g1_inf = np.array([0, 0, 0, self.first["a"][1], self.first["b_g1"][1]], dtype=np.uint8)
        g2 = np.ascontiguousarray(np.stack([self.beta_g2, self.delta_g2, self.first["b_g2"][0]]))
        g2_inf = np.array([0, 0, self.first["b_g2"][1]], dtype=np.uint8)
        h = ctypes.c_uint64(0)
        try:
            _lib.check(_lib.lib().zkm_groth16_pk_create(self.curve, _ptr(handles), _ptr(g1), _ptr(g1_inf), _ptr(g2),
                                                        _ptr(g2_inf), ctypes.byref(h)))
        except Exception:
            self.msms.release()
            raise
        self.handle = h.value

    def release(self):
        if self.handle:
            _lib.check(_lib.lib().zkm_groth16_pk_release(self.handle))
            self.handle = 0
        self.msms.release()

    def prove_device(self, d_a: int, d_b: int, d_c: int, log_n: int, d_assignment: int, num_inputs: int, r: int, s: int,
                     d_out: int, stream: int = 0):
        """Device form of `create_proof` (zkm_groth16_prove_device): d_a, d_b, d_c (2^log_n Montgomery Fr each, consumed)
        and d_assignment (num_inputs + num_aux canonical scalars) are device pointers; d_out receives the records A, B,
        C (2 W1 + 1, 2 W2 + 1, 2 W1 + 1 words; last word 0 finite, 1 infinity, 2 invalid scalar).  Enqueued on `stream`
        without a host wait; r and s are reduced modulo the scalar modulus."""
        rl, sl = (_scalar_limbs(self.curve, v % FR_MODULUS[self.curve]) for v in (r, s))
        _lib.check(_lib.lib().zkm_groth16_prove_device(
            self.handle, ctypes.c_void_p(d_a), ctypes.c_void_p(d_b), ctypes.c_void_p(d_c), int(log_n),
            ctypes.c_void_p(d_assignment), int(num_inputs), self.num_vars - int(num_inputs), _ptr(rl), _ptr(sl),
            ctypes.c_void_p(d_out), ctypes.c_void_p(stream)))


def create_proof(pk: ProvingKey, r: int, s: int, a, b, c, input_assignment, aux_assignment) -> Proof:
    """ark_groth16::create_proof_with_reduction_and_matrices (ark-groth16 0.3.0 src/prover.rs) after constraint
    synthesis: `a`, `b`, `c` are the evaluation vectors handed to the witness map (Montgomery Fr, domain size n),
    `input_assignment` (without the leading one) and `aux_assignment` the canonical (`into_repr`) assignments,
    r and s the prover's blinding scalars (reduced modulo the scalar modulus)."""
    curve = pk.curve
    S = FR_WORDS[curve]
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, S)
    b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, S)
    c = np.ascontiguousarray(c, dtype=np.uint64).reshape(-1, S)
    n = len(a)
    log_n = n.bit_length() - 1
    if n == 0 or (1 << log_n) != n or len(b) != n or len(c) != n:
        raise ValueError("a, b, c must have the same power-of-two length")
    inputs = np.ascontiguousarray(input_assignment, dtype=np.uint64).reshape(-1, S)
    aux = np.ascontiguousarray(aux_assignment, dtype=np.uint64).reshape(-1, S)
    full = np.ascontiguousarray(np.concatenate([inputs, aux]))
    rl, sl = (_scalar_limbs(curve, v % FR_MODULUS[curve]) for v in (r, s))
    W1, W2 = coord_words(curve, 1), coord_words(curve, 2)
    axy, bxy, cxy = np.zeros(2 * W1, dtype=np.uint64), np.zeros(2 * W2, dtype=np.uint64), np.zeros(2 * W1, dtype=np.uint64)
    inf = np.zeros(3, dtype=np.uint8)
    p = lambda x: ctypes.c_void_p(x.ctypes.data)
    _lib.check(_lib.lib().zkm_groth16_prove(pk.handle, p(a), p(b), p(c), log_n, _ptr(full), len(inputs), len(aux), p(rl),
                                            p(sl), p(axy), ctypes.c_void_p(inf.ctypes.data), p(bxy),
                                            ctypes.c_void_p(inf.ctypes.data + 1), p(cxy), ctypes.c_void_p(inf.ctypes.data + 2)))
    return Proof(a=AffinePoint(curve, 1, axy, bool(inf[0])), b=AffinePoint(curve, 2, bxy, bool(inf[1])),
                 c=AffinePoint(curve, 1, cxy, bool(inf[2])))
