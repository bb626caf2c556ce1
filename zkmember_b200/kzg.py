"""Host-side mirror of the hot part of ark-poly-commit 0.3.0's KZG10 (SURVEY.md 8f row 3).

    KZG10.commit(powers, coeffs[, gamma_powers, blinding_coeffs])   `KZG10::commit`  (src/kzg10/mod.rs)
    KZG10.commit_batch(powers, [coeffs, ...])                        the commitments of one prover round in one call
    KZG10.open(powers, coeffs, point[, gamma_powers, blinding])      `KZG10::open`: witness polynomial + its commitment
    KZG10.setup(curve, max_degree, beta, g, gamma_g)                 `KZG10::setup`: the two power vectors of the SRS

reached from /root/reference/benches/marlin.rs:202,311 through MarlinKZG10::{commit, open}.  Same meaning as upstream:
`commit` skips the leading zero coefficients, converts with `into_repr()` and runs
`VariableBaseMSM::multi_scalar_mul(&powers.powers_of_g[z..], &coeffs)`; with a blinding polynomial it adds
`multi_scalar_mul(&powers.powers_of_gamma_g, &blinding).into_affine()`.  `open` divides p(X) - p(z) by (X - z) --
on the device -- and commits the quotient; with a blinding polynomial it adds the hiding witness and returns
`random_v = blinding.evaluate(z)`.  Sampling the blinding polynomial stays the caller's RNG (unchanged host code).
The SRS powers are registered on the device once (`Powers`); every call then uploads only coefficients.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np

from . import _lib
from .msm import AffinePoint, FixedBaseMSM, RegisteredBases, coord_words, _curve_id
from .serialize import FR_MODULUS


class Powers(RegisteredBases):
    """powers_of_g (or powers_of_gamma_g) of a KZG10 committer key, resident in HBM."""

    def __init__(self, curve, powers_of_g, precompute: bool = False, shard: bool = False, device=None):
        super().__init__(curve, 1, powers_of_g, precompute=precompute, shard=shard, device=device)


@dataclass
class OpeningProof:
    """ark_poly_commit::kzg10::Proof { w, random_v }."""
    w: AffinePoint
    random_v: np.ndarray | None      # Montgomery Fr limbs, None without hiding


def _coeffs(powers: RegisteredBases, coeffs) -> np.ndarray:
    return np.ascontiguousarray(coeffs, dtype=np.uint64).reshape(-1, _lib.FR_WORDS[powers.curve])


def _p(a):
    return ctypes.c_void_p(a.ctypes.data if a is not None and a.size else 0)


@dataclass
class UniversalParams:
    """The group vectors of ark_poly_commit::kzg10::UniversalParams that KZG10::setup builds by fixed-base batches
    (Montgomery affine records + infinity bytes)."""
    powers_of_g: np.ndarray            # (max_degree + 1, 2 W): beta^i g
    powers_of_g_inf: np.ndarray
    powers_of_gamma_g: np.ndarray      # (max_degree + 2, 2 W): beta^i gamma_g, with the extra power upstream appends
    powers_of_gamma_g_inf: np.ndarray


def _powers_of_beta(curve: int, beta, count: int) -> np.ndarray:
    """Montgomery limbs of beta^0 .. beta^(count - 1), computed on the host like upstream's `cur *= &beta` loop."""
    S = _lib.FR_WORDS[curve]
    r = FR_MODULUS[curve]
    R = 1 << (64 * S)
    b_mont = int.from_bytes(np.ascontiguousarray(beta, dtype=np.uint64).reshape(S).tobytes(), "little")
    if b_mont >= r:
        raise ValueError("beta is not a canonical Montgomery Fr element")
    b = b_mont * pow(R, -1, r) % r
    out = bytearray(8 * S * count)
    cur = R % r                        # Montgomery one; mont(beta^i) = mont(beta^(i-1)) * beta mod r
    for i in range(count):
        out[8 * S * i:8 * S * (i + 1)] = cur.to_bytes(8 * S, "little")
        cur = cur * b % r
    return np.frombuffer(bytes(out), dtype=np.uint64).reshape(count, S)


class KZG10:
    @staticmethod
    def setup(curve, max_degree: int, beta, g, gamma_g) -> UniversalParams:
        """KZG10::setup (ark-poly-commit 0.3.0 src/kzg10/mod.rs) after its random draws: `beta` is one Montgomery Fr
        element (S words), `g` / `gamma_g` the two G1 generators (AffinePoint or 2 W words).  powers_of_g[i] = beta^i g
        for i <= max_degree; powers_of_gamma_g[i] = beta^i gamma_g for i <= max_degree + 1 (upstream pushes one more
        power so that up to max_degree queries can be supported).  Both vectors are fixed-base batches on the GPU."""
        cid = _curve_id(curve)
        if max_degree < 1:
            raise ValueError("max_degree must be at least 1 (upstream: DegreeIsZero)")
        pw = _powers_of_beta(cid, beta, max_degree + 2)
        g_xy, g_inf = FixedBaseMSM.multi_scalar_mul(g, pw[:max_degree + 1], curve=cid, group=1)
        gg_xy, gg_inf = FixedBaseMSM.multi_scalar_mul(gamma_g, pw, curve=cid, group=1)
        return UniversalParams(g_xy, g_inf, gg_xy, gg_inf)

    @staticmethod
    def commit(powers: RegisteredBases, coeffs, gamma_powers: RegisteredBases | None = None, blinding_coeffs=None) -> AffinePoint:
        """coeffs: (d + 1, S) uint64 Montgomery Fr, low degree first (DensePolynomial::coeffs)."""
        c = _coeffs(powers, coeffs)
        if len(c) > powers.n:
            raise ValueError("polynomial degree %d exceeds the %d registered powers" % (len(c) - 1, powers.n))
        W = coord_words(powers.curve, 1)
        out = np.zeros(2 * W, dtype=np.uint64)
        oinf = np.zeros(1, dtype=np.uint8)
        L = _lib.lib()
        if gamma_powers is None or blinding_coeffs is None:
            _lib.check(L.zkm_kzg_commit(powers.handle, _p(c), len(c), _p(out), _p(oinf)))
        else:
            b = _coeffs(powers, blinding_coeffs)
            _lib.check(L.zkm_kzg_commit_hiding(powers.handle, gamma_powers.handle, _p(c), len(c), _p(b), len(b), _p(out), _p(oinf)))
        return AffinePoint(powers.curve, 1, out, bool(oinf[0]))

    @staticmethod
    def commit_batch(powers: RegisteredBases, polys) -> list:
        """Non-hiding commitments of several polynomials over the same powers, issued concurrently in ONE call."""
        cs = [_coeffs(powers, p) for p in polys]
        k = len(cs)
        W = coord_words(powers.curve, 1)
        out = np.zeros((max(k, 1), 2 * W), dtype=np.uint64)
        oinf = np.zeros(max(k, 1), dtype=np.uint8)
        ptrs = (ctypes.c_void_p * max(k, 1))(*[c.ctypes.data if c.size else 0 for c in cs])
        ns = (ctypes.c_size_t * max(k, 1))(*[len(c) for c in cs])
        _lib.check(_lib.lib().zkm_kzg_commit_batch(powers.handle, k, ctypes.cast(ptrs, ctypes.c_void_p),
                                                   ctypes.cast(ns, ctypes.c_void_p), _p(out), _p(oinf)))
        return [AffinePoint(powers.curve, 1, out[i].copy(), bool(oinf[i])) for i in range(k)]

    @staticmethod
    def open(powers: RegisteredBases, coeffs, point, gamma_powers: RegisteredBases | None = None, blinding_coeffs=None) -> OpeningProof:
        """point: one Montgomery Fr element (S words)."""
        c = _coeffs(powers, coeffs)
        S = _lib.FR_WORDS[powers.curve]
        z = np.ascontiguousarray(point, dtype=np.uint64).reshape(S)
        W = coord_words(powers.curve, 1)
        out = np.zeros(2 * W, dtype=np.uint64)
        oinf = np.zeros(1, dtype=np.uint8)
        rv = np.zeros(S, dtype=np.uint64)
        hiding = gamma_powers is not None and blinding_coeffs is not None
        b = _coeffs(powers, blinding_coeffs) if hiding else None
        _lib.check(_lib.lib().zkm_kzg_open(powers.handle, gamma_powers.handle if hiding else 0, _p(c), len(c),
                                           _p(b) if hiding else ctypes.c_void_p(0), len(b) if hiding else 0, _p(z), _p(out),
                                           _p(oinf), _p(rv)))
        return OpeningProof(AffinePoint(powers.curve, 1, out, bool(oinf[0])), rv if hiding else None)
