"""TEST INFRASTRUCTURE ONLY (oracle) -- never imported by the product path.

Exact restatement of ark-poly-commit 0.3.0's MarlinKZG10 (src/marlin/marlin_pc/mod.rs), written from upstream's
per-polynomial loops rather than from the batched form the library runs:

  commit(p)        comm = KZG10::commit(powers_of_g, p) [+ MSM(powers_of_gamma_g, rand)]
                   bounded p (bound d): shifted_comm = MSM(powers_of_g[D - d ..], p) [+ MSM(powers_of_gamma_g, shifted_rand)]
  open at z        counter k from 0; every p: xi^k p into P and xi^k rand into R, k += 1; a bounded p also
                   xi^k X^(D - d) q_(p, z) into the shifted witness, xi^k q_(shifted_rand, z) into the hiding witness,
                   xi^k shifted_rand(z) into random_v, k += 1.
                   w = MSM(powers_of_g, q_(P, z)) + MSM(powers_of_g, shifted witness) + MSM(powers_of_gamma_g, q_(R, z) +
                   hiding parts); random_v = R(z) + shifted parts   (two MSMs over powers_of_g, as upstream)
  batch_open       one proof per point label in sorted order, the point's labels sorted (BTreeMap / BTreeSet)
  open_combinations  each LC -> sum a_t p_t with its one degree bound; LCTerm::One (label None) only in evaluations
  batch_check      per point, C = sum xi^k (comm - v g) + xi^(k+1) (shifted_comm - v g^(beta^(D - d))), then
                   e(C - random_v gamma_g + z W, h) = e(W, beta h)   on the exact BLS12-381 pairing of pairing.py

Polynomials are lists of canonical integers; points are oracle/py/exact.py affine tuples.
"""
from typing import Dict, List, Optional, Sequence, Tuple

from . import exact, pairing
from .kzg_exact import evaluate, witness_polynomial
from .params import BLS12_381, CurveParams


class Srs:
    def __init__(self, curve: CurveParams, powers: Sequence, gamma_powers: Sequence):
        self.curve = curve
        self.powers = list(powers)
        self.gamma_powers = list(gamma_powers)
        self.D = len(self.powers) - 1
        self.G = exact.Group(curve, 1)

    def msm(self, bases, coeffs, start: int = 0):
        return self.G.msm_naive(bases[start:start + len(coeffs)], list(coeffs))


def _padd(r: int, a: List[int], b: Sequence[int], k: int = 1, shift: int = 0) -> List[int]:
    n = max(len(a), len(b) + shift)
    out = list(a) + [0] * (n - len(a))
    for i, v in enumerate(b):
        out[i + shift] = (out[i + shift] + k * v) % r
    return out


def commit(srs: Srs, coeffs, bound: Optional[int] = None, rand=None, shifted_rand=None):
    G = srs.G
    comm = srs.msm(srs.powers, coeffs)
    if rand:
        comm = G.add(comm, srs.msm(srs.gamma_powers, rand))
    if bound is None:
        return comm, None
    shifted = srs.msm(srs.powers, coeffs, srs.D - bound)
    if shifted_rand:
        shifted = G.add(shifted, srs.msm(srs.gamma_powers, shifted_rand))
    return comm, shifted


def open_point(srs: Srs, polys: Sequence[Tuple], z: int, xi: int):
    """polys: (coeffs, bound, rand, shifted_rand) in opening order.  Returns (w, random_v)."""
    r = srs.curve.fr.modulus
    P, R, shifted_w, shifted_rw, shifted_rv = [], [], [], [], 0
    k = 0
    for coeffs, bound, rand, shifted_rand in polys:
        c = pow(xi, k, r)
        P = _padd(r, P, coeffs, c)
        R = _padd(r, R, rand or [], c)
        k += 1
        if bound is not None:
            c = pow(xi, k, r)
            shifted_w = _padd(r, shifted_w, witness_polynomial(r, coeffs, z), c, srs.D - bound)
            if shifted_rand:
                shifted_rw = _padd(r, shifted_rw, witness_polynomial(r, shifted_rand, z), c)
                shifted_rv = (shifted_rv + c * evaluate(r, shifted_rand, z)) % r
            k += 1
    G = srs.G
    w = G.add(srs.msm(srs.powers, witness_polynomial(r, P, z)), srs.msm(srs.powers, shifted_w))
    hw = _padd(r, witness_polynomial(r, R, z), shifted_rw)
    w = G.add(w, srs.msm(srs.gamma_powers, hw))
    return w, (evaluate(r, R, z) + shifted_rv) % r


def _group(query_set):
    pts: Dict[str, Tuple[int, set]] = {}
    for lab, (pl, z) in query_set:
        pts.setdefault(pl, (z, set()))[1].add(lab)
    return [(pl, pts[pl][0], sorted(pts[pl][1])) for pl in sorted(pts)]


def batch_open(srs: Srs, polys: Dict[str, Tuple], query_set, xi: int):
    """polys: label -> (coeffs, bound, rand, shifted_rand).  Returns ({point_label: (w, random_v)}, {(label, pl): v})."""
    r = srs.curve.fr.modulus
    proofs, evals = {}, {}
    for pl, z, labels in _group(query_set):
        proofs[pl] = open_point(srs, [polys[lab] for lab in labels], z, xi)
        for lab in labels:
            evals[(lab, pl)] = evaluate(r, polys[lab][0], z)
    return proofs, evals


def combine(srs: Srs, lcs: Dict[str, Sequence[Tuple]], polys: Dict[str, Tuple]) -> Tuple[Dict[str, Tuple], Dict[str, int]]:
    """lcs: label -> [(coefficient, poly label or None)].  Returns (the LC polynomials, the constant of each LC)."""
    r = srs.curve.fr.modulus
    out, ones = {}, {}
    for lab, terms in lcs.items():
        real = [(a, l) for a, l in terms if l is not None]
        ones[lab] = sum(a for a, l in terms if l is None) % r
        bound = None
        if len(terms) == 1 and real and polys[real[0][1]][1] is not None:
            assert real[0][0] % r == 1
            bound = polys[real[0][1]][1]
        else:
            assert all(polys[l][1] is None for _, l in real)
        p, rd, srd = [], [], []
        for a, l in real:
            c, _, rand, srand = polys[l]
            p = _padd(r, p, c, a)
            rd = _padd(r, rd, rand or [], a)
            srd = _padd(r, srd, srand or [], a)
        out[lab] = (p, bound, rd, srd if bound is not None else None)
    return out, ones


def open_combinations(srs: Srs, lcs, polys, query_set, xi: int):
    r = srs.curve.fr.modulus
    lc_polys, ones = combine(srs, lcs, polys)
    proofs, evals = batch_open(srs, lc_polys, query_set, xi)
    return proofs, {key: (v + ones[key[0]]) % r for key, v in evals.items()}


def batch_check(srs: Srs, h, beta_h, comms: Dict[str, Tuple], bounds: Dict[str, Optional[int]], query_set,
                evals: Dict[Tuple[str, str], int], proofs: Dict[str, Tuple], xi: int) -> bool:
    """MarlinKZG10::batch_check on BLS12-381 with one challenge; comms: label -> (comm, shifted_comm)."""
    assert srs.curve is BLS12_381
    r = srs.curve.fr.modulus
    G = srs.G
    g, gamma_g = srs.powers[0], srs.gamma_powers[0]
    for pl, z, labels in _group(query_set):
        C, v, k = None, 0, 0
        for lab in labels:
            val = evals[(lab, pl)]
            c = pow(xi, k, r)
            C = G.add(C, G.mul(comms[lab][0], c))
            v = (v + c * val) % r
            k += 1
            if bounds[lab] is not None:
                c = pow(xi, k, r)
                shift_power = srs.powers[srs.D - bounds[lab]]
                adjusted = G.add(comms[lab][1], G.neg(G.mul(shift_power, val)))
                C = G.add(C, G.mul(adjusted, c))
                k += 1
        w, random_v = proofs[pl]
        lhs = G.add(G.add(C, G.neg(G.mul(g, v))), G.neg(G.mul(gamma_g, random_v or 0)))
        lhs = G.add(lhs, G.mul(w, z))
        if not pairing.pairing_product_is_one([(lhs, h), (G.neg(w), beta_h)]):
            return False
    return True
