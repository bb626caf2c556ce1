"""Host-side mirror of ark-poly-commit 0.3.0's MarlinKZG10 (src/marlin/marlin_pc/mod.rs): the polynomial commitment
Marlin calls, with degree bounds and batch openings.

    MarlinKZG10.commit(ck, polys, rands)                          one `zkm_kzg_commit_many` call per 23 items
    MarlinKZG10.batch_open(ck, polys, query_set, xi, rands)       one `zkm_kzg_open_batch` call
    MarlinKZG10.open_combinations(ck, lcs, polys, query_set, xi, rands)

The MarlinKZG10 bookkeeping lives here and the group and polynomial work on the GPU.  A polynomial p with degree bound d
has a second commitment over powers_of_g[D - d ..] (D = max degree of the registered powers), with its own hiding term.
Opening at a point z walks the point's polynomials (sorted by label, as upstream's BTreeSet) with a counter k from 0:
p contributes xi^k p to the main witness, and a bounded p also xi^(k+1) X^(D - d) q_(p, z) with its shifted
randomness.  The library folds the xi powers and the linear-combination coefficients into one coefficient per term and
divides each combination once.  Blinding polynomials are the caller's RNG, as in `KZG10`.
Field elements are Montgomery Fr limbs (numpy uint64, S words each) at the interface, integers mod r inside.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from .kzg import Powers, _p
from .msm import AffinePoint, coord_words
from .serialize import FR_MODULUS

MAX_ITEMS = 23     # MSM pairs one call takes at once (two lanes each out of the 48 of a device)


def _to_int(curve: int, limbs) -> int:
    """Montgomery limbs -> canonical integer."""
    S = _lib.FR_WORDS[curve]
    m = int.from_bytes(np.ascontiguousarray(limbs, dtype=np.uint64).reshape(S).tobytes(), "little")
    r = FR_MODULUS[curve]
    return m * pow(1 << (64 * S), -1, r) % r


def _to_mont(curve: int, v: int) -> np.ndarray:
    S = _lib.FR_WORDS[curve]
    r = FR_MODULUS[curve]
    return np.frombuffer((v % r * (1 << (64 * S)) % r).to_bytes(8 * S, "little"), dtype=np.uint64).copy()


def _coeffs(curve: int, c) -> np.ndarray:
    """(n, S) limbs without trailing zero coefficients, as DensePolynomial keeps them (the library's bound checks count
    every coefficient it is given)."""
    S = _lib.FR_WORDS[curve]
    a = np.ascontiguousarray(c if c is not None else np.zeros((0, S)), dtype=np.uint64).reshape(-1, S)
    nz = np.flatnonzero(a.any(axis=1))
    return a[:nz[-1] + 1] if len(nz) else a[:0]


def degree(c: np.ndarray) -> int:
    """DensePolynomial::degree: index of the top non-zero coefficient (0 for the zero polynomial)."""
    nz = np.flatnonzero(c.any(axis=1)) if c.size else []
    return int(nz[-1]) if len(nz) else 0


@dataclass
class CommitterKey:
    """ark_poly_commit::marlin_pc::CommitterKey: `powers` holds powers_of_g[0..=D], `gamma_powers` powers_of_gamma_g."""
    powers: Powers
    gamma_powers: Powers | None
    supported_degree: int
    enforced_degree_bounds: list | None = None

    @property
    def max_degree(self) -> int:
        return self.powers.n - 1

    def shift(self, bound: int) -> int:
        if not self.enforced_degree_bounds or bound not in self.enforced_degree_bounds:
            raise ValueError("degree bound %d is not among the enforced bounds %s" % (bound, self.enforced_degree_bounds))
        return self.max_degree - bound


@dataclass
class LabeledPolynomial:
    label: str
    coeffs: np.ndarray                  # (n, S) Montgomery Fr, low degree first
    degree_bound: int | None = None
    hiding_bound: int | None = None


@dataclass
class Randomness:
    """marlin_pc::Randomness: the blinding polynomial of the commitment and, with a degree bound, of the shifted one."""
    rand: np.ndarray | None = None
    shifted_rand: np.ndarray | None = None


@dataclass
class Commitment:
    comm: AffinePoint
    shifted_comm: AffinePoint | None = None


@dataclass
class Proof:
    """kzg10::Proof { w, random_v }; random_v: Montgomery limbs, None when no polynomial at the point is hiding."""
    w: AffinePoint
    random_v: np.ndarray | None


@dataclass
class LinearCombination:
    """(coefficient, label) terms; the label None is LCTerm::One.  Coefficients are canonical integers mod r."""
    label: str
    terms: list = field(default_factory=list)


def _check_degrees(ck: CommitterKey, p: LabeledPolynomial, c: np.ndarray):
    d = degree(c)
    if d > ck.supported_degree:
        raise ValueError("%s: degree %d exceeds the supported degree %d" % (p.label, d, ck.supported_degree))
    if p.degree_bound is not None:
        ck.shift(p.degree_bound)
        if d > p.degree_bound:
            raise ValueError("%s: degree %d exceeds its degree bound %d" % (p.label, d, p.degree_bound))


class MarlinKZG10:
    @staticmethod
    def commit(ck: CommitterKey, polys, rands=None) -> list:
        """MarlinKZG10::commit after its random draws: rands[i] (Randomness or None) are polys[i]'s blinding
        polynomials.  Returns one Commitment per polynomial."""
        curve = ck.powers.curve
        rands = rands or [None] * len(polys)
        items = []       # (coeffs, shift, blind)
        for p, rd in zip(polys, rands):
            c = _coeffs(curve, p.coeffs)
            _check_degrees(ck, p, c)
            items.append((c, 0, None if rd is None else rd.rand))
            if p.degree_bound is not None:
                items.append((c, ck.shift(p.degree_bound), None if rd is None else rd.shifted_rand))
        pts = []
        for k in range(0, len(items), MAX_ITEMS):
            pts += _commit_many(ck, items[k:k + MAX_ITEMS])
        out, k = [], 0
        for p in polys:
            if p.degree_bound is None:
                out.append(Commitment(pts[k]))
                k += 1
            else:
                out.append(Commitment(pts[k], pts[k + 1]))
                k += 2
        return out

    @staticmethod
    def batch_open(ck: CommitterKey, polys, query_set, xi: int, rands=None):
        """MarlinKZG10::batch_open with one opening challenge xi (canonical integer).  query_set: (label, (point_label,
        point)) with the point a canonical integer.  Returns ({point_label: Proof}, {(label, point_label): value})."""
        curve = ck.powers.curve
        rands = rands or [None] * len(polys)
        by_label = {p.label: (p, rd) for p, rd in zip(polys, rands)}
        points = _group_queries(query_set)
        terms, groups = [], []
        for pl, (z, labels) in points:
            k = 0
            for lab in labels:
                p, rd = by_label[lab]
                _check_degrees(ck, p, _coeffs(curve, p.coeffs))
                terms.append((len(groups), lab, None if rd is None else rd.rand, 0, pow(xi, k, FR_MODULUS[curve]), (lab, pl)))
                k += 1
                if p.degree_bound is not None:
                    terms.append((len(groups), lab, None if rd is None else rd.shifted_rand, ck.shift(p.degree_bound),
                                  pow(xi, k, FR_MODULUS[curve]), None))
                    k += 1
            groups.append((pl, z))
        proofs, ev = _open_batch(ck, {p.label: p.coeffs for p in polys}, groups, terms)
        return proofs, {key: v for key, v in ev if key is not None}

    @staticmethod
    def open_combinations(ck: CommitterKey, lcs, polys, query_set, xi: int, rands=None):
        """MarlinKZG10::open_combinations: every LinearCombination becomes a polynomial with its terms' degree bound (at
        most one, and then the LC is that polynomial alone with coefficient 1); LCTerm::One only enters the evaluation.
        Returns ({point_label: Proof}, {(lc_label, point_label): value})."""
        curve = ck.powers.curve
        r = FR_MODULUS[curve]
        rands = rands or [None] * len(polys)
        by_label = {p.label: (p, rd) for p, rd in zip(polys, rands)}
        by_lc = {lc.label: lc for lc in lcs}
        points = _group_queries(query_set)
        terms, groups, ones = [], [], {}
        for pl, (z, labels) in points:
            k = 0
            for lab in labels:
                lc = by_lc[lab]
                real = [(a, l) for a, l in lc.terms if l is not None]
                ones[(lab, pl)] = sum(a for a, l in lc.terms if l is None) % r
                bounded = [l for _, l in real if by_label[l][0].degree_bound is not None]
                if bounded and (len(lc.terms) != 1 or real[0][0] % r != 1):    # upstream counts LCTerm::One too
                    raise ValueError("%s: a degree-bounded polynomial must be alone in its combination, with coefficient 1" % lab)
                for a, l in real:
                    p, rd = by_label[l]
                    _check_degrees(ck, p, _coeffs(curve, p.coeffs))
                    terms.append((len(groups), l, None if rd is None else rd.rand, 0, pow(xi, k, r) * a % r, (lab, pl, a)))
                k += 1
                if bounded:
                    p, rd = by_label[bounded[0]]
                    terms.append((len(groups), p.label, None if rd is None else rd.shifted_rand, ck.shift(p.degree_bound),
                                  pow(xi, k, r), None))
                    k += 1
            groups.append((pl, z))
        proofs, ev = _open_batch(ck, {p.label: p.coeffs for p in polys}, groups, terms)
        evals = dict(ones)
        for key, v in ev:
            if key is not None:
                lab, pl, a = key
                evals[(lab, pl)] = (evals[(lab, pl)] + a * v) % r
        return proofs, evals


def _group_queries(query_set):
    """upstream's BTreeMap<point_label, (point, BTreeSet<label>)>, in order."""
    pts = {}
    for lab, (pl, z) in query_set:
        pts.setdefault(pl, (z, set()))[1].add(lab)
    return [(pl, (pts[pl][0], sorted(pts[pl][1]))) for pl in sorted(pts)]


def _commit_many(ck: CommitterKey, items) -> list:
    curve = ck.powers.curve
    k = len(items)
    W = coord_words(curve, 1)
    out = np.zeros((max(k, 1), 2 * W), dtype=np.uint64)
    oinf = np.zeros(max(k, 1), dtype=np.uint8)
    cs = [c for c, _, _ in items]
    bs = [_coeffs(curve, b) for _, _, b in items]
    if any(len(b) for b in bs) and ck.gamma_powers is None:
        raise ValueError("hiding commitments need powers_of_gamma_g")
    arr = lambda ct, vals: ctypes.cast((ct * max(len(vals), 1))(*vals), ctypes.c_void_p)
    ptrs = arr(ctypes.c_void_p, [c.ctypes.data if c.size else 0 for c in cs])
    ns = arr(ctypes.c_size_t, [len(c) for c in cs])
    sh = arr(ctypes.c_size_t, [s for _, s, _ in items])
    bptrs = arr(ctypes.c_void_p, [b.ctypes.data if b.size else 0 for b in bs])
    nbs = arr(ctypes.c_size_t, [len(b) for b in bs])
    _lib.check(_lib.lib().zkm_kzg_commit_many(ck.powers.handle, ck.gamma_powers.handle if ck.gamma_powers else 0, k, ptrs, ns,
                                              sh, bptrs, nbs, _p(out), _p(oinf)))
    return [AffinePoint(curve, 1, out[i].copy(), bool(oinf[i])) for i in range(k)]


def _open_batch(ck: CommitterKey, coeffs_by_label: dict, groups, terms):
    """groups: [(point_label, z)]; terms: (group, poly label, blinding coeffs or None, shift, coefficient, key).
    Returns ({point_label: Proof}, [(key, value of the term's polynomial at its point)])."""
    curve = ck.powers.curve
    S = _lib.FR_WORDS[curve]
    W = coord_words(curve, 1)
    labels = sorted({t[1] for t in terms})
    pidx = {lab: i for i, lab in enumerate(labels)}
    polys = [_coeffs(curve, coeffs_by_label[lab]) for lab in labels]
    blinds = [_coeffs(curve, t[2]) for t in terms]
    bidx = [i if t[2] is not None and len(blinds[i]) else -1 for i, t in enumerate(terms)]
    hiding = {g for (g, *_), b in zip(terms, bidx) if b >= 0}
    if hiding and ck.gamma_powers is None:
        raise ValueError("hiding openings need powers_of_gamma_g")
    npt, nt = len(groups), len(terms)
    arr = lambda ct, vals: ctypes.cast((ct * max(len(vals), 1))(*vals), ctypes.c_void_p)
    cp = arr(ctypes.c_void_p, [c.ctypes.data if c.size else 0 for c in polys])
    cn = arr(ctypes.c_size_t, [len(c) for c in polys])
    bp = arr(ctypes.c_void_p, [b.ctypes.data if b.size else 0 for b in blinds])
    bn = arr(ctypes.c_size_t, [len(b) for b in blinds])
    zs = np.concatenate([_to_mont(curve, z) for _, z in groups]) if groups else np.zeros(S, np.uint64)
    tp = arr(ctypes.c_int32, [t[0] for t in terms])
    tq = arr(ctypes.c_int32, [pidx[t[1]] for t in terms])
    tb = arr(ctypes.c_int32, bidx)
    ts = arr(ctypes.c_size_t, [t[3] for t in terms])
    tc = np.concatenate([_to_mont(curve, t[4]) for t in terms]) if terms else np.zeros(S, np.uint64)
    w = np.zeros((max(npt, 1), 2 * W), dtype=np.uint64)
    winf = np.zeros(max(npt, 1), dtype=np.uint8)
    rv = np.zeros((max(npt, 1), S), dtype=np.uint64)
    ev = np.zeros((max(nt, 1), S), dtype=np.uint64)
    _lib.check(_lib.lib().zkm_kzg_open_batch(ck.powers.handle, ck.gamma_powers.handle if ck.gamma_powers else 0, len(polys), cp, cn,
                                             nt, bp, bn, npt, _p(zs), nt, tp, tq, tb, ts, _p(tc), _p(w), _p(winf), _p(rv), _p(ev)))
    proofs = {pl: Proof(AffinePoint(curve, 1, w[i].copy(), bool(winf[i])), rv[i].copy() if i in hiding else None)
              for i, (pl, _) in enumerate(groups)}
    return proofs, [(t[5], _to_int(curve, ev[i])) for i, t in enumerate(terms)]
