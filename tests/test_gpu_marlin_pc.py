"""MarlinKZG10 on the GPU (zkm_kzg_commit_many, zkm_kzg_open_batch[_device]): exact bytes against the restatement in
oracle/py/marlin_pc_exact.py on three curves, GPU proofs through the BLS12-381 pairing check, a Marlin-sized opening
against the C++ oracle's MSM of exact witness coefficients, the device form, concurrent calls and the error codes."""
import ctypes
import random
import threading

import numpy as np
import pytest

from oracle import capi
from oracle.py import exact, kzg_exact as kx, marlin_pc_exact as mx
from oracle.py.params import BLS12_381, BN254, BW6_761

CURVES = [BLS12_381, BN254, BW6_761]
D = 64
BOUNDS = [30, 62, 64]


@pytest.fixture(scope="module")
def zkm():
    import zkmember_b200 as z
    z.init(0)
    return z


def _arr(curve, pts):
    return np.stack([np.frombuffer(exact.point_to_bytes(curve, 1, Q)[0], dtype=np.uint64) for Q in pts])


def _mont(fr, vals):
    return capi.ints_to_limbs([fr.to_mont(v) for v in vals], fr.limbs64).reshape(-1, fr.limbs64)


def _pt(curve, ap):
    return exact.point_from_bytes(curve, 1, ap.xy.tobytes(), 1 if ap.infinity else 0)


class Setup:
    def __init__(self, curve, seed):
        from zkmember_b200.kzg import Powers
        from zkmember_b200.marlin_pc import CommitterKey
        self.curve, fr = curve, curve.fr
        r = self.r = fr.modulus
        rng = self.rng = random.Random(seed)
        G = exact.Group(curve, 1)
        self.beta, gamma = rng.randrange(2, r), rng.randrange(2, r)
        self.srs = mx.Srs(curve, [G.mul(G.gen, pow(self.beta, i, r)) for i in range(D + 1)],
                          [G.mul(G.gen, gamma * pow(self.beta, i, r) % r) for i in range(D + 2)])
        self.pg = Powers(curve.curve_id, _arr(curve, self.srs.powers))
        self.pgg = Powers(curve.curve_id, _arr(curve, self.srs.gamma_powers))
        self.ck = CommitterKey(self.pg, self.pgg, D, BOUNDS)
        rnd = lambda n: [rng.randrange(r) for _ in range(n)]
        c_lead = [0, 0, 0] + rnd(20)                          # leading zeros
        z_root = rng.randrange(r)
        f = rnd(10)                                            # p(X) = (X - z_root) f(X): a root at z_root
        p_root = [0] * 11
        for i, v in enumerate(f):
            p_root[i + 1] = (p_root[i + 1] + v) % r
            p_root[i] = (p_root[i] - z_root * v) % r
        self.z_root = z_root
        self.polys = {   # label -> (coeffs, bound, rand, shifted_rand)
            "a": (rnd(41), None, rnd(3), None),
            "b": (rnd(31), 30, rnd(3), rnd(3)),
            "c": (rnd(65), 64, rnd(2), rnd(2)),               # d = D
            "d": (c_lead, None, None, None),                   # no hiding
            "e": ([], None, rnd(2), None),                     # the zero polynomial
            "f": (p_root, 62, None, None),                     # bounded, no hiding
        }

    def labeled(self):
        from zkmember_b200.marlin_pc import LabeledPolynomial, Randomness
        fr = self.curve.fr
        m = lambda v: _mont(fr, v) if v else None
        ps = [LabeledPolynomial(lab, _mont(fr, c) if c else np.zeros((0, fr.limbs64), np.uint64), b) for lab, (c, b, _, _) in
              self.polys.items()]
        rs = [Randomness(m(rd), m(srd)) if rd or srd else None for (_, _, rd, srd) in self.polys.values()]
        return ps, rs


@pytest.fixture(scope="module", params=CURVES, ids=lambda c: c.name)
def setup(zkm, request):
    return Setup(request.param, 100 + request.param.curve_id)


@pytest.mark.gpu
def test_commit_many_exact(setup):
    from zkmember_b200.marlin_pc import MarlinKZG10
    ps, rs = setup.labeled()
    got = MarlinKZG10.commit(setup.ck, ps, rs)
    for p, cm in zip(ps, got):
        want = mx.commit(setup.srs, *setup.polys[p.label])
        assert _pt(setup.curve, cm.comm) == want[0], p.label
        if want[1] is None:
            assert cm.shifted_comm is None
        else:
            assert _pt(setup.curve, cm.shifted_comm) == want[1], p.label


@pytest.mark.gpu
def test_bounded_polynomial_with_trailing_zero_coefficients(setup):
    """A degree-30 polynomial handed in with 40 coefficients fits its bound (DensePolynomial has no trailing zeros)."""
    from zkmember_b200.marlin_pc import LabeledPolynomial, MarlinKZG10
    s = setup
    c = [s.rng.randrange(s.r) for _ in range(31)]
    p = LabeledPolynomial("t", np.concatenate([_mont(s.curve.fr, c), np.zeros((9, s.curve.fr.limbs64), np.uint64)]), 30)
    cm = MarlinKZG10.commit(s.ck, [p])[0]
    want = mx.commit(s.srs, c, 30)
    assert _pt(s.curve, cm.comm) == want[0] and _pt(s.curve, cm.shifted_comm) == want[1]
    proofs, evals = MarlinKZG10.batch_open(s.ck, [p], [("t", ("z", 9))], 5)
    wp, we = mx.batch_open(s.srs, {"t": (c, 30, None, None)}, [("t", ("z", 9))], 5)
    _same_proofs(s, proofs, wp)
    assert evals == we


def _queries(s):
    zb, zg = s.rng.randrange(s.r), s.z_root
    return [("a", ("beta", zb)), ("b", ("beta", zb)), ("c", ("beta", zb)), ("d", ("beta", zb)), ("e", ("beta", zb)),
            ("a", ("gamma", zg)), ("c", ("gamma", zg)), ("f", ("gamma", zg)), ("d", ("zero", 0)), ("b", ("zero", 0))]


def _same_proofs(s, got, want):
    assert sorted(got) == sorted(want)
    for pl, (w, rv) in want.items():
        assert _pt(s.curve, got[pl].w) == w, pl
        grv = 0 if got[pl].random_v is None else s.curve.fr.from_mont(capi.limbs_to_ints(got[pl].random_v.reshape(1, -1))[0])
        assert grv == rv, pl


@pytest.mark.gpu
def test_batch_open_exact(setup):
    from zkmember_b200.marlin_pc import MarlinKZG10
    s = setup
    ps, rs = s.labeled()
    qs = _queries(s)
    xi = s.rng.randrange(s.r)
    proofs, evals = MarlinKZG10.batch_open(s.ck, ps, qs, xi, rs)
    wp, we = mx.batch_open(s.srs, s.polys, qs, xi)
    _same_proofs(s, proofs, wp)
    assert evals == we
    assert evals[("f", "gamma")] == 0                           # z a root of f


@pytest.mark.gpu
def test_open_combinations_exact(setup):
    from zkmember_b200.marlin_pc import LinearCombination, MarlinKZG10
    s = setup
    ps, rs = s.labeled()
    r = s.r
    k1, k2 = s.rng.randrange(r), s.rng.randrange(r)
    lcs = {"outer": [(1, "a"), (k1, "d"), (k2, None)], "inner": [(k2, "a"), (1, "e"), (5, None)], "g1": [(1, "b")],
           "g2": [(1, "c")]}
    zb, zg = s.rng.randrange(r), s.rng.randrange(r)
    qs = [("outer", ("beta", zb)), ("g1", ("beta", zb)), ("inner", ("gamma", zg)), ("g2", ("gamma", zg)), ("outer", ("gamma", zg))]
    xi = s.rng.randrange(r)
    proofs, evals = MarlinKZG10.open_combinations(s.ck, [LinearCombination(k, v) for k, v in lcs.items()], ps, qs, xi, rs)
    wp, we = mx.open_combinations(s.srs, lcs, s.polys, qs, xi)
    _same_proofs(s, proofs, wp)
    assert evals == we


@pytest.mark.gpu
def test_gpu_proofs_pass_the_pairing_check_and_tampered_ones_fail(zkm):
    from zkmember_b200.marlin_pc import MarlinKZG10
    s = Setup(BLS12_381, 7)
    ps, rs = s.labeled()
    keep = {"a", "b", "c"}
    ps = [p for p in ps if p.label in keep]
    rs = [rd for p, rd in zip(s.labeled()[0], s.labeled()[1]) if p.label in keep]
    comms = {p.label: (_pt(s.curve, c.comm), c.shifted_comm and _pt(s.curve, c.shifted_comm))
             for p, c in zip(ps, MarlinKZG10.commit(s.ck, ps, rs))}
    zb, zg = s.rng.randrange(s.r), s.rng.randrange(s.r)
    qs = [("a", ("beta", zb)), ("c", ("beta", zb)), ("a", ("gamma", zg)), ("b", ("gamma", zg))]
    xi = s.rng.randrange(s.r)
    proofs, evals = MarlinKZG10.batch_open(s.ck, ps, qs, xi, rs)
    fr = s.curve.fr
    pr = {pl: (_pt(s.curve, p.w), fr.from_mont(capi.limbs_to_ints(p.random_v.reshape(1, -1))[0])) for pl, p in proofs.items()}
    G2 = exact.Group(s.curve, 2)
    bounds = {lab: s.polys[lab][1] for lab in keep}
    check = lambda **o: mx.batch_check(s.srs, G2.gen, G2.mul(G2.gen, s.beta), o.get("comms", comms), bounds, qs,
                                       o.get("evals", evals), o.get("proofs", pr), xi)
    assert check()
    bad = dict(evals)
    bad[("b", "gamma")] = (bad[("b", "gamma")] + 1) % s.r
    assert not check(evals=bad)
    assert not check(proofs={"beta": pr["gamma"], "gamma": pr["gamma"]})


def _raw_open(s, polys, blinds, zs, terms, device=False, evals=True):
    """zkm_kzg_open_batch[_device] with explicit terms (point, poly, blind, shift, coefficient int)."""
    import torch
    from zkmember_b200 import _lib
    cid, fr = s.curve.curve_id, s.curve.fr
    S, W = fr.limbs64, 2 * capi.coord_words(cid, 1)
    arr = lambda ct, v: ctypes.cast((ct * max(len(v), 1))(*v), ctypes.c_void_p)
    P = [_mont(fr, c) if c else np.zeros((0, S), np.uint64) for c in polys]
    B = [_mont(fr, c) if c else np.zeros((0, S), np.uint64) for c in blinds]
    zsm, tc = _mont(fr, zs), _mont(fr, [t[4] for t in terms])
    args_t = [arr(ctypes.c_int32, [t[i] for t in terms]) for i in range(3)] + [arr(ctypes.c_size_t, [t[3] for t in terms])]
    p = lambda a: ctypes.c_void_p(a.ctypes.data)
    L = _lib.lib()
    if not device:
        w = np.zeros((len(zs), W), np.uint64)
        wi = np.zeros(len(zs), np.uint8)
        rv = np.zeros((len(zs), S), np.uint64)
        ev = np.zeros((max(len(terms), 1), S), np.uint64)
        rc = L.zkm_kzg_open_batch(s.pg.handle, s.pgg.handle, len(P), arr(ctypes.c_void_p, [a.ctypes.data if a.size else 0 for a in P]),
                                  arr(ctypes.c_size_t, [len(a) for a in P]), len(B),
                                  arr(ctypes.c_void_p, [a.ctypes.data if a.size else 0 for a in B]),
                                  arr(ctypes.c_size_t, [len(a) for a in B]), len(zs), p(zsm), len(terms), *args_t, p(tc), p(w), p(wi),
                                  p(rv), p(ev) if evals else None)
        return rc, (np.concatenate([w, wi[:, None].astype(np.uint64)], axis=1), rv, ev[:len(terms)])
    dev = lambda a: torch.from_numpy(a.view(np.int64).copy()).cuda() if a.size else torch.zeros(2, dtype=torch.int64, device="cuda")
    dP, dB = [dev(a) for a in P], [dev(a) for a in B]
    dw = torch.zeros(len(zs) * (W + 1), dtype=torch.int64, device="cuda")
    drv = torch.zeros(len(zs) * S, dtype=torch.int64, device="cuda")
    dev_ = torch.zeros(max(len(terms), 1) * S, dtype=torch.int64, device="cuda")
    rc = L.zkm_kzg_open_batch_device(s.pg.handle, s.pgg.handle, len(P), arr(ctypes.c_void_p, [t.data_ptr() for t in dP]),
                                     arr(ctypes.c_size_t, [len(a) for a in P]), len(B), arr(ctypes.c_void_p, [t.data_ptr() for t in dB]),
                                     arr(ctypes.c_size_t, [len(a) for a in B]), len(zs), p(zsm), len(terms), *args_t, p(tc),
                                     ctypes.c_void_p(dw.data_ptr()), ctypes.c_void_p(drv.data_ptr()), ctypes.c_void_p(dev_.data_ptr()),
                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    u = lambda t: t.cpu().numpy().view(np.uint64)
    return rc, (u(dw).reshape(len(zs), W + 1), u(drv).reshape(len(zs), S), u(dev_).reshape(-1, S)[:len(terms)])


@pytest.mark.gpu
def test_device_form_equals_the_host_form(setup):
    s = setup
    r = s.r
    polys = [v[0] for v in s.polys.values()]
    blinds = [s.polys["a"][2], s.polys["b"][3]]
    zs = [s.rng.randrange(r), 0]
    terms = [(0, 0, 0, 0, 1), (0, 1, 1, D - 30, s.rng.randrange(r)), (1, 2, -1, 0, 3), (1, 0, 0, 0, 5), (0, 4, -1, 7, 9)]
    rc, host = _raw_open(s, polys, blinds, zs, terms)
    assert rc == 0
    rc, devr = _raw_open(s, polys, blinds, zs, terms, device=True)
    assert rc == 0
    for a, b in zip(host, devr):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_eight_concurrent_calls(setup):
    from zkmember_b200.marlin_pc import MarlinKZG10
    s = setup
    ps, rs = s.labeled()
    jobs = []
    for k in range(8):
        z = s.rng.randrange(s.r)
        jobs.append(([("a", ("p", z)), ("b", ("p", z)), ("c", ("q", (z + k) % s.r))], s.rng.randrange(s.r)))
    want = [mx.batch_open(s.srs, s.polys, qs, xi) for qs, xi in jobs]
    got = [None] * 8

    def run(k):
        got[k] = MarlinKZG10.batch_open(s.ck, ps, jobs[k][0], jobs[k][1], rs)
    th = [threading.Thread(target=run, args=(k,)) for k in range(8)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for k in range(8):
        _same_proofs(s, got[k][0], want[k][0])
        assert got[k][1] == want[k][1]


@pytest.mark.gpu
def test_errors(zkm):
    from zkmember_b200 import _lib
    from zkmember_b200.kzg import Powers
    s = Setup(BN254, 3)
    polys, blinds = [s.polys["a"][0]], [s.polys["a"][2]]
    z = [5]
    assert _raw_open(s, polys, blinds, z, [(1, 0, -1, 0, 1)])[0] == -1           # point out of range
    assert _raw_open(s, polys, blinds, z, [(0, 1, -1, 0, 1)])[0] == -1           # polynomial out of range
    assert _raw_open(s, polys, blinds, z, [(0, 0, 1, 0, 1)])[0] == -1            # blinding polynomial out of range
    assert _raw_open(s, polys, blinds, z, [(0, 0, 0, D - 39, 1)])[0] == 0        # 41 coefficients: 40 witness ones, to D + 1
    assert _raw_open(s, polys, blinds, z, [(0, 0, 0, D - 38, 1)])[0] == -6       # one past the registered powers
    g2 = capi.progression(s.curve.curve_id, 2, 3, 5, 8)
    h = ctypes.c_uint64(0)
    _lib.check(_lib.lib().zkm_bases_register(s.curve.curve_id, 2, ctypes.c_void_p(g2.ctypes.data), None, 8, ctypes.byref(h)))
    s.pgg_saved, s.pg_saved = s.pgg, s.pg
    s.pgg = type("H", (), {"handle": h.value})()
    assert _raw_open(s, polys, blinds, z, [(0, 0, 0, 0, 1)])[0] == -1            # a G2 registration
    s.pgg = s.pgg_saved
    other = Powers(BLS12_381.curve_id, capi.progression(BLS12_381.curve_id, 1, 3, 5, 8))
    s.pgg = other
    assert _raw_open(s, polys, blinds, z, [(0, 0, 0, 0, 1)])[0] == -1            # another curve
    s.pgg = s.pgg_saved
    _lib.check(_lib.lib().zkm_bases_release(h.value))
    pts = capi.progression(s.curve.curve_id, 1, 3, 5, D + 1)
    _lib.check(_lib.lib().zkm_bases_register(s.curve.curve_id, 1, ctypes.c_void_p(pts.ctypes.data), None, D + 1, ctypes.byref(h)))
    _lib.check(_lib.lib().zkm_bases_release(h.value))
    s.pg = type("H", (), {"handle": h.value})()
    assert _raw_open(s, polys, blinds, z, [(0, 0, -1, 0, 1)])[0] == -6           # a released handle
    s.pg = s.pg_saved
    assert _raw_open(s, polys, blinds, z, [(0, 0, -1, 0, 1)] * 65536)[0] == -1   # more terms than one grid holds


@pytest.mark.gpu
def test_marlin_sized_open_against_the_cpp_oracle(zkm):
    """|H| = 2^15, |K| = 2^17, D = 6 |K|: zkMember's opening at beta (g_1 bounded by |H| - 2, z_b, t and a mask) and gamma
    (g_2 bounded by |K| - 2 and the inner-sumcheck combination), W_i against capi.msm of exact witness coefficients."""
    from zkmember_b200.kzg import Powers
    curve = BLS12_381
    cid, fr = curve.curve_id, curve.fr
    r = fr.modulus
    H, K = 1 << 15, 1 << 17
    Dm = 6 * K
    bases = capi.progression(cid, 1, 11, 13, Dm + 1)
    gbases = capi.progression(cid, 1, 17, 19, Dm + 2)
    s = type("S", (), {})()
    s.curve, s.pg, s.pgg = curve, Powers(cid, bases), Powers(cid, gbases)
    rng = random.Random(5)
    rnd = lambda n: [rng.randrange(r) for _ in range(n)]
    polys = [rnd(H - 1), rnd(2 * H), rnd(H), rnd(3 * H), rnd(K - 1), rnd(6 * K - 5), rnd(3 * K)]   # g1 zb t mask g2 a b
    blinds = [rnd(2) for _ in polys] + [rnd(2), rnd(2)]
    zb, zg = rng.randrange(r), rng.randrange(r)
    x = [rng.randrange(r) for _ in range(12)]
    terms = [(0, 0, 0, 0, x[0]), (0, 0, 7, Dm - (H - 2), x[1]), (0, 1, 1, 0, x[2]), (0, 2, 2, 0, x[3]), (0, 3, 3, 0, x[4]),
             (1, 4, 4, 0, x[5]), (1, 4, 8, Dm - (K - 2), x[6]), (1, 5, 5, 0, x[7]), (1, 6, 6, 0, x[8]), (1, 1, 1, 0, x[9])]
    rc, (w, rv, ev) = _raw_open(s, polys, blinds, [zb, zg], terms)
    assert rc == 0, _lib_err()
    for i, z in enumerate((zb, zg)):
        wg, wh, rvi = [], [], 0
        for (pt, pi, bi, sh, c) in terms:
            if pt != i:
                continue
            wg = mx._padd(r, wg, kx.witness_polynomial(r, polys[pi], z), c, sh)
            wh = mx._padd(r, wh, kx.witness_polynomial(r, blinds[bi], z), c)
            rvi = (rvi + c * kx.evaluate(r, blinds[bi], z)) % r
        G = exact.Group(curve, 1)
        pg = exact.point_from_bytes(curve, 1, capi.msm(cid, 1, bases[:len(wg)], capi.ints_to_limbs(wg, fr.limbs64))[0].tobytes(), 0)
        ph = exact.point_from_bytes(curve, 1, capi.msm(cid, 1, gbases[:len(wh)], capi.ints_to_limbs(wh, fr.limbs64))[0].tobytes(), 0)
        want = G.add(pg, ph)
        assert exact.point_from_bytes(curve, 1, w[i, :-1].tobytes(), int(w[i, -1])) == want
        assert fr.from_mont(capi.limbs_to_ints(rv[i:i + 1])[0]) == rvi
    for t, (pt, pi, _, _, _) in enumerate(terms):
        assert fr.from_mont(capi.limbs_to_ints(ev[t:t + 1])[0]) == kx.evaluate(r, polys[pi], (zb, zg)[pt])


def _lib_err():
    from zkmember_b200 import _lib
    return _lib.load().zkm_last_error()
