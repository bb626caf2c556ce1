"""Fixed-base batch scalar multiplication (zkm_fixed_base_msm / FixedBaseMSM.multi_scalar_mul), the replacement of
ark-ec 0.3.0 FixedBaseMSM + batch_normalization_into_affine in the two setup paths.  Outputs are normalised affine
points, so the bar is byte equality with the exact big-int group law (oracle/py/exact.py); large batches are checked
on sampled indices, for normalisation, and by a weighted-sum identity evaluated with the variable-base MSM (a kernel
path that shares nothing with the fixed-base one)."""
import ctypes
import random

import numpy as np
import pytest

from oracle import capi
from oracle.py import exact, groth16_setup as gs, kzg_exact as kx
from oracle.py.params import BLS12_381, BN254, BW6_761

pytestmark = pytest.mark.gpu

PAIRS = [(c, g) for c in (BLS12_381, BN254, BW6_761) for g in (1, 2)]
PID = lambda p: "%s-g%d" % (p[0].name, p[1])


@pytest.fixture(scope="module")
def zkm():
    import zkmember_b200 as z
    z.init(0)
    return z


def _mont(curve, vals):
    return capi.ints_to_limbs([curve.fr.to_mont(v % curve.fr.modulus) for v in vals], curve.fr.limbs64)


def _rec(curve, g, P):
    xy, inf = exact.point_to_bytes(curve, g, P)
    return np.frombuffer(xy, dtype=np.uint64), inf


def _same(curve, g, xy_row, inf, P):
    want_xy, want_inf = _rec(curve, g, P)
    return int(inf) == want_inf and xy_row.tobytes() == want_xy.tobytes()


_CACHE = {}


def _base_and_edges(curve, g):
    """A random base B = k G and the edge scalars with their exact multiples (computed once per pair, incrementally
    where possible: the 2^k chain by doublings)."""
    key = (curve.name, g)
    if key in _CACHE:
        return _CACHE[key]
    G = exact.Group(curve, g)
    r, bits = curve.fr.modulus, curve.fr.bits
    rng = random.Random(1000 + 10 * curve.curve_id + g)
    B = G.mul(G.gen, rng.randrange(2, r))
    vals, pts = [], []

    def add(v, P=None):
        vals.append(v % r)
        pts.append(P if P is not None or v % r == 0 else G.mul(B, v % r))

    for v in (0, 1, 2, r - 1, r - 2, r - 3):
        add(v)
    P, negB = B, G.neg(B)
    for k in range(bits):                       # 2^k and 2^k - 1: every window boundary of every width
        if (1 << k) < r:
            add(1 << k, P)
            add((1 << k) - 1, G.add(P, negB) if k else None)
        P = G.double(P)
    for c in range(2, 21):                      # digits that carry into the next signed window
        W = (bits + c) // c
        for w in sorted({0, 1, W // 2, W - 2}):
            for pat in ((1 << c) - 1, (1 << (c - 1)) + 1, 1 << (c - 1)):
                v = pat << (c * w)
                if 0 < v < r:
                    add(v)
    top = (r >> (bits - 8)) << (bits - 8)       # the top window full
    add(top - 1)
    add(top - (1 << (bits - 9)))
    for i in (3, 17, 40):                       # repeated scalars
        add(vals[i], pts[i])
    _CACHE[key] = (B, vals, pts)
    return _CACHE[key]


@pytest.mark.parametrize("pair", PAIRS, ids=PID)
def test_fixed_base_small_exact(zkm, pair):
    curve, g = pair
    B, vals, pts = _base_and_edges(curve, g)
    base = _rec(curve, g, B)[0]
    for n in (1, 2, 31, 33, 257, len(vals)):
        xy, inf = zkm.FixedBaseMSM.multi_scalar_mul(base, _mont(curve, vals[:n]), curve=curve.name, group=g)
        assert xy.shape == (n, base.size) and inf.shape == (n,)
        for i in range(n):
            assert _same(curve, g, xy[i], inf[i], pts[i]), "n=%d i=%d scalar=%#x" % (n, i, vals[i])
    # a base at infinity: every output at infinity; n = 0 succeeds
    zero_xy, _ = _rec(curve, g, None)
    base_inf = zkm.AffinePoint(curve.curve_id, g, zero_xy, True)
    xy, inf = zkm.FixedBaseMSM.multi_scalar_mul(base_inf, _mont(curve, vals[:40]), curve=curve.name, group=g)
    assert inf.all() and all(xy[i].tobytes() == zero_xy.tobytes() for i in range(40))
    xy, inf = zkm.FixedBaseMSM.multi_scalar_mul(base, np.zeros((0, curve.fr.limbs64), np.uint64), curve=curve.name, group=g)
    assert xy.shape[0] == 0 and inf.shape == (0,)


def _rand_mont(curve, n, seed):
    """Random Montgomery limbs below 2^(bits - 1) (< r): the canonical values s = m R^-1 are spread over Fr."""
    S, bits = curve.fr.limbs64, curve.fr.bits
    rng = np.random.Generator(np.random.PCG64(seed))
    m = rng.integers(0, 1 << 64, size=(n, S), dtype=np.uint64)
    m[:, S - 1] &= np.uint64((1 << (bits - 1 - 64 * (S - 1))) - 1)
    return m


def _weighted_sum_mod_r(curve, m, rw):
    """sum_i rw_i * s_i mod r with s_i = m_i R^-1: exact limb products in 16-bit pieces (no uint64 overflow)."""
    r = curve.fr.modulus
    S = m.shape[1]
    m16 = m.view(np.uint16).reshape(len(m), 4 * S).astype(np.uint64)
    r16 = rw.view(np.uint16).reshape(len(rw), 4).astype(np.uint64)
    total = 0
    for lo in range(0, len(m), 1 << 20):
        mb, rb = m16[lo:lo + (1 << 20)], r16[lo:lo + (1 << 20)]
        for a in range(4):
            sums = (rb[:, a:a + 1] * mb).sum(axis=0, dtype=np.uint64)
            total += sum(int(v) << (16 * (a + k)) for k, v in enumerate(sums))
    return total * pow(1 << (64 * S), -1, r) % r


def _assert_normalised(curve, g, xy):
    q = curve.fq.modulus
    L = curve.fq.limbs64
    ql = [(q >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(L)]
    a = xy.reshape(len(xy), -1, L)
    lt = np.zeros(a.shape[:2], dtype=bool)
    eq = np.ones(a.shape[:2], dtype=bool)
    for k in range(L - 1, -1, -1):
        lt |= eq & (a[..., k] < np.uint64(ql[k]))
        eq &= a[..., k] == np.uint64(ql[k])
    assert lt.all(), "a coordinate is not reduced below q"


def _check_large(zkm, curve, g, n, seed):
    B, vals, pts = _base_and_edges(curve, g)
    base = _rec(curve, g, B)[0]
    m = _rand_mont(curve, n, seed)
    k = min(len(vals), n // 4)
    m[:k] = _mont(curve, vals[:k])                  # the edge scalars at the front: every width this n selects
    xy, inf = zkm.FixedBaseMSM.multi_scalar_mul(base, m, curve=curve.name, group=g)
    for i in range(k):
        assert _same(curve, g, xy[i], inf[i], pts[i]), "edge %d" % i
    G = exact.Group(curve, g)
    rinv = pow(1 << (64 * curve.fr.limbs64), -1, curve.fr.modulus)
    rng = random.Random(seed)
    for i in rng.sample(range(n), 256):
        s = capi.limbs_to_ints(m[i:i + 1])[0] * rinv % curve.fr.modulus
        assert _same(curve, g, xy[i], inf[i], G.mul(B, s) if s else None), "index %d" % i
    _assert_normalised(curve, g, xy)
    rw = np.random.Generator(np.random.PCG64(seed + 1)).integers(0, 1 << 64, size=n, dtype=np.uint64)
    rsc = np.zeros((n, curve.fr.limbs64), dtype=np.uint64)
    rsc[:, 0] = rw
    lhs = zkm.VariableBaseMSM.multi_scalar_mul(xy, rsc, curve=curve.name, group=g, infinity=inf)
    rhs = G.mul(B, _weighted_sum_mod_r(curve, m, rw))
    assert _same(curve, g, lhs.xy, lhs.infinity, rhs), "weighted-sum identity"


@pytest.mark.parametrize("log_n", [10, 16, 20])
@pytest.mark.parametrize("pair", PAIRS, ids=PID)
def test_fixed_base_large(zkm, pair, log_n):
    _check_large(zkm, pair[0], pair[1], 1 << log_n, 0xF1B0 + log_n)


def test_fixed_base_bls12_381_g1_2p24(zkm):
    _check_large(zkm, BLS12_381, 1, 1 << 24, 0xF1B024)


@pytest.mark.parametrize("pair", PAIRS, ids=PID)
def test_fixed_base_equals_synthetic_progression(zkm, pair):
    """s_i = a0 + i d over the generator equals the per-point double-and-add generator, byte for byte."""
    import torch
    curve, g = pair
    n, a0, d = 1 << 20, 0x1234567, 0x9E3779B1
    W2 = _rec(curve, g, None)[0].size
    r, R = curve.fr.modulus, 1 << (64 * curve.fr.limbs64)
    S = curve.fr.limbs64
    raw = b"".join(((a0 + i * d) * R % r).to_bytes(8 * S, "little") for i in range(n))
    m = np.frombuffer(raw, dtype=np.uint64).reshape(n, S)
    xy, inf = zkm.FixedBaseMSM.multi_scalar_mul(capi.generator_mont(curve.curve_id, g), m, curve=curve.name, group=g)
    assert not inf.any()
    d_b = torch.empty((n, W2), dtype=torch.int64, device="cuda")
    L = zkm.load()
    zkm._lib.check(L.zkm_testgen_progression_device(curve.curve_id, g, a0, d, n, ctypes.c_void_p(d_b.data_ptr()),
                                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert np.array_equal(d_b.cpu().numpy().view(np.uint64), xy)


@pytest.mark.parametrize("pair", PAIRS, ids=PID)
def test_fixed_base_device_entry_point(zkm, pair):
    import torch
    curve, g = pair
    B, vals, pts = _base_and_edges(curve, g)
    base = _rec(curve, g, B)[0]
    n = 5000
    m = _rand_mont(curve, n, 77 + curve.curve_id)
    m[:50] = _mont(curve, vals[:50])                 # zero among them: an infinity output
    want_xy, want_inf = zkm.FixedBaseMSM.multi_scalar_mul(base, m, curve=curve.name, group=g)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_s = torch.from_numpy(m.view(np.int64)).to("cuda")
        d_xy = torch.empty((n, base.size), dtype=torch.int64, device="cuda")
        d_inf = torch.empty(n, dtype=torch.uint8, device="cuda")
        zkm.FixedBaseMSM.multi_scalar_mul_device(base, d_s.data_ptr(), n, d_xy.data_ptr(), d_inf.data_ptr(), curve=curve.name,
                                                 group=g, stream=stream.cuda_stream)
    stream.synchronize()
    assert np.array_equal(d_xy.cpu().numpy().view(np.uint64), want_xy)
    assert np.array_equal(d_inf.cpu().numpy(), want_inf)
    # the device outputs registered as bases without a host round trip give the MSM of the host-registered copy
    L = zkm.load()
    h = ctypes.c_uint64(0)
    zkm._lib.check(L.zkm_bases_register_device(curve.curve_id, g, ctypes.c_void_p(d_xy.data_ptr()),
                                               ctypes.c_void_p(d_inf.data_ptr()), n, ctypes.byref(h)))
    try:
        sc = capi.random_scalars(curve.curve_id, n, seed=5)
        W2 = base.size
        out = np.zeros(W2, dtype=np.uint64)
        oinf = np.zeros(1, dtype=np.uint8)
        zkm._lib.check(L.zkm_msm_registered(h.value, 0, ctypes.c_void_p(sc.ctypes.data), n, ctypes.c_void_p(out.ctypes.data),
                                            ctypes.c_void_p(oinf.ctypes.data)))
        host = zkm.RegisteredBases(curve.curve_id, g, want_xy, want_inf)
        try:
            ref = host.msm(sc)
        finally:
            host.release()
        assert out.tobytes() == ref.xy.tobytes() and bool(oinf[0]) == ref.infinity
    finally:
        zkm._lib.check(L.zkm_bases_release(h.value))
    # a scalar >= r in the host entry point
    bad = m[:8].copy()
    bad[3] = capi.ints_to_limbs([curve.fr.modulus], curve.fr.limbs64)[0]
    with pytest.raises(zkm.ZkmError) as e:
        zkm.FixedBaseMSM.multi_scalar_mul(base, bad, curve=curve.name, group=g)
    assert e.value.code == -5


def _arr(curve, g, pts):
    xy = np.stack([_rec(curve, g, Q)[0] for Q in pts])
    inf = np.array([_rec(curve, g, Q)[1] for Q in pts], dtype=np.uint8)
    return xy, inf


def _setup_scalars(curve, cs, seed):
    """The field side of oracle/py/groth16_setup.generate_parameters, restated with the same draws from the same seeded
    RNG: the trapdoor and the scalar of every point of every query, in the order ark-groth16 0.3.0 src/generator.rs
    feeds them to its fixed-base batches.  The test below checks that the points built from them on the GPU are exactly
    the points generate_parameters returns."""
    p = curve.fr.modulus
    rng = random.Random(seed)
    log_n = cs.domain_log()
    n = 1 << log_n
    t = rng.randrange(2, p)
    while pow(t, n, p) == 1:
        t = rng.randrange(2, p)
    alpha, beta, gamma, delta = (rng.randrange(1, p) for _ in range(4))
    u = gs.lagrange_at(curve.fr, log_n, t)
    nv = cs.num_variables
    a, b, c = [0] * nv, [0] * nv, [0] * nv
    for j in range(cs.num_instance):
        a[j] = u[cs.num_constraints + j]
    for i in range(cs.num_constraints):
        for j, coef in cs.A[i].items():
            a[j] = (a[j] + u[i] * coef) % p
        for j, coef in cs.B[i].items():
            b[j] = (b[j] + u[i] * coef) % p
        for j, coef in cs.C[i].items():
            c[j] = (c[j] + u[i] * coef) % p
    zt = (pow(t, n, p) - 1) % p
    dinv, ginv = pow(delta, -1, p), pow(gamma, -1, p)
    abc = [(beta * a[j] + alpha * b[j] + c[j]) % p for j in range(nv)]
    return {
        "alpha": alpha, "beta": beta, "gamma": gamma, "delta": delta,
        "a_query": a, "b_g1_query": b, "b_g2_query": b,
        "h_query": [zt * dinv % p * pow(t, i, p) % p for i in range(n - 1)],
        "l_query": [abc[j] * dinv % p for j in range(cs.num_instance, nv)],
        "gamma_abc_g1": [abc[j] * ginv % p for j in range(cs.num_instance)],
    }


def _kzg_setup(curve, max_degree, beta, g, gamma_g):
    """KZG10::setup (ark-poly-commit 0.3.0 src/kzg10/mod.rs) for given draws, in exact arithmetic: powers_of_g[i] =
    beta^i g for i <= max_degree, powers_of_gamma_g[i] = beta^i gamma_g for i <= max_degree + 1 (upstream pushes
    last * beta after the fixed-base batch, "to support up to D queries"); beta^i by the running product from one."""
    p = curve.fr.modulus
    G = exact.Group(curve, 1)
    pw, cur = [], 1
    for _ in range(max_degree + 2):
        pw.append(cur)
        cur = cur * beta % p
    return [G.mul(g, b) for b in pw[:max_degree + 1]], [G.mul(gamma_g, b) for b in pw]


@pytest.mark.parametrize("circuit", ["cubic", "gadgets"])
def test_groth16_setup_fixed_base_end_to_end(zkm, circuit):
    from zkmember_b200.groth16 import ProvingKey, create_proof
    C = BLS12_381
    P = C.fr.modulus
    cs, z = gs.cubic_circuit(0xC0FFEE, P) if circuit == "cubic" else gs.random_circuit(num_constraints=27, num_inputs=3, seed=11, p=P)
    par = gs.generate_parameters(C, cs, seed=3)
    sc = _setup_scalars(C, cs, seed=3)
    g1, g2 = capi.generator_mont(C.curve_id, 1), capi.generator_mont(C.curve_id, 2)
    built = {}
    for name, g in (("a_query", 1), ("b_g1_query", 1), ("b_g2_query", 2), ("h_query", 1), ("l_query", 1), ("gamma_abc_g1", 1)):
        built[name] = zkm.FixedBaseMSM.multi_scalar_mul(g1 if g == 1 else g2, _mont(C, sc[name]), curve=C.name, group=g)
        want = par["vk"][name] if name == "gamma_abc_g1" else par["pk"][name]
        wxy, winf = _arr(C, g, want)
        assert np.array_equal(built[name][0], wxy) and np.array_equal(built[name][1], winf), name
    one = lambda g, k: zkm.FixedBaseMSM.multi_scalar_mul(g1 if g == 1 else g2, _mont(C, [k]), curve=C.name, group=g)[0][0]
    zpk = ProvingKey(C.name, one(1, sc["alpha"]), one(1, sc["beta"]), one(2, sc["beta"]), one(1, sc["delta"]), one(2, sc["delta"]),
                     built["a_query"][0], built["b_g1_query"][0], built["b_g2_query"][0], built["h_query"][0], built["l_query"][0],
                     infinity={"a": built["a_query"][1], "b_g1": built["b_g1_query"][1], "b_g2": built["b_g2_query"][1],
                               "h": built["h_query"][1], "l": built["l_query"][1]}, precompute=False)
    rng = random.Random(99)
    r, s = rng.randrange(P), rng.randrange(P)
    a, b, c = cs.evaluation_vectors(z, P)
    inputs, aux = z[1:cs.num_instance], z[cs.num_instance:]
    try:
        canon = lambda v: capi.ints_to_limbs(v, C.fr.limbs64)
        proof = create_proof(zpk, r, s, _mont(C, a), _mont(C, b), _mont(C, c), canon(inputs), canon(aux))
    finally:
        zpk.release()
    pt = lambda ap, g: exact.point_from_bytes(C, g, ap.xy.tobytes(), 1 if ap.infinity else 0)
    A, Bp, Cc = pt(proof.a, 1), pt(proof.b, 2), pt(proof.c, 1)
    assert gs.verify_proof(C, par["vk"], inputs, A, Bp, Cc)
    bad = list(inputs)
    bad[-1] = (bad[-1] + 1) % P
    assert not gs.verify_proof(C, par["vk"], bad, A, Bp, Cc)


@pytest.mark.parametrize("curve", [BLS12_381, BN254, BW6_761], ids=lambda c: c.name)
def test_kzg10_setup_end_to_end(zkm, curve):
    from zkmember_b200.kzg import KZG10, Powers
    p = curve.fr.modulus
    rng = random.Random(31 + curve.curve_id)
    G = exact.Group(curve, 1)
    beta = rng.randrange(2, p)
    g, gamma_g = G.mul(G.gen, rng.randrange(2, p)), G.mul(G.gen, rng.randrange(2, p))
    max_degree = 24
    up = KZG10.setup(curve.name, max_degree, _mont(curve, [beta])[0], _rec(curve, 1, g)[0], _rec(curve, 1, gamma_g)[0])
    want_g, want_gg = _kzg_setup(curve, max_degree, beta, g, gamma_g)
    assert len(want_g) == max_degree + 1 and len(want_gg) == max_degree + 2
    assert np.array_equal(up.powers_of_g, _arr(curve, 1, want_g)[0]) and not up.powers_of_g_inf.any()
    assert np.array_equal(up.powers_of_gamma_g, _arr(curve, 1, want_gg)[0]) and not up.powers_of_gamma_g_inf.any()
    pw, gw = Powers(curve.name, up.powers_of_g), Powers(curve.name, up.powers_of_gamma_g)
    try:
        coeffs = [rng.randrange(p) for _ in range(max_degree + 1)]
        blind = [rng.randrange(p) for _ in range(3)]
        got = KZG10.commit(pw, _mont(curve, coeffs), gw, _mont(curve, blind))
        assert exact.point_from_bytes(curve, 1, got.xy.tobytes(), int(got.infinity)) == kx.commit(curve, want_g, coeffs, want_gg, blind)
        zpt = rng.randrange(p)
        pr = KZG10.open(pw, _mont(curve, coeffs), _mont(curve, [zpt])[0], gw, _mont(curve, blind))
        w, rv = kx.open_(curve, want_g, coeffs, zpt, want_gg, blind)
        assert exact.point_from_bytes(curve, 1, pr.w.xy.tobytes(), int(pr.w.infinity)) == w
        assert capi.limbs_to_ints(pr.random_v[None, :])[0] == curve.fr.to_mont(rv)
    finally:
        pw.release()
        gw.release()
