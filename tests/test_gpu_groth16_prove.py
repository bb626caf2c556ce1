"""Groth16 `create_proof` as one device-resident call (zkm_groth16_pk_create / zkm_groth16_prove[_device]): proof bytes
against the exact restatement of ark-groth16 0.3.0 src/prover.rs (oracle/py/groth16_exact.py), edge scalars, genuine
circuits through the pairing verifier, zkMember sizes against the per-call orchestration the one call replaces, the
device form, concurrency, placement of the G2 query on another device, key lifetime and argument errors."""
import ctypes
import random
import threading

import numpy as np
import pytest

from oracle import capi
from oracle.py import exact, groth16_exact as gx, groth16_setup as gs
from oracle.py.params import BLS12_381, BN254, BW6_761

pytestmark = pytest.mark.gpu

CURVES = [BLS12_381, BN254, BW6_761]
ERR_ARG, ERR_SCALAR_RANGE, ERR_HANDLE = -1, -5, -6


@pytest.fixture(scope="module")
def zkm():
    import zkmember_b200 as z
    z.init(0)
    return z


def _arr(curve, g, pts):
    xy = np.stack([np.frombuffer(exact.point_to_bytes(curve, g, P)[0], dtype=np.uint64) for P in pts])
    inf = np.array([exact.point_to_bytes(curve, g, P)[1] for P in pts], dtype=np.uint8)
    return xy, inf


def _device_key(curve, pk, precompute=True):
    """zkmember_b200.groth16.ProvingKey from an exact proving key (dict of exact points, None = infinity)."""
    from zkmember_b200.groth16 import ProvingKey
    q = {k: _arr(curve, 2 if k == "b_g2_query" else 1, pk[k]) for k in ("a_query", "b_g1_query", "b_g2_query", "h_query", "l_query")}
    one = lambda g, P: _arr(curve, g, [P])[0][0]
    return ProvingKey(curve.name, one(1, pk["alpha_g1"]), one(1, pk["beta_g1"]), one(2, pk["beta_g2"]), one(1, pk["delta_g1"]),
                      one(2, pk["delta_g2"]), q["a_query"][0], q["b_g1_query"][0], q["b_g2_query"][0], q["h_query"][0],
                      q["l_query"][0], infinity={"a": q["a_query"][1], "b_g1": q["b_g1_query"][1], "b_g2": q["b_g2_query"][1],
                                                 "h": q["h_query"][1], "l": q["l_query"][1]}, precompute=precompute)


def _exact_pk(curve, rng, n, num_inputs, m):
    """Shaped like test_groth16_proof._pk: arbitrary points, infinity and repeats in the b queries."""
    G1, G2 = exact.Group(curve, 1), exact.Group(curve, 2)
    p1 = G1.progression(rng.randrange(1, 1 << 20), rng.randrange(1, 1 << 20), 3 * (m + 1) + (n - 1) + (m - num_inputs) + 3)
    p2 = G2.progression(rng.randrange(1, 1 << 20), rng.randrange(1, 1 << 20), (m + 1) + 2)
    it1, it2 = iter(p1), iter(p2)
    pk = {"alpha_g1": next(it1), "beta_g1": next(it1), "delta_g1": next(it1), "beta_g2": next(it2), "delta_g2": next(it2)}
    pk["a_query"] = [next(it1) for _ in range(m + 1)]
    pk["b_g1_query"] = [next(it1) for _ in range(m + 1)]
    pk["b_g2_query"] = [next(it2) for _ in range(m + 1)]
    pk["h_query"] = [next(it1) for _ in range(n - 1)]
    pk["l_query"] = [next(it1) for _ in range(m - num_inputs)]
    for i in (2, 5):
        pk["b_g1_query"][i] = None
        pk["b_g2_query"][i] = None
    pk["b_g1_query"][7] = pk["b_g1_query"][6]
    pk["b_g2_query"][8] = pk["b_g2_query"][9]
    return pk


def _prove(curve, dpk, r, s, a, b, c, inputs, aux):
    from zkmember_b200.groth16 import create_proof
    fr = curve.fr
    mont = lambda v: capi.ints_to_limbs([fr.to_mont(x) for x in v], fr.limbs64)
    canon = lambda v: capi.ints_to_limbs(v, fr.limbs64)
    return create_proof(dpk, r, s, mont(a), mont(b), mont(c), canon(inputs), canon(aux))


def _instance(curve, seed, log_n=4, num_inputs=2, m=13, zero_assignment=False):
    rng = random.Random(seed)
    fr = curve.fr
    n = 1 << log_n
    pk = _exact_pk(curve, rng, n, num_inputs, m)
    a, b, c = ([rng.randrange(fr.modulus) for _ in range(n)] for _ in range(3))
    inputs = [0 if zero_assignment else rng.randrange(fr.modulus) for _ in range(num_inputs)]
    aux = [0 if zero_assignment else rng.choice([0, 1, rng.randrange(fr.modulus)]) for _ in range(m - num_inputs)]
    return pk, a, b, c, inputs, aux, rng


# 1. exact bytes
@pytest.mark.parametrize("curve", CURVES, ids=lambda c: c.name)
@pytest.mark.parametrize("precompute", [False, True])
def test_proof_bytes_equal_exact_prover(zkm, curve, precompute):
    pk, a, b, c, inputs, aux, rng = _instance(curve, 77 + curve.curve_id)
    r, s = rng.randrange(curve.fr.modulus), rng.randrange(curve.fr.modulus)
    dpk = _device_key(curve, pk, precompute)
    try:
        got = _prove(curve, dpk, r, s, a, b, c, inputs, aux).serialize()
    finally:
        dpk.release()
    assert got == gx.serialize_proof(curve, *gx.create_proof(curve, pk, r, s, a, b, c, inputs, aux))


# 2. edge scalars, and a key whose A is the identity (arkworks' zero encoding)
@pytest.mark.parametrize("curve", CURVES, ids=lambda c: c.name)
def test_edge_scalars(zkm, curve):
    P = curve.fr.modulus
    pk, a, b, c, inputs, aux, rng = _instance(curve, 5 + curve.curve_id)
    _, _, _, _, zin, zaux, _ = _instance(curve, 5 + curve.curve_id, zero_assignment=True)
    dpk = _device_key(curve, pk)
    try:
        cases = [(0, 123), (456, 0), (0, 0), (P - 1, P - 1), (P - 1, 7)]
        for r, s in cases:
            got = _prove(curve, dpk, r, s, a, b, c, inputs, aux).serialize()
            assert got == gx.serialize_proof(curve, *gx.create_proof(curve, pk, r, s, a, b, c, inputs, aux)), (r, s)
        got = _prove(curve, dpk, 11, 13, a, b, c, zin, zaux).serialize()
        assert got == gx.serialize_proof(curve, *gx.create_proof(curve, pk, 11, 13, a, b, c, zin, zaux))
    finally:
        dpk.release()
    # A = r delta + alpha + a_0 + MSM(a_query[1..], z) = identity: r = 0, zero assignment, a_0 = -alpha
    G1 = exact.Group(curve, 1)
    pk["a_query"][0] = G1.neg(pk["alpha_g1"])
    dpk = _device_key(curve, pk)
    try:
        proof = _prove(curve, dpk, 0, 99, a, b, c, zin, zaux)
    finally:
        dpk.release()
    assert proof.a.infinity
    assert np.array_equal(proof.a.xy, _arr(curve, 1, [None])[0][0])      # x = 0, y = 1 (Montgomery)
    assert proof.serialize() == gx.serialize_proof(curve, *gx.create_proof(curve, pk, 0, 99, a, b, c, zin, zaux))


# 3. genuine circuits through the pairing verifier
@pytest.mark.parametrize("circuit", ["cubic", "gadgets"])
def test_genuine_circuit_verifies(zkm, circuit):
    C, P = BLS12_381, BLS12_381.fr.modulus
    if circuit == "cubic":
        cs, z = gs.cubic_circuit(0xBEEF, P)
    else:
        cs, z = gs.random_circuit(num_constraints=21, num_inputs=3, seed=17, p=P)
    par = gs.generate_parameters(C, cs, seed=8)
    rng = random.Random(3)
    r, s = rng.randrange(P), rng.randrange(P)
    a, b, c = cs.evaluation_vectors(z, P)
    inputs, aux = z[1:cs.num_instance], z[cs.num_instance:]
    dpk = _device_key(C, par["pk"])
    try:
        proof = _prove(C, dpk, r, s, a, b, c, inputs, aux)
    finally:
        dpk.release()
    pt = lambda ap, g: exact.point_from_bytes(C, g, ap.xy.tobytes(), 1 if ap.infinity else 0)
    A, B, Cc = pt(proof.a, 1), pt(proof.b, 2), pt(proof.c, 1)
    assert gs.verify_proof(C, par["vk"], inputs, A, B, Cc)
    bad = list(inputs)
    bad[0] = (bad[0] + 1) % P
    assert not gs.verify_proof(C, par["vk"], bad, A, B, Cc)


# ---------------------------------------------------------------------------------------- zkMember sizes
def _synthetic(cid, log_n, seed, precompute=True):
    """A key of zkMember's shape from progressions (known discrete logs), 50 % infinity in the b queries, witness-like
    assignment.  Returns (ProvingKey, kwargs of create_proof)."""
    from zkmember_b200.groth16 import ProvingKey
    n = 1 << log_n
    m, num_inputs = n - 5, 3
    num_aux = m - num_inputs
    rng = np.random.Generator(np.random.PCG64(seed))
    g1 = capi.progression(cid, 1, 3 + seed, 7, 3 * m + n + 8)
    g2 = capi.progression(cid, 2, 5 + seed, 11, m + 3)
    inf_b1 = (rng.random(m + 1) < 0.5).astype(np.uint8)
    inf_b2 = (rng.random(m + 1) < 0.5).astype(np.uint8)
    pk = ProvingKey(cid, g1[-1], g1[-2], g2[-1], g1[-3], g2[-2], g1[:m + 1], g1[m + 1:2 * m + 2], g2[:m + 1],
                    g1[2 * m + 2:2 * m + 1 + n], g1[2 * m + 1 + n:2 * m + 1 + n + num_aux],
                    infinity={"b_g1": inf_b1, "b_g2": inf_b2}, precompute=precompute)
    abc = [capi.random_field_elements(cid, n, seed=seed + k) for k in range(3)]
    full = capi.random_scalars(cid, m, seed=seed + 9, kind="witness")
    args = dict(r=int(rng.integers(1, 1 << 62)) ** 4, s=int(rng.integers(1, 1 << 62)) ** 4, a=abc[0], b=abc[1], c=abc[2],
                input_assignment=full[:num_inputs], aux_assignment=full[num_inputs:])
    return pk, args


def _old_create_proof(pk, r, s, a, b, c, input_assignment, aux_assignment):
    """The parent revision's create_proof: host witness map, five host MSM calls, assembly by four tiny MSMs."""
    from zkmember_b200.groth16 import witness_map
    from zkmember_b200.kzg import KZG10
    from zkmember_b200.msm import VariableBaseMSM, FR_WORDS
    from zkmember_b200.serialize import Proof, FR_MODULUS
    curve = pk.curve
    S = FR_WORDS[curve]

    def lincomb(group, terms):
        xy = np.stack([t[0] for t in terms])
        inf = np.array([1 if t[1] else 0 for t in terms], dtype=np.uint8)
        sc = np.stack([np.array([((t[2] % FR_MODULUS[curve]) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(S)],
                                dtype=np.uint64) for t in terms])
        return VariableBaseMSM.multi_scalar_mul(xy, sc, curve=curve, group=group, infinity=inf)

    h = witness_map(a, b, c, curve=curve)
    n = len(h)
    inputs = np.ascontiguousarray(input_assignment, dtype=np.uint64).reshape(-1, S)
    aux = np.ascontiguousarray(aux_assignment, dtype=np.uint64).reshape(-1, S)
    full = np.concatenate([inputs, aux])
    h_acc = KZG10.commit(pk.msms.h, h[:n - 1])
    l_acc = pk.msms.l.msm(aux)
    a_acc = pk.msms.a.msm(full)
    b1_acc = pk.msms.b_g1.msm(full)
    b2_acc = pk.msms.b_g2.msm(full)
    g_a = lincomb(1, [(pk.delta_g1, False, r), (*pk.first["a"], 1), (a_acc.xy, a_acc.infinity, 1), (pk.alpha_g1, False, 1)])
    g1_b = lincomb(1, [(pk.delta_g1, False, s), (*pk.first["b_g1"], 1), (b1_acc.xy, b1_acc.infinity, 1), (pk.beta_g1, False, 1)])
    g2_b = lincomb(2, [(pk.delta_g2, False, s), (*pk.first["b_g2"], 1), (b2_acc.xy, b2_acc.infinity, 1), (pk.beta_g2, False, 1)])
    g_c = lincomb(1, [(g_a.xy, g_a.infinity, s), (g1_b.xy, g1_b.infinity, r), (pk.delta_g1, False, -(r * s)),
                      (l_acc.xy, l_acc.infinity, 1), (h_acc.xy, h_acc.infinity, 1)])
    return Proof(a=g_a, b=g2_b, c=g_c)


# 4. zkMember sizes against the per-call orchestration
@pytest.mark.parametrize("cid,log_n", [(0, 15), (0, 16), (2, 15), (2, 16)], ids=["bls12_381-15", "bls12_381-16", "bw6_761-15",
                                                                               "bw6_761-16"])
def test_zkmember_sizes_equal_per_call_orchestration(zkm, cid, log_n):
    from zkmember_b200.groth16 import create_proof
    pk, args = _synthetic(cid, log_n, seed=40 + log_n)
    try:
        got = create_proof(pk, **args)
        want = _old_create_proof(pk, **args)
    finally:
        pk.release()
    assert got.serialize() == want.serialize()
    assert got.a == want.a and got.b == want.b and got.c == want.c


# ---------------------------------------------------------------------------------------- device form
def _dev(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.int64).copy()).cuda()


def _records(pk, args):
    """Run the device form; returns the three records (uint64) and the launches it made."""
    import torch
    import zkmember_b200 as z
    from zkmember_b200.msm import coord_words
    cid = pk.curve
    n = len(args["a"])
    log_n = n.bit_length() - 1
    full = np.concatenate([args["input_assignment"], args["aux_assignment"]])
    d_a, d_b, d_c, d_z = _dev(args["a"]), _dev(args["b"]), _dev(args["c"]), _dev(full)
    W1, W2 = coord_words(cid, 1), coord_words(cid, 2)
    d_out = torch.zeros(2 * (2 * W1 + 1) + 2 * W2 + 1 + 2, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    before = z.launch_count()
    pk.prove_device(d_a.data_ptr(), d_b.data_ptr(), d_c.data_ptr(), log_n, d_z.data_ptr(), len(args["input_assignment"]),
                    args["r"], args["s"], d_out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    launches = z.launch_count() - before
    torch.cuda.synchronize()
    out = d_out.cpu().numpy().view(np.uint64)
    return out[:2 * W1 + 1], out[2 * W1 + 1:2 * W1 + 2 * W2 + 2], out[2 * W1 + 2 * W2 + 2:4 * W1 + 2 * W2 + 3], launches


@pytest.mark.parametrize("cid", [0, 1, 2], ids=["bls12_381", "bn254", "bw6_761"])
def test_device_form_equals_host_form(zkm, cid):
    from zkmember_b200._lib import ZkmError
    from zkmember_b200.groth16 import create_proof
    from zkmember_b200.msm import FR_WORDS
    pk, args = _synthetic(cid, 10, seed=3)
    try:
        want = create_proof(pk, **args)
        ra, rb, rc, _ = _records(pk, args)
        _, _, _, l1 = _records(pk, args)
        _, _, _, l2 = _records(pk, args)
        assert l1 == l2 and l1 > 0
        for rec, p in ((ra, want.a), (rb, want.b), (rc, want.c)):
            assert rec[-1] == (1 if p.infinity else 0)
            assert np.array_equal(rec[:-1], p.xy)
        # a non-canonical assignment element: flag 2 in every record of the device form, ZKM_ERR_SCALAR_RANGE from the host form
        bad = dict(args)
        aux = np.array(args["aux_assignment"], copy=True)
        aux[5] = capi.ints_to_limbs([CURVES[cid].fr.modulus], FR_WORDS[cid])[0]
        bad["aux_assignment"] = aux
        ra, rb, rc, _ = _records(pk, bad)
        assert ra[-1] == 2 and rb[-1] == 2 and rc[-1] == 2
        with pytest.raises(ZkmError) as e:
            create_proof(pk, **bad)
        assert e.value.code == ERR_SCALAR_RANGE
    finally:
        pk.release()


# 6. concurrency
def test_concurrent_proofs_equal_sequential(zkm):
    from zkmember_b200.groth16 import create_proof
    pk, args = _synthetic(0, 12, seed=21)
    jobs = []
    for k in range(8):
        j = dict(args)
        j["aux_assignment"] = capi.random_scalars(0, len(args["aux_assignment"]), seed=100 + k, kind="witness")
        j["r"], j["s"] = 1000 + k, 2000 + 3 * k
        jobs.append(j)
    try:
        seq = [create_proof(pk, **j).serialize() for j in jobs]
        par = [None] * 8
        errs = []

        def run(k):
            try:
                par[k] = create_proof(pk, **jobs[k]).serialize()
            except Exception as e:   # surfaced below
                errs.append(e)
        th = [threading.Thread(target=run, args=(k,)) for k in range(8)]
        for t in th:
            t.start()
        for t in th:
            t.join()
    finally:
        pk.release()
    assert not errs
    assert par == seq
    assert len(set(seq)) == 8


# 8. lifetime and errors
def test_key_outlives_handles_and_errors(zkm):
    from zkmember_b200 import _lib
    from zkmember_b200.groth16 import create_proof
    pk, args = _synthetic(0, 9, seed=8)
    want = create_proof(pk, **args).serialize()
    pk.msms.release()                          # the five registrations go; the key keeps its references
    assert create_proof(pk, **args).serialize() == want
    L = _lib.lib()
    S = 4
    n = len(args["a"])
    full = np.ascontiguousarray(np.concatenate([args["input_assignment"], args["aux_assignment"]]))
    ni, na = len(args["input_assignment"]), len(args["aux_assignment"])
    out1, out2, out3 = np.zeros(12, np.uint64), np.zeros(24, np.uint64), np.zeros(12, np.uint64)
    inf = np.zeros(3, np.uint8)
    p = lambda x: ctypes.c_void_p(x.ctypes.data)
    one = np.array([1, 0, 0, 0], np.uint64)

    def call(handle=None, log_n=n.bit_length() - 1, ni=ni, na=na, r=one, s=one):
        return L.zkm_groth16_prove(pk.handle if handle is None else handle, p(args["a"]), p(args["b"]), p(args["c"]), log_n,
                                   p(full), ni, na, p(r), p(s), p(out1), p(inf), p(out2), ctypes.c_void_p(inf.ctypes.data + 1),
                                   p(out3), ctypes.c_void_p(inf.ctypes.data + 2))
    assert call() == 0
    assert call(ni=ni + 1) == ERR_ARG                                   # num_inputs + num_aux != len(a_query) - 1
    assert call(ni=ni + 1, na=na - 1) == ERR_ARG                        # len(l_query) != num_aux
    assert call(log_n=n.bit_length() - 3) == ERR_ARG                    # len(h_query) > 2^log_n
    modulus = capi.ints_to_limbs([BLS12_381.fr.modulus], S)[0]
    assert call(r=modulus) == ERR_SCALAR_RANGE
    assert call(s=modulus) == ERR_SCALAR_RANGE
    # handles of the wrong group / curve / length
    from zkmember_b200.msm import RegisteredBases
    g1 = capi.progression(0, 1, 1, 1, 8)
    g2 = capi.progression(0, 2, 1, 1, 8)
    bn1 = capi.progression(1, 1, 1, 1, 8)
    regs = [RegisteredBases(0, 1, g1), RegisteredBases(0, 1, g1), RegisteredBases(0, 1, g1), RegisteredBases(0, 1, g1),
            RegisteredBases(0, 2, g2), RegisteredBases(0, 1, g1[:7]), RegisteredBases(1, 1, bn1)]
    pts1, pts2 = np.ascontiguousarray(np.tile(g1[0], (5, 1))), np.ascontiguousarray(np.tile(g2[0], (3, 1)))
    z5, z3 = np.zeros(5, np.uint8), np.zeros(3, np.uint8)

    def create(idx, curve=0):
        hs = np.array([regs[i].handle for i in idx], dtype=np.uint64)
        h = ctypes.c_uint64(0)
        rc = L.zkm_groth16_pk_create(curve, p(hs), p(pts1), p(z5), p(pts2), p(z3), ctypes.byref(h))
        if rc == 0:
            assert L.zkm_groth16_pk_release(h.value) == 0
        return rc
    try:
        assert create([0, 1, 2, 3, 4]) == 0
        assert create([0, 1, 2, 3, 0]) == ERR_ARG           # b_g2 of group 1
        assert create([0, 1, 4, 3, 4]) == ERR_ARG           # a of group 2
        assert create([0, 1, 5, 3, 4]) == ERR_ARG           # a shorter than b_g1
        assert create([0, 6, 2, 3, 4]) == ERR_ARG           # a BN254 registration in a BLS12-381 key
        assert create([0, 1, 2, 3, 4], curve=7) == ERR_ARG  # unknown curve
    finally:
        for rg in regs:
            rg.release()
    handle = pk.handle
    pk.release()
    assert call(handle=handle) == ERR_HANDLE
    assert L.zkm_groth16_pk_release(handle) == ERR_HANDLE


# 7. placement: b_g2 registered on device index 1 of a process that owns two devices
def test_g2_query_on_another_device():
    import zkmember_b200 as z
    from zkmember_b200.groth16 import create_proof
    z.shutdown()
    try:
        L = z.load()
        z.init([0, 1] if L.zkm_device_count() >= 2 else [0, 0])
        assert z._lib.initialised_devices() == 2
        pk, args = _synthetic(0, 11, seed=31)
        try:
            got = create_proof(pk, **args)
            want = _old_create_proof(pk, **args)
        finally:
            pk.release()
        assert got.serialize() == want.serialize()
    finally:
        z.shutdown()
        z.init(0)
