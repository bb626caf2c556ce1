"""MarlinKZG10 (degree-bounded commitments, batch opening) on the CPU side: the exact restatement in
oracle/py/marlin_pc_exact.py on a genuine BLS12-381 SRS with known beta passes MarlinKZG10's pairing check and the check
rejects tampered proofs; the three C entry points exist and refuse to run without an initialised GPU; the C++ wrapper
compiles and links; the Rust patch routes by the fields' moduli through the sys crate."""
import ctypes
import os
import random
import re
import subprocess

import numpy as np
import pytest

from oracle.py import exact, marlin_pc_exact as mx
from oracle.py.params import BLS12_381

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("zkm_kzg_commit_many", "zkm_kzg_open_batch", "zkm_kzg_open_batch_device")
D = 64
BOUNDS = (30, 62)


@pytest.fixture(scope="module")
def setup():
    curve = BLS12_381
    r = curve.fr.modulus
    rng = random.Random(2026)
    beta, gamma = rng.randrange(2, r), rng.randrange(2, r)
    G1, G2 = exact.Group(curve, 1), exact.Group(curve, 2)
    srs = mx.Srs(curve, [G1.mul(G1.gen, pow(beta, i, r)) for i in range(D + 1)],
                 [G1.mul(G1.gen, gamma * pow(beta, i, r) % r) for i in range(D + 2)])
    rnd = lambda n: [rng.randrange(r) for _ in range(n)]
    polys = {   # label -> (coeffs, bound, rand, shifted_rand); hiding bound 1
        "a": (rnd(41), None, rnd(2), None),
        "b": (rnd(31), 30, rnd(2), rnd(2)),
        "c": (rnd(51), 62, rnd(2), rnd(2)),
    }
    comms = {lab: mx.commit(srs, *p) for lab, p in polys.items()}
    zb, zg = rng.randrange(r), rng.randrange(r)
    query_set = [("a", ("beta", zb)), ("c", ("beta", zb)), ("a", ("gamma", zg)), ("b", ("gamma", zg)), ("c", ("gamma", zg))]
    xi = rng.randrange(r)
    proofs, evals = mx.batch_open(srs, polys, query_set, xi)
    bounds = {lab: p[1] for lab, p in polys.items()}
    return dict(srs=srs, polys=polys, h=G2.gen, beta_h=G2.mul(G2.gen, beta), comms=comms, bounds=bounds, query_set=query_set,
                evals=evals, proofs=proofs, xi=xi)


def _check(s, **over):
    a = dict(s, **over)
    return mx.batch_check(a["srs"], a["h"], a["beta_h"], a["comms"], a["bounds"], a["query_set"], a["evals"], a["proofs"], a["xi"])


def test_restatement_passes_the_pairing_check(setup):
    assert _check(setup)


def test_pairing_check_rejects_a_wrong_evaluation(setup):
    r = BLS12_381.fr.modulus
    evals = dict(setup["evals"])
    evals[("b", "gamma")] = (evals[("b", "gamma")] + 1) % r
    assert not _check(setup, evals=evals)


def test_pairing_check_rejects_the_unshifted_commitment_in_place_of_the_shifted_one(setup):
    comms = dict(setup["comms"])
    comms["c"] = (comms["c"][0], comms["c"][0])
    assert not _check(setup, comms=comms)


def test_pairing_check_rejects_a_proof_of_the_other_point(setup):
    p = setup["proofs"]
    assert not _check(setup, proofs={"beta": p["gamma"], "gamma": p["gamma"]})


def test_open_combinations_of_single_polynomials_is_batch_open(setup):
    lcs = {lab: [(1, lab)] for lab in ("a", "b", "c")}
    proofs, evals = mx.open_combinations(setup["srs"], lcs, setup["polys"], setup["query_set"], setup["xi"])
    assert proofs == setup["proofs"] and evals == setup["evals"]


def test_bounded_polynomial_must_be_alone_in_its_combination_one_included():
    """upstream counts LCTerm::One in `lc.len()`: {1 * g, c * One} with a bounded g is EquationHasDegreeBounds."""
    from types import SimpleNamespace
    from zkmember_b200.marlin_pc import CommitterKey, LabeledPolynomial, LinearCombination, MarlinKZG10
    ck = CommitterKey(SimpleNamespace(curve=0, n=D + 1), None, D, list(BOUNDS))
    g = LabeledPolynomial("g", np.ones((31, 4), np.uint64), 30)
    with pytest.raises(ValueError):
        MarlinKZG10.open_combinations(ck, [LinearCombination("lc", [(1, "g"), (3, None)])], [g], [("lc", ("beta", 5))], 7)
    with pytest.raises(ValueError):
        MarlinKZG10.open_combinations(ck, [LinearCombination("lc", [(2, "g")])], [g], [("lc", ("beta", 5))], 7)


def test_symbols_exported():
    from zkmember_b200 import _lib
    L = _lib.load()
    for name in NAMES:
        assert name in _lib.SYMBOLS
        assert hasattr(L, name)


def test_not_initialised_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from zkmember_b200 import _lib
    L = _lib.load()
    p = lambda a: ctypes.c_void_p(a.ctypes.data)
    v = np.zeros((8, 4), np.uint64)
    ptrs = (ctypes.c_void_p * 1)(v.ctypes.data)
    n = (ctypes.c_size_t * 1)(8)
    i0 = (ctypes.c_int32 * 1)(0)
    im = (ctypes.c_int32 * 1)(-1)
    out = np.zeros(16, np.uint64)
    inf = np.zeros(2, np.uint8)
    assert L.zkm_kzg_commit_many(1, 2, 1, ptrs, n, n, None, None, p(out), p(inf)) == -3           # ZKM_ERR_NOT_INIT
    assert L.zkm_kzg_open_batch(1, 2, 1, ptrs, n, 0, None, None, 1, p(v), 1, i0, i0, im, n, p(v), p(out), p(inf), p(out),
                                p(out)) == -3
    assert L.zkm_kzg_open_batch_device(1, 2, 1, ptrs, n, 0, None, None, 1, p(v), 1, i0, i0, im, n, p(v), p(out), p(out), p(out),
                                       None) == -3


def test_cpp_marlin_pc_source_compiles_and_links(tmp_path):
    exe = tmp_path / "marlin_pc"
    lib_dir = os.path.join(ROOT, "zkmember_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o", str(exe),
                           os.path.join(ROOT, "tests", "cpp", "test_marlin_pc.cpp"), "-L" + lib_dir, "-lzkm_b200",
                           "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath," + lib_dir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    import torch
    if not torch.cuda.is_available():
        assert subprocess.run([str(exe)]).returncode == 0     # zkm::Error (not initialised): no CPU fallback


def test_rust_marlin_pc_patch_routes_through_gpu_group_with_one_powers_registration():
    s = open(os.path.join(ROOT, "rust", "patches", "ark_poly_commit_marlin_pc.rs")).read()
    assert not re.findall(r"const \w+: \[u64; \d+\]", s)           # routes by the variable-base patch's moduli table
    assert "use ark_ec::msm::{gpu_group, registered, GroupId};" in s
    assert s.count("gpu_group::<E::G1Affine>()") == 2 and "upstream::commit" in s
    assert "upstream::open_combinations_individual_opening_challenges" in s
    for name in ("zkm_kzg_commit_many", "zkm_kzg_open_batch", "zkm_bases_register_ex"):
        assert "sys::" + name in s
    # ck.powers and ck.shifted_powers become ONE registration of powers_of_g[0..=max_degree], shifts are absolute
    assert "ck.shifted_powers" in s and "ck.max_degree + 1" in s and "shifts.push(max_degree - d)" in s
    assert "registered(g1, &ck.powers_of_gamma_g)" in s
    # only accessors the sibling patches define
    v = open(os.path.join(ROOT, "rust", "patches", "ark_ec_variable_base.rs")).read()
    f = open(os.path.join(ROOT, "rust", "patches", "ark_ff_raw_limbs.rs")).read()
    for m in set(re.findall(r"\.(zkm_\w+)\(", s)) | set(re.findall(r"::(zkm_\w+)\(", s)) - {n for n in re.findall(r"sys::(zkm_\w+)", s)}:
        assert ("fn %s(" % m) in v + f, m
    assert "fn commit<" in s and "fn open_combinations_individual_opening_challenges<" in s
    assert "num_polys = lc.len()" in s                               # upstream counts LCTerm::One in the bound rule
    assert "zkmember-gpu-sys = { path =" in s
