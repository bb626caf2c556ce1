"""Groth16 create_proof as one call, on the CPU side: the four C entry points exist and refuse to run without an
initialised GPU (no CPU fallback), the C++ layer's Groth16ProvingKey / create_proof compiles and links, and the Rust
prover patch routes through gpu_group with extern items that match the header."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("zkm_groth16_pk_create", "zkm_groth16_pk_release", "zkm_groth16_prove", "zkm_groth16_prove_device")


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
    handles = np.arange(1, 6, dtype=np.uint64)
    g1, g2 = np.zeros(5 * 12, np.uint64), np.zeros(3 * 24, np.uint64)
    i1, i2 = np.zeros(5, np.uint8), np.zeros(3, np.uint8)
    h = ctypes.c_uint64(0)
    assert L.zkm_groth16_pk_create(0, p(handles), p(g1), p(i1), p(g2), p(i2), ctypes.byref(h)) == -3     # ZKM_ERR_NOT_INIT
    assert L.zkm_groth16_pk_release(1) == -3
    v = np.zeros((16, 4), np.uint64)
    one = np.array([1, 0, 0, 0], np.uint64)
    out = np.zeros(24, np.uint64)
    inf = np.zeros(3, np.uint8)
    assert L.zkm_groth16_prove(1, p(v), p(v), p(v), 4, p(v), 2, 3, p(one), p(one), p(out), p(inf), p(out), p(inf), p(out),
                               p(inf)) == -3
    assert L.zkm_groth16_prove_device(1, p(v), p(v), p(v), 4, p(v), 2, 3, p(one), p(one), p(out), ctypes.c_void_p(0)) == -3


def test_cpp_groth16_source_compiles_and_links(tmp_path):
    exe = tmp_path / "g16"
    lib_dir = os.path.join(ROOT, "zkmember_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o", str(exe),
                           os.path.join(ROOT, "tests", "cpp", "test_groth16_prove.cpp"), "-L" + lib_dir, "-lzkm_b200",
                           "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath," + lib_dir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    import torch
    if not torch.cuda.is_available():
        assert subprocess.run([str(exe)]).returncode == 0     # zkm::Error (not initialised): no CPU fallback


def test_rust_prover_patch_routes_through_gpu_group():
    s = open(os.path.join(ROOT, "rust", "patches", "ark_groth16_prover.rs")).read()
    assert not re.findall(r"const \w+: \[u64; \d+\]", s)           # routes by the variable-base patch's table
    assert "gpu_group::<E::G1Affine>()" in s and "upstream::create_proof" in s
    for name in ("zkm_groth16_prove", "zkm_groth16_pk_create", "zkm_groth16_pk_release"):
        assert "sys::" + name in s
    lib = open(os.path.join(ROOT, "rust", "zkmember-gpu-sys", "src", "lib.rs")).read()
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "zkm_b200.h")).read(), flags=re.S)
    for name in NAMES:
        rs = re.search(r"pub fn %s\s*\((.*?)\)\s*->\s*i32;" % name, lib, re.S)
        c = re.search(r"\b%s\s*\(([^;]*?)\)\s*;" % name, header, re.S)
        assert rs and c, name
        rs_types = [p.split(":")[1].strip() for p in rs.group(1).split(",") if p.strip()]
        c_types = [" ".join(p.split()[:-1]) for p in c.group(1).split(",") if p.strip()]
        assert len(rs_types) == len(c_types), name
        for rt, ct in zip(rs_types, c_types):          # pointers stay pointers, of the same mutability and width
            assert rt.startswith("*") == ct.endswith("*"), (name, rt, ct)
            if rt.startswith("*"):
                assert ("const" in rt) == ct.startswith("const"), (name, rt, ct)


def test_rust_prover_patch_defines_the_witness_map_split():
    s = open(os.path.join(ROOT, "rust", "patches", "ark_groth16_prover.rs")).read()
    # the first half of witness_map is spelled out as an edit of src/r1cs_to_qap.rs, and witness_map calls it
    assert re.search(r"//\s+pub fn evaluation_vectors<F: PrimeField, D: EvaluationDomain<F>>\(", s)
    assert re.search(r"//.*Self::evaluation_vectors::<F, D>\(prover\)", s)
    assert "R1CStoQAP::evaluation_vectors::<E::Fr, GeneralEvaluationDomain<E::Fr>>(cs.clone())" in s
    # ark-ec re-exports the variable-base module's public items at ark_ec::msm (its module is private)
    assert "use ark_ec::msm::{gpu_group, registered, GroupId};" in s
    assert "zkmember-gpu-sys = { path =" in s
    v = open(os.path.join(ROOT, "rust", "patches", "ark_ec_variable_base.rs")).read()
    for item in ("pub struct GroupId", "pub fn gpu_group<", "pub fn registered<"):
        assert item in v
