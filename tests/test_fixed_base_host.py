"""Fixed-base batch scalar multiplication on the CPU side: the two C entry points exist and refuse to run without an
initialised GPU (no CPU fallback), the Python wrappers reject malformed shapes before any device work, the Rust patch
routes without modulus constants of its own, and the C++ wrapper compiles against the header."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_symbols_exported():
    from zkmember_b200 import _lib
    L = _lib.load()
    for name in ("zkm_fixed_base_msm", "zkm_fixed_base_msm_device"):
        assert name in _lib.SYMBOLS
        assert hasattr(L, name)


def test_not_initialised_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from zkmember_b200 import _lib
    L = _lib.load()
    base = np.zeros(12, dtype=np.uint64)
    s = np.zeros((4, 4), dtype=np.uint64)
    out = np.zeros((4, 12), dtype=np.uint64)
    inf = np.zeros(4, dtype=np.uint8)
    p = lambda a: ctypes.c_void_p(a.ctypes.data)
    assert L.zkm_fixed_base_msm(0, 1, p(base), 0, p(s), 4, p(out), p(inf)) == -3        # ZKM_ERR_NOT_INIT
    assert L.zkm_fixed_base_msm(0, 1, p(base), 0, p(s), 0, p(out), p(inf)) == -3
    assert L.zkm_fixed_base_msm_device(0, 1, p(base), 0, ctypes.c_void_p(0), 0, ctypes.c_void_p(0), ctypes.c_void_p(0),
                                       ctypes.c_void_p(0)) == -3
    # argument errors are reported before the device is needed
    assert L.zkm_fixed_base_msm(7, 1, p(base), 0, p(s), 4, p(out), p(inf)) == -1         # unknown curve
    assert L.zkm_fixed_base_msm(0, 3, p(base), 0, p(s), 4, p(out), p(inf)) == -1         # unknown group
    assert L.zkm_fixed_base_msm(0, 1, p(base), 0, ctypes.c_void_p(0), 4, p(out), p(inf)) == -1   # null with n > 0


def test_python_wrappers_reject_malformed_shapes():
    from zkmember_b200 import AffinePoint, FixedBaseMSM
    from zkmember_b200.kzg import KZG10
    good = np.zeros(12, dtype=np.uint64)
    with pytest.raises(ValueError):
        FixedBaseMSM.multi_scalar_mul(np.zeros(11, dtype=np.uint64), np.zeros((2, 4), dtype=np.uint64))   # base size
    with pytest.raises(ValueError):
        FixedBaseMSM.multi_scalar_mul(good, np.zeros(7, dtype=np.uint64))                                  # scalar words
    with pytest.raises(ValueError):
        FixedBaseMSM.multi_scalar_mul(good, np.zeros((2, 4), dtype=np.uint64), group=3)
    with pytest.raises(ValueError):                                                                        # G2 point as G1 base
        FixedBaseMSM.multi_scalar_mul(AffinePoint(0, 2, np.zeros(24, dtype=np.uint64), False), np.zeros((2, 4), np.uint64))
    with pytest.raises(ValueError):
        KZG10.setup("bls12_381", 0, np.zeros(4, dtype=np.uint64), good, good)                             # DegreeIsZero
    with pytest.raises(ValueError):
        KZG10.setup("bls12_381", 4, np.full(4, 0xFFFFFFFFFFFFFFFF, dtype=np.uint64), good, good)           # beta >= r


def test_rust_fixed_base_patch_names_no_modulus_constants():
    s = open(os.path.join(ROOT, "rust", "patches", "ark_ec_fixed_base.rs")).read()
    assert not re.findall(r"const \w+: \[u64; \d+\]", s)
    assert "zkm_fixed_base_msm" in s and "gpu_group" in s


def test_cpp_wrapper_compiles_against_the_header(tmp_path):
    src = tmp_path / "fb.cpp"
    src.write_text(
        '#include "zkm_b200.hpp"\n'
        "int main() {\n"
        "    zkm::G1Affine<zkm::Bls12_381> g{};\n"
        "    std::vector<zkm::Bls12_381::Fr> s(3);\n"
        "    try { auto v = zkm::FixedBaseMSM::multi_scalar_mul(g, s); return (int)v.size(); }\n"
        "    catch (const zkm::Error&) { return 0; }\n"
        "}\n")
    exe = tmp_path / "fb"
    lib_dir = os.path.join(ROOT, "zkmember_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o", str(exe),
                           str(src), "-L" + lib_dir, "-lzkm_b200", "-L/usr/local/cuda/lib64", "-lcudart",
                           "-Wl,-rpath," + lib_dir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    import torch
    if not torch.cuda.is_available():
        assert subprocess.run([str(exe)]).returncode == 0     # zkm::Error (not initialised): no CPU fallback
