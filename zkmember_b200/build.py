"""Build recipe for libzkm_b200.so (hand-written CUDA for sm_100a + the C ABI of include/zkm_b200.h).

nvcc cross-compiles here without a GPU; the .so is built IN-TREE (zkmember_b200/lib/) so that it
travels to the GPU box with the repo snapshot.  Translation units are compiled in parallel and
cached by a hash of their sources + flags (build/*.o, git-ignored).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ_DIR = os.path.join(ROOT, "build", "obj")
LIB_DIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIB_DIR, "libzkm_b200.so")

UNITS = [   # the slowest units first: with fewer cores than units they must start right away
    "zkm_msm_bw6.cu",
    "zkm_msm_g2_bls.cu",
    "zkm_msm_bw6_pair.cu",
    "zkm_fixed_base_bw6.cu",
    "zkm_fixed_base_bls.cu",
    "zkm_api.cu",
    "zkm_ntt_bls.cu",
    "zkm_ntt_bn.cu",
    "zkm_msm.cu",
    "zkm_msm_g1_bls.cu",
    "zkm_msm_g1_bn.cu",
    "zkm_msm_g2_bn.cu",
    "zkm_ntt_bw6.cu",
    "zkm_fixed_base_bn.cu",
    "zkm_groth16_bw6.cu",
    "zkm_groth16_bls.cu",
    "zkm_groth16_bn.cu",
    "zkm_kzg_bls.cu",
    "zkm_kzg_bw6.cu",
    "zkm_kzg_bn.cu",
]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


BASE_HEADERS = ["zkm_common.cuh", "zkm_curve.cuh", "zkm_field.cuh", "zkm_fpmul_u.cuh", "zkm_arith.cuh", "zkm_constants.cuh"]
UNIT_HEADERS = {
    "zkm_api.cu": ["zkm_groth16_ops.cuh", "zkm_kzg_ops.cuh"],
    "zkm_ntt_bls.cu": ["zkm_ntt.cuh"],
    "zkm_ntt_bn.cu": ["zkm_ntt.cuh"],
    "zkm_msm.cu": ["zkm_msm.cuh"],
    "zkm_msm_g1_bls.cu": ["zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_msm_g2_bls.cu": ["zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_msm_g1_bn.cu": ["zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_msm_g2_bn.cu": ["zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_ntt_bw6.cu": ["zkm_ntt.cuh"],
    "zkm_msm_bw6.cu": ["zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_msm_bw6_pair.cu": ["zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_fixed_base_bls.cu": ["zkm_fixed_base.cuh", "zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_fixed_base_bn.cu": ["zkm_fixed_base.cuh", "zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_fixed_base_bw6.cu": ["zkm_fixed_base.cuh", "zkm_msm.cuh", "zkm_msm_curve.cuh", "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_groth16_bls.cu": ["zkm_groth16.cuh", "zkm_groth16_ops.cuh", "zkm_fixed_base.cuh", "zkm_msm.cuh", "zkm_msm_curve.cuh",
                           "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_groth16_bn.cu": ["zkm_groth16.cuh", "zkm_groth16_ops.cuh", "zkm_fixed_base.cuh", "zkm_msm.cuh", "zkm_msm_curve.cuh",
                          "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_groth16_bw6.cu": ["zkm_groth16.cuh", "zkm_groth16_ops.cuh", "zkm_fixed_base.cuh", "zkm_msm.cuh", "zkm_msm_curve.cuh",
                           "zkm_msm_affine.cuh", "zkm_msm_quad.cuh"],
    "zkm_kzg_bls.cu": ["zkm_kzg.cuh", "zkm_kzg_ops.cuh"],
    "zkm_kzg_bn.cu": ["zkm_kzg.cuh", "zkm_kzg_ops.cuh"],
    "zkm_kzg_bw6.cu": ["zkm_kzg.cuh", "zkm_kzg_ops.cuh"],
}


def _headers_digest(unit: str) -> bytes:
    """Hash of exactly the headers `unit` includes (so touching one kernel family does not rebuild all)."""
    h = hashlib.sha256()
    paths = [os.path.join(ROOT, "include", "zkm_b200.h")]
    paths += [os.path.join(CSRC, n) for n in BASE_HEADERS + UNIT_HEADERS[unit]]
    for path in paths:
        h.update(os.path.basename(path).encode())
        h.update(open(path, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.digest()


def _compile(unit: str, verbose: bool) -> str:
    src = os.path.join(CSRC, unit)
    hdr = _headers_digest(unit)
    key = hashlib.sha256(hdr + open(src, "rb").read()).hexdigest()[:16]
    obj = os.path.join(OBJ_DIR, unit.replace(".cu", "") + "." + key + ".o")
    if os.path.exists(obj):
        return obj
    for old in os.listdir(OBJ_DIR):
        if old.startswith(unit.replace(".cu", "") + "."):
            os.remove(os.path.join(OBJ_DIR, old))
    cmd = [_nvcc()] + NVCC_FLAGS + ["-c", src, "-o", obj + ".tmp"]
    if verbose:
        print("[zkm build]", " ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    os.replace(obj + ".tmp", obj)
    return obj


def build(verbose: bool = True, jobs: int | None = None) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    jobs = jobs or min(len(UNITS), os.cpu_count() or 4)
    with ThreadPoolExecutor(max_workers=jobs) as ex:
        objs = list(ex.map(lambda u: _compile(u, verbose), UNITS))
    stamp = hashlib.sha256("".join(objs).encode()).hexdigest()
    stamp_file = LIB + ".stamp"
    if os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-lcudart"]
    if verbose:
        print("[zkm build]", " ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    open(stamp_file, "w").write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(verbose=True))
