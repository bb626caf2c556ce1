"""The device headers (zkm_field.cuh / zkm_curve.cuh) compiled for the HOST with -DZKM_HOST_EMU:
the very limb schedules the kernels use (two-accumulator CIOS on 32-bit limbs, XYZZ formulas with
their exceptional cases) run on the CPU and are compared with exact big-int arithmetic.
Test vehicle only -- nothing in the shipped library is built with ZKM_HOST_EMU."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.py import exact
from oracle.py.params import BLS12_381, BN254, BW6_761

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_emu", "emu_field.cpp")
OUT = os.path.join(HERE, "host_emu", "_build", "libzkm_emu.so")
CSRC = os.path.join(os.path.dirname(HERE), "zkmember_b200", "csrc")


@pytest.fixture(scope="module")
def emu():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("zkm_arith.cuh", "zkm_field.cuh", "zkm_curve.cuh", "zkm_constants.cuh",
                                                     "zkm_fpmul_u.cuh")]
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-DZKM_HOST_EMU", "-x", "c++", "-shared", "-fPIC", "-o", OUT, SRC])
    return ctypes.CDLL(OUT)


FIELDS = {0: BLS12_381.fq, 1: BLS12_381.fr, 2: BN254.fq, 3: BN254.fr, 4: BW6_761.fq, 5: BW6_761.fr}


def _limbs32(v, n):
    return [(v >> (32 * i)) & 0xFFFFFFFF for i in range(n)]


def _p(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))


@pytest.mark.parametrize("fid", [0, 1, 2, 3, 4, 5])
def test_fp_ops(emu, fid):
    fp = FIELDS[fid]
    p, n = fp.modulus, fp.limbs32
    rng = np.random.default_rng(fid)
    vals = [0, 1, 2, p - 1, p - 2, (p - 1) // 2] + [int.from_bytes(rng.bytes(104), "little") % p for _ in range(60)]
    A = np.array([_limbs32(fp.to_mont(v), n) for v in vals], dtype=np.uint32)
    B = np.array([_limbs32(fp.to_mont(v), n) for v in reversed(vals)], dtype=np.uint32)
    out = np.zeros_like(A)
    ops = {0: lambda a, b: a * b % p, 1: lambda a, b: (a + b) % p, 2: lambda a, b: (a - b) % p, 3: lambda a, b: (-a) % p,
           4: lambda a, b: a * a % p, 6: lambda a, b: 2 * a % p, 8: lambda a, b: a * b % p}
    for op, f in ops.items():
        assert emu.emu_fp_op(fid, op, _p(A), _p(B), _p(out), len(vals)) == 0
        for i, (a, b) in enumerate(zip(vals, reversed(vals))):
            got = sum(int(out[i, j]) << (32 * j) for j in range(n))
            assert got == fp.to_mont(f(a, b)), (fid, op, i)
    nz = [v for v in vals if v][:10]
    A2 = np.array([_limbs32(fp.to_mont(v), n) for v in nz], dtype=np.uint32)
    out2 = np.zeros_like(A2)
    assert emu.emu_fp_op(fid, 5, _p(A2), _p(A2), _p(out2), len(nz)) == 0
    for i, a in enumerate(nz):
        assert sum(int(out2[i, j]) << (32 * j) for j in range(n)) == fp.to_mont(pow(a, -1, p))
    # binary-EGCD inverse == Fermat inverse, incl. 1, p-1, small values and inv(0) = 0
    edge = [1, 2, 3, p - 1, p - 2, (p + 1) // 2] + [int.from_bytes(rng.bytes(104), "little") % p for _ in range(30)]
    A3 = np.array([_limbs32(fp.to_mont(v), n) for v in edge], dtype=np.uint32)
    o5, o7 = np.zeros_like(A3), np.zeros_like(A3)
    assert emu.emu_fp_op(fid, 5, _p(A3), _p(A3), _p(o5), len(edge)) == 0
    assert emu.emu_fp_op(fid, 7, _p(A3), _p(A3), _p(o7), len(edge)) == 0
    assert np.array_equal(o5, o7)
    for i, a in enumerate(edge):
        assert sum(int(o5[i, j]) << (32 * j) for j in range(n)) == fp.to_mont(pow(a, -1, p))
    Z = np.zeros((1, n), dtype=np.uint32)
    oz = np.ones_like(Z)
    assert emu.emu_fp_op(fid, 5, _p(Z), _p(Z), _p(oz), 1) == 0 and not oz.any()


@pytest.mark.parametrize("fid", [0, 1, 2, 3, 4, 5])
def test_fp_mul_unsaturated_extreme_limbs(emu, fid):
    """The carry-free column product (zkm_fpmul_u.cuh) on RAW representatives chosen to maximise the column sums:
    p - 1, all-ones below the modulus width, every r-bit limb saturated, sparse patterns, and 2000 random pairs;
    the unsaturated product and squaring and the saturated CIOS (ops 0 / 4) must all equal x * y * R^-1 mod p."""
    fp = FIELDS[fid]
    p, n = fp.modulus, fp.limbs32
    Rinv = pow(1 << (32 * n), -1, p)
    rng = np.random.default_rng(100 + fid)
    top = (1 << (p.bit_length() - 1)) - 1
    raw = [0, 1, p - 1, p - 2, top, top - 1, (1 << (p.bit_length() - 1)), p >> 1, (p - 1) ^ 0x5555555555555555]
    for r in (29, 30):
        m = 0
        for i in range(0, p.bit_length() + r, r):
            m |= ((1 << r) - 1) << i
        raw += [m % p, (m >> 1) % p, (m & top)]
    raw = [v % p for v in raw]
    raw += [int.from_bytes(rng.bytes(104), "little") % p for _ in range(2000)]
    A = np.array([_limbs32(v, n) for v in raw], dtype=np.uint32)
    B = np.array([_limbs32(v, n) for v in raw[::-1]], dtype=np.uint32)
    for op in (0, 8, 4, 9):
        out = np.zeros_like(A)
        assert emu.emu_fp_op(fid, op, _p(A), _p(B), _p(out), len(raw)) == 0
        for i, (a, b) in enumerate(zip(raw, raw[::-1])):
            want = (a * (a if op in (4, 9) else b) * Rinv) % p
            assert sum(int(out[i, j]) << (32 * j) for j in range(n)) == want, (fid, op, i)
    # every ordered pair of the extreme values
    ext = raw[:15]
    pa = [a for a in ext for _ in ext]
    pb = [b for _ in ext for b in ext]
    A = np.array([_limbs32(v, n) for v in pa], dtype=np.uint32)
    B = np.array([_limbs32(v, n) for v in pb], dtype=np.uint32)
    out = np.zeros_like(A)
    assert emu.emu_fp_op(fid, 8, _p(A), _p(B), _p(out), len(pa)) == 0
    for i, (a, b) in enumerate(zip(pa, pb)):
        assert sum(int(out[i, j]) << (32 * j) for j in range(n)) == (a * b * Rinv) % p, (fid, i)


@pytest.mark.parametrize("curve", [BLS12_381, BN254, BW6_761], ids=lambda c: c.name)
@pytest.mark.parametrize("g", [1, 2])
def test_xyzz_group_law_with_exceptional_cases(emu, curve, g):
    """madd / add / dbl / to_affine incl. identity operands, P + P and P + (-P)."""
    G = exact.Group(curve, g)
    fq = curve.fq
    deg = curve.coord_degree(g)
    n = fq.limbs32 * deg
    pts = G.progression(3, 5, 6)

    def coord(c):
        if deg == 1:
            return _limbs32(fq.to_mont(c), fq.limbs32)
        return _limbs32(fq.to_mont(c[0]), fq.limbs32) + _limbs32(fq.to_mont(c[1]), fq.limbs32)

    one = 1 if deg == 1 else (1, 0)
    zero = 0 if deg == 1 else (0, 0)

    def xyzz(P):
        if P is None:
            return coord(zero) * 4
        return coord(P[0]) + coord(P[1]) + coord(one) + coord(one)

    def aff(P):
        return coord(P[0]) + coord(P[1])

    cases = [(pts[0], pts[1]), (None, pts[2]), (pts[3], pts[3]), (pts[4], G.neg(pts[4])), (pts[5], pts[0])]
    Pbuf = np.array([xyzz(a) for a, _ in cases], dtype=np.uint32)
    Qaff = np.array([aff(b) for _, b in cases], dtype=np.uint32)
    Qx = np.array([xyzz(b) for _, b in cases], dtype=np.uint32)
    out = np.zeros_like(Pbuf)
    aout = np.zeros((len(cases), 2 * n), dtype=np.uint32)
    inf = np.zeros(len(cases), dtype=np.uint8)
    cid = curve.curve_id

    def check(res, want_list):
        assert emu.emu_curve_op(cid, g, 3, _p(res), _p(res), _p(aout), inf.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), len(cases)) == 0
        for i, want in enumerate(want_list):
            if want is None:
                assert inf[i] == 1, i
            else:
                assert inf[i] == 0, i
                assert list(aout[i]) == aff(want), i

    u8 = inf.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
    assert emu.emu_curve_op(cid, g, 0, _p(Pbuf), _p(Qaff), _p(out), u8, len(cases)) == 0   # madd
    check(out.copy(), [G.add(a, b) for a, b in cases])
    assert emu.emu_curve_op(cid, g, 1, _p(Pbuf), _p(Qx), _p(out), u8, len(cases)) == 0     # add
    check(out.copy(), [G.add(a, b) for a, b in cases])
    assert emu.emu_curve_op(cid, g, 2, _p(Pbuf), _p(Qx), _p(out), u8, len(cases)) == 0     # dbl
    check(out.copy(), [G.double(a) for a, _ in cases])


def test_constants_header_is_up_to_date():
    root = os.path.dirname(HERE)
    assert subprocess.call([sys.executable, os.path.join(root, "tools", "gen_constants.py"), "--check"]) == 0
