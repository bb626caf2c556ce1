"""Host-side mirror of ark-ec 0.3.0's MSM interfaces.

    VariableBaseMSM.multi_scalar_mul(bases, scalars) -> affine point
    FixedBaseMSM.multi_scalar_mul(base, scalars)     -> n affine points s_i * base (the setup paths)

replaces `ark_ec::msm::VariableBaseMSM::multi_scalar_mul` (src/msm/variable_base.rs; pin
/root/reference/Cargo.lock:179-180) + `into_affine()`, the call ark-groth16's create_proof makes
five times per proof (reached from /root/reference/benches/groth16.rs:115) and KZG10::commit makes
per polynomial (benches/marlin.rs:202,311).  Same argument meaning as upstream: `bases` are
affine points with Montgomery coordinates, `scalars` are canonical BigInteger256 (`into_repr()`),
the sum runs over min(len(bases), len(scalars)) pairs, zero scalars and points at infinity are
legal, and the empty sum is the identity.  Arrays are numpy uint64 in arkworks' limb layout; the
computation happens on the GPU through the C ABI (include/zkm_b200.h) -- no CPU path exists.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np

from . import _lib

L64 = {_lib.CURVE_BLS12_381: 6, _lib.CURVE_BN254: 4, _lib.CURVE_BW6_761: 12}
FR_WORDS = _lib.FR_WORDS


def coord_words(curve: int, group: int) -> int:
    """u64 words per coordinate: Fq (G1) or Fq2 (G2); BW6-761's G2 is a curve over Fq as well."""
    if curve == _lib.CURVE_BW6_761:
        return L64[curve]
    return L64[curve] * (2 if group == 2 else 1)


def _curve_id(curve) -> int:
    if isinstance(curve, str):
        return _lib.CURVE_IDS[curve]
    return int(curve)


@dataclass
class AffinePoint:
    """GroupAffine{x, y, infinity}: `xy` holds x then y (each L64 words; G2: c0 then c1), Montgomery."""
    curve: int
    group: int
    xy: np.ndarray
    infinity: bool

    def to_bytes(self) -> bytes:
        return self.xy.tobytes() + bytes([1 if self.infinity else 0])

    def __eq__(self, other):
        return (isinstance(other, AffinePoint) and self.curve == other.curve and self.group == other.group
                and self.infinity == other.infinity and np.array_equal(self.xy, other.xy))


def _as_u64(a, cols: int, name: str) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint64)
    if a.size % cols:
        raise ValueError("%s: size %d is not a multiple of %d words" % (name, a.size, cols))
    return a.reshape(-1, cols)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None and a.size else ctypes.c_void_p(0)


class RegisteredBases:
    """Bases uploaded once to HBM (a proving-key query vector or the KZG powers), used by handle.
    The proving key is static across proofs (/root/reference/benches/groth16.rs:107-115)."""

    def __init__(self, curve, group: int, bases, infinity=None, *, precompute: bool = False, shard: bool = False,
                 device: int | None = None, _device_ptr=None, _n=None):
        """precompute: also store the window multiples (ZKM_REG_PRECOMPUTE); shard: split the bases over all
        initialised GPUs (ZKM_REG_SHARD); device: index of the initialised GPU that holds them (ZKM_REG_DEVICE)."""
        self.curve = _curve_id(curve)
        self.group = int(group)
        L = _lib.lib()
        W = coord_words(self.curve, self.group)
        h = ctypes.c_uint64(0)
        flags = (_lib.REG_PRECOMPUTE if precompute else 0) | (_lib.REG_SHARD if shard else 0)
        if device is not None:
            flags |= _lib.REG_DEVICE(device)
        if _device_ptr is not None:
            self.n = int(_n)
            _lib.check(L.zkm_bases_register_ex(self.curve, self.group, ctypes.c_void_p(_device_ptr),
                                               ctypes.c_void_p(0), self.n, flags, ctypes.byref(h)))
        else:
            b = _as_u64(bases, 2 * W, "bases")
            self.n = len(b)
            inf = None
            if infinity is not None:
                inf = np.ascontiguousarray(infinity, dtype=np.uint8)
                if len(inf) != self.n:
                    raise ValueError("infinity flags: expected %d, got %d" % (self.n, len(inf)))
            _lib.check(L.zkm_bases_register_ex(self.curve, self.group, _ptr(b), _ptr(inf), self.n, flags, ctypes.byref(h)))
        self.handle = h.value

    @classmethod
    def from_device(cls, curve, group: int, device_ptr: int, n: int, **kw) -> "RegisteredBases":
        return cls(curve, group, None, _device_ptr=device_ptr, _n=n, **kw)

    def release(self):
        if self.handle:
            _lib.check(_lib.lib().zkm_bases_release(self.handle))
            self.handle = 0

    def msm(self, scalars, offset: int = 0, n: int | None = None) -> AffinePoint:
        s = _as_u64(scalars, FR_WORDS[self.curve], "scalars")
        avail = self.n - offset
        n = min(len(s), avail) if n is None else n
        W = coord_words(self.curve, self.group)
        out = np.zeros(2 * W, dtype=np.uint64)
        oinf = np.zeros(1, dtype=np.uint8)
        _lib.check(_lib.lib().zkm_msm_registered(self.handle, offset, _ptr(s), n, _ptr(out), _ptr(oinf)))
        return AffinePoint(self.curve, self.group, out, bool(oinf[0]))

    def msm_device(self, d_scalars_ptr: int, n: int, d_out_ptr: int, offset: int = 0, stream: int = 0):
        """Device-resident variant: scalars and the (2W+1)-word result record stay in HBM."""
        _lib.check(_lib.lib().zkm_msm_registered_device(self.handle, offset, ctypes.c_void_p(d_scalars_ptr), n,
                                                        ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(stream)))


class VariableBaseMSM:
    """Namesake of ark_ec::msm::VariableBaseMSM."""

    @staticmethod
    def multi_scalar_mul(bases, scalars, *, curve="bls12_381", group: int = 1, infinity=None) -> AffinePoint:
        cid = _curve_id(curve)
        W = coord_words(cid, group)
        b = _as_u64(bases, 2 * W, "bases")
        s = _as_u64(scalars, FR_WORDS[cid], "scalars")
        n = min(len(b), len(s))          # upstream: size = min(bases.len(), scalars.len())
        inf = None
        if infinity is not None:
            inf = np.ascontiguousarray(infinity, dtype=np.uint8)
            if len(inf) < n:
                raise ValueError("infinity flags: expected at least %d, got %d" % (n, len(inf)))
        out = np.zeros(2 * W, dtype=np.uint64)
        oinf = np.zeros(1, dtype=np.uint8)
        L = _lib.lib()
        fn = L.zkm_msm_g1 if group == 1 else L.zkm_msm_g2
        _lib.check(fn(cid, _ptr(b), _ptr(inf), _ptr(s), n, _ptr(out), _ptr(oinf)))
        return AffinePoint(cid, group, out, bool(oinf[0]))


def _base_record(base, cid: int, group: int):
    """(xy words, infinity flag) of ONE affine base: an AffinePoint or its 2 W words."""
    W = coord_words(cid, group)
    if isinstance(base, AffinePoint):
        if base.curve != cid or base.group != group:
            raise ValueError("base is a point of curve %d group %d, not curve %d group %d" % (base.curve, base.group, cid, group))
        xy, inf = base.xy, base.infinity
    else:
        xy, inf = base, False
    xy = np.ascontiguousarray(xy, dtype=np.uint64)
    if xy.size != 2 * W:
        raise ValueError("base: expected %d words (one affine point), got %d" % (2 * W, xy.size))
    return xy.reshape(2 * W), 1 if inf else 0


class FixedBaseMSM:
    """Namesake of ark_ec::msm::FixedBaseMSM: get_window_table + multi_scalar_mul + batch_normalization_into_affine in
    one call (the window width is the library's choice)."""

    @staticmethod
    def multi_scalar_mul(base, scalars, curve="bls12_381", group: int = 1):
        """s_i * base for every Montgomery Fr element s_i of `scalars` ((n, S) uint64, as upstream's &[G::ScalarField]).
        Returns (xy (n, 2W) uint64 Montgomery affine, inf (n,) uint8).  An element >= r raises ZKM_ERR_SCALAR_RANGE."""
        cid = _curve_id(curve)
        if group not in (1, 2):
            raise ValueError("group must be 1 or 2, got %r" % (group,))
        W = coord_words(cid, group)
        xy_b, inf_b = _base_record(base, cid, group)
        s = _as_u64(scalars, FR_WORDS[cid], "scalars")
        n = len(s)
        out = np.zeros((n, 2 * W), dtype=np.uint64)
        oinf = np.zeros(n, dtype=np.uint8)
        _lib.check(_lib.lib().zkm_fixed_base_msm(cid, group, _ptr(xy_b), inf_b, _ptr(s), n, _ptr(out), _ptr(oinf)))
        return out, oinf

    @staticmethod
    def multi_scalar_mul_device(base, d_scalars_ptr: int, n: int, d_out_xy_ptr: int, d_out_inf_ptr: int, curve="bls12_381",
                                group: int = 1, stream: int = 0):
        """Device-resident variant: n Montgomery scalars and the n affine records + infinity bytes stay in HBM; enqueued on
        `stream` without a host wait.  Scalars are not range-checked here."""
        cid = _curve_id(curve)
        xy_b, inf_b = _base_record(base, cid, group)
        _lib.check(_lib.lib().zkm_fixed_base_msm_device(cid, group, _ptr(xy_b), inf_b, ctypes.c_void_p(d_scalars_ptr), n,
                                                        ctypes.c_void_p(d_out_xy_ptr), ctypes.c_void_p(d_out_inf_ptr),
                                                        ctypes.c_void_p(stream)))


def msm_window_bits(curve, group: int, n: int) -> int:
    return int(_lib.load().zkm_msm_window_bits(_curve_id(curve), group, n))


def msm_batch_device(items, stream: int = 0):
    """Concurrent MSMs over registered bases, device resident (the create_proof pattern).
    items: iterable of (RegisteredBases, d_scalars_ptr, n, d_out_ptr[, offset])."""
    items = list(items)
    k = len(items)
    handles = (ctypes.c_uint64 * k)(*[it[0].handle for it in items])
    offsets = (ctypes.c_size_t * k)(*[(it[4] if len(it) > 4 else 0) for it in items])
    scal = (ctypes.c_void_p * k)(*[it[1] for it in items])
    ns = (ctypes.c_size_t * k)(*[it[2] for it in items])
    outs = (ctypes.c_void_p * k)(*[it[3] for it in items])
    _lib.check(_lib.lib().zkm_msm_batch_registered_device(k, ctypes.cast(handles, ctypes.c_void_p), ctypes.cast(offsets, ctypes.c_void_p),
                                                          ctypes.cast(scal, ctypes.c_void_p), ctypes.cast(ns, ctypes.c_void_p),
                                                          ctypes.cast(outs, ctypes.c_void_p), ctypes.c_void_p(stream)))
