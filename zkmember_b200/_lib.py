"""ctypes binding of libzkm_b200.so -- the C ABI declared in include/zkm_b200.h.

The library is hand-written CUDA for sm_100a; this module only loads it and turns error codes
into exceptions.  There is NO CPU fallback: if the shared object is missing, or no B200 is
visible, every compute call raises.
"""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libzkm_b200.so")

CURVE_BLS12_381 = 0
CURVE_BN254 = 1
CURVE_BW6_761 = 2
CURVE_IDS = {"bls12_381": CURVE_BLS12_381, "bn254": CURVE_BN254, "bw6_761": CURVE_BW6_761}
# u64 words of an Fr element / canonical scalar (BigInteger256; BigInteger384 for BW6-761)
FR_WORDS = {CURVE_BLS12_381: 4, CURVE_BN254: 4, CURVE_BW6_761: 6}

ERR_NAMES = {
    -1: "ZKM_ERR_ARG", -2: "ZKM_ERR_CUDA", -3: "ZKM_ERR_NOT_INIT", -4: "ZKM_ERR_DOMAIN",
    -5: "ZKM_ERR_SCALAR_RANGE", -6: "ZKM_ERR_HANDLE", -7: "ZKM_ERR_OOM",
}

# every symbol include/zkm_b200.h declares (tests check that the .so exports each one)
SYMBOLS = [
    "zkm_init", "zkm_shutdown", "zkm_last_error", "zkm_device_count", "zkm_version",
    "zkm_msm_g1", "zkm_msm_g2", "zkm_bases_register", "zkm_bases_release", "zkm_msm_registered",
    "zkm_ntt", "zkm_domain_constants", "zkm_ntt_device", "zkm_msm_registered_device",
    "zkm_bases_register_device", "zkm_points_sum_device", "zkm_set_option", "zkm_launch_count",
    "zkm_msm_window_bits", "zkm_testgen_progression_device", "zkm_profile_last_msm", "zkm_witness_map", "zkm_witness_map_device", "zkm_fr_into_repr_device", "zkm_kzg_commit", "zkm_msm_batch_registered_device",
    "zkm_init_mask", "zkm_init_devices", "zkm_initialised_devices", "zkm_bases_register_ex", "zkm_kzg_commit_batch",
    "zkm_kzg_commit_hiding", "zkm_kzg_open", "zkm_profile_last_msm_counts", "zkm_msm_cache_clear", "zkm_msm_cache_stats",
    "zkm_fixed_base_msm", "zkm_fixed_base_msm_device",
    "zkm_groth16_pk_create", "zkm_groth16_pk_release", "zkm_groth16_prove", "zkm_groth16_prove_device",
    "zkm_kzg_commit_many", "zkm_kzg_open_batch", "zkm_kzg_open_batch_device",
]

# zkm_bases_register_ex flags (include/zkm_b200.h)
REG_PRECOMPUTE = 1
REG_SHARD = 2


def REG_DEVICE(i: int) -> int:
    return (int(i) + 1) << 8



class ZkmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("%s (%d): %s" % (ERR_NAMES.get(code, "ZKM_ERR"), code, msg))
        self.code = code


class DomainError(ZkmError, ValueError):
    """log_n exceeds the two-adicity of Fr (upstream: Radix2EvaluationDomain::new returns None)."""


_lib = None
_inited_device = None


def load():
    """Load the shared library (no CUDA call yet).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "zkmember_b200: %s is missing -- build it with `python -m zkmember_b200.build` "
            "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    u64p, u8p, vp = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p
    i32, u32, sz, u64 = ctypes.c_int32, ctypes.c_uint32, ctypes.c_size_t, ctypes.c_uint64
    L.zkm_init.argtypes = [i32]
    L.zkm_init_mask.argtypes = [u32]
    L.zkm_init_devices.argtypes = [ctypes.c_void_p, i32]
    L.zkm_bases_register_ex.argtypes = [i32, i32, u64p, u8p, sz, u32, ctypes.POINTER(u64)]
    L.zkm_kzg_commit_batch.argtypes = [u64, i32, ctypes.c_void_p, ctypes.c_void_p, u64p, u8p]
    L.zkm_kzg_commit_hiding.argtypes = [u64, u64, u64p, sz, u64p, sz, u64p, u8p]
    L.zkm_kzg_open.argtypes = [u64, u64, u64p, sz, u64p, sz, u64p, u64p, u8p, u64p]
    L.zkm_profile_last_msm_counts.argtypes = [ctypes.c_void_p]
    L.zkm_msm_cache_stats.argtypes = [ctypes.c_void_p]
    L.zkm_shutdown.restype = None
    L.zkm_last_error.restype = ctypes.c_char_p
    L.zkm_version.restype = ctypes.c_char_p
    L.zkm_msm_g1.argtypes = [i32, u64p, u8p, u64p, sz, u64p, u8p]
    L.zkm_msm_g2.argtypes = [i32, u64p, u8p, u64p, sz, u64p, u8p]
    L.zkm_bases_register.argtypes = [i32, i32, u64p, u8p, sz, ctypes.POINTER(u64)]
    L.zkm_bases_register_device.argtypes = [i32, i32, u64p, u8p, sz, ctypes.POINTER(u64)]
    L.zkm_bases_release.argtypes = [u64]
    L.zkm_msm_registered.argtypes = [u64, sz, u64p, sz, u64p, u8p]
    L.zkm_msm_registered_device.argtypes = [u64, sz, u64p, sz, u64p, vp]
    L.zkm_points_sum_device.argtypes = [i32, i32, u64p, sz, u64p, vp]
    L.zkm_ntt.argtypes = [i32, u64p, u32, i32, i32]
    L.zkm_ntt_device.argtypes = [i32, u64p, u64p, u32, i32, i32, vp]
    L.zkm_domain_constants.argtypes = [i32, u32, u64p]
    L.zkm_set_option.argtypes = [ctypes.c_char_p, ctypes.c_int64]
    L.zkm_profile_last_msm.argtypes = [ctypes.c_void_p]
    L.zkm_fr_into_repr_device.argtypes = [i32, u64p, u64p, sz, vp]
    L.zkm_msm_batch_registered_device.argtypes = [i32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                  ctypes.c_void_p, ctypes.c_void_p, vp]
    L.zkm_kzg_commit.argtypes = [u64, u64p, sz, u64p, u8p]
    L.zkm_witness_map.argtypes = [i32, u64p, u64p, u64p, u32, u64p]
    L.zkm_witness_map_device.argtypes = [i32, u64p, u64p, u64p, u32, u64p, vp]
    L.zkm_launch_count.argtypes = [i32]
    L.zkm_launch_count.restype = u64
    L.zkm_msm_window_bits.argtypes = [i32, i32, sz]
    L.zkm_testgen_progression_device.argtypes = [i32, i32, u64, u64, sz, u64p, vp]
    L.zkm_fixed_base_msm.argtypes = [i32, i32, u64p, ctypes.c_uint8, u64p, sz, u64p, u8p]
    L.zkm_fixed_base_msm_device.argtypes = [i32, i32, u64p, ctypes.c_uint8, u64p, sz, u64p, u8p, vp]
    L.zkm_groth16_pk_create.argtypes = [i32, ctypes.c_void_p, u64p, u8p, u64p, u8p, ctypes.POINTER(u64)]
    L.zkm_groth16_pk_release.argtypes = [u64]
    L.zkm_groth16_prove.argtypes = [u64, u64p, u64p, u64p, u32, u64p, sz, sz, u64p, u64p, u64p, u8p, u64p, u8p, u64p, u8p]
    L.zkm_groth16_prove_device.argtypes = [u64, u64p, u64p, u64p, u32, u64p, sz, sz, u64p, u64p, u64p, vp]
    L.zkm_kzg_commit_many.argtypes = [u64, u64, i32, vp, vp, vp, vp, vp, u64p, u8p]
    L.zkm_kzg_open_batch.argtypes = [u64, u64, i32, vp, vp, i32, vp, vp, i32, u64p, i32, vp, vp, vp, vp, u64p, u64p, u8p, u64p,
                                     u64p]
    L.zkm_kzg_open_batch_device.argtypes = [u64, u64, i32, vp, vp, i32, vp, vp, i32, u64p, i32, vp, vp, vp, vp, u64p, u64p, u64p,
                                            u64p, vp]
    _lib = L
    return L


def check(rc: int):
    if rc == 0:
        return
    msg = (load().zkm_last_error() or b"").decode("utf-8", "replace")
    if rc == -4:
        raise DomainError(rc, msg)
    raise ZkmError(rc, msg)


def init(device=None):
    """Bind this process to one GPU (default: LOCAL_RANK, else 0) -- one process per GPU -- or, given a list of CUDA
    ordinals, to several GPUs of the box (one process, many GPUs: `zkm_init_devices`; the first entry is the primary
    device; a repeated ordinal gives separate lane sets on the same GPU, used to test the sharded paths on one GPU)."""
    global _inited_device
    L = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    key = tuple(device) if isinstance(device, (list, tuple)) else int(device)
    if _inited_device == key:
        return L
    if isinstance(key, tuple):
        arr = (ctypes.c_int32 * len(key))(*key)
        check(L.zkm_init_devices(ctypes.cast(arr, ctypes.c_void_p), len(key)))
    else:
        check(L.zkm_init(key))
    _inited_device = key
    return L


def initialised_devices() -> int:
    return int(load().zkm_initialised_devices())


def lib():
    """The initialised library (initialises on first use)."""
    if _inited_device is None:
        return init()
    return _lib


def shutdown():
    global _inited_device
    if _lib is not None:
        _lib.zkm_shutdown()
    _inited_device = None


def set_option(key: str, value: int):
    check(lib().zkm_set_option(key.encode(), int(value)))


def launch_count(reset: bool = False) -> int:
    return int(load().zkm_launch_count(1 if reset else 0))
