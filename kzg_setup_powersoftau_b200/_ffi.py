"""ctypes binding of libptau_b200.so (include/ptau_b200.h).

The library is the product; this module only marshals pointers and sizes.  It
fails loudly if the shared library has not been built (there is no fallback of
any kind -- see __graft_entry__.build()).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PTAU_LIB selects an alternative build of the same library (A/B kernel experiments)
LIB_PATH = os.environ.get("PTAU_LIB") or os.path.join(_HERE, "libptau_b200.so")

# constants mirrored from include/ptau_b200.h (checked by tests/test_host_logic.py)
G1, G2 = 1, 2
FMT_ZCASH_UNCOMPRESSED, FMT_ZCASH_COMPRESSED, FMT_ARK_UNCOMPRESSED, FMT_ARK_MONT_LIMBS = 1, 2, 3, 4
CHECK_ON_CURVE, CHECK_SUBGROUP, CHECK_REJECT_INFINITY = 2, 4, 8
CHECKS_LOAD = 0
CHECKS_READ = CHECK_SUBGROUP
CHECKS_DECOMPRESS = 0
CHECKS_STRICT = CHECK_ON_CURVE | CHECK_SUBGROUP | CHECK_REJECT_INFINITY
OK = 0
BAD_NON_CANONICAL, BAD_FLAGS, BAD_INFINITY, BAD_NOT_ON_CURVE, BAD_NOT_IN_SUBGROUP = 1, 2, 3, 4, 5
BAD_NOT_POWERS = 6
ERR_CUDA, ERR_ARG, ERR_SIZE, ERR_NOMEM, ERR_IO, ERR_DIGEST, ERR_EXISTS = -1, -2, -3, -4, -5, -6, -7
FILE_SKIP_DIGEST, FILE_NO_UNCOMPRESSED, FILE_FSYNC = 1, 2, 4
VARIANT_KGZ, VARIANT_FASTKGZ = 1, 2
STATUS_NONE = 0xFFFFFFFFFFFFFFFF
POWERS_RESPONSE, POWERS_KGZ, POWERS_FASTKGZ = 1, 2, 3
REL_GENERATORS, REL_TAU_G1, REL_TAU_G2, REL_ALPHA_G1, REL_BETA_G1, REL_BETA_G2, REL_KEY = 0, 1, 2, 3, 4, 5, 6

BAD_NAMES = {
    BAD_NON_CANONICAL: "NON_CANONICAL",
    BAD_FLAGS: "BAD_FLAGS",
    BAD_INFINITY: "INFINITY",
    BAD_NOT_ON_CURVE: "NOT_ON_CURVE",
    BAD_NOT_IN_SUBGROUP: "NOT_IN_SUBGROUP",
    BAD_NOT_POWERS: "NOT_POWERS",
}
REL_NAMES = ("GENERATORS", "TAU_G1", "TAU_G2", "ALPHA_G1", "BETA_G1", "BETA_G2", "KEY")


class Timing(C.Structure):
    _fields_ = [
        ("n_gpus", C.c_int),
        ("wall_ms", C.c_double),
        ("gpu_ms", C.c_double * 8),
        ("kernel_ms", C.c_double * 8),
        ("h2d_bytes", C.c_uint64 * 8),
        ("d2h_bytes", C.c_uint64 * 8),
        ("kernel_launches", C.c_uint64),
    ]


_SIGNATURES = {
    "ptau_device_count": (C.c_int, []),
    "ptau_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_int), C.c_size_t]),
    "ptau_destroy": (None, [C.c_void_p]),
    "ptau_strerror": (C.c_char_p, [C.c_int]),
    "ptau_last_error": (C.c_char_p, [C.c_void_p]),
    "ptau_last_timing": (C.c_int, [C.c_void_p, C.POINTER(Timing)]),
    "ptau_host_alloc": (C.c_void_p, [C.c_size_t]),
    "ptau_host_free": (None, [C.c_void_p]),
    "ptau_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "ptau_host_unregister": (C.c_int, [C.c_void_p]),
    "ptau_record_size": (C.c_size_t, [C.c_int, C.c_int]),
    "ptau_response_size": (C.c_uint64, [C.c_uint64]),
    "ptau_uncompressed_size": (C.c_uint64, [C.c_uint64]),
    "ptau_setup_size": (C.c_uint64, [C.c_int, C.c_uint64]),
    "ptau_convert": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_uint,
         C.POINTER(C.c_uint64), C.POINTER(C.c_int)],
    ),
    "ptau_convert_device": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_uint,
         C.c_uint64, C.c_void_p, C.c_void_p],
    ),
    "ptau_status_decode": (C.c_int, [C.c_uint64, C.POINTER(C.c_uint64)]),
    "ptau_generate": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_uint64, C.c_size_t, C.c_void_p],
    ),
    "ptau_generate_device": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_uint64, C.c_size_t, C.c_void_p,
         C.c_void_p],
    ),
    "ptau_preprocess": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
         C.c_uint64, C.c_uint, C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_int)],
    ),
    "ptau_preprocess_uncompressed": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint,
         C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_int)],
    ),
    "ptau_load_setup": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint, C.c_void_p, C.c_uint64,
         C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_int)],
    ),
    "ptau_load_phase1": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint, C.c_void_p, C.c_uint64, C.c_void_p,
         C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_int)],
    ),
    "ptau_preprocess_files": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint, C.c_char_p, C.c_uint, C.c_uint,
         C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_int)],
    ),
    "ptau_load_setup_file": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_char_p, C.c_uint64, C.c_uint, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int)],
    ),
    "ptau_blake2b_file": (C.c_int, [C.c_char_p, C.c_char_p]),
    "ptau_kzg_commit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ptau_kzg_powers_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "ptau_kzg_powers_free": (None, [C.c_void_p]),
    "ptau_kzg_commit_resident": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ptau_kzg_quotient": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ptau_kzg_open": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
         C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "ptau_kzg_check": (C.c_int, [C.c_void_p] * 8 + [C.c_size_t, C.c_void_p]),
    "ptau_pairing_product2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "ptau_g2_prepare": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "ptau_msm_g2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ptau_verify_powers": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_char_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int),
         C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p],
    ),
    "ptau_selftest_fq_op": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "ptau_microbench": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib() -> C.CDLL:
    """Load libptau_b200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libptau_b200.so is missing (%s). Build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C kzg_setup_powersoftau_b200/csrc`. There is no CPU fallback." % LIB_PATH
            )
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def strerror(code: int) -> str:
    return lib().ptau_strerror(code).decode()
