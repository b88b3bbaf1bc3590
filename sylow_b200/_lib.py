"""ctypes binding of libsylow_b200.so (include/sylow_b200.h).  Fails loudly if the CUDA library is
missing or no CUDA device is usable - there is no CPU fallback."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_size_t, c_uint64, c_void_p

from .build import LIB_PATH

_lib = None

OK = 0
ERR_ARG, ERR_CUDA, ERR_NOT_ON_CURVE, ERR_NOT_IN_SUBGROUP, ERR_CANNOT_HASH, ERR_DECODE, ERR_NOMEM = range(-1, -8, -1)
HASH_KECCAK256 = 0
HASH_SHA256 = 1
HASH_SHAKE128 = 2

# every symbol include/sylow_b200.h declares (tests/test_capi_symbols.py checks the header against this)
_P = c_void_p
_SIGNATURES = {
    "sylow_b200_create": (c_int, [POINTER(c_void_p), c_int]),
    "sylow_b200_create_multi": (c_int, [POINTER(c_void_p), POINTER(c_int), c_int]),
    "sylow_b200_device_count": (c_int, [_P]),
    "sylow_b200_device_ctx": (c_void_p, [_P, c_int]),
    "sylow_b200_destroy": (c_int, [_P]),
    "sylow_b200_strerror": (c_char_p, [c_int]),
    "sylow_b200_last_cuda_error": (c_int, [_P]),
    "sylow_b200_launch_count": (c_uint64, [_P]),
    "sylow_b200_pairing_batch": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P]),
    "sylow_b200_miller_loop_batch": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P]),
    "sylow_b200_miller_product": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P]),
    "sylow_b200_final_exp_batch": (c_int, [_P, _P, c_size_t, _P]),
    "sylow_b200_fp12_product": (c_int, [_P, _P, c_size_t, _P]),
    "sylow_b200_pairing_check_batch": (c_int, [_P, _P, _P, _P, _P, c_size_t, c_size_t, _P]),
    "sylow_b200_g2_precompute": (c_int, [_P, _P, c_size_t, _P]),
    "sylow_b200_miller_loop_precomputed": (c_int, [_P, _P, _P, _P, c_size_t, _P]),
    "sylow_b200_pairing_check_fixed_batch": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_size_t, _P]),
    "sylow_b200_pairing_check_fixed_batch_dev": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_size_t, _P, _P]),
    "sylow_b200_tables_to_device": (c_int, [_P, _P, c_size_t, _P, _P]),
    "sylow_b200_miller_loop_precomputed_batch": (c_int, [_P, _P, _P, _P, c_size_t, _P]),
    "sylow_b200_miller_product_precomputed": (c_int, [_P, _P, _P, _P, c_size_t, _P]),
    "sylow_b200_g2_precompute_dev": (c_int, [_P, _P, c_size_t, _P, _P]),
    "sylow_b200_miller_product_precomputed_dev": (c_int, [_P, _P, c_size_t, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_g1_validate_batch": (c_int, [_P, _P, _P, c_size_t, _P]),
    "sylow_b200_g2_validate_batch": (c_int, [_P, _P, _P, c_size_t, _P]),
    "sylow_b200_g1_from_be_bytes_batch": (c_int, [_P, _P, c_size_t, c_int, _P, _P, _P]),
    "sylow_b200_g2_from_be_bytes_batch": (c_int, [_P, _P, c_size_t, c_int, _P, _P, _P]),
    "sylow_b200_g1_to_be_bytes_batch": (c_int, [_P, _P, _P, c_size_t, c_int, _P]),
    "sylow_b200_g2_to_be_bytes_batch": (c_int, [_P, _P, _P, c_size_t, c_int, _P]),
    "sylow_b200_eip197_pairing_check_batch": (c_int, [_P, _P, c_size_t, c_size_t, _P, _P]),
    "sylow_b200_gt_mul_batch": (c_int, [_P, _P, _P, c_size_t, _P]),
    "sylow_b200_g1_mul_batch": (c_int, [_P, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_g2_mul_batch": (c_int, [_P, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_hash_to_g1_batch": (c_int, [_P, _P, _P, c_size_t, _P, c_size_t, c_int, _P, _P]),
    "sylow_b200_g1_sum": (c_int, [_P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_g1_msm": (c_int, [_P, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_g1_msm_bucket": (c_int, [_P, _P, _P, _P, c_size_t, c_int, _P, _P]),
    "sylow_b200_lagrange_coefficients_batch": (c_int, [_P, _P, c_size_t, c_size_t, _P]),
    "sylow_b200_threshold_aggregate_batch": (c_int, [_P, _P, _P, _P, c_size_t, c_size_t, _P, _P]),
    "sylow_b200_verify_batch_same_signer": (c_int, [_P, _P, c_int, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_int, _P,
                                                    POINTER(c_int)]),
    "sylow_b200_expand_message_batch": (c_int, [_P, _P, _P, c_size_t, _P, c_size_t, c_int, c_size_t, _P]),
    "sylow_b200_hash_to_field_batch": (c_int, [_P, _P, _P, c_size_t, _P, c_size_t, c_int, _P]),
    "sylow_b200_sign_batch": (c_int, [_P, _P, _P, _P, c_size_t, _P, c_size_t, c_int, _P, _P]),
    "sylow_b200_verify_each": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_int, _P]),
    "sylow_b200_verify_batch_partial": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_int, _P, c_uint64,
                                                _P]),
    "sylow_b200_verify_batch_finish": (c_int, [_P, _P, c_size_t, POINTER(c_int)]),
    "sylow_b200_verify_batch": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_int, _P, POINTER(c_int)]),
    "sylow_b200_hash_failed_dev": (c_int, [_P, _P, POINTER(c_int)]),
    "sylow_b200_batch_weights": (c_int, [_P, _P, c_uint64, c_size_t, _P]),
    "sylow_b200_pairing_batch_dev": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_miller_loop_batch_dev": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_miller_product_dev": (c_int, [_P, _P, _P, _P, _P, c_size_t, _P, _P]),
    "sylow_b200_final_exp_batch_dev": (c_int, [_P, _P, c_size_t, _P, _P]),
    "sylow_b200_pairing_check_batch_dev": (c_int, [_P, _P, _P, _P, _P, c_size_t, c_size_t, _P, _P]),
    "sylow_b200_g1_mul_batch_dev": (c_int, [_P, _P, _P, _P, c_size_t, _P, _P, _P]),
    "sylow_b200_g2_mul_batch_dev": (c_int, [_P, _P, _P, _P, c_size_t, _P, _P, _P]),
    "sylow_b200_hash_to_g1_batch_dev": (c_int, [_P, _P, _P, c_size_t, _P, c_size_t, c_int, _P, _P, _P]),
    "sylow_b200_verify_batch_partial_dev": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_size_t, _P, c_size_t, c_int, _P,
                                                    c_uint64, _P, _P]),
    "sylow_b200_fp_op_batch": (c_int, [_P, c_int, _P, _P, c_size_t, _P]),
    "sylow_b200_fp12_op_batch": (c_int, [_P, c_int, _P, _P, c_size_t, _P]),
    "sylow_b200_imad_probe": (c_int, [_P, c_int, c_int, c_int, c_int, POINTER(c_float), POINTER(c_double)]),
}


class SylowB200Error(RuntimeError):
    def __init__(self, status: int, where: str, cuda_error: int = 0):
        self.status = status
        self.cuda_error = cuda_error
        msg = load().sylow_b200_strerror(status).decode()
        if cuda_error:
            msg += " (cudaError %d)" % cuda_error
        super().__init__("%s: %s" % (where, msg))


def load():
    """Load libsylow_b200.so; raise (never fall back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SYLOW_B200_LIB", LIB_PATH)  # tuning experiments load alternative builds
    if not os.path.exists(path):
        raise RuntimeError(
            "libsylow_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `python -m sylow_b200.build`. There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)
