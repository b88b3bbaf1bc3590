"""ctypes binding of libsylow_b200.so.  Prototypes and constants are read from include/sylow_b200.h when this module
is imported, so the header is the one declaration of the C ABI.  Fails loudly if the CUDA library is missing or no
CUDA device is usable - there is no CPU fallback."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_size_t, c_uint64, c_void_p

from . import _header
from .build import LIB_PATH

_lib = None

_CONSTS, _FUNCS = _header.parse()
# the header's SYLOW_B200_* constants without the prefix: OK, ERR_ARG ... ERR_NOMEM, HASH_KECCAK256, HASH_SHA256,
# HASH_SHAKE128
globals().update({name[len("SYLOW_B200_"):]: int(value) for name, value in _CONSTS})

# A pointer is a c_void_p unless the binding reads or writes through it as a ctypes object.  An integer type missing
# from _INTS fails the import: a narrower ctypes type would truncate the argument, so it has to be mapped by hand.
_INTS = {"int": c_int, "size_t": c_size_t, "uint64_t": c_uint64}
_POINTERS = {("int", 1): POINTER(c_int), ("float", 1): POINTER(c_float), ("double", 1): POINTER(c_double),
             ("sylow_b200_ctx", 2): POINTER(c_void_p), ("char", 1): c_char_p}


def _ctypes_type(t: _header.CType):
    return _POINTERS.get((t.base, t.stars), c_void_p) if t.stars else _INTS[t.base]


_PROTOTYPES = {name: (_ctypes_type(ret), [_ctypes_type(t) for _, t in params]) for name, params, ret in _FUNCS}


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
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_PROTOTYPES)
