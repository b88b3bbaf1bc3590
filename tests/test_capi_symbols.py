"""CPU tier: the C-ABI library builds for sm_100a, loads, and exports every symbol the header declares.
No compute calls (there is no GPU here)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from sylow_b200 import _lib, build

    build.build_library()
    return _lib.load()


def _declared():
    with open(os.path.join(ROOT, "include", "sylow_b200.h")) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sylow_b200_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported(lib):
    from sylow_b200 import _lib

    declared = _declared()
    assert len(declared) >= 30
    assert declared == _lib.exported_symbols(), "header and ctypes signature table disagree"
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "sylow_b200", "libsylow_b200.so")],
                                  text=True)
    exported = set(re.findall(r"\bT (sylow_b200_\w+)", out))
    assert set(declared) <= exported, set(declared) - exported


def test_ctypes_prototypes_from_the_header(lib):
    """_lib.py derives argtypes/restype from the header.  Pin the entry points whose types are not plain data pointers,
    and the three bench.py calls through Engine._lib with c_void_p / None pointers."""
    from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_size_t, c_uint64, c_void_p as P

    pins = {
        "sylow_b200_create": (c_int, [POINTER(P), c_int]),
        "sylow_b200_create_multi": (c_int, [POINTER(P), POINTER(c_int), c_int]),
        "sylow_b200_strerror": (c_char_p, [c_int]),
        "sylow_b200_device_ctx": (P, [P, c_int]),
        "sylow_b200_launch_count": (c_uint64, [P]),
        "sylow_b200_imad_probe": (c_int, [P, c_int, c_int, c_int, c_int, POINTER(c_float), POINTER(c_double)]),
        "sylow_b200_hash_failed_dev": (c_int, [P, P, POINTER(c_int)]),
        "sylow_b200_pairing_batch": (c_int, [P, P, P, P, P, c_size_t, P]),
        "sylow_b200_verify_batch": (c_int, [P, P, P, P, P, P, P, c_size_t, P, c_size_t, c_int, P, POINTER(c_int)]),
        "sylow_b200_verify_batch_partial": (c_int, [P, P, P, P, P, P, P, c_size_t, P, c_size_t, c_int, P, c_uint64, P]),
    }
    for name, (res, args) in pins.items():
        fn = getattr(lib, name)
        assert (fn.restype, list(fn.argtypes)) == (res, args), name


def test_strerror_and_arg_checks(lib):
    assert lib.sylow_b200_strerror(0) == b"ok"
    assert b"argument" in lib.sylow_b200_strerror(-1)
    assert lib.sylow_b200_create(None, 0) == -1  # NULL out pointer is rejected before any CUDA call
    assert lib.sylow_b200_destroy(None) == -1


def test_library_targets_sm100a_with_imad_wide_carry_chains():
    """The Montgomery product must compile to IMAD.WIDE.U32(.X) carry chains (DESIGN.md, fp.cuh)."""
    so = os.path.join(ROOT, "sylow_b200", "libsylow_b200.so")
    sass = subprocess.check_output(["cuobjdump", "-sass", so], text=True)
    assert "sm_100a" in sass
    fp_op = sass[sass.index("k_fp_op"):]
    fp_op = fp_op[:fp_op.index("Function :")]
    assert fp_op.count("IMAD.WIDE.U32.X") > 100


def test_rust_bindings_are_in_sync_with_the_header():
    """ffi/sylow-cuda-sys/src/lib.rs is generated from include/sylow_b200.h (tools/gen_rust_ffi.py)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gen_rust_ffi.py"), "--check"])
    assert r.returncode == 0, "run tools/gen_rust_ffi.py"
