"""CPU tier: the per-item bodies of pointwise addition (csrc/group_law.cuh: add_pair, run by k_g1_add / k_g2_add) and
of the EIP-196 steps (decode_be_item, g1_validate_item, eip196_scalar_item, eip196_finish_item), compiled for the host
from the device source (tests/hostsim/group_law.cu), against oracle.bn254_py and the pinned EIP-196 vectors."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import bn254_py as o
from tests import wire as w

HERE = os.path.dirname(os.path.abspath(__file__))
R = o.R_ORDER
GROUPS = [(0, o.FpOps, o.G1_GEN), (1, o.Fp2Ops, o.G2_GEN)]
ERR_DECODE, ERR_NOT_ON_CURVE = -6, -3


@pytest.fixture(scope="module")
def gl(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("group_law") / "libgroup_law.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "group_law.cu")])
    return ctypes.CDLL(so)


def _zero(F):
    return o.proj_to_affine(F, o.proj_zero(F))


def _mul(F, gen, k):
    return o.proj_to_affine(F, o.proj_mul(F, o.affine_to_proj(F, gen), k % R))


def _neg(F, p):
    return o.g1_affine_neg(p) if F is o.FpOps else o.g2_affine_neg(p)


def _expect(F, a, b, subtract):
    b = _neg(F, b) if subtract else b
    return o.proj_to_affine(F, o.proj_add(F, o.affine_to_proj(F, a), o.affine_to_proj(F, b)))


def _add(gl, g2, F, a, b, subtract):
    width = 128 if g2 else 64
    enc = w.g2_b if g2 else w.g1_b
    out = ctypes.create_string_buffer(width)
    inf = ctypes.c_uint8()
    gl.hs_add_pair(ctypes.c_int(g2), enc(a), ctypes.c_int(int(a[2])), enc(b), ctypes.c_int(int(b[2])),
                   ctypes.c_int(int(subtract)), out, ctypes.byref(inf))
    return (w.b_g2 if g2 else w.b_g1)(out.raw, inf.value)


@pytest.mark.parametrize("g2,F,gen", GROUPS, ids=["g1", "g2"])
@pytest.mark.parametrize("subtract", [False, True], ids=["add", "sub"])
def test_add_pair_edge_cases(gl, g2, F, gen, subtract):
    rng = random.Random(3 + g2)
    a, b = _mul(F, gen, rng.randrange(1, R)), _mul(F, gen, rng.randrange(1, R))
    O = _zero(F)
    cases = [(O, O), (O, b), (a, O), (a, a), (a, _neg(F, a)), (a, b), (b, a)]
    for x, y in cases:
        assert _add(gl, g2, F, x, y, subtract) == _expect(F, x, y, subtract), (x, y)
    # the named identities, stated directly
    assert _add(gl, g2, F, a, a, True) == O                                  # a - a
    assert _add(gl, g2, F, a, O, True) == a                                  # a - O
    assert _add(gl, g2, F, O, a, True) == _neg(F, a)                         # O - a


@pytest.mark.parametrize("g2,F,gen", GROUPS, ids=["g1", "g2"])
def test_add_pair_doubles_and_cancels(gl, g2, F, gen):
    k = 0x1234567890ABCDEF
    a = _mul(F, gen, k)
    assert _add(gl, g2, F, a, a, False) == _mul(F, gen, 2 * k)
    assert _add(gl, g2, F, a, _neg(F, a), False) == _zero(F)


@pytest.mark.parametrize("g2,F,gen", GROUPS, ids=["g1", "g2"])
def test_add_pair_random(gl, g2, F, gen):
    rng = random.Random(17 + g2)
    for i in range(200):
        k1, k2 = rng.randrange(R), rng.randrange(R)
        a, b = _mul(F, gen, k1), _mul(F, gen, k2)
        sub = bool(i & 1)
        got = _add(gl, g2, F, a, b, sub)
        assert got == _expect(F, a, b, sub)
        assert got == _mul(F, gen, k1 - k2 if sub else k1 + k2)


def _be(*vals) -> bytes:
    return b"".join(int(v).to_bytes(32, "big") for v in vals)


def _eip196_add(gl, inp: bytes):
    out = ctypes.create_string_buffer(64)
    st = ctypes.c_int8()
    gl.hs_eip196_add(inp, out, ctypes.byref(st))
    return out.raw, st.value


def _decode(gl, inp: bytes, mul: int):
    pts = ctypes.create_string_buffer(128)
    infs = (ctypes.c_uint8 * 2)()
    sts = (ctypes.c_int8 * 2)()
    k = ctypes.create_string_buffer(32)
    gl.hs_eip196_decode(inp, ctypes.c_int(mul), pts, infs, sts, k)
    return pts.raw, list(infs), list(sts), w.b_fp(k.raw)


def _finish(gl, pt, inf, st_a, st_b):
    out = ctypes.create_string_buffer(64)
    st = ctypes.c_int8()
    gl.hs_eip196_finish(w.g1_b(pt), ctypes.c_int(int(inf)), ctypes.c_int(st_a), ctypes.c_int(st_b), out,
                        ctypes.byref(st))
    return out.raw, st.value


def _eip196_mul(gl, inp: bytes):
    """decode / validate / scalar steps of the host simulation, the multiplication by the oracle, then the epilogue"""
    pts, infs, sts, k = _decode(gl, inp, 1)
    p = w.b_g1(pts[:64], infs[0])
    q = _zero(o.FpOps) if p[2] else o.proj_to_affine(o.FpOps, o.proj_mul(o.FpOps, o.affine_to_proj(o.FpOps, p), k))
    return _finish(gl, q, q[2], sts[0], 0)


def test_eip196_add_kat(gl, kats):
    out, st = _eip196_add(gl, bytes.fromhex(kats["eip196_add"]["input"]))
    assert st == 0 and out.hex() == kats["eip196_add"]["expected"]


def test_eip196_mul_kat(gl, kats):
    out, st = _eip196_mul(gl, bytes.fromhex(kats["eip196_mul"]["input"]))
    assert st == 0 and out.hex() == kats["eip196_mul"]["expected"]


def test_eip196_scalar_is_big_endian(gl):
    s = random.Random(9).getrandbits(256)
    assert _decode(gl, _be(1, 2, s), 1)[3] == s


# (first point, expected status): the point is placed first and second in ecAdd and is ecMul's point
BAD = [((o.P, 2), ERR_DECODE), ((1, o.P), ERR_DECODE), ((0x31 << 248, 2), ERR_DECODE),
       ((1, 3), ERR_NOT_ON_CURVE), ((0, 1), ERR_NOT_ON_CURVE)]


@pytest.mark.parametrize("pt,status", BAD, ids=["x=p", "y=p", "top-byte", "(1,3)", "(0,1)"])
def test_eip196_failed_inputs(gl, pt, status):
    g = (1, 2)
    for inp in (_be(*pt, *g), _be(*g, *pt)):
        assert _eip196_add(gl, inp) == (bytes(64), status)
    assert _eip196_mul(gl, _be(*pt, 5)) == (bytes(64), status)


def test_eip196_infinity(gl):
    assert _eip196_add(gl, bytes(128)) == (bytes(64), 0)                        # (0,0) + (0,0)
    g = _be(1, 2)
    assert _eip196_add(gl, g + bytes(64)) == (g, 0)                             # P + O
    assert _eip196_add(gl, bytes(64) + g) == (g, 0)                             # O + P
    assert _eip196_add(gl, g + _be(1, o.P - 2)) == (bytes(64), 0)               # P + (-P)
    assert _eip196_mul(gl, bytes(64) + _be(7)) == (bytes(64), 0)                # k O
    assert _eip196_mul(gl, g + _be(R)) == (bytes(64), 0)                        # r P
    assert _eip196_mul(gl, g + _be(0)) == (bytes(64), 0)                        # 0 P


def test_eip196_finish_folds_first_error(gl):
    g = (1, 2, False)
    assert _finish(gl, g, False, 0, 0) == (_be(1, 2), 0)
    assert _finish(gl, g, False, ERR_DECODE, ERR_NOT_ON_CURVE) == (bytes(64), ERR_DECODE)
    assert _finish(gl, g, False, 0, ERR_NOT_ON_CURVE) == (bytes(64), ERR_NOT_ON_CURVE)
    assert _finish(gl, g, True, 0, 0) == (bytes(64), 0)
