"""CPU tier: the per-thread body of fixed-base multiplication by a generator (csrc/curve.cuh: scalar_reduce_r,
scalar_digit, proj_add_mixed and gen_scalar_mul, run by k_g1_mul_gen / k_g2_mul_gen), compiled for the host from the
device source (tests/hostsim/generator_mul.cu), against oracle.bn254_py.  The table is built here from the oracle."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import bn254_py as o
from tests import wire as w

HERE = os.path.dirname(os.path.abspath(__file__))
R = o.R_ORDER
MONT = 1 << 256
GROUPS = [(0, o.FpOps, o.G1_GEN), (1, o.Fp2Ops, o.G2_GEN)]


@pytest.fixture(scope="module")
def gm(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("generator_mul") / "libgenerator_mul.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "generator_mul.cu")])
    lib = ctypes.CDLL(so)
    c, nw, e = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    lib.hs_gen_params(ctypes.byref(c), ctypes.byref(nw), ctypes.byref(e))
    lib.params = (c.value, nw.value, e.value)
    return lib


def _coords(F, v):
    return [v] if F is o.FpOps else list(v)


def _pt_b(F, *coords) -> bytes:
    return b"".join(w.fp_b(c) for v in coords for c in _coords(F, v))


def _read(F, raw: bytes, inf: int):
    return w.b_g1(raw, inf) if F is o.FpOps else w.b_g2(raw, inf)


def _expect(F, gen, k):
    return o.proj_to_affine(F, o.proj_mul(F, o.affine_to_proj(F, gen), k % R))


@pytest.fixture(scope="module")
def tables(gm):
    """Device form of the table of each generator: T[w][j] = (j + 1) 2^(C w) G, affine, Montgomery form."""
    c, nw, ne = gm.params
    out = {}
    for g2, F, gen in GROUPS:
        base = o.affine_to_proj(F, gen)
        rows = []
        for _ in range(nw):
            acc = base
            for _ in range(ne):
                x, y, inf = o.proj_to_affine(F, acc)
                assert not inf
                rows.append(b"".join(w.fp_b(v * MONT % o.P) for v in _coords(F, x) + _coords(F, y)))
                acc = o.proj_add(F, acc, base)
            for _ in range(c):
                base = o.proj_double(F, base)
        out[g2] = b"".join(rows)
    return out


def _digits(gm, k):
    nw = gm.params[1]
    d = (ctypes.c_int * nw)()
    red = ctypes.create_string_buffer(32)
    gm.hs_gen_digits(w.fp_b(k), d, red)
    return list(d), w.b_fp(red.raw)


def _mul(gm, tables, g2, F, k):
    out = ctypes.create_string_buffer(128 if g2 else 64)
    inf = ctypes.c_uint8()
    tab = tables[g2]
    gm.hs_gen_mul(ctypes.c_int(g2), tab, ctypes.c_size_t(len(tab)), w.fp_b(k), out, ctypes.byref(inf))
    return _read(F, out.raw, inf.value)


def _edge_scalars(c, nw):
    """The reduction's edges, digits at +-2^(C-1) and carries across every window boundary."""
    ks = [0, 1, 2, R - 1, R, R + 1] + [m * R for m in range(2, 6)] + [o.P - 1, o.P, MONT - 1]
    ks += [int.from_bytes(bytes([b]) * 32, "little") for b in (0x80, 0x7F, 0xFF)]
    ks += [int.from_bytes(bytes([b]) * 32, "little") % (1 << 253) for b in (0x80, 0x7F, 0xFF)]
    half = 1 << (c - 1)
    below = nw - 1  # windows fully below 2^254
    ks.append(sum(half << (c * i) for i in range(below)))            # every digit +2^(C-1), no carry
    ks.append(sum((half + 1) << (c * i) for i in range(below)))      # every digit negative, a carry into each window
    ks.append(sum(((1 << c) - 1) << (c * i) for i in range(below)))  # all ones: one carry rippling through every window
    ks.append((1 << (c * below)) - half)                             # a borrow ending at the top window
    ks += [half << (c * i) for i in range(nw)] + [((1 << c) - 1) << (c * i) for i in range(below)]
    return ks


def _random_scalars(n, seed):
    rng = random.Random(seed)
    return [rng.getrandbits(256) for _ in range(n)]


def test_recoding_reconstructs_k_mod_r(gm):
    c, nw, ne = gm.params
    assert nw * c >= 254 and ne == 1 << (c - 1)
    for k in _edge_scalars(c, nw) + _random_scalars(500, 1):
        d, red = _digits(gm, k)
        assert red == k % R, hex(k)
        assert all(abs(x) <= ne for x in d), (hex(k), d)
        assert sum(x << (c * i) for i, x in enumerate(d)) == k % R, hex(k)


def test_recoding_hits_the_digit_bound(gm):
    c, nw, ne = gm.params
    d, _ = _digits(gm, sum(ne << (c * i) for i in range(nw - 1)))
    assert d[:nw - 1] == [ne] * (nw - 1)
    d, _ = _digits(gm, sum((ne + 1) << (c * i) for i in range(nw - 1)))
    assert d[0] == 1 - ne and all(x == 2 - ne for x in d[1:nw - 1]) and d[nw - 1] == 1


@pytest.mark.parametrize("g2,F,gen", GROUPS, ids=["g1", "g2"])
def test_mixed_addition(gm, g2, F, gen):
    rng = random.Random(5 + g2)
    width = 128 if g2 else 64
    e = _expect(F, gen, rng.randrange(1, R))
    ex, ey = e[0], e[1]
    scale = (lambda a, z: F.mul(a, z))
    z = (rng.randrange(1, o.P) if F is o.FpOps else (rng.randrange(o.P), rng.randrange(o.P)))

    def run(acc):
        out = ctypes.create_string_buffer(width)
        inf = ctypes.c_uint8()
        gm.hs_add_mixed(ctypes.c_int(g2), _pt_b(F, *acc), _pt_b(F, ex, ey), out, ctypes.byref(inf))
        return _read(F, out.raw, inf.value)

    e_proj = (scale(ex, z), scale(ey, z), z)
    assert run(o.proj_zero(F)) == e                                              # acc = O
    assert run(e_proj) == o.proj_to_affine(F, o.proj_double(F, e_proj))          # acc = e
    assert run(o.proj_neg(F, e_proj)) == o.proj_to_affine(F, o.proj_zero(F))    # acc = -e
    a = o.affine_to_proj(F, _expect(F, gen, rng.randrange(1, R)))
    a = (scale(a[0], z), scale(a[1], z), z)
    assert run(a) == o.proj_to_affine(F, o.proj_add(F, a, o.affine_to_proj(F, e)))  # generic


@pytest.mark.parametrize("g2,F,gen", GROUPS, ids=["g1", "g2"])
def test_multiplication_edge_scalars(gm, tables, g2, F, gen):
    c, nw, _ = gm.params
    for k in _edge_scalars(c, nw):
        assert _mul(gm, tables, g2, F, k) == _expect(F, gen, k), hex(k)


@pytest.mark.parametrize("g2,F,gen", GROUPS, ids=["g1", "g2"])
def test_multiplication_random_scalars(gm, tables, g2, F, gen):
    for k in _random_scalars(200, 11 + g2):
        assert _mul(gm, tables, g2, F, k) == _expect(F, gen, k), hex(k)
