"""CPU tier: the per-thread bodies of the Groth16 kernels (csrc/groth16.cuh, run by k_groth16_assemble,
k_groth16_fr_partial and k_groth16_fr_final), compiled for the host from the device source (tests/hostsim/groth16.cu),
against oracle.bn254_py and the Groth16 reference of tests/groth16_ref.py.  The device form of the key is built here
from the oracle; only its -alpha, IC_0 and IC_i tables are read by these bodies."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import bn254_py as o
from tests import groth16_ref as g
from tests import wire as w

HERE = os.path.dirname(os.path.abspath(__file__))
R = o.R_ORDER
MONT = 1 << 256
EDGE_X = [0, 1, R - 1, R, R + 1, MONT - 1]


@pytest.fixture(scope="module")
def hs(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("groth16") / "libgroth16.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "groth16.cu")])
    lib = ctypes.CDLL(so)
    v = [ctypes.c_size_t() for _ in range(4)]
    lib.hs_g16_layout(*[ctypes.byref(x) for x in v])
    lib.layout = [x.value for x in v]
    return lib


_TABLES = {}


def _table(p):
    """gen_scalar_mul's table of p: T[w][j] = (j + 1) 2^(8 w) p, affine x || y in Montgomery form"""
    if p not in _TABLES:
        base = o.affine_to_proj(o.FpOps, p)
        rows = []
        for _ in range(32):
            acc = base
            for _ in range(128):
                x, y, inf = o.proj_to_affine(o.FpOps, acc)
                assert not inf
                rows.append(w.fp_b(x * MONT % o.P) + w.fp_b(y * MONT % o.P))
                acc = o.proj_add(o.FpOps, acc, base)
            for _ in range(8):
                base = o.proj_double(o.FpOps, base)
        _TABLES[p] = b"".join(rows)
    return _TABLES[p]


def _device_key(hs, vk):
    neg_alpha, ic0, tables, table_bytes = hs.layout
    alpha, _, _, _, ic = vk
    out = bytearray(tables + (len(ic) - 1) * table_bytes)
    out[neg_alpha:neg_alpha + 64] = w.g1_b(o.g1_affine_neg(alpha))
    out[ic0:ic0 + 64] = w.g1_b(ic[0])
    for i, p in enumerate(ic[1:]):
        out[tables + i * table_bytes:tables + (i + 1) * table_bytes] = _table(p)
    return bytes(out)


def _assemble(hs, key, l, xs, proof, inf):
    rec, b = ctypes.create_string_buffer(256), ctypes.create_string_buffer(128)
    rec_inf, b_inf, ok = (ctypes.c_uint8 * 4)(), ctypes.c_uint8(), ctypes.c_int()
    x = b"".join(v.to_bytes(32, "little") for v in xs) or bytes(32)
    hs.hs_g16_assemble(key, ctypes.c_size_t(len(key)), ctypes.c_size_t(l), x, g.proof_bytes(proof),
                       None if inf is None else bytes(inf), rec, rec_inf, b, ctypes.byref(b_inf), ctypes.byref(ok))
    return rec.raw, list(rec_inf), b.raw, b_inf.value, bool(ok.value)


@pytest.mark.parametrize("l", [0, 1, 3, 16])
def test_assembly_body(hs, l):
    td = g.Trapdoor(l, 50 + l)
    vk = td.vk()
    key = _device_key(hs, vk)
    rng = random.Random(l)
    cases = [[rng.randrange(R) for _ in range(l)] for _ in range(3)]
    if l:
        cases += [[e] + [rng.randrange(R) for _ in range(l - 1)] for e in EDGE_X]
        cases.append([R - 1] * l)
    flags = [None, (0, 0, 0), (1, 0, 0), (0, 0, 1), (0, 1, 0), (1, 1, 1)]
    for t, xs in enumerate(cases):
        a, b_, c = td.proof_scalars([v % R for v in xs])
        proof = (g.g1_mul(a), g.g2_mul(b_), g.g1_mul(c))
        inf = flags[t % len(flags)]
        rec, rec_inf, b, b_inf, ok = _assemble(hs, key, l, xs, proof, inf)
        fl = inf or (0, 0, 0)
        neg_l = o.g1_affine_neg(g.public_term(vk[4], [v % R for v in xs]))
        neg_c = proof[2] if fl[2] else o.g1_affine_neg(proof[2])
        assert rec == w.g1_b(proof[0]) + w.g1_b(o.g1_affine_neg(vk[0])) + w.g1_b(neg_l) + w.g1_b(neg_c), (t, xs)
        assert rec_inf == [fl[0], 0, int(neg_l[2]), fl[2]]
        assert (b, b_inf) == (w.g2_b(proof[1]), fl[1])
        assert ok == all(v < R for v in xs), xs
        if t < 2 and fl == (0, 0, 0):  # the verifier equation on the assembled record
            assert g.groth16_verify(vk, proof, xs) == ok


def test_public_term_at_infinity(hs):
    """IC_0 + x IC_1 = O (x = -u_0 / u_1): the record carries -L as (0, 1) with its flag set"""
    td = g.Trapdoor(1, 77)
    vk = td.vk()
    key = _device_key(hs, vk)
    x = -td.u[0] * pow(td.u[1], -1, R) % R
    proof = (g.g1_mul(2), g.g2_mul(3), g.g1_mul(5))
    rec, rec_inf, _, _, ok = _assemble(hs, key, 1, [x], proof, None)
    assert ok and rec_inf[2] == 1 and rec[128:192] == w.g1_b((0, 1, True))


@pytest.mark.parametrize("threads", [1, 7, 256])
def test_weighted_sums(hs, threads):
    rng = random.Random(threads)
    for n in (1, 2, 33, 300):
        r = [rng.getrandbits(64) | 1 for _ in range(n)]
        xs = [rng.randrange(R) for _ in range(n)]
        xs[0] = R - 1
        rr = (ctypes.c_uint64 * n)(*r)
        out, ok = ctypes.create_string_buffer(32), ctypes.c_int()
        hs.hs_g16_weighted_sum(b"".join(v.to_bytes(32, "little") for v in xs), rr, ctypes.c_size_t(n),
                               ctypes.c_size_t(threads), out, ctypes.byref(ok))
        assert w.b_fp(out.raw) == sum(a * b for a, b in zip(xs, r)) % R and ok.value == 1
        hs.hs_g16_weighted_sum(None, rr, ctypes.c_size_t(n), ctypes.c_size_t(threads), out, ctypes.byref(ok))
        assert w.b_fp(out.raw) == sum(r) % R and ok.value == 1
        for bad in (R, R + 1, MONT - 1):
            xb = list(xs)
            xb[n // 2] = bad
            hs.hs_g16_weighted_sum(b"".join(v.to_bytes(32, "little") for v in xb), rr, ctypes.c_size_t(n),
                                   ctypes.c_size_t(threads), out, ctypes.byref(ok))
            assert ok.value == 0, bad
