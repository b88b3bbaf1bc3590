"""GPU tier (-m gpu): pointwise G1 / G2 addition and subtraction (g1/g2_add_batch and their `_dev` forms) against the
Python oracle across SY_G1/G2_ADD_AFF_MIN_BATCH and against the C oracle's scalar multiplication at 2^16 + 3; group-law
cross-checks at 2^20 / 2^18 points; streams, the multi-device context and the argument rules; the EIP-196 ecAdd / ecMul
bodies against the pinned vectors, failed inputs and the equivalent composition of existing entry points; the sylow.py
operators and the C++ mirror."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = o.R_ORDER
GROUPS = {"g1": (64, o.FpOps), "g2": (128, o.Fp2Ops)}
ERR_DECODE, ERR_NOT_ON_CURVE = -6, -3


def _threshold(g) -> int:
    src = open(os.path.join(ROOT, "sylow_b200", "csrc", "sylow_b200.cu")).read()
    return int(re.search(r"#define SY_%s_ADD_AFF_MIN_BATCH (\d+)" % g.upper(), src).group(1))


T = {g: _threshold(g) for g in ("g1", "g2")}


@pytest.fixture(scope="module")
def eng():
    import sylow_b200

    e = sylow_b200.Engine(0)
    yield e
    e.close()


def _k(n, seed):
    return np.random.default_rng(seed).integers(0, 256, size=(n, 32), dtype=np.uint8)


def _operands(eng, g, n, seed):
    """a, b = random multiples of the generator with infinity flags mixed in, b[i] = a[i] at every 5th item and
    b[i] = -a[i] at every 7th."""
    width, _ = GROUPS[g]
    a, _ = getattr(eng, g + "_mul_generator_batch")(_k(n, seed))
    b, _ = getattr(eng, g + "_mul_generator_batch")(_k(n, seed + 1))
    rng = np.random.default_rng(seed + 2)
    same, opp = np.arange(0, n, 5), np.arange(3, n, 7)
    b[same] = a[same]
    neg, _ = getattr(eng, g + "_mul_batch")(a[opp], np.tile(np.frombuffer(w.fp_b(R - 1), np.uint8), (len(opp), 1)))
    b[opp] = neg
    a_inf = (rng.random(n) < 0.1).astype(np.uint8)
    b_inf = (rng.random(n) < 0.1).astype(np.uint8)
    return a, b, a_inf, b_inf


def _pt(g, row, inf):
    F = GROUPS[g][1]
    return o.proj_to_affine(F, o.proj_zero(F)) if inf else (w.b_g1 if g == "g1" else w.b_g2)(bytes(row), False)


def _oracle(g, a, b, sub):
    F = GROUPS[g][1]
    if sub:
        b = o.g1_affine_neg(b) if g == "g1" else o.g2_affine_neg(b)
    return o.proj_to_affine(F, o.proj_add(F, o.affine_to_proj(F, a), o.affine_to_proj(F, b)))


def _read(g, row, inf):
    return (w.b_g1 if g == "g1" else w.b_g2)(bytes(row), inf)


@pytest.mark.parametrize("g", ["g1", "g2"])
@pytest.mark.parametrize("dn", [None, 7, -1, 0, 5], ids=["1", "7", "T-1", "T", "T+5"])
@pytest.mark.parametrize("sub", [False, True], ids=["add", "sub"])
def test_against_python_oracle(eng, g, dn, sub):
    """n = 1, 7 and around SY_G*_ADD_AFF_MIN_BATCH = T: below it each thread converts its own point, from it
    k_g*_batch_affine does."""
    n = 1 if dn is None else dn if dn == 7 else T[g] + dn
    a, b, ai, bi = _operands(eng, g, n, 100 + n)
    out, inf = getattr(eng, g + "_add_batch")(a, b, ai, bi, subtract=sub)
    for i in range(n):
        exp = _oracle(g, _pt(g, a[i], ai[i]), _pt(g, b[i], bi[i]), sub)
        assert _read(g, out[i], inf[i]) == exp, i


@pytest.mark.parametrize("g", ["g1", "g2"])
@pytest.mark.parametrize("sub", [False, True], ids=["add", "sub"])
def test_against_c_oracle(eng, g, sub):
    """n = 2^16 + 3: a = k1 P, b = k2 P by the C oracle's scalar multiplication, so a +- b = (k1 +- k2) P by the same;
    infinite operands are flagged at random and their scalar taken as 0."""
    from oracle import c_oracle as c

    n = (1 << 16) + 3
    width, _ = GROUPS[g]
    rng = np.random.default_rng(7 + sub)
    p, _ = getattr(eng, g + "_mul_generator_batch")(_k(n, 5))
    k1 = [int(x) for x in rng.integers(0, 1 << 62, n)]
    k2 = [int(x) for x in rng.integers(0, 1 << 62, n)]
    for i in range(0, n, 11):
        k2[i] = k1[i]
    ai = (rng.random(n) < 0.05).astype(np.uint8)
    bi = (rng.random(n) < 0.05).astype(np.uint8)
    k1 = [0 if ai[i] else k1[i] for i in range(n)]
    k2 = [0 if bi[i] else k2[i] for i in range(n)]
    mul = getattr(c, g + "_mul_batch")
    enc = lambda ks: np.frombuffer(b"".join(w.fp_b(k % R) for k in ks), np.uint8).reshape(-1, 32)
    a, _ = mul(p, enc(k1))
    b, _ = mul(p, enc(k2))
    ref, ref_inf = mul(p, enc([x - y if sub else x + y for x, y in zip(k1, k2)]))
    out, inf = getattr(eng, g + "_add_batch")(a, b, ai, bi, subtract=sub)
    assert (out == ref).all() and (inf == ref_inf).all()


@pytest.mark.parametrize("g,lg", [("g1", 20), ("g2", 18)])
def test_group_law_cross_checks(eng, g, lg):
    n = 1 << lg
    width, _ = GROUPS[g]
    k1, k2 = _k(n, 40), _k(n, 41)
    a, a_inf = getattr(eng, g + "_mul_generator_batch")(k1)
    two = np.tile(np.frombuffer(w.fp_b(2), np.uint8), (n, 1))
    dbl, dbl_inf = getattr(eng, g + "_mul_batch")(a, two)
    s, s_inf = getattr(eng, g + "_add_batch")(a, a)
    assert (s == dbl).all() and (s_inf == dbl_inf).all()                     # a + a == 2 a
    z, z_inf = getattr(eng, g + "_add_batch")(a, a, subtract=True)
    assert z_inf.all()                                                         # a - a == O
    b, _ = getattr(eng, g + "_mul_generator_batch")(k2)
    ksum = [(w.b_fp(bytes(x)) + w.b_fp(bytes(y))) % R for x, y in zip(k1, k2)]
    kk = np.frombuffer(b"".join(w.fp_b(k) for k in ksum), np.uint8).reshape(-1, 32)
    ref, ref_inf = getattr(eng, g + "_mul_generator_batch")(kk)
    s, s_inf = getattr(eng, g + "_add_batch")(a, b)
    assert (s == ref).all() and (s_inf == ref_inf).all()                     # k1 G + k2 G == (k1 + k2) G


def test_dev_forms_on_a_torch_stream(eng):
    import torch

    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(dev)
    for g in ("g1", "g2"):
        width, _ = GROUPS[g]
        for n in (T[g] - 3, T[g] + 1):
            a, b, ai, bi = _operands(eng, g, n, 60 + n)
            for sub in (False, True):
                ref, ref_inf = getattr(eng, g + "_add_batch")(a, b, ai, bi, subtract=sub)
                with torch.cuda.stream(st):
                    t = [torch.from_numpy(x).to(dev) for x in (a, b, ai, bi)]
                    d_out = torch.empty((n, width), dtype=torch.uint8, device=dev)
                    d_inf = torch.empty(n, dtype=torch.uint8, device=dev)
                    getattr(eng, g + "_add_batch_dev")(t[0], t[1], d_out, d_inf, t[2], t[3], subtract=sub)
                    d_out2 = torch.empty((n, width), dtype=torch.uint8, device=dev)
                    getattr(eng, g + "_add_batch_dev")(t[0], t[1], d_out2, None, t[2], t[3], subtract=sub)
                st.synchronize()
                assert (d_out.cpu().numpy() == ref).all() and (d_inf.cpu().numpy() == ref_inf).all()
                assert (d_out2.cpu().numpy() == ref).all()


def test_multi_device_context(eng):
    """{0, 0}: the host forms shard over the slots and give the single context's bytes; `_dev` forms are rejected."""
    import sylow_b200
    import torch
    from sylow_b200._lib import ERR_ARG, SylowB200Error

    multi = sylow_b200.Engine([0, 0])
    try:
        for n in (1, 7, 50, T["g2"] + 1):
            for g in ("g1", "g2"):
                a, b, ai, bi = _operands(eng, g, n, 80 + n)
                x = getattr(eng, g + "_add_batch")(a, b, ai, bi, subtract=n & 1)
                y = getattr(multi, g + "_add_batch")(a, b, ai, bi, subtract=n & 1)
                assert (x[0] == y[0]).all() and (x[1] == y[1]).all()
        inp = _mul_inputs(eng, 1001, 3)
        for name in ("eip196_add_batch", "eip196_mul_batch"):
            data = _add_inputs(eng, 1001, 4) if name == "eip196_add_batch" else inp
            x, y = getattr(eng, name)(data), getattr(multi, name)(data)
            assert (x[0] == y[0]).all() and (x[1] == y[1]).all()
        dev = torch.device("cuda", 0)
        d = torch.zeros((8, 64), dtype=torch.uint8, device=dev)
        with pytest.raises(SylowB200Error) as err:
            multi.g1_add_batch_dev(d, d, torch.empty_like(d))
        assert err.value.status == ERR_ARG
    finally:
        multi.close()


@pytest.mark.parametrize("g", ["g1", "g2"])
def test_argument_rules(eng, g):
    from sylow_b200 import _lib as L

    width, _ = GROUPS[g]
    a = np.zeros((5, width), np.uint8)
    out = np.empty((5, width), np.uint8)
    fn = getattr(eng._lib, "sylow_b200_%s_add_batch" % g)
    assert fn(eng._h, None, None, None, None, 0, 0, None, None) == L.OK
    assert fn(eng._h, None, None, a.ctypes.data, None, 5, 0, out.ctypes.data, None) == L.ERR_ARG
    assert fn(eng._h, a.ctypes.data, None, None, None, 5, 0, out.ctypes.data, None) == L.ERR_ARG
    assert fn(eng._h, a.ctypes.data, None, a.ctypes.data, None, 5, 0, None, None) == L.ERR_ARG
    assert fn(None, a.ctypes.data, None, a.ctypes.data, None, 5, 0, out.ctypes.data, None) == L.ERR_ARG
    dev = getattr(eng._lib, "sylow_b200_%s_add_batch_dev" % g)
    assert dev(eng._h, None, None, None, None, 0, 0, None, None, None) == L.OK
    assert dev(eng._h, None, None, None, None, 5, 0, out.ctypes.data, None, None) == L.ERR_ARG
    # out_inf may be null; the Python form checks row counts before the call
    assert fn(eng._h, a.ctypes.data, None, a.ctypes.data, None, 5, 1, out.ctypes.data, None) == L.OK
    with pytest.raises(ValueError):
        getattr(eng, g + "_add_batch")(a, a[:4])
    with pytest.raises(ValueError):
        getattr(eng, g + "_add_batch")(a, a, a_inf=np.zeros(4, np.uint8))
    for name, wd in (("eip196_add_batch", 128), ("eip196_mul_batch", 96)):
        f = getattr(eng._lib, "sylow_b200_" + name)
        buf = np.zeros((5, wd), np.uint8)
        st = np.empty(5, np.int8)
        assert f(eng._h, None, 0, None, None) == L.OK
        assert f(eng._h, None, 5, out.ctypes.data, st.ctypes.data) == L.ERR_ARG
        assert f(eng._h, buf.ctypes.data, 5, None, st.ctypes.data) == L.ERR_ARG
        assert f(eng._h, buf.ctypes.data, 5, out.ctypes.data, None) == L.ERR_ARG
        with pytest.raises(ValueError):
            getattr(eng, name)(np.zeros((5, wd - 1), np.uint8))


# ---------------------------------------------------------------------------------------------- EIP-196
def _be(*vals) -> bytes:
    return b"".join(int(v).to_bytes(32, "big") for v in vals)


def _rows(bs):
    return np.frombuffer(b"".join(bs), np.uint8).reshape(len(bs), -1).copy()


def test_eip196_kats(eng, kats):
    out, st = eng.eip196_add_batch(_rows([bytes.fromhex(kats["eip196_add"]["input"])]))
    assert st[0] == 0 and bytes(out[0]).hex() == kats["eip196_add"]["expected"]
    out, st = eng.eip196_mul_batch(_rows([bytes.fromhex(kats["eip196_mul"]["input"])]))
    assert st[0] == 0 and bytes(out[0]).hex() == kats["eip196_mul"]["expected"]


BAD = [((o.P, 2), ERR_DECODE), ((1, o.P), ERR_DECODE), ((0x31 << 248, 2), ERR_DECODE), ((1, 3), ERR_NOT_ON_CURVE),
       ((0, 1), ERR_NOT_ON_CURVE)]


def test_eip196_failed_inputs(eng):
    g = (1, 2)
    add_in, add_st, mul_in, mul_st = [], [], [], []
    for pt, status in BAD:
        add_in += [_be(*pt, *g), _be(*g, *pt)]
        add_st += [status, status]
        mul_in.append(_be(*pt, 5))
        mul_st.append(status)
    add_in.append(_be(*BAD[0][0], *BAD[3][0]))  # two failures: the first point's status
    add_st.append(ERR_DECODE)
    add_in.append(bytes(128))  # (0,0) + (0,0)
    add_st.append(0)
    out, st = eng.eip196_add_batch(_rows(add_in))
    assert list(st) == add_st and not out.any()
    out, st = eng.eip196_mul_batch(_rows(mul_in))
    assert list(st) == mul_st and not out.any()


def test_eip196_mul_edge_scalars(eng):
    p = w.rand_g1(__import__("random").Random(5))
    ks = [0, 1, R, R + 1, (1 << 256) - 1]
    rows = [_be(p[0], p[1], k) for k in ks] + [bytes(64) + _be(k) for k in ks]
    out, st = eng.eip196_mul_batch(_rows(rows))
    assert not st.any()
    for i, k in enumerate(ks):
        q = o.proj_to_affine(o.FpOps, o.proj_mul(o.FpOps, o.affine_to_proj(o.FpOps, p), k % R))
        assert bytes(out[i]) == (bytes(64) if q[2] else _be(q[0], q[1])), k
    assert not out[len(ks):].any()  # k O = O


def _mul_inputs(eng, n, seed):
    """valid points (a few infinite, a few invalid) || random 256-bit big-endian scalars"""
    pts, _ = eng.g1_mul_generator_batch(_k(n, seed))
    be = eng.g1_to_be_bytes_batch(pts, scrubbed=True)
    be[::97] = 0
    be[5::101, 63] ^= 1  # off the curve
    return np.concatenate([be, _k(n, seed + 1)], axis=1)


def _add_inputs(eng, n, seed):
    a = _mul_inputs(eng, n, seed)[:, :64]
    b = _mul_inputs(eng, n, seed + 7)[:, :64]
    b[::13] = a[::13]
    return np.concatenate([a, b], axis=1)


def test_eip196_mul_matches_composition(eng):
    """2^16 inputs: byte-equal to g1_from_be_bytes_batch -> g1_mul_batch -> g1_to_be_bytes_batch(scrubbed), with
    failed inputs zeroed."""
    n = 1 << 16
    inp = _mul_inputs(eng, n, 300)
    out, st = eng.eip196_mul_batch(inp)
    pts, inf, st_ref = eng.g1_from_be_bytes_batch(inp[:, :64], eip_mode=True)
    m, m_inf = eng.g1_mul_batch(pts, np.ascontiguousarray(inp[:, 64:][:, ::-1]), inf)
    ref = eng.g1_to_be_bytes_batch(m, m_inf, scrubbed=True)
    ref[st_ref != 0] = 0
    assert (st == st_ref).all() and (st != 0).any() and (out == ref).all()


def test_eip196_add_matches_composition(eng):
    n = 1 << 16
    inp = _add_inputs(eng, n, 400)
    out, st = eng.eip196_add_batch(inp)
    pa, ia, sa = eng.g1_from_be_bytes_batch(inp[:, :64], eip_mode=True)
    pb, ib, sb = eng.g1_from_be_bytes_batch(inp[:, 64:], eip_mode=True)
    s, s_inf = eng.g1_add_batch(pa, pb, ia, ib)
    ref = eng.g1_to_be_bytes_batch(s, s_inf, scrubbed=True)
    st_ref = np.where(sa != 0, sa, sb)
    ref[st_ref != 0] = 0
    assert (st == st_ref).all() and (st != 0).any() and (out == ref).all()


# ---------------------------------------------------------------------------------------------- bindings
def test_sylow_operators():
    import random

    from sylow_b200 import sylow

    rng = random.Random(12)
    for _ in range(3):
        p, q = w.rand_g1(rng), w.rand_g1(rng)
        a, b = sylow.G1Affine(p[0], p[1], False), sylow.G1Affine(q[0], q[1], False)
        s, d = a + b, a - b
        assert (s.x, s.y, s.infinity) == _oracle("g1", p, q, False)
        assert (d.x, d.y, d.infinity) == _oracle("g1", p, q, True)
        assert (a - a).is_zero() and a + sylow.G1Affine.zero() == a and a + a == a * 2
        p2, q2 = w.rand_g2(rng), w.rand_g2(rng)
        a2, b2 = sylow.G2Affine(p2[0], p2[1], False), sylow.G2Affine(q2[0], q2[1], False)
        s2, d2 = a2 + b2, a2 - b2
        assert (s2.x, s2.y, s2.infinity) == _oracle("g2", p2, q2, False)
        assert (d2.x, d2.y, d2.infinity) == _oracle("g2", p2, q2, True)
        assert (a2 - a2).is_zero() and sylow.G2Affine.zero() - a2 == -a2


def test_cpp_header_group_law(tmp_path):
    """include/sylow_b200.hpp: g1_add_batch / g2_add_batch against g*_mul_batch, and a two-slot MultiEngine."""
    exe = str(tmp_path / "test_hpp_group_law")
    libdir = os.path.join(ROOT, "sylow_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "test_hpp_group_law.cpp"),
                           "-o", exe, "-L" + libdir, "-lsylow_b200", "-Wl,-rpath," + libdir, "-pthread"])
    out = subprocess.check_output([exe], text=True).splitlines()
    tag = {l.split()[0]: l.split()[1:] for l in out}
    assert tag["G1"] == ["1"] and tag["G2"] == ["1"] and tag["INF"] == ["1"] and tag["MULTI"] == ["1"]
