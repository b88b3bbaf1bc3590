"""GPU tier (-m gpu): fixed-base multiplication by the G1 and G2 generators (g1/g2_mul_generator_batch and their `_dev`
forms) against the variable-base ladder on the repeated generator, byte for byte, outputs and infinity flags together;
argument rules, the lazy table build, streams, the multi-device context, the C oracle, KeyPair.generate and the C++
mirror."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w

pytestmark = pytest.mark.gpu

R = o.R_ORDER
GROUPS = {"g1": (64, w.g1_b(o.G1_GEN)), "g2": (128, w.g2_b(o.G2_GEN))}
EDGES = [0, 1, 2, R - 1, R, R + 1] + [m * R for m in range(2, 6)] + [o.P - 1, o.P, (1 << 256) - 1] + \
    [int.from_bytes(bytes([b]) * 32, "little") for b in (0x80, 0x7F, 0xFF)]


@pytest.fixture(scope="module")
def eng():
    import sylow_b200

    e = sylow_b200.Engine(0)
    yield e
    e.close()


def _scalars(n, seed):
    """n random 256-bit scalars with the edge scalars first, in the middle and last (cyclically for small n)."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    edges = np.frombuffer(b"".join(w.fp_b(e) for e in EDGES), np.uint8).reshape(-1, 32)
    m = len(edges)
    if n < 3 * m:
        k[:] = edges[np.arange(n) % m]
    else:
        k[:m] = edges
        k[n // 2: n // 2 + m] = edges
        k[n - m:] = edges
    return k


def _ladder(eng, g, k):
    width, gen = GROUPS[g]
    pts = np.tile(np.frombuffer(gen, np.uint8), (k.shape[0], 1))
    return getattr(eng, g + "_mul_batch")(pts, k)


@pytest.mark.parametrize("g", ["g1", "g2"])
@pytest.mark.parametrize("n", [1, 7, 32767, 32768, (1 << 16) + 3])
def test_matches_ladder_on_repeated_generator(eng, g, n):
    """Straddles SY_AFF_MIN_BATCH (32 768): below it each thread converts its own point, from it
    k_g*_batch_affine does."""
    k = _scalars(n, n)
    out, inf = getattr(eng, g + "_mul_generator_batch")(k)
    ref, ref_inf = _ladder(eng, g, k)
    assert (out == ref).all() and (inf == ref_inf).all()
    assert inf[: len(EDGES)].tolist()[:11] == [1, 0, 0, 0, 1, 0, 1, 1, 1, 1, 0][: min(n, 11)]


@pytest.mark.parametrize("g", ["g1", "g2"])
def test_argument_rules(eng, g):
    import sylow_b200._lib as L

    width = GROUPS[g][0]
    fn = getattr(eng._lib, "sylow_b200_%s_mul_generator_batch" % g)
    k = _scalars(5, 3)
    out = np.zeros((5, width), np.uint8)
    # out_inf = NULL: the same points
    assert fn(eng._h, k.ctypes.data, 5, out.ctypes.data, None) == L.OK
    assert (out == _ladder(eng, g, k)[0]).all()
    # n = 0 returns 0 whatever the pointers; a null scalar or output pointer with n > 0 is ERR_ARG
    assert fn(eng._h, None, 0, None, None) == L.OK
    assert fn(eng._h, None, 5, out.ctypes.data, None) == L.ERR_ARG
    assert fn(eng._h, k.ctypes.data, 5, None, None) == L.ERR_ARG
    assert fn(None, k.ctypes.data, 5, out.ctypes.data, None) == L.ERR_ARG
    dev = getattr(eng._lib, "sylow_b200_%s_mul_generator_batch_dev" % g)
    assert dev(eng._h, None, 0, None, None, None) == L.OK
    assert dev(eng._h, None, 5, out.ctypes.data, None, None) == L.ERR_ARG
    # the existing entry points keep rejecting a null point pointer
    mul = getattr(eng._lib, "sylow_b200_%s_mul_batch" % g)
    assert mul(eng._h, None, None, k.ctypes.data, 5, out.ctypes.data, None) == L.ERR_ARG


def test_first_call_builds_the_table_once():
    """A fresh context builds each table on its first call (ladder + conversion launches), then reuses it."""
    import sylow_b200

    e = sylow_b200.Engine(0)
    try:
        for g in ("g1", "g2"):
            k = _scalars(40, 7)
            ref = _ladder(e, g, k)
            before = e.launch_count
            first = getattr(e, g + "_mul_generator_batch")(k)
            built = e.launch_count - before
            before = e.launch_count
            second = getattr(e, g + "_mul_generator_batch")(k)
            assert e.launch_count - before == 1 and built == 3  # k_g*_mul + k_fp_convert, then k_g*_mul_gen
            for a in (first, second):
                assert (a[0] == ref[0]).all() and (a[1] == ref[1]).all()
    finally:
        e.close()


def test_dev_forms_on_a_torch_stream(eng):
    import torch

    dev = torch.device("cuda", 0)
    n = 40000
    k = _scalars(n, 11)
    st = torch.cuda.Stream(dev)
    for g in ("g1", "g2"):
        width = GROUPS[g][0]
        ref, ref_inf = _ladder(eng, g, k)
        with torch.cuda.stream(st):
            d_k = torch.from_numpy(k).to(dev, non_blocking=False)
            d_out = torch.empty((n, width), dtype=torch.uint8, device=dev)
            d_inf = torch.empty(n, dtype=torch.uint8, device=dev)
            getattr(eng, g + "_mul_generator_batch_dev")(d_k, d_out, d_inf)
            d_out2 = torch.empty((n, width), dtype=torch.uint8, device=dev)
            getattr(eng, g + "_mul_generator_batch_dev")(d_k, d_out2)  # d_out_inf = None
        st.synchronize()
        assert (d_out.cpu().numpy() == ref).all() and (d_inf.cpu().numpy() == ref_inf).all()
        assert (d_out2.cpu().numpy() == ref).all()


def test_multi_device_context():
    """{0, 0}: the host forms shard like g*_mul_batch and give the single context's bytes; `_dev` forms are rejected."""
    import sylow_b200
    import torch
    from sylow_b200._lib import ERR_ARG, SylowB200Error

    single, multi = sylow_b200.Engine(0), sylow_b200.Engine([0, 0])
    try:
        for n in (1, 7, 50, 40001):
            k = _scalars(n, 20 + n)
            for g in ("g1", "g2"):
                a = getattr(single, g + "_mul_generator_batch")(k)
                b = getattr(multi, g + "_mul_generator_batch")(k)
                assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
        dev = torch.device("cuda", 0)
        d_k = torch.from_numpy(_scalars(8, 1)).to(dev)
        for g in ("g1", "g2"):
            with pytest.raises(SylowB200Error) as err:
                getattr(multi, g + "_mul_generator_batch_dev")(d_k, torch.empty((8, GROUPS[g][0]), dtype=torch.uint8,
                                                                              device=dev))
            assert err.value.status == ERR_ARG
    finally:
        single.close()
        multi.close()


def test_sample_against_c_oracle(eng):
    """The C oracle restates the reference, whose scalar is an Fp value (below p), so it is given k mod r: the same group
    element, since k G = (k mod r) G.  Its 256-digit NAF does not cover scalars from 2^255 on."""
    from oracle import c_oracle as c

    k = _scalars(4096, 31)
    idx = np.r_[0:24, 2048:2072, 4072:4096, random.Random(3).sample(range(4096), 64)]
    k_r = np.frombuffer(b"".join(w.fp_b(w.b_fp(bytes(row)) % R) for row in k[idx]), np.uint8).reshape(-1, 32)
    for g in ("g1", "g2"):
        out, inf = getattr(eng, g + "_mul_generator_batch")(k)
        width, gen = GROUPS[g]
        pts = np.tile(np.frombuffer(gen, np.uint8), (len(idx), 1))
        ref, ref_inf = getattr(c, g + "_mul_batch")(pts, k_r)
        assert (out[idx] == ref).all() and (inf[idx] == ref_inf).all()


def test_keypair_generate():
    from sylow_b200 import sylow

    for _ in range(3):
        kp = sylow.KeyPair.generate()
        assert kp.public_key == sylow.G2Affine.generator() * kp.secret_key


def test_cpp_header_generator(tmp_path):
    """include/sylow_b200.hpp: KeyPair::generate's pk from g2_mul_generator_batch equals g2_mul_batch({g2}, {sk})."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_hpp_generator")
    libdir = os.path.join(root, "sylow_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", os.path.join(root, "tests", "cpp", "test_hpp_generator.cpp"),
                           "-o", exe, "-L" + libdir, "-lsylow_b200", "-Wl,-rpath," + libdir, "-pthread"])
    out = subprocess.check_output([exe], text=True).splitlines()
    tag = {l.split()[0]: l.split()[1:] for l in out}
    assert tag["PK"] == ["1"] and tag["G1"] == ["1"] and tag["G2"] == ["1"]
    assert tag["INF"] == ["1", "1"] and tag["MULTI"] == ["1"] and tag["EMPTY"] == ["1"]
