"""CPU tier: the per-thread body of the Miller loops over per-pair G2 tables (csrc/miller_tables.cuh:
miller_tables_item, run by k_miller_tables<M>), compiled for the host from the device source
(tests/hostsim/miller_tables.cu), against oracle.bn254_py.glued_miller_loop for M = 1, 2 and 4 pairs per item."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import bn254_py as o
from tests import wire as w

HERE = os.path.dirname(os.path.abspath(__file__))
R = 1 << 256
ZERO = o.fp12_from_list([0] * 12)


@pytest.fixture(scope="module")
def mt(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("miller_tables") / "libmiller_tables.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "miller_tables.cu")])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def pool():
    """Four G2 points (the generator first) with their oracle tables, and six G1 points (the generator first)."""
    rng = random.Random(87)
    qs = [o.G2_GEN] + [w.rand_g2(rng) for _ in range(3)]
    ps = [o.G1_GEN] + [w.rand_g1(rng) for _ in range(5)]
    return [o.g2_precompute(q) for q in qs], ps


def _device_table(coeffs) -> bytes:
    """The library's device form: 87 triples of Fp2, Montgomery limbs, 192 bytes per triple."""
    return b"".join(w.fp_b(c * R % o.P) for ell in coeffs for fp2 in ell for c in fp2)


def _run(mt, m, tables, ps, item, idx=None, inf=None):
    tb = b"".join(_device_table(t) for t in tables)
    g1 = b"".join(w.g1_b(p) for p in ps)
    idx_a = None if idx is None else (ctypes.c_uint32 * len(idx))(*idx)
    inf_a = None if inf is None else (ctypes.c_uint8 * len(inf))(*inf)
    out = ctypes.create_string_buffer(384)
    mt.hs_miller_tables(ctypes.c_int(m), tb, ctypes.c_size_t(len(tables)), idx_a, g1, inf_a, ctypes.c_size_t(len(ps)),
                        ctypes.c_size_t(item), out)
    return w.b_fp12(out.raw)


def _expect(tables, ps, m, item, idx=None, inf=None):
    ks = range(item * m, item * m + m)
    used = [k for k in ks if not (inf and inf[k])]
    t = [tables[idx[k] if idx else k] for k in used]
    return o.glued_miller_loop(t, [ps[k] for k in used])


@pytest.mark.parametrize("m", [1, 2, 4])
def test_tables_of_generator_and_random_points(mt, pool, m):
    tables, ps = pool
    n = 2 * m  # two items, so that the second one's offsets are exercised
    tabs = [tables[k % 4] for k in range(n)]
    g1 = [ps[k % 6] for k in range(n)]
    for item in range(2):
        assert _run(mt, m, tabs, g1, item) == _expect(tabs, g1, m, item)


@pytest.mark.parametrize("m", [1, 2, 4])
def test_repeated_and_permuted_indices(mt, pool, m):
    tables, ps = pool
    rng = random.Random(m)
    n = 2 * m
    g1 = [ps[rng.randrange(6)] for _ in range(n)]
    for idx in ([3, 0, 2, 1, 1, 3, 0, 0][:n], [rng.randrange(4) for _ in range(n)], [2] * n):
        for item in range(2):
            assert _run(mt, m, tables, g1, item, idx=idx) == _expect(tables, g1, m, item, idx=idx), (idx, item)


@pytest.mark.parametrize("m", [1, 2, 4])
def test_skip_first_and_last_pair(mt, pool, m):
    tables, ps = pool
    g1 = [ps[(k + 1) % 6] for k in range(m)]
    idx = [(k + 2) % 4 for k in range(m)]
    for inf in ([1] + [0] * (m - 1), [0] * (m - 1) + [1], [1] * m):
        got = _run(mt, m, tables, g1, 0, idx=idx, inf=inf)
        assert got == _expect(tables, g1, m, 0, idx=idx, inf=inf), inf
    assert _run(mt, m, tables, g1, 0, idx=idx, inf=[1] * m) == o.FP12_ONE


@pytest.mark.parametrize("m", [1, 2, 4])
def test_out_of_range_index_gives_zero(mt, pool, m):
    tables, ps = pool
    g1 = ps[:m]
    for bad in range(m):
        for v in (4, 5, 0xffffffff):
            idx = [k % 4 for k in range(m)]
            idx[bad] = v
            assert _run(mt, m, tables, g1, 0, idx=idx) == ZERO, (bad, v)
    # a flagged-infinite pair with a bad index still makes the item zero: the index is checked whatever the flag
    idx = [4] + [0] * (m - 1)
    assert _run(mt, m, tables, g1, 0, idx=idx, inf=[1] * m) == ZERO
